"""The backward pass of the fp16-split tensor-core path gives bit-identical gradients from run to run: its sums over rows
(weight gradients of the GEMMs, bias gradients, the head's weight / bias sums) are stored per CTA / sample chunk and
added in a fixed order, not with float atomics."""
import pytest
import torch


@pytest.mark.gpu
@pytest.mark.parametrize("obs,act,n", [(128, 8, 40000),   # bench shape: register path of the head backward
                                       (32, 12, 5000)])   # act > 8: generic head path
def test_backward_is_bit_reproducible(obs, act, n):
    from rlinf_b200.policy import MLPPolicy

    pol = MLPPolicy(obs_dim=obs, action_dim=act, seed=3)
    g = torch.Generator(device="cuda").manual_seed(0)
    states = torch.randn(n, obs, device="cuda", generator=g)
    action = torch.randn(n, act, device="cuda", generator=g)
    d_lp, d_ent = (torch.randn(n, act, device="cuda", generator=g) for _ in range(2))
    d_v = torch.randn(n, 1, device="cuda", generator=g)
    grads = []
    for _ in range(3):
        pol.forward_train(states, action)
        pol.flat_grads.zero_()
        pol.backward(d_lp, d_v, d_ent)
        grads.append(pol.flat_grads.clone())
    assert torch.isfinite(grads[0]).all() and grads[0].abs().sum() > 0
    for name, seg in pol.named_grads():
        assert seg.abs().sum() > 0, name
    assert torch.equal(grads[0], grads[1]) and torch.equal(grads[0], grads[2])
