"""INTEGRATION.md's install() against the reference's registries, as recorded from the unmodified reference in
tests/golden/golden_install.npz (tests/golden/make_golden_install.py).  The checks: install() replaces every entry the
reference registers and accepts every parameter its callables name with the same defaults; the kwargs the reference's
own dispatchers (`calculate_adv_and_returns`, `policy_loss`, registry.py:77-124) hand the registered callable, for the
kwargs its workers build, reach the replacement without a TypeError / KeyError, and without a GPU the replacement then
refuses to compute on the host (Rb200Error) instead of falling back."""
import inspect
import json

import numpy as np
import pytest
import torch


def _meta(g):
    return json.loads(str(g["install_json"]))


@pytest.fixture()
def installed(golden):
    g = golden("install")
    meta = _meta(g)

    def stand_ins(names):
        return {name: (lambda name=name: name) for name in names}

    regs = {key: stand_ins(meta["registries"][key]) for key in ("adv", "loss", "loss_scale")}
    saved = tuple(dict(regs[key]) for key in ("adv", "loss", "loss_scale"))
    import rlinf_b200.plugin as plugin

    done = plugin.install(regs["adv"], regs["loss"], regs["loss_scale"])
    return regs, saved, done, g, meta


def test_install_replaces_every_reference_entry(installed):
    regs, saved, done, _, meta = installed
    import rlinf_b200.algorithms as A

    assert sorted(done["adv"]) == sorted(saved[0]) == sorted(A.ADV_REGISTRY)
    assert sorted(done["loss"]) == sorted(saved[1]) == sorted(A.LOSS_REGISTRY)
    assert sorted(done["loss_scale"]) == sorted(saved[2]) == sorted(A.LOSS_SCALE_REGISTRY)
    for name, fn in regs["adv"].items():
        assert fn is A.ADV_REGISTRY[name]
    # signature compatibility: every parameter the reference callable names is accepted by the replacement
    for key, new_reg in (("adv", A.ADV_REGISTRY), ("loss", A.LOSS_REGISTRY)):
        for name, old_params in meta["signatures"][key].items():
            new_sig = inspect.signature(new_reg[name])
            new_kw = any(p.kind is inspect.Parameter.VAR_KEYWORD for p in new_sig.parameters.values())
            for p in old_params:
                pname, default = p["name"], p["default"]
                if p["kind"] in ("VAR_KEYWORD", "VAR_POSITIONAL"):
                    continue
                assert pname in new_sig.parameters or new_kw, (name, pname)
                if pname == "loss_agg_func":
                    continue  # a callable default (masked_mean): the aggregation is selected inside the fused kernel
                assert "callable" not in default, (name, pname)
                if pname in new_sig.parameters and "value" in default:
                    assert new_sig.parameters[pname].default == default["value"], (name, pname)  # same defaults (e.g. A1)


def test_reference_dispatchers_reach_the_cuda_callables(installed):
    regs, _, _, g, meta = installed
    from rlinf_b200._lib import Rb200Error

    if torch.cuda.is_available():
        pytest.skip("checks the refusal to compute without a GPU: on a GPU the call would simply succeed")
    kinds = {(c["kind"], c["name"]) for c in meta["calls"]}
    assert {("adv", t) for t in ("gae", "grpo", "raw", "reinpp")} <= kinds
    assert {("loss", t) for t in ("actor_critic", "actor", "decoupled_actor_critic")} <= kinds
    for i, call in enumerate(meta["calls"]):
        kw = dict(call["scalars"])
        kw.update({k: torch.from_numpy(np.array(g[f"call_{i}__{k}"])) for k in call["tensors"]})
        with pytest.raises(Rb200Error):
            regs[call["kind"]][call["name"]](**kw)


def test_logits_wrappers_are_signature_compatible_with_the_reference(golden):
    """SURVEY 8(f)3 drop-ins: rlinf_b200.ops.compute_logprobs_from_logits / compute_entropy_from_logits take the reference's
    positional and keyword arguments (rlinf/utils/utils.py:454-512) and, without a GPU, refuse to compute on the host."""
    want_params = _meta(golden("install"))["logits_params"]
    from rlinf_b200 import ops
    from rlinf_b200._lib import Rb200Error

    for name in ("compute_logprobs_from_logits", "compute_entropy_from_logits"):
        want = want_params[name]
        got = list(inspect.signature(getattr(ops, name)).parameters)
        assert got == want, (name, got, want)
    if not torch.cuda.is_available():
        logits, target = torch.randn(2, 3, 11), torch.randint(0, 11, (2, 3))
        with pytest.raises((Rb200Error, RuntimeError, AssertionError, OSError)):
            ops.compute_logprobs_from_logits(logits, target, op_type="torch")
