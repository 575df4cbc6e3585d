"""One MLP forward+backward at the config-2 mini-batch size (for ncu per-kernel timing) + event timing."""
import sys, torch
sys.path.insert(0, '.')
from rlinf_b200.policy import MLPPolicy
n = int(sys.argv[1]) if len(sys.argv) > 1 else 262144
pol = MLPPolicy(obs_dim=128, action_dim=8, seed=0)
states = torch.randn(n, 128, device='cuda'); action = torch.randn(n, 8, device='cuda')
dl = torch.randn(n, 8, device='cuda') / n; dv = torch.randn(n, 1, device='cuda') / n
for _ in range(2):
    out = pol.forward_train(states, action, compute_entropy=False); pol.backward(dl, dv, None)
torch.cuda.synchronize()
e = [torch.cuda.Event(enable_timing=True) for _ in range(3)]
e[0].record(); out = pol.forward_train(states, action, compute_entropy=False); e[1].record(); pol.backward(dl, dv, None); e[2].record()
torch.cuda.synchronize()
print(f"n={n}: fwd {e[0].elapsed_time(e[1]):.3f} ms  bwd {e[1].elapsed_time(e[2]):.3f} ms", flush=True)
