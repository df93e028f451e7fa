"""W1 microbench timing (configs[3]): tensor-pipe vs SIMT kernel, bf16 storage."""
import sys, os
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT); sys.path.insert(0, os.path.join(ROOT, "tests"))
import torch, common
common.package()
from dgtd_b200.twig.ops.functions import texture_diffusion_func as OP
S, C = 1024, 256
g = torch.Generator().manual_seed(0)
x = torch.randn(1, S, S, C, generator=g).cuda()
wgt = torch.rand(1, 49, S, S, generator=g).cuda()
xb = x.to(torch.bfloat16)
def t(fn, n=5):
    for _ in range(2): fn()
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    torch.cuda.synchronize(); a.record()
    for _ in range(n): fn()
    b.record(); torch.cuda.synchronize()
    return a.elapsed_time(b) / n
for impl in sys.argv[1:] or ["tc", "simt"]:
    for T in (1, 4):
        ms = t(lambda: OP.message_passing_tiled(xb, wgt, T, impl=impl))
        nbytes = (2 * C * 2 + 49 * 4) * S * S
        print(f"bf16 {impl} T={T}: {ms:.4f} ms  per-step {ms / T:.4f} ms  {nbytes * T / ms / 1e6:.0f} GB/s  hbm_frac {nbytes * T / ms / 1e6 / 6549:.3f}")
for impl in ("tc", "simt"):
    for T in (1, 4):
        ms = t(lambda: OP.message_passing_tiled(x, wgt, T, impl=impl))
        nbytes = (2 * C * 4 + 49 * 4) * S * S
        print(f"fp32 {impl} T={T}: {ms:.4f} ms  per-step {ms / T:.4f} ms  {nbytes * T / ms / 1e6:.0f} GB/s  hbm_frac {nbytes * T / ms / 1e6 / 6549:.3f}")
