"""Time the d-sweeping 32 -> 32 conv kernel at the cfg-3 shape (B=16, 128^3) in three configurations (GPU box):
plain | + GroupNorm partial sums in the epilogue | both + residual."""
import os, sys
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import torch
import b200dm
from b200dm import ops, _lib as L

B, S = (int(sys.argv[1]) if len(sys.argv) > 1 else 16), (int(sys.argv[2]) if len(sys.argv) > 2 else 128)
dev = torch.device("cuda", 0)
x = torch.randn(B, S, S, S, 32, device=dev).to(L.ACT_DTYPE)
res = torch.randn(B, S, S, S, 32, device=dev).to(L.ACT_DTYPE)
w = torch.randn(3, 3, 3, 32, 32) * 0.03
desc = ops.make_conv_desc(L.CONV_DIRECT, B, (S, S, S), 32, 0, 32, 3, 1, None, None)
wp = ops.pack_conv_weights(desc, w, False).to(dev)
bias = torch.zeros(32, device=dev)


def timed(plan, n=5):
    for _ in range(2):
        plan.run()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(n):
        plan.run()
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) / n


for name, gn, rs in (("plain", 0, 0), ("gn partials", 1, 0), ("gn partials + residual", 1, 1)):
    y = torch.empty_like(x)
    plan = ops.ConvPlan(desc, x, wp, y, bias=bias, residual=res if rs else None)
    assert plan.info["halo"] == 3
    if gn:
        plan.gn_partials()
    ms = timed(plan)
    fl = 2.0 * 27 * 32 * 32 * B * S ** 3
    print(f"{name:22s} {ms:7.3f} ms  {fl / ms / 1e9:7.1f} TFLOP/s   flag {L.debug_flag()}")
