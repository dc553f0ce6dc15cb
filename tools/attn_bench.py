"""Time the flash attention kernel (CUDA events).  python tools/attn_bench.py B L D [iters]"""
import os, sys
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import torch
import b200dm
from b200dm import ops, _lib

B, L, D = [int(v) for v in sys.argv[1:4]]
iters = int(sys.argv[4]) if len(sys.argv) > 4 else 10
dev = torch.device("cuda", 0)
q = torch.randn(B, L, D, device=dev).to(_lib.ACT_DTYPE)
k = torch.randn(B, L, D, device=dev).to(_lib.ACT_DTYPE)
vt = torch.randn(B, D, L, device=dev).to(_lib.ACT_DTYPE)
o = torch.empty_like(q)
plan = ops.AttnPlan(q, k, vt, o, D ** -0.5)
for _ in range(3):
    plan.run()
torch.cuda.synchronize()
assert _lib.debug_flag() == 0
e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
e0.record()
for _ in range(iters):
    plan.run()
e1.record()
torch.cuda.synchronize()
ms = e0.elapsed_time(e1) / iters
print(f"flash attention B{B} L{L} D{D}: {ms*1e3:.1f} us  {plan.flops/ms/1e9:.1f} TFLOP/s (4*B*L^2*D)")
