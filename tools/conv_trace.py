"""Per-role clock64 timeline of CTA 0 of the halo conv kernel (tuning aid, GPU box)."""
import os, sys
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import ctypes as C
import torch
import b200dm
from b200dm import ops, _lib

a = [int(v) for v in sys.argv[1:]]
B, D, H, W, c0, c1, cout = a[:7]
dev = torch.device("cuda", 0)
w = torch.randn(3, 3, 3, c0 + c1, cout) * 0.05
desc = ops.make_conv_desc(0, B, (D, H, W), c0, c1, cout, 3, 1)
wp = ops.pack_conv_weights(desc, w).to(dev)
x0 = torch.randn(B, D, H, W, c0, device=dev).bfloat16()
x1 = torch.randn(B, D, H, W, c1, device=dev).bfloat16() if c1 else None
y = torch.empty(B, D, H, W, cout, device=dev, dtype=torch.bfloat16)
kw = {}
if os.environ.get("EPI") == "1":     # the ResidualBlock conv1 form: + temb row (device-side t), folded norm2, swish
    desc = ops.make_conv_desc(0, B, (D, H, W), c0, c1, cout, 3, 1, "silu", None, torch.bfloat16, chan_bias_rows=1)
    kw = dict(chan_bias=torch.randn(1000, cout, device=dev), t_dev=torch.tensor([500, 499, 0, 0], dtype=torch.int32, device=dev),
              out_affine=(torch.rand(cout, device=dev) + 0.5, torch.randn(cout, device=dev) * 0.1))
if os.environ.get("RES") == "1":     # the conv2 form: + residual
    kw = dict(residual=torch.randn(B, D, H, W, cout, device=dev).bfloat16())
if os.environ.get("F32") == "1" or os.environ.get("FUSE"):   # the U-Net's output conv: fp32 eps
    desc = ops.make_conv_desc(0, B, (D, H, W), c0, c1, cout, 3, 1, None, None, torch.float32)
    y = torch.empty(B, D, H, W, cout, device=dev, dtype=torch.float32)
plan = ops.ConvPlan(desc, x0, wp, y, x1=x1, bias=torch.zeros(cout, device=dev), **kw)
if os.environ.get("FUSE"):           # ... with the reverse-diffusion update in its epilogue (FUSE=ddpm|ddim)
    betas = b200dm.Betas(1000).to(dev)
    xt = torch.randn(B, D, H, W, cout, device=dev)
    xb = torch.empty(B, D, H, W, cout, device=dev, dtype=torch.bfloat16)
    ud = ops.make_update_desc(betas, xt[0].numel(), B, 500, 499, 1 if os.environ["FUSE"] == "ddim" else 0, 7, 0, _lib.F32)
    assert plan.set_fused_update(ud, xt, xt, xb)
for _ in range(3):
    plan.run()
tr = torch.zeros(4 * 2048, dtype=torch.int64, device=dev)
_lib.check(_lib.lib().b200dm_conv_plan_set_trace(plan.h, C.c_void_p(tr.data_ptr())))
plan.run()
torch.cuda.synchronize()
t = tr.cpu().view(4, 2048)
names = {1: "tile:begin", 2: "tile:tmem_empty ok", 3: "kd:slabs ready", 4: "kd:issued", 5: "b?", 6: "b:waited", 7: "b:pre", 10: "epi:wait", 11: "epi:tmem_full ok", 12: "epi:done", 13: "epi:buf free", 14: "epi:tile written", 15: "epi:synced", 16: "epi:acc in regs", 17: "epi:half done", 18: "epi:loop top", 19: "epi:tile decoded", 20: "epi:bias staged"}
t0 = min(int(v) >> 8 for v in t[0] if int(v) != 0)
names.update({30: "tail:roles done", 31: "tail:block synced", 32: "tail:cluster synced"})
for region, label in ((0, "MMA"), (1, "EPI"), (2, "SLAB"), (3, "TAIL")):
    prev = None
    out = []
    for v in t[region]:
        v = int(v)
        if v == 0:
            break
        clk, tag = (v >> 8) - t0, v & 0xff
        out.append(f"{names.get(tag, 'slab'+str(tag-20))}@{clk}" + (f"(+{clk-prev})" if prev is not None else ""))
        prev = clk
    print(label, len(out))
    for i in range(0, min(len(out), int(os.environ.get('NEV', '60'))), 6):
        print("   ", "  ".join(out[i:i + 6]))
