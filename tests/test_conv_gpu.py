"""GPU parity: tcgen05 implicit-GEMM conv (all variants) vs the oracle's Keras-semantics conv.

Inputs and weights are representable in the 16-bit storage type, accumulation is fp32 on both sides, so the only
difference on fp32 outputs is summation order: tolerance A * max|y| absolute (A set from the measured spread, 4x margin),
plus U (the storage type's unit roundoff, its largest relative rounding error) per 16-bit rounding on 16-bit outputs.
"""
import numpy as np
import pytest
import torch

from b200dm import _lib
from oracle import ops as O

pytestmark = pytest.mark.gpu

ACT = _lib.ACT_DTYPE
U = 2 ** -8 if _lib.precision() == "bf16" else 2 ** -11   # unit roundoff of the storage type: its largest relative rounding error
A = 2e-5   # fp32 accumulation in another order: measured <= 3.6e-6 of max|y| in either build (B200)


def _r(t):  # storage-representable fp32
    return t.to(ACT).to(torch.float32)


def _rand(shape, seed, scale=1.0):
    g = torch.Generator().manual_seed(seed)
    return _r(torch.randn(shape, generator=g) * scale)


def _close(y, ref, tol=A, what=""):
    y = y.float().cpu()
    err = (y - ref).abs().max().item()
    den = ref.abs().max().item() + 1e-12
    print(f"{what}: rel max err {err / den:.3e} (bound {tol:.3e})")
    assert err <= tol * den, f"{what}: max abs err {err:.4e} vs max|ref| {den:.4e} (rel {err/den:.3e})"


def _check_flag():
    from b200dm import _lib
    torch.cuda.synchronize()
    assert _lib.debug_flag() == 0, "tcgen05/TMA pipeline watchdog fired"


CASES = [
    # B, S, cin, cout
    (2, 8, 64, 64),
    (1, 16, 8, 64),
    (2, 4, 128, 256),
    (1, 16, 32, 32),
    (1, 8, 192, 64),
    (3, 8, 64, 16),
    (1, 32, 64, 64),
]


@pytest.mark.parametrize("B,S,cin,cout", CASES)
def test_conv3_same(cuda, B, S, cin, cout):
    from b200dm import ops
    x = _rand((B, S, S, S, cin), 1)
    w = _rand((3, 3, 3, cin, cout), 2, 1.0 / np.sqrt(27 * cin))
    b = torch.randn(cout, generator=torch.Generator().manual_seed(3))
    ref = O.conv3d(x, w, b)
    y = ops.conv3d(x.to(cuda, ACT), w, bias=b.to(cuda), y_dtype=torch.float32)
    _check_flag()
    _close(y, ref, what=f"conv3 B{B} S{S} {cin}->{cout}")


def test_conv3_bf16_out_and_epilogue(cuda):
    from b200dm import ops
    B, S, cin, cout = 2, 8, 64, 128
    x = _rand((B, S, S, S, cin), 1)
    w = _rand((3, 3, 3, cin, cout), 2, 1.0 / np.sqrt(27 * cin))
    b = torch.randn(cout, generator=torch.Generator().manual_seed(3))
    cbias = torch.randn(B, cout, generator=torch.Generator().manual_seed(4))
    res = _rand((B, S, S, S, cout), 5)
    ref = O.swish(O.conv3d(x, w, b) + cbias[:, None, None, None, :]) + res
    y = ops.conv3d(x.to(cuda, ACT), w, bias=b.to(cuda), chan_bias=cbias.to(cuda), act="silu",
                   residual=res.to(cuda, ACT))
    _check_flag()
    assert y.dtype == ACT
    _close(y, ref, tol=A + U, what="conv3 + bias + temb + silu + residual (16-bit out)")


def test_conv3_pair_slab_tiles(cuda):
    """8 x 8 planes (the U-Net's 8^3 level): pair-slab halo tiles, two K segments, odd depth (ragged last pair)."""
    from b200dm import ops
    for (B, D, c0, c1, cout) in ((2, 8, 256, 256, 256), (1, 5, 64, 0, 64)):
        x0 = _rand((B, D, 8, 8, c0), 1)
        x1 = _rand((B, D, 8, 8, c1), 6) if c1 else None
        w = _rand((3, 3, 3, c0 + c1, cout), 2, 1.0 / np.sqrt(27 * (c0 + c1)))
        b = torch.randn(cout, generator=torch.Generator().manual_seed(3))
        res = _rand((B, D, 8, 8, cout), 5)
        xin = x0 if x1 is None else torch.cat([x0, x1], -1)
        ref = O.conv3d(xin, w, b) + res
        y = ops.conv3d(x0.to(cuda, ACT), w, bias=b.to(cuda), residual=res.to(cuda, ACT),
                       x1=None if x1 is None else x1.to(cuda, ACT))
        _check_flag()
        _close(y, ref, tol=A + U, what=f"pair-slab conv3 B{B} D{D} {c0}+{c1}->{cout}")


def test_conv3_two_segments(cuda):
    from b200dm import ops
    B, S, c0, c1, cout = 2, 8, 64, 32, 64
    x0, x1 = _rand((B, S, S, S, c0), 1), _rand((B, S, S, S, c1), 6)
    w = _rand((3, 3, 3, c0 + c1, cout), 2, 1.0 / np.sqrt(27 * (c0 + c1)))
    ref = O.conv3d(torch.cat([x0, x1], -1), w)
    y = ops.conv3d(x0.to(cuda, ACT), w, x1=x1.to(cuda, ACT), y_dtype=torch.float32)
    _check_flag()
    _close(y, ref, what="conv3 over [x, skip] K-segments")


def test_conv1(cuda):
    from b200dm import ops
    B, S, cin, cout = 2, 8, 96, 64
    x = _rand((B, S, S, S, cin), 1)
    w = _rand((1, 1, 1, cin, cout), 2, 1.0 / np.sqrt(cin))
    ref = torch.relu(O.conv3d(x, w))
    y = ops.conv3d(x.to(cuda, ACT), w, act="relu", y_dtype=torch.float32)
    _check_flag()
    _close(y, ref, what="conv1 + relu")


def test_conv_head_cout1(cuda):
    from b200dm import ops
    B, S, cin = 1, 16, 32
    x = _rand((B, S, S, S, cin), 1)
    w = _rand((3, 3, 3, cin, 1), 2, 1.0 / np.sqrt(27 * cin))
    b = torch.tensor([0.25])
    ref = O.conv3d(x, w, b)
    y = ops.conv3d(x.to(cuda, ACT), w, bias=b.to(cuda), y_dtype=torch.float32)
    _check_flag()
    _close(y, ref, what="conv3 32->1 head")


@pytest.mark.parametrize("S,c", [(8, 64), (16, 128)])
def test_conv3_stride2_tf_same(cuda, S, c):
    """TF 'same' for even input, k=3, s=2 pads (0,1): NOT torch padding=1."""
    from b200dm import ops
    x = _rand((2, S, S, S, c), 1)
    w = _rand((3, 3, 3, c, c), 2, 1.0 / np.sqrt(27 * c))
    ref = O.conv3d(x, w, stride=2)
    y = ops.conv3d(x.to(cuda, ACT), w, stride=2, y_dtype=torch.float32)
    _check_flag()
    assert tuple(y.shape) == tuple(ref.shape)
    _close(y, ref, what="conv3 stride 2")


@pytest.mark.parametrize("S,c", [(4, 64), (8, 128)])
def test_upsample_conv_parity_fold(cuda, S, c):
    from b200dm import ops, _lib
    x = _rand((2, S, S, S, c), 1)
    w = _rand((3, 3, 3, c, c), 2, 1.0 / np.sqrt(27 * c))
    b = torch.randn(c, generator=torch.Generator().manual_seed(3))
    ref = O.conv3d(O.upsample_nearest2(x), w, b)
    y = ops.conv3d(x.to(cuda, ACT), w, bias=b.to(cuda), mode=_lib.CONV_PARITY, y_dtype=torch.float32)
    _check_flag()
    # folded taps are summed in fp32 then rounded to the storage type once: the reference's taps are not; two ulps of a weight
    _close(y, ref, tol=A + 2 * U, what="UpSampling3D(2)+Conv3 as 8 parity sub-convs")


@pytest.mark.parametrize("S,cin,cout", [(4, 128, 64), (8, 64, 32)])
def test_conv_transpose_k4s2(cuda, S, cin, cout):
    from b200dm import ops, _lib
    x = _rand((2, S, S, S, cin), 1)
    w = _rand((4, 4, 4, cout, cin), 2, 1.0 / np.sqrt(8 * cin))
    b = torch.randn(cout, generator=torch.Generator().manual_seed(3))
    ref = O.conv3d_transpose(x, w, b)
    y = ops.conv3d(x.to(cuda, ACT), w, bias=b.to(cuda), mode=_lib.CONV_PARITY, transposed=True, y_dtype=torch.float32)
    _check_flag()
    _close(y, ref, what="Conv3DTranspose k4 s2")


@pytest.mark.parametrize("S,cin,cout,transposed", [(16, 128, 128, False), (16, 64, 64, True), (16, 64, 32, True), (16, 64, 32, False),
                                                   (16, 96, 32, True)])
def test_up_conv_halo_kernel_bf16(cuda, S, cin, cout, transposed):
    """bf16-output x2 up-convolutions on planes that fill the 8 x 16 halo tile run conv_halo_up_kernel (CTA pairs, staged
    TMA stores through the parity maps); C_out = 32 takes the N = 32 tiles with 64-byte staged rows (the decoders' last
    ConvT, vqgan_attn_cp.py:404-412).  Tolerance: one output rounding (U) on top of the fp32 bound."""
    from b200dm import ops, _lib
    x = _rand((2, S, S, S, cin), 1)
    b = torch.randn(cout, generator=torch.Generator().manual_seed(3))
    if transposed:
        w = _rand((4, 4, 4, cout, cin), 2, 1.0 / np.sqrt(8 * cin))
        ref = O.conv3d_transpose(x, w, b)
        tol = A + U
    else:
        w = _rand((3, 3, 3, cin, cout), 2, 1.0 / np.sqrt(27 * cin))
        ref = O.conv3d(O.upsample_nearest2(x), w, b)
        tol = A + 3 * U   # + the folded taps' weight rounding (test_upsample_conv_parity_fold)
    y = ops.conv3d(x.to(cuda, ACT), w, bias=b.to(cuda), mode=_lib.CONV_PARITY, transposed=transposed, y_dtype=ACT)
    _check_flag()
    assert tuple(y.shape) == tuple(ref.shape)
    _close(y, ref, tol=tol, what="x2 up-conv (halo up kernel), bf16 out")


def test_prelu_postact_epilogue(cuda):
    """monai ResUnit tail: relu(x + PReLU(conv(h)))  (vqvae3d_monai.py:233-234), BN folded by the host."""
    from b200dm import ops
    B, S, c = 2, 8, 64
    h, x = _rand((B, S, S, S, c), 1), _rand((B, S, S, S, c), 7)
    w = _rand((3, 3, 3, c, c), 2, 1.0 / np.sqrt(27 * c))
    alpha = _r(torch.rand(S, S, S, c, generator=torch.Generator().manual_seed(8)) * 0.3)
    ref = torch.relu(x + O.prelu(O.conv3d(h, w), alpha))
    y = ops.conv3d(h.to(cuda, ACT), w, prelu_alpha=alpha.to(cuda, ACT),
                   residual=x.to(cuda, ACT), post_act="relu", y_dtype=torch.float32)
    _check_flag()
    _close(y, ref, what="PReLU + residual + ReLU epilogue")


def test_batched_gemm_and_transposed_store(cuda):
    from b200dm import ops, _lib
    B, L, Cc = 2, 512, 256
    q, k = _rand((B, L, Cc), 1), _rand((B, L, Cc), 2)
    s = ops.batched_gemm(q.to(cuda, ACT), k.to(cuda, ACT))
    _check_flag()
    _close(s, torch.einsum("blc,bLc->blL", q, k), what="Q K^T")
    # V^T via a transposed-store 1^3 conv
    x = _rand((B, 8, 8, 8, Cc), 3)
    w = _rand((1, 1, 1, Cc, Cc), 4, 1.0 / 16)
    desc = ops.make_conv_desc(_lib.CONV_DIRECT, B, (8, 8, 8), Cc, 0, Cc, 1, 1, y_dtype=ACT, transposed_store=True)
    wp = ops.pack_conv_weights(desc, w).to(cuda)
    vt = torch.empty(B, Cc, L, dtype=ACT, device=cuda)
    bv = _rand((Cc,), 6)
    plan = ops.ConvPlan(desc, x.to(cuda, ACT), wp, vt, bias=bv.to(cuda))
    plan.run()
    _check_flag()
    ref = (O.conv3d(x, w) + bv).reshape(B, L, Cc).transpose(1, 2)
    _close(vt, ref, tol=A + U, what="transposed store (operand swap)")
    # small volume (tile spans samples): the scalar transposed path
    xs = _rand((B, 4, 4, 4, Cc), 7)
    descs = ops.make_conv_desc(_lib.CONV_DIRECT, B, (4, 4, 4), Cc, 0, Cc, 1, 1, y_dtype=ACT, transposed_store=True)
    vts = torch.empty(B, Cc, 64, dtype=ACT, device=cuda)
    ops.ConvPlan(descs, xs.to(cuda, ACT), ops.pack_conv_weights(descs, w).to(cuda), vts, bias=bv.to(cuda)).run()
    _check_flag()
    _close(vts, (O.conv3d(xs, w) + bv).reshape(B, 64, Cc).transpose(1, 2), tol=A + U, what="transposed store (scalar path)")
    p = _r(torch.softmax(torch.randn(B, L, L, generator=torch.Generator().manual_seed(5)), -1))
    o = ops.batched_gemm(p.to(cuda, ACT), vt)
    _check_flag()
    _close(o, torch.einsum("blL,bcL->blc", p, vt.float().cpu()), what="P V")


HALO_CASES = [
    # B, (D,H,W), c0, c1, cout: each with the automatic kernel choice (use_halo = 0) against the per-tap kernel (use_halo = -1)
    (1, (16, 16, 16), 64, 0, 64),
    (2, (5, 24, 12), 64, 32, 64),      # odd depth, ragged H/W tiles, two K-segments
    (1, (16, 16, 16), 8, 0, 32),       # C_in = 8 (TMA zero-fills the 64-channel chunk)
    (1, (8, 16, 8), 128, 0, 256),      # two N tiles
    (1, (16, 32, 32), 32, 0, 1),       # decoder head, C_out = 1
    (8, (32, 32, 32), 64, 0, 64),      # cfg-2 level-0 shape: TD=2, CTA pairs
    (3, (32, 32, 32), 64, 0, 128),
    (1, (5, 16, 8), 64, 0, 128),       # odd tile count: N = 128 tiles on one CTA (3-tap weight stages x 2)
]


@pytest.mark.parametrize("B,dhw,c0,c1,cout", HALO_CASES)
def test_conv3_halo_kernel(cuda, B, dhw, c0, c1, cout):
    """Persistent halo-reuse kernel (shifted SWIZZLE_128B descriptors over TMA-staged halo slabs) vs the oracle,
    and bit-for-bit against the per-tap kernel (same bf16 products, fp32 accumulation; order may differ)."""
    from b200dm import ops, _lib
    D, H, W = dhw
    x0 = _rand((B, D, H, W, c0), 1)
    x1 = _rand((B, D, H, W, c1), 6) if c1 else None
    cin = c0 + c1
    w = _rand((3, 3, 3, cin, cout), 2, 1.0 / np.sqrt(27 * cin))
    b = torch.randn(cout, generator=torch.Generator().manual_seed(3))
    res = _rand((B, D, H, W, cout), 5)
    xin = torch.cat([x0, x1], -1) if c1 else x0
    big = B * D * H * W * cin * cout > 2e10
    ys = {}
    for m in (0, -1):
        desc = ops.make_conv_desc(_lib.CONV_DIRECT, B, dhw, c0, c1, cout, 3, 1, y_dtype=torch.float32, use_halo=m)
        wp = ops.pack_conv_weights(desc, w).to(cuda)
        y = torch.empty(B, D, H, W, cout, dtype=torch.float32, device=cuda)
        ops.ConvPlan(desc, x0.to(cuda, ACT), wp, y, x1=x1.to(cuda, ACT) if c1 else None,
                     bias=b.to(cuda), residual=res.to(cuda, ACT)).run()
        _check_flag()
        ys[m] = y.cpu()
    d = (ys[0] - ys[-1]).abs().max().item() / ys[-1].abs().max().item()
    print(f"halo vs per-tap kernel: rel max diff {d:.3e}")
    assert d < 2e-5
    if not big:
        ref = O.conv3d(xin, w, b) + res
        _close(ys[0], ref, what=f"halo conv B{B} {dhw} {c0}+{c1}->{cout}")


@pytest.mark.parametrize("B,S,cin,cout,halo", [(2, 8, 64, 128, -1), (1, 16, 64, 64, 0), (2, 16, 32, 96, 0), (4, 4, 64, 64, -1)])
def test_conv_out_affine_fuses_consumer_batchnorm(cuda, B, S, cin, cout, halo):
    """ResidualBlock conv1 -> +temb -> BN(norm2) -> swish (dm3d.py:237-244) in ONE epilogue: the folded BN of the
    consumer is applied to the fp32 accumulator.  (4,4,...) covers tiles that span several samples (per-row temb)."""
    from b200dm import ops
    g = torch.Generator().manual_seed(9)
    x = _rand((B, S, S, S, cin), 1)
    w = _rand((3, 3, 3, cin, cout), 2, 1.0 / np.sqrt(27 * cin))
    b = torch.randn(cout, generator=g)
    temb = torch.randn(B, cout, generator=g)
    gamma, beta = torch.rand(cout, generator=g) + 0.5, torch.randn(cout, generator=g) * 0.1
    mean, var = torch.randn(cout, generator=g) * 0.1, torch.rand(cout, generator=g) + 0.5
    ref = O.swish(O.batchnorm_infer(O.conv3d(x, w, b) + temb[:, None, None, None, :], gamma, beta, mean, var))
    sc, sh = ops.bn_fold(gamma.to(cuda), beta.to(cuda), mean.to(cuda), var.to(cuda), 1e-3)
    y = ops.conv3d(x.to(cuda, ACT), w, bias=b.to(cuda), chan_bias=temb.to(cuda), act="silu", out_affine=(sc, sh),
                   y_dtype=torch.float32, use_halo=halo)
    _check_flag()
    _close(y, ref, what=f"conv3 + temb + BN + swish fused, B{B} S{S} {cin}->{cout}")


@pytest.mark.parametrize("shape", [(2, 9, 13, 40), (1, 16, 16, 16), (1, 3, 8, 32), (2, 33, 24, 70)])
def test_conv3_head_stencil_kernel(cuda, shape):
    """C_in = 32 -> C_out = 1 (vqgan_attn_cp.py:424-427, the decoder's head): the HBM-bound stencil-reduce kernel
    (conv_stencil.cuh) on ragged volumes (partial h / w tiles, several d ranges), fp32 and 16-bit outputs, bias + activation."""
    from b200dm import ops, _lib as L
    B, D, H, W = shape
    x = _rand((B, D, H, W, 32), 1)
    w = _rand((3, 3, 3, 32, 1), 2, 1.0 / np.sqrt(27 * 32))
    b = torch.tensor([0.37])
    ref = O.conv3d(x, w, b)
    xd = x.to(cuda, L.ACT_DTYPE)
    desc = ops.make_conv_desc(L.CONV_DIRECT, B, (D, H, W), 32, 0, 1, 3, 1, None, None, torch.float32)
    y = torch.empty(B, D, H, W, 1, dtype=torch.float32, device=cuda)
    plan = ops.ConvPlan(desc, xd, ops.pack_conv_weights(desc, w, False).to(cuda), y, bias=b.to(cuda))
    assert plan.info["halo"] == 2, "expected the stencil plan"
    plan.run()
    _check_flag()
    _close(y, ref, tol=2e-5, what=f"stencil head {shape} fp32 out")
    # against the tensor-core halo / per-tap path on the same inputs (use_halo = -1 switches the stencil and halo kernels off)
    y2 = ops.conv3d(xd, w, bias=b.to(cuda), y_dtype=torch.float32, use_halo=-1)
    _close(y, y2.float().cpu(), tol=2e-5, what="stencil vs per-tap GEMM kernel")
    y16 = ops.conv3d(xd, w, bias=b.to(cuda), act="silu")
    _check_flag()
    _close(y16, O.swish(ref), tol=A + U, what="stencil head + silu (16-bit out)")


@pytest.mark.parametrize("shape,extras", [((2, 20, 16, 8), False), ((1, 35, 24, 12), True), ((3, 9, 48, 40), True)])
def test_conv3_sweep32_kernel(cuda, shape, extras):
    """C_in = C_out = 32 (the decoders' residual units, vqgan_attn_cp.py:250-276): the d-sweeping kernel -- three kd taps per
    N = 96 MMA into a TMEM ring, weights resident, SWIZZLE_64B slabs -- on ragged volumes (partial h / w tiles, several d ranges,
    ring wrap-around), with bias + output affine + SiLU + residual, and its GroupNorm partial sums against a direct evaluation."""
    from b200dm import ops, _lib as L
    B, D, H, W = shape
    x = _rand((B, D, H, W, 32), 1)
    w = _rand((3, 3, 3, 32, 32), 2, 1.0 / np.sqrt(27 * 32))
    b = torch.randn(32, generator=torch.Generator().manual_seed(3))
    xd = x.to(cuda, L.ACT_DTYPE)
    desc = ops.make_conv_desc(L.CONV_DIRECT, B, (D, H, W), 32, 0, 32, 3, 1, "silu" if extras else None, None)
    y = torch.empty(B, D, H, W, 32, dtype=L.ACT_DTYPE, device=cuda)
    res = _rand((B, D, H, W, 32), 5) if extras else None
    sc = torch.rand(32, generator=torch.Generator().manual_seed(6)) + 0.5
    sh = torch.randn(32, generator=torch.Generator().manual_seed(7))
    plan = ops.ConvPlan(desc, xd, ops.pack_conv_weights(desc, w, False).to(cuda), y, bias=b.to(cuda),
                        residual=None if res is None else res.to(cuda, L.ACT_DTYPE),
                        out_affine=(sc.to(cuda), sh.to(cuda)) if extras else None)
    assert plan.info["halo"] == 3, "expected the d-sweeping plan"
    ws, rows = plan.gn_partials()
    plan.run()
    _check_flag()
    ref = O.conv3d(x, w, b)
    if extras:
        ref = O.swish(ref * sc + sh) + res
    _close(y, ref, tol=A + U, what=f"sweep32 {shape}")
    # the same layer on the halo kernel (tuning switch off -> use_halo = -1 selects the per-tap GEMM): agree to one 16-bit ulp
    y2 = ops.conv3d(xd, w, bias=b.to(cuda), use_halo=-1, act="silu" if extras else None,
                    residual=None if res is None else res.to(cuda, L.ACT_DTYPE), out_affine=(sc.to(cuda), sh.to(cuda)) if extras else None)
    _close(y, y2.float().cpu(), tol=A + 2 * U, what="sweep32 vs per-tap GEMM kernel")
    # GroupNorm statistics from the epilogue's partial sums (of the stored values) vs a direct evaluation, 8 groups
    mr = torch.empty(B, 8, 2, dtype=torch.float32, device=cuda)
    L.check(L.lib().b200dm_gn_finalize(L.ptr(ws), B, rows, 32, 8, D * H * W, 1e-6, L.ptr(mr), L.stream()))
    torch.cuda.synchronize()
    yf = y.float().cpu().reshape(B, -1, 8, 4).double()
    mean = yf.mean(dim=(1, 3))
    var = yf.var(dim=(1, 3), unbiased=False)
    assert torch.allclose(mr[..., 0].cpu().double(), mean, rtol=1e-4, atol=1e-5)
    assert torch.allclose(mr[..., 1].cpu().double(), 1.0 / torch.sqrt(var + 1e-6), rtol=1e-4)
