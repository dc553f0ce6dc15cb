"""The 16-bit storage type at its edges, in either build (bf16 or fp16, tests/test_fp16_build_gpu.py runs this file in both):
every reference is computed from the same stored 16-bit inputs.

* store rounding: each conv epilogue family's 16-bit store is the round-to-nearest-even of the same conv's fp32 output
  (operands on a coarse power-of-two grid, so that the fp32 result is exact whichever kernel and summation order computes it);
* subnormal operands (fp16 below 2^-14) through the tensor cores and the stencil head's mma.sync, against fp64;
* flash attention when most unnormalised probabilities underflow in the storage type;
* norm_act_ex / stats_f32 (csrc/norm_ex.cu, the vqgan_gnorm / vqgan_stride decoders' GroupNorm passes) against fp64.
"""
import ctypes

import numpy as np
import pytest
import torch

from b200dm import _lib as L
from oracle import ops as O

pytestmark = pytest.mark.gpu

ACT = L.ACT_DTYPE
FP16 = ACT == torch.float16
U = 2 ** -8 if L.precision() == "bf16" else 2 ** -11   # unit roundoff of the storage type: its largest relative rounding error
A = 2e-5   # fp32 accumulation in another order than the reference (tests/test_conv_gpu.py)


def _flag_ok():
    torch.cuda.synchronize()
    assert L.debug_flag() == 0, "tcgen05/TMA pipeline watchdog fired"


def _rand(shape, seed, scale=1.0):
    g = torch.Generator().manual_seed(seed)
    return (torch.randn(shape, generator=g) * scale).to(ACT).float()


def _ordered(t):
    """16-bit values as integers in value order (adjacent representable values differ by 1; +0 and -0 are both 0)."""
    b = t.contiguous().view(torch.int16).int()
    mag = b & 0x7FFF
    return torch.where(b < 0, -mag, mag)


# ------------------------------------------------------------------------------------------------ store rounding
def _conv(cuda, x, w, y_dtype, mode=L.CONV_DIRECT, stride=1, use_halo=0, residual=None, transposed_store=False, transposed=False,
          bias_scale=1.0):
    """One conv + bias (multiples of bias_scale / 8 in [-bias_scale, bias_scale]) through ConvPlan with the given output type."""
    from b200dm import ops
    B, D, H, W, cin = x.shape
    k = w.shape[0]
    cout = w.shape[3] if transposed else w.shape[4]
    desc = ops.make_conv_desc(mode, B, (D, H, W), cin, 0, cout, k, stride, None, None, y_dtype, use_halo=use_halo,
                              transposed_store=transposed_store)
    wp = ops.pack_conv_weights(desc, w, transposed).to(cuda)
    od, oh, ow = ops.conv_out_shape(mode, (D, H, W), stride)
    shape = (B, cout, od * oh * ow) if transposed_store else (B, od, oh, ow, cout)
    y = torch.empty(shape, dtype=L.storage(y_dtype), device=cuda)
    b = (torch.arange(cout, device=cuda) % 17 - 8).float() / 8
    ops.ConvPlan(desc, x.to(cuda, ACT), wp, y, bias=b * bias_scale, residual=residual).run()
    _flag_ok()
    return y.cpu()


STORE_CASES = {
    # name: (x shape, C_out, conv kwargs, residual); the 16-bit and the fp32 run may take different kernels (the sweep32, pair
    # slab and halo up kernels store 16-bit only): exact operands make their fp32 values identical all the same
    "direct": ((2, 8, 8, 8, 64), 32, dict(use_halo=-1), False),
    "staged": ((2, 8, 8, 8, 64), 64, dict(use_halo=-1), False),
    "staged_residual": ((2, 8, 8, 8, 64), 128, dict(use_halo=-1), True),
    "halo_cta_pair": ((2, 16, 16, 16, 64), 64, {}, False),
    "halo_n32_residual": ((1, 8, 16, 16, 64), 32, {}, True),
    "pair_slab": ((2, 8, 8, 8, 256), 256, {}, False),
    "halo_up64": ((2, 4, 16, 16, 64), 64, dict(mode=L.CONV_PARITY), False),
    "halo_up32": ((2, 4, 16, 16, 64), 32, dict(mode=L.CONV_PARITY), False),
    "convT_halo_up32": ((2, 4, 16, 16, 64), 32, dict(mode=L.CONV_PARITY, transposed=True), False),
    "sweep32": ((2, 20, 16, 8, 32), 32, {}, False),
    "stencil_head": ((1, 9, 13, 40, 32), 1, {}, False),
    "stride2": ((2, 16, 16, 16, 64), 64, dict(stride=2), False),
    "transposed_store": ((2, 8, 8, 8, 256), 256, dict(transposed_store=True), False),
}


def _grid(shape, seed, scale):
    """Integers in [-8, 8] times scale / 8 (scale a power of two): every product and sum of a conv is exact in fp32."""
    return torch.randint(-8, 9, shape, generator=torch.Generator().manual_seed(seed)).float() * (scale / 8)


def _store_operands(name, xscale=1.0, wscale=1.0):
    """Grid inputs and weights of a STORE_CASES conv whose outputs (and bias) are of the order of xscale * wscale."""
    shape, cout, kw, res = STORE_CASES[name]
    cin = shape[-1]
    k = 4 if kw.get("transposed") else (1 if kw.get("transposed_store") else 3)
    x = _grid(shape, 1, xscale)
    wshape = (k, k, k, cout, cin) if kw.get("transposed") else (k, k, k, cin, cout)
    w = _grid(wshape, 2, wscale * 2.0 ** -round(np.log2(np.sqrt(k ** 3 * cin))))
    assert torch.equal(x.to(ACT).float(), x) and torch.equal(w.to(ACT).float(), w)
    return x, w, cout, dict(kw, bias_scale=xscale * wscale), res


def _store_check(y16, y32, what):
    want = y32.float().to(ACT)
    fin = torch.isfinite(want)
    frac = (y16.float() == want.float()).float().mean().item()
    ulps = (_ordered(y16) - _ordered(want)).abs()[fin]
    print(f"{what}: {frac:.6f} of {y16.numel()} bit-equal to round(fp32), max {int(ulps.max()) if ulps.numel() else 0} ulp")
    assert not torch.isnan(y16.float()).any()
    assert frac == 1.0, f"{what}: only {frac:.6f} bit-equal to the fp32 output rounded to nearest"


@pytest.mark.parametrize("name", list(STORE_CASES))
def test_store_rounds_the_fp32_result_to_nearest(cuda, name):
    """The 16-bit output of every epilogue family is the fp32 output of the same conv rounded to nearest, ties to even, bit for
    bit (the grid operands give many exact ties): a truncating or otherwise mis-rounding store fails."""
    x, w, cout, kw, res = _store_operands(name)
    r = _grid(tuple(STORE_CASES[name][0][:-1]) + (cout,), 5, 1.0).to(cuda, ACT) if res else None
    y32 = _conv(cuda, x, w, torch.float32, residual=r, **kw)
    y16 = _conv(cuda, x, w, ACT, residual=r, **kw)
    assert y16.dtype == ACT and y16.shape == y32.shape and y32.abs().max() > 0.5
    _store_check(y16, y32, name)


@pytest.mark.parametrize("name", ["halo_cta_pair", "sweep32", "direct"])
def test_store_of_subnormal_outputs(cuda, name):
    """Outputs around 2^-20 (fp16 subnormals; normal in bf16) are rounded like the fp32 result, not flushed."""
    x, w, cout, kw, res = _store_operands(name, xscale=2.0 ** -10, wscale=2.0 ** -10)
    y32 = _conv(cuda, x, w, torch.float32, **kw)
    y16 = _conv(cuda, x, w, ACT, **kw)
    if FP16:
        assert (y32.abs() < 2 ** -14).float().mean() > 0.9 and (y16 != 0).float().mean() > 0.9
    _store_check(y16, y32, f"{name}, outputs ~2^-20")


@pytest.mark.skipif(not FP16, reason="bf16 has fp32's range")
@pytest.mark.parametrize("name", ["halo_cta_pair", "staged", "direct"])
def test_store_overflows_to_inf(cuda, name):
    """fp16 outputs straddling 65504: +-inf wherever the fp32 result rounds to it, never NaN and never clamped to +-65504."""
    x, w, cout, kw, res = _store_operands(name, wscale=2.0 ** 17)
    y32 = _conv(cuda, x, w, torch.float32, **kw).float()
    y16 = _conv(cuda, x, w, ACT, **kw).float()
    big = y32.abs() >= 65536          # past the rounding boundary 65520 by far more than the fp32 spread of two kernels
    small = y32.abs() < 65472         # below it by two fp16 ulps
    print(f"{name}: {big.float().mean().item():.3%} of outputs overflow")
    assert big.any() and small.any()
    assert not torch.isnan(y16).any()
    assert torch.equal(y16[big], torch.sign(y32[big]) * float("inf"))
    assert torch.isfinite(y16[small]).all()
    _store_check(y16.to(ACT), y32, f"{name}, outputs up to {y32.abs().max().item():.0f}")


# ------------------------------------------------------------------------------------------------ subnormal operands
SUB_CASES = {
    # name: (x shape, C_out, use_halo, y_dtype)
    "halo": ((1, 16, 16, 16, 64), 64, 0, torch.float32),
    "per_tap_gemm": ((1, 16, 16, 16, 64), 64, -1, torch.float32),
    "stencil_head": ((1, 16, 16, 16, 32), 1, 0, torch.float32),
    "sweep32": ((2, 20, 16, 8, 32), 32, 0, ACT),
}


@pytest.mark.parametrize("operand", ["x", "w"])
@pytest.mark.parametrize("name", list(SUB_CASES))
def test_subnormal_operands(cuda, name, operand):
    """Activations (or weights) scaled by 2^-16 -- mostly below fp16's 2^-14, normal in bf16 -- and the other operand scaled up
    to keep outputs O(1), against fp64 on the stored values.  A flush of subnormal operands to zero would be an O(1) error."""
    from b200dm import ops
    shape, cout, halo, y_dtype = SUB_CASES[name]
    cin = shape[-1]
    xs, ws = (2.0 ** -16, 2.0 ** 8) if operand == "x" else (2.0 ** 8, 2.0 ** -16)
    x = _rand(shape, 1, xs)
    w = _rand((3, 3, 3, cin, cout), 2, ws / np.sqrt(27 * cin))
    small = x if operand == "x" else w
    if FP16:
        assert (small.abs() < 2 ** -14).float().mean() > 0.5
    ref = O.conv3d(x.double(), w.double()).float()
    y = ops.conv3d(x.to(cuda, ACT), w, y_dtype=y_dtype, use_halo=halo)
    _flag_ok()
    y = y.float().cpu()
    err = (y - ref).abs().max().item() / ref.abs().max().item()
    print(f"{name}, {operand} x 2^-16: rel max err {err:.3e}")
    assert err <= A + (U if y_dtype != torch.float32 else 0), err


# ------------------------------------------------------------------------------------------------ attention underflow
@pytest.mark.parametrize("Lk", [32768, 131072])
def test_attention_normalisation_when_p_underflows(cuda, Lk):
    """One key at the row maximum (the first, so that the running maximum is exact from the first tile on), Lk - 1 keys 25.5
    binades below it, identical value rows: softmax returns that value row exactly.  In fp16 those p (2^-25.5) round to 0 before
    P.V; were they still counted in the normaliser l, the output would be 2.8e-3 low at 131072 keys (5.7 ulps)."""
    from b200dm import ops
    B, Lq, D = 1, 256, 64
    q = torch.zeros(B, Lq, D)
    q[..., 0] = 1.0
    k = torch.zeros(B, Lk, D)
    k[:, 1:, 0] = -25.5 * np.log(2.0)
    v0 = (_rand((1, 1, D), 3) + 0.5).to(ACT).float()
    vt = v0.reshape(1, D, 1).expand(B, D, Lk).contiguous()
    low = k[0, 1, 0].to(ACT).float().item() / np.log(2.0)
    assert -26 < low < -25
    o = ops.attention(q.to(cuda, ACT), k.to(cuda, ACT), vt.to(cuda, ACT), 1.0)
    _flag_ok()
    o = o.cpu()
    want = v0.to(ACT).expand(B, Lq, D)
    ulps = (_ordered(o) - _ordered(want)).abs().max().item()
    rel = ((o.float() - want.float()) / want.float()).mean().item()
    print(f"attention Lk {Lk}, p = 2^{low:.2f}: mean rel err {rel:.2e}, max {ulps} ulp")
    assert ulps <= 1


# ------------------------------------------------------------------------------------------------ norm_act_ex / stats_f32
EX_CASES = [
    # C, kind, groups, upsample, prelu, residual, act, post_act, x fp32, y fp32
    (16, 0, 1, False, True, True, "silu", "relu", False, False),     # vector kernel
    (32, 1, 8, True, True, False, None, None, False, False),         # vector, upsample + GroupNorm (vqgan_stride)
    (64, 1, 1, False, False, True, None, "relu", False, False),      # vector, residual unit tail (vqgan_gnorm)
    (16, 1, 8, False, True, True, "relu", None, False, True),        # C % 8 == 0 but fp32 out: scalar kernel
    (12, 0, 1, False, True, True, "silu", None, False, False),       # scalar kernel (C % 8 != 0)
    (2, 1, 1, True, True, True, None, "relu", True, True),           # the 2-channel fp32 network output
    (1, 1, 1, False, False, False, "silu", None, True, True),
    (2, 1, 2, True, False, False, None, None, True, False),
]


@pytest.mark.parametrize("C,kind,groups,up,prelu,res,act,post,xf,yf", EX_CASES)
def test_norm_act_ex(cuda, C, kind, groups, up, prelu, res, act, post, xf, yf):
    """y = post_act(residual + act(PReLU_alpha(a x[src] + b))) against fp64 on the same stored inputs."""
    g = torch.Generator().manual_seed(C * 10 + kind)
    B, ind = 2, (4, 6, 8)
    outd = tuple(2 * s for s in ind) if up else ind
    x = torch.randn(B, *ind, C, generator=g) * 2 + 0.3
    x = x if xf else x.to(ACT).float()
    if kind == 0:
        a, b = torch.rand(C, generator=g) + 0.5, torch.randn(C, generator=g) * 0.2
        mr = None
        aa, bb = a.double().expand(B, C), b.double().expand(B, C)
    else:
        a, b = torch.rand(C, generator=g) + 0.5, torch.randn(C, generator=g) * 0.2    # gamma, beta
        mr = torch.stack([torch.randn(B, groups, generator=g) * 0.3 + 0.3, torch.rand(B, groups, generator=g) + 0.3], -1)
        m, r = (mr[..., i].double().repeat_interleave(C // groups, 1) for i in (0, 1))
        aa = r * a.double()
        bb = b.double() - m * aa
    alpha = (torch.rand(*outd, C, generator=g) * 0.4).to(ACT).float() if prelu else None
    resid = torch.randn(B, *outd, C, generator=g).to(ACT).float() if res else None
    # fp64 reference
    xs = x.double()
    if up:
        xs = xs.repeat_interleave(2, 1).repeat_interleave(2, 2).repeat_interleave(2, 3)
    ref = xs * aa[:, None, None, None, :] + bb[:, None, None, None, :]
    if prelu:
        ref = ref.clamp(min=0) + alpha.double() * ref.clamp(max=0)
    ops_act = {None: lambda t: t, "silu": lambda t: t * torch.sigmoid(t), "relu": lambda t: t.clamp(min=0)}
    ref = ops_act[act](ref)
    if res:
        ref = ref + resid.double()
    ref = ops_act[post](ref)
    # kernel
    d = L.NormExDesc()
    d.batch, (d.out_d, d.out_h, d.out_w), d.c = B, outd, C
    d.kind, d.groups, d.act, d.post_act, d.upsample = kind, groups, L.ACT[act], L.ACT[post], int(up)
    d.x_dtype, d.y_dtype = (L.F32 if xf else L.BF16), (L.F32 if yf else L.BF16)
    dev = lambda t, dt=torch.float32: None if t is None else t.to(cuda, dt).contiguous()  # noqa: E731
    xd = dev(x, torch.float32 if xf else ACT)
    y = torch.empty(B, *outd, C, dtype=torch.float32 if yf else ACT, device=cuda)
    keep = (dev(a), dev(b), dev(mr), dev(alpha, ACT), dev(resid, ACT))
    L.check(L.lib().b200dm_norm_act_ex(ctypes.byref(d), L.ptr(xd), *(L.ptr(t) for t in keep), L.ptr(y), L.stream()))
    _flag_ok()
    err = (y.cpu().double() - ref).abs()
    bound = (0 if yf else U) * ref.abs() + 1e-5 * ref.abs().max()   # one rounding to the storage type: <= U relative
    print(f"norm_act_ex C{C} kind{kind}: max err {err.max().item():.2e}, max excess {(err - bound).max().item():.2e}")
    assert bool((err <= bound).all())


@pytest.mark.parametrize("per_sample", [127, 1000, 12345 * 3])
def test_stats_f32(cuda, per_sample):
    """Per-sample mean and rstd of an fp32 tensor with |mean| / std = 1e4, at sizes that do not divide into the 128 chunks."""
    g = torch.Generator().manual_seed(per_sample)
    B = 3
    mean = torch.tensor([100.0, -300.0, 0.5])
    std = mean.abs() * 1e-4
    x = (torch.randn(B, per_sample, generator=g, dtype=torch.float64) * std[:, None].double() + mean[:, None].double()).float()
    eps = 1e-6
    ws = torch.empty(L.lib().b200dm_stats_f32_workspace(B), dtype=torch.uint8, device=cuda)
    mr = torch.empty(B, 2, dtype=torch.float32, device=cuda)
    xd = x.to(cuda)
    L.check(L.lib().b200dm_stats_f32(L.ptr(xd), B, per_sample, eps, L.ptr(mr), L.ptr(ws), ws.numel(), L.stream()))
    _flag_ok()
    xs = x.double()
    m = xs.mean(1)
    rstd = 1 / torch.sqrt(((xs - m[:, None]) ** 2).mean(1) + eps)
    got = mr.cpu().double()
    print(f"stats_f32 n={per_sample}: mean rel err {((got[:, 0] - m) / m).abs().max().item():.2e}, "
          f"rstd rel err {((got[:, 1] - rstd) / rstd).abs().max().item():.2e}")
    assert torch.allclose(got[:, 0], m, rtol=1e-7, atol=0)
    assert torch.allclose(got[:, 1], rstd, rtol=1e-5, atol=0)
