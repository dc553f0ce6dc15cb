"""The normalisation and row-reduction kernels (csrc/norm.cu, csrc/norm_ex.cu, the d-sweeping conv's GroupNorm partials) element
by element against fp64 references computed on the device from the same stored 16-bit inputs, in either storage build.

GroupNorm statistics are held to the bn_stats contract: |m^ - m| <= eps_s * sigma (+ the fp32 rounding of the stored mean) and
|r^ / r - 1| <= eps_s with eps_s = 5e-6, also for groups whose |mean| is ~150 standard deviations -- where one-pass fp32 sums
of x and x^2 cancel.  The apply passes, LayerNorm, softmax and dense are held to U * |ref| (the storage type's unit roundoff)
plus a per-element fp32 term stated in each test."""
import ctypes
import math

import numpy as np
import pytest
import torch

from b200dm import _lib as L

pytestmark = pytest.mark.gpu

ACT = L.ACT_DTYPE
BF16 = L.precision() == "bf16"
U = 2 ** -8 if BF16 else 2 ** -11             # unit roundoff of the storage type
ETA = 2.0 ** -134 if BF16 else 2.0 ** -25     # half the storage type's smallest subnormal
E32 = 2.0 ** -24                              # fp32 unit roundoff
EPS_STATS = 5e-6                              # GroupNorm statistics bound (bn_stats' contract)
OFFSETS = [0.0, 8.0, 64.0, 150.0]             # |mean| / std of the generated groups
SIGMA = 2.0                                   # 300 +- 2: several fp16 ulps (0.25), about one bf16 ulp (2)
LAMBDA = {None: 1.0, "relu": 1.0, "silu": 1.1}   # Lipschitz constants of the activations


def _gen(seed):
    return torch.Generator(device="cuda").manual_seed(seed)


def _act64(z, act):
    if act == "silu":
        return z * torch.sigmoid(z)
    if act == "relu":
        return torch.relu(z)
    return z


def _report(what, err, bound):
    """worst err / bound over the case, printed for the record; the assertion names the first failing element."""
    ratio = (err / bound).max().item()
    print(f"{what}: worst err/bound {ratio:.3f}")
    if not ratio <= 1.0:
        i = int(torch.argmax(torch.nan_to_num(err / bound, nan=float("inf"))).item())
        raise AssertionError(f"{what}: element {i}: err {err.flatten()[i].item():.3e} > bound {bound.flatten()[i].item():.3e}")
    return ratio


# ------------------------------------------------------------------ GroupNorm statistics
def _grouped_input(B, V, C, G, seed, const_group=False, spread_group=False):
    """(B, V, C) stored 16-bit tensor; (sample, group) k has mean OFFSETS[k % 4] * SIGMA (alternating sign) and std SIGMA.
    const_group: group 0 of sample 0 is one constant.  spread_group: the channels of the last group sit 50 sigma apart."""
    g = _gen(seed)
    k = torch.arange(B * G, device="cuda") + seed
    mean = (torch.tensor(OFFSETS, device="cuda")[k % 4] * SIGMA * torch.where(k % 3 == 1, -1.0, 1.0)).reshape(B, 1, G, 1)
    x = torch.randn(B, V, G, C // G, generator=g, device="cuda") * SIGMA + mean
    if spread_group and C // G > 1:
        x[:, :, -1, :] += (torch.arange(C // G, device="cuda") - (C // G) / 2) * 50 * SIGMA
    if const_group:
        x[0, :, 0, :] = 3.25
    return x.reshape(B, V, C).to(ACT)


def _gn_ref(x, G):
    """fp64 (mean, variance) per (sample, group) of the stored values, two-pass"""
    B, C = x.shape[0], x.shape[-1]
    xg = x.double().reshape(B, -1, G, C // G).transpose(1, 2).reshape(B, G, -1)
    m = xg.mean(-1)
    return m, ((xg - m[..., None]) ** 2).mean(-1)


def _check_stats(mr, x, G, eps, what):
    m, v = _gn_ref(x, G)
    mr = mr.double()
    eps64 = float(np.float32(eps))
    r = 1.0 / torch.sqrt(v + eps64)
    em = _report(f"{what} mean", (mr[..., 0] - m).abs(), EPS_STATS * v.sqrt() + E32 * m.abs())
    er = _report(f"{what} rstd", (mr[..., 1] / r - 1).abs(), torch.full_like(r, EPS_STATS))
    return max(em, er)


def _gn_stats(x, G, eps):
    from b200dm import ops
    return ops.gn_stats(x.reshape(x.shape[0], -1, 1, 1, x.shape[-1]), G, eps)


@pytest.mark.parametrize("C", [8, 16, 32, 64, 128, 256, 512])
def test_gn_stats_against_fp64(cuda, C):
    """ops.gn_stats (gn_partial_kernel -> gn_final_kernel) over groups {1, 8, 32, C}, voxels {1, 63, 64, 65, 1000, 32^3}
    (below 64 voxels some of the 64 chunks are empty) and batch {1, 3}, groups at |mean|/std 0, 8, 64, 150, a constant group
    (rstd = eps^-1/2) and a group whose channels' means are 50 std apart.  Bound: |m^ - m| <= 5e-6 sigma + 2^-24 |m| and
    |r^/r - 1| <= 5e-6 for every (sample, group); two runs are bit-identical."""
    worst = 0.0
    case = 0
    for G in sorted({1, 8, 32, C}):
        if C % G:
            continue
        for V in [1, 63, 64, 65, 1000, 32 ** 3]:
            for B in ([1] if V == 32 ** 3 and C > 64 else [1, 3]):
                case += 1
                x = _grouped_input(B, V, C, G, case, const_group=case % 2 == 0, spread_group=case % 3 == 0)
                mr = _gn_stats(x, G, 1e-6)
                worst = max(worst, _check_stats(mr, x, G, 1e-6, f"gn_stats C{C} G{G} V{V} B{B}"))
                if V == 1000:
                    assert torch.equal(mr, _gn_stats(x, G, 1e-6)), "gn_stats is not bit-reproducible"
    print(f"gn_stats C{C}: worst err/bound {worst:.3f} over {case} cases")


def test_gn_stats_cfg3_size(cuda):
    """The cfg-3 decoder's statistics pass: 128^3 x 32, 32 groups, B = 1, groups at |mean|/std up to 150.  Same bound."""
    x = _grouped_input(1, 128 ** 3, 32, 32, 7, const_group=True)
    mr = _gn_stats(x, 32, 1e-6)
    _check_stats(mr, x, 32, 1e-6, "gn_stats 128^3 x 32, 32 groups")
    assert torch.equal(mr, _gn_stats(x, 32, 1e-6))


@pytest.mark.parametrize("shape,extras", [((2, 20, 16, 8), False), ((1, 35, 24, 12), True), ((3, 9, 48, 40), True),
                                          ((1, 128, 128, 128), False)])
def test_sweep_gn_partials_against_fp64(cuda, shape, extras):
    """GroupNorm statistics from the d-sweeping conv's epilogue partials + b200dm_gn_finalize on ragged volumes and at 128^3,
    with the stored y shifted to |mean|/std up to ~150 by the conv bias (or by out_affine's shift when the epilogue also runs
    affine + SiLU + residual), 8 groups with different offsets.  Against fp64 statistics of the stored y: the same bound as
    gn_stats; two runs are bit-identical."""
    from b200dm import ops
    B, D, H, W = shape
    g = torch.Generator().manual_seed(11)
    x = torch.randn(B, D, H, W, 32, generator=g).to(ACT)
    w = torch.randn(3, 3, 3, 32, 32, generator=g) / math.sqrt(27 * 32)
    shift = torch.tensor([OFFSETS[(c // 4) % 4] for c in range(32)]) * torch.where(torch.arange(32) % 8 < 4, 1.0, -1.0)
    b = torch.randn(32, generator=g) * 0.1 + (0 if extras else shift)
    sc = torch.rand(32, generator=g) + 0.5
    sh = shift if extras else None
    res = torch.randn(B, D, H, W, 32, generator=g).to(ACT).to(cuda) if extras else None
    desc = ops.make_conv_desc(L.CONV_DIRECT, B, (D, H, W), 32, 0, 32, 3, 1, "silu" if extras else None, None)
    y = torch.empty(B, D, H, W, 32, dtype=ACT, device=cuda)
    plan = ops.ConvPlan(desc, x.to(cuda), ops.pack_conv_weights(desc, w, False).to(cuda), y, bias=b.to(cuda), residual=res,
                        out_affine=(sc.to(cuda), sh.to(cuda)) if extras else None)
    assert plan.info["halo"] == 3, "expected the d-sweeping plan"
    ws, rows = plan.gn_partials()

    def stats():
        plan.run()
        mr = torch.empty(B, 8, 2, dtype=torch.float32, device=cuda)
        L.check(L.lib().b200dm_gn_finalize(L.ptr(ws), B, rows, 32, 8, D * H * W, 1e-6, L.ptr(mr), L.stream()))
        torch.cuda.synchronize()
        assert L.debug_flag() == 0
        return mr

    mr = stats()
    yd = y.reshape(B, -1, 32)
    m, v = _gn_ref(yd, 8)
    assert (m.abs() / v.sqrt()).max().item() > 30, "the stored y should have |mean| >> std in some group"
    _check_stats(mr, yd, 8, 1e-6, f"sweep partials {shape}{' +extras' if extras else ''}")
    assert torch.equal(mr, stats()), "sweep GroupNorm statistics are not bit-reproducible"


def test_stats_f32_offset(cuda):
    """b200dm_stats_f32 (fp32 input, fp64 accumulation) at |mean|/std = 150: the GroupNorm statistics bound."""
    B, n = 2, 300_001
    x = torch.randn(B, n, generator=_gen(3), device="cuda", dtype=torch.float32) * 2 + torch.tensor([[300.0], [-17.0]], device="cuda")
    ws = torch.empty(L.lib().b200dm_stats_f32_workspace(B) // 8, dtype=torch.float64, device=cuda)
    mr = torch.empty(B, 1, 2, dtype=torch.float32, device=cuda)
    L.check(L.lib().b200dm_stats_f32(L.ptr(x), B, n, 1e-6, L.ptr(mr), L.ptr(ws), ws.numel() * 8, L.stream()))
    m = x.double().mean(-1, keepdim=True)
    v = ((x.double() - m) ** 2).mean(-1, keepdim=True)
    r = 1.0 / torch.sqrt(v + float(np.float32(1e-6)))
    _report("stats_f32 mean", (mr[..., 0].double() - m).abs(), EPS_STATS * v.sqrt() + E32 * m.abs())
    _report("stats_f32 rstd", (mr[..., 1].double() / r - 1).abs(), torch.full_like(r, EPS_STATS))


# ------------------------------------------------------------------ apply passes
def _norm_act_path(voxels, C, B):
    """Which index path bind_norm_act_fwd's grid gives norm_act_kernel: 'octet' when gridDim.x * 256 is a multiple of C / 8
    (each thread keeps one channel octet), else 'generic'.  The grid is at most ceil(want / B) blocks per sample; when that
    covers fewer than all vectors of a sample it is rounded up to a multiple of C / 8 / gcd(C / 8, 256) (octet path) whatever
    the occupancy, and a one-block grid (want = 1) is exact."""
    c8n = C // 8
    items = voxels * c8n
    if 256 % c8n == 0:
        return "octet"
    want = -(-(-(-(items * B + 3) // 4)) // 256)
    if -(-want // B) * 256 < items:
        return "octet"
    assert want == 1, "the path of this shape depends on the occupancy"
    return "generic"


def _stats_f32(x, G):
    """fp32 (B, G, 2) (mean, rstd) from fp64 statistics: the input of the apply passes (gn_stats takes only C / 8 | 256)"""
    m, v = _gn_ref(x, G)
    return torch.stack([m, 1.0 / torch.sqrt(v + float(np.float32(1e-6)))], -1).float()


def _apply_bound(ref, x, a, m, beta, act, c=8):
    """U |r| + Lambda c 2^-24 (|x a| + |m a| + |beta|) + eta: storage rounding, the fp32 fold b = beta - m a and fma"""
    return U * ref.abs() + LAMBDA[act] * c * E32 * ((x * a).abs() + (m * a).abs() + beta.abs()) + ETA


# (c0, c1, voxels, B): generic-path shapes (C / 8 does not divide 256, one block), octet-path shapes (large) with the same C,
# concat boundaries at octets 1, 3 and 8, voxel counts that leave a partial 4-vector unrolled tail
NORM_ACT_CASES = [(24, 0, 9, 1), (40, 0, 13, 1), (8, 40, 5, 1), (64, 8, 7, 1), (64, 40, 3, 3), (24, 40, 11, 3),
                  (24, 0, 100_003, 1), (40, 0, 64_001, 2), (8, 40, 50_001, 1), (64, 8, 40_003, 3), (64, 40, 30_001, 1),
                  (8, 8, 1_001, 3), (24, 8, 997, 2), (64, 0, 1_234_567, 1)]


def _case_id(c):
    c0, c1, V, B = c
    return f"{c0}+{c1}-V{V}-B{B}-{_norm_act_path(V, c0 + c1, B)}"


@pytest.mark.parametrize("case", NORM_ACT_CASES, ids=_case_id)
@pytest.mark.parametrize("kind", [0, 1])
@pytest.mark.parametrize("act", [None, "silu", "relu"])
def test_norm_act_against_fp64(cuda, case, kind, act):
    """norm_act_kernel (both index paths, named in the id) over [x0 | x1]: kind 0 with (scale, shift), kind 1 with fp32
    (mean, rstd) that the kernel and the fp64 reference both read, so the apply pass is tested on its own terms; per-sample
    statistics differ (B = 3) and groups sit at |mean|/std up to 150.  Bound per element:
    |y - r| <= U |r| + Lambda 8 2^-24 (|x a| + |m a| + |beta|) + eta."""
    from b200dm import ops
    c0, c1, V, B = case
    C = c0 + c1
    G = 4 if C % 32 else 8
    xc = _grouped_input(B, V, C, G, c0 * 7 + c1 + V)
    x0, x1 = xc[..., :c0].contiguous(), (xc[..., c0:].contiguous() if c1 else None)
    g = _gen(5)
    gamma = torch.rand(C, generator=g, device="cuda") + 0.5
    beta = torch.randn(C, generator=g, device="cuda")
    x64 = xc.double()
    if kind == 0:
        mr = None
        a64, b64, m64 = gamma.double(), beta.double(), torch.zeros((), dtype=torch.float64, device="cuda")
        z = x64 * a64 + b64
    else:
        mr = _stats_f32(xc, G)
        m64 = mr[..., 0].double().repeat_interleave(C // G, 1)[:, None, :]
        r64 = mr[..., 1].double().repeat_interleave(C // G, 1)[:, None, :]
        a64, b64 = r64 * gamma.double(), beta.double()
        z = (x64 - m64) * a64 + b64
    ref = _act64(z, act)
    y = ops.norm_act(x0.reshape(B, V, 1, 1, c0), gamma, beta, act=act, x1=None if x1 is None else x1.reshape(B, V, 1, 1, c1),
                     kind=kind, groups=G, mean_rstd=mr)
    err = (y.reshape(B, V, C).double() - ref).abs()
    _report(f"norm_act kind{kind} {act} {_case_id(case)}", err, _apply_bound(ref, x64, a64, m64, b64, act))


@pytest.mark.parametrize("C,V,B", [(32, 4099, 3), (8, 65, 1), (96, 777, 2), (24, 100_003, 1)])
def test_norm_act_ex_groupnorm_against_fp64(cuda, C, V, B):
    """norm_act_ex kind 1 (GroupNorm apply + SiLU, vector path) with fp32 (mean, rstd) that kernel and reference both read:
    the norm_act bound."""
    from b200dm import ops
    G = 8 if C % 64 == 0 or C == 32 else 4
    x = _grouped_input(B, V, C, G, V)
    g = _gen(6)
    gamma = torch.rand(C, generator=g, device="cuda") + 0.5
    beta = torch.randn(C, generator=g, device="cuda")
    mr = _stats_f32(x, G)
    y = torch.empty(B, V, 1, 1, C, dtype=ACT, device=cuda)
    d = L.NormExDesc()
    d.batch, d.out_d, d.out_h, d.out_w, d.c = B, V, 1, 1, C
    d.kind, d.groups, d.act, d.post_act, d.upsample = 1, G, L.ACT["silu"], L.ACT[None], 0
    d.x_dtype, d.y_dtype = L.BF16, L.BF16
    L.check(L.lib().b200dm_norm_act_ex(ctypes.byref(d), L.ptr(x), L.ptr(gamma), L.ptr(beta), L.ptr(mr), None, None,
                                       L.ptr(y), L.stream()))
    m64 = mr[..., 0].double().repeat_interleave(C // G, 1)[:, None, :]
    a64 = mr[..., 1].double().repeat_interleave(C // G, 1)[:, None, :] * gamma.double()
    x64 = x.double()
    ref = _act64((x64 - m64) * a64 + beta.double(), "silu")
    err = (y.reshape(B, V, C).double() - ref).abs()
    _report(f"norm_act_ex C{C} V{V} B{B}", err, _apply_bound(ref, x64, a64, m64, beta.double(), "silu"))


def test_gn_stats_then_norm_act_end_to_end(cuda):
    """gn_stats -> norm_act (SiLU) at |mean|/std up to 150 against fp64 GroupNorm + SiLU of the stored input (statistics in
    fp64 too): U |r| + 1.1 (8 2^-24 (|x a| + |m a| + |beta|) + 2 eps_s |a| (|x - m| + sigma)) + eta, the apply bound plus the
    statistics bound carried through the affine."""
    from b200dm import ops
    B, V, C, G = 2, 40_000, 64, 8
    x = _grouped_input(B, V, C, G, 21)
    g = _gen(8)
    gamma = torch.rand(C, generator=g, device="cuda") + 0.5
    beta = torch.randn(C, generator=g, device="cuda")
    mr = ops.gn_stats(x.reshape(B, V, 1, 1, C), G, 1e-6)
    y = ops.norm_act(x.reshape(B, V, 1, 1, C), gamma, beta, act="silu", kind=1, groups=G, mean_rstd=mr)
    m, v = _gn_ref(x, G)
    rstd = 1.0 / torch.sqrt(v + float(np.float32(1e-6)))
    m64 = m.repeat_interleave(C // G, 1)[:, None, :]
    s64 = v.sqrt().repeat_interleave(C // G, 1)[:, None, :]
    a64 = rstd.repeat_interleave(C // G, 1)[:, None, :] * gamma.double()
    x64 = x.double()
    ref = _act64((x64 - m64) * a64 + beta.double(), "silu")
    bound = _apply_bound(ref, x64, a64, m64, beta.double(), "silu") + 1.1 * 2 * EPS_STATS * a64.abs() * ((x64 - m64).abs() + s64)
    _report("gn_stats -> norm_act end to end", (y.reshape(B, V, C).double() - ref).abs(), bound)


# ------------------------------------------------------------------ LayerNorm
@pytest.mark.parametrize("C", [8, 200, 256, 264, 512, 520, 1024])
@pytest.mark.parametrize("n_out", [1, 2, 3])
def test_layernorm_against_fp64(cuda, C, n_out):
    """layernorm_kernel (kVecPerLane 1 / 2 / 4, with and without partial lanes) over 1, 7 and more rows than one resident grid
    of warps (grid-stride loop), n_out distinct affines, rows at |mean|/std up to 150 and a constant row.  Bound per element:
    U |r| + 2^-24 (64 rstd mean|x| |gamma| + 32 |x^ gamma| + 4 |beta|) + eta -- the fp32 row mean's rounding (warp tree of
    <= 37 terms) carried through rstd, the variance sum and rsqrtf, and the affine."""
    from b200dm import ops
    sms = torch.cuda.get_device_properties(0).multi_processor_count
    g = _gen(C + n_out)
    for rows in (1, 7, sms * 8 * 8 + 37):
        mean = torch.tensor(OFFSETS, device="cuda")[torch.arange(rows, device="cuda") % 4] * SIGMA
        x = (torch.randn(rows, C, generator=g, device="cuda") * SIGMA + mean[:, None])
        x[rows // 2] = -5.5   # constant row: x^ = 0, y = beta
        x = x.to(ACT)
        gs = [torch.rand(C, generator=g, device="cuda") + 0.5 for _ in range(n_out)]
        bs = [torch.randn(C, generator=g, device="cuda") for _ in range(n_out)]
        ys = ops.layernorm(x, gs, bs, 1e-3)
        x64 = x.double()
        m = x64.mean(-1, keepdim=True)
        r = 1.0 / torch.sqrt(((x64 - m) ** 2).mean(-1, keepdim=True) + float(np.float32(1e-3)))
        xh = (x64 - m) * r
        for o, (y, ga, be) in enumerate(zip(ys, gs, bs)):
            ga, be = ga.double(), be.double()
            ref = xh * ga + be
            bound = U * ref.abs() + E32 * (64 * r * x64.abs().mean(-1, keepdim=True) * ga.abs() + 32 * (xh * ga).abs() + 4 * be.abs()) + ETA
            _report(f"layernorm C{C} rows{rows} out{o}", (y.double() - ref).abs(), bound)


# ------------------------------------------------------------------ softmax
@pytest.mark.parametrize("cols", [1, 31, 255, 256, 257, 4096, 32768])
def test_softmax_rows_against_fp64(cuda, cols):
    """softmax_rows_kernel at several scales, rows above the 148 * 8 grid cap (small cols), rows whose scores span more than
    the exponent range (p underflows) and rows of identical scores.  The reference is fp64 softmax of fl32(s * scale), the
    kernel's first operation.  Bound per element: |p - r| <= U r + 2^-24 (16 + cols / 128 + 2 |s scale - max|) r + eta:
    __expf's argument rounding, ex2.approx, and the fp32 row sum of <= cols / 256 + 8 serial terms."""
    from b200dm import ops
    sms = torch.cuda.get_device_properties(0).multi_processor_count
    rows = sms * 8 + 41 if cols <= 257 else 64
    g = _gen(cols)
    s = torch.randn(rows, cols, generator=g, device="cuda") * 3
    s[1] = torch.linspace(-400, 400, cols, device="cuda")   # exp of the span under- / overflows fp32 without the max shift
    s[2] = 1.75                                             # identical scores: p = 1 / cols
    s[3] = torch.randn(cols, generator=g, device="cuda") * 60 + 200
    for scale in (0.125, 1.0, 2.5):
        p = ops.softmax_rows(s, scale)
        z = (s * scale).double()   # fl32(s * scale), exactly
        mx = z.max(-1, keepdim=True).values
        ref = torch.softmax(z, -1)
        bound = U * ref + E32 * (16 + cols / 128 + 2 * (z - mx).abs()) * ref + ETA
        _report(f"softmax cols{cols} rows{rows} scale{scale}", (p.double() - ref).abs(), bound)


# ------------------------------------------------------------------ dense
@pytest.mark.parametrize("M", [1, 8, 9, 37])
@pytest.mark.parametrize("K", [1, 128, 1280])
def test_dense_f32_against_fp64(cuda, M, K):
    """dense_f32_kernel, N not a multiple of 128, every act_in x act_out.  Bound per element:
    |y - r| <= (K + 8) 2^-24 Lambda (sum_k |x'_k| |w_kn| + |b_n|) + 4 2^-24 |r|, x' = act_in(x)."""
    from b200dm import ops
    g = _gen(M * 10_000 + K)
    N = 1000
    x = torch.randn(M, K, generator=g, device="cuda") * 2
    w = torch.randn(K, N, generator=g, device="cuda") / math.sqrt(K)
    b = torch.randn(N, generator=g, device="cuda")
    for act_in in (None, "silu"):
        for act_out in (None, "silu", "relu"):
            y = ops.dense_f32(x, w, b, act_in=act_in, act_out=act_out)
            xi = _act64(x.double(), act_in)
            ref = _act64(xi @ w.double() + b.double(), act_out)
            bound = (K + 8) * E32 * LAMBDA[act_out] * (xi.abs() @ w.double().abs() + b.double().abs()) + 4 * E32 * ref.abs()
            _report(f"dense M{M} K{K} {act_in}->{act_out}", (y.double() - ref).abs(), bound)


# ------------------------------------------------------------------ casts, bn_fold
def _special_f32(n, g):
    """n fp32 values: normal, NaN, +-inf, fp32 and storage subnormals, values that overflow the storage type, exact ties"""
    x = torch.randn(n, generator=g, device="cuda") * 10
    fin = torch.finfo(ACT)
    specials = [float("nan"), float("inf"), -float("inf"), 0.0, -0.0, 1e-40, -3e-39, fin.tiny * 0.75, fin.tiny / 3,
                fin.max * 1.5, -fin.max * 1.01, fin.max, fin.tiny * fin.eps]
    one = 1.0 + fin.eps / 2                       # half-way between 1 and its successor: ties round to even (1)
    specials += [one, 1.0 + 1.5 * fin.eps, -(1.0 + 2.5 * fin.eps), 3 * (1.0 + fin.eps / 2)]
    k = min(n, len(specials))
    x[:k] = torch.tensor(specials[:k], device="cuda")
    return x[torch.randperm(n, generator=g, device="cuda")] if n > 1 else x


def _same_or_both_nan(y, ref):
    nan = torch.isnan(ref)
    assert torch.equal(torch.isnan(y), nan)
    bits = torch.int16 if y.element_size() == 2 else torch.int32
    assert torch.equal(y[~nan].view(bits), ref[~nan].view(bits)), "conversion differs from torch's"


@pytest.mark.parametrize("n", list(range(1, 18)) + [8 * 1000 + 5, 1_000_003])
def test_cast_bit_identical_to_torch(cuda, n):
    """b200dm_cast fp32 -> 16-bit and back is torch's round-to-nearest-even conversion bit for bit (NaN stays NaN; its
    payload is not compared) for every n mod 8 (the scalar tail) and NaN, +-inf, subnormals, overflow to inf and ties."""
    from b200dm import ops
    x = _special_f32(n, _gen(n))
    y = ops.cast(x, ACT)
    _same_or_both_nan(y, x.to(ACT))
    h = torch.randn(n, generator=_gen(n + 1), device="cuda").to(ACT)
    h[: min(n, 4)] = torch.tensor([float("nan"), float("inf"), torch.finfo(ACT).tiny / 4, -0.0][: min(n, 4)], device="cuda").to(ACT)
    _same_or_both_nan(ops.cast(h, torch.float32), h.float())


def test_bn_fold_against_fp64(cuda):
    """bn_fold: scale = gamma rsqrt(var + eps) within 2 fp32 ulps of fp64; shift = beta - mean scale within 2 fp32 ulps of
    |beta| + |mean scale| (its terms' magnitude: the subtraction may cancel)."""
    from b200dm import ops
    g = _gen(9)
    C = 1000
    gamma = torch.randn(C, generator=g, device="cuda")
    beta = torch.randn(C, generator=g, device="cuda")
    mean = torch.randn(C, generator=g, device="cuda") * 100
    var = torch.rand(C, generator=g, device="cuda") ** 4 * 100
    sc, sh = ops.bn_fold(gamma, beta, mean, var, 1e-3)
    s64 = gamma.double() / torch.sqrt((var.double() + float(np.float32(1e-3))))
    h64 = beta.double() - mean.double() * s64

    def ulp(v):
        f = v.abs().float()
        return (torch.nextafter(f, torch.full_like(f, float("inf"))) - f).double()

    _report("bn_fold scale", (sc.double() - s64).abs(), 2 * ulp(s64))
    _report("bn_fold shift", (sh.double() - h64).abs(), 2 * ulp(beta.double().abs() + (mean.double() * s64).abs()))
