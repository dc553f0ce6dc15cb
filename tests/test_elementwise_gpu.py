"""GPU parity for the HBM-bound kernels: fused DDPM/DDIM update + Philox, norm+act(+concat), GN stats,
LayerNorm, softmax, dense, VQ argmin+gather -- each against the oracle on the same seeded inputs."""
import numpy as np
import pytest
import torch

from oracle import ops as O, sampler as OS, philox as OP, first_stage as OF, init as OI
from b200dm import _lib
from oracle.schedule import Betas

pytestmark = pytest.mark.gpu

ACT = _lib.ACT_DTYPE
U = 2 ** -8 if _lib.precision() == "bf16" else 2 ** -11   # unit roundoff of the storage type: its largest relative rounding error


def _r(t):
    return t.to(ACT).to(torch.float32)


@pytest.mark.parametrize("t", [999, 500, 1, 0])
def test_ddpm_update_injected_noise_bit_exact(cuda, t):
    """fp32 arithmetic in the reference's op order: posterior mean/clip/noise-add must match the oracle
    to <= 1 ulp (sigma goes through expf/logf: tolerance 2e-7 relative, stated)."""
    from b200dm import ops
    T = 1000
    tabs = ops.ScheduleTables(T, cuda)
    b = Betas(T)
    for k in ops.ScheduleTables.NAMES:
        assert np.array_equal(tabs.host[k], getattr(b, k)), k
    shape = (2, 8, 8, 8, 16)
    x, eps, z = OI.normal(shape, 1), OI.normal(shape, 2), OI.normal(shape, 3)
    ref = OS.ddpm_step(b, x, eps, t, z)
    y = ops.ddpm_update(tabs, x.to(cuda), eps.to(cuda), t, noise=z.to(cuda))
    err = (y.cpu() - ref).abs().max().item()
    assert err <= 4e-7 * max(1.0, ref.abs().max().item()), err
    if t == 0:
        assert torch.equal(y.cpu(), torch.clamp(OS.sample(b, x, eps, 0)[0], -1, 1))
    # 16-bit eps input + 16-bit copy of the output
    eb = _r(eps)
    y2, y2b = ops.ddpm_update(tabs, x.to(cuda), eb.to(cuda, ACT), t, noise=z.to(cuda), want_bf16=True)
    ref2 = OS.ddpm_step(b, x, eb, t, z)
    assert (y2.cpu() - ref2).abs().max().item() <= 4e-7 * max(1.0, ref2.abs().max().item())
    assert torch.equal(y2b.cpu(), y2.cpu().to(ACT))


def test_ddim_update(cuda):
    from b200dm import ops
    T = 1000
    tabs, b = ops.ScheduleTables(T, cuda), Betas(T)
    shape = (2, 4, 4, 4, 8)
    x, eps = OI.normal(shape, 1), OI.normal(shape, 2)
    for t, tp in [(996, 992), (4, 0), (0, -1)]:
        ref = OS.ddim_step(b, x, eps, t, tp)
        y = ops.ddpm_update(tabs, x.to(cuda), eps.to(cuda), t, sampler=1, t_prev=tp)
        assert (y.cpu() - ref).abs().max().item() <= 1e-6 * max(1.0, ref.abs().max().item())


def test_philox_stream_matches_oracle(cuda):
    from b200dm import ops
    seed, step = 1234, 17
    n = 4 * 4 * 4 * 8
    x = ops.philox_normal((3, 4, 4, 4, 8), seed, sample_id0=5, step=step, stream_id=0)
    ref = OP.normal(seed, step, [5, 6, 7], n, stream=0).reshape(3, 4, 4, 4, 8)
    err = np.abs(x.cpu().numpy() - ref).max()
    assert err <= 2e-5, err  # logf/sincospif vs numpy log/sin/cos
    big = ops.philox_normal((2, 32, 32, 32, 8), seed, 0, 3, 0).cpu().numpy()
    assert abs(big.mean()) < 5e-3 and abs(big.std() - 1) < 5e-3
    # the update kernel draws the same stream in-register
    T = 1000
    tabs, b = ops.ScheduleTables(T, cuda), Betas(T)
    shape = (3, 4, 4, 4, 8)
    xt, eps = OI.normal(shape, 1), OI.normal(shape, 2)
    y = ops.ddpm_update(tabs, xt.to(cuda), eps.to(cuda), step, seed=seed, sample_id0=5)
    ref = OS.ddpm_step(b, xt, eps, step, torch.from_numpy(ref))
    assert (y.cpu() - ref).abs().max().item() <= 1e-5


@pytest.mark.parametrize("act", [None, "silu", "relu"])
def test_bn_act_concat(cuda, act):
    from b200dm import ops
    B, S, c0, c1 = 2, 8, 64, 32
    g = torch.Generator().manual_seed(0)
    x0, x1 = _r(torch.randn(B, S, S, S, c0, generator=g)), _r(torch.randn(B, S, S, S, c1, generator=g))
    C = c0 + c1
    gamma, beta = torch.rand(C, generator=g) + 0.5, torch.randn(C, generator=g) * 0.1
    mean, var = torch.randn(C, generator=g) * 0.1, torch.rand(C, generator=g) + 0.5
    ref = O.batchnorm_infer(torch.cat([x0, x1], -1), gamma, beta, mean, var)
    ref = O.swish(ref) if act == "silu" else (torch.relu(ref) if act == "relu" else ref)
    sc, sh = ops.bn_fold(gamma.to(cuda), beta.to(cuda), mean.to(cuda), var.to(cuda), 1e-3)
    y = ops.norm_act(x0.to(cuda, ACT), sc, sh, act=act, x1=x1.to(cuda, ACT))
    err = (y.float().cpu() - ref).abs().max().item()
    assert err <= U * ref.abs().max().item() + 1e-6, err


@pytest.mark.parametrize("C,G,S", [(32, 32, 16), (64, 32, 8), (128, 32, 8), (64, 8, 8)])
def test_groupnorm_silu(cuda, C, G, S):
    from b200dm import ops
    B = 2
    g = torch.Generator().manual_seed(0)
    x = _r(torch.randn(B, S, S, S, C, generator=g) * 2 + 0.3)
    gamma, beta = torch.rand(C, generator=g) + 0.5, torch.randn(C, generator=g) * 0.1
    ref = O.swish(O.groupnorm(x, gamma, beta, G, 1e-6))
    xb = x.to(cuda, ACT)
    mr = ops.gn_stats(xb, G, 1e-6)
    xg = x.reshape(B, -1, G, C // G)
    assert (mr[..., 0].cpu() - xg.mean(dim=(1, 3))).abs().max().item() < 1e-5
    y = ops.norm_act(xb, gamma.to(cuda), beta.to(cuda), act="silu", kind=1, groups=G, mean_rstd=mr)
    err = (y.float().cpu() - ref).abs().max().item()
    assert err <= U * ref.abs().max().item() + 1e-5, err


def test_layernorm3(cuda):
    from b200dm import ops
    g = torch.Generator().manual_seed(0)
    x = _r(torch.randn(2, 8, 8, 8, 256, generator=g))
    gs = [torch.rand(256, generator=g) + 0.5 for _ in range(3)]
    bs = [torch.randn(256, generator=g) * 0.1 for _ in range(3)]
    ys = ops.layernorm(x.to(cuda, ACT), [t.to(cuda) for t in gs], [t.to(cuda) for t in bs], 1e-3)
    for y, ga, be in zip(ys, gs, bs):
        ref = O.layernorm(x, ga, be)
        assert (y.float().cpu() - ref).abs().max().item() <= U * ref.abs().max().item() + 1e-5


def test_softmax_and_dense(cuda):
    from b200dm import ops
    g = torch.Generator().manual_seed(0)
    s = torch.randn(64, 512, generator=g) * 3
    p = ops.softmax_rows(s.to(cuda), 0.25)
    ref = torch.softmax(s * 0.25, -1)
    assert (p.float().cpu() - ref).abs().max().item() <= U * ref.max().item()
    x, w, b = torch.randn(37, 128, generator=g), torch.randn(128, 1000, generator=g) * 0.1, torch.randn(1000, generator=g)
    y = ops.dense_f32(x.to(cuda), w.to(cuda), b.to(cuda), act_in="silu", act_out="silu")
    ref = O.swish(O.dense(O.swish(x), w, b))
    assert (y.cpu() - ref).abs().max().item() <= 1e-4


@pytest.mark.parametrize("N,D,K,layout", [(4096, 64, 256, "DK"), (5000, 256, 1024, "KD"), (128, 16, 7, "KD")])
def test_vq_indices_bit_exact(cuda, N, D, K, layout):
    """Indices must equal the exact-arithmetic argmin wherever the fp32 formula is unambiguous
    (fp64 margin > 1e-5 * distance); on well-separated inputs that is every row."""
    from b200dm import ops
    cb = OI.codebook(K, D, layout, seed=3)
    x = OI.normal((N, D), 7, 0.5 if layout == "KD" else 0.05)
    idx64, margin = OF.get_code_indices_exact(x, cb, layout)
    idx32 = OF.get_code_indices(x, cb, layout)
    cb_kd = (cb.t() if layout == "DK" else cb).contiguous()
    hist = torch.zeros(K, dtype=torch.int32, device=cuda)
    idx, q = ops.vq_argmin_gather(x.to(cuda), cb_kd.to(cuda), hist=hist)
    idx = idx.cpu()
    d_best = OF.code_distances(x.double(), cb.double(), layout).min(1).values
    safe = margin > 1e-5 * d_best.abs().clamp(min=1e-6)
    assert torch.equal(idx[safe], idx64[safe]), f"{(idx[safe] != idx64[safe]).sum().item()} mismatches on unambiguous rows"
    assert torch.equal(idx[safe], idx32[safe])
    assert (idx != idx64).sum().item() <= (~safe).sum().item()
    assert torch.equal(q.cpu(), cb_kd[idx])          # gather is exact
    assert torch.equal(hist.cpu().long(), torch.bincount(idx, minlength=K))


def test_vq_ties_take_lowest_index_and_empty(cuda):
    from b200dm import ops
    cb = torch.tensor([[1.0, 0, 0, 0], [1.0, 0, 0, 0], [0, 1.0, 0, 0]])  # codes 0 and 1 identical
    x = torch.tensor([[0.9, 0, 0, 0], [0, 0.8, 0, 0], [0.5, 0.5, 0, 0]])
    idx, q = ops.vq_argmin_gather(x.to(cuda), cb.to(cuda))
    assert idx.cpu().tolist() == [0, 2, 0]
    idx, q = ops.vq_argmin_gather(torch.empty(0, 4, device=cuda), cb.to(cuda))
    assert idx.numel() == 0


def _vq_both(x, cb_kd, cuda, **kw):
    """(idx, q, hist) of the fp32 SIMT kernel and of the tensor-core candidate search on the same device inputs."""
    from b200dm import ops
    xd, cbd = x.to(cuda), cb_kd.to(cuda)
    K = cb_kd.shape[0]
    out = []
    for tc in (None, "auto"):
        hist = torch.zeros(K, dtype=torch.int32, device=cuda)
        stats = torch.zeros(3, dtype=torch.int64, device=cuda)
        idx, q = ops.vq_argmin_gather(xd, cbd, hist=hist, tc_ws=tc, stats=stats, **kw)
        out.append((idx.cpu(), q.cpu(), hist.cpu(), stats.cpu()))
    return out


@pytest.mark.parametrize("N,D,K", [(5000, 256, 1024), (777, 64, 128), (4096, 128, 512), (1000, 192, 256), (128 * 300 + 5, 256, 2048)])
@pytest.mark.parametrize("x16", [False, True])
def test_vq_tensor_core_search_is_bit_identical(cuda, N, D, K, x16):
    """vq_tc_kernel (fp16 hi/lo split MMAs -> candidates inside the proven margin -> exact fp32 chain for them) returns the
    indices, rows and histogram of vq_kernel bit for bit: random rows, rows that ARE codes, duplicated codes (exact ties ->
    lowest index), codes one ulp apart, tiny and huge row scales, zero rows."""
    from b200dm import _lib as L
    g = torch.Generator().manual_seed(N + D + K)
    cb = (torch.rand(K, D, generator=g) - 0.5) * 0.1
    cb[K // 2] = cb[3]                                   # exact duplicate: index 3 must win
    cb[K // 2 + 1] = cb[5]
    cb[K // 2 + 1, 7] = torch.nextafter(cb[5, 7], torch.tensor(1.0))   # one ulp apart
    cb[K - 1] = cb[9] * (1 + 2 ** -20)
    x = torch.randn(N, D, generator=g) * 0.5
    x[:64] = cb[torch.randint(0, K, (64,), generator=g)]  # rows equal to codes
    x[64:96] = cb[[3, 5, 9, K // 2 + 1] * 8] + torch.randn(32, D, generator=g) * 1e-6
    x[96:128] = 0.5 * (cb[3] + cb[11]) + torch.randn(32, D, generator=g) * 1e-7   # equidistant to two codes up to noise
    # tiny / huge but finite in the input type: 1e-9 / 1e9 are 0 / inf in fp16
    tiny, huge = (2.0 ** -12, 2.0 ** 12) if x16 and ACT == torch.float16 else (1e-9, 1e9)
    x[128:160] *= tiny
    x[160:192] *= huge
    x[192:200] = 0
    x[200:232] = cb[torch.randint(0, K, (32,), generator=g)] * 40   # large ||x||: fl(||x||^2 + ||e||^2) is coarse, many fp32 ties
    if x16:
        x = x.to(ACT)
        assert torch.isfinite(x).all() and (x[128:160] != 0).any()
    (i0, q0, h0, _), (i1, q1, h1, st) = _vq_both(x, cb, cuda)
    assert L.debug_flag() == 0
    assert torch.equal(i0, i1), f"{(i0 != i1).sum().item()} of {N} indices differ (first rows {torch.nonzero(i0 != i1)[:8].flatten().tolist()})"
    assert torch.equal(q0, q1) and torch.equal(h0, h1)
    assert int(st[2]) <= 64 + 8, f"full-scan fallbacks: {st.tolist()}"   # only the out-of-range rows (1e-9 scale is in range)
    print(f"N={N} D={D} K={K}: rechecked rows {int(st[0])} ({int(st[1])} candidates), full scans {int(st[2])}")


def test_vq_tensor_core_search_nonfinite_and_cfg3_margin(cuda):
    """NaN / inf rows take the full exact scan (code 0 for NaN rows, like vq_kernel); at the cfg-3 shape the candidate margin
    has headroom: indices stay identical with the margin shrunk 8x (B200DM_TUNING hook), so the error bound of the fp16-split
    products is not tight."""
    import os
    from b200dm import _lib as L
    g = torch.Generator().manual_seed(5)
    K, D, N = 1024, 256, 128 * 1024
    cb = (torch.rand(K, D, generator=g) - 0.5) * 0.1
    x = torch.randn(N, D, generator=g) * 0.5
    x[5, 17] = float("nan")
    x[300, 0] = float("inf")
    x[301, 3] = -float("inf")
    (i0, q0, h0, _), (i1, q1, h1, st) = _vq_both(x, cb, cuda)
    assert torch.equal(i0, i1) and torch.equal(h0, h1) and int(i1[5]) == 0
    assert 3 <= int(st[2]) <= 8, st.tolist()
    frac = int(st[0]) / N
    os.environ["B200DM_TUNING"], os.environ["B200DM_VQ_MARGIN_SCALE"] = "1", "0.125"
    try:
        (_, _, _, _), (i2, _, _, st2) = _vq_both(x, cb, cuda)
    finally:
        del os.environ["B200DM_TUNING"], os.environ["B200DM_VQ_MARGIN_SCALE"]
    print(f"cfg-3 rows rechecked: {frac:.4%} at the proven margin, {int(st2[0]) / N:.4%} at 1/8 of it; mismatches at 1/8: {(i2 != i0).sum().item()}")
    assert torch.equal(i2, i0)
    assert L.debug_flag() == 0


@pytest.mark.parametrize("layout", ["DK", "KD"])
def test_vq_distribution_matrix(cuda, layout):
    """VectorQuantizer.get_code_indices(x, distribution=True) (vqvae3d_monai.py:165-177): the (N, K) squared-distance matrix
    ||x||^2 + ||e||^2 - 2 x.e itself, in the argmin's own fp32 arithmetic -- its row argmin IS get_code_indices(x), and it
    matches the oracle's fp32 matrix to rounding (different summation order of the D-term dot products)."""
    import b200dm
    N, D, K = 333, 64, 96
    vq = b200dm.VectorQuantizer(K, D, layout=layout)
    cb = OI.codebook(K, D, layout, seed=3)
    vq.set_embeddings(cb)
    x = OI.normal((N, D), 7, 0.5 if layout == "KD" else 0.05)
    dist = vq.get_code_indices(x.to(cuda), distribution=True)
    assert tuple(dist.shape) == (N, K) and dist.dtype == torch.float32
    ref = OF.code_distances(x, cb, layout)
    scale = ref.abs().max().item()
    assert (dist.cpu() - ref).abs().max().item() <= 2e-6 * max(scale, 1.0)
    idx = vq.get_code_indices(x.to(cuda))
    assert torch.equal(dist.argmin(1).cpu(), idx.cpu())      # torch.argmin: first minimum, like tf.argmin
