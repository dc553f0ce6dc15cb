"""GPU parity at BASELINE.json's FULL sizes, where the CPU oracle would take minutes to hours: size-independent properties.

cfg-2 (conditional U-Net, 32^3 x 256 latent, batch 8): batch-permutation equivariance of the whole denoise chain (samples are
independent -- the property multi-GPU sharding rests on); exact homogeneity of the conv kernels (scaling the input by a power of
two scales the fp32 accumulators exactly); cfg-3 VQ (524288 rows, K = 1024): idempotence on codebook rows and agreement with a
float64 check of sampled rows."""
import types

import numpy as np
import pytest
import torch

from b200dm import _lib
from oracle import init as OI, first_stage as OF

pytestmark = pytest.mark.gpu

ACT = _lib.ACT_DTYPE
U = 2 ** -8 if _lib.precision() == "bf16" else 2 ** -11   # unit roundoff of the storage type: its largest relative rounding error


def _flag_ok():
    from b200dm import _lib
    torch.cuda.synchronize()
    assert _lib.debug_flag() == 0, "tcgen05/TMA pipeline watchdog fired"


def test_cfg2_chain_is_batch_permutation_equivariant(cuda):
    import b200dm
    S, C, B, T = 32, 256, 8, 1000
    dm = b200dm.ConditionalDiffusionModel(S, 1024, C, None, types.SimpleNamespace(timesteps=T, num_gpus=1, kernel_resize=False, bs=B))
    shape = (B, S, S, S, C)
    g = torch.Generator().manual_seed(5)
    x_T = torch.randn(shape, generator=g)
    ctx = torch.tensor([0, 1, 1, 0, 1, 0, 0, 1])
    # injected noise is zero -> the chain is a deterministic function of (x_T, ctx) per sample
    zero = {i: torch.zeros(1) .expand(shape) for i in range(T)}
    lat = dm.generate(shape, last_step=T - 3, x_T=x_T, context=ctx, noise=lambda i: zero[i]).cpu()
    _flag_ok()
    assert torch.isfinite(lat).all()
    perm = torch.tensor([3, 0, 7, 1, 6, 2, 5, 4])
    lat_p = dm.generate(shape, last_step=T - 3, x_T=x_T[perm], context=ctx[perm], noise=lambda i: zero[i]).cpu()
    _flag_ok()
    assert torch.equal(lat_p, lat[perm]), "a sample's latents depend on its position / neighbours in the batch"
    # and the samples really differ from each other and from their input
    assert (lat[0] - lat[1]).abs().max() > 1e-3 and (lat - x_T).abs().max() > 1e-3


@pytest.mark.parametrize("case", ["halo64", "halo128", "halo32", "halo32s", "pair", "gemm1", "down", "up", "up8", "up32"])
def test_fullsize_convs_are_exactly_homogeneous(cuda, case):
    """y(4 x) == 4 y(x) bit for bit (no bias): every product and partial sum scales by an exact power of two, so any
    dropped / duplicated tap, tile or K chunk at the full cfg-2 shapes shows up, without an oracle run.  Exact where y is a
    normal number of the storage type; a subnormal y (1 in ~2e4 outputs in fp16, none in bf16) is rounded on a grid that
    does not scale, so 4 y(x) and y(4 x) may differ there by up to one quantum of the scaled grid."""
    from b200dm import ops, _lib
    B = 8
    cfg = dict(halo64=(32, 64, 64, 3, 1, _lib.CONV_DIRECT), halo128=(16, 128, 128, 3, 1, _lib.CONV_DIRECT),
               halo32=(32, 256, 32, 3, 1, _lib.CONV_DIRECT), halo32s=(32, 32, 32, 3, 1, _lib.CONV_DIRECT),
               pair=(8, 256, 256, 3, 1, _lib.CONV_DIRECT), gemm1=(8, 256, 1024, 1, 1, _lib.CONV_DIRECT),
               down=(32, 64, 64, 3, 2, _lib.CONV_DIRECT), up=(16, 128, 128, 3, 1, _lib.CONV_PARITY),
               up8=(8, 256, 256, 3, 1, _lib.CONV_PARITY), up32=(32, 64, 32, 3, 1, _lib.CONV_PARITY))[case]
    S, cin, cout, k, stride, mode = cfg
    g = torch.Generator().manual_seed(1)
    x = torch.randn(B, S, S, S, cin, generator=g).to(ACT)
    w = (torch.randn(k, k, k, cin, cout, generator=g) / np.sqrt(k ** 3 * cin)).to(ACT).float()
    y1 = ops.conv3d(x.to(cuda), w, mode=mode, stride=stride, y_dtype=ACT).float()
    y4 = ops.conv3d((x.float() * 4).to(ACT).to(cuda), w, mode=mode, stride=stride, y_dtype=ACT).float()
    _flag_ok()
    assert torch.isfinite(y1).all() and y1.abs().max() > 0.1
    normal = y1.abs() >= torch.finfo(ACT).tiny
    assert torch.equal(y4[normal], y1[normal] * 4)
    assert bool(((y4 - y1 * 4).abs()[~normal] <= 4 * torch.finfo(ACT).tiny * torch.finfo(ACT).eps).all())
    # spot-check 64 output voxels against a direct fp64 evaluation of the Keras 'same' / upsample+conv definition
    xs, idx = x.float(), torch.randint(0, y1.shape[1], (64, 3), generator=g)
    for (d, h, ww) in idx.tolist():
        n = (d + h + ww) % B
        acc = torch.zeros(cout, dtype=torch.float64)
        for kd in range(k):
            for kh in range(k):
                for kw in range(k):
                    if mode == _lib.CONV_PARITY:      # conv3 on the nearest-upsampled tensor, pad 1
                        pd, ph, pw = d + kd - 1, h + kh - 1, ww + kw - 1
                        if min(pd, ph, pw) < 0 or max(pd, ph, pw) >= 2 * S:
                            continue
                        src = xs[n, pd // 2, ph // 2, pw // 2]
                    else:                              # TF 'same': pad_before = total // 2 (0 for k3 s2 on even sizes)
                        pb = max((y1.shape[1] - 1) * stride + k - S, 0) // 2
                        pd, ph, pw = d * stride + kd - pb, h * stride + kh - pb, ww * stride + kw - pb
                        if min(pd, ph, pw) < 0 or max(pd, ph, pw) >= S:
                            continue
                        src = xs[n, pd, ph, pw]
                    acc += src.double() @ w[kd, kh, kw].double()
        got = y1[n, d, h, ww].cpu().double()
        assert (got - acc).abs().max() <= 5 * U * acc.abs().max() + 1e-3, (case, d, h, ww)


def test_cfg3_vq_fullsize_properties(cuda):
    import b200dm
    N, K, D = 16 * 32 ** 3, 1024, 256
    vq = b200dm.VectorQuantizer(K, D, layout="KD")
    cb = OI.codebook(K, D, "KD", seed=3)
    vq.set_embeddings(cb)
    g = torch.Generator().manual_seed(7)
    want = torch.randint(0, K, (N,), generator=g)
    rows = cb[want]                                    # every input row IS a codebook row
    q, idx, perp = vq.quantize(rows.view(16, 32, 32, 32, D).to(cuda))
    assert torch.equal(idx.cpu(), want), "codebook rows do not map to themselves"
    assert torch.equal(q.cpu().view(N, D), rows)       # gather is exact; quantize(quantize(x)) == quantize(x)
    assert 0.9 * K < perp <= K
    assert int(vq.codebooks_used.sum()) == N
    # noisy rows: float64 check of 512 sampled rows (first-min on ties)
    x = rows[:4096] + 0.02 * torch.randn(4096, D, generator=g)
    idx2 = vq.get_code_indices(x.to(cuda)).cpu()
    d64 = (x[:512].double() ** 2).sum(1, keepdim=True) + (cb.double() ** 2).sum(1)[None] - 2 * x[:512].double() @ cb.double().t()
    best = d64.argmin(1)
    margin = d64.sort(1).values
    clear = (margin[:, 1] - margin[:, 0]) > 1e-4       # away from fp32-level near ties
    assert torch.equal(idx2[:512][clear], best[clear])
