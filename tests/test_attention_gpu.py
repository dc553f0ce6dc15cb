"""GPU parity of the flash-style tcgen05 attention kernel (csrc/attention.cu) vs the oracle's attention_core
(softmax(q k^T * scale) v over flattened voxel tokens; networks/dm3d.py:51-61, conditional_dm3d.py:162-184).

Tolerance (stated): q, k, v are 16-bit on both sides, scores / softmax statistics / accumulation are fp32 on both sides; the
kernel rounds the UNNORMALISED probabilities to the storage type before P.V (the oracle does not round them) and writes 16-bit
outputs: rel-L2 <= 1.28 U, max-abs <= 5.12 U * max|ref|, U the unit roundoff of the storage type (2^-8 bf16, 2^-11 fp16).

Element by element, against fp64 (ref64): with p_i = exp(scale s_i - max), r = sum p_i v_i / sum p_i (+ residual) and
W_c = sum p_i |v_ic| / sum p_i,

    |o - r| <= U |r| + ETA + (KAPPA U + EPS) W_c

U |r| and ETA are the output's rounding (ETA: half the storage type's smallest subnormal, for outputs below its normal range);
KAPPA U W_c is the rounding of each p to the storage type before P.V (KAPPA = 2 in fp16, where the row sum adds the rounded
p and so errs too); EPS W_c is what fp32 adds: score accumulation, ex2.approx and the fp32 sums of O and l.  The bound holds
while the kernel's p stay in the storage type's normal range (p >= 2^-14 in fp16; always in bf16), which every input below
keeps to.  A wrong correction factor, mask or residual moves whole rows or tiles by far more than U, wherever it lands."""
import math

import numpy as np
import pytest
import torch

from b200dm import _lib
from oracle import ops as O

pytestmark = pytest.mark.gpu

ACT = _lib.ACT_DTYPE
U = 2 ** -8 if _lib.precision() == "bf16" else 2 ** -11   # unit roundoff of the storage type: its largest relative rounding error
KAPPA = 1 if _lib.precision() == "bf16" else 2
ETA = 2 ** -134 if _lib.precision() == "bf16" else 2 ** -25
# fp32's share, measured on a B200 over every case of this file in both builds: none was needed.  The error beyond the output's
# rounding, (|o - r| - U |r| - ETA) / W, peaked at 0.56 U (bf16) and 0.61 U (fp16), inside KAPPA U, and at 0.08 U on the cfg-4
# staircase rows, whose scores reach ~2400 log2 units
EPS = 0.0

# The two constants of flash_attn_kernel (csrc/attention.cu) the constructions below are built around: the key tile per head
# dim (b200dm_attention_plan_create: bkv) and the reference-max threshold (`grow`: a tile max above m_ref + 8, log2 units).
BKV = {64: 128, 128: 128, 256: 64}
GROW = 8.0
LOG2E = math.log2(math.e)


def _r(t, dtype=None):
    return t.to(dtype or ACT).to(torch.float32)


def _rand(shape, seed, scale=1.0, dtype=None):
    return _r(torch.randn(shape, generator=torch.Generator().manual_seed(seed)) * scale, dtype)


def _run(cuda, q, k, v, scale, residual=None, strided=False):
    """strided: q and k are the column blocks [:, :, :D] / [:, :, D:] of (B, L, 2D) tensors (the fused [q | k] Dense layout)
    whose other half is NaN, so a read outside the block would show."""
    from b200dm import ops, _lib
    vt = v.transpose(1, 2).contiguous()
    dq, dk = q.to(cuda, ACT), k.to(cuda, ACT)
    if strided:
        D = q.shape[-1]
        wq = torch.full((*q.shape[:2], 2 * D), float("nan"), dtype=ACT, device=cuda)
        wk = torch.full((*k.shape[:2], 2 * D), float("nan"), dtype=ACT, device=cuda)
        wq[..., :D], wk[..., D:] = dq, dk
        dq, dk = wq[..., :D], wk[..., D:]
    o = ops.attention(dq, dk, vt.to(cuda, ACT), scale, residual=None if residual is None else residual.to(cuda, ACT))
    torch.cuda.synchronize()
    assert _lib.debug_flag() == 0, "tcgen05/TMA pipeline watchdog fired"
    return o.float().cpu()


def ref64(q, k, v, scale, residual=None):
    """fp64 softmax(scale q k^T) v (+ residual) and W = softmax(scale q k^T) |v|, the weight the element-wise bound scales by."""
    s = torch.einsum("bld,bLd->blL", q.double(), k.double()) * scale
    p = torch.exp(s - s.amax(-1, keepdim=True))
    l = p.sum(-1, keepdim=True)
    v = v.double()
    r = torch.bmm(p, v) / l
    w = torch.bmm(p, v.abs()) / l
    return (r if residual is None else r + residual.double()), w


def check_elementwise(o, r, w, what):
    """Assert |o - r| <= U |r| + ETA + (KAPPA U + EPS) W for every element; print the largest share of W the error takes
    beyond the output's rounding (at most KAPPA U + EPS)."""
    err = (o.double() - r).abs()
    excess = err - (U * r.abs() + ETA + (KAPPA * U + EPS) * w)
    pos = w > 0
    share = ((err - U * r.abs() - ETA)[pos] / w[pos]).max().item() if pos.any() else 0.0
    print(f"{what}: max (|o - r| - U|r| - ETA) / W = {share:.3e} = {share / U:.3f} U")
    if excess.max().item() > 0:
        b, i, c = np.unravel_index(int(excess.argmax()), err.shape)
        raise AssertionError(
            f"{what}: {int((excess > 0).sum())} of {err.numel()} elements out of bound; worst at sample {b} row {i} channel "
            f"{c}: o {o[b, i, c].item():.6g} ref {r[b, i, c].item():.6g} W {w[b, i, c].item():.3g}\n"
            f"  that row, channels 0-7 (with tile-indicator values channel j is key tile j's softmax mass):\n"
            f"  kernel {o[b, i, :8].double().numpy()}\n  fp64   {r[b, i, :8].numpy()}")


# ------------------------------------------------------------------ inputs built to drive the online-softmax branches
def replay_ref_max(s_log2, bkv):
    """CPU replay of the kernel's reference-maximum rule over scores s_log2 = scale log2(e) q.k (..., Lk).
    Returns (grow, rise), both (..., ntile): whether tile j moved the reference max (tile 0 always does), and by how much
    the tile's max exceeds the reference max in force before it (+inf for tile 0)."""
    m_ref = torch.full(s_log2.shape[:-1], -math.inf, dtype=torch.float64)
    grow, rise = [], []
    for j0 in range(0, s_log2.shape[-1], bkv):
        mx = s_log2[..., j0:j0 + bkv].amax(-1)
        g = mx > m_ref + GROW
        grow.append(g)
        rise.append(mx - m_ref)
        m_ref = torch.where(g, mx, m_ref)
    return torch.stack(grow, -1), torch.stack(rise, -1)


# tile levels (log2 units of scale s) per construction
LEVELS = {
    "staircase": lambda nt: [9.5 * j for j in range(nt)],                      # every tile corrects
    "threshold": lambda nt: [16 * (j // 2) + 7.5 * (j % 2) for j in range(nt)],    # rises 7.5, 8.5, ...: skip, take, ...
    "huge_jump": lambda nt: [0.0, 3.0, 1.0][:nt - 1] + [150.0],                # factor 2^-147: ex2.approx.ftz flushes it to 0
    "dominant_first": lambda nt: [0.0] + [-8.0, -4.0, -9.0][:nt - 1],
    "dominant_last": lambda nt: [0.0, -3.0, 2.0][:nt - 1] + [20.0],
    "masked_tail": lambda nt: [-31.0] * nt,                                    # a key past Lk would score 0, above all of them
}
KINDS = list(LEVELS)
NTILE = {"staircase": 5, "threshold": 6, "huge_jump": 4, "dominant_first": 4, "dominant_last": 4, "masked_tail": 4}


def keyed_inputs(kind, B, Lq, D, values="random", ntile=None, seed=0, check_rows=None, dtype=None):
    """q, k, v (fp32 holding storage-type values) and Lk for one construction, scale = D^-0.5.
    Every row sees the same per-key score offset: q[..., 0:2] = 1 and k[..., 0:2] = hi, lo with hi + lo the offset (one 16-bit
    value cannot place a level to the fraction of a log2 unit the threshold case needs).  A key of tile j sits u in [0, 3]
    log2 units below level j, one key per tile at u = 0, plus small random components that make the rows differ.
    values: "random" (1 + N(0, 1): every channel's output is order 1) or "indicator" (channel c is 1 for the keys of tile c:
    the output reads each tile's softmax mass).  The claims of the construction are asserted with replay_ref_max on the rows
    check_rows (all by default)."""
    dtype = dtype or ACT
    bkv = BKV[D]
    nt = ntile or NTILE[kind]
    Lk = nt * bkv if kind != "masked_tail" else (nt - 1) * bkv + 40
    scale = D ** -0.5
    c = scale * LOG2E
    g = torch.Generator().manual_seed(seed)
    level = torch.tensor(LEVELS[kind](nt), dtype=torch.float64)
    tile = torch.arange(Lk) // bkv
    u = 3 * torch.rand(B, Lk, generator=g, dtype=torch.float64)
    u[:, torch.arange(0, Lk, bkv) + torch.randint(0, 40, (nt,), generator=g)] = 0
    off = (level[tile] - u) / c
    hi = off.to(dtype).double()
    lo = (off - hi).to(dtype).double()
    q = _r(torch.randn(B, Lq, D, generator=g) * 0.2, dtype)
    k = _r(torch.randn(B, Lk, D, generator=g) * 0.2, dtype)
    q[..., :2] = 1
    k[..., 0], k[..., 1] = hi.float(), lo.float()
    if values == "random":
        v = _r(1 + torch.randn(B, Lk, D, generator=g), dtype)
    else:
        v = (tile[None, :, None] % D == torch.arange(D)).float().expand(B, Lk, D).contiguous()

    qc = q if check_rows is None else q[:, check_rows]
    s = torch.einsum("bld,bLd->blL", qc.double(), k.double()) * c
    grow, rise = replay_ref_max(s, bkv)
    later = grow[..., 1:]
    if kind == "staircase":
        assert later.all(), "staircase: a row skips a correction"
    elif kind == "threshold":
        assert later[..., 1::2].all() and not later[..., 0::2].any(), "threshold: corrections not taken and skipped in turn"
        assert rise[..., 1::2].min() > 7, "threshold: no row reaches p = 2^7 unrescaled"
    elif kind == "huge_jump":
        assert later[..., -1].all() and rise[..., -1].min() > 126 and not later[..., :-1].any(), "huge_jump: last rise <= 126"
    elif kind == "dominant_first":
        assert not later.any(), "dominant_first: a later tile moves the reference max"
    elif kind == "dominant_last":
        assert later[..., -1].all(), "dominant_last: the last tile does not correct"
    else:
        assert Lk % bkv and s.max() <= -30, "masked_tail: Lk a multiple of the key tile, or a real key scores above -30"
    if kind.startswith("dominant"):
        p = torch.softmax(s / LOG2E, -1)
        j = 0 if kind == "dominant_first" else nt - 1
        assert p[..., j * bkv:(j + 1) * bkv].sum(-1).min() > 0.9, f"{kind}: tile {j} holds less than 0.9 of the mass"
    return q, k, v, Lk


CASES = [
    # B, Lq, Lk, D, residual
    (2, 512, 512, 256, True),     # cfg-2 attention site: 8^3 tokens, d = 256
    (8, 512, 512, 256, False),
    (1, 64, 64, 256, False),      # cfg-1: 4^3 tokens
    (2, 8, 8, 256, True),         # 2^3 tokens (S=8 test networks): one ragged tile
    (1, 1024, 1024, 64, False),   # d = 64 (cfg-4 geometry, short)
    (1, 200, 72, 128, True),      # ragged query and key counts, d = 128
    (2, 4096, 4096, 64, False),   # many key tiles: online-softmax reference-max updates
]


@pytest.mark.parametrize("B,Lq,Lk,D,res", CASES)
def test_flash_attention_matches_oracle(cuda, B, Lq, Lk, D, res):
    q, k, v = _rand((B, Lq, D), 1), _rand((B, Lk, D), 2), _rand((B, Lk, D), 3)
    r = _rand((B, Lq, D), 4) if res else None
    scale = float(D) ** -0.5
    ref = O.attention_core(q, k, v, scale)
    if res:
        ref = ref + r
    o = _run(cuda, q, k, v, scale, r)
    rel = ((o - ref).norm() / ref.norm()).item()
    mx = (o - ref).abs().max().item() / ref.abs().max().item()
    print(f"attention B{B} Lq{Lq} Lk{Lk} D{D}: rel-L2 {rel:.3e} max-abs/max {mx:.3e}")
    assert rel <= 1.28 * U and mx <= 5.12 * U, (rel, mx)
    check_elementwise(o, *ref64(q, k, v, scale, r), f"B{B} Lq{Lq} Lk{Lk} D{D}{' +res' if res else ''}")


def test_flash_attention_peaked_scores(cuda):
    """Large score range (|s*scale| up to ~40): exercises the lazy rescale of the TMEM accumulator."""
    B, L, D = 1, 1024, 64
    q, k, v = _rand((B, L, D), 1, 3.0), _rand((B, L, D), 2, 3.0), _rand((B, L, D), 3)
    scale = float(D) ** -0.5
    ref = O.attention_core(q, k, v, scale)
    o = _run(cuda, q, k, v, scale)
    rel = ((o - ref).norm() / ref.norm()).item()
    print(f"peaked scores: rel-L2 {rel:.3e}")
    assert rel <= 2.05 * U, rel


def test_flash_attention_full_size_properties(cuda):
    """cfg-4 size (L = 32768 tokens, d = 64), where the oracle's (L, L) score matrix is 4 GiB: size-independent properties.
    (1) identical value rows -> every output row equals that row (softmax weights sum to 1);
    (2) zero keys -> uniform weights -> every output row equals the mean value row."""
    B, L, D = 1, 32768, 64
    q = _rand((B, L, D), 1)
    k = _rand((B, L, D), 2)
    v0 = _rand((1, 1, D), 3)
    o = _run(cuda, q, k, v0.expand(B, L, D).contiguous(), D ** -0.5)
    assert (o - v0).abs().max().item() <= 5.12 * U * v0.abs().max().item()
    v = _rand((B, L, D), 4)
    o = _run(cuda, q, torch.zeros(B, L, D), v, D ** -0.5)
    mean = v.mean(1, keepdim=True)
    assert (o - mean).abs().max().item() <= 2e-3 + 5.12 * U * mean.abs().max().item()


def test_flash_attention_strided_q_k(cuda):
    """q and k as column blocks of one wider projection output (fused [q | k] Dense): row stride 2D, k 2D*2 bytes... offset D."""
    from b200dm import ops, _lib
    B, L, D = 2, 512, 256
    qk = _rand((B, L, 2 * D), 1)
    v = _rand((B, L, D), 2)
    dqk = qk.to(cuda, ACT)
    o = ops.attention(dqk[..., :D], dqk[..., D:], v.transpose(1, 2).contiguous().to(cuda, ACT), D ** -0.5)
    torch.cuda.synchronize()
    assert _lib.debug_flag() == 0
    ref = O.attention_core(qk[..., :D], qk[..., D:], v, D ** -0.5)
    o = o.float().cpu()
    assert ((o - ref).norm() / ref.norm()).item() <= 1.28 * U
    check_elementwise(o, *ref64(qk[..., :D], qk[..., D:], v, D ** -0.5), f"strided q/k B{B} L{L} D{D}")


# B, Lq, Lk, D, residual, strided q/k: every Lq in {8, 127, 128, 129, 200} and Lk in {8, BKV - 8, BKV, BKV + 8, 3 BKV + 8} at
# each head dim, B in {1, 3}, with and without a residual; strided at d = 64 and 128 (d = 256: test_flash_attention_strided_q_k)
GRID = [
    (1, 8, 8, 64, False, False),
    (3, 127, 120, 64, True, False),
    (3, 129, 128, 64, False, True),
    (1, 200, 136, 64, True, True),
    (3, 128, 392, 64, True, False),
    (1, 127, 392, 64, False, False),
    (3, 200, 8, 64, True, False),
    (1, 129, 8, 128, True, False),
    (3, 8, 120, 128, False, True),
    (1, 128, 128, 128, True, False),
    (3, 200, 136, 128, True, True),
    (3, 127, 392, 128, False, False),
    (1, 200, 392, 128, True, True),
    (3, 128, 120, 128, False, False),
    (3, 127, 8, 256, False, False),
    (1, 129, 56, 256, True, False),
    (3, 128, 64, 256, True, False),
    (1, 8, 72, 256, False, False),
    (3, 200, 200, 256, True, False),
    (1, 128, 200, 256, False, False),
    (3, 129, 72, 256, True, False),
]


@pytest.mark.parametrize("B,Lq,Lk,D,res,strided", GRID)
def test_flash_attention_shape_grid(cuda, B, Lq, Lk, D, res, strided):
    q, k, v = _rand((B, Lq, D), 11), _rand((B, Lk, D), 12), _rand((B, Lk, D), 13)
    r = _rand((B, Lq, D), 14) if res else None
    o = _run(cuda, q, k, v, D ** -0.5, r, strided)
    check_elementwise(o, *ref64(q, k, v, D ** -0.5, r), f"B{B} Lq{Lq} Lk{Lk} D{D}{' +res' if res else ''}{' strided' if strided else ''}")


# every construction at every head dim with both kinds of values, and once with a residual (the head dim rotating)
CONSTRUCTED = [(kind, D, values, False) for kind in KINDS for D in (64, 128, 256) for values in ("random", "indicator")]
CONSTRUCTED += [(kind, (64, 128, 256)[i % 3], "random", True) for i, kind in enumerate(KINDS)]


@pytest.mark.parametrize("kind,D,values,res", CONSTRUCTED)
def test_flash_attention_constructed_scores(cuda, kind, D, values, res):
    B, Lq = 2, 200
    q, k, v, Lk = keyed_inputs(kind, B, Lq, D, values)
    r = _rand((B, Lq, D), 5) if res else None
    o = _run(cuda, q, k, v, D ** -0.5, r)
    check_elementwise(o, *ref64(q, k, v, D ** -0.5, r), f"{kind} D{D} Lk{Lk} {values}{' +res' if res else ''}")


@pytest.mark.parametrize("keys", ["random", "staircase"])
def test_flash_attention_cfg4_rows(cuda, keys):
    """cfg-4 size (B = 1, L = 32768, d = 64) against fp64 on 512 query rows: the first and last query tile and 256 rows across
    the range.  Staircase keys: 256 key tiles, every one a correction, scores up to ~2400 log2 units."""
    B, L, D = 1, 32768, 64
    rows = torch.cat([torch.arange(128), torch.linspace(128, L - 129, 256).long(), torch.arange(L - 128, L)])
    if keys == "random":
        q, k, v = _rand((B, L, D), 21), _rand((B, L, D), 22), _rand((B, L, D), 23)
    else:
        q, k, v, _ = keyed_inputs("staircase", B, L, D, ntile=L // BKV[D], check_rows=rows)
    o = _run(cuda, q, k, v, D ** -0.5)
    check_elementwise(o[:, rows], *ref64(q[:, rows], k, v, D ** -0.5), f"cfg-4 {keys} keys, {len(rows)} rows")


@pytest.mark.parametrize("D", [64, 128, 256])
def test_flash_attention_deterministic(cuda, D):
    """One AttnPlan run twice, and the same attention recorded in a step program: bit-identical outputs."""
    from b200dm import ops, _lib
    from b200dm.program import Program
    B, Lq = 2, 200
    q, k, v, Lk = keyed_inputs("staircase", B, Lq, D)
    dq, dk, dvt = q.to(cuda, ACT), k.to(cuda, ACT), v.transpose(1, 2).contiguous().to(cuda, ACT)
    dr = _rand((B, Lq, D), 6).to(cuda, ACT)
    o1 = torch.empty(B, Lq, D, dtype=ACT, device=cuda)
    plan = ops.AttnPlan(dq, dk, dvt, o1, D ** -0.5, dr)
    a = plan.run().clone()
    b = plan.run().clone()
    o2 = torch.empty_like(o1)
    pr = Program(cuda)
    pr.attention(dq, dk, dvt, o2, D ** -0.5, dr)
    pr.run()
    torch.cuda.synchronize()
    assert _lib.debug_flag() == 0
    assert torch.equal(a.view(torch.int16), b.view(torch.int16)), "AttnPlan: second run differs from the first"
    assert torch.equal(a.view(torch.int16), o2.view(torch.int16)), "Program.attention differs from AttnPlan"
