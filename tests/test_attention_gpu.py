"""GPU parity of the flash-style tcgen05 attention kernel (csrc/attention.cu) vs the oracle's attention_core
(softmax(q k^T * scale) v over flattened voxel tokens; networks/dm3d.py:51-61, conditional_dm3d.py:162-184).

Tolerance (stated): q, k, v are 16-bit on both sides, scores / softmax statistics / accumulation are fp32 on both sides; the
kernel rounds the UNNORMALISED probabilities to the storage type before P.V (the oracle does not round them) and writes 16-bit
outputs: rel-L2 <= 1.28 U, max-abs <= 5.12 U * max|ref|, U the unit roundoff of the storage type (2^-8 bf16, 2^-11 fp16)."""
import numpy as np
import pytest
import torch

from b200dm import _lib
from oracle import ops as O

pytestmark = pytest.mark.gpu

ACT = _lib.ACT_DTYPE
U = 2 ** -8 if _lib.precision() == "bf16" else 2 ** -11   # unit roundoff of the storage type: its largest relative rounding error


def _r(t):
    return t.to(ACT).to(torch.float32)


def _rand(shape, seed, scale=1.0):
    return _r(torch.randn(shape, generator=torch.Generator().manual_seed(seed)) * scale)


def _run(cuda, q, k, v, scale, residual=None):
    from b200dm import ops, _lib
    vt = v.transpose(1, 2).contiguous()
    o = ops.attention(q.to(cuda, ACT), k.to(cuda, ACT), vt.to(cuda, ACT), scale,
                      residual=None if residual is None else residual.to(cuda, ACT))
    torch.cuda.synchronize()
    assert _lib.debug_flag() == 0, "tcgen05/TMA pipeline watchdog fired"
    return o.float().cpu()


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
