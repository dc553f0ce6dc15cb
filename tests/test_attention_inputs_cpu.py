"""The attention test's constructed inputs and its replay of the kernel's reference-maximum rule (test_attention_gpu.py), without a
device: the replay on hand-made tile maxima, and each construction in both storage types, doing what its GPU test relies on."""
import importlib.util
import os

import pytest
import torch

_spec = importlib.util.spec_from_file_location("attention_gpu_cases", os.path.join(os.path.dirname(__file__), "test_attention_gpu.py"))
A = importlib.util.module_from_spec(_spec)
_spec.loader.exec_module(A)


def test_replay_follows_the_threshold():
    # one row, key tile 2: tile maxima 0, 7.9, 8.1, 20, 27.5, 28.5 against the reference max in force
    s = torch.tensor([[0.0, -1.0, 7.9, 3.0, 8.1, 0.0, -5.0, 20.0, 27.5, 1.0, 28.5, 28.0]], dtype=torch.float64)
    grow, rise = A.replay_ref_max(s, 2)
    assert grow.tolist() == [[True, False, True, True, False, True]]
    assert torch.allclose(rise[0, 1:], torch.tensor([7.9, 8.1, 11.9, 7.5, 8.5], dtype=torch.float64))


@pytest.mark.parametrize("dtype", [torch.bfloat16, torch.float16])
@pytest.mark.parametrize("D", [64, 128, 256])
@pytest.mark.parametrize("kind", A.KINDS)
def test_construction_claims(kind, D, dtype):
    """keyed_inputs asserts each construction's claims itself; here, in addition, what the GPU tests rely on."""
    q, k, v, Lk = A.keyed_inputs(kind, 2, 200, D, "indicator", dtype=dtype)
    bkv = A.BKV[D]
    for t in (q, k):   # the inputs are storage-type values
        assert torch.equal(t, t.to(dtype).float())
    s = torch.einsum("bld,bLd->blL", q.double(), k.double()) * D ** -0.5 * A.LOG2E
    grow, rise = A.replay_ref_max(s, bkv)
    assert grow.shape[-1] == -(-Lk // bkv) == A.NTILE[kind]
    if kind == "staircase":     # every row corrects at every tile after the first
        assert grow.all()
    if kind == "threshold":     # corrections taken and skipped, p up to ~2^7.5 before a rescale
        assert grow[..., 1:].any() and not grow[..., 1:].all() and rise[..., 1:][~grow[..., 1:]].max() > 7
    if kind == "masked_tail":   # keys past Lk would score 0 and outweigh every real key by 2^30
        assert Lk % bkv != 0 and s.max() <= -30
    # indicator values: channel c is 1 exactly for the keys of tile c
    tile = torch.arange(Lk) // bkv
    assert torch.equal(v[0, :, : grow.shape[-1]], (tile[:, None] == torch.arange(grow.shape[-1])).float())
    assert not v[..., grow.shape[-1]:].any()


def test_staircase_at_cfg4_size_corrects_every_tile():
    rows = torch.tensor([0, 1, 16384, 32767])
    q, k, v, Lk = A.keyed_inputs("staircase", 1, 32768, 64, ntile=256, check_rows=rows, dtype=torch.bfloat16)
    assert Lk == 32768


def test_elementwise_bound_catches_a_tile_mass_error():
    """The bound is tight enough that one tile's mass off by 2 % fails, in both builds' U."""
    q, k, v, Lk = A.keyed_inputs("staircase", 1, 8, 64, "indicator")
    r, w = A.ref64(q, k, v, 64 ** -0.5)
    A.check_elementwise(r.float(), r, w, "exact")
    bad = r.clone()
    bad[..., 2] *= 1.02
    with pytest.raises(AssertionError, match="channel 2"):
        A.check_elementwise(bad.float(), r, w, "tile 2 mass + 2 %")
