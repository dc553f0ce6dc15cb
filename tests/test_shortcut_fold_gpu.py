"""The 1^3 shortcut of a width-changing ResidualBlock folded into conv2's K loop (b200dm_conv_plan_set_shortcut).

At the cfg-2 U-Net's folded geometries (batch 8) the folded conv2 is compared with the two-launch form built through the same
public API (the shortcut conv stores its output in the 16-bit type, conv2 adds it as its residual): they differ by that one
removed rounding.  Both are also checked against an fp64 evaluation of the Keras definition at sampled voxels, the folded
form for exact homogeneity, and the compiled cfg-2 program for its launch count and FLOPs.
"""
import numpy as np
import pytest
import torch
import torch.nn.functional as F

pytestmark = pytest.mark.gpu

# S, conv2 width, shortcut C_in of x, of skip: down.0.res.0 (ragged 32-channel x), up.0.res.1, up.0.res.2 (ragged skip),
# up.1.res.1 (16^3), up.2.res.0 (8^3, pair-slab tiles)
CASES = [(32, 64, 32, 0), (32, 64, 128, 64), (32, 64, 64, 32), (16, 128, 256, 128), (8, 256, 256, 256)]
B = 8


def _flag_ok():
    from b200dm import _lib
    torch.cuda.synchronize()
    assert _lib.debug_flag() == 0, "tcgen05/TMA pipeline watchdog fired"


def _operands(S, w, c0, c1, seed):
    from b200dm import _lib as L
    g = torch.Generator().manual_seed(seed)
    act = lambda c: torch.randn(B, S, S, S, c, generator=g).to(L.ACT_DTYPE)  # noqa: E731
    h, x, skip = act(w), act(c0), act(c1) if c1 else None
    w2 = (torch.randn(3, 3, 3, w, w, generator=g) / np.sqrt(27 * w)).to(L.ACT_DTYPE).float()
    wsc = (torch.randn(1, 1, 1, c0 + c1, w, generator=g) / np.sqrt(c0 + c1)).to(L.ACT_DTYPE).float()
    b2, bsc = torch.randn(w, generator=g) * 0.1, torch.randn(w, generator=g) * 0.1
    return h, x, skip, w2, wsc, b2, bsc


def _folded(cuda, h, x, skip, w2, wsc, b2, bsc):
    """conv2(h) + b2 + Wsc [x | skip] + bsc in one launch; biases None: no bias."""
    from b200dm import _lib as L, ops
    S, w = h.shape[1], h.shape[-1]
    desc = ops.make_conv_desc(L.CONV_DIRECT, B, (S, S, S), w, 0, w, 3, 1)
    sdesc = ops.make_conv_desc(L.CONV_DIRECT, B, (S, S, S), x.shape[-1], skip.shape[-1] if skip is not None else 0, w, 1, 1)
    wp = ops.pack_conv_weights(desc, w2).to(cuda)
    y = torch.empty(B, S, S, S, w, dtype=L.ACT_DTYPE, device=cuda)
    hd, xd, sd = h.to(cuda), x.to(cuda), skip.to(cuda) if skip is not None else None
    plan = ops.ConvPlan(desc, hd, wp, y, bias=b2.to(cuda) if b2 is not None else None)
    wf = ops.fold_shortcut_weights(wp, sdesc, ops.pack_conv_weights(sdesc, wsc))
    assert plan.set_shortcut(xd, sd, wf, (b2 + bsc).to(cuda) if b2 is not None else None)
    assert plan.info["halo"] == 1
    plan.run()
    _flag_ok()
    return y.float().cpu()


def _ref64(h, x, skip, w2, wsc, b2, bsc, vox):
    """fp64 Keras definition at voxels [(n, d, h, w)]: 'same' 3^3 conv of h + 1^3 conv of the concat [x | skip] + both biases."""
    hp = F.pad(h.double(), (0, 0, 1, 1, 1, 1, 1, 1))
    xs = torch.cat([x, skip], dim=-1).double() if skip is not None else x.double()
    out = []
    for n, d, hh, ww in vox:
        patch = hp[n, d:d + 3, hh:hh + 3, ww:ww + 3, :]                       # (3, 3, 3, C)
        v = torch.einsum("abci,abcio->o", patch, w2.double()) + b2.double()
        v += xs[n, d, hh, ww] @ wsc[0, 0, 0].double() + bsc.double()
        out.append(v)
    return torch.stack(out)


def _voxels(S, seed, k=48):
    g = torch.Generator().manual_seed(seed)
    vox = torch.randint(0, S, (k, 4), generator=g)
    vox[:, 0] %= B
    vox[:4, 1:] = torch.tensor([[0, 0, 0], [S - 1, S - 1, S - 1], [0, S - 1, 0], [S - 1, 0, S - 1]])   # corners: zero padding
    return [tuple(v) for v in vox.tolist()]


@pytest.mark.parametrize("S,w,c0,c1", CASES)
def test_folded_matches_two_launch_form(cuda, S, w, c0, c1):
    from b200dm import _lib as L, ops
    h, x, skip, w2, wsc, b2, bsc = _operands(S, w, c0, c1, seed=S + c0 + c1)
    yf = _folded(cuda, h, x, skip, w2, wsc, b2, bsc)
    # two-launch form: the shortcut conv stores r in the 16-bit type, conv2 reads it back as its residual
    r = ops.conv3d(x.to(cuda), wsc, bias=bsc.to(cuda), x1=skip.to(cuda) if skip is not None else None)
    y2 = ops.conv3d(h.to(cuda), w2, bias=b2.to(cuda), residual=r)
    _flag_ok()
    r, y2 = r.float().cpu(), y2.float().cpu()
    assert torch.isfinite(yf).all() and yf.abs().max() > 0.5
    # the removed rounding of r (<= u |r|) plus the output rounding of either form (<= u |y| each); u = unit roundoff of the
    # storage type; the fp32 sums of the two forms differ in order only (1e-5 of max|y|)
    u = torch.finfo(L.ACT_DTYPE).eps / 2
    err = (yf - y2).abs()
    bound = u * (r.abs() + 2 * y2.abs()) * 1.01 + 1e-5 * y2.abs().max()
    assert bool((err <= bound).all()), f"max excess {(err - bound).max().item():.3e}, max err {err.max().item():.3e}"
    assert (yf != y2).any(), "the folded form should skip the shortcut's rounding"
    vox = _voxels(S, seed=7)
    ref = _ref64(h, x, skip, w2, wsc, b2, bsc, vox)
    got = torch.stack([yf[v] for v in vox]).double()
    tol = u * ref.abs() + 1e-3 * ref.abs().max()
    assert bool(((got - ref).abs() <= tol).all()), f"vs fp64 Keras definition: max err {(got - ref).abs().max().item():.3e}"


@pytest.mark.parametrize("S,w,c0,c1", CASES)
def test_folded_is_exactly_homogeneous(cuda, S, w, c0, c1):
    """y(4 h, 4 x) == 4 y(h, x) bit for bit without bias: a dropped or duplicated shortcut chunk, slab or tap shows up.  Exact
    where y is a normal number of the storage type; a subnormal y (fp16 only) may differ by one quantum of the scaled grid."""
    from b200dm import _lib as L
    h, x, skip, w2, wsc, _, _ = _operands(S, w, c0, c1, seed=3 * S + c0)
    four = lambda t: (t.float() * 4).to(L.ACT_DTYPE) if t is not None else None  # noqa: E731
    y1 = _folded(cuda, h, x, skip, w2, wsc, None, None)
    y4 = _folded(cuda, four(h), four(x), four(skip), w2, wsc, None, None)
    assert y1.abs().max() > 0.5
    normal = y1.abs() >= torch.finfo(L.ACT_DTYPE).tiny
    assert torch.equal(y4[normal], y1[normal] * 4)
    assert bool(((y4 - y1 * 4).abs()[~normal] <= 4 * torch.finfo(L.ACT_DTYPE).tiny * torch.finfo(L.ACT_DTYPE).eps).all())


def test_cfg2_program_folds_every_width_change(cuda, monkeypatch):
    """The cfg-2 U-Net launches 12 fewer kernels per step with the shortcuts folded, with the same algorithmic FLOPs."""
    import b200dm
    from b200dm import ops

    def compiled():
        net = b200dm.build_model(32, 256, [64, 128, 256], [False, False, True, True], context_dim=1)
        net.compile(8, 1000)
        return net.prog

    folded = compiled()
    n_fold, fl_fold = folded.num_launches, folded.flops
    assert not any(note.endswith(".shortcut") for _, note, _ in folded.log)
    del folded
    monkeypatch.setattr(ops.ConvPlan, "set_shortcut", lambda self, *a: False)   # the two-launch form everywhere
    two = compiled()
    assert sum(1 for _, note, _ in two.log if note.endswith(".shortcut")) == 12
    assert two.num_launches - n_fold == 12
    assert fl_fold == pytest.approx(two.flops, rel=1e-12)
