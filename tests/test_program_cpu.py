"""Step-program ops are checked and sized when they are recorded, without a GPU: b200dm_program_add_X refuses a malformed
op with the code and b200dm_last_error() text of the direct entry point b200dm_X, and records nothing; a well-formed
program counts the launches its ops bind.  Every pointer below is a placeholder: nothing is launched or dereferenced."""
import ctypes as C
import os

import pytest

FAKE = 1 << 20   # 16-byte aligned placeholder device address


@pytest.fixture(scope="module")
def L():
    import __graft_entry__
    from b200dm import _lib
    if not os.path.exists(_lib._LIB_PATH):
        __graft_entry__.build()
    return _lib


@pytest.fixture
def prog(L):
    h = C.c_void_p()
    assert L.lib().b200dm_program_create(C.byref(h)) == 0
    yield h
    L.lib().b200dm_program_destroy(h)


def norm_desc(L, c0, c1=0, kind=0, groups=1, voxels=512, batch=2):
    return L.NormDesc(voxels=voxels, batch=batch, c0=c0, c1=c1, kind=kind, groups=groups, act=L.ACT_SILU,
                      x_dtype=L.BF16, y_dtype=L.BF16)


def ptrs(*addrs):
    return (C.c_void_p * len(addrs))(*addrs)


def malformed_ops(L):
    """(kind, direct entry point's arguments without the stream) -> the same op recorded through b200dm_program_add_<kind>."""
    upd = L.UpdateDesc(n_per_sample=4096, batch=2, sampler=2, t=5)   # sampler 2 does not exist
    for f in ("beta", "sqrt_alpha", "alpha_bar", "alpha_bar_prev", "sqrt_alpha_bar", "sqrt_alpha_bar_prev", "sqrt_one_minus_alpha_bar"):
        setattr(upd, f, FAKE)
    ex = L.NormExDesc(batch=1, out_d=3, out_h=4, out_w=4, c=8, kind=0, groups=1, upsample=1, x_dtype=L.BF16, y_dtype=L.BF16)
    ws = 1 << 30
    return [
        ("norm_act", "b200dm_norm_act_fwd", (C.byref(norm_desc(L, 12)), FAKE, None, FAKE, FAKE, None, FAKE)),
        ("norm_act", "b200dm_norm_act_fwd", (C.byref(norm_desc(L, 64, 64)), FAKE, None, FAKE, FAKE, None, FAKE)),   # x1 missing
        ("gn_stats", "b200dm_gn_stats", (C.byref(norm_desc(L, 24, kind=1, groups=3)), FAKE, 1e-6, FAKE, FAKE, ws)),
        ("gn_stats", "b200dm_gn_stats", (C.byref(norm_desc(L, 64, kind=1, groups=8)), FAKE, 1e-6, FAKE, FAKE, 16)),
        ("bn_stats", "b200dm_bn_stats", (FAKE, 4096, 12, FAKE, FAKE, 1e-3, FAKE, FAKE, FAKE, ws)),
        ("gn_finalize", "b200dm_gn_finalize", (FAKE, 2, 16, 30, 7, 4096, 1e-6, FAKE)),
        ("layernorm", "b200dm_layernorm_fwd", (FAKE, 4096, 12, 1e-3, 1, ptrs(FAKE), ptrs(FAKE), ptrs(FAKE))),
        ("layernorm", "b200dm_layernorm_fwd", (FAKE, 4096, 64, 1e-3, 2, ptrs(FAKE, FAKE + 4), ptrs(FAKE, FAKE), ptrs(FAKE, FAKE))),
        ("norm_act_ex", "b200dm_norm_act_ex", (C.byref(ex), FAKE, FAKE, FAKE, None, None, None, FAKE)),
        ("stats_f32", "b200dm_stats_f32", (FAKE, 2, 4096, 1e-6, FAKE, FAKE, 8)),
        ("softmax", "b200dm_softmax_rows", (FAKE, FAKE, 64, 0, 0.125)),
        ("update", "b200dm_ddpm_update", (C.byref(upd), FAKE, FAKE, None, FAKE, None)),
        ("step_advance", "b200dm_step_advance", (None, 1)),
    ]


def test_malformed_op_is_refused_when_recorded(L, prog):
    lib = L.lib()
    assert lib.b200dm_program_add_step_advance(prog, FAKE, 1) == 0
    for kind, direct, args in malformed_ops(L):
        rc = getattr(lib, direct)(*args, None)
        msg = lib.b200dm_last_error()
        assert rc == -1 and msg.startswith(direct[len("b200dm_"):].encode() + b":"), (direct, rc, msg)
        assert lib.b200dm_program_set_lane(prog, 99) != 0   # leaves another message behind
        assert getattr(lib, "b200dm_program_add_" + kind)(prog, *args) == rc, kind
        assert lib.b200dm_last_error() == msg, kind
        assert (lib.b200dm_program_num_ops(prog), lib.b200dm_program_num_launches(prog)) == (1, 1), kind


def test_null_program_is_refused(L):
    lib = L.lib()
    assert lib.b200dm_program_add_step_advance(None, FAKE, 1) == -1
    assert lib.b200dm_last_error() == b"program_add_step_advance: null program"


def test_launch_count_is_the_sum_of_the_bound_launches(L, prog):
    lib = L.lib()
    gn = norm_desc(L, 64, kind=1, groups=8)
    assert lib.b200dm_program_add_gn_stats(prog, C.byref(gn), FAKE, 1e-6, FAKE, FAKE, lib.b200dm_gn_stats_workspace(C.byref(gn))) == 0
    assert lib.b200dm_program_add_bn_stats(prog, FAKE, 4096, 64, FAKE, FAKE, 1e-3, FAKE, FAKE, FAKE, lib.b200dm_bn_stats_workspace(64)) == 0
    assert lib.b200dm_program_add_norm_act(prog, C.byref(norm_desc(L, 64, 32)), FAKE, FAKE, FAKE, FAKE, None, FAKE) == 0
    assert lib.b200dm_program_add_stats_f32(prog, FAKE, 2, 4096, 1e-6, FAKE, FAKE, lib.b200dm_stats_f32_workspace(2)) == 0
    assert lib.b200dm_program_add_gn_finalize(prog, FAKE, 2, 16, 64, 8, 4096, 1e-6, FAKE) == 0
    assert lib.b200dm_program_num_ops(prog) == 5
    assert lib.b200dm_program_num_launches(prog) == 2 + 4 + 1 + 2 + 1
