"""CPU checks of the drop-in boundary: libb200dm.so loads, exports every symbol include/b200dm.h declares, the ctypes
structs mirror the C structs, host-side entry points (no device work) behave, and the product path FAILS LOUDLY without a
GPU instead of falling back to anything.  No compute call is made here."""
import ctypes as C
import os
import re
import subprocess
import sys

import numpy as np
import pytest
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
HEADER = os.path.join(ROOT, "include", "b200dm.h")


@pytest.fixture(scope="module")
def L():
    import __graft_entry__  # noqa: F401  (puts ROOT on sys.path)
    import b200dm
    from b200dm import _lib
    if not os.path.exists(_lib._LIB_PATH):
        __graft_entry__.build()
    return _lib


def header_functions():
    src = open(HEADER).read()
    src = re.sub(r"/\*.*?\*/", "", src, flags=re.S)
    return sorted(set(re.findall(r"\b(b200dm_[a-z0-9_]+)\s*\(", src)))


def test_header_symbols_exported(L):
    lib = L.lib()
    names = header_functions()
    assert len(names) >= 30
    for n in names:
        assert hasattr(lib, n), f"{n} declared in include/b200dm.h but not exported by libb200dm.so"
    # the ctypes table binds exactly the header's functions: nothing undeclared is called from Python
    assert sorted(L.EXPORTED_SYMBOLS) == names


def test_dynamic_symbol_table_has_c_linkage(L):
    out = subprocess.run(["nm", "-D", "--defined-only", L._LIB_PATH], capture_output=True, text=True).stdout
    exported = {ln.split()[-1] for ln in out.splitlines() if " T " in ln}
    for n in header_functions():
        assert n in exported, f"{n} is not an unmangled (extern \"C\") export"


def test_version_and_error_string(L):
    lib = L.lib()
    assert lib.b200dm_version() == 101
    assert isinstance(lib.b200dm_last_error(), bytes)


def test_struct_layouts_match_header(L):
    """sizeof / field offsets of the ctypes mirrors equal what gcc computes for include/b200dm.h."""
    prog = r'''
#include <stdio.h>
#include <stddef.h>
#include "b200dm.h"
int main(void){
  printf("%zu %zu %zu %zu\n", sizeof(b200dm_update_desc), sizeof(b200dm_norm_desc), sizeof(b200dm_vq_desc), sizeof(b200dm_conv_desc));
  printf("%zu %zu %zu %zu\n", offsetof(b200dm_update_desc, t_dev), offsetof(b200dm_update_desc, seed), offsetof(b200dm_update_desc, eps_dtype), offsetof(b200dm_norm_desc, y_dtype));
  printf("%zu %zu %zu\n", offsetof(b200dm_vq_desc, q_dtype), offsetof(b200dm_conv_desc, use_halo), offsetof(b200dm_conv_desc, reserved));
  return 0; }'''
    import tempfile
    with tempfile.TemporaryDirectory() as td:
        src, exe = os.path.join(td, "t.c"), os.path.join(td, "t")
        open(src, "w").write(prog)
        subprocess.run(["gcc", "-I", os.path.join(ROOT, "include"), src, "-o", exe], check=True)   # header is plain C
        rows = [[int(v) for v in ln.split()] for ln in subprocess.run([exe], capture_output=True, text=True).stdout.splitlines()]
    assert rows[0] == [C.sizeof(L.UpdateDesc), C.sizeof(L.NormDesc), C.sizeof(L.VqDesc), C.sizeof(L.ConvDesc)]
    assert rows[1] == [L.UpdateDesc.t_dev.offset, L.UpdateDesc.seed.offset, L.UpdateDesc.eps_dtype.offset, L.NormDesc.y_dtype.offset]
    assert rows[2] == [L.VqDesc.q_dtype.offset, L.ConvDesc.use_halo.offset, L.ConvDesc.reserved.offset]


def test_weight_packer_is_a_permutation_of_the_keras_kernel(L):
    """b200dm_conv_pack_weights is host-side: every Keras kernel entry (rounded to bf16) appears in the packed image,
    the rest is zero padding."""
    from b200dm import ops
    rng = np.random.default_rng(0)
    for (k, cin, cout, stride) in [(3, 32, 64, 1), (1, 96, 64, 1), (3, 64, 64, 2), (3, 8, 64, 1)]:
        w = torch.from_numpy(rng.standard_normal((k, k, k, cin, cout)).astype(np.float32))
        desc = ops.make_conv_desc(L.CONV_DIRECT, 1, (8, 8, 8), cin, 0, cout, k, stride)
        packed = ops.pack_conv_weights(desc, w)
        assert packed.dtype == torch.bfloat16 and packed.numel() * 2 == L.lib().b200dm_conv_packed_weight_bytes(C.byref(desc))
        a = np.sort(packed.float().numpy().ravel())
        b = np.sort(w.to(torch.bfloat16).float().numpy().ravel())
        nz = a[a != 0]
        assert np.array_equal(nz, b[b != 0])
        assert abs(packed.float().sum().item() - w.to(torch.bfloat16).float().sum().item()) < 1e-2 * w.numel() ** 0.5


def test_upsample_fold_presums_taps(L):
    """PARITY mode with a 3^3 kernel folds UpSampling3D(2)+Conv3D (dm3d.py:271-274) into 8 parity kernels of 2^3 taps:
    per parity the folded taps sum to the sum of all 27 taps."""
    from b200dm import ops
    w = torch.from_numpy(np.random.default_rng(1).standard_normal((3, 3, 3, 64, 64)).astype(np.float32))
    desc = ops.make_conv_desc(L.CONV_PARITY, 1, (4, 4, 4), 64, 0, 64, 3, 1)
    packed = ops.pack_conv_weights(desc, w).float()
    per_parity = packed.reshape(8, -1).sum(1)
    assert torch.allclose(per_parity, w.sum().expand(8), rtol=0, atol=2.0)   # bf16 rounding of 3.3e4 folded terms


def test_bad_descriptor_is_rejected_without_a_gpu(L):
    from b200dm import ops
    desc = ops.make_conv_desc(L.CONV_DIRECT, 1, (8, 8, 8), 32, 0, 64, 5, 1)   # ksize 5 is not a reference layer
    assert L.lib().b200dm_conv_packed_weight_bytes(C.byref(desc)) == 0
    assert L.lib().b200dm_last_error() != b""


@pytest.mark.skipif(torch.cuda.is_available(), reason="checks the no-GPU behaviour")
def test_product_path_fails_loudly_without_gpu(L):
    import types
    import b200dm
    with pytest.raises(L.B200dmError):
        b200dm.ops.cast(torch.zeros(4), torch.bfloat16)
    dm = b200dm.DiffusionModel(8, 256, 8, None, types.SimpleNamespace(timesteps=4, num_gpus=1, kernel_resize=False, bs=1))
    with pytest.raises(L.B200dmError):
        dm.generate((1, 8, 8, 8, 8))
    with pytest.raises(L.B200dmError):
        b200dm.VectorQuantizer(16, 8).quantize(torch.zeros(1, 2, 2, 2, 8))
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--steps", "1"], capture_output=True, text=True)
    assert r.returncode != 0 and "no CPU fallback" in (r.stderr + r.stdout)


def test_product_package_never_imports_the_oracle():
    pkg = os.path.join(ROOT, "3d-condtional-stable-diffusion_b200")
    for dirpath, _, files in os.walk(pkg):
        for f in files:
            if f.endswith((".py", ".cu", ".cuh", ".h")):
                src = open(os.path.join(dirpath, f)).read()
                assert not re.search(r"^\s*(from|import)\s+oracle\b", src, flags=re.M), f"{f} imports the oracle"


def test_fp16_storage_build_exports_the_same_abi(L):
    """libb200dm_f16.so (same sources, -DB200DM_ACT_FP16): same symbols, reports its storage type; the selection is per process."""
    path = L._LIBS["fp16"]
    assert os.path.exists(path), "build.py builds both storage variants"
    lib16 = C.CDLL(path)
    for n in header_functions():
        assert hasattr(lib16, n), n
    lib16.b200dm_storage_dtype.restype = C.c_char_p
    assert lib16.b200dm_storage_dtype() == b"fp16"
    assert L.lib().b200dm_storage_dtype() == L.precision().encode()
    code = ("import os,sys; os.environ['B200DM_PRECISION']='fp16'; sys.path.insert(0, %r); import torch, b200dm; from b200dm import _lib as L; "
            "assert L.precision()=='fp16' and L.ACT_DTYPE is torch.float16 and L.lib().b200dm_storage_dtype()==b'fp16'; "
            "import pytest\ntry:\n    L.set_precision('bf16'); raise SystemExit(3)\nexcept L.B200dmError:\n    pass") % ROOT
    r = subprocess.run([sys.executable, "-c", code], capture_output=True, text=True)
    assert r.returncode == 0, r.stderr


@pytest.mark.parametrize("precision,other", [("fp16", "bfloat16"), ("bf16", "float16")])
def test_other_16bit_type_is_rejected_before_the_device(precision, other):
    """A 16-bit tensor of the type the loaded build does not store is an error naming both types, raised before any device
    check: the kernels take raw pointers and would otherwise read bf16 bits as fp16 (or the reverse)."""
    code = f"""
import os, sys
os.environ['B200DM_PRECISION'] = {precision!r}
sys.path.insert(0, {ROOT!r})
import torch, b200dm
from b200dm import ops, _lib as L
bad = torch.zeros(1, 4, 4, 4, 64, dtype=torch.{other})
f32 = torch.zeros(1, 4, 4, 4, 64)
one = torch.ones(64)
desc = ops.make_conv_desc(L.CONV_DIRECT, 1, (4, 4, 4), 64, 0, 64, 1, 1)
calls = dict(
    ConvPlan=lambda: ops.ConvPlan(desc, bad, torch.zeros(64 * 64, dtype=L.ACT_DTYPE), torch.zeros(1, 4, 4, 4, 64, dtype=L.ACT_DTYPE)),
    norm_act=lambda: ops.norm_act(bad, one, one),
    gn_stats=lambda: ops.gn_stats(bad, 8, 1e-6),
    layernorm=lambda: ops.layernorm(bad, [one], [one]),
    bn_stats=lambda: ops.bn_stats(bad, one, one),
    q_sample=lambda: ops.q_sample(ops.ScheduleTables(4), f32, torch.zeros(1, dtype=torch.int32), out16=bad),
    noise_loss=lambda: ops.noise_loss(bad, 1.0),
    batched_gemm=lambda: ops.batched_gemm(bad[0, 0], bad[0, 0]),
)
for name, call in calls.items():
    try:
        call()
    except L.B200dmError as e:
        msg = str(e)
        assert str(L.ACT_DTYPE) in msg and 'torch.{other}' in msg, (name, msg)
    else:
        raise SystemExit(name + ': no error')
print('rejected', len(calls))
"""
    r = subprocess.run([sys.executable, "-c", code], capture_output=True, text=True)
    assert r.returncode == 0, r.stdout + r.stderr
    assert "rejected 8" in r.stdout
