"""The kernel and model test files again in the fp16 storage build (libb200dm_f16.so, B200DM_PRECISION=fp16), one child
process per file: the storage type is chosen once per process.  The files are written for either build (tolerances in units
of the storage type's ulp), so the fp16 run checks the code only that build compiles -- its conversions, the tcgen05 and TMA
format codes, the stencil head's mma.sync, host weight rounding, attention's P rounding -- at 8x the sensitivity."""
import os
import subprocess
import sys
import time

import pytest

pytestmark = pytest.mark.gpu

HERE = os.path.dirname(os.path.abspath(__file__))
FILES = ["test_conv_gpu.py", "test_attention_gpu.py", "test_elementwise_gpu.py", "test_fullsize_gpu.py", "test_shortcut_fold_gpu.py",
         "test_model_gpu.py", "test_train_forward_gpu.py", "test_storage_edges_gpu.py", "test_norm_gpu.py"]


@pytest.mark.skipif(os.environ.get("B200DM_PRECISION", "bf16") != "bf16", reason="already the fp16 child run")
@pytest.mark.parametrize("name", FILES)
def test_file_passes_in_fp16_build(cuda, name):
    env = dict(os.environ, B200DM_PRECISION="fp16")
    t0 = time.perf_counter()
    r = subprocess.run([sys.executable, "-m", "pytest", os.path.join(HERE, name), "-m", "gpu", "-q", "-p", "no:cacheprovider"],
                       env=env, cwd=os.path.dirname(HERE), capture_output=True, text=True)
    tail = r.stdout.strip().splitlines()[-1] if r.stdout.strip() else ""
    print(f"fp16 build, {name}: {tail} ({time.perf_counter() - t0:.0f} s)")
    assert r.returncode == 0, r.stdout[-6000:] + r.stderr[-2000:]
