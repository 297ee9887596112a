"""Host-side logic of the CUDA library on a machine without a GPU: the library's own objects are linked against a
pretend CUDA runtime (tests/native/fake_cudart.cpp: device memory is host memory, kernels do nothing) and driven by
the sanitizer probes' drivers under AddressSanitizer's allocator -- the batch ABI on good / damaged / all-invalid
inputs and a few hundred thousand random, mostly wrong, raw ABI calls.  Nothing may crash, overrun a buffer or hang.
(The long runs, with the library itself instrumented, are tests/native/host_fake_gpu_fuzz.sh.)"""
import glob
import os
import shutil
import subprocess

import numpy as np
import pytest

from tests import golden as golden_set

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
OBJ = sorted(glob.glob(os.path.join(ROOT, "lilliput_b200", "csrc", "build", "*.o")))
CUDA_INC = os.path.join(os.environ.get("CUDA_HOME", "/usr/local/cuda"), "include")


@pytest.fixture(scope="module")
def fake(tmp_path_factory):
    if not shutil.which("g++") or len(OBJ) < 10 or not os.path.exists(os.path.join(CUDA_INC, "cuda_runtime.h")):
        pytest.skip("needs g++, the CUDA headers and the library's objects (run __graft_entry__.build() first)")
    d = str(tmp_path_factory.mktemp("fake_gpu"))
    san = ["-fsanitize=address", "-fno-omit-frame-pointer"]
    nat = os.path.join(ROOT, "tests", "native")

    def run(cmd):
        r = subprocess.run(cmd, cwd=d, capture_output=True, text=True, timeout=600)
        assert r.returncode == 0, " ".join(cmd) + "\n" + r.stderr[-3000:]

    run(["g++", "-O1", "-g", "-std=c++17", "-fPIC", *san, "-I" + CUDA_INC, "-c", os.path.join(nat, "fake_cudart.cpp"),
         "-o", "fake_cudart.o"])
    run(["g++", "-shared", *san, "-o", "liblp_fake.so", *OBJ, "fake_cudart.o"])
    inc = ["-I" + os.path.join(ROOT, "include"), "-I" + os.path.join(ROOT, "lilliput_b200", "csrc"), "-I" + CUDA_INC]
    for src, exe in [("host_batch_fake_gpu.cpp", "batch_fake"), ("host_abi_misuse_fake_gpu.cpp", "misuse_fake"),
                     ("host_transform_fuzz.cpp", "transform_fake")]:
        run(["g++", "-O1", "-g", "-std=c++17", *san, *inc, os.path.join(nat, src), "-o", exe, "-L.", "-llp_fake",
             "-Wl,-rpath," + d])
    g = golden_set.load("golden")
    w = np.load(os.path.join(ROOT, "tests", "golden", "webp_golden.npz"))
    seeds = []
    for k, a in [("c1_input", g["c1_input"]), ("jpeg_31", g["jpeg_31"]), ("jpegvar_420_0", g["jpegvar_420_0"]),
                 ("webp_anim_lossy", w["webp_anim_lossy"]), ("webp_lossless_rgba", w["webp_lossless_rgba"])]:
        p = os.path.join(d, k)
        open(p, "wb").write(a.tobytes())
        seeds.append(p)
    for k in g.files:
        if k.startswith(("gif_", "png_")) and g[k].dtype == np.uint8 and g[k].ndim == 1 and g[k].size < 30000:
            p = os.path.join(d, k)
            open(p, "wb").write(g[k].tobytes())
            seeds.append(p)
    return d, seeds


def _run(d, cmd, extra_env=None):
    env = dict(os.environ, ASAN_OPTIONS="detect_leaks=0:allocator_may_return_null=1:max_allocation_size_mb=8192")
    env.update(extra_env or {})
    r = subprocess.run(cmd, cwd=d, env=env, capture_output=True, text=True, timeout=900)
    tail = (r.stdout + r.stderr)[-3000:]
    assert r.returncode == 0 and "done:" in r.stdout, tail
    assert "ERROR: AddressSanitizer" not in r.stderr and "runtime error" not in r.stderr, tail


def test_batch_abi_host_side(fake):
    d, seeds = fake
    _run(d, ["./batch_fake", "12", *seeds[:3]])


@pytest.mark.parametrize("env", [{}, {"LP_FAKE_CHAOS": "1"}, {"LP_RESIZE_TAB_CAP": "2", "LP_JPEG_ENC_CONST_CAP": "2"}],
                         ids=["plain", "chaos", "tiny_caches"])
def test_raw_abi_misuse_host_side(fake, env):
    d, seeds = fake
    _run(d, ["./misuse_fake", "300000", "5", *seeds], env)


def test_transform_host_side(fake):
    d, seeds = fake
    _run(d, ["./transform_fake", "1500", *seeds])
