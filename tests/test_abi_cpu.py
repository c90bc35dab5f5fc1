"""CPU-side checks of the drop-in boundary: the C-ABI library builds, loads, exports every symbol that
include/nb200.h declares, and refuses to run without a CUDA device (no CPU fallback on the product path)."""
import ctypes as C
import os
import subprocess
import sys

import pytest

import nexus_zkvm_b200 as nb
from nexus_zkvm_b200 import build as nb_build

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
NO_DEVICE_ENV = dict(os.environ, CUDA_VISIBLE_DEVICES="")   # a child process that sees no CUDA device, GPU machine or not


@pytest.fixture(scope="module")
def built():
    return nb_build.build()


def test_header_compiles_as_c(tmp_path):
    src = tmp_path / "t.c"
    src.write_text('#include "nb200.h"\nint main(void){return NB200_OK;}\n')
    subprocess.check_call(["/usr/bin/gcc", "-std=c99", "-Wall", "-Werror", "-I", os.path.join(ROOT, "include"), "-c", str(src), "-o", str(tmp_path / "t.o")])


def test_library_exports_every_declared_symbol(built):
    L = C.CDLL(built)
    syms = nb.exported_symbols()
    assert len(syms) >= 25
    missing = [s for s in syms if not hasattr(L, s)]
    assert not missing, missing


def test_no_cpu_fallback_without_device(built):
    """Runs in a child process with every CUDA device hidden, so it holds on a machine with a GPU too."""
    code = ("import nexus_zkvm_b200 as nb\n"
            "try:\n    nb.Context(0)\nexcept nb.Nb200Error as e:\n    print(e)\nelse:\n    raise SystemExit('a context was created')\n")
    r = subprocess.run([sys.executable, "-c", code], cwd=ROOT, env=NO_DEVICE_ENV, capture_output=True, text=True, timeout=120)
    assert r.returncode == 0, r.stdout + r.stderr
    assert "no CPU fallback" in r.stdout or "no CUDA device" in r.stdout


def test_product_sources_do_not_reference_oracle():
    for root, _, files in os.walk(os.path.join(ROOT, "nexus_zkvm_b200")):
        if os.path.basename(root) == "build":
            continue
        for f in files:
            if f.endswith((".py", ".cu", ".cuh", ".h", ".cc")):
                txt = open(os.path.join(root, f)).read()
                assert "oracle" not in txt.replace("no oracle", ""), f"{f} mentions the oracle"


def test_kernel_sources_and_cache_keys_without_a_gpu():
    """The generated CUDA C of an AIR's kernels is available without a device; the cache key is stable and distinguishes kernels."""
    from nexus_zkvm_b200 import build as B, machine as M
    a = B.kernel_sources(M.AddMachine(log_size=8, n_lanes=1).words)
    b = B.kernel_sources(M.AddMachine(log_size=8, n_lanes=2).words)
    assert len(a) >= 2 and len(b) >= 2               # constraint + logup program of the main component
    assert all(b"extern \"C\" __global__" in src and b"nbjit" in src for _k, src in a)
    keys = [k for k, _ in a + b]
    assert len(set(keys)) == len(keys)
    assert [k for k, _ in B.kernel_sources(M.AddMachine(log_size=8, n_lanes=1).words)] == [k for k, _ in a]


def test_native_host_example_builds_and_fails_loudly_without_a_gpu(tmp_path):
    """examples/prove_demo.cc compiles against include/nb200.h, links against the library, and — on a machine without a CUDA
    device (here: every device hidden from it) — stops at nb200_ctx_create instead of computing anything on the CPU.  The success
    path is tests/test_gpu_native_host.py."""
    from nexus_zkvm_b200 import machine as M
    from tests.native_job import build_demo, write_job
    exe = build_demo()
    m = M.AddMachine(log_size=8, n_lanes=1)
    cols, mult = m.fill_main_trace(seed=1)
    write_job(tmp_path / "job.bin", m, cols, mult, dict(pow_bits=5, log_blowup=1, log_last=0, n_queries=3))
    r = subprocess.run([exe, str(tmp_path / "job.bin"), str(tmp_path / "proof.bin")], env=NO_DEVICE_ENV, capture_output=True, text=True,
                       timeout=120)
    assert r.returncode == 3 and "no context" in r.stderr
    assert not (tmp_path / "proof.bin").exists()
