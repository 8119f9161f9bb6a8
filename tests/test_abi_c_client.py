"""The header is valid C99 and the ABI is callable from a plain C program (tests/abi_kat.c)."""
import os
import subprocess

import pytest

import gficf_b200

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(HERE)


@pytest.fixture(scope="module")
def exe(tmp_path_factory):
    """The C client, built into a temporary directory (the source tree may be read-only)."""
    path = str(tmp_path_factory.mktemp("abi") / "abi_kat")
    lib = gficf_b200.library_path()
    cmd = ["gcc", "-std=c99", "-Wall", "-Wextra", "-Werror", "-pedantic", "-I" + os.path.join(ROOT, "include"),
           os.path.join(HERE, "abi_kat.c"), lib, "-Wl,-rpath," + os.path.dirname(lib), "-o", path]
    r = subprocess.run(cmd, capture_output=True, text=True)
    assert r.returncode == 0, r.stderr
    return path


def test_c_client_compiles_and_fails_loudly_without_gpu(exe):
    r = subprocess.run([exe], capture_output=True, text=True, timeout=120)
    if gficf_b200.lib().gficf_cuda_device_count() == 0:
        assert r.returncode == 3 and "no CUDA device" in r.stdout  # GFICF_E_CUDA, never a CPU answer
    else:
        assert r.returncode == 0, r.stdout


@pytest.mark.gpu
def test_c_client_known_answers(cuda, exe):
    r = subprocess.run([exe], capture_output=True, text=True, timeout=120)
    assert r.returncode == 0 and "abi_kat ok" in r.stdout, r.stdout + r.stderr
