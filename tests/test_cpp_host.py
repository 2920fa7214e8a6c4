"""The C++ host-side mirror of the reference's Go host layer (nornicdb_b200/host/nornic_cuda.hpp) compiles against the
C ABI and behaves like the Go code: error paths without a GPU, the reference's cuda_test.go / gpu_test.go cases with one."""
import os
import subprocess

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


@pytest.fixture(scope="module")
def host_binary(knn_lib, tmp_path_factory):
    # Built fresh into a temporary directory: the source tree may be read-only, and a binary left there from an earlier
    # build could be linked against another copy of the library.
    src = os.path.join(ROOT, "tests", "cpp", "host_mirror_test.cpp")
    lib = os.path.join(ROOT, "nornicdb_b200", "libnornic_knn.so")
    out = str(tmp_path_factory.mktemp("host_mirror") / "host_mirror_test")
    subprocess.run(["/usr/bin/g++", "-std=c++17", "-O1", "-Wall", "-I", ROOT, src, "-L", os.path.dirname(lib), "-lnornic_knn",
                    f"-Wl,-rpath,{os.path.dirname(lib)}", "-lpthread", "-o", out], check=True, cwd=ROOT)
    return out


def test_host_mirror_error_paths_without_gpu(host_binary):
    from nornicdb_b200 import cuda
    if cuda.IsAvailable():
        pytest.skip("GPU present: the full run below covers it")
    out = subprocess.run([host_binary, "--no-gpu"], capture_output=True, text=True)
    assert out.returncode == 0, out.stdout + out.stderr
    assert "host mirror ok" in out.stdout


@pytest.mark.gpu
def test_host_mirror_reference_cases_on_gpu(host_binary):
    out = subprocess.run([host_binary], capture_output=True, text=True, timeout=120)
    assert out.returncode == 0, out.stdout + out.stderr
    assert "host mirror ok" in out.stdout
