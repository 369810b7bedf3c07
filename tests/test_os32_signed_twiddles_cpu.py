"""fir_os32_kernel's signed lanes and register indices (DESIGN.md section 4.2, step 8), checked on the CPU.

tools/os32_host_check.cpp runs one 1024-point overlap-save block the way the kernel does -- the same 32-point
transforms, the same step-twiddle helper (os32_step) and the same 16-row table builder (os32_signed_twiddles) from
os64_core.cuh, the same row shifts of the landing read, the tap spectrum and the store -- and compares every forward bin
of every lane and register, and every alias-free output, with a double-precision DFT and convolution.  Its --fault
switches break one conjugate flag or one lane's shift on purpose; the check has to catch each of them."""
import os
import shutil
import subprocess

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


@pytest.fixture(scope="module")
def host_check(tmp_path_factory):
    cxx = shutil.which("g++") or shutil.which("c++")
    assert cxx, "a host C++ compiler is needed (nvcc needs one as well)"
    exe = str(tmp_path_factory.mktemp("os32") / "os32_host_check")
    subprocess.run([cxx, "-std=c++17", "-O2", "-w", "-I", os.path.join(ROOT, "pothoscomms_b200", "csrc"), "-o", exe,
                    os.path.join(ROOT, "tools", "os32_host_check.cpp")], check=True)
    return exe


@pytest.mark.parametrize("K", [9, 256, 448])
def test_every_lane_and_register_matches_the_dft(host_check, K):
    r = subprocess.run([host_check, str(K)], capture_output=True, text=True)
    assert r.returncode == 0, r.stdout + r.stderr
    assert "-> ok" in r.stdout and "every output once: yes" in r.stdout


@pytest.mark.parametrize("fault", ["conj:1", "conj:15", "conj:16", "conj:17", "conj:31", "lane:16", "lane:23", "lane:31"])
def test_one_wrong_conjugate_or_lane_shift_fails(host_check, fault):
    r = subprocess.run([host_check, "--fault", fault, "256"], capture_output=True, text=True)
    assert r.returncode == 1 and "FAIL" in r.stdout, r.stdout + r.stderr
