"""The tangent-factored 32-point transforms of os64_core.cuh (DESIGN.md section 4.2, step 9), checked on the CPU.

tools/dft32_tangent_check.cpp runs dft32_dit and dft32_dif, forward and inverse, on random, full-scale (+-1 per part) and
full-scale tone inputs against a double-precision DFT, next to a copy of the plain form they replaced (a complex multiply
per twiddle, then the butterfly).  The tangent form's relative RMS error must be at most 1.5 times the plain form's, and
every output register must hold the value the plain form puts there: the register order is unchanged."""
import os
import shutil
import subprocess

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


@pytest.fixture(scope="module")
def dft32_check(tmp_path_factory):
    cxx = shutil.which("g++") or shutil.which("c++")
    assert cxx, "a host C++ compiler is needed (nvcc needs one as well)"
    exe = str(tmp_path_factory.mktemp("dft32") / "dft32_tangent_check")
    subprocess.run([cxx, "-std=c++17", "-O2", "-w", "-I", os.path.join(ROOT, "pothoscomms_b200", "csrc"), "-o", exe,
                    os.path.join(ROOT, "tools", "dft32_tangent_check.cpp")], check=True)
    return exe


@pytest.mark.parametrize("kind", ["random", "fullscale", "tone"])
@pytest.mark.parametrize("direction", ["fwd", "inv"])
@pytest.mark.parametrize("form", ["dit", "dif"])
def test_tangent_form_matches_the_dft_and_the_plain_form(dft32_check, form, direction, kind):
    r = subprocess.run([dft32_check, form, direction, kind], capture_output=True, text=True)
    assert r.returncode == 0 and r.stdout.count("-> ok") == 1, r.stdout + r.stderr
