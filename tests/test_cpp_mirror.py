"""The C++ host mirror (include/scann_b200.hpp) compiles against the C ABI (CPU check) and passes the
reference's unit-test sequences on a GPU (-m gpu)."""
import os
import subprocess

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
SRC = os.path.join(ROOT, "tests", "cpp", "test_hpp_mirror.cpp")


def _build(pkg, out_dir):
    """Compiles the mirror test into out_dir (the source tree may be read-only) and returns the executable."""
    lib = pkg.build_lib.build()
    libdir = os.path.dirname(lib)
    exe = str(out_dir / "test_hpp_mirror.bin")
    cmd = ["g++", "-std=c++17", "-O1", "-Wall", "-I", os.path.join(ROOT, "include"), SRC, "-o", exe, "-L", libdir,
           "-lscann_b200", f"-Wl,-rpath,{libdir}"]
    subprocess.check_call(cmd)
    return exe


def test_cpp_mirror_compiles_and_links(pkg, tmp_path):
    assert os.path.exists(_build(pkg, tmp_path))


def test_c_header_is_plain_c(pkg, tmp_path):
    # the ABI header must be consumable from C (no C++-isms)
    probe = tmp_path / "_probe.c"
    probe.write_text('#include "scann_b200.h"\nint main(void){ return scann_version() > 0 ? 0 : 1; }\n')
    subprocess.check_call(["gcc", "-std=c99", "-Wall", "-Werror", "-I", os.path.join(ROOT, "include"), "-c", str(probe),
                           "-o", str(tmp_path / "_probe.o")])


@pytest.mark.gpu
def test_cpp_mirror_runs_reference_unit_tests(gpu_lib, tmp_path):
    exe = _build(gpu_lib, tmp_path)
    out = subprocess.run([exe], capture_output=True, text=True, timeout=120)
    assert out.returncode == 0, out.stdout + out.stderr
    assert "hpp mirror ok" in out.stdout
