"""The reference's two test programs, rewritten in C++ against the splpak_type mirror and linked
against the product library's C ABI (no Python in the loop)."""
import os
import subprocess

import pytest

import splpak_b200 as sp

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
SRC = os.path.join(ROOT, "tests", "cpp", "splpak_test_linear.cpp")


def _build(tmp_path):
    """The executable goes to a temporary directory: the source tree may be read-only."""
    exe = str(tmp_path / "splpak_test_linear.bin")
    libdir = os.path.dirname(sp.lib_path(False))
    subprocess.run(["g++", "-O2", "-std=c++17", SRC, "-o", exe, f"-L{libdir}", "-lsplpak_b200",
                    f"-Wl,-rpath,{libdir}", "-L/usr/local/cuda/lib64", "-Wl,-rpath,/usr/local/cuda/lib64"],
                   check=True)
    return exe


def test_cpp_mirror_compiles_and_links(tmp_path):
    """CPU: the header-only mirror compiles against include/splpak_b200.h and links to the library."""
    assert os.path.exists(_build(tmp_path))


@pytest.mark.gpu
def test_reference_test_programs_in_cpp(tmp_path):
    r = subprocess.run([_build(tmp_path)], capture_output=True, text=True)
    assert r.returncode == 0, r.stdout + r.stderr
    assert "splcw ierror = 0" in r.stdout and r.stdout.strip().endswith("ok")
