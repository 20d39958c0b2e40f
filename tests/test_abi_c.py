"""The C ABI used from plain C (examples/abi_demo.c): builds against include/kgr_msm.h + libkgr_msm.so with gcc only.
CPU: the program must fail loudly without a device (no CPU fallback).  GPU: its MSM identities hold on G1 and G2."""
import os
import subprocess

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


@pytest.fixture(scope="module")
def demo(tmp_path_factory):
    """The demo program, built into a temporary directory: the source tree may be read-only."""
    from kogarashi_b200 import _lib
    _lib.build()
    exe = str(tmp_path_factory.mktemp("abi_demo") / "abi_demo")
    libdir = os.path.join(ROOT, "kogarashi_b200")
    subprocess.check_call(["gcc", "-O2", "-Wall", "-Werror", "-I", os.path.join(ROOT, "include"), "-o", exe, os.path.join(ROOT, "examples", "abi_demo.c"),
                           "-L", libdir, "-lkgr_msm", f"-Wl,-rpath,{libdir}"])
    return exe


def test_header_compiles_as_c_and_program_fails_loudly_without_a_device(demo):
    import torch
    if torch.cuda.is_available():
        pytest.skip("a GPU is present")
    out = subprocess.run([demo], capture_output=True, text=True, timeout=120)
    assert out.returncode == 3 and "no CPU fallback" in out.stdout, out.stdout + out.stderr


@pytest.mark.gpu
def test_c_program_msm_identities(demo):
    out = subprocess.run([demo], capture_output=True, text=True, timeout=300)
    assert out.returncode == 0 and out.stdout.count(": yes") == 3, out.stdout + out.stderr
