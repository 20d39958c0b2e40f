"""CPU test of the Groth16 evaluation kernel's body (k_r1cs_evaluate): run position by position on the host (tests/host_emu_groth16.cpp), its
three NTT buffers must equal cs.evaluate() of the restated reference (oracle/groth16_ref.py), zero padded and permuted by bit reversal, word
for word."""
import os
import subprocess

import numpy as np
import pytest
from conftest import ROOT
from groth16_r1cs_util import csr_from_r1cs, edge_circuit, evaluations_bitrev, mont

from oracle import groth16_ref as G

EXE = os.path.join(ROOT, "tests", "_build", "host_emu_groth16")


@pytest.fixture(scope="module")
def host_emu_groth16():
    os.makedirs(os.path.dirname(EXE), exist_ok=True)
    src = os.path.join(ROOT, "tests", "host_emu_groth16.cpp")
    deps = [src] + [os.path.join(ROOT, "kogarashi_b200", "csrc", f) for f in ("field.cuh", "r1cs_kernels.cuh")]
    if not os.path.exists(EXE) or any(os.path.getmtime(d) > os.path.getmtime(EXE) for d in deps):
        subprocess.check_call(["g++", "-O2", "-std=c++17", "-Wno-unknown-pragmas", "-o", EXE, src])
    return EXE


def _circuit(name):
    if name == "example":
        return G.example_circuit(3, 35), ()
    if name == "edge":
        return edge_circuit()
    steps = int(name.split("_")[1])
    return G.chain_circuit(steps, 3)[0], ()


# (circuit, log_n): m = 4 on its own domain and on a much larger one; chains with m = 3 * steps + 1 not a power of two (301 -> 512,
# 4 -> 8) and exactly one (16); the chain of 100 steps with an empty row, a 300-term row, coefficients 1 and r - 1, duplicated columns
CASES = [("example", 2), ("example", 5), ("chain_100", 9), ("chain_1", 3), ("chain_5", 4), ("edge", 9), ("edge", 10)]


@pytest.mark.parametrize("name,log_n", CASES)
def test_r1cs_evaluate_body_on_cpu(host_emu_groth16, tmp_path, name, log_n):
    cs, split = _circuit(name)
    m, n_z, mats = csr_from_r1cs(cs, split_rows=split)
    assert (1 << log_n) >= m
    inp, outp = tmp_path / "in.bin", tmp_path / "out.bin"
    with open(inp, "wb") as f:
        f.write(np.array([log_n, m, n_z], dtype=np.uint32).tobytes())
        for row_ptr, cols, coeffs in mats:
            f.write(row_ptr.tobytes() + cols.tobytes() + coeffs.tobytes())
        f.write(mont(cs.x + cs.w).tobytes())
    out = subprocess.run([host_emu_groth16, str(inp), str(outp)], capture_output=True, text=True, timeout=600)
    assert out.returncode == 0 and out.stdout.startswith("OK"), out.stdout + out.stderr
    got = np.fromfile(outp, dtype=np.uint64).reshape(3, 1 << log_n, 4)
    for k, exp in enumerate(evaluations_bitrev(cs, log_n)):
        assert (got[k] == exp).all(), f"matrix {'ABC'[k]}"
