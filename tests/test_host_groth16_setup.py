"""CPU test of the Groth16 setup kernels' bodies (setup_kernels.cuh): the powers of tau, the column index and bounded-segment column sums of A, B
and C against the Lagrange basis, and the scalar formula, run thread index by thread index on the host (tests/host_emu_groth16_setup.cpp) in the
pass structure of the device, must equal crs_exponents of the restated reference (oracle/groth16_ref.py) word for word: u, v, w per variable, ic,
l and h."""
import os
import subprocess

import numpy as np
import pytest
from conftest import ROOT
from groth16_r1cs_util import csr_from_r1cs, edge_circuit, mont

from oracle import groth16_ref as G
from oracle import pyref as B
from test_groth16 import SETUP_SEED

EXE = os.path.join(ROOT, "tests", "_build", "host_emu_groth16_setup")


@pytest.fixture(scope="module")
def host_emu_setup():
    os.makedirs(os.path.dirname(EXE), exist_ok=True)
    src = os.path.join(ROOT, "tests", "host_emu_groth16_setup.cpp")
    deps = [src] + [os.path.join(ROOT, "kogarashi_b200", "csrc", f) for f in ("field.cuh", "r1cs_kernels.cuh", "setup_kernels.cuh")]
    if not os.path.exists(EXE) or any(os.path.getmtime(d) > os.path.getmtime(EXE) for d in deps):
        subprocess.check_call(["g++", "-O2", "-std=c++17", "-Wno-unknown-pragmas", "-o", EXE, src])
    return EXE


def _circuit(name):
    if name == "example":
        return G.example_circuit(3, 35), ()
    if name == "edge":
        return edge_circuit()
    return G.chain_circuit(int(name.split("_")[1]), 3)[0], ()


# the example (m = n = 4); the edge circuit (an empty row, a 300-term row, coefficients 1 and r - 1, duplicated columns); a chain of m = 301 (not a
# power of two); a chain of m = 2^10, whose constant column in A and B spans two thirds of the rows (three passes of partial sums)
@pytest.mark.parametrize("name", ["example", "edge", "chain_100", "chain_341"])
def test_setup_bodies_match_crs_exponents(host_emu_setup, tmp_path, name):
    cs, split = _circuit(name)
    E, trap, uvw = G.crs_exponents(cs, B.XorShift128(SETUP_SEED))
    k, n = E["k"], E["n"]
    m, n_z, mats = csr_from_r1cs(cs, split_rows=split)
    tau = trap["tau"]
    lagr = G.lagrange_at(n, pow(G.ROOT_OF_UNITY, 1 << (G.S - k), G.R), tau)
    inp, outp = tmp_path / "in.bin", tmp_path / "out.bin"
    with open(inp, "wb") as f:
        f.write(np.array([k, m, n_z, cs.l], dtype=np.uint32).tobytes())
        for row_ptr, cols, coeffs in mats:
            f.write(row_ptr.tobytes() + cols.tobytes() + coeffs.tobytes())
        f.write(mont([trap[x] for x in ("alpha", "beta", "gamma", "delta", "tau")]).tobytes())
        f.write(mont(lagr).tobytes())
    out = subprocess.run([host_emu_setup, str(inp), str(outp)], capture_output=True, text=True, timeout=600)
    assert out.returncode == 0 and out.stdout.startswith("OK"), out.stdout + out.stderr
    got = np.fromfile(outp, dtype=np.uint64).reshape(-1, 4)
    parts, off = {}, 0
    for key, size in (("powers", n), ("u", n_z), ("v", n_z), ("w", n_z), ("ext", n_z), ("h", m - 1)):
        parts[key], off = got[off: off + size], off + size
    assert off == got.shape[0]
    assert (parts["powers"] == mont([pow(tau, i, G.R) for i in range(n)])).all()
    for j, key in enumerate("uvw"):
        assert (parts[key] == mont([t[j] for t in uvw])).all(), key
    assert (parts["u"] == mont(E["a"])).all() and (parts["v"] == mont(E["b_g1"])).all()
    assert (parts["ext"][: cs.l] == mont(E["ic"])).all()
    assert (parts["ext"][cs.l:] == mont(E["l"])).all()
    assert (parts["h"] == mont(E["h"])).all()
