"""CPU tests of the relaxed-R1CS check's per-row body (body_relaxed_row in kogarashi_b200/csrc/r1cs_kernels.cuh, the body of k_relaxed_check behind
kgr_nova_is_sat) compiled with g++ (tests/host_emu_nova_sat.cpp): the violation flag of every row must equal a Python big-integer evaluation of
(A z)_i (B z)_i = u (C z)_i + E_i (nova/src/relaxed_r1cs.rs:80-146), u = z[0] relaxed or 1 strict, E = 0 when absent."""
import os
import subprocess

import numpy as np
import pytest
from conftest import ROOT
from nova_util import chain_r1cs, csr_from_rows, example_r1cs, example_z, mont

from oracle import pyref as B

EXE = os.path.join(ROOT, "tests", "_build", "host_emu_nova_sat")
FIELDS = [(0, B.FQ), (1, B.FR)]


@pytest.fixture(scope="module")
def emu():
    os.makedirs(os.path.dirname(EXE), exist_ok=True)
    src = os.path.join(ROOT, "tests", "host_emu_nova_sat.cpp")
    deps = [src] + [os.path.join(ROOT, "kogarashi_b200", "csrc", f) for f in ("field.cuh", "r1cs_kernels.cuh")]
    if not os.path.exists(EXE) or any(os.path.getmtime(d) > os.path.getmtime(EXE) for d in deps):
        subprocess.check_call(["g++", "-O2", "-std=c++17", "-Wno-unknown-pragmas", "-o", EXE, src])
    return EXE


def _flags(emu, fid, p, m, n_z, mats, z, e, strict):
    """Run the body on every row; z, e: Python ints (e None: no E)."""
    words = [fid, m, n_z, int(strict), int(e is not None)]
    for row_ptr, cols, coeffs in mats:
        words += [int(x) for x in row_ptr] + [int(x) for x in cols] + [int(x) for x in np.asarray(coeffs, dtype=np.uint64).reshape(-1)]
    words += [int(x) for x in mont(z, p).reshape(-1)]
    if e is not None:
        words += [int(x) for x in mont(e, p).reshape(-1)] if m else []
    out = subprocess.run([emu], input=" ".join(map(str, words)), capture_output=True, text=True, timeout=600)
    assert out.returncode == 0 and out.stdout.startswith("FLAGS"), out.stdout + out.stderr
    got = out.stdout.split()[1] if m else ""
    return [c == "1" for c in got]


def _rows(mat, p):
    row_ptr, cols, coeffs = mat
    co = [B.from_mont(B.limbs_to_int(c), p) for c in np.asarray(coeffs, dtype=np.uint64).reshape(-1, 4)]
    return [[(int(cols[j]), co[j]) for j in range(int(row_ptr[i]), int(row_ptr[i + 1]))] for i in range(len(row_ptr) - 1)]


def _products(mats, z, p):
    return [[sum(c * z[col] for col, c in row) % p for row in _rows(mat, p)] for mat in mats]


def _expect(mats, z, e, strict, p):
    az, bz, cz = _products(mats, z, p)
    u = 1 if strict else z[0]
    return [(az[i] * bz[i] - u * cz[i] - (e[i] if e is not None else 0)) % p != 0 for i in range(len(az))]


def _random_shape(rng, m, n_z, p):
    """Empty rows, unit and non-unit coefficients, the constant column 0 in about a third of the rows, one long row."""
    mats = []
    for _ in range(3):
        rows = []
        for i in range(m):
            kind = int(rng.integers(0, 8))
            nnz = 0 if kind == 0 else (min(n_z, 40) if i == m // 2 else int(rng.integers(1, 5)))
            cols = set(int(c) for c in rng.choice(n_z, size=nnz, replace=False))
            if kind in (1, 2) and nnz:
                cols.add(0)
            rows.append({c: (1 if rng.integers(0, 2) else int(rng.integers(2, 1 << 62)) ** 4 % p) for c in cols})
        mats.append(csr_from_rows(rows, p))
    return tuple(mats)


def _fold(mats, z1, z2, e1, r, p):
    """One NIFS fold with big integers: T = AZ1 o BZ2 + AZ2 o BZ1 - u1 CZ2 - u2 CZ1 (prover.rs:53-90), z = z1 + r z2, E = e1 + r T."""
    (a1, b1, c1), (a2, b2, c2) = _products(mats, z1, p), _products(mats, z2, p)
    t = [(a1[i] * b2[i] + a2[i] * b1[i] - z1[0] * c2[i] - z2[0] * c1[i]) % p for i in range(len(a1))]
    return [(x + r * y) % p for x, y in zip(z1, z2)], [(x + r * y) % p for x, y in zip(e1, t)]


@pytest.mark.parametrize("fid,p", FIELDS)
@pytest.mark.parametrize("strict,with_e", [(False, True), (False, False), (True, False)])
def test_random_shapes_match_big_integers(emu, fid, p, strict, with_e):
    rng = np.random.default_rng(100 + 10 * fid + 2 * strict + with_e)
    for m, n_z in ((1, 1), (37, 5), (300, 120)):
        mats = _random_shape(rng, m, n_z, p)
        z = [int(rng.integers(0, 1 << 62)) ** 4 % p for _ in range(n_z)]
        if rng.integers(0, 2):
            z[0] = 1
        az, bz, cz = _products(mats, z, p)
        u = 1 if strict else z[0]
        # E chosen so that every row holds, then about half the rows disturbed: both outcomes on every shape
        e = [(az[i] * bz[i] - u * cz[i]) % p for i in range(m)] if with_e else None
        if with_e:
            for i in range(m):
                if rng.integers(0, 2):
                    e[i] = (e[i] + int(rng.integers(1, 1 << 62))) % p
        got = _flags(emu, fid, p, m, n_z, mats, z, e, strict)
        assert got == _expect(mats, z, e, strict, p)
        if with_e:
            assert 0 < sum(got) < m or m == 1


@pytest.mark.parametrize("fid,p", FIELDS)
def test_folded_instance_and_tampering(emu, fid, p):
    m, n_z, mats, z1 = chain_r1cs(60, 3, p)
    z2 = chain_r1cs(60, 4, p)[3]
    # strict instances hold, and the relaxed instance of one fold (u != 1, E != 0) holds
    assert not any(_flags(emu, fid, p, m, n_z, mats, z1, None, True))
    z, e = _fold(mats, z1, z2, [0] * m, 0x1234567890ABCDEF1234567890ABCDEF % p, p)
    assert z[0] != 1 and any(e)
    assert not any(_flags(emu, fid, p, m, n_z, mats, z, e, False))
    # rows broken through E: exactly those rows
    bad_rows = [0, 17, m - 1]
    e_bad = list(e)
    for i in bad_rows:
        e_bad[i] = (e_bad[i] + 1) % p
    got = _flags(emu, fid, p, m, n_z, mats, z, e_bad, False)
    assert [i for i, f in enumerate(got) if f] == bad_rows
    # one witness entry changed: the rows that reference that column
    col = 10
    z_bad = list(z)
    z_bad[col] = (z_bad[col] + 5) % p
    got = _flags(emu, fid, p, m, n_z, mats, z_bad, e, False)
    refs = {i for mat in mats for i, row in enumerate(_rows(mat, p)) if any(c == col for c, _ in row)}
    assert got == _expect(mats, z_bad, e, False, p) and {i for i, f in enumerate(got) if f} == refs
    # strict mode takes u = 1 whatever z[0] holds: the folded z (z[0] != 1) with E dropped is judged against u = 1
    got = _flags(emu, fid, p, m, n_z, mats, z, None, True)
    assert got == _expect(mats, z, None, True, p) and any(got)


@pytest.mark.parametrize("fid,p", FIELDS)
def test_example_strict_with_u_not_one(emu, fid, p):
    """The reference's 4-constraint example: satisfied with z[0] = 1; with z[0] = 2 the strict check still uses u = 1, so the rows that
    read column 0 (the constant 5 of row 3, the B column of rows 2 and 3) decide."""
    m, n_z, mats = example_r1cs(p)
    z = example_z(3, p)
    assert _flags(emu, fid, p, m, n_z, mats, z, None, True) == [False] * 4
    assert _flags(emu, fid, p, m, n_z, mats, z, [0] * m, False) == [False] * 4
    z2 = [2] + z[1:]
    got = _flags(emu, fid, p, m, n_z, mats, z2, None, True)
    assert got == _expect(mats, z2, None, True, p) and got[:2] == [False, False] and any(got[2:])
