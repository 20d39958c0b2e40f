"""CPU test of kogarashi_b200/csrc/pairing.cuh: the tower arithmetic, the Frobenius and twist constants, the cyclotomic square, the sparse line
product, the final exponentiation, reduced pairings and the per-proof Groth16 verify body, compiled with g++ (tests/host_emu_pairing.cpp) and
compared limb for limb with the flat big-integer pairing of oracle/pairing_ref.py, which shares no formula with the device tower."""
import os
import random
import subprocess

import numpy as np
import pytest
from conftest import ROOT

from oracle import groth16_ref as G
from oracle import pairing_ref as E
from oracle import pyref as B

EXE = os.path.join(ROOT, "tests", "_build", "host_emu_pairing")
P = E.P
RNG = random.Random(20261022)


@pytest.fixture(scope="module")
def emu(tmp_path_factory):
    os.makedirs(os.path.dirname(EXE), exist_ok=True)
    src = os.path.join(ROOT, "tests", "host_emu_pairing.cpp")
    deps = [src] + [os.path.join(ROOT, "kogarashi_b200", "csrc", f) for f in ("field.cuh", "modinv.cuh", "curve.cuh", "pairing.cuh")]
    if not os.path.exists(EXE) or any(os.path.getmtime(d) > os.path.getmtime(EXE) for d in deps):
        subprocess.check_call(["g++", "-O2", "-std=c++17", "-Wno-unknown-pragmas", "-o", EXE, src])
    tmp = tmp_path_factory.mktemp("pairing")

    def run(op, words):
        fin, fout = tmp / "in.bin", tmp / "out.bin"
        np.asarray(words, dtype=np.uint64).tofile(fin)
        subprocess.check_call([EXE, op, str(fin), str(fout)])
        return np.fromfile(fout, dtype=np.uint64)
    return run


def mont_words(vals):
    out = []
    for v in vals:
        m = v % P * B.R256 % P
        out += [(m >> (64 * k)) & 0xFFFFFFFFFFFFFFFF for k in range(4)]
    return out


def unmont(words):
    r_inv = pow(B.R256, -1, P)
    return [sum(int(words[4 * i + k]) << (64 * k) for k in range(4)) * r_inv % P for i in range(len(words) // 4)]


def rand_tower(n=12):
    return [RNG.randrange(P) for _ in range(n)]


def gt_words(flat):
    return [int(w) for w in E.gt_to_words(flat)]


def g1_words(p):
    return mont_words([0, 0]) + [1] if p is None else mont_words(list(p)) + [0]


def g2_words(q):
    return mont_words([0, 0, 0, 0]) + [1] if q is None else mont_words([*q[0], *q[1]]) + [0]


# ---- Fq6 as the v-part of the flat field: c0 + c1 w^2 + c2 w^4 -----------------------------------------------------------------------
def fq6_flat(t):
    return E.tower_to_flat(list(t) + [0] * 6)


def test_fq6_ops(emu):
    n = 6
    ins, exp = [], []
    for _ in range(n):
        a, b = rand_tower(6), rand_tower(6)
        ins += mont_words(a) + mont_words(b)
        fa, fb = fq6_flat(a), fq6_flat(b)
        for r in (E.f12_mul(fa, fb), E.f12_mul(fa, fa), E.f12_inv(fa)):
            t = E.flat_to_tower(r)
            assert t[6:] == (0,) * 6
            exp += list(t[:6])
    got = unmont(emu("fq6", ins))
    assert got == exp


def test_fq12_ops(emu):
    n = 5
    ins, exp = [], []
    for _ in range(n):
        a, b = rand_tower(), rand_tower()
        ins += mont_words(a) + mont_words(b)
        fa, fb = E.tower_to_flat(a), E.tower_to_flat(b)
        res = [E.f12_mul(fa, fb), E.f12_mul(fa, fa), E.f12_inv(fa)] + [E.f12_pow(fa, P ** k) for k in (1, 2, 3)]
        for r in res:
            exp += list(E.flat_to_tower(r))
    assert unmont(emu("fq12", ins)) == exp


def test_cyclotomic_square(emu):
    ins, exp_easy = [], []
    for _ in range(4):
        a = rand_tower()
        ins += mont_words(a)
        exp_easy.append(E.f12_pow(E.tower_to_flat(a), (P ** 6 - 1) * (P ** 2 + 1)))
    got = unmont(emu("cyc", ins))
    for i, e in enumerate(exp_easy):
        easy, cyc, sq = got[36 * i: 36 * i + 12], got[36 * i + 12: 36 * i + 24], got[36 * i + 24: 36 * i + 36]
        assert E.tower_to_flat(easy) == e
        assert cyc == sq == list(E.flat_to_tower(E.f12_mul(e, e)))


def test_sparse_line_product(emu):
    ins, exp = [], []
    for _ in range(5):
        f, l0, l3, l4 = rand_tower(), rand_tower(2), rand_tower(2), rand_tower(2)
        ins += mont_words(f) + mont_words(l0 + l3 + l4)
        line = E.tower_to_flat(l0 + [0] * 4 + l3 + l4 + [0, 0])
        exp += list(E.flat_to_tower(E.f12_mul(E.tower_to_flat(f), line)))
    assert unmont(emu("m034", ins)) == exp


def _f2pow(a, e):
    acc = (1, 0)
    for bit in bin(e)[2:]:
        acc = G.f2_mul(acc, acc)
        if bit == "1":
            acc = G.f2_mul(acc, a)
    return acc


def test_frobenius_and_twist_constants(emu):
    got = unmont(emu("consts", []))
    exp = []
    for k in (1, 2, 3):
        for e in range(1, 6):
            exp += list(_f2pow((9, 1), e * (P ** k - 1) // 6))
    b = G.G2_B
    assert G.f2_mul(b, (9, 1)) == (3, 0)                 # b' = 3 / xi
    exp += list(b) + list(G.f2_add(G.f2_add(b, b), b))
    assert got == exp
    # the untwisting constants of pi(Q), pi^2(Q) and the sign of -pi^2(Q)
    assert _f2pow((9, 1), (P ** 2 - 1) // 2) == (P - 1, 0)


def test_final_exponentiation(emu):
    ins, exp = [], []
    for _ in range(3):
        a = rand_tower()
        ins += mont_words(a)
        exp += gt_words(E.final_exp(E.tower_to_flat(a)))
    assert [int(w) for w in emu("fexp", ins)] == exp


def _rand_g1():
    return E.G1.mul(E.G1.g, RNG.randrange(1, E.R))


def _rand_g2():
    return G.g2_mul(G.G2_GEN, RNG.randrange(1, E.R))


def test_reduced_pairings(emu):
    pairs = [(_rand_g1(), _rand_g2()) for _ in range(3)] + [(None, _rand_g2()), (_rand_g1(), None), (E.G1.g, G.G2_GEN)]
    ins, exp = [], []
    for p, q in pairs:
        ins += g1_words(p) + g2_words(q)
        exp += [1] + gt_words(E.pairing(p, q))
    got = [int(w) for w in emu("pair", ins)]
    assert got == exp
    one = gt_words(E.ONE)
    assert got[49 * 3 + 1: 49 * 4] == one and got[49 * 4 + 1: 49 * 5] == one


def test_pair_refuses_invalid_points(emu):
    p, q = _rand_g1(), _rand_g2()
    off_curve = (p[0], (p[1] + 1) % P)
    ins = g1_words(off_curve) + g2_words(q) + g1_words(p) + g2_words(((q[0][0] + 1, q[0][1]), q[1])) + g1_words((P, 2)) + g2_words(q)
    got = emu("pair", ins)
    assert [int(got[49 * i]) for i in range(3)] == [0, 0, 0]


def example_setup():
    from test_groth16 import PROVE_SEED, SETUP_SEED
    P_, trap, uvw = G.setup(B.XorShift128(SETUP_SEED))
    proof, internals = G.create_proof(P_, B.XorShift128(PROVE_SEED), 3, 35)
    return P_, proof, internals


def verify_words(vk, proofs, inputs_rows):
    n_public = len(vk["ic"]) - 1
    w = [n_public, len(proofs)]
    for pt in (vk["alpha_g1"], vk["beta_g1"], vk["delta_g1"]):
        w += g1_words(pt)
    for pt in (vk["beta_g2"], vk["gamma_g2"], vk["delta_g2"]):
        w += g2_words(pt)
    for pt in vk["ic"]:
        w += g1_words(pt)
    for pr in proofs:
        w += g1_words(pr["a"]) + g2_words(pr["b"]) + g1_words(pr["c"])
    for row in inputs_rows:
        for x in row:
            m = x % E.R * B.R256 % E.R
            w += [(m >> (64 * k)) & 0xFFFFFFFFFFFFFFFF for k in range(4)]
    return w


def test_verify_body_on_the_example_proof(emu):
    P_, proof, internals = example_setup()
    vk = P_["vk"]
    pub = internals["inputs"][1:]
    g1 = E.G1
    tampered = [dict(proof, a=g1.add(proof["a"], g1.g)), dict(proof, a=proof["c"], c=proof["a"]),
                dict(proof, b=G.g2_add(proof["b"], G.G2_GEN)), dict(proof, c=None)]
    proofs = [proof] + tampered + [proof]
    inputs = [pub] * 5 + [[pub[0], (pub[1] + 1) % E.R]]
    got = [int(v) for v in emu("verify", verify_words(vk, proofs, inputs))]
    assert got == [1, 0, 0, 0, 0, 0]
