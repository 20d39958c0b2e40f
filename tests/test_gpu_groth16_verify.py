"""Groth16 verification on the B200 (kgr_groth16_verify, groth16.Groth16Verifier): proofs from a setup whose toxic waste is never shown to the
check verify at several batch sizes; the restated reference's example proof verifies; one tampered proof in a batch of 64 gets verdict 0 and
only it (the batched check fails and the per-proof fallback runs); verdicts agree with oracle/pairing_ref.py; every refusal of the header; and
the launch count of a call grows with k only by the levels of the product tree."""
import ctypes
import random

import numpy as np
import pytest
from groth16_r1cs_util import csr_from_r1cs, mont
from test_groth16 import PROVE_SEED, SETUP_SEED, _pts

from oracle import groth16_ref as G
from oracle import pairing_ref as E
from oracle import pyref as B

pytestmark = pytest.mark.gpu
R = G.R
P = G.Q


def _fq(words):
    return B.from_mont(B.limbs_to_int([int(w) for w in words]), P)


def _fq_words(v):
    return B.int_to_limbs(B.to_mont(v % P, P))


def g1_of(row):
    return None if int(row[8]) else (_fq(row[0:4]), _fq(row[4:8]))


def g2_of(row):
    return None if int(row[16]) else ((_fq(row[0:4]), _fq(row[4:8])), (_fq(row[8:12]), _fq(row[12:16])))


def g1_row(p):
    return np.array([0] * 8 + [1] if p is None else _fq_words(p[0]) + _fq_words(p[1]) + [0], dtype=np.uint64)


def g2_row(q):
    return np.array([0] * 16 + [1] if q is None else [w for v in (*q[0], *q[1]) for w in _fq_words(v)] + [0], dtype=np.uint64)


class Key:
    """A chain circuit of m = 3 steps + 1 constraints set up on the device with random toxic waste, and a pool of proofs for several x0."""

    def __init__(self, steps, x0s, per_x0, seed):
        from kogarashi_b200.groth16 import Groth16Prover, Groth16Verifier, setup
        from kogarashi_b200.nova import FIELD_FR, DeviceVec, R1csShape
        cs0, _ = G.chain_circuit(steps, 3)
        m, n_z, mats = csr_from_r1cs(cs0)
        self.shape = R1csShape(FIELD_FR, m, n_z, *mats)
        self.params = setup(self.shape, cs0.l)
        self.verifier = Groth16Verifier.from_params(self.params)
        prover = Groth16Prover.from_params(self.params)
        rng = random.Random(seed)
        self.proofs, self.inputs = [], []
        for x0 in x0s:
            cs, out = G.chain_circuit(steps, x0)
            z = DeviceVec(FIELD_FR, mont(cs.x + cs.w))
            for _ in range(per_x0):
                A, Bp, C, _ = prover.prove_r1cs(self.params.log_n, self.shape, z, cs.l, rng.randrange(1, R), rng.randrange(1, R))
                self.proofs.append((A, Bp, C))
                self.inputs.append([x0 % R, out])
            z.free()
        prover.free()

    def batch(self, k):
        idx = [i % len(self.proofs) for i in range(k)]
        return [self.proofs[i] for i in idx], [list(self.inputs[i]) for i in idx]


@pytest.fixture(scope="module")
def k():
    import kogarashi_b200 as kk
    kk.init()
    return kk


@pytest.fixture(scope="module")
def key10(k):
    return Key(341, [3, 5, 12345, R - 1], 4, seed=10)


@pytest.fixture(scope="module")
def key10b(k):
    return Key(341, [3], 1, seed=11)


@pytest.mark.parametrize("n", [1, 2, 3, 64, 1000, 4096])
def test_valid_proofs_pass(key10, n):
    proofs, inputs = key10.batch(n)
    assert key10.verifier.verify(proofs, inputs).all()


def test_valid_proofs_pass_2p12(k):
    key = Key(1365, [7, 99], 2, seed=12)
    assert key.params.log_n == 12
    for n in (1, 3, 64):
        proofs, inputs = key.batch(n)
        assert key.verifier.verify(proofs, inputs).all()


def test_reference_example_proof_passes(k):
    from kogarashi_b200.groth16 import Groth16Verifier
    Pm, _, _ = G.setup(B.XorShift128(SETUP_SEED))
    proof, internals = G.create_proof(Pm, B.XorShift128(PROVE_SEED), 3, 35)
    vk = Pm["vk"]
    vk_g1 = np.stack([g1_row(vk[n]) for n in ("alpha_g1", "beta_g1", "delta_g1")])
    vk_g2 = np.stack([g2_row(vk[n]) for n in ("beta_g2", "gamma_g2", "delta_g2")])
    ver = Groth16Verifier(vk_g1, vk_g2, _pts(vk["ic"]))
    pr = (g1_row(proof["a"]), g2_row(proof["b"]), g1_row(proof["c"]))
    pub = internals["inputs"][1:]
    assert ver.verify([pr], [pub]).tolist() == [True]
    assert ver.verify([pr, pr], [pub, [pub[0], pub[1] + 1]]).tolist() == [True, False]
    ver.free()


def _tamper(mode, proof, inputs, other):
    A, Bp, C = (np.array(x, dtype=np.uint64) for x in proof)
    inputs = list(inputs)
    if mode == "a_plus_g1":
        A = g1_row(E.G1.add(g1_of(A), E.G1.g))
    elif mode == "b_plus_g2":
        Bp = g2_row(G.g2_add(g2_of(Bp), G.G2_GEN))
    elif mode == "c_plus_g1":
        C = g1_row(E.G1.add(g1_of(C), E.G1.g))
    elif mode == "swap_a_c":
        A, C = C, A
    elif mode == "input_plus_one":
        inputs[0] = (inputs[0] + 1) % R
    elif mode == "other_key":
        A, Bp, C = (np.array(x, dtype=np.uint64) for x in other)
    elif mode in ("identity_a", "identity_b", "identity_c"):
        t = {"identity_a": A, "identity_b": Bp, "identity_c": C}[mode]
        t[-1] = 1
    elif mode == "off_curve_a":
        x, y = g1_of(A)
        A = g1_row((x, y + 1))
    elif mode == "coordinate_ge_p":
        A[0:4] = B.int_to_limbs(B.limbs_to_int(A[0:4].tolist()) + P)
    elif mode == "b_outside_g2":
        from test_gpu_pairing import twist_point_outside_g2
        Bp = g2_row(twist_point_outside_g2(5))
    return (A, Bp, C), inputs


TAMPER = ["a_plus_g1", "b_plus_g2", "c_plus_g1", "swap_a_c", "input_plus_one", "other_key", "identity_a", "identity_b", "identity_c",
          "off_curve_a", "coordinate_ge_p", "b_outside_g2"]


@pytest.mark.parametrize("mode", TAMPER)
def test_one_tampered_proof_in_64(key10, key10b, mode):
    proofs, inputs = key10.batch(64)
    at = 37
    proofs[at], inputs[at] = _tamper(mode, proofs[at], inputs[at], key10b.proofs[0])
    got = key10.verifier.verify(proofs, inputs)
    exp = np.ones(64, dtype=bool)
    exp[at] = False
    assert (got == exp).all(), np.nonzero(got != exp)


def test_verdicts_agree_with_the_oracle(key10, key10b):
    proofs, inputs = key10.batch(8)
    for i, mode in ((1, "c_plus_g1"), (4, "other_key"), (6, "input_plus_one")):
        proofs[i], inputs[i] = _tamper(mode, proofs[i], inputs[i], key10b.proofs[0])
    got = key10.verifier.verify(proofs, inputs)
    host = key10.params.download()
    vk1, vk2 = host["vk_g1"], host["vk_g2"]
    ic_pts, ic_inf = host["ic"]
    vk = dict(alpha_g1=g1_of(vk1[0]), beta_g2=g2_of(vk2[0]), gamma_g2=g2_of(vk2[1]), delta_g2=g2_of(vk2[2]),
              ic=[None if f else (_fq(p[0:4]), _fq(p[4:8])) for p, f in zip(ic_pts, ic_inf)])
    exp = [E.verify(vk, dict(a=g1_of(pr[0]), b=g2_of(pr[1]), c=g1_of(pr[2])), x) for pr, x in zip(proofs, inputs)]
    assert got.tolist() == exp == [True, False, True, True, False, True, False, True]


def _raw_call(key, proofs, inputs, rho, ic=None, vk_g1=None, vk_g2=None, n_public=None, null=None):
    """kgr_groth16_verify through ctypes with every argument under the test's control -> return code."""
    from kogarashi_b200 import _lib
    L = _lib.lib()
    u64p = ctypes.POINTER(ctypes.c_uint64)
    arr = lambda a: None if a is None else np.ascontiguousarray(a, dtype=np.uint64)
    vk_g1 = arr(key.verifier.vk_g1 if vk_g1 is None else vk_g1)
    vk_g2 = arr(key.verifier.vk_g2 if vk_g2 is None else vk_g2)
    pr = np.stack([np.concatenate([np.asarray(x, dtype=np.uint64).reshape(-1) for x in p[:3]]) for p in proofs])
    xs = np.stack([mont(x) for x in inputs])
    rho = arr(rho)
    ok = np.zeros(len(proofs) + 1, dtype=np.uint32)
    ptr = lambda a: None if a is None else a.ctypes.data_as(u64p)
    args = [ptr(vk_g1), ptr(vk_g2), (key.verifier.ic if ic is None else ic)._h, ptr(pr), len(proofs), ptr(xs),
            2 if n_public is None else n_public, ptr(rho), ok.ctypes.data_as(ctypes.POINTER(ctypes.c_uint32))]
    if null is not None:
        args[null] = None
    return L.kgr_groth16_verify(*args)


def test_every_refusal(k, key10):
    E_ARG = -3
    proofs, inputs = key10.batch(3)
    rho = np.arange(1, 7, dtype=np.uint64).reshape(3, 2)
    assert _raw_call(key10, proofs, inputs, rho) == 0
    for null in (0, 1, 3, 5, 8):
        assert _raw_call(key10, proofs, inputs, rho, null=null) == E_ARG, null
    assert _raw_call(key10, proofs, inputs, None) == E_ARG                      # k >= 2 without rho
    zero = rho.copy()
    zero[1] = 0
    assert _raw_call(key10, proofs, inputs, zero) == E_ARG                      # a zero rho_i
    assert _raw_call(key10, proofs, inputs, rho, n_public=1) == E_ARG           # n_public + 1 != ic->n
    from kogarashi_b200 import _lib
    L = _lib.lib()
    # an input >= r: r itself as a raw Montgomery word pattern
    xs_bad = np.stack([mont(x) for x in inputs])
    xs_bad[2, 1] = B.int_to_limbs(R)
    pr = np.stack([np.concatenate([np.asarray(x, dtype=np.uint64).reshape(-1) for x in p[:3]]) for p in proofs])
    ok = np.zeros(3, dtype=np.uint32)
    u64p = ctypes.POINTER(ctypes.c_uint64)
    rc = L.kgr_groth16_verify(key10.verifier.vk_g1.ctypes.data_as(u64p), key10.verifier.vk_g2.ctypes.data_as(u64p), key10.verifier.ic._h,
                              pr.ctypes.data_as(u64p), 3, xs_bad.ctypes.data_as(u64p), 2, rho.ctypes.data_as(u64p),
                              ok.ctypes.data_as(ctypes.POINTER(ctypes.c_uint32)))
    assert rc == E_ARG
    # identity gamma or delta, an invalid vk point
    for j in (1, 2):
        vk2 = key10.verifier.vk_g2.copy()
        vk2[j, 16] = 1
        assert _raw_call(key10, proofs, inputs, rho, vk_g2=vk2) == E_ARG, j
    vk1 = key10.verifier.vk_g1.copy()
    vk1[0, 4:8] = B.int_to_limbs(B.limbs_to_int(vk1[0, 4:8].tolist()) ^ 1)
    assert _raw_call(key10, proofs, inputs, rho, vk_g1=vk1) == E_ARG
    # ic of the wrong curve
    from kogarashi_b200.msm import Bases
    g2 = Bases(k.BN254_G2, np.array([g2_row(G.G2_GEN)[:16]] * 3))
    assert _raw_call(key10, proofs, inputs, rho, ic=g2) == E_ARG
    g2.free()
    # k == 0: nothing to do
    assert L.kgr_groth16_verify(key10.verifier.vk_g1.ctypes.data_as(u64p), key10.verifier.vk_g2.ctypes.data_as(u64p), key10.verifier.ic._h, None, 0,
                                None, 2, None, None) == 0


def test_launch_count_grows_only_with_the_product_tree(key10):
    import kogarashi_b200 as kk

    def launches(n, tamper=None):
        proofs, inputs = key10.batch(n)
        if tamper:
            proofs[1], inputs[1] = _tamper(tamper, proofs[1], inputs[1], None)
        before = kk.launch_count()
        got = key10.verifier.verify(proofs, inputs)
        return kk.launch_count() - before, got

    def levels(n):
        lv = 0
        while n > 1:
            n, lv = (n + 1) // 2, lv + 1
        return lv

    c64, ok64 = launches(64)
    c4096, ok4096 = launches(4096)
    assert ok64.all() and ok4096.all()
    assert c4096 - c64 == levels(4096) - levels(64) == 6
    cbad, okbad = launches(64, "c_plus_g1")
    assert okbad.sum() == 63 and not okbad[1]
    assert cbad > c64


def test_stale_ic_after_reinit():
    import kogarashi_b200 as kk
    from kogarashi_b200.groth16 import Groth16Verifier
    kk.init()
    Pm, _, _ = G.setup(B.XorShift128(SETUP_SEED))
    proof, internals = G.create_proof(Pm, B.XorShift128(PROVE_SEED), 3, 35)
    vk = Pm["vk"]
    ver = Groth16Verifier(np.stack([g1_row(vk[n]) for n in ("alpha_g1", "beta_g1", "delta_g1")]),
                          np.stack([g2_row(vk[n]) for n in ("beta_g2", "gamma_g2", "delta_g2")]), _pts(vk["ic"]))
    pr = (g1_row(proof["a"]), g2_row(proof["b"]), g1_row(proof["c"]))
    assert ver.verify([pr], [internals["inputs"][1:]]).all()
    kk.init()
    with pytest.raises(kk.KgrError, match="error -3"):
        ver.verify([pr], [internals["inputs"][1:]])
    ver.free()


def test_multi_device_context_is_refused():
    import kogarashi_b200 as kk
    from kogarashi_b200.groth16 import Groth16Verifier
    try:
        kk.init([0, 0])
    except kk.KgrError:
        kk.init()
        pytest.skip("this driver refuses two engines on one device")
    try:
        Pm, _, _ = G.setup(B.XorShift128(SETUP_SEED))
        vk = Pm["vk"]
        ver = Groth16Verifier(np.stack([g1_row(vk[n]) for n in ("alpha_g1", "beta_g1", "delta_g1")]),
                              np.stack([g2_row(vk[n]) for n in ("beta_g2", "gamma_g2", "delta_g2")]), _pts(vk["ic"]))
        with pytest.raises(kk.KgrError, match="error -3"):
            ver.verify([(g1_row(None), g2_row(None), g1_row(None))], [[1, 2]])
        ver.free()
    finally:
        kk.init()
