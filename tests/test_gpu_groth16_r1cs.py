"""Groth16 from the constraint system on the GPU (kgr_groth16_prove_r1cs): the R1CS evaluations A z, B z, C z computed on the device from a
registered shape and a resident assignment, H, and every query with its scalars read from z in device memory.  Checked against the
restated reference's proof bytes, against the host-evaluation path (kgr_groth16_msms), against the discrete logs of the proof elements,
query by query against kgr_msm, after a device-side producer of z, and for every argument it refuses."""
import numpy as np
import pytest
from groth16_r1cs_util import csr_from_r1cs, mont
from test_groth16 import PROVE_SEED, SETUP_SEED, _enc, _pts, _pts_g2

from oracle import groth16_ref as G
from oracle import pyref as B

pytestmark = pytest.mark.gpu

_SETUPS = {}


def _chain_setup(steps):
    """Host side of a chain circuit of 3 * steps + 1 constraints: CRS exponents, toxic waste, CSR, assignment, evaluations (cached per size)."""
    if steps not in _SETUPS:
        cs, _ = G.chain_circuit(steps, 3)
        E, trap, uvw = G.crs_exponents(cs, B.XorShift128(SETUP_SEED))
        m, n_z, mats = csr_from_r1cs(cs)
        evals = tuple(mont(v) for v in cs.evaluate())
        rng = B.XorShift128(PROVE_SEED)
        r, s = rng.random_field(B.FR), rng.random_field(B.FR)
        _SETUPS[steps] = dict(cs=cs, E=E, trap=trap, uvw=uvw, m=m, n_z=n_z, mats=mats, evals=evals, z=mont(cs.x + cs.w), xs=mont(cs.x), ws=mont(cs.w),
                              r=r, s=s)
    return _SETUPS[steps]


def _points(k, curve, exps):
    from kogarashi_b200 import msm as M
    return M.fixed_base_mul(curve, mont(exps)), np.array([1 if e % G.R == 0 else 0 for e in exps], dtype=np.uint8)


def _prover(st, precompute=False):
    import kogarashi_b200 as k
    from kogarashi_b200.groth16 import Groth16Prover
    E, trap = st["E"], st["trap"]
    vk = _points(k, k.BN254_G1, [trap["delta"], trap["alpha"], trap["beta"]])[0]
    vk2 = _points(k, k.BN254_G2, [trap["delta"], trap["beta"]])[0]
    g1 = [_points(k, k.BN254_G1, E[name]) for name in ("a", "b_g1", "h", "l")]
    return Groth16Prover(vk[0], vk[1], vk[2], *g1[0], *g1[1], *g1[2], *g1[3], vk2[0], vk2[1], *_points(k, k.BN254_G2, E["b_g1"]), precompute=precompute)


def _resident(st):
    from kogarashi_b200.nova import FIELD_FR, DeviceVec, R1csShape
    return R1csShape(FIELD_FR, st["m"], st["n_z"], *st["mats"]), DeviceVec(FIELD_FR, st["z"])


def test_example_circuit_proof_bytes_from_the_constraint_system():
    """groth16/examples/simple.rs through prove_r1cs: the 259-byte proof of the restated reference under the same randomness."""
    import kogarashi_b200 as k
    from kogarashi_b200.groth16 import Groth16G1Prover, Groth16Prover
    from kogarashi_b200.nova import FIELD_FR, DeviceVec, R1csShape
    k.init()
    P, trap, uvw = G.setup(B.XorShift128(SETUP_SEED))
    proof, internals = G.create_proof(P, B.XorShift128(PROVE_SEED), 3, 35)
    vk = P["vk"]
    one = lambda p: _pts([p])[0][0]
    one2 = lambda p: _pts_g2([p])[0][0]
    g1_args = (*_pts(P["a"]), *_pts(P["b_g1"]), *_pts(P["h"]), *_pts(P["l"]))
    prover = Groth16Prover(one(vk["delta_g1"]), one(vk["alpha_g1"]), one(vk["beta_g1"]), *g1_args, one2(vk["delta_g2"]), one2(vk["beta_g2"]),
                           *_pts_g2(P["b_g2"]))
    cs = G.example_circuit(3, 35)
    m, n_z, mats = csr_from_r1cs(cs)
    shape, z = R1csShape(FIELD_FR, m, n_z, *mats), DeviceVec(FIELD_FR, mont(cs.x + cs.w))
    A, Bp, C, q = prover.prove_r1cs(2, shape, z, cs.l, internals["r"], internals["s"])
    assert _enc(A) + _enc(Bp) + _enc(C) == G.proof_bytes(proof)
    assert [B.from_mont(B.limbs_to_int(x), B.FR) for x in q] == internals["q"]
    g1 = Groth16G1Prover(one(vk["delta_g1"]), one(vk["alpha_g1"]), one(vk["beta_g1"]), *g1_args)
    A1, C1, q1 = g1.prove_r1cs(2, shape, z, cs.l, internals["r"], internals["s"])
    assert (A1 == A).all() and (C1 == C).all() and (q1 == q).all()
    prover.free()
    g1.free()


@pytest.mark.parametrize("steps,precompute", [(341, False), (341, True), (1365, False), (1365, True), (21845, False), (21845, True)])
def test_chain_circuit_matches_host_evaluation_path(steps, precompute):
    """2^10, 2^12 and 2^16 constraints: the same proof and q as prove_from_evaluations on host-evaluated a, b, c, q equal to the oracle's H,
    A, B, C equal to their discrete logs; with a host thread per lane and with every lane driven from the calling thread."""
    import kogarashi_b200 as k
    from oracle import oracle as A_
    k.init()
    st = _chain_setup(steps)
    E, cs = st["E"], st["cs"]
    prover = _prover(st, precompute)
    shape, z = _resident(st)
    q_ref, n_ref = A_.groth16_h(E["k"], *st["evals"])
    q_int = [B.from_mont(B.limbs_to_int(x), B.FR) for x in q_ref[:n_ref]]
    a_exp, b_exp, c_exp, pairing_ok = G.expected_exponents(st["trap"], st["uvw"], cs.x, cs.w, q_int, E["n"], st["r"], st["s"])
    assert pairing_ok
    for lane_threads in (1, 0):
        k.set_param("lane_threads", lane_threads)
        try:
            A, Bp, C, q = prover.prove_r1cs(E["k"], shape, z, cs.l, st["r"], st["s"])
            A0, B0, C0, q0 = prover.prove_from_evaluations(E["k"], *st["evals"], st["xs"], st["ws"], st["r"], st["s"])
        finally:
            k.set_param("lane_threads", 1)
        assert (A == A0).all() and (Bp == B0).all() and (C == C0).all() and q.shape == q0.shape and (q == q0).all(), lane_threads
        assert q.shape[0] == n_ref and (q == q_ref[:n_ref]).all()
        assert _enc(A) == G.encode_g1(G.G1.mul(G.G1.g, a_exp))
        assert _enc(C) == G.encode_g1(G.G1.mul(G.G1.g, c_exp))
        assert _enc(Bp) == G.encode_g2(G.g2_mul(G.G2_GEN, b_exp))
    prover.free()


def test_each_query_equals_kgr_msm():
    """The five projective outputs, normalised, against kgr_msm on the same handles with host scalars z, z[l:] and q: a CRS shorter than n_z
    (zip), identity CRS entries, h shorter than the domain, and an assignment without aux (the l query has no pairs: the identity)."""
    import kogarashi_b200 as k
    from kogarashi_b200.msm import Bases, groth16_prove_r1cs
    k.init()
    st = _chain_setup(341)
    E, n_z, l = st["E"], st["n_z"], st["cs"].l
    assert n_z > 1000 and len(E["h"]) < (1 << E["k"])
    ident = lambda exps, idx: [0 if i in idx else e for i, e in enumerate(exps)]
    a = Bases(k.BN254_G1, *_points(k, k.BN254_G1, E["a"][: n_z - 7]))                             # shorter than z
    b_g1 = Bases(k.BN254_G1, *_points(k, k.BN254_G1, ident(E["b_g1"], {0, 3, 500})))            # identity entries
    h = Bases(k.BN254_G1, *_points(k, k.BN254_G1, E["h"]))
    lq = Bases(k.BN254_G1, *_points(k, k.BN254_G1, ident(E["l"], {1, 2})))
    b_g2 = Bases(k.BN254_G2, *_points(k, k.BN254_G2, E["b_g1"][: n_z // 2]))
    shape, z = _resident(st)
    zh = st["z"]
    aff = lambda curve, p: k.to_affine(curve, p)
    for n_inputs in (l, n_z):
        res, q, _ = groth16_prove_r1cs(E["k"], shape, z, n_inputs, h, lq, a, b_g1, b_g2, [])
        assert (aff(0, res["h"]) == aff(0, k.msm_curve_addition(h, q))).all()
        assert (aff(0, res["a"]) == aff(0, k.msm_curve_addition(a, zh))).all()
        assert (aff(0, res["b_g1"]) == aff(0, k.msm_curve_addition(b_g1, zh))).all()
        assert (aff(2, res["b_g2"]) == aff(2, k.msm_curve_addition(b_g2, zh))).all()
        if n_inputs < n_z:
            assert (aff(0, res["l"]) == aff(0, k.msm_curve_addition(lq, zh[n_inputs:]))).all()
            assert not int(aff(0, res["l"])[8])
        else:
            assert int(aff(0, res["l"])[8]) == 1
    for b in (a, b_g1, h, lq, b_g2):
        b.free()


def test_assignment_produced_on_the_device():
    """z = z1 + z2 * r written by kgr_vec_fold_device immediately before the call: the same proof as from an uploaded copy of z."""
    import kogarashi_b200 as k
    from kogarashi_b200.nova import FIELD_FR, DeviceVec
    k.init()
    st = _chain_setup(1365)
    E, cs = st["E"], st["cs"]
    prover = _prover(st)
    shape, z_up = _resident(st)
    z_int = cs.x + cs.w
    rng = B.XorShift128(bytes(range(60, 76)))
    rr = rng.random_field(B.FR)
    z2 = [rng.random_field(B.FR) for _ in z_int]
    z1 = [(v - w * rr) % G.R for v, w in zip(z_int, z2)]
    d1, d2, out = DeviceVec(FIELD_FR, mont(z1)), DeviceVec(FIELD_FR, mont(z2)), DeviceVec(FIELD_FR, n=len(z_int))
    d1.fold(d2, mont([rr])[0], out=out)
    got = prover.prove_r1cs(E["k"], shape, out, cs.l, st["r"], st["s"])
    exp = prover.prove_r1cs(E["k"], shape, z_up, cs.l, st["r"], st["s"])
    assert all((g == e).all() for g, e in zip(got, exp))
    assert (out.download() == st["z"]).all()
    prover.free()


def test_refusals():
    """Every refused argument returns KGR_E_ARG before any work, and a valid call still succeeds afterwards."""
    import kogarashi_b200 as k
    from kogarashi_b200.msm import Bases, groth16_prove_r1cs
    from kogarashi_b200.nova import FIELD_FQ, FIELD_FR, DeviceVec, R1csShape
    st = _chain_setup(5)
    E, m, n_z, l = st["E"], st["m"], st["n_z"], st["cs"].l

    def make():
        g1 = lambda name: Bases(k.BN254_G1, *_points(k, k.BN254_G1, E[name]))
        shape, z = _resident(st)
        return dict(shape=shape, z=z, h=g1("h"), l=g1("l"), a=g1("a"), b_g1=g1("b_g1"), b_g2=Bases(k.BN254_G2, *_points(k, k.BN254_G2, E["b_g1"])))

    def call(o, log_n=None, n_inputs=None, **kw):
        args = dict(o, **kw)
        return groth16_prove_r1cs(E["k"] if log_n is None else log_n, args["shape"], args["z"], l if n_inputs is None else n_inputs, args["h"],
                                  args["l"], args["a"], args["b_g1"], args["b_g2"], [], want_q=False)

    def refused(fn):
        with pytest.raises(k.KgrError, match="kgr error -3"):
            fn()

    k.init()
    o = make()
    valid = call(o)[0]
    grumpkin = Bases(k.GRUMPKIN, np.zeros((1, 8), dtype=np.uint64), np.ones(1, dtype=np.uint8))
    cases = [
        lambda: call(o, shape=R1csShape(FIELD_FQ, m, n_z, *st["mats"])),
        lambda: call(o, z=DeviceVec(FIELD_FQ, st["z"])),
        lambda: call(o, z=DeviceVec(FIELD_FR, np.concatenate([st["z"], st["z"][:1]]))),
        lambda: call(o, n_inputs=0),
        lambda: call(o, n_inputs=n_z + 1),
        lambda: call(o, log_n=0),
        lambda: call(o, log_n=29),
        lambda: call(o, log_n=E["k"] - 1),
        lambda: call(o, h=o["b_g2"]),
        lambda: call(o, l=grumpkin),
        lambda: call(o, a=o["b_g2"]),
        lambda: call(o, b_g1=o["b_g2"]),
        lambda: call(o, b_g2=o["b_g1"]),
    ]
    assert (1 << (E["k"] - 1)) < m
    for case in cases:
        refused(case)
        res = call(o)[0]
        assert all((k.to_affine(2 if q == "b_g2" else 0, res[q]) == k.to_affine(2 if q == "b_g2" else 0, valid[q])).all() for q in res)
    # a context of two engines on one device: registered bases are split into two shards
    k.init([0, 0])
    try:
        refused(lambda: call(make()))
    finally:
        k.init()
    # handles from before the last kgr_init: the shape, the vector, a query
    old = make()
    k.init()
    fresh = make()
    for name in ("shape", "z", "a"):
        refused(lambda: call(fresh, **{name: old[name]}))
        res = call(fresh)[0]
        assert (k.to_affine(0, res["a"]) == k.to_affine(0, valid["a"])).all()
