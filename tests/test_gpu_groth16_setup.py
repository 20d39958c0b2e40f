"""Groth16 parameter generation on the GPU (kgr_groth16_setup, groth16.setup): every query and vk element against the restated reference's setup
and against crs_exponents, a hot column that holds every row, a valid proof at 2^20 constraints checked without the oracle, determinism, every
refusal, and the lifetime of the handles it returns."""
import ctypes

import numpy as np
import pytest
from groth16_r1cs_util import csr_from_r1cs, edge_circuit, mont
from test_groth16 import PROVE_SEED, SETUP_SEED, _enc, _pts, _pts_g2

from oracle import groth16_ref as G
from oracle import pyref as B

pytestmark = pytest.mark.gpu

R = G.R
_LAGR = {}


def _lagr(k, tau):
    if (k, tau) not in _LAGR:
        _LAGR[(k, tau)] = G.lagrange_at(1 << k, pow(G.ROOT_OF_UNITY, 1 << (G.S - k), R), tau)
    return _LAGR[(k, tau)]


def _need_gib(gib):
    import torch
    free = torch.cuda.mem_get_info()[0]
    if free < gib << 30:
        pytest.skip(f"needs {gib} GiB of free device memory, {free / 2**30:.1f} GiB free")


def _resident(cs, split=()):
    from kogarashi_b200.nova import FIELD_FR, DeviceVec, R1csShape
    m, n_z, mats = csr_from_r1cs(cs, split_rows=split)
    return R1csShape(FIELD_FR, m, n_z, *mats), DeviceVec(FIELD_FR, mont(cs.x + cs.w))


def _toxic(trap):
    return [trap[x] for x in ("alpha", "beta", "gamma", "delta", "tau")]


def _same_points(got, inf, ref_xy, ref_inf):
    """Downloaded query vs the reference's encoding: equal flags, equal coordinates of every non-identity, (0, 0) for every identity."""
    assert (inf == ref_inf).all()
    assert (got[ref_inf == 0] == ref_xy[ref_inf == 0]).all()
    assert not got[ref_inf == 1].any()


def _fixed(curve, exps):
    from kogarashi_b200.msm import fixed_base_mul
    return fixed_base_mul(curve, mont(exps))


def test_example_circuit_matches_reference_setup_and_proof_bytes():
    """zksnark.rs:17-127 on the example circuit under the toxic waste of XorShift128(SETUP_SEED): every point byte-equal to the restated
    reference's setup, and the 259-byte proof from Groth16Prover.from_params."""
    import kogarashi_b200 as k
    from kogarashi_b200.groth16 import Groth16Prover, setup
    k.init()
    P, trap, uvw = G.setup(B.XorShift128(SETUP_SEED))
    proof, internals = G.create_proof(P, B.XorShift128(PROVE_SEED), 3, 35)
    cs = G.example_circuit(3, 35)
    shape, z = _resident(cs)
    params = setup(shape, cs.l, toxic=_toxic(trap))
    assert params.log_n == 2
    host = params.download()
    for name in ("a", "b_g1", "ic", "l", "h"):
        _same_points(*host[name], *_pts(P[name]))
    _same_points(*host["b_g2"], *_pts_g2(P["b_g2"]))
    vk = P["vk"]
    for i, name in enumerate(("alpha_g1", "beta_g1", "delta_g1")):
        _same_points(host["vk_g1"][i:i + 1, :8], host["vk_g1"][i:i + 1, 8].astype(np.uint8), *_pts([vk[name]]))
    for i, name in enumerate(("beta_g2", "gamma_g2", "delta_g2")):
        _same_points(host["vk_g2"][i:i + 1, :16], host["vk_g2"][i:i + 1, 16].astype(np.uint8), *_pts_g2([vk[name]]))
    prover = Groth16Prover.from_params(params)
    assert params.a is None and params.b_g2 is None and params.ic is not None
    A, Bp, C, q = prover.prove_r1cs(params.log_n, shape, z, cs.l, internals["r"], internals["s"])
    assert _enc(A) + _enc(Bp) + _enc(C) == G.proof_bytes(proof)
    prover.free()
    params.free()


CHAINS = [("chain_341", 341), ("chain_1365", 1365), ("chain_21845", 21845), ("chain_100", 100), ("edge", None)]


@pytest.mark.parametrize("name,steps", CHAINS)
def test_queries_match_crs_exponents(name, steps):
    """Chains of 2^10, 2^12 and 2^16 constraints, m = 301 and the edge circuit: each query equals fixed_base_mul of crs_exponents, identities
    included; for m = 2^k the proof of prove_r1cs has the discrete logs of expected_exponents and satisfies the Groth16 equation."""
    import kogarashi_b200 as k
    from kogarashi_b200.groth16 import Groth16Prover, setup
    k.init()
    cs, split = edge_circuit() if steps is None else (G.chain_circuit(steps, 3)[0], ())
    E, trap, uvw = G.crs_exponents(cs, B.XorShift128(SETUP_SEED))
    shape, z = _resident(cs, split)
    params = setup(shape, cs.l, toxic=_toxic(trap))
    assert params.log_n == E["k"]
    host = params.download()
    for name_q in ("a", "b_g1", "ic", "l", "h"):
        exps = E[name_q]
        _same_points(*host[name_q], _fixed(k.BN254_G1, exps), np.array([e % R == 0 for e in exps], dtype=np.uint8))
    _same_points(*host["b_g2"], _fixed(k.BN254_G2, E["b_g1"]), np.array([e % R == 0 for e in E["b_g1"]], dtype=np.uint8))
    if cs.m == E["n"]:
        rng = B.XorShift128(PROVE_SEED)
        r, s = rng.random_field(R), rng.random_field(R)
        prover = Groth16Prover.from_params(params)
        A, Bp, C, q = prover.prove_r1cs(params.log_n, shape, z, cs.l, r, s)
        q_int = [B.from_mont(B.limbs_to_int(x), B.FR) for x in q]
        a_exp, b_exp, c_exp, pairing_ok = G.expected_exponents(trap, uvw, cs.x, cs.w, q_int, E["n"], r, s)
        assert pairing_ok
        assert _enc(A) == G.encode_g1(G.G1.mul(G.G1.g, a_exp))
        assert _enc(Bp) == G.encode_g2(G.g2_mul(G.G2_GEN, b_exp))
        assert _enc(C) == G.encode_g1(G.G1.mul(G.G1.g, c_exp))
        prover.free()
    params.free()


def _k20_toxic():
    rng = B.XorShift128(bytes(range(100, 116)))
    return [rng.random_field(R) for _ in range(5)]


def test_hot_column_of_every_row():
    """2^20 rows whose B holds the constant column in every row (coefficients 2, 3, ...) beside one column of its own: that column's b_g1 and b_g2
    points and 256 sampled others against Python sums over the closed-form Lagrange basis."""
    import kogarashi_b200 as k
    from kogarashi_b200.groth16 import setup
    from kogarashi_b200.nova import FIELD_FR, R1csShape
    k.init()
    _need_gib(8)
    K = 20
    m = 1 << K
    al, be, ga, de, tau = _k20_toxic()
    rows = np.arange(m, dtype=np.uint32)
    one = mont([1])[0]
    mat_a = (np.arange(m + 1, dtype=np.uint32), rows + 1, np.tile(one, (m, 1)))
    b_cols = np.stack([np.zeros(m, dtype=np.uint32), rows + 1], axis=1).reshape(-1)
    b_coeffs = np.stack([mont([i + 2 for i in range(m)]), np.tile(one, (m, 1))], axis=1).reshape(-1, 4)
    mat_b = (np.arange(0, 2 * m + 1, 2, dtype=np.uint32), b_cols, b_coeffs)
    mat_c = (np.arange(m + 1, dtype=np.uint32), ((rows * 7) % m + 1).astype(np.uint32), np.tile(mont([3])[0], (m, 1)))
    shape = R1csShape(FIELD_FR, m, m + 1, mat_a, mat_b, mat_c)
    params = setup(shape, 1, toxic=[al, be, ga, de, tau])
    assert params.log_n == K
    lagr = _lagr(K, tau)
    v0 = sum((i + 2) * l for i, l in enumerate(lagr)) % R
    sample = [int(j) for j in np.random.default_rng(7).choice(np.arange(1, m + 1), 256, replace=False)]
    exps = [v0] + [lagr[j - 1] for j in sample]
    for b, curve in ((params.b_g1, k.BN254_G1), (params.b_g2, k.BN254_G2)):
        got = np.stack([b.download(j, 1)[0] for j in [0] + sample])
        assert (got == _fixed(curve, exps)).all()
    params.free()
    shape.free()


def test_valid_proof_at_2_20_constraints():
    """A chain of 349525 steps (m = 2^20): the proof from setup + prove_r1cs checked without the oracle.  U, V, W = sum_i l_i (Az, Bz, Cz)_i in
    Python integers, the input part from the instance columns only; A, B, C must have the discrete logs these give, H(tau) Z(tau) = UV - W, and
    the Groth16 equation holds in the exponent.  256 entries of every query against fixed_base_mul of Python values."""
    import kogarashi_b200 as k
    from kogarashi_b200.groth16 import Groth16Prover, setup
    k.init()
    _need_gib(8)
    K = 20
    cs, _ = G.chain_circuit(349525, 3)
    assert cs.m == 1 << K
    al, be, ga, de, tau = _k20_toxic()
    shape, z = _resident(cs)
    params = setup(shape, cs.l, toxic=[al, be, ga, de, tau])
    assert params.log_n == K
    lagr = _lagr(K, tau)
    zv = cs.x + cs.w
    l_in, n_z = cs.l, len(zv)
    cols = [cs.columns(mat) for mat in (cs.a, cs.b, cs.c)]
    ev = lambda col: sum(lagr[i] * co for co, i in col) % R
    uvw_of = lambda j: tuple(ev(xs[j] if j < l_in else ws[j - l_in]) for xs, ws in cols)
    # 256 entries of every query
    rng = np.random.default_rng(11)
    pick = lambda n: sorted(int(j) for j in rng.choice(n, min(256, n), replace=False))
    ja, jl, jh = pick(n_z), pick(n_z - l_in), pick(cs.m - 1)
    uvw_a = {j: uvw_of(j) for j in ja}
    uvw_l = {j: uvw_of(l_in + j) for j in jl}
    zt = (pow(tau, 1 << K, R) - 1) % R
    checks = [(params.a, k.BN254_G1, ja, [uvw_a[j][0] for j in ja]), (params.b_g1, k.BN254_G1, ja, [uvw_a[j][1] for j in ja]),
              (params.b_g2, k.BN254_G2, ja, [uvw_a[j][1] for j in ja]),
              (params.ic, k.BN254_G1, list(range(l_in)), [(be * u + al * v + w) * pow(ga, -1, R) for u, v, w in map(uvw_of, range(l_in))]),
              (params.l, k.BN254_G1, jl, [(be * uvw_l[j][0] + al * uvw_l[j][1] + uvw_l[j][2]) * pow(de, -1, R) for j in jl]),
              (params.h, k.BN254_G1, jh, [pow(tau, i, R) * zt * pow(de, -1, R) for i in jh])]
    for b, curve, idx, exps in checks:
        got = np.stack([b.download(j, 1)[0] for j in idx])
        assert (got == _fixed(curve, exps)).all()
    # the proof
    a_ev, b_ev, c_ev = cs.evaluate()
    U, V, W = (sum(l * x for l, x in zip(lagr, v)) % R for v in (a_ev, b_ev, c_ev))
    in_part = sum(zv[j] * (be * u + al * v + w) for j, (u, v, w) in enumerate(map(uvw_of, range(l_in)))) % R
    rr = B.XorShift128(PROVE_SEED)
    r, s = rr.random_field(R), rr.random_field(R)
    prover = Groth16Prover.from_params(params)
    A, Bp, C, q = prover.prove_r1cs(params.log_n, shape, z, cs.l, r, s)
    q_int = [B.from_mont(B.limbs_to_int(x), B.FR) for x in q]
    ht = 0
    for c in reversed(q_int):
        ht = (ht * tau + c) % R
    assert ht * zt % R == (U * V - W) % R
    a_exp = (al + r * de + U) % R
    b_exp = (be + s * de + V) % R
    aux_part = (be * U + al * V + W - in_part) % R
    c_exp = ((aux_part + ht * zt) * pow(de, -1, R) + s * a_exp + r * b_exp - r * s * de) % R
    assert (a_exp * b_exp - (al * be + in_part + c_exp * de)) % R == 0
    assert _enc(A) == G.encode_g1(G.G1.mul(G.G1.g, a_exp))
    assert _enc(Bp) == G.encode_g2(G.g2_mul(G.G2_GEN, b_exp))
    assert _enc(C) == G.encode_g1(G.G1.mul(G.G1.g, c_exp))
    prover.free()
    params.free()


def test_deterministic_across_calls_and_sizes():
    import kogarashi_b200 as k
    from kogarashi_b200.groth16 import setup
    k.init()
    cs = G.chain_circuit(341, 3)[0]
    other = G.chain_circuit(100, 3)[0]
    toxic = _k20_toxic()
    shape, _ = _resident(cs)
    shape_o, _ = _resident(other)
    p1 = setup(shape, cs.l, toxic=toxic)
    p_other = setup(shape_o, other.l, toxic=toxic[::-1])
    p2 = setup(shape, cs.l, toxic=toxic)
    d1, d2 = p1.download(), p2.download()
    for key in d1:
        if key == "log_n":
            assert d1[key] == d2[key]
        elif isinstance(d1[key], tuple):
            assert all((a == b).all() for a, b in zip(d1[key], d2[key])), key
        else:
            assert (d1[key] == d2[key]).all(), key
    for p in (p1, p2, p_other):
        p.free()


def _raw_setup(shape, n_inputs, toxic, g2=True, drop=None):
    """kgr_groth16_setup with every output handle preset to a non-NULL value -> (rc, handle values after the call)."""
    import kogarashi_b200 as k
    u64p = ctypes.POINTER(ctypes.c_uint64)
    tox = mont(toxic)
    hs = [ctypes.c_void_p(0x1000 + i) for i in range(6)]
    refs = [ctypes.byref(h) for h in hs]
    if not g2:
        refs[4] = None
    log_n = ctypes.c_uint32(99)
    vk1, vk2 = np.zeros((3, 9), dtype=np.uint64), np.zeros((3, 17), dtype=np.uint64)
    args = [shape._h if shape is not None else None, n_inputs, tox.ctypes.data_as(u64p), ctypes.byref(log_n), *refs, vk1.ctypes.data_as(u64p),
            vk2.ctypes.data_as(u64p)]
    if drop is not None:
        args[drop] = None
    rc = k.lib().kgr_groth16_setup(*args)
    return rc, [h.value for h in hs]


def test_refusals_leave_outputs_null():
    import kogarashi_b200 as k
    from kogarashi_b200.nova import FIELD_FQ, FIELD_FR, R1csShape
    k.init()
    cs = G.chain_circuit(5, 3)[0]
    m, n_z, mats = csr_from_r1cs(cs)
    toxic = _k20_toxic()
    old = R1csShape(FIELD_FR, m, n_z, *mats)
    k.init()
    shape = R1csShape(FIELD_FR, m, n_z, *mats)

    def refused(*a, **kw):
        rc, hs = _raw_setup(*a, **kw)
        assert rc == -3, k.lib().kgr_last_error()
        drop = kw.get("drop")
        not_passed = {drop - 4} if drop is not None and 4 <= drop < 10 else set()   # an output slot the call was not given
        assert all(h is None for i, h in enumerate(hs) if i not in not_passed)

    refused(None, cs.l, toxic)
    for drop in (2, 3, 4, 5, 6, 7, 9, 10):  # toxic, log_n_out, h, l, a, b_g1, ic, vk_g1
        refused(shape, cs.l, toxic, drop=drop)
    refused(shape, cs.l, toxic, drop=11)    # b_g2 given without vk_g2
    refused(old, cs.l, toxic)
    refused(R1csShape(FIELD_FQ, m, n_z, *mats), cs.l, toxic)
    refused(shape, 0, toxic)
    refused(shape, n_z + 1, toxic)
    refused(shape, cs.l, toxic[:2] + [0] + toxic[3:])
    refused(shape, cs.l, toxic[:3] + [0] + toxic[4:])
    rc, hs = _raw_setup(shape, cs.l, toxic, g2=False)    # valid, G1 only; vk_g2 is still filled
    assert rc == 0 and all(hs[i] for i in (0, 1, 2, 3, 5))
    for i in (0, 1, 2, 3, 5):
        k.lib().kgr_bases_free(ctypes.c_void_p(hs[i]))
    # toxic values >= r (not reduced): the raw limbs of r itself
    u64p = ctypes.POINTER(ctypes.c_uint64)
    bad = mont(toxic)
    bad[4] = B.int_to_limbs(R)
    out = [ctypes.c_void_p(1) for _ in range(6)]
    rc = k.lib().kgr_groth16_setup(shape._h, cs.l, bad.ctypes.data_as(u64p), ctypes.byref(ctypes.c_uint32()), *[ctypes.byref(h) for h in out],
                                   np.zeros(27, dtype=np.uint64).ctypes.data_as(u64p), np.zeros(51, dtype=np.uint64).ctypes.data_as(u64p))
    assert rc == -3 and all(h.value is None for h in out)
    # a context of two engines (on one device): refused as in prove_r1cs
    k.init([0, 0])
    try:
        refused(R1csShape(FIELD_FR, m, n_z, *mats), cs.l, toxic)
    finally:
        k.init()
    # m > 2^28: a shape of 2^28 + 1 empty rows
    _need_gib(24)
    big_m = (1 << 28) + 1
    rp = np.zeros(big_m + 1, dtype=np.uint32)
    empty = (rp, np.zeros(0, dtype=np.uint32), np.zeros((0, 4), dtype=np.uint64))
    big = R1csShape(FIELD_FR, big_m, 1, empty, empty, empty)
    refused(big, 1, toxic)
    big.free()


def test_free_shutdown_and_stale_handles():
    """kgr_bases_free returns the queries' device memory, kgr_shutdown leaves the handles freeable, and handles from before a kgr_init are refused."""
    import torch

    import kogarashi_b200 as k
    from kogarashi_b200.groth16 import Groth16Prover, setup
    k.init()
    cs = G.chain_circuit(21845, 3)[0]
    shape, z = _resident(cs)
    toxic = _k20_toxic()
    setup(shape, cs.l, toxic=toxic).free()            # the engine's cached tables exist from here on
    torch.cuda.synchronize()
    f0 = torch.cuda.mem_get_info()[0]
    params = setup(shape, cs.l, toxic=toxic)
    f1 = torch.cuda.mem_get_info()[0]
    used = f0 - f1
    assert used >= (3 * 65536 * 64 + 65536 * 128)     # a, b_g1, l + h (G1) and b_g2
    params.free()
    f2 = torch.cuda.mem_get_info()[0]
    assert abs(f2 - f0) < used // 4
    params = setup(shape, cs.l, toxic=toxic)
    k.lib().kgr_shutdown()
    params.free()
    f3 = torch.cuda.mem_get_info()[0]
    assert f3 >= f0 - used // 4
    k.init()
    shape, z = _resident(cs)
    old = setup(shape, cs.l, toxic=toxic)
    k.init()
    shape, z = _resident(cs)
    with pytest.raises(k.KgrError, match="kgr error -3"):
        k.msm_curve_addition(old.a, mont(cs.x + cs.w))
    prover = Groth16Prover.from_params(old)
    with pytest.raises(k.KgrError, match="kgr error -3"):
        prover.prove_r1cs(old.log_n, shape, z, cs.l, 1, 2)
    prover.free()
    old.free()
