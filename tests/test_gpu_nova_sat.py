"""kgr_nova_is_sat / R1csShape.is_sat(_relaxed) on the GPU: R1csShape::is_sat and the relaxed check (nova/src/relaxed_r1cs.rs:80-146) on resident
vectors, both curves.  Expected commitments come from the oracle's Pedersen commitment of the downloaded vectors, never from the code under
test; expected violation counts and first rows from host evaluations of the CSR."""
import ctypes

import numpy as np
import pytest
from nova_util import chain_r1cs, example_r1cs, example_z, ints, mont

from oracle import oracle as A
from oracle import pyref as B

pytestmark = pytest.mark.gpu
CURVES = [A.GRUMPKIN, A.BN254_G1]
W_OFF = 3            # z = (u, x0, out | w) for the chain and (1, input, out | w) for the example
KGR_E_ARG = -3


@pytest.fixture(scope="module")
def k():
    import kogarashi_b200 as kk
    kk.init()
    return kk


def _field(curve):
    fid = A.SCALAR_FIELD[curve]
    return fid, (B.FQ if fid == A.FIELD_FQ else B.FR)


def _key(k, curve, n, seed=7):
    pts = A.random_points(curve, n, seed=bytes(range(seed, seed + 16)))
    return k.PedersenCommitment(curve, pts), pts


def _commit(curve, pts, v):
    """The oracle's PedersenCommitment::commit of a downloaded vector, zipped with the key (pedersen.rs:16-17)."""
    v = np.asarray(v, dtype=np.uint64).reshape(-1, 4)
    n = min(len(v), len(pts))
    return A.pedersen_commit(curve, pts[:n], v[:n])


def _circuit(name, p, x):
    if name == "example":
        m, n_z, mats = example_r1cs(p)
        return m, n_z, mats, example_z(x, p)
    return chain_r1cs(700, x, p)


def _host_check(fid, p, m, mats, z, e):
    """(count, first) of rows violating (A z) o (B z) = u (C z) + E, u = z[0], from the oracle's sparse products."""
    az, bz, cz = (ints(A.sparse_prod(fid, m, mat, z), p) for mat in mats)
    u = ints(z[:1], p)[0]
    ev = ints(e, p)
    bad = [i for i in range(m) if (az[i] * bz[i] - u * cz[i] - ev[i]) % p]
    return len(bad), (bad[0] if bad else m)


def _fold_step(nova, shape, d_z1, d_z2, d_e, d_t, r):
    nova.cross_term_device(shape, d_z1, d_z2, t=d_t)
    d_z1.fold(d_z2, r)
    d_e.fold(d_t, r)


@pytest.mark.parametrize("circuit", ["example", "chain700"])
@pytest.mark.parametrize("curve", CURVES)
def test_satisfied_instances(k, curve, circuit):
    """A strict instance, then the relaxed instances after one and after two device folds: satisfied, both commitments equal."""
    from kogarashi_b200 import nova
    fid, p = _field(curve)
    m, n_z, mats, z1 = _circuit(circuit, p, 3)
    shape = nova.R1csShape(fid, m, n_z, *mats)
    ck, pts = _key(k, curve, max(m, n_z))
    d_z1 = nova.DeviceVec(fid, mont(z1, p))
    rep = shape.is_sat(d_z1, W_OFF, ck=ck, commit_w=_commit(curve, pts, mont(z1, p)[W_OFF:]))
    assert rep and rep == (True, 0, m, True, None, True)
    assert shape.is_sat(d_z1, W_OFF) == (True, 0, m, None, None, True)
    d_z2 = nova.DeviceVec(fid, mont(_circuit(circuit, p, 4)[3], p))
    d_e, d_t = nova.DeviceVec(fid, n=m), nova.DeviceVec(fid, n=m)
    r = mont([0x0F1E2D3C4B5A69788796A5B4C3D2E1F0 % p], p)[0]
    for step in range(2):
        if step:
            d_z2.write(0, mont(_circuit(circuit, p, 9)[3], p))
        _fold_step(nova, shape, d_z1, d_z2, d_e, d_t, r)
        z, e = d_z1.download(), d_e.download()
        assert ints(z[:1], p)[0] != 1 and e.any()
        rep = shape.is_sat_relaxed(d_z1, d_e, W_OFF, ck=ck, commit_w=_commit(curve, pts, z[W_OFF:]), commit_e=_commit(curve, pts, e))
        assert rep == (True, 0, m, True, True, True), (step, rep)
        assert shape.is_sat_relaxed(d_z1, d_e, W_OFF) == (True, 0, m, None, None, True)
        # the strict check of a relaxed instance fails on u (and on every row where E or u matters)
        assert not shape.is_sat(d_z1, W_OFF).u_ok
    for v in (d_z1, d_z2, d_e, d_t):
        v.free()
    shape.free()


@pytest.mark.parametrize("curve", CURVES)
def test_tampering(k, curve):
    from kogarashi_b200 import nova
    fid, p = _field(curve)
    m, n_z, mats, z1 = chain_r1cs(700, 3, p)
    shape = nova.R1csShape(fid, m, n_z, *mats)
    ck, pts = _key(k, curve, max(m, n_z), seed=21)
    d_z, d_z2 = nova.DeviceVec(fid, mont(z1, p)), nova.DeviceVec(fid, mont(chain_r1cs(700, 5, p)[3], p))
    d_e, d_t = nova.DeviceVec(fid, n=m), nova.DeviceVec(fid, n=m)
    _fold_step(nova, shape, d_z, d_z2, d_e, d_t, mont([0xABCDEF0123456789 % p], p)[0])
    z, e = d_z.download(), d_e.download()
    cw, ce = _commit(curve, pts, z[W_OFF:]), _commit(curve, pts, e)
    assert shape.is_sat_relaxed(d_z, d_e, W_OFF, ck=ck, commit_w=cw, commit_e=ce)
    # one E entry changed: exactly that row
    for row in (0, 1234, m - 1):
        d_e.write(row, mont([ints(e[row:row + 1], p)[0] + 1], p))
        rep = shape.is_sat_relaxed(d_z, d_e, W_OFF)
        assert rep == (False, 1, row, None, None, True), (row, rep)
        d_e.write(row, e[row:row + 1])
    # one witness entry changed: the rows that reference that column, from the CSR on the host
    for col in (W_OFF, 1000, n_z - 1):
        refs = sorted({i for (row_ptr, cols, _) in mats for i in range(m) if col in cols[row_ptr[i]:row_ptr[i + 1]]})
        zb = z.copy()
        zb[col] = mont([ints(z[col:col + 1], p)[0] + 5], p)[0]
        d_z.write(col, zb[col:col + 1])
        rep = shape.is_sat_relaxed(d_z, d_e, W_OFF, ck=ck, commit_w=cw)
        assert (rep.violations, rep.first_violation) == (len(refs), refs[0]) == _host_check(fid, p, m, mats, zb, e), col
        assert not rep and rep.commit_w is False
        d_z.write(col, z[col:col + 1])
    # u changed
    zb = z.copy()
    zb[0] = mont([ints(z[:1], p)[0] + 1], p)[0]
    d_z.write(0, zb[:1])
    rep = shape.is_sat_relaxed(d_z, d_e, W_OFF)
    assert not rep and (rep.violations, rep.first_violation) == _host_check(fid, p, m, mats, zb, e) and rep.violations > 0
    d_z.write(0, z[:1])
    # a commitment of another vector: status 0 while the relation still holds
    rep = shape.is_sat_relaxed(d_z, d_e, W_OFF, ck=ck, commit_w=ce, commit_e=ce)
    assert rep == (False, 0, m, False, True, True)
    rep = shape.is_sat_relaxed(d_z, d_e, W_OFF, ck=ck, commit_w=cw, commit_e=cw)
    assert rep == (False, 0, m, True, False, True)
    assert shape.is_sat_relaxed(d_z, d_e, W_OFF, ck=ck, commit_w=cw, commit_e=ce)
    # strict mode with z[0] != 1: u reported, and the rows judged with u = 1
    d_s = nova.DeviceVec(fid, mont(z1, p))
    assert shape.is_sat(d_s, W_OFF, ck=ck, commit_w=_commit(curve, pts, mont(z1, p)[W_OFF:]))
    d_s.write(0, mont([2], p))
    rep = shape.is_sat(d_s, W_OFF)
    assert not rep and not rep.u_ok and rep.commit_w is None and rep.violations > 0
    for v in (d_z, d_z2, d_e, d_t, d_s):
        v.free()
    shape.free()


@pytest.mark.parametrize("curve", CURVES)
def test_identity_commitment(k, curve):
    """E all zero commits to the identity: equal to an identity (0, R, 1), different from a non-identity; W = z[n_z ..] is empty."""
    from kogarashi_b200 import nova
    fid, p = _field(curve)
    base_p = B.FR if fid == A.FIELD_FQ else B.FQ
    m, n_z, mats, z = chain_r1cs(50, 3, p)
    shape = nova.R1csShape(fid, m, n_z, *mats)
    ck, pts = _key(k, curve, max(m, n_z), seed=33)
    ident = np.concatenate([np.zeros(4, dtype=np.uint64), mont([1], base_p)[0], np.ones(1, dtype=np.uint64)])
    assert A.pedersen_commit(curve, pts[:m], np.zeros((m, 4), dtype=np.uint64))[8] == 1
    d_z, d_e = nova.DeviceVec(fid, mont(z, p)), nova.DeviceVec(fid, n=m)
    cw = _commit(curve, pts, mont(z, p)[W_OFF:])
    assert cw[8] == 0
    assert shape.is_sat_relaxed(d_z, d_e, W_OFF, ck=ck, commit_w=cw, commit_e=ident) == (True, 0, m, True, True, True)
    assert shape.is_sat_relaxed(d_z, d_e, W_OFF, ck=ck, commit_e=cw).commit_e is False
    assert shape.is_sat_relaxed(d_z, d_e, W_OFF, ck=ck, commit_w=ident).commit_w is False
    assert shape.is_sat(d_z, n_z, ck=ck, commit_w=ident).commit_w is True
    assert shape.is_sat(d_z, n_z, ck=ck, commit_w=cw).commit_w is False
    for v in (d_z, d_e):
        v.free()
    shape.free()


@pytest.mark.parametrize("curve", CURVES)
def test_grid_wide_reduction(k, curve):
    """2^16 + 3 rows (513 blocks of 128): violations only in the last block, scattered over many blocks, and in every row."""
    from kogarashi_b200 import nova
    fid, p = _field(curve)
    m, n_z, mats, z = chain_r1cs(21846, 3, p)
    assert m >= 1 << 16 and m % 128 != 0
    shape = nova.R1csShape(fid, m, n_z, *mats)
    d_z = nova.DeviceVec(fid, mont(z, p))
    last_block = (m - 1) // 128 * 128
    rng = np.random.default_rng(5)
    cases = [[m - 1], [last_block, m - 2, m - 1], sorted(rng.choice(m, size=700, replace=False).tolist()),
             sorted(rng.choice(np.arange(128, m, 128), size=300, replace=False).tolist()), list(range(m))]
    one = mont([1], p)[0]
    for rows in cases:
        e = np.zeros((m, 4), dtype=np.uint64)
        e[rows] = one
        d_e = nova.DeviceVec(fid, e)
        rep = shape.is_sat_relaxed(d_z, d_e, W_OFF)
        assert rep == (False, len(rows), rows[0], None, None, True), (len(rows), rep)
        d_e.free()
    d_e = nova.DeviceVec(fid, n=m)
    assert shape.is_sat_relaxed(d_z, d_e, W_OFF) == (True, 0, m, None, None, True)
    d_e.free()
    d_z.free()
    shape.free()


@pytest.mark.parametrize("curve", CURVES)
def test_sees_the_fold_just_enqueued(k, curve):
    """is_sat_relaxed right after a fold on the same vectors judges the folded values: z folded alone breaks the relation, E folded too
    restores it, and the commitments of the folded vectors match."""
    from kogarashi_b200 import nova
    fid, p = _field(curve)
    m, n_z, mats, z1 = chain_r1cs(700, 3, p)
    z2 = chain_r1cs(700, 8, p)[3]
    shape = nova.R1csShape(fid, m, n_z, *mats)
    ck, pts = _key(k, curve, max(m, n_z), seed=40)
    d_z1, d_z2 = nova.DeviceVec(fid, mont(z1, p)), nova.DeviceVec(fid, mont(z2, p))
    d_e, d_t = nova.DeviceVec(fid, n=m), nova.DeviceVec(fid, n=m)
    rm = mont([0x77665544332211 % p], p)[0]
    nova.cross_term_device(shape, d_z1, d_z2, t=d_t)
    t = d_t.download()
    zf = A.vec_fold(fid, mont(z1, p), mont(z2, p), rm)
    ef = A.vec_fold(fid, np.zeros_like(t), t, rm)
    d_z1.fold(d_z2, rm)
    rep = shape.is_sat_relaxed(d_z1, d_e, W_OFF, ck=ck, commit_w=_commit(curve, pts, zf[W_OFF:]))
    assert not rep and rep.violations > 0 and rep.commit_w is True
    d_e.fold(d_t, rm)
    assert shape.is_sat_relaxed(d_z1, d_e, W_OFF, ck=ck, commit_w=_commit(curve, pts, zf[W_OFF:]), commit_e=_commit(curve, pts, ef))
    for v in (d_z1, d_z2, d_e, d_t):
        v.free()
    shape.free()


def _rc(k, shape, z, e, w_off, ck, cw, ce, report=None):
    """Raw kgr_nova_is_sat: (return code, report).  A refused call must leave the report untouched."""
    u64p = ctypes.POINTER(ctypes.c_uint64)
    rep = np.full(6, 7, dtype=np.uint64) if report is None else report
    h = lambda x: getattr(getattr(x, "g", x), "_h", None) if x is not None else None
    arr = lambda a: np.ascontiguousarray(a, dtype=np.uint64).ctypes.data_as(u64p) if a is not None else None
    keep = [np.ascontiguousarray(a, dtype=np.uint64) if a is not None else None for a in (cw, ce)]
    rc = k.lib().kgr_nova_is_sat(h(shape), h(z), h(e), w_off, h(ck), arr(keep[0]), arr(keep[1]),
                                 rep.ctypes.data_as(u64p) if report is not False else None)
    return rc, rep


def test_refusals(k):
    from kogarashi_b200 import nova
    curve = A.BN254_G1
    fid, p = _field(curve)
    m, n_z, mats, z = chain_r1cs(20, 3, p)
    shape = nova.R1csShape(fid, m, n_z, *mats)
    ck, pts = _key(k, curve, max(m, n_z), seed=50)
    d_z, d_e = nova.DeviceVec(fid, mont(z, p)), nova.DeviceVec(fid, n=m)
    cw = _commit(curve, pts, mont(z, p)[W_OFF:])
    ok_rc, rep = _rc(k, shape, d_z, d_e, W_OFF, ck, cw, cw)
    assert ok_rc == 0 and list(rep) == [0, 0, m, 1, 0, 1]
    other_f = nova.DeviceVec(1 - fid, n=n_z)
    grumpkin_ck = k.PedersenCommitment(A.GRUMPKIN, A.random_points(A.GRUMPKIN, 8))
    g2_ck = k.Bases(A.BN254_G2, A.random_points(A.BN254_G2, 8))
    short_z, short_e = nova.DeviceVec(fid, n=n_z - 1), nova.DeviceVec(fid, n=m - 1)
    refused = {
        "null shape": (None, d_z, d_e, W_OFF, None, None, None),
        "null z": (shape, None, d_e, W_OFF, None, None, None),
        "z of the other field": (shape, other_f, d_e, W_OFF, None, None, None),
        "e of the other field": (shape, d_z, nova.DeviceVec(1 - fid, n=m), W_OFF, None, None, None),
        "key of the other scalar field": (shape, d_z, d_e, W_OFF, grumpkin_ck, cw, None),
        "G2 key": (shape, d_z, d_e, W_OFF, g2_ck, None, None),
        "short z": (shape, short_z, d_e, W_OFF, None, None, None),
        "short e": (shape, d_z, short_e, W_OFF, None, None, None),
        "w_off 0": (shape, d_z, d_e, 0, None, None, None),
        "w_off past n_z": (shape, d_z, d_e, n_z + 1, None, None, None),
        "commit_w without key": (shape, d_z, d_e, W_OFF, None, cw, None),
        "commit_e without key": (shape, d_z, d_e, W_OFF, None, None, cw),
        "commit_e in strict mode": (shape, d_z, None, W_OFF, ck, cw, cw),
    }
    for what, args in refused.items():
        rc, rep = _rc(k, *args)
        assert rc == KGR_E_ARG and (rep == 7).all(), what
    assert _rc(k, shape, d_z, d_e, W_OFF, None, None, None, report=False)[0] == KGR_E_ARG
    assert _rc(k, shape, d_z, None, n_z, ck, cw, None)[0] == 0          # w_off = n_z: an empty W is allowed
    with pytest.raises(k.KgrError):
        shape.is_sat_relaxed(d_z, d_e, W_OFF, commit_e=cw)
    # a key split over two engines (two shards)
    k.init([0, 0])
    try:
        shape2 = nova.R1csShape(fid, m, n_z, *mats)
        z2 = nova.DeviceVec(fid, mont(z, p))
        split = k.PedersenCommitment(curve, pts)                       # registered as two shards, one per engine
        assert _rc(k, shape2, z2, None, W_OFF, split, cw, None)[0] == KGR_E_ARG
        assert _rc(k, shape2, z2, None, W_OFF, None, None, None)[0] == 0
    finally:
        k.init()
    # everything from before the last kgr_init is stale
    shape3 = nova.R1csShape(fid, m, n_z, *mats)
    z3, e3 = nova.DeviceVec(fid, mont(z, p)), nova.DeviceVec(fid, n=m)
    ck3 = k.PedersenCommitment(curve, pts)
    assert _rc(k, shape3, z3, e3, W_OFF, ck3, cw, None)[0] == 0
    for what, args in {"stale shape": (shape, z3, e3, W_OFF, None, None, None), "stale z": (shape3, d_z, e3, W_OFF, None, None, None),
                       "stale e": (shape3, z3, d_e, W_OFF, None, None, None), "stale key": (shape3, z3, e3, W_OFF, ck, cw, None)}.items():
        rc, rep = _rc(k, *args)
        assert rc == KGR_E_ARG and (rep == 7).all(), what
    for v in (z3, e3):
        v.free()
    shape3.free()
