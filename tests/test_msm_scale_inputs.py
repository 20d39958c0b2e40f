"""Inputs with known discrete logarithms for the large-input MSM tests (test_gpu_msm_scale.py), and the CPU check that ties their
cheap reference to the oracle's MSM.

Every base is drawn from a pool of points k_j * G whose k_j are known (plus their negations and exact duplicates, so that equal and opposite
points share buckets at every size), about 1/64 of the bases are identities.  Then sum_i s_i * P_i = (sum_i s_i k_i) * G: one threaded field
dot product and one scalar multiplication give the exact group element of an MSM of any size, and any wrong bucket changes it."""
import functools

import numpy as np
import pytest
from conftest import same_affine

from oracle import oracle as A
from oracle import pyref as B

POOL = 4096
MIXES = ("nova", "one_bucket", "rm1", "small", "uniform", "canonical_unreduced")
CURVES = (A.BN254_G1, A.GRUMPKIN, A.BN254_G2)
SCALARS_MONTGOMERY, SCALARS_CANONICAL = 0, 1   # scalar formats of the C ABI (include/kgr_msm.h)


def scalar_modulus(curve):
    return B.FR if A.SCALAR_FIELD[curve] == A.FIELD_FR else B.FQ


def _base_field(curve):
    return A.BASE_FIELD.get(curve, A.FIELD_FQ)  # G2 coordinates are pairs of Fq elements


def _mont(vals, p):
    return np.array([B.int_to_limbs(B.to_mont(int(v) % p, p)) for v in vals], dtype=np.uint64).reshape(-1, 4)


@functools.lru_cache(maxsize=None)
def pool(curve):
    """(points, k): POOL points k_j * G, their negations (-k_j) * G, and exact copies of the first POOL / 8.  Shared: index, do not modify."""
    pts, ks = A.random_points(curve, POOL, seed=bytes(range(70, 86)), return_scalars=True)
    cl, bf, fid = A.coord_limbs(curve), _base_field(curve), A.SCALAR_FIELD[curve]
    neg = pts.copy()
    for i in range(POOL):
        for h in range(cl, 2 * cl, 4):
            neg[i, h:h + 4] = A.field_op(bf, "neg", pts[i, h:h + 4])
    neg_ks = np.stack([A.field_op(fid, "neg", k) for k in ks])
    dup = slice(0, POOL // 8)
    return np.concatenate([pts, neg, pts[dup]]), np.concatenate([ks, neg_ks, ks[dup]])


def make_bases(curve, n, seed):
    """(points, inf, k) for n bases drawn from the curve's pool; about 1/64 are identities (flag set, coordinates zero, k = 0)."""
    pool_pts, pool_ks = pool(curve)
    rng = np.random.default_rng(seed)
    idx = rng.integers(0, pool_pts.shape[0], n)
    pts, ks = pool_pts[idx], pool_ks[idx]
    inf = (rng.integers(0, 64, n) == 0).astype(np.uint8)
    pts[inf == 1] = 0
    ks[inf == 1] = 0
    return pts, inf, ks


def make_scalars(curve, mix, n, seed):
    """(scalars as passed to the MSM, their format, the same values as reduced Montgomery limbs) for one of MIXES:
      nova                 half 0, a quarter 1, the rest uniform (Nova's witnesses and cross terms)
      one_bucket           every scalar equal: each window has one bucket that holds every point
      rm1                  7 / 8 of them r - 1: signed-digit carries run through the top window
      small                values below 2^16: only the low windows hold any point
      uniform              uniform in [0, r)
      canonical_unreduced  canonical-format values >= r (and r itself), read modulo r"""
    fid, p = A.SCALAR_FIELD[curve], scalar_modulus(curve)
    rng = np.random.default_rng(seed)
    one = A.field_op(fid, "to_mont", np.array([1, 0, 0, 0], dtype=np.uint64))
    fseed = bytes(rng.integers(0, 256, 16, dtype=np.uint8))
    if mix == "uniform":
        sc = A.random_field(fid, n, seed=fseed)
    elif mix == "nova":
        sc = A.random_field(fid, n, seed=fseed)
        kind = rng.integers(0, 4, n)
        sc[kind < 2] = 0
        sc[kind == 2] = one
    elif mix == "one_bucket":
        sc = np.tile(A.random_field(fid, 1, seed=fseed), (n, 1))
    elif mix == "rm1":
        sc = A.random_field(fid, n, seed=fseed)
        sc[rng.integers(0, 8, n) != 0] = A.field_op(fid, "neg", one)
    elif mix == "small":
        vals = np.concatenate([[0, 1, 0xFFFF], rng.integers(0, 1 << 16, POOL - 3)])
        sc = _mont(vals, p)[rng.integers(0, POOL, n)]
    elif mix == "canonical_unreduced":
        top = p >> 192
        raw = rng.integers(0, 1 << 63, (POOL, 4), dtype=np.uint64) * np.uint64(2) + rng.integers(0, 2, (POOL, 4), dtype=np.uint64)
        raw[:, 3] = np.maximum(raw[:, 3], np.uint64(top + 1))          # top limb above r's: every value > r
        raw[0] = np.uint64(0xFFFFFFFFFFFFFFFF)                          # 2^256 - 1
        raw[1] = B.int_to_limbs(p)                                      # r itself reads as 0
        raw[2] = B.int_to_limbs(p + 1)
        red = _mont([B.limbs_to_int(x) for x in raw], p)
        idx = rng.integers(0, POOL, n)
        return raw[idx], SCALARS_CANONICAL, red[idx]
    else:
        raise ValueError(mix)
    return sc, SCALARS_MONTGOMERY, sc


def generator_proj(curve):
    one = A.field_op(_base_field(curve), "to_mont", np.array([1, 0, 0, 0], dtype=np.uint64))
    z = np.concatenate([one, np.zeros(4, dtype=np.uint64)]) if curve == A.BN254_G2 else one
    return np.concatenate([A.generator(curve), z])


def checksum(curve, ks, sc_mont):
    """(sum_i k_i s_i) * G, affine: the MSM of bases k_i * G with scalars s_i (Montgomery in, field_dot is exact)."""
    s = A.field_dot(A.SCALAR_FIELD[curve], ks, sc_mont)
    return A.to_affine(curve, A.scalar_point(curve, generator_proj(curve), s))


@pytest.mark.parametrize("curve", CURVES)
def test_pool_points_are_multiples_of_the_generator(curve):
    """Originals, negations and duplicates of the pool, and the bases drawn from it, are k * G for the k they carry."""
    pts, ks = pool(curve)
    assert pts.shape[0] == 2 * POOL + POOL // 8
    sample = np.r_[0:8, POOL:POOL + 8, 2 * POOL:2 * POOL + 8, POOL - 1, 2 * POOL - 1, pts.shape[0] - 1]
    assert (A.fixed_base(curve, ks[sample]) == pts[sample]).all()
    bpts, inf, bks = make_bases(curve, 4096, seed=1)
    assert 0 < int(inf.sum()) < 4096 // 16
    assert not bpts[inf == 1].any() and not bks[inf == 1].any()
    assert (A.fixed_base(curve, bks[:256]) == bpts[:256]).all()          # identities: k = 0 gives the (0, 0) encoding


@pytest.mark.parametrize("mix", MIXES)
@pytest.mark.parametrize("curve", CURVES)
def test_checksum_matches_oracle_msm(curve, mix):
    """At 2^12 points the O(n) reference equals the oracle's MSM for every scalar mix, with repeated, opposite and identity bases."""
    n = 1 << 12
    pts, inf, ks = make_bases(curve, n, seed=2)
    sc, fmt, sc_mont = make_scalars(curve, mix, n, seed=3)
    exp = checksum(curve, ks, sc_mont)
    assert same_affine(exp, A.to_affine(curve, A.msm(curve, pts, sc_mont, inf=inf)))
    assert not exp[-1]                                                    # not the identity: a wrong bucket cannot hide behind zero
    p = scalar_modulus(curve)
    vals = [B.limbs_to_int(x) % p if fmt else B.from_mont(B.limbs_to_int(x), p) for x in sc]
    assert vals == [B.from_mont(B.limbs_to_int(x), p) for x in sc_mont]
    if mix == "nova":
        assert 0.4 < np.mean([v == 0 for v in vals]) < 0.6 and 0.2 < np.mean([v == 1 for v in vals]) < 0.3
    elif mix == "one_bucket":
        assert len(set(vals)) == 1
    elif mix == "rm1":
        assert np.mean([v == p - 1 for v in vals]) > 0.8
    elif mix == "small":
        assert max(vals) < 1 << 16
    elif mix == "canonical_unreduced":
        assert all(B.limbs_to_int(x) >= p for x in sc)
