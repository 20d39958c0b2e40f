"""kgr_pairing on the B200: reduced optimal-ate pairings limb for limb against the flat big-integer pairing of oracle/pairing_ref.py, pairs with an
identity, the product form against the product of single values, bilinearity on device-made points, and the refusal of invalid points."""
import random

import numpy as np
import pytest
from groth16_r1cs_util import mont

from oracle import groth16_ref as G
from oracle import pairing_ref as E
from oracle import pyref as B

pytestmark = pytest.mark.gpu
R = E.R
P = E.P


def fq_words(vals):
    return [w for v in vals for w in B.int_to_limbs(B.to_mont(v % P, P))]


def g1_rows(points):
    return np.array([fq_words([0, 0]) + [1] if p is None else fq_words(p) + [0] for p in points], dtype=np.uint64).reshape(-1, 9)


def g2_rows(points):
    return np.array([fq_words([0] * 4) + [1] if q is None else fq_words([*q[0], *q[1]]) + [0] for q in points], dtype=np.uint64).reshape(-1, 17)


def device_points(curve, scalars):
    from kogarashi_b200.msm import fixed_base_mul
    xy = fixed_base_mul(curve, mont(scalars))
    return np.concatenate([xy, np.zeros((xy.shape[0], 1), dtype=np.uint64)], axis=1)


@pytest.fixture(scope="module")
def k():
    import kogarashi_b200 as kk
    kk.init()
    return kk


def test_pairings_match_the_oracle(k):
    rng = random.Random(1)
    a = [rng.randrange(1, R) for _ in range(16)]
    b = [rng.randrange(1, R) for _ in range(16)]
    got = k.pairing(device_points(k.BN254_G1, a), device_points(k.BN254_G2, b))
    base = E.pairing(E.G1.g, G.G2_GEN)
    for i in range(16):
        assert [int(w) for w in got[i]] == E.gt_to_words(E.f12_pow(base, a[i] * b[i] % R)), i
    # two pairs evaluated by the oracle's own Miller loop, not through bilinearity
    p, q = E.G1.mul(E.G1.g, a[0]), G.g2_mul(G.G2_GEN, b[0])
    p2, q2 = E.G1.mul(E.G1.g, a[1]), G.g2_mul(G.G2_GEN, 3)
    got2 = k.pairing(g1_rows([p, p2]), g2_rows([q, q2]))
    assert [int(w) for w in got2[0]] == E.gt_to_words(E.pairing(p, q))
    assert [int(w) for w in got2[1]] == E.gt_to_words(E.pairing(p2, q2))


def test_identity_pairs_give_one(k):
    one = E.gt_to_words(E.ONE)
    p, q = E.G1.mul(E.G1.g, 5), G.g2_mul(G.G2_GEN, 7)
    got = k.pairing(g1_rows([None, p, None]), g2_rows([q, None, None]))
    for row in got:
        assert [int(w) for w in row] == one
    # the flag wins over the coordinates
    rows1 = g1_rows([p])
    rows1[0, 8] = 1
    assert [int(w) for w in k.pairing(rows1, g2_rows([q]))[0]] == one
    assert [int(w) for w in k.pairing_product(np.zeros((0, 9), np.uint64), np.zeros((0, 17), np.uint64))] == one


def test_product_equals_product_of_values(k):
    rng = random.Random(2)
    n = 37
    a = [rng.randrange(1, R) for _ in range(n)]
    b = [rng.randrange(1, R) for _ in range(n)]
    g1, g2 = device_points(k.BN254_G1, a), device_points(k.BN254_G2, b)
    g1[5, 8] = 1                        # one identity pair inside the product
    each = k.pairing(g1, g2)
    acc = E.ONE
    for row in each:
        acc = E.f12_mul(acc, E.words_to_gt(row))
    assert [int(w) for w in k.pairing_product(g1, g2)] == E.gt_to_words(acc)


def test_bilinearity_on_device_points(k):
    rng = random.Random(3)
    n = 256
    a = [rng.randrange(1, R) for _ in range(n)]
    b = [rng.randrange(1, R) for _ in range(n)]
    lhs = k.pairing(device_points(k.BN254_G1, a), device_points(k.BN254_G2, b))
    rhs = k.pairing(device_points(k.BN254_G1, [1] * n), device_points(k.BN254_G2, [x * y % R for x, y in zip(a, b)]))
    assert (lhs == rhs).all()
    assert len({tuple(r) for r in lhs.tolist()}) == n
    # e(P, Q)^r = 1 is e(P, [r] Q) = e(P, O); e(-P, Q) e(P, Q) = 1
    g1 = device_points(k.BN254_G1, [a[0], R - a[0]])
    g2 = device_points(k.BN254_G2, [b[0], b[0]])
    assert [int(w) for w in k.pairing_product(g1, g2)] == E.gt_to_words(E.ONE)


def _f2_pow(a, e):
    acc = (1, 0)
    for bit in bin(e)[2:]:
        acc = G.f2_mul(acc, acc)
        if bit == "1":
            acc = G.f2_mul(acc, a)
    return acc


def f2_sqrt(a):
    """Square root in Fq2 (p = 3 mod 4), or None."""
    a1 = _f2_pow(a, (P - 3) // 4)
    alpha = G.f2_mul(G.f2_mul(a1, a1), a)
    x0 = G.f2_mul(a1, a)
    if alpha == (P - 1, 0):
        y = G.f2_mul((0, 1), x0)
    else:
        y = G.f2_mul(_f2_pow(G.f2_add((1, 0), alpha), (P - 1) // 2), x0)
    return y if G.f2_mul(y, y) == a else None


def twist_point_outside_g2(seed):
    rng = random.Random(seed)
    while True:
        x = (rng.randrange(P), rng.randrange(P))
        y = f2_sqrt(G.f2_add(G.f2_mul(G.f2_mul(x, x), x), G.G2_B))
        if y is not None:
            assert G.g2_on_curve((x, y)) and E._g2_mul_raw((x, y), R) is not None
            return (x, y)


def test_invalid_points_are_refused(k):
    from kogarashi_b200 import KgrError
    p, q = E.G1.mul(E.G1.g, 11), G.g2_mul(G.G2_GEN, 13)
    for g1, g2 in ((g1_rows([(p[0], p[1] + 1)]), g2_rows([q])),            # off the curve
                   (g1_rows([p]), g2_rows([twist_point_outside_g2(4)])),    # on the twist, outside G2
                   (g1_rows([p]), g2_rows([((q[0][0] + 1, q[0][1]), q[1])]))):  # off the twist
        for fn in (k.pairing, k.pairing_product):
            with pytest.raises(KgrError, match="error -3"):
                fn(np.concatenate([g1_rows([p]), g1]), np.concatenate([g2_rows([q]), g2]))
    # a coordinate >= p (x + p as a 256-bit integer is the same residue)
    bad = g1_rows([p])
    x = B.limbs_to_int(bad[0, :4].tolist()) + P
    bad[0, :4] = B.int_to_limbs(x)
    with pytest.raises(KgrError, match="error -3"):
        k.pairing(bad, g2_rows([q]))
