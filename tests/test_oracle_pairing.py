"""Pins of oracle/pairing_ref.py, the flat big-integer BN254 pairing the device pairing is compared with.  No external pairing vectors exist
offline, so the oracle is pinned by what only a correct reduced pairing satisfies — the tower map is a ring isomorphism, bilinearity in both
arguments, non-degeneracy, values of order r — and by the Groth16 check accepting the restated reference's example proof
(groth16/examples/simple.rs:54-75) and rejecting a wrong public output, swapped A and C, and a proof under another key."""
import random

from test_groth16 import PROVE_SEED, SETUP_SEED

from oracle import groth16_ref as G
from oracle import pairing_ref as E
from oracle import pyref as B

RNG = random.Random(97)
P, R = E.P, E.R


def test_tower_flat_map_is_a_ring_isomorphism():
    for _ in range(4):
        a = [RNG.randrange(P) for _ in range(12)]
        b = [RNG.randrange(P) for _ in range(12)]
        fa, fb = E.tower_to_flat(a), E.tower_to_flat(b)
        assert E.flat_to_tower(fa) == tuple(a)
        assert E.tower_to_flat([(x + y) % P for x, y in zip(a, b)]) == E.f12_add(fa, fb)
        # the product in the tower, written out by hand over Fq2 with v^3 = xi, w^2 = v: (a0 + a1 w)(b0 + b1 w) = a0 b0 + a1 b1 v + (a0 b1 + a1 b0) w
        prod = E.f12_mul(fa, fb)
        a0, a1 = E.tower_to_flat(a[:6] + [0] * 6), E.tower_to_flat([0] * 6 + a[6:])
        b0, b1 = E.tower_to_flat(b[:6] + [0] * 6), E.tower_to_flat([0] * 6 + b[6:])
        assert prod == E.f12_add(E.f12_add(E.f12_mul(a0, b0), E.f12_mul(a0, b1)), E.f12_add(E.f12_mul(a1, b0), E.f12_mul(a1, b1)))
        assert E.f12_mul(fa, E.f12_inv(fa)) == E.ONE


def test_bilinearity():
    a, b = RNG.randrange(1, R), RNG.randrange(1, R)
    p, q = E.G1.mul(E.G1.g, RNG.randrange(1, R)), G.g2_mul(G.G2_GEN, RNG.randrange(1, R))
    e = E.pairing(p, q)
    assert E.pairing(E.G1.mul(p, a), G.g2_mul(q, b)) == E.f12_pow(e, a * b % R)
    q2 = G.g2_mul(G.G2_GEN, RNG.randrange(1, R))
    assert E.pairing(p, G.g2_add(q, q2)) == E.f12_mul(e, E.pairing(p, q2))
    assert E.pairing(E.g1_neg(p), q) == E.f12_inv(e)


def test_non_degenerate_and_of_order_r():
    e = E.pairing(E.G1.g, G.G2_GEN)
    assert e != E.ONE
    assert E.f12_pow(e, R) == E.ONE
    assert E.pairing(None, G.G2_GEN) == E.ONE and E.pairing(E.G1.g, None) == E.ONE


def test_reference_example_proof_verifies():
    Pm, _, _ = G.setup(B.XorShift128(SETUP_SEED))
    proof, internals = G.create_proof(Pm, B.XorShift128(PROVE_SEED), 3, 35)
    vk, pub = Pm["vk"], internals["inputs"][1:]
    assert pub == [3, 35]
    assert E.verify(vk, proof, pub)
    assert not E.verify(vk, proof, [3, 36])                                   # a wrong public output
    assert not E.verify(vk, dict(proof, a=proof["c"], c=proof["a"]), pub)     # A and C swapped
    other, _, _ = G.setup(B.XorShift128(bytes(range(200, 216))))
    assert not E.verify(other["vk"], proof, pub)                              # a proof under another key
