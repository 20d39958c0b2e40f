"""oracle/pairing_ref.py — TEST INFRASTRUCTURE: big-integer BN254 optimal-ate pairing and Groth16 verifier, written independently of the
device's tower (kogarashi_b200/csrc/pairing.cuh).

Fq12 is the flat field Fq[w] / (w^12 - 18 w^6 + 82), with u = w^6 - 9 (so u^2 = -1, the Fq2 of bn254/src/fq2) and xi = 9 + u = w^6.
A twist point (x, y) over Fq2 untwists to (x w^2, y w^3) on y^2 = x^3 + 3.  The Miller loop uses affine lines over the untwisted points
(py_ecc's textbook form); the final exponentiation is plain square-and-multiply by (p^12 - 1) / r.  Nothing here shares a formula, a
constant or a coordinate system with the device code, so agreement limb for limb pins both.

No external pairing known-answer vectors are available offline; this file is pinned by algebraic properties (tests/test_oracle_pairing.py:
bilinearity, non-degeneracy, order r) and by the restated reference's example proof verifying (groth16/src/verifier.rs, proof.rs:39-48).
"""
from . import groth16_ref as G
from . import pyref as B

P = B.FQ
R = B.FR
U = 4965661367192848881                      # the BN parameter: p = 36u^4 + 36u^3 + 24u^2 + 6u + 1
ATE = 6 * U + 2
FINAL_EXP = (P ** 12 - 1) // R
assert 36 * U ** 4 + 36 * U ** 3 + 24 * U ** 2 + 6 * U + 1 == P

# ---- flat Fq12: tuples of 12 ints ------------------------------------------------------------------
def f12(coeffs=None):
    c = [0] * 12
    for i, v in (coeffs or {}).items():
        c[i] = v % P
    return tuple(c)


ONE = f12({0: 1})


def f12_add(a, b):
    return tuple((x + y) % P for x, y in zip(a, b))


def f12_sub(a, b):
    return tuple((x - y) % P for x, y in zip(a, b))


def f12_neg(a):
    return tuple((-x) % P for x in a)


def f12_mul(a, b):
    t = [0] * 23
    for i, x in enumerate(a):
        if x:
            for j, y in enumerate(b):
                t[i + j] += x * y
    for k in range(22, 11, -1):       # w^k = w^(k-12) (18 w^6 - 82)
        c = t[k]
        if c:
            t[k - 6] += 18 * c
            t[k - 12] -= 82 * c
    return tuple(v % P for v in t[:12])


def f12_scale(a, s):
    return tuple(x * s % P for x in a)


def f12_pow(a, e):
    acc = ONE
    for bit in bin(e)[2:]:
        acc = f12_mul(acc, acc)
        if bit == "1":
            acc = f12_mul(acc, a)
    return acc


def _poly_divmod(a, b):
    """Polynomials over Fq as coefficient lists, lowest first; b has a non-zero leading coefficient."""
    a = list(a)
    q = [0] * max(1, len(a) - len(b) + 1)
    inv = pow(b[-1], -1, P)
    for k in range(len(a) - len(b), -1, -1):
        c = a[k + len(b) - 1] * inv % P
        q[k] = c
        if c:
            for j, bj in enumerate(b):
                a[k + j] = (a[k + j] - c * bj) % P
    return q, _trim(a[: len(b) - 1])


def _trim(a):
    a = list(a)
    while len(a) > 1 and a[-1] == 0:
        a.pop()
    return a or [0]


def _poly_mul(a, b):
    t = [0] * (len(a) + len(b) - 1)
    for i, x in enumerate(a):
        for j, y in enumerate(b):
            t[i + j] = (t[i + j] + x * y) % P
    return _trim(t)


def _poly_sub(a, b):
    n = max(len(a), len(b))
    return _trim([((a[i] if i < len(a) else 0) - (b[i] if i < len(b) else 0)) % P for i in range(n)])


def f12_inv(a):
    """Extended Euclid against the modulus w^12 - 18 w^6 + 82."""
    r0, r1 = [82, 0, 0, 0, 0, 0, P - 18, 0, 0, 0, 0, 0, 1], _trim(a)
    s0, s1 = [0], [1]
    while r1 != [0]:
        q, r = _poly_divmod(r0, r1)
        r0, r1 = r1, r
        s0, s1 = s1, _poly_sub(s0, _poly_mul(q, s1))
    assert len(r0) == 1 and r0[0], "not invertible"
    c = pow(r0[0], -1, P)
    s0 = [x * c % P for x in s0] + [0] * 12
    return tuple(s0[:12])


def fq2_to_f12(a, k=0):
    """(a0 + a1 u) w^k in the flat basis: a0 + a1 (w^6 - 9)."""
    c = {}
    c[k] = (a[0] - 9 * a[1])
    c[k + 6] = c.get(k + 6, 0) + a[1]
    return f12(c)


# ---- the device's tower <-> flat: Fq12 = Fq6[w]/(w^2 - v), Fq6 = Fq2[v]/(v^3 - xi), so v = w^2 --------------------------------------
# tower coefficient order c0.c0, c0.c1, c0.c2, c1.c0, c1.c1, c1.c2 (each an Fq2 pair) multiplies w^0, w^2, w^4, w^1, w^3, w^5
_TOWER_POW = (0, 2, 4, 1, 3, 5)


def tower_to_flat(t):
    """t: 12 ints (c0.c0.c0, c0.c0.c1, c0.c1.c0, ..., c1.c2.c1) -> flat Fq12."""
    acc = f12()
    for i, k in enumerate(_TOWER_POW):
        acc = f12_add(acc, fq2_to_f12((t[2 * i], t[2 * i + 1]), k))
    return acc


def flat_to_tower(a):
    """Inverse of tower_to_flat: coefficient of w^k (k < 6) is b0 + b1 w^6 with w^6 = u + 9, i.e. (b0 + 9 b1) + b1 u."""
    out = [0] * 12
    for i, k in enumerate(_TOWER_POW):
        b0, b1 = a[k], a[k + 6]
        out[2 * i], out[2 * i + 1] = (b0 + 9 * b1) % P, b1 % P
    return tuple(out)


# ---- points over Fq12 --------------------------------------------------------------------------------
def untwist(q):
    """Twist point (x, y) over Fq2 -> (x w^2, y w^3) on y^2 = x^3 + 3 over Fq12."""
    if q is None:
        return None
    return fq2_to_f12(q[0], 2), fq2_to_f12(q[1], 3)


def embed_g1(p):
    return None if p is None else (f12({0: p[0]}), f12({0: p[1]}))


def _add12(a, b):
    if a is None:
        return b
    if b is None:
        return a
    if a[0] == b[0]:
        if f12_add(a[1], b[1]) == f12():
            return None
        lam = f12_mul(f12_scale(f12_mul(a[0], a[0]), 3), f12_inv(f12_scale(a[1], 2)))
    else:
        lam = f12_mul(f12_sub(b[1], a[1]), f12_inv(f12_sub(b[0], a[0])))
    x = f12_sub(f12_sub(f12_mul(lam, lam), a[0]), b[0])
    return x, f12_sub(f12_mul(lam, f12_sub(a[0], x)), a[1])


def _line(a, b, t):
    """The line through a and b (tangent if equal) evaluated at t; a vertical line if b = -a."""
    if a[0] != b[0]:
        lam = f12_mul(f12_sub(b[1], a[1]), f12_inv(f12_sub(b[0], a[0])))
    elif a[1] == b[1]:
        lam = f12_mul(f12_scale(f12_mul(a[0], a[0]), 3), f12_inv(f12_scale(a[1], 2)))
    else:
        return f12_sub(t[0], a[0])
    return f12_sub(f12_mul(lam, f12_sub(t[0], a[0])), f12_sub(t[1], a[1]))


def _frob_point(q, k):
    e = P ** k
    return f12_pow(q[0], e), f12_pow(q[1], e)


def miller(p, q):
    """Optimal-ate Miller loop f_{6u+2,Q}(P) l_{[6u+2]Q, pi(Q)}(P) l_{.., -pi^2(Q)}(P), not reduced.  p: G1 affine tuple or None; q: twist
    point over Fq2 or None."""
    if p is None or q is None:
        return ONE
    pt, qt = embed_g1(p), untwist(q)
    r, f = qt, ONE
    for bit in bin(ATE)[3:]:
        f = f12_mul(f12_mul(f, f), _line(r, r, pt))
        r = _add12(r, r)
        if bit == "1":
            f = f12_mul(f, _line(r, qt, pt))
            r = _add12(r, qt)
    q1 = _frob_point(qt, 1)
    q2 = _frob_point(qt, 2)
    nq2 = (q2[0], f12_neg(q2[1]))
    f = f12_mul(f, _line(r, q1, pt))
    r = _add12(r, q1)
    f = f12_mul(f, _line(r, nq2, pt))
    return f


def final_exp(f):
    return f12_pow(f, FINAL_EXP)


def pairing(p, q):
    """Reduced optimal-ate pairing e(P, Q) in the flat basis."""
    return final_exp(miller(p, q))


def pairing_product(pairs):
    f = ONE
    for p, q in pairs:
        f = f12_mul(f, miller(p, q))
    return final_exp(f)


# ---- encodings shared with the device ABI ----------------------------------------------------------------
def gt_to_words(a):
    """flat Fq12 -> (48,) list of uint64 words: 12 Montgomery Fq elements in tower order, 4 little-endian words each."""
    out = []
    for v in flat_to_tower(a):
        m = v * B.R256 % P
        out += [(m >> (64 * k)) & 0xFFFFFFFFFFFFFFFF for k in range(4)]
    return out


def words_to_gt(w):
    r_inv = pow(B.R256, -1, P)
    t = [sum(int(w[4 * i + k]) << (64 * k) for k in range(4)) * r_inv % P for i in range(12)]
    return tower_to_flat(t)


# ---- Groth16 verification (groth16/src/verifier.rs; the check of proof.rs:39-48) --------------------------------------------
G1 = G.G1


def g1_neg(p):
    return None if p is None else (p[0], (-p[1]) % P)


def _g2_mul_raw(q, k):
    """[k]Q without reducing k mod r (g2_mul reduces, which would hide a point outside G2)."""
    acc = None
    while k:
        if k & 1:
            acc = G.g2_add(acc, q)
        q = G.g2_add(q, q)
        k >>= 1
    return acc


def g1_valid(p):
    return p is None or (0 <= p[0] < P and 0 <= p[1] < P and (p[1] * p[1] - p[0] ** 3 - 3) % P == 0)


def g2_valid(q):
    if q is None:
        return True
    if not all(0 <= c < P for c in (*q[0], *q[1])):
        return False
    return G.g2_on_curve(q) and _g2_mul_raw(q, R) is None


def verify(vk, proof, inputs):
    """vk: dict alpha_g1, beta_g2, gamma_g2, delta_g2, ic (list of G1 points, ic[0] for the constant one); proof: dict a, b, c;
    inputs: the public inputs WITHOUT the leading one.  e(A, B) == e(alpha, beta) e(IC(x), gamma) e(C, delta)."""
    if not (g1_valid(proof["a"]) and g2_valid(proof["b"]) and g1_valid(proof["c"])):
        return False
    ic = vk["ic"]
    if len(inputs) + 1 != len(ic):
        raise ValueError("input count does not match the verifying key")
    acc = ic[0]
    for x, pt in zip(inputs, ic[1:]):
        acc = G1.add(acc, G1.mul(pt, x % R)) if pt is not None else acc
    f = pairing_product([(proof["a"], proof["b"]), (g1_neg(vk["alpha_g1"]), vk["beta_g2"]), (g1_neg(acc), vk["gamma_g2"]),
                         (g1_neg(proof["c"]), vk["delta_g2"])])
    return f == ONE
