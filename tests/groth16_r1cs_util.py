"""Helpers for the Groth16-from-R1CS tests: the constraint systems of oracle/groth16_ref.py as CSR over z = x ++ w, the layout
kgr_r1cs_register takes (Wire::Instance(i) -> i, Wire::Witness(i) -> l + i, zkstd/src/matrix.rs:41-44)."""
import numpy as np

from oracle import groth16_ref as G
from oracle import pyref as B


def mont(vals):
    cache, out = {}, np.zeros((len(vals), 4), dtype=np.uint64)
    for i, v in enumerate(vals):
        v %= G.R
        if v not in cache:
            cache[v] = B.int_to_limbs(B.to_mont(v, B.FR))
        out[i] = cache[v]
    return out


def csr_from_r1cs(cs, split_rows=()):
    """-> m, n_z, (A, B, C) with each matrix (row_ptr, cols, coeffs Montgomery).  In the rows of `split_rows` (indices into every matrix) the
    first term is stored as two entries of the same column whose coefficients add up to it: a duplicated column."""
    l = cs.l

    def mat(rows):
        row_ptr, cols, co = [0], [], []
        for i, row in enumerate(rows):
            for t, ((kind, w), v) in enumerate(row.items()):
                col = w if kind == "x" else l + w
                if t == 0 and i in split_rows:
                    cols += [col, col]
                    co += [12345, v - 12345]
                elif v % G.R:
                    cols.append(col)
                    co.append(v)
            row_ptr.append(len(cols))
        return np.array(row_ptr, dtype=np.uint32), np.array(cols, dtype=np.uint32), mont(co)

    return cs.m, cs.l + cs.m_l_1, tuple(mat(rows) for rows in (cs.a, cs.b, cs.c))


def edge_circuit():
    """A chain of 100 steps (m = 301) plus rows the chain lacks: an empty row, a row of 300 terms with coefficients 1 and r - 1 among random
    ones, and a row with coefficient r - 1 on the constant.  -> (cs, rows to store with a duplicated column)."""
    cs, _ = G.chain_circuit(100, 3)
    rng = B.XorShift128(bytes(range(40, 56)))
    cs.a.append({}), cs.b.append({("x", 0): 1}), cs.c.append({})
    long_row = {("w", i): (1 if i % 3 == 0 else G.R - 1 if i % 3 == 1 else rng.random_field(G.R)) for i in range(300)}
    cs.a.append(long_row), cs.b.append({("x", 0): 1}), cs.c.append(dict(long_row))
    cs.a.append({("x", 0): G.R - 1, ("w", 7): 1}), cs.b.append({("x", 1): G.R - 1}), cs.c.append({("w", 2): 3})
    return cs, (0, 5, cs.m - 2, cs.m - 1)


def bitrev(i, k):
    return int(format(i, f"0{k}b")[::-1], 2)


def evaluations_bitrev(cs, k):
    """cs.evaluate() zero padded to 2^k and permuted by bit reversal: what the evaluation kernel leaves in the three NTT buffers."""
    n = 1 << k
    perm = np.array([bitrev(i, k) for i in range(n)])
    bufs = []
    for ev in cs.evaluate():
        padded = np.zeros((n, 4), dtype=np.uint64)
        padded[: len(ev)] = mont(ev)
        buf = np.zeros_like(padded)
        buf[perm] = padded
        bufs.append(buf)
    return bufs
