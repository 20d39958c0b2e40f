"""Mirror of the vector work of nova's folding prover over the C ABI (SURVEY.md §8f row N4).

Reference:
  zkstd/src/matrix.rs:36-48                 SparseMatrix::prod(m, l, z)        row i: sum of coeff * z[wire]
  nova/src/prover.rs:53-90                  Prover::compute_cross_term          T = AZ1∘BZ2 + AZ2∘BZ1 − u1·CZ2 − u2·CZ1
  nova/src/prover.rs:35                     self.ck.commit(&t)
  nova/src/relaxed_r1cs/witness.rs:56-71    RelaxedR1csWitness::fold            e = e1 + t·r,  w = w1 + w2·r
  nova/src/relaxed_r1cs.rs:80-146           R1csShape::is_sat(_relaxed)         (A z)∘(B z) = u·(C z) + E, commit(W) (and commit(E))
Vectors are (n, 4) uint64 Montgomery arrays of the constraint system's field (FIELD_FQ for nova's GrumpkinDriver, FIELD_FR
for Bn254Driver); z = (u, x, w) is passed whole, matrices are CSR over flat column indices into z.
"""
import collections
import ctypes

import numpy as np

from . import _lib
from .msm import _c, _u64

FIELD_FQ, FIELD_FR = 0, 1
_u32p = ctypes.POINTER(ctypes.c_uint32)
_u64p = ctypes.POINTER(ctypes.c_uint64)


class SatReport(collections.namedtuple("SatReport", "sat violations first_violation commit_w commit_e u_ok")):
    """kgr_nova_is_sat's report.  `bool(report)` is `sat`.  violations: rows with (A z)_i (B z)_i != u (C z)_i + E_i; first_violation: the
    lowest such row (m if none); commit_w / commit_e: True equal, False different, None not checked; u_ok: relaxed, or z[0] == 1."""
    __slots__ = ()

    def __bool__(self):
        return self.sat

    @classmethod
    def _from_words(cls, r):
        status = {0: False, 1: True, 2: None}
        return cls(bool(r[0]), int(r[1]), int(r[2]), status[int(r[3])], status[int(r[4])], bool(r[5]))


class R1csShape:
    """A, B, C resident on the GPU (kgr_r1cs_register).  Each matrix is (row_ptr[m+1] uint32, cols[nnz] uint32, coeffs (nnz, 4) uint64)."""

    def __init__(self, field, m, n_z, a, b, c):
        _lib.ensure_init()
        self.field, self.m, self.n_z = field, m, n_z
        keep = []
        rp, cl, cf = (_u32p * 3)(), (_u32p * 3)(), (_u64p * 3)()
        for k, (row_ptr, cols, coeffs) in enumerate((a, b, c)):
            row_ptr = _c(row_ptr, np.uint32)
            cols = _c(cols, np.uint32)
            coeffs = _c(coeffs).reshape(-1, 4)
            assert row_ptr.shape[0] == m + 1 and cols.shape[0] == coeffs.shape[0] == int(row_ptr[-1])
            keep += [row_ptr, cols, coeffs]
            rp[k] = row_ptr.ctypes.data_as(_u32p)
            cl[k] = cols.ctypes.data_as(_u32p)
            cf[k] = coeffs.ctypes.data_as(_u64p)
        h = ctypes.c_void_p()
        _lib.check(_lib.lib().kgr_r1cs_register(field, m, n_z, rp, cl, cf, ctypes.byref(h)))
        self._h = h

    def prod(self, which, z):
        """SparseMatrix::prod: which = 0 A, 1 B, 2 C -> (m, 4)."""
        z = _c(z).reshape(-1, 4)
        assert z.shape[0] == self.n_z
        out = np.zeros((self.m, 4), dtype=np.uint64)
        _lib.check(_lib.lib().kgr_r1cs_mul(self._h, which, _u64(z), _u64(out)))
        return out

    def cross_term(self, z1, z2, ck=None, want_t=True):
        """compute_cross_term; with a commitment key (`Bases` or `PedersenCommitment`) also commit(T) from the device-resident T.
        -> T (m, 4) [, commit (9,)]"""
        z1, z2 = _c(z1).reshape(-1, 4), _c(z2).reshape(-1, 4)
        assert z1.shape[0] == self.n_z and z2.shape[0] == self.n_z
        t = np.zeros((self.m, 4), dtype=np.uint64) if want_t else None
        bases = getattr(ck, "g", ck)
        commit = np.zeros(9, dtype=np.uint64) if bases is not None else None
        _lib.check(_lib.lib().kgr_nova_cross_term(self._h, _u64(z1), _u64(z2), _u64(t) if t is not None else None,
                                                  bases._h if bases is not None else None, _u64(commit) if commit is not None else None))
        return (t, commit) if bases is not None else t

    def is_sat(self, z, w_off, ck=None, commit_w=None):
        """R1csShape::is_sat (relaxed_r1cs.rs:117-146) on the resident z = (1, x, w) (`DeviceVec`): (A z) o (B z) = C z for every row, and
        with a key (`Bases` or `PedersenCommitment`) commit(z[w_off ..]) == commit_w when commit_w (9,) is given.  -> SatReport"""
        return self._is_sat(z, None, w_off, ck, commit_w, None)

    def is_sat_relaxed(self, z, e, w_off, ck=None, commit_w=None, commit_e=None):
        """The relaxed relation (relaxed_r1cs.rs:80-114): (A z) o (B z) = u (C z) + E with u = z[0], z and E resident (`DeviceVec`); each
        expected commitment is checked only when given.  -> SatReport"""
        return self._is_sat(z, e, w_off, ck, commit_w, commit_e)

    def _is_sat(self, z, e, w_off, ck, commit_w, commit_e):
        bases = getattr(ck, "g", ck)
        keep = [_c(c).reshape(9) if c is not None else None for c in (commit_w, commit_e)]
        report = np.zeros(6, dtype=np.uint64)
        _lib.check(_lib.lib().kgr_nova_is_sat(self._h, z._h, e._h if e is not None else None, w_off, bases._h if bases is not None else None,
                                              *[_u64(c) if c is not None else None for c in keep], _u64(report)))
        return SatReport._from_words(report)

    def last_timing(self):
        ms = (ctypes.c_float * 3)()
        _lib.check(_lib.lib().kgr_r1cs_last_timing(self._h, ms))
        return dict(h2d=float(ms[0]), cross_term=float(ms[1]), commit=float(ms[2]))

    def free(self):
        if getattr(self, "_h", None):
            _lib.lib().kgr_r1cs_free(self._h)
            self._h = None

    def __del__(self):
        try:
            self.free()
        except Exception:
            pass


def vec_fold(field, a, b, r):
    """a + b * r element-wise (RelaxedR1csWitness::fold): a, b (n, 4); r (4,) Montgomery."""
    _lib.ensure_init()
    a, b, r = _c(a).reshape(-1, 4), _c(b).reshape(-1, 4), _c(r).reshape(4)
    assert a.shape == b.shape
    out = np.zeros_like(a)
    _lib.check(_lib.lib().kgr_vec_fold(field, _u64(a), _u64(b), _u64(r), a.shape[0], _u64(out)))
    return out


class DeviceVec:
    """A vector of field elements that stays on the GPU between folding steps (kgr_vec_t): nova's z = (u, x, w), E, T.
    `RelaxedR1csWitness { w, e }` (nova/src/relaxed_r1cs/witness.rs:20-21) with both members resident is two of these."""

    def __init__(self, field, values=None, n=None):
        _lib.ensure_init()
        self.field = field
        h = ctypes.c_void_p()
        if values is not None:
            v = _c(values).reshape(-1, 4)
            self.n = v.shape[0]
            _lib.check(_lib.lib().kgr_vec_upload(field, _u64(v), self.n, ctypes.byref(h)))
        else:
            self.n = int(n)
            _lib.check(_lib.lib().kgr_vec_upload(field, None, self.n, ctypes.byref(h)))
        self._h = h

    def __len__(self):
        return self.n

    def download(self, off=0, n=None):
        n = self.n - off if n is None else n
        out = np.zeros((n, 4), dtype=np.uint64)
        _lib.check(_lib.lib().kgr_vec_download(self._h, off, n, _u64(out)))
        return out

    def write(self, off, values):
        v = _c(values).reshape(-1, 4)
        _lib.check(_lib.lib().kgr_vec_write(self._h, off, _u64(v), v.shape[0]))

    def fold(self, other, r, out=None):
        """self + other * r element-wise on the device (witness.rs:67-68); out defaults to self (in place) and is returned."""
        out = out or self
        r = _c(r).reshape(4)
        _lib.check(_lib.lib().kgr_vec_fold_device(self._h, other._h, _u64(r), out._h))
        return out

    def commit(self, ck, off=0, n=None):
        """PedersenCommitment::commit of elements [off, off + n) without leaving the device -> (9,) x, y, is_infinity."""
        bases = getattr(ck, "g", ck)
        n = self.n - off if n is None else n
        out = np.zeros(9, dtype=np.uint64)
        _lib.check(_lib.lib().kgr_pedersen_commit_vec(bases._h, self._h, off, n, _u64(out)))
        return out

    def free(self):
        if getattr(self, "_h", None):
            _lib.lib().kgr_vec_free(self._h)
            self._h = None

    def __del__(self):
        try:
            self.free()
        except Exception:
            pass


def cross_term_device(shape, z1, z2, t=None, ck=None):
    """compute_cross_term with z1, z2 (DeviceVec) resident; T stays in `t` (DeviceVec) — -> commit (9,) when a key is given."""
    bases = getattr(ck, "g", ck)
    commit = np.zeros(9, dtype=np.uint64) if bases is not None else None
    _lib.check(_lib.lib().kgr_nova_cross_term_device(shape._h, z1._h, z2._h, t._h if t is not None else None, bases._h if bases is not None else None,
                                                     _u64(commit) if commit is not None else None))
    return commit
