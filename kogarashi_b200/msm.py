"""Host-side mirror of the reference's MSM entry point over the C ABI.

Reference interface mirrored here (paths relative to the Kogarashi repo):
  groth16/src/msm.rs:6   pub fn msm_curve_addition<C: BNAffine>(bases: &[C], coeffs: &[C::Scalar]) -> C::Extended
Semantics kept: pairs = zip(coeffs, bases) (msm.rs:25), identity bases allowed, the result is a
projective representative (compare after to_affine).  Arrays are numpy uint64 views of the
reference's own limbs: points (n, 8) = x||y Montgomery, scalars (n, 4) Montgomery (`Fr.0`).
"""
import ctypes

import numpy as np

from . import _lib

BN254_G1 = 0   # bn_254::G1Affine, scalars bn_254::Fr
GRUMPKIN = 1   # grumpkin::Affine, scalars bn_254::Fq
BN254_G2 = 2   # bn_254::G2Affine (coordinates in Fq2 = c0 || c1), scalars bn_254::Fr  (next row N3, groth16/src/prover.rs:64-65)
SCALARS_MONTGOMERY = 0
SCALARS_CANONICAL = 1

_u64p = ctypes.POINTER(ctypes.c_uint64)
_u8p = ctypes.POINTER(ctypes.c_uint8)


def _u64(a):
    return a.ctypes.data_as(_u64p)


def _c(a, dtype=np.uint64):
    return np.ascontiguousarray(a, dtype=dtype)


def coord_limbs(curve):
    """uint64 limbs per coordinate: 4, or 8 for G2 (an Fq2 element c0 || c1)."""
    return 8 if curve == BN254_G2 else 4


class Bases:
    """A base vector resident on the GPU(s) (kgr_bases_register): a Groth16 CRS query or a Pedersen ck."""

    def __init__(self, curve, points=None, inf=None, _handle=None, _n=None):
        _lib.ensure_init()
        self.curve = curve
        if _handle is not None:
            self._h, self.n = _handle, _n
            return
        pts = _c(points).reshape(-1, 2 * coord_limbs(curve))
        self.n = pts.shape[0]
        h = ctypes.c_void_p()
        infp = None
        if inf is not None:
            inf = _c(inf, np.uint8)
            assert inf.shape[0] == self.n
            infp = inf.ctypes.data_as(_u8p)
        _lib.check(_lib.lib().kgr_bases_register(curve, _u64(pts), infp, self.n, ctypes.byref(h)))
        self._h = h

    @classmethod
    def generate(cls, curve, n, seed, return_scalars=False, first=0):
        """n points k_i*G computed on the device from a seed — SYNTHETIC BENCHMARK / TEST INPUTS ONLY: the k_i come from a public 64-bit
        splitmix64 stream, so every discrete logarithm is known and a commitment key built this way is not binding.  `first`: global index
        of point 0 (a shard of a larger vector)."""
        _lib.ensure_init()
        h = ctypes.c_void_p()
        ks = np.zeros((n, 4), dtype=np.uint64) if return_scalars else None
        _lib.check(_lib.lib().kgr_bases_generate_at(curve, seed, first, n, ctypes.byref(h), _u64(ks) if ks is not None else None))
        b = cls(curve, _handle=h, _n=n)
        return (b, ks) if return_scalars else b

    def __len__(self):
        return self.n

    def precompute(self, window_bits=0):
        """kgr_bases_precompute: build the 2^(c*w) * P_i table so that MSMs on this vector run window-collapsed."""
        _lib.check(_lib.lib().kgr_bases_precompute(self._h, window_bits))
        return self

    def download(self, off=0, n=None):
        """Copy registered points back to the host as (n, 8) uint64 (identity entries read (0, 0))."""
        n = self.n - off if n is None else n
        out = np.zeros((n, 2 * coord_limbs(self.curve)), dtype=np.uint64)
        _lib.check(_lib.lib().kgr_bases_download(self._h, off, n, _u64(out)))
        return out

    def free(self):
        if getattr(self, "_h", None):
            _lib.lib().kgr_bases_free(self._h)
            self._h = None

    def __del__(self):
        try:
            self.free()
        except Exception:
            pass


def msm_curve_addition(bases, coeffs, curve=BN254_G1, inf=None, scalar_fmt=SCALARS_MONTGOMERY, base_off=0):
    """sum_i coeffs[i] * bases[i] over the first min(len) pairs -> (12,) uint64 projective (X, Y, Z).

    `bases` is either a registered `Bases` (device-resident, only the scalars are uploaded) or an
    (n, 8) uint64 array (uploaded for this call, like the reference's by-slice signature)."""
    _lib.ensure_init()
    sc = _c(coeffs).reshape(-1, 4)
    if isinstance(bases, Bases):
        curve = bases.curve
    out = np.zeros(3 * coord_limbs(curve), dtype=np.uint64)
    L = _lib.lib()
    if isinstance(bases, Bases):
        n = min(sc.shape[0], bases.n - base_off)
        _lib.check(L.kgr_msm(bases._h, base_off, _u64(sc), scalar_fmt, n, _u64(out)))
    else:
        pts = _c(bases).reshape(-1, 2 * coord_limbs(curve))
        infp = None
        if inf is not None:
            inf = _c(inf, np.uint8)
            infp = inf.ctypes.data_as(_u8p)
        _lib.check(L.kgr_msm_oneshot(curve, _u64(pts), infp, pts.shape[0], _u64(sc), scalar_fmt, sc.shape[0], _u64(out)))
    return out


class _Job(ctypes.Structure):
    _fields_ = [("bases", ctypes.c_void_p), ("base_off", ctypes.c_size_t), ("scalars", _u64p), ("scalar_fmt", ctypes.c_int),
                ("n", ctypes.c_size_t), ("out", _u64p)]


def msm_batch(jobs, scalar_fmt=SCALARS_MONTGOMERY):
    """kgr_msm_batch: jobs = [(Bases, coeffs[, base_off[, scalar_fmt]]), ...] -> list of projective results.  Independent MSMs
    on registered vectors (the prover's h, l, a, b_g1, b_g2 queries, prover.rs:51-65) overlap on separate lanes of the device."""
    _lib.ensure_init()
    arr, keep, outs = _job_array(jobs, scalar_fmt)
    _lib.check(_lib.lib().kgr_msm_batch(ctypes.cast(arr, ctypes.c_void_p), len(jobs)))
    return outs


def _job_array(jobs, scalar_fmt):
    arr = (_Job * max(len(jobs), 1))()
    keep, outs = [], []
    for i, job in enumerate(jobs):
        bases, coeffs = job[0], _c(job[1]).reshape(-1, 4)
        off = job[2] if len(job) > 2 else 0
        fmt = job[3] if len(job) > 3 else scalar_fmt
        out = np.zeros(3 * coord_limbs(bases.curve), dtype=np.uint64)
        keep.append(coeffs)
        outs.append(out)
        arr[i] = _Job(bases._h.value if hasattr(bases._h, "value") else bases._h, off, _u64(coeffs), fmt, min(coeffs.shape[0], bases.n - off), _u64(out))
    return arr, keep, outs


def groth16_msms(log_n, a_evals, b_evals, c_evals, h_bases, jobs, scalar_fmt=SCALARS_MONTGOMERY, want_q=True):
    """kgr_groth16_msms: prover.rs:36-65 in one call.  H is computed on the device and goes into msm(h_bases, q) without leaving it; `jobs` (as in
    msm_batch) overlap on other lanes.  -> (h_point (12,), q (stripped, (len, 4)) or None, [job results])."""
    _lib.ensure_init()
    a, b, c = (_c(x).reshape(-1, 4) for x in (a_evals, b_evals, c_evals))
    assert a.shape == b.shape == c.shape
    arr, keep, outs = _job_array(jobs, scalar_fmt)
    h_out = np.zeros(12, dtype=np.uint64)
    q = np.zeros((1 << log_n, 4), dtype=np.uint64) if want_q else None
    q_len = ctypes.c_size_t()
    _lib.check(_lib.lib().kgr_groth16_msms(log_n, _u64(a), _u64(b), _u64(c), a.shape[0], h_bases._h, _u64(h_out), _u64(q) if want_q else None,
                                           ctypes.byref(q_len), ctypes.cast(arr, ctypes.c_void_p), len(jobs)))
    return h_out, (q[: q_len.value] if want_q else None), outs


def groth16_prove_r1cs(log_n, shape, z, n_inputs, h, l, a, b_g1, b_g2, jobs, want_q=True):
    """kgr_groth16_prove_r1cs: prover.rs:32-65 from a registered R1CS shape (nova.R1csShape over Fr) and the resident assignment z = x ++ w
    (nova.DeviceVec; x = the n_inputs instance elements, the constant one first).  b_g2 may be None (G1 only); `jobs` as in msm_batch.
    -> ({"h", "l", "a", "b_g1"[, "b_g2"]: projective results}, q (stripped) or None, [job results])."""
    _lib.ensure_init()
    arr, keep, outs = _job_array(jobs, SCALARS_MONTGOMERY)
    out = np.zeros(72, dtype=np.uint64)
    q = np.zeros((1 << log_n, 4), dtype=np.uint64) if want_q else None
    q_len = ctypes.c_size_t()
    _lib.check(_lib.lib().kgr_groth16_prove_r1cs(log_n, shape._h, z._h, n_inputs, h._h, l._h, a._h, b_g1._h, b_g2._h if b_g2 is not None else None,
                                                 _u64(out), _u64(q) if want_q else None, ctypes.byref(q_len), ctypes.cast(arr, ctypes.c_void_p), len(jobs)))
    res = {"h": out[0:12], "l": out[12:24], "a": out[24:36], "b_g1": out[36:48]}
    if b_g2 is not None:
        res["b_g2"] = out[48:72]
    return res, (q[: q_len.value] if want_q else None), outs


SETUP_QUERIES = ("h", "l", "a", "b_g1", "b_g2", "ic")


def groth16_setup(shape, n_inputs, toxic, g2=True):
    """kgr_groth16_setup: groth16/src/zksnark.rs:17-127 on the device from a registered R1CS shape (nova.R1csShape over Fr).  toxic: (5, 4) uint64
    Montgomery alpha, beta, gamma, delta, tau.  -> (log_n, {query name: Bases} (no "b_g2" without g2), vk_g1 (3, 9), vk_g2 (3, 17) or None)."""
    _lib.ensure_init()
    toxic = _c(toxic).reshape(5, 4)
    handles = [ctypes.c_void_p() for _ in SETUP_QUERIES]
    log_n = ctypes.c_uint32()
    vk_g1 = np.zeros((3, 9), dtype=np.uint64)
    vk_g2 = np.zeros((3, 17), dtype=np.uint64) if g2 else None
    refs = [ctypes.byref(h) if name != "b_g2" or g2 else None for name, h in zip(SETUP_QUERIES, handles)]
    _lib.check(_lib.lib().kgr_groth16_setup(shape._h, n_inputs, _u64(toxic), ctypes.byref(log_n), *refs, _u64(vk_g1), _u64(vk_g2) if g2 else None))
    L = _lib.lib()
    queries = {name: Bases(BN254_G2 if name == "b_g2" else BN254_G1, _handle=h, _n=L.kgr_bases_len(h))
               for name, h in zip(SETUP_QUERIES, handles) if name != "b_g2" or g2}
    return int(log_n.value), queries, vk_g1, vk_g2


def groth16_setup_timing():
    """Device time (ms) per phase of the last groth16_setup (kgr_groth16_setup_last_timing)."""
    ms = (ctypes.c_float * 10)()
    _lib.check(_lib.lib().kgr_groth16_setup_last_timing(ms))
    keys = ["powers_idft", "columns", "scalars", "a", "b_g1", "ic", "l", "h", "b_g2", "vk"]
    return dict(zip(keys, [float(x) for x in ms]))


def _pair_rows(g1, g2):
    g1 = _c(g1).reshape(-1, 9)
    g2 = _c(g2).reshape(-1, 17)
    if g1.shape[0] != g2.shape[0]:
        raise ValueError("g1 and g2 must hold the same number of points")
    return g1, g2


def pairing(g1, g2):
    """kgr_pairing op 0: the reduced optimal-ate pairing e(P_i, Q_i) per pair.  g1: (n, 9) x, y, is_infinity; g2: (n, 17) x.c0 x.c1 y.c0 y.c1,
    is_infinity (Montgomery).  -> (n, 48) uint64: 12 Montgomery Fq elements per value in tower order (include/kgr_msm.h)."""
    _lib.ensure_init()
    g1, g2 = _pair_rows(g1, g2)
    out = np.zeros((g1.shape[0], 48), dtype=np.uint64)
    _lib.check(_lib.lib().kgr_pairing(_u64(g1), _u64(g2), g1.shape[0], 0, _u64(out)))
    return out


def pairing_product(g1, g2):
    """kgr_pairing op 1: prod_i e(P_i, Q_i) with one final exponentiation.  -> (48,) uint64."""
    _lib.ensure_init()
    g1, g2 = _pair_rows(g1, g2)
    out = np.zeros(48, dtype=np.uint64)
    _lib.check(_lib.lib().kgr_pairing(_u64(g1), _u64(g2), g1.shape[0], 1, _u64(out)))
    return out


def groth16_verify(vk_g1, vk_g2, ic, proofs, inputs, rho):
    """kgr_groth16_verify.  vk_g1 (3, 9), vk_g2 (3, 17), ic: Bases of n_public + 1 G1 points, proofs (k, 35), inputs (k, n_public, 4) Montgomery
    Fr, rho (k, 2) uint64 or None.  -> (k,) bool."""
    _lib.ensure_init()
    vk_g1, vk_g2, proofs = _c(vk_g1).reshape(3, 9), _c(vk_g2).reshape(3, 17), _c(proofs).reshape(-1, 35)
    k, n_public = proofs.shape[0], ic.n - 1
    inputs = _c(inputs).reshape(k, n_public, 4) if n_public else np.zeros((k, 0, 4), dtype=np.uint64)
    ok = np.zeros(k, dtype=np.uint32)
    rp = None
    if rho is not None:
        rho = _c(rho).reshape(k, 2)
        rp = _u64(rho)
    _lib.check(_lib.lib().kgr_groth16_verify(_u64(vk_g1), _u64(vk_g2), ic._h, _u64(proofs), k, _u64(inputs) if inputs.size else None, n_public, rp,
                                             ok.ctypes.data_as(ctypes.POINTER(ctypes.c_uint32))))
    return ok.astype(bool)


def msm_device(bases, d_scalars_ptr, n, scalar_fmt=SCALARS_MONTGOMERY, base_off=0):
    """MSM with the scalars already in device memory (raw pointer, n x 4 uint64)."""
    out = np.zeros(3 * coord_limbs(bases.curve), dtype=np.uint64)
    _lib.check(_lib.lib().kgr_msm_device(bases._h, base_off, ctypes.c_void_p(d_scalars_ptr), scalar_fmt, n, _u64(out)))
    return out


def to_affine(curve, proj):
    """BNProjective::to_affine (zkstd/src/macros/curve/weierstrass.rs:57-66) -> (9,) x, y, is_infinity ((17,) for G2)."""
    proj = _c(proj)
    out = np.zeros(2 * coord_limbs(curve) + 1, dtype=np.uint64)
    _lib.check(_lib.lib().kgr_to_affine(curve, _u64(proj), _u64(out)))
    return out


def proj_add(curve, a, b):
    a, b = _c(a), _c(b)
    out = np.zeros(3 * coord_limbs(curve), dtype=np.uint64)
    _lib.check(_lib.lib().kgr_proj_add(curve, _u64(a), _u64(b), _u64(out)))
    return out


def last_timing(dev=0):
    ms = (ctypes.c_float * 9)()
    shape = (ctypes.c_uint32 * 6)()
    _lib.check(_lib.lib().kgr_last_timing(dev, ms, shape))
    keys = ["total", "count", "scan", "fill", "accumulate", "fixup", "reduce", "h2d", "host_finish"]
    return dict(zip(keys, [float(x) for x in ms])), dict(zip(["c", "W", "B", "L", "K", "n"], [int(x) for x in shape]))


def event_record(idx, dev=0):
    _lib.check(_lib.lib().kgr_event_record(dev, idx))


def event_elapsed_ms(a, b, dev=0):
    ms = ctypes.c_float()
    _lib.check(_lib.lib().kgr_event_elapsed_ms(dev, a, b, ctypes.byref(ms)))
    return float(ms.value)


def launch_count(dev=0):
    c = ctypes.c_uint64()
    _lib.check(_lib.lib().kgr_launch_count(dev, ctypes.byref(c)))
    return int(c.value)


def msm_oneshot_ptr(curve, xy_ptr, n_bases, sc_ptr, n_scalars, scalar_fmt=SCALARS_MONTGOMERY):
    """kgr_msm_oneshot on raw host pointers (e.g. pinned torch tensors): bases and scalars are uploaded inside the call."""
    out = np.zeros(3 * coord_limbs(curve), dtype=np.uint64)
    L = _lib.lib()
    _lib.check(L.kgr_msm_oneshot(curve, ctypes.cast(xy_ptr, _u64p), None, n_bases, ctypes.cast(sc_ptr, _u64p), scalar_fmt, n_scalars, _u64(out)))
    return out


def msm_host_ptr(bases, sc_ptr, n, scalar_fmt=SCALARS_MONTGOMERY, base_off=0):
    """kgr_msm on a raw host pointer to the scalars (registered bases)."""
    out = np.zeros(3 * coord_limbs(bases.curve), dtype=np.uint64)
    _lib.check(_lib.lib().kgr_msm(bases._h, base_off, ctypes.cast(sc_ptr, _u64p), scalar_fmt, n, _u64(out)))
    return out


def set_param(name, value):
    _lib.check(_lib.lib().kgr_set_param(name.encode(), int(value)))


def microbench():
    _lib.ensure_init()
    r = (ctypes.c_double * 8)()
    _lib.check(_lib.lib().kgr_microbench(r))
    keys = ["imad_gops", "imad_hi_gops", "imad_wide_gops", "imad_wide_x_gops", "iadd3_gops", "fq_mul_gops", "xyzz_madd_gops", "sm_mhz"]
    return dict(zip(keys, [float(x) for x in r]))


def test_field_op(field, op, a, b=None):
    _lib.ensure_init()
    a = _c(a).reshape(-1, 4)
    out = np.zeros_like(a)
    bp = None
    if b is not None:
        b = _c(b).reshape(-1, 4)
        bp = _u64(b)
    _lib.check(_lib.lib().kgr_test_field_op(field, op, _u64(a), bp, a.shape[0], _u64(out)))
    return out


def test_point_op(curve, op, a, b, a_inf=None, b_inf=None):
    _lib.ensure_init()
    cl = coord_limbs(curve)
    a, b = _c(a).reshape(-1, 2 * cl), _c(b).reshape(-1, 2 * cl)
    out = np.zeros((a.shape[0], 3 * cl), dtype=np.uint64)
    ai = _c(a_inf, np.uint8) if a_inf is not None else None
    bi = _c(b_inf, np.uint8) if b_inf is not None else None
    _lib.check(_lib.lib().kgr_test_point_op(curve, op, _u64(a), ai.ctypes.data_as(_u8p) if ai is not None else None, _u64(b),
                                            bi.ctypes.data_as(_u8p) if bi is not None else None, a.shape[0], _u64(out)))
    return out


def fixed_base_mul(curve, k):
    _lib.ensure_init()
    k = _c(k).reshape(-1, 4)
    out = np.zeros((k.shape[0], 2 * coord_limbs(curve)), dtype=np.uint64)
    _lib.check(_lib.lib().kgr_fixed_base_mul(curve, _u64(k), k.shape[0], _u64(out)))
    return out
