"""oracle/oracle.py — TEST INFRASTRUCTURE: ctypes front-end to libzkstd_oracle.so (Oracle A).

Only tests/, __graft_entry__.smoke() and bench.py's cpu_baseline / --impl reference legs import
this.  Array conventions equal include/kgr_msm.h: points (n, 8) uint64 = x||y Montgomery limbs,
optional (n,) uint8 infinity flags, scalars (n, 4) uint64 Montgomery, projective result (12,).
For BN254_G2 every coordinate is 8 limbs (c0 || c1): points (n, 16), projective (24,), affine (17,).
"""
import ctypes
import os
import subprocess

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
_LIB_PATH = os.path.join(_HERE, "libzkstd_oracle.so")

BN254_G1, GRUMPKIN, BN254_G2 = 0, 1, 2
FIELD_FQ, FIELD_FR = 0, 1
# base / scalar field ids per curve
BASE_FIELD = {BN254_G1: FIELD_FQ, GRUMPKIN: FIELD_FR}
SCALAR_FIELD = {BN254_G1: FIELD_FR, GRUMPKIN: FIELD_FQ, BN254_G2: FIELD_FR}


def coord_limbs(curve):
    """uint64 limbs per coordinate: 4, or 8 for G2 (Fq2 = c0 || c1, bn254/src/fqn.rs)."""
    return 8 if curve == BN254_G2 else 4

OPS = dict(add=0, sub=1, mul=2, square=3, double=4, neg=5, invert=6, mont_reduce=7, to_mont=8, from_u512=9)


def build(force=False):
    src = [os.path.join(_HERE, f) for f in ("zkstd_oracle.cpp", "zkstd_oracle.hpp")]
    if force or not os.path.exists(_LIB_PATH) or any(
            os.path.exists(s) and os.path.getmtime(s) > os.path.getmtime(_LIB_PATH) for s in src):
        subprocess.check_call(["make", "-C", _HERE, "-s"])
    return _LIB_PATH


def _owned_private(path, kind):
    """True if `path` is a `kind` (stat.S_ISDIR / S_ISREG), not a symlink, owned by this user and writable by nobody else: only then is
    a shared object found there ours to load."""
    import stat
    st = os.lstat(path)
    return kind(st.st_mode) and st.st_uid == os.getuid() and not st.st_mode & (stat.S_IWGRP | stat.S_IWOTH)


def _native_path():
    """libzkstd_oracle.<tag>.so: the same source built with -march=native on THIS host (the portable .so travels between machines with
    different CPUs).  Built at first use into the user's cache directory ($XDG_CACHE_HOME or ~/.cache, kogarashi-oracle/), not into the
    source tree, which a benchmark run must leave as it found it (and which may be read-only); the tag hashes the CPU and the sources, so
    checkouts of different versions never share a build.  Nothing is loaded from that directory unless it and the file belong to this
    user and are writable by no one else.  None if any of this is not possible (no compiler, no private cache directory), in which case
    the portable build is used."""
    if os.environ.get("ZKO_PORTABLE"):
        return None
    try:
        import hashlib
        import stat
        with open("/proc/cpuinfo") as f:
            model = next((line for line in f if line.startswith(("model name", "flags"))), "")
            flags = next((line for line in f if line.startswith("flags")), "")
        h = hashlib.sha1((model + flags).encode())
        for name in ("zkstd_oracle.cpp", "zkstd_oracle.hpp"):
            with open(os.path.join(_HERE, name), "rb") as f:
                h.update(f.read())
        base = os.environ.get("XDG_CACHE_HOME") or os.path.join(os.path.expanduser("~"), ".cache")
        cache = os.path.join(base, "kogarashi-oracle")
        os.makedirs(cache, mode=0o700, exist_ok=True)
        if not _owned_private(cache, stat.S_ISDIR):
            return None
        path = os.path.join(cache, f"libzkstd_oracle.{h.hexdigest()[:10]}.so")
        if not os.path.lexists(path):
            tmp = f"{path}.{os.getpid()}.tmp"
            subprocess.check_call(["make", "-C", _HERE, "-s", "native", f"OUT={tmp}"], stdout=subprocess.DEVNULL, stderr=subprocess.DEVNULL)
            os.chmod(tmp, 0o700)
            os.replace(tmp, path)
        return path if _owned_private(path, stat.S_ISREG) else None
    except Exception:
        return None


def _pick_build():
    """The faster of the portable and the -march=native build on this host, by a 2^13-point MSM on all host threads (best of 3).  The
    flag alone is not a win everywhere: on the build container the native code is ~10 % faster on one thread and ~40 % SLOWER with all
    eight threads busy, so the baseline takes whichever build this host runs faster."""
    native = _native_path()
    if native is None:
        return _LIB_PATH
    import time
    best = (None, None)
    u64p = ctypes.POINTER(ctypes.c_uint64)
    for path in (_LIB_PATH, native):
        try:
            L = ctypes.CDLL(path)
            n = 1 << 13
            threads = os.cpu_count() or 1
            k = np.zeros((n, 4), dtype=np.uint64)
            xy = np.zeros((n, 8), dtype=np.uint64)
            out = np.zeros(12, dtype=np.uint64)
            L.zko_bench_scalars(0, ctypes.c_uint64(1), ctypes.c_uint64(0), ctypes.c_size_t(n), k.ctypes.data_as(u64p))
            L.zko_fixed_base(0, k.ctypes.data_as(u64p), ctypes.c_size_t(n), threads, xy.ctypes.data_as(u64p))
            dt = None
            for _ in range(3):
                t0 = time.perf_counter()
                L.zko_msm(0, xy.ctypes.data_as(u64p), None, ctypes.c_size_t(n), k.ctypes.data_as(u64p), ctypes.c_size_t(n), threads, out.ctypes.data_as(u64p))
                t1 = time.perf_counter() - t0
                dt = t1 if dt is None else min(dt, t1)
            if best[0] is None or dt < best[0]:
                best = (dt, path)
        except Exception:
            continue
    return best[1] or _LIB_PATH


_lib = None
LOADED_PATH = None


def lib():
    global _lib, LOADED_PATH
    if _lib is None:
        if not os.path.exists(_LIB_PATH):
            build()
        LOADED_PATH = _pick_build()
        L = ctypes.CDLL(LOADED_PATH)
        u64p = ctypes.POINTER(ctypes.c_uint64)
        u8p = ctypes.POINTER(ctypes.c_uint8)
        L.zko_field_op.argtypes = [ctypes.c_int, ctypes.c_int, u64p, u64p, u64p]
        L.zko_msm.argtypes = [ctypes.c_int, u64p, u8p, ctypes.c_size_t, u64p, ctypes.c_size_t, ctypes.c_int, u64p]
        L.zko_pedersen_commit.argtypes = [ctypes.c_int, u64p, u8p, ctypes.c_size_t, u64p, ctypes.c_size_t, u64p]
        L.zko_to_affine.argtypes = [ctypes.c_int, u64p, u64p]
        L.zko_point_op.argtypes = [ctypes.c_int, ctypes.c_int, u64p, u64p, u64p]
        L.zko_scalar_point.argtypes = [ctypes.c_int, u64p, u64p, u64p]
        L.zko_generator.argtypes = [ctypes.c_int, u64p]
        L.zko_random_field.argtypes = [ctypes.c_int, u8p, ctypes.c_size_t, u64p]
        L.zko_random_points.argtypes = [ctypes.c_int, u8p, ctypes.c_size_t, ctypes.c_int, u64p, u64p]
        L.zko_bench_scalars.argtypes = [ctypes.c_int, ctypes.c_uint64, ctypes.c_uint64, ctypes.c_size_t, u64p]
        L.zko_fixed_base.argtypes = [ctypes.c_int, u64p, ctypes.c_size_t, ctypes.c_int, u64p]
        L.zko_field_dot.argtypes = [ctypes.c_int, u64p, u64p, ctypes.c_size_t, ctypes.c_int, u64p]
        L.zko_xorshift_u64.argtypes = [u8p, ctypes.c_size_t, u64p]
        L.zko_fft.argtypes = [ctypes.c_size_t, ctypes.c_int, u64p, ctypes.c_size_t, u64p, ctypes.POINTER(ctypes.c_size_t)]
        L.zko_groth16_h.argtypes = [ctypes.c_size_t, u64p, u64p, u64p, ctypes.c_size_t, u64p, ctypes.POINTER(ctypes.c_size_t)]
        u32p = ctypes.POINTER(ctypes.c_uint32)
        L.zko_sparse_prod.argtypes = [ctypes.c_int, ctypes.c_size_t, u32p, u32p, u64p, u64p, ctypes.c_size_t, u64p]
        L.zko_cross_term.argtypes = [ctypes.c_int, ctypes.c_size_t, ctypes.POINTER(u32p), ctypes.POINTER(u32p), ctypes.POINTER(u64p), u64p, u64p,
                                     ctypes.c_size_t, u64p]
        L.zko_vec_fold.argtypes = [ctypes.c_int, u64p, u64p, u64p, ctypes.c_size_t, u64p]
        L.zko_window_bits.argtypes = [ctypes.c_size_t]
        L.zko_window_bits.restype = ctypes.c_size_t
        L.zko_get_at.argtypes = [ctypes.c_size_t, ctypes.c_size_t, u8p]
        L.zko_get_at.restype = ctypes.c_size_t
        _lib = L
    return _lib


def _u64(a):
    return a.ctypes.data_as(ctypes.POINTER(ctypes.c_uint64))


def _u8(a):
    return a.ctypes.data_as(ctypes.POINTER(ctypes.c_uint8))


def _c(a, dtype=np.uint64):
    return np.ascontiguousarray(a, dtype=dtype)


DEFAULT_SEED = bytes.fromhex("5962be5d763d318d17db37325406bce5")  # pallet/nova/src/tests.rs:69-74


def _seed(seed):
    s = np.frombuffer(bytes(seed), dtype=np.uint8).copy()
    assert s.size == 16
    return s


def field_op(field_id, op, a, b=None):
    a = _c(a)
    out = np.zeros(4, dtype=np.uint64)
    bb = _c(b) if b is not None else np.zeros(4, dtype=np.uint64)
    rc = lib().zko_field_op(field_id, OPS[op], _u64(a), _u64(bb), _u64(out))
    if rc == 1:
        return None
    assert rc == 0
    return out


def msm(curve, points, scalars, inf=None, threads=None):
    points, scalars = _c(points).reshape(-1, 2 * coord_limbs(curve)), _c(scalars).reshape(-1, 4)
    out = np.zeros(3 * coord_limbs(curve), dtype=np.uint64)
    infp = _u8(_c(inf, np.uint8)) if inf is not None else None
    rc = lib().zko_msm(curve, _u64(points), infp, points.shape[0], _u64(scalars), scalars.shape[0],
                       threads or os.cpu_count() or 1, _u64(out))
    assert rc == 0
    return out


def pedersen_commit(curve, points, scalars, inf=None):
    points, scalars = _c(points).reshape(-1, 2 * coord_limbs(curve)), _c(scalars).reshape(-1, 4)
    out = np.zeros(2 * coord_limbs(curve) + 1, dtype=np.uint64)
    infp = _u8(_c(inf, np.uint8)) if inf is not None else None
    assert lib().zko_pedersen_commit(curve, _u64(points), infp, points.shape[0], _u64(scalars), scalars.shape[0], _u64(out)) == 0
    return out


def to_affine(curve, proj):
    """-> (9,) uint64: x(4) y(4) is_infinity ((17,) for G2)."""
    proj = _c(proj)
    out = np.zeros(2 * coord_limbs(curve) + 1, dtype=np.uint64)
    assert lib().zko_to_affine(curve, _u64(proj), _u64(out)) == 0
    return out


def point_op(curve, op, a, b=None, out_len=None):
    a = _c(a)
    bb = _c(b) if b is not None else np.zeros(3 * coord_limbs(curve), dtype=np.uint64)
    out = np.zeros(out_len or 3 * coord_limbs(curve), dtype=np.uint64)
    assert lib().zko_point_op(curve, op, _u64(a), _u64(bb), _u64(out)) == 0
    return out


def scalar_point(curve, proj, scalar):
    proj, scalar = _c(proj), _c(scalar)
    out = np.zeros(3 * coord_limbs(curve), dtype=np.uint64)
    assert lib().zko_scalar_point(curve, _u64(proj), _u64(scalar), _u64(out)) == 0
    return out


def generator(curve):
    out = np.zeros(2 * coord_limbs(curve), dtype=np.uint64)
    assert lib().zko_generator(curve, _u64(out)) == 0
    return out


def random_field(field_id, n, seed=DEFAULT_SEED):
    out = np.zeros((n, 4), dtype=np.uint64)
    s = _seed(seed)
    assert lib().zko_random_field(field_id, _u8(s), n, _u64(out)) == 0
    return out


def random_points(curve, n, seed=DEFAULT_SEED, threads=None, return_scalars=False):
    xy = np.zeros((n, 2 * coord_limbs(curve)), dtype=np.uint64)
    ks = np.zeros((n, 4), dtype=np.uint64)
    s = _seed(seed)
    assert lib().zko_random_points(curve, _u8(s), n, threads or os.cpu_count() or 1, _u64(xy), _u64(ks)) == 0
    return (xy, ks) if return_scalars else xy


def bench_scalars(curve, seed, first, n):
    """Bench input support (not reference code): k_i = from_u512(splitmix64 stream of (seed, first + i)) in the curve's scalar field, the
    stream kgr_bases_generate_at uses on the device."""
    out = np.zeros((n, 4), dtype=np.uint64)
    assert lib().zko_bench_scalars(curve, seed, first, n, _u64(out)) == 0
    return out


def fixed_base(curve, k, threads=None):
    """Bench input support: k_i * G as affine points (identity -> (0, 0), the device encoding) via a byte-window table and add_mixed."""
    k = _c(k).reshape(-1, 4)
    xy = np.zeros((k.shape[0], 2 * coord_limbs(curve)), dtype=np.uint64)
    assert lib().zko_fixed_base(curve, _u64(k), k.shape[0], threads or os.cpu_count() or 1, _u64(xy)) == 0
    return xy


def field_dot(field_id, a, b, threads=None):
    """sum a_i * b_i (Montgomery in / out): with bases k_i * G an MSM must equal (sum k_i s_i) * G."""
    a, b = _c(a).reshape(-1, 4), _c(b).reshape(-1, 4)
    assert a.shape == b.shape
    out = np.zeros(4, dtype=np.uint64)
    assert lib().zko_field_dot(field_id, _u64(a), _u64(b), a.shape[0], threads or os.cpu_count() or 1, _u64(out)) == 0
    return out


def xorshift_u64(n, seed=DEFAULT_SEED):
    out = np.zeros(n, dtype=np.uint64)
    s = _seed(seed)
    assert lib().zko_xorshift_u64(_u8(s), n, _u64(out)) == 0
    return out


FFT_OPS = dict(dft=0, idft=1, coset_dft=2, coset_idft=3)


def fft(k, op, values):
    """groth16/src/fft.rs on Fr: returns (2^k, 4) uint64 and the stripped length (idft variants drop trailing zeros)."""
    v = _c(values).reshape(-1, 4)
    out = np.zeros((1 << k, 4), dtype=np.uint64)
    n_out = ctypes.c_size_t()
    assert lib().zko_fft(k, FFT_OPS[op], _u64(v), v.shape[0], _u64(out), ctypes.byref(n_out)) == 0
    return out, int(n_out.value)


def groth16_h(k, a, b, c):
    """prover.rs:36-47: H coefficients from the R1CS evaluation vectors."""
    a, b, c = (_c(x).reshape(-1, 4) for x in (a, b, c))
    out = np.zeros((1 << k, 4), dtype=np.uint64)
    n_out = ctypes.c_size_t()
    assert lib().zko_groth16_h(k, _u64(a), _u64(b), _u64(c), a.shape[0], _u64(out), ctypes.byref(n_out)) == 0
    return out, int(n_out.value)


def _u32(a):
    return a.ctypes.data_as(ctypes.POINTER(ctypes.c_uint32))


def sparse_prod(field_id, m, mat, z):
    """zkstd/src/matrix.rs:36-48: mat = (row_ptr[m+1], cols[nnz], coeffs (nnz, 4)) over flat column indices; -> (m, 4)."""
    rp, cl, cf = _c(mat[0], np.uint32), _c(mat[1], np.uint32), _c(mat[2]).reshape(-1, 4)
    z = _c(z).reshape(-1, 4)
    out = np.zeros((m, 4), dtype=np.uint64)
    assert lib().zko_sparse_prod(field_id, m, _u32(rp), _u32(cl), _u64(cf), _u64(z), z.shape[0], _u64(out)) == 0
    return out


def cross_term(field_id, m, a, b, c, z1, z2):
    """nova/src/prover.rs:53-90 compute_cross_term with z1 = (u1, x1, w1), z2 = (u2, x2, w2)."""
    u32p, u64p = ctypes.POINTER(ctypes.c_uint32), ctypes.POINTER(ctypes.c_uint64)
    keep = []
    rp, cl, cf = (u32p * 3)(), (u32p * 3)(), (u64p * 3)()
    for k, mat in enumerate((a, b, c)):
        arrs = (_c(mat[0], np.uint32), _c(mat[1], np.uint32), _c(mat[2]).reshape(-1, 4))
        keep.append(arrs)
        rp[k], cl[k], cf[k] = _u32(arrs[0]), _u32(arrs[1]), _u64(arrs[2])
    z1, z2 = _c(z1).reshape(-1, 4), _c(z2).reshape(-1, 4)
    out = np.zeros((m, 4), dtype=np.uint64)
    assert lib().zko_cross_term(field_id, m, rp, cl, cf, _u64(z1), _u64(z2), z1.shape[0], _u64(out)) == 0
    return out


def vec_fold(field_id, a, b, r):
    a, b, r = _c(a).reshape(-1, 4), _c(b).reshape(-1, 4), _c(r).reshape(4)
    out = np.zeros_like(a)
    assert lib().zko_vec_fold(field_id, _u64(a), _u64(b), _u64(r), a.shape[0], _u64(out)) == 0
    return out


def window_bits(n):
    return int(lib().zko_window_bits(n))


def get_at(segment, c, bytes32):
    b = np.frombuffer(bytes(bytes32), dtype=np.uint8).copy()
    return int(lib().zko_get_at(segment, c, _u8(b)))
