"""ctypes binding of libkgr_msm.so (the C ABI in include/kgr_msm.h).

The library is built in tree by `make -C kogarashi_b200/csrc` (or __graft_entry__.build()).  There
is deliberately no fallback: if the shared object is missing or no CUDA device is usable, every
entry point raises.
"""
import ctypes
import os
import subprocess

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "libkgr_msm.so")
CSRC = os.path.join(_HERE, "csrc")

EXPORTS = [
    "kgr_init", "kgr_shutdown", "kgr_last_error", "kgr_device_count", "kgr_bases_register", "kgr_bases_free",
    "kgr_bases_len", "kgr_msm", "kgr_msm_oneshot", "kgr_msm_device", "kgr_pedersen_commit", "kgr_to_affine",
    "kgr_proj_add", "kgr_set_param", "kgr_last_timing", "kgr_test_field_op", "kgr_test_point_op",
    "kgr_fixed_base_mul", "kgr_bases_generate", "kgr_microbench", "kgr_bases_download", "kgr_event_record",
    "kgr_event_elapsed_ms", "kgr_launch_count", "kgr_bases_precompute", "kgr_ntt", "kgr_ntt_device", "kgr_groth16_h",
    "kgr_bases_generate_at", "kgr_vec_upload", "kgr_vec_download", "kgr_vec_free", "kgr_vec_len", "kgr_vec_write", "kgr_vec_fold_device", "kgr_msm_vec",
    "kgr_pedersen_commit_vec", "kgr_nova_cross_term_device", "kgr_host_alloc", "kgr_host_free", "kgr_msm_batch", "kgr_groth16_msms", "kgr_groth16_prove_r1cs", "kgr_groth16_setup", "kgr_groth16_setup_last_timing", "kgr_r1cs_register", "kgr_r1cs_free", "kgr_r1cs_mul", "kgr_nova_cross_term", "kgr_r1cs_last_timing", "kgr_vec_fold",
    "kgr_pairing", "kgr_groth16_verify", "kgr_nova_is_sat",
]


class KgrError(RuntimeError):
    pass


def build(force=False):
    """Compile the CUDA engine for sm_100a (nvcc cross-compiles without a GPU)."""
    srcs = [os.path.join(CSRC, f) for f in os.listdir(CSRC) if f.endswith((".cu", ".cuh"))]
    srcs.append(os.path.join(_HERE, "..", "include", "kgr_msm.h"))
    stale = (not os.path.exists(LIB_PATH)) or any(os.path.getmtime(s) > os.path.getmtime(LIB_PATH) for s in srcs)
    if force or stale:
        subprocess.check_call(["make", "-C", CSRC, "-s"])
    return LIB_PATH


_lib = None


def lib():
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise KgrError(f"{LIB_PATH} is missing: build it with `make -C {CSRC}` (no CPU fallback exists)")
    L = ctypes.CDLL(LIB_PATH)
    u64p, u8p, vp = ctypes.POINTER(ctypes.c_uint64), ctypes.POINTER(ctypes.c_uint8), ctypes.c_void_p
    sz, ci = ctypes.c_size_t, ctypes.c_int
    L.kgr_init.argtypes = [ctypes.POINTER(ci), ci]
    L.kgr_last_error.restype = ctypes.c_char_p
    L.kgr_bases_register.argtypes = [ci, u64p, u8p, sz, ctypes.POINTER(vp)]
    L.kgr_bases_free.argtypes = [vp]
    L.kgr_bases_precompute.argtypes = [vp, ci]
    L.kgr_ntt.argtypes = [ctypes.c_uint, ci, u64p, sz, u64p, ctypes.POINTER(sz)]
    L.kgr_ntt_device.argtypes = [ctypes.c_uint, ci, vp]
    L.kgr_groth16_h.argtypes = [ctypes.c_uint, u64p, u64p, u64p, sz, u64p, ctypes.POINTER(sz)]
    L.kgr_bases_len.argtypes = [vp]
    L.kgr_bases_len.restype = sz
    L.kgr_msm.argtypes = [vp, sz, u64p, ci, sz, u64p]
    L.kgr_msm_oneshot.argtypes = [ci, u64p, u8p, sz, u64p, ci, sz, u64p]
    L.kgr_msm_device.argtypes = [vp, sz, vp, ci, sz, u64p]
    L.kgr_pedersen_commit.argtypes = [vp, u64p, ci, sz, u64p]
    L.kgr_to_affine.argtypes = [ci, u64p, u64p]
    L.kgr_proj_add.argtypes = [ci, u64p, u64p, u64p]
    L.kgr_set_param.argtypes = [ctypes.c_char_p, ctypes.c_long]
    L.kgr_last_timing.argtypes = [ci, ctypes.POINTER(ctypes.c_float), ctypes.POINTER(ctypes.c_uint32)]
    L.kgr_test_field_op.argtypes = [ci, ci, u64p, u64p, sz, u64p]
    L.kgr_test_point_op.argtypes = [ci, ci, u64p, u8p, u64p, u8p, sz, u64p]
    L.kgr_fixed_base_mul.argtypes = [ci, u64p, sz, u64p]
    L.kgr_bases_generate.argtypes = [ci, ctypes.c_uint64, sz, ctypes.POINTER(vp), u64p]
    L.kgr_bases_generate_at.argtypes = [ci, ctypes.c_uint64, ctypes.c_uint64, sz, ctypes.POINTER(vp), u64p]
    L.kgr_microbench.argtypes = [ctypes.POINTER(ctypes.c_double)]
    L.kgr_bases_download.argtypes = [vp, sz, sz, u64p]
    L.kgr_event_record.argtypes = [ci, ci]
    L.kgr_event_elapsed_ms.argtypes = [ci, ci, ci, ctypes.POINTER(ctypes.c_float)]
    L.kgr_launch_count.argtypes = [ci, ctypes.POINTER(ctypes.c_uint64)]
    u32p = ctypes.POINTER(ctypes.c_uint32)
    L.kgr_r1cs_register.argtypes = [ci, sz, sz, ctypes.POINTER(u32p), ctypes.POINTER(u32p), ctypes.POINTER(u64p), ctypes.POINTER(vp)]
    L.kgr_msm_batch.argtypes = [vp, sz]
    L.kgr_groth16_msms.argtypes = [ctypes.c_uint, u64p, u64p, u64p, sz, vp, u64p, u64p, ctypes.POINTER(sz), vp, sz]
    L.kgr_groth16_prove_r1cs.argtypes = [ctypes.c_uint, vp, vp, sz, vp, vp, vp, vp, vp, u64p, u64p, ctypes.POINTER(sz), vp, sz]
    L.kgr_groth16_setup.argtypes = [vp, sz, u64p, ctypes.POINTER(ctypes.c_uint32)] + [ctypes.POINTER(vp)] * 6 + [u64p, u64p]
    L.kgr_groth16_setup_last_timing.argtypes = [ctypes.POINTER(ctypes.c_float)]
    L.kgr_r1cs_free.argtypes = [vp]
    L.kgr_r1cs_mul.argtypes = [vp, ci, u64p, u64p]
    L.kgr_nova_cross_term.argtypes = [vp, u64p, u64p, u64p, vp, u64p]
    L.kgr_r1cs_last_timing.argtypes = [vp, ctypes.POINTER(ctypes.c_float)]
    L.kgr_vec_fold.argtypes = [ci, u64p, u64p, u64p, sz, u64p]
    L.kgr_vec_upload.argtypes = [ci, u64p, sz, ctypes.POINTER(vp)]
    L.kgr_vec_download.argtypes = [vp, sz, sz, u64p]
    L.kgr_vec_free.argtypes = [vp]
    L.kgr_vec_len.argtypes = [vp]
    L.kgr_vec_len.restype = sz
    L.kgr_vec_write.argtypes = [vp, sz, u64p, sz]
    L.kgr_vec_fold_device.argtypes = [vp, vp, u64p, vp]
    L.kgr_msm_vec.argtypes = [vp, sz, vp, sz, sz, u64p]
    L.kgr_pedersen_commit_vec.argtypes = [vp, vp, sz, sz, u64p]
    L.kgr_nova_cross_term_device.argtypes = [vp, vp, vp, vp, vp, u64p]
    L.kgr_nova_is_sat.argtypes = [vp, vp, vp, sz, vp, u64p, u64p, u64p]
    L.kgr_host_alloc.argtypes = [sz, ctypes.POINTER(vp)]
    L.kgr_host_free.argtypes = [vp]
    L.kgr_pairing.argtypes = [u64p, u64p, sz, ci, u64p]
    L.kgr_groth16_verify.argtypes = [u64p, u64p, vp, u64p, sz, u64p, sz, u64p, u32p]
    _lib = L
    return L


def check(rc):
    if rc != 0:
        raise KgrError(f"kgr error {rc}: {lib().kgr_last_error().decode(errors='replace')}")


_initialised = False


def init(devices=None):
    """kgr_init: devices=None -> the current CUDA device of this process."""
    global _initialised
    L = lib()
    if devices is None:
        check(L.kgr_init(None, 0))
    else:
        arr = (ctypes.c_int * len(devices))(*devices)
        check(L.kgr_init(arr, len(devices)))
    _initialised = True


def ensure_init():
    if not _initialised:
        init()
