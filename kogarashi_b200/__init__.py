"""kogarashi_b200 — B200-native (sm_100a) multi-scalar multiplication for Kogarashi's BN254 G1 and
Grumpkin curves, behind the reference's own entry points (groth16::msm::msm_curve_addition,
nova::PedersenCommitment::commit).  The product is the CUDA engine in csrc/ behind the C ABI in
include/kgr_msm.h; this package is the thin host mirror used by tests and bench.py."""
from ._lib import KgrError, build, init, lib  # noqa: F401
from .msm import (BN254_G1, BN254_G2, GRUMPKIN, SCALARS_CANONICAL, SCALARS_MONTGOMERY, Bases, event_elapsed_ms, event_record,  # noqa: F401
                  last_timing, launch_count, msm_host_ptr, msm_oneshot_ptr,
                  microbench, groth16_msms, groth16_prove_r1cs, msm_batch, msm_curve_addition, msm_device, pairing, pairing_product, proj_add, set_param, to_affine)
from .fft import Fft  # noqa: F401
from .pedersen import PedersenCommitment  # noqa: F401
from .groth16 import Groth16Verifier, ProverSubVersionCrsAttack  # noqa: F401
