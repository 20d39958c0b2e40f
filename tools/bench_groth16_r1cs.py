"""Groth16 proof from the constraint system (kgr_groth16_prove_r1cs) against the proof from host evaluations (kgr_groth16_msms), on the chain
circuit (the example's x^3 + x + 5 iterated) at 2^16 and 2^20 constraints.  One JSON line per size, also written to DIR/groth16_r1cs.jsonl:
  prove_from_evaluations_ms  best-of-N wall time after warm-up, a, b, c given as host arrays (the old path's input)
  prove_r1cs_ms              the same for prove_r1cs with the shape registered and z resident
  z_upload_ms                best-of-N wall time of the DeviceVec upload of z (what a caller with z in host memory adds to prove_r1cs)
  host_evaluate_s            cs.evaluate() as the old path needs it: the C++ oracle's SparseMatrix::prod (zkstd/src/matrix.rs:36-48) x 3, one core
  same_proof                 A, B, C and q of the two paths byte for byte, and the oracle's evaluations equal the host ones
  device_crs_setup_s         wall time of groth16.setup, which generates the CRS both provers use on the device
  h2d_bytes_per_call         per path, from the shapes
usage: python tools/bench_groth16_r1cs.py --out DIR [--logm 16 20] [--steps 5] [--warmup 3]"""
import argparse
import json
import os
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))
import kogarashi_b200 as k  # noqa: E402
from groth16_r1cs_util import csr_from_r1cs, mont  # noqa: E402
from kogarashi_b200.groth16 import Groth16Prover, setup  # noqa: E402
from kogarashi_b200.nova import FIELD_FR, DeviceVec, R1csShape  # noqa: E402
from oracle import groth16_ref as G  # noqa: E402
from oracle import oracle as A  # noqa: E402
from oracle import pyref as B  # noqa: E402


def _wall(fn):
    t0 = time.perf_counter()
    fn()
    return time.perf_counter() - t0


def card():
    """Name and power limit of device 0, read in the same run as the timings (nvidia-smi query only)."""
    try:
        q = subprocess.run(["nvidia-smi", "-i", "0", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True, text=True).stdout
    except OSError as e:
        return {"name": "unknown", "power_limit": f"nvidia-smi failed: {e}"}
    name, power = (q.strip().split(", ") + ["unknown"])[:2]
    return {"name": name, "power_limit": power}


def bench(logm, steps, warmup):
    t0 = time.perf_counter()
    cs, _ = G.chain_circuit(((1 << logm) - 1) // 3, 3)
    m, n_z, mats = csr_from_r1cs(cs)
    evals = tuple(mont(v) for v in cs.evaluate())
    z, xs, ws = mont(cs.x + cs.w), mont(cs.x), mont(cs.w)
    setup_s = time.perf_counter() - t0
    shape, zv = R1csShape(FIELD_FR, m, n_z, *mats), DeviceVec(FIELD_FR, z)
    rng = B.XorShift128(A.DEFAULT_SEED)
    t0 = time.perf_counter()
    params = setup(shape, cs.l, toxic=[rng.random_field(B.FR) for _ in range(5)])   # the CRS on the device (zksnark.rs:17-127)
    crs_s = time.perf_counter() - t0
    log_n = params.log_n
    prover = Groth16Prover.from_params(params)
    rng = B.XorShift128(bytes(range(1, 17)))
    r, s = rng.random_field(B.FR), rng.random_field(B.FR)
    old = lambda: prover.prove_from_evaluations(log_n, *evals, xs, ws, r, s)
    new = lambda: prover.prove_r1cs(log_n, shape, zv, cs.l, r, s)
    for _ in range(warmup):
        old(), new()
    t_old, t_new = [], []
    for _ in range(steps):   # alternated, so that both see the same state of the shared host
        t_old.append(_wall(old))
        t_new.append(_wall(new))
    same = all((a == b).all() and a.shape == b.shape for a, b in zip(old(), new()))
    t_up = []
    for _ in range(steps):
        t0 = time.perf_counter()
        DeviceVec(FIELD_FR, z).free()
        t_up.append(time.perf_counter() - t0)
    t_eval = []
    for _ in range(max(1, min(steps, 3))):
        t0 = time.perf_counter()
        host = [A.sparse_prod(A.FIELD_FR, m, mat, z) for mat in mats]
        t_eval.append(time.perf_counter() - t0)
    same = same and all((h == e).all() for h, e in zip(host, evals))
    l, el = cs.l, 32
    blind = (2 + 2) * el   # the two blinding jobs of Groth16Prover: [r, 1] and [s, 1]
    rec = {
        "workload": "Groth16 create_proof of the chain circuit (x^3 + x + 5 iterated) after synthesis: prover.rs:32-98",
        "constraints": m, "n_z": n_z, "log_n": log_n, "steps": steps, "warmup": warmup,
        "prove_from_evaluations_ms": min(t_old) * 1e3, "prove_r1cs_ms": min(t_new) * 1e3, "z_upload_ms": min(t_up) * 1e3,
        "host_evaluate_s": min(t_eval), "host_evaluate_cores": 1,
        "host_evaluate_note": "C++ oracle SparseMatrix::prod x 3 (A z, B z, C z), a serial loop on one core; the Python restatement is not timed",
        "same_proof": bool(same),
        "h2d_bytes_per_call": {"prove_from_evaluations": 3 * m * el + 3 * n_z * el + (n_z - l) * el + blind, "prove_r1cs": blind,
                               "z_upload_if_z_is_on_the_host": n_z * el,
                               "note": "old: a, b, c + z for the a, b_g1, b_g2 lanes + aux for l + blinding scalars; new: blinding scalars only"},
        "python_setup_s": setup_s, "device_crs_setup_s": crs_s, "card": card(),
    }
    shape.free(), zv.free(), prover.free(), params.free()
    return rec


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", required=True)
    ap.add_argument("--logm", type=int, nargs="+", default=[16, 20])
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=3)
    a = ap.parse_args()
    os.makedirs(a.out, exist_ok=True)
    k.init()
    with open(os.path.join(a.out, "groth16_r1cs.jsonl"), "w") as f:
        for logm in a.logm:
            rec = bench(logm, a.steps, a.warmup)
            print(json.dumps(rec), flush=True)
            f.write(json.dumps(rec) + "\n")
            f.flush()


if __name__ == "__main__":
    main()
