"""Groth16 parameter generation on the device (groth16.setup, kgr_groth16_setup, zksnark.rs:17-127) on the chain circuit (the example's
x^3 + x + 5 iterated) at 2^16, 2^20 and 2^22 constraints.  One JSON line per size, also written to DIR/groth16_setup.jsonl:
  setup_ms          best-of-N wall time of setup() after warm-up (all queries G1 and G2 plus the vk, ending in a device synchronise)
  phases_ms         device time per phase of that call (kgr_groth16_setup_last_timing): powers of tau + idft, column index + sums, scalars, and the
                    fixed-base multiplications of a, b_g1, ic, l, h, b_g2 and the vk
  points            points per query, and G1 / G2 fixed-base rates (points / ms of their phases)
  python_exponents_s  (at --python-logm only) the host path the tests used before: crs_exponents in Python integers, then kgr_fixed_base_mul per
                    query with the scalars uploaded, and the points registered again as Bases
  same_as_python    (with python_exponents_s) every query downloaded from setup() equals the points of the host path
  card              name and power limit of device 0, read in the same run
usage: python tools/bench_groth16_setup.py --out DIR [--logm 16 20 22] [--steps 3] [--warmup 1] [--python-logm 16]"""
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
from kogarashi_b200 import msm as M  # noqa: E402
from kogarashi_b200.groth16 import setup  # noqa: E402
from kogarashi_b200.nova import FIELD_FR, R1csShape  # noqa: E402
from oracle import groth16_ref as G  # noqa: E402
from oracle import pyref as B  # noqa: E402

SEED = bytes(range(100, 116))


def card():
    """Name and power limit of device 0, read in the same run as the timings (nvidia-smi query only)."""
    try:
        q = subprocess.run(["nvidia-smi", "-i", "0", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True, text=True).stdout
    except OSError as e:
        return {"name": "unknown", "power_limit": f"nvidia-smi failed: {e}"}
    name, power = (q.strip().split(", ") + ["unknown"])[:2]
    return {"name": name, "power_limit": power}


def python_path(cs):
    """What the tests did before setup(): every CRS exponent in Python integers, the points by kgr_fixed_base_mul, then registered as Bases."""
    t0 = time.perf_counter()
    E, trap, _ = G.crs_exponents(cs, B.XorShift128(SEED))
    t_exp = time.perf_counter() - t0
    out = {}
    for name in ("a", "b_g1", "ic", "l", "h"):
        out[name] = M.fixed_base_mul(k.BN254_G1, mont(E[name]))
    out["b_g2"] = M.fixed_base_mul(k.BN254_G2, mont(E["b_g1"]))
    bases = [M.Bases(k.BN254_G2 if name == "b_g2" else k.BN254_G1, pts) for name, pts in out.items()]
    for b in bases:
        b.free()
    return time.perf_counter() - t0, t_exp, out


def bench(logm, steps, warmup, with_python):
    cs, _ = G.chain_circuit(((1 << logm) - 1) // 3, 3)
    m, n_z, mats = csr_from_r1cs(cs)
    shape = R1csShape(FIELD_FR, m, n_z, *mats)
    rng = B.XorShift128(SEED)
    toxic = [rng.random_field(B.FR) for _ in range(5)]
    for _ in range(warmup):
        setup(shape, cs.l, toxic=toxic).free()
    best, phases, last = None, None, None
    for _ in range(steps):
        if last is not None:
            last.free()
        t0 = time.perf_counter()
        params = setup(shape, cs.l, toxic=toxic)
        t = time.perf_counter() - t0
        if best is None or t < best:
            best, phases = t, M.groth16_setup_timing()
        last = params
    counts = {name: len(getattr(last, name)) for name in ("a", "b_g1", "b_g2", "ic", "l", "h")}
    g1_ms = sum(phases[q] for q in ("a", "b_g1", "ic", "l", "h"))
    rec = {
        "workload": "Groth16 ZkSnark::setup of the chain circuit (x^3 + x + 5 iterated): zksnark.rs:17-127 on the device",
        "constraints": m, "n_z": n_z, "log_n": last.log_n, "nnz": [int(mt[0][-1]) for mt in mats], "steps": steps, "warmup": warmup,
        "setup_ms": best * 1e3, "phases_ms": phases, "points": counts,
        "g1_fixed_base_points_per_ms": sum(counts[q] for q in ("a", "b_g1", "ic", "l", "h")) / g1_ms if g1_ms else None,
        "g2_fixed_base_points_per_ms": counts["b_g2"] / phases["b_g2"] if phases["b_g2"] else None,
        "card": card(),
    }
    if with_python:
        t_py, t_exp, pts = python_path(cs)
        host = last.download()
        rec["python_exponents_s"] = t_py
        rec["python_exponents_integer_part_s"] = t_exp
        rec["same_as_python"] = bool(all((host[name][0] == pts[name]).all() for name in pts))
    last.free()
    shape.free()
    return rec


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", required=True)
    ap.add_argument("--logm", type=int, nargs="+", default=[16, 20, 22])
    ap.add_argument("--steps", type=int, default=3)
    ap.add_argument("--warmup", type=int, default=1)
    ap.add_argument("--python-logm", type=int, nargs="*", default=[16])
    a = ap.parse_args()
    os.makedirs(a.out, exist_ok=True)
    k.init()
    with open(os.path.join(a.out, "groth16_setup.jsonl"), "w") as f:
        for logm in a.logm:
            rec = bench(logm, a.steps, a.warmup, logm in a.python_logm)
            print(json.dumps(rec), flush=True)
            f.write(json.dumps(rec) + "\n")
            f.flush()


if __name__ == "__main__":
    main()
