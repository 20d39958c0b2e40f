"""Groth16 verification and the BN254 pairing on the device (kgr_groth16_verify, kgr_pairing).  One JSON line per measurement, also written to
DIR/groth16_verify.jsonl:
  verify     proofs verified per second at k proofs and n_public public inputs, all valid (the batched check) and with one invalid proof (the
             batched check fails, then every proof is checked on its own); ms = best of --steps calls after --warmup, device events
             (kgr_event_record) around the call
  pairing    kgr_pairing at n pairs: op 0 (n reduced pairings) in pairings/s, op 1 (one product, one final exponentiation) in pairs/s
  roofline   Fq multiplications per Miller loop and per final exponentiation (counted from pairing.cuh, see FQ_MULS), the Fq-multiplication rate of
             kgr_microbench measured in the same run, and the share of that rate the op-0 pairing rate implies
  card       name and power limit of device 0, read in the same run
The proofs are synthetic but valid: the verifying key and the proofs are made from known discrete logarithms (A = a G1, B = b G2,
C = (a b - alpha beta - gamma sum_j x_j u_j) / delta G1 with ic_j = u_j G1), a pool of 256 distinct proofs repeated up to k.
usage: python tools/bench_groth16_verify.py --out DIR [--k 1 64 1024 16384] [--n-public 1 32] [--pairs 65536] [--steps 3] [--warmup 1]"""
import argparse
import json
import os
import random
import subprocess
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))
import kogarashi_b200 as k  # noqa: E402
from groth16_r1cs_util import mont  # noqa: E402
from kogarashi_b200 import msm as M  # noqa: E402
from kogarashi_b200.groth16 import Groth16Verifier  # noqa: E402
from oracle import groth16_ref as G  # noqa: E402

R = G.R
POOL = 256

# Fq multiplications (an Fq2 product = 3, an Fq2 square = 2) per step of pairing.cuh:
#   Fq12 mul 54 (3 Fq6 mul of 6 Fq2 mul), Fq12 sqr 36, cyclotomic sqr 18, line evaluation 43 (2 x 2 for the G1 coordinates + sparse 034 product 39),
#   doubling step 24, addition step 37, pi(Q) 6, -pi^2(Q) 3, Frobenius of an Fq12 15.
#   Miller loop: 63 Fq12 sqr + 64 (doubling + line) + 36 (addition + line) + 2 (addition + line) + 9        = 9605
#   final exponentiation: easy part 216 (+ one Fq inversion), hard part 7 Frobenius + 3 x (62 cyclotomic sqr + 27 mul) + 13 mul + 4 cyclotomic sqr
#   = 105 + 7722 + 702 + 72 = 8601                                                                              = 8817
FQ_MULS = {"miller_loop": 63 * 36 + 64 * (24 + 43) + 36 * (37 + 43) + 2 * (37 + 43) + 9,
           "final_exp": 216 + 7 * 15 + 3 * (62 * 18 + 27 * 54) + 13 * 54 + 4 * 18}


def card():
    try:
        q = subprocess.run(["nvidia-smi", "-i", "0", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True, text=True).stdout
    except OSError as e:
        return {"name": "unknown", "power_limit": f"nvidia-smi failed: {e}"}
    name, power = (q.strip().split(", ") + ["unknown"])[:2]
    return {"name": name, "power_limit": power}


def with_flag(xy):
    return np.concatenate([xy, np.zeros((xy.shape[0], 1), dtype=np.uint64)], axis=1)


def synthetic(n_public, seed):
    """-> verifier, proofs (POOL, 35), inputs (POOL, n_public, 4): a valid pool from known exponents."""
    rng = random.Random(seed)
    al, be, ga, de = (rng.randrange(1, R) for _ in range(4))
    u = [rng.randrange(1, R) for _ in range(n_public + 1)]
    vk_g1 = with_flag(M.fixed_base_mul(k.BN254_G1, mont([al, be, de])))
    vk_g2 = with_flag(M.fixed_base_mul(k.BN254_G2, mont([be, ga, de])))
    ic = M.fixed_base_mul(k.BN254_G1, mont(u))
    a = [rng.randrange(1, R) for _ in range(POOL)]
    b = [rng.randrange(1, R) for _ in range(POOL)]
    xs = [[rng.randrange(R) for _ in range(n_public)] for _ in range(POOL)]
    dinv = pow(de, -1, R)
    c = [(ai * bi - al * be - ga * (u[0] + sum(x * uj for x, uj in zip(xi, u[1:])))) * dinv % R for ai, bi, xi in zip(a, b, xs)]
    A, Bq, C = with_flag(M.fixed_base_mul(k.BN254_G1, mont(a))), with_flag(M.fixed_base_mul(k.BN254_G2, mont(b))), with_flag(M.fixed_base_mul(k.BN254_G1, mont(c)))
    proofs = np.concatenate([A, Bq, C], axis=1)
    inputs = np.stack([mont(x) for x in xs]) if n_public else np.zeros((POOL, 0, 4), dtype=np.uint64)
    ver = Groth16Verifier(vk_g1, vk_g2, (ic, np.zeros(n_public + 1, dtype=np.uint8)))
    return ver, proofs, inputs


def timed(fn, steps, warmup):
    for _ in range(warmup):
        out = fn()
    best = None
    for _ in range(steps):
        M.event_record(0)
        out = fn()
        M.event_record(1)
        ms = M.event_elapsed_ms(0, 1)
        best = ms if best is None else min(best, ms)
    return best, out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", required=True)
    ap.add_argument("--k", type=int, nargs="+", default=[1, 64, 1024, 16384])
    ap.add_argument("--n-public", type=int, nargs="+", default=[1, 32])
    ap.add_argument("--pairs", type=int, default=1 << 16)
    ap.add_argument("--steps", type=int, default=3)
    ap.add_argument("--warmup", type=int, default=1)
    args = ap.parse_args()
    os.makedirs(args.out, exist_ok=True)
    k.init()
    lines = [{"card": card()}]
    rng = np.random.default_rng(5)
    for npub in args.n_public:
        ver, pool, pool_x = synthetic(npub, seed=npub)
        for kk in args.k:
            idx = np.arange(kk) % POOL
            proofs, inputs = pool[idx].copy(), pool_x[idx].copy()
            rho = rng.integers(1, 1 << 63, size=(kk, 2), dtype=np.uint64)
            for case in ("all_valid", "one_invalid"):
                pr = proofs.copy()
                if case == "one_invalid":
                    pr[kk // 2, 26:35] = pool[(kk // 2 + 1) % POOL, 26:35]      # another proof's C
                ms, ok = timed(lambda: ver.verify(pr, inputs, rho if kk >= 2 else None), args.steps, args.warmup)
                expect = kk - (case == "one_invalid")
                assert int(ok.sum()) == expect and (case == "all_valid" or not ok[kk // 2]), (npub, kk, case, int(ok.sum()))
                lines.append({"verify": {"k": kk, "n_public": npub, "case": case, "ms": round(ms, 4), "proofs_per_s": round(kk / (ms * 1e-3), 1)}})
                print(json.dumps(lines[-1]), flush=True)
        ver.free()
    n = args.pairs
    a = [int(x) for x in rng.integers(1, 1 << 62, size=256)]
    g1 = with_flag(M.fixed_base_mul(k.BN254_G1, mont(a)))[np.arange(n) % 256]
    g2 = with_flag(M.fixed_base_mul(k.BN254_G2, mont(a[::-1])))[np.arange(n) % 256]
    ms0, _ = timed(lambda: M.pairing(g1, g2), args.steps, args.warmup)
    ms1, _ = timed(lambda: M.pairing_product(g1, g2), args.steps, args.warmup)
    lines.append({"pairing": {"n": n, "op0_ms": round(ms0, 3), "op0_pairings_per_s": round(n / (ms0 * 1e-3), 1), "op1_ms": round(ms1, 3),
                              "op1_pairs_per_s": round(n / (ms1 * 1e-3), 1)}})
    print(json.dumps(lines[-1]), flush=True)
    mb = M.microbench()
    per_pairing = FQ_MULS["miller_loop"] + FQ_MULS["final_exp"]
    lines.append({"roofline": {"fq_muls": FQ_MULS, "fq_mul_gops": mb["fq_mul_gops"],
                               "op0_share_of_fq_mul_rate": round(n / (ms0 * 1e-3) * per_pairing / (mb["fq_mul_gops"] * 1e9), 4)}})
    print(json.dumps(lines[0]), flush=True)
    print(json.dumps(lines[-1]), flush=True)
    with open(os.path.join(args.out, "groth16_verify.jsonl"), "w") as f:
        for ln in lines:
            f.write(json.dumps(ln) + "\n")


if __name__ == "__main__":
    main()
