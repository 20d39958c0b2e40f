"""Measurement harness for the "next" rows N2 (Fr NTT) and N1 (G1 side of the Groth16 prover) — not the headline bench.
Uses the oracle exactly like bench.py does: as the checker and as the CPU baseline timed on the host cores.
Writes gpurun_out/next_rows_<tag>.json."""
import json
import os
import sys
import time

import numpy as np

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import kogarashi_b200 as k  # noqa: E402
from kogarashi_b200 import msm as M  # noqa: E402
from kogarashi_b200.groth16 import Groth16Prover  # noqa: E402
from oracle import groth16_ref as G  # noqa: E402
from oracle import oracle as A  # noqa: E402
from oracle import pyref as B  # noqa: E402

IMAD_PEAK = 148 * 64 * 1.965e9


def bench_ntt(logn, out):
    import torch
    n = 1 << logn
    x = A.random_field(A.FIELD_FR, n, seed=bytes(range(16)))
    f = k.Fft(logn)
    d = torch.from_numpy(x.view(np.int64)).cuda()
    torch.cuda.synchronize()
    f.transform_device("dft", d.data_ptr())
    best = min(_timed(lambda: f.transform_device("dft", d.data_ptr())) for _ in range(10))
    # parity at this size: device dft == restated reference dft
    t0 = time.perf_counter()
    exp, _ = A.fft(logn, "dft", x)
    cpu_s = time.perf_counter() - t0
    got = f.dft(x)
    e2e = min(_wall(lambda: f.dft(x)) for _ in range(3))
    butterflies = n // 2 * logn
    rec = {"row": "N2 Fr NTT (groth16/src/fft.rs dft)", "log_n": logn, "device_ms": best, "melem_per_s": n / best / 1e3,
           "bit_exact_with_oracle": bool((got == exp).all()),
           "e2e_host_buffers_ms": e2e * 1e3, "cpu_baseline": {"seconds": cpu_s, "cores": 1, "kind": "port", "melem_per_s": n / cpu_s / 1e6},
           "roofline": {"bound": "imad", "algorithmic_imads": butterflies * 264, "achieved_T_per_s": butterflies * 264 / (best * 1e-3) / 1e12,
                        "peak_T_per_s": IMAD_PEAK / 1e12, "frac": butterflies * 264 / (best * 1e-3) / IMAD_PEAK,
                        "hbm_gbs_algorithmic": 64 * n / (best * 1e-3) / 1e9,
                        "note": "one 254-bit Montgomery product (264 IMAD) per butterfly, n/2*log2(n) butterflies; 64 B/element algorithmic traffic: multiplier-bound, not HBM-bound"}}
    out.append(rec)
    print(json.dumps(rec), flush=True)


def _timed(fn):
    fn()
    return k.last_timing(0)[0]["total"]


def _wall(fn):
    t0 = time.perf_counter()
    fn()
    return time.perf_counter() - t0


def bench_groth16(logm, out, steps=5, warmup=5, cpu_steps=1, cpu_warmup=0):
    """GPU: best of `steps` proofs after `warmup` warm-up proofs; CPU baseline: best of `cpu_steps` runs after `cpu_warmup`.  Returns the
    last proof (A, B, C as affine limb arrays) of the default (not precomputed) prover."""
    t0 = time.perf_counter()
    cs, _ = G.chain_circuit(((1 << logm) - 1) // 3, 3)
    E, trap, uvw = G.crs_exponents(cs, B.XorShift128(A.DEFAULT_SEED))
    setup_s = time.perf_counter() - t0
    mont = lambda vals: np.array([B.int_to_limbs(B.to_mont(v, B.FR)) for v in vals], dtype=np.uint64).reshape(-1, 4)

    def points(exps):
        return M.fixed_base_mul(k.BN254_G1, mont(exps)), np.array([1 if e == 0 else 0 for e in exps], dtype=np.uint8)

    def points_g2(exps):
        return M.fixed_base_mul(k.BN254_G2, mont(exps)), np.array([1 if e == 0 else 0 for e in exps], dtype=np.uint8)

    vk = points([trap["delta"], trap["alpha"], trap["beta"]])[0]
    vk2 = points_g2([trap["delta"], trap["beta"]])[0]
    crs = [points(E[name]) for name in ("a", "b_g1", "h", "l")]
    crs_g2 = points_g2(E["b_g1"])  # b_g2: the exponents of b_g1 on the G2 generator (zksnark.rs:177-185)
    a_ev, b_ev, c_ev = (mont(v) for v in cs.evaluate())
    xs, ws = mont(cs.x), mont(cs.w)
    rng = B.XorShift128(bytes(range(1, 17)))
    r, s = rng.random_field(B.FR), rng.random_field(B.FR)
    res, proof = {}, None
    for pre in (False, True):
        prover = Groth16Prover(vk[0], vk[1], vk[2], *crs[0], *crs[1], *crs[2], *crs[3], vk2[0], vk2[1], *crs_g2, precompute=pre)
        for _ in range(warmup):   # warm-up: lanes, NTT tables, workspaces
            prover.prove_from_evaluations(E["k"], a_ev, b_ev, c_ev, xs, ws, r, s)
        wall = min(_wall(lambda: prover.prove_from_evaluations(E["k"], a_ev, b_ev, c_ev, xs, ws, r, s)) for _ in range(steps))
        Ap, Bp, Cp, q = prover.prove_from_evaluations(E["k"], a_ev, b_ev, c_ev, xs, ws, r, s)
        res["precomputed" if pre else "normal"] = wall * 1e3
        if not pre:
            proof = (Ap, Bp, Cp)
        prover.free()
    q_int = [B.from_mont(B.limbs_to_int(x), B.FR) for x in q]
    a_exp, b_exp, c_exp, pairing_ok = G.expected_exponents(trap, uvw, cs.x, cs.w, q_int, E["n"], r, s)
    enc = lambda aff: np.asarray(aff[:-1], dtype="<u8").tobytes() + bytes([int(aff[-1])])
    ok = (pairing_ok and enc(Ap) == G.encode_g1(G.G1.mul(G.G1.g, a_exp)) and enc(Cp) == G.encode_g1(G.G1.mul(G.G1.g, c_exp))
          and enc(Bp) == G.encode_g2(G.g2_mul(G.G2_GEN, b_exp)))
    # CPU baseline: the same work with the restated reference code (7 FFTs + the six G1 and two G2 MSMs of prover.rs:51-65)
    cores = os.cpu_count() or 1
    l = cs.l
    best = None
    for it in range(cpu_warmup + cpu_steps):
        t0 = time.perf_counter()
        q_ref, n_ref = A.groth16_h(E["k"], a_ev, b_ev, c_ev)
        fft_s = time.perf_counter() - t0
        t0 = time.perf_counter()
        for pts_inf, sc in ((crs[2], q_ref[:n_ref]), (crs[3], ws), (crs[0], xs), ((crs[0][0][l:], crs[0][1][l:]), ws), (crs[1], xs), ((crs[1][0][l:], crs[1][1][l:]), ws)):
            A.msm(A.BN254_G1, pts_inf[0], sc, inf=pts_inf[1], threads=cores)
        for pts_inf, sc in ((crs_g2, xs), ((crs_g2[0][l:], crs_g2[1][l:]), ws)):
            A.msm(A.BN254_G2, pts_inf[0], sc, inf=pts_inf[1], threads=cores)
        msm_s = time.perf_counter() - t0
        if it >= cpu_warmup and (best is None or fft_s + msm_s < best[0] + best[1]):
            best = (fft_s, msm_s)
    fft_s, msm_s = best
    rec = {"row": "N1+N3 Groth16 create_proof after witness generation (7 FFTs + six G1 MSMs + two G2 MSMs + assembly of A, B, C)",
           "constraints": cs.m, "log_n": E["k"], "gpu_wall_ms": res, "checked_against_discrete_logs": bool(ok),
           "h_bit_exact_with_oracle": bool(q.shape[0] == n_ref and (q == q_ref[:n_ref]).all()),
           "cpu_baseline": {"fft_seconds": fft_s, "msm_seconds": msm_s, "total_seconds": fft_s + msm_s, "cores": cores, "kind": "port",
                            "note": "restated reference FFTs (recursion halves forked like rayon::join, fft.rs:180-183) + the eight reference-algorithm MSMs on all cores"},
           "speedup_vs_cpu_baseline": {m: (fft_s + msm_s) * 1e3 / v for m, v in res.items()}, "setup_python_s": setup_s}
    out.append(rec)
    print(json.dumps(rec), flush=True)
    return proof


def bench_g2(logn, out):
    """N3: one G2 MSM (prover.rs:64-65) with device-resident bases, host scalars; CPU baseline = the reference algorithm over Fq2."""
    n = 1 << logn
    bases, ks = k.Bases.generate(k.BN254_G2, n, seed=5, return_scalars=True)
    sc = A.random_field(A.FIELD_FR, n, seed=bytes(range(16)))
    k.msm_curve_addition(bases, sc)
    best, phases, shape = None, None, None
    for _ in range(5):
        got = k.msm_curve_addition(bases, sc)
        t, sh = k.last_timing(0)
        dev = t["total"] - t["h2d"]
        if best is None or dev < best:
            best, phases, shape = dev, t, sh
    wall = min(_wall(lambda: k.msm_curve_addition(bases, sc)) for _ in range(3)) * 1e3
    cores = os.cpu_count() or 1
    ns = min(n, 1 << 18)
    pts = bases.download(0, ns)
    t0 = time.perf_counter()
    cpu = A.msm(A.BN254_G2, pts, sc[:ns], threads=cores)
    cpu_s = time.perf_counter() - t0
    same = bool((A.to_affine(A.BN254_G2, cpu) == k.to_affine(k.BN254_G2, k.msm_curve_addition(bases, sc[:ns]))).all()) if ns < n else \
        bool((A.to_affine(A.BN254_G2, cpu) == k.to_affine(k.BN254_G2, got)).all())
    rec = {"row": "N3 BN254 G2 MSM", "log_n": logn, "device_ms": best, "mpoints_per_s": n / best / 1e3, "e2e_registered_ms": wall, "shape": shape,
           "phases_ms": {a: round(b, 3) for a, b in phases.items()}, "bit_exact_with_oracle_on_sample": same,
           "cpu_baseline": {"mpoints_per_s": ns / cpu_s / 1e6, "cores": cores, "kind": "port", "sample": f"one MSM over the first 2^{int(np.log2(ns))} pairs, {cpu_s:.2f} s"},
           "roofline": {"bound": "imad", "note": "madd over Fq2 = 8 products x 3 + 2 squares x 2 = 28 Fq multiplications (10 on G1)"}}
    rec["speedup_vs_cpu_baseline"] = rec["mpoints_per_s"] / rec["cpu_baseline"]["mpoints_per_s"]
    out.append(rec)
    print(json.dumps(rec), flush=True)
    bases.free()


def bench_nova(steps, out):
    """N4: Nova's compute_cross_term + commit(T) + witness fold (nova/src/prover.rs:33-47) on the chained x^3 + x + 5 circuit over Fq
    (GrumpkinDriver): T stays on the device for the commitment MSM.  CPU baseline = the restated reference loops (single thread, like the
    reference) and, for the commitment, the reference's naive fold of scalar multiplications (pedersen.rs:15-20) on a bounded sample."""
    sys.path.insert(0, os.path.join(os.path.dirname(os.path.abspath(__file__)), "..", "tests"))
    from nova_util import chain_r1cs
    from kogarashi_b200 import nova
    p, fid, curve = B.FQ, A.FIELD_FQ, k.GRUMPKIN
    t0 = time.perf_counter()
    m, n_z, mats, z1_int = chain_r1cs(steps, 3, p)
    z2_int = chain_r1cs(steps, 4, p)[3]
    R256 = 1 << 256
    to_m = lambda vals: np.frombuffer(b"".join((v * R256 % p).to_bytes(32, "little") for v in vals), dtype=np.uint64).reshape(-1, 4).copy()
    z1, z2 = to_m(z1_int), to_m(z2_int)
    build_s = time.perf_counter() - t0
    nnz = [int(mt[0][-1]) for mt in mats]
    shape = nova.R1csShape(fid, m, n_z, *mats)
    ck = k.Bases.generate(curve, m, seed=9)
    shape.cross_term(z1, z2, ck=ck, want_t=False)
    best = None
    for _ in range(5):
        w0 = time.perf_counter()
        t_dev, commit = shape.cross_term(z1, z2, ck=ck, want_t=False)
        wall = (time.perf_counter() - w0) * 1e3
        tm = shape.last_timing()
        if best is None or wall < best[0]:
            best = (wall, tm)
    t_host, commit2 = shape.cross_term(z1, z2, ck=ck)
    rm = to_m([0x0123456789ABCDEF0123456789ABCDEF])[0]
    fold_wall = min(_wall(lambda: nova.vec_fold(fid, z1, z2, rm)) for _ in range(3)) * 1e3
    # CPU restatement
    t0 = time.perf_counter()
    t_ref = A.cross_term(fid, m, *mats, z1, z2)
    cpu_ct = time.perf_counter() - t0
    t0 = time.perf_counter()
    f_ref = A.vec_fold(fid, z1, z2, rm)
    cpu_fold = time.perf_counter() - t0
    ns = min(m, 1 << 11)
    pts = ck.download(0, ns)
    t0 = time.perf_counter()
    A.pedersen_commit(curve, pts, t_ref[:ns])
    cpu_commit_per_elem = (time.perf_counter() - t0) / ns
    cores = os.cpu_count() or 1
    t0 = time.perf_counter()
    ns2 = min(m, 1 << 18)
    msm_ref = A.msm(curve, ck.download(0, ns2), t_ref[:ns2], threads=cores)
    cpu_msm_rate = ns2 / (time.perf_counter() - t0)
    ok = bool((t_host == t_ref).all() and (nova.vec_fold(fid, z1, z2, rm) == f_ref).all() and (commit == commit2).all())
    if ns2 == m:
        ok = ok and bool((A.to_affine(curve, msm_ref) == commit).all())
    total_nnz = sum(nnz)
    rec = {"row": "N4 Nova compute_cross_term + commit(T) + fold (Fq / Grumpkin)", "constraints": m, "z_len": n_z, "nnz": nnz,
           "gpu_ms": {"call_wall": best[0], "h2d_z1_z2": best[1]["h2d"], "cross_term_kernel": best[1]["cross_term"], "commit_msm": best[1]["commit"],
                      "vec_fold_call_wall_host_buffers": fold_wall},
           "cross_term_algorithmic": {"bytes": total_nnz * (36 + 64) + m * 32, "gb_per_s": (total_nnz * 100 + m * 32) / (best[1]["cross_term"] * 1e-3) / 1e9,
                                      "note": "per non-zero: 32 B coefficient + 4 B column + two 32 B z gathers; per row 32 B of T written; bound: HBM / L2 gathers"},
           "bit_exact_with_oracle": ok,
           "cpu_baseline": {"cross_term_seconds": cpu_ct, "fold_seconds": cpu_fold, "kind": "port", "cores": 1,
                            "commit_reference_naive_seconds_extrapolated": cpu_commit_per_elem * m,
                            "commit_sample": f"pedersen.rs:15-20 fold of scalar multiplications over the first {ns} elements, extrapolated linearly",
                            "commit_as_reference_msm_seconds": m / cpu_msm_rate, "msm_cores": cores},
           "python_build_s": build_s}
    rec["speedup_cross_term_kernel_vs_cpu"] = cpu_ct * 1e3 / best[1]["cross_term"]
    out.append(rec)
    print(json.dumps(rec), flush=True)
    shape.free()
    ck.free()


def main():
    tag = sys.argv[1] if len(sys.argv) > 1 else "r01"
    os.makedirs("gpurun_out", exist_ok=True)
    k.init([0])
    out = []
    only = sys.argv[2] if len(sys.argv) > 2 else None
    if only == "nova":
        for steps in (21845, 349525):
            bench_nova(steps, out)
        json.dump(out, open(f"gpurun_out/next_rows_{tag}.json", "w"), indent=1)
        return
    for logn in (16, 20, 22):
        bench_ntt(logn, out)
    for logn in (16, 20):
        bench_g2(logn, out)
    for logm in (12, 16):
        bench_groth16(logm, out)
    for steps in (21845, 349525):   # 2^16 and 2^20 constraints
        bench_nova(steps, out)
    json.dump(out, open(f"gpurun_out/next_rows_{tag}.json", "w"), indent=1)


if __name__ == "__main__":
    main()
