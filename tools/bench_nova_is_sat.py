"""Nova's relaxed-R1CS check on resident vectors (kgr_nova_is_sat; nova/src/relaxed_r1cs.rs:80-146, reached by RecursiveProof::verify):
(A z) o (B z) = u (C z) + E row by row, plus commit(W) and commit(E), on a relaxed instance made by one device fold (u != 1, E != 0).

  python tools/bench_nova_is_sat.py [log2 constraints ...]        (default 15 18 20; both curves each)

One JSON line per (size, curve).  Timings are wall clock around a call that ends in a synchronise, best of 5 after two warm-up calls:
  relation_ms            ck = NULL: the relation kernel alone (memsets, kernel, 12-byte copy)
  relation_device_ms     the same call between two CUDA events on the library's stream (best of 5)
  full_ms                relation + commit(W) + commit(E), the MSMs on two lanes beside the relation
  commits_sequential_ms  the same two commitments through kgr_pedersen_commit_vec, one after the other
  cpu_ms                 the CPU restatement on all host cores, timed once (it takes seconds): oracle.sparse_prod x 3, oracle.field_op for the
                         products and the compare, oracle.msm for both commitments.  Its commitments are the expected values of the device call,
                         and both verdicts must say satisfied.
relation_bytes: what the relation kernel must read, from the shape: per matrix the row offsets, the coefficients and column indices once, and
32 B per z gather; 32 B of E per row.  relation_gbs = relation_bytes / relation_device_ms.  The 2^15 size is SURVEY's estimate of Nova's
augmented circuit, not a measurement of it.
"""
import json
import os
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))
import kogarashi_b200 as k  # noqa: E402
from kogarashi_b200 import nova  # noqa: E402
from nova_util import chain_r1cs, mont  # noqa: E402
from oracle import oracle as A  # noqa: E402
from oracle import pyref as B  # noqa: E402

W_OFF = 3  # z = (u, x0, out | w)


def best(f, reps=5):
    f()
    f()
    ts = []
    for _ in range(reps):
        t0 = time.perf_counter()
        f()
        ts.append(time.perf_counter() - t0)
    return min(ts) * 1e3


def device():
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True, text=True, timeout=60)
        name, power = [s.strip() for s in out.stdout.splitlines()[0].split(",")]
        return name, power
    except Exception as ex:  # the numbers still stand; the line says the query failed
        return f"unknown ({ex})", "unknown"


def cpu_check(fid, m, mats, z, e, g, curve, cores):
    """The restated reference on the host: the three products, then (A z)_i (B z)_i == u (C z)_i + E_i per row, then both commitments."""
    az, bz, cz = (A.sparse_prod(fid, m, mat, z) for mat in mats)
    u = z[0]
    ok = True
    for i in range(m):
        lhs = A.field_op(fid, "mul", az[i], bz[i])
        rhs = A.field_op(fid, "add", A.field_op(fid, "mul", u, cz[i]), e[i])
        ok &= bool((lhs == rhs).all())
    n_w = min(len(z) - W_OFF, len(g))
    cw = A.to_affine(curve, A.msm(curve, g[:n_w], z[W_OFF:W_OFF + n_w], threads=cores))
    ce = A.to_affine(curve, A.msm(curve, g[:min(m, len(g))], e[:min(m, len(g))], threads=cores))
    return ok, cw, ce


def run(log_m, curve, dev):
    fid = A.SCALAR_FIELD[curve]
    p = B.FQ if fid == A.FIELD_FQ else B.FR
    steps = ((1 << log_m) - 1) // 3
    m, n_z, mats, z1 = chain_r1cs(steps, 3, p)
    z2 = chain_r1cs(steps, 5, p)[3]
    shape = nova.R1csShape(fid, m, n_z, *mats)
    ck = k.PedersenCommitment.new_benchmark(curve, max(m, n_z).bit_length(), seed=11)
    d_z, d_z2 = nova.DeviceVec(fid, mont(z1, p)), nova.DeviceVec(fid, mont(z2, p))
    d_e, d_t = nova.DeviceVec(fid, n=m), nova.DeviceVec(fid, n=m)
    r = mont([0x1F2E3D4C5B6A79880123456789ABCDEF % p], p)[0]
    nova.cross_term_device(shape, d_z, d_z2, t=d_t)
    d_z.fold(d_z2, r)
    d_e.fold(d_t, r)
    z, e = d_z.download(), d_e.download()
    cores = os.cpu_count() or 1
    t0 = time.perf_counter()
    cpu_ok, cw, ce = cpu_check(fid, m, mats, z, e, ck.g.download(), curve, cores)
    cpu_ms = (time.perf_counter() - t0) * 1e3

    rec = {"row": "N4 Nova relaxed-R1CS check (kgr_nova_is_sat)", "device": dev[0], "power_limit": dev[1], "curve": "grumpkin" if curve == A.GRUMPKIN else "bn254_g1",
           "constraints": m, "n_z": n_z, "nnz": [int(mat[0][-1]) for mat in mats], "cores": cores}
    rep = shape.is_sat_relaxed(d_z, d_e, W_OFF, ck=ck, commit_w=cw, commit_e=ce)
    rec["report"] = list(rep)
    rec["sat_device"], rec["sat_cpu"] = bool(rep), cpu_ok
    rec["relation_ms"] = best(lambda: shape.is_sat_relaxed(d_z, d_e, W_OFF))
    dev_ms = []
    for _ in range(7):
        k.event_record(0)
        shape.is_sat_relaxed(d_z, d_e, W_OFF)
        k.event_record(1)
        dev_ms.append(k.event_elapsed_ms(0, 1))
    rec["relation_device_ms"] = min(dev_ms[2:])
    rec["full_ms"] = best(lambda: shape.is_sat_relaxed(d_z, d_e, W_OFF, ck=ck, commit_w=cw, commit_e=ce))
    rec["commits_sequential_ms"] = best(lambda: (d_z.commit(ck, off=W_OFF), d_e.commit(ck)))
    rec["cpu_ms"] = cpu_ms
    gathers = sum(int(mat[0][-1]) for mat in mats)
    rec["relation_bytes"] = sum(4 * (m + 1) + 36 * int(mat[0][-1]) for mat in mats) + 32 * gathers + 32 * m
    rec["relation_gbs"] = rec["relation_bytes"] / rec["relation_device_ms"] / 1e6
    rec["overlap_saves_ms"] = rec["relation_ms"] + rec["commits_sequential_ms"] - rec["full_ms"]
    rec["speedup_vs_cpu"] = cpu_ms / rec["full_ms"]
    for v in (d_z, d_z2, d_e, d_t):
        v.free()
    shape.free()
    return rec


def main():
    sizes = [int(a) for a in sys.argv[1:]] or [15, 18, 20]
    k.init([0])
    dev = device()
    for log_m in sizes:
        for curve in (A.GRUMPKIN, A.BN254_G1):
            rec = run(log_m, curve, dev)
            print(json.dumps(rec), flush=True)
            assert rec["sat_device"] and rec["sat_cpu"], rec


if __name__ == "__main__":
    main()
