#!/usr/bin/env python
"""bench.py — BN254 G1 MSM throughput (Mpoints/s) on B200 and Groth16 prove latency, the metric BASELINE.json names.

  python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--quick] [--dump-outputs DIR]
  python -m torch.distributed.run --nnodes=1 --nproc-per-node N --master-addr 127.0.0.1 --master-port P bench.py --gpus N ...

The run writes nothing into the source tree (it may be read-only): no bytecode, and the CPU oracle's -march=native build goes to a temp dir.
--dump-outputs DIR writes what the timed path computed in its last step, as affine points: the headline MSM's result (DIR/msm_affine.npy) or,
with --workload groth16, the proof (DIR/proof_{a,b,c}.npy), so that two builds can be compared output for output on the same seeded inputs.

Inputs (both arms, every N): bases P_i = k_i * G with k_i = from_u512(splitmix64 stream of (BASE_SEED, i)) — generated on the device by
kgr_bases_generate_at in our arm and by the oracle's restatement of the same stream in the reference arm — and scalars s_i drawn by numpy
in blocks of 2^18 (seed (SCALAR_SEED, block)), uniform below the modulus.  Global index i: a shard of the vector is the same numbers
whatever the sharding.

N = 1   workload = BASELINE configs[1]: one 2^20-point BN254 G1 MSM.
        `value`        bases and scalars resident in HBM, device time from the engine's CUDA events, L2 flushed between steps
        `e2e`          kgr_msm_oneshot = msm_curve_addition on host slices: points AND scalars uploaded from pinned memory in every call
        `e2e_pageable` the same call with both vectors in ordinary (pageable) memory, as a Rust Vec or a numpy array is; `e2e_registered`: scalars only
        `roofline`     integer-multiply roofline (SURVEY.md 8d), whole pipeline + the dominant kernel; `cpu_baseline` = oracle on the host cores
        `north_star`   2^24 points (the north-star size): device time, roofline, e2e, FULL comparison with the restated reference MSM
        `grumpkin_2p20`, `groth16_2p16`   BASELINE configs[2] and [3]; `g2_2p18` the G2 query's MSM (row N3); `ntt_2p20` the Fr transform (row N2); `nova_ivc_step_32k` Nova's folding vector work (row N4, tools/bench_ivc_step.py in a child process);  `strong_scaling_base`   2^26 / 2^24 points on this one GPU
N > 1   workload = BASELINE configs[4], STRONG scaling: ONE 2^26-point MSM sharded evenly over the N ranks (contiguous shards, no data-path
        collective); a step = every rank's MSM + all_gather of one 96-byte point per rank + the host sum on rank 0, timed by wall clock between
        barriers.  `value`: scalars resident in HBM; `e2e`: scalars uploaded from pinned host memory every step (bases registered).
        `checksum_ok`: the combined point equals (sum k_i s_i) * G, with sum k_i s_i accumulated per rank by the oracle and all-gathered.
        `weak_scaling` keeps round 1's figure (independent 2^20-point MSMs per GPU); `inprocess` is ONE kgr_msm call over kgr_init([0..N-1])
        issued by rank 0 while the other ranks wait on a CPU barrier.
--impl reference   the reference's CPU algorithm (C++ restatement in oracle/: rustc / cargo are absent) on all host cores, same inputs.
"""
import argparse
import json
import math
import os
import statistics
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

FR_TOP = 0x30644E72E131A029  # top limb of r (bn254/src/fr.rs:11-16) = top limb of q (fq.rs:10-15)
UNIT = "Mpoints/s"
BASE_SEED, SCALAR_SEED, SC_BLOCK = 1000, 77, 1 << 18
CURVE_IDS = {"bn254_g1": 0, "grumpkin": 1, "bn254_g2": 2}
METRICS = {"bn254_g1": "bn254_g1_msm_throughput", "grumpkin": "grumpkin_msm_throughput", "bn254_g2": "bn254_g2_msm_throughput"}
IMAD_PEAK_T = 148 * 64 * 1.965e9 / 1e12  # nominal; kgr_microbench measured 18.4-18.5 T mad.lo.u32/s on this pool (profiles/r01_microbench.md)


def kernel_sources_sha():
    """sha256 over the CUDA kernel sources (not the host engine): ties an ncu capture in profiles/ncu_traffic.json to the kernels it measured."""
    import hashlib
    h = hashlib.sha256()
    d = os.path.join(ROOT, "kogarashi_b200", "csrc")
    for name in sorted(os.listdir(d)):
        if name.endswith(".cuh") or (name.startswith("kernels_") and name.endswith(".cu")):
            h.update(name.encode())
            h.update(open(os.path.join(d, name), "rb").read())
    return h.hexdigest()[:16]


def measured_traffic(n, curve_name):
    """DRAM bytes (read + write) of the dominant phase per launch from the committed `ncu --set full` capture — only for the workload it was
    taken on (2^20-point BN254 G1 / Grumpkin MSM: same kernels, same sizes) and only while the kernel sources still hash to the captured ones;
    otherwise None (a stale constant is worse than no number)."""
    try:
        t = json.load(open(os.path.join(ROOT, "profiles", "ncu_traffic.json")))
        if n == (1 << 20) and curve_name in ("bn254_g1", "grumpkin") and t.get("kernel_sources_sha") == kernel_sources_sha():
            sort_bytes = sum(v["bytes"] for kname, v in t["per_kernel_dram_bytes"].items() if kname.startswith("k_sort_"))
            return t["accumulate_phase_dram_bytes"], t["capture"], sort_bytes
    except Exception:
        pass
    return None, None, None


def ref_window_bits(n):  # groth16/src/msm.rs:7-14
    if n < 4:
        return 1
    if n < 32:
        return 3
    return (n.bit_length() * 69) // 100 + 2


def algorithmic_imads(n, curve_name="bn254_g1", dominant_only=False):
    """SURVEY.md 8(d): A(n) = n*W + 2*(2^c - 1)*W point adds with the reference's c and W = ceil(254/c); 11 field multiplications per add
    (reference mixed add 9M+2S; 31 over Fq2); 264 32-bit IMADs per multiplication.  dominant_only: the n*W bucket additions alone."""
    c = ref_window_bits(n)
    W = math.ceil(254 / c)
    adds = n * W + (0 if dominant_only else 2 * ((1 << c) - 1) * W)
    return adds * (31 if curve_name == "bn254_g2" else 11) * 264


def scalars_range(first, n):
    """s_i for global indices [first, first + n): (n, 4) uint64 Montgomery limbs (any value below the modulus is a valid residue)."""
    out = np.empty((n, 4), dtype=np.uint64)
    pos = 0
    b = first // SC_BLOCK
    while pos < n:
        rng = np.random.default_rng([SCALAR_SEED, b])
        blk = rng.integers(0, 1 << 63, size=(SC_BLOCK, 4), dtype=np.uint64) * np.uint64(2) + rng.integers(0, 2, size=(SC_BLOCK, 4), dtype=np.uint64)
        blk[:, 3] = rng.integers(0, FR_TOP, size=SC_BLOCK, dtype=np.uint64)  # top limb < top limb of the modulus  =>  value < modulus
        lo = max(first, b * SC_BLOCK) - b * SC_BLOCK
        take = min(SC_BLOCK - lo, n - pos)
        out[pos:pos + take] = blk[lo:lo + take]
        pos += take
        b += 1
    return out


def workload_config(args, world):
    """The `config` object: identical text in both arms for the same command line."""
    if args.workload == "groth16":
        return {"workload": f"Groth16 create_proof after witness generation, chained x^3 + x + 5 circuit, 2^{args.logm} constraints"}
    if world > 1:
        return {"workload": f"{args.curve} MSM, ONE 2^{args.strong_logn}-point MSM sharded over {world} GPUs (strong scaling, BASELINE configs[4])",
                "points_total": 1 << args.strong_logn, "inputs": "bases k_i*G (splitmix64 stream, seed 1000), uniform scalars (numpy blocks, seed 77)"}
    return {"workload": f"{args.curve} MSM, 2^{args.logn} points on 1 GPU (BASELINE configs[1])", "points_total": 1 << args.logn,
            "inputs": "bases k_i*G (splitmix64 stream, seed 1000), uniform scalars (numpy blocks, seed 77)"}


class ClockSampler:
    """SM clock / throttle reasons sampled through NVML in a thread while the timed region runs
    (the same counters `nvidia-smi --query-gpu=clocks.sm,clocks_event_reasons.*` prints)."""

    def __init__(self, gpu_index, period_s=0.004):
        self.gpu, self.period, self.rows, self.stop_flag, self.thread, self.h = gpu_index, period_s, [], False, None, None
        try:
            import pynvml
            self.nv = pynvml
            pynvml.nvmlInit()
            self.h = pynvml.nvmlDeviceGetHandleByIndex(gpu_index)
        except Exception:
            self.nv = None

    def _loop(self):
        nv = self.nv
        while not self.stop_flag:
            try:
                sm = nv.nvmlDeviceGetClockInfo(self.h, nv.NVML_CLOCK_SM)
                reasons = nv.nvmlDeviceGetCurrentClocksEventReasons(self.h) if hasattr(nv, "nvmlDeviceGetCurrentClocksEventReasons") \
                    else nv.nvmlDeviceGetCurrentClocksThrottleReasons(self.h)
                self.rows.append((sm, reasons))
            except Exception:
                pass
            time.sleep(self.period)

    def start(self):
        if self.nv is None or self.h is None:
            return
        self.thread = threading.Thread(target=self._loop, daemon=True)
        self.thread.start()

    def stop(self):
        self.stop_flag = True
        if self.thread:
            self.thread.join(timeout=1.0)
        if self.nv is None or not self.rows:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": [], "samples": 0}
        nv = self.nv
        smax = nv.nvmlDeviceGetMaxClockInfo(self.h, nv.NVML_CLOCK_SM)
        names = {"hw_slowdown": 0x8, "sw_power_cap": 0x4, "hw_thermal_slowdown": 0x40, "sw_thermal_slowdown": 0x20, "hw_power_brake_slowdown": 0x80}
        seen = set()
        for _, r in self.rows:
            for name, bit in names.items():
                if r & bit:
                    seen.add(name)
        sm = [x for x, _ in self.rows]
        return {"sm_mhz": statistics.median(sm), "sm_max_mhz": smax, "reasons": sorted(seen), "samples": len(sm)}


# ---- checker side (oracle): only used to verify results and as the CPU baseline -----------------------------------------------------------
def expected_from_dot(curve, dot_mont):
    """(sum k_i s_i) * G as an affine point, by the oracle's double-and-add on the generator."""
    from oracle import oracle as A
    g = A.generator(curve)
    one = A.field_op(A.FIELD_FR if curve == A.GRUMPKIN else A.FIELD_FQ, "to_mont", np.array([1, 0, 0, 0], dtype=np.uint64))
    z = np.concatenate([one, np.zeros(4, dtype=np.uint64)]) if curve == A.BN254_G2 else one  # Z = 1 (in Fq2: 1 + 0u)
    return A.to_affine(curve, A.scalar_point(curve, np.concatenate([g, z]), dot_mont))


def dot_of_shard(curve, ks, sc):
    from oracle import oracle as A
    return A.field_dot(A.SCALAR_FIELD[curve], ks, sc)


def cpu_msm(curve, pts, sc, threads):
    from oracle import oracle as A
    t0 = time.perf_counter()
    out = A.msm(curve, pts, sc, threads=threads)
    return time.perf_counter() - t0, out


# ---- one single-GPU measurement ------------------------------------------------------------------------------------------------------------
def measure_single(k, torch, curve_name, logn, steps, warmup, local_rank, flush, first=0, seed=BASE_SEED, want_e2e=True, full_cpu=False, cpu_sample_logn=None,
                   sampler=None, want_precompute=False):
    """value / e2e / roofline / checksum of one MSM of 2^logn points on the current GPU.  Returns (record, device_ms_per_step, affine result)."""
    from oracle import oracle as A  # checker only
    curve = CURVE_IDS[curve_name]
    n = 1 << logn
    pt_bytes = 128 if curve == k.BN254_G2 else 64
    bases, ks = k.Bases.generate(curve, n, seed=seed, return_scalars=True, first=first)
    sc = scalars_range(first, n)
    sc_pinned = torch.from_numpy(sc.view(np.int64)).pin_memory()
    d_sc = sc_pinned.cuda(non_blocking=False)
    torch.cuda.synchronize()
    for _ in range(warmup):
        out = k.msm_device(bases, d_sc.data_ptr(), n)
    if sampler:
        sampler.start()
    launches0 = k.launch_count(0)
    dev_ms, phases = 0.0, {}
    t_wall0 = time.perf_counter()
    for _ in range(steps):
        flush.zero_()
        torch.cuda.synchronize()
        out = k.msm_device(bases, d_sc.data_ptr(), n)
        ms, shape = k.last_timing(0)
        dev_ms += ms["total"]
        for key, v in ms.items():
            phases[key] = phases.get(key, 0.0) + v / steps
    torch.cuda.synchronize()
    wall_ms = (time.perf_counter() - t_wall0) * 1e3
    clocks = sampler.stop() if sampler else None
    launches = k.launch_count(0) - launches0
    ms_per_step = dev_ms / steps
    aff = k.to_affine(curve, out)
    rec = {"points": n, "clocks": clocks, "ms_per_step": ms_per_step, "value": n / ms_per_step / 1e3, "unit": UNIT, "steps": steps, "warmup": warmup, "phases_ms": phases, "shape": shape,
           "wall_ms_per_step": wall_ms / steps, "gpu_launches": launches}
    # ---- roofline --------------------------------------------------------------------------------------------------------------------------
    alg = algorithmic_imads(n, curve_name)
    g2 = curve_name == "bn254_g2"
    exec_imads = (n * shape["W"] * (28 if g2 else 10) + 2 * shape["W"] * shape["B"] * (40 if g2 else 14)) * 264
    acc_alg = algorithmic_imads(n, curve_name, dominant_only=True)
    sort_ms = phases.get("count", 0) + phases.get("scan", 0) + phases.get("fill", 0)
    sort_bytes = n * 32 + n * shape["W"] * 4  # scalars read once + one 4-byte entry written per (scalar, window)
    rec["roofline"] = {
        "bound": "imad", "achieved": alg / (ms_per_step * 1e-3) / 1e12, "peak": IMAD_PEAK_T, "unit": "T IMAD/s", "frac": alg / (ms_per_step * 1e-3) / 1e12 / IMAD_PEAK_T,
        "traffic": measured_traffic(n, curve_name)[0], "traffic_source": measured_traffic(n, curve_name)[1],
        "kernel": "whole pipeline (all kernels of one MSM); dominant kernel below; traffic = DRAM bytes of the dominant phase per launch (ncu), null when the kernels changed since the capture",
        "algorithmic_imads_per_launch": alg,
        "peak_source": "148 SM x 64 IMAD/clk x 1.965 GHz; kgr_microbench measured 18.4-18.5 T mad.lo.u32/s on this pool (MEASURED_PEAKS.json has no integer figure)",
        "executed": {"imads_per_launch": exec_imads, "frac": exec_imads / (ms_per_step * 1e-3) / 1e12 / IMAD_PEAK_T,
                     "note": "additions this implementation issues (signed digits, its own window size, XYZZ formulas) x products per addition x 264"},
        "dominant_kernel": {"name": "accumulate phase: batched-affine levels (k_affine_den / k_batch_inv / k_affine_add) + k_accumulate", "ms": phases.get("accumulate"), "algorithmic_imads": acc_alg,
                            "frac": acc_alg / (phases["accumulate"] * 1e-3) / 1e12 / IMAD_PEAK_T if phases.get("accumulate") else None},
        "sort": {"kernels": "k_sort_digits + k_sort_scan + k_sort_partition + k_sort_buckets (or k_count + scan + k_fill below 2^21 entries)", "bound": "hbm", "ms": sort_ms,
                 "algorithmic_bytes": sort_bytes, "achieved_gbs": sort_bytes / (sort_ms * 1e-3) / 1e9 if sort_ms else None},
        "hbm": {"achieved_gbs": (pt_bytes + 32) * n / (ms_per_step * 1e-3) / 1e9, "note": f"{pt_bytes + 32} B/point algorithmic traffic; the path is multiply-bound, not HBM-bound"}}
    sort_traffic = measured_traffic(n, curve_name)[2]
    if sort_traffic and sort_ms:  # what the two partition passes really move (ncu): digit words, payloads and fine bytes are written and read again
        rec["roofline"]["sort"]["traffic"] = sort_traffic
        rec["roofline"]["sort"]["traffic_gbs"] = sort_traffic / (sort_ms * 1e-3) / 1e9
    try:
        peaks = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
        rec["roofline"]["hbm"]["peak_gbs"] = peaks.get("hbm_gbs")
        if sort_ms and peaks.get("hbm_gbs"):
            rec["roofline"]["sort"]["frac"] = rec["roofline"]["sort"]["achieved_gbs"] / peaks["hbm_gbs"]
            if sort_traffic:
                rec["roofline"]["sort"]["frac_of_traffic"] = rec["roofline"]["sort"]["traffic_gbs"] / peaks["hbm_gbs"]
    except Exception:
        pass
    # ---- e2e: host buffers through the reference-facing calls ----------------------------------------------------------------------------
    if want_e2e:
        pts_host = bases.download()
        pts_pinned = torch.from_numpy(pts_host.view(np.int64)).pin_memory()
        e2e_steps = max(2, min(steps, 10))
        for _ in range(2):
            k.msm_oneshot_ptr(curve, pts_pinned.data_ptr(), n, sc_pinned.data_ptr(), n)
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        for _ in range(e2e_steps):
            out_e2e = k.msm_oneshot_ptr(curve, pts_pinned.data_ptr(), n, sc_pinned.data_ptr(), n)
        e2e_ms = (time.perf_counter() - t0) * 1e3 / e2e_steps
        k.msm_host_ptr(bases, sc_pinned.data_ptr(), n)
        t0 = time.perf_counter()
        for _ in range(e2e_steps):
            out_reg = k.msm_host_ptr(bases, sc_pinned.data_ptr(), n)
        reg_ms = (time.perf_counter() - t0) * 1e3 / e2e_steps
        assert (k.to_affine(curve, out_e2e) == aff).all() and (k.to_affine(curve, out_reg) == aff).all()
        pieces = max(1, min(4, n >> 19))
        rec["e2e"] = {"value": n / e2e_ms / 1e3, "unit": UNIT, "h2d_bytes_per_step": (pt_bytes + 32) * n, "d2h_bytes_per_step": pieces * shape["W"] * 2 * pt_bytes,
                      "ms_per_step": e2e_ms, "steps": e2e_steps, "call": "kgr_msm_oneshot (points + scalars uploaded from pinned host memory every call)"}
        rec["e2e_registered"] = {"value": n / reg_ms / 1e3, "unit": UNIT, "h2d_bytes_per_step": 32 * n, "d2h_bytes_per_step": shape["W"] * 2 * pt_bytes,
                                 "ms_per_step": reg_ms, "call": "kgr_msm (bases registered once, scalars uploaded every call)"}
        if n <= (1 << 22):  # the same call from ORDINARY (pageable) memory — what a Rust Vec or a numpy array is: staged through pinned slots by host threads
            sc_page = np.ascontiguousarray(sc)
            for _ in range(2):
                k.msm_oneshot_ptr(curve, pts_host.ctypes.data, n, sc_page.ctypes.data, n)
            t0 = time.perf_counter()
            for _ in range(e2e_steps):
                out_pg = k.msm_oneshot_ptr(curve, pts_host.ctypes.data, n, sc_page.ctypes.data, n)
            pg_ms = (time.perf_counter() - t0) * 1e3 / e2e_steps
            assert (k.to_affine(curve, out_pg) == aff).all()
            rec["e2e_pageable"] = {"value": n / pg_ms / 1e3, "unit": UNIT, "ms_per_step": pg_ms, "h2d_bytes_per_step": (pt_bytes + 32) * n,
                                   "call": "kgr_msm_oneshot with points and scalars in pageable host memory (no cudaHostAlloc / kgr_host_alloc on the caller's side)"}
    else:
        pts_host = None
    # ---- optional mode for reused vectors (CRS / Pedersen key): window table built once at registration ---------------------------------
    if want_precompute:
        t0 = time.perf_counter()
        bases.precompute(0)
        build_s = time.perf_counter() - t0
        for _ in range(warmup):
            out_pre = k.msm_device(bases, d_sc.data_ptr(), n)
        pre_ms = 0.0
        for _ in range(steps):
            flush.zero_()
            torch.cuda.synchronize()
            out_pre = k.msm_device(bases, d_sc.data_ptr(), n)
            pre_ms += k.last_timing(0)[0]["total"]
        assert (k.to_affine(curve, out_pre) == aff).all()
        rec["precomputed_bases"] = {"note": "secondary, NOT the headline: bases registered with kgr_bases_precompute (table 2^(c*w)*P_i built once, W x the memory)",
                                    "value": n / (pre_ms / steps) / 1e3, "unit": UNIT, "ms_per_step": pre_ms / steps, "table_build_s": build_s, "shape": k.last_timing(0)[1]}
    # ---- checks (oracle = checker) ---------------------------------------------------------------------------------------------------------
    rec["checksum_ok"] = bool((expected_from_dot(curve, dot_of_shard(curve, ks, sc)) == aff).all())
    cores = os.cpu_count() or 1
    if full_cpu or cpu_sample_logn:
        s_logn = logn if full_cpu else min(cpu_sample_logn, logn)
        ns = 1 << s_logn
        if pts_host is None:
            pts_host = bases.download(0, ns)
        secs, cpu_out = cpu_msm(curve, pts_host[:ns], sc[:ns], cores)
        rec["cpu_baseline"] = {"value": ns / secs / 1e6, "unit": UNIT, "cores": cores, "kind": "port", "oracle_build": os.path.basename(A.LOADED_PATH or ""),
                               "sample": f"one MSM over the first 2^{s_logn} pairs of the same inputs, {secs:.2f} s, C++ restatement of the reference algorithm (c={ref_window_bits(ns)})"}
        if ns == n:
            rec["cpu_baseline"]["bit_exact_with_gpu"] = bool((A.to_affine(curve, cpu_out) == aff).all())
    bases.free()
    del d_sc, sc_pinned
    return rec, ms_per_step, aff


# ---- strong scaling: one MSM of 2^logn_total points over `world` ranks (world == 1: the base point of the curve) ---------------------------
def measure_strong(k, torch, dist, sharding, curve_name, logn_total, world, rank, steps, warmup, barrier, sampler=None):
    curve = CURVE_IDS[curve_name]
    n_total = 1 << logn_total
    first, count = sharding.shard_range(n_total, world, rank)
    bases, ks = k.Bases.generate(curve, count, seed=BASE_SEED, return_scalars=True, first=first)
    sc = scalars_range(first, count)
    sc_pinned = torch.from_numpy(sc.view(np.int64)).pin_memory()
    d_sc = sc_pinned.cuda(non_blocking=False)
    dot = dot_of_shard(curve, ks, sc)  # checker input, outside the timed regions
    del ks
    torch.cuda.synchronize()

    def step(resident):
        part = k.msm_device(bases, d_sc.data_ptr(), count) if resident else k.msm_host_ptr(bases, sc_pinned.data_ptr(), count)
        parts = sharding.gather_partials(part, device="cuda")  # one 96-byte point per rank
        return sharding.combine_partials(curve, parts) if rank == 0 else None, k.last_timing(0)[0]

    res, clocks = {}, None
    launches0 = k.launch_count(0)
    for resident in (True, False):
        for _ in range(warmup):
            total, _ = step(resident)
        barrier()
        if sampler and resident:
            sampler.start()
        t0 = time.perf_counter()
        dev = 0.0
        for _ in range(steps):
            total, tm = step(resident)
            dev += tm["total"]
        barrier()
        wall = (time.perf_counter() - t0) * 1e3 / steps
        if sampler and resident:
            clocks = sampler.stop()
        stats = torch.tensor([wall, dev / steps], dtype=torch.float64, device="cuda")
        if world > 1:
            dist.all_reduce(stats, op=dist.ReduceOp.MAX)
        res["resident" if resident else "host_scalars"] = {"wall_ms_per_step": float(stats[0]), "max_rank_device_ms": float(stats[1]), "total": total}
    launches = (k.launch_count(0) - launches0) // (2 * (steps + warmup))
    W = k.last_timing(0)[1]["W"]
    # checksum over all ranks
    dots = sharding.gather_partials(dot, device="cuda")
    out = None
    if rank == 0:
        from oracle import oracle as A
        from oracle import pyref as B
        r = B.FQ if curve == A.GRUMPKIN else B.FR
        acc = sum(B.limbs_to_int(d) for d in dots) % r  # Montgomery residues add like the values they stand for
        exp = expected_from_dot(curve, np.array(B.int_to_limbs(acc), dtype=np.uint64))
        aff = [k.to_affine(curve, res[m]["total"]) for m in ("resident", "host_scalars")]
        out = {"points_total": n_total, "points_per_gpu": count, "n_gpus": world,
               "value": n_total / res["resident"]["wall_ms_per_step"] / 1e3, "ms_per_step": res["resident"]["wall_ms_per_step"],
               "max_rank_device_ms": res["resident"]["max_rank_device_ms"],
               "e2e": {"value": n_total / res["host_scalars"]["wall_ms_per_step"] / 1e3, "unit": UNIT, "ms_per_step": res["host_scalars"]["wall_ms_per_step"],
                       "h2d_bytes_per_step": 32 * n_total, "d2h_bytes_per_step": world * max(1, min(4, count >> 21)) * W * 128,
                       "h2d_gbs_per_gpu_averaged_over_the_step": 32 * count / (res["host_scalars"]["wall_ms_per_step"] * 1e-3) / 1e9,
                       "call": "kgr_msm per rank (bases registered, scalars uploaded from pinned host memory every step) + all_gather of the partial points + host sum"},
               "checksum_ok": bool((exp == aff[0]).all() and (exp == aff[1]).all()), "result_is_identity": bool(int(aff[0][-1])), "affine": aff[0],
               "clocks": clocks, "gpu_launches_per_step_per_rank": launches,
               "timing": "wall clock between barriers around K steps (MSM on every rank + all_gather of one point per rank + host sum on rank 0), max over ranks"}
    bases.free()
    del d_sc, sc_pinned
    return out


def measure_inprocess(k, curve_name, logn_total, n_dev, steps):
    """The product's own sharding: kgr_init over n_dev devices in THIS process, one kgr_msm call with host scalars."""
    import torch
    curve = CURVE_IDS[curve_name]
    n = 1 << logn_total
    k.init(list(range(n_dev)))
    bases, ks = k.Bases.generate(curve, n, seed=BASE_SEED, return_scalars=True)
    sc = scalars_range(0, n)
    sc_pinned = torch.from_numpy(sc.view(np.int64)).pin_memory()
    for _ in range(2):
        out = k.msm_host_ptr(bases, sc_pinned.data_ptr(), n)
    t0 = time.perf_counter()
    for _ in range(steps):
        out = k.msm_host_ptr(bases, sc_pinned.data_ptr(), n)
    ms = (time.perf_counter() - t0) * 1e3 / steps
    aff = k.to_affine(curve, out)
    ok = bool((expected_from_dot(curve, dot_of_shard(curve, ks, sc)) == aff).all())
    bases.free()
    return {"call": f"one kgr_msm over kgr_init([0..{n_dev - 1}]) in one process, bases registered (sharded over the devices), host scalars from pinned memory",
            "points_total": n, "n_gpus": n_dev, "ms_per_step": ms, "value": n / ms / 1e3, "unit": UNIT, "steps": steps, "checksum_ok": ok, "affine": aff}


def run_reference(args, rank, world):
    """--impl reference: the reference's own CPU algorithm (C++ restatement; rustc/cargo are absent) on the host cores, on the first pairs of
    the SAME vectors our arm uses (bases from the oracle's restatement of the device generator's stream)."""
    if rank != 0:
        return
    from oracle import oracle as A
    cores = os.cpu_count() or 1
    cid = CURVE_IDS[args.curve]
    n_full = 1 << (args.strong_logn if world > 1 else args.logn)
    # bound the per-step sample so that the whole run (input generation included) stays within a few minutes
    cal_n = 1 << 13
    kk = A.bench_scalars(cid, BASE_SEED, 0, cal_n)
    t0 = time.perf_counter()
    pts_cal = A.fixed_base(cid, kk)
    gen_rate = cal_n / (time.perf_counter() - t0)
    secs, _ = cpu_msm(cid, pts_cal, scalars_range(0, cal_n), cores)
    rate = cal_n / secs
    n_s = n_full
    while n_s > cal_n and ((args.steps + args.warmup) * n_s / rate > 120.0 or n_s / gen_rate > 60.0):
        n_s //= 2
    pts = A.fixed_base(cid, A.bench_scalars(cid, BASE_SEED, 0, n_s))
    sc = scalars_range(0, n_s)
    for _ in range(args.warmup):
        cpu_msm(cid, pts, sc, cores)
    t0 = time.perf_counter()
    for _ in range(args.steps):
        cpu_msm(cid, pts, sc, cores)
    dt = time.perf_counter() - t0
    value = n_s * args.steps / dt / 1e6
    sample = (f"{args.steps} x MSM over the first 2^{int(math.log2(n_s))} pairs of the workload's own vectors (c={ref_window_bits(n_s)}; the full 2^{int(math.log2(n_full))} "
              f"would use c={ref_window_bits(n_full)}), all points distinct")
    line = {"impl": "reference", "metric": METRICS[args.curve], "value": value, "unit": UNIT, "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup,
            "ms_per_step": dt / args.steps * 1e3, "higher_is_better": True, "scaling": "strong" if world > 1 else "weak", "vs_baseline": None,
            "dtype": "u64 limbs (Montgomery Fq/Fr)", "data": "synthetic", "config": workload_config(args, world), "sample_points_per_step": n_s,
            "cpu_baseline": {"value": value, "unit": UNIT, "cores": cores, "kind": "port", "sample": sample, "oracle_build": os.path.basename(A.LOADED_PATH or "")},
            "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
            "note": "C++ restatement of groth16::msm::msm_curve_addition + zkstd arithmetic (oracle/), std::thread over windows like rayon; the Rust reference cannot be compiled in this image"}
    print(json.dumps(line), flush=True)


def groth16_record(args, steps=5, warmup=5, cpu_steps=1, cpu_warmup=0):
    import contextlib
    import importlib.util
    import io
    spec = importlib.util.spec_from_file_location("bench_next_rows", os.path.join(ROOT, "tools", "bench_next_rows.py"))
    rows = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(rows)
    out = []
    with contextlib.redirect_stdout(io.StringIO()):
        # Measured twice.  In a process that has not run any multi-threaded CPU work yet the call is ~25 % slower however many warm-up proofs
        # precede it (the per-lane host threads run on cores at idle clocks; tools/probe_prover_host.py).  The second pass runs after the CPU
        # baseline of the first has used all host cores, which is the state of a prover process that has generated a witness; both figures are reported.
        rows.bench_groth16(args.logm, out, steps, warmup, cpu_steps, cpu_warmup)
        proof = rows.bench_groth16(args.logm, out, steps, warmup, cpu_steps, cpu_warmup)
    return out[1], out[0], proof


def run_groth16(args, rank):
    """Groth16 prove latency (BASELINE metric, second half; config #4 scaled as SURVEY H7 suggests): create_proof after witness generation —
    7 FFTs, six G1 and two G2 MSMs, assembly of A, B, C — on the chained x^3 + x + 5 circuit with 2^logm constraints, host buffers in, three
    affine points out.  `--impl reference` times the restated reference code on the same inputs (FFT halves forked like rayon::join, the eight MSMs on all
    cores).  Either arm takes the best of --steps timed runs after --warmup warm-up runs.  The proof is checked against its discrete logs
    computed from the toxic waste; --dump-outputs writes it (ours only)."""
    if rank != 0:
        return
    import kogarashi_b200 as k
    k.init([int(os.environ.get("LOCAL_RANK", "0"))])
    ours = args.impl != "reference"
    if ours:
        rec, first, proof = groth16_record(args, steps=args.steps, warmup=args.warmup)
        if args.dump_outputs:
            dump_outputs(args.dump_outputs, {"proof_a": proof[0], "proof_b": proof[1], "proof_c": proof[2]})
        timing = f"wall clock around Groth16Prover.prove_from_evaluations, best of {args.steps} after {args.warmup} warm-up proofs; CRS registered on the GPU"
        cpu_sample = "the whole workload once: "
    else:
        rec, first, _ = groth16_record(args, cpu_steps=args.steps, cpu_warmup=args.warmup)
        timing = f"wall clock around the restated reference H pipeline and the eight MSMs, best of {args.steps} after {args.warmup} warm-up runs"
        cpu_sample = f"the whole workload, best of {args.steps} after {args.warmup} warm-up runs: "
    cpu_ms = rec["cpu_baseline"]["total_seconds"] * 1e3
    value = rec["gpu_wall_ms"]["normal"] if ours else cpu_ms
    line = {"metric": "groth16_prove_latency", "value": value, "unit": "ms", "n_gpus": 1, "steps": args.steps, "warmup": args.warmup, "ms_per_step": value, "higher_is_better": False,
            "scaling": "weak", "vs_baseline": None, "dtype": "u32 limbs (Montgomery Fq/Fr/Fq2)" if ours else "u64 limbs (Montgomery)", "data": "synthetic",
            "config": workload_config(args, 1),
            "timing": timing,
            "e2e": {"value": value, "unit": "ms", "h2d_bytes_per_step": (3 * rec["constraints"] + 4 * rec["constraints"]) * 32 if ours else 0,
                    "d2h_bytes_per_step": (1 << rec["log_n"]) * 32 if ours else 0},
            "cpu_baseline": {"value": cpu_ms, "unit": "ms", "cores": rec["cpu_baseline"]["cores"], "kind": "port",
                             "sample": cpu_sample + rec["cpu_baseline"]["note"]},
            "roofline": None, "proof_checked_against_discrete_logs": rec["checked_against_discrete_logs"], "h_bit_exact_with_oracle": rec["h_bit_exact_with_oracle"]}
    if ours:
        line["gpu_launches"] = int(k.launch_count(0))
        line["precomputed_crs_tables_ms"] = rec["gpu_wall_ms"]["precomputed"]
        line["idle_host_ms"] = first["gpu_wall_ms"]["normal"]   # first pass: no multi-threaded CPU work in this process before it
    else:
        line["impl"] = "reference"
    print(json.dumps(line), flush=True)


def strip(rec):
    """Drop the raw affine arrays before printing."""
    if isinstance(rec, dict):
        return {key: strip(v) for key, v in rec.items() if key != "affine"}
    return rec


def dump_outputs(dirname, points):
    """points: {name: affine point (x, y as Montgomery limbs, then is_infinity)} -> DIR/<name>.npy, each a float64 array of shape (words, 2)
    holding every uint64 limb as its low and high 32-bit halves, which float64 holds exactly.  Points are stored in affine form, not as the
    projective X, Y, Z the MSM engine returns: the sort places a bucket's points with atomic cursors, so their order and with it the
    projective representative of the same group element change from run to run; the affine form depends on the inputs alone."""
    os.makedirs(dirname, exist_ok=True)
    for name, a in points.items():
        a = np.asarray(a, dtype=np.uint64)
        np.save(os.path.join(dirname, name + ".npy"), np.stack([a & np.uint64(0xFFFFFFFF), a >> np.uint64(32)], axis=-1).astype(np.float64))


def main():
    sys.dont_write_bytecode = True  # the modules this run imports leave no __pycache__ in the tree
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--logn", type=int, default=20, help="log2 of the points of the N = 1 workload (BASELINE configs[1]: 2^20 on 1 B200) and of the weak-scaling shard")
    ap.add_argument("--strong-logn", type=int, default=26, help="log2 of the total points of the strong-scaling MSM (N > 1, and the strong_scaling_base of N = 1)")
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--curve", default="bn254_g1", choices=["bn254_g1", "grumpkin", "bn254_g2"],
                    help="grumpkin = BASELINE configs[2] (Nova secondary-curve commitment shape); bn254_g2 = next row N3 (the b_g2 MSMs of the Groth16 prover)")
    ap.add_argument("--cpu-sample-logn", type=int, default=20)
    ap.add_argument("--quick", action="store_true", help="main line only: skip north_star / grumpkin / groth16 / strong_scaling_base (N = 1) and weak / 2^24 / inprocess (N > 1)")
    ap.add_argument("--workload", default="msm", choices=["msm", "groth16"],
                    help="groth16 = the other half of BASELINE's metric: prove latency (create_proof after witness generation) on the chained example circuit")
    ap.add_argument("--logm", type=int, default=16, help="log2 of the constraint count for --workload groth16")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="write what the timed path computed in its last step: the MSM result as DIR/msm_affine.npy, or with --workload groth16 the "
                         "proof as DIR/proof_{a,b,c}.npy. Points are stored in affine form (x, y, is_infinity), not as the projective X, Y, Z the "
                         "engine returns, whose representative changes from run to run with the order of the bucket additions; float64, each uint64 "
                         "limb as its low and high 32-bit halves")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "ours":
        ap.error("--dump-outputs applies to --impl ours: the reference arm's sample size is chosen by a timing calibration, so its result "
                 "is not a fixed function of the arguments")
    args.warmup = max(args.warmup, 3) if args.impl == "ours" else args.warmup

    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))

    if args.workload == "groth16":
        run_groth16(args, rank)
        return
    if args.impl == "reference":
        run_reference(args, rank, world)
        return

    import torch
    import torch.distributed as dist

    import kogarashi_b200 as k
    from kogarashi_b200 import sharding

    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device (there is no CPU fallback)")
    torch.cuda.set_device(local_rank)
    cpu_group = None
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))
        cpu_group = dist.new_group(backend="gloo")  # CPU-side barrier for the in-process leg (an NCCL barrier would keep the other GPUs busy)
    k.init([local_rank])
    flush = torch.empty(512 << 20, dtype=torch.uint8, device="cuda")
    curve = CURVE_IDS[args.curve]

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    common = {"metric": METRICS[args.curve], "unit": UNIT, "n_gpus": world, "steps": args.steps, "warmup": args.warmup, "higher_is_better": True, "vs_baseline": None,
              "dtype": "u32 limbs (Montgomery Fq/Fr, 8x32-bit)", "data": "synthetic", "config": workload_config(args, world)}

    if world == 1:
        sampler = ClockSampler(local_rank)
        rec, ms_per_step, aff = measure_single(k, torch, args.curve, args.logn, args.steps, args.warmup, local_rank, flush, want_e2e=True, full_cpu=args.logn <= 20,
                                               cpu_sample_logn=args.cpu_sample_logn, sampler=sampler, want_precompute=not args.quick)
        if args.dump_outputs:
            dump_outputs(args.dump_outputs, {"msm_affine": aff})
        clocks = rec["clocks"]
        line = dict(common)
        line.update({"value": rec["value"], "ms_per_step": ms_per_step, "scaling": "weak", "l2": "flushed between steps (512 MiB write)",
                     "timing": "sum of per-step CUDA-event durations on the engine stream; wall_ms_per_step includes the flush and host gaps", "clocks": clocks})
        for key in ("wall_ms_per_step", "phases_ms", "shape", "gpu_launches", "e2e", "e2e_registered", "e2e_pageable", "roofline", "checksum_ok", "cpu_baseline", "precomputed_bases"):
            if key in rec:
                line[key] = rec[key]
        if not args.quick and args.curve == "bn254_g1":
            # BASELINE configs [4]/north star, [2], [3] and the N = 1 point of the strong-scaling curve, so that one driver run covers them
            ns, _, _ = measure_single(k, torch, "bn254_g1", 24, 3, 3, local_rank, flush, want_e2e=True, full_cpu=True)
            ns["note"] = "north-star size: 2^24-point BN254 G1 MSM on one B200; cpu_baseline.bit_exact_with_gpu compares with the restated reference MSM over ALL 2^24 pairs"
            line["north_star"] = ns
            gr, _, _ = measure_single(k, torch, "grumpkin", 20, 5, 3, local_rank, flush, want_e2e=True, full_cpu=True)
            gr["note"] = "BASELINE configs[2]: Grumpkin MSM, 2^20 points (Nova secondary-curve commitment shape)"
            line["grumpkin_2p20"] = gr
            try:  # SURVEY 8(f) row N3: the G2 query of the prover (prover.rs:64-65), same pipeline over Fq2 coordinates
                g2, _, _ = measure_single(k, torch, "bn254_g2", 18, 5, 3, local_rank, flush, want_e2e=True, full_cpu=True)
                g2["note"] = "row N3: BN254 G2 MSM, 2^18 points (Fq2 coordinates, 128-byte points); cpu_baseline = the restated reference algorithm over Fq2, all pairs"
                line["g2_2p18"] = g2
            except Exception as ex:
                line["g2_2p18"] = {"error": repr(ex)}
            try:  # SURVEY 8(f) row N2: the radix-2 transform of groth16/src/fft.rs on bn254 Fr, 2^20 elements, bit-exact with the restated reference dft
                from oracle import oracle as A
                nn = 1 << 20
                xv = A.random_field(A.FIELD_FR, nn, seed=bytes(range(16)))
                f = k.Fft(20)
                dv = torch.from_numpy(xv.view(np.int64)).cuda()
                torch.cuda.synchronize()
                f.transform_device("dft", dv.data_ptr())
                ntt_ms = []
                for _ in range(10):
                    f.transform_device("dft", dv.data_ptr())
                    ntt_ms.append(k.last_timing(0)[0]["total"])
                t0 = time.perf_counter()
                exp_v, _ = A.fft(20, "dft", xv)
                cpu_s = time.perf_counter() - t0
                t0 = time.perf_counter()
                got_v = f.dft(xv)
                e2e_s = time.perf_counter() - t0
                bf = nn // 2 * 20
                line["ntt_2p20"] = {"metric": "fr_ntt_time", "unit": "ms", "value": min(ntt_ms), "melem_per_s": nn / min(ntt_ms) / 1e3, "bit_exact_with_oracle": bool((got_v == exp_v).all()),
                                    "e2e_host_buffers_ms": e2e_s * 1e3, "cpu_baseline": {"value": cpu_s * 1e3, "unit": "ms", "kind": "port", "cores": "recursion halves forked like rayon::join"},
                                    "roofline": {"bound": "imad", "algorithmic_imads": bf * 264, "frac": bf * 264 / (min(ntt_ms) * 1e-3) / 1e12 / IMAD_PEAK_T,
                                                 "note": "one 254-bit Montgomery product (264 IMAD) per butterfly, n/2 * log2(n) butterflies"},
                                    "note": "row N2: dft of 2^20 Fr elements resident in HBM (device time, best of 10)"}
            except Exception as ex:
                line["ntt_2p20"] = {"error": repr(ex)}
            try:
                g16, first, _ = groth16_record(args)
                line["groth16_2p16"] = {"metric": "groth16_prove_latency", "unit": "ms", "value": g16["gpu_wall_ms"]["normal"], "idle_host_ms": first["gpu_wall_ms"]["normal"],
                                        "precomputed_crs_tables_ms": g16["gpu_wall_ms"]["precomputed"], "constraints": g16["constraints"],
                                        "cpu_baseline": {"value": g16["cpu_baseline"]["total_seconds"] * 1e3, "unit": "ms", "cores": g16["cpu_baseline"]["cores"], "kind": "port",
                                                         "fft_ms": g16["cpu_baseline"]["fft_seconds"] * 1e3, "msm_ms": g16["cpu_baseline"]["msm_seconds"] * 1e3,
                                                         "sample": "the whole workload once: " + g16["cpu_baseline"]["note"]},
                                        "proof_checked_against_discrete_logs": g16["checked_against_discrete_logs"], "h_bit_exact_with_oracle": g16["h_bit_exact_with_oracle"],
                                        "note": "BASELINE configs[3] scaled: create_proof after witness generation, chained x^3 + x + 5 circuit, wall clock, best of 5"}
            except Exception as ex:  # the secondary figure must not take the headline down with it
                line["groth16_2p16"] = {"error": repr(ex)}
            try:  # SURVEY 8(f) row N4: one Nova IVC step's vector work on one curve (commit(W), cross term, commit(T), two folds), state resident on the GPU
                import subprocess
                env = dict(os.environ, CUDA_VISIBLE_DEVICES=os.environ.get("CUDA_VISIBLE_DEVICES", str(local_rank)))
                outp = subprocess.run([sys.executable, "-B", os.path.join(ROOT, "tools", "bench_ivc_step.py"), "15", "1"], capture_output=True, text=True, timeout=300, env=env)
                recs = [json.loads(l) for l in outp.stdout.splitlines() if l.startswith("{")]
                line["nova_ivc_step_32k"] = recs[-1] if recs else {"error": (outp.stderr or "no output")[-300:]}
            except Exception as ex:
                line["nova_ivc_step_32k"] = {"error": repr(ex)}
            k.init([local_rank])
            base = {}
            for lg in sorted({24, args.strong_logn}):
                base[f"2p{lg}"] = strip(measure_strong(k, torch, dist, sharding, "bn254_g1", lg, 1, 0, 3, 2, barrier))
            line["strong_scaling_base"] = base
        print(json.dumps(strip(line)), flush=True)
        return

    # ---- N > 1: strong scaling of one MSM -----------------------------------------------------------------------------------------------
    main_rec = measure_strong(k, torch, dist, sharding, args.curve, args.strong_logn, world, rank, args.steps, args.warmup, barrier, sampler=ClockSampler(local_rank))
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, {"msm_affine": main_rec["affine"]})
    extra = {}
    if not args.quick:
        extra["strong_2p24"] = measure_strong(k, torch, dist, sharding, args.curve, 24, world, rank, args.steps, args.warmup, barrier)
        # weak scaling as in round 1: an independent 2^logn-point MSM per GPU, device events, max over ranks
        wrec, w_ms, w_aff = measure_single(k, torch, args.curve, args.logn, args.steps, args.warmup, local_rank, flush, first=rank << args.logn, want_e2e=True)
        stats = torch.tensor([w_ms, wrec["e2e"]["ms_per_step"], wrec["e2e_registered"]["ms_per_step"], 0.0 if wrec["checksum_ok"] else 1.0], dtype=torch.float64, device="cuda")
        dist.all_reduce(stats, op=dist.ReduceOp.MAX)
        n = 1 << args.logn
        extra["weak_scaling"] = {"note": "independent 2^%d-point MSMs, one per GPU (round-1 figure): per-rank CUDA events / wall clock, max over ranks" % args.logn,
                                 "value": world * n / float(stats[0]) / 1e3, "ms_per_step": float(stats[0]), "e2e_value": world * n / float(stats[1]) / 1e3,
                                 "e2e_registered_value": world * n / float(stats[2]) / 1e3, "checksum_ok_all_ranks": float(stats[3]) == 0.0, "unit": UNIT}
    # ---- the product's own sharding, from rank 0 alone; the other ranks wait on a CPU barrier with their GPUs idle ----------------------
    if not args.quick:
        torch.cuda.synchronize()
        dist.barrier(group=cpu_group)
        if rank == 0:
            try:
                inproc = {}
                for lg in sorted({24, args.strong_logn}):
                    r = measure_inprocess(k, args.curve, lg, world, 3)
                    ref = main_rec if lg == args.strong_logn else extra["strong_2p24"]
                    r["same_point_as_torchrun"] = bool((r["affine"] == ref["affine"]).all())
                    inproc[f"2p{lg}"] = r
                extra["inprocess"] = inproc
            except Exception as ex:
                extra["inprocess"] = {"error": repr(ex)}
        dist.barrier(group=cpu_group)
    if rank == 0:
        line = dict(common)
        line.update({"value": main_rec["value"], "ms_per_step": main_rec["ms_per_step"], "scaling": "strong", "timing": main_rec["timing"], "clocks": main_rec["clocks"],
                     "l2": "inputs larger than L2 (a 2^%d-point shard is %d MiB of bases + scalars)" % (args.strong_logn - int(math.log2(world)), (96 << (args.strong_logn - int(math.log2(world)))) >> 20),
                     "points_per_gpu": main_rec["points_per_gpu"], "max_rank_device_ms": main_rec["max_rank_device_ms"], "e2e": main_rec["e2e"],
                     "checksum_ok": main_rec["checksum_ok"], "result_is_identity": main_rec["result_is_identity"], "gpu_launches": main_rec["gpu_launches_per_step_per_rank"] * world,
                     "roofline": {"bound": "imad", "peak": IMAD_PEAK_T * world, "unit": "T IMAD/s", "traffic": None,
                                  "achieved": algorithmic_imads(1 << args.strong_logn) / (main_rec["ms_per_step"] * 1e-3) / 1e12,
                                  "frac": algorithmic_imads(1 << args.strong_logn) / (main_rec["ms_per_step"] * 1e-3) / 1e12 / (IMAD_PEAK_T * world),
                                  "note": "algorithmic IMADs of ONE 2^%d-point reference MSM over the wall time of the sharded call, against N x the per-GPU IMAD peak" % args.strong_logn}})
        line.update(extra)
        print(json.dumps(strip(line)), flush=True)
    dist.barrier(group=cpu_group)
    dist.destroy_process_group()


if __name__ == "__main__":
    main()
