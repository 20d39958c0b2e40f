// msm.cu — kernels, per-GPU engine and the C ABI (include/kgr_msm.h) of the MSM engine.
//
// One Engine per selected GPU: its own stream, grow-only workspace in HBM, pinned staging for the
// scalar upload and the 128-byte result.  A registered base vector is split into contiguous
// shards, one per GPU (SURVEY §8e); kgr_msm enqueues the whole pipeline on every GPU from one host
// thread per device, each GPU returns one XYZZ point, and the host adds them with the same
// field/curve code compiled for the CPU (field.cuh host bodies).  No NCCL, no CPU fallback for
// the MSM itself.
//
// Layout of this file:
//   1. error plumbing, Params, DevBuf, NttDomain, Engine (one per GPU and per lane: stream, events, grow-only workspaces)
//   2. window-size cost models, make_shape, enqueue_msm (the kernel pipeline of one MSM on one engine), collect_timing
//   3. shards / handles, upload, combine_partials (host Horner + sum over GPUs), run_msm (sharding, pipelined pieces, oneshot uploads),
//      lane_start / lane_finish (kgr_msm_batch), host conversions between the reference's projective form and XYZZ
//   4. test hooks, generator constants, fixed-base table, NTT domain tables and enqueue
//   5. extern "C": init / params / bases / msm / batch / oneshot / pedersen, NTT + Groth16 H, R1CS + Nova cross term, timing, test + bench hooks
#include <cuda_runtime.h>

#include <algorithm>
#include <atomic>
#include <chrono>
#include <cmath>
#include <condition_variable>
#include <cstdio>
#include <cstring>
#include <functional>
#include <map>
#include <memory>
#include <mutex>
#include <string>
#include <thread>
#include <type_traits>
#include <vector>

#include "../../include/kgr_msm.h"
#include "launch.cuh"
#include "pairing.cuh"
#include "r1cs_kernels.cuh"
#include "setup_kernels.cuh"

namespace kgr {

// ---- error plumbing ---------------------------------------------------------------------------
static thread_local std::string g_err;
static int fail(int code, const std::string &msg) {
    g_err = msg;
    return code;
}
struct CudaError {
    cudaError_t e;
    const char *what;
    int line;
};
#define CK(expr)                                                      \
    do {                                                              \
        cudaError_t _e = (expr);                                      \
        if (_e != cudaSuccess) throw CudaError{_e, #expr, __LINE__};  \
    } while (0)

// ---- engine -----------------------------------------------------------------------------------
struct Params {
    long window_bits = 0, chunk = 0, reduce_fanin = 16, final_on_device = 0, running_sum_stop = 4096, sort_mode = -1, reduce_mode = 1, affine_levels = -1, oneshot_split = 0, oneshot_growth = 0, lane_threads = 1, dense_x = -1;
};
// Tuning state is per calling thread (kgr_set_param changes the calling thread's copy only): an entry point snapshots it once and hands the
// snapshot to every engine it drives (Engine::params), so a kgr_set_param on one thread never changes an MSM in flight on another, and the
// library's own worker threads (lanes, devices) see the caller's values.
static thread_local Params t_params;

template <class T> struct DevBuf {
    T *p = nullptr;
    size_t cap = 0;
    void ensure(size_t n) {
        if (n <= cap) return;
        if (p) CK(cudaFree(p));
        p = nullptr;
        cap = 0;
        size_t want = n + n / 8;
        CK(cudaMalloc(&p, want * sizeof(T)));
        cap = want;
    }
    void release() {
        if (p) cudaFree(p);
        p = nullptr;
        cap = 0;
    }
};

// Radix-2 domain over bn254 Fr (groth16/src/fft.rs:27-90): tables live in HBM, built once per size.
struct NttDomain {
    uint32_t k = 0;
    DevBuf<uint8_t> tw, inv_tw, cosets, inv_cosets;  // omega^i (n/2), omega^-i (n/2), 7^i (n), 7^-i (n)
    Fp<FrP> n_inv, z_inv;                            // 1/n (fft.rs:86), 1/(7^n - 1) (fft.rs:139-153)
    ~NttDomain() {
        tw.release(); inv_tw.release(); cosets.release(); inv_cosets.release();
    }
};

enum { EV_START, EV_H2D, EV_COUNT, EV_SCAN, EV_FILL, EV_ACC, EV_FIXUP, EV_END, EV_N };

// Worker threads that stay alive between calls (the staging copies of upload_from_host / download_to_host).  Starting and joining seven
// std::threads per buffer — each paying the CUDA runtime's per-thread initialisation at its first call — cost more than the copies they ran:
// a 2^20-point oneshot call from pageable memory took 7.3 ms with 8 threads and 6.6 ms with 4 (pinned memory: 4.4 ms).
struct StagePool {
    std::mutex mu;
    std::condition_variable cv_work, cv_done;
    std::vector<std::thread> workers;
    const std::function<void(size_t)> *job = nullptr;
    size_t n_job = 0, next = 0, done = 0;
    bool stop = false;
    explicit StagePool(size_t n_workers) {
        for (size_t i = 0; i < n_workers; i++) workers.emplace_back([this]() { loop(); });
    }
    ~StagePool() {
        {
            std::lock_guard<std::mutex> lk(mu);
            stop = true;
        }
        cv_work.notify_all();
        for (auto &t : workers) t.join();
    }
    void loop() {
        std::unique_lock<std::mutex> lk(mu);
        for (;;) {
            cv_work.wait(lk, [&]() { return stop || next < n_job; });
            if (stop) return;
            const size_t idx = next++;
            const std::function<void(size_t)> *f = job;
            lk.unlock();
            (*f)(idx);
            lk.lock();
            if (++done == n_job) cv_done.notify_all();
        }
    }
    // f(0) .. f(n - 1), f(0) on the calling thread; returns when all have finished
    void run(size_t n, const std::function<void(size_t)> &f) {
        if (n == 0) return;
        {
            std::lock_guard<std::mutex> lk(mu);
            job = &f;
            n_job = n;
            next = 1;
            done = 0;
        }
        if (n > 1) cv_work.notify_all();
        f(0);
        std::unique_lock<std::mutex> lk(mu);
        if (++done < n_job) cv_done.wait(lk, [&]() { return done >= n_job; });
        n_job = 0;
        next = 0;
        job = nullptr;
    }
};

struct Engine {
    Params params;  // snapshot of the caller's tuning state for the MSM being enqueued
    int dev = -1;
    int sm_count = 0;
    cudaStream_t st = nullptr;
    cudaStream_t st_copy = nullptr;   // second stream: oneshot base upload overlaps count/scan/fill
    cudaEvent_t ev_pts = nullptr;     // bases of the current oneshot call are on the device
    cudaEvent_t ev_sc = nullptr;      // scalars of the current call are on the device (orders the two uploads)
    cudaEvent_t ev_fork = nullptr, ev_join = nullptr;  // fold reduce: the big upper-half sums run on st_copy beside the deep fold levels
    cudaEvent_t ev_input = nullptr;   // kgr_groth16_prove_r1cs: everything enqueued on st before the call (the resident z) is complete
    bool wait_pts = false;
    cudaEvent_t ev[EV_N] = {};
    cudaEvent_t ev_piece_sc[16] = {}, ev_piece_pts[16] = {};  // piece k's scalars / points are on the device (recorded on st_copy)
    cudaEvent_t ev_up0 = nullptr, ev_up1 = nullptr;            // around the uploads of a host-buffer call (timed: feeds h2d_gbs)
    double h2d_gbs = 42.0;       // host -> device rate the last host-buffer calls of this engine saw (moving average; pinned H2D on this pool: 42 - 55 GB/s)
    cudaEvent_t pev[16][6] = {};      // per-piece phase marks of a streamed call (enqueue_msm)
    size_t n_pev = 0;
    uint32_t n_pieces = 1;            // pieces of the last MSM enqueued on this engine
    DevBuf<uint32_t> counts, offsets, tile_sums, entries, scalars, worklist, tail_bucket, digits;
    DevBuf<uint32_t> coarse_counts, coarse_off, coarse_cursor, part_pay;  // radix-partition sort (kernels_sort.cu)
    DevBuf<uint32_t> lvl_off[5], lvl_cnt, lvl_pre, lvl_tot;                                // batched-affine levels (affine_kernels.cuh): offsets per level
    DevBuf<uint8_t> lvl_nodes[2];                                          // ... and their node arrays (ping-pong)
    DevBuf<uint8_t> lvl_x;                                                 // dense copy of the x coordinates of the bases (level-0 denominators)
    DevBuf<uint8_t> part_fine;
    DevBuf<uint8_t> piece_acc;  // bucket sums of one piece of a streamed call (enqueue_msm)
    DevBuf<uint8_t> fix_partial;  // slice sums of the hot buckets (k_fixup_long)
    DevBuf<uint32_t> fix_counter;  // ... and their arrival counters (zero between launches)
    DevBuf<uint8_t> bucket_acc, head, tail, lvl_s[2], lvl_a[2], result, fold_f, fold_partial, fold_v;  // raw bytes, cast per curve
    uint32_t *h_result = nullptr;                                         // pinned, 256 x 32 words (window sums)
    uint32_t n_result = 0;                                                // XYZZ points in h_result for the last MSM
    uint32_t result_c = 0;                                                // window bits to apply between them (0: already combined)
    uint8_t *h_stage = nullptr;                                           // pinned ring for uploads from pageable memory (upload_from_host)
    std::unique_ptr<StagePool> stage_pool;                                // its copy threads, started at first use
    cudaEvent_t stage_ev[16] = {};                                         // slot s may be refilled once its last copy has completed
    size_t counts_zeroed = 0;  // counts[0..counts_zeroed) are known to be zero
    float last_ms[9] = {};
    uint32_t last_shape[6] = {};
    int acc_blocks_per_sm[3] = {0, 0, 0};
    uint64_t launches = 0;            // kernels of this library launched on this engine since init
    cudaEvent_t user_ev[4] = {};      // kgr_event_record / kgr_event_elapsed_ms
    cudaEvent_t aux_ev[3] = {};       // phase marks of the R1CS calls (kgr_r1cs_last_timing)
    DevBuf<uint32_t> sat_result;      // kgr_nova_is_sat: violation count, first violating row, z[0] == 1
    DevBuf<uint8_t> oneshot_pts, oneshot_inf;  // device copy of the bases of kgr_msm_oneshot
    std::map<uint32_t, std::shared_ptr<struct NttDomain>> ntt_domains;  // per log2(n): twiddle / coset tables in HBM
    DevBuf<uint8_t> ntt_buf[3];
    DevBuf<uint8_t> fixed_table[3];   // per curve: d * 2^(8 j) * G, built on first use (kgr_fixed_base_mul / kgr_bases_generate)

    void init(int device) {
        dev = device;
        CK(cudaSetDevice(dev));
        cudaDeviceProp prop;
        CK(cudaGetDeviceProperties(&prop, dev));
        sm_count = prop.multiProcessorCount;
        CK(cudaStreamCreateWithFlags(&st, cudaStreamNonBlocking));
        CK(cudaStreamCreateWithFlags(&st_copy, cudaStreamNonBlocking));
        CK(cudaEventCreateWithFlags(&ev_pts, cudaEventDisableTiming));
        CK(cudaEventCreateWithFlags(&ev_sc, cudaEventDisableTiming));
        CK(cudaEventCreateWithFlags(&ev_fork, cudaEventDisableTiming));
        CK(cudaEventCreateWithFlags(&ev_join, cudaEventDisableTiming));
        CK(cudaEventCreateWithFlags(&ev_input, cudaEventDisableTiming));
        for (auto &e : ev) CK(cudaEventCreate(&e));
        for (auto &e : user_ev) CK(cudaEventCreate(&e));
        for (auto &e : aux_ev) CK(cudaEventCreate(&e));
        CK(cudaMallocHost(&h_result, 256 * 64 * sizeof(uint32_t)));  // up to 255 window sums of the widest XYZZ point (G2)
        acc_blocks_per_sm[0] = Launch<Bn254G1>::accumulate_blocks_per_sm();
        acc_blocks_per_sm[1] = Launch<GrumpkinC>::accumulate_blocks_per_sm();
        acc_blocks_per_sm[2] = Launch<Bn254G2>::accumulate_blocks_per_sm();
    }
    void destroy() {
        if (dev < 0) return;
        cudaSetDevice(dev);
        cudaStreamSynchronize(st);
        counts.release(); offsets.release(); tile_sums.release(); entries.release(); scalars.release(); worklist.release(); tail_bucket.release(); digits.release(); fix_partial.release(); fix_counter.release();
        coarse_counts.release(); coarse_off.release(); coarse_cursor.release(); part_pay.release(); part_fine.release();
        for (auto &b : lvl_off) b.release();
        lvl_cnt.release(); lvl_pre.release(); lvl_tot.release(); lvl_nodes[0].release(); lvl_nodes[1].release(); lvl_x.release();
        piece_acc.release();
        bucket_acc.release(); head.release(); tail.release(); result.release(); fold_f.release(); fold_partial.release(); fold_v.release();
        for (auto &t : fixed_table) t.release();
        for (int i = 0; i < 2; i++) { lvl_s[i].release(); lvl_a[i].release(); }
        if (h_result) cudaFreeHost(h_result);
        stage_pool.reset();
        if (h_stage) cudaFreeHost(h_stage);
        h_stage = nullptr;
        for (auto &e : stage_ev) if (e) { cudaEventDestroy(e); e = nullptr; }
        for (auto &e : ev) if (e) cudaEventDestroy(e);
        for (size_t k = 0; k < n_pev; k++)
            for (auto &pe : pev[k]) if (pe) cudaEventDestroy(pe);
        n_pev = 0;
        for (auto &x : ev_piece_sc) if (x) { cudaEventDestroy(x); x = nullptr; }
        if (ev_up0) { cudaEventDestroy(ev_up0); ev_up0 = nullptr; }
        if (ev_up1) { cudaEventDestroy(ev_up1); ev_up1 = nullptr; }
        for (auto &x : ev_piece_pts) if (x) { cudaEventDestroy(x); x = nullptr; }
        for (auto &e : user_ev) if (e) cudaEventDestroy(e);
        for (auto &e : aux_ev) if (e) cudaEventDestroy(e);
        sat_result.release();
        oneshot_pts.release(); oneshot_inf.release();
        ntt_domains.clear();
        for (auto &b : ntt_buf) b.release();
        if (st) cudaStreamDestroy(st);
        if (st_copy) cudaStreamDestroy(st_copy);
        if (ev_pts) cudaEventDestroy(ev_pts);
        if (ev_sc) cudaEventDestroy(ev_sc);
        if (ev_fork) cudaEventDestroy(ev_fork);
        if (ev_join) cudaEventDestroy(ev_join);
        if (ev_input) cudaEventDestroy(ev_input);
        dev = -1;
    }
};

// Host -> device copy of a caller buffer on stream st.  Pinned / registered memory goes straight to cudaMemcpyAsync.  Ordinary (pageable)
// memory — what a Rust Vec or a numpy array is — would be staged by the driver through one thread at ~12 GB/s on this box (a 2^20-point oneshot
// call: 11.4 ms against 5.0 ms from pinned buffers); here a few host threads copy 4-MiB chunks into a ring of pinned slots and enqueue the
// slot copies themselves, so the link is fed at several times that rate.  Returns when every chunk has been enqueued.
static constexpr size_t STAGE_CHUNK = 2u << 20, STAGE_SLOTS = 16, STAGE_THREADS = 8;
static size_t stage_threads_now() {  // development knob (KGR_STAGE_THREADS): number of staging threads actually used, <= STAGE_THREADS
    static const size_t v = [] {
        const char *e = getenv("KGR_STAGE_THREADS");
        long x = e ? atol(e) : (long)STAGE_THREADS;
        return (size_t)std::min<long>(std::max<long>(x, 1), (long)STAGE_THREADS);
    }();
    return v;
}
static void upload_from_host(Engine &e, void *dst, const void *src, size_t bytes, cudaStream_t st) {
    if (!bytes) return;
    cudaPointerAttributes at;
    bool pageable = true;
    if (cudaPointerGetAttributes(&at, src) == cudaSuccess) pageable = (at.type == cudaMemoryTypeUnregistered);
    else cudaGetLastError();
    if (!pageable || bytes < 2 * STAGE_CHUNK) {
        CK(cudaMemcpyAsync(dst, src, bytes, cudaMemcpyHostToDevice, st));
        return;
    }
    if (!e.h_stage) {
        CK(cudaMallocHost(&e.h_stage, STAGE_CHUNK * STAGE_SLOTS));
        for (auto &ev : e.stage_ev) CK(cudaEventCreateWithFlags(&ev, cudaEventDisableTiming));
    }
    const size_t n_chunks = (bytes + STAGE_CHUNK - 1) / STAGE_CHUNK;
    const size_t n_threads = std::min(stage_threads_now(), n_chunks);
    std::vector<cudaError_t> errs(n_threads, cudaSuccess);
    auto worker = [&](size_t t) {
        cudaError_t ce = cudaSetDevice(e.dev);
        // thread t owns the slots t and t + STAGE_THREADS and the chunks t, t + n_threads, ...
        for (size_t c = t, use = 0; c < n_chunks && ce == cudaSuccess; c += n_threads, use++) {
            size_t slot = t + (use & 1) * STAGE_THREADS, off = c * STAGE_CHUNK, len = std::min(STAGE_CHUNK, bytes - off);
            uint8_t *buf = e.h_stage + slot * STAGE_CHUNK;
            ce = cudaEventSynchronize(e.stage_ev[slot]);  // a never-recorded event is complete
            if (ce != cudaSuccess) break;
            std::memcpy(buf, (const uint8_t *)src + off, len);
            ce = cudaMemcpyAsync((uint8_t *)dst + off, buf, len, cudaMemcpyHostToDevice, st);
            if (ce == cudaSuccess) ce = cudaEventRecord(e.stage_ev[slot], st);
        }
        errs[t] = ce;
    };
    if (!e.stage_pool) e.stage_pool.reset(new StagePool(STAGE_THREADS - 1));
    e.stage_pool->run(n_threads, worker);
    for (cudaError_t ce : errs)
        if (ce != cudaSuccess) throw CudaError{ce, "upload_from_host", __LINE__};
}

// Device -> host copy into a caller buffer, same staging for pageable destinations.  Returns when the data is in `dst` (it synchronises the copies
// it issued; everything enqueued on st before the call has completed by then as well).
static void download_to_host(Engine &e, void *dst, const void *src, size_t bytes, cudaStream_t st) {
    if (!bytes) return;
    cudaPointerAttributes at;
    bool pageable = true;
    if (cudaPointerGetAttributes(&at, dst) == cudaSuccess) pageable = (at.type == cudaMemoryTypeUnregistered);
    else cudaGetLastError();
    if (!pageable || bytes < 2 * STAGE_CHUNK) {
        CK(cudaMemcpyAsync(dst, src, bytes, cudaMemcpyDeviceToHost, st));
        CK(cudaStreamSynchronize(st));
        return;
    }
    if (!e.h_stage) {
        CK(cudaMallocHost(&e.h_stage, STAGE_CHUNK * STAGE_SLOTS));
        for (auto &ev : e.stage_ev) CK(cudaEventCreateWithFlags(&ev, cudaEventDisableTiming));
    }
    for (auto &ev : e.stage_ev) CK(cudaEventSynchronize(ev));  // no upload may still be reading a slot
    const size_t n_chunks = (bytes + STAGE_CHUNK - 1) / STAGE_CHUNK;
    const size_t n_threads = std::min(STAGE_THREADS, n_chunks);
    std::vector<cudaError_t> errs(n_threads, cudaSuccess);
    auto worker = [&](size_t t) {
        cudaError_t ce = cudaSetDevice(e.dev);
        // two slots per thread: the copy of chunk i + 1 into one slot runs while chunk i is copied out of the other
        size_t first = t, use = 0;
        auto issue = [&](size_t c, size_t u) {
            size_t slot = t + (u & 1) * STAGE_THREADS, off = c * STAGE_CHUNK, len = std::min(STAGE_CHUNK, bytes - off);
            cudaError_t r = cudaMemcpyAsync(e.h_stage + slot * STAGE_CHUNK, (const uint8_t *)src + off, len, cudaMemcpyDeviceToHost, st);
            if (r == cudaSuccess) r = cudaEventRecord(e.stage_ev[slot], st);
            return r;
        };
        if (first < n_chunks && ce == cudaSuccess) ce = issue(first, 0);
        for (size_t c = first; c < n_chunks && ce == cudaSuccess; c += n_threads, use++) {
            size_t nxt = c + n_threads;
            if (nxt < n_chunks) ce = issue(nxt, use + 1);
            if (ce != cudaSuccess) break;
            size_t slot = t + (use & 1) * STAGE_THREADS, off = c * STAGE_CHUNK, len = std::min(STAGE_CHUNK, bytes - off);
            ce = cudaEventSynchronize(e.stage_ev[slot]);
            if (ce == cudaSuccess) std::memcpy((uint8_t *)dst + off, e.h_stage + slot * STAGE_CHUNK, len);
        }
        errs[t] = ce;
    };
    if (!e.stage_pool) e.stage_pool.reset(new StagePool(STAGE_THREADS - 1));
    e.stage_pool->run(n_threads, worker);
    for (cudaError_t ce : errs)
        if (ce != cudaSuccess) throw CudaError{ce, "download_to_host", __LINE__};
}

static std::mutex g_mu;
static std::vector<Engine> g_engines;
static uint64_t g_generation = 0;  // bumped by every kgr_init
// Extra engines (stream + workspaces) on the device of g_engines[0]: independent MSMs of one kgr_msm_batch call overlap on them.
static std::vector<std::vector<std::unique_ptr<Engine>>> g_lanes;  // [engine index][lane - 1]; lane 0 of a device is g_engines[index] itself
static constexpr size_t MAX_LANES = 8;
static void destroy_lanes() {
    for (auto &v : g_lanes)
        for (auto &l : v) l->destroy();
    g_lanes.clear();
}
static void ensure_lanes(size_t eng, size_t k) {
    if (g_lanes.size() < g_engines.size()) g_lanes.resize(g_engines.size());
    while (g_lanes[eng].size() + 1 < k) {
        std::unique_ptr<Engine> l(new Engine);
        l->init(g_engines[eng].dev);
        g_lanes[eng].push_back(std::move(l));
    }
}
static Engine &lane_of(size_t eng, size_t i) { return i == 0 ? g_engines[eng] : *g_lanes[eng][i - 1]; }

// Cost model for the window size (ns).  Small inputs (no batched-affine levels, counting sort), fitted to profiles/r01_phase_sweep.md:
//   accumulate 0.174 per entry; counting sort 0.0155 per entry growing with the histogram size G
//   (random L2 atomics + sector-granular scatter); reduce 0.4 ms fixed + 0.7 per bucket;
//   a thin top window (few leading scalar bits) concentrates n / 2^t entries in 2^t buckets.
// From 2^19 points on (batched-affine levels, radix-partition sort, quad reduction tail), refitted to profiles/r02_sweep_c_levels_quad_reduce.txt
// and the 2^24 - 2^26 sweeps of r02 (DESIGN section 4): accumulate 0.139 + 0.35 / (entries per bucket) per entry (short buckets: fewer useful
// affine levels, more flushes), sort 0.011 per entry, reduce 0.25 ms + 0.6 per bucket; the top window's digits fall into 2^(top_bits - 1 - F)
// coarse bins of the sort, each placed by ONE CTA at ~0.7 ns per element (c = 19 at 2^25: + 24 ms), and beyond 4096 coarse bins the sort
// falls back to the counting sort.  2^25 points: c = 20 (72.6 ms) instead of 17 (76.6); 2^24 stays at 17 (38.6 against 39.2).
static uint32_t choose_window_bits(uint32_t n, const Params &P) {
    if (P.window_bits > 0) return (uint32_t)std::min<long>(std::max<long>(P.window_bits, 1), 24);
    double best = 1e300;
    // c >= 9: with fewer than 256 buckets per window the bucket reduction falls back to serial running sums, which is never faster
    // from 2^8 points on (sweeps in profiles/r01_phase_sweep.md); a handful of points (the prover's blinding sums) is cheapest with tiny windows
    const uint32_t c_min = n < 64 ? 1 : 9;
    uint32_t best_c = c_min;
    for (uint32_t c = c_min; c <= 22; c++) {
        double W = std::ceil(255.0 / c), B = std::ldexp(1.0, (int)c - 1), G = W * B;
        int top_bits = 255 - (int)c * ((int)W - 1);  // bits of the top window incl. the carry bit
        double cost;
        if (n >= (1u << 19)) {
            const double per_bucket = (double)n / B;
            cost = (double)n * W * (0.139 + 0.35 / per_bucket + 0.011) + 0.6 * G + 0.25e6;
            const int F = std::min(8, (int)c - 1);
            const double used_bins = top_bits - 1 > F ? std::ldexp(1.0, top_bits - 1 - F) : 1.0;
            cost += 0.7 * (double)n / used_bins;
            if (c >= 22) cost += 0.5 * (double)n * W;
        } else {
            double lg = std::log2(G);
            double sort_ns = 0.0155 + (lg > 19 ? 0.008 * (lg - 19) : 0.0);
            cost = (double)n * W * (0.174 + sort_ns) + 0.7 * G + (G > 64 ? 0.4e6 : 0.1e6);
        }
        if (top_bits < (int)c) cost += 0.08e6;       // a thin top window fills few buckets: the hot-bucket fix-up path runs
        if (top_bits < 8 && top_bits < (int)c) cost += 0.08 * n * (8 - top_bits);
        if (cost < best) { best = cost; best_c = c; }
    }
    return best_c;
}

// Window size for the collapsed mode: one bucket set shared by all windows, so the reduce term depends on B, not W * B.
// Fitted to the sweeps in profiles/r01_precompute.md (ns): accumulate 0.16 per entry (0.08 ms floor: one chunk of 16 adds);
// count and fill are bound by atomics on the B shared counters — 0.245 per entry at B <= 256 falling like B^-0.6 to the
// 0.008 streaming floor; single-window reduce 0.17 ms + 0.017 ms per bit of c (+ 0.9 per bucket beyond 2^16); a thin top
// window (fewer leading bits than c) makes a few buckets hot and costs ~0.25 ms of fix-up.  `mul_weight`: field
// multiplications per coordinate product (1, or 3 for G2) scales everything that is curve arithmetic.
static uint32_t choose_window_bits_collapsed(uint32_t n, double mul_weight) {
    double best = 1e300;
    uint32_t best_c = 9;
    for (uint32_t c = 9; c <= 23; c++) {  // below c = 9 all entries share <= 128 counters and buckets: never the fastest
        double W = std::ceil(255.0 / c), B = std::ldexp(1.0, (int)c - 1), entries = (double)n * W;
        double atomic_ns = std::min(0.245, std::max(0.008, 0.072 * std::pow(1024.0 / B, 0.6)));
        double acc = std::max(entries * 0.16, 0.08e6);
        double reduce = 0.17e6 + 0.017e6 * c + 0.9 * std::max(0.0, B - 65536.0);
        int top_bits = 255 - (int)c * ((int)W - 1);
        double hot = top_bits < (int)c ? std::min(0.25e6, entries * 0.05) : 0.0;
        double cost = (acc + reduce + hot) * mul_weight + 2.0 * entries * atomic_ns;
        if (cost < best) { best = cost; best_c = c; }
    }
    return best_c;
}

// table_c == 0: normal mode.  Otherwise the bases pointer is a precomputed table built for window size table_c.
static MsmShape make_shape(const Params &P, uint32_t n, int blocks_per_sm, int sm_count, uint32_t table_c = 0, uint32_t table_stride = 0, uint32_t table_off = 0,
                           uint64_t entries_override = 0) {
    MsmShape sh;
    sh.n = n;
    sh.c = table_c ? table_c : choose_window_bits(n, P);
    sh.W = (255 + sh.c - 1) / sh.c;
    sh.B = 1u << (sh.c - 1);
    sh.G = table_c ? sh.B : sh.W * sh.B;
    sh.gstride = table_c ? 0 : sh.B;
    sh.pstride = table_c ? table_stride : 0;
    sh.poff = table_c ? table_off : 0;
    sh.K = (uint32_t)P.reduce_fanin;
    uint64_t M = entries_override ? entries_override : (uint64_t)n * sh.W;
    if (P.chunk > 0) {
        sh.L = (uint32_t)P.chunk;
    } else {
        // pick the chunk length that minimises (waves x (L + per-chunk overhead)) for this GPU
        uint64_t concurrent = (uint64_t)std::max(1, blocks_per_sm) * TPB_ACC * std::max(1, sm_count);
        double best = 1e300;
        uint32_t bestL = 32;
        // short lists (one wave whatever L is): the chain of L dependent additions per thread is the latency of the kernel, and the quad fix-up sums
        // the pieces of a cut bucket cheaply, so L goes down to 4 as long as a typical bucket is cut into <= ~4 pieces (more than
        // FIXUP_INLINE_MAX pieces take the hot-bucket path): 2^10 points 0.38 -> 0.32 ms, 2^12 0.37 -> 0.34 ms
        const uint64_t per_bucket = M / std::max<uint64_t>(1, sh.G);
        const uint32_t L_lo = (uint32_t)std::min<uint64_t>(16, std::max<uint64_t>(4, (per_bucket / 4 + 3) & ~3ull));
        for (uint32_t L = L_lo; L <= 256; L += 4) {
            uint64_t chunks = (M + L - 1) / L;
            uint64_t waves = (chunks + concurrent - 1) / concurrent;
            double cost = (double)waves * (L + 2.0);
            if (cost < best - 1e-9) { best = cost; bestL = L; }
        }
        sh.L = bestL;
    }
    return sh;
}

// One piece of a host-buffer call that is streamed over PCIe: pairs [first, first + count) of the call, usable once ev_sc (its scalars are on
// the device) and ev_pts (its points are; nullptr for registered bases) have fired.
struct StreamPiece {
    size_t first, count;
    cudaEvent_t ev_sc, ev_pts;
    // number of pieces whose events have been RECORDED (a wait on an event that was never recorded is a no-op, so the waits of piece k must
    // not be enqueued before that); nullptr: all of them were recorded before enqueue_msm was called
    const std::atomic<size_t> *recorded;
};
enum { PE_BEGIN, PE_COUNT, PE_SCAN, PE_FILL, PE_ACC, PE_FIXUP, PE_N };
constexpr size_t MAX_PIECES = 16;

// Enqueue one MSM over n pairs on engine e.  d_scalars: device pointer (n x 8 words).
// pieces (optional, more than one): the call's inputs arrive piece by piece.  Every piece is sorted and accumulated as soon as it is on the
// device, with the window size of the whole call, its bucket sums are added to one shared, zero-initialised bucket set (k_bucket_merge), and
// ONE bucket reduction closes the call.  (Round 1 ran the pieces as independent MSMs on separate lanes: each paid its own reduction and the smaller window size
// of a smaller MSM, 2 x 1.9 ms for the two halves of a 2^20-point call against 3.5 ms for the whole, profiles/r02_e2e.md.)
template <class C>
static void enqueue_msm(Engine &e, const AffinePt<C> *d_bases, const uint32_t *d_scalars, int is_mont, uint32_t n, uint32_t table_c = 0,
                        uint32_t table_stride = 0, uint32_t table_off = 0, const std::vector<StreamPiece> *pieces = nullptr) {
    typedef XyzzPt<C> X;
    typedef Launch<C> K;
    const Params &P = e.params;
    const bool streamed = pieces && pieces->size() > 1;
    if (streamed && pieces->size() > MAX_PIECES) throw CudaError{cudaErrorInvalidValue, "too many pieces", __LINE__};
    uint32_t n_piece_max = n;
    if (streamed) {
        n_piece_max = 0;
        for (auto &pc : *pieces) n_piece_max = std::max<uint32_t>(n_piece_max, (uint32_t)pc.count);
    }
    MsmShape sh = make_shape(P, n, e.acc_blocks_per_sm[C::ID], e.sm_count, table_c, table_stride, table_off);
    const uint32_t nwin = table_c ? 1u : sh.W;  // independent bucket sets to reduce
    uint64_t M64 = (uint64_t)n_piece_max * sh.W;
    if (M64 >= (1ull << 32) - 1) throw CudaError{cudaErrorInvalidValue, "n * windows exceeds 2^32 entries", __LINE__};
    const uint32_t Mmax = (uint32_t)M64;  // entries of the largest piece
    uint32_t cnt1 = (sh.B + sh.K - 1) / sh.K;

    size_t G1 = (size_t)sh.G + 1;
    if (e.counts.cap < G1) e.counts_zeroed = 0;
    e.counts.ensure(G1);
    e.offsets.ensure(G1 + 4);
    e.tile_sums.ensure(LaunchUtil::scan_tiles((uint32_t)G1) + 1);
    e.entries.ensure((size_t)Mmax + 1);
    e.bucket_acc.ensure((size_t)sh.G * sizeof(X));
    for (int i = 0; i < 2; i++) {
        e.lvl_s[i].ensure((size_t)nwin * cnt1 * sizeof(X));
        e.lvl_a[i].ensure((size_t)nwin * cnt1 * sizeof(X));
    }
    e.result.ensure(sizeof(X));
    if (e.counts_zeroed < G1) {
        CK(cudaMemsetAsync(e.counts.p, 0, e.counts.cap * sizeof(uint32_t), e.st));
        e.counts_zeroed = e.counts.cap;
    }
    X *piece_dst = (X *)e.bucket_acc.p;  // where a piece's bucket sums go: the call's bucket set itself unless the call is streamed
    if (streamed) {
        CK(cudaMemsetAsync(e.bucket_acc.p, 0, (size_t)sh.G * sizeof(X), e.st));  // all-zero words: XYZZ identity (zz = 0)
        e.piece_acc.ensure((size_t)sh.G * sizeof(X));
        piece_dst = (X *)e.piece_acc.p;
        for (size_t k = e.n_pev; k < pieces->size(); k++) {
            for (auto &ev : e.pev[k]) CK(cudaEventCreate(&ev));
            e.n_pev = k + 1;
        }
    }
    e.n_pieces = streamed ? (uint32_t)pieces->size() : 1;

    const uint32_t *off_final = e.offsets.p;
    // ---- one piece: sort, (batched-affine levels,) accumulate, fix-up ------------------------------------------------------------------------------
    auto run_piece = [&](const AffinePt<C> *bases_k, const uint32_t *scalars_k, uint32_t n_k, uint32_t poff_k, cudaEvent_t ev_sc, cudaEvent_t ev_pts, cudaEvent_t *pe) {
        MsmShape shp = make_shape(P, n, e.acc_blocks_per_sm[C::ID], e.sm_count, table_c, table_stride, poff_k, (uint64_t)n_k * sh.W);
        shp.n = n_k;
        const uint32_t Mk = n_k * sh.W;
        uint32_t chunks = (Mk + shp.L - 1) / shp.L;  // re-derived below when batched-affine levels shorten the list
        e.head.ensure((size_t)chunks * sizeof(X));
        e.tail.ensure((size_t)chunks * sizeof(X));
        e.tail_bucket.ensure((size_t)chunks + 1);
        if (ev_sc) CK(cudaStreamWaitEvent(e.st, ev_sc, 0));
        CK(cudaEventRecord(pe[PE_BEGIN], e.st));
        // sort_mode 2: two block-local radix partitions (kernels_sort.cu); 1: counting sort with a window-major fill from stored digits (scatter
        // region per window stays in L2); 0: counting sort, one thread per scalar recodes again and scatters into all windows;
        // -1 (auto): radix partitions from 2^21 entries on (below, the second pass costs more than the atomics it saves: 2^16 points 0.91 vs 0.85 ms,
        // 2^18 points 1.44 vs 1.48 ms, profiles/r02_sort.md)
        SortPlan pl;
        const bool radix = (P.sort_mode == 2 || (P.sort_mode < 0 && Mk >= (1u << 21))) && LaunchSort::plan(shp, pl);
        if (radix) {
            const size_t cw = LaunchSort::coarse_words(pl);
            if (e.coarse_counts.cap < cw) {
                e.coarse_counts.ensure(cw);
                CK(cudaMemsetAsync(e.coarse_counts.p, 0, e.coarse_counts.cap * sizeof(uint32_t), e.st));  // k_sort_scan leaves it zero again
            }
            e.coarse_off.ensure(cw);
            e.coarse_cursor.ensure(cw);
            e.digits.ensure((size_t)Mmax + 1);
            e.part_pay.ensure((size_t)Mmax + 1);
            e.part_fine.ensure((size_t)Mmax + 16);
            e.launches += LaunchSort::run(e.st, std::is_same<typename C::Scalar, FqP>::value ? 0 : 1, e.sm_count, pl, scalars_k, is_mont, e.digits.p, e.coarse_counts.p,
                                          e.coarse_off.p, e.coarse_cursor.p, e.part_pay.p, e.part_fine.p, e.entries.p, e.offsets.p, pe[PE_COUNT], pe[PE_SCAN]);
            CK(cudaEventRecord(pe[PE_FILL], e.st));
        } else {
            const bool window_major = P.sort_mode == 1 || (P.sort_mode < 0 && (uint64_t)Mk * 4 > (96ull << 20));
            if (window_major) e.digits.ensure((size_t)Mmax + 1);
            K::count(e.st, shp, scalars_k, is_mont, e.counts.p, window_major ? e.digits.p : nullptr);
            CK(cudaEventRecord(pe[PE_COUNT], e.st));
            LaunchUtil::exclusive_scan(e.st, e.counts.p, e.offsets.p, (uint32_t)G1, e.tile_sums.p);
            e.launches += 2 + LaunchUtil::scan_launches((uint32_t)G1);
            CK(cudaEventRecord(pe[PE_SCAN], e.st));
            if (window_major) K::fill_window(e.st, shp, e.digits.p, e.counts.p, e.offsets.p, e.entries.p);
            else K::fill(e.st, shp, scalars_k, is_mont, e.counts.p, e.offsets.p, e.entries.p);
            CK(cudaEventRecord(pe[PE_FILL], e.st));
        }
        if (ev_pts) CK(cudaStreamWaitEvent(e.st, ev_pts, 0));
        if (e.wait_pts) {
            CK(cudaStreamWaitEvent(e.st, e.ev_pts, 0));
            e.wait_pts = false;
        }
        // affine_levels r > 0 (8-word coordinates only): r levels of pairwise batched-affine sums inside every bucket (affine_kernels.cuh) leave
        // ceil(len / 2^r) affine nodes per bucket; the XYZZ kernel then sums those instead of the base points.  -1 (auto), from the sweeps in
        // profiles/r02_affine.md and r02_e2e.md: none below 8e6 entries or 16 entries per bucket (the three extra kernels per level cost more than they
        // save: 2^18 points 1.44 vs 1.43 ms), 1 up to 1.2e7 (a 2^19-point piece of a streamed 2^20 call: 4.77 vs 4.91 ms), 2 up to 3e7 entries
        // (2^20: 3.48 vs 3.82 ms), then 3, and 4 from 128 entries per bucket on (2^24: 39.3 vs 42.9 ms)
        const uint32_t *off_k = e.offsets.p;
        bool levels_ran = false;
        if constexpr (C::ID != Bn254G2::ID) {
            uint32_t levels = (uint32_t)std::max<long>(P.affine_levels, 0);
            if (P.affine_levels < 0) {
                const double per_bucket = (double)Mk / (double)sh.G;
                levels = (Mk < 8000000u || per_bucket < 16.0) ? 0u : Mk < 12000000u ? 1u : Mk < 30000000u ? 2u : per_bucket >= 128.0 ? 4u : 3u;
            }
            if (levels > 0 && Mk >= 2) {
                uint32_t out_max[5], m_in = Mk;
                for (uint32_t l = 0; l < levels; l++) {
                    out_max[l] = (uint32_t)(((uint64_t)m_in + std::min<uint64_t>(sh.G, m_in) + 1) / 2);  // sum of ceil(len / 2) over the non-empty buckets
                    m_in = out_max[l];
                }
                uint32_t *off[6] = {e.offsets.p};
                for (uint32_t l = 0; l < levels; l++) {
                    e.lvl_off[l].ensure(G1 + 4);
                    off[l + 1] = e.lvl_off[l].p;
                }
                e.lvl_cnt.ensure(G1 + 4);
                e.lvl_nodes[0].ensure((size_t)out_max[0] * sizeof(AffinePt<C>));
                if (levels > 1) e.lvl_nodes[1].ensure((size_t)out_max[1] * sizeof(AffinePt<C>));
                AffinePt<C> *nodes[2] = {(AffinePt<C> *)e.lvl_nodes[0].p, (AffinePt<C> *)e.lvl_nodes[1].p};
                size_t pre_words, tot_words;
                K::affine_scratch_words(out_max[0], pre_words, tot_words);
                e.lvl_pre.ensure(pre_words);
                e.lvl_tot.ensure(tot_words);
                // dense x copy for the level-0 denominators ("dense_x": -1 auto, 0 off, 1 on).  Measured (accumulate phase, ms): 2^20 2.70 -> 2.69,
                // 2^21 4.94 -> 4.80, 2^22 9.23 -> 8.98, 2^23 18.12 -> 17.83, 2^24 35.62 -> 35.46, 2^26 no change: a gathered 32-byte x out of a
                // 64-byte point costs a wider DRAM fetch than one out of a dense array; below 2^21 points the copy costs what it saves
                void *xs = nullptr;
                const bool want_x = !table_c && (P.dense_x > 0 || (P.dense_x < 0 && n_k > (1u << 20) && n_k <= (1u << 24)));
                if (want_x) {
                    e.lvl_x.ensure((size_t)n_k * sizeof(typename C::Elem));
                    xs = e.lvl_x.p;
                }
                e.launches += K::affine_levels(e.st, levels, sh.G, bases_k, e.entries.p, off, nodes, out_max, e.lvl_cnt.p, e.tile_sums.p, e.lvl_pre.p, e.lvl_tot.p, n_k, xs);
                // the XYZZ kernel sums what is left: chunk length re-chosen for the shorter list
                MsmShape sh2 = make_shape(P, n, e.acc_blocks_per_sm[C::ID], e.sm_count, table_c, table_stride, poff_k, out_max[levels - 1]);
                shp.L = sh2.L;
                chunks = (out_max[levels - 1] + shp.L - 1) / shp.L;
                e.head.ensure((size_t)chunks * sizeof(X));
                e.tail.ensure((size_t)chunks * sizeof(X));
                e.tail_bucket.ensure((size_t)chunks + 1);
                off_k = off[levels];
                shp.chunks = P.chunk > 0 ? 0u : chunks;  // the chunk length follows the entries actually on the device (eff_chunk_len) unless it is forced
                K::accumulate(e.st, shp, chunks, nodes[(levels - 1) & 1], off_k, nullptr, piece_dst, (X *)e.head.p, (X *)e.tail.p, e.tail_bucket.p);
                levels_ran = true;
            }
        }
        if (!levels_ran) {
            shp.chunks = P.chunk > 0 ? 0u : chunks;
            K::accumulate(e.st, shp, chunks, bases_k, e.offsets.p, e.entries.p, piece_dst, (X *)e.head.p, (X *)e.tail.p, e.tail_bucket.p);
        }
        CK(cudaEventRecord(pe[PE_ACC], e.st));
        {
            const size_t rec = K::fixup_records_max(chunks);
            e.worklist.ensure(4 * rec + 4);
            e.fix_partial.ensure(rec * sizeof(X));
            if (e.fix_counter.cap < rec) {
                e.fix_counter.ensure(rec);
                CK(cudaMemsetAsync(e.fix_counter.p, 0, e.fix_counter.cap * sizeof(uint32_t), e.st));  // k_fixup_long leaves it zero again
            }
        }
        CK(cudaMemsetAsync(e.worklist.p, 0, sizeof(uint32_t), e.st));
        K::fixup(e.st, shp, chunks, e.sm_count, off_k, piece_dst, (const X *)e.head.p, (const X *)e.tail.p, e.tail_bucket.p, e.worklist.p + 4, e.worklist.p,
                 (X *)e.fix_partial.p, e.fix_counter.p);
        if (streamed) {
            K::bucket_merge(e.st, sh.G, off_k, piece_dst, (X *)e.bucket_acc.p);
            e.launches++;
        }
        CK(cudaEventRecord(pe[PE_FIXUP], e.st));
        e.launches += 4;  // accumulate, fixup, fixup_long (+ memset)
        off_final = off_k;
        sh.L = shp.L;
    };
    if (streamed) {
        for (size_t k = 0; k < pieces->size(); k++) {
            const StreamPiece &pc = (*pieces)[k];
            if (pc.recorded)
                while (pc.recorded->load(std::memory_order_acquire) <= k) std::this_thread::yield();  // the uploader thread is still staging this piece
            // window table: same base pointer, shifted column; plain vector: shifted pointer
            run_piece(table_c ? d_bases : d_bases + pc.first, d_scalars + 8 * pc.first, (uint32_t)pc.count, table_c ? table_off + (uint32_t)pc.first : 0u, pc.ev_sc,
                      pc.ev_pts, e.pev[k]);
        }
        off_final = nullptr;  // every bucket is defined (zero-initialised): the reduction reads them all
    } else {
        cudaEvent_t pe[PE_N] = {e.ev[EV_H2D], e.ev[EV_COUNT], e.ev[EV_SCAN], e.ev[EV_FILL], e.ev[EV_ACC], e.ev[EV_FIXUP]};
        const bool one = pieces && pieces->size() == 1;  // a host-buffer call small enough for one upload: still wait for it
        run_piece(d_bases, d_scalars, n, table_off, one ? (*pieces)[0].ev_sc : nullptr, one ? (*pieces)[0].ev_pts : nullptr, pe);
    }
    // Reduce.  reduce_mode 1 (default, B >= 256): fold reduce — parallel halving folds + plain sums of the upper halves
    // (kernels_curve.cuh).  reduce_mode 0: running-sum levels (fan-in K) while many elements per window remain, then one
    // parallel weighting pass and block-level tree sums.
    const X *win = nullptr;
    if (P.reduce_mode == 1 && sh.B >= 256) {
        uint32_t nb = sh.c - 1, chunks_max = K::fold_chunks_max(sh.B);
        e.fold_f.ensure((size_t)nwin * sh.B * sizeof(X));
        e.fold_partial.ensure((size_t)nwin * nb * chunks_max * sizeof(X));
        e.fold_v.ensure((size_t)nwin * nb * sizeof(X));
        e.launches += K::fold_reduce(e.st, e.st_copy, e.ev_fork, e.ev_join, nwin, sh.B, (const X *)e.bucket_acc.p, off_final, (X *)e.fold_f.p, (X *)e.fold_partial.p, (X *)e.fold_v.p,
                                     (X *)e.lvl_a[0].p);
        win = (const X *)e.lvl_a[0].p;
    } else {
        uint32_t cnt = sh.B, m_log2 = 0, klog = 0;
        while ((1u << klog) < sh.K) klog++;
        const X *in_s = (const X *)e.bucket_acc.p, *in_a = nullptr;
        int pp = 0;
        do {
            uint32_t cnt_out = (cnt + sh.K - 1) / sh.K;
            X *os = (X *)e.lvl_s[pp].p, *oa = (X *)e.lvl_a[pp].p;
            K::reduce(e.st, nwin, cnt, sh.K, m_log2, in_s, in_a, os, oa, in_a ? nullptr : off_final);
            e.launches++;
            in_s = os;
            in_a = oa;
            cnt = cnt_out;
            m_log2 += klog;
            pp ^= 1;
        } while (cnt > (uint32_t)P.running_sum_stop);
        win = in_a;  // [nwin] once cnt == 1
        if (cnt > 1) {
            X *v = (X *)e.lvl_s[pp].p;
            K::weight(e.st, nwin, cnt, m_log2, in_s, in_a, v);
            e.launches++;
            const X *tin = v;
            X *tout = (X *)e.lvl_a[pp].p;
            while (cnt > 1) {
                uint32_t blocks = (cnt + TPB_TREE - 1) / TPB_TREE;
                K::tree_sum(e.st, nwin, tin, cnt, tout);
                e.launches++;
                cnt = blocks;
                X *nxt = (X *)tin;
                tin = tout;
                tout = nxt;
            }
            win = tin;
        }
    }
    if (P.final_on_device && !table_c) {
        K::final_horner(e.st, sh, win, (X *)e.result.p);
        e.launches++;
        CK(cudaMemcpyAsync(e.h_result, e.result.p, sizeof(X), cudaMemcpyDeviceToHost, e.st));
        e.n_result = 1;
        e.result_c = 0;
    } else {
        // one D2H copy of the W window sums; the host applies the c doublings between windows
        // (254 sequential doublings: ~1 ms on one GPU thread, ~0.1 ms on a host core)
        CK(cudaMemcpyAsync(e.h_result, win, (size_t)nwin * sizeof(X), cudaMemcpyDeviceToHost, e.st));
        e.n_result = nwin;
        e.result_c = sh.c;
    }
    CK(cudaEventRecord(e.ev[EV_END], e.st));
    CK(cudaGetLastError());
    e.last_shape[0] = sh.c; e.last_shape[1] = sh.W; e.last_shape[2] = sh.B; e.last_shape[3] = sh.L; e.last_shape[4] = sh.K; e.last_shape[5] = n;
}

static void collect_timing(Engine &e) {
    auto el = [&](int a, int b) {
        float ms = 0;
        cudaEventElapsedTime(&ms, e.ev[a], e.ev[b]);
        return ms;
    };
    if (e.n_pieces > 1) {  // streamed call: phases summed over the pieces; the waits for the uploads count as h2d
        auto pel = [&](size_t k, int a, int b) {
            float ms = 0;
            cudaEventElapsedTime(&ms, e.pev[k][a], e.pev[k][b]);
            return ms;
        };
        for (int q = 1; q <= 7; q++) e.last_ms[q] = 0;
        e.last_ms[0] = el(EV_START, EV_END);
        float busy = 0;
        for (size_t k = 0; k < e.n_pieces; k++) {
            e.last_ms[1] += pel(k, PE_BEGIN, PE_COUNT);
            e.last_ms[2] += pel(k, PE_COUNT, PE_SCAN);
            e.last_ms[3] += pel(k, PE_SCAN, PE_FILL);
            e.last_ms[4] += pel(k, PE_FILL, PE_ACC);   // includes the wait for the piece's points
            e.last_ms[5] += pel(k, PE_ACC, PE_FIXUP);
            busy += pel(k, PE_BEGIN, PE_FIXUP);
        }
        cudaEventElapsedTime(&e.last_ms[6], e.pev[e.n_pieces - 1][PE_FIXUP], e.ev[EV_END]);
        e.last_ms[7] = e.last_ms[0] - busy - e.last_ms[6];
        return;
    }
    e.last_ms[0] = el(EV_START, EV_END);
    e.last_ms[7] = el(EV_START, EV_H2D);
    e.last_ms[1] = el(EV_H2D, EV_COUNT);
    e.last_ms[2] = el(EV_COUNT, EV_SCAN);
    e.last_ms[3] = el(EV_SCAN, EV_FILL);
    e.last_ms[4] = el(EV_FILL, EV_ACC);
    e.last_ms[5] = el(EV_ACC, EV_FIXUP);
    e.last_ms[6] = el(EV_FIXUP, EV_END);
}

struct Shard {
    int eng = 0;
    int dev = -1;  // CUDA device of d_pts / d_table (valid after a later kgr_init re-numbered the engines)
    size_t first = 0, count = 0;
    void *d_pts = nullptr;
    void *d_table = nullptr;  // kgr_bases_precompute: W * count affine points, table[w * count + i] = 2^(c*w) * P_i
    uint32_t table_c = 0;
};
}  // namespace kgr

struct kgr_bases {
    int curve = 0;
    size_t n = 0;
    uint64_t generation = 0;  // kgr_init that created it: a handle from an earlier kgr_init is refused by every call but kgr_bases_free
    std::vector<kgr::Shard> shards;
    ~kgr_bases() {  // device memory goes with the handle, also when registration fails half way
        for (auto &s : shards) {
            if (s.dev < 0) continue;
            cudaSetDevice(s.dev);
            if (s.d_pts) cudaFree(s.d_pts);
            if (s.d_table) cudaFree(s.d_table);
        }
    }
};

// An R1CS shape (A, B, C in CSR) resident on the first device (nova/src/relaxed_r1cs.rs R1csShape).
struct kgr_r1cs {
    int field = 0;
    size_t m = 0, n_z = 0;
    uint64_t generation = 0;  // kgr_init that created it (checked by kgr_groth16_prove_r1cs and kgr_groth16_setup)
    size_t nnz[3] = {0, 0, 0};
    kgr::DevBuf<uint32_t> row_ptr[3], cols[3], coeffs[3], z1, z2, t;
    float ms[3] = {0, 0, 0};  // last cross term: H2D of z1 / z2, kernel, commit MSM
    kgr::Csr csr(int i) const { return kgr::Csr{row_ptr[i].p, cols[i].p, coeffs[i].p}; }
};

// A vector of field elements resident on the first device (nova: z, E, T between folding steps).
struct kgr_vec {
    int field = 0;
    size_t n = 0;
    uint64_t generation = 0;
    kgr::DevBuf<uint32_t> d;
};

namespace kgr {

template <class C> static void upload_shard(Engine &e, Shard &s, const uint64_t *xy, const uint8_t *inf) {
    CK(cudaSetDevice(e.dev));
    s.dev = e.dev;
    CK(cudaMalloc(&s.d_pts, std::max<size_t>(s.count, 1) * sizeof(AffinePt<C>)));
    if (s.count == 0) return;
    upload_from_host(e, s.d_pts, xy + (sizeof(AffinePt<C>) / 8) * s.first, s.count * sizeof(AffinePt<C>), e.st);
    if (inf) {
        uint8_t *d_inf = nullptr;
        CK(cudaMalloc(&d_inf, s.count));
        CK(cudaMemcpyAsync(d_inf, inf + s.first, s.count, cudaMemcpyHostToDevice, e.st));
        Launch<C>::fold_inf(e.st, (AffinePt<C> *)s.d_pts, d_inf, (uint32_t)s.count);
        CK(cudaStreamSynchronize(e.st));
        CK(cudaFree(d_inf));
    }
    CK(cudaStreamSynchronize(e.st));
}

static void make_shards(std::vector<Shard> &shards, size_t n) {
    size_t ne = g_engines.size();
    size_t per = (n + ne - 1) / ne;
    for (size_t i = 0; i < ne; i++) {
        Shard s;
        s.eng = (int)i;
        s.first = std::min(n, i * per);
        s.count = std::min(n, (i + 1) * per) - s.first;
        shards.push_back(s);
    }
}

// Host side of the result: per GPU, Horner over its W window sums (c doublings between windows —
// what msm.rs:41 does with c*i doublings per window), then the sum over GPUs and the conversion to
// the reference's projective form.  Runs on the CPU build of field.cuh / curve.cuh.
struct Partial {
    const uint32_t *pts;
    uint32_t count, c;
};
template <class C> static void combine_partials(const std::vector<Partial> &parts, uint64_t *out) {
    constexpr size_t XW = sizeof(XyzzPt<C>) / 4;  // words per XYZZ point
    XyzzPt<C> acc = xyzz_identity<C>();
    for (const Partial &p : parts) {
        if (!p.count) continue;
        XyzzPt<C> r;
        std::memcpy(&r, p.pts + XW * (size_t)(p.count - 1), sizeof r);
        for (uint32_t w = p.count - 1; w-- > 0;) {
            for (uint32_t d = 0; d < p.c; d++) r = xyzz_dbl(r);
            XyzzPt<C> q;
            std::memcpy(&q, p.pts + XW * (size_t)w, sizeof q);
            xyzz_add(r, q);
        }
        xyzz_add(acc, r);
    }
    typename C::Elem o[3];
    xyzz_to_projective(acc, o);
    std::memcpy(out, o, sizeof o);
}

struct HostPts {
    const uint64_t *xy;
    const uint8_t *inf;
};

static bool is_pageable(const void *p) {
    cudaPointerAttributes at;
    if (cudaPointerGetAttributes(&at, p) == cudaSuccess) return at.type == cudaMemoryTypeUnregistered;
    cudaGetLastError();
    return true;
}

// Run an MSM over [off, off+n) of a sharded base vector.  scalars: host pointer unless on_device.
// hp != nullptr: the bases themselves come from host memory for this call only (kgr_msm_oneshot).
// A host-buffer call is bound by PCIe upload + pipeline in sequence (the bucket accumulation of a point needs the point).  MSM is linear, so
// every device's share is cut into pieces that are uploaded back to back on the copy stream while the pieces already on the device are sorted
// and accumulated INTO one shared bucket set (enqueue_msm, StreamPiece); one bucket reduction closes the call.
template <class C>
static void run_msm(std::vector<Shard> &shards, size_t off, const uint64_t *scalars, bool on_device, int fmt, size_t n, uint64_t *out,
                    const HostPts *hp) {
    struct Job {
        Engine *e;
        const AffinePt<C> *pts;
        size_t pt_first, sc_first, count;
        uint32_t table_c, table_stride, table_off;
    };
    const Params P = t_params;  // the calling thread's tuning state, handed to every engine this call drives
    std::vector<Job> jobs;
    for (auto &s : shards) {
        size_t lo = std::max(off, s.first), hi = std::min(off + n, s.first + s.count);
        if (lo >= hi) continue;
        if (!hp && s.d_table)
            jobs.push_back(Job{&g_engines[s.eng], (const AffinePt<C> *)s.d_table, lo, lo - off, hi - lo, s.table_c, (uint32_t)s.count, (uint32_t)(lo - s.first)});
        else
            jobs.push_back(Job{&g_engines[s.eng], hp ? nullptr : (const AffinePt<C> *)s.d_pts + (lo - s.first), lo, lo - off, hi - lo, 0, 0, 0});
    }
    if (on_device && jobs.size() > 1) throw CudaError{cudaErrorInvalidValue, "device-resident scalars need a single-device range", __LINE__};
    int is_mont = (fmt == KGR_SCALARS_MONTGOMERY);
    std::vector<CudaError> errs(jobs.size(), CudaError{cudaSuccess, "", 0});
    auto launch = [&](size_t j) {
        try {
            Job &jb = jobs[j];
            Engine &e = *jb.e;
            e.params = P;
            CK(cudaSetDevice(e.dev));
            CK(cudaEventRecord(e.ev[EV_START], e.st));
            if (on_device) {
                enqueue_msm<C>(e, jb.pts, reinterpret_cast<const uint32_t *>(scalars) + 8 * jb.sc_first, is_mont, (uint32_t)jb.count, jb.table_c, jb.table_stride, jb.table_off);
            } else {
                // pieces: "oneshot_split" / "oneshot_growth" or automatic (tools/probe_e2e_growth.py, profiles/r02_e2e.md).  Nothing overlaps the FIRST
                // piece's upload, so it is the smallest; piece i + 1 is `growth` times piece i, as long as its upload still ends before the
                // pipeline is through with the pieces before it (points + scalars: 1.75 ms of PCIe against 2.35 ms of pipeline per 2^20 pairs, so
                // growth <= 1.3 for long calls; scalars only: a third of the traffic, growth 3).  Each piece pays its sort's fixed part, shorter
                // buckets for the batched-affine levels and a merge pass over all buckets (0.1 - 0.3 ms), which bounds their number:
                // points + scalars 2^20: 2 pieces x 1.7 (4.63 ms; equal halves 4.88, one piece 5.25), 2^24: 5 x 1.3 (46.7; four equal pieces 49.0, one 66.0);
                // scalars only 2^20: one piece (4.25), 2^24: 3 x 3.0 (42.4; equal 44.7, one 49.0).
                size_t lg = 0;
                while (((size_t)2 << lg) <= jb.count) lg++;  // floor(log2(count))
                size_t k_auto = hp ? (lg < 20 ? 1 : lg < 22 ? 2 : lg == 22 ? 3 : lg == 23 ? 4 : 5) : (lg < 22 ? 1 : lg < 24 ? 2 : 3);
                size_t k = P.oneshot_split > 0 ? (size_t)P.oneshot_split : k_auto;
                k = std::min<size_t>(std::min<size_t>(k, MAX_PIECES), std::max<size_t>(jb.count, 1));
                // growth = 1.3 x (pipeline time of the call) / (upload time of the call), from what this engine measured on its last calls: with a fast
                // link the pipeline is the bottleneck and the pieces grow (the first upload overlaps nothing), with a slow or contended link (eight
                // processes uploading at once) the uploads are, and the pieces shrink (after the last byte only the last piece's work remains).  With the
                // default rate (42 GB/s): 2^20 points + scalars 1.7, 2^24 1.3, scalars only 3 — the values the sweeps of profiles/r02_e2e.md found.
                const double up_bytes = (double)jb.count * (32.0 + (hp ? (double)sizeof(AffinePt<C>) : 0.0));
                // device time per pair: 3.1 ns at 2^20, 2.6 at 2^22, 2.3 from 2^24 on (section 4 of DESIGN.md); Fq2 coordinates cost 3.5 times that
                const double ns_per_pair = (jb.count >= (1u << 23) ? 2.35 : jb.count >= (1u << 21) ? 2.6 : 3.1) * (C::ID == Bn254G2::ID ? 3.5 : 1.0);
                const double up_ms = up_bytes / (e.h2d_gbs * 1e6), dev_ms = ns_per_pair * (double)jb.count * 1e-6;
                const double growth = P.oneshot_growth > 0 ? (double)P.oneshot_growth / 100.0 : std::min(3.0, std::max(0.6, 1.3 * dev_ms / up_ms));
                std::vector<size_t> cut(k + 1, 0);
                {
                    double tot_w = 0, w = 1, acc_w = 0;
                    for (size_t i = 0; i < k; i++, w *= growth) tot_w += w;
                    w = 1;
                    for (size_t i = 0; i < k; i++, w *= growth) {
                        acc_w += w;
                        cut[i + 1] = i + 1 == k ? jb.count : std::min<size_t>(jb.count, (size_t)((double)jb.count * (acc_w / tot_w)));
                    }
                }
                e.scalars.ensure(std::max<size_t>(jb.count, 1) * 8);
                if (hp) {
                    e.oneshot_pts.ensure(std::max<size_t>(jb.count, 1) * sizeof(AffinePt<C>));
                    if (hp->inf) e.oneshot_inf.ensure(std::max<size_t>(jb.count, 1));
                    jb.pts = (const AffinePt<C> *)e.oneshot_pts.p;
                }
                std::vector<StreamPiece> pieces;
                for (size_t i = 0; i < k; i++) {
                    size_t lo = cut[i], hi = cut[i + 1];
                    if (lo >= hi && !(i + 1 == k && pieces.empty())) continue;  // an empty piece of a tiny call (the last one is kept if nothing else exists)
                    if (!e.ev_piece_sc[i]) {
                        CK(cudaEventCreateWithFlags(&e.ev_piece_sc[i], cudaEventDisableTiming));
                        CK(cudaEventCreateWithFlags(&e.ev_piece_pts[i], cudaEventDisableTiming));
                    }
                    pieces.push_back(StreamPiece{lo, hi - lo, e.ev_piece_sc[i], hp ? e.ev_piece_pts[i] : nullptr, nullptr});
                }
                std::atomic<size_t> recorded(0);
                CudaError up_err{cudaSuccess, "", 0};
                // uploads, piece after piece on the copy stream (scalars first: the sort only needs them); the copy stream starts after
                // everything enqueued on the main stream so far (the previous call's kernels may still read the buffers)
                auto upload_all = [&]() {
                    try {
                        CK(cudaSetDevice(e.dev));
                        CK(cudaStreamWaitEvent(e.st_copy, e.ev[EV_START], 0));
                        if (!e.ev_up0) {
                            CK(cudaEventCreate(&e.ev_up0));
                            CK(cudaEventCreate(&e.ev_up1));
                        }
                        CK(cudaEventRecord(e.ev_up0, e.st_copy));
                        for (size_t i = 0; i < pieces.size(); i++) {
                            const StreamPiece &pc = pieces[i];
                            upload_from_host(e, e.scalars.p + 8 * pc.first, scalars + 4 * (jb.sc_first + pc.first), pc.count * 32, e.st_copy);
                            CK(cudaEventRecord(pc.ev_sc, e.st_copy));
                            if (hp) {
                                AffinePt<C> *dst = (AffinePt<C> *)e.oneshot_pts.p + pc.first;
                                upload_from_host(e, dst, hp->xy + (sizeof(AffinePt<C>) / 8) * (jb.pt_first + pc.first), pc.count * sizeof(AffinePt<C>), e.st_copy);
                                if (hp->inf) {
                                    CK(cudaMemcpyAsync(e.oneshot_inf.p + pc.first, hp->inf + jb.pt_first + pc.first, pc.count, cudaMemcpyHostToDevice, e.st_copy));
                                    Launch<C>::fold_inf(e.st_copy, dst, e.oneshot_inf.p + pc.first, (uint32_t)pc.count);
                                    e.launches++;
                                }
                                CK(cudaEventRecord(pc.ev_pts, e.st_copy));
                            }
                            if (i + 1 == pieces.size()) CK(cudaEventRecord(e.ev_up1, e.st_copy));
                            recorded.store(i + 1, std::memory_order_release);
                        }
                    } catch (CudaError &ce) {
                        up_err = ce;
                        recorded.store(pieces.size(), std::memory_order_release);  // never leave the enqueueing thread waiting
                    }
                };
                // Pinned sources: the copies are enqueued at once, from this thread.  Pageable sources are staged through pinned slots by host
                // threads (upload_from_host), which takes as long as the transfer itself: a second thread does that while this one enqueues the
                // pieces that are already on their way.
                const bool threaded = pieces.size() > 1 && (is_pageable(scalars) || (hp && is_pageable(hp->xy)));
                std::thread uploader;
                if (threaded) {
                    for (auto &pc : pieces) pc.recorded = &recorded;
                    uploader = std::thread(upload_all);
                } else {
                    upload_all();
                }
                try {
                    enqueue_msm<C>(e, jb.pts, e.scalars.p, is_mont, (uint32_t)jb.count, jb.table_c, jb.table_stride, jb.table_off, &pieces);
                } catch (...) {
                    if (uploader.joinable()) uploader.join();
                    throw;
                }
                if (uploader.joinable()) uploader.join();
                if (up_err.e != cudaSuccess) throw up_err;
                CK(cudaStreamSynchronize(e.st));
                collect_timing(e);
                // what this call saw, for the piece sizes of the next one (calls large enough for the figures to mean something)
                float up_meas = 0;
                if (jb.count >= (1u << 18) && cudaEventSynchronize(e.ev_up1) == cudaSuccess && cudaEventElapsedTime(&up_meas, e.ev_up0, e.ev_up1) == cudaSuccess &&
                    up_meas > 0.05f) {
                    const double rate = up_bytes / (up_meas * 1e6);
                    e.h2d_gbs = 0.5 * e.h2d_gbs + 0.5 * std::min(80.0, std::max(2.0, rate));
                }
                cudaGetLastError();
                return;
            }
            CK(cudaStreamSynchronize(e.st));
            collect_timing(e);
        } catch (CudaError &ce) {
            errs[j] = ce;
        }
    };
    if (jobs.size() <= 1) {
        for (size_t j = 0; j < jobs.size(); j++) launch(j);
    } else {
        std::vector<std::thread> th;
        for (size_t j = 0; j < jobs.size(); j++) th.emplace_back(launch, j);
        for (auto &t : th) t.join();
    }
    for (auto &ce : errs)
        if (ce.e != cudaSuccess) throw ce;
    std::vector<Partial> parts;
    for (auto &jb : jobs) parts.push_back(Partial{jb.e->h_result, jb.e->n_result, jb.e->result_c});
    auto t0 = std::chrono::steady_clock::now();
    combine_partials<C>(parts, out);
    float host_ms = std::chrono::duration<float, std::milli>(std::chrono::steady_clock::now() - t0).count();
    for (auto &jb : jobs) {
        jb.e->last_ms[8] = host_ms;
        jb.e->last_ms[0] += host_ms;  // total = device events + host finish
    }
}

// ---- kgr_msm_batch: one single-shard MSM per lane, started without waiting and finished later --------------------------
template <class C> static void lane_enqueue(Engine &e, const Shard &s, size_t off, const uint32_t *d_scalars, int fmt, size_t n) {
    size_t first = off - s.first;
    if (s.d_table)
        enqueue_msm<C>(e, (const AffinePt<C> *)s.d_table, d_scalars, fmt == KGR_SCALARS_MONTGOMERY, (uint32_t)n, s.table_c, (uint32_t)s.count, (uint32_t)first);
    else
        enqueue_msm<C>(e, (const AffinePt<C> *)s.d_pts + first, d_scalars, fmt == KGR_SCALARS_MONTGOMERY, (uint32_t)n);
}
template <class C> static void lane_start(Engine &e, const Params &P, const Shard &s, size_t off, const uint64_t *scalars, int fmt, size_t n) {
    e.params = P;
    CK(cudaSetDevice(e.dev));
    CK(cudaEventRecord(e.ev[EV_START], e.st));
    e.scalars.ensure(std::max<size_t>(n, 1) * 8);
    upload_from_host(e, e.scalars.p, scalars, n * 32, e.st);
    lane_enqueue<C>(e, s, off, e.scalars.p, fmt, n);
}
// Montgomery scalars already on the lane's device; the lane's stream first waits for `ready` (recorded where the scalars were produced)
template <class C> static void lane_start_device(Engine &e, const Params &P, const Shard &s, size_t off, const uint32_t *d_scalars, size_t n, cudaEvent_t ready) {
    e.params = P;
    CK(cudaSetDevice(e.dev));
    CK(cudaStreamWaitEvent(e.st, ready, 0));
    CK(cudaEventRecord(e.ev[EV_START], e.st));
    lane_enqueue<C>(e, s, off, d_scalars, KGR_SCALARS_MONTGOMERY, n);
}
template <class C> static void lane_finish(Engine &e, uint64_t *out) {
    CK(cudaSetDevice(e.dev));
    CK(cudaStreamSynchronize(e.st));
    collect_timing(e);
    std::vector<Partial> parts{Partial{e.h_result, e.n_result, e.result_c}};
    combine_partials<C>(parts, out);
}

// in: 3 coordinates, out: x, y (Montgomery) and one trailing word = is_infinity
template <class C> static void proj_to_affine_host(const uint64_t *in, uint64_t *out) {
    typedef typename C::Elem E;
    constexpr size_t EB = sizeof(E), EL = sizeof(E) / 8;
    E x, y, z;
    std::memcpy(&x, in, EB);
    std::memcpy(&y, in + EL, EB);
    std::memcpy(&z, in + 2 * EL, EB);
    if (fp_is_zero(z)) {
        E zero = El<E>::zero(), one = El<E>::one();
        std::memcpy(out, &zero, EB);
        std::memcpy(out + EL, &one, EB);
        out[2 * EL] = 1;
        return;
    }
    E zi = fp_inv(z);
    E ax = fp_mul(x, zi), ay = fp_mul(y, zi);
    std::memcpy(out, &ax, EB);
    std::memcpy(out + EL, &ay, EB);
    out[2 * EL] = 0;
}

// (X : Y : Z) homogeneous -> XYZZ with zz = Z^2, zzz = Z^3, X' = X*Z, Y' = Y*Z^2
template <class C> static XyzzPt<C> proj_to_xyzz_host(const uint64_t *in) {
    typedef typename C::Elem E;
    constexpr size_t EB = sizeof(E), EL = sizeof(E) / 8;
    E x, y, z;
    std::memcpy(&x, in, EB);
    std::memcpy(&y, in + EL, EB);
    std::memcpy(&z, in + 2 * EL, EB);
    if (fp_is_zero(z)) return xyzz_identity<C>();
    XyzzPt<C> r;
    r.zz = fp_sqr(z);
    r.zzz = fp_mul(r.zz, z);
    r.x = fp_mul(x, z);
    r.y = fp_mul(y, r.zz);
    return r;
}

template <class F, int FIELD_ID> static int test_field_op(Engine &e, int op, const uint64_t *a, const uint64_t *b, size_t n, uint64_t *out) {
    CK(cudaSetDevice(e.dev));
    Fp<F> *da = nullptr, *db = nullptr, *dout = nullptr;
    CK(cudaMalloc(&da, n * 32));
    CK(cudaMalloc(&dout, n * 32));
    // uploads go on the engine stream: it is non-blocking, so a legacy-stream cudaMemcpy from pageable memory would not be ordered before the kernel
    CK(cudaMemcpyAsync(da, a, n * 32, cudaMemcpyHostToDevice, e.st));
    if (b) {
        CK(cudaMalloc(&db, n * 32));
        CK(cudaMemcpyAsync(db, b, n * 32, cudaMemcpyHostToDevice, e.st));
    }
    LaunchUtil::field_op(e.st, FIELD_ID, op, da, db, dout, (uint32_t)n);
    CK(cudaGetLastError());
    CK(cudaStreamSynchronize(e.st));
    CK(cudaMemcpy(out, dout, n * 32, cudaMemcpyDeviceToHost));
    cudaFree(da);
    cudaFree(dout);
    if (db) cudaFree(db);
    return 0;
}

template <class C>
static int test_point_op(Engine &e, int op, const uint64_t *a, const uint8_t *ainf, const uint64_t *b, const uint8_t *binf, size_t n, uint64_t *out) {
    CK(cudaSetDevice(e.dev));
    Shard sa, sb;
    sa.count = sb.count = n;
    upload_shard<C>(e, sa, a, ainf);
    upload_shard<C>(e, sb, b, binf);
    uint32_t *dout = nullptr;
    const size_t PB = 3 * sizeof(typename C::Elem);  // bytes per projective result
    CK(cudaMalloc(&dout, n * PB));
    Launch<C>::point_op(e.st, op, (AffinePt<C> *)sa.d_pts, (AffinePt<C> *)sb.d_pts, dout, (uint32_t)n);
    CK(cudaGetLastError());
    CK(cudaStreamSynchronize(e.st));
    CK(cudaMemcpy(out, dout, n * PB, cudaMemcpyDeviceToHost));
    cudaFree(dout);
    cudaFree(sa.d_pts);
    cudaFree(sb.d_pts);
    return 0;
}

template <class C> static AffinePt<C> generator_affine();
template <> AffinePt<Bn254G1> generator_affine<Bn254G1>() {  // bn254/src/params.rs:8-9: (1, 2)
    AffinePt<Bn254G1> g;
    g.x = fp_one<FqP>();
    Fp<FqP> two = fp_zero<FqP>();
    two.v[0] = 2;
    g.y = fp_to_mont(two);
    return g;
}
template <> AffinePt<GrumpkinC> generator_affine<GrumpkinC>() {  // grumpkin/src/params.rs:4-11 (Montgomery limbs as stored)
    AffinePt<GrumpkinC> g;
    g.x = fp_one<FrP>();
    const uint64_t gy[4] = {0x11b2dff1448c41d8ULL, 0x23d3446f21c77dc3ULL, 0xaa7b8cf435dfafbbULL, 0x14b34cf69dc25d68ULL};
    std::memcpy(&g.y, gy, 32);
    return g;
}

template <> AffinePt<Bn254G2> generator_affine<Bn254G2>() {  // bn254/src/params.rs:15-42 (canonical limbs there; Montgomery here)
    const uint64_t c[4][4] = {{0x46debd5cd992f6edULL, 0x674322d4f75edaddULL, 0x426a00665e5c4479ULL, 0x1800deef121f1e76ULL},
                              {0x97e485b7aef312c2ULL, 0xf1aa493335a9e712ULL, 0x7260bfb731fb5d25ULL, 0x198e9393920d483aULL},
                              {0x4ce6cc0166fa7daaULL, 0xe3d1e7690c43d37bULL, 0x4aab71808dcb408fULL, 0x12c85ea5db8c6debULL},
                              {0x55acdadcd122975bULL, 0xbc4b313370b38ef3ULL, 0xec9e99ad690c3395ULL, 0x090689d0585ff075ULL}};
    Fp<FqP> m[4];
    for (int i = 0; i < 4; i++) {
        std::memcpy(&m[i], c[i], 32);
        m[i] = fp_to_mont(m[i]);
    }
    AffinePt<Bn254G2> g;
    g.x = Fp2<FqP>{m[0], m[1]};
    g.y = Fp2<FqP>{m[2], m[3]};
    return g;
}

// The generator's window table on engine e (built once per curve and device).
template <class C> static const AffinePt<C> *fixed_table(Engine &e) {
    DevBuf<uint8_t> &buf = e.fixed_table[C::ID];
    if (!buf.p) {
        buf.ensure(Launch<C>::fixed_table_points() * sizeof(AffinePt<C>));
        Launch<C>::fixed_table(e.st, generator_affine<C>(), (AffinePt<C> *)buf.p);
        e.launches++;
        CK(cudaGetLastError());
    }
    return (const AffinePt<C> *)buf.p;
}

template <class C> static void generate_shard(Engine &e, Shard &s, uint64_t seed, uint64_t first, uint64_t *k_out) {
    typedef Fp<typename C::Scalar> S;
    CK(cudaSetDevice(e.dev));
    s.dev = e.dev;
    CK(cudaMalloc(&s.d_pts, std::max<size_t>(s.count, 1) * sizeof(AffinePt<C>)));
    if (!s.count) return;
    S *dk = nullptr;
    CK(cudaMalloc(&dk, s.count * sizeof(S)));
    uint32_t n = (uint32_t)s.count;
    Launch<C>::gen_scalars(e.st, seed, first + (uint64_t)s.first, n, dk);
    Launch<C>::fixed_base(e.st, dk, fixed_table<C>(e), n, (AffinePt<C> *)s.d_pts);
    CK(cudaGetLastError());
    CK(cudaStreamSynchronize(e.st));
    if (k_out) CK(cudaMemcpy(k_out + 4 * s.first, dk, s.count * sizeof(S), cudaMemcpyDeviceToHost));
    CK(cudaFree(dk));
}

// A new single-shard handle on engine e holding k[i] * G for i < n (device scalars, Montgomery): a zero scalar gives (0, 0), the identity as
// registered handles store it (k_fold_inf).
template <class C> static std::unique_ptr<kgr_bases> fixed_base_handle(Engine &e, int curve, const void *d_k, size_t n) {
    std::unique_ptr<kgr_bases> b(new kgr_bases);
    b->curve = curve;
    b->n = n;
    b->generation = g_generation;
    make_shards(b->shards, n);
    Shard &s = b->shards[0];
    s.dev = e.dev;
    CK(cudaMalloc(&s.d_pts, std::max<size_t>(n, 1) * sizeof(AffinePt<C>)));
    if (n) {
        Launch<C>::fixed_base(e.st, (const Fp<typename C::Scalar> *)d_k, fixed_table<C>(e), (uint32_t)n, (AffinePt<C> *)s.d_pts);
        e.launches++;
        CK(cudaGetLastError());
    }
    return b;
}

static double ubench_mode(Engine &e, int mode, uint32_t *sink, double ops_per_thread_iter) {
    const int iters = 2000, blocks = e.sm_count * 8, tpb = 256;
    LaunchUtil::ubench(e.st, mode, blocks, sink, 10);
    cudaEvent_t a, b;
    CK(cudaEventCreate(&a));
    CK(cudaEventCreate(&b));
    CK(cudaEventRecord(a, e.st));
    LaunchUtil::ubench(e.st, mode, blocks, sink, iters);
    CK(cudaEventRecord(b, e.st));
    CK(cudaStreamSynchronize(e.st));
    float ms = 0;
    CK(cudaEventElapsedTime(&ms, a, b));
    cudaEventDestroy(a);
    cudaEventDestroy(b);
    return (double)blocks * tpb * iters * ops_per_thread_iter / (ms * 1e-3) / 1e9;
}

// ---- Fr NTT (SURVEY.md 8f N2) -----------------------------------------------------------------------
static Fp<FrP> fr_from_u64(uint64_t v) {
    Fp<FrP> x = fp_zero<FrP>();
    x.v[0] = (uint32_t)v;
    x.v[1] = (uint32_t)(v >> 32);
    return fp_to_mont(x);
}
static Fp<FrP> fr_pow2k(Fp<FrP> x, uint32_t squarings) {
    for (uint32_t i = 0; i < squarings; i++) x = fp_sqr(x);
    return x;
}
static NttDomain &ntt_domain(Engine &e, uint32_t k) {
    auto it = e.ntt_domains.find(k);
    if (it != e.ntt_domains.end()) return *it->second;
    auto d = std::make_shared<NttDomain>();
    d->k = k;
    const uint32_t n = 1u << k;
    // fr.rs:60-65 ROOT_OF_UNITY = to_mont_form(limbs); S = 28 (fr.rs:53); omega = root^(2^(S-k)) (fft.rs:35)
    Fp<FrP> root = fp_zero<FrP>();
    const uint64_t rl[4] = {0xd34f1ed960c37c9cULL, 0x3215cf6dd39329c8ULL, 0x98865ea93dd31f74ULL, 0x03ddb9f5166d18b7ULL};
    std::memcpy(root.v, rl, 32);
    root = fp_to_mont(root);
    Fp<FrP> omega = fr_pow2k(root, 28 - k), omega_inv = fp_inv(omega);
    Fp<FrP> g = fr_from_u64(7), g_inv = fp_inv(g);  // MULTIPLICATIVE_GENERATOR (fr.rs:18,21)
    d->n_inv = fp_inv(fr_from_u64(n));
    Fp<FrP> gn = fr_pow2k(g, k);                     // 7^(2^k)
    d->z_inv = fp_inv(fp_sub(gn, fp_one<FrP>()));
    d->tw.ensure((size_t)std::max(1u, n / 2) * 32);
    d->inv_tw.ensure((size_t)std::max(1u, n / 2) * 32);
    d->cosets.ensure((size_t)n * 32);
    d->inv_cosets.ensure((size_t)n * 32);
    LaunchNtt::pow_table(e.st, d->tw.p, &omega, std::max(1u, n / 2));
    LaunchNtt::pow_table(e.st, d->inv_tw.p, &omega_inv, std::max(1u, n / 2));
    LaunchNtt::pow_table(e.st, d->cosets.p, &g, n);
    LaunchNtt::pow_table(e.st, d->inv_cosets.p, &g_inv, n);
    CK(cudaGetLastError());
    CK(cudaStreamSynchronize(e.st));
    e.launches += 4;
    e.ntt_domains[k] = d;
    return *d;
}
// op: 0 dft, 1 idft, 2 coset_dft, 3 coset_idft (fft.rs:92-127), in place on 2^k device elements
static void ntt_enqueue(Engine &e, NttDomain &d, void *buf, int op) {
    const uint32_t n = 1u << d.k;
    switch (op) {
        case 0: e.launches += LaunchNtt::transform(e.st, buf, d.tw.p, d.k); break;
        case 1:
            e.launches += LaunchNtt::transform(e.st, buf, d.inv_tw.p, d.k);
            LaunchNtt::scale(e.st, buf, nullptr, &d.n_inv, n);
            e.launches++;
            break;
        case 2:
            LaunchNtt::scale(e.st, buf, d.cosets.p, nullptr, n);
            e.launches += 1 + LaunchNtt::transform(e.st, buf, d.tw.p, d.k);
            break;
        default:
            e.launches += LaunchNtt::transform(e.st, buf, d.inv_tw.p, d.k);
            LaunchNtt::scale(e.st, buf, d.inv_cosets.p, &d.n_inv, n);
            e.launches++;
            break;
    }
}
static size_t stripped_len(const uint64_t *v, size_t n) {  // Coefficients::new (poly.rs:61-63)
    while (n && !(v[4 * (n - 1)] | v[4 * (n - 1) + 1] | v[4 * (n - 1) + 2] | v[4 * (n - 1) + 3])) n--;
    return n;
}
static void upload_padded(Engine &e, void *dbuf, const uint64_t *src, size_t n_in, size_t n) {
    size_t m = std::min(n_in, n);
    upload_from_host(e, dbuf, src, m * 32, e.st);
    if (m < n) CK(cudaMemsetAsync((uint8_t *)dbuf + m * 32, 0, (n - m) * 32, e.st));
}

// prover.rs:36-47 on the three evaluation vectors in e.ntt_buf[0..2] (2^k elements each; in bit-reversed order when bitrev_input), enqueued on
// e.st: leaves the 2^k coefficients of H in e.ntt_buf[0] (device).
static void enqueue_groth16_h_transforms(Engine &e, NttDomain &d, bool bitrev_input) {
    const size_t n = (size_t)1 << d.k;
    for (int i = 0; i < 3; i++) {
        // idft then coset_dft (prover.rs:36-41); the 1/n and coset scalings are one elementwise pass
        if (bitrev_input) e.launches += LaunchNtt::transform_bitrev_input(e.st, e.ntt_buf[i].p, d.inv_tw.p, d.k);
        else e.launches += LaunchNtt::transform(e.st, e.ntt_buf[i].p, d.inv_tw.p, d.k);
        LaunchNtt::scale(e.st, e.ntt_buf[i].p, d.cosets.p, &d.n_inv, (uint32_t)n);
        e.launches += 1 + LaunchNtt::transform(e.st, e.ntt_buf[i].p, d.tw.p, d.k);
    }
    LaunchNtt::h_pointwise(e.st, e.ntt_buf[0].p, e.ntt_buf[1].p, e.ntt_buf[2].p, &d.z_inv, (uint32_t)n);  // prover.rs:43-46
    e.launches++;
    ntt_enqueue(e, d, e.ntt_buf[0].p, 3);                                                             // coset_idft, prover.rs:47
}
// The same from host evaluations: uploads a, b, c (m evaluations each, zero padded) first.
static void enqueue_groth16_h(Engine &e, NttDomain &d, const uint64_t *a, const uint64_t *b, const uint64_t *c, size_t m) {
    const size_t n = (size_t)1 << d.k;
    const uint64_t *src[3] = {a, b, c};
    for (int i = 0; i < 3; i++) {
        e.ntt_buf[i].ensure(n * 32);
        upload_padded(e, e.ntt_buf[i].p, src[i], m, n);
    }
    CK(cudaEventRecord(e.ev[EV_H2D], e.st));
    enqueue_groth16_h_transforms(e, d, false);
}


static int guarded(const std::function<int()> &f) {
    try {
        return f();
    } catch (CudaError &ce) {
        char buf[512];
        std::snprintf(buf, sizeof buf, "CUDA error %d (%s) at msm.cu:%d: %s", (int)ce.e, cudaGetErrorString(ce.e), ce.line, ce.what);
        cudaGetLastError();
        return fail(ce.e == cudaErrorInvalidValue ? KGR_E_ARG : KGR_E_CUDA, buf);
    } catch (std::exception &ex) {
        return fail(KGR_E_CUDA, std::string("exception: ") + ex.what());
    } catch (...) {
        return fail(KGR_E_CUDA, "unknown exception");
    }
}

static inline size_t affine_bytes(int curve) { return curve == KGR_CURVE_BN254_G2 ? 128 : 64; }  // x || y

#define DISPATCH(curve, CALL)                                              \
    do {                                                                   \
        if ((curve) == KGR_CURVE_BN254_G1) { CALL(Bn254G1); }              \
        else if ((curve) == KGR_CURVE_GRUMPKIN) { CALL(GrumpkinC); }       \
        else if ((curve) == KGR_CURVE_BN254_G2) { CALL(Bn254G2); }         \
        else return fail(KGR_E_ARG, "unknown curve id");                   \
    } while (0)

// f((C *)nullptr) for the curve type C of an id already validated (DISPATCH for code that cannot return an error code)
template <class F> static void with_curve(int curve, F &&f) {
    if (curve == KGR_CURVE_BN254_G1) f((Bn254G1 *)nullptr);
    else if (curve == KGR_CURVE_GRUMPKIN) f((GrumpkinC *)nullptr);
    else f((Bn254G2 *)nullptr);
}

}  // namespace kgr

using namespace kgr;

extern "C" {

const char *kgr_last_error(void) { return g_err.c_str(); }

int kgr_init(const int *devices, int n_devices) {
    std::lock_guard<std::mutex> lk(g_mu);
    return guarded([&]() -> int {
        int count = 0;
        cudaError_t ce = cudaGetDeviceCount(&count);
        if (ce != cudaSuccess || count == 0) {
            cudaGetLastError();
            return fail(KGR_E_NO_DEVICE, std::string("no CUDA device: ") + cudaGetErrorString(ce));
        }
        destroy_lanes();
        for (auto &e : g_engines) e.destroy();
        g_engines.clear();
        std::vector<int> devs;
        if (!devices || n_devices <= 0) {
            int cur = 0;
            CK(cudaGetDevice(&cur));
            devs.push_back(cur);
        } else {
            for (int i = 0; i < n_devices; i++) {
                if (devices[i] < 0 || devices[i] >= count) return fail(KGR_E_ARG, "device index out of range");
                devs.push_back(devices[i]);
            }
        }
        g_engines.resize(devs.size());
        for (size_t i = 0; i < devs.size(); i++) g_engines[i].init(devs[i]);
        g_generation++;
        return KGR_OK;
    });
}

int kgr_shutdown(void) {
    std::lock_guard<std::mutex> lk(g_mu);
    destroy_lanes();
    for (auto &e : g_engines) e.destroy();
    g_engines.clear();
    return KGR_OK;
}

int kgr_device_count(void) { return (int)g_engines.size(); }

int kgr_set_param(const char *name, long value) {
    std::string s(name ? name : "");
    if (s == "window_bits") t_params.window_bits = value;
    else if (s == "chunk") t_params.chunk = value;
    else if (s == "reduce_fanin") {
        if (value < 2 || (value & (value - 1))) return fail(KGR_E_ARG, "reduce_fanin must be a power of two >= 2");
        t_params.reduce_fanin = value;
    } else if (s == "final_on_device") t_params.final_on_device = value;
    else if (s == "running_sum_stop") t_params.running_sum_stop = std::max<long>(1, value);
    else if (s == "sort_mode") t_params.sort_mode = value;
    else if (s == "reduce_mode") t_params.reduce_mode = value;
    else if (s == "lane_threads") t_params.lane_threads = value ? 1 : 0;
    else if (s == "oneshot_split") t_params.oneshot_split = std::min<long>(std::max<long>(value, 0), (long)MAX_LANES);
    else if (s == "oneshot_growth") t_params.oneshot_growth = std::min<long>(std::max<long>(value, 0), 1000);
    else if (s == "affine_levels") t_params.affine_levels = std::min<long>(std::max<long>(value, -1), 5);
    else if (s == "dense_x") t_params.dense_x = std::min<long>(std::max<long>(value, -1), 1);
    else return fail(KGR_E_ARG, "unknown parameter");
    return KGR_OK;
}

int kgr_bases_register(int curve, const uint64_t *xy, const uint8_t *inf, size_t n, kgr_bases_t **out) {
    std::lock_guard<std::mutex> lk(g_mu);
    if (g_engines.empty()) return fail(KGR_E_NOT_INIT, "kgr_init has not been called");
    if (!out || (!xy && n)) return fail(KGR_E_ARG, "null pointer");
    if (curve < KGR_CURVE_BN254_G1 || curve > KGR_CURVE_BN254_G2) return fail(KGR_E_ARG, "unknown curve id");
    if (n >= (1ull << 31)) return fail(KGR_E_TOO_LARGE, "at most 2^31 - 1 bases per vector");
    return guarded([&]() -> int {
        std::unique_ptr<kgr_bases> b(new kgr_bases);  // frees the shards uploaded so far if a later one throws
        b->curve = curve;
        b->n = n;
        b->generation = g_generation;
        make_shards(b->shards, n);
#define CALL(C) for (auto &s : b->shards) upload_shard<C>(g_engines[s.eng], s, xy, inf)
        DISPATCH(curve, CALL);
#undef CALL
        *out = b.release();
        return KGR_OK;
    });
}

int kgr_bases_free(kgr_bases_t *b) {
    std::lock_guard<std::mutex> lk(g_mu);
    if (!b) return KGR_OK;
    delete b;  // ~kgr_bases frees the shards on the devices they were allocated on, whatever kgr_init has done since
    return KGR_OK;
}

size_t kgr_bases_len(const kgr_bases_t *b) { return b ? b->n : 0; }

int kgr_bases_precompute(kgr_bases_t *b, int window_bits) {
    std::lock_guard<std::mutex> lk(g_mu);
    if (g_engines.empty()) return fail(KGR_E_NOT_INIT, "kgr_init has not been called");
    if (!b) return fail(KGR_E_ARG, "null pointer");
    if (b->generation != g_generation) return fail(KGR_E_ARG, "base handle was created before the last kgr_init");
    if (window_bits < 0 || window_bits > 24) return fail(KGR_E_ARG, "window_bits out of range");
    return guarded([&]() -> int {
        for (auto &s : b->shards) {
            if (!s.count) continue;
            Engine &e = g_engines[s.eng];
            CK(cudaSetDevice(e.dev));
            uint32_t c = window_bits ? (uint32_t)window_bits : choose_window_bits_collapsed((uint32_t)s.count, b->curve == KGR_CURVE_BN254_G2 ? 3.0 : 1.0);
            uint32_t W = (255 + c - 1) / c;
            if ((uint64_t)W * s.count >= (1ull << 31)) return fail(KGR_E_TOO_LARGE, "precomputed table would exceed 2^31 points");
            if (s.d_table) CK(cudaFree(s.d_table));
            s.d_table = nullptr;
            s.table_c = 0;
            CK(cudaMalloc(&s.d_table, (size_t)W * s.count * affine_bytes(b->curve)));
#define CALL(C) Launch<C>::precompute(e.st, (uint32_t)s.count, c, W, (uint32_t)s.count, (const AffinePt<C> *)s.d_pts, (AffinePt<C> *)s.d_table)
            DISPATCH(b->curve, CALL);
#undef CALL
            CK(cudaGetLastError());
            CK(cudaStreamSynchronize(e.st));
            s.table_c = c;
        }
        return KGR_OK;
    });
}

static int msm_common(kgr_bases_t *b, size_t off, const uint64_t *scalars, bool on_device, int fmt, size_t n, uint64_t *out) {
    if (g_engines.empty()) return fail(KGR_E_NOT_INIT, "kgr_init has not been called");
    if (!b || !out || (!scalars && n)) return fail(KGR_E_ARG, "null pointer");
    if (b->generation != g_generation) return fail(KGR_E_ARG, "base handle was created before the last kgr_init");
    if (off > b->n || n > b->n - off) return fail(KGR_E_ARG, "range exceeds the registered vector");
    if (fmt != KGR_SCALARS_MONTGOMERY && fmt != KGR_SCALARS_CANONICAL) return fail(KGR_E_ARG, "unknown scalar format");
    return guarded([&]() -> int {
#define CALL(C) run_msm<C>(b->shards, off, scalars, on_device, fmt, n, out, nullptr)
        DISPATCH(b->curve, CALL);
#undef CALL
        return KGR_OK;
    });
}

int kgr_msm(kgr_bases_t *b, size_t off, const uint64_t *scalars, int fmt, size_t n, uint64_t *out) {
    std::lock_guard<std::mutex> lk(g_mu);
    return msm_common(b, off, scalars, false, fmt, n, out);
}

int kgr_msm_device(kgr_bases_t *b, size_t off, const void *d_scalars, int fmt, size_t n, uint64_t *out) {
    std::lock_guard<std::mutex> lk(g_mu);
    return msm_common(b, off, (const uint64_t *)d_scalars, true, fmt, n, out);
}

int kgr_msm_batch(const kgr_msm_job_t *jobs, size_t n_jobs) {
    if (!jobs && n_jobs) return fail(KGR_E_ARG, "null pointer");
    bool overlap;
    {
        std::lock_guard<std::mutex> lk(g_mu);
        if (g_engines.empty()) return fail(KGR_E_NOT_INIT, "kgr_init has not been called");
        overlap = g_engines.size() == 1 && n_jobs > 1;
        for (size_t j = 0; j < n_jobs && overlap; j++) {
            const kgr_msm_job_t &jb = jobs[j];
            if (!jb.bases || jb.bases->shards.size() != 1) overlap = false;
        }
    }
    if (!overlap) {  // several devices (every MSM is already spread over all of them) or a single job: plain sequence
        for (size_t j = 0; j < n_jobs; j++) {
            int rc = kgr_msm(jobs[j].bases, jobs[j].base_off, jobs[j].scalars, jobs[j].scalar_fmt, jobs[j].n, jobs[j].out);
            if (rc) return rc;
        }
        return KGR_OK;
    }
    std::lock_guard<std::mutex> lk(g_mu);
    for (size_t j = 0; j < n_jobs; j++) {
        const kgr_msm_job_t &jb = jobs[j];
        if (!jb.out || (!jb.scalars && jb.n)) return fail(KGR_E_ARG, "null pointer");
        if (jb.base_off > jb.bases->n || jb.n > jb.bases->n - jb.base_off) return fail(KGR_E_ARG, "range exceeds the registered vector");
        if (jb.scalar_fmt != KGR_SCALARS_MONTGOMERY && jb.scalar_fmt != KGR_SCALARS_CANONICAL) return fail(KGR_E_ARG, "unknown scalar format");
        if (jb.bases->curve < KGR_CURVE_BN254_G1 || jb.bases->curve > KGR_CURVE_BN254_G2) return fail(KGR_E_ARG, "unknown curve id");
        if (jb.bases->generation != g_generation) return fail(KGR_E_ARG, "base handle was created before the last kgr_init");
    }
    const Params P = t_params;
    return guarded([&]() -> int {
        size_t n_lanes = std::min(n_jobs, MAX_LANES);
        ensure_lanes(0, n_lanes);
        auto lane = [&](size_t i) -> Engine & { return lane_of(0, i); };
        // one host thread per lane: it takes the next job, enqueues it on its lane (uploads + ~25 launches), waits and finishes it on the
        // host (Horner over the window sums), so neither the enqueue work nor the host finish of one job delays another lane
        std::vector<CudaError> errs(n_lanes, CudaError{cudaSuccess, "", 0});
        std::vector<int> rcs(n_lanes, KGR_OK);
        std::vector<std::string> msgs(n_lanes);  // kgr_last_error is per thread: a worker's text is carried back to the caller
        auto worker = [&](size_t li) {
            try {
                // static assignment (job j on lane j mod lanes): a lane sees the same jobs in every call of a repeated batch, so its grow-only
                // workspaces settle after the first call instead of being re-allocated whenever a bigger job lands on it
                for (size_t j = li; j < n_jobs; j += n_lanes) {
                    const kgr_msm_job_t &jb = jobs[j];
                    rcs[li] = [&]() -> int {
                        if (jb.n == 0) {  // empty sum: the identity (msm.rs:45-47 folds nothing)
#define CALL(C) combine_partials<C>(std::vector<Partial>(), jb.out)
                            DISPATCH(jb.bases->curve, CALL);
#undef CALL
                            return KGR_OK;
                        }
#define CALL(C) lane_start<C>(lane(li), P, jb.bases->shards[0], jb.base_off, jb.scalars, jb.scalar_fmt, jb.n); lane_finish<C>(lane(li), jb.out)
                        DISPATCH(jb.bases->curve, CALL);
#undef CALL
                        return KGR_OK;
                    }();
                    if (rcs[li]) {
                        msgs[li] = g_err;
                        break;
                    }
                }
            } catch (CudaError &ce) {
                errs[li] = ce;
            }
        };
        std::vector<std::thread> th;
        for (size_t li = 1; li < n_lanes; li++) th.emplace_back(worker, li);
        worker(0);
        for (auto &t : th) t.join();
        for (auto &ce : errs)
            if (ce.e != cudaSuccess) throw ce;
        for (size_t li = 0; li < n_lanes; li++)
            if (rcs[li]) return fail(rcs[li], msgs[li]);
        return KGR_OK;
    });
}

int kgr_msm_oneshot(int curve, const uint64_t *xy, const uint8_t *inf, size_t n_bases, const uint64_t *scalars, int fmt, size_t n_scalars,
                    uint64_t *out) {
    std::lock_guard<std::mutex> lk(g_mu);
    if (g_engines.empty()) return fail(KGR_E_NOT_INIT, "kgr_init has not been called");
    size_t n = std::min(n_bases, n_scalars);  // zip semantics, groth16/src/msm.rs:25
    if (!out || (n && (!xy || !scalars))) return fail(KGR_E_ARG, "null pointer");
    if (n >= (1ull << 31)) return fail(KGR_E_TOO_LARGE, "at most 2^31 - 1 pairs per call");
    if (fmt != KGR_SCALARS_MONTGOMERY && fmt != KGR_SCALARS_CANONICAL) return fail(KGR_E_ARG, "unknown scalar format");
    return guarded([&]() -> int {
        std::vector<Shard> shards;
        make_shards(shards, n);
        HostPts hp{xy, inf};
#define CALL(C) run_msm<C>(shards, 0, scalars, false, fmt, n, out, &hp)
        DISPATCH(curve, CALL);
#undef CALL
        return KGR_OK;
    });
}

int kgr_bases_download(const kgr_bases_t *b, size_t off, size_t n, uint64_t *xy_out) {
    std::lock_guard<std::mutex> lk(g_mu);
    if (!b || (!xy_out && n)) return fail(KGR_E_ARG, "null pointer");
    if (b->generation != g_generation) return fail(KGR_E_ARG, "base handle was created before the last kgr_init");
    if (off > b->n || n > b->n - off) return fail(KGR_E_ARG, "range exceeds the registered vector");
    return guarded([&]() -> int {
        for (auto &s : b->shards) {
            size_t lo = std::max(off, s.first), hi = std::min(off + n, s.first + s.count);
            if (lo >= hi) continue;
            CK(cudaSetDevice(g_engines[s.eng].dev));
            const size_t ab = affine_bytes(b->curve);
            CK(cudaMemcpy(xy_out + (ab / 8) * (lo - off), (const uint8_t *)s.d_pts + ab * (lo - s.first), ab * (hi - lo), cudaMemcpyDeviceToHost));
        }
        return KGR_OK;
    });
}

int kgr_event_record(int dev, int idx) {
    std::lock_guard<std::mutex> lk(g_mu);
    if (dev < 0 || dev >= (int)g_engines.size() || idx < 0 || idx >= 4) return fail(KGR_E_ARG, "bad device slot / event index");
    return guarded([&]() -> int {
        Engine &e = g_engines[dev];
        CK(cudaSetDevice(e.dev));
        CK(cudaEventRecord(e.user_ev[idx], e.st));
        return KGR_OK;
    });
}

int kgr_event_elapsed_ms(int dev, int idx_a, int idx_b, float *ms) {
    std::lock_guard<std::mutex> lk(g_mu);
    if (dev < 0 || dev >= (int)g_engines.size() || idx_a < 0 || idx_a >= 4 || idx_b < 0 || idx_b >= 4 || !ms)
        return fail(KGR_E_ARG, "bad device slot / event index");
    return guarded([&]() -> int {
        Engine &e = g_engines[dev];
        CK(cudaSetDevice(e.dev));
        CK(cudaEventSynchronize(e.user_ev[idx_b]));
        CK(cudaEventElapsedTime(ms, e.user_ev[idx_a], e.user_ev[idx_b]));
        return KGR_OK;
    });
}

int kgr_launch_count(int dev, uint64_t *count) {
    std::lock_guard<std::mutex> lk(g_mu);
    if (dev < 0 || dev >= (int)g_engines.size() || !count) return fail(KGR_E_ARG, "bad device slot");
    *count = g_engines[dev].launches;
    if ((size_t)dev < g_lanes.size())
        for (auto &l : g_lanes[dev]) *count += l->launches;
    return KGR_OK;
}

int kgr_to_affine(int curve, const uint64_t *in, uint64_t *out) {
    if (!in || !out) return fail(KGR_E_ARG, "null pointer");
#define CALL(C) proj_to_affine_host<C>(in, out)
    DISPATCH(curve, CALL);
#undef CALL
    return KGR_OK;
}

int kgr_proj_add(int curve, const uint64_t *a, const uint64_t *b, uint64_t *out) {
    if (!a || !b || !out) return fail(KGR_E_ARG, "null pointer");
#define CALL(C)                                                   \
    {                                                             \
        XyzzPt<C> x = proj_to_xyzz_host<C>(a), y = proj_to_xyzz_host<C>(b); \
        xyzz_add(x, y);                                           \
        typename C::Elem o[3];                                    \
        xyzz_to_projective(x, o);                                 \
        std::memcpy(out, o, sizeof o);                            \
    }
    DISPATCH(curve, CALL);
#undef CALL
    return KGR_OK;
}

int kgr_pedersen_commit(kgr_bases_t *ck, const uint64_t *scalars, int fmt, size_t n, uint64_t *out) {
    if (!ck) return fail(KGR_E_ARG, "null pointer");
    uint64_t proj[24];
    size_t pairs = std::min(n, ck->n);  // m.iter().zip(self.g.iter()), nova/src/pedersen.rs:16-17
    int rc = kgr_msm(ck, 0, scalars, fmt, pairs, proj);
    if (rc) return rc;
    return kgr_to_affine(ck->curve, proj, out);
}

int kgr_ntt(unsigned log_n, int op, const uint64_t *in, size_t n_in, uint64_t *out, size_t *n_out) {
    std::lock_guard<std::mutex> lk(g_mu);
    if (g_engines.empty()) return fail(KGR_E_NOT_INIT, "kgr_init has not been called");
    if (log_n < 1 || log_n > 28 || op < 0 || op > 3 || !out || (!in && n_in)) return fail(KGR_E_ARG, "bad argument");
    return guarded([&]() -> int {
        Engine &e = g_engines[0];
        CK(cudaSetDevice(e.dev));
        NttDomain &d = ntt_domain(e, log_n);
        const size_t n = (size_t)1 << log_n;
        e.ntt_buf[0].ensure(n * 32);
        CK(cudaEventRecord(e.ev[EV_START], e.st));
        upload_padded(e, e.ntt_buf[0].p, in, n_in, n);
        CK(cudaEventRecord(e.ev[EV_H2D], e.st));
        ntt_enqueue(e, d, e.ntt_buf[0].p, op);
        CK(cudaEventRecord(e.ev[EV_ACC], e.st));
        download_to_host(e, out, e.ntt_buf[0].p, n * 32, e.st);
        CK(cudaEventRecord(e.ev[EV_END], e.st));
        CK(cudaGetLastError());
        CK(cudaStreamSynchronize(e.st));
        std::memset(e.last_ms, 0, sizeof e.last_ms);
        cudaEventElapsedTime(&e.last_ms[0], e.ev[EV_START], e.ev[EV_END]);
        cudaEventElapsedTime(&e.last_ms[7], e.ev[EV_START], e.ev[EV_H2D]);
        cudaEventElapsedTime(&e.last_ms[4], e.ev[EV_H2D], e.ev[EV_ACC]);
        if (n_out) *n_out = (op == 1 || op == 3) ? stripped_len(out, n) : n;
        return KGR_OK;
    });
}

int kgr_ntt_device(unsigned log_n, int op, void *d_data) {
    std::lock_guard<std::mutex> lk(g_mu);
    if (g_engines.empty()) return fail(KGR_E_NOT_INIT, "kgr_init has not been called");
    if (log_n < 1 || log_n > 28 || op < 0 || op > 3 || !d_data) return fail(KGR_E_ARG, "bad argument");
    return guarded([&]() -> int {
        Engine &e = g_engines[0];
        CK(cudaSetDevice(e.dev));
        NttDomain &d = ntt_domain(e, log_n);
        CK(cudaEventRecord(e.ev[EV_START], e.st));
        ntt_enqueue(e, d, d_data, op);
        CK(cudaEventRecord(e.ev[EV_END], e.st));
        CK(cudaGetLastError());
        CK(cudaStreamSynchronize(e.st));
        std::memset(e.last_ms, 0, sizeof e.last_ms);
        cudaEventElapsedTime(&e.last_ms[0], e.ev[EV_START], e.ev[EV_END]);
        e.last_ms[4] = e.last_ms[0];
        return KGR_OK;
    });
}

int kgr_groth16_h(unsigned log_n, const uint64_t *a, const uint64_t *b, const uint64_t *c, size_t m, uint64_t *out, size_t *n_out) {
    std::lock_guard<std::mutex> lk(g_mu);
    if (g_engines.empty()) return fail(KGR_E_NOT_INIT, "kgr_init has not been called");
    if (log_n < 1 || log_n > 28 || !a || !b || !c || !out) return fail(KGR_E_ARG, "bad argument");
    return guarded([&]() -> int {
        Engine &e = g_engines[0];
        CK(cudaSetDevice(e.dev));
        NttDomain &d = ntt_domain(e, log_n);
        const size_t n = (size_t)1 << log_n;
        CK(cudaEventRecord(e.ev[EV_START], e.st));
        enqueue_groth16_h(e, d, a, b, c, m);
        CK(cudaEventRecord(e.ev[EV_ACC], e.st));
        download_to_host(e, out, e.ntt_buf[0].p, n * 32, e.st);
        CK(cudaEventRecord(e.ev[EV_END], e.st));
        CK(cudaGetLastError());
        CK(cudaStreamSynchronize(e.st));
        std::memset(e.last_ms, 0, sizeof e.last_ms);
        cudaEventElapsedTime(&e.last_ms[0], e.ev[EV_START], e.ev[EV_END]);
        cudaEventElapsedTime(&e.last_ms[7], e.ev[EV_START], e.ev[EV_H2D]);
        cudaEventElapsedTime(&e.last_ms[4], e.ev[EV_H2D], e.ev[EV_ACC]);
        if (n_out) *n_out = stripped_len(out, n);
        return KGR_OK;
    });
}

int kgr_groth16_msms(unsigned log_n, const uint64_t *a, const uint64_t *b, const uint64_t *c, size_t m, kgr_bases_t *h, uint64_t *h_out, uint64_t *q_out,
                     size_t *q_len, const kgr_msm_job_t *jobs, size_t n_jobs) {
    if (log_n < 1 || log_n > 28 || !a || !b || !c || !h || !h_out || (!jobs && n_jobs)) return fail(KGR_E_ARG, "bad argument");
    if (h->curve != KGR_CURVE_BN254_G1) return fail(KGR_E_ARG, "the h query must be a BN254 G1 vector (its scalars are the Fr coefficients of H, its result 12 words)");
    const size_t n = (size_t)1 << log_n;
    bool fused;
    {
        std::lock_guard<std::mutex> lk(g_mu);
        if (g_engines.empty()) return fail(KGR_E_NOT_INIT, "kgr_init has not been called");
        fused = g_engines.size() == 1 && h->curve == KGR_CURVE_BN254_G1 && h->shards.size() == 1 && n_jobs < MAX_LANES;
        for (size_t j = 0; j < n_jobs && fused; j++)
            if (!jobs[j].bases || jobs[j].bases->shards.size() != 1) fused = false;
    }
    if (!fused) {  // several devices: the same steps one after the other
        std::vector<uint64_t> q(n * 4);
        size_t len = 0;
        int rc = kgr_groth16_h(log_n, a, b, c, m, q.data(), &len);
        if (rc) return rc;
        if (q_out) std::memcpy(q_out, q.data(), n * 32);
        if (q_len) *q_len = len;
        rc = kgr_msm(h, 0, q.data(), KGR_SCALARS_MONTGOMERY, std::min(len, h->n), h_out);
        if (rc) return rc;
        return kgr_msm_batch(jobs, n_jobs);
    }
    std::lock_guard<std::mutex> lk(g_mu);
    for (size_t j = 0; j < n_jobs; j++) {
        const kgr_msm_job_t &jb = jobs[j];
        if (!jb.out || (!jb.scalars && jb.n)) return fail(KGR_E_ARG, "null pointer");
        if (jb.base_off > jb.bases->n || jb.n > jb.bases->n - jb.base_off) return fail(KGR_E_ARG, "range exceeds the registered vector");
        if (jb.scalar_fmt != KGR_SCALARS_MONTGOMERY && jb.scalar_fmt != KGR_SCALARS_CANONICAL) return fail(KGR_E_ARG, "unknown scalar format");
        if (jb.bases->curve < KGR_CURVE_BN254_G1 || jb.bases->curve > KGR_CURVE_BN254_G2) return fail(KGR_E_ARG, "unknown curve id");
        if (jb.bases->generation != g_generation) return fail(KGR_E_ARG, "base handle was created before the last kgr_init");
    }
    if (h->generation != g_generation) return fail(KGR_E_ARG, "base handle was created before the last kgr_init");
    const Params P = t_params;
    return guarded([&]() -> int {
        const size_t n_lanes = std::min(n_jobs + 1, MAX_LANES);
        ensure_lanes(0, n_lanes);
        std::vector<CudaError> errs(n_lanes, CudaError{cudaSuccess, "", 0});
        std::vector<int> rcs(n_lanes, KGR_OK);
        std::vector<std::string> msgs(n_lanes);
        // lane 0: H on the device, then the h query with q as device-resident scalars (no D2H / H2D of q on the critical path)
        const size_t nh = std::min(n, h->n);  // zip(q, h): coefficients beyond the degree are zero, so the unstripped q gives the same sum
        auto h_start = [&]() {
            Engine &e = g_engines[0];
            e.params = P;
            CK(cudaSetDevice(e.dev));
            NttDomain &d = ntt_domain(e, log_n);
            CK(cudaEventRecord(e.ev[EV_START], e.st));
            enqueue_groth16_h(e, d, a, b, c, m);
            const Shard &sh = h->shards[0];
            if (nh) {
                const uint32_t *d_q = reinterpret_cast<const uint32_t *>(e.ntt_buf[0].p);
                if (sh.d_table) enqueue_msm<Bn254G1>(e, (const AffinePt<Bn254G1> *)sh.d_table, d_q, 1, (uint32_t)nh, sh.table_c, (uint32_t)sh.count, 0);
                else enqueue_msm<Bn254G1>(e, (const AffinePt<Bn254G1> *)sh.d_pts, d_q, 1, (uint32_t)nh);
            }
        };
        auto h_finish = [&]() {
            Engine &e = g_engines[0];
            if (nh) {
                lane_finish<Bn254G1>(e, h_out);
            } else {
                CK(cudaSetDevice(e.dev));
                CK(cudaStreamSynchronize(e.st));
                combine_partials<Bn254G1>(std::vector<Partial>(), h_out);
            }
            if (q_out) {
                download_to_host(e, q_out, e.ntt_buf[0].p, n * 32, e.st);
                if (q_len) *q_len = stripped_len(q_out, n);
            }
        };
        if (!P.lane_threads) {
            // one host thread: enqueue everything (lane 0 first), then collect in order.  Slower than a thread per lane when the host cores are awake,
            // less sensitive to sleeping cores (profiles/r01_next_rows.md)
            h_start();
            for (size_t j = 0; j < n_jobs; j++) {
                const kgr_msm_job_t &jb = jobs[j];
                if (jb.n == 0) continue;
#define CALL(C) lane_start<C>(lane_of(0, 1 + j), P, jb.bases->shards[0], jb.base_off, jb.scalars, jb.scalar_fmt, jb.n)
                DISPATCH(jb.bases->curve, CALL);
#undef CALL
            }
            h_finish();
            for (size_t j = 0; j < n_jobs; j++) {
                const kgr_msm_job_t &jb = jobs[j];
                if (jb.n == 0) {
#define CALL(C) combine_partials<C>(std::vector<Partial>(), jb.out)
                    DISPATCH(jb.bases->curve, CALL);
#undef CALL
                    continue;
                }
#define CALL(C) lane_finish<C>(lane_of(0, 1 + j), jb.out)
                DISPATCH(jb.bases->curve, CALL);
#undef CALL
            }
            return KGR_OK;
        }
        auto h_worker = [&]() {
            try {
                h_start();
                h_finish();
            } catch (CudaError &ce) {
                errs[0] = ce;
            }
        };
        auto worker = [&](size_t li) {
            try {
                for (size_t j = li - 1; j < n_jobs; j += n_lanes - 1) {  // static assignment, lanes 1 .. n_lanes - 1 (lane 0 runs H and the h query)
                    const kgr_msm_job_t &jb = jobs[j];
                    rcs[li] = [&]() -> int {
                        if (jb.n == 0) {
#define CALL(C) combine_partials<C>(std::vector<Partial>(), jb.out)
                            DISPATCH(jb.bases->curve, CALL);
#undef CALL
                            return KGR_OK;
                        }
#define CALL(C) lane_start<C>(lane_of(0, li), P, jb.bases->shards[0], jb.base_off, jb.scalars, jb.scalar_fmt, jb.n); lane_finish<C>(lane_of(0, li), jb.out)
                        DISPATCH(jb.bases->curve, CALL);
#undef CALL
                        return KGR_OK;
                    }();
                    if (rcs[li]) {
                        msgs[li] = g_err;
                        break;
                    }
                }
            } catch (CudaError &ce) {
                errs[li] = ce;
            }
        };
        std::vector<std::thread> th;
        for (size_t li = 1; li < n_lanes; li++) th.emplace_back(worker, li);
        h_worker();
        for (auto &t : th) t.join();
        for (auto &ce : errs)
            if (ce.e != cudaSuccess) throw ce;
        for (size_t li = 0; li < n_lanes; li++)
            if (rcs[li]) return fail(rcs[li], msgs[li]);
        return KGR_OK;
    });
}

int kgr_last_timing(int dev, float ms[8], uint32_t shape[6]) {
    std::lock_guard<std::mutex> lk(g_mu);
    if (dev < 0 || dev >= (int)g_engines.size()) return fail(KGR_E_ARG, "device slot out of range");
    if (ms) std::memcpy(ms, g_engines[dev].last_ms, sizeof(float) * 9);
    if (shape) std::memcpy(shape, g_engines[dev].last_shape, sizeof(uint32_t) * 6);
    return KGR_OK;
}

int kgr_test_field_op(int field, int op, const uint64_t *a, const uint64_t *b, size_t n, uint64_t *out) {
    std::lock_guard<std::mutex> lk(g_mu);
    if (g_engines.empty()) return fail(KGR_E_NOT_INIT, "kgr_init has not been called");
    return guarded([&]() -> int {
        if (field == 0) return test_field_op<FqP, 0>(g_engines[0], op, a, b, n, out);
        if (field == 1) return test_field_op<FrP, 1>(g_engines[0], op, a, b, n, out);
        return fail(KGR_E_ARG, "unknown field id");
    });
}

int kgr_test_point_op(int curve, int op, const uint64_t *a_xy, const uint8_t *a_inf, const uint64_t *b_xy, const uint8_t *b_inf, size_t n,
                      uint64_t *out) {
    std::lock_guard<std::mutex> lk(g_mu);
    if (g_engines.empty()) return fail(KGR_E_NOT_INIT, "kgr_init has not been called");
    return guarded([&]() -> int {
#define CALL(C) return test_point_op<C>(g_engines[0], op, a_xy, a_inf, b_xy, b_inf, n, out)
        DISPATCH(curve, CALL);
#undef CALL
    });
}

int kgr_fixed_base_mul(int curve, const uint64_t *k, size_t n, uint64_t *out_xy) {
    std::lock_guard<std::mutex> lk(g_mu);
    if (g_engines.empty()) return fail(KGR_E_NOT_INIT, "kgr_init has not been called");
    return guarded([&]() -> int {
        Engine &e = g_engines[0];
        CK(cudaSetDevice(e.dev));
        void *dk = nullptr, *dp = nullptr;
        CK(cudaMalloc(&dk, n * 32 + 32));
        const size_t ab = affine_bytes(curve);
        CK(cudaMalloc(&dp, n * ab + ab));
        CK(cudaMemcpyAsync(dk, k, n * 32, cudaMemcpyHostToDevice, e.st));
#define CALL(C) Launch<C>::fixed_base(e.st, (const Fp<C::Scalar> *)dk, fixed_table<C>(e), (uint32_t)n, (AffinePt<C> *)dp)
        DISPATCH(curve, CALL);
#undef CALL
        CK(cudaGetLastError());
        CK(cudaStreamSynchronize(e.st));
        CK(cudaMemcpy(out_xy, dp, n * ab, cudaMemcpyDeviceToHost));
        cudaFree(dk);
        cudaFree(dp);
        return KGR_OK;
    });
}

int kgr_bases_generate(int curve, uint64_t seed, size_t n, kgr_bases_t **out, uint64_t *k_out) { return kgr_bases_generate_at(curve, seed, 0, n, out, k_out); }

int kgr_bases_generate_at(int curve, uint64_t seed, uint64_t first, size_t n, kgr_bases_t **out, uint64_t *k_out) {
    std::lock_guard<std::mutex> lk(g_mu);
    if (g_engines.empty()) return fail(KGR_E_NOT_INIT, "kgr_init has not been called");
    if (!out) return fail(KGR_E_ARG, "null pointer");
    if (curve < KGR_CURVE_BN254_G1 || curve > KGR_CURVE_BN254_G2) return fail(KGR_E_ARG, "unknown curve id");
    if (n >= (1ull << 31)) return fail(KGR_E_TOO_LARGE, "at most 2^31 - 1 bases per vector");
    return guarded([&]() -> int {
        std::unique_ptr<kgr_bases> b(new kgr_bases);
        b->curve = curve;
        b->n = n;
        b->generation = g_generation;
        make_shards(b->shards, n);
#define CALL(C) for (auto &s : b->shards) generate_shard<C>(g_engines[s.eng], s, seed, first, k_out)
        DISPATCH(curve, CALL);
#undef CALL
        *out = b.release();
        return KGR_OK;
    });
}

// ---- Nova folding vector work (row N4) ------------------------------------------------------------------------------
int kgr_r1cs_register(int field, size_t m, size_t n_z, const uint32_t *const row_ptr[3], const uint32_t *const cols[3], const uint64_t *const coeffs[3],
                      kgr_r1cs_t **out) {
    std::lock_guard<std::mutex> lk(g_mu);
    if (g_engines.empty()) return fail(KGR_E_NOT_INIT, "kgr_init has not been called");
    if ((field != 0 && field != 1) || !row_ptr || !cols || !coeffs || !out) return fail(KGR_E_ARG, "bad argument");
    if (m >= (1ull << 31) || n_z >= (1ull << 31) || n_z == 0) return fail(KGR_E_TOO_LARGE, "at most 2^31 - 1 rows / columns, at least one column");
    for (int k = 0; k < 3; k++) {
        if (!row_ptr[k]) return fail(KGR_E_ARG, "null row_ptr");
        if (row_ptr[k][0] != 0) return fail(KGR_E_ARG, "row_ptr must start at 0");
        for (size_t i = 0; i < m; i++)
            if (row_ptr[k][i + 1] < row_ptr[k][i]) return fail(KGR_E_ARG, "row_ptr must be non-decreasing");
        size_t nnz = row_ptr[k][m];
        if (nnz && (!cols[k] || !coeffs[k])) return fail(KGR_E_ARG, "null cols / coeffs");
        for (size_t j = 0; j < nnz; j++)
            if (cols[k][j] >= n_z) return fail(KGR_E_ARG, "column index out of range");
    }
    return guarded([&]() -> int {
        Engine &e = g_engines[0];
        CK(cudaSetDevice(e.dev));
        std::unique_ptr<kgr_r1cs> s(new kgr_r1cs);
        s->field = field;
        s->m = m;
        s->n_z = n_z;
        s->generation = g_generation;
        for (int k = 0; k < 3; k++) {
            size_t nnz = row_ptr[k][m];
            s->nnz[k] = nnz;
            s->row_ptr[k].ensure(m + 1);
            s->cols[k].ensure(std::max<size_t>(nnz, 1));
            s->coeffs[k].ensure(std::max<size_t>(nnz, 1) * 8);
            CK(cudaMemcpyAsync(s->row_ptr[k].p, row_ptr[k], (m + 1) * sizeof(uint32_t), cudaMemcpyHostToDevice, e.st));
            if (nnz) {
                CK(cudaMemcpyAsync(s->cols[k].p, cols[k], nnz * sizeof(uint32_t), cudaMemcpyHostToDevice, e.st));
                upload_from_host(e, s->coeffs[k].p, coeffs[k], nnz * 32, e.st);
            }
        }
        s->z1.ensure(n_z * 8);
        s->z2.ensure(n_z * 8);
        s->t.ensure(std::max<size_t>(m, 1) * 8);
        CK(cudaStreamSynchronize(e.st));
        *out = s.release();
        return KGR_OK;
    });
}

int kgr_r1cs_free(kgr_r1cs_t *s) {
    std::lock_guard<std::mutex> lk(g_mu);
    if (!s) return KGR_OK;
    if (!g_engines.empty()) cudaSetDevice(g_engines[0].dev);
    for (int k = 0; k < 3; k++) { s->row_ptr[k].release(); s->cols[k].release(); s->coeffs[k].release(); }
    s->z1.release(); s->z2.release(); s->t.release();
    delete s;
    return KGR_OK;
}

int kgr_r1cs_mul(kgr_r1cs_t *s, int which, const uint64_t *z, uint64_t *out) {
    std::lock_guard<std::mutex> lk(g_mu);
    if (g_engines.empty()) return fail(KGR_E_NOT_INIT, "kgr_init has not been called");
    if (!s || which < 0 || which > 2 || !z || (!out && s->m)) return fail(KGR_E_ARG, "bad argument");
    return guarded([&]() -> int {
        Engine &e = g_engines[0];
        CK(cudaSetDevice(e.dev));
        upload_from_host(e, s->z1.p, z, s->n_z * 32, e.st);
        LaunchR1cs::spmv(e.st, s->field, (uint32_t)s->m, s->csr(which), s->z1.p, s->t.p);
        e.launches++;
        CK(cudaGetLastError());
        download_to_host(e, out, s->t.p, s->m * 32, e.st);
        CK(cudaStreamSynchronize(e.st));
        return KGR_OK;
    });
}

int kgr_nova_cross_term(kgr_r1cs_t *s, const uint64_t *z1, const uint64_t *z2, uint64_t *t_out, kgr_bases_t *ck, uint64_t *commit_out) {
    std::lock_guard<std::mutex> lk(g_mu);
    if (g_engines.empty()) return fail(KGR_E_NOT_INIT, "kgr_init has not been called");
    if (!s || !z1 || !z2 || (ck && !commit_out)) return fail(KGR_E_ARG, "bad argument");
    if (ck) {
        // the commitment key's scalar field must be the field of the constraint system (nova/src/driver.rs: Grumpkin <-> Fq, G1 <-> Fr)
        int scalar_field = ck->curve == KGR_CURVE_GRUMPKIN ? 0 : 1;
        if (scalar_field != s->field) return fail(KGR_E_ARG, "commitment key curve does not match the R1CS field");
        if (ck->shards.size() != 1 || ck->shards[0].eng != 0) return fail(KGR_E_ARG, "the commitment key must live on the first device only");
    }
    return guarded([&]() -> int {
        Engine &e = g_engines[0];
        CK(cudaSetDevice(e.dev));
        CK(cudaEventRecord(e.aux_ev[0], e.st));
        upload_from_host(e, s->z1.p, z1, s->n_z * 32, e.st);
        upload_from_host(e, s->z2.p, z2, s->n_z * 32, e.st);
        CK(cudaEventRecord(e.aux_ev[1], e.st));
        LaunchR1cs::cross_term(e.st, s->field, (uint32_t)s->m, s->csr(0), s->csr(1), s->csr(2), s->z1.p, s->z2.p, s->t.p);
        e.launches++;
        CK(cudaGetLastError());
        CK(cudaEventRecord(e.aux_ev[2], e.st));
        if (t_out) download_to_host(e, t_out, s->t.p, s->m * 32, e.st);
        CK(cudaStreamSynchronize(e.st));
        cudaEventElapsedTime(&s->ms[0], e.aux_ev[0], e.aux_ev[1]);
        cudaEventElapsedTime(&s->ms[1], e.aux_ev[1], e.aux_ev[2]);
        s->ms[2] = 0;
        if (ck) {
            // PedersenCommitment::commit(&t) (nova/src/prover.rs:35) straight from the device-resident cross term: no H2D of scalars
            uint64_t proj[24];
            size_t pairs = std::min(s->m, ck->n);
#define CALL(C) run_msm<C>(ck->shards, 0, reinterpret_cast<const uint64_t *>(s->t.p), true, KGR_SCALARS_MONTGOMERY, pairs, proj, nullptr)
            DISPATCH(ck->curve, CALL);
#undef CALL
            s->ms[2] = e.last_ms[0];
#define CALL(C) proj_to_affine_host<C>(proj, commit_out)
            DISPATCH(ck->curve, CALL);
#undef CALL
        }
        return KGR_OK;
    });
}

int kgr_r1cs_last_timing(const kgr_r1cs_t *s, float ms[3]) {
    if (!s || !ms) return fail(KGR_E_ARG, "null pointer");
    for (int i = 0; i < 3; i++) ms[i] = s->ms[i];
    return KGR_OK;
}

int kgr_vec_fold(int field, const uint64_t *a, const uint64_t *b, const uint64_t r[4], size_t n, uint64_t *out) {
    std::lock_guard<std::mutex> lk(g_mu);
    if (g_engines.empty()) return fail(KGR_E_NOT_INIT, "kgr_init has not been called");
    if ((field != 0 && field != 1) || !r || (n && (!a || !b || !out))) return fail(KGR_E_ARG, "bad argument");
    if (n >= (1ull << 31)) return fail(KGR_E_TOO_LARGE, "at most 2^31 - 1 elements");
    if (!n) return KGR_OK;
    return guarded([&]() -> int {
        Engine &e = g_engines[0];
        CK(cudaSetDevice(e.dev));
        e.ntt_buf[0].ensure(n * 32);
        e.ntt_buf[1].ensure(n * 32);
        upload_from_host(e, e.ntt_buf[0].p, a, n * 32, e.st);
        upload_from_host(e, e.ntt_buf[1].p, b, n * 32, e.st);
        uint32_t r8[8];
        std::memcpy(r8, r, 32);
        LaunchR1cs::vec_fold(e.st, field, (uint32_t)n, (const uint32_t *)e.ntt_buf[0].p, (const uint32_t *)e.ntt_buf[1].p, r8, (uint32_t *)e.ntt_buf[0].p);
        e.launches++;
        CK(cudaGetLastError());
        download_to_host(e, out, e.ntt_buf[0].p, n * 32, e.st);
        CK(cudaStreamSynchronize(e.st));
        return KGR_OK;
    });
}

// ---- device-resident vectors (Nova residency) ------------------------------------------------------------------------------------------------
static int vec_check(const kgr_vec *v) {
    if (!v) return fail(KGR_E_ARG, "null vector");
    if (v->generation != g_generation) return fail(KGR_E_ARG, "vector handle was created before the last kgr_init");
    return KGR_OK;
}

int kgr_vec_upload(int field, const uint64_t *host, size_t n, kgr_vec_t **out) {
    std::lock_guard<std::mutex> lk(g_mu);
    if (g_engines.empty()) return fail(KGR_E_NOT_INIT, "kgr_init has not been called");
    if ((field != 0 && field != 1) || !out) return fail(KGR_E_ARG, "bad argument");
    if (n >= (1ull << 31)) return fail(KGR_E_TOO_LARGE, "at most 2^31 - 1 elements");
    return guarded([&]() -> int {
        Engine &e = g_engines[0];
        CK(cudaSetDevice(e.dev));
        std::unique_ptr<kgr_vec> v(new kgr_vec);
        v->field = field;
        v->n = n;
        v->generation = g_generation;
        v->d.ensure(std::max<size_t>(n, 1) * 8);
        if (host) upload_from_host(e, v->d.p, host, n * 32, e.st);
        else CK(cudaMemsetAsync(v->d.p, 0, std::max<size_t>(n, 1) * 32, e.st));
        CK(cudaStreamSynchronize(e.st));
        *out = v.release();
        return KGR_OK;
    });
}

int kgr_vec_free(kgr_vec_t *v) {
    std::lock_guard<std::mutex> lk(g_mu);
    if (!v) return KGR_OK;
    if (!g_engines.empty()) cudaSetDevice(g_engines[0].dev);
    v->d.release();
    delete v;
    return KGR_OK;
}

size_t kgr_vec_len(const kgr_vec_t *v) { return v ? v->n : 0; }

int kgr_vec_download(const kgr_vec_t *v, size_t off, size_t n, uint64_t *host) {
    std::lock_guard<std::mutex> lk(g_mu);
    if (g_engines.empty()) return fail(KGR_E_NOT_INIT, "kgr_init has not been called");
    if (int rc = vec_check(v)) return rc;
    if (off > v->n || n > v->n - off || (!host && n)) return fail(KGR_E_ARG, "range exceeds the vector");
    return guarded([&]() -> int {
        Engine &e = g_engines[0];
        CK(cudaSetDevice(e.dev));
        download_to_host(e, host, v->d.p + 8 * off, n * 32, e.st);
        return KGR_OK;
    });
}

int kgr_vec_write(kgr_vec_t *v, size_t off, const uint64_t *host, size_t n) {
    std::lock_guard<std::mutex> lk(g_mu);
    if (g_engines.empty()) return fail(KGR_E_NOT_INIT, "kgr_init has not been called");
    if (int rc = vec_check(v)) return rc;
    if (off > v->n || n > v->n - off || (!host && n)) return fail(KGR_E_ARG, "range exceeds the vector");
    return guarded([&]() -> int {
        Engine &e = g_engines[0];
        CK(cudaSetDevice(e.dev));
        upload_from_host(e, v->d.p + 8 * off, host, n * 32, e.st);
        CK(cudaStreamSynchronize(e.st));
        return KGR_OK;
    });
}

int kgr_vec_fold_device(const kgr_vec_t *a, const kgr_vec_t *b, const uint64_t r[4], kgr_vec_t *out) {
    std::lock_guard<std::mutex> lk(g_mu);
    if (g_engines.empty()) return fail(KGR_E_NOT_INIT, "kgr_init has not been called");
    if (int rc = vec_check(a)) return rc;
    if (int rc = vec_check(b)) return rc;
    if (int rc = vec_check(out)) return rc;
    if (!r) return fail(KGR_E_ARG, "null pointer");
    if (a->field != b->field || a->field != out->field) return fail(KGR_E_ARG, "vectors of different fields");
    if (a->n < out->n || b->n < out->n) return fail(KGR_E_ARG, "inputs shorter than the output vector");
    if (!out->n) return KGR_OK;
    return guarded([&]() -> int {
        Engine &e = g_engines[0];
        CK(cudaSetDevice(e.dev));
        uint32_t r8[8];
        std::memcpy(r8, r, 32);
        LaunchR1cs::vec_fold(e.st, out->field, (uint32_t)out->n, a->d.p, b->d.p, r8, out->d.p);
        e.launches++;
        CK(cudaGetLastError());
        CK(cudaStreamSynchronize(e.st));
        return KGR_OK;
    });
}

int kgr_msm_vec(kgr_bases_t *b, size_t base_off, const kgr_vec_t *scalars, size_t sc_off, size_t n, uint64_t *out) {
    std::lock_guard<std::mutex> lk(g_mu);
    if (g_engines.empty()) return fail(KGR_E_NOT_INIT, "kgr_init has not been called");
    if (int rc = vec_check(scalars)) return rc;
    if (!b) return fail(KGR_E_ARG, "null pointer");
    if (sc_off > scalars->n || n > scalars->n - sc_off) return fail(KGR_E_ARG, "range exceeds the scalar vector");
    if ((b->curve == KGR_CURVE_GRUMPKIN ? 0 : 1) != scalars->field) return fail(KGR_E_ARG, "the vector's field is not the scalar field of the curve");
    if (b->shards.size() != 1 || b->shards[0].eng != 0) return fail(KGR_E_ARG, "the bases must live on the first device only");
    return msm_common(b, base_off, reinterpret_cast<const uint64_t *>(scalars->d.p + 8 * sc_off), true, KGR_SCALARS_MONTGOMERY, n, out);
}

int kgr_pedersen_commit_vec(kgr_bases_t *ck, const kgr_vec_t *m, size_t sc_off, size_t n, uint64_t *out) {
    if (!ck || !m) return fail(KGR_E_ARG, "null pointer");
    uint64_t proj[24];
    size_t pairs = std::min(n, ck->n);  // m.iter().zip(self.g.iter()), nova/src/pedersen.rs:16-17
    int rc = kgr_msm_vec(ck, 0, m, sc_off, pairs, proj);
    if (rc) return rc;
    return kgr_to_affine(ck->curve, proj, out);
}

int kgr_nova_cross_term_device(kgr_r1cs_t *s, const kgr_vec_t *z1, const kgr_vec_t *z2, kgr_vec_t *t, kgr_bases_t *ck, uint64_t *commit_out) {
    std::lock_guard<std::mutex> lk(g_mu);
    if (g_engines.empty()) return fail(KGR_E_NOT_INIT, "kgr_init has not been called");
    if (!s || (ck && !commit_out)) return fail(KGR_E_ARG, "bad argument");
    if (int rc = vec_check(z1)) return rc;
    if (int rc = vec_check(z2)) return rc;
    if (t)
        if (int rc = vec_check(t)) return rc;
    if (z1->field != s->field || z2->field != s->field || (t && t->field != s->field)) return fail(KGR_E_ARG, "vector field does not match the R1CS field");
    if (z1->n < s->n_z || z2->n < s->n_z || (t && t->n < s->m)) return fail(KGR_E_ARG, "vector shorter than the shape needs");
    if (ck) {
        int scalar_field = ck->curve == KGR_CURVE_GRUMPKIN ? 0 : 1;
        if (scalar_field != s->field) return fail(KGR_E_ARG, "commitment key curve does not match the R1CS field");
        if (ck->shards.size() != 1 || ck->shards[0].eng != 0) return fail(KGR_E_ARG, "the commitment key must live on the first device only");
        if (ck->generation != g_generation) return fail(KGR_E_ARG, "base handle was created before the last kgr_init");
    }
    return guarded([&]() -> int {
        Engine &e = g_engines[0];
        CK(cudaSetDevice(e.dev));
        uint32_t *d_t = t ? t->d.p : s->t.p;
        CK(cudaEventRecord(e.aux_ev[1], e.st));
        LaunchR1cs::cross_term(e.st, s->field, (uint32_t)s->m, s->csr(0), s->csr(1), s->csr(2), z1->d.p, z2->d.p, d_t);
        e.launches++;
        CK(cudaGetLastError());
        CK(cudaEventRecord(e.aux_ev[2], e.st));
        s->ms[0] = 0;
        s->ms[2] = 0;
        if (ck) {
            uint64_t proj[24];
            size_t pairs = std::min(s->m, ck->n);
#define CALL(C) run_msm<C>(ck->shards, 0, reinterpret_cast<const uint64_t *>(d_t), true, KGR_SCALARS_MONTGOMERY, pairs, proj, nullptr)
            DISPATCH(ck->curve, CALL);
#undef CALL
            s->ms[2] = e.last_ms[0];
#define CALL(C) proj_to_affine_host<C>(proj, commit_out)
            DISPATCH(ck->curve, CALL);
#undef CALL
        } else {
            CK(cudaStreamSynchronize(e.st));
        }
        cudaEventElapsedTime(&s->ms[1], e.aux_ev[1], e.aux_ev[2]);
        return KGR_OK;
    });
}

// ---- Groth16 from the constraint system (row N1: groth16/src/prover.rs:32-65 after synthesis) ------------------------------------------------
static int query_check(const kgr_bases *b, int curve, const char *name) {
    if (b->curve != curve) return fail(KGR_E_ARG, std::string("the ") + name + " query must be a BN254 " + (curve == KGR_CURVE_BN254_G2 ? "G2" : "G1") + " vector");
    if (b->generation != g_generation) return fail(KGR_E_ARG, "base handle was created before the last kgr_init");
    if (b->shards.size() != 1 || b->shards[0].eng != 0) return fail(KGR_E_ARG, "the bases must live on the first device only (a single-device context)");
    return KGR_OK;
}

int kgr_groth16_prove_r1cs(unsigned log_n, const kgr_r1cs_t *cs, const kgr_vec_t *z, size_t n_inputs, kgr_bases_t *h, kgr_bases_t *l, kgr_bases_t *a,
                           kgr_bases_t *b_g1, kgr_bases_t *b_g2, uint64_t *out, uint64_t *q_out, size_t *q_len, const kgr_msm_job_t *jobs, size_t n_jobs) {
    std::lock_guard<std::mutex> lk(g_mu);
    if (g_engines.empty()) return fail(KGR_E_NOT_INIT, "kgr_init has not been called");
    if (!cs || !h || !l || !a || !b_g1 || !out || (!jobs && n_jobs)) return fail(KGR_E_ARG, "null pointer");
    if (int rc = vec_check(z)) return rc;
    if (cs->generation != g_generation) return fail(KGR_E_ARG, "R1CS shape was registered before the last kgr_init");
    if (cs->field != 1 || z->field != 1) return fail(KGR_E_ARG, "the shape and the assignment must be over Fr (field 1)");
    if (z->n != cs->n_z) return fail(KGR_E_ARG, "the assignment must have n_z elements (z = x ++ w)");
    if (n_inputs == 0 || n_inputs > cs->n_z) return fail(KGR_E_ARG, "n_inputs must be in 1 .. n_z (the instance starts with the constant one)");
    if (log_n < 1 || log_n > 28 || ((size_t)1 << log_n) < cs->m) return fail(KGR_E_ARG, "log_n must be in 1 .. 28 with 2^log_n >= m");
    if (int rc = query_check(h, KGR_CURVE_BN254_G1, "h")) return rc;
    if (int rc = query_check(l, KGR_CURVE_BN254_G1, "l")) return rc;
    if (int rc = query_check(a, KGR_CURVE_BN254_G1, "a")) return rc;
    if (int rc = query_check(b_g1, KGR_CURVE_BN254_G1, "b_g1")) return rc;
    if (b_g2)
        if (int rc = query_check(b_g2, KGR_CURVE_BN254_G2, "b_g2")) return rc;
    for (size_t j = 0; j < n_jobs; j++) {
        const kgr_msm_job_t &jb = jobs[j];
        if (!jb.bases || !jb.out || (!jb.scalars && jb.n)) return fail(KGR_E_ARG, "null pointer");
        if (jb.base_off > jb.bases->n || jb.n > jb.bases->n - jb.base_off) return fail(KGR_E_ARG, "range exceeds the registered vector");
        if (jb.scalar_fmt != KGR_SCALARS_MONTGOMERY && jb.scalar_fmt != KGR_SCALARS_CANONICAL) return fail(KGR_E_ARG, "unknown scalar format");
        if (jb.bases->curve < KGR_CURVE_BN254_G1 || jb.bases->curve > KGR_CURVE_BN254_G2) return fail(KGR_E_ARG, "unknown curve id");
        if (int rc = query_check(jb.bases, jb.bases->curve, "job")) return rc;
    }
    const Params P = t_params;
    return guarded([&]() -> int {
        const size_t n = (size_t)1 << log_n, n_z = cs->n_z;
        // the MSMs besides h, longest first (G2: 3x the arithmetic per point) so that the others overlap with it; pairs = zip (msm.rs:25)
        struct Item {
            kgr_bases *b;
            const uint32_t *d_sc;     // scalars in z on the device, or
            const kgr_msm_job_t *job;  // a job with host scalars
            size_t n;
            uint64_t *out;
        };
        std::vector<Item> work;
        auto add = [&](kgr_bases *b, const uint32_t *d_sc, const kgr_msm_job_t *job, size_t pairs, uint64_t *o) {
            if (pairs) work.push_back(Item{b, d_sc, job, pairs, o});
            else with_curve(b->curve, [&](auto tag) { combine_partials<std::remove_pointer_t<decltype(tag)>>(std::vector<Partial>(), o); });
        };
        if (b_g2) add(b_g2, z->d.p, nullptr, std::min(b_g2->n, n_z), out + 48);                          // b_g2_inputs + b_g2_aux (prover.rs:64-65)
        add(a, z->d.p, nullptr, std::min(a->n, n_z), out + 24);                                            // a_inputs + a_aux (:58-59)
        add(b_g1, z->d.p, nullptr, std::min(b_g1->n, n_z), out + 36);                                      // b_g1_inputs + b_g1_aux (:61-62)
        add(l, z->d.p + 8 * n_inputs, nullptr, std::min(l->n, n_z - n_inputs), out + 12);                 // l: aux only (:56)
        for (size_t j = 0; j < n_jobs; j++) add(jobs[j].bases, nullptr, &jobs[j], jobs[j].n, jobs[j].out);
        const size_t n_lanes = std::min(work.size() + 1, MAX_LANES);
        ensure_lanes(0, n_lanes);
        Engine &e0 = g_engines[0];
        CK(cudaSetDevice(e0.dev));
        CK(cudaEventRecord(e0.ev_input, e0.st));  // z is complete once this event is: every lane waits for it before reading z
        auto start = [&](const Item &it, Engine &ln) {
            with_curve(it.b->curve, [&](auto tag) {
                typedef std::remove_pointer_t<decltype(tag)> C;
                if (it.job) lane_start<C>(ln, P, it.b->shards[0], it.job->base_off, it.job->scalars, it.job->scalar_fmt, it.n);
                else lane_start_device<C>(ln, P, it.b->shards[0], 0, it.d_sc, it.n, e0.ev_input);
            });
        };
        auto finish = [&](const Item &it, Engine &ln) {
            with_curve(it.b->curve, [&](auto tag) { lane_finish<std::remove_pointer_t<decltype(tag)>>(ln, it.out); });
        };
        // lane 0: the evaluations A z, B z, C z straight into the NTT buffers, H, then the h query on the device-resident q
        const size_t nh = std::min(n, h->n);
        auto h_start = [&]() {
            Engine &e = e0;
            e.params = P;
            NttDomain &d = ntt_domain(e, log_n);
            CK(cudaEventRecord(e.ev[EV_START], e.st));
            uint32_t *bufs[3];
            for (int i = 0; i < 3; i++) {
                e.ntt_buf[i].ensure(n * 32);
                bufs[i] = reinterpret_cast<uint32_t *>(e.ntt_buf[i].p);
            }
            LaunchR1cs::evaluate(e.st, log_n, (uint32_t)cs->m, cs->csr(0), cs->csr(1), cs->csr(2), z->d.p, bufs);
            e.launches++;
            CK(cudaGetLastError());
            CK(cudaEventRecord(e.ev[EV_H2D], e.st));
            enqueue_groth16_h_transforms(e, d, true);
            if (nh) lane_enqueue<Bn254G1>(e, h->shards[0], 0, bufs[0], KGR_SCALARS_MONTGOMERY, nh);
        };
        auto h_finish = [&]() {
            Engine &e = e0;
            if (nh) {
                lane_finish<Bn254G1>(e, out);
            } else {
                CK(cudaSetDevice(e.dev));
                CK(cudaStreamSynchronize(e.st));
                combine_partials<Bn254G1>(std::vector<Partial>(), out);
            }
            if (q_out) {
                download_to_host(e, q_out, e.ntt_buf[0].p, n * 32, e.st);
                if (q_len) *q_len = stripped_len(q_out, n);
            }
        };
        if (!P.lane_threads) {  // one host thread (as kgr_groth16_msms): a lane that gets a second MSM finishes its first one before
            h_start();
            std::vector<long> pending(n_lanes, -1);
            for (size_t j = 0; j < work.size(); j++) {
                const size_t li = 1 + j % (n_lanes - 1);
                if (pending[li] >= 0) finish(work[pending[li]], lane_of(0, li));
                start(work[j], lane_of(0, li));
                pending[li] = (long)j;
            }
            h_finish();
            for (size_t li = 1; li < n_lanes; li++)
                if (pending[li] >= 0) finish(work[pending[li]], lane_of(0, li));
            return KGR_OK;
        }
        std::vector<CudaError> errs(n_lanes, CudaError{cudaSuccess, "", 0});
        auto worker = [&](size_t li) {
            try {
                for (size_t j = li - 1; j < work.size(); j += n_lanes - 1) {
                    start(work[j], lane_of(0, li));
                    finish(work[j], lane_of(0, li));
                }
            } catch (CudaError &ce) {
                errs[li] = ce;
            }
        };
        std::vector<std::thread> th;
        for (size_t li = 1; li < n_lanes; li++) th.emplace_back(worker, li);
        try {
            h_start();
            h_finish();
        } catch (CudaError &ce) {
            errs[0] = ce;
        }
        for (auto &t : th) t.join();
        for (auto &ce : errs)
            if (ce.e != cudaSuccess) throw ce;
        return KGR_OK;
    });
}

// ---- Nova: R1csShape::is_sat / is_sat_relaxed on resident vectors (nova/src/relaxed_r1cs.rs:80-146) -----------------------------------------
// zkstd affine equality (macros/curve/weierstrass/group.rs:5-13) of two x[4] y[4] is_infinity values: an identity equals only an identity
static bool affine_eq9(const uint64_t *a, const uint64_t *b) {
    if (a[8] || b[8]) return a[8] && b[8];
    return std::memcmp(a, b, 64) == 0;
}

int kgr_nova_is_sat(const kgr_r1cs_t *s, const kgr_vec_t *z, const kgr_vec_t *e, size_t w_off, kgr_bases_t *ck, const uint64_t *commit_w,
                    const uint64_t *commit_e, uint64_t *report) {
    std::lock_guard<std::mutex> lk(g_mu);
    if (g_engines.empty()) return fail(KGR_E_NOT_INIT, "kgr_init has not been called");
    if (!s || !z || !report) return fail(KGR_E_ARG, "null pointer");
    if (int rc = vec_check(z)) return rc;
    if (e)
        if (int rc = vec_check(e)) return rc;
    if (s->generation != g_generation) return fail(KGR_E_ARG, "R1CS shape was registered before the last kgr_init");
    if (z->field != s->field || (e && e->field != s->field)) return fail(KGR_E_ARG, "vector field does not match the R1CS field");
    if (z->n < s->n_z || (e && e->n < s->m)) return fail(KGR_E_ARG, "vector shorter than the shape needs");
    if (w_off < 1 || w_off > s->n_z) return fail(KGR_E_ARG, "w_off must be in 1 .. n_z (W = z[w_off ..] follows u and x)");
    if ((commit_w || commit_e) && !ck) return fail(KGR_E_ARG, "an expected commitment needs the commitment key");
    if (commit_e && !e) return fail(KGR_E_ARG, "commit_e in strict mode: there is no E");
    if (ck) {
        if (ck->curve != KGR_CURVE_BN254_G1 && ck->curve != KGR_CURVE_GRUMPKIN) return fail(KGR_E_ARG, "the commitment key must be a BN254 G1 or Grumpkin vector");
        if ((ck->curve == KGR_CURVE_GRUMPKIN ? 0 : 1) != s->field) return fail(KGR_E_ARG, "commitment key curve does not match the R1CS field");
        if (ck->generation != g_generation) return fail(KGR_E_ARG, "base handle was created before the last kgr_init");
        if (ck->shards.size() != 1 || ck->shards[0].eng != 0) return fail(KGR_E_ARG, "the commitment key must live on the first device only");
    }
    const Params P = t_params;
    return guarded([&]() -> int {
        uint64_t rep[6] = {0, 0, 0, 2, 2, 1};
        struct Commit {
            const uint32_t *d_sc;  // the committed vector in device memory
            size_t n;              // pairs: zip with ck.g (pedersen.rs:16-17)
            const uint64_t *expect;
            uint64_t *status;
        };
        std::vector<Commit> work;
        if (commit_w) work.push_back(Commit{z->d.p + 8 * w_off, std::min(s->n_z - w_off, ck->n), commit_w, &rep[3]});
        if (commit_e) work.push_back(Commit{e->d.p, std::min(s->m, ck->n), commit_e, &rep[4]});
        ensure_lanes(0, 1 + work.size());
        Engine &e0 = g_engines[0];
        CK(cudaSetDevice(e0.dev));
        CK(cudaEventRecord(e0.ev_input, e0.st));  // z and E are complete once this event is: the commitment lanes wait for it before reading them
        // lane 0: the relation.  It runs no MSM in this call, so its pinned result buffer takes the three result words.
        uint32_t *res = e0.h_result;
        auto relation_start = [&]() {
            e0.sat_result.ensure(3);
            CK(cudaMemsetAsync(e0.sat_result.p, 0, 3 * sizeof(uint32_t), e0.st));
            CK(cudaMemsetAsync(e0.sat_result.p + 1, 0xFF, sizeof(uint32_t), e0.st));
            LaunchR1cs::relaxed_check(e0.st, s->field, (uint32_t)s->m, s->csr(0), s->csr(1), s->csr(2), z->d.p, e ? e->d.p : nullptr, !e, e0.sat_result.p);
            e0.launches++;
            CK(cudaGetLastError());
            CK(cudaMemcpyAsync(res, e0.sat_result.p, 3 * sizeof(uint32_t), cudaMemcpyDeviceToHost, e0.st));
        };
        auto relation_finish = [&]() {
            CK(cudaSetDevice(e0.dev));
            CK(cudaStreamSynchronize(e0.st));
        };
        // lanes 1, 2: commit(W), commit(E) from the resident scalars
        auto commit_start = [&](const Commit &c, Engine &ln) {
            if (c.n) with_curve(ck->curve, [&](auto tag) { lane_start_device<std::remove_pointer_t<decltype(tag)>>(ln, P, ck->shards[0], 0, c.d_sc, c.n, e0.ev_input); });
        };
        auto commit_finish = [&](const Commit &c, Engine &ln) {
            uint64_t proj[24], aff[17];
            with_curve(ck->curve, [&](auto tag) {
                typedef std::remove_pointer_t<decltype(tag)> C;
                if (c.n) lane_finish<C>(ln, proj);
                else combine_partials<C>(std::vector<Partial>(), proj);
                proj_to_affine_host<C>(proj, aff);
            });
            *c.status = affine_eq9(aff, c.expect) ? 1 : 0;
        };
        if (!P.lane_threads) {
            relation_start();
            for (size_t j = 0; j < work.size(); j++) commit_start(work[j], lane_of(0, 1 + j));
            relation_finish();
            for (size_t j = 0; j < work.size(); j++) commit_finish(work[j], lane_of(0, 1 + j));
        } else {
            std::vector<CudaError> errs(1 + work.size(), CudaError{cudaSuccess, "", 0});
            std::vector<std::thread> th;
            for (size_t j = 0; j < work.size(); j++)
                th.emplace_back([&, j]() {
                    try {
                        commit_start(work[j], lane_of(0, 1 + j));
                        commit_finish(work[j], lane_of(0, 1 + j));
                    } catch (CudaError &ce) {
                        errs[1 + j] = ce;
                    }
                });
            try {
                relation_start();
                relation_finish();
            } catch (CudaError &ce) {
                errs[0] = ce;
            }
            for (auto &t : th) t.join();
            for (auto &ce : errs)
                if (ce.e != cudaSuccess) throw ce;
        }
        rep[1] = res[0];
        rep[2] = res[0] ? res[1] : s->m;
        if (!e) rep[5] = res[2];
        rep[0] = (rep[1] == 0 && rep[5] == 1 && rep[3] != 0 && rep[4] != 0) ? 1 : 0;
        std::memcpy(report, rep, sizeof rep);
        return KGR_OK;
    });
}

// ---- Groth16 parameter generation (groth16/src/zksnark.rs:17-127) on the device ---------------------------------------------------------
static float g_setup_ms[10] = {};  // phases of the last kgr_groth16_setup (kgr_groth16_setup_last_timing)

static bool fr_canonical(const uint64_t *w) {  // w < r: the field code takes fully reduced residues only
    for (int i = 3; i >= 0; i--) {
        const uint64_t r = ((uint64_t)FrP::mod(2 * i + 1) << 32) | FrP::mod(2 * i);
        if (w[i] != r) return w[i] < r;
    }
    return false;
}

int kgr_groth16_setup(const kgr_r1cs_t *cs, size_t n_inputs, const uint64_t toxic[20], uint32_t *log_n_out, kgr_bases_t **h, kgr_bases_t **l,
                      kgr_bases_t **a, kgr_bases_t **b_g1, kgr_bases_t **b_g2, kgr_bases_t **ic, uint64_t *vk_g1, uint64_t *vk_g2) {
    std::lock_guard<std::mutex> lk(g_mu);
    for (kgr_bases_t **o : {h, l, a, b_g1, b_g2, ic})
        if (o) *o = nullptr;
    if (g_engines.empty()) return fail(KGR_E_NOT_INIT, "kgr_init has not been called");
    if (!cs || !toxic || !log_n_out || !h || !l || !a || !b_g1 || !ic || !vk_g1 || (b_g2 && !vk_g2)) return fail(KGR_E_ARG, "null pointer");
    if (cs->generation != g_generation) return fail(KGR_E_ARG, "R1CS shape was registered before the last kgr_init");
    if (cs->field != 1) return fail(KGR_E_ARG, "the shape must be over Fr (field 1)");
    if (n_inputs == 0 || n_inputs > cs->n_z) return fail(KGR_E_ARG, "n_inputs must be in 1 .. n_z (the instance starts with the constant one)");
    uint32_t k = 1;
    while (((size_t)1 << k) < cs->m) k++;
    if (k > 28) return fail(KGR_E_ARG, "m exceeds 2^28, the largest Fr domain");
    for (int i = 0; i < 5; i++)
        if (!fr_canonical(toxic + 4 * i)) return fail(KGR_E_ARG, "toxic waste must be reduced modulo r");
    for (int i : {2, 3})
        if (!(toxic[4 * i] | toxic[4 * i + 1] | toxic[4 * i + 2] | toxic[4 * i + 3])) return fail(KGR_E_ARG, "gamma and delta must be non-zero");
    if (g_engines.size() != 1) return fail(KGR_E_ARG, "setup needs a single-device context (the queries live on the first device, unsplit)");
    return guarded([&]() -> int {
        Engine &e = g_engines[0];
        CK(cudaSetDevice(e.dev));
        const size_t n = (size_t)1 << k, n_z = cs->n_z, n_h = cs->m ? cs->m - 1 : 0;
        Fp<FrP> t[5];  // alpha, beta, gamma, delta, tau
        for (int i = 0; i < 5; i++) std::memcpy(&t[i], toxic + 4 * i, 32);
        const Fp<FrP> &tau = t[4];
        SetupConsts<FrP> consts{t[0], t[1], fp_inv(t[2]), fp_inv(t[3]), fp_zero<FrP>()};
        consts.h_coeff = fp_mul(fp_sub(fr_pow2k(tau, k), fp_one<FrP>()), consts.delta_inv);  // (tau^n - 1) / delta (zksnark.rs:52-53)
        const uint32_t log_t = LaunchSetup::tau_log_t(k);
        const Fp<FrP> tau_t = fr_pow2k(tau, log_t);
        const size_t nnz_max = std::max({cs->nnz[0], cs->nnz[1], cs->nnz[2], (size_t)1});
        struct Scratch {
            DevBuf<uint8_t> lo, hi, lagr, hs, uvw[3], ext, vals[2], vk_k, vk_pts;
            DevBuf<uint32_t> cnt, ptr[2], tile_sums;
            ~Scratch() {
                for (auto *b : {&lo, &hi, &lagr, &hs, &uvw[0], &uvw[1], &uvw[2], &ext, &vals[0], &vals[1], &vk_k, &vk_pts}) b->release();
                for (auto *b : {&cnt, &ptr[0], &ptr[1], &tile_sums}) b->release();
            }
        } sc;
        sc.lo.ensure(((size_t)1 << log_t) * 32);
        sc.hi.ensure((n >> log_t) * 32);
        sc.lagr.ensure(n * 32);
        sc.hs.ensure(std::max<size_t>(n_h, 1) * 32);
        for (auto &b : sc.uvw) b.ensure(n_z * 32);
        sc.ext.ensure(n_z * 32);
        for (auto &b : sc.vals) b.ensure(nnz_max * 32);
        sc.cnt.ensure(n_z + 1);
        for (auto &b : sc.ptr) b.ensure(n_z + 1);
        sc.tile_sums.ensure(LaunchUtil::scan_tiles((uint32_t)n_z + 1));
        sc.vk_k.ensure(6 * 32);
        sc.vk_pts.ensure(3 * sizeof(AffinePt<Bn254G1>) + 3 * sizeof(AffinePt<Bn254G2>));
        // vk scalars: alpha, beta, delta (G1) then beta, gamma, delta (G2)
        const Fp<FrP> vk_k[6] = {t[0], t[1], t[3], t[1], t[2], t[3]};
        CK(cudaMemcpyAsync(sc.vk_k.p, vk_k, sizeof vk_k, cudaMemcpyHostToDevice, e.st));
        // one-time tables (cached per engine), outside the timed phases
        NttDomain &d = ntt_domain(e, k);
        fixed_table<Bn254G1>(e);
        if (b_g2 || vk_g2) fixed_table<Bn254G2>(e);
        cudaEvent_t ev[11] = {};
        struct Events {
            cudaEvent_t *ev;
            ~Events() {
                for (int i = 0; i < 11; i++)
                    if (ev[i]) cudaEventDestroy(ev[i]);
            }
        } ev_guard{ev};
        for (auto &x : ev) CK(cudaEventCreate(&x));
        int mark = 0;
        auto phase = [&]() { CK(cudaEventRecord(ev[mark++], e.st)); };
        phase();
        // powers of tau (the first m - 1 also into h, zksnark.rs:51-57), then the Lagrange basis at tau = idft of the powers (zksnark.rs:60)
        LaunchNtt::pow_table(e.st, sc.lo.p, &tau, 1u << log_t);
        LaunchNtt::pow_table(e.st, sc.hi.p, &tau_t, (uint32_t)(n >> log_t));
        e.launches += 2 + LaunchSetup::tau_powers(e.st, k, sc.lo.p, sc.hi.p, sc.lagr.p, (uint32_t)n_h, sc.hs.p);
        ntt_enqueue(e, d, sc.lagr.p, 1);
        CK(cudaGetLastError());
        phase();
        // u, v, w per variable (zksnark.rs:62-87: eval_at_tau of the columns of A, B, C)
        uint32_t *ptr[2] = {sc.ptr[0].p, sc.ptr[1].p};
        for (int i = 0; i < 3; i++) {
            void *vals[2] = {sc.vals[0].p, sc.vals[1].p};
            CK(cudaMemsetAsync(sc.cnt.p, 0, (n_z + 1) * sizeof(uint32_t), e.st));
            e.launches += LaunchSetup::column_sums(e.st, (uint32_t)cs->m, (uint32_t)n_z, cs->csr(i), (uint32_t)cs->nnz[i], sc.lagr.p, sc.cnt.p, ptr, vals,
                                                   sc.tile_sums.p, sc.uvw[i].p);
            CK(cudaGetLastError());
        }
        phase();
        e.launches += LaunchSetup::scalars(e.st, (uint32_t)n_z, (uint32_t)n_inputs, (uint32_t)n_h, &consts, sc.uvw[0].p, sc.uvw[1].p, sc.uvw[2].p, sc.ext.p,
                                           sc.hs.p);
        CK(cudaGetLastError());
        phase();
        // the queries: a_j = u_j, b_j = v_j, ic / l from ext, h (zksnark.rs:51-87)
        std::unique_ptr<kgr_bases> qa = fixed_base_handle<Bn254G1>(e, KGR_CURVE_BN254_G1, sc.uvw[0].p, n_z);
        phase();
        std::unique_ptr<kgr_bases> qb1 = fixed_base_handle<Bn254G1>(e, KGR_CURVE_BN254_G1, sc.uvw[1].p, n_z);
        phase();
        std::unique_ptr<kgr_bases> qic = fixed_base_handle<Bn254G1>(e, KGR_CURVE_BN254_G1, sc.ext.p, n_inputs);
        phase();
        std::unique_ptr<kgr_bases> ql = fixed_base_handle<Bn254G1>(e, KGR_CURVE_BN254_G1, sc.ext.p + 32 * n_inputs, n_z - n_inputs);
        phase();
        std::unique_ptr<kgr_bases> qh = fixed_base_handle<Bn254G1>(e, KGR_CURVE_BN254_G1, sc.hs.p, n_h);
        phase();
        std::unique_ptr<kgr_bases> qb2;
        if (b_g2) qb2 = fixed_base_handle<Bn254G2>(e, KGR_CURVE_BN254_G2, sc.uvw[1].p, n_z);
        phase();
        AffinePt<Bn254G1> *vk1 = (AffinePt<Bn254G1> *)sc.vk_pts.p;
        AffinePt<Bn254G2> *vk2 = (AffinePt<Bn254G2> *)(vk1 + 3);
        Launch<Bn254G1>::fixed_base(e.st, (const Fp<FrP> *)sc.vk_k.p, fixed_table<Bn254G1>(e), 3, vk1);
        e.launches++;
        if (vk_g2) {
            Launch<Bn254G2>::fixed_base(e.st, (const Fp<FrP> *)sc.vk_k.p + 3, fixed_table<Bn254G2>(e), 3, vk2);
            e.launches++;
        }
        CK(cudaGetLastError());
        phase();
        uint64_t pts[3 * 8 + 3 * 16];
        CK(cudaMemcpyAsync(pts, sc.vk_pts.p, sizeof pts, cudaMemcpyDeviceToHost, e.st));
        CK(cudaStreamSynchronize(e.st));
        for (int i = 0; i < 10; i++) CK(cudaEventElapsedTime(&g_setup_ms[i], ev[i], ev[i + 1]));
        auto put = [](const uint64_t *xy, int words, uint64_t *o) {  // x y is_infinity; the identity reads (0, 0, 1) as in kgr_bases_download
            uint64_t any = 0;
            for (int w = 0; w < words; w++) any |= (o[w] = xy[w]);
            o[words] = any ? 0 : 1;
        };
        for (int i = 0; i < 3; i++) put(pts + 8 * i, 8, vk_g1 + 9 * i);
        if (vk_g2)
            for (int i = 0; i < 3; i++) put(pts + 24 + 16 * i, 16, vk_g2 + 17 * i);
        *log_n_out = k;
        *a = qa.release();
        *b_g1 = qb1.release();
        *ic = qic.release();
        *l = ql.release();
        *h = qh.release();
        if (b_g2) *b_g2 = qb2.release();
        return KGR_OK;
    });
}

int kgr_groth16_setup_last_timing(float ms[10]) {
    std::lock_guard<std::mutex> lk(g_mu);
    if (!ms) return fail(KGR_E_ARG, "null pointer");
    std::memcpy(ms, g_setup_ms, sizeof g_setup_ms);
    return KGR_OK;
}

// ---- BN254 pairing and Groth16 verification (groth16/src/verifier.rs: the check of proof.rs:39-48) on the device --------------------------
int kgr_pairing(const uint64_t *g1, const uint64_t *g2, size_t n, int op, uint64_t *out) {
    std::lock_guard<std::mutex> lk(g_mu);
    if (g_engines.empty()) return fail(KGR_E_NOT_INIT, "kgr_init has not been called");
    if (!out || (n && (!g1 || !g2))) return fail(KGR_E_ARG, "null pointer");
    if (op != 0 && op != 1) return fail(KGR_E_ARG, "op must be 0 (one value per pair) or 1 (the product)");
    if (n >= (1ull << 31)) return fail(KGR_E_TOO_LARGE, "at most 2^31 - 1 pairs");
    if (n == 0) {
        if (op == 1) {
            const Fq12 one = fq12_one();
            std::memcpy(out, &one, sizeof one);
        }
        return KGR_OK;
    }
    return guarded([&]() -> int {
        Engine &e = g_engines[0];
        CK(cudaSetDevice(e.dev));
        struct Scratch {
            DevBuf<uint64_t> g1, g2;
            DevBuf<uint8_t> p, q, f[2], gt;
            DevBuf<uint32_t> bad;
            ~Scratch() {
                g1.release(), g2.release(), bad.release();
                for (auto *b : {&p, &q, &f[0], &f[1], &gt}) b->release();
            }
        } sc;
        typedef LaunchPairing L;
        sc.g1.ensure(9 * n), sc.g2.ensure(17 * n), sc.p.ensure(n * L::G1_BYTES), sc.q.ensure(n * L::G2_BYTES), sc.bad.ensure(1);
        sc.f[0].ensure(n * L::FQ12_BYTES), sc.f[1].ensure(((n + 1) / 2) * L::FQ12_BYTES), sc.gt.ensure((op ? 1 : n) * L::FQ12_BYTES);
        CK(cudaMemcpyAsync(sc.g1.p, g1, 72 * n, cudaMemcpyHostToDevice, e.st));
        CK(cudaMemcpyAsync(sc.g2.p, g2, 136 * n, cudaMemcpyHostToDevice, e.st));
        CK(cudaMemsetAsync(sc.bad.p, 0, 4, e.st));
        L::load(e.st, (uint32_t)n, sc.g1.p, sc.g2.p, sc.p.p, sc.q.p, sc.bad.p);
        L::miller(e.st, (uint32_t)n, sc.p.p, sc.q.p, sc.f[0].p);
        e.launches += 2;
        int root = 0;
        void *fb[2] = {sc.f[0].p, sc.f[1].p};
        if (op == 1) e.launches += L::product_tree(e.st, (uint32_t)n, fb, nullptr, root);
        L::final_exp(e.st, op ? 1u : (uint32_t)n, sc.f[root].p, sc.gt.p, nullptr, nullptr);
        e.launches++;
        CK(cudaGetLastError());
        uint32_t bad = 0;
        CK(cudaMemcpyAsync(&bad, sc.bad.p, 4, cudaMemcpyDeviceToHost, e.st));
        CK(cudaStreamSynchronize(e.st));
        if (bad) return fail(KGR_E_ARG, "a G1 point off the curve, a G2 point off the twist or outside G2, or a coordinate >= p");
        CK(cudaMemcpyAsync(out, sc.gt.p, (op ? 1 : n) * L::FQ12_BYTES, cudaMemcpyDeviceToHost, e.st));
        CK(cudaStreamSynchronize(e.st));
        return KGR_OK;
    });
}

int kgr_groth16_verify(const uint64_t *vk_g1, const uint64_t *vk_g2, kgr_bases_t *ic, const uint64_t *proofs, size_t k, const uint64_t *inputs,
                       size_t n_public, const uint64_t *rho, uint32_t *ok) {
    std::lock_guard<std::mutex> lk(g_mu);
    if (g_engines.empty()) return fail(KGR_E_NOT_INIT, "kgr_init has not been called");
    if (!vk_g1 || !vk_g2 || !ic || (k && (!proofs || !ok || (n_public && !inputs)))) return fail(KGR_E_ARG, "null pointer");
    if (int rc = query_check(ic, KGR_CURVE_BN254_G1, "ic")) return rc;
    if (n_public + 1 != ic->n) return fail(KGR_E_ARG, "ic must hold n_public + 1 points (ic_0 carries the constant one)");
    if (g_engines.size() != 1) return fail(KGR_E_ARG, "verification needs a single-device context");
    if (k >= (1ull << 31) || (k && n_public >= (1ull << 31) / k)) return fail(KGR_E_TOO_LARGE, "too many proofs or inputs");
    if (k >= 2) {
        if (!rho) return fail(KGR_E_ARG, "a batch of two or more proofs needs rho");
        for (size_t i = 0; i < k; i++)
            if (!(rho[2 * i] | rho[2 * i + 1])) return fail(KGR_E_ARG, "every rho_i must be non-zero");
    }
    for (size_t i = 0; i < k * n_public; i++)
        if (!fr_canonical(inputs + 4 * i)) return fail(KGR_E_ARG, "public inputs must be reduced modulo r");
    G1A vk1[3];
    G2A vk2[3];
    for (int j = 0; j < 3; j++)
        if (!load_g1(vk_g1 + 9 * j, vk1[j])) return fail(KGR_E_ARG, "a G1 point of the verifying key is invalid");
    uint32_t present = 0;
    for (int j = 0; j < 3; j++) {
        if (!load_g2(vk_g2 + 17 * j, vk2[j])) return fail(KGR_E_ARG, "a G2 point of the verifying key is invalid (off the twist or outside G2)");
        if (!affine_is_identity(vk2[j])) present |= 1u << j;
    }
    if ((present & 6u) != 6u) return fail(KGR_E_ARG, "gamma and delta must not be the identity");
    if (k == 0) return KGR_OK;
    return guarded([&]() -> int {
        typedef LaunchPairing L;
        Engine &e = g_engines[0];
        CK(cudaSetDevice(e.dev));
        const uint32_t K = (uint32_t)k, NP = (uint32_t)n_public;
        struct Scratch {
            DevBuf<uint64_t> proofs, inputs, rho;
            DevBuf<uint8_t> a, b, c, valid, canon, fixed, lines, f[2], sums[2], rho_a, rho_mont, colsum, fbatch, ic_tab, ic_x;
            DevBuf<uint32_t> ok;
            ~Scratch() {
                proofs.release(), inputs.release(), rho.release(), ok.release();
                for (auto *x : {&a, &b, &c, &valid, &canon, &fixed, &lines, &f[0], &f[1], &sums[0], &sums[1], &rho_a, &rho_mont, &colsum, &fbatch, &ic_tab,
                                &ic_x})
                    x->release();
            }
        } sc;
        sc.proofs.ensure(35 * k), sc.inputs.ensure(std::max<size_t>(4 * k * n_public, 1));
        sc.a.ensure(k * L::G1_BYTES), sc.b.ensure(k * L::G2_BYTES), sc.c.ensure(k * L::G1_BYTES), sc.valid.ensure(k);
        sc.canon.ensure(std::max<size_t>(k * n_public, 1) * 32), sc.lines.ensure(3 * MILLER_LINES * L::LINE_BYTES);
        sc.fixed.ensure(2 * L::G1_BYTES + 3 * L::G2_BYTES);  // alpha, the batched IC sum, beta, gamma, delta
        sc.f[0].ensure(k * L::FQ12_BYTES), sc.f[1].ensure(((k + 1) / 2) * L::FQ12_BYTES), sc.ok.ensure(k + 1);
        uint8_t *d_alpha = sc.fixed.p, *d_icsum = sc.fixed.p + L::G1_BYTES, *d_vk2 = sc.fixed.p + 2 * L::G1_BYTES;
        CK(cudaMemcpyAsync(sc.proofs.p, proofs, 35 * 8 * k, cudaMemcpyHostToDevice, e.st));
        if (n_public) CK(cudaMemcpyAsync(sc.inputs.p, inputs, 32 * k * n_public, cudaMemcpyHostToDevice, e.st));
        CK(cudaMemcpyAsync(d_alpha, &vk1[0], sizeof(G1A), cudaMemcpyHostToDevice, e.st));
        CK(cudaMemcpyAsync(d_vk2, vk2, sizeof vk2, cudaMemcpyHostToDevice, e.st));
        L::validate_proofs(e.st, K, sc.proofs.p, sc.inputs.p, NP, sc.a.p, sc.b.p, sc.c.p, sc.valid.p, sc.canon.p);
        L::lines(e.st, 3, d_vk2, sc.lines.p);
        e.launches += 2;
        CK(cudaGetLastError());
        std::vector<uint8_t> valid(k);
        if (k >= 2) {
            // one random linear combination of the k checks: a single final exponentiation
            sc.rho.ensure(2 * k), sc.rho_a.ensure(k * L::G1_BYTES), sc.rho_mont.ensure(k * 32), sc.colsum.ensure((n_public + 1) * 32);
            sc.sums[0].ensure(2 * k * L::XYZZ_BYTES), sc.sums[1].ensure(2 * ((k + 1) / 2) * L::XYZZ_BYTES), sc.fbatch.ensure(L::FQ12_BYTES);
            CK(cudaMemcpyAsync(sc.rho.p, rho, 16 * k, cudaMemcpyHostToDevice, e.st));
            L::batch_prep(e.st, K, sc.rho.p, sc.valid.p, sc.a.p, sc.c.p, d_alpha, sc.rho_a.p, sc.sums[0].p, sc.rho_mont.p);
            L::batch_colsum(e.st, K, NP, sc.rho_mont.p, sc.inputs.p, sc.colsum.p);
            e.launches += 2;
            CK(cudaGetLastError());
            // sum_i rho_i IC(x_i) = (sum_i rho_i) ic_0 + sum_j s_j ic_{j+1}: one MSM over the ic handle with device-resident scalars
            uint64_t proj[12], aff[9];
            run_msm<Bn254G1>(ic->shards, 0, reinterpret_cast<const uint64_t *>(sc.colsum.p), true, KGR_SCALARS_MONTGOMERY, n_public + 1, proj, nullptr);
            proj_to_affine_host<Bn254G1>(proj, aff);
            G1A icsum{};
            if (!aff[8]) std::memcpy(&icsum, aff, sizeof icsum);
            CK(cudaMemcpyAsync(d_icsum, &icsum, sizeof icsum, cudaMemcpyHostToDevice, e.st));
            L::miller(e.st, K, sc.rho_a.p, sc.b.p, sc.f[0].p);
            e.launches++;
            int root = 0;
            void *fb[2] = {sc.f[0].p, sc.f[1].p}, *sb[2] = {sc.sums[0].p, sc.sums[1].p};
            e.launches += L::product_tree(e.st, K, fb, sb, root);
            L::batch_fixed(e.st, sc.f[root].p, sc.sums[root].p, d_icsum, sc.lines.p, present, sc.fbatch.p);
            L::final_exp(e.st, 1, sc.fbatch.p, nullptr, nullptr, sc.ok.p + k);
            e.launches += 2;
            CK(cudaGetLastError());
            uint32_t batch_ok = 0;
            CK(cudaMemcpyAsync(&batch_ok, sc.ok.p + k, 4, cudaMemcpyDeviceToHost, e.st));
            CK(cudaMemcpyAsync(valid.data(), sc.valid.p, k, cudaMemcpyDeviceToHost, e.st));
            CK(cudaStreamSynchronize(e.st));
            if (batch_ok) {
                for (size_t i = 0; i < k; i++) ok[i] = valid[i];
                return KGR_OK;
            }
        }
        // every proof on its own: IC(x_i) by Straus over the ic points, one multi-Miller loop and one final exponentiation per thread
        const void *ic_pts = ic->shards[0].d_pts;
        sc.ic_tab.ensure(std::max<size_t>(16 * n_public, 1) * L::G1_BYTES), sc.ic_x.ensure(k * L::G1_BYTES);
        if (NP) {
            L::ic_table(e.st, NP, ic_pts, sc.ic_tab.p);
            e.launches++;
        }
        L::ic_straus(e.st, K, NP, ic_pts, sc.ic_tab.p, sc.canon.p, sc.ic_x.p);
        L::verify_miller(e.st, K, sc.a.p, sc.b.p, sc.c.p, d_alpha, sc.ic_x.p, sc.lines.p, present, sc.f[0].p);
        L::final_exp(e.st, K, sc.f[0].p, nullptr, sc.valid.p, sc.ok.p);
        e.launches += 3;
        CK(cudaGetLastError());
        CK(cudaMemcpyAsync(ok, sc.ok.p, 4 * k, cudaMemcpyDeviceToHost, e.st));
        CK(cudaStreamSynchronize(e.st));
        return KGR_OK;
    });
}

int kgr_host_alloc(size_t bytes, void **out) {
    if (!out) return fail(KGR_E_ARG, "null pointer");
    {
        std::lock_guard<std::mutex> lk(g_mu);
        if (g_engines.empty()) return fail(KGR_E_NOT_INIT, "kgr_init has not been called");
        cudaSetDevice(g_engines[0].dev);
    }
    return guarded([&]() -> int {
        CK(cudaHostAlloc(out, std::max<size_t>(bytes, 1), cudaHostAllocPortable));
        return KGR_OK;
    });
}

int kgr_host_free(void *p) {
    if (p) cudaFreeHost(p);
    return KGR_OK;
}

int kgr_microbench(double r[8]) {
    std::lock_guard<std::mutex> lk(g_mu);
    if (g_engines.empty()) return fail(KGR_E_NOT_INIT, "kgr_init has not been called");
    return guarded([&]() -> int {
        Engine &e = g_engines[0];
        CK(cudaSetDevice(e.dev));
        uint32_t *sink = nullptr;
        CK(cudaMalloc(&sink, 4096));
        r[0] = ubench_mode(e, 0, sink, 64);
        r[1] = ubench_mode(e, 1, sink, 64);
        r[2] = ubench_mode(e, 2, sink, 64);
        r[3] = ubench_mode(e, 3, sink, 8 * 4);  // 4 wide mads per chain, 8 chains per iteration
        r[4] = ubench_mode(e, 4, sink, 64);
        cudaEvent_t a, b;
        CK(cudaEventCreate(&a));
        CK(cudaEventCreate(&b));
        float ms = 0;
        {
            const int iters = 500, blocks = e.sm_count * 8;
            LaunchUtil::ubench_fmul(e.st, blocks, sink, 4);
            CK(cudaEventRecord(a, e.st));
            LaunchUtil::ubench_fmul(e.st, blocks, sink, iters);
            CK(cudaEventRecord(b, e.st));
            CK(cudaStreamSynchronize(e.st));
            CK(cudaEventElapsedTime(&ms, a, b));
            r[5] = (double)blocks * 256 * iters * 2 / (ms * 1e-3) / 1e9;
        }
        {
            AffinePt<Bn254G1> g = generator_affine<Bn254G1>();
            XyzzPt<Bn254G1> d = xyzz_dbl_affine(g);
            AffinePt<Bn254G1> g2 = xyzz_to_affine(d);
            const int iters = 200, blocks = e.sm_count * 16;
            LaunchUtil::ubench_madd(e.st, blocks, sink, g, g2, 4);
            CK(cudaEventRecord(a, e.st));
            LaunchUtil::ubench_madd(e.st, blocks, sink, g, g2, iters);
            CK(cudaEventRecord(b, e.st));
            CK(cudaStreamSynchronize(e.st));
            CK(cudaEventElapsedTime(&ms, a, b));
            r[6] = (double)blocks * 128 * iters / (ms * 1e-3) / 1e9;
        }
        {
            uint64_t *d = nullptr, h[2];
            CK(cudaMalloc(&d, 16));
            LaunchUtil::clock_probe(e.st, d);
            CK(cudaStreamSynchronize(e.st));
            CK(cudaMemcpy(h, d, 16, cudaMemcpyDeviceToHost));
            cudaFree(d);
            r[7] = (double)h[1] / (double)h[0] * 1e3;  // cycles per ns -> MHz
        }
        cudaEventDestroy(a);
        cudaEventDestroy(b);
        cudaFree(sink);
        CK(cudaGetLastError());
        return KGR_OK;
    });
}

}  // extern "C"
