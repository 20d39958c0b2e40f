// launch.cuh — host-callable launchers, one set per curve.  The engine (msm.cu) sees only these
// declarations; the kernels are compiled in kernels_g1.cu / kernels_grumpkin.cu / kernels_util.cu so the
// three translation units build in parallel.
#pragma once
#include <cuda_runtime.h>

#include <cstring>

#include "msm_kernels.cuh"

namespace kgr {

constexpr int TPB_SCALAR = 256;
constexpr int TPB_ACC = 128;
constexpr int TPB_RED = 64;
constexpr int TPB_TREE = 128;

template <class C> struct Launch {
    typedef XyzzPt<C> X;
    typedef AffinePt<C> A;
    typedef Fp<typename C::Scalar> S;
    static int accumulate_blocks_per_sm();
    static void count(cudaStream_t st, const MsmShape &sh, const uint32_t *scalars, int is_mont, uint32_t *counts, uint32_t *digits);
    static void fill_window(cudaStream_t st, const MsmShape &sh, const uint32_t *digits, uint32_t *counts, const uint32_t *offsets, uint32_t *entries);
    static void fill(cudaStream_t st, const MsmShape &sh, const uint32_t *scalars, int is_mont, uint32_t *counts, const uint32_t *offsets, uint32_t *entries);
    static void accumulate(cudaStream_t st, const MsmShape &sh, uint32_t chunks, const A *bases, const uint32_t *offsets, const uint32_t *entries, X *bucket_acc,
                           X *head, X *tail, uint32_t *tail_bucket);
    // Batched-affine tree levels (affine_kernels.cuh): level i reads off[i] / node array i (level 0: entries over bases) and writes off[i + 1] /
    // nodes[i & 1]; cnt: G + 1 words of scratch.  Returns the number of launches.  out_max[i]: host-side bound of the nodes of level i + 1.
    // pre: 8 words per node of the largest level, tot: 8 words per thread (affine_scratch_words gives both sizes for out_max[0])
    static int affine_levels(cudaStream_t st, uint32_t levels, uint32_t G, const A *bases, const uint32_t *entries, uint32_t *const off[], A *const nodes[2],
                             const uint32_t out_max[], uint32_t *cnt, uint32_t *tile_sums, uint32_t *pre, uint32_t *tot, uint32_t n_bases, void *xs);
    static void affine_scratch_words(uint32_t out_max0, size_t &pre_words, size_t &tot_words);
    // worklist: 4 words per record, fixup_records_max(chunks) records; partial: one XYZZ point per record; counter: one word per record, zero on
    // entry and left zero
    static size_t fixup_records_max(uint32_t chunks);
    static void fixup(cudaStream_t st, const MsmShape &sh, uint32_t chunks, int sm_count, const uint32_t *offsets, X *bucket_acc, const X *head, const X *tail,
                      const uint32_t *tail_bucket, uint32_t *worklist, uint32_t *worklist_len, X *partial, uint32_t *counter);
    static void bucket_merge(cudaStream_t st, uint32_t G, const uint32_t *piece_offsets, const X *piece_acc, X *bucket_acc);
    static void reduce(cudaStream_t st, uint32_t n_windows, uint32_t cnt_in, uint32_t K, uint32_t m_log2, const X *in_s, const X *in_a, X *out_s, X *out_a,
                       const uint32_t *bucket_offsets);
    static void weight(cudaStream_t st, uint32_t n_windows, uint32_t cnt, uint32_t m_log2, const X *in_s, const X *in_a, X *out);
    static void tree_sum(cudaStream_t st, uint32_t n_windows, const X *in, uint32_t cnt_in, X *out);
    // fold reduce (B >= 256): returns the number of kernels launched; F: n_windows * B points, partial: n_windows * nb * chunks_max,
    // V: n_windows * nb, out: n_windows
    // st2 / ev_fork / ev_join: a second stream on which the sums of the big upper halves (levels 1..3, 7/8 of that work) overlap the deep,
    // latency-bound fold levels
    static int fold_reduce(cudaStream_t st, cudaStream_t st2, cudaEvent_t ev_fork, cudaEvent_t ev_join, uint32_t n_windows, uint32_t B, const X *buckets,
                           const uint32_t *bucket_offsets, X *F, X *partial, X *V, X *out);
    static uint32_t fold_chunks_max(uint32_t B);
    static void final_horner(cudaStream_t st, const MsmShape &sh, const X *win_a, X *out);
    static void fold_inf(cudaStream_t st, A *pts, const uint8_t *inf, uint32_t n);
    static void precompute(cudaStream_t st, uint32_t n, uint32_t c, uint32_t W, uint32_t stride, const A *pts, A *table);
    static void point_op(cudaStream_t st, int op, const A *a, const A *b, uint32_t *out24, uint32_t n);
    static void gen_scalars(cudaStream_t st, uint64_t seed, uint64_t first, uint32_t n, S *out);
    static size_t fixed_table_points();  // entries of the table below
    static void fixed_table(cudaStream_t st, const A &g, A *table);
    static void fixed_base(cudaStream_t st, const S *k, const A *table, uint32_t n, A *out);
};

// Bucket sort by two block-local radix partitions (kernels_sort.cu): bucket index = (coarse bin << F) | fine bits.
struct SortPlan {
    uint32_t n, c, W;
    uint32_t nseg;            // independent bucket sets: W, or 1 when all windows share the buckets (precomputed window table)
    uint32_t nbins, F;        // coarse bins per segment, fine bits per bin (<= 8)
    uint32_t T;               // digits per partition tile
    uint32_t cap;             // elements of one bin that k_sort_buckets places in shared memory
    uint32_t pstride, poff;   // entry payload = w * pstride + poff + i  (MsmShape)
};
struct LaunchSort {
    // false: this shape is left to the counting sort (k_count / k_fill)
    static bool plan(const MsmShape &sh, SortPlan &pl);
    static size_t coarse_words(const SortPlan &pl);  // words of coarse_counts / coarse_off / cursor
    // scalar_field: 0 Fq, 1 Fr.  digits / part_pay / entries: n * W words, part_fine: n * W bytes, offsets: G + 1 words.  Returns the launches.
    static int run(cudaStream_t st, int scalar_field, int sm_count, const SortPlan &pl, const uint32_t *scalars, int is_mont, uint32_t *digits,
                   uint32_t *coarse_counts, uint32_t *coarse_off, uint32_t *cursor, uint32_t *part_pay, uint8_t *part_fine, uint32_t *entries, uint32_t *offsets,
                   cudaEvent_t ev_digits, cudaEvent_t ev_scan);
};

struct LaunchUtil {
    // field: 0 Fq, 1 Fr (test hook for the PTX carry chains)
    static void field_op(cudaStream_t st, int field, int op, const void *a, const void *b, void *out, uint32_t n);
    static void exclusive_scan(cudaStream_t st, const uint32_t *in, uint32_t *out, uint32_t len, uint32_t *tile_sums);
    static uint32_t scan_tiles(uint32_t len);
    static int scan_launches(uint32_t len);
    static void ubench(cudaStream_t st, int mode, int blocks, uint32_t *sink, int iters);          // modes 0..4
    static void ubench_fmul(cudaStream_t st, int blocks, void *sink, int iters);
    static void ubench_madd(cudaStream_t st, int blocks, void *sink, const AffinePt<Bn254G1> &p, const AffinePt<Bn254G1> &q, int iters);
    static void clock_probe(cudaStream_t st, uint64_t *out2);
};

// Fr NTT (kernels_ntt.cu).  Field elements are passed as opaque 32-byte Montgomery values.
struct LaunchNtt {
    static int passes(uint32_t k);
    static void pow_table(cudaStream_t st, void *out, const void *base32, uint32_t n);
    static void scale(cudaStream_t st, void *d, const void *table, const void *c32, uint32_t n);
    static void h_pointwise(cudaStream_t st, void *a, const void *b, const void *c, const void *zinv32, uint32_t n);
    static int transform(cudaStream_t st, void *d, const void *tw, uint32_t k);
    // the same transform of input already in bit-reversed order: the butterfly passes only
    static int transform_bitrev_input(cudaStream_t st, void *d, const void *tw, uint32_t k);
};

// Nova folding vector work (kernels_r1cs.cu).  field: 0 Fq, 1 Fr.
struct Csr;
struct LaunchR1cs {
    static void spmv(cudaStream_t st, int field, uint32_t m, const Csr &mat, const uint32_t *z, uint32_t *out);
    static void cross_term(cudaStream_t st, int field, uint32_t m, const Csr &a, const Csr &b, const Csr &c, const uint32_t *z1, const uint32_t *z2, uint32_t *t);
    static void vec_fold(cudaStream_t st, int field, uint32_t n, const uint32_t *a, const uint32_t *b, const uint32_t r8[8], uint32_t *out);
    // (A z) o (B z) = u (C z) + E row by row (e == nullptr: E = 0; strict: u = 1).  result: 3 words, on entry {0, 0xFFFFFFFF, 0}; on exit
    // [0] violating rows, [1] the first of them (0xFFFFFFFF if none), [2] strict only: z[0] == 1
    static void relaxed_check(cudaStream_t st, int field, uint32_t m, const Csr &a, const Csr &b, const Csr &c, const uint32_t *z, const uint32_t *e,
                              bool strict, uint32_t *result);
    // Groth16 (Fr only): A z, B z, C z over 2^k positions, zero padded, each stored at its bit-reversed index of out[0..2] (2^k elements each)
    static void evaluate(cudaStream_t st, uint32_t k, uint32_t m, const Csr &a, const Csr &b, const Csr &c, const uint32_t *z, uint32_t *const out[3]);
};

// Groth16 parameter generation over Fr (kernels_setup.cu, bodies in setup_kernels.cuh).  Each returns the kernels it launched.
struct LaunchSetup {
    // tau^i for i < 2^k from lo[j] = tau^j (j < 2^tau_log_t(k)) and hi[b] = tau^(2^tau_log_t(k) * b); out[0 .. n_h) is copied to h
    static uint32_t tau_log_t(uint32_t k) { return (k + 1) / 2; }
    static int tau_powers(cudaStream_t st, uint32_t k, const void *lo, const void *hi, void *out, uint32_t n_h, void *h);
    // out[j] = sum over the entries (i, j) of mat of coeff * lagr[i], j < n_z.  cnt: n_z + 1 words, zero on entry; ptr[0..1]: n_z + 1 words each;
    // vals[0..1]: nnz elements each; tile_sums: LaunchUtil::scan_tiles(n_z + 1) words
    static int column_sums(cudaStream_t st, uint32_t m, uint32_t n_z, const Csr &mat, uint32_t nnz, const void *lagr, uint32_t *cnt, uint32_t *const ptr[2],
                           void *const vals[2], uint32_t *tile_sums, void *out);
    // consts: alpha, beta, 1/gamma, 1/delta, (tau^n - 1)/delta (setup_kernels.cuh: SetupConsts); ext: n_z elements; h: n_h elements, tau^i on entry
    static int scalars(cudaStream_t st, uint32_t n_z, uint32_t n_inputs, uint32_t n_h, const void *consts, const void *u, const void *v, const void *w,
                       void *ext, void *h);
};

// BN254 pairing and Groth16 verification (kernels_pairing.cu, bodies in pairing.cuh).  Points are device affine forms (G1 64 bytes, G2 128
// bytes, the identity (0, 0)), Fq12 values 384 bytes, lines 192 bytes (MILLER_LINES per fixed G2 point), XYZZ G1 points 128 bytes.
struct LaunchPairing {
    static constexpr size_t G1_BYTES = 64, G2_BYTES = 128, FQ12_BYTES = 384, LINE_BYTES = 192, XYZZ_BYTES = 128;
    // ABI rows (9 / 17 words) -> device points; *bad |= 1 if any point is invalid
    static void load(cudaStream_t st, uint32_t n, const uint64_t *g1, const uint64_t *g2, void *p, void *q, uint32_t *bad);
    // proofs: k x 35 words; valid: k bytes; inputs_canon: k x n_public canonical Fr (32 bytes)
    static void validate_proofs(cudaStream_t st, uint32_t k, const uint64_t *proofs, const uint64_t *inputs, uint32_t n_public, void *a, void *b, void *c,
                                uint8_t *valid, void *inputs_canon);
    static void lines(cudaStream_t st, uint32_t n, const void *q, void *table);
    static void miller(cudaStream_t st, uint32_t n, const void *p, const void *q, void *f);
    // ceil(log2 n) levels ping-ponging between f[0] and f[1] (and sums[0] / sums[1], 2 XYZZ points per element, unless sums == nullptr); the
    // product lands in element 0 of buffer `root`.  Returns the launches.
    static int product_tree(cudaStream_t st, uint32_t n, void *f[2], void *sums[2], int &root);
    static int tree_levels(uint32_t n);
    static void final_exp(cudaStream_t st, uint32_t n, const void *f, void *out_gt, const uint8_t *valid, uint32_t *ok);
    // rho: k x 2 words; sums: 2 XYZZ points per proof (rho_i C_i, rho_i alpha); rho_mont: k x 32 bytes
    static void batch_prep(cudaStream_t st, uint32_t k, const uint64_t *rho, const uint8_t *valid, const void *a, const void *c, const void *alpha,
                           void *rho_a, void *sums, void *rho_mont);
    static void batch_colsum(cudaStream_t st, uint32_t k, uint32_t n_public, const void *rho_mont, const uint64_t *inputs, void *out);
    static void batch_fixed(cudaStream_t st, const void *f_root, const void *sums_root, const void *ic_sum, const void *lines, uint32_t present, void *out);
    static void ic_table(cudaStream_t st, uint32_t n_public, const void *ic, void *table);
    static void ic_straus(cudaStream_t st, uint32_t k, uint32_t n_public, const void *ic, const void *table, const void *inputs_canon, void *ic_x);
    static void verify_miller(cudaStream_t st, uint32_t k, const void *a, const void *b, const void *c, const void *alpha, const void *ic_x,
                              const void *lines, uint32_t present, void *f);
};

}  // namespace kgr
