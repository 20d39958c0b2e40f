/* kgr_msm.h — C ABI of the B200-native MSM engine for Kogarashi's BN254 G1 and Grumpkin curves, and of the rows built around it
 * (BN254 G2 MSM, Fr NTT + Groth16 H polynomial, Nova folding vector work).
 *
 * The reference has no FFI for this path: the boundary is two Rust functions,
 *   groth16/src/msm.rs:6        fn msm_curve_addition<C: BNAffine>(bases: &[C], coeffs: &[C::Scalar]) -> C::Extended
 *   nova/src/pedersen.rs:15     fn PedersenCommitment::<C>::commit(&self, m: &DenseVectors<C::Scalar>) -> C
 * and the zkstd trait surface they are generic over (zkstd/src/traits/curve/weierstrass.rs:7-97,
 * zkstd/src/traits/field.rs:13-40).  This header is what a Rust `extern "C"` block (see
 * INTEGRATION.md and rust/kogarashi-msm-b200) or any other FFI binds instead.
 *
 * Data formats (all little endian, plain pointers, caller-owned for the duration of the call):
 *   points   n x 8 uint64   x[4] || y[4], Montgomery limbs exactly as stored in bn_254::Fq /
 *                           bn_254::Fr (`inner()`, bn254/src/fq.rs:102, fr.rs:118)
 *   inf      n x uint8      is_infinity flags (bn254/src/g1.rs:21); NULL = no identity points
 *   scalars  n x 4 uint64   KGR_SCALARS_MONTGOMERY: the in-memory form (`Fr.0`, fr.rs:71);
 *                           KGR_SCALARS_CANONICAL:  `to_raw_bytes()` output read as 4 LE words
 *                           (zkstd/src/macros/field.rs:102-104), must be < the scalar modulus
 *   result   12 uint64      homogeneous projective X[4] Y[4] Z[4] in Montgomery form, i.e. the
 *                           fields of G1Projective / grumpkin::Projective (g1.rs:119); identity =
 *                           (0, R, 0) as in zkstd/src/macros/curve/weierstrass/group.rs:106-110.
 *                           Any representative of the correct group element may be returned;
 *                           compare after to_affine (macros/curve/weierstrass.rs:57-66).  The
 *                           representative is NOT stable from run to run: the order of the entries inside
 *                           a bucket depends on the order in which thread blocks claim their ranges, and a
 *                           different summation order gives a different (X : Y : Z) of the same point.
 *                           The normalised affine point is bit-identical every time.
 *
 * Every function returns 0 on success or a negative KGR_E_* code; kgr_last_error() gives the
 * text for the calling thread.  No C++ exception crosses this boundary.  There is no CPU
 * fallback: without a usable CUDA device kgr_init fails with KGR_E_NO_DEVICE.
 */
#ifndef KGR_MSM_H
#define KGR_MSM_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

/* KGR_CURVE_BN254_G2 (next row N3; bn254/src/g2.rs:15-21, the b_g2 queries of groth16/src/prover.rs:64-65): coordinates are
 * Fq2 elements c0 || c1 (fqn.rs), so wherever a size below says 4 limbs per coordinate G2 uses 8: points n x 16 uint64,
 * projective results 24, affine results 17 (x[8] y[8] is_infinity). */
enum { KGR_CURVE_BN254_G1 = 0, KGR_CURVE_GRUMPKIN = 1, KGR_CURVE_BN254_G2 = 2 };
enum { KGR_SCALARS_MONTGOMERY = 0, KGR_SCALARS_CANONICAL = 1 };
enum {
    KGR_OK = 0,
    KGR_E_NO_DEVICE = -1,   /* no CUDA device / driver */
    KGR_E_CUDA = -2,        /* a CUDA runtime call failed (see kgr_last_error) */
    KGR_E_ARG = -3,         /* bad argument */
    KGR_E_NOT_INIT = -4,    /* kgr_init has not been called */
    KGR_E_TOO_LARGE = -5    /* exceeds the engine's limits */
};

typedef struct kgr_bases kgr_bases_t; /* opaque handle: a point vector resident on the GPUs */

/* Select the GPUs of this process.  devices == NULL or n_devices == 0: the current device only.
 * Large MSMs are sharded evenly over the listed devices, each returns one partial point
 * (one D2H copy per GPU) and the host adds them; no NCCL is involved. */
int kgr_init(const int *devices, int n_devices);
int kgr_shutdown(void);
const char *kgr_last_error(void);
int kgr_device_count(void); /* devices selected by kgr_init (0 before) */

/* Upload a base vector once (Groth16 CRS queries `params.{h,l,a,b_g1}`, groth16/src/prover.rs:51-62;
 * Pedersen `ck.g`, nova/src/pedersen.rs:6-13).  The vector is split into contiguous shards, one per device. */
int kgr_bases_register(int curve, const uint64_t *xy, const uint8_t *inf, size_t n, kgr_bases_t **out);
int kgr_bases_free(kgr_bases_t *bases);
size_t kgr_bases_len(const kgr_bases_t *bases);

/* Optional, for vectors that are reused many times (a CRS, a Pedersen key): build the table
 * 2^(c*w) * P_i for every window w on the device (W x the memory of the vector; one-time cost of about
 * 254 doublings + W inversions per point).  Afterwards every kgr_msm* call on this handle runs in
 * window-collapsed mode: all windows share one bucket set, so the bucket reduction shrinks W-fold and
 * the 254 final doublings disappear.  window_bits = 0 picks c from the cost model.  The result is the
 * same group element. */
int kgr_bases_precompute(kgr_bases_t *bases, int window_bits);

/* sum_{i<n} scalars[i] * bases[base_off + i]   (replaces msm_curve_addition, groth16/src/msm.rs:6-48).
 * Host scalars; the H2D copy of the scalars and the 96-byte D2H of the result are part of the call. */
int kgr_msm(kgr_bases_t *bases, size_t base_off, const uint64_t *scalars, int scalar_fmt, size_t n, uint64_t *out /* [12] */);

/* Several independent MSMs on registered vectors in one call — the prover's h, l, a, b_g1 and b_g2 queries (groth16/src/prover.rs:51-65,
 * SURVEY row N1: "overlap the MSMs on streams").  Same results as calling kgr_msm on each job in order.  With one device selected the
 * jobs run on up to eight independent lanes (stream + workspace) of that device, so the latency-bound tail of one MSM overlaps the
 * bulk of the next; with several devices every MSM is already spread over all of them and the jobs run in sequence. */
typedef struct kgr_msm_job {
    kgr_bases_t *bases;
    size_t base_off;
    const uint64_t *scalars;
    int scalar_fmt;
    size_t n;
    uint64_t *out; /* [12], or [24] for G2 */
} kgr_msm_job_t;
int kgr_msm_batch(const kgr_msm_job_t *jobs, size_t n_jobs);

/* Same with everything passed from host memory each call; pairs = min(n_bases, n_scalars) exactly
 * like coeffs.iter().zip(bases.iter()) (msm.rs:25). */
int kgr_msm_oneshot(int curve, const uint64_t *xy, const uint8_t *inf, size_t n_bases, const uint64_t *scalars, int scalar_fmt,
                    size_t n_scalars, uint64_t *out /* [12] */);

/* Scalars already resident on the device that holds the bases (single-device contexts only):
 * d_scalars is a device pointer to n x 4 uint64.  Used for kernel-only timing and by callers
 * that produce scalars on the GPU. */
int kgr_msm_device(kgr_bases_t *bases, size_t base_off, const void *d_scalars, int scalar_fmt, size_t n, uint64_t *out /* [12] */);

/* Copy n registered points starting at `off` back to the host (x||y Montgomery; identity entries
 * come back as (0, 0), the device encoding). */
int kgr_bases_download(const kgr_bases_t *bases, size_t off, size_t n, uint64_t *xy_out);

/* PedersenCommitment::commit (nova/src/pedersen.rs:15-20): MSM followed by to_affine.
 * out = x[4] y[4] is_infinity (identity -> (0, R, 1) as in group.rs:22-26). */
int kgr_pedersen_commit(kgr_bases_t *ck, const uint64_t *scalars, int scalar_fmt, size_t n, uint64_t *out /* [9] */);

/* Projective -> affine normalisation on the host (zkstd/src/macros/curve/weierstrass.rs:57-66);
 * out = x[4] y[4] is_infinity. */
int kgr_to_affine(int curve, const uint64_t *in, uint64_t *out);
/* a + b on the host for two projective points (used to combine per-GPU / per-rank partial sums). */
int kgr_proj_add(int curve, const uint64_t *a, const uint64_t *b, uint64_t *out);

/* ---- Fr NTT (next row N2: groth16/src/fft.rs) --------------------------------------------------
 * Radix-2 transforms over bn254 Fr on a domain of size 2^log_n, semantics of groth16/src/fft.rs:92-127:
 * op 0 dft, 1 idft, 2 coset_dft, 3 coset_idft.  in: n_in <= 2^log_n Montgomery elements (zero padded like
 * prepare_fft, fft.rs:157-162); out: 2^log_n elements; *n_out: length after Coefficients::new stripped the
 * trailing zeros (idft variants, poly.rs:61-63), else 2^log_n.  Host buffers. */
int kgr_ntt(unsigned log_n, int op, const uint64_t *in, size_t n_in, uint64_t *out, size_t *n_out);
/* Same transform in place on 2^log_n elements already in device memory (no stripping). */
int kgr_ntt_device(unsigned log_n, int op, void *d_data);
/* groth16/src/prover.rs:36-47 in one call: q = coset_idft((coset_dft(idft(a)) * coset_dft(idft(b)) - coset_dft(idft(c))) / Z).
 * a, b, c: the m R1CS evaluations each (host, Montgomery); out: 2^log_n elements, *n_out after stripping. */
int kgr_groth16_h(unsigned log_n, const uint64_t *a, const uint64_t *b, const uint64_t *c, size_t m, uint64_t *out, size_t *n_out);

/* ---- Nova folding vector work (next row N4: nova/src/prover.rs:53-90, relaxed_r1cs/witness.rs:56-71) ----------------
 * An R1CS shape: A, B, C as CSR over flat column indices into z = (u, x, w) — the caller resolves Wire::Instance(i) -> i and
 * Wire::Witness(i) -> i + l (zkstd/src/matrix.rs:41-44) when it builds the arrays.  field: 0 = Fq (nova's GrumpkinDriver),
 * 1 = Fr (Bn254Driver).  row_ptr[k]: m + 1 offsets, cols[k]: nnz column indices, coeffs[k]: nnz x 4 uint64 Montgomery; k = A, B, C.
 * The shape lives on the first device of kgr_init. */
typedef struct kgr_r1cs kgr_r1cs_t;
int kgr_r1cs_register(int field, size_t m, size_t n_z, const uint32_t *const row_ptr[3], const uint32_t *const cols[3],
                      const uint64_t *const coeffs[3], kgr_r1cs_t **out);
int kgr_r1cs_free(kgr_r1cs_t *shape);
/* SparseMatrix::prod (matrix.rs:36-48): out (m x 4) = M z, which = 0 A, 1 B, 2 C; z: n_z x 4 uint64 Montgomery, host buffers. */
int kgr_r1cs_mul(kgr_r1cs_t *shape, int which, const uint64_t *z, uint64_t *out);
/* compute_cross_term (prover.rs:53-90): T = AZ1 o BZ2 + AZ2 o BZ1 - u1 CZ2 - u2 CZ1 with u1 = z1[0], u2 = z2[0] (the reference passes
 * z2 = (1, x2, w2)), in one fused kernel.  t_out (m x 4, host) may be NULL.  With ck != NULL the Pedersen commitment of T
 * (prover.rs:35, `self.ck.commit(&t)`) is computed from the device-resident T without copying it: commit_out = x[4] y[4] is_infinity.
 * ck must be registered on the first device only and its scalar field must equal `field`. */
int kgr_nova_cross_term(kgr_r1cs_t *shape, const uint64_t *z1, const uint64_t *z2, uint64_t *t_out, kgr_bases_t *ck, uint64_t *commit_out);
/* ms[0] H2D of z1 and z2, ms[1] cross-term kernel, ms[2] commitment MSM (device events + host finish) of the last kgr_nova_cross_term. */
int kgr_r1cs_last_timing(const kgr_r1cs_t *shape, float ms[3]);
/* RelaxedR1csWitness::fold (witness.rs:67-68): out[i] = a[i] + b[i] * r over `field`; host buffers, n x 4 uint64 Montgomery
 * (kgr_vec_fold_device below keeps all three vectors on the GPU). */
int kgr_vec_fold(int field, const uint64_t *a, const uint64_t *b, const uint64_t r[4], size_t n, uint64_t *out);

/* ---- device-resident vectors (Nova: z = (u, x, w), E and T stay on the GPU between folding steps) ----------------------------------
 * nova/src/relaxed_r1cs/witness.rs:20-21,56-71 and nova/src/ivc.rs:160-205: every IVC step commits the new witness, computes and commits the
 * cross term and folds (w, e) — with host buffers each of those vectors crosses PCIe in both directions per step.  A kgr_vec_t is a vector
 * of field elements (field 0 = Fq, 1 = Fr; Montgomery, n x 4 uint64) on the first device of kgr_init. */
typedef struct kgr_vec kgr_vec_t;
int kgr_vec_upload(int field, const uint64_t *host, size_t n, kgr_vec_t **out);   /* host == NULL: n zero elements */
int kgr_vec_download(const kgr_vec_t *v, size_t off, size_t n, uint64_t *host);
int kgr_vec_free(kgr_vec_t *v);
size_t kgr_vec_len(const kgr_vec_t *v);
/* Overwrite elements [off, off + n) from host memory (the step's public inputs / fresh witness entering a resident z). */
int kgr_vec_write(kgr_vec_t *v, size_t off, const uint64_t *host, size_t n);
/* RelaxedR1csWitness::fold on the device: out[i] = a[i] + b[i] * r for i < n = len(out); out may be a or b.  (witness.rs:67-68) */
int kgr_vec_fold_device(const kgr_vec_t *a, const kgr_vec_t *b, const uint64_t r[4], kgr_vec_t *out);
/* sum_{i<n} scalars[sc_off + i] * bases[base_off + i] with the scalars taken from a resident vector (their field must be the curve's scalar
 * field; bases on the first device only): the commitment `ck.commit(&w)` of a witness that never left the GPU (w = z[1 + l ..]). */
int kgr_msm_vec(kgr_bases_t *bases, size_t base_off, const kgr_vec_t *scalars, size_t sc_off, size_t n, uint64_t *out /* [12] */);
/* PedersenCommitment::commit of the elements [sc_off, sc_off + n) of a resident vector: out = x[4] y[4] is_infinity. */
int kgr_pedersen_commit_vec(kgr_bases_t *ck, const kgr_vec_t *m, size_t sc_off, size_t n, uint64_t *out /* [9] */);
/* kgr_nova_cross_term with z1, z2 resident (n_z elements each) and T left in the resident vector t (m elements; NULL: internal buffer).
 * With ck != NULL also commit(T).  No host <-> device traffic except the 72-byte commitment. */
int kgr_nova_cross_term_device(kgr_r1cs_t *shape, const kgr_vec_t *z1, const kgr_vec_t *z2, kgr_vec_t *t, kgr_bases_t *ck, uint64_t *commit_out);
/* R1csShape::is_sat (strict, e == NULL) / the relaxed check (e != NULL) on resident vectors (nova/src/relaxed_r1cs.rs:80-146): for every row
 * i < m, (A z)_i (B z)_i = u (C z)_i + E_i with z = (u, x, w) flat (z->n >= n_z), u = z[0] and E = e[0, m) when relaxed, u = 1 and E = 0 when
 * strict.  W = z[w_off, n_z).  With ck (a BN254 G1 or Grumpkin key whose scalar field is the shape's field, one shard on the first device):
 * commit(W) is compared with commit_w and commit(E) with commit_e, each zipped with ck.g (pedersen.rs:15-20, min length) and compared as zkstd
 * compares affine points (group.rs:5-13: an identity equals only an identity, otherwise x and y limb for limb).  Expected commitments use the
 * layout kgr_pedersen_commit* returns, x[4] y[4] is_infinity.  Either may be NULL, which skips that check: which commitments the reference's
 * relaxed check re-derives (W only, or W and E) is not recorded here, so the caller chooses; the strict check re-derives commit(W) (:143).
 * The relation runs on the library's stream, the two MSMs on two further lanes at the same time ("lane_threads" as kgr_groth16_msms).  Work
 * enqueued on the library's stream before the call (a fold or cross term writing z or e) is complete before z or e is read.
 * report[6]: [0] sat (1 iff every check made holds)  [1] rows violating (A z)o(B z) = u (C z) + E  [2] first violating row (m if none)
 *            [3] commit(W) == commit_w: 1 equal, 0 different, 2 not checked  [4] commit(E) == commit_e: same  [5] u: 1 if relaxed or z[0] == 1
 * An unsatisfied instance is KGR_OK with report[0] == 0, not an error.
 * Refused with KGR_E_ARG before any work: a NULL shape, z or report; a shape, vector or key from before the last kgr_init; vector fields that
 * differ from the shape's; a ck of another scalar field, another curve or more than one shard; z->n < n_z or e->n < m; w_off outside 1 .. n_z;
 * commit_w or commit_e without ck; commit_e in strict mode. */
int kgr_nova_is_sat(const kgr_r1cs_t *shape, const kgr_vec_t *z, const kgr_vec_t *e, size_t w_off, kgr_bases_t *ck,
                    const uint64_t *commit_w /* [9] or NULL */, const uint64_t *commit_e /* [9] or NULL */, uint64_t *report /* [6] */);

/* Page-locked host memory for callers that marshal into a reusable arena instead of a fresh pageable buffer per call (a Rust Vec is
 * pageable: the library then stages it through its own pinned ring, one extra copy).  cudaHostAlloc / cudaFreeHost underneath. */
int kgr_host_alloc(size_t bytes, void **out);
int kgr_host_free(void *p);

/* groth16/src/prover.rs:36-65 as one call (row N1): the H coefficients are computed on the device (as kgr_groth16_h), fed to the h query
 * `msm(params.h, q)` without leaving the device, and the other queries of the prover (`jobs`: l, a, b_g1, b_g2, blinding sums ...) overlap with that
 * on separate lanes like kgr_msm_batch.  h must be a BN254 G1 vector; h_out: its projective result [12].  q_out (2^log_n x 4, host) and q_len
 * (length after stripping trailing zeros) are optional.  Same results as kgr_groth16_h + kgr_msm + kgr_msm_batch. */
int kgr_groth16_msms(unsigned log_n, const uint64_t *a, const uint64_t *b, const uint64_t *c, size_t m, kgr_bases_t *h, uint64_t *h_out, uint64_t *q_out,
                     size_t *q_len, const kgr_msm_job_t *jobs, size_t n_jobs);

/* groth16/src/prover.rs:32-65 from the constraint system: cs.evaluate() (r1cs.rs:137-142) on the device from the registered shape cs (field 1 = Fr)
 * and the resident assignment z = cs.x() ++ cs.w() (z->n == n_z of the shape; the first n_inputs elements are the instance, the constant one first),
 * H as kgr_groth16_h, then the queries with scalars read from z on the device:
 *   h: q (2^log_n coefficients, never leaving the device)   l: z[n_inputs ..]   a, b_g1, b_g2: z (inputs and aux fused, as prover.rs:58-65)
 * out: h[12] l[12] a[12] b_g1[12] b_g2[24] projective results (b_g2 == NULL: a G1-only prover, the last 24 words are not written).
 * jobs: further MSMs with host scalars (the blinding sums) on the other lanes, as in kgr_groth16_msms.  q_out / q_len as there.
 * Pairs are zipped (msm.rs:25): h min(2^log_n, len), a / b_g1 / b_g2 min(len, n_z), l min(len, n_z - n_inputs); no pairs gives the identity.
 * Requires 2^log_n >= m (nothing is truncated) and a single-device context: every handle on the first device, unsplit.  Work enqueued on the
 * library's stream before the call (kgr_vec_fold_device, kgr_nova_cross_term_device writing z) is complete before z is read. */
int kgr_groth16_prove_r1cs(unsigned log_n, const kgr_r1cs_t *cs, const kgr_vec_t *z, size_t n_inputs, kgr_bases_t *h, kgr_bases_t *l, kgr_bases_t *a,
                           kgr_bases_t *b_g1, kgr_bases_t *b_g2, uint64_t *out, uint64_t *q_out, size_t *q_len, const kgr_msm_job_t *jobs, size_t n_jobs);

/* groth16/src/zksnark.rs:17-127 (ZkSnark::setup) on the device, from a shape registered over Fr (field 1) and its number of instance variables
 * (the constant one included, z = x ++ w as kgr_groth16_prove_r1cs).  toxic: alpha, beta, gamma, delta, tau, 4 x u64 Montgomery each (< r).
 * With n = 2^k, k = max(1, ceil(log2 m)), l_i = L_i(tau) over that domain and u_j, v_j, w_j = sum_i A/B/C[i][j] * l_i:
 *   a_j = u_j * G1   b_g1_j = v_j * G1   b_g2_j = v_j * G2   ic_j (j < n_inputs) = (beta u_j + alpha v_j + w_j) / gamma * G1
 *   l_j (j >= n_inputs) = (beta u_j + alpha v_j + w_j) / delta * G1   h_i = tau^i (tau^n - 1) / delta * G1 for i < m - 1
 * Outputs are new single-shard handles on the first device, ready for kgr_groth16_prove_r1cs:
 *   a, b_g1, b_g2: n_z points   ic: n_inputs   l: n_z - n_inputs   h: m - 1   (the identity, stored (0, 0), where the exponent is 0)
 * vk_g1: alpha, beta, delta (3 x 9: x[4] y[4] is_infinity);  vk_g2: beta, gamma, delta (3 x 17); an identity reads (0, 0, 1).
 * *log_n_out = k.  b_g2 == NULL: no G2 query is built (vk_g2 may then be NULL too; it is filled whenever it is given).
 * The h query has m - 1 entries, as the reference builds it.  H = (AB - C) / Z has up to n - 1 coefficients, so for m < 2^k a proof can need
 * entries the query lacks: proofs are guaranteed valid for m = 2^k only.
 * Refused with KGR_E_ARG before any work, every output handle left NULL: a NULL required pointer, a shape registered before the last kgr_init,
 * a shape over Fq, n_inputs == 0 or > n_z, k > 28, toxic values >= r, gamma == 0 or delta == 0, a context of more than one device.
 * On a later failure everything allocated is freed. */
int kgr_groth16_setup(const kgr_r1cs_t *cs, size_t n_inputs, const uint64_t toxic[20], uint32_t *log_n_out, kgr_bases_t **h, kgr_bases_t **l,
                      kgr_bases_t **a, kgr_bases_t **b_g1, kgr_bases_t **b_g2, kgr_bases_t **ic, uint64_t *vk_g1, uint64_t *vk_g2);
/* Device time (ms, CUDA events) of the phases of the last kgr_groth16_setup: [0] powers of tau + idft, [1] column index + sums of A, B, C,
 * [2] scalars, fixed-base multiplications of [3] a, [4] b_g1, [5] ic, [6] l, [7] h, [8] b_g2, [9] vk.  The one-time NTT and generator tables
 * of a device are built before [0] and are not included. */
int kgr_groth16_setup_last_timing(float ms[10]);

/* Reduced optimal-ate pairing on BN254 (the map the Groth16 check of groth16/src/proof.rs:39-48 evaluates).
 * g1: n x 9 words (x[4] y[4] is_infinity, Montgomery Fq), g2: n x 17 (x.c0 x.c1 y.c0 y.c1 is_infinity); a set flag means the identity.
 * op 0: out = n x 48 words, e(P_i, Q_i) each;  op 1: out = 48 words, prod_i e(P_i, Q_i) (one final exponentiation; n == 0 gives 1).
 * Gt is 12 Fq elements, Montgomery, order c0.c0.c0, c0.c0.c1, c0.c1.c0, ..., c1.c2.c1 (Fq12 = c0 + c1 w, Fq6 = c0 + c1 v + c2 v^2,
 * w^2 = v, v^3 = 9 + u).  A pair with an identity contributes 1.
 * Points off their curve, a G2 point outside G2, or a coordinate >= p: KGR_E_ARG. */
int kgr_pairing(const uint64_t *g1, const uint64_t *g2, size_t n, int op, uint64_t *out);

/* Groth16 verification of k proofs against one verifying key (groth16/src/verifier.rs).  vk_g1: alpha, beta, delta (3 x 9), vk_g2: beta,
 * gamma, delta (3 x 17), the layout kgr_groth16_setup writes; ic: a BN254 G1 handle of n_public + 1 points (ic_0 carries the constant one).
 * proofs: k x 35 = A[9] B[17] C[9], the prover's output.  inputs: k x n_public x 4 Montgomery Fr, the instance WITHOUT its leading one.
 * ok[i] = 1 iff  e(A_i, B_i) = e(alpha, beta) e(ic_0 + sum_j x_ij ic_{j+1}, gamma) e(C_i, delta)  and every point of proof i is valid (each
 * coordinate < p, A and C on the curve, B on the twist and in G2; a set is_infinity flag is the identity).  A failing proof gets 0, not an error.
 * k >= 2 needs rho (k x 2 words, 128-bit, non-zero, unpredictable to whoever made the proofs): one batched check
 *   prod_i e(rho_i A_i, B_i) * e(-sum_i rho_i IC(x_i), gamma) * e(-sum_i rho_i C_i, delta) * e(-(sum_i rho_i) alpha, beta) == 1
 * over the valid proofs; if it fails, every proof is checked on its own.  k == 1: the per-proof check (rho ignored).
 * KGR_E_ARG before any work: NULL pointers, ic not a single-shard G1 handle of the current kgr_init, n_public + 1 != ic->n, an input >= r,
 * k >= 2 without rho or with a zero rho_i, an invalid verifying-key point, an identity gamma or delta, a context of more than one device.
 * k == 0: KGR_OK, nothing done. */
int kgr_groth16_verify(const uint64_t *vk_g1, const uint64_t *vk_g2, kgr_bases_t *ic, const uint64_t *proofs, size_t k,
                       const uint64_t *inputs, size_t n_public, const uint64_t *rho, uint32_t *ok);

/* Tuning knobs: "window_bits" (0 = auto), "chunk" (entries per accumulate thread, 0 = auto),
 * "reduce_fanin" (power of two), "running_sum_stop" (elements per window below which the reduce
 * switches from running sums to the parallel weighting pass), "final_on_device" (1: Horner over
 * windows in a one-thread kernel and one point per GPU in the D2H copy; 0 (default): the W window
 * sums come back in one D2H copy and the host applies the doublings), "sort_mode" (-1 auto, 0 counting sort with a per-scalar fill,
 * 1 counting sort with a window-major fill from stored digits, 2 two block-local radix partitions: the default from 2^21 entries on), "reduce_mode" (1 fold reduce, 0 running sums), "affine_levels" (levels of pairwise batched-affine
 * sums inside every bucket before the XYZZ accumulation, affine_kernels.cuh: -1 (default) automatic from the entry count, 0 none, 1..5; 8-word curves only),
 * "dense_x" (a dense copy of the x coordinates for the level-0 denominators of the batched-affine levels: -1 (default) automatic, 0 off, 1 on),
 * "oneshot_split" (pieces a large single-device kgr_msm_oneshot call is cut into so that uploads
 * overlap the pipeline; 0 (default) = automatic: 2 pieces from 2^20 pairs to 5 from 2^24 when points and scalars are uploaded, 2 - 3 from 2^22 for scalars only; 1 = off), "oneshot_growth" (size of piece i + 1
 * in percent of piece i: the first upload overlaps nothing, so it is the smallest; 0 (default) = automatic, 100 = equal pieces), "lane_threads" (kgr_groth16_msms: 1 (default) one
 * host thread per lane, 0 everything enqueued from the calling thread). */
/* The tuning state belongs to the CALLING THREAD: kgr_set_param changes the values used by MSMs this thread issues afterwards (the
 * library's own worker threads inherit the caller's snapshot) and never those of a call in flight on another thread. */
int kgr_set_param(const char *name, long value);

/* Per-phase time (ms) of the last MSM on device slot `dev`, CUDA events on the engine's stream:
 * [1] count, [2] scan, [3] fill, [4] accumulate, [5] fixup, [6] reduce (+ D2H of the window sums),
 * [7] H2D of scalars (and bases for oneshot); [8] host finish (Horner over windows + sum over GPUs,
 * host clock); [0] total = device events start..end + [8].  shape = {c, W, B, L, K, n}.  For a host-buffer call that was cut into pipelined
 * pieces ("oneshot_split") the phases are summed over the pieces (they overlap, so they can exceed the total), [0] spans the first piece's start
 * to the last piece's end, and c, W, B, L describe the first piece. */
int kgr_last_timing(int dev, float ms[9], uint32_t shape[6]);

/* CUDA events on the engine's own stream (the stream every kernel of this library is launched
 * on), for timing a region of calls from outside: 4 event slots per device slot. */
int kgr_event_record(int dev, int idx);
int kgr_event_elapsed_ms(int dev, int idx_a, int idx_b, float *ms);
/* Number of kernels this library has launched on device slot `dev` since kgr_init. */
int kgr_launch_count(int dev, uint64_t *count);

/* ---- test / bench utilities (exercise the same device code the MSM uses) ------------------- */
/* Elementwise field ops on the device: field 0 = Fq, 1 = Fr; op 0 add 1 sub 2 mul 3 sqr 4 neg
 * 5 from_mont 6 to_mont 7 inv (Fermat) 8 dbl 9 inv (safegcd divsteps).  a, b, out: host arrays of n x 4 uint64. */
int kgr_test_field_op(int field, int op, const uint64_t *a, const uint64_t *b, size_t n, uint64_t *out);
/* Elementwise point ops: op 0: proj(a_xyzz-from-affine madd b_affine), i.e. a + b for affine inputs with flags
 * (inf bytes may be NULL); out n x 12 projective. op 1: a + a.  op 2: a + b computed through xyzz_add. */
int kgr_test_point_op(int curve, int op, const uint64_t *a_xy, const uint8_t *a_inf, const uint64_t *b_xy, const uint8_t *b_inf, size_t n,
                      uint64_t *out);
/* out[i] = k[i] * G as affine (x||y Montgomery), computed on the device (fixed-base double-and-add +
 * batched normalisation).  k: host n x 4 uint64, Montgomery form of the curve's scalar field. */
int kgr_fixed_base_mul(int curve, const uint64_t *k, size_t n, uint64_t *out_xy);
/* Same but leaves the points on the device as a registered base vector (for large benchmarks).
 * Scalars are derived on the device from a 64-bit seed (splitmix64 -> 8 words -> from_u512 like
 * zkstd/src/arithmetic/limbs/bits_256/represent.rs:18-28,80-103).  If k_out != NULL it receives the n scalars (Montgomery). */
int kgr_bases_generate(int curve, uint64_t seed, size_t n, kgr_bases_t **out, uint64_t *k_out);
/* The same stream from global index `first` on: point i of the result is point first + i of kgr_bases_generate(curve, seed, ...), so
 * processes that each hold one shard of a large synthetic vector (bench.py under torchrun) together hold the vector a single process would
 * generate.  Benchmark / test inputs only: the discrete logarithms are public. */
int kgr_bases_generate_at(int curve, uint64_t seed, uint64_t first, size_t n, kgr_bases_t **out, uint64_t *k_out);
/* Integer-pipe microbenchmark on device slot 0: fills results[0..7] with giga-ops/s of
 * [0] IMAD (mad.lo.u32), [1] IMAD.HI, [2] IMAD.WIDE.U32, [3] IMAD.WIDE.U32.X carry chains,
 * [4] IADD3, [5] field multiplications (Fq), [6] XYZZ mixed adds, [7] SM clock MHz seen. */
int kgr_microbench(double results[8]);

#ifdef __cplusplus
}
#endif
#endif /* KGR_MSM_H */
