// kernels_pairing.cu — the BN254 pairing and the Groth16 verifier on the device (bodies in pairing.cuh).  One pairing, or one proof's set of
// pairs, per thread.  Built with KGR_FP2_CALLS: the Fq2 and Fq6 products are shared __noinline__ calls, without which the Fq12 loop overflows
// the instruction cache.
#define KGR_FP2_CALLS 1
#include <cuda_runtime.h>

#include "launch.cuh"
#include "pairing.cuh"

namespace kgr {

constexpr int TPB_PAIR = 64;

// kgr_pairing input: ABI rows -> device points; bad[0] |= 1 for any invalid point
__global__ void __launch_bounds__(TPB_PAIR) k_pairing_load(uint32_t n, const uint64_t *g1, const uint64_t *g2, G1A *p, G2A *q, uint32_t *bad) {
    const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    bool ok = load_g1(g1 + 9 * (size_t)i, p[i]);
    ok = load_g2(g2 + 17 * (size_t)i, q[i]) && ok;
    if (!ok) atomicOr(bad, 1u);
}
__global__ void __launch_bounds__(TPB_PAIR) k_validate_proofs(uint32_t k, const uint64_t *proofs, const uint64_t *inputs, uint32_t n_public, G1A *a,
                                                               G2A *b, G1A *c, uint8_t *valid, Fp<FrP> *inputs_canon) {
    body_validate_proof(blockIdx.x * blockDim.x + threadIdx.x, k, proofs, inputs, n_public, a, b, c, valid, inputs_canon);
}
__global__ void __launch_bounds__(TPB_PAIR) k_pairing_lines(uint32_t n, const G2A *q, Line *table) {
    body_pairing_lines(blockIdx.x * blockDim.x + threadIdx.x, n, q, table);
}
// f_i = Miller(P_i, Q_i), lines on the fly
__global__ void __launch_bounds__(TPB_PAIR) k_miller(uint32_t n, const G1A *p, const G2A *q, Fq12 *f) {
    const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    f[i] = miller_one(p[i], q[i]);
}
// One level of the product tree: out[i] = in[2i] in[2i+1] (in[2i] alone for the odd tail); with sums != nullptr the same level also adds the
// two G1 sums of the batched check (rho_i C_i and rho_i alpha).
__global__ void __launch_bounds__(TPB_PAIR) k_product_level(uint32_t n, const Fq12 *in, Fq12 *out, const XyzzPt<Bn254G1> *sums_in,
                                                             XyzzPt<Bn254G1> *sums_out) {
    const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x, m = (n + 1) / 2;
    if (i >= m) return;
    const bool pair = 2 * i + 1 < n;
    out[i] = pair ? fq12_mul(in[2 * i], in[2 * i + 1]) : in[2 * i];
    if (sums_in) {
        for (int s = 0; s < 2; s++) {
            XyzzPt<Bn254G1> acc = sums_in[2 * (2 * i) + s];
            if (pair) xyzz_add(acc, sums_in[2 * (2 * i + 1) + s]);
            sums_out[2 * i + s] = acc;
        }
    }
}
// out_gt (if set) = final_exp(f_i); ok (if set) = valid_i (if set) && final_exp(f_i) == 1
__global__ void __launch_bounds__(TPB_PAIR) k_final_exp(uint32_t n, const Fq12 *f, Fq12 *out_gt, const uint8_t *valid, uint32_t *ok) {
    const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    Fq12 g = final_exp(f[i]);
    if (out_gt) out_gt[i] = g;
    if (ok) ok[i] = (!valid || valid[i]) && fq12_is_one(g);
}
// Batched check, per proof: rho_i A_i (affine, for its Miller loop), rho_i C_i and rho_i alpha (XYZZ, summed by the product tree), rho_i in
// Montgomery form for the column sums.  An invalid proof takes part with rho_i = 0.
__global__ void __launch_bounds__(TPB_PAIR) k_batch_prep(uint32_t k, const uint64_t *rho, const uint8_t *valid, const G1A *a, const G1A *c,
                                                          const G1A *alpha, G1A *rho_a, XyzzPt<Bn254G1> *sums, Fp<FrP> *rho_mont) {
    const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= k) return;
    const bool v = valid[i];
    const uint64_t lo = v ? rho[2 * i] : 0, hi = v ? rho[2 * i + 1] : 0;
    rho_a[i] = g1_affine(g1_mul_u128(a[i], lo, hi));
    sums[2 * i] = g1_mul_u128(c[i], lo, hi);
    sums[2 * i + 1] = g1_mul_u128(*alpha, lo, hi);
    Fp<FrP> r = fp_zero<FrP>();
    r.v[0] = (uint32_t)lo, r.v[1] = (uint32_t)(lo >> 32), r.v[2] = (uint32_t)hi, r.v[3] = (uint32_t)(hi >> 32);
    rho_mont[i] = fp_to_mont(r);
}
// Column sums of the batched check: out[0] = sum_i rho_i, out[j + 1] = sum_i rho_i x_ij (Montgomery Fr), one block per column
__global__ void __launch_bounds__(256) k_batch_colsum(uint32_t k, uint32_t n_public, const Fp<FrP> *rho_mont, const uint64_t *inputs, Fp<FrP> *out) {
    __shared__ Fp<FrP> part[256];
    const uint32_t col = blockIdx.x;
    Fp<FrP> acc = fp_zero<FrP>();
    for (uint32_t i = threadIdx.x; i < k; i += blockDim.x) {
        if (col == 0) {
            acc = fp_add(acc, rho_mont[i]);
        } else {
            Fp<FrP> x;
            const uint64_t *xw = inputs + 4 * ((size_t)i * n_public + col - 1);
            for (int q = 0; q < 4; q++) x.v[2 * q] = (uint32_t)xw[q], x.v[2 * q + 1] = (uint32_t)(xw[q] >> 32);
            acc = fp_add(acc, fp_mul(rho_mont[i], x));
        }
    }
    part[threadIdx.x] = acc;
    __syncthreads();
    for (uint32_t s = blockDim.x / 2; s; s >>= 1) {
        if (threadIdx.x < s) part[threadIdx.x] = fp_add(part[threadIdx.x], part[threadIdx.x + s]);
        __syncthreads();
    }
    if (threadIdx.x == 0) out[col] = part[0];
}
// Batched check, one thread: f_root e(-sum rho_i alpha, beta) e(-sum rho_i IC(x_i), gamma) e(-sum rho_i C_i, delta) from the line tables
__global__ void k_batch_fixed(const Fq12 *f_root, const XyzzPt<Bn254G1> *sums_root, const G1A *ic_sum, const Line *lines, uint32_t present, Fq12 *out) {
    if (blockIdx.x * blockDim.x + threadIdx.x) return;
    G1A fixed[3] = {g1_neg(g1_affine(sums_root[1])), g1_neg(*ic_sum), g1_neg(g1_affine(sums_root[0]))};
    G1A none{fp_zero<FqP>(), fp_zero<FqP>()};
    G2A none2{fq2_zero(), fq2_zero()};
    *out = fq12_mul(*f_root, miller_groth16(none, none2, fixed, lines, present));
}
// Per-proof path
__global__ void __launch_bounds__(TPB_PAIR) k_ic_table(uint32_t n_public, const G1A *ic, G1A *table) {
    body_ic_table(blockIdx.x * blockDim.x + threadIdx.x, n_public, ic, table);
}
__global__ void __launch_bounds__(TPB_PAIR) k_ic_straus(uint32_t k, uint32_t n_public, const G1A *ic, const G1A *table, const Fp<FrP> *inputs_canon,
                                                         G1A *ic_x) {
    const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= k) return;
    ic_x[i] = ic_combination(ic[0], table, inputs_canon + (size_t)i * n_public, n_public);
}
__global__ void __launch_bounds__(TPB_PAIR) k_verify_miller(uint32_t k, const G1A *a, const G2A *b, const G1A *c, const G1A *alpha, const G1A *ic_x,
                                                             const Line *lines, uint32_t present, Fq12 *f) {
    const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= k) return;
    G1A fixed[3] = {g1_neg(*alpha), g1_neg(ic_x[i]), g1_neg(c[i])};
    f[i] = miller_groth16(a[i], b[i], fixed, lines, present);
}

static inline unsigned blocks(size_t n, int tpb) { return (unsigned)((n + tpb - 1) / tpb); }

void LaunchPairing::load(cudaStream_t st, uint32_t n, const uint64_t *g1, const uint64_t *g2, void *p, void *q, uint32_t *bad) {
    k_pairing_load<<<blocks(n, TPB_PAIR), TPB_PAIR, 0, st>>>(n, g1, g2, (G1A *)p, (G2A *)q, bad);
}
void LaunchPairing::validate_proofs(cudaStream_t st, uint32_t k, const uint64_t *proofs, const uint64_t *inputs, uint32_t n_public, void *a, void *b,
                                    void *c, uint8_t *valid, void *inputs_canon) {
    k_validate_proofs<<<blocks(k, TPB_PAIR), TPB_PAIR, 0, st>>>(k, proofs, inputs, n_public, (G1A *)a, (G2A *)b, (G1A *)c, valid, (Fp<FrP> *)inputs_canon);
}
void LaunchPairing::lines(cudaStream_t st, uint32_t n, const void *q, void *table) {
    k_pairing_lines<<<1, 32, 0, st>>>(n, (const G2A *)q, (Line *)table);
}
void LaunchPairing::miller(cudaStream_t st, uint32_t n, const void *p, const void *q, void *f) {
    k_miller<<<blocks(n, TPB_PAIR), TPB_PAIR, 0, st>>>(n, (const G1A *)p, (const G2A *)q, (Fq12 *)f);
}
int LaunchPairing::product_tree(cudaStream_t st, uint32_t n, void *f[2], void *sums[2], int &root) {
    int launches = 0, cur = 0;
    while (n > 1) {
        const uint32_t m = (n + 1) / 2;
        k_product_level<<<blocks(m, TPB_PAIR), TPB_PAIR, 0, st>>>(n, (const Fq12 *)f[cur], (Fq12 *)f[cur ^ 1],
                                                                  sums ? (const XyzzPt<Bn254G1> *)sums[cur] : nullptr,
                                                                  sums ? (XyzzPt<Bn254G1> *)sums[cur ^ 1] : nullptr);
        launches++;
        cur ^= 1;
        n = m;
    }
    root = cur;
    return launches;
}
int LaunchPairing::tree_levels(uint32_t n) {
    int l = 0;
    for (; n > 1; n = (n + 1) / 2) l++;
    return l;
}
void LaunchPairing::final_exp(cudaStream_t st, uint32_t n, const void *f, void *out_gt, const uint8_t *valid, uint32_t *ok) {
    k_final_exp<<<blocks(n, TPB_PAIR), TPB_PAIR, 0, st>>>(n, (const Fq12 *)f, (Fq12 *)out_gt, valid, ok);
}
void LaunchPairing::batch_prep(cudaStream_t st, uint32_t k, const uint64_t *rho, const uint8_t *valid, const void *a, const void *c, const void *alpha,
                               void *rho_a, void *sums, void *rho_mont) {
    k_batch_prep<<<blocks(k, TPB_PAIR), TPB_PAIR, 0, st>>>(k, rho, valid, (const G1A *)a, (const G1A *)c, (const G1A *)alpha, (G1A *)rho_a,
                                                           (XyzzPt<Bn254G1> *)sums, (Fp<FrP> *)rho_mont);
}
void LaunchPairing::batch_colsum(cudaStream_t st, uint32_t k, uint32_t n_public, const void *rho_mont, const uint64_t *inputs, void *out) {
    k_batch_colsum<<<n_public + 1, 256, 0, st>>>(k, n_public, (const Fp<FrP> *)rho_mont, inputs, (Fp<FrP> *)out);
}
void LaunchPairing::batch_fixed(cudaStream_t st, const void *f_root, const void *sums_root, const void *ic_sum, const void *lines, uint32_t present,
                                void *out) {
    k_batch_fixed<<<1, 32, 0, st>>>((const Fq12 *)f_root, (const XyzzPt<Bn254G1> *)sums_root, (const G1A *)ic_sum, (const Line *)lines, present,
                                    (Fq12 *)out);
}
void LaunchPairing::ic_table(cudaStream_t st, uint32_t n_public, const void *ic, void *table) {
    k_ic_table<<<blocks(n_public, TPB_PAIR), TPB_PAIR, 0, st>>>(n_public, (const G1A *)ic, (G1A *)table);
}
void LaunchPairing::ic_straus(cudaStream_t st, uint32_t k, uint32_t n_public, const void *ic, const void *table, const void *inputs_canon, void *ic_x) {
    k_ic_straus<<<blocks(k, TPB_PAIR), TPB_PAIR, 0, st>>>(k, n_public, (const G1A *)ic, (const G1A *)table, (const Fp<FrP> *)inputs_canon, (G1A *)ic_x);
}
void LaunchPairing::verify_miller(cudaStream_t st, uint32_t k, const void *a, const void *b, const void *c, const void *alpha, const void *ic_x,
                                  const void *lines, uint32_t present, void *f) {
    k_verify_miller<<<blocks(k, TPB_PAIR), TPB_PAIR, 0, st>>>(k, (const G1A *)a, (const G2A *)b, (const G1A *)c, (const G1A *)alpha, (const G1A *)ic_x,
                                                              (const Line *)lines, present, (Fq12 *)f);
}

}  // namespace kgr
