// kernels_r1cs.cu — sparse R1CS matrix-vector products, the Nova cross term, the relaxed-R1CS check and the witness fold (row N4), Fq and Fr.
// One thread per row; a row's coefficients stream (32 B each, read once for both z vectors), the z entries are 32-byte gathers.
#include <cuda_runtime.h>

#include "launch.cuh"
#include "r1cs_kernels.cuh"

namespace kgr {

template <class P> __global__ void __launch_bounds__(128) k_spmv(uint32_t m, Csr mat, const uint32_t *z, uint32_t *out) {
    body_spmv<P>(blockIdx.x * blockDim.x + threadIdx.x, m, mat, z, out);
}
template <class P> __global__ void __launch_bounds__(128) k_cross_term(uint32_t m, Csr a, Csr b, Csr c, const uint32_t *z1, const uint32_t *z2, uint32_t *t) {
    body_cross_term<P>(blockIdx.x * blockDim.x + threadIdx.x, m, a, b, c, z1, z2, t);
}
// result[0] += rows violating the relation, result[1] = min(violating row), one atomic of each per warp with a violation; strict: result[2] =
// (z[0] == 1).  The grid has at least one block, so row 0's thread exists also for m == 0.
template <class P>
__global__ void __launch_bounds__(128) k_relaxed_check(uint32_t m, Csr a, Csr b, Csr c, const uint32_t *z, const uint32_t *e, bool strict, uint32_t *result) {
    const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
    const uint32_t bad = __ballot_sync(0xFFFFFFFFu, body_relaxed_row<P>(i, m, a, b, c, z, e, strict));
    if ((threadIdx.x & 31) == 0 && bad) {
        atomicAdd(&result[0], (uint32_t)__popc(bad));
        atomicMin(&result[1], i + (uint32_t)__ffs(bad) - 1);
    }
    if (strict && i == 0) result[2] = fp_eq(ld_elem<P>(z, 0), fp_one<P>()) ? 1u : 0u;
}
template <class P> __global__ void __launch_bounds__(256) k_vec_fold(uint32_t n, const uint32_t *a, const uint32_t *b, Fp<P> r, uint32_t *out) {
    body_vec_fold<P>(blockIdx.x * blockDim.x + threadIdx.x, n, a, b, r, out);
}

__global__ void __launch_bounds__(128) k_r1cs_evaluate(uint32_t k, uint32_t m, Csr a, Csr b, Csr c, const uint32_t *z, uint32_t *out_a, uint32_t *out_b,
                                                        uint32_t *out_c) {
    body_r1cs_evaluate<FrP>(blockIdx.x * blockDim.x + threadIdx.x, k, m, a, b, c, z, out_a, out_b, out_c);
}

static inline unsigned blocks_for(size_t n, unsigned tpb) { return (unsigned)((n + tpb - 1) / tpb); }

void LaunchR1cs::evaluate(cudaStream_t st, uint32_t k, uint32_t m, const Csr &a, const Csr &b, const Csr &c, const uint32_t *z, uint32_t *const out[3]) {
    k_r1cs_evaluate<<<blocks_for((size_t)1 << k, 128), 128, 0, st>>>(k, m, a, b, c, z, out[0], out[1], out[2]);
}

void LaunchR1cs::spmv(cudaStream_t st, int field, uint32_t m, const Csr &mat, const uint32_t *z, uint32_t *out) {
    if (!m) return;
    if (field == 0) k_spmv<FqP><<<blocks_for(m, 128), 128, 0, st>>>(m, mat, z, out);
    else k_spmv<FrP><<<blocks_for(m, 128), 128, 0, st>>>(m, mat, z, out);
}
void LaunchR1cs::cross_term(cudaStream_t st, int field, uint32_t m, const Csr &a, const Csr &b, const Csr &c, const uint32_t *z1, const uint32_t *z2, uint32_t *t) {
    if (!m) return;
    if (field == 0) k_cross_term<FqP><<<blocks_for(m, 128), 128, 0, st>>>(m, a, b, c, z1, z2, t);
    else k_cross_term<FrP><<<blocks_for(m, 128), 128, 0, st>>>(m, a, b, c, z1, z2, t);
}
void LaunchR1cs::relaxed_check(cudaStream_t st, int field, uint32_t m, const Csr &a, const Csr &b, const Csr &c, const uint32_t *z, const uint32_t *e,
                               bool strict, uint32_t *result) {
    const unsigned blocks = blocks_for(m ? m : 1, 128);
    if (field == 0) k_relaxed_check<FqP><<<blocks, 128, 0, st>>>(m, a, b, c, z, e, strict, result);
    else k_relaxed_check<FrP><<<blocks, 128, 0, st>>>(m, a, b, c, z, e, strict, result);
}
void LaunchR1cs::vec_fold(cudaStream_t st, int field, uint32_t n, const uint32_t *a, const uint32_t *b, const uint32_t r8[8], uint32_t *out) {
    if (!n) return;
    if (field == 0) {
        Fp<FqP> r;
        for (int i = 0; i < 8; i++) r.v[i] = r8[i];
        k_vec_fold<FqP><<<blocks_for(n, 256), 256, 0, st>>>(n, a, b, r, out);
    } else {
        Fp<FrP> r;
        for (int i = 0; i < 8; i++) r.v[i] = r8[i];
        k_vec_fold<FrP><<<blocks_for(n, 256), 256, 0, st>>>(n, a, b, r, out);
    }
}

}  // namespace kgr
