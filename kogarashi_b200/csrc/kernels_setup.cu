// kernels_setup.cu — the data-parallel steps of the Groth16 parameter generation (groth16/src/zksnark.rs:17-127) over bn254 Fr:
// powers of tau, the column sums of A, B and C against the Lagrange basis (setup_kernels.cuh), and the elementwise scalar formula.
// The Lagrange basis itself is an inverse NTT (kernels_ntt.cu) and the points are the fixed-base kernel of kernels_curve.cuh.
#include <cuda_runtime.h>

#include <algorithm>

#include "launch.cuh"
#include "setup_kernels.cuh"

namespace kgr {

__global__ void __launch_bounds__(256) k_tau_powers(uint32_t n, uint32_t log_t, const uint32_t *lo, const uint32_t *hi, uint32_t *out, uint32_t n_h,
                                                     uint32_t *h) {
    body_tau_powers<FrP>(blockIdx.x * blockDim.x + threadIdx.x, n, log_t, lo, hi, out, n_h, h);
}
__global__ void __launch_bounds__(256) k_col_count(uint32_t nnz, const uint32_t *cols, uint32_t *cnt) {
    body_col_count(blockIdx.x * blockDim.x + threadIdx.x, nnz, cols, cnt);
}
__global__ void __launch_bounds__(256) k_col_scatter(uint32_t nnz, uint32_t m, Csr mat, const uint32_t *lagr, const uint32_t *col_ptr, uint32_t *cnt,
                                                      uint32_t *vals) {
    body_col_scatter<FrP>(blockIdx.x * blockDim.x + threadIdx.x, nnz, m, mat, lagr, col_ptr, cnt, vals);
}
__global__ void __launch_bounds__(256) k_seg_count(uint32_t n_z, const uint32_t *ptr, uint32_t *cnt) {
    body_seg_count(blockIdx.x * blockDim.x + threadIdx.x, n_z, ptr, cnt);
}
__global__ void __launch_bounds__(256) k_seg_sum(uint32_t n_z, const uint32_t *ptr, const uint32_t *vals, const uint32_t *out_ptr, uint32_t *out) {
    body_seg_sum<FrP>(blockIdx.x * blockDim.x + threadIdx.x, n_z, ptr, vals, out_ptr, out);
}
__global__ void __launch_bounds__(256) k_col_final(uint32_t n_z, const uint32_t *ptr, const uint32_t *vals, uint32_t *out) {
    body_col_final<FrP>(blockIdx.x * blockDim.x + threadIdx.x, n_z, ptr, vals, out);
}
__global__ void __launch_bounds__(256) k_setup_scalars(uint32_t n_z, uint32_t n_inputs, uint32_t n_h, SetupConsts<FrP> k, const uint32_t *u,
                                                        const uint32_t *v, const uint32_t *w, uint32_t *ext, uint32_t *h) {
    body_setup_scalars<FrP>(blockIdx.x * blockDim.x + threadIdx.x, n_z, n_inputs, n_h, k, u, v, w, ext, h);
}

static inline unsigned blocks256(size_t n) { return (unsigned)((n + 255) / 256); }

int LaunchSetup::tau_powers(cudaStream_t st, uint32_t k, const void *lo, const void *hi, void *out, uint32_t n_h, void *h) {
    k_tau_powers<<<blocks256((size_t)1 << k), 256, 0, st>>>(1u << k, tau_log_t(k), (const uint32_t *)lo, (const uint32_t *)hi, (uint32_t *)out, n_h,
                                                                 (uint32_t *)h);
    return 1;
}

int LaunchSetup::column_sums(cudaStream_t st, uint32_t m, uint32_t n_z, const Csr &mat, uint32_t nnz, const void *lagr, uint32_t *cnt, uint32_t *const ptr[2],
                             void *const vals[2], uint32_t *tile_sums, void *out) {
    int launches = 0;
    if (nnz) {
        k_col_count<<<blocks256(nnz), 256, 0, st>>>(nnz, mat.cols, cnt);
        launches++;
    }
    LaunchUtil::exclusive_scan(st, cnt, ptr[0], n_z + 1, tile_sums);
    launches += LaunchUtil::scan_launches(n_z + 1);
    if (nnz) {
        k_col_scatter<<<blocks256(nnz), 256, 0, st>>>(nnz, m, mat, (const uint32_t *)lagr, ptr[0], cnt, (uint32_t *)vals[0]);
        launches++;
    }
    // values per column <= nnz; after each level a column of len values holds ceil(len / COL_SEG), and the level's total is at most
    // min(len_total, len_total / COL_SEG + n_z)
    int cur = 0;
    size_t total = nnz;
    for (uint32_t lv = col_sum_levels(nnz); lv; lv--) {
        k_seg_count<<<blocks256((size_t)n_z + 1), 256, 0, st>>>(n_z, ptr[cur], cnt);
        LaunchUtil::exclusive_scan(st, cnt, ptr[cur ^ 1], n_z + 1, tile_sums);
        total = std::min(total, total / COL_SEG + n_z);
        k_seg_sum<<<blocks256(total), 256, 0, st>>>(n_z, ptr[cur], (const uint32_t *)vals[cur], ptr[cur ^ 1], (uint32_t *)vals[cur ^ 1]);
        launches += 2 + LaunchUtil::scan_launches(n_z + 1);
        cur ^= 1;
    }
    k_col_final<<<blocks256(n_z), 256, 0, st>>>(n_z, ptr[cur], (const uint32_t *)vals[cur], (uint32_t *)out);
    return launches + 1;
}

int LaunchSetup::scalars(cudaStream_t st, uint32_t n_z, uint32_t n_inputs, uint32_t n_h, const void *consts, const void *u, const void *v, const void *w,
                         void *ext, void *h) {
    SetupConsts<FrP> k;
    memcpy(&k, consts, sizeof k);
    k_setup_scalars<<<blocks256(std::max(n_z, n_h)), 256, 0, st>>>(n_z, n_inputs, n_h, k, (const uint32_t *)u, (const uint32_t *)v, (const uint32_t *)w,
                                                                     (uint32_t *)ext, (uint32_t *)h);
    return 1;
}

}  // namespace kgr
