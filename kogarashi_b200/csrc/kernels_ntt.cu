// kernels_ntt.cu — radix-2 NTT over bn254 Fr on the device (SURVEY.md §8f row N2).
//
// Replaces groth16/src/fft.rs:92-218 (dft / idft / coset variants: bit-reversal + recursive DIT butterflies,
// `butterfly_arithmetic` :195-218) for the prover's seven transforms (groth16/src/prover.rs:36-47).  A transform is
//   bit-reversal permutation, then ceil(k / 10) passes; a pass keeps a tile of 2^s elements in shared memory
//   (word-major, conflict-free) and runs s butterfly stages on it: t = b * w; b = a - t; a = a + t.
// Tiles of pass p are the index sets { hi | j << (p*s) | lo }, so every global access is one full 32-byte sector.
// Field elements are fully reduced Montgomery residues, hence the result is bit-identical to the reference's
// regardless of the butterfly schedule.  The kernel is bound by the integer multiplier (one 254-bit product per
// butterfly, n/2 * k products), not by HBM: 64 B moved per 10 products.
#include <cuda_runtime.h>

#include "launch.cuh"

namespace kgr {

typedef Fp<FrP> Fr;

__device__ __forceinline__ Fr ld_fr(const Fr *p) {
    const uint4 *q = reinterpret_cast<const uint4 *>(p);
    uint4 a = q[0], b = q[1];
    Fr r;
    r.v[0] = a.x; r.v[1] = a.y; r.v[2] = a.z; r.v[3] = a.w;
    r.v[4] = b.x; r.v[5] = b.y; r.v[6] = b.z; r.v[7] = b.w;
    return r;
}
__device__ __forceinline__ void st_fr(Fr *p, const Fr &r) {
    uint4 *q = reinterpret_cast<uint4 *>(p);
    q[0] = make_uint4(r.v[0], r.v[1], r.v[2], r.v[3]);
    q[1] = make_uint4(r.v[4], r.v[5], r.v[6], r.v[7]);
}

// fft.rs:157-162 prepare_fft: swap (i, reverse(i)) for i < reverse(i)
__global__ void k_ntt_bitrev(Fr *d, uint32_t k) {
    uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= (1u << k)) return;
    uint32_t r = __brev(i) >> (32 - k);
    if (i < r) {
        Fr a = ld_fr(d + i), b = ld_fr(d + r);
        st_fr(d + i, b);
        st_fr(d + r, a);
    }
}

// One pass: stages p_shift+1 .. p_shift+s of a size-2^k transform.  Each thread owns one butterfly per stage.
// tiles_per_block * 2^(s-1) threads per block; shared memory: tiles_per_block * 2^s elements, word-major per tile.
__global__ void k_ntt_pass(Fr *d, const Fr *__restrict__ tw, uint32_t k, uint32_t p_shift, uint32_t s) {
    extern __shared__ uint32_t sm[];
    const uint32_t T = 1u << s, half_t = T >> 1;
    const uint32_t b = blockIdx.x * blockDim.x + threadIdx.x;  // global butterfly slot
    const uint32_t tile = b >> (s - 1), tid = b & (half_t - 1);
    const uint32_t tile_in_block = threadIdx.x >> (s - 1);
    uint32_t *tsm = sm + tile_in_block * (8 * T);
    const uint32_t lo = tile & ((1u << p_shift) - 1), hi = tile >> p_shift;
    const size_t base = ((size_t)hi << (p_shift + s)) | lo;
    {
        Fr x0 = ld_fr(d + (base | ((size_t)tid << p_shift)));
        Fr x1 = ld_fr(d + (base | ((size_t)(tid + half_t) << p_shift)));
#pragma unroll
        for (int l = 0; l < 8; l++) {
            tsm[l * T + tid] = x0.v[l];
            tsm[l * T + tid + half_t] = x1.v[l];
        }
    }
    __syncthreads();
    for (uint32_t u = 1; u <= s; u++) {
        const uint32_t half = 1u << (u - 1);
        const uint32_t r = tid & (half - 1);
        const uint32_t j = ((tid >> (u - 1)) << u) | r;
        // twiddle of global stage t = p_shift + u for the butterfly whose lower index has low bits (r << p_shift | lo)
        const uint32_t e = ((r << p_shift) | lo) << (k - (p_shift + u));
        Fr a, bb;
#pragma unroll
        for (int l = 0; l < 8; l++) {
            a.v[l] = tsm[l * T + j];
            bb.v[l] = tsm[l * T + j + half];
        }
        Fr t = e ? fp_mul(bb, ld_fr(tw + e)) : bb;  // twiddle 1 for e == 0 (fft.rs:201-205)
        Fr hi_v = fp_sub(a, t), lo_v = fp_add(a, t);
#pragma unroll
        for (int l = 0; l < 8; l++) {
            tsm[l * T + j] = lo_v.v[l];
            tsm[l * T + j + half] = hi_v.v[l];
        }
        __syncthreads();
    }
    {
        Fr x0, x1;
#pragma unroll
        for (int l = 0; l < 8; l++) {
            x0.v[l] = tsm[l * T + tid];
            x1.v[l] = tsm[l * T + tid + half_t];
        }
        st_fr(d + (base | ((size_t)tid << p_shift)), x0);
        st_fr(d + (base | ((size_t)(tid + half_t) << p_shift)), x1);
    }
}

// d[i] *= table[i]  (coset shift, fft.rs:110-116 / 121-126), optionally also by a constant (n^-1, fft.rs:104)
__global__ void k_ntt_scale(Fr *d, const Fr *__restrict__ table, Fr c, int use_c, uint32_t n) {
    uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    Fr x = ld_fr(d + i);
    if (table) x = fp_mul(x, ld_fr(table + i));
    if (use_c) x = fp_mul(x, c);
    st_fr(d + i, x);
}

// out[i] = base^i  (twiddle and coset tables, fft.rs:36-67)
__global__ void k_pow_table(Fr *out, Fr base, uint32_t n) {
    uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    Fr acc = fp_one<FrP>();
    for (int bit = 31 - __clz(i | 1); bit >= 0; bit--) {
        acc = fp_sqr(acc);
        if ((i >> bit) & 1) acc = fp_mul(acc, base);
    }
    st_fr(out + i, acc);
}

// a[i] = (a[i] * b[i] - c[i]) * zinv   (prover.rs:43-46 with divide_by_z_on_coset, fft.rs:149-153)
__global__ void k_h_pointwise(Fr *a, const Fr *__restrict__ b, const Fr *__restrict__ c, Fr zinv, uint32_t n) {
    uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    Fr x = fp_sub(fp_mul(ld_fr(a + i), ld_fr(b + i)), ld_fr(c + i));
    st_fr(a + i, fp_mul(x, zinv));
}

static inline unsigned cdivu(size_t a, unsigned b) { return (unsigned)((a + b - 1) / b); }

int LaunchNtt::passes(uint32_t k) { return k == 0 ? 0 : (int)((k + 9) / 10); }

void LaunchNtt::pow_table(cudaStream_t st, void *out, const void *base32, uint32_t n) {
    Fr b;
    memcpy(&b, base32, 32);
    k_pow_table<<<cdivu(n, 128), 128, 0, st>>>((Fr *)out, b, n);
}
void LaunchNtt::scale(cudaStream_t st, void *d, const void *table, const void *c32, uint32_t n) {
    Fr c = fp_one<FrP>();
    if (c32) memcpy(&c, c32, 32);
    k_ntt_scale<<<cdivu(n, 128), 128, 0, st>>>((Fr *)d, (const Fr *)table, c, c32 != nullptr, n);
}
void LaunchNtt::h_pointwise(cudaStream_t st, void *a, const void *b, const void *c, const void *zinv32, uint32_t n) {
    Fr z;
    memcpy(&z, zinv32, 32);
    k_h_pointwise<<<cdivu(n, 128), 128, 0, st>>>((Fr *)a, (const Fr *)b, (const Fr *)c, z, n);
}
// In-place transform with the given twiddle table (forward or inverse): bit reversal + passes.  Returns kernels launched.
int LaunchNtt::transform(cudaStream_t st, void *d, const void *tw, uint32_t k) {
    if (k == 0) return 0;
    k_ntt_bitrev<<<cdivu((size_t)1 << k, 256), 256, 0, st>>>((Fr *)d, k);
    return 1 + transform_bitrev_input(st, d, tw, k);
}
int LaunchNtt::transform_bitrev_input(cudaStream_t st, void *d, const void *tw, uint32_t k) {
    if (k == 0) return 0;
    const uint32_t n = 1u << k;
    int launches = 0;
    const uint32_t np = (k + 9) / 10;
    uint32_t done = 0;
    for (uint32_t p = 0; p < np; p++) {
        uint32_t s = (k - done + (np - p) - 1) / (np - p);  // spread the stages evenly over the passes
        uint32_t half_t = 1u << (s - 1);
        uint32_t threads = half_t > 256 ? half_t : 256;
        if (threads > n / 2) threads = n / 2;
        uint32_t tiles_per_block = threads / half_t;
        size_t smem = (size_t)tiles_per_block * 8 * (1u << s) * sizeof(uint32_t);
        k_ntt_pass<<<(n / 2) / threads, threads, smem, st>>>((Fr *)d, (const Fr *)tw, k, done, s);
        done += s;
        launches++;
    }
    return launches;
}

}  // namespace kgr
