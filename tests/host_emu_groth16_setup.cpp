// tests/host_emu_groth16_setup.cpp — runs the bodies of the Groth16 setup kernels (kogarashi_b200/csrc/setup_kernels.cuh, compiled for the host
// with the emulated carry chains) in the order and with the pass structure LaunchSetup uses (kernels_setup.cu), one thread index after another;
// tests/test_host_groth16_setup.py compares the results with crs_exponents of oracle/groth16_ref.py.  The Lagrange basis (an inverse NTT on the
// device) is an input here.
// usage: host_emu_groth16_setup <in> <out>
//   in:  u32 k, m, n_z, n_inputs; per matrix A, B, C: u32 row_ptr[m + 1], u32 cols[nnz], u64 coeffs[nnz][4]; u64 toxic[5][4] (alpha, beta, gamma,
//        delta, tau); u64 lagr[2^k][4]  (all field elements Montgomery)
//   out: u64 powers[2^k][4], u[n_z][4], v[n_z][4], w[n_z][4], ext[n_z][4], h[m - 1][4]
#include <algorithm>
#include <cstdlib>
#include <cstdio>
#include <cstring>
#include <vector>

#define KGR_HOST_EMULATE_CHAINS 1
#include "../kogarashi_b200/csrc/setup_kernels.cuh"

using namespace kgr;
typedef Fp<FrP> Fr;

template <class T> static bool rd(FILE *f, std::vector<T> &v, size_t n) {
    v.resize(n ? n : 1);
    return fread(v.data(), sizeof(T), n, f) == n;
}
static Fr fr_at(const std::vector<uint64_t> &v, size_t i) {
    Fr r;
    std::memcpy(&r, v.data() + 4 * i, 32);
    return r;
}
static std::vector<uint32_t> exclusive_scan(const std::vector<uint32_t> &in) {
    std::vector<uint32_t> out(in.size());
    uint32_t acc = 0;
    for (size_t i = 0; i < in.size(); i++) out[i] = acc, acc += in[i];
    return out;
}
static uint32_t *w32(std::vector<uint64_t> &v) { return reinterpret_cast<uint32_t *>(v.data()); }

// LaunchSetup::column_sums, thread by thread; the scatter runs its entries backwards (the device's slot order is whatever the atomics give)
static void column_sums(uint32_t m, uint32_t n_z, const Csr &mat, uint32_t nnz, const uint32_t *lagr, uint32_t *out) {
    std::vector<uint32_t> cnt(n_z + 1, 0), ptr[2];
    std::vector<uint64_t> vals[2];
    vals[0].assign(4 * std::max(nnz, 1u), 0x5a5a5a5a5a5a5a5aULL);
    vals[1] = vals[0];
    for (uint32_t e = 0; e < nnz + 3; e++) body_col_count(e, nnz, mat.cols, cnt.data());
    ptr[0] = exclusive_scan(cnt);
    for (uint32_t e = nnz + 3; e-- > 0;) body_col_scatter<FrP>(e, nnz, m, mat, lagr, ptr[0].data(), cnt.data(), w32(vals[0]));
    for (uint32_t c = 0; c <= n_z; c++)
        if (cnt[c]) { fprintf(stderr, "scatter left cnt[%u] = %u\n", c, cnt[c]); exit(3); }
    int cur = 0;
    size_t total = nnz;
    for (uint32_t lv = col_sum_levels(nnz); lv; lv--) {
        for (uint32_t c = 0; c <= n_z + 2; c++) body_seg_count(c, n_z, ptr[cur].data(), cnt.data());
        ptr[cur ^ 1] = exclusive_scan(cnt);
        total = std::min(total, total / COL_SEG + n_z);
        if (ptr[cur ^ 1][n_z] > total) { fprintf(stderr, "level bound %zu < %u partial sums\n", total, ptr[cur ^ 1][n_z]); exit(3); }
        for (uint32_t s = 0; s < total + 3; s++) body_seg_sum<FrP>(s, n_z, ptr[cur].data(), w32(vals[cur]), ptr[cur ^ 1].data(), w32(vals[cur ^ 1]));
        cur ^= 1;
    }
    for (uint32_t c = 0; c < n_z; c++)
        if (ptr[cur][c + 1] - ptr[cur][c] > COL_SEG) { fprintf(stderr, "column %u keeps %u values\n", c, ptr[cur][c + 1] - ptr[cur][c]); exit(3); }
    for (uint32_t c = 0; c < n_z + 3; c++) body_col_final<FrP>(c, n_z, ptr[cur].data(), w32(vals[cur]), out);
}

int main(int argc, char **argv) {
    if (argc < 3) { fprintf(stderr, "usage: host_emu_groth16_setup in out\n"); return 2; }
    FILE *f = fopen(argv[1], "rb");
    if (!f) { perror(argv[1]); return 2; }
    uint32_t hdr[4];
    if (fread(hdr, 4, 4, f) != 4) return 2;
    const uint32_t k = hdr[0], m = hdr[1], n_z = hdr[2], n_inputs = hdr[3], n = 1u << k, n_h = m ? m - 1 : 0;
    std::vector<uint32_t> row_ptr[3], cols[3];
    std::vector<uint64_t> coeffs[3], toxic, lagr;
    Csr mats[3];
    for (int i = 0; i < 3; i++) {
        if (!rd(f, row_ptr[i], m + 1)) return 2;
        const uint32_t nnz = row_ptr[i][m];
        if (!rd(f, cols[i], nnz) || !rd(f, coeffs[i], 4 * (size_t)nnz)) return 2;
        mats[i] = Csr{row_ptr[i].data(), cols[i].data(), reinterpret_cast<const uint32_t *>(coeffs[i].data())};
    }
    if (!rd(f, toxic, 20) || !rd(f, lagr, 4 * (size_t)n)) return 2;
    fclose(f);
    const Fr tau = fr_at(toxic, 4);
    // the two power tables (pow_table on the device), then one product per power
    const uint32_t log_t = (k + 1) / 2;
    std::vector<uint64_t> lo(4 << log_t), hi(4 * (size_t)(n >> log_t)), powers(4 * (size_t)n, 0x5a5a5a5a5a5a5a5aULL), h(4 * std::max(n_h, 1u));
    Fr x = fp_one<FrP>(), tau_t = tau;
    for (uint32_t i = 0; i < log_t; i++) tau_t = fp_sqr(tau_t);
    for (uint32_t j = 0; j < (1u << log_t); j++, x = fp_mul(x, tau)) el_store(w32(lo) + 8 * j, x);
    x = fp_one<FrP>();
    for (uint32_t b = 0; b < (n >> log_t); b++, x = fp_mul(x, tau_t)) el_store(w32(hi) + 8 * b, x);
    for (uint32_t i = 0; i < n + 3; i++) body_tau_powers<FrP>(i, n, log_t, w32(lo), w32(hi), w32(powers), n_h, w32(h));
    std::vector<uint64_t> uvw[3], ext(4 * (size_t)n_z, 0x5a5a5a5a5a5a5a5aULL);
    for (int i = 0; i < 3; i++) {
        uvw[i].assign(4 * (size_t)n_z, 0x5a5a5a5a5a5a5a5aULL);
        column_sums(m, n_z, mats[i], row_ptr[i][m], w32(lagr), w32(uvw[i]));
    }
    Fr tau_n = tau;
    for (uint32_t i = 0; i < k; i++) tau_n = fp_sqr(tau_n);
    SetupConsts<FrP> consts{fr_at(toxic, 0), fr_at(toxic, 1), fp_inv(fr_at(toxic, 2)), fp_inv(fr_at(toxic, 3)), fp_zero<FrP>()};
    consts.h_coeff = fp_mul(fp_sub(tau_n, fp_one<FrP>()), consts.delta_inv);
    for (uint32_t i = 0; i < std::max(n_z, n_h) + 3; i++)
        body_setup_scalars<FrP>(i, n_z, n_inputs, n_h, consts, w32(uvw[0]), w32(uvw[1]), w32(uvw[2]), w32(ext), w32(h));
    FILE *g = fopen(argv[2], "wb");
    if (!g) { perror(argv[2]); return 2; }
    fwrite(powers.data(), 8, 4 * (size_t)n, g);
    for (int i = 0; i < 3; i++) fwrite(uvw[i].data(), 8, 4 * (size_t)n_z, g);
    fwrite(ext.data(), 8, 4 * (size_t)n_z, g);
    fwrite(h.data(), 8, 4 * (size_t)n_h, g);
    fclose(g);
    printf("OK k=%u m=%u n_z=%u\n", k, m, n_z);
    return 0;
}
