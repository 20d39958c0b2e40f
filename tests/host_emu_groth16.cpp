// tests/host_emu_groth16.cpp — runs the per-position body of k_r1cs_evaluate (kogarashi_b200/csrc/r1cs_kernels.cuh, compiled for the host
// with the emulated carry chains) for every position of the domain and writes the three NTT buffers it fills; tests/test_host_groth16.py
// compares them with cs.evaluate() of oracle/groth16_ref.py, zero padded and permuted by bit reversal.
// usage: host_emu_groth16 <in> <out>
//   in:  u32 k, m, n_z; per matrix A, B, C: u32 row_ptr[m + 1], u32 cols[nnz], u64 coeffs[nnz][4] (Montgomery); u64 z[n_z][4] (Montgomery)
//   out: u64 a[2^k][4], b[2^k][4], c[2^k][4]
#include <cstdio>
#include <cstring>
#include <vector>

#define KGR_HOST_EMULATE_CHAINS 1
#include "../kogarashi_b200/csrc/r1cs_kernels.cuh"

using namespace kgr;

template <class T> static bool rd(FILE *f, std::vector<T> &v, size_t n) {
    v.resize(n ? n : 1);
    return fread(v.data(), sizeof(T), n, f) == n;
}

int main(int argc, char **argv) {
    if (argc < 3) { fprintf(stderr, "usage: host_emu_groth16 in out\n"); return 2; }
    FILE *f = fopen(argv[1], "rb");
    if (!f) { perror(argv[1]); return 2; }
    uint32_t hdr[3];
    if (fread(hdr, 4, 3, f) != 3) return 2;
    const uint32_t k = hdr[0], m = hdr[1], n_z = hdr[2];
    std::vector<uint32_t> row_ptr[3], cols[3];
    std::vector<uint64_t> coeffs[3], z;
    Csr mats[3];
    for (int i = 0; i < 3; i++) {
        if (!rd(f, row_ptr[i], m + 1)) return 2;
        const uint32_t nnz = row_ptr[i][m];
        if (!rd(f, cols[i], nnz) || !rd(f, coeffs[i], 4 * (size_t)nnz)) return 2;
        mats[i] = Csr{row_ptr[i].data(), cols[i].data(), reinterpret_cast<const uint32_t *>(coeffs[i].data())};
    }
    if (!rd(f, z, 4 * (size_t)n_z)) return 2;
    fclose(f);
    const size_t n = (size_t)1 << k;
    // stale contents the kernel must overwrite: the zero padding is written, not assumed
    std::vector<uint64_t> out[3];
    uint32_t *outw[3];
    for (int i = 0; i < 3; i++) {
        out[i].assign(4 * n, 0x5a5a5a5a5a5a5a5aULL);
        outw[i] = reinterpret_cast<uint32_t *>(out[i].data());
    }
    const uint32_t *zw = reinterpret_cast<const uint32_t *>(z.data());
    for (uint32_t i = 0; i < n + 3; i++)   // indices >= 2^k must be ignored
        body_r1cs_evaluate<FrP>(i, k, m, mats[0], mats[1], mats[2], zw, outw[0], outw[1], outw[2]);
    FILE *g = fopen(argv[2], "wb");
    if (!g) { perror(argv[2]); return 2; }
    for (int i = 0; i < 3; i++) fwrite(out[i].data(), 8, 4 * n, g);
    fclose(g);
    printf("OK k=%u m=%u n_z=%u\n", k, m, n_z);
    return 0;
}
