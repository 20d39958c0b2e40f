// tests/host_emu_nova_sat.cpp — runs body_relaxed_row (kogarashi_b200/csrc/r1cs_kernels.cuh, the per-row body of k_relaxed_check, compiled
// for the host with the emulated carry chains) on every row of an instance read from stdin and prints the violation flag of each row.
// stdin (whitespace-separated decimal): field m n_z strict has_e, then for A, B, C: row_ptr[m + 1], cols[nnz], coeffs[nnz x 4 limbs], then
// z[n_z x 4], then e[m x 4] if has_e.  All elements Montgomery.  stdout: "FLAGS " and one '0' / '1' per row; rows m .. m + 2 are called too
// and must report no violation.
#include <cstdio>
#include <cstdlib>
#include <iostream>
#include <vector>

#define KGR_HOST_EMULATE_CHAINS 1
#include "../kogarashi_b200/csrc/r1cs_kernels.cuh"

using namespace kgr;

template <class P> static int run(uint32_t m, uint32_t n_z, bool strict, bool has_e) {
    struct Mat {
        std::vector<uint32_t> row_ptr, cols;
        std::vector<uint64_t> coeffs;
    } mats[3];
    Csr csr[3];
    for (int k = 0; k < 3; k++) {
        Mat &mt = mats[k];
        mt.row_ptr.resize(m + 1);
        for (auto &x : mt.row_ptr) std::cin >> x;
        const uint32_t nnz = mt.row_ptr[m];
        mt.cols.resize(nnz + 1);
        mt.coeffs.resize(4 * (size_t)nnz + 4);
        for (uint32_t j = 0; j < nnz; j++) std::cin >> mt.cols[j];
        for (size_t j = 0; j < 4 * (size_t)nnz; j++) std::cin >> mt.coeffs[j];
        csr[k] = Csr{mt.row_ptr.data(), mt.cols.data(), reinterpret_cast<const uint32_t *>(mt.coeffs.data())};
    }
    std::vector<uint64_t> z(4 * (size_t)n_z), e(has_e ? 4 * (size_t)m + 4 : 0);
    for (auto &x : z) std::cin >> x;
    for (size_t j = 0; j < 4 * (size_t)m && has_e; j++) std::cin >> e[j];
    if (!std::cin) { fprintf(stderr, "short input\n"); return 2; }
    const uint32_t *zw = reinterpret_cast<const uint32_t *>(z.data()), *ew = has_e ? reinterpret_cast<const uint32_t *>(e.data()) : nullptr;
    std::string flags;
    for (uint32_t i = 0; i < m; i++) flags += body_relaxed_row<P>(i, m, csr[0], csr[1], csr[2], zw, ew, strict) ? '1' : '0';
    for (uint32_t i = m; i < m + 3; i++)
        if (body_relaxed_row<P>(i, m, csr[0], csr[1], csr[2], zw, ew, strict)) { fprintf(stderr, "row %u >= m reported\n", i); return 1; }
    printf("FLAGS %s\n", flags.c_str());
    return 0;
}

int main() {
    int field, strict, has_e;
    uint32_t m, n_z;
    if (!(std::cin >> field >> m >> n_z >> strict >> has_e)) { fprintf(stderr, "usage: host_emu_nova_sat < instance\n"); return 2; }
    return field == 0 ? run<FqP>(m, n_z, strict, has_e) : run<FrP>(m, n_z, strict, has_e);
}
