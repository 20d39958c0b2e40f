// r1cs_kernels.cuh — per-row bodies of the Nova folding prover's vector work (SURVEY.md §8f row N4), host + device.
//
// Reference: zkstd/src/matrix.rs:36-48 `SparseMatrix::prod` (row i: sum of coeff * z[wire]), nova/src/prover.rs:53-90
// `compute_cross_term` (T = AZ1∘BZ2 + AZ2∘BZ1 − u1·CZ2 − u2·CZ1), nova/src/relaxed_r1cs/witness.rs:56-71 `fold`
// (e = e1 + t·r, w = w1 + w2·r).  Matrices are CSR with flat column indices into z = (u, x, w) — the caller resolves
// `Wire::Instance(i) -> i`, `Wire::Witness(i) -> i + l` (matrix.rs:41-44) once when it registers the shape.
// All values are fully reduced Montgomery residues, so every result is bit-identical to the reference's regardless of the
// summation schedule.
#pragma once
#include "field.cuh"

namespace kgr {

struct Csr {
    const uint32_t *row_ptr;   // m + 1
    const uint32_t *cols;      // nnz
    const uint32_t *coeffs;    // nnz x 8 words, Montgomery
};

template <class P> KGR_HD Fp<P> ld_elem(const uint32_t *base, size_t idx) {
    Fp<P> r;
    el_load(r, base + 8 * idx);
    return r;
}

// sum_j coeff_j * z[col_j] over row i for one or two vectors at once (coefficients are read once).
// R1CS coefficients are mostly 1: that product is skipped.
template <class P, int NZ> KGR_HD void row_dot(const Csr &mat, uint32_t i, const uint32_t *const z[NZ], Fp<P> out[NZ]) {
    for (int v = 0; v < NZ; v++) out[v] = fp_zero<P>();
    const Fp<P> one = fp_one<P>();
    for (uint32_t j = mat.row_ptr[i], end = mat.row_ptr[i + 1]; j < end; j++) {
        Fp<P> c = ld_elem<P>(mat.coeffs, j);
        uint32_t col = mat.cols[j];
        bool unit = fp_eq(c, one);
        for (int v = 0; v < NZ; v++) {
            Fp<P> x = ld_elem<P>(z[v], col);
            out[v] = fp_add(out[v], unit ? x : fp_mul(c, x));
        }
    }
}

// SparseMatrix::prod: out[i] = (M z)[i]
template <class P> KGR_HD void body_spmv(uint32_t i, uint32_t m, const Csr &mat, const uint32_t *z, uint32_t *out) {
    if (i >= m) return;
    const uint32_t *zs[1] = {z};
    Fp<P> r[1];
    row_dot<P, 1>(mat, i, zs, r);
    el_store(out + 8 * (size_t)i, r[0]);
}

// compute_cross_term, one row: all six products and the combination stay in registers; u1 = z1[0], u2 = z2[0].
template <class P> KGR_HD void body_cross_term(uint32_t i, uint32_t m, const Csr &a, const Csr &b, const Csr &c, const uint32_t *z1, const uint32_t *z2, uint32_t *t) {
    if (i >= m) return;
    const uint32_t *zs[2] = {z1, z2};
    Fp<P> az[2], bz[2], cz[2];
    row_dot<P, 2>(a, i, zs, az);
    row_dot<P, 2>(b, i, zs, bz);
    row_dot<P, 2>(c, i, zs, cz);
    Fp<P> u1 = ld_elem<P>(z1, 0), u2 = ld_elem<P>(z2, 0);
    Fp<P> r = fp_add(fp_mul(az[1], bz[0]), fp_mul(az[0], bz[1]));   // AZ2∘BZ1 + AZ1∘BZ2
    r = fp_sub(r, fp_mul(cz[1], u1));                               // − u1·CZ2
    r = fp_sub(r, fp_mul(cz[0], u2));                               // − u2·CZ1
    el_store(t + 8 * (size_t)i, r);
}

// R1csShape::is_sat_relaxed / is_sat, one row (nova/src/relaxed_r1cs.rs:80-146): true iff row i VIOLATES (A z)_i (B z)_i = u (C z)_i + E_i.
// u = z[0], or the constant one when strict (is_sat); e == nullptr: E = 0.  Rows i >= m never violate.
template <class P>
KGR_HD bool body_relaxed_row(uint32_t i, uint32_t m, const Csr &a, const Csr &b, const Csr &c, const uint32_t *z, const uint32_t *e, bool strict) {
    if (i >= m) return false;
    const uint32_t *zs[1] = {z};
    Fp<P> az, bz, cz;
    row_dot<P, 1>(a, i, zs, &az);
    row_dot<P, 1>(b, i, zs, &bz);
    row_dot<P, 1>(c, i, zs, &cz);
    Fp<P> rhs = strict ? cz : fp_mul(ld_elem<P>(z, 0), cz);
    if (e) rhs = fp_add(rhs, ld_elem<P>(e, i));
    return !fp_eq(fp_mul(az, bz), rhs);
}

// The k low bits of i reversed (fft.rs:157-162 swaps i and this index)
KGR_HD uint32_t bitrev_k(uint32_t i, uint32_t k) {
#ifdef __CUDA_ARCH__
    return __brev(i) >> (32 - k);
#else
    uint32_t r = 0;
    for (uint32_t b = 0; b < k; b++) r |= ((i >> b) & 1u) << (k - 1 - b);
    return r;
#endif
}

// cs.evaluate() (zkstd/src/r1cs.rs:137-142) straight into the three NTT buffers of the Groth16 H pipeline (groth16/src/prover.rs:36-41):
// position i < 2^k holds row i of A z, B z, C z (zero for m <= i, the padding of prepare_fft, fft.rs:157-162) and is stored at bitrev_k(i),
// so the first transform of each buffer starts with its butterflies.  k >= 1.
template <class P>
KGR_HD void body_r1cs_evaluate(uint32_t i, uint32_t k, uint32_t m, const Csr &a, const Csr &b, const Csr &c, const uint32_t *z, uint32_t *out_a,
                               uint32_t *out_b, uint32_t *out_c) {
    if (i >= (1u << k)) return;
    Fp<P> r[3] = {fp_zero<P>(), fp_zero<P>(), fp_zero<P>()};
    if (i < m) {
        const uint32_t *zs[1] = {z};
        row_dot<P, 1>(a, i, zs, &r[0]);
        row_dot<P, 1>(b, i, zs, &r[1]);
        row_dot<P, 1>(c, i, zs, &r[2]);
    }
    const size_t j = 8 * (size_t)bitrev_k(i, k);
    el_store(out_a + j, r[0]);
    el_store(out_b + j, r[1]);
    el_store(out_c + j, r[2]);
}

// out[i] = a[i] + b[i] * r   (witness.rs:67-68)
template <class P> KGR_HD void body_vec_fold(uint32_t i, uint32_t n, const uint32_t *a, const uint32_t *b, const Fp<P> &r, uint32_t *out) {
    if (i >= n) return;
    el_store(out + 8 * (size_t)i, fp_add(ld_elem<P>(a, i), fp_mul(ld_elem<P>(b, i), r)));
}

}  // namespace kgr
