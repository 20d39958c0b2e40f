// setup_kernels.cuh — per-thread bodies of the Groth16 parameter generation (groth16/src/zksnark.rs:17-127), host + device.
//
// The setup needs, per variable j of z = x ++ w, u_j = sum_i A[i][j] * l_i with l_i = L_i(tau) (and v_j, w_j from B and C): a transposed
// sparse product, while the shape is stored as CSR by rows.  The column sums run in passes of bounded work per thread:
//   1. count the entries of every column (atomics), exclusive scan -> col_ptr;
//   2. scatter: each entry writes coeff * l_row to a free slot of its column (the slot order depends on the atomics; field addition is exact,
//      so no sum depends on it);
//   3. while a column may hold more than COL_SEG values: every run of COL_SEG values of a column becomes one partial sum (one thread each);
//   4. one thread per column adds its last <= COL_SEG values.
// A column can hold every row (the constant one in B of most circuits), so no thread ever walks a whole column.
// All values are fully reduced Montgomery residues, so every result is bit-identical to the reference's.
#pragma once
#include "r1cs_kernels.cuh"

namespace kgr {

constexpr uint32_t COL_SEG = 32;  // values one thread adds in a pass of the column sums

// passes of step 3 for a matrix whose longest column has at most max_len entries
inline uint32_t col_sum_levels(size_t max_len) {
    uint32_t levels = 0;
    while (max_len > COL_SEG) {
        max_len = (max_len + COL_SEG - 1) / COL_SEG;
        levels++;
    }
    return levels;
}

KGR_HD uint32_t kgr_atomic_add(uint32_t *p, uint32_t v) {
#ifdef __CUDA_ARCH__
    return atomicAdd(p, v);
#else
    uint32_t old = *p;
    *p = old + v;
    return old;
#endif
}
KGR_HD uint32_t kgr_atomic_sub(uint32_t *p, uint32_t v) {
#ifdef __CUDA_ARCH__
    return atomicSub(p, v);
#else
    uint32_t old = *p;
    *p = old - v;
    return old;
#endif
}

// the index r of the last ptr[r] <= x over ptr[0..len] (non-decreasing, ptr[0] <= x): the row of entry x in CSR, the column of a segment
KGR_HD uint32_t seg_of(const uint32_t *ptr, uint32_t len, uint32_t x) {
    uint32_t lo = 0, hi = len;  // ptr[lo] <= x < ptr[hi] (ptr[len] is treated as +inf)
    while (hi - lo > 1) {
        uint32_t mid = lo + (hi - lo) / 2;
        if (ptr[mid] <= x) lo = mid;
        else hi = mid;
    }
    return lo;
}

// tau^i for i < n from tau^j (j < 2^log_t, lo) and tau^(2^log_t * b) (hi): one product per element.  The first n_h powers also go to h.
template <class P> KGR_HD void body_tau_powers(uint32_t i, uint32_t n, uint32_t log_t, const uint32_t *lo, const uint32_t *hi, uint32_t *out, uint32_t n_h,
                                               uint32_t *h) {
    if (i >= n) return;
    Fp<P> x = fp_mul(ld_elem<P>(hi, i >> log_t), ld_elem<P>(lo, i & ((1u << log_t) - 1)));
    el_store(out + 8 * (size_t)i, x);
    if (i < n_h) el_store(h + 8 * (size_t)i, x);
}

// step 1: cnt[col] += 1 per entry (cnt: n_z + 1 words, zero on entry)
KGR_HD void body_col_count(uint32_t e, uint32_t nnz, const uint32_t *cols, uint32_t *cnt) {
    if (e >= nnz) return;
    kgr_atomic_add(cnt + cols[e], 1);
}

// step 2: vals[col_ptr[col] + slot] = coeff * lagr[row]; cnt holds the counts of step 1 and is left zero
template <class P> KGR_HD void body_col_scatter(uint32_t e, uint32_t nnz, uint32_t m, const Csr &mat, const uint32_t *lagr, const uint32_t *col_ptr,
                                                uint32_t *cnt, uint32_t *vals) {
    if (e >= nnz) return;
    const uint32_t row = seg_of(mat.row_ptr, m, e), col = mat.cols[e];
    const Fp<P> c = ld_elem<P>(mat.coeffs, e), l = ld_elem<P>(lagr, row);
    const uint32_t pos = col_ptr[col] + kgr_atomic_sub(cnt + col, 1) - 1;
    el_store(vals + 8 * (size_t)pos, fp_eq(c, fp_one<P>()) ? l : fp_mul(c, l));
}

// step 3, count: column c gets ceil(len / COL_SEG) partial sums (cnt[n_z] = 0 for the scan's total)
KGR_HD void body_seg_count(uint32_t c, uint32_t n_z, const uint32_t *ptr, uint32_t *cnt) {
    if (c > n_z) return;
    cnt[c] = c == n_z ? 0 : (ptr[c + 1] - ptr[c] + COL_SEG - 1) / COL_SEG;
}

template <class P> KGR_HD Fp<P> sum_range(const uint32_t *vals, uint32_t first, uint32_t end) {
    Fp<P> acc = fp_zero<P>();
    for (uint32_t j = first; j < end; j++) acc = fp_add(acc, ld_elem<P>(vals, j));
    return acc;
}

// step 3, sum: partial sum s of column c = the values [ptr[c] + COL_SEG * (s - out_ptr[c]), + COL_SEG) of that column
template <class P> KGR_HD void body_seg_sum(uint32_t s, uint32_t n_z, const uint32_t *ptr, const uint32_t *vals, const uint32_t *out_ptr, uint32_t *out) {
    if (s >= out_ptr[n_z]) return;
    const uint32_t c = seg_of(out_ptr, n_z, s);
    const uint32_t first = ptr[c] + COL_SEG * (s - out_ptr[c]), end = ptr[c + 1] < first + COL_SEG ? ptr[c + 1] : first + COL_SEG;
    el_store(out + 8 * (size_t)s, sum_range<P>(vals, first, end));
}

// step 4: out[c] = the sum of the (at most COL_SEG) values of column c, zero for an empty column
template <class P> KGR_HD void body_col_final(uint32_t c, uint32_t n_z, const uint32_t *ptr, const uint32_t *vals, uint32_t *out) {
    if (c >= n_z) return;
    el_store(out + 8 * (size_t)c, sum_range<P>(vals, ptr[c], ptr[c + 1]));
}

// The scalars of zksnark.rs:62-87 that are not u or v themselves (a_j = u_j, b_j = v_j):
//   ext[j] = (beta u_j + alpha v_j + w_j) / gamma for j < n_inputs (ic), / delta otherwise (l = ext[n_inputs ..]);
//   h[i] *= (tau^n - 1) / delta for i < n_h (h holds tau^i on entry, zksnark.rs:51-57).
template <class P> struct SetupConsts {
    Fp<P> alpha, beta, gamma_inv, delta_inv, h_coeff;
};
template <class P> KGR_HD void body_setup_scalars(uint32_t i, uint32_t n_z, uint32_t n_inputs, uint32_t n_h, const SetupConsts<P> &k, const uint32_t *u,
                                                  const uint32_t *v, const uint32_t *w, uint32_t *ext, uint32_t *h) {
    if (i < n_z) {
        Fp<P> t = fp_add(fp_add(fp_mul(k.beta, ld_elem<P>(u, i)), fp_mul(k.alpha, ld_elem<P>(v, i))), ld_elem<P>(w, i));
        el_store(ext + 8 * (size_t)i, fp_mul(t, i < n_inputs ? k.gamma_inv : k.delta_inv));
    }
    if (i < n_h) el_store(h + 8 * (size_t)i, fp_mul(ld_elem<P>(h, i), k.h_coeff));
}

}  // namespace kgr
