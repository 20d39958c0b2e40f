// pairing.cuh — the BN254 optimal-ate pairing over the Fq / Fq2 of field.cuh: the Fq6 / Fq12 tower, line functions of the D-type twist,
// the Miller loop (lines on the fly or from a precomputed table) and the final exponentiation to exactly (p^12 - 1) / r.
//
// Tower (the zkcrypto / arkworks layout, bn254/src/fqn.rs):  Fq6 = Fq2[v] / (v^3 - xi), xi = 9 + u;  Fq12 = Fq6[w] / (w^2 - v).  So w^6 = xi
// and the twist E': y^2 = x^3 + 3/xi untwists by (x, y) -> (x w^2, y w^3).  A line through twist points evaluated at an affine G1 point P
// is, up to a factor in Fq2 that the final exponentiation removes,  c0 yP + c1 xP w + c2 v w  (the sparse "034" form).
//
// Every function is KGR_HD: the host emulation (tests/host_emu_pairing.cpp) compiles this header with g++.  With KGR_FP2_CALLS on the
// device the Fq2 products (field.cuh) and the Fq6 products below are __noinline__ calls: an inlined Fq12 Miller loop does not fit the
// instruction cache (profiles/r01_g2.md).
#pragma once
#include "curve.cuh"
#include "modinv.cuh"

namespace kgr {

typedef Fp<FqP> Fq;
typedef Fp2<FqP> Fq2;
struct Fq6 {
    Fq2 c0, c1, c2;
};
struct Fq12 {
    Fq6 c0, c1;
};

// ---- constants (Montgomery limbs; tests/test_host_pairing.py recomputes every one with Python's pow) --------------------------------------
struct PairingConsts {
    // FROB[k-1][e-1] = xi^(e (p^k - 1) / 6), k = 1..3, e = 1..5: Frob^k(c w^e) = c^(p^k) FROB[k-1][e-1] w^e.  The untwisted Frobenius of a
    // twist point uses e = 2 (x) and e = 3 (y): pi(Q) = (conj(x) FROB[0][1], conj(y) FROB[0][2]), pi^2(Q) = (x FROB[1][1], y FROB[1][2]) with
    // FROB[1][2] = -1.
    static KGR_HD Fq2 frob(int k, int e) {
        constexpr uint32_t F[3][5][2][8] = {
            {{{0x33144907u, 0xaf9ba696u, 0x87afb78au, 0xca6b1d73u, 0xf08a2087u, 0x11bded5eu, 0x1a1f3a7cu, 0x02f34d75u},
              {0x4c492d72u, 0xa222ae23u, 0x565de15bu, 0xd00f02a4u, 0x53dfc926u, 0xdc2ff3a2u, 0xb3899551u, 0x10a75716u}},
             {{0x4563ab30u, 0xb5773b10u, 0xa9aa6454u, 0x347f91c8u, 0x242e0991u, 0x7a007127u, 0x118214ecu, 0x1956bcd8u},
              {0xa0aa4757u, 0x6e849f1eu, 0x89f89141u, 0xaa1c7b6du, 0xfae0ca3au, 0xb6e713cdu, 0x4e82ebc3u, 0x26694fbbu}},
             {{0x2936b629u, 0xe4bbdd0cu, 0xe133bacbu, 0xbb30f162u, 0xf9645366u, 0x31a9d1b6u, 0xa500f8ddu, 0x253570beu},
              {0x5ffe77c7u, 0xa1d77ce4u, 0x7826d1dbu, 0x07affd11u, 0xbb7edc6bu, 0x6d16bd27u, 0x85defeccu, 0x2c872002u}},
             {{0x843abe92u, 0x7361d77fu, 0x273411fbu, 0xa5bb2bd3u, 0x4b3e2399u, 0x9c941f31u, 0xbb9fd3ecu, 0x15df9cddu},
              {0x4bd8c949u, 0x5dddfd15u, 0xa4445b60u, 0x62cb29a5u, 0x0c7dd2b9u, 0x37bc870au, 0x3171f0fdu, 0x24830a9du}},
             {{0x41690fe7u, 0xc970692fu, 0x27694b0bu, 0xe2403421u, 0x83c459e8u, 0x32bee66bu, 0x0ab08841u, 0x12aabcedu},
              {0x40aebfa9u, 0x0d485d23u, 0xab2fcc57u, 0x05193418u, 0x8a4910f5u, 0xd3b0a40bu, 0x35d2925au, 0x2f21ebb5u}}},
            {{{0x00fa1bf2u, 0xca8d8005u, 0x68b39769u, 0xf0c5d614u, 0xad0d4418u, 0x0e201271u, 0xbad856e6u, 0x04290f65u}, {0, 0, 0, 0, 0, 0, 0, 0}},
             {{0x13e80b9cu, 0x3350c88eu, 0xdb5e56b9u, 0x7dce557cu, 0xb615564au, 0x6001b4b8u, 0x020217e0u, 0x2682e617u}, {0, 0, 0, 0, 0, 0, 0, 0}},
             {{0x12edefaau, 0x68c34889u, 0x72aabf4fu, 0x8d087f68u, 0x09081231u, 0x51e1a247u, 0x4729c0fau, 0x2259d6b1u}, {0, 0, 0, 0, 0, 0, 0, 0}},
             {{0xd782e155u, 0x71930c11u, 0xffbe3323u, 0xa6bb947cu, 0xd4741444u, 0xaa303344u, 0x26594943u, 0x2c3b3f0du}, {0, 0, 0, 0, 0, 0, 0, 0}},
             {{0xc494f1abu, 0x08cfc388u, 0x8d1373d4u, 0x19b31514u, 0xcb6c0213u, 0x584e90fdu, 0xdf2f8849u, 0x09e1685bu}, {0, 0, 0, 0, 0, 0, 0, 0}}},
            {{{0x4e46d97du, 0x36531618u, 0xd4c96d9fu, 0x0af7129eu, 0xca1009b5u, 0x659da72fu, 0x83a20d23u, 0x08116d89u},
              {0xc39c1939u, 0xb1df4af7u, 0x8a73bf7fu, 0x3d9f0287u, 0x8caf0ae0u, 0x9b222092u, 0xeff054a6u, 0x26684515u}},
             {{0x16ad6badu, 0xc9af22f7u, 0x4aa662b2u, 0xb311782au, 0xe248c7f4u, 0x19eeaf64u, 0xe3439f82u, 0x20273e77u},
              {0xf7ce93acu, 0xacc02860u, 0x7ba76b4cu, 0x3933d581u, 0x446c8467u, 0x69e6188bu, 0x4417cc55u, 0x0a46036du}},
             {{0xaf46471eu, 0x5764af0au, 0x873e0fc1u, 0xdc50792eu, 0x881d04f6u, 0x86a673ffu, 0x3c30a74cu, 0x0b2eddb4u},
              {0x787e8580u, 0x9a490f32u, 0xf04af8b1u, 0x8fd16d7fu, 0xc6027bf2u, 0x4b39888eu, 0x5b52a15du, 0x03dd2e70u}},
             {{0x7b6762dfu, 0x448a93a5u, 0x28fdeadfu, 0xbfd62df5u, 0x0e9bd47au, 0xd858f5d0u, 0x3476ec58u, 0x06b03d4du},
              {0xbcc936d1u, 0x2b19daf4u, 0x56f4299fu, 0xa1a54e7au, 0x5adeaef1u, 0xb533eee0u, 0x84dda0b2u, 0x170c812bu}},
             {{0x75cf559fu, 0xe0bc4b22u, 0xc154e60fu, 0xc238b945u, 0x929a7d5eu, 0x803982a5u, 0xf7e4a37eu, 0x15ce052du},
              {0xbf3799a7u, 0x2d28efbdu, 0x1ad60773u, 0x9b097e3cu, 0xaf4a535bu, 0x982d4113u, 0xe3056063u, 0x24e18991u}}}};
        Fq2 r;
#pragma unroll
        for (int i = 0; i < 8; i++) {
            r.c0.v[i] = F[k - 1][e - 1][0][i];
            r.c1.v[i] = F[k - 1][e - 1][1][i];
        }
        return r;
    }
    // b' = 3 / xi, the twist's constant (bn254/src/params.rs:44-57), and 3 b'
    static KGR_HD Fq2 twist_b() {
        constexpr uint32_t B[2][8] = {{0x77b802a8u, 0x3bf938e3u, 0x3633535du, 0x020b1b27u, 0x49755260u, 0x26b7edf0u, 0x4384a86du, 0x2514c632u},
                                      {0xd1dcff67u, 0x38e7ecccu, 0x93ce0d3eu, 0x65f0b37du, 0x22ac00aau, 0xd749d0ddu, 0x4a688d4du, 0x0141b9ceu}};
        Fq2 r;
#pragma unroll
        for (int i = 0; i < 8; i++) r.c0.v[i] = B[0][i], r.c1.v[i] = B[1][i];
        return r;
    }
    static KGR_HD Fq2 twist_b3() {
        constexpr uint32_t B[2][8] = {{0xb62e0d6au, 0x3baa927cu, 0xd1b664fdu, 0xd71e7c52u, 0xd95d4664u, 0x03873e63u, 0x082ab8f4u, 0x0e75b5b1u},
                                      {0x7596fe35u, 0xaab7c666u, 0xbb6a27bau, 0x31d21a78u, 0x680401ffu, 0x85dd7297u, 0xdf39a7e9u, 0x03c52d6au}};
        Fq2 r;
#pragma unroll
        for (int i = 0; i < 8; i++) r.c0.v[i] = B[0][i], r.c1.v[i] = B[1][i];
        return r;
    }
};

// The BN parameter u = 4965661367192848881 (63 bits) and the optimal-ate loop length 6u + 2 = 0x1_9d797039be763ba8 (65 bits, binary: 64
// doublings and 36 additions), then the two additions with pi(Q) and -pi^2(Q).
constexpr uint64_t BN_U = 0x44e992b44a6909f1ull;
constexpr uint64_t ATE_LO = 0x9d797039be763ba8ull;  // 6u + 2 without its top bit (bit 64)
constexpr int ATE_DOUBLINGS = 64;
constexpr int ATE_ADDITIONS = 36;  // popcount(6u + 2) - 1
constexpr int MILLER_LINES = ATE_DOUBLINGS + ATE_ADDITIONS + 2;

// ---- Fq2 helpers ------------------------------------------------------------------------------------------------------------------------
KGR_HD Fq2 fq2_conj(const Fq2 &a) { return Fq2{a.c0, fp_neg(a.c1)}; }
KGR_HD Fq2 fq2_mul_fq(const Fq2 &a, const Fq &s) { return Fq2{fp_mul(a.c0, s), fp_mul(a.c1, s)}; }
// a (9 + u) = (9 a0 - a1) + (a0 + 9 a1) u
KGR_HD Fq2 fq2_mul_xi(const Fq2 &a) {
    Fq2 a8 = fp_dbl(fp_dbl(fp_dbl(a)));
    Fq2 a9 = fp_add(a8, a);
    return Fq2{fp_sub(a9.c0, a.c1), fp_add(a9.c1, a.c0)};
}
KGR_HD Fq2 fq2_zero() { return El<Fq2>::zero(); }
KGR_HD Fq2 fq2_one() { return El<Fq2>::one(); }

// ---- Fq6 --------------------------------------------------------------------------------------------------------------------------------
KGR_HD Fq6 fq6_zero() { return Fq6{fq2_zero(), fq2_zero(), fq2_zero()}; }
KGR_HD Fq6 fq6_one() { return Fq6{fq2_one(), fq2_zero(), fq2_zero()}; }
KGR_HD Fq6 fq6_add(const Fq6 &a, const Fq6 &b) { return Fq6{fp_add(a.c0, b.c0), fp_add(a.c1, b.c1), fp_add(a.c2, b.c2)}; }
KGR_HD Fq6 fq6_sub(const Fq6 &a, const Fq6 &b) { return Fq6{fp_sub(a.c0, b.c0), fp_sub(a.c1, b.c1), fp_sub(a.c2, b.c2)}; }
KGR_HD Fq6 fq6_neg(const Fq6 &a) { return Fq6{fp_neg(a.c0), fp_neg(a.c1), fp_neg(a.c2)}; }
KGR_HD Fq6 fq6_dbl(const Fq6 &a) { return Fq6{fp_dbl(a.c0), fp_dbl(a.c1), fp_dbl(a.c2)}; }
// a v = (xi a2, a0, a1)
KGR_HD Fq6 fq6_mul_v(const Fq6 &a) { return Fq6{fq2_mul_xi(a.c2), a.c0, a.c1}; }
KGR_HD Fq6 fq6_mul_fq2(const Fq6 &a, const Fq2 &s) { return Fq6{fp_mul(a.c0, s), fp_mul(a.c1, s), fp_mul(a.c2, s)}; }
KGR_HD bool fq6_eq(const Fq6 &a, const Fq6 &b) { return fp_eq(a.c0, b.c0) && fp_eq(a.c1, b.c1) && fp_eq(a.c2, b.c2); }

// Karatsuba: 6 Fq2 products
KGR_HD Fq6 fq6_mul_inline(const Fq6 &a, const Fq6 &b) {
    Fq2 t0 = fp_mul(a.c0, b.c0), t1 = fp_mul(a.c1, b.c1), t2 = fp_mul(a.c2, b.c2);
    Fq2 c0 = fp_add(fq2_mul_xi(fp_sub(fp_sub(fp_mul(fp_add(a.c1, a.c2), fp_add(b.c1, b.c2)), t1), t2)), t0);
    Fq2 c1 = fp_add(fp_sub(fp_sub(fp_mul(fp_add(a.c0, a.c1), fp_add(b.c0, b.c1)), t0), t1), fq2_mul_xi(t2));
    Fq2 c2 = fp_add(fp_sub(fp_sub(fp_mul(fp_add(a.c0, a.c2), fp_add(b.c0, b.c2)), t0), t2), t1);
    return Fq6{c0, c1, c2};
}
// Chung-Hasan SQR2: 2 Fq2 products and 3 squares
KGR_HD Fq6 fq6_sqr_inline(const Fq6 &a) {
    Fq2 s0 = fp_sqr(a.c0);
    Fq2 s1 = fp_dbl(fp_mul(a.c0, a.c1));
    Fq2 s2 = fp_sqr(fp_add(fp_sub(a.c0, a.c1), a.c2));
    Fq2 s3 = fp_dbl(fp_mul(a.c1, a.c2));
    Fq2 s4 = fp_sqr(a.c2);
    return Fq6{fp_add(s0, fq2_mul_xi(s3)), fp_add(s1, fq2_mul_xi(s4)), fp_sub(fp_sub(fp_add(fp_add(s1, s2), s3), s0), s4)};
}
// a (b0 + b1 v): 5 Fq2 products
KGR_HD Fq6 fq6_mul_01_inline(const Fq6 &a, const Fq2 &b0, const Fq2 &b1) {
    Fq2 aa = fp_mul(a.c0, b0), bb = fp_mul(a.c1, b1);
    Fq2 c0 = fp_add(fq2_mul_xi(fp_mul(a.c2, b1)), aa);
    Fq2 c1 = fp_sub(fp_sub(fp_mul(fp_add(a.c0, a.c1), fp_add(b0, b1)), aa), bb);
    Fq2 c2 = fp_add(fp_sub(fp_mul(fp_add(a.c0, a.c2), b0), aa), bb);
    return Fq6{c0, c1, c2};
}
#if defined(__CUDA_ARCH__) && defined(KGR_FP2_CALLS)
__device__ __noinline__ Fq6 fq6_mul_call(Fq6 a, Fq6 b) { return fq6_mul_inline(a, b); }
__device__ __noinline__ Fq6 fq6_sqr_call(Fq6 a) { return fq6_sqr_inline(a); }
__device__ __noinline__ Fq6 fq6_mul_01_call(Fq6 a, Fq2 b0, Fq2 b1) { return fq6_mul_01_inline(a, b0, b1); }
KGR_HD Fq6 fq6_mul(const Fq6 &a, const Fq6 &b) { return fq6_mul_call(a, b); }
KGR_HD Fq6 fq6_sqr(const Fq6 &a) { return fq6_sqr_call(a); }
KGR_HD Fq6 fq6_mul_01(const Fq6 &a, const Fq2 &b0, const Fq2 &b1) { return fq6_mul_01_call(a, b0, b1); }
#else
KGR_HD Fq6 fq6_mul(const Fq6 &a, const Fq6 &b) { return fq6_mul_inline(a, b); }
KGR_HD Fq6 fq6_sqr(const Fq6 &a) { return fq6_sqr_inline(a); }
KGR_HD Fq6 fq6_mul_01(const Fq6 &a, const Fq2 &b0, const Fq2 &b1) { return fq6_mul_01_inline(a, b0, b1); }
#endif

// 1/a down the tower to one Fq inversion (fp_inv_fast, safegcd); zero maps to zero
KGR_HD Fq6 fq6_inv(const Fq6 &a) {
    Fq2 t0 = fp_sub(fp_sqr(a.c0), fq2_mul_xi(fp_mul(a.c1, a.c2)));
    Fq2 t1 = fp_sub(fq2_mul_xi(fp_sqr(a.c2)), fp_mul(a.c0, a.c1));
    Fq2 t2 = fp_sub(fp_sqr(a.c1), fp_mul(a.c0, a.c2));
    Fq2 d = fp_add(fp_mul(a.c0, t0), fq2_mul_xi(fp_add(fp_mul(a.c2, t1), fp_mul(a.c1, t2))));
    Fq2 di = fp_inv_fast(d);
    return Fq6{fp_mul(t0, di), fp_mul(t1, di), fp_mul(t2, di)};
}

// ---- Fq12 -------------------------------------------------------------------------------------------------------------------------------
KGR_HD Fq12 fq12_one() { return Fq12{fq6_one(), fq6_zero()}; }
KGR_HD bool fq12_eq(const Fq12 &a, const Fq12 &b) { return fq6_eq(a.c0, b.c0) && fq6_eq(a.c1, b.c1); }
KGR_HD bool fq12_is_one(const Fq12 &a) { return fq12_eq(a, fq12_one()); }
KGR_HD Fq12 fq12_conj(const Fq12 &a) { return Fq12{a.c0, fq6_neg(a.c1)}; }
// Karatsuba over Fq6: 3 Fq6 products
KGR_HD Fq12 fq12_mul(const Fq12 &a, const Fq12 &b) {
    Fq6 t0 = fq6_mul(a.c0, b.c0), t1 = fq6_mul(a.c1, b.c1);
    Fq6 c1 = fq6_sub(fq6_sub(fq6_mul(fq6_add(a.c0, a.c1), fq6_add(b.c0, b.c1)), t0), t1);
    return Fq12{fq6_add(t0, fq6_mul_v(t1)), c1};
}
// complex squaring: 2 Fq6 products
KGR_HD Fq12 fq12_sqr(const Fq12 &a) {
    Fq6 ab = fq6_mul(a.c0, a.c1);
    Fq6 c0 = fq6_sub(fq6_sub(fq6_mul(fq6_add(a.c0, a.c1), fq6_add(a.c0, fq6_mul_v(a.c1))), ab), fq6_mul_v(ab));
    return Fq12{c0, fq6_dbl(ab)};
}
// (a0 - a1 w) / (a0^2 - v a1^2)
KGR_HD Fq12 fq12_inv(const Fq12 &a) {
    Fq6 d = fq6_inv(fq6_sub(fq6_sqr(a.c0), fq6_mul_v(fq6_sqr(a.c1))));
    return Fq12{fq6_mul(a.c0, d), fq6_neg(fq6_mul(a.c1, d))};
}
// Frob^k, k = 1, 2, 3: coefficient c of w^e goes to c^(p^k) xi^(e (p^k - 1) / 6); c^(p^k) = conj(c) for odd k.  Coefficient (i, j) of the
// tower (Fq6 index i, Fq2 index j) multiplies w^(i + 2 j).
KGR_HD Fq12 fq12_frob(const Fq12 &a, int k) {
    auto f = [&](const Fq2 &c, int e) {
        Fq2 x = (k & 1) ? fq2_conj(c) : c;
        return e ? fp_mul(x, PairingConsts::frob(k, e)) : x;
    };
    return Fq12{Fq6{f(a.c0.c0, 0), f(a.c0.c1, 2), f(a.c0.c2, 4)}, Fq6{f(a.c1.c0, 1), f(a.c1.c1, 3), f(a.c1.c2, 5)}};
}
// f (l0 + l3 w + l4 v w): 13 Fq2 products instead of 18
KGR_HD Fq12 fq12_mul_034(const Fq12 &f, const Fq2 &l0, const Fq2 &l3, const Fq2 &l4) {
    Fq6 a = fq6_mul_fq2(f.c0, l0);
    Fq6 b = fq6_mul_01(f.c1, l3, l4);
    Fq6 e = fq6_mul_01(fq6_add(f.c0, f.c1), fp_add(l0, l3), l4);
    return Fq12{fq6_add(a, fq6_mul_v(b)), fq6_sub(fq6_sub(e, a), b)};
}
// Granger-Scott squaring in the cyclotomic subgroup (valid only after the easy part of the final exponentiation): three Fq4 squarings over
// the pairs (c0.c0, c1.c1), (c1.c0, c0.c2), (c0.c1, c1.c2) with Fq4 = Fq2[y] / (y^2 - xi).
KGR_HD void fq4_sqr(const Fq2 &a, const Fq2 &b, Fq2 &t0, Fq2 &t1) {  // (a + b y)^2 = t0 + t1 y
    Fq2 ab = fp_mul(a, b);
    t0 = fp_sub(fp_sub(fp_mul(fp_add(a, b), fp_add(fq2_mul_xi(b), a)), ab), fq2_mul_xi(ab));
    t1 = fp_dbl(ab);
}
KGR_HD Fq12 fq12_cyclotomic_sqr(const Fq12 &f) {
    Fq2 t0, t1, t2, t3, t4, t5;
    fq4_sqr(f.c0.c0, f.c1.c1, t0, t1);
    fq4_sqr(f.c1.c0, f.c0.c2, t2, t3);
    fq4_sqr(f.c0.c1, f.c1.c2, t4, t5);
    Fq12 r;
    auto three_minus_two = [](const Fq2 &t, const Fq2 &z) { return fp_add(fp_dbl(fp_sub(t, z)), t); };  // 3 t - 2 z
    auto three_plus_two = [](const Fq2 &t, const Fq2 &z) { return fp_add(fp_dbl(fp_add(t, z)), t); };   // 3 t + 2 z
    r.c0.c0 = three_minus_two(t0, f.c0.c0);
    r.c1.c1 = three_plus_two(t1, f.c1.c1);
    r.c1.c0 = three_plus_two(fq2_mul_xi(t5), f.c1.c0);
    r.c0.c2 = three_minus_two(t4, f.c0.c2);
    r.c0.c1 = three_minus_two(t2, f.c0.c1);
    r.c1.c2 = three_plus_two(t3, f.c1.c2);
    return r;
}

// ---- lines and the Miller loop ---------------------------------------------------------------------------------------------------------
struct G2Proj {  // homogeneous projective over Fq2: x = X / Z, y = Y / Z
    Fq2 x, y, z;
};
struct Line {  // c0 yP + c1 xP w + c2 v w
    Fq2 c0, c1, c2;
};
typedef AffinePt<Bn254G1> G1A;
typedef AffinePt<Bn254G2> G2A;

// T = 2T; the tangent at T scaled by -2YZ:  (-2YZ, 3X^2, 3b'Z^2 - Y^2)
KGR_HD Line dbl_step(G2Proj &t) {
    Fq2 a = fp_mul(t.x, t.y);  // X Y
    Fq2 b = fp_sqr(t.y);
    Fq2 c = fp_sqr(t.z);
    Fq2 e = fp_mul(c, PairingConsts::twist_b3());  // 3 b' Z^2
    Fq2 f = fp_add(fp_dbl(e), e);
    Fq2 h = fp_sub(fp_sqr(fp_add(t.y, t.z)), fp_add(b, c));  // 2 Y Z
    Fq2 j = fp_sqr(t.x);
    // (XY (b - f) / 2, ((b + f) / 2)^2 - 3 e^2, b h) scaled by 4 so that nothing is halved: the same point
    Fq2 e2 = fp_sqr(e);
    Fq2 bf = fp_add(b, f);
    t.x = fp_dbl(fp_mul(a, fp_sub(b, f)));
    t.y = fp_sub(fp_sqr(bf), fp_dbl(fp_dbl(fp_add(fp_dbl(e2), e2))));
    t.z = fp_dbl(fp_dbl(fp_mul(b, h)));
    return Line{fp_neg(h), fp_add(fp_dbl(j), j), fp_sub(e, b)};
}
// T = T + Q (Q affine, Q != +-T); the line through T and Q scaled by (X - x2 Z):  (X - x2 Z, -(Y - y2 Z), (Y - y2 Z) x2 - (X - x2 Z) y2)
KGR_HD Line add_step(G2Proj &t, const G2A &q) {
    Fq2 theta = fp_sub(t.y, fp_mul(q.y, t.z));
    Fq2 lambda = fp_sub(t.x, fp_mul(q.x, t.z));
    Fq2 c = fp_sqr(theta);
    Fq2 d = fp_sqr(lambda);
    Fq2 e = fp_mul(lambda, d);
    Fq2 f = fp_mul(t.z, c);
    Fq2 g = fp_mul(t.x, d);
    Fq2 h = fp_sub(fp_add(e, f), fp_dbl(g));
    Fq2 j = fp_sub(fp_mul(theta, q.x), fp_mul(lambda, q.y));
    t.x = fp_mul(lambda, h);
    t.y = fp_sub(fp_mul(theta, fp_sub(g, h)), fp_mul(e, t.y));
    t.z = fp_mul(t.z, e);
    return Line{lambda, fp_neg(theta), j};
}
// pi(Q) and -pi^2(Q) of the untwisted point, back on the twist
KGR_HD G2A frob_q1(const G2A &q) {
    G2A r;
    r.x = fp_mul(fq2_conj(q.x), PairingConsts::frob(1, 2));
    r.y = fp_mul(fq2_conj(q.y), PairingConsts::frob(1, 3));
    return r;
}
KGR_HD G2A frob_neg_q2(const G2A &q) {  // y pi^2 = -y: the negation cancels
    G2A r;
    r.x = fp_mul(q.x, PairingConsts::frob(2, 2));
    r.y = q.y;
    return r;
}
KGR_HD Fq12 line_eval(const Fq12 &f, const Line &l, const G1A &p) {
    return fq12_mul_034(f, fq2_mul_fq(l.c0, p.y), fq2_mul_fq(l.c1, p.x), l.c2);
}

// Writes the MILLER_LINES lines of Q in the order the Miller loop consumes them (per bit: the doubling, then the addition if the bit is set;
// then pi(Q), -pi^2(Q)).  Q must not be the identity.
template <class Sink> KGR_HD void miller_lines(const G2A &q, Sink &&sink) {
    G2Proj t{q.x, q.y, fq2_one()};
    int s = 0;
    for (int i = ATE_DOUBLINGS - 1; i >= 0; i--) {
        sink(s++, dbl_step(t));
        if ((ATE_LO >> i) & 1) sink(s++, add_step(t, q));
    }
    sink(s++, add_step(t, frob_q1(q)));
    sink(s++, add_step(t, frob_neg_q2(q)));
}

// Multi-Miller loop: at most one pair (p_fly, q_fly) with lines on the fly (use_fly) and n_tab pairs (p_tab[j], lines tab[j]) read from
// precomputed tables of MILLER_LINES lines each.  One squaring of f per iteration is shared by all pairs.  Identity inputs are the caller's
// to drop (a pair with P = O or Q = O contributes 1).
template <class TabRead>
KGR_HD Fq12 miller_multi(bool use_fly, const G1A &p_fly, const G2A &q_fly, int n_tab, const G1A *p_tab, TabRead &&tab) {
    Fq12 f = fq12_one();
    G2Proj t{q_fly.x, q_fly.y, fq2_one()};
    int s = 0;
    for (int i = ATE_DOUBLINGS - 1; i >= 0; i--) {
        if (i != ATE_DOUBLINGS - 1) f = fq12_sqr(f);
        if (use_fly) f = line_eval(f, dbl_step(t), p_fly);
        for (int j = 0; j < n_tab; j++) f = line_eval(f, tab(j, s), p_tab[j]);
        s++;
        if ((ATE_LO >> i) & 1) {
            if (use_fly) f = line_eval(f, add_step(t, q_fly), p_fly);
            for (int j = 0; j < n_tab; j++) f = line_eval(f, tab(j, s), p_tab[j]);
            s++;
        }
    }
    if (use_fly) f = line_eval(f, add_step(t, frob_q1(q_fly)), p_fly);
    for (int j = 0; j < n_tab; j++) f = line_eval(f, tab(j, s), p_tab[j]);
    s++;
    if (use_fly) f = line_eval(f, add_step(t, frob_neg_q2(q_fly)), p_fly);
    for (int j = 0; j < n_tab; j++) f = line_eval(f, tab(j, s), p_tab[j]);
    return f;
}
KGR_HD Fq12 miller_one(const G1A &p, const G2A &q) {
    if (affine_is_identity(p) || affine_is_identity(q)) return fq12_one();
    return miller_multi(true, p, q, 0, (const G1A *)nullptr, [](int, int) { return Line{}; });
}

// ---- final exponentiation to exactly (p^12 - 1) / r ------------------------------------------------------------------------------------
// a^u for a in the cyclotomic subgroup
KGR_HD Fq12 cyclotomic_exp_u(const Fq12 &a) {
    Fq12 r = a;
    for (int i = 61; i >= 0; i--) {
        r = fq12_cyclotomic_sqr(r);
        if ((BN_U >> i) & 1) r = fq12_mul(r, a);
    }
    return r;
}
// Easy part f^((p^6 - 1)(p^2 + 1)); hard part (p^4 - p^2 + 1) / r by the vectorial addition chain of Scott et al. (ePrint 2008/490), which
// computes that exponent exactly (three exponentiations by u).  Zero maps to zero.
KGR_HD Fq12 final_exp(const Fq12 &f) {
    Fq12 t = fq12_mul(fq12_conj(f), fq12_inv(f));
    t = fq12_mul(fq12_frob(t, 2), t);
    Fq12 fp1 = fq12_frob(t, 1), fp2 = fq12_frob(t, 2), fp3 = fq12_frob(fp2, 1);
    Fq12 fu = cyclotomic_exp_u(t), fu2 = cyclotomic_exp_u(fu), fu3 = cyclotomic_exp_u(fu2);
    Fq12 y3 = fq12_conj(fq12_frob(fu, 1));
    Fq12 fu2p = fq12_frob(fu2, 1), fu3p = fq12_frob(fu3, 1);
    Fq12 y2 = fq12_frob(fu2, 2);
    Fq12 y0 = fq12_mul(fq12_mul(fp1, fp2), fp3);
    Fq12 y1 = fq12_conj(t);
    Fq12 y5 = fq12_conj(fu2);
    Fq12 y4 = fq12_conj(fq12_mul(fu, fu2p));
    Fq12 y6 = fq12_conj(fq12_mul(fu3, fu3p));
    Fq12 t0 = fq12_mul(fq12_mul(fq12_cyclotomic_sqr(y6), y4), y5);
    Fq12 t1 = fq12_mul(fq12_mul(y3, y5), t0);
    t0 = fq12_mul(t0, y2);
    t1 = fq12_cyclotomic_sqr(fq12_mul(fq12_cyclotomic_sqr(t1), t0));
    t0 = fq12_mul(t1, y1);
    t1 = fq12_mul(t1, y0);
    t0 = fq12_cyclotomic_sqr(t0);
    return fq12_mul(t0, t1);
}

// ---- point validation ------------------------------------------------------------------------------------------------------------------
// words < p (as stored, before any arithmetic)
KGR_HD bool fq_canonical(const Fq &a) {
    for (int i = 7; i >= 0; i--)
        if (a.v[i] != FqP::mod(i)) return a.v[i] < FqP::mod(i);
    return false;
}
KGR_HD bool g1_on_curve(const G1A &p) {  // y^2 = x^3 + 3
    Fq one = fp_one<FqP>();
    Fq three = fp_add(fp_dbl(one), one);
    return fp_eq(fp_sqr(p.y), fp_add(fp_mul(fp_sqr(p.x), p.x), three));
}
KGR_HD bool g2_on_twist(const G2A &q) {  // y^2 = x^3 + 3 / xi
    return fp_eq(fp_sqr(q.y), fp_add(fp_mul(fp_sqr(q.x), q.x), PairingConsts::twist_b()));
}
// [r] Q = O by double-and-add in XYZZ over Fq2 (curve.cuh): the twist has a cofactor of about 2^254, so being on it does not place Q in G2
KGR_HD bool g2_in_subgroup(const G2A &q) {
    XyzzPt<Bn254G2> acc = xyzz_from_affine(q);  // the top bit of r
    for (int i = 252; i >= 0; i--) {
        acc = xyzz_dbl(acc);
        if ((FrP::mod(i >> 5) >> (i & 31)) & 1) xyzz_madd(acc, q);
    }
    return xyzz_is_identity(acc);
}

// ---- kernel bodies (kernels_pairing.cu; tests/host_emu_pairing.cpp runs the same bodies on the host) -------------------------------------
// ABI points are 64-bit words: G1 x[4] y[4] is_infinity, G2 x.c0 x.c1 y.c0 y.c1 is_infinity, Montgomery Fq.  The flag means the identity
// whatever the coordinates say; the device's identity is (0, 0).
KGR_HD void words_to_fq(const uint64_t *w, Fq &a) {
    for (int k = 0; k < 4; k++) {
        a.v[2 * k] = (uint32_t)w[k];
        a.v[2 * k + 1] = (uint32_t)(w[k] >> 32);
    }
}
// false: a coordinate >= p, or off the curve
KGR_HD bool load_g1(const uint64_t *w, G1A &p) {
    p.x = fp_zero<FqP>();
    p.y = fp_zero<FqP>();
    if (w[8]) return true;
    G1A t;
    words_to_fq(w, t.x);
    words_to_fq(w + 4, t.y);
    if (!fq_canonical(t.x) || !fq_canonical(t.y) || !g1_on_curve(t)) return false;
    p = t;
    return true;
}
// false: a coordinate >= p, off the twist, or outside G2
KGR_HD bool load_g2(const uint64_t *w, G2A &q) {
    q.x = fq2_zero();
    q.y = fq2_zero();
    if (w[16]) return true;
    G2A t;
    words_to_fq(w, t.x.c0);
    words_to_fq(w + 4, t.x.c1);
    words_to_fq(w + 8, t.y.c0);
    words_to_fq(w + 12, t.y.c1);
    if (!fq_canonical(t.x.c0) || !fq_canonical(t.x.c1) || !fq_canonical(t.y.c0) || !fq_canonical(t.y.c1)) return false;
    if (!g2_on_twist(t) || !g2_in_subgroup(t)) return false;
    q = t;
    return true;
}
KGR_HD G1A g1_neg(const G1A &p) { return G1A{p.x, fp_neg(p.y)}; }
// XYZZ -> affine with one safegcd inversion; the identity -> (0, 0)
KGR_HD G1A g1_affine(const XyzzPt<Bn254G1> &p) {
    if (xyzz_is_identity(p)) return G1A{fp_zero<FqP>(), fp_zero<FqP>()};
    Fq t = fp_inv_fast(fp_mul(p.zz, p.zzz));
    return G1A{fp_mul(p.x, fp_mul(t, p.zzz)), fp_mul(p.y, fp_mul(t, p.zz))};
}
// [k] P for a 128-bit k (lo, hi) by double-and-add from the top bit
KGR_HD XyzzPt<Bn254G1> g1_mul_u128(const G1A &p, uint64_t lo, uint64_t hi) {
    XyzzPt<Bn254G1> acc = xyzz_identity<Bn254G1>();
    for (int i = 127; i >= 0; i--) {
        acc = xyzz_dbl(acc);
        if (((i >= 64 ? hi >> (i - 64) : lo >> i) & 1)) xyzz_madd(acc, p);
    }
    return acc;
}

// Proof i of k (35 words: A[9] B[17] C[9]): every point valid?  Writes the device forms (an invalid point as the identity) and, for the
// per-proof path, the public inputs (Montgomery Fr) converted to canonical integers for the Straus windows.
KGR_HD void body_validate_proof(uint32_t i, uint32_t k, const uint64_t *proofs, const uint64_t *inputs, uint32_t n_public, G1A *a, G2A *b, G1A *c,
                                uint8_t *valid, Fp<FrP> *inputs_canon) {
    if (i >= k) return;
    const uint64_t *w = proofs + 35 * (size_t)i;
    bool ok = load_g1(w, a[i]);
    ok = load_g2(w + 9, b[i]) && ok;
    ok = load_g1(w + 26, c[i]) && ok;
    valid[i] = ok;
    for (uint32_t j = 0; j < n_public; j++) {
        Fp<FrP> x;
        const uint64_t *xw = inputs + 4 * ((size_t)i * n_public + j);
        for (int q = 0; q < 4; q++) x.v[2 * q] = (uint32_t)xw[q], x.v[2 * q + 1] = (uint32_t)(xw[q] >> 32);
        inputs_canon[(size_t)i * n_public + j] = fp_from_mont(x);
    }
}

// The lines of fixed G2 point j (not the identity) into table[j * MILLER_LINES ...]
KGR_HD void body_pairing_lines(uint32_t j, uint32_t n, const G2A *q, Line *table) {
    if (j >= n) return;
    Line *t = table + (size_t)j * MILLER_LINES;
    miller_lines(q[j], [&](int s, const Line &l) { t[s] = l; });
}

// Straus over the ic points: table[j * 16 + d] = d ic_{j+1} (d < 16, affine); IC(x) = ic_0 + sum_j x_j ic_{j+1}, 4-bit windows whose doublings
// are shared by all ic points.
KGR_HD void body_ic_table(uint32_t j, uint32_t n_public, const G1A *ic, G1A *table) {
    if (j >= n_public) return;
    const G1A p = ic[j + 1];
    XyzzPt<Bn254G1> acc = xyzz_identity<Bn254G1>();
    table[16 * j] = G1A{fp_zero<FqP>(), fp_zero<FqP>()};
    for (int d = 1; d < 16; d++) {
        xyzz_madd(acc, p);
        table[16 * j + d] = g1_affine(acc);
    }
}
KGR_HD G1A ic_combination(const G1A &ic0, const G1A *table, const Fp<FrP> *x, uint32_t n_public) {
    XyzzPt<Bn254G1> acc = xyzz_from_affine(ic0);
    XyzzPt<Bn254G1> sum = xyzz_identity<Bn254G1>();
    for (int wnd = 63; wnd >= 0; wnd--) {
        for (int d = 0; d < 4; d++) sum = xyzz_dbl(sum);
        for (uint32_t j = 0; j < n_public; j++) {
            uint32_t nib = (x[j].v[wnd >> 3] >> (4 * (wnd & 7))) & 15u;
            if (nib) xyzz_madd(sum, table[16 * j + nib]);
        }
    }
    xyzz_add(acc, sum);
    return g1_affine(acc);
}

// The multi-Miller loop of one Groth16 check against the fixed points beta, gamma, delta (lines in `lines`, 3 x MILLER_LINES; bit j of
// `present`: fixed point j is not the identity):  e(A, B) e(-alpha, beta) e(-IC, gamma) e(-C, delta), unreduced.  g1_fixed holds the G1
// points that pair with beta, gamma, delta, already negated.
KGR_HD Fq12 miller_groth16(const G1A &a, const G2A &b, const G1A g1_fixed[3], const Line *lines, uint32_t present) {
    G1A p[3];
    int idx[3], n = 0;
    for (int j = 0; j < 3; j++)
        if (((present >> j) & 1) && !affine_is_identity(g1_fixed[j])) p[n] = g1_fixed[j], idx[n++] = j;
    const bool fly = !affine_is_identity(a) && !affine_is_identity(b);
    return miller_multi(fly, a, b, n, p, [&](int j, int s) { return lines[(size_t)idx[j] * MILLER_LINES + s]; });
}

}  // namespace kgr
