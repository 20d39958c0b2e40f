// tests/host_emu_pairing.cpp — runs the tower arithmetic, the Miller loop, the final exponentiation and the kernel bodies of
// kogarashi_b200/csrc/pairing.cuh on the host (g++, emulated carry chains); tests/test_host_pairing.py compares the results with the flat
// big-integer pairing of oracle/pairing_ref.py.
// usage: host_emu_pairing <op> <in> <out>; in and out are little-endian u64 words, field elements Montgomery, Fq12 as 48 words in tower order
//   fq6     n x (a[24], b[24])           -> n x (a b, a^2, 1/a)
//   fq12    n x (a[48], b[48])           -> n x (a b, a^2, 1/a, Frob(a), Frob^2(a), Frob^3(a))
//   cyc     n x a[48]                    -> n x (e = a^((p^6-1)(p^2+1)), cyclotomic square of e, e^2)
//   m034    n x (f[48], l0 l3 l4 [24])   -> n x f (l0 + l3 w + l4 v w)
//   fexp    n x f[48]                    -> n x final_exp(f)
//   pair    n x (g1[9], g2[17])          -> n x (valid, e(P, Q)[48])
//   consts  (nothing)                    -> FROB[3][5] (16 words each), b', 3b'
//   verify  n_public, k, vk_g1[3][9], vk_g2[3][17], ic[n_public + 1][9], proofs[k][35], inputs[k][n_public][4]  -> k verdicts
//           (the per-proof path of kgr_groth16_verify: validation, line tables, Straus for IC(x), multi-Miller, final exponentiation)
#include <cstdio>
#include <cstring>
#include <string>
#include <vector>

#define KGR_HOST_EMULATE_CHAINS 1
#include "../kogarashi_b200/csrc/pairing.cuh"

using namespace kgr;

template <class T> static T get(const uint64_t *&p) {
    T r;
    std::memcpy(&r, p, sizeof r);
    p += sizeof r / 8;
    return r;
}
template <class T> static void put(std::vector<uint64_t> &o, const T &v) {
    size_t at = o.size();
    o.resize(at + sizeof v / 8);
    std::memcpy(o.data() + at, &v, sizeof v);
}

int main(int argc, char **argv) {
    if (argc < 4) { fprintf(stderr, "usage: host_emu_pairing op in out\n"); return 2; }
    const std::string op = argv[1];
    std::vector<uint64_t> in;
    {
        FILE *f = fopen(argv[2], "rb");
        if (!f) { perror(argv[2]); return 2; }
        uint64_t w;
        while (fread(&w, 8, 1, f) == 1) in.push_back(w);
        fclose(f);
    }
    const uint64_t *p = in.data(), *end = in.data() + in.size();
    std::vector<uint64_t> out;
    if (op == "fq6") {
        while (p < end) {
            Fq6 a = get<Fq6>(p), b = get<Fq6>(p);
            put(out, fq6_mul(a, b)), put(out, fq6_sqr(a)), put(out, fq6_inv(a));
        }
    } else if (op == "fq12") {
        while (p < end) {
            Fq12 a = get<Fq12>(p), b = get<Fq12>(p);
            put(out, fq12_mul(a, b)), put(out, fq12_sqr(a)), put(out, fq12_inv(a));
            for (int k = 1; k <= 3; k++) put(out, fq12_frob(a, k));
        }
    } else if (op == "cyc") {
        while (p < end) {
            Fq12 a = get<Fq12>(p);
            Fq12 e = fq12_mul(fq12_conj(a), fq12_inv(a));
            e = fq12_mul(fq12_frob(e, 2), e);
            put(out, e), put(out, fq12_cyclotomic_sqr(e)), put(out, fq12_sqr(e));
        }
    } else if (op == "m034") {
        while (p < end) {
            Fq12 f = get<Fq12>(p);
            Fq2 l0 = get<Fq2>(p), l3 = get<Fq2>(p), l4 = get<Fq2>(p);
            put(out, fq12_mul_034(f, l0, l3, l4));
        }
    } else if (op == "fexp") {
        while (p < end) put(out, final_exp(get<Fq12>(p)));
    } else if (op == "pair") {
        while (p < end) {
            G1A a;
            G2A b;
            bool ok = load_g1(p, a);
            ok = load_g2(p + 9, b) && ok;
            p += 26;
            out.push_back(ok);
            put(out, final_exp(miller_one(a, b)));
        }
    } else if (op == "consts") {
        for (int k = 1; k <= 3; k++)
            for (int e = 1; e <= 5; e++) put(out, PairingConsts::frob(k, e));
        put(out, PairingConsts::twist_b()), put(out, PairingConsts::twist_b3());
    } else if (op == "verify") {
        const uint32_t n_public = (uint32_t)*p++, k = (uint32_t)*p++;
        G1A vk1[3];
        G2A vk2[3];
        for (int j = 0; j < 3; j++)
            if (!load_g1(p + 9 * j, vk1[j])) { fprintf(stderr, "bad vk_g1\n"); return 3; }
        p += 27;
        uint32_t present = 0;
        for (int j = 0; j < 3; j++) {
            if (!load_g2(p + 17 * j, vk2[j])) { fprintf(stderr, "bad vk_g2\n"); return 3; }
            if (!affine_is_identity(vk2[j])) present |= 1u << j;
        }
        p += 51;
        std::vector<G1A> ic(n_public + 1);
        for (uint32_t j = 0; j <= n_public; j++, p += 9)
            if (!load_g1(p, ic[j])) { fprintf(stderr, "bad ic\n"); return 3; }
        const uint64_t *proofs = p, *inputs = p + 35 * (size_t)k;
        std::vector<G1A> a(k), c(k), table(16 * (size_t)n_public + 1);
        std::vector<G2A> b(k);
        std::vector<uint8_t> valid(k);
        std::vector<Fp<FrP>> xs((size_t)k * n_public + 1);
        std::vector<Line> lines(3 * MILLER_LINES);
        for (uint32_t i = 0; i < k + 2; i++) body_validate_proof(i, k, proofs, inputs, n_public, a.data(), b.data(), c.data(), valid.data(), xs.data());
        for (uint32_t j = 0; j < 3; j++)
            if ((present >> j) & 1) body_pairing_lines(j, 3, vk2, lines.data());
        for (uint32_t j = 0; j < n_public + 1; j++) body_ic_table(j, n_public, ic.data(), table.data());
        for (uint32_t i = 0; i < k; i++) {
            G1A icx = ic_combination(ic[0], table.data(), xs.data() + (size_t)i * n_public, n_public);
            G1A fixed[3] = {g1_neg(vk1[0]), g1_neg(icx), g1_neg(c[i])};
            Fq12 f = miller_groth16(a[i], b[i], fixed, lines.data(), present);
            out.push_back(valid[i] && fq12_is_one(final_exp(f)));
        }
    } else {
        fprintf(stderr, "unknown op %s\n", op.c_str());
        return 2;
    }
    FILE *g = fopen(argv[3], "wb");
    if (!g) { perror(argv[3]); return 2; }
    fwrite(out.data(), 8, out.size(), g);
    fclose(g);
    return 0;
}
