// Self-test kernels behind bbs_selftest_* (include/bbs_b200.h): they expose the field, G1 and pairing
// layers one level below the BBS operations so the parity tests can pin each layer against the oracle.
#pragma once
#include "kernels.cuh"

namespace bbs {

// op: the operation (low byte; list at bbs_selftest_field) | FIELD_TEST_MONT.  With FIELD_TEST_MONT the operands are taken as
// Montgomery words and the result is returned as one, so a chosen limb pattern reaches the multiplication chains as it is.
constexpr int FIELD_TEST_MONT = 0x100;
constexpr int FIELD_TEST_LAST_OP = 13;
BBS_HD bool field_test_on_fp(int op) { return op <= 4 || op == 7 || op == 9 || op == 10; }

struct FieldTestArgs { int op; const uint8_t* a; const uint8_t* b; uint8_t* out; };

// the operations both kinds of field have; false if op is not one of them
template <class F> BBS_HD bool field_test_common(int op, uint32_t* r, const uint32_t* a, const uint32_t* b) {
    if (op == 0 || op == 5) fe_mul<F>(r, a, b);
    else if (op == 1 || op == 11) fe_add<F>(r, a, b);
    else if (op == 2 || op == 12) fe_sub<F>(r, a, b);
    else if (op == 3 || op == 6) fe_inv<F>(r, a);
    else if (op == 7 || op == 8) fe_inv_vt<F>(r, a);
    else if (op == 10 || op == 13) fe_neg<F>(r, a);
    else return false;
    return true;
}

template <class C> BBS_HD void field_test_item(const FieldTestArgs& t, uint32_t i) {
    using Fp = typename C::Fp;
    using Fr = typename C::Fr;
    const int op = t.op & 0xff;
    const bool mont = (t.op & FIELD_TEST_MONT) != 0;
    if (field_test_on_fp(op)) {
        constexpr int N = Fp::N;
        BBS_A16 uint32_t a[N], b[N], r[N];
        limbs_from_le<N>(a, t.a + (size_t)i * 4 * N);
        limbs_from_le<N>(b, t.b + (size_t)i * 4 * N);
        if (!mont) { fe_to_mont<Fp>(a, a); fe_to_mont<Fp>(b, b); }
        if (!field_test_common<Fp>(op, r, a, b)) {
            if (op == 9) fe_sqr<Fp>(r, a);
            else if (!fe_sqrt<Fp>(r, a)) bn_zero<N>(r);
        }
        if (!mont) fe_from_mont<Fp>(r, r);
        limbs_to_le<N>(t.out + (size_t)i * 4 * N, r);
    } else {
        BBS_A16 uint32_t a[8], b[8], r[8];
        limbs_from_le<8>(a, t.a + (size_t)i * 32);
        limbs_from_le<8>(b, t.b + (size_t)i * 32);
        if (!mont) { fe_to_mont<Fr>(a, a); fe_to_mont<Fr>(b, b); }
        field_test_common<Fr>(op, r, a, b);
        if (!mont) fe_from_mont<Fr>(r, r);
        limbs_to_le<8>(t.out + (size_t)i * 32, r);
    }
}


struct G1MulTestArgs { const uint8_t* pts; const uint8_t* sc; uint8_t* out; };
template <class C> BBS_HD void g1_mul_test_item(const G1MulTestArgs& t, uint32_t i) {
    BBS_A16 uint32_t A[G1A], k[8], R[G1J];
    uint8_t* o = t.out + (size_t)i * C::G1_BYTES;
    int st = g1_decompress<C>(A, t.pts + (size_t)i * C::G1_BYTES);
    limbs_from_le<8>(k, t.sc + (size_t)i * 32);
    if (st == PT_BAD) { for (int j = 0; j < C::G1_BYTES; j++) o[j] = 0xff; return; }
    // canonical scalars take the production path (windowed GLV, g1_mul_scalar); others the plain double-and-add
    if (st == PT_INF) g1_set_inf<C>(R);
    else if (fe_is_canonical<typename C::Fr>(k)) g1_mul_scalar<C>(R, A, k);
    else g1_mul_affine<C>(R, A, k, 256);
    g1_compress<C>(o, R);
}

// The G1 group law (bbs_selftest_g1): one operation per item on Jacobian operands, so the test can reach the rare-case
// branches of the additions (P + P, P + (-P), identities) with one point under several Z.
enum : int { G1_TEST_ADD = 0, G1_TEST_ADD_MIXED = 1, G1_TEST_DBL = 2, G1_TEST_MSM2 = 3, G1_TEST_MSM3 = 4 };
constexpr int G1_TEST_LAST_OP = G1_TEST_MSM3;
BBS_HD int g1_test_points(int op) { return op == G1_TEST_MSM2 ? 2 : op == G1_TEST_MSM3 ? 3 : 1; }

struct G1TestArgs { int op; const uint8_t* p; const uint8_t* q; const uint8_t* sc; uint8_t* out; };
// canonical little-endian (X, Y, Z) -> Montgomery Jacobian
template <class C> BBS_HD void g1_test_load(uint32_t* r, const uint8_t* in) {
    for (int k = 0; k < 3; k++) {
        limbs_from_le<C::Fp::N>(r + k * FPN, in + k * 4 * C::Fp::N);
        fe_to_mont<typename C::Fp>(r + k * FPN, r + k * FPN);
    }
}
template <class C, int NP> BBS_HD void g1_test_msm(uint32_t* R, const uint8_t* p, const uint8_t* sc) {
    BBS_A16 uint32_t P[NP][G1J], k[NP][8];
    const uint32_t* pts[NP];
    const uint32_t* ks[NP];
    for (int j = 0; j < NP; j++) {
        g1_test_load<C>(P[j], p + (size_t)j * 12 * C::Fp::N);
        limbs_from_le<8>(k[j], sc + (size_t)j * 32);
        pts[j] = g1_is_inf<C>(P[j]) ? nullptr : P[j];       // affine (x, y): Z only marks the identity
        ks[j] = k[j];
    }
    g1_msm_scalar<C, NP>(R, pts, ks);
}
template <class C> BBS_HD void g1_test_item(const G1TestArgs& t, uint32_t i) {
    constexpr size_t PB = 12 * C::Fp::N;         // bytes of one Jacobian operand
    const int np = g1_test_points(t.op);
    const uint8_t* p = t.p + (size_t)i * np * PB;
    BBS_A16 uint32_t R[G1J];
    if (t.op == G1_TEST_MSM2) g1_test_msm<C, 2>(R, p, t.sc + (size_t)i * 2 * 32);
    else if (t.op == G1_TEST_MSM3) g1_test_msm<C, 3>(R, p, t.sc + (size_t)i * 3 * 32);
    else {
        BBS_A16 uint32_t P[G1J], Q[G1J];
        g1_test_load<C>(P, p);
        if (t.op == G1_TEST_DBL) g1_dbl<C>(R, P);
        else {
            g1_test_load<C>(Q, t.q + (size_t)i * PB);
            if (t.op == G1_TEST_ADD) g1_add<C>(R, P, Q); else g1_add_mixed<C>(R, P, Q);
        }
    }
    g1_compress<C>(t.out + (size_t)i * C::G1_BYTES, R);
}

struct PairTestPrepArgs { const uint8_t* q; uint32_t* W; uint32_t* lines; uint32_t* st; };
template <class C> BBS_HD void pair_test_prep_item(const PairTestPrepArgs& t, uint32_t i) {
    if (i == 0) {
        int s = g2_decompress<C>(t.W, t.q);
        t.st[0] = (uint32_t)s;
        if (s == PT_OK) g2_precompute_lines<C>(t.lines, t.W, 0);
    } else {
        g2_precompute_lines<C>(t.lines, C::G2(), 1);
    }
}
struct PairTestArgs { const uint8_t* p; const uint8_t* r; const uint32_t* lines; const uint32_t* st; uint8_t* status; };
template <class C> BBS_HD void pair_test_item(const PairTestArgs& t, uint32_t i) {
    BBS_A16 uint32_t P[G1A], R[G1A], a0[3 * FPN], a1[3 * FPN], f[F12N];
    int sp = g1_decompress<C>(P, t.p + (size_t)i * C::G1_BYTES);
    int sr = g1_decompress<C>(R, t.r + (size_t)i * C::G1_BYTES);
    if (sp == PT_BAD || sr == PT_BAD || t.st[0] == PT_BAD) { t.status[i] = ST_ERR_MALFORMED; return; }
    bn_copy<2 * C::Fp::N>(a0, P); fe_set_one<typename C::Fp>(a0 + 2 * FPN);
    bn_copy<2 * C::Fp::N>(a1, R); fe_set_one<typename C::Fp>(a1 + 2 * FPN);
    miller2<C>(f, t.lines, a0, sp == PT_INF || t.st[0] == PT_INF, a1, sr == PT_INF);
    t.status[i] = final_exp_is_one<C>(f) ? ST_ACCEPT : ST_REJECT;
}

}  // namespace bbs
