// Per-item bodies of every kernel on the path, written as plain functions of (args, item index) so the
// same source runs as a CUDA kernel (one thread per item; `launch.cuh`) and, in tests only, as a host
// loop (BBS_HOSTSIM) for GPU-less debugging.
//
//   ctx creation : ctx_decode_item, ctx_domain_item, ctx_table_item, ctx_lines_item
//   per-item hdr : item_domain_item                (calculate_domain + K per item, bbs_*_hdr calls)
//   hashing      : h2s_item                      (msg_to_scalars, interface_utilities.rs:76-88)
//   verify       : verify_g1_item -> pairing_item (core_verify, verify.rs:53-93)
//   sign         : sign_item                      (core_sign, sign.rs:63-133)
//   proof verify : proof_g1_item -> pairing_item  (core_proof_verify, proof_verify.rs:64-188)
#pragma once
#include "g2.cuh"
#include "sha256.cuh"
#include "h2c.cuh"

namespace bbs {

// per-item status bytes (include/bbs_b200.h)
enum : uint8_t {
    ST_REJECT = 0,            // Ok(false)
    ST_ACCEPT = 1,            // Ok(true)
    ST_ERR_MSG_GEN_LEN = 2,   // InvalidMessageAndGeneratorsLength (sign.rs:26, proof_gen.rs:66)
    ST_ERR_DISCLOSED_INDEX = 3,  // InvalidDisclosedIndex (proof_gen.rs:62-65)
    ST_ERR_IDX_MSG_LEN = 4,   // InvalidIndicesAndMessagesLength (proof_gen.rs:72-74)
    ST_ERR_MALFORMED = 5,     // undecodable point / non-canonical scalar / the reference's panic cases
    ST_ERR_DISCLOSED_LEN = 6, // InvalidDisclosedIndicesLength (proof_gen.rs:139-141)
    ST_ERR_RANDOM_LEN = 7,    // InvalidRandomScalarsAndUndisclosedIndicesLength (proof_gen.rs:232-234)
};

// Fixed-base tables: entry (g, w, d) = (d * 2^(BITS w)) * base_g in affine form, d = 1 .. 2^BITS - 1.
//   The scalar is split with the GLV endomorphism (g1.cuh: k = k1 + k2 lambda, both < 2^128) and BOTH halves use the same
//   table (phi of an entry is (beta x, y): one extra multiplication), so 16-bit windows need only 8 windows: 16 mixed
//   additions per generator from a 50 MB (BLS12-381) / 34 MB (BN254) table per generator, 96- / 64-byte gathers from HBM.
//   The host simulation (tests only) builds its tables on CPU cores and uses 8-bit windows.
//   A context may instead be built with SMALL tables (bbs_ctx_create_ex, BBS_CTX_SMALL_TABLES): 8-bit windows, 16 windows,
//   32 additions per generator from a 390 KB (BLS12-381) table per generator that stays resident in L2 -- 128 x less memory
//   and table-building work, for roughly twice the fixed-base additions.
#ifndef BBS_TAB_BITS_GLV
#ifdef BBS_HOSTSIM
#define BBS_TAB_BITS_GLV 8
#else
#define BBS_TAB_BITS_GLV 16
#endif
#endif
constexpr int TAB_BITS_SMALL = 8;
// geometry of a context's tables for a window width chosen at creation
struct TabGeom {
    int bits, windows;
    uint32_t entries;
    BBS_HD explicit TabGeom(uint32_t b) : bits((int)b), windows((128 + (int)b - 1) / (int)b), entries((1u << b) - 1u) {}
};
BBS_HD uint32_t tab_digit(const TabGeom& G, const uint32_t* s, int nlimbs, int w) {      // s: canonical limbs
    const int bit = w * G.bits, word = bit >> 5, off = bit & 31;
    uint64_t v = s[word];
    if (word + 1 < nlimbs) v |= (uint64_t)s[word + 1] << 32;
    return (uint32_t)(v >> off) & G.entries;
}
constexpr int MAX_L = 256;
// per-issuer flags of an issuer set (below): identity public key, identity K, unusable key
enum : uint32_t { ISS_W_INF = 1, ISS_K_INF = 2, ISS_BAD = 4 };

// Read-only per-issuer state living in device memory (built once by bbs_ctx_create)
struct CtxView {
    uint32_t L;               // message generators H_1..H_L
    uint32_t w_inf;           // public key is the identity
    uint32_t k_inf;           // K = P1 + Q1*domain is the identity
    uint32_t tab_bits;        // window width of `tab` (16, or 8 for small tables)
    uint32_t dst_h2s_len, dst_map_len;
    const uint8_t* dst_h2s;   // api_id || "H2S_"
    const uint8_t* dst_map;   // api_id || "MAP_MSG_TO_SCALAR_AS_HASH_"
    const uint32_t* gens;     // (L+1) affine points: Q1, H_1..H_L
    const uint32_t* W;        // affine G2 public key
    const uint32_t* K;        // affine K
    const uint32_t* domain;   // canonical limbs (8)
    const uint32_t* tab;      // fixed-base tables: generator index g in [0, L] (0 = K, j = H_j)
    const uint32_t* lines;    // line table for (W, BP2)
};

// ---- ctx creation ----------------------------------------------------------------------------------
struct CtxDecodeArgs {
    const uint8_t* gens_comp; const uint8_t* pk_comp; uint32_t n_gens;
    uint32_t* gens; uint32_t* W; uint32_t* status;   // status[j]: PT_* per generator, status[n_gens]: pk
};
template <class C> BBS_HD void ctx_decode_item(const CtxDecodeArgs& a, uint32_t i) {
    if (i < a.n_gens) a.status[i] = g1_decompress<C>(a.gens + i * G1A, a.gens_comp + i * C::G1_BYTES);
    else a.status[i] = g2_decompress<C>(a.W, a.pk_comp);
}

struct CtxDomainArgs {
    const uint8_t* pk_comp; const uint8_t* gens_comp; uint32_t L;
    const uint8_t* api_id; uint32_t api_id_len; const uint8_t* header; uint32_t header_len;
    const uint8_t* dst_h2s; uint32_t dst_h2s_len;
    const uint32_t* gens; uint32_t* domain; uint32_t* K; uint32_t* k_inf;
    uint32_t* prefix;          // optional: the hash state after domain_prefix (SHA_STATE_WORDS), for per-item headers
};
// Sha256 state as plain words: h, the partial block w, fill, total
constexpr int SHA_STATE_WORDS = 26;
BBS_HD void sha_store(uint32_t* dst, const Sha256& s) {
    for (int k = 0; k < 8; k++) dst[k] = s.h[k];
    for (int k = 0; k < 16; k++) dst[8 + k] = s.w[k];
    dst[24] = s.fill; dst[25] = s.total;
}
BBS_HD void sha_load(Sha256& s, const uint32_t* src) {
    for (int k = 0; k < 8; k++) s.h[k] = src[k];
    for (int k = 0; k < 16; k++) s.w[k] = src[8 + k];
    s.fill = src[24]; s.total = src[25];
}
// calculate_domain (core_utilities.rs:24-63) in two parts.  The prefix Z_pad || comp(pk) || I2OSP(L, 8) || comp(Q1) ..
// comp(H_L) || api_id does not depend on the header, so a per-item-header context keeps the state after it.
template <class C> BBS_HD void domain_prefix(Xmd48& x, const CtxDomainArgs& a) {
    x.begin();
    x.s.update(a.pk_comp, C::G2_BYTES);
    x.s.put_be64(a.L);
    x.s.update(a.gens_comp, (a.L + 1) * C::G1_BYTES);
    x.s.update(a.api_id, a.api_id_len);
}
// ... then I2OSP(header_len, 8) || header, expanded and reduced to the domain scalar (canonical limbs)
template <class C> BBS_HD void domain_finish(Xmd48& x, const uint8_t* header, uint32_t header_len, const uint8_t* dst,
                                             uint32_t dst_len, uint32_t* dom) {
    x.s.put_be64(header_len);
    x.s.update(header, header_len);
    BBS_A16 uint32_t okm[12];
    x.finish(dst, dst_len, okm);
    okm48_to_scalar<typename C::Fr>(dom, okm);
}
// calculate_domain + K = P1 + Q1*domain (verify.rs:81-82)
template <class C> BBS_HD void ctx_domain_item(const CtxDomainArgs& a, uint32_t) {
    Xmd48 x;
    domain_prefix<C>(x, a);
    if (a.prefix) sha_store(a.prefix, x.s);
    BBS_A16 uint32_t dom[8];
    domain_finish<C>(x, a.header, a.header_len, a.dst_h2s, a.dst_h2s_len, dom);
    bn_copy<8>(a.domain, dom);
    BBS_A16 uint32_t acc[G1J], p1[G1J];
    g1_mul_affine<C>(acc, a.gens, dom, 256);
    g1_from_affine<C>(p1, C::P1());
    g1_add<C>(acc, acc, p1);
    *a.k_inf = g1_to_affine_vt<C>(a.K, acc) ? 0u : 1u;
}

// q1_slot != 0: generator slot q1_slot is Q1 again (slot L + 1 of a per-item-header context)
struct CtxTableArgs { const uint32_t* K; const uint32_t* gens; uint32_t* tab; uint32_t* wbase; uint32_t tab_bits; uint32_t q1_slot; };
// entry (g, w, d) = (d * 2^(BITS w)) * base_g in affine form, in two steps:
//   ctx_wbase_item: the window bases 2^(BITS w) * base_g, affine (one thread per (g, w); a K at infinity gives zeros);
//   ctx_table_item: d * window base by a BITS-bit double-and-add, then to affine.
template <class C> BBS_HD void ctx_wbase_item(const CtxTableArgs& a, uint32_t i) {
    const TabGeom G(a.tab_bits);
    const uint32_t TAB_WINDOWS = (uint32_t)G.windows;
    const int TAB_BITS = G.bits;
    const uint32_t w = i % TAB_WINDOWS, g = i / TAB_WINDOWS;
    const uint32_t* base = g == 0 ? a.K : a.gens + (g == a.q1_slot ? 0u : g) * G1A;
    BBS_A16 uint32_t acc[G1J];
    g1_from_affine<C>(acc, base);
    if (bn_is_zero<2 * C::Fp::N>(base)) g1_set_inf<C>(acc);          // K at infinity is stored as zeros
    for (uint32_t k = 0; k < w * TAB_BITS; k++) g1_dbl<C>(acc, acc);
    g1_to_affine_vt<C>(a.wbase + (size_t)i * G1A, acc);
}
// Jacobian d * window base for table entry i; false when the base is the identity
template <class C> BBS_HD bool ctx_table_head(uint32_t* acc, const CtxTableArgs& a, uint32_t i) {
    const TabGeom G(a.tab_bits);
    const uint32_t TAB_ENTRIES = G.entries;
    const int TAB_BITS = G.bits;
    const uint32_t d = i % TAB_ENTRIES + 1;
    const uint32_t* wb = a.wbase + (size_t)(i / TAB_ENTRIES) * G1A;      // (g, w) = i / ENTRIES
    if (bn_is_zero<2 * C::Fp::N>(wb)) { g1_set_inf<C>(acc); return false; }
    BBS_A16 uint32_t k[1] = {d};
    g1_mul_affine<C>(acc, wb, k, TAB_BITS);
    return true;
}
// one entry with its own inversion (host simulation; the CUDA build uses ctx_table_kernel below)
template <class C> BBS_HD void ctx_table_item(const CtxTableArgs& a, uint32_t i) {
    BBS_A16 uint32_t acc[G1J];
    ctx_table_head<C>(acc, a, i);
    g1_to_affine<C>(a.tab + (size_t)i * G1A, acc);
}

struct CtxLinesArgs { const uint32_t* W; uint32_t w_inf; uint32_t* lines; };
template <class C> BBS_HD void ctx_lines_item(const CtxLinesArgs& a, uint32_t i) {
    if (i == 0) { if (!a.w_inf) g2_precompute_lines<C>(a.lines, a.W, 0); }
    else g2_precompute_lines<C>(a.lines, C::G2(), 1);
}

// Line table of the cooperative pairing kernel (M-type twist): entry (line, pair) = (Bc / A, 1 / A), i.e. the line scaled to
// constant term 1 (any Fp2 factor dies in the final exponentiation).  A == 0 (a tangent / chord through the origin,
// impossible for an honest key) is reported so that the context falls back to the per-thread kernel.
struct CtxLinesCoopArgs { const uint32_t* lines; uint32_t* lines2; uint32_t* degenerate; uint32_t w_inf; };
// one (line, pair) entry: raw (A, Bc) at `src` -> cooperative entry at `dst`; false when the line is degenerate
template <class C> BBS_HD bool lines_coop_one(uint32_t* dst, const uint32_t* src, bool skip) {
    if (skip) { bn_zero<4 * C::Fp::N>(dst); return true; }
    if (!C::M_TWIST) {
        // D-type twist (BN254): the constant term of the line is the item's y, so the line is normalised per item
        // (pairing_coop.cuh POINT_RATIO) and the table keeps (Bc, A) as they are: never degenerate
        f2_copy<C>(dst, src + F2N);
        f2_copy<C>(dst + F2N, src);
        return true;
    }
    if (f2_is_zero<C>(src)) { bn_zero<4 * C::Fp::N>(dst); return false; }
    BBS_A16 uint32_t ai[F2N], bp[F2N];
    f2_inv_vt<C>(ai, src);
    f2_mul<C>(bp, src + F2N, ai);
    f2_copy<C>(dst, bp);
    f2_copy<C>(dst + F2N, ai);
    return true;
}
template <class C> BBS_HD void ctx_lines_coop_item(const CtxLinesCoopArgs& a, uint32_t i) {
    const uint32_t* src = a.lines + (size_t)i * LINE_WORDS;
    uint32_t* dst = a.lines2 + ((size_t)(i >> 1) * 4 + (i & 1) * 2) * F2N;
    if (!lines_coop_one<C>(dst, src, (i & 1) == 0 && a.w_inf)) *a.degenerate = 1;
}
// the same for a chunk of an issuer set: entry t = (issuer, line, pair); pair 1 (BP2) is copied from the shared table
struct IssLinesCoopArgs {
    const uint32_t* raw; uint32_t raw_stride; const uint32_t* bp2_coop; uint32_t* coop; uint32_t coop_stride;
    uint32_t* flags; uint32_t first; uint32_t n_lines;
};
template <class C> BBS_HD void iss_lines_coop_item(const IssLinesCoopArgs& a, uint32_t t) {
    const uint32_t per = 2 * a.n_lines, local = t / per, j = t % per, i = a.first + local;
    uint32_t* dst = a.coop + (size_t)i * a.coop_stride + ((size_t)(j >> 1) * 4 + (j & 1) * 2) * F2N;
    if (j & 1) { bn_copy<4 * C::Fp::N>(dst, a.bp2_coop + ((size_t)(j >> 1) * 4 + 2) * F2N); return; }
    const uint32_t fl = a.flags[i];
    const uint32_t* src = a.raw + (size_t)local * a.raw_stride + (size_t)j * LINE_WORDS;
    if (!lines_coop_one<C>(dst, src, (fl & (ISS_BAD | ISS_W_INF)) != 0)) a.flags[i] = fl | ISS_BAD;   // degenerate line: see bbs_b200.h
}

// ---- issuer sets: many issuer keys over ONE generator list (multi-issuer batches, SURVEY 8f-4) -------------------
// `&self` (the public key) is per call in the reference (verify.rs:18-30): a batch may name a different issuer per item.
// Everything that depends on the key is small -- W (G2), domain, K = P1 + Q1 * domain, the Miller-loop lines of W -- and
// lives in per-issuer arrays; the fixed-base tables of H_1..H_L depend only on (suite, api_id, L) and are shared.
struct IssuerSetView {
    const uint32_t* K;          // n_issuers x affine K_i
    const uint32_t* flags;      // n_issuers x ISS_*
    const uint32_t* lines;      // n_issuers x line table, `line_stride` words apart (cooperative layout on the GPU, raw
                                // (A, Bc) layout in the host simulation)
    uint32_t line_stride;
    uint32_t n_issuers;
    const uint32_t* domains;    // n_issuers x 8 words: calculate_domain of issuer i (proof verification hashes it into the challenge)
};

struct IssDecodeArgs { const uint8_t* pks; uint32_t* W; uint32_t* flags; };
template <class C> BBS_HD void iss_decode_item(const IssDecodeArgs& a, uint32_t i) {
    const int st = g2_decompress<C>(a.W + (size_t)i * 4 * C::Fp::N, a.pks + (size_t)i * C::G2_BYTES);
    a.flags[i] = st == PT_BAD ? (uint32_t)ISS_BAD : (st == PT_INF ? (uint32_t)ISS_W_INF : 0u);
}
struct IssDomainArgs { CtxDomainArgs base; const uint8_t* pks; uint32_t* domains; uint32_t* K; uint32_t* flags; };
template <class C> BBS_HD void iss_domain_item(const IssDomainArgs& a, uint32_t i) {
    if (a.flags[i] & ISS_BAD) return;
    CtxDomainArgs d = a.base;
    uint32_t kinf = 0;
    d.pk_comp = a.pks + (size_t)i * C::G2_BYTES;
    d.domain = a.domains + (size_t)i * 8;
    d.K = a.K + (size_t)i * G1A;
    d.k_inf = &kinf;
    ctx_domain_item<C>(d, 0);
    if (kinf) a.flags[i] |= ISS_K_INF;
}
struct IssLinesArgs { const uint32_t* W; const uint32_t* flags; uint32_t* raw; uint32_t raw_stride; uint32_t first; };
template <class C> BBS_HD void iss_lines_item(const IssLinesArgs& a, uint32_t t) {
    const uint32_t i = a.first + t;
    if (a.flags[i] & (ISS_BAD | ISS_W_INF)) return;
    g2_precompute_lines<C>(a.raw + (size_t)t * a.raw_stride, a.W + (size_t)i * 4 * C::Fp::N, 0);
}

// ---- msg_to_scalars ----------------------------------------------------------------------------------
struct H2sArgs {
    const uint8_t* msgs; const uint64_t* offsets;   // message t = msgs[offsets[t] .. offsets[t+1])
    const uint8_t* dst; uint32_t dst_len;
    uint8_t* out;                                   // 32-byte little-endian scalars
};
template <class C> BBS_HD void h2s_item(const H2sArgs& a, uint32_t t) {
    BBS_A16 uint32_t s[8];
    uint64_t b = a.offsets[t], e = a.offsets[t + 1];
    hash_to_scalar<typename C::Fr>(s, a.msgs + b, (uint32_t)(e - b), a.dst, a.dst_len);
    limbs_to_le<8>(a.out + (size_t)t * 32, s);
}

// ---- fixed-base MSM over the window tables -------------------------------------------------------------
// acc += s * base_g, s canonical limbs (8)
template <class C> BBS_HDN void tab_accumulate(uint32_t* acc, const CtxView& cx, uint32_t g, const uint32_t* s) {
    const TabGeom G(cx.tab_bits);
    const uint32_t* tg = cx.tab + (size_t)g * G.windows * G.entries * G1A;
    BBS_A16 uint32_t k1[5], k2[5];
    glv_split<C>(k1, k2, s);
    for (int w = 0; w < G.windows; w++) {
        uint32_t d1 = tab_digit(G, k1, 5, w), d2 = tab_digit(G, k2, 5, w);
        if (d1) {
            BBS_A16 uint32_t e[G1A];
            const uint32_t* src = tg + ((size_t)w * G.entries + (d1 - 1)) * G1A;
            bn_copy<2 * C::Fp::N>(e, src);                               // 96- / 64-byte gather as 128-bit loads
            g1_add_mixed<C>(acc, acc, e);
        }
        if (d2) {
            BBS_A16 uint32_t e[G1A], t[FPN];
            const uint32_t* src = tg + ((size_t)w * G.entries + (d2 - 1)) * G1A;
            bn_copy<2 * C::Fp::N>(e, src);
            fe_mul<typename C::Fp>(t, e, C::GLV_BETA());            // phi(x, y) = (beta x, y)
            bn_copy<C::Fp::N>(e, t);
            g1_add_mixed<C>(acc, acc, e);
        }
    }
}

// pair-argument record handed from the G1 kernels to the pairing kernel
#define PAIR_WORDS (6 * C::Fp::N)
enum : uint32_t { FL_SKIP0 = 1, FL_SKIP1 = 2, FL_DONE = 4 };   // FL_DONE: status already final, no pairing

// ---- per-item headers (bbs_*_hdr) ------------------------------------------------------------------------
// A call with a header per item hashes domain_i and builds K_i = P1 + Q1 * domain_i per item (item_domain_kernel below) into
// arrays indexed by item; W and the line tables stay the context's.  K == nullptr: every item uses the context's K and domain.
struct ItemKeyView {
    const uint32_t* K;         // n x affine K_i (zeros for the identity)
    const uint32_t* domains;   // n x 8 words, canonical limbs
    const uint32_t* flags;     // n x (ISS_K_INF or 0)
};
// K, domain and identity flags (ISS_W_INF | ISS_K_INF) of item i
template <class C> BBS_HD uint32_t item_key(const CtxView& cx, const ItemKeyView& it, uint32_t i, const uint32_t*& K,
                                            const uint32_t*& domain) {
    const uint32_t w = cx.w_inf ? (uint32_t)ISS_W_INF : 0u;
    if (!it.K) { K = cx.K; domain = cx.domain; return w | (cx.k_inf ? (uint32_t)ISS_K_INF : 0u); }
    K = it.K + (size_t)i * G1A; domain = it.domains + (size_t)i * 8;
    return w | it.flags[i];
}
// domain of item i alone: sign and proof gen read it where they hash it, so that no pointer is held across the G1 work
// (that cost those kernels spill slots)
template <class C> BBS_HD const uint32_t* item_domain(const CtxView& cx, const ItemKeyView& it, uint32_t i) {
    return it.K ? it.domains + (size_t)i * 8 : cx.domain;
}
// presentation header of item i: the call's shared ph, or ph[ph_off[i] .. ph_off[i+1]) when the call has one per item
BBS_HD const uint8_t* item_ph(const uint8_t* ph, uint32_t ph_len, const uint64_t* ph_off, uint32_t i, uint32_t& len) {
    if (!ph_off) { len = ph_len; return ph; }
    len = (uint32_t)(ph_off[i + 1] - ph_off[i]);
    return ph + ph_off[i];
}

struct ItemDomainArgs {
    CtxView ctx;
    const uint32_t* prefix;                         // hash state after domain_prefix (SHA_STATE_WORDS)
    const uint8_t* headers; const uint64_t* hdr_off;  // header i = headers[hdr_off[i] .. hdr_off[i+1])
    uint32_t* domains; uint32_t* K; uint32_t* flags;  // the arrays of ItemKeyView
};
// domain_i (written out) and the Jacobian K_i; Q1's window table is slot L + 1 of a per-item-header context
template <class C> BBS_HD void item_domain_head(const ItemDomainArgs& a, uint32_t i, uint32_t* Kj) {
    Xmd48 x;
    sha_load(x.s, a.prefix);
    const uint64_t b = a.hdr_off[i];
    BBS_A16 uint32_t dom[8];
    domain_finish<C>(x, a.headers + b, (uint32_t)(a.hdr_off[i + 1] - b), a.ctx.dst_h2s, a.ctx.dst_h2s_len, dom);
    bn_copy<8>(a.domains + (size_t)i * 8, dom);
    g1_from_affine<C>(Kj, C::P1());
    tab_accumulate<C>(Kj, a.ctx, a.ctx.L + 1, dom);
}
// K_i to affine with zinv = 1 / Z (unused for the identity)
template <class C> BBS_HD void item_domain_tail(const ItemDomainArgs& a, uint32_t i, const uint32_t* Kj, const uint32_t* zinv) {
    using F = typename C::Fp;
    uint32_t* K = a.K + (size_t)i * G1A;
    if (g1_is_inf_ool<C>(Kj)) { bn_zero<2 * C::Fp::N>(K); a.flags[i] = ISS_K_INF; return; }
    BBS_A16 uint32_t zi2[FPN];
    fe_sqr<F>(zi2, zinv);
    fe_mul<F>(K, Kj, zi2);
    fe_mul<F>(zi2, zi2, zinv);
    fe_mul<F>(K + FPN, Kj + FPN, zi2);
    a.flags[i] = 0;
}
// one item, its own inversion (host simulation; the CUDA build uses item_domain_kernel)
template <class C> BBS_HD void item_domain_item(const ItemDomainArgs& a, uint32_t i) {
    BBS_A16 uint32_t Kj[G1J], z[FPN];
    item_domain_head<C>(a, i, Kj);
    if (!g1_is_inf_ool<C>(Kj)) fe_inv<typename C::Fp>(z, Kj + 2 * FPN);
    item_domain_tail<C>(a, i, Kj, z);
}

// ---- core_verify, G1 half ------------------------------------------------------------------------------
struct VerifyG1Args {
    CtxView ctx;
    const uint8_t* sigs;       // n x (G1 compressed || LE32 e)   (ark CanonicalSerialize of Signature, sign.rs:18-22)
    const uint8_t* scalars;    // n x n_msgs x LE32
    uint32_t n_msgs;
    uint32_t* pair; uint32_t* flags; uint8_t* status;
    const uint32_t* item_issuer;   // multi-issuer batches: issuer of item i in `iss` (nullptr: the context's own key)
    IssuerSetView iss;
    // split path (verify_g1_split_kernel + verify_g1_combine_kernel): per item the Jacobian e*A and B and a state byte
    uint32_t* part_v; uint32_t* part_f; uint8_t* part_st;
    ItemKeyView item;              // per-item headers (not with issuer sets)
};
enum : uint8_t { VST_PA = 3, VST_VDONE = 4, VST_FBAD = 8 };      // part_st: PT_* of A | status already final | bad scalar
// the key-dependent inputs of item i: K and the two identity flags
template <class C> BBS_HD uint32_t verify_issuer(const VerifyG1Args& a, uint32_t i, const uint32_t*& K) {
    if (!a.item_issuer) { const uint32_t* domain; return item_key<C>(a.ctx, a.item, i, K, domain); }
    const uint32_t s = a.item_issuer[i];
    if (s >= a.iss.n_issuers) { K = a.ctx.K; return ISS_BAD; }
    K = a.iss.K + (size_t)s * G1A;
    return a.iss.flags[s];
}
// Part 1: everything up to the Jacobian point Cc = e A - B.  Returns false when the item's status is already final.
template <class C> BBS_HD bool verify_g1_head(const VerifyG1Args& a, uint32_t i, uint32_t* Cc, int& pa) {
    const CtxView& cx = a.ctx;
    if (a.n_msgs != cx.L) { a.status[i] = ST_ERR_MSG_GEN_LEN; a.flags[i] = FL_DONE; return false; }   // verify.rs:68-71
    const uint32_t* Kp;
    const uint32_t ifl = verify_issuer<C>(a, i, Kp);
    if (ifl & ISS_BAD) { a.status[i] = ST_ERR_MALFORMED; a.flags[i] = FL_DONE; return false; }        // undecodable issuer key
    const uint8_t* sig = a.sigs + (size_t)i * (C::G1_BYTES + 32);
    BBS_A16 uint32_t A[G1A], e[8];
    pa = g1_decompress<C>(A, sig);
    bool ok = pa != PT_BAD && fr_from_le32<C>(e, sig + C::G1_BYTES);
    // B = P1 + Q1*domain + sum H_j m_j  (verify.rs:81-86), K = P1 + Q1*domain hoisted into the context
    BBS_A16 uint32_t B[G1J];
    if (ifl & ISS_K_INF) g1_set_inf<C>(B); else g1_from_affine<C>(B, Kp);
    const uint8_t* sc = a.scalars + (size_t)i * a.n_msgs * 32;
    for (uint32_t j = 0; j < a.n_msgs && ok; j++) {
        BBS_A16 uint32_t m[8];
        ok = fr_from_le32<C>(m, sc + j * 32);
        if (ok) tab_accumulate<C>(B, cx, j + 1, m);
    }
    if (!ok) { a.status[i] = ST_ERR_MALFORMED; a.flags[i] = FL_DONE; return false; }
    // e(A, W + e BP2) e(B, -BP2) == 1  <=>  e(A, W) e(eA - B, BP2) == 1   (SURVEY 8a note (i))
    g1_neg<C>(Cc, B);
    if (pa == PT_OK) {
        BBS_A16 uint32_t eA[G1J];
        g1_mul_scalar<C>(eA, A, e);
        g1_add<C>(Cc, Cc, eA);
    }
    // first pairing argument: A itself (affine)
    uint32_t* pr = a.pair + (size_t)i * PAIR_WORDS;
    bn_copy<2 * C::Fp::N>(pr, A); fe_set_one<typename C::Fp>(pr + 2 * FPN);
    return true;
}
// Part 2: both pairing arguments leave the kernel affine, (x, y, 1): the cooperative pairing kernel normalises its
// lines to constant term 1, which needs Z = 1 (pairing_coop.cuh).  zinv = 1 / Z of Cc (unused for the identity).
template <class C> BBS_HD void verify_g1_tail(const VerifyG1Args& a, uint32_t i, const uint32_t* Cc, const uint32_t* zinv, int pa) {
    using F = typename C::Fp;
    uint32_t* pr = a.pair + (size_t)i * PAIR_WORDS;
    const bool cfin = !g1_is_inf_ool<C>(Cc);
    if (cfin) {
        BBS_A16 uint32_t zi2[FPN];
        fe_sqr<F>(zi2, zinv);
        fe_mul<F>(pr + 3 * FPN, Cc, zi2);
        fe_mul<F>(zi2, zi2, zinv);
        fe_mul<F>(pr + 4 * FPN, Cc + FPN, zi2);
    } else {
        bn_zero<2 * C::Fp::N>(pr + 3 * FPN);
    }
    fe_set_one<F>(pr + 5 * FPN);
    uint32_t fl = 0;
    const uint32_t* Kp;
    if (pa == PT_INF || (verify_issuer<C>(a, i, Kp) & ISS_W_INF)) fl |= FL_SKIP0;
    if (!cfin) fl |= FL_SKIP1;
    a.flags[i] = fl;
}
// one item, its own inversion (host simulation; the CUDA build uses verify_g1_kernel below)
template <class C> BBS_HD void verify_g1_item(const VerifyG1Args& a, uint32_t i) {
    BBS_A16 uint32_t Cc[G1J], zinv[FPN];
    int pa = PT_BAD;
    if (!verify_g1_head<C>(a, i, Cc, pa)) return;
    if (!g1_is_inf_ool<C>(Cc)) fe_inv<typename C::Fp>(zinv, Cc + 2 * FPN);
    verify_g1_tail<C>(a, i, Cc, zinv, pa);
}

// ---- the same work as two independent tasks per item (CUDA build, verify_g1_split_kernel) --------------------------------
// One thread per item is a serial chain of ~5,300 field multiplications; at the headline batch (65,536 items = 443 threads
// per SM) every item is resident at once and the kernel time is that chain's latency.  Split per item into the
// variable-base task V (decode + subgroup test of A, e*A: ~3,400 multiplications) and the fixed-base task F
// (B = K + sum tab: ~1,900), 2n tasks go through the block scheduler -- V blocks first, F blocks fill in behind -- and the
// critical path per item shrinks to V.  A small third kernel joins them (C = e*A - B, one inversion per block, flags).
template <class C> BBS_HD void verify_task_v(const VerifyG1Args& a, uint32_t i) {
    const CtxView& cx = a.ctx;
    a.part_st[i] = VST_VDONE;
    if (a.n_msgs != cx.L) { a.status[i] = ST_ERR_MSG_GEN_LEN; a.flags[i] = FL_DONE; return; }          // verify.rs:68-71
    const uint32_t* Kp;
    const uint32_t ifl = verify_issuer<C>(a, i, Kp);
    if (ifl & ISS_BAD) { a.status[i] = ST_ERR_MALFORMED; a.flags[i] = FL_DONE; return; }
    const uint8_t* sig = a.sigs + (size_t)i * (C::G1_BYTES + 32);
    BBS_A16 uint32_t A[G1A], e[8];
    const int pa = g1_decompress<C>(A, sig);
    if (pa == PT_BAD || !fr_from_le32<C>(e, sig + C::G1_BYTES)) { a.status[i] = ST_ERR_MALFORMED; a.flags[i] = FL_DONE; return; }
    uint32_t* pv = a.part_v + (size_t)i * G1J;
    if (pa == PT_OK) {
        BBS_A16 uint32_t eA[G1J];
        g1_mul_scalar<C>(eA, A, e);
        g1_copy<C>(pv, eA);
    }
    uint32_t* pr = a.pair + (size_t)i * PAIR_WORDS;
    bn_copy<2 * C::Fp::N>(pr, A); fe_set_one<typename C::Fp>(pr + 2 * FPN);
    a.part_st[i] = (uint8_t)pa;
}
template <class C> BBS_HD void verify_task_f(const VerifyG1Args& a, uint32_t i, uint8_t* fbad) {
    const CtxView& cx = a.ctx;
    *fbad = 0;
    if (a.n_msgs != cx.L) return;
    const uint32_t* Kp;
    const uint32_t ifl = verify_issuer<C>(a, i, Kp);
    if (ifl & ISS_BAD) return;
    BBS_A16 uint32_t B[G1J];
    if (ifl & ISS_K_INF) g1_set_inf<C>(B); else g1_from_affine<C>(B, Kp);
    const uint8_t* sc = a.scalars + (size_t)i * a.n_msgs * 32;
    bool ok = true;
    for (uint32_t j = 0; j < a.n_msgs && ok; j++) {
        BBS_A16 uint32_t m[8];
        ok = fr_from_le32<C>(m, sc + j * 32);
        if (ok) tab_accumulate<C>(B, cx, j + 1, m);
    }
    if (!ok) { *fbad = 1; return; }
    g1_copy<C>(a.part_f + (size_t)i * G1J, B);
}

// join, part 1: Cc = e*A - B; false when the item's status is already final
template <class C> BBS_HD bool verify_join_head(const VerifyG1Args& a, uint32_t i, const uint8_t* fbad, uint32_t* Cc, int& pa) {
    const uint8_t st = a.part_st[i];
    if (st & VST_VDONE) return false;
    if (fbad[i]) { a.status[i] = ST_ERR_MALFORMED; a.flags[i] = FL_DONE; return false; }
    pa = st & VST_PA;
    BBS_A16 uint32_t B[G1J];
    g1_copy<C>(B, a.part_f + (size_t)i * G1J);
    g1_neg<C>(Cc, B);                                  // e(A, W) e(eA - B, BP2) == 1   (SURVEY 8a note (i))
    if (pa == PT_OK) g1_add<C>(Cc, Cc, a.part_v + (size_t)i * G1J);
    return true;
}
// the join with one inversion per item (host simulation of verify_g1_combine_kernel)
template <class C> BBS_HD void verify_join_item(const VerifyG1Args& a, uint32_t i, const uint8_t* fbad) {
    using F = typename C::Fp;
    BBS_A16 uint32_t Cc[G1J], z[FPN];
    int pa = PT_BAD;
    if (!verify_join_head<C>(a, i, fbad, Cc, pa)) return;
    if (!g1_is_inf_ool<C>(Cc)) fe_inv<F>(z, Cc + 2 * FPN); else fe_set_one<F>(z);
    verify_g1_tail<C>(a, i, Cc, z, pa);
}

#if defined(__CUDACC__) && !defined(BBS_HOSTSIM)
// Block-wide simultaneous inversion (Montgomery's trick as a product tree in shared memory): one Fermat inversion per
// block instead of one per thread.  On a SIMT machine an inversion costs the warp the same whether one lane or all
// 32 need it, so the saving comes from the other warps of the block: 7 of 8 skip their ~490 multiplications and pay
// ~25 for the tree instead.  z must be non-zero in every thread (pass 1 for items without a point); TPB a power of 2.
// VT: the root is inverted by the variable-time binary Euclid instead of the Fermat ladder (public data only).  Measured:
// context creation 2x, sign_kernel -6.5 %, verify_g1_kernel<Bn> (64-thread blocks) -2.8 %, but verify_g1_kernel<Bls>
// (256-thread blocks) +5 %, so the callers choose.
template <class F, int TPB, bool VT> __device__ __forceinline__ void block_batch_inverse(uint32_t* z, uint32_t (*tree)[F::N]) {
    constexpr int N = F::N;
    const int t = threadIdx.x;
    // leaves at tree[TPB + t], node k = product of its children 2k, 2k+1, root at tree[1]
    bn_copy<N>(tree[TPB + t], z);
    __syncthreads();
    for (int w = TPB / 2; w >= 1; w >>= 1) {
        if (t < w) fe_mul<F>(tree[w + t], tree[2 * (w + t)], tree[2 * (w + t) + 1]);
        __syncthreads();
    }
    if (t == 0) {
        BBS_A16 uint32_t r[N];
        if (VT) fe_inv_vt<F>(r, tree[1]); else fe_inv<F>(r, tree[1]);
        bn_copy<N>(tree[1], r);
    }
    __syncthreads();
    // going down: inv(left) = inv(parent) * right, inv(right) = inv(parent) * left
    for (int w = 1; w < TPB; w <<= 1) {
        if (t < w) {
            BBS_A16 uint32_t l[N], r[N], ip[N];
            bn_copy<N>(ip, tree[w + t]);
            bn_copy<N>(l, tree[2 * (w + t)]);
            bn_copy<N>(r, tree[2 * (w + t) + 1]);
            fe_mul<F>(tree[2 * (w + t)], ip, r);
            fe_mul<F>(tree[2 * (w + t) + 1], ip, l);
        }
        __syncthreads();
    }
    bn_copy<N>(z, tree[TPB + t]);
}

// table entries with one inversion per block
template <class C, int TPB> __global__ void __launch_bounds__(TPB, 4) ctx_table_kernel(const CtxTableArgs a, uint32_t n) {
    using F = typename C::Fp;
    __shared__ BBS_A16 uint32_t tree[2 * TPB][C::Fp::N];
    const uint32_t i = blockIdx.x * TPB + threadIdx.x;
    BBS_A16 uint32_t acc[G1J], z[FPN];
    const bool live = i < n && ctx_table_head<C>(acc, a, i) && !g1_is_inf_ool<C>(acc);
    if (live) bn_copy<C::Fp::N>(z, acc + 2 * FPN); else fe_set_one<F>(z);
    block_batch_inverse<F, TPB, true>(z, tree);
    if (i < n) {
        uint32_t* dst = a.tab + (size_t)i * G1A;
        if (live) {
            BBS_A16 uint32_t zi2[FPN];
            fe_sqr<F>(zi2, z);
            fe_mul<F>(dst, acc, zi2);
            fe_mul<F>(zi2, zi2, z);
            fe_mul<F>(dst + FPN, acc + FPN, zi2);
        } else {
            bn_zero<2 * C::Fp::N>(dst);
        }
    }
}

template <class C, int TPB, int MINB> __global__ void __launch_bounds__(TPB, MINB) verify_g1_kernel(const VerifyG1Args a, uint32_t n) {
    using F = typename C::Fp;
    __shared__ BBS_A16 uint32_t tree[2 * TPB][C::Fp::N];
    const uint32_t i = blockIdx.x * TPB + threadIdx.x;
    BBS_A16 uint32_t Cc[G1J], z[FPN];
    int pa = PT_BAD;
    const bool live = i < n && verify_g1_head<C>(a, i, Cc, pa);
    if (live && !g1_is_inf_ool<C>(Cc)) bn_copy<C::Fp::N>(z, Cc + 2 * FPN); else fe_set_one<F>(z);
#ifdef BBS_NO_BATCH_INV
    { uint32_t zz[FPN]; fe_inv<F>(zz, z); bn_copy<C::Fp::N>(z, zz); (void)tree; }
#else
    block_batch_inverse<F, TPB, (TPB < 256)>(z, tree);
#endif
    if (live) verify_g1_tail<C>(a, i, Cc, z, pa);
}

// 2 * nb blocks: the first nb run task V for items [0, n), the next nb task F.  `fbad` (one byte per item) is written by F.
template <class C, int TPB, int MINB> __global__ void __launch_bounds__(TPB, MINB)
verify_g1_split_kernel(const VerifyG1Args a, uint32_t n, uint32_t nb, uint8_t* fbad) {
    const bool var = blockIdx.x < nb;
    const uint32_t i = (blockIdx.x - (var ? 0u : nb)) * TPB + threadIdx.x;
    if (i >= n) return;
    if (var) verify_task_v<C>(a, i); else verify_task_f<C>(a, i, fbad + i);
}
template <class C, int TPB> __global__ void __launch_bounds__(TPB, 2)
verify_g1_combine_kernel(const VerifyG1Args a, uint32_t n, const uint8_t* fbad) {
    using F = typename C::Fp;
    __shared__ BBS_A16 uint32_t tree[2 * TPB][C::Fp::N];
    const uint32_t i = blockIdx.x * TPB + threadIdx.x;
    BBS_A16 uint32_t Cc[G1J], z[FPN];
    int pa = PT_BAD;
    const bool live = i < n && verify_join_head<C>(a, i, fbad, Cc, pa);
    if (live && !g1_is_inf_ool<C>(Cc)) bn_copy<C::Fp::N>(z, Cc + 2 * FPN); else fe_set_one<F>(z);
    block_batch_inverse<F, TPB, true>(z, tree);
    if (live) verify_g1_tail<C>(a, i, Cc, z, pa);
}
#endif

#if defined(__CUDACC__) && !defined(BBS_HOSTSIM)
// domain_i and K_i of a call with per-item headers, one inversion per block for the affine K_i
template <class C, int TPB> __global__ void __launch_bounds__(TPB, 4) item_domain_kernel(const ItemDomainArgs a, uint32_t n) {
    using F = typename C::Fp;
    __shared__ BBS_A16 uint32_t tree[2 * TPB][C::Fp::N];
    const uint32_t i = blockIdx.x * TPB + threadIdx.x;
    BBS_A16 uint32_t Kj[G1J], z[FPN];
    const bool live = i < n;
    if (live) item_domain_head<C>(a, i, Kj);
    if (live && !g1_is_inf_ool<C>(Kj)) bn_copy<C::Fp::N>(z, Kj + 2 * FPN); else fe_set_one<F>(z);
    block_batch_inverse<F, TPB, true>(z, tree);
    if (live) item_domain_tail<C>(a, i, Kj, z);
}
#endif

// ---- pairing half (shared by verify and proof verify) ----------------------------------------------------
struct PairingArgs {
    const uint32_t* lines; const uint32_t* pair; const uint32_t* flags; uint8_t* status;
    const uint32_t* item_issuer; uint32_t line_stride;     // multi-issuer: lines + item_issuer[i] * line_stride
};
template <class C> BBS_HD void pairing_item(const PairingArgs& a, uint32_t i) {
    uint32_t fl = a.flags[i];
    if (fl & FL_DONE) return;
    const uint32_t* lines = a.item_issuer ? a.lines + (size_t)a.item_issuer[i] * a.line_stride : a.lines;
    BBS_A16 uint32_t P[PAIR_WORDS], f[F12N];
    const uint32_t* src = a.pair + (size_t)i * PAIR_WORDS;
    for (int j = 0; j < PAIR_WORDS; j++) P[j] = src[j];
    miller2<C>(f, lines, P, (fl & FL_SKIP0) != 0, P + 3 * FPN, (fl & FL_SKIP1) != 0);
    a.status[i] = final_exp_is_one<C>(f) ? ST_ACCEPT : ST_REJECT;
}

// ---- core_sign -----------------------------------------------------------------------------------------
struct SignArgs {
    CtxView ctx;
    const uint32_t* sk;        // canonical limbs (8) in a device buffer that the host clears after the call: the secret never
                               // travels in the kernel-parameter bank (key_gen.rs:29: SecretKey is Zeroize + ZeroizeOnDrop)
    const uint8_t* scalars; uint32_t n_msgs;
    uint8_t* sigs_out;         // n x (G1 compressed || LE32 e)
    uint8_t* b_out;            // optional: n x G1 compressed B (row a7)
    uint8_t* status;
    ItemKeyView item;          // per-item headers
};
// core_sign in three parts around its three inversions (1 / B.Z, 1 / (sk + e), 1 / A.Z), so that the CUDA build can take
// each of them once per block (sign_kernel below) while the host simulation inverts per item (sign_item).
// Part 1: B (Jacobian), e, and sk + e in Montgomery form.  false: the item's status is final.
// PER_ITEM = false: a call without per-item headers; the per-item reads are compiled out (sign_kernel)
template <class C, bool PER_ITEM> BBS_HD bool sign_head(const SignArgs& a, uint32_t i, uint32_t* B, uint32_t* e, uint32_t* sm) {
    using Fr = typename C::Fr;
    const CtxView& cx = a.ctx;
    const ItemKeyView item = PER_ITEM ? a.item : ItemKeyView{};
    if (a.n_msgs != cx.L) { a.status[i] = ST_ERR_MSG_GEN_LEN; return false; }     // sign.rs:76-79
    const uint8_t* sc = a.scalars + (size_t)i * a.n_msgs * 32;
    // e = H2S(BE(sk) || BE(m_1..m_L) || BE(domain), api_id || "H2S_")   (sign.rs:90-118)
    Xmd48 x;
    x.begin();
    BBS_A16 uint32_t sk[8];
    for (int k = 0; k < 8; k++) sk[k] = a.sk[k];
    for (int k = 7; k >= 0; k--) x.s.update_words(&sk[k], 1);
    {
        const uint32_t *Kp, *domain;
        if (item_key<C>(cx, item, i, Kp, domain) & ISS_K_INF) g1_set_inf<C>(B); else g1_from_affine<C>(B, Kp);
    }
    bool ok = true;
    for (uint32_t j = 0; j < a.n_msgs && ok; j++) {
        BBS_A16 uint32_t m[8];
        ok = fr_from_le32<C>(m, sc + j * 32);
        if (!ok) break;
        for (int k = 7; k >= 0; k--) x.s.update_words(&m[k], 1);
        tab_accumulate<C>(B, cx, j + 1, m);                                      // sign.rs:120-126
    }
    if (!ok) { a.status[i] = ST_ERR_MALFORMED; return false; }
    const uint32_t* domain = item_domain<C>(cx, item, i);
    for (int k = 7; k >= 0; k--) x.s.update_words(&domain[k], 1);
    BBS_A16 uint32_t okm[12], s[8];
    x.finish(cx.dst_h2s, cx.dst_h2s_len, okm);
    okm48_to_scalar<Fr>(e, okm);
    fe_add<Fr>(s, sk, e);
    if (bn_is_zero<8>(s)) { a.status[i] = ST_ERR_MALFORMED; return false; }        // sign.rs:129 panics
    fe_to_mont<Fr>(sm, s);
    return true;
}
// Part 2: A = B * (sk + e)^-1 (sign.rs:130) with the windowed GLV multiplication; B is normalised first (its affine form is
// also what the optional B output serialises).  zinv = 1 / B.Z (unused for the identity), sinv = (sk + e)^-1 (Montgomery).
template <class C> BBS_HD void sign_mid(uint32_t* Aj, uint32_t* Baff, bool& bfin, const uint32_t* B, const uint32_t* zinv,
                                        const uint32_t* sinv) {
    using F = typename C::Fp;
    BBS_A16 uint32_t s[8];
    fe_from_mont<typename C::Fr>(s, sinv);
    bfin = !g1_is_inf_ool<C>(B);
    if (bfin) {
        BBS_A16 uint32_t zi2[FPN];
        fe_sqr<F>(zi2, zinv);
        fe_mul<F>(Baff, B, zi2);
        fe_mul<F>(zi2, zi2, zinv);
        fe_mul<F>(Baff + FPN, B + FPN, zi2);
        g1_mul_scalar<C>(Aj, Baff, s);
    } else {
        bn_zero<2 * C::Fp::N>(Baff);
        g1_set_inf<C>(Aj);
    }
}
// Part 3: serialise.  zinv = 1 / A.Z (unused for the identity)
template <class C> BBS_HD void sign_tail(const SignArgs& a, uint32_t i, const uint32_t* Aj, const uint32_t* zinv, const uint32_t* e,
                                         const uint32_t* Baff, bool bfin) {
    using F = typename C::Fp;
    uint8_t* out = a.sigs_out + (size_t)i * (C::G1_BYTES + 32);
    BBS_A16 uint32_t aff[G1A];
    const bool afin = !g1_is_inf_ool<C>(Aj);
    if (afin) {
        BBS_A16 uint32_t zi2[FPN];
        fe_sqr<F>(zi2, zinv);
        fe_mul<F>(aff, Aj, zi2);
        fe_mul<F>(zi2, zi2, zinv);
        fe_mul<F>(aff + FPN, Aj + FPN, zi2);
    } else {
        bn_zero<2 * C::Fp::N>(aff);
    }
    g1_compress_affine<C>(out, aff, !afin);
    limbs_to_le<8>(out + C::G1_BYTES, e);
    if (a.b_out) g1_compress_affine<C>(a.b_out + (size_t)i * C::G1_BYTES, Baff, !bfin);
    a.status[i] = ST_ACCEPT;
}
// one item, its own inversions (host simulation; the CUDA build uses sign_kernel below)
template <class C> BBS_HD void sign_item(const SignArgs& a, uint32_t i) {
    using F = typename C::Fp;
    BBS_A16 uint32_t B[G1J], e[8], sm[8], zinv[FPN], Aj[G1J], Baff[G1A];
    if (!sign_head<C, true>(a, i, B, e, sm)) return;
    if (!g1_is_inf_ool<C>(B)) fe_inv<F>(zinv, B + 2 * FPN);
    fe_inv<typename C::Fr>(sm, sm);
    bool bfin;
    sign_mid<C>(Aj, Baff, bfin, B, zinv, sm);
    if (!g1_is_inf_ool<C>(Aj)) fe_inv<F>(zinv, Aj + 2 * FPN);
    sign_tail<C>(a, i, Aj, zinv, e, Baff, bfin);
}

#if defined(__CUDACC__) && !defined(BBS_HOSTSIM)
// the three inversions of core_sign, each taken once per block (block_batch_inverse: Montgomery's trick as a product tree)
// PER_ITEM = false (calls without per-item headers): the per-item reads are compiled out, so that these calls run the code
// they ran before per-item headers existed
template <class C, int TPB, int MINB, bool PER_ITEM> __global__ void __launch_bounds__(TPB, MINB) sign_kernel(const SignArgs a, uint32_t n) {
    using F = typename C::Fp;
    using Fr = typename C::Fr;
    __shared__ BBS_A16 uint32_t tree[2 * TPB][C::Fp::N];
    const uint32_t i = blockIdx.x * TPB + threadIdx.x;
    BBS_A16 uint32_t B[G1J], e[8], sm[8], z[FPN], Aj[G1J], Baff[G1A];
    const bool live = i < n && sign_head<C, PER_ITEM>(a, i, B, e, sm);
    if (live && !g1_is_inf_ool<C>(B)) bn_copy<C::Fp::N>(z, B + 2 * FPN); else fe_set_one<F>(z);
    if (!live) fe_set_one<Fr>(sm);
    block_batch_inverse<F, TPB, true>(z, tree);
    __syncthreads();
    block_batch_inverse<Fr, TPB, false>(sm, (uint32_t (*)[Fr::N])tree);      // 1 / (sk + e): secret, constant-time ladder
    __syncthreads();
    bool bfin = false;
    if (live) sign_mid<C>(Aj, Baff, bfin, B, z, sm);
    if (live && !g1_is_inf_ool<C>(Aj)) bn_copy<C::Fp::N>(z, Aj + 2 * FPN); else fe_set_one<F>(z);
    block_batch_inverse<F, TPB, true>(z, tree);
    if (live) sign_tail<C>(a, i, Aj, z, e, Baff, bfin);
    // the tree held products and inverses of the secret values sk + e: leave no trace in shared memory
    __syncthreads();
    bn_zero<C::Fp::N>(tree[threadIdx.x]); bn_zero<C::Fp::N>(tree[TPB + threadIdx.x]);
}
#endif

// ---- core_proof_verify, G1 half ---------------------------------------------------------------------------
struct ProofG1Args {
    CtxView ctx;
    const uint8_t* proofs;         // n x (3 G1 compressed || LE32 e^, r1^, r3^, c)
    const uint8_t* commitments;    // flat LE32 scalars m^_j
    const uint64_t* commit_off;    // n+1, in scalars
    const uint32_t* dis_idx;       // flat disclosed indexes
    const uint8_t* dis_scalars;    // flat LE32 disclosed message scalars (same indexing as dis_idx)
    const uint64_t* dis_off;       // n+1
    const uint8_t* ph; uint32_t ph_len;
    uint32_t* pair; uint32_t* flags; uint8_t* status;
    // split path (proof_g1_split_kernel + proof_g1_join_kernel): Jacobian T1, D*r3^, fixed-base part of T2; state bytes
    uint32_t* part_t1; uint32_t* part_v2; uint32_t* part_f; uint8_t* part_st;
    // issuer sets (split path only): proof i is checked under issuer item_issuer[i]; K_i * c is variable-base then
    const uint32_t* item_issuer; IssuerSetView iss;
    // per-item headers (split path only, as issuer sets); per-item ph: ph[ph_off[i] .. ph_off[i+1]) (nullptr: shared ph)
    ItemKeyView item; const uint64_t* ph_off;
};
// K_i has no window table when it is per item (issuer sets, per-item headers): K_i * c is then part of task V2.
// PER_ITEM (here and in the proof_task_* / proof_join_* functions) = false: a call without per-item headers or phs, whose
// kernels are compiled without the per-item reads (the host simulation passes true: the reads check for themselves)
template <bool PER_ITEM> BBS_HD bool proof_k_variable(const ProofG1Args& a) { return a.item_issuer || (PER_ITEM && a.item.K); }
template <bool PER_ITEM> BBS_HD const uint64_t* proof_ph_off(const ProofG1Args& a) { return PER_ITEM ? a.ph_off : nullptr; }
template <class C> BBS_HD void proof_g1_item(const ProofG1Args& a, uint32_t i) {
    using F = typename C::Fp;
    using Fr = typename C::Fr;
    const CtxView& cx = a.ctx;
    constexpr int GB = C::G1_BYTES;
    const uint8_t* pf = a.proofs + (size_t)i * (3 * GB + 128);
    uint64_t cb = a.commit_off[i], U = a.commit_off[i + 1] - cb;
    uint64_t db = a.dis_off[i], R = a.dis_off[i + 1] - db;
    uint64_t L = R + U;
#define PROOF_FAIL(code) { a.status[i] = (code); a.flags[i] = FL_DONE; return; }
    // proof_verify.rs:139-150, in the reference's order
    BBS_A16 uint32_t mask[MAX_L / 32];
    for (int k = 0; k < MAX_L / 32; k++) mask[k] = 0;
    bool dup = false;
    for (uint64_t k = 0; k < R; k++) {
        uint32_t idx = a.dis_idx[db + k];
        if (idx >= L) PROOF_FAIL(ST_ERR_DISCLOSED_INDEX)
        if (idx < MAX_L) { dup |= (mask[idx >> 5] >> (idx & 31)) & 1; mask[idx >> 5] |= 1u << (idx & 31); }
    }
    if (L != cx.L) PROOF_FAIL(ST_ERR_MSG_GEN_LEN)
    if (dup) PROOF_FAIL(ST_ERR_MALFORMED)     // the reference indexes out of bounds and panics (proof_verify.rs:179)
    BBS_A16 uint32_t Ab[G1A], Bb[G1A], D[G1A], ecap[8], r1cap[8], r3cap[8], c[8];
    int pA = g1_decompress<C>(Ab, pf), pB = g1_decompress<C>(Bb, pf + GB), pD = g1_decompress<C>(D, pf + 2 * GB);
    bool ok = pA != PT_BAD && pB != PT_BAD && pD != PT_BAD;
    ok = ok && fr_from_le32<C>(ecap, pf + 3 * GB) && fr_from_le32<C>(r1cap, pf + 3 * GB + 32) &&
         fr_from_le32<C>(r3cap, pf + 3 * GB + 64) && fr_from_le32<C>(c, pf + 3 * GB + 96);
    if (!ok) PROOF_FAIL(ST_ERR_MALFORMED)
    // T1 = Bbar*c + Abar*e^ + D*r1^   (proof_verify.rs:163-164): one windowed three-point multi-scalar product
    BBS_A16 uint32_t T1[G1J], T2[G1J];
    {
        const uint32_t* pts[3] = {pB == PT_OK ? Bb : nullptr, pA == PT_OK ? Ab : nullptr, pD == PT_OK ? D : nullptr};
        const uint32_t* ks[3] = {c, ecap, r1cap};
        g1_msm_scalar<C, 3>(T1, pts, ks);
    }
    // T2 = Bv*c + D*r3^ + sum H_undisclosed m^   with Bv*c = K*c + sum H_disclosed (c m)   (:165-182)
    BBS_A16 uint32_t cm[8];
    fe_to_mont<Fr>(cm, c);
    g1_set_inf<C>(T2);
    if (!cx.k_inf) tab_accumulate<C>(T2, cx, 0, c);
    for (uint64_t k = 0; k < R; k++) {
        BBS_A16 uint32_t m[8];
        if (!fr_from_le32<C>(m, a.dis_scalars + (db + k) * 32)) PROOF_FAIL(ST_ERR_MALFORMED)
        fe_mul<Fr>(m, m, cm);                                   // c * m_k, canonical
        tab_accumulate<C>(T2, cx, a.dis_idx[db + k] + 1, m);
    }
    {
        uint64_t k = 0;
        for (uint32_t j = 0; j < (uint32_t)L; j++) {
            if ((mask[j >> 5] >> (j & 31)) & 1) continue;
            BBS_A16 uint32_t m[8];
            if (!fr_from_le32<C>(m, a.commitments + (cb + k) * 32)) PROOF_FAIL(ST_ERR_MALFORMED)
            tab_accumulate<C>(T2, cx, j + 1, m);
            k++;
        }
    }
    if (pD == PT_OK) {
        BBS_A16 uint32_t t[G1J];
        g1_mul_scalar<C>(t, D, r3cap);
        g1_add<C>(T2, T2, t);
    }
    // challenge (proof_gen.rs:272-328)
    Xmd48 x;
    x.begin();
    x.s.put_be64(R);
    for (uint64_t k = 0; k < R; k++) {
        BBS_A16 uint32_t m[8];
        x.s.put_be64(a.dis_idx[db + k]);
        limbs_from_le<8>(m, a.dis_scalars + (db + k) * 32);
        for (int q = 7; q >= 0; q--) x.s.update_words(&m[q], 1);
    }
    x.s.update(pf, 3 * GB);                                     // canonical encodings of Abar, Bbar, D
    {
        // one shared inversion for T1, T2 (Montgomery's trick)
        bool i1 = g1_is_inf_ool<C>(T1), i2 = g1_is_inf_ool<C>(T2);
        BBS_A16 uint32_t z1[FPN], z2[FPN], zz[FPN], t[FPN], aff[G1A];
        uint8_t enc[GB];
        if (i1) fe_set_one<F>(z1); else bn_copy<C::Fp::N>(z1, T1 + 2 * FPN);
        if (i2) fe_set_one<F>(z2); else bn_copy<C::Fp::N>(z2, T2 + 2 * FPN);
        fe_mul<F>(zz, z1, z2); fe_inv<F>(zz, zz);
        fe_mul<F>(t, zz, z2);                                   // 1/z1
        fe_mul<F>(zz, zz, z1);                                  // 1/z2
        fe_sqr<F>(z1, t); fe_mul<F>(aff, T1, z1); fe_mul<F>(z1, z1, t); fe_mul<F>(aff + FPN, T1 + FPN, z1);
        g1_compress_affine<C>(enc, aff, i1); x.s.update(enc, GB);
        fe_sqr<F>(z2, zz); fe_mul<F>(aff, T2, z2); fe_mul<F>(z2, z2, zz); fe_mul<F>(aff + FPN, T2 + FPN, z2);
        g1_compress_affine<C>(enc, aff, i2); x.s.update(enc, GB);
    }
    for (int q = 7; q >= 0; q--) x.s.update_words(&cx.domain[q], 1);
    uint32_t ph_len;
    const uint8_t* ph = item_ph(a.ph, a.ph_len, a.ph_off, i, ph_len);
    x.s.put_be64(ph_len);
    x.s.update(ph, ph_len);
    BBS_A16 uint32_t okm[12], c2[8];
    x.finish(cx.dst_h2s, cx.dst_h2s_len, okm);
    okm48_to_scalar<Fr>(c2, okm);
    if (!bn_eq<8>(c2, c)) PROOF_FAIL(ST_REJECT)                 // proof_verify.rs:108-110: no pairing
    // e(Abar, W) e(Bbar, -BP2) = e(Abar, W) e(-Bbar, BP2)      (proof_verify.rs:112-115)
    uint32_t* pr = a.pair + (size_t)i * PAIR_WORDS;
    bn_copy<2 * C::Fp::N>(pr, Ab); fe_set_one<F>(pr + 2 * FPN);
    bn_copy<C::Fp::N>(pr + 3 * FPN, Bb); fe_neg<F>(pr + 4 * FPN, Bb + FPN); fe_set_one<F>(pr + 5 * FPN);
    uint32_t fl = 0;
    if (pA == PT_INF || cx.w_inf) fl |= FL_SKIP0;
    if (pB == PT_INF) fl |= FL_SKIP1;
    a.flags[i] = fl;
#undef PROOF_FAIL
}

// ---- core_proof_verify, G1 half, as three independent tasks per proof + a join (CUDA build) -----------------------------
// One thread per proof is a serial chain of ~16,500 field multiplications.  Tasks: V1 = the checks of
// proof_verify.rs:139-150, decoding + subgroup tests of Abar, Bbar, D and T1 (~8,400); F = the fixed-base part of T2,
// K*c + sum H_disclosed (c m) + sum H_undisclosed m^ (~5,800); V2 = D * r3^ (~2,500, decodes D again).  The join adds the
// two parts of T2, normalises T1 and T2 with one inversion per block, hashes the challenge and writes the pairing record.
// Statuses are those of proof_g1_item: V1 owns every status of the checks and decodings, F only reports a non-canonical
// message / commitment scalar (the same ERR_MALFORMED), the join owns the challenge comparison.
struct ProofShape { uint64_t cb, U, db, R, L; uint32_t mask[MAX_L / 32]; };
enum : uint8_t { PST_DONE = 0x80 };       // part_st[i]: status final | PT_* of Abar, Bbar, D in bits 0-1, 2-3, 4-5
// the checks of proof_verify.rs:139-150 in the reference's order; 0 = fine, else the status
template <class C> BBS_HD uint8_t proof_shape(const ProofG1Args& a, uint32_t i, ProofShape& s) {
    s.cb = a.commit_off[i]; s.U = a.commit_off[i + 1] - s.cb;
    s.db = a.dis_off[i]; s.R = a.dis_off[i + 1] - s.db;
    s.L = s.R + s.U;
    for (int k = 0; k < MAX_L / 32; k++) s.mask[k] = 0;
    bool dup = false;
    for (uint64_t k = 0; k < s.R; k++) {
        uint32_t idx = a.dis_idx[s.db + k];
        if (idx >= s.L) return ST_ERR_DISCLOSED_INDEX;
        if (idx < MAX_L) { dup |= (s.mask[idx >> 5] >> (idx & 31)) & 1; s.mask[idx >> 5] |= 1u << (idx & 31); }
    }
    if (s.L != a.ctx.L) return ST_ERR_MSG_GEN_LEN;
    if (dup) return ST_ERR_MALFORMED;     // the reference indexes out of bounds and panics (proof_verify.rs:179)
    return 0;
}
// the key-dependent inputs of proof i: K, domain and the identity flags (issuer sets: per item)
template <class C, bool PER_ITEM> BBS_HD uint32_t proof_issuer(const ProofG1Args& a, uint32_t i, const uint32_t*& K, const uint32_t*& domain) {
    K = a.ctx.K; domain = a.ctx.domain;
    if (!a.item_issuer) return item_key<C>(a.ctx, PER_ITEM ? a.item : ItemKeyView{}, i, K, domain);
    const uint32_t s = a.item_issuer[i];
    if (s >= a.iss.n_issuers) return ISS_BAD;
    K = a.iss.K + (size_t)s * G1A; domain = a.iss.domains + (size_t)s * 8;
    return a.iss.flags[s];
}
template <class C, bool PER_ITEM> BBS_HD void proof_task_v1(const ProofG1Args& a, uint32_t i) {
    using F = typename C::Fp;
    constexpr int GB = C::G1_BYTES;
    const uint8_t* pf = a.proofs + (size_t)i * (3 * GB + 128);
    a.part_st[i] = PST_DONE;
    ProofShape sh;
    const uint8_t err = proof_shape<C>(a, i, sh);
    if (err) { a.status[i] = err; a.flags[i] = FL_DONE; return; }
    {
        const uint32_t *Kp, *dom;
        if (proof_issuer<C, PER_ITEM>(a, i, Kp, dom) & ISS_BAD) { a.status[i] = ST_ERR_MALFORMED; a.flags[i] = FL_DONE; return; }   // undecodable issuer key
    }
    BBS_A16 uint32_t Ab[G1A], Bb[G1A], D[G1A], ecap[8], r1cap[8], r3cap[8], c[8];
    int pA = g1_decompress<C>(Ab, pf), pB = g1_decompress<C>(Bb, pf + GB), pD = g1_decompress<C>(D, pf + 2 * GB);
    bool ok = pA != PT_BAD && pB != PT_BAD && pD != PT_BAD;
    ok = ok && fr_from_le32<C>(ecap, pf + 3 * GB) && fr_from_le32<C>(r1cap, pf + 3 * GB + 32) &&
         fr_from_le32<C>(r3cap, pf + 3 * GB + 64) && fr_from_le32<C>(c, pf + 3 * GB + 96);
    if (!ok) { a.status[i] = ST_ERR_MALFORMED; a.flags[i] = FL_DONE; return; }
    // T1 = Bbar*c + Abar*e^ + D*r1^   (proof_verify.rs:163-164)
    {
        BBS_A16 uint32_t T1[G1J];
        const uint32_t* pts[3] = {pB == PT_OK ? Bb : nullptr, pA == PT_OK ? Ab : nullptr, pD == PT_OK ? D : nullptr};
        const uint32_t* ks[3] = {c, ecap, r1cap};
        g1_msm_scalar<C, 3>(T1, pts, ks);
        g1_copy<C>(a.part_t1 + (size_t)i * G1J, T1);
    }
    // e(Abar, W) e(Bbar, -BP2) = e(Abar, W) e(-Bbar, BP2)      (proof_verify.rs:112-115); the join sets the flags
    uint32_t* pr = a.pair + (size_t)i * PAIR_WORDS;
    bn_copy<2 * C::Fp::N>(pr, Ab); fe_set_one<F>(pr + 2 * FPN);
    bn_copy<C::Fp::N>(pr + 3 * FPN, Bb); fe_neg<F>(pr + 4 * FPN, Bb + FPN); fe_set_one<F>(pr + 5 * FPN);
    a.part_st[i] = (uint8_t)(pA | (pB << 2) | (pD << 4));
}
template <class C, bool PER_ITEM> BBS_HD void proof_task_v2(const ProofG1Args& a, uint32_t i) {
    constexpr int GB = C::G1_BYTES;
    const uint8_t* pf = a.proofs + (size_t)i * (3 * GB + 128);
    ProofShape sh;
    if (proof_shape<C>(a, i, sh)) return;
    BBS_A16 uint32_t D[G1A], r3cap[8], t[G1J];
    if (proof_k_variable<PER_ITEM>(a)) {
        // issuer sets / per-item headers: K_i has no window table, so K_i * c joins D * r3^ in one two-point multiplication
        const uint32_t *Kp, *dom;
        const uint32_t ifl = proof_issuer<C, PER_ITEM>(a, i, Kp, dom);
        BBS_A16 uint32_t c[8], Ka[G1A];
        const int pD = g1_decompress<C>(D, pf + 2 * GB);
        if ((ifl & ISS_BAD) || pD == PT_BAD || !fr_from_le32<C>(r3cap, pf + 3 * GB + 64) || !fr_from_le32<C>(c, pf + 3 * GB + 96)) return;
        bn_copy<2 * C::Fp::N>(Ka, Kp);
        const uint32_t* pts[2] = {pD == PT_OK ? D : nullptr, (ifl & ISS_K_INF) ? nullptr : Ka};
        const uint32_t* ks[2] = {r3cap, c};
        g1_msm_scalar<C, 2>(t, pts, ks);
        g1_copy<C>(a.part_v2 + (size_t)i * G1J, t);
        return;
    }
    if (g1_decompress<C>(D, pf + 2 * GB) != PT_OK || !fr_from_le32<C>(r3cap, pf + 3 * GB + 64)) return;   // V1 reports what is wrong
    g1_mul_scalar<C>(t, D, r3cap);
    g1_copy<C>(a.part_v2 + (size_t)i * G1J, t);
}
template <class C, bool PER_ITEM> BBS_HD void proof_task_f(const ProofG1Args& a, uint32_t i, uint8_t* fbad) {
    using Fr = typename C::Fr;
    const CtxView& cx = a.ctx;
    constexpr int GB = C::G1_BYTES;
    const uint8_t* pf = a.proofs + (size_t)i * (3 * GB + 128);
    *fbad = 0;
    ProofShape sh;
    if (proof_shape<C>(a, i, sh)) return;
    BBS_A16 uint32_t c[8], cm[8], T2[G1J];
    if (!fr_from_le32<C>(c, pf + 3 * GB + 96)) return;                                  // V1 reports it
    // Bv*c = K*c + sum H_disclosed (c m), then sum H_undisclosed m^   (proof_verify.rs:165-182)
    fe_to_mont<Fr>(cm, c);
    g1_set_inf<C>(T2);
    if (!proof_k_variable<PER_ITEM>(a) && !cx.k_inf) tab_accumulate<C>(T2, cx, 0, c);    // else K_i * c is part of task V2
    for (uint64_t k = 0; k < sh.R; k++) {
        BBS_A16 uint32_t m[8];
        if (!fr_from_le32<C>(m, a.dis_scalars + (sh.db + k) * 32)) { *fbad = 1; return; }
        fe_mul<Fr>(m, m, cm);                                   // c * m_k, canonical
        tab_accumulate<C>(T2, cx, a.dis_idx[sh.db + k] + 1, m);
    }
    uint64_t k = 0;
    for (uint32_t j = 0; j < (uint32_t)sh.L; j++) {
        if ((sh.mask[j >> 5] >> (j & 31)) & 1) continue;
        BBS_A16 uint32_t m[8];
        if (!fr_from_le32<C>(m, a.commitments + (sh.cb + k) * 32)) { *fbad = 1; return; }
        tab_accumulate<C>(T2, cx, j + 1, m);
        k++;
    }
    g1_copy<C>(a.part_f + (size_t)i * G1J, T2);
}
// join, part 1: T2 = F part (+ V2 part); false when the item's status is already final
template <class C, bool PER_ITEM> BBS_HD bool proof_join_head(const ProofG1Args& a, uint32_t i, const uint8_t* fbad, uint32_t* T1, uint32_t* T2, uint8_t& st) {
    st = a.part_st[i];
    if (st & PST_DONE) return false;
    if (fbad[i]) { a.status[i] = ST_ERR_MALFORMED; a.flags[i] = FL_DONE; return false; }
    g1_copy<C>(T1, a.part_t1 + (size_t)i * G1J);
    g1_copy<C>(T2, a.part_f + (size_t)i * G1J);
    if (((st >> 4) & 3) == PT_OK || proof_k_variable<PER_ITEM>(a)) g1_add<C>(T2, T2, a.part_v2 + (size_t)i * G1J);
    return true;
}
// join, part 2: zinv = 1 / (Z(T1) Z(T2)) with identities counted as Z = 1; challenge (proof_gen.rs:272-328), comparison, flags
template <class C, bool PER_ITEM> BBS_HD void proof_join_tail(const ProofG1Args& a, uint32_t i, const uint32_t* T1, const uint32_t* T2, const uint32_t* zinv, uint8_t st) {
    using F = typename C::Fp;
    using Fr = typename C::Fr;
    const CtxView& cx = a.ctx;
    constexpr int GB = C::G1_BYTES;
    const uint8_t* pf = a.proofs + (size_t)i * (3 * GB + 128);
    const uint64_t db = a.dis_off[i], R = a.dis_off[i + 1] - db;
    const uint32_t *Kp, *domain;
    const uint32_t ifl = proof_issuer<C, PER_ITEM>(a, i, Kp, domain);
    Xmd48 x;
    x.begin();
    x.s.put_be64(R);
    for (uint64_t k = 0; k < R; k++) {
        BBS_A16 uint32_t m[8];
        x.s.put_be64(a.dis_idx[db + k]);
        limbs_from_le<8>(m, a.dis_scalars + (db + k) * 32);
        for (int q = 7; q >= 0; q--) x.s.update_words(&m[q], 1);
    }
    x.s.update(pf, 3 * GB);                                     // canonical encodings of Abar, Bbar, D
    {
        const bool i1 = g1_is_inf_ool<C>(T1), i2 = g1_is_inf_ool<C>(T2);
        BBS_A16 uint32_t z1[FPN], z2[FPN], t[FPN], zz[FPN], aff[G1A];
        uint8_t enc[GB];
        if (i1) fe_set_one<F>(z1); else bn_copy<C::Fp::N>(z1, T1 + 2 * FPN);
        if (i2) fe_set_one<F>(z2); else bn_copy<C::Fp::N>(z2, T2 + 2 * FPN);
        fe_mul<F>(t, zinv, z2);                                 // 1/z1
        fe_mul<F>(zz, zinv, z1);                                // 1/z2
        fe_sqr<F>(z1, t); fe_mul<F>(aff, T1, z1); fe_mul<F>(z1, z1, t); fe_mul<F>(aff + FPN, T1 + FPN, z1);
        g1_compress_affine<C>(enc, aff, i1); x.s.update(enc, GB);
        fe_sqr<F>(z2, zz); fe_mul<F>(aff, T2, z2); fe_mul<F>(z2, z2, zz); fe_mul<F>(aff + FPN, T2 + FPN, z2);
        g1_compress_affine<C>(enc, aff, i2); x.s.update(enc, GB);
    }
    for (int q = 7; q >= 0; q--) x.s.update_words(&domain[q], 1);
    uint32_t ph_len;
    const uint8_t* ph = item_ph(a.ph, a.ph_len, proof_ph_off<PER_ITEM>(a), i, ph_len);
    x.s.put_be64(ph_len);
    x.s.update(ph, ph_len);
    BBS_A16 uint32_t okm[12], c2[8], c[8];
    x.finish(cx.dst_h2s, cx.dst_h2s_len, okm);
    okm48_to_scalar<Fr>(c2, okm);
    limbs_from_le<8>(c, pf + 3 * GB + 96);
    if (!bn_eq<8>(c2, c)) { a.status[i] = ST_REJECT; a.flags[i] = FL_DONE; return; }      // proof_verify.rs:108-110: no pairing
    uint32_t fl = 0;
    if ((st & 3) == PT_INF || (ifl & ISS_W_INF)) fl |= FL_SKIP0;
    if (((st >> 2) & 3) == PT_INF) fl |= FL_SKIP1;
    a.flags[i] = fl;
}

// the join with one inversion per proof (host simulation of proof_g1_join_kernel)
template <class C, bool PER_ITEM> BBS_HD void proof_join_item(const ProofG1Args& a, uint32_t i, const uint8_t* fbad) {
    using F = typename C::Fp;
    BBS_A16 uint32_t T1[G1J], T2[G1J], z[FPN];
    uint8_t st = 0;
    if (!proof_join_head<C, PER_ITEM>(a, i, fbad, T1, T2, st)) return;
    fe_set_one<F>(z);
    if (!g1_is_inf_ool<C>(T1)) bn_copy<C::Fp::N>(z, T1 + 2 * FPN);
    if (!g1_is_inf_ool<C>(T2)) fe_mul<F>(z, z, T2 + 2 * FPN);
    fe_inv<F>(z, z);
    proof_join_tail<C, PER_ITEM>(a, i, T1, T2, z, st);
}

// ---- core_proof_gen (proof_gen.rs:116-365: proof_init, proof_challenge_calculate, proof_finalize) ---------------
// The reference draws its random scalars from the thread RNG (or the mocked stream with feature testvector_bls12_381);
// here the caller supplies them (5 + U per item), which is what makes the output reproducible and comparable.
struct ProofGenArgs {
    CtxView ctx;
    const uint8_t* sigs;           // n x (G1 compressed || LE32 e)
    const uint8_t* scalars;        // n x n_msgs x LE32 message scalars (all messages)
    uint32_t n_msgs;
    const uint32_t* dis_idx;       // flat disclosed indexes
    const uint64_t* dis_off;       // n+1
    const uint8_t* rand;           // flat LE32 random scalars
    const uint64_t* rand_off;      // n+1 (item i owns 5 + U_i scalars)
    const uint64_t* commit_off;    // n+1: where item i's U_i commitments go in commitments_out
    const uint8_t* ph; uint32_t ph_len;
    uint8_t* proofs_out;           // n x (3 G1 compressed || LE32 e^, r1^, r3^, c)
    uint8_t* commitments_out;      // flat LE32
    uint8_t* status;
    ItemKeyView item;              // per-item headers
    const uint64_t* ph_off;        // per-item ph: ph[ph_off[i] .. ph_off[i+1]) (nullptr: shared ph)
};
// PER_ITEM = false: the calls without per-item headers / phs; their kernel is compiled without the per-item reads, which
// cost it spill slots (proof generation runs at the register cap)
template <class C, bool PER_ITEM> BBS_HD void proof_gen_item(const ProofGenArgs& a, uint32_t i) {
    using F = typename C::Fp;
    using Fr = typename C::Fr;
    const CtxView& cx = a.ctx;
    const ItemKeyView item = PER_ITEM ? a.item : ItemKeyView{};
    const uint64_t* ph_off = PER_ITEM ? a.ph_off : nullptr;
    constexpr int GB = C::G1_BYTES;
    const uint64_t L = a.n_msgs;
    const uint64_t db = a.dis_off[i], R = a.dis_off[i + 1] - db;
    const uint64_t rb = a.rand_off[i], NR = a.rand_off[i + 1] - rb;
    const uint64_t cb = a.commit_off[i], U = a.commit_off[i + 1] - cb;
#define GEN_FAIL(code) { a.status[i] = (code); return; }
    if (R > L) GEN_FAIL(ST_ERR_DISCLOSED_LEN)                                   // proof_gen.rs:139-141
    BBS_A16 uint32_t mask[MAX_L / 32];
    for (int k = 0; k < MAX_L / 32; k++) mask[k] = 0;
    uint64_t distinct = 0;
    for (uint64_t k = 0; k < R; k++) {
        uint32_t idx = a.dis_idx[db + k];
        if (idx >= L) GEN_FAIL(ST_ERR_DISCLOSED_INDEX)                          // :143-147
        if (idx < MAX_L && !((mask[idx >> 5] >> (idx & 31)) & 1)) { mask[idx >> 5] |= 1u << (idx & 31); distinct++; }
    }
    if (L != cx.L) GEN_FAIL(ST_ERR_MSG_GEN_LEN)                                 // :228-230
    // the reference de-duplicates the disclosed set (:154-158); its scalar count check is :232-234
    if (NR != (L - distinct) + 5 || U != L - distinct) GEN_FAIL(ST_ERR_RANDOM_LEN)
    const uint8_t* sig = a.sigs + (size_t)i * (GB + 32);
    const uint8_t* sc = a.scalars + (size_t)i * L * 32;
    BBS_A16 uint32_t A[G1A], e[8], rs[5][8];
    int pa = g1_decompress<C>(A, sig);
    bool ok = pa != PT_BAD && fr_from_le32<C>(e, sig + GB);
    for (int k = 0; k < 5 && ok; k++) ok = fr_from_le32<C>(rs[k], a.rand + (rb + k) * 32);
    if (!ok) GEN_FAIL(ST_ERR_MALFORMED)
    // B = P1 + Q1*domain + sum H_j m_j   (:247-253)
    BBS_A16 uint32_t B[G1J];
    {
        const uint32_t *Kp, *domain;
        if (item_key<C>(cx, item, i, Kp, domain) & ISS_K_INF) g1_set_inf<C>(B); else g1_from_affine<C>(B, Kp);
    }
    for (uint32_t j = 0; j < (uint32_t)L; j++) {
        BBS_A16 uint32_t m[8];
        if (!fr_from_le32<C>(m, sc + j * 32)) GEN_FAIL(ST_ERR_MALFORMED)
        tab_accumulate<C>(B, cx, j + 1, m);
    }
    // D = B r1 ; Abar = A (r0 r1)   (:254-255)
    BBS_A16 uint32_t r0m[8], r01[8], Baff[G1A], Dj[G1J], Abj[G1J];
    fe_to_mont<Fr>(r0m, rs[0]);
    fe_mul<Fr>(r01, r0m, rs[1]);                               // r0 r1, canonical
    bool bfin = g1_to_affine<C>(Baff, B);
    if (bfin) g1_mul_scalar<C>(Dj, Baff, rs[1]); else g1_set_inf<C>(Dj);
    if (pa == PT_OK) g1_mul_scalar<C>(Abj, A, r01); else g1_set_inf<C>(Abj);
    // normalise D and Abar with one inversion (they are multiplied again and serialised)
    BBS_A16 uint32_t Daff[G1A], Abaff[G1A];
    bool dfin = !g1_is_inf_ool<C>(Dj), afin = !g1_is_inf_ool<C>(Abj);
    {
        BBS_A16 uint32_t z1[FPN], z2[FPN], zz[FPN], t[FPN];
        if (dfin) bn_copy<C::Fp::N>(z1, Dj + 2 * FPN); else fe_set_one<F>(z1);
        if (afin) bn_copy<C::Fp::N>(z2, Abj + 2 * FPN); else fe_set_one<F>(z2);
        fe_mul<F>(zz, z1, z2); fe_inv<F>(zz, zz);
        fe_mul<F>(t, zz, z2);                                   // 1/z1
        fe_mul<F>(zz, zz, z1);                                  // 1/z2
        fe_sqr<F>(z1, t); fe_mul<F>(Daff, Dj, z1); fe_mul<F>(z1, z1, t); fe_mul<F>(Daff + FPN, Dj + FPN, z1);
        fe_sqr<F>(z2, zz); fe_mul<F>(Abaff, Abj, z2); fe_mul<F>(z2, z2, zz); fe_mul<F>(Abaff + FPN, Abj + FPN, z2);
    }
    // Bbar = D r0 - Abar e ; T1 = Abar r2 + D r3   (:256-257)
    BBS_A16 uint32_t ne[8], Bbj[G1J], T1[G1J], T2[G1J];
    fe_neg<Fr>(ne, e);
    const uint32_t* pts[2] = {dfin ? Daff : nullptr, afin ? Abaff : nullptr};
    {
        const uint32_t* ks[2] = {rs[0], ne};
        g1_msm_scalar<C, 2>(Bbj, pts, ks);
        const uint32_t* kt[2] = {rs[3], rs[2]};
        g1_msm_scalar<C, 2>(T1, pts, kt);
    }
    // T2 = D r4 + sum_{undisclosed} H_j r_{5+k}   (:258-263)
    if (dfin) g1_mul_scalar<C>(T2, Daff, rs[4]); else g1_set_inf<C>(T2);
    {
        uint64_t k = 0;
        for (uint32_t j = 0; j < (uint32_t)L; j++) {
            if ((mask[j >> 5] >> (j & 31)) & 1) continue;
            BBS_A16 uint32_t m[8];
            if (!fr_from_le32<C>(m, a.rand + (rb + 5 + k) * 32)) GEN_FAIL(ST_ERR_MALFORMED)
            tab_accumulate<C>(T2, cx, j + 1, m);
            k++;
        }
    }
    // serialise Bbar, T1, T2 with one shared inversion
    uint8_t* out = a.proofs_out + (size_t)i * (3 * GB + 128);
    uint8_t encT1[GB], encT2[GB];
    {
        uint32_t* P[3] = {Bbj, T1, T2};
        bool inf[3];
        BBS_A16 uint32_t z[3][FPN], pre[3][FPN], inv[FPN], t[FPN], aff[G1A];
        for (int k = 0; k < 3; k++) {
            inf[k] = g1_is_inf_ool<C>(P[k]);
            if (inf[k]) fe_set_one<F>(z[k]); else bn_copy<C::Fp::N>(z[k], P[k] + 2 * FPN);
        }
        bn_copy<C::Fp::N>(pre[0], z[0]);
        fe_mul<F>(pre[1], pre[0], z[1]);
        fe_mul<F>(pre[2], pre[1], z[2]);
        fe_inv<F>(inv, pre[2]);
        for (int k = 2; k >= 0; k--) {
            BBS_A16 uint32_t zi[FPN], zi2[FPN];
            if (k > 0) { fe_mul<F>(zi, inv, pre[k - 1]); fe_mul<F>(t, inv, z[k]); bn_copy<C::Fp::N>(inv, t); }
            else bn_copy<C::Fp::N>(zi, inv);
            fe_sqr<F>(zi2, zi); fe_mul<F>(aff, P[k], zi2); fe_mul<F>(zi2, zi2, zi); fe_mul<F>(aff + FPN, P[k] + FPN, zi2);
            uint8_t* dst = k == 0 ? out + GB : (k == 1 ? encT1 : encT2);
            g1_compress_affine<C>(dst, aff, inf[k]);
        }
    }
    g1_compress_affine<C>(out, Abaff, !afin);
    g1_compress_affine<C>(out + 2 * GB, Daff, !dfin);
    // challenge (:272-328): disclosed indexes sorted and de-duplicated (:154-158), messages looked up by index (:186-189)
    Xmd48 x;
    x.begin();
    x.s.put_be64(distinct);
    for (uint32_t j = 0; j < (uint32_t)L; j++) {
        if (!((mask[j >> 5] >> (j & 31)) & 1)) continue;
        BBS_A16 uint32_t m[8];
        x.s.put_be64(j);
        limbs_from_le<8>(m, sc + j * 32);
        for (int q = 7; q >= 0; q--) x.s.update_words(&m[q], 1);
    }
    x.s.update(out, 3 * GB);
    x.s.update(encT1, GB);
    x.s.update(encT2, GB);
    const uint32_t* domain = item_domain<C>(cx, item, i);
    for (int q = 7; q >= 0; q--) x.s.update_words(&domain[q], 1);
    uint32_t ph_len;
    const uint8_t* ph = item_ph(a.ph, a.ph_len, ph_off, i, ph_len);
    x.s.put_be64(ph_len);
    x.s.update(ph, ph_len);
    BBS_A16 uint32_t okm[12], c[8], cm[8];
    x.finish(cx.dst_h2s, cx.dst_h2s_len, okm);
    okm48_to_scalar<Fr>(c, okm);
    fe_to_mont<Fr>(cm, c);
    // proof_finalize (:331-365)
    BBS_A16 uint32_t r1m[8], r3[8], t[8], v[8];
    if (bn_is_zero<8>(rs[1])) GEN_FAIL(ST_ERR_MALFORMED)                       // :347 `inverse().unwrap()` panics
    fe_to_mont<Fr>(r1m, rs[1]); fe_inv<Fr>(r1m, r1m); fe_from_mont<Fr>(r3, r1m);
    fe_mul<Fr>(t, cm, e); fe_add<Fr>(v, rs[2], t); limbs_to_le<8>(out + 3 * GB, v);             // e^ = r2 + e c
    fe_mul<Fr>(t, cm, rs[0]); fe_sub<Fr>(v, rs[3], t); limbs_to_le<8>(out + 3 * GB + 32, v);     // r1^ = r3 - r0 c
    fe_mul<Fr>(t, cm, r3); fe_sub<Fr>(v, rs[4], t); limbs_to_le<8>(out + 3 * GB + 64, v);        // r3^ = r4 - c / r1
    limbs_to_le<8>(out + 3 * GB + 96, c);
    {
        uint64_t k = 0;
        for (uint32_t j = 0; j < (uint32_t)L; j++) {
            if ((mask[j >> 5] >> (j & 31)) & 1) continue;
            BBS_A16 uint32_t m[8], rk[8];
            limbs_from_le<8>(m, sc + j * 32);
            limbs_from_le<8>(rk, a.rand + (rb + 5 + k) * 32);
            fe_mul<Fr>(t, cm, m); fe_add<Fr>(v, rk, t);                                          // m^ = r_{5+k} + m c
            limbs_to_le<8>(a.commitments_out + (cb + k) * 32, v);
            k++;
        }
    }
    a.status[i] = ST_ACCEPT;
#undef GEN_FAIL
}

#if defined(__CUDACC__) && !defined(BBS_HOSTSIM)
// 3 * nb blocks: V1 for items [0, n), then F, then V2 (longest tasks first)
// PER_ITEM = false (no per-item headers or phs): the per-item reads are compiled out, as in sign_kernel
template <class C, int TPB, int MINB, bool PER_ITEM> __global__ void __launch_bounds__(TPB, MINB)
proof_g1_split_kernel(const ProofG1Args a, uint32_t n, uint32_t nb, uint8_t* fbad) {
    const uint32_t kind = blockIdx.x / nb;
    const uint32_t i = (blockIdx.x - kind * nb) * TPB + threadIdx.x;
    if (i >= n) return;
    if (kind == 0) proof_task_v1<C, PER_ITEM>(a, i); else if (kind == 1) proof_task_f<C, PER_ITEM>(a, i, fbad + i); else proof_task_v2<C, PER_ITEM>(a, i);
}
template <class C, int TPB, bool PER_ITEM> __global__ void __launch_bounds__(TPB, 4) proof_g1_join_kernel(const ProofG1Args a, uint32_t n,
                                                                                            const uint8_t* fbad) {
    using F = typename C::Fp;
    __shared__ BBS_A16 uint32_t tree[2 * TPB][C::Fp::N];
    const uint32_t i = blockIdx.x * TPB + threadIdx.x;
    BBS_A16 uint32_t T1[G1J], T2[G1J], z[FPN];
    uint8_t st = 0;
    const bool live = i < n && proof_join_head<C, PER_ITEM>(a, i, fbad, T1, T2, st);
    fe_set_one<F>(z);
    if (live) {
        if (!g1_is_inf_ool<C>(T1)) bn_copy<C::Fp::N>(z, T1 + 2 * FPN);
        if (!g1_is_inf_ool<C>(T2)) fe_mul<F>(z, z, T2 + 2 * FPN);
    }
    block_batch_inverse<F, TPB, true>(z, tree);
    if (live) proof_join_tail<C, PER_ITEM>(a, i, T1, T2, z, st);
}
#endif

}  // namespace bbs
