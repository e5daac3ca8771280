// C ABI (include/bbs_b200.h) of the B200 batch engine.  Host code here only moves bytes and enqueues
// kernels; every field / curve / pairing / hash operation of the path runs on the GPU (kernels.cuh).
#include "../../include/bbs_b200.h"
#include "launchers.cuh"

#include <algorithm>
#include <new>
#include <string>
#include <vector>

using namespace bbs;

namespace {

constexpr int TPB_HEAVY = 128;   // G1 / pairing kernels
constexpr int TPB_LIGHT = 128;   // hashing

// CUDA events on the launching stream: mark k sits before kernel k of a batch call (last mark = end)
struct ProfEvents {
    static constexpr int MAX = 10;
#ifndef BBS_HOSTSIM
    cudaEvent_t ev[MAX] = {};
    int used = 0;
    // the per-item domain kernel of a bbs_*_hdr call is timed by its own pair of events and reported in slot xslot, after
    // the call's other slots; every call's chain of marks starts at slot 0 or 1, which forgets the previous call's xslot
    cudaEvent_t xev[2] = {};
    int xslot = -1;
    int mark(int slot, rt_stream_t s) {
        if (slot >= MAX) return 0;
        if (slot <= 1) xslot = -1;
        if (!ev[slot]) RT_CHECK(cudaEventCreate(&ev[slot]));
        RT_CHECK(cudaEventRecord(ev[slot], s));
        used = slot + 1;
        return 0;
    }
    int read(float* ms, int n) {
        for (int i = 0; i < n; i++) ms[i] = 0.f;
        for (int i = 0; i + 1 < used && i < n; i++) {
            if (!ev[i] || !ev[i + 1]) continue;       // slot never marked by the last call (e.g. no hashing kernel)
            RT_CHECK(cudaEventSynchronize(ev[i + 1]));
            RT_CHECK(cudaEventElapsedTime(&ms[i], ev[i], ev[i + 1]));
        }
        if (xslot >= 0 && xslot < n && xev[0] && xev[1]) {
            RT_CHECK(cudaEventSynchronize(xev[1]));
            RT_CHECK(cudaEventElapsedTime(&ms[xslot], xev[0], xev[1]));
        }
        return 0;
    }
    int mark_extra(int k, rt_stream_t s) {
        if (!xev[k]) RT_CHECK(cudaEventCreate(&xev[k]));
        RT_CHECK(cudaEventRecord(xev[k], s));
        return 0;
    }
    void release() {
        for (auto& e : ev) if (e) { cudaEventDestroy(e); e = nullptr; }
        for (auto& e : xev) if (e) { cudaEventDestroy(e); e = nullptr; }
    }
#else
    int xslot = -1;
    int mark(int, rt_stream_t) { return 0; }
    int mark_extra(int, rt_stream_t) { return 0; }
    int read(float* ms, int n) { for (int i = 0; i < n; i++) ms[i] = 0.f; return 0; }
    void release() {}
#endif
};

struct Ctx {
    int curve = 0, device = 0;
    uint32_t L = 0;
    size_t api_id_len = 0, header_len = 0;
    rt_stream_t stream = nullptr;
#ifndef BBS_HOSTSIM
    cudaStream_t copy_stream = nullptr;        // uploads of the chunked host-buffer paths (rlc): overlap with compute
    cudaEvent_t copy_done[8] = {};
    cudaStream_t down_stream = nullptr;        // downloads of the chunked signing path
    cudaEvent_t comp_done[8] = {};
#endif
    uint64_t launches = 0;
    bool profile = false;            // bbs_ctx_set_profiling: CUDA events around each kernel of a batch call
    ProfEvents prof;
    DevBuf pk_comp, gens_comp, api_id, header, dst_h2s, dst_map;
    DevBuf gens, W, K, domain, tab, wbase, lines, lines_coop, misc, prefix;
    bool coop = false;               // cooperative pairing kernel usable (no degenerate line)
    bool force_per_thread = false;   // bbs_ctx_use_per_thread_pairing: the fallback kernel on request (tests)
    bool per_item_header = false;    // BBS_CTX_PER_ITEM_HEADER: Q1 table in slot L + 1 and the domain prefix state in `prefix`
    uint32_t rlc_windows = 0;        // bbs_ctx_set_rlc_windows: digits per 128-bit value of the bucket MSM (0 = cost model)
    CtxView view{};
    // grow-only scratch for the batch calls
    DevBuf s_rand, s_rand_off, s_sk, s_g1v, s_g1f, s_g1st, s_g1t;
    size_t split_max = 0;            // batches up to this size take the two-task G1 path (bbs_ctx_set_g1_split)
    uint32_t pair_split_max = 32;    // batches up to this size (<= 32) run the pairing with two warps per role (bbs_ctx_set_pairing_split)
    DevBuf s_gscr, s_rlc_pt, s_rlc_sc, s_rlc_parts, s_rlc_bad, s_msm_pts, s_msm_kv, s_msm_idx, s_msm_entries, s_msm_buckets;
    DevBuf s_sigs, s_scalars, s_msgs, s_offsets, s_pair, s_flags, s_status, s_out, s_out2;
    DevBuf s_commit, s_commit_off, s_dis_idx, s_dis_scalars, s_dis_off, s_ph, s_dis_msgs, s_dis_msg_off;
    DevBuf s_hdr, s_hdr_off, s_ph_off, s_ik, s_idom, s_ifl;     // per-item headers / phs and the ItemKeyView arrays
    DevBuf s_rlcp;                   // rlc proof calls: the combined pairing record, its flag word and its status
    template <class Fn> void each_buffer(Fn f) {
        DevBuf* all[] = {&pk_comp, &gens_comp, &api_id, &header, &dst_h2s, &dst_map, &gens, &W, &K, &domain, &tab, &wbase,
                         &lines, &lines_coop, &s_rand, &s_rand_off, &s_sk, &s_g1v, &s_g1f, &s_g1st, &s_g1t, &s_gscr, &s_rlc_pt, &s_rlc_sc, &s_rlc_parts, &s_rlc_bad, &s_msm_pts, &s_msm_kv, &s_msm_idx, &s_msm_entries, &s_msm_buckets, &misc, &s_sigs, &s_scalars, &s_msgs, &s_offsets, &s_pair, &s_flags, &s_status, &s_out,
                         &s_out2, &s_commit, &s_commit_off, &s_dis_idx, &s_dis_scalars, &s_dis_off, &s_ph, &s_dis_msgs,
                         &s_dis_msg_off, &prefix, &s_hdr, &s_hdr_off, &s_ph_off, &s_ik, &s_idom, &s_ifl, &s_rlcp};
        for (DevBuf* b : all) f(b);
    }
    void release_all() { each_buffer([](DevBuf* b) { b->release(); }); }
    size_t bytes() { size_t t = 0; each_buffer([&](DevBuf* b) { t += b->cap; }); return t; }
};

// Many issuer keys over one generator list (bbs_issuer_set_create): `base` owns everything the issuers share -- decoded
// generators, the fixed-base tables of H_1..H_L, the BP2 lines, the batch scratch and the stream (its own key is the
// identity and is never used) -- and the arrays below hold what depends on the key, ~26 KB per issuer on BLS12-381.
struct IssuerSet {
    Ctx* base = nullptr;
    size_t n_issuers = 0;
    uint32_t line_stride = 0;        // words between two issuers' line tables
    DevBuf pks, W, K, domains, flags, lines, item_issuer;
    size_t per_issuer_bytes() const { return pks.cap + W.cap + K.cap + domains.cap + flags.cap + lines.cap; }
    void release_all() { for (DevBuf* b : {&pks, &W, &K, &domains, &flags, &lines, &item_issuer}) b->release(); }
    IssuerSetView view() const {
        return IssuerSetView{(const uint32_t*)K.p, (const uint32_t*)flags.p, (const uint32_t*)lines.p, line_stride,
                             (uint32_t)n_issuers, (const uint32_t*)domains.p};
    }
};

// The messages of a host-buffer batch call: byte messages `msgs` with their count + 1 offsets `off`, or (off == nullptr)
// their scalars, 32 bytes each
struct MsgIn { const uint8_t* scalars; const uint8_t* msgs; const uint64_t* off; };

// The random-linear-combination form of a call with per-item statuses (bbs_rlc_*proof_verify_batch*,
// bbs_rlc_*verify_batch_status*): the 32-byte coefficient seed and where the combined check's verdict goes (may be null)
struct RlcProofIn { const uint8_t* seed; uint8_t* combined; };

#define TRY(expr) do { int rc_ = (expr); if (rc_) return rc_; } while (0)
#define PROF(c, slot, s) do { if ((c)->profile) TRY((c)->prof.mark(slot, s)); } while (0)

int arg_error(const char* what) { rt_set_error("bad argument", what); return BBS_E_ARG; }

// The kernels index items and flat message slots with 32-bit counters.
bool counts_fit(size_t n, size_t per_item) {
    if (n > 0xffffffffull) return false;
    return per_item == 0 || n <= 0xffffffffull / per_item;
}
// Per-item byte strings (headers, phs): n + 1 offsets that never decrease, each item shorter than 2^28 bytes so that every
// hash input built from one stays below the 2^29 bytes that Sha256 counts.
constexpr uint64_t MAX_ITEM_BYTES = 1ull << 28;
int check_items(size_t n, const uint8_t* bytes, const uint64_t* off, const char* what) {
    for (size_t i = 0; i < n; i++) {
        if (off[i + 1] < off[i]) { rt_set_error("bad argument", (std::string(what) + " offsets decrease").c_str()); return BBS_E_ARG; }
        if (off[i + 1] - off[i] >= MAX_ITEM_BYTES) {
            rt_set_error("bad argument", (std::string(what) + " longer than 2^28 bytes").c_str());
            return BBS_E_ARG;
        }
    }
    if (off[n] != off[0] && !bytes) return arg_error("null per-item byte strings");
    return BBS_OK;
}
#define CHECK_COUNTS(n, per_item) do { if (!counts_fit((n), (per_item))) return arg_error("batch too large: n and n * n_msgs must fit in 32 bits"); } while (0)

template <class C>
struct Impl {
    static constexpr size_t SIG = C::G1_BYTES + 32;
    static constexpr size_t PROOF = 3 * C::G1_BYTES + 128;

    static int create(Ctx* c, const uint8_t* pk, const uint8_t* gens, uint32_t n_gens, const uint8_t* header,
                      size_t header_len, const uint8_t* api_id, size_t api_id_len, uint32_t flags) {
        const TabGeom G((flags & BBS_CTX_SMALL_TABLES) ? (uint32_t)TAB_BITS_SMALL : (uint32_t)BBS_TAB_BITS_GLV);
        const uint32_t L = n_gens - 1;
        const bool per_item = (flags & BBS_CTX_PER_ITEM_HEADER) != 0;
        const uint32_t n_tabs = per_item ? L + 2 : L + 1;        // K, H_1..H_L (, Q1)
        c->L = L;
        c->api_id_len = api_id_len; c->header_len = header_len;
        rt_stream_t s = c->stream;
        std::vector<uint8_t> dsth(api_id, api_id + api_id_len), dstm(api_id, api_id + api_id_len);
        const char* h2s = "H2S_";                            // verify.rs / core_utilities.rs:60
        const char* map = "MAP_MSG_TO_SCALAR_AS_HASH_";      // interface_utilities.rs:82
        dsth.insert(dsth.end(), h2s, h2s + 4);
        dstm.insert(dstm.end(), map, map + 26);
        if (dstm.size() > 255) return arg_error("dst size is invalid (api_id too long; utilities_helper.rs:50-52)");
        TRY(c->pk_comp.reserve(C::G2_BYTES));
        TRY(c->gens_comp.reserve((size_t)n_gens * C::G1_BYTES));
        TRY(c->api_id.reserve(api_id_len));
        TRY(c->header.reserve(header_len));
        TRY(c->dst_h2s.reserve(dsth.size()));
        TRY(c->dst_map.reserve(dstm.size()));
        TRY(c->gens.reserve((size_t)n_gens * 2 * C::Fp::N * 4));
        TRY(c->W.reserve(4 * C::Fp::N * 4));
        TRY(c->K.reserve(2 * C::Fp::N * 4));
        TRY(c->domain.reserve(32));
        TRY(c->misc.reserve((n_gens + 2) * 4));
        if (per_item) TRY(c->prefix.reserve(SHA_STATE_WORDS * 4));
        const size_t tab_entries = (size_t)n_tabs * G.windows * G.entries;
        TRY(c->tab.reserve(tab_entries * 2 * C::Fp::N * 4));
        const int n_lines = ate_line_count<C>();
        TRY(c->lines.reserve((size_t)n_lines * 2 * 4 * C::Fp::N * 4));
        TRY(rt_h2d(c->pk_comp.p, pk, C::G2_BYTES, s));
        TRY(rt_h2d(c->gens_comp.p, gens, (size_t)n_gens * C::G1_BYTES, s));
        TRY(rt_h2d(c->api_id.p, api_id, api_id_len, s));
        TRY(rt_h2d(c->header.p, header, header_len, s));
        TRY(rt_h2d(c->dst_h2s.p, dsth.data(), dsth.size(), s));
        TRY(rt_h2d(c->dst_map.p, dstm.data(), dstm.size(), s));
        TRY(rt_memset(c->lines.p, 0, (size_t)n_lines * 2 * 4 * C::Fp::N * 4, s));
        uint32_t* d_status = (uint32_t*)c->misc.p;
        // 1. decode generators and public key
        CtxDecodeArgs da{(const uint8_t*)c->gens_comp.p, (const uint8_t*)c->pk_comp.p, n_gens, (uint32_t*)c->gens.p,
                         (uint32_t*)c->W.p, d_status};
        TRY((launch_ctx_decode<C>(da, n_gens + 1, s)));
        std::vector<uint32_t> st(n_gens + 2);
        TRY(rt_d2h(st.data(), d_status, (n_gens + 1) * 4, s));
        TRY(rt_sync(s));
        for (uint32_t j = 0; j < n_gens; j++)
            if (st[j] != PT_OK) return arg_error("generator is not a valid non-identity G1 encoding");
        if (st[n_gens] == PT_BAD) return arg_error("public key is not a valid G2 encoding");
        const uint32_t w_inf = st[n_gens] == PT_INF;
        // 2. domain and K
        uint32_t* d_kinf = d_status + n_gens + 1;
        CtxDomainArgs dom{(const uint8_t*)c->pk_comp.p, (const uint8_t*)c->gens_comp.p, L,
                          (const uint8_t*)c->api_id.p, (uint32_t)api_id_len, (const uint8_t*)c->header.p,
                          (uint32_t)header_len, (const uint8_t*)c->dst_h2s.p, (uint32_t)dsth.size(),
                          (const uint32_t*)c->gens.p, (uint32_t*)c->domain.p, (uint32_t*)c->K.p, d_kinf,
                          per_item ? (uint32_t*)c->prefix.p : nullptr};
        TRY((launch_ctx_domain<C>(dom, 1, s)));
        uint32_t k_inf = 0;
        TRY(rt_d2h(&k_inf, d_kinf, 4, s));
        TRY(rt_sync(s));
        // 3. window tables, 4. line tables
        TRY(c->wbase.reserve((size_t)n_tabs * G.windows * 2 * C::Fp::N * 4));
        CtxTableArgs ta{(const uint32_t*)c->K.p, (const uint32_t*)c->gens.p, (uint32_t*)c->tab.p, (uint32_t*)c->wbase.p,
                        (uint32_t)G.bits, per_item ? L + 1 : 0u};
        TRY((launch_ctx_table<C>(ta, n_tabs, s)));
        CtxLinesArgs la{(const uint32_t*)c->W.p, w_inf, (uint32_t*)c->lines.p};
        TRY((launch_ctx_lines<C>(la, 2, s)));
        TRY(rt_sync(s));
        c->launches += 4;
        // 5. normalised line table of the cooperative pairing kernel
        c->coop = false;
#ifndef BBS_HOSTSIM
        {
            TRY(c->lines_coop.reserve((size_t)n_lines * 2 * 4 * C::Fp::N * 4));
            uint32_t* d_deg = d_status;
            TRY(rt_memset(d_deg, 0, 4, s));
            CtxLinesCoopArgs lc{(const uint32_t*)c->lines.p, (uint32_t*)c->lines_coop.p, d_deg, w_inf};
            TRY((launch_ctx_lines_coop<C>(lc, (uint32_t)(2 * n_lines), s)));
            uint32_t deg = 0;
            TRY(rt_d2h(&deg, d_deg, 4, s));
            TRY(rt_sync(s));
            c->launches += 1;
            c->coop = deg == 0;
        }
#endif
        CtxView& v = c->view;
        v.L = L; v.w_inf = w_inf; v.k_inf = k_inf; v.tab_bits = (uint32_t)G.bits;
        v.dst_h2s = (const uint8_t*)c->dst_h2s.p; v.dst_h2s_len = (uint32_t)dsth.size();
        v.dst_map = (const uint8_t*)c->dst_map.p; v.dst_map_len = (uint32_t)dstm.size();
        v.gens = (const uint32_t*)c->gens.p; v.W = (const uint32_t*)c->W.p; v.K = (const uint32_t*)c->K.p;
        v.domain = (const uint32_t*)c->domain.p; v.tab = (const uint32_t*)c->tab.p;
        v.lines = (const uint32_t*)c->lines.p;
        c->per_item_header = per_item;
#ifndef BBS_HOSTSIM
        c->split_max = (size_t)-1;       // the two-task G1 path is faster at every batch size measured (DESIGN 4.2)
#endif
        return BBS_OK;
    }

    static int h2s_dev(Ctx* c, size_t count, const uint8_t* d_msgs, const uint64_t* d_off, uint8_t* d_out, rt_stream_t s) {
        H2sArgs a{d_msgs, d_off, c->view.dst_map, c->view.dst_map_len, d_out};
        TRY((launch_h2s<C>(a, (uint32_t)count, s)));
        c->launches += count ? 1 : 0;
        return BBS_OK;
    }

    // S != nullptr: multi-issuer batch, item i is checked against the lines of issuer d_item_issuer[i] of the set.
    // The records and flags are the batch's (s_pair, s_flags) unless d_pair / d_flags name others.
    static int pairing_dev(Ctx* c, size_t n, uint8_t* d_status, rt_stream_t s, const IssuerSet* S = nullptr,
                           const uint32_t* d_pair = nullptr, const uint32_t* d_flags = nullptr) {
        const uint32_t* d_issuer = S ? (const uint32_t*)S->item_issuer.p : nullptr;
        if (!d_pair) { d_pair = (const uint32_t*)c->s_pair.p; d_flags = (const uint32_t*)c->s_flags.p; }
#ifndef BBS_HOSTSIM
        if (S || (c->coop && !c->force_per_thread)) {
            TRY(c->s_gscr.reserve(coop_gscratch_size<C>(n)));
            CoopArgs ca{(const uint32_t*)(S ? S->lines.p : c->lines_coop.p), d_pair, d_flags, d_status, (uint32_t*)c->s_gscr.p, (uint32_t)n, d_issuer,
                        S ? S->line_stride : 0u, c->pair_split_max};
            TRY((launch_pairing_coop<C>(ca, s)));
            c->launches += n ? 1 : 0;
            return BBS_OK;
        }
#endif
        PairingArgs pa{S ? (const uint32_t*)S->lines.p : c->view.lines, d_pair, d_flags, d_status, d_issuer,
                       S ? S->line_stride : 0u};
        TRY((launch_pairing<C>(pa, (uint32_t)n, s)));
        c->launches += n ? 1 : 0;
        return BBS_OK;
    }

    // G1 half of core_verify for items [first, first + n) of a batch whose pair records / flags / statuses are indexed by the
    // batch (scratch of the task split is per launch: reserve it for the largest launch BEFORE a chunked sequence starts)
    static int verify_g1_dev(Ctx* c, size_t n, size_t first, const uint8_t* d_sigs, const uint8_t* d_scalars, uint32_t n_msgs,
                             uint8_t* d_status, rt_stream_t s, const IssuerSet* S = nullptr, const ItemKeyView* item = nullptr) {
        VerifyG1Args a{c->view, d_sigs + first * SIG, d_scalars + first * n_msgs * 32, n_msgs,
                       (uint32_t*)c->s_pair.p + first * 6 * C::Fp::N, (uint32_t*)c->s_flags.p + first, d_status + first};
        if (n <= c->split_max) {
            TRY(c->s_g1v.reserve(n * 3 * C::Fp::N * 4));
            TRY(c->s_g1f.reserve(n * 3 * C::Fp::N * 4));
            TRY(c->s_g1st.reserve(2 * n));
            a.part_v = (uint32_t*)c->s_g1v.p; a.part_f = (uint32_t*)c->s_g1f.p; a.part_st = (uint8_t*)c->s_g1st.p;
        }
        if (S) {
            a.item_issuer = (const uint32_t*)S->item_issuer.p + first;
            a.iss = S->view();
        }
        if (item) a.item = ItemKeyView{item->K + first * 2 * C::Fp::N, item->domains + first * 8, item->flags + first};
        TRY((launch_verify_g1<C>(a, (uint32_t)n, s)));
        c->launches += n ? (a.part_v ? 2 : 1) : 0;
        return BBS_OK;
    }
    static int core_verify_dev(Ctx* c, size_t n, const uint8_t* d_sigs, const uint8_t* d_scalars, uint32_t n_msgs,
                               uint8_t* d_status, rt_stream_t s, const IssuerSet* S = nullptr, const ItemKeyView* item = nullptr) {
        TRY(c->s_pair.reserve(n * 6 * C::Fp::N * 4));
        TRY(c->s_flags.reserve(n * 4));
        PROF(c, 1, s);
        TRY(verify_g1_dev(c, n, 0, d_sigs, d_scalars, n_msgs, d_status, s, S, item));
        PROF(c, 2, s);
        TRY(pairing_dev(c, n, d_status, s, S));
        PROF(c, 3, s);
        if (item) c->prof.xslot = 3;
        return BBS_OK;
    }

    // ---- per-item headers (bbs_*_hdr) ----------------------------------------------------------------------
    // domain_i, K_i and the K_i-is-identity flags of items [0, n) into the call's scratch; `item` is what the consumers read
    static int item_keys_dev(Ctx* c, size_t n, const uint8_t* d_headers, const uint64_t* d_hdr_off, ItemKeyView& item,
                             rt_stream_t s) {
        TRY(c->s_ik.reserve(n * 2 * C::Fp::N * 4));
        TRY(c->s_idom.reserve(n * 32));
        TRY(c->s_ifl.reserve(n * 4));
        ItemDomainArgs a{c->view, (const uint32_t*)c->prefix.p, d_headers, d_hdr_off, (uint32_t*)c->s_idom.p,
                         (uint32_t*)c->s_ik.p, (uint32_t*)c->s_ifl.p};
        if (c->profile) TRY(c->prof.mark_extra(0, s));
        TRY((launch_item_domain<C>(a, (uint32_t)n, s)));
        if (c->profile) TRY(c->prof.mark_extra(1, s));
        c->launches += n ? 1 : 0;
        item = ItemKeyView{(const uint32_t*)c->s_ik.p, (const uint32_t*)c->s_idom.p, (const uint32_t*)c->s_ifl.p};
        return BBS_OK;
    }
    // host headers staged, then item_keys_dev
    static int item_keys(Ctx* c, size_t n, const uint8_t* headers, const uint64_t* hdr_off, ItemKeyView& item) {
        TRY(stage(c->s_hdr, headers, hdr_off[n], c->stream));
        TRY(stage(c->s_hdr_off, hdr_off, (n + 1) * 8, c->stream));
        return item_keys_dev(c, n, (const uint8_t*)c->s_hdr.p, (const uint64_t*)c->s_hdr_off.p, item, c->stream);
    }
    static int core_verify_hdr_dev(Ctx* c, size_t n, const uint8_t* d_sigs, const uint8_t* d_scalars, uint32_t n_msgs,
                                   const uint8_t* d_headers, const uint64_t* d_hdr_off, uint8_t* d_status, rt_stream_t s) {
        ItemKeyView item{};
        TRY(item_keys_dev(c, n, d_headers, d_hdr_off, item, s));
        return core_verify_dev(c, n, d_sigs, d_scalars, n_msgs, d_status, s, nullptr, &item);
    }
#ifndef BBS_HOSTSIM
    // ---- chunked host-buffer pipelines (verify, sign, rlc) ----------------------------------------------------------
    // Bounds of up to 8 chunks covering [0, n): chunks of `first` items, or (doubling) of sizes doubling from `first`, where
    // a remainder below `first` and everything past the 8th chunk joins the last chunk.  Returns the number of chunks.
    static int plan_chunks(size_t n, size_t first, bool doubling, size_t bounds[9]) {
        int k = 0;
        bounds[0] = 0;
        for (size_t at = 0, cur = first; at < n; cur = doubling ? 2 * cur : cur) {
            size_t take = std::min(n - at, cur);
            if (doubling && (n - at - take < first || k == 7)) take = n - at;
            at += take;
            bounds[++k] = at;
        }
        return k;
    }
    // Queues the uploads of every chunk on the copy stream, with event copy_done[k] after chunk k: the signatures (unless
    // sigs == nullptr) into s_sigs, and the byte messages and offsets into s_msgs / s_offsets or the scalars into
    // s_scalars.  The copy stream first waits for everything already queued on the compute stream, so that no buffer of a
    // previous call is overwritten early.
    static int upload_chunks(Ctx* c, size_t n, int n_chunks, const size_t* bounds, const uint8_t* sigs, const MsgIn& in,
                             uint32_t n_msgs, rt_stream_t s) {
        const size_t count = n * n_msgs;
        if (sigs) TRY(c->s_sigs.reserve(n * SIG));
        TRY(c->s_scalars.reserve(count * 32));
        if (in.off) {
            TRY(c->s_msgs.reserve(in.off[count]));
            TRY(c->s_offsets.reserve((count + 1) * 8));
        }
        if (!c->copy_stream) RT_CHECK(cudaStreamCreateWithFlags(&c->copy_stream, cudaStreamNonBlocking));
        if (!c->copy_done[0]) for (auto& e : c->copy_done) RT_CHECK(cudaEventCreateWithFlags(&e, cudaEventDisableTiming));
        RT_CHECK(cudaEventRecord(c->copy_done[7], s));
        RT_CHECK(cudaStreamWaitEvent(c->copy_stream, c->copy_done[7], 0));
        for (int k = 0; k < n_chunks; k++) {
            const size_t i0 = bounds[k], i1 = bounds[k + 1], m0 = i0 * n_msgs, m1 = i1 * n_msgs;
            if (sigs) TRY(rt_h2d((uint8_t*)c->s_sigs.p + i0 * SIG, sigs + i0 * SIG, (i1 - i0) * SIG, c->copy_stream));
            if (in.off) {
                TRY(rt_h2d((uint8_t*)c->s_msgs.p + in.off[m0], in.msgs + in.off[m0], in.off[m1] - in.off[m0], c->copy_stream));
                TRY(rt_h2d((uint64_t*)c->s_offsets.p + m0, in.off + m0, (m1 - m0 + 1) * 8, c->copy_stream));
            } else {
                TRY(rt_h2d((uint8_t*)c->s_scalars.p + m0 * 32, in.scalars + m0 * 32, (m1 - m0) * 32, c->copy_stream));
            }
            RT_CHECK(cudaEventRecord(c->copy_done[k], c->copy_stream));
        }
        return BBS_OK;
    }

    // Host buffers of a LARGE verify batch (>= 2 * VERIFY_CHUNK items) in up to 8 chunks of doubling size: all uploads are
    // queued on the copy stream with one event per chunk; the compute stream hashes (byte messages) and runs the G1 half of
    // chunk k while chunk k + 1 is in flight; ONE pairing launch over the whole batch follows (it is 3/4 of the work and
    // loses nothing to chunking that way).  Statuses are those of the one-shot path: the items are independent.
    static constexpr size_t VERIFY_CHUNK = 131072;
    static int verify_chunked(Ctx* c, size_t n, const uint8_t* sigs, const MsgIn& in, uint32_t n_msgs, uint8_t* status) {
        rt_stream_t s = c->stream;
        size_t bounds[9];
        const int n_chunks = plan_chunks(n, VERIFY_CHUNK, true, bounds);
        size_t largest = 0;
        for (int k = 0; k < n_chunks; k++) largest = std::max(largest, bounds[k + 1] - bounds[k]);
        TRY(c->s_status.reserve(n));
        TRY(c->s_pair.reserve(n * 6 * C::Fp::N * 4));
        TRY(c->s_flags.reserve(n * 4));
        if (largest <= c->split_max) {                   // no reallocation between the chunk launches
            TRY(c->s_g1v.reserve(largest * 3 * C::Fp::N * 4));
            TRY(c->s_g1f.reserve(largest * 3 * C::Fp::N * 4));
            TRY(c->s_g1st.reserve(2 * largest));
        }
        TRY(upload_chunks(c, n, n_chunks, bounds, sigs, in, n_msgs, s));
        int rc = BBS_OK;
        for (int k = 0; k < n_chunks && !rc; k++) {
            const size_t i0 = bounds[k], i1 = bounds[k + 1], m0 = i0 * n_msgs, m1 = i1 * n_msgs;
            RT_CHECK(cudaStreamWaitEvent(s, c->copy_done[k], 0));
            if (in.off) rc = h2s_dev(c, m1 - m0, (const uint8_t*)c->s_msgs.p, (const uint64_t*)c->s_offsets.p + m0,
                                     (uint8_t*)c->s_scalars.p + m0 * 32, s);
            if (!rc) rc = verify_g1_dev(c, i1 - i0, i0, (const uint8_t*)c->s_sigs.p, (const uint8_t*)c->s_scalars.p, n_msgs,
                                        (uint8_t*)c->s_status.p, s);
        }
        if (!rc) rc = pairing_dev(c, n, (uint8_t*)c->s_status.p, s);
        if (rc) { cudaStreamSynchronize(c->copy_stream); rt_sync(s); return rc; }
        return finish_status(c, n, status);
    }
#endif

    // ---- issuer sets ------------------------------------------------------------------------------------
    // per-issuer state for n keys on top of an existing base context: decode + subgroup test, domain and K, the ate walk
    // of every key (one thread per issuer), normalised for the cooperative kernel
    static int issuer_set_build(IssuerSet* S, const uint8_t* pks, size_t n, uint8_t* issuer_status) {
        Ctx* c = S->base;
        rt_stream_t s = c->stream;
        constexpr size_t FN = C::Fp::N;
        const uint32_t n_lines = (uint32_t)ate_line_count<C>();
        const uint32_t stride = n_lines * 2 * 4 * (uint32_t)FN;          // words per issuer: lines x 2 pairs x (2 Fp2)
        S->n_issuers = n;
        S->line_stride = stride;
        TRY(S->pks.reserve(n * C::G2_BYTES));
        TRY(S->W.reserve(n * 4 * FN * 4));
        TRY(S->K.reserve(n * 2 * FN * 4));
        TRY(S->domains.reserve(n * 32));
        TRY(S->flags.reserve(n * 4));
        TRY(S->lines.reserve(n * (size_t)stride * 4));
        TRY(rt_h2d(S->pks.p, pks, n * C::G2_BYTES, s));
        IssDecodeArgs da{(const uint8_t*)S->pks.p, (uint32_t*)S->W.p, (uint32_t*)S->flags.p};
        TRY((launch_iss_decode<C>(da, (uint32_t)n, s)));
        IssDomainArgs dom{};
        dom.base = CtxDomainArgs{nullptr, (const uint8_t*)c->gens_comp.p, c->L, (const uint8_t*)c->api_id.p, (uint32_t)c->api_id_len,
                                 (const uint8_t*)c->header.p, (uint32_t)c->header_len, c->view.dst_h2s, c->view.dst_h2s_len,
                                 c->view.gens, nullptr, nullptr, nullptr};
        dom.pks = (const uint8_t*)S->pks.p; dom.domains = (uint32_t*)S->domains.p; dom.K = (uint32_t*)S->K.p;
        dom.flags = (uint32_t*)S->flags.p;
        TRY((launch_iss_domain<C>(dom, (uint32_t)n, s)));
        c->launches += 2;
        const size_t chunk = std::min<size_t>(n, 4096);
        DevBuf raw;
        int rc = raw.reserve(chunk * (size_t)stride * 4);
        for (size_t first = 0; !rc && first < n; first += chunk) {
            const uint32_t cnt = (uint32_t)std::min(chunk, n - first);
            IssLinesArgs la{(const uint32_t*)S->W.p, (const uint32_t*)S->flags.p, (uint32_t*)raw.p, stride, (uint32_t)first};
            rc = launch_iss_lines<C>(la, cnt, s);
#ifndef BBS_HOSTSIM
            IssLinesCoopArgs lc{(const uint32_t*)raw.p, stride, (const uint32_t*)c->lines_coop.p, (uint32_t*)S->lines.p, stride,
                                (uint32_t*)S->flags.p, (uint32_t)first, n_lines};
            if (!rc) rc = launch_iss_lines_coop<C>(lc, cnt * 2 * n_lines, s);
#else
            // host simulation: the per-thread pairing kernel reads the raw (A, Bc) layout; pair 1 = the base context's BP2 lines
            for (uint32_t t = 0; t < cnt; t++) {
                uint32_t* dst = (uint32_t*)S->lines.p + (first + t) * (size_t)stride;
                const uint32_t* src = (const uint32_t*)raw.p + t * (size_t)stride;
                const uint32_t* bp2 = (const uint32_t*)c->lines.p;
                for (uint32_t k = 0; k < n_lines; k++) {
                    memcpy(dst + (2 * k) * 4 * FN, src + (2 * k) * 4 * FN, 4 * FN * 4);
                    memcpy(dst + (2 * k + 1) * 4 * FN, bp2 + (2 * k + 1) * 4 * FN, 4 * FN * 4);
                }
            }
#endif
            c->launches += 2;
        }
        if (!rc) rc = rt_sync(s);
        raw.release();
        TRY(rc);
        std::vector<uint32_t> fl(n);
        TRY(rt_d2h(fl.data(), S->flags.p, n * 4, s));
        TRY(rt_sync(s));
        for (size_t i = 0; i < n; i++) issuer_status[i] = (fl[i] & ISS_BAD) ? (uint8_t)ST_ERR_MALFORMED : (uint8_t)ST_ACCEPT;
        return BBS_OK;
    }

    static int verify_dev(Ctx* c, size_t n, const uint8_t* d_sigs, const uint8_t* d_msgs, const uint64_t* d_off,
                          uint32_t n_msgs, uint8_t* d_status, rt_stream_t s) {
        TRY(c->s_scalars.reserve(n * n_msgs * 32));
        PROF(c, 0, s);
        TRY(h2s_dev(c, n * n_msgs, d_msgs, d_off, (uint8_t*)c->s_scalars.p, s));
        return core_verify_dev(c, n, d_sigs, (const uint8_t*)c->s_scalars.p, n_msgs, d_status, s);
    }

    static int core_sign_dev(Ctx* c, const uint8_t* sk, size_t n, const uint8_t* d_scalars, uint32_t n_msgs,
                             uint8_t* d_sigs, uint8_t* d_b, uint8_t* d_status, rt_stream_t s, const ItemKeyView* item = nullptr) {
        SignArgs a{};
        a.ctx = c->view;
        if (item) a.item = *item;
        uint32_t skl[8];
        limbs_from_le<8>(skl, sk);
        const bool canon = fe_is_canonical<typename C::Fr>(skl);
        int rc = canon ? c->s_sk.reserve(32) : arg_error("secret key scalar is not canonical");
        if (!rc) rc = rt_h2d(c->s_sk.p, skl, 32, s);       // pageable source: staged before the call returns
        volatile uint32_t* wipe = skl;
        for (int i = 0; i < 8; i++) wipe[i] = 0;
        TRY(rc);
        a.sk = (const uint32_t*)c->s_sk.p;
        a.scalars = d_scalars; a.n_msgs = n_msgs; a.sigs_out = d_sigs; a.b_out = d_b; a.status = d_status;
        PROF(c, 1, s);
        rc = launch_sign<C>(a, (uint32_t)n, s);
        c->launches += n ? 1 : 0;
        int rc2 = rt_memset(c->s_sk.p, 0, 32, s);           // SecretKey is ZeroizeOnDrop (key_gen.rs:29)
        TRY(rc);
        TRY(rc2);
        PROF(c, 2, s);
        if (item) c->prof.xslot = 2;
        return BBS_OK;
    }

    static int core_proof_verify_dev(Ctx* c, size_t n, const uint8_t* d_proofs, const uint8_t* d_commit,
                                     const uint64_t* d_commit_off, const uint32_t* d_idx, const uint8_t* d_dis_scalars,
                                     const uint64_t* d_dis_off, const uint8_t* d_ph, size_t ph_len, uint8_t* d_status,
                                     rt_stream_t s, const IssuerSet* S = nullptr, const ItemKeyView* item = nullptr,
                                     const uint64_t* d_ph_off = nullptr, const RlcProofIn* rlc = nullptr) {
        TRY(c->s_pair.reserve(n * 6 * C::Fp::N * 4));
        TRY(c->s_flags.reserve(n * 4));
        ProofG1Args a{c->view, d_proofs, d_commit, d_commit_off, d_idx, d_dis_scalars, d_dis_off, d_ph,
                      (uint32_t)ph_len, (uint32_t*)c->s_pair.p, (uint32_t*)c->s_flags.p, d_status};
        if (S) {                           // issuer sets go through the task split (kernels.cuh proof_task_*) at every size
            a.item_issuer = (const uint32_t*)S->item_issuer.p;
            a.iss = S->view();
        }
        a.ph_off = d_ph_off;
        if (item) a.item = *item;         // per-item headers, like issuer sets, take the task split at every size
        if (S || item || n <= c->split_max) {
            TRY(c->s_g1t.reserve(n * 3 * C::Fp::N * 4));
            TRY(c->s_g1v.reserve(n * 3 * C::Fp::N * 4));
            TRY(c->s_g1f.reserve(n * 3 * C::Fp::N * 4));
            TRY(c->s_g1st.reserve(2 * n));
            a.part_t1 = (uint32_t*)c->s_g1t.p; a.part_v2 = (uint32_t*)c->s_g1v.p; a.part_f = (uint32_t*)c->s_g1f.p;
            a.part_st = (uint8_t*)c->s_g1st.p;
        }
        PROF(c, 1, s);
        TRY((launch_proof_g1<C>(a, (uint32_t)n, s)));
        c->launches += n ? (a.part_t1 ? 2 : 1) : 0;
        PROF(c, 2, s);
#ifndef BBS_HOSTSIM
        if (rlc) {
            TRY(rlc_proof_pairing_dev(c, n, *rlc, d_status, s));
            if (item) c->prof.xslot = 9;
            return BBS_OK;
        }
#endif
        TRY(pairing_dev(c, n, d_status, s, S));
        PROF(c, 3, s);
        if (item) c->prof.xslot = 3;
        return BBS_OK;
    }
    // bbs_core_proof_verify_batch_hdr_dev: d_hdr_off == nullptr = the context's header
    static int core_proof_verify_hdr_dev(Ctx* c, size_t n, const uint8_t* d_proofs, const uint8_t* d_commit,
                                         const uint64_t* d_commit_off, const uint32_t* d_idx, const uint8_t* d_dis_scalars,
                                         const uint64_t* d_dis_off, const uint8_t* d_headers, const uint64_t* d_hdr_off,
                                         const uint8_t* d_phs, const uint64_t* d_ph_off, uint8_t* d_status, rt_stream_t s) {
        ItemKeyView item{};
        if (d_hdr_off) TRY(item_keys_dev(c, n, d_headers, d_hdr_off, item, s));
        return core_proof_verify_dev(c, n, d_proofs, d_commit, d_commit_off, d_idx, d_dis_scalars, d_dis_off, d_phs, 0, d_status,
                                     s, nullptr, d_hdr_off ? &item : nullptr, d_ph_off);
    }

    // ---- core_proof_gen (proof_gen.rs:116-365) -----------------------------------------------------------
    // ph_off != nullptr: per-item phs in `ph`; hdr_off != nullptr: per-item headers (bbs_*proof_gen_batch_hdr)
    static int proof_gen(Ctx* c, size_t n, const uint8_t* sigs, const MsgIn& in, uint32_t n_msgs, const uint32_t* idx,
                         const uint64_t* dis_off, const uint8_t* rand, const uint64_t* rand_off, const uint64_t* commit_off,
                         const uint8_t* ph, size_t ph_len, uint8_t* proofs_out, uint8_t* commitments_out, uint8_t* status,
                         const uint64_t* ph_off = nullptr, const uint8_t* headers = nullptr, const uint64_t* hdr_off = nullptr) {
        rt_stream_t s = c->stream;
        TRY(stage_scalars(c, n * n_msgs, in, c->s_msgs, c->s_offsets, c->s_scalars, false));
        ItemKeyView item{};
        if (hdr_off) TRY(item_keys(c, n, headers, hdr_off, item));
        if (ph_off) {
            ph_len = ph_off[n];
            TRY(stage(c->s_ph_off, ph_off, (n + 1) * 8, s));
        }
        TRY(stage(c->s_sigs, sigs, n * SIG, s));
        TRY(stage(c->s_dis_idx, idx, dis_off[n] * 4, s));
        TRY(stage(c->s_dis_off, dis_off, (n + 1) * 8, s));
        TRY(stage(c->s_rand, rand, rand_off[n] * 32, s));
        TRY(stage(c->s_rand_off, rand_off, (n + 1) * 8, s));
        TRY(stage(c->s_commit_off, commit_off, (n + 1) * 8, s));
        TRY(stage(c->s_ph, ph, ph_len, s));
        TRY(c->s_out.reserve(n * PROOF));
        TRY(c->s_commit.reserve(commit_off[n] * 32));
        TRY(c->s_status.reserve(n));
        TRY(rt_memset(c->s_out.p, 0, n * PROOF, s));
        TRY(rt_memset(c->s_commit.p, 0, commit_off[n] * 32, s));
        ProofGenArgs a{c->view, (const uint8_t*)c->s_sigs.p, (const uint8_t*)c->s_scalars.p, n_msgs,
                       (const uint32_t*)c->s_dis_idx.p, (const uint64_t*)c->s_dis_off.p, (const uint8_t*)c->s_rand.p,
                       (const uint64_t*)c->s_rand_off.p, (const uint64_t*)c->s_commit_off.p, (const uint8_t*)c->s_ph.p,
                       (uint32_t)ph_len, (uint8_t*)c->s_out.p, (uint8_t*)c->s_commit.p, (uint8_t*)c->s_status.p};
        a.item = item;
        a.ph_off = ph_off ? (const uint64_t*)c->s_ph_off.p : nullptr;
        TRY((launch_proof_gen<C>(a, (uint32_t)n, s)));
        c->launches += n ? 1 : 0;
        TRY(rt_d2h(proofs_out, c->s_out.p, n * PROOF, s));
        TRY(rt_d2h(commitments_out, c->s_commit.p, commit_off[n] * 32, s));
        return finish_status(c, n, status);
    }

    // ---- random-linear-combination batch mode (rlc.cuh) ---------------------------------------------
#ifndef BBS_HOSTSIM
    // digits per 128-bit value for the bucket MSM.  Cost in field multiplications: 11 per bucket addition, inflated by the
    // quantisation of buckets over the persistent threads of msm_bucket_kernel (u buckets per thread), plus ~47 per bucket
    // for the reduction (measured on B200 at n = 65,536 and 524,288: profiles/summary_r01.md).  `values`: 128-bit values
    // per item (3 for signatures, 2 for proofs).
    static MsmPlan rlc_plan(size_t n, uint32_t force, double values = 3.0) {   // force != 0: bbs_ctx_set_rlc_windows (tests)
        uint32_t best = 32;
        double best_cost = 1e300;
        for (uint32_t W = 8; W <= 32; W++) {
            const uint32_t c = (128 + W - 1) / W, rows = 2 * W;
            double used = 0;                                   // buckets that can be non-empty
            for (uint32_t w = 0; w < W; w++) used += (double)(1u << (((w + 1) * 128) / W - (w * 128) / W));
            used *= rows / W;
            const double u = used / (148.0 * 512.0);
            const double cost = 11.0 * values * W * (double)n * (1.0 + 1.0 / u) + 47.0 * rows * (double)(1u << c);
            if (force ? force == W : cost < best_cost) { best = W; best_cost = cost; }
        }
        MsmPlan p;
        p.W = best;
        p.c = (128 + best - 1) / best;
        p.rows = 2 * p.W;
        p.chunk = 16u;
        const uint32_t threads = (1u << p.c) / p.chunk;
        p.red_blocks = (threads + RLC_TPB - 1) / RLC_TPB;
        return p;
    }
    // The upload, hashing and prep stages of a shard: its host buffers are fed in up to 8 chunks, chunk k + 1 uploaded on
    // the copy stream while chunk k is hashed (byte messages) and prepared on the compute stream.  `mode` (RLC_PREP_*):
    // RLC_PREP_VERDICT sets the word s_rlc_bad when an item is malformed; the status modes write the malformed items'
    // statuses and every item's flag word into s_status / s_flags and set s_rlc_bad when some item is well formed, and
    // RLC_PREP_STATUS_HDR reads the items' domains from `item`.  Reserves the MSM scratch that rlc_msm_dev uses after it.
    static int rlc_prep_dev(Ctx* c, size_t n, const uint8_t* sigs, const MsgIn& in, uint32_t n_msgs, const uint8_t* seed,
                            uint64_t index_base, int mode, const ItemKeyView* item, MsmPlan& plan, rt_stream_t s) {
        if (n >= (1ull << 31)) return arg_error("rlc shard too large");
        const uint32_t blocks = (uint32_t)((n + RLC_TPB - 1) / RLC_TPB);
        const uint32_t sc_rows = n_msgs + 1 + (mode == RLC_PREP_STATUS_HDR ? 1u : 0u);
        plan = rlc_plan(n, c->rlc_windows);
        const size_t nb = (size_t)plan.rows << plan.c, PT = 3 * C::Fp::N * 4;
        TRY(c->s_rlc_sc.reserve((size_t)(blocks ? blocks : 1) * sc_rows * 32));
        TRY(c->s_rlc_parts.reserve(2 * C::G1_BYTES));
        TRY(c->s_rlc_bad.reserve(4));
        if (mode != RLC_PREP_VERDICT) {
            TRY(c->s_status.reserve(n));
            TRY(c->s_flags.reserve(n * 4));
        }
        TRY(c->s_msm_pts.reserve((n ? n : 1) * 2 * C::Fp::N * 4));
        TRY(c->s_msm_kv.reserve((n ? n : 1) * 48));
        TRY(c->s_msm_idx.reserve((3 * nb + 5) * 4));                        // next (4 words) | counts | offsets (nb + 1) | cursor
        TRY(c->s_msm_entries.reserve((n ? n : 1) * 3 * plan.W * 4));
        TRY(c->s_msm_buckets.reserve(nb * PT));
        TRY(c->s_rlc_pt.reserve((size_t)plan.rows * plan.red_blocks * PT));
        uint32_t* next = (uint32_t*)c->s_msm_idx.p;
        uint32_t* counts = next + 4;
        uint32_t* offsets = counts + nb;
        uint32_t* cursor = offsets + nb + 1;
        TRY(rt_memset(c->s_rlc_bad.p, 0, 4, s));
        TRY(rt_memset(next, 0, (nb + 4) * 4, s));
        RlcPrepArgs pa{};
        RlcArgs& a = pa.base;
        a.ctx = c->view; a.n_msgs = n_msgs;
        for (int i = 0; i < 8; i++)
            a.seed[i] = ((uint32_t)seed[4 * i] << 24) | ((uint32_t)seed[4 * i + 1] << 16) | ((uint32_t)seed[4 * i + 2] << 8) | seed[4 * i + 3];
        a.bad = (uint32_t*)c->s_rlc_bad.p;
        pa.plan = plan; pa.counts = counts;
        pa.live = (uint32_t*)c->s_rlc_bad.p;
        // chunk = a whole number of waves of the prep kernel (4 blocks of RLC_TPB items per SM), at most 8 chunks; chunk
        // boundaries are multiples of the block size, so the blocks' partial sums keep their global index
        int sms = 0;
        RT_CHECK(cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, c->device));
        const size_t wave = (size_t)4 * sms * RLC_TPB;
        const size_t waves = std::max<size_t>(2, ((n + 7) / 8 + wave - 1) / wave);
        size_t bounds[9];
        const int n_chunks = plan_chunks(n, waves * wave, false, bounds);
        TRY(upload_chunks(c, n, n_chunks, bounds, sigs, in, n_msgs, s));      // after the memsets: the copy stream waits for them
        PROF(c, 0, s);
        for (int k = 0; k < n_chunks; k++) {
            const size_t i0 = bounds[k], i1 = bounds[k + 1], m0 = i0 * n_msgs, m1 = i1 * n_msgs;
            RT_CHECK(cudaStreamWaitEvent(s, c->copy_done[k], 0));
            if (in.off)
                TRY(h2s_dev(c, m1 - m0, (const uint8_t*)c->s_msgs.p, (const uint64_t*)c->s_offsets.p + m0,
                            (uint8_t*)c->s_scalars.p + m0 * 32, s));
            if (k == 0) PROF(c, 1, s);          // slot 0: first chunk's upload wait + hashing; slot 1: everything chunked after it
            a.sigs = (const uint8_t*)c->s_sigs.p + i0 * SIG; a.scalars = (const uint8_t*)c->s_scalars.p + m0 * 32;
            a.n = (uint32_t)(i1 - i0);
            a.index_base = index_base + i0;
            a.sc_part = (uint32_t*)c->s_rlc_sc.p + (i0 / RLC_TPB) * sc_rows * 8;
            pa.pts = (uint32_t*)c->s_msm_pts.p + i0 * 2 * C::Fp::N; pa.kv = (uint32_t*)c->s_msm_kv.p + i0 * 12;
            if (mode != RLC_PREP_VERDICT) {
                pa.status = (uint8_t*)c->s_status.p + i0; pa.flags = (uint32_t*)c->s_flags.p + i0;
                pa.domains = item ? item->domains + i0 * 8 : nullptr;
            }
            TRY((launch_rlc_prep<C>(pa, (uint32_t)((i1 - i0 + RLC_TPB - 1) / RLC_TPB), mode, s)));
            c->launches += 1;
        }
        PROF(c, 2, s);
        return BBS_OK;
    }
    // scan, scatter, buckets, reduction and finish over the prepared shard: comp(S1) || comp(S2) in c->s_rlc_parts and the
    // pairing record of the two sums, its flag word and status at pair / flags / status (index 0)
    static int rlc_msm_dev(Ctx* c, size_t n, const MsmPlan& plan, uint32_t n_msgs, bool hdr, uint32_t* pair, uint32_t* flags,
                           uint8_t* status, rt_stream_t s) {
        const uint32_t blocks = (uint32_t)((n + RLC_TPB - 1) / RLC_TPB);
        const size_t nb = (size_t)plan.rows << plan.c;
        uint32_t* next = (uint32_t*)c->s_msm_idx.p;
        uint32_t* counts = next + 4;
        uint32_t* offsets = counts + nb;
        uint32_t* cursor = offsets + nb + 1;
        TRY(launch_msm_scan(counts, offsets, cursor, (uint32_t)nb, s));
        MsmScatterArgs sa{plan, (const uint32_t*)c->s_msm_kv.p, cursor, (uint32_t*)c->s_msm_entries.p, (uint32_t)n};
        TRY((launch_msm_scatter<C>(sa, s)));
        PROF(c, 3, s);
        MsmBucketArgs ba{offsets, (const uint32_t*)c->s_msm_entries.p, (const uint32_t*)c->s_msm_pts.p,
                         (uint32_t*)c->s_msm_buckets.p, next, (uint32_t)nb};
        TRY((launch_msm_bucket<C>(ba, s)));
        PROF(c, 4, s);
        MsmReduceArgs ra{plan, (const uint32_t*)c->s_msm_buckets.p, (uint32_t*)c->s_rlc_pt.p};
        TRY((launch_msm_reduce<C>(ra, s)));
        PROF(c, 5, s);
        RlcMsmFinishArgs f{c->view, plan, (const uint32_t*)c->s_rlc_pt.p, (const uint32_t*)c->s_rlc_sc.p, blocks, n_msgs,
                           (uint8_t*)c->s_rlc_parts.p, pair, flags, status};
        TRY((launch_rlc_msm_finish<C>(f, hdr, s)));
        PROF(c, 6, s);
        c->launches += (n ? 5 : 3);
        return BBS_OK;
    }
    // shard -> comp(S1) || comp(S2) in c->s_rlc_parts (and the pairing record of the two sums in s_pair); *bad != 0 when an
    // item was malformed
    static int rlc_partial_dev(Ctx* c, size_t n, const uint8_t* sigs, const MsgIn& in, uint32_t n_msgs, const uint8_t* seed,
                               uint64_t index_base, uint32_t* bad, rt_stream_t s) {
        MsmPlan plan;
        TRY(rlc_prep_dev(c, n, sigs, in, n_msgs, seed, index_base, RLC_PREP_VERDICT, nullptr, plan, s));
        TRY(c->s_pair.reserve(6 * C::Fp::N * 4));
        TRY(c->s_flags.reserve(4));
        TRY(c->s_status.reserve(1));
        TRY(rlc_msm_dev(c, n, plan, n_msgs, false, (uint32_t*)c->s_pair.p, (uint32_t*)c->s_flags.p, (uint8_t*)c->s_status.p, s));
        TRY(rt_d2h(bad, c->s_rlc_bad.p, 4, s));
        return BBS_OK;
    }
    static int rlc_partial(Ctx* c, size_t n, const uint8_t* sigs, const MsgIn& in, uint32_t n_msgs, const uint8_t* seed,
                           uint64_t index_base, uint8_t* parts_out, uint8_t* status) {
        rt_stream_t s = c->stream;
        if (n_msgs != c->L) { *status = ST_ERR_MSG_GEN_LEN; return BBS_OK; }
        uint32_t bad = 0;
        TRY(rlc_partial_dev(c, n, sigs, in, n_msgs, seed, index_base, &bad, s));
        TRY(rt_d2h(parts_out, c->s_rlc_parts.p, 2 * C::G1_BYTES, s));
        TRY(rt_sync(s));
        *status = bad ? ST_ERR_MALFORMED : ST_ACCEPT;
        return BBS_OK;
    }
    // one shard = the whole batch: the finish kernel's pairing record goes straight to the pairing kernel
    static int rlc_verify(Ctx* c, size_t n, const uint8_t* sigs, const MsgIn& in, uint32_t n_msgs, const uint8_t* seed,
                          uint8_t* verdict) {
        rt_stream_t s = c->stream;
        if (n_msgs != c->L) { *verdict = ST_ERR_MSG_GEN_LEN; return BBS_OK; }
        uint32_t bad = 0;
        TRY(rlc_partial_dev(c, n, sigs, in, n_msgs, seed, 0, &bad, s));
        TRY(pairing_dev(c, 1, (uint8_t*)c->s_status.p, s));
        PROF(c, 7, s);
        TRY(finish_status(c, 1, verdict));             // synchronises: `bad` has arrived too
        if (bad) *verdict = ST_ERR_MALFORMED;
        return BBS_OK;
    }
    // Per-item statuses by one random linear combination (bbs_rlc_*verify_batch_status*; hdr_off != nullptr: a header per
    // item).  The prep kernel decides the malformed items and leaves them out of the sums; if any item is left, ONE pairing
    // checks the combination of all of them (its record, flag word and verdict in s_rlcp, apart from the items' arrays).
    // If it holds, those items are accepted; if not, the per-item G1 half and pairing decide every item from the buffers
    // already on the device.  Profiling slots: see include/bbs_b200.h.
    static int rlc_verify_status(Ctx* c, size_t n, const uint8_t* sigs, const MsgIn& in, uint32_t n_msgs, const RlcProofIn& rlc,
                                 uint8_t* status, const uint8_t* headers = nullptr, const uint64_t* hdr_off = nullptr) {
        rt_stream_t s = c->stream;
        uint8_t verdict = ST_ACCEPT;
        if (n_msgs != c->L) {                                                // verify.rs:68-71, for every item
            std::fill(status, status + n, (uint8_t)ST_ERR_MSG_GEN_LEN);
            if (rlc.combined) *rlc.combined = verdict;
            return BBS_OK;
        }
        constexpr size_t PW = 6 * C::Fp::N;
        ItemKeyView item{};
        if (hdr_off) TRY(item_keys(c, n, headers, hdr_off, item));
        TRY(c->s_rlcp.reserve((PW + 2) * 4));                               // record | flags | status
        MsmPlan plan;
        TRY(rlc_prep_dev(c, n, sigs, in, n_msgs, rlc.seed, 0, hdr_off ? RLC_PREP_STATUS_HDR : RLC_PREP_STATUS,
                         hdr_off ? &item : nullptr, plan, s));
        uint32_t live = 0;
        TRY(rt_d2h(&live, c->s_rlc_bad.p, 4, s));
        TRY(rt_sync(s));
        if (live) {                                                          // else every status is final already
            uint32_t* pair = (uint32_t*)c->s_rlcp.p;
            uint8_t* verdict_d = (uint8_t*)(pair + PW + 1);
            TRY(rlc_msm_dev(c, n, plan, n_msgs, hdr_off != nullptr, pair, pair + PW, verdict_d, s));
            TRY(pairing_dev(c, 1, verdict_d, s, nullptr, pair, pair + PW));
            TRY(rt_d2h(&verdict, verdict_d, 1, s));
            TRY(rt_sync(s));
            PROF(c, 7, s);
            if (verdict == ST_ACCEPT) {
                TRY((launch_rlc_proof_accept<C>((const uint32_t*)c->s_flags.p, (uint8_t*)c->s_status.p, (uint32_t)n, s)));
                c->launches += 1;
                PROF(c, 8, s);
            } else {
                TRY(rlc_status_fallback(c, n, n_msgs, hdr_off ? &item : nullptr, s));
            }
            PROF(c, 9, s);
        }
        TRY(finish_status(c, n, status));
        if (hdr_off) c->prof.xslot = 9;
        if (rlc.combined) *rlc.combined = verdict;
        return BBS_OK;
    }
    // the per-item path over the signatures and scalars that rlc_prep_dev left in s_sigs / s_scalars: the G1 half in the
    // chunks of verify_chunked (its scratch reserved for the largest first), then one pairing launch
    static int rlc_status_fallback(Ctx* c, size_t n, uint32_t n_msgs, const ItemKeyView* item, rt_stream_t s) {
        size_t bounds[9];
        const int n_chunks = plan_chunks(n, VERIFY_CHUNK, true, bounds);
        size_t largest = 0;
        for (int k = 0; k < n_chunks; k++) largest = std::max(largest, bounds[k + 1] - bounds[k]);
        TRY(c->s_pair.reserve(n * 6 * C::Fp::N * 4));
        if (largest <= c->split_max) {
            TRY(c->s_g1v.reserve(largest * 3 * C::Fp::N * 4));
            TRY(c->s_g1f.reserve(largest * 3 * C::Fp::N * 4));
            TRY(c->s_g1st.reserve(2 * largest));
        }
        for (int k = 0; k < n_chunks; k++)
            TRY(verify_g1_dev(c, bounds[k + 1] - bounds[k], bounds[k], (const uint8_t*)c->s_sigs.p, (const uint8_t*)c->s_scalars.p,
                              n_msgs, (uint8_t*)c->s_status.p, s, nullptr, item));
        PROF(c, 8, s);
        return pairing_dev(c, n, (uint8_t*)c->s_status.p, s);
    }
    // n_parts x (comp(S1) || comp(S2)) -> one verdict byte
    static int rlc_combine(Ctx* c, size_t n_parts, const uint8_t* parts, uint8_t* verdict) {
        rt_stream_t s = c->stream;
        TRY(stage(c->s_sigs, parts, n_parts * 2 * C::G1_BYTES, s));
        TRY(c->s_pair.reserve(6 * C::Fp::N * 4));
        TRY(c->s_flags.reserve(4));
        TRY(c->s_status.reserve(1));
        RlcCombineArgs a{c->view, (const uint8_t*)c->s_sigs.p, (uint32_t)n_parts, (uint32_t*)c->s_pair.p,
                         (uint32_t*)c->s_flags.p, (uint8_t*)c->s_status.p};
        TRY((launch_rlc_combine<C>(a, s)));
        c->launches += 1;
        TRY(pairing_dev(c, 1, (uint8_t*)c->s_status.p, s));
        return finish_status(c, 1, verdict);
    }
    // The pairing half of a proof batch by one random linear combination (rlc_msm.cuh, proof batches): after the G1 half,
    // the items without FL_DONE are checked with ONE pairing of S1 = sum r_i Abar_i and S2 = sum r_i (-Bbar_i).  If it
    // holds they are accepted; if not, the per-item pairing kernel decides them from their records, which the MSM leaves
    // intact (the combined record has its own slot, s_rlcp).  Profiling slots 2..8: prep, scan + scatter, buckets,
    // reduction, finish, combined pairing, acceptance or per-item pairing.
    static int rlc_proof_pairing_dev(Ctx* c, size_t n, const RlcProofIn& rlc, uint8_t* d_status, rt_stream_t s) {
        const MsmPlan plan = rlc_plan(n, c->rlc_windows, 2.0);
        const size_t nb = (size_t)plan.rows << plan.c, PT = 3 * C::Fp::N * 4, PW = 6 * C::Fp::N;
        TRY(c->s_msm_kv.reserve(n * 48));
        TRY(c->s_msm_idx.reserve((3 * nb + 5) * 4));                        // next (4 words) | counts | offsets (nb + 1) | cursor
        TRY(c->s_msm_entries.reserve(n * 2 * plan.W * 4));
        TRY(c->s_msm_buckets.reserve(nb * PT));
        TRY(c->s_rlc_pt.reserve((size_t)plan.rows * plan.red_blocks * PT));
        TRY(c->s_rlc_parts.reserve(2 * C::G1_BYTES));
        TRY(c->s_rlc_bad.reserve(4));
        TRY(c->s_rlcp.reserve((PW + 2) * 4));                               // record | flags | status
        uint32_t* next = (uint32_t*)c->s_msm_idx.p;
        uint32_t* counts = next + 4;
        uint32_t* offsets = counts + nb;
        uint32_t* cursor = offsets + nb + 1;
        uint32_t* pair = (uint32_t*)c->s_rlcp.p;
        uint8_t* verdict_d = (uint8_t*)(pair + PW + 1);
        TRY(rt_memset(c->s_rlc_bad.p, 0, 4, s));
        TRY(rt_memset(next, 0, (nb + 4) * 4, s));
        RlcProofPrepArgs pa{};
        pa.plan = plan; pa.flags = (const uint32_t*)c->s_flags.p; pa.kv = (uint32_t*)c->s_msm_kv.p; pa.counts = counts;
        pa.live = (uint32_t*)c->s_rlc_bad.p; pa.n = (uint32_t)n;
        for (int i = 0; i < 8; i++)
            pa.seed[i] = ((uint32_t)rlc.seed[4 * i] << 24) | ((uint32_t)rlc.seed[4 * i + 1] << 16) |
                         ((uint32_t)rlc.seed[4 * i + 2] << 8) | rlc.seed[4 * i + 3];
        TRY((launch_rlc_proof_prep<C>(pa, s)));
        c->launches += 1;
        PROF(c, 3, s);
        uint32_t live = 0;
        TRY(rt_d2h(&live, c->s_rlc_bad.p, 4, s));
        TRY(rt_sync(s));
        uint8_t verdict = ST_ACCEPT;
        if (live) {                                                          // else every status is final already
            TRY(launch_msm_scan(counts, offsets, cursor, (uint32_t)nb, s));
            MsmScatterArgs sa{plan, (const uint32_t*)c->s_msm_kv.p, cursor, (uint32_t*)c->s_msm_entries.p, (uint32_t)n};
            TRY((launch_msm_scatter<C>(sa, s)));
            PROF(c, 4, s);
            MsmBucketArgs ba{offsets, (const uint32_t*)c->s_msm_entries.p, (const uint32_t*)c->s_pair.p,
                             (uint32_t*)c->s_msm_buckets.p, next, (uint32_t)nb};
            TRY((launch_msm_bucket_pair<C>(ba, s)));
            PROF(c, 5, s);
            MsmReduceArgs ra{plan, (const uint32_t*)c->s_msm_buckets.p, (uint32_t*)c->s_rlc_pt.p};
            TRY((launch_msm_reduce<C>(ra, s)));
            PROF(c, 6, s);
            // the signature mode's finish kernel with no prep blocks and no messages: its Fr sums and fixed-base term are
            // zero, so it yields S1 and S2 as they are
            RlcMsmFinishArgs f{c->view, plan, (const uint32_t*)c->s_rlc_pt.p, nullptr, 0u, 0u, (uint8_t*)c->s_rlc_parts.p,
                               pair, pair + PW, verdict_d};
            TRY((launch_rlc_msm_finish<C>(f, false, s)));
            c->launches += 5;
            PROF(c, 7, s);
            TRY(pairing_dev(c, 1, verdict_d, s, nullptr, pair, pair + PW));
            TRY(rt_d2h(&verdict, verdict_d, 1, s));
            TRY(rt_sync(s));
            PROF(c, 8, s);
            if (verdict == ST_ACCEPT) {
                TRY((launch_rlc_proof_accept<C>((const uint32_t*)c->s_flags.p, d_status, (uint32_t)n, s)));
                c->launches += 1;
            } else {
                TRY(pairing_dev(c, n, d_status, s));
            }
            PROF(c, 9, s);
        }
        if (rlc.combined) *rlc.combined = verdict;
        return BBS_OK;
    }
#endif

    // ---- host-buffer calls ------------------------------------------------------------------------------------------
    static int stage(DevBuf& b, const void* h, size_t bytes, rt_stream_t s) {
        TRY(b.reserve(bytes));
        return rt_h2d(b.p, h, bytes, s);
    }
    static int finish_status(Ctx* c, size_t n, uint8_t* status) {
        TRY(rt_d2h(status, c->s_status.p, n, c->stream));
        return rt_sync(c->stream);
    }
    // the `count` message scalars of `in` into `out`: staged, or the byte messages staged into `msgs` / `off` and hashed.
    // With `prof`, profiling slot 0 brackets the hashing kernel.
    static int stage_scalars(Ctx* c, size_t count, const MsgIn& in, DevBuf& msgs, DevBuf& off, DevBuf& out, bool prof) {
        rt_stream_t s = c->stream;
        if (!in.off) return stage(out, in.scalars, count * 32, s);
        TRY(stage(msgs, in.msgs, in.off[count], s));
        TRY(stage(off, in.off, (count + 1) * 8, s));
        TRY(out.reserve(count * 32));
        if (prof) PROF(c, 0, s);
        return h2s_dev(c, count, (const uint8_t*)msgs.p, (const uint64_t*)off.p, (uint8_t*)out.p, s);
    }

    static int msg_to_scalars(Ctx* c, size_t count, const uint8_t* msgs, const uint64_t* off, uint8_t* out) {
        TRY(stage_scalars(c, count, MsgIn{nullptr, msgs, off}, c->s_msgs, c->s_offsets, c->s_scalars, false));
        TRY(rt_d2h(out, c->s_scalars.p, count * 32, c->stream));
        return rt_sync(c->stream);
    }
    // verify / core_verify; hdr_off != nullptr: a header per item (bbs_*verify_batch_hdr); S != nullptr: the issuer of each
    // item in item_issuer (bbs_*verify_batch_multi, c = S->base)
    static int verify(Ctx* c, size_t n, const uint8_t* sigs, const MsgIn& in, uint32_t n_msgs, uint8_t* status,
                      const uint8_t* headers = nullptr, const uint64_t* hdr_off = nullptr, IssuerSet* S = nullptr,
                      const uint32_t* item_issuer = nullptr) {
#ifndef BBS_HOSTSIM
        if (!hdr_off && !S && n >= 2 * VERIFY_CHUNK) return verify_chunked(c, n, sigs, in, n_msgs, status);
#endif
        rt_stream_t s = c->stream;
        ItemKeyView item{};
        if (hdr_off) TRY(item_keys(c, n, headers, hdr_off, item));
        if (S) TRY(stage(S->item_issuer, item_issuer, n * 4, s));
        TRY(stage(c->s_sigs, sigs, n * SIG, s));
        TRY(c->s_status.reserve(n));
        TRY(stage_scalars(c, n * n_msgs, in, c->s_msgs, c->s_offsets, c->s_scalars, true));
        TRY(core_verify_dev(c, n, (const uint8_t*)c->s_sigs.p, (const uint8_t*)c->s_scalars.p, n_msgs, (uint8_t*)c->s_status.p,
                            s, S, hdr_off ? &item : nullptr));
        return finish_status(c, n, status);
    }
#ifndef BBS_HOSTSIM
    // Host buffers of a LARGE signing batch (>= 2 * SIGN_CHUNK items), in up to 8 chunks of doubling size: all uploads are queued on the copy
    // stream with one event per chunk, the compute stream hashes and signs chunk k while chunk k + 1 is in flight, and a
    // third stream brings the signatures of chunk k - 1 back (H2D and D2H run on separate copy engines).  The items are
    // independent, so the results are those of the one-shot path; 1.7 GB per 4 M signatures cross the bus either way.
    // Chunk sizes double from SIGN_CHUNK: the first upload (the only one nothing hides) is small, and few launches keep the
    // kernel's tail effects (~3 % per launch at 524,288 items) down.
    static constexpr size_t SIGN_CHUNK = 262144;
    static int sign_chunked(Ctx* c, const uint8_t* sk, size_t n, const MsgIn& in, uint32_t n_msgs, uint8_t* sigs_out,
                            uint8_t* b_out, uint8_t* status) {
        rt_stream_t s = c->stream;
        size_t bounds[9];
        const int n_chunks = plan_chunks(n, SIGN_CHUNK, true, bounds);
        TRY(c->s_out.reserve(n * SIG));
        TRY(c->s_out2.reserve(n * C::G1_BYTES));
        TRY(c->s_status.reserve(n));
        if (!c->down_stream) RT_CHECK(cudaStreamCreateWithFlags(&c->down_stream, cudaStreamNonBlocking));
        if (!c->comp_done[0]) for (auto& e : c->comp_done) RT_CHECK(cudaEventCreateWithFlags(&e, cudaEventDisableTiming));
        TRY(rt_memset(c->s_out.p, 0, n * SIG, s));
        TRY(upload_chunks(c, n, n_chunks, bounds, nullptr, in, n_msgs, s));
        int rc = BBS_OK;
        for (int k = 0; k < n_chunks && !rc; k++) {
            const size_t i0 = bounds[k], i1 = bounds[k + 1], m0 = i0 * n_msgs, m1 = i1 * n_msgs, cnt = i1 - i0;
            RT_CHECK(cudaStreamWaitEvent(s, c->copy_done[k], 0));
            if (in.off) rc = h2s_dev(c, m1 - m0, (const uint8_t*)c->s_msgs.p, (const uint64_t*)c->s_offsets.p + m0,
                                     (uint8_t*)c->s_scalars.p + m0 * 32, s);
            if (!rc) rc = core_sign_dev(c, sk, cnt, (const uint8_t*)c->s_scalars.p + m0 * 32, n_msgs, (uint8_t*)c->s_out.p + i0 * SIG,
                                        b_out ? (uint8_t*)c->s_out2.p + i0 * C::G1_BYTES : nullptr, (uint8_t*)c->s_status.p + i0, s);
            if (rc) break;
            RT_CHECK(cudaEventRecord(c->comp_done[k], s));
            RT_CHECK(cudaStreamWaitEvent(c->down_stream, c->comp_done[k], 0));
            rc = rt_d2h(sigs_out + i0 * SIG, (uint8_t*)c->s_out.p + i0 * SIG, cnt * SIG, c->down_stream);
            if (!rc && b_out) rc = rt_d2h(b_out + i0 * C::G1_BYTES, (uint8_t*)c->s_out2.p + i0 * C::G1_BYTES, cnt * C::G1_BYTES, c->down_stream);
            if (!rc) rc = rt_d2h(status + i0, (uint8_t*)c->s_status.p + i0, cnt, c->down_stream);
        }
        // the signer's staging copies of the messages and their scalars do not outlive the call (also on an error path:
        // everything queued so far is drained first)
        cudaStreamSynchronize(c->copy_stream);
        int rc2 = rt_memset(c->s_scalars.p, 0, n * n_msgs * 32, s);
        if (!rc2 && c->s_msgs.p && c->s_msgs.cap) rc2 = rt_memset(c->s_msgs.p, 0, c->s_msgs.cap, s);
        cudaStreamSynchronize(c->down_stream);
        const int rc3 = rt_sync(s);
        return rc ? rc : (rc2 ? rc2 : rc3);
    }
#endif
    // sign / core_sign; hdr_off != nullptr: a header per item (bbs_*sign_batch_hdr)
    static int sign(Ctx* c, const uint8_t* sk, size_t n, const MsgIn& in, uint32_t n_msgs, uint8_t* sigs_out, uint8_t* b_out,
                    uint8_t* status, const uint8_t* headers = nullptr, const uint64_t* hdr_off = nullptr) {
#ifndef BBS_HOSTSIM
        if (!hdr_off && n >= 2 * SIGN_CHUNK) return sign_chunked(c, sk, n, in, n_msgs, sigs_out, b_out, status);
#endif
        rt_stream_t s = c->stream;
        ItemKeyView item{};
        if (hdr_off) TRY(item_keys(c, n, headers, hdr_off, item));
        TRY(stage_scalars(c, n * n_msgs, in, c->s_msgs, c->s_offsets, c->s_scalars, true));
        TRY(c->s_out.reserve(n * SIG));
        TRY(c->s_out2.reserve(n * C::G1_BYTES));
        TRY(c->s_status.reserve(n));
        TRY(rt_memset(c->s_out.p, 0, n * SIG, s));
        TRY(core_sign_dev(c, sk, n, (const uint8_t*)c->s_scalars.p, n_msgs, (uint8_t*)c->s_out.p,
                          b_out ? (uint8_t*)c->s_out2.p : nullptr, (uint8_t*)c->s_status.p, s, hdr_off ? &item : nullptr));
        TRY(rt_d2h(sigs_out, c->s_out.p, n * SIG, s));
        if (b_out) TRY(rt_d2h(b_out, c->s_out2.p, n * C::G1_BYTES, s));
        // the signer's staging copies of the messages and their scalars do not outlive the call
        TRY(rt_memset(c->s_scalars.p, 0, n * (size_t)n_msgs * 32, s));
        if (c->s_msgs.p && c->s_msgs.cap) TRY(rt_memset(c->s_msgs.p, 0, c->s_msgs.cap, s));
        return finish_status(c, n, status);
    }
    // proof_verify / core_proof_verify: `dis` holds the disclosed messages (or their scalars); ph_off != nullptr: per-item
    // phs in `ph`; hdr_off != nullptr: per-item headers (bbs_*proof_verify_batch_hdr); S != nullptr: the issuer of each
    // item in item_issuer (bbs_*proof_verify_batch_multi, c = S->base); rlc != nullptr: the pairing half by one random
    // linear combination (bbs_rlc_*proof_verify_batch*)
    static int proof_verify(Ctx* c, size_t n, const uint8_t* proofs, const uint8_t* commit, const uint64_t* commit_off,
                            const uint32_t* idx, const MsgIn& dis, const uint64_t* dis_off, const uint8_t* ph, size_t ph_len,
                            uint8_t* status, IssuerSet* S = nullptr, const uint32_t* item_issuer = nullptr,
                            const uint64_t* ph_off = nullptr, const uint8_t* headers = nullptr, const uint64_t* hdr_off = nullptr,
                            const RlcProofIn* rlc = nullptr) {
        rt_stream_t s = c->stream;
        TRY(stage_scalars(c, dis_off[n], dis, c->s_dis_msgs, c->s_dis_msg_off, c->s_dis_scalars, false));
        ItemKeyView item{};
        if (hdr_off) TRY(item_keys(c, n, headers, hdr_off, item));
        if (ph_off) {
            ph_len = ph_off[n];
            TRY(stage(c->s_ph_off, ph_off, (n + 1) * 8, s));
        }
        if (S) TRY(stage(S->item_issuer, item_issuer, n * 4, s));
        TRY(stage(c->s_sigs, proofs, n * PROOF, s));
        TRY(stage(c->s_commit, commit, commit_off[n] * 32, s));
        TRY(stage(c->s_commit_off, commit_off, (n + 1) * 8, s));
        TRY(stage(c->s_dis_idx, idx, dis_off[n] * 4, s));
        TRY(stage(c->s_dis_off, dis_off, (n + 1) * 8, s));
        TRY(stage(c->s_ph, ph, ph_len, s));
        TRY(c->s_status.reserve(n));
        TRY(core_proof_verify_dev(c, n, (const uint8_t*)c->s_sigs.p, (const uint8_t*)c->s_commit.p,
                                  (const uint64_t*)c->s_commit_off.p, (const uint32_t*)c->s_dis_idx.p,
                                  (const uint8_t*)c->s_dis_scalars.p, (const uint64_t*)c->s_dis_off.p,
                                  (const uint8_t*)c->s_ph.p, ph_len, (uint8_t*)c->s_status.p, s, S, hdr_off ? &item : nullptr,
                                  ph_off ? (const uint64_t*)c->s_ph_off.p : nullptr, rlc));
        return finish_status(c, n, status);
    }
};

#include "selftest_host.inc"
#include "imad_peak.inc"

Ctx* as_ctx(bbs_ctx* p) { return reinterpret_cast<Ctx*>(p); }

// 32 bytes from the operating system's CSPRNG: the default coefficient seed of the random-linear-combination mode, drawn
// after the batch has been handed over (a seed the submitter of the batch can predict voids the mode's soundness)
int fresh_seed(uint8_t out[32]) {
    FILE* f = fopen("/dev/urandom", "rb");
    const size_t got = f ? fread(out, 1, 32, f) : 0;
    if (f) fclose(f);
    if (got != 32) { rt_set_error("rlc", "cannot read /dev/urandom for the coefficient seed"); return -1; }
    return 0;
}

// per-item headers (hdr_off != NULL) need a context created with the flag
int check_hdr_flag(Ctx* c, const uint64_t* hdr_off) {
    if (c && hdr_off && !c->per_item_header) return arg_error("per-item headers need a context created with BBS_CTX_PER_ITEM_HEADER");
    return BBS_OK;
}
// the per-item header arguments of a *_hdr call: `required` (verify / sign) or NULL = the context's header (proofs)
int check_hdr_args(Ctx* c, size_t n, const uint8_t* headers, const uint64_t* hdr_off, bool required) {
    if (!c) return arg_error("null context");
    if (!hdr_off) return required ? arg_error("hdr_off is null") : BBS_OK;
    TRY(check_hdr_flag(c, hdr_off));
    return check_items(n, headers, hdr_off, "header");
}
// the flat commitment and disclosed-index counts of a proof call
int check_flat_counts(size_t n, const uint64_t* commit_off, const uint64_t* dis_off) {
    if (commit_off[n] > 0xffffffffull || dis_off[n] > 0xffffffffull) return arg_error("batch too large: flat counts must fit in 32 bits");
    return BBS_OK;
}
#define DISPATCH(c, call)                                              \
    do {                                                               \
        if (!(c)) return arg_error("null context");                    \
        if (rt_set_device((c)->device)) return BBS_E_CUDA;             \
        if ((c)->curve == BBS_CURVE_BLS12_381) return Impl<Bls>::call; \
        return Impl<Bn>::call;                                         \
    } while (0)

}  // namespace

extern "C" {

size_t bbs_g1_bytes(int curve) { return curve == BBS_CURVE_BLS12_381 ? 48 : (curve == BBS_CURVE_BN254 ? 32 : 0); }
size_t bbs_g2_bytes(int curve) { return 2 * bbs_g1_bytes(curve); }
size_t bbs_signature_bytes(int curve) { return bbs_g1_bytes(curve) ? bbs_g1_bytes(curve) + 32 : 0; }
size_t bbs_proof_fixed_bytes(int curve) { return bbs_g1_bytes(curve) ? 3 * bbs_g1_bytes(curve) + 128 : 0; }
const char* bbs_last_error(void) { return rt_errbuf(); }

int bbs_create_generators(int curve, int device, const uint8_t* api_id, size_t api_id_len, uint32_t count, uint8_t* out) {
    if (curve != BBS_CURVE_BLS12_381 && curve != BBS_CURVE_BN254) return arg_error("unknown curve id");
    if (!out || (api_id_len && !api_id)) return arg_error("null");
    if (api_id_len > 128) return arg_error("api_id too long");
    if (count == 0) return BBS_OK;
    if (rt_set_device(device)) return BBS_E_CUDA;
    const size_t gb = bbs_g1_bytes(curve);
    DevBuf d_api, d_v, d_out;
    int rc = d_api.reserve(api_id_len + 1);
    if (!rc) rc = d_v.reserve((size_t)count * 48);
    if (!rc) rc = d_out.reserve((size_t)count * gb);
    if (!rc) rc = rt_h2d(d_api.p, api_id, api_id_len, nullptr);
    if (!rc) {
        GenSeedArgs sa{(const uint8_t*)d_api.p, (uint32_t)api_id_len, count, (uint8_t*)d_v.p};
        rc = launch_gen_seed(sa, nullptr);
    }
    if (!rc) {
        GenPointArgs pa{(const uint8_t*)d_api.p, (uint32_t)api_id_len, (const uint8_t*)d_v.p, (uint8_t*)d_out.p};
        rc = curve == BBS_CURVE_BLS12_381 ? launch_gen_point<Bls>(pa, count, nullptr) : launch_gen_point<Bn>(pa, count, nullptr);
    }
    if (!rc) rc = rt_d2h(out, d_out.p, (size_t)count * gb, nullptr);
    if (!rc) rc = rt_sync(nullptr);
    d_api.release(); d_v.release(); d_out.release();
    return rc;
}

int bbs_ctx_create_ex(int curve, int device, uint32_t flags, const uint8_t* pk, const uint8_t* generators, uint32_t n_generators,
                      const uint8_t* header, size_t header_len, const uint8_t* api_id, size_t api_id_len, bbs_ctx** out) {
    if (!out) return arg_error("out is null");
    *out = nullptr;
    if (curve != BBS_CURVE_BLS12_381 && curve != BBS_CURVE_BN254) return arg_error("unknown curve id");
    if (flags & ~(uint32_t)(BBS_CTX_SMALL_TABLES | BBS_CTX_PER_ITEM_HEADER)) return arg_error("unknown context flag");
    if (!pk || !generators || n_generators < 1) return arg_error("pk / generators missing");
    if (n_generators - 1 > BBS_MAX_MESSAGES) return arg_error("too many generators");
    if ((header_len && !header) || (api_id_len && !api_id)) return arg_error("null header / api_id");
    if (rt_set_device(device)) return BBS_E_CUDA;
    Ctx* c = new (std::nothrow) Ctx();
    if (!c) return arg_error("out of host memory");
    c->curve = curve; c->device = device;
    int rc = rt_stream_create(&c->stream);
    if (!rc) {
        rc = curve == BBS_CURVE_BLS12_381
                 ? Impl<Bls>::create(c, pk, generators, n_generators, header, header_len, api_id, api_id_len, flags)
                 : Impl<Bn>::create(c, pk, generators, n_generators, header, header_len, api_id, api_id_len, flags);
    }
    if (rc) { c->release_all(); rt_stream_destroy(c->stream); delete c; return rc; }
    *out = reinterpret_cast<bbs_ctx*>(c);
    return BBS_OK;
}
int bbs_ctx_create(int curve, int device, const uint8_t* pk, const uint8_t* generators, uint32_t n_generators,
                   const uint8_t* header, size_t header_len, const uint8_t* api_id, size_t api_id_len, bbs_ctx** out) {
    return bbs_ctx_create_ex(curve, device, 0, pk, generators, n_generators, header, header_len, api_id, api_id_len, out);
}

void bbs_ctx_destroy(bbs_ctx* p) {
    Ctx* c = as_ctx(p);
    if (!c) return;
    rt_set_device(c->device);
    rt_sync(c->stream);
    // batch inputs (messages, scalars, signatures, random scalars of the prover) are wiped before the memory goes back
    for (DevBuf* b : {&c->s_sk, &c->s_rand, &c->s_scalars, &c->s_msgs, &c->s_sigs, &c->s_dis_scalars, &c->s_dis_msgs, &c->s_commit,
                      &c->s_out, &c->s_out2, &c->s_rlc_sc, &c->s_msm_kv})
        if (b->p && b->cap) rt_memset(b->p, 0, b->cap, c->stream);
    rt_sync(c->stream);
    c->release_all();
    c->prof.release();
#ifndef BBS_HOSTSIM
    for (auto& e : c->copy_done) if (e) cudaEventDestroy(e);
    for (auto& e : c->comp_done) if (e) cudaEventDestroy(e);
    if (c->copy_stream) cudaStreamDestroy(c->copy_stream);
    if (c->down_stream) cudaStreamDestroy(c->down_stream);
#endif
    rt_stream_destroy(c->stream);
    delete c;
}

int bbs_ctx_domain(bbs_ctx* p, uint8_t out[32]) {
    Ctx* c = as_ctx(p);
    if (!c || !out) return arg_error("null");
    if (rt_set_device(c->device)) return BBS_E_CUDA;
    TRY(rt_d2h(out, c->domain.p, 32, c->stream));
    return rt_sync(c->stream);
}

uint64_t bbs_ctx_launch_count(bbs_ctx* p) { return p ? as_ctx(p)->launches : 0; }

const char* bbs_build_info(void) {
#ifdef BBS_HOSTSIM
    return "host-simulation (tests only; not a product build)";
#else
    return "cuda sm_100a";
#endif
}

int bbs_ctx_set_rlc_windows(bbs_ctx* p, uint32_t windows) {
    if (!p) return arg_error("null context");
    if (windows != 0 && (windows < 8 || windows > 32)) return arg_error("windows must be 0 (cost model) or 8..32");
    as_ctx(p)->rlc_windows = windows;
    return BBS_OK;
}

int bbs_ctx_set_g1_split(bbs_ctx* p, size_t max_items) {
    if (!p) return arg_error("null context");
    as_ctx(p)->split_max = max_items;
    return BBS_OK;
}

int bbs_ctx_set_pairing_split(bbs_ctx* p, size_t max_items) {
    if (!p) return arg_error("null context");
    as_ctx(p)->pair_split_max = (uint32_t)std::min<size_t>(max_items, 32);
    return BBS_OK;
}

int bbs_ctx_use_per_thread_pairing(bbs_ctx* p, int on) {
    if (!p) return arg_error("null context");
    as_ctx(p)->force_per_thread = on != 0;
    return BBS_OK;
}

int bbs_ctx_set_profiling(bbs_ctx* p, int on) {
    if (!p) return arg_error("null context");
    as_ctx(p)->profile = on != 0;
    return BBS_OK;
}
int bbs_ctx_kernel_times(bbs_ctx* p, float* ms, int n) {
    Ctx* c = as_ctx(p);
    if (!c || !ms) return arg_error("null");
    if (rt_set_device(c->device)) return BBS_E_CUDA;
    return c->prof.read(ms, n);
}
int bbs_imad_peak(int device, int iters, int mode, double* gprod_per_s, float* ms_out) {
    if (rt_set_device(device)) return BBS_E_CUDA;
    return imad_peak(iters, mode, gprod_per_s, ms_out);
}

int bbs_msg_to_scalars(bbs_ctx* p, size_t count, const uint8_t* msgs, const uint64_t* off, uint8_t* out) {
    Ctx* c = as_ctx(p);
    if (count && (!off || !out)) return arg_error("null");
    if (!count) return BBS_OK;
    CHECK_COUNTS(count, 1);
    DISPATCH(c, msg_to_scalars(c, count, msgs, off, out));
}
int bbs_core_verify_batch(bbs_ctx* p, size_t n, const uint8_t* sigs, const uint8_t* scalars, uint32_t n_msgs, uint8_t* status) {
    Ctx* c = as_ctx(p);
    if (!n) return BBS_OK;
    if (!sigs || !status || (n_msgs && !scalars)) return arg_error("null");
    CHECK_COUNTS(n, n_msgs);
    DISPATCH(c, verify(c, n, sigs, MsgIn{scalars, nullptr, nullptr}, n_msgs, status));
}
int bbs_verify_batch(bbs_ctx* p, size_t n, const uint8_t* sigs, const uint8_t* msgs, const uint64_t* off, uint32_t n_msgs,
                     uint8_t* status) {
    Ctx* c = as_ctx(p);
    if (!n) return BBS_OK;
    if (!sigs || !status || !off) return arg_error("null");
    CHECK_COUNTS(n, n_msgs);
    DISPATCH(c, verify(c, n, sigs, MsgIn{nullptr, msgs, off}, n_msgs, status));
}
int bbs_core_sign_batch(bbs_ctx* p, const uint8_t sk[32], size_t n, const uint8_t* scalars, uint32_t n_msgs,
                        uint8_t* sigs_out, uint8_t* b_out, uint8_t* status) {
    Ctx* c = as_ctx(p);
    if (!n) return BBS_OK;
    if (!sk || !sigs_out || !status || (n_msgs && !scalars)) return arg_error("null");
    CHECK_COUNTS(n, n_msgs);
    DISPATCH(c, sign(c, sk, n, MsgIn{scalars, nullptr, nullptr}, n_msgs, sigs_out, b_out, status));
}
int bbs_sign_batch(bbs_ctx* p, const uint8_t sk[32], size_t n, const uint8_t* msgs, const uint64_t* off, uint32_t n_msgs,
                   uint8_t* sigs_out, uint8_t* b_out, uint8_t* status) {
    Ctx* c = as_ctx(p);
    if (!n) return BBS_OK;
    if (!sk || !sigs_out || !status || !off) return arg_error("null");
    CHECK_COUNTS(n, n_msgs);
    DISPATCH(c, sign(c, sk, n, MsgIn{nullptr, msgs, off}, n_msgs, sigs_out, b_out, status));
}
int bbs_core_proof_verify_batch(bbs_ctx* p, size_t n, const uint8_t* proofs, const uint8_t* commit,
                                const uint64_t* commit_off, const uint32_t* idx, const uint8_t* dis_scalars,
                                const uint64_t* dis_off, const uint8_t* ph, size_t ph_len, uint8_t* status) {
    Ctx* c = as_ctx(p);
    if (!n) return BBS_OK;
    if (!proofs || !commit_off || !dis_off || !status) return arg_error("null");
    CHECK_COUNTS(n, 1);
    TRY(check_flat_counts(n, commit_off, dis_off));
    DISPATCH(c, proof_verify(c, n, proofs, commit, commit_off, idx, MsgIn{dis_scalars, nullptr, nullptr}, dis_off, ph, ph_len, status));
}
int bbs_proof_verify_batch(bbs_ctx* p, size_t n, const uint8_t* proofs, const uint8_t* commit, const uint64_t* commit_off,
                           const uint32_t* idx, const uint8_t* dis_msgs, const uint64_t* dis_msg_off,
                           const uint64_t* dis_off, const uint8_t* ph, size_t ph_len, uint8_t* status) {
    Ctx* c = as_ctx(p);
    if (!n) return BBS_OK;
    if (!proofs || !commit_off || !dis_off || !dis_msg_off || !status) return arg_error("null");
    CHECK_COUNTS(n, 1);
    TRY(check_flat_counts(n, commit_off, dis_off));
    DISPATCH(c, proof_verify(c, n, proofs, commit, commit_off, idx, MsgIn{nullptr, dis_msgs, dis_msg_off}, dis_off, ph, ph_len, status));
}

int bbs_core_proof_gen_batch(bbs_ctx* p, size_t n, const uint8_t* sigs, const uint8_t* scalars, uint32_t n_msgs,
                             const uint32_t* idx, const uint64_t* dis_off, const uint8_t* rand, const uint64_t* rand_off,
                             const uint64_t* commit_off, const uint8_t* ph, size_t ph_len, uint8_t* proofs_out,
                             uint8_t* commitments_out, uint8_t* status) {
    Ctx* c = as_ctx(p);
    if (!n) return BBS_OK;
    if (!sigs || !dis_off || !rand || !rand_off || !commit_off || !proofs_out || !status) return arg_error("null");
    CHECK_COUNTS(n, n_msgs);
    if (n_msgs > BBS_MAX_MESSAGES) return arg_error("n_msgs exceeds BBS_MAX_MESSAGES");
    DISPATCH(c, proof_gen(c, n, sigs, MsgIn{scalars, nullptr, nullptr}, n_msgs, idx, dis_off, rand, rand_off, commit_off, ph,
                          ph_len, proofs_out, commitments_out, status));
}
int bbs_proof_gen_batch(bbs_ctx* p, size_t n, const uint8_t* sigs, const uint8_t* msgs, const uint64_t* off, uint32_t n_msgs,
                        const uint32_t* idx, const uint64_t* dis_off, const uint8_t* rand, const uint64_t* rand_off,
                        const uint64_t* commit_off, const uint8_t* ph, size_t ph_len, uint8_t* proofs_out,
                        uint8_t* commitments_out, uint8_t* status) {
    Ctx* c = as_ctx(p);
    if (!n) return BBS_OK;
    if (!sigs || !off || !dis_off || !rand || !rand_off || !commit_off || !proofs_out || !status) return arg_error("null");
    CHECK_COUNTS(n, n_msgs);
    if (n_msgs > BBS_MAX_MESSAGES) return arg_error("n_msgs exceeds BBS_MAX_MESSAGES");
    DISPATCH(c, proof_gen(c, n, sigs, MsgIn{nullptr, msgs, off}, n_msgs, idx, dis_off, rand, rand_off, commit_off, ph, ph_len,
                          proofs_out, commitments_out, status));
}

// ---- per-item headers and presentation headers ------------------------------------------------------------------
int bbs_core_verify_batch_hdr(bbs_ctx* p, size_t n, const uint8_t* sigs, const uint8_t* scalars, uint32_t n_msgs,
                              const uint8_t* headers, const uint64_t* hdr_off, uint8_t* status) {
    Ctx* c = as_ctx(p);
    if (!n) return BBS_OK;
    if (!sigs || !status || (n_msgs && !scalars)) return arg_error("null");
    CHECK_COUNTS(n, n_msgs);
    TRY(check_hdr_args(c, n, headers, hdr_off, true));
    DISPATCH(c, verify(c, n, sigs, MsgIn{scalars, nullptr, nullptr}, n_msgs, status, headers, hdr_off));
}
int bbs_verify_batch_hdr(bbs_ctx* p, size_t n, const uint8_t* sigs, const uint8_t* msgs, const uint64_t* off, uint32_t n_msgs,
                         const uint8_t* headers, const uint64_t* hdr_off, uint8_t* status) {
    Ctx* c = as_ctx(p);
    if (!n) return BBS_OK;
    if (!sigs || !status || !off) return arg_error("null");
    CHECK_COUNTS(n, n_msgs);
    TRY(check_hdr_args(c, n, headers, hdr_off, true));
    DISPATCH(c, verify(c, n, sigs, MsgIn{nullptr, msgs, off}, n_msgs, status, headers, hdr_off));
}
int bbs_core_sign_batch_hdr(bbs_ctx* p, const uint8_t sk[32], size_t n, const uint8_t* scalars, uint32_t n_msgs,
                            const uint8_t* headers, const uint64_t* hdr_off, uint8_t* sigs_out, uint8_t* b_out, uint8_t* status) {
    Ctx* c = as_ctx(p);
    if (!n) return BBS_OK;
    if (!sk || !sigs_out || !status || (n_msgs && !scalars)) return arg_error("null");
    CHECK_COUNTS(n, n_msgs);
    TRY(check_hdr_args(c, n, headers, hdr_off, true));
    DISPATCH(c, sign(c, sk, n, MsgIn{scalars, nullptr, nullptr}, n_msgs, sigs_out, b_out, status, headers, hdr_off));
}
int bbs_sign_batch_hdr(bbs_ctx* p, const uint8_t sk[32], size_t n, const uint8_t* msgs, const uint64_t* off, uint32_t n_msgs,
                       const uint8_t* headers, const uint64_t* hdr_off, uint8_t* sigs_out, uint8_t* b_out, uint8_t* status) {
    Ctx* c = as_ctx(p);
    if (!n) return BBS_OK;
    if (!sk || !sigs_out || !status || !off) return arg_error("null");
    CHECK_COUNTS(n, n_msgs);
    TRY(check_hdr_args(c, n, headers, hdr_off, true));
    DISPATCH(c, sign(c, sk, n, MsgIn{nullptr, msgs, off}, n_msgs, sigs_out, b_out, status, headers, hdr_off));
}
int bbs_core_proof_verify_batch_hdr(bbs_ctx* p, size_t n, const uint8_t* proofs, const uint8_t* commit,
                                    const uint64_t* commit_off, const uint32_t* idx, const uint8_t* dis_scalars,
                                    const uint64_t* dis_off, const uint8_t* headers, const uint64_t* hdr_off,
                                    const uint8_t* phs, const uint64_t* ph_off, uint8_t* status) {
    Ctx* c = as_ctx(p);
    if (!n) return BBS_OK;
    if (!proofs || !commit_off || !dis_off || !status || !ph_off) return arg_error("null");
    CHECK_COUNTS(n, 1);
    TRY(check_flat_counts(n, commit_off, dis_off));
    TRY(check_hdr_args(c, n, headers, hdr_off, false));
    TRY(check_items(n, phs, ph_off, "ph"));
    DISPATCH(c, proof_verify(c, n, proofs, commit, commit_off, idx, MsgIn{dis_scalars, nullptr, nullptr}, dis_off, phs, 0, status,
                             nullptr, nullptr, ph_off, headers, hdr_off));
}
int bbs_proof_verify_batch_hdr(bbs_ctx* p, size_t n, const uint8_t* proofs, const uint8_t* commit, const uint64_t* commit_off,
                               const uint32_t* idx, const uint8_t* dis_msgs, const uint64_t* dis_msg_off, const uint64_t* dis_off,
                               const uint8_t* headers, const uint64_t* hdr_off, const uint8_t* phs, const uint64_t* ph_off,
                               uint8_t* status) {
    Ctx* c = as_ctx(p);
    if (!n) return BBS_OK;
    if (!proofs || !commit_off || !dis_off || !dis_msg_off || !status || !ph_off) return arg_error("null");
    CHECK_COUNTS(n, 1);
    TRY(check_flat_counts(n, commit_off, dis_off));
    TRY(check_hdr_args(c, n, headers, hdr_off, false));
    TRY(check_items(n, phs, ph_off, "ph"));
    DISPATCH(c, proof_verify(c, n, proofs, commit, commit_off, idx, MsgIn{nullptr, dis_msgs, dis_msg_off}, dis_off, phs, 0, status,
                             nullptr, nullptr, ph_off, headers, hdr_off));
}
int bbs_core_proof_gen_batch_hdr(bbs_ctx* p, size_t n, const uint8_t* sigs, const uint8_t* scalars, uint32_t n_msgs,
                                 const uint32_t* idx, const uint64_t* dis_off, const uint8_t* rand, const uint64_t* rand_off,
                                 const uint64_t* commit_off, const uint8_t* headers, const uint64_t* hdr_off, const uint8_t* phs,
                                 const uint64_t* ph_off, uint8_t* proofs_out, uint8_t* commitments_out, uint8_t* status) {
    Ctx* c = as_ctx(p);
    if (!n) return BBS_OK;
    if (!sigs || !dis_off || !rand || !rand_off || !commit_off || !proofs_out || !status || !ph_off) return arg_error("null");
    CHECK_COUNTS(n, n_msgs);
    if (n_msgs > BBS_MAX_MESSAGES) return arg_error("n_msgs exceeds BBS_MAX_MESSAGES");
    TRY(check_hdr_args(c, n, headers, hdr_off, false));
    TRY(check_items(n, phs, ph_off, "ph"));
    DISPATCH(c, proof_gen(c, n, sigs, MsgIn{scalars, nullptr, nullptr}, n_msgs, idx, dis_off, rand, rand_off, commit_off, phs, 0,
                          proofs_out, commitments_out, status, ph_off, headers, hdr_off));
}
int bbs_proof_gen_batch_hdr(bbs_ctx* p, size_t n, const uint8_t* sigs, const uint8_t* msgs, const uint64_t* off, uint32_t n_msgs,
                            const uint32_t* idx, const uint64_t* dis_off, const uint8_t* rand, const uint64_t* rand_off,
                            const uint64_t* commit_off, const uint8_t* headers, const uint64_t* hdr_off, const uint8_t* phs,
                            const uint64_t* ph_off, uint8_t* proofs_out, uint8_t* commitments_out, uint8_t* status) {
    Ctx* c = as_ctx(p);
    if (!n) return BBS_OK;
    if (!sigs || !off || !dis_off || !rand || !rand_off || !commit_off || !proofs_out || !status || !ph_off) return arg_error("null");
    CHECK_COUNTS(n, n_msgs);
    if (n_msgs > BBS_MAX_MESSAGES) return arg_error("n_msgs exceeds BBS_MAX_MESSAGES");
    TRY(check_hdr_args(c, n, headers, hdr_off, false));
    TRY(check_items(n, phs, ph_off, "ph"));
    DISPATCH(c, proof_gen(c, n, sigs, MsgIn{nullptr, msgs, off}, n_msgs, idx, dis_off, rand, rand_off, commit_off, phs, 0,
                          proofs_out, commitments_out, status, ph_off, headers, hdr_off));
}

// ---- issuer sets (multi-issuer batches) -------------------------------------------------------------------
int bbs_issuer_set_create(int curve, int device, size_t n_issuers, const uint8_t* pks, const uint8_t* generators,
                          uint32_t n_generators, const uint8_t* header, size_t header_len, const uint8_t* api_id,
                          size_t api_id_len, uint8_t* issuer_status, bbs_issuer_set** out) {
    if (!out) return arg_error("out is null");
    *out = nullptr;
    if (!n_issuers || !pks || !issuer_status) return arg_error("issuer keys / status missing");
    if (n_issuers > 0xffffffffull) return arg_error("too many issuers");
    // the shared part is an ordinary context whose own key is the identity (never used by the multi-issuer calls)
    uint8_t ident[96] = {0};
    if (curve == BBS_CURVE_BLS12_381) ident[0] = 0xc0; else ident[63] = 0x40;
    bbs_ctx* base = nullptr;
    int rc = bbs_ctx_create(curve, device, ident, generators, n_generators, header, header_len, api_id, api_id_len, &base);
    if (rc) return rc;
    IssuerSet* S = new (std::nothrow) IssuerSet();
    if (!S) { bbs_ctx_destroy(base); return arg_error("out of host memory"); }
    S->base = as_ctx(base);
#ifndef BBS_HOSTSIM
    if (!S->base->coop) rc = arg_error("degenerate BP2 line table");
#endif
    if (!rc) rc = curve == BBS_CURVE_BLS12_381 ? Impl<Bls>::issuer_set_build(S, pks, n_issuers, issuer_status)
                                               : Impl<Bn>::issuer_set_build(S, pks, n_issuers, issuer_status);
    if (rc) { S->release_all(); bbs_ctx_destroy(base); delete S; return rc; }
    *out = reinterpret_cast<bbs_issuer_set*>(S);
    return BBS_OK;
}
void bbs_issuer_set_destroy(bbs_issuer_set* p) {
    IssuerSet* S = reinterpret_cast<IssuerSet*>(p);
    if (!S) return;
    rt_set_device(S->base->device);
    rt_sync(S->base->stream);
    S->release_all();
    bbs_ctx_destroy(reinterpret_cast<bbs_ctx*>(S->base));
    delete S;
}
uint64_t bbs_issuer_set_memory_bytes(bbs_issuer_set* p, uint64_t* shared_bytes) {
    IssuerSet* S = reinterpret_cast<IssuerSet*>(p);
    if (!S) return 0;
    if (shared_bytes) *shared_bytes = S->base->bytes() + S->item_issuer.cap;
    return S->per_issuer_bytes();
}
uint64_t bbs_ctx_memory_bytes(bbs_ctx* p) { return p ? as_ctx(p)->bytes() : 0; }

#define DISPATCH_SET(S, call)                                                    \
    do {                                                                         \
        if (!(S)) return arg_error("null issuer set");                           \
        if (rt_set_device((S)->base->device)) return BBS_E_CUDA;                 \
        if ((S)->base->curve == BBS_CURVE_BLS12_381) return Impl<Bls>::call;     \
        return Impl<Bn>::call;                                                   \
    } while (0)

int bbs_verify_batch_multi(bbs_issuer_set* p, size_t n, const uint32_t* item_issuer, const uint8_t* sigs, const uint8_t* msgs,
                           const uint64_t* off, uint32_t n_msgs, uint8_t* status) {
    IssuerSet* S = reinterpret_cast<IssuerSet*>(p);
    if (!n) return BBS_OK;
    if (!item_issuer || !sigs || !status || !off) return arg_error("null");
    CHECK_COUNTS(n, n_msgs);
    DISPATCH_SET(S, verify(S->base, n, sigs, MsgIn{nullptr, msgs, off}, n_msgs, status, nullptr, nullptr, S, item_issuer));
}
int bbs_core_verify_batch_multi(bbs_issuer_set* p, size_t n, const uint32_t* item_issuer, const uint8_t* sigs,
                                const uint8_t* scalars, uint32_t n_msgs, uint8_t* status) {
    IssuerSet* S = reinterpret_cast<IssuerSet*>(p);
    if (!n) return BBS_OK;
    if (!item_issuer || !sigs || !status || (n_msgs && !scalars)) return arg_error("null");
    CHECK_COUNTS(n, n_msgs);
    DISPATCH_SET(S, verify(S->base, n, sigs, MsgIn{scalars, nullptr, nullptr}, n_msgs, status, nullptr, nullptr, S, item_issuer));
}

int bbs_core_proof_verify_batch_multi(bbs_issuer_set* p, size_t n, const uint32_t* item_issuer, const uint8_t* proofs,
                                      const uint8_t* commit, const uint64_t* commit_off, const uint32_t* idx,
                                      const uint8_t* dis_scalars, const uint64_t* dis_off, const uint8_t* ph, size_t ph_len,
                                      uint8_t* status) {
    IssuerSet* S = reinterpret_cast<IssuerSet*>(p);
    if (!n) return BBS_OK;
    if (!item_issuer || !proofs || !commit_off || !dis_off || !status) return arg_error("null");
    CHECK_COUNTS(n, 1);
    TRY(check_flat_counts(n, commit_off, dis_off));
    DISPATCH_SET(S, proof_verify(S->base, n, proofs, commit, commit_off, idx, MsgIn{dis_scalars, nullptr, nullptr}, dis_off, ph,
                                 ph_len, status, S, item_issuer));
}
int bbs_proof_verify_batch_multi(bbs_issuer_set* p, size_t n, const uint32_t* item_issuer, const uint8_t* proofs,
                                 const uint8_t* commit, const uint64_t* commit_off, const uint32_t* idx, const uint8_t* dis_msgs,
                                 const uint64_t* dis_msg_off, const uint64_t* dis_off, const uint8_t* ph, size_t ph_len,
                                 uint8_t* status) {
    IssuerSet* S = reinterpret_cast<IssuerSet*>(p);
    if (!n) return BBS_OK;
    if (!item_issuer || !proofs || !commit_off || !dis_off || !dis_msg_off || !status) return arg_error("null");
    CHECK_COUNTS(n, 1);
    TRY(check_flat_counts(n, commit_off, dis_off));
    DISPATCH_SET(S, proof_verify(S->base, n, proofs, commit, commit_off, idx, MsgIn{nullptr, dis_msgs, dis_msg_off}, dis_off, ph,
                                 ph_len, status, S, item_issuer));
}

// ---- random-linear-combination batch mode ----------------------------------------------------------------
#ifndef BBS_HOSTSIM
int bbs_rlc_partial_core(bbs_ctx* p, size_t n, const uint8_t* sigs, const uint8_t* scalars, uint32_t n_msgs,
                         const uint8_t seed[32], uint64_t index_base, uint8_t* parts_out, uint8_t* status) {
    Ctx* c = as_ctx(p);
    if (!seed || !parts_out || !status || (n && !sigs) || (n && n_msgs && !scalars)) return arg_error("null (shards must share one seed)");
    CHECK_COUNTS(n, n_msgs);
    DISPATCH(c, rlc_partial(c, n, sigs, MsgIn{scalars, nullptr, nullptr}, n_msgs, seed, index_base, parts_out, status));
}
int bbs_rlc_partial(bbs_ctx* p, size_t n, const uint8_t* sigs, const uint8_t* msgs, const uint64_t* off, uint32_t n_msgs,
                    const uint8_t seed[32], uint64_t index_base, uint8_t* parts_out, uint8_t* status) {
    Ctx* c = as_ctx(p);
    if (!seed || !parts_out || !status || !off || (n && !sigs)) return arg_error("null (shards must share one seed)");
    CHECK_COUNTS(n, n_msgs);
    DISPATCH(c, rlc_partial(c, n, sigs, MsgIn{nullptr, msgs, off}, n_msgs, seed, index_base, parts_out, status));
}
int bbs_rlc_combine(bbs_ctx* p, size_t n_parts, const uint8_t* parts, uint8_t* verdict) {
    Ctx* c = as_ctx(p);
    if (!parts || !verdict || !n_parts) return arg_error("null");
    DISPATCH(c, rlc_combine(c, n_parts, parts, verdict));
}
int bbs_rlc_core_verify_batch(bbs_ctx* p, size_t n, const uint8_t* sigs, const uint8_t* scalars, uint32_t n_msgs,
                              const uint8_t seed[32], uint8_t* verdict) {
    Ctx* c = as_ctx(p);
    if (!verdict || (n && !sigs) || (n && n_msgs && !scalars)) return arg_error("null");
    CHECK_COUNTS(n, n_msgs);
    uint8_t fresh[32];
    if (!seed) { if (fresh_seed(fresh)) return BBS_E_ARG; seed = fresh; }
    DISPATCH(c, rlc_verify(c, n, sigs, MsgIn{scalars, nullptr, nullptr}, n_msgs, seed, verdict));
}
int bbs_rlc_verify_batch(bbs_ctx* p, size_t n, const uint8_t* sigs, const uint8_t* msgs, const uint64_t* off,
                         uint32_t n_msgs, const uint8_t seed[32], uint8_t* verdict) {
    Ctx* c = as_ctx(p);
    if (!verdict || !off || (n && !sigs)) return arg_error("null");
    CHECK_COUNTS(n, n_msgs);
    uint8_t fresh[32];
    if (!seed) { if (fresh_seed(fresh)) return BBS_E_ARG; seed = fresh; }
    DISPATCH(c, rlc_verify(c, n, sigs, MsgIn{nullptr, msgs, off}, n_msgs, seed, verdict));
}
// proof verification with the pairing half by one random linear combination: the arguments of the call without rlc_,
// then the seed (NULL = drawn here, after the batch has been handed over) and the combined check's verdict
#define RLC_PROOF_ARGS(seed, combined)                                                                              \
    if (!n) { if (combined) *(combined) = BBS_ST_ACCEPT; return BBS_OK; }                                           \
    if (n >= (1ull << 31)) return arg_error("batch too large for the rlc mode: n must be below 2^31");             \
    uint8_t fresh[32];                                                                                              \
    if (!seed) { if (fresh_seed(fresh)) return BBS_E_ARG; seed = fresh; }                                           \
    const RlcProofIn rlc{seed, combined}
int bbs_rlc_core_proof_verify_batch(bbs_ctx* p, size_t n, const uint8_t* proofs, const uint8_t* commit,
                                    const uint64_t* commit_off, const uint32_t* idx, const uint8_t* dis_scalars,
                                    const uint64_t* dis_off, const uint8_t* ph, size_t ph_len, const uint8_t* seed,
                                    uint8_t* status, uint8_t* combined) {
    Ctx* c = as_ctx(p);
    if (n && (!proofs || !commit_off || !dis_off || !status)) return arg_error("null");
    CHECK_COUNTS(n, 1);
    if (n) TRY(check_flat_counts(n, commit_off, dis_off));
    RLC_PROOF_ARGS(seed, combined);
    DISPATCH(c, proof_verify(c, n, proofs, commit, commit_off, idx, MsgIn{dis_scalars, nullptr, nullptr}, dis_off, ph, ph_len, status,
                             nullptr, nullptr, nullptr, nullptr, nullptr, &rlc));
}
int bbs_rlc_proof_verify_batch(bbs_ctx* p, size_t n, const uint8_t* proofs, const uint8_t* commit, const uint64_t* commit_off,
                               const uint32_t* idx, const uint8_t* dis_msgs, const uint64_t* dis_msg_off,
                               const uint64_t* dis_off, const uint8_t* ph, size_t ph_len, const uint8_t* seed, uint8_t* status,
                               uint8_t* combined) {
    Ctx* c = as_ctx(p);
    if (n && (!proofs || !commit_off || !dis_off || !dis_msg_off || !status)) return arg_error("null");
    CHECK_COUNTS(n, 1);
    if (n) TRY(check_flat_counts(n, commit_off, dis_off));
    RLC_PROOF_ARGS(seed, combined);
    DISPATCH(c, proof_verify(c, n, proofs, commit, commit_off, idx, MsgIn{nullptr, dis_msgs, dis_msg_off}, dis_off, ph, ph_len, status,
                             nullptr, nullptr, nullptr, nullptr, nullptr, &rlc));
}
int bbs_rlc_core_proof_verify_batch_hdr(bbs_ctx* p, size_t n, const uint8_t* proofs, const uint8_t* commit,
                                        const uint64_t* commit_off, const uint32_t* idx, const uint8_t* dis_scalars,
                                        const uint64_t* dis_off, const uint8_t* headers, const uint64_t* hdr_off,
                                        const uint8_t* phs, const uint64_t* ph_off, const uint8_t* seed, uint8_t* status,
                                        uint8_t* combined) {
    Ctx* c = as_ctx(p);
    if (n && (!proofs || !commit_off || !dis_off || !status || !ph_off)) return arg_error("null");
    CHECK_COUNTS(n, 1);
    if (n) {
        TRY(check_flat_counts(n, commit_off, dis_off));
        TRY(check_hdr_args(c, n, headers, hdr_off, false));
        TRY(check_items(n, phs, ph_off, "ph"));
    }
    RLC_PROOF_ARGS(seed, combined);
    DISPATCH(c, proof_verify(c, n, proofs, commit, commit_off, idx, MsgIn{dis_scalars, nullptr, nullptr}, dis_off, phs, 0, status,
                             nullptr, nullptr, ph_off, headers, hdr_off, &rlc));
}
int bbs_rlc_proof_verify_batch_hdr(bbs_ctx* p, size_t n, const uint8_t* proofs, const uint8_t* commit,
                                   const uint64_t* commit_off, const uint32_t* idx, const uint8_t* dis_msgs,
                                   const uint64_t* dis_msg_off, const uint64_t* dis_off, const uint8_t* headers,
                                   const uint64_t* hdr_off, const uint8_t* phs, const uint64_t* ph_off, const uint8_t* seed,
                                   uint8_t* status, uint8_t* combined) {
    Ctx* c = as_ctx(p);
    if (n && (!proofs || !commit_off || !dis_off || !dis_msg_off || !status || !ph_off)) return arg_error("null");
    CHECK_COUNTS(n, 1);
    if (n) {
        TRY(check_flat_counts(n, commit_off, dis_off));
        TRY(check_hdr_args(c, n, headers, hdr_off, false));
        TRY(check_items(n, phs, ph_off, "ph"));
    }
    RLC_PROOF_ARGS(seed, combined);
    DISPATCH(c, proof_verify(c, n, proofs, commit, commit_off, idx, MsgIn{nullptr, dis_msgs, dis_msg_off}, dis_off, phs, 0, status,
                             nullptr, nullptr, ph_off, headers, hdr_off, &rlc));
}
// signature verification with per-item statuses by one random linear combination: the arguments of the call without
// rlc_ and _status, then the seed and the combined check's verdict, as the proof calls above
int bbs_rlc_core_verify_batch_status(bbs_ctx* p, size_t n, const uint8_t* sigs, const uint8_t* scalars, uint32_t n_msgs,
                                     const uint8_t* seed, uint8_t* status, uint8_t* combined) {
    Ctx* c = as_ctx(p);
    if (n && (!sigs || !status || (n_msgs && !scalars))) return arg_error("null");
    CHECK_COUNTS(n, n_msgs);
    RLC_PROOF_ARGS(seed, combined);
    DISPATCH(c, rlc_verify_status(c, n, sigs, MsgIn{scalars, nullptr, nullptr}, n_msgs, rlc, status));
}
int bbs_rlc_verify_batch_status(bbs_ctx* p, size_t n, const uint8_t* sigs, const uint8_t* msgs, const uint64_t* off,
                                uint32_t n_msgs, const uint8_t* seed, uint8_t* status, uint8_t* combined) {
    Ctx* c = as_ctx(p);
    if (n && (!sigs || !status || !off)) return arg_error("null");
    CHECK_COUNTS(n, n_msgs);
    RLC_PROOF_ARGS(seed, combined);
    DISPATCH(c, rlc_verify_status(c, n, sigs, MsgIn{nullptr, msgs, off}, n_msgs, rlc, status));
}
int bbs_rlc_core_verify_batch_status_hdr(bbs_ctx* p, size_t n, const uint8_t* sigs, const uint8_t* scalars, uint32_t n_msgs,
                                         const uint8_t* headers, const uint64_t* hdr_off, const uint8_t* seed, uint8_t* status,
                                         uint8_t* combined) {
    Ctx* c = as_ctx(p);
    if (n && (!sigs || !status || (n_msgs && !scalars))) return arg_error("null");
    CHECK_COUNTS(n, n_msgs);
    if (n) TRY(check_hdr_args(c, n, headers, hdr_off, true));
    RLC_PROOF_ARGS(seed, combined);
    DISPATCH(c, rlc_verify_status(c, n, sigs, MsgIn{scalars, nullptr, nullptr}, n_msgs, rlc, status, headers, hdr_off));
}
int bbs_rlc_verify_batch_status_hdr(bbs_ctx* p, size_t n, const uint8_t* sigs, const uint8_t* msgs, const uint64_t* off,
                                    uint32_t n_msgs, const uint8_t* headers, const uint64_t* hdr_off, const uint8_t* seed,
                                    uint8_t* status, uint8_t* combined) {
    Ctx* c = as_ctx(p);
    if (n && (!sigs || !status || !off)) return arg_error("null");
    CHECK_COUNTS(n, n_msgs);
    if (n) TRY(check_hdr_args(c, n, headers, hdr_off, true));
    RLC_PROOF_ARGS(seed, combined);
    DISPATCH(c, rlc_verify_status(c, n, sigs, MsgIn{nullptr, msgs, off}, n_msgs, rlc, status, headers, hdr_off));
}
#else
int bbs_rlc_partial_core(bbs_ctx*, size_t, const uint8_t*, const uint8_t*, uint32_t, const uint8_t*, uint64_t, uint8_t*, uint8_t*) { rt_set_error("rlc", "needs the CUDA build"); return BBS_E_CUDA; }
int bbs_rlc_partial(bbs_ctx*, size_t, const uint8_t*, const uint8_t*, const uint64_t*, uint32_t, const uint8_t*, uint64_t, uint8_t*, uint8_t*) { rt_set_error("rlc", "needs the CUDA build"); return BBS_E_CUDA; }
int bbs_rlc_combine(bbs_ctx*, size_t, const uint8_t*, uint8_t*) { rt_set_error("rlc", "needs the CUDA build"); return BBS_E_CUDA; }
int bbs_rlc_core_verify_batch(bbs_ctx*, size_t, const uint8_t*, const uint8_t*, uint32_t, const uint8_t*, uint8_t*) { rt_set_error("rlc", "needs the CUDA build"); return BBS_E_CUDA; }
int bbs_rlc_verify_batch(bbs_ctx*, size_t, const uint8_t*, const uint8_t*, const uint64_t*, uint32_t, const uint8_t*, uint8_t*) { rt_set_error("rlc", "needs the CUDA build"); return BBS_E_CUDA; }
int bbs_rlc_core_proof_verify_batch(bbs_ctx*, size_t, const uint8_t*, const uint8_t*, const uint64_t*, const uint32_t*, const uint8_t*, const uint64_t*, const uint8_t*, size_t, const uint8_t*, uint8_t*, uint8_t*) { rt_set_error("rlc", "needs the CUDA build"); return BBS_E_CUDA; }
int bbs_rlc_proof_verify_batch(bbs_ctx*, size_t, const uint8_t*, const uint8_t*, const uint64_t*, const uint32_t*, const uint8_t*, const uint64_t*, const uint64_t*, const uint8_t*, size_t, const uint8_t*, uint8_t*, uint8_t*) { rt_set_error("rlc", "needs the CUDA build"); return BBS_E_CUDA; }
int bbs_rlc_core_proof_verify_batch_hdr(bbs_ctx*, size_t, const uint8_t*, const uint8_t*, const uint64_t*, const uint32_t*, const uint8_t*, const uint64_t*, const uint8_t*, const uint64_t*, const uint8_t*, const uint64_t*, const uint8_t*, uint8_t*, uint8_t*) { rt_set_error("rlc", "needs the CUDA build"); return BBS_E_CUDA; }
int bbs_rlc_proof_verify_batch_hdr(bbs_ctx*, size_t, const uint8_t*, const uint8_t*, const uint64_t*, const uint32_t*, const uint8_t*, const uint64_t*, const uint64_t*, const uint8_t*, const uint64_t*, const uint8_t*, const uint64_t*, const uint8_t*, uint8_t*, uint8_t*) { rt_set_error("rlc", "needs the CUDA build"); return BBS_E_CUDA; }
int bbs_rlc_core_verify_batch_status(bbs_ctx*, size_t, const uint8_t*, const uint8_t*, uint32_t, const uint8_t*, uint8_t*, uint8_t*) { rt_set_error("rlc", "needs the CUDA build"); return BBS_E_CUDA; }
int bbs_rlc_verify_batch_status(bbs_ctx*, size_t, const uint8_t*, const uint8_t*, const uint64_t*, uint32_t, const uint8_t*, uint8_t*, uint8_t*) { rt_set_error("rlc", "needs the CUDA build"); return BBS_E_CUDA; }
int bbs_rlc_core_verify_batch_status_hdr(bbs_ctx*, size_t, const uint8_t*, const uint8_t*, uint32_t, const uint8_t*, const uint64_t*, const uint8_t*, uint8_t*, uint8_t*) { rt_set_error("rlc", "needs the CUDA build"); return BBS_E_CUDA; }
int bbs_rlc_verify_batch_status_hdr(bbs_ctx*, size_t, const uint8_t*, const uint8_t*, const uint64_t*, uint32_t, const uint8_t*, const uint64_t*, const uint8_t*, uint8_t*, uint8_t*) { rt_set_error("rlc", "needs the CUDA build"); return BBS_E_CUDA; }
#endif

int bbs_msg_to_scalars_dev(bbs_ctx* p, size_t count, const uint8_t* d_msgs, const uint64_t* d_off, uint8_t* d_out, void* stream) {
    Ctx* c = as_ctx(p);
    CHECK_COUNTS(count, 1);
    DISPATCH(c, h2s_dev(c, count, d_msgs, d_off, d_out, (rt_stream_t)stream));
}
int bbs_core_verify_batch_dev(bbs_ctx* p, size_t n, const uint8_t* d_sigs, const uint8_t* d_scalars, uint32_t n_msgs,
                              uint8_t* d_status, void* stream) {
    Ctx* c = as_ctx(p);
    CHECK_COUNTS(n, n_msgs);
    DISPATCH(c, core_verify_dev(c, n, d_sigs, d_scalars, n_msgs, d_status, (rt_stream_t)stream));
}
int bbs_verify_batch_dev(bbs_ctx* p, size_t n, const uint8_t* d_sigs, const uint8_t* d_msgs, const uint64_t* d_off,
                         uint32_t n_msgs, uint8_t* d_status, void* stream) {
    Ctx* c = as_ctx(p);
    CHECK_COUNTS(n, n_msgs);
    DISPATCH(c, verify_dev(c, n, d_sigs, d_msgs, d_off, n_msgs, d_status, (rt_stream_t)stream));
}
int bbs_core_sign_batch_dev(bbs_ctx* p, const uint8_t sk[32], size_t n, const uint8_t* d_scalars, uint32_t n_msgs,
                            uint8_t* d_sigs, uint8_t* d_b, uint8_t* d_status, void* stream) {
    Ctx* c = as_ctx(p);
    if (!sk) return arg_error("null");
    CHECK_COUNTS(n, n_msgs);
    DISPATCH(c, core_sign_dev(c, sk, n, d_scalars, n_msgs, d_sigs, d_b, d_status, (rt_stream_t)stream));
}
int bbs_core_proof_verify_batch_dev(bbs_ctx* p, size_t n, const uint8_t* d_proofs, const uint8_t* d_commit,
                                    const uint64_t* d_commit_off, const uint32_t* d_idx, const uint8_t* d_dis_scalars,
                                    const uint64_t* d_dis_off, const uint8_t* d_ph, size_t ph_len, uint8_t* d_status,
                                    void* stream) {
    Ctx* c = as_ctx(p);
    CHECK_COUNTS(n, 1);
    DISPATCH(c, core_proof_verify_dev(c, n, d_proofs, d_commit, d_commit_off, d_idx, d_dis_scalars, d_dis_off, d_ph,
                                      ph_len, d_status, (rt_stream_t)stream));
}

// device-buffer forms: the offsets are device memory and, as for every *_dev call, the caller's contract
int bbs_core_verify_batch_hdr_dev(bbs_ctx* p, size_t n, const uint8_t* d_sigs, const uint8_t* d_scalars, uint32_t n_msgs,
                                  const uint8_t* d_headers, const uint64_t* d_hdr_off, uint8_t* d_status, void* stream) {
    Ctx* c = as_ctx(p);
    CHECK_COUNTS(n, n_msgs);
    if (!d_hdr_off) return arg_error("hdr_off is null");
    TRY(check_hdr_flag(c, d_hdr_off));
    DISPATCH(c, core_verify_hdr_dev(c, n, d_sigs, d_scalars, n_msgs, d_headers, d_hdr_off, d_status, (rt_stream_t)stream));
}
int bbs_core_proof_verify_batch_hdr_dev(bbs_ctx* p, size_t n, const uint8_t* d_proofs, const uint8_t* d_commit,
                                        const uint64_t* d_commit_off, const uint32_t* d_idx, const uint8_t* d_dis_scalars,
                                        const uint64_t* d_dis_off, const uint8_t* d_headers, const uint64_t* d_hdr_off,
                                        const uint8_t* d_phs, const uint64_t* d_ph_off, uint8_t* d_status, void* stream) {
    Ctx* c = as_ctx(p);
    CHECK_COUNTS(n, 1);
    if (!d_ph_off) return arg_error("ph_off is null");
    TRY(check_hdr_flag(c, d_hdr_off));
    DISPATCH(c, core_proof_verify_hdr_dev(c, n, d_proofs, d_commit, d_commit_off, d_idx, d_dis_scalars, d_dis_off, d_headers,
                                          d_hdr_off, d_phs, d_ph_off, d_status, (rt_stream_t)stream));
}

int bbs_selftest_field(int curve, int device, int op, size_t n, const uint8_t* a, const uint8_t* b, uint8_t* out) {
    if (rt_set_device(device)) return BBS_E_CUDA;
    if (curve == BBS_CURVE_BLS12_381) return selftest_field<Bls>(op, n, a, b, out);
    if (curve == BBS_CURVE_BN254) return selftest_field<Bn>(op, n, a, b, out);
    return arg_error("unknown curve id");
}
int bbs_selftest_g1_mul(int curve, int device, size_t n, const uint8_t* pts, const uint8_t* sc, uint8_t* out) {
    if (rt_set_device(device)) return BBS_E_CUDA;
    if (curve == BBS_CURVE_BLS12_381) return selftest_g1_mul<Bls>(n, pts, sc, out);
    if (curve == BBS_CURVE_BN254) return selftest_g1_mul<Bn>(n, pts, sc, out);
    return arg_error("unknown curve id");
}
int bbs_selftest_g1(int curve, int device, int op, size_t n, const uint8_t* p, const uint8_t* q, const uint8_t* sc,
                    uint8_t* out) {
    if (rt_set_device(device)) return BBS_E_CUDA;
    if (curve == BBS_CURVE_BLS12_381) return selftest_g1<Bls>(op, n, p, q, sc, out);
    if (curve == BBS_CURVE_BN254) return selftest_g1<Bn>(op, n, p, q, sc, out);
    return arg_error("unknown curve id");
}
int bbs_selftest_pairing(int curve, int device, size_t n, const uint8_t* p_points, const uint8_t* r_points,
                         const uint8_t* q_point, uint8_t* status) {
    if (rt_set_device(device)) return BBS_E_CUDA;
    if (curve == BBS_CURVE_BLS12_381) return selftest_pairing<Bls>(n, p_points, r_points, q_point, status);
    if (curve == BBS_CURVE_BN254) return selftest_pairing<Bn>(n, p_points, r_points, q_point, status);
    return arg_error("unknown curve id");
}

}  // extern "C"
