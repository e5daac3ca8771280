// Bucket (Pippenger) multi-scalar multiplication for the random-linear-combination mode (rlc.cuh): the two sums
//     S1 = sum r_i A_i          S2' = sum (r_i e_i) A_i            (verify.rs:88-92 folded over the batch)
// are the north star's "two large MSMs per GPU".  Every item contributes three 128-bit values:
//     v0 = r_i                                  -> bucket rows [0, W)            (S1)
//     (v1, v2) = GLV halves of r_i e_i (g1.cuh glv_split), v2 acting on phi(A_i) = (beta x, y)  -> rows [W, 2W), shared
// cut into W digits of near-equal width (digit w = bits [128 w / W, 128 (w + 1) / W), at most c bits: equal bucket loads in
// every row, whatever W).  Pipeline (all on the context's stream):
//     rlc_prep_kernel    decompress A_i, coefficients, GLV split; histogram of the non-zero digits; Fr partial sums
//     msm_scan_kernel    bucket sizes -> offsets (exclusive scan)
//     msm_scatter_kernel item references sorted by bucket (counting sort; order inside a bucket is irrelevant)
//     msm_bucket_kernel  one thread per bucket: sum of its points (Jacobian += affine)
//     msm_reduce_kernel  sum_d d * bucket[d] per row by chunked running sums
//     rlc_msm_finish_kernel   rows -> S1, S2' (Horner over the windows), minus the fixed-base term, compressed
// Same group elements as the per-item scalar multiplications (and as the oracle): only the addition order differs.
#pragma once
#include "rlc.cuh"

#ifdef __CUDACC__
namespace bbs {

struct MsmPlan {
    uint32_t c;          // widest digit, bits: a row holds 2^c buckets
    uint32_t W;          // digits per 128-bit value
    uint32_t rows;       // bucket rows: 2W
    uint32_t chunk;      // buckets per thread in msm_reduce_kernel
    uint32_t red_blocks; // blocks per row in msm_reduce_kernel
};
__device__ __forceinline__ uint32_t msm_digit_start(uint32_t w, uint32_t W) { return (w * 128u) / W; }
__device__ __forceinline__ uint32_t msm_digit_bits(uint32_t w, uint32_t W) { return msm_digit_start(w + 1, W) - msm_digit_start(w, W); }
__device__ __forceinline__ uint32_t msm_digit(const uint32_t* v /*4 words, global*/, uint32_t w, uint32_t W) {
    const uint32_t bit = msm_digit_start(w, W), word = bit >> 5, off = bit & 31;
    uint64_t x = v[word];
    if (word < 3) x |= (uint64_t)v[word + 1] << 32;
    return (uint32_t)(x >> off) & ((1u << msm_digit_bits(w, W)) - 1u);
}
__device__ __forceinline__ uint32_t msm_row(uint32_t stream, uint32_t w, uint32_t W) { return (stream == 0 ? 0u : W) + w; }

struct RlcPrepArgs {
    RlcArgs base;            // pt_part unused
    MsmPlan plan;
    uint32_t* pts;           // n x affine Montgomery
    uint32_t* kv;            // n x 3 x 4 words
    uint32_t* counts;        // rows << c, zeroed by the caller
};
template <class C> __global__ void __launch_bounds__(RLC_TPB, 4) rlc_prep_kernel(const RlcPrepArgs pa) {
    using Fr = typename C::Fr;
    __shared__ BBS_A16 uint32_t ss[RLC_TPB][8];
    const RlcArgs& a = pa.base;
    const uint32_t i = blockIdx.x * RLC_TPB + threadIdx.x;
    const bool valid = i < a.n;
    BBS_A16 uint32_t rm[8], r[8];
    bn_zero<8>(rm);
    bn_zero<8>(r);
    bool ok = true;
    const uint8_t* sc = a.scalars + (size_t)(valid ? i : 0) * a.n_msgs * 32;
    if (valid) {
        const uint8_t* sig = a.sigs + (size_t)i * (C::G1_BYTES + 32);
        BBS_A16 uint32_t A[G1A], e[8], kv[12];
        for (int k = 0; k < 12; k++) kv[k] = 0;
        int st = g1_decompress<C>(A, sig);
        ok = st != PT_BAD && fr_from_le32<C>(e, sig + C::G1_BYTES);
        rlc_coeff(r, a.seed, a.index_base + i);
        fe_to_mont<Fr>(rm, r);
        if (ok && st == PT_OK) {
            BBS_A16 uint32_t ae[8];
            fe_mul<Fr>(ae, rm, e);                  // r_i e_i mod r, canonical
            for (int k = 0; k < 4; k++) kv[k] = r[k];
            BBS_A16 uint32_t k1[5], k2[5];
            glv_split<C>(k1, k2, ae);
            for (int k = 0; k < 4; k++) { kv[4 + k] = k1[k]; kv[8 + k] = k2[k]; }
            uint32_t* dst = pa.pts + (size_t)i * G1A;
            for (int k = 0; k < G1A; k++) dst[k] = A[k];
        }
        uint32_t* kd = pa.kv + (size_t)i * 12;
        for (int k = 0; k < 12; k++) kd[k] = kv[k];
        if (ok && st == PT_OK) {
            const uint32_t c = pa.plan.c, W = pa.plan.W;
            for (uint32_t s = 0; s < 3; s++)
                for (uint32_t w = 0; w < W; w++) {
                    const uint32_t d = msm_digit(kd + 4 * s, w, W);
                    if (d) atomicAdd(pa.counts + ((size_t)msm_row(s, w, W) << c) + d, 1u);
                }
        }
    }
    // scalars: sum r_i, sum r_i m_ij
    uint32_t* scp = a.sc_part + (size_t)blockIdx.x * (a.n_msgs + 1) * 8;
    rlc_block_sum_fr<C>(ss, r);
    if (threadIdx.x == 0) bn_copy<8>(scp, ss[0]);
    __syncthreads();
    for (uint32_t j = 0; j < a.n_msgs; j++) {
        BBS_A16 uint32_t t[8];
        bn_zero<8>(t);
        if (valid && ok) {
            BBS_A16 uint32_t m[8];
            if (fr_from_le32<C>(m, sc + j * 32)) fe_mul<Fr>(t, rm, m); else ok = false;
        }
        rlc_block_sum_fr<C>(ss, t);
        if (threadIdx.x == 0) bn_copy<8>(scp + (j + 1) * 8, ss[0]);
        __syncthreads();
    }
    if (valid && !ok) atomicOr(a.bad, 1u);
}

constexpr int MSM_SCAN_TPB = 1024;
// offsets[b] = sum_{b' < b} counts[b'] (nb + 1 entries); cursor = copy of offsets for the scatter.  One block: every warp
// scans a contiguous slice 32 elements at a time (coalesced loads, shuffle scan), then the slice totals are scanned.
template <int TPB_ = MSM_SCAN_TPB> __global__ void __launch_bounds__(MSM_SCAN_TPB, 1) msm_scan_kernel(const uint32_t* counts, uint32_t* offsets, uint32_t* cursor, uint32_t nb) {
    __shared__ uint32_t wsum[MSM_SCAN_TPB / 32];
    const uint32_t lane = threadIdx.x & 31, warp = threadIdx.x >> 5, nw = MSM_SCAN_TPB / 32;
    const uint32_t per = ((nb + nw - 1) / nw + 31) / 32 * 32;
    const uint32_t lo = min(nb, warp * per), hi = min(nb, lo + per);
    uint32_t s = 0;
    for (uint32_t i = lo + lane; i < hi; i += 32) s += counts[i];
    for (int d = 16; d >= 1; d >>= 1) s += __shfl_xor_sync(0xffffffffu, s, d);
    if (lane == 0) wsum[warp] = s;
    __syncthreads();
    uint32_t run = 0;
    for (uint32_t k = 0; k < warp; k++) run += wsum[k];
    for (uint32_t i0 = lo; i0 < hi; i0 += 32) {
        const uint32_t i = i0 + lane;
        const uint32_t v = i < hi ? counts[i] : 0u;
        uint32_t x = v;
        for (int d = 1; d < 32; d <<= 1) { uint32_t y = __shfl_up_sync(0xffffffffu, x, d); if (lane >= (uint32_t)d) x += y; }
        if (i < hi) { offsets[i] = run + x - v; cursor[i] = run + x - v; }
        run += __shfl_sync(0xffffffffu, x, 31);
    }
    if (warp == nw - 1 && lane == 0) offsets[nb] = run;
}

struct MsmScatterArgs { MsmPlan plan; const uint32_t* kv; uint32_t* cursor; uint32_t* entries; uint32_t n; };
template <class C> __global__ void __launch_bounds__(128) msm_scatter_kernel(const MsmScatterArgs a) {
    const uint32_t i = blockIdx.x * 128 + threadIdx.x;
    if (i >= a.n) return;
    const uint32_t c = a.plan.c, W = a.plan.W;
    const uint32_t* kd = a.kv + (size_t)i * 12;
    for (uint32_t s = 0; s < 3; s++)
        for (uint32_t w = 0; w < W; w++) {
            const uint32_t d = msm_digit(kd + 4 * s, w, W);
            if (d) {
                const uint32_t pos = atomicAdd(a.cursor + ((size_t)msm_row(s, w, W) << c) + d, 1u);
                a.entries[pos] = i | (s == 2 ? 0x80000000u : 0u);
            }
        }
}

struct MsmBucketArgs { const uint32_t* offsets; const uint32_t* entries; const uint32_t* pts; uint32_t* buckets; uint32_t* next; uint32_t nb; };
// Persistent threads (grid = resident capacity): every lane takes the next unprocessed bucket from a global counter and
// adds its points one per trip of ONE flat loop, so lanes whose bucket ends early fetch another bucket while the rest of
// the warp keeps adding: bucket sizes (Poisson around n / 2^c) no longer cost max-over-lanes per warp.
// PAIR = false: pts = n affine points, entry bit 31 = phi(point).  PAIR = true: pts = the proof pairing records
// (PAIR_WORDS per item), entry bit 31 = the record's second point (-Bbar at word 3 FPN) instead of its first (Abar).
template <class C, bool PAIR> __device__ __forceinline__ void msm_bucket_run(const MsmBucketArgs& a) {
    using F = typename C::Fp;
    BBS_A16 uint32_t acc[G1J];
    uint32_t b = 0, j = 0, end = 0;
    bool have = false;
    for (;;) {
        if (j == end) {
            if (have) {
                uint32_t* dst = a.buckets + (size_t)b * G1J;
                for (int k = 0; k < G1J; k++) dst[k] = acc[k];
            }
            b = atomicAdd(a.next, 1u);
            if (b >= a.nb) break;
            have = true;
            j = a.offsets[b];
            end = a.offsets[b + 1];
            g1_set_inf<C>(acc);
            continue;
        }
        const uint32_t e = a.entries[j++];
        const uint4* src = PAIR ? (const uint4*)(a.pts + (size_t)(e & 0x7fffffffu) * PAIR_WORDS + ((e >> 31) ? 3 * FPN : 0))
                                : (const uint4*)(a.pts + (size_t)(e & 0x7fffffffu) * G1A);
        BBS_A16 uint32_t p[G1A];
#pragma unroll
        for (int q = 0; q < G1A / 4; q++) { uint4 v = __ldg(src + q); p[4 * q] = v.x; p[4 * q + 1] = v.y; p[4 * q + 2] = v.z; p[4 * q + 3] = v.w; }
        if (!PAIR && (e >> 31)) {
            BBS_A16 uint32_t t[FPN];
            fe_mul<F>(t, p, C::GLV_BETA());            // phi(x, y) = (beta x, y)
            bn_copy<C::Fp::N>(p, t);
        }
        g1_add_mixed<C>(acc, acc, p);
    }
}
template <class C> __global__ void __launch_bounds__(128, 4) msm_bucket_kernel(const MsmBucketArgs a) { msm_bucket_run<C, false>(a); }
template <class C> __global__ void __launch_bounds__(128, 4) msm_bucket_pair_kernel(const MsmBucketArgs a) { msm_bucket_run<C, true>(a); }

struct MsmReduceArgs { MsmPlan plan; const uint32_t* buckets; uint32_t* row_part; };     // row_part[row][block][Jacobian]
// grid (red_blocks, rows): thread t of a row owns the digits t*chunk + 1 .. t*chunk + chunk and produces
// sum_j (t*chunk + j) bucket[t*chunk + j] = tot + (t*chunk) run  by running sums; the block adds its threads' points
template <class C> __global__ void __launch_bounds__(RLC_TPB, 4) msm_reduce_kernel(const MsmReduceArgs a) {
    __shared__ BBS_A16 uint32_t sp[RLC_TPB][3 * C::Fp::N];
    const uint32_t c = a.plan.c, chunk = a.plan.chunk, row = blockIdx.y;
    const uint32_t t = blockIdx.x * RLC_TPB + threadIdx.x, base = t * chunk, nd = 1u << msm_digit_bits(row % a.plan.W, a.plan.W);
    BBS_A16 uint32_t P[G1J];
    g1_set_inf<C>(P);
    if (base < nd) {
        BBS_A16 uint32_t run[G1J];
        g1_set_inf<C>(run);
        const uint32_t* brow = a.buckets + ((size_t)row << c) * G1J;
        for (uint32_t j = chunk; j >= 1; j--) {
            const uint32_t d = base + j;
            if (d < nd) g1_add<C>(run, run, brow + (size_t)d * G1J);
            g1_add<C>(P, P, run);
        }
        if (base) {
            BBS_A16 uint32_t m[G1J];
            g1_set_inf<C>(m);
            for (int bit = (int)c - 1; bit >= 0; bit--) {
                g1_dbl<C>(m, m);
                if ((base >> bit) & 1u) g1_add<C>(m, m, run);
            }
            g1_add<C>(P, P, m);
        }
    }
    rlc_block_sum_points<C>(sp, P);
    if (threadIdx.x == 0) g1_copy<C>(a.row_part + ((size_t)row * a.plan.red_blocks + blockIdx.x) * G1J, sp[0]);
}

struct RlcMsmFinishArgs {
    CtxView ctx;
    MsmPlan plan;
    const uint32_t* row_part; const uint32_t* sc_part;
    uint32_t n_blocks, n_msgs;     // n_blocks: blocks of rlc_prep_kernel (sc_part rows)
    uint8_t* parts_out;            // comp(S1) || comp(S2)
    uint32_t* pair; uint32_t* flags; uint8_t* status;     // pairing record of (S1, S2) for the single-shard verdict
};
// one block: rows -> S1 and S2' by Horner over the windows (two independent chains in warps 0 and 1) while warp 3 sums
// the fixed-base term F = (sum r_i) K + sum_j (sum_i r_i m_ij) H_j, one generator per lane; then S2 = S2' - F, and the two
// points are normalised in two warps: compressed for the host-combined multi-GPU path (rlc_combine) and written as the
// pairing record (x, y, 1) that the single-shard verdict feeds straight to the pairing kernel.
template <class C> __global__ void __launch_bounds__(RLC_TPB, 1) rlc_msm_finish_kernel(const RlcMsmFinishArgs a) {
    using Fr = typename C::Fr;
    using F = typename C::Fp;
    __shared__ BBS_A16 uint32_t sp[RLC_TPB][3 * C::Fp::N];
    __shared__ BBS_A16 uint32_t ss[RLC_TPB][8];
    __shared__ BBS_A16 uint32_t sums[MAX_L + 1][8];
    __shared__ BBS_A16 uint32_t res[3][3 * C::Fp::N];        // S1, S2', F
    __shared__ BBS_A16 uint32_t sf[32][3 * C::Fp::N];        // warp 3: partial sums of F
    __shared__ uint32_t skip[2];
    const CtxView& cx = a.ctx;
    const uint32_t t = threadIdx.x, W = a.plan.W, rows = a.plan.rows;
    // Fr sums over the prep blocks
    for (uint32_t j = 0; j <= a.n_msgs; j++) {
        BBS_A16 uint32_t v[8];
        bn_zero<8>(v);
        for (uint32_t b = t; b < a.n_blocks; b += RLC_TPB) fe_add<Fr>(v, v, a.sc_part + ((size_t)b * (a.n_msgs + 1) + j) * 8);
        rlc_block_sum_fr<C>(ss, v);
        if (t == 0) bn_copy<8>(sums[j], ss[0]);
        __syncthreads();
    }
    // row totals (rows <= 64): tpr threads per row add the reduce blocks' partial points, then a small tree per row
    const uint32_t tpr = rows <= 16 ? 8u : rows <= 32 ? 4u : rows <= 64 ? 2u : 1u;
    BBS_A16 uint32_t acc[G1J];
    {
        const uint32_t row = t / tpr, sub = t % tpr;
        g1_set_inf<C>(acc);
        if (row < rows)
            for (uint32_t b = sub; b < a.plan.red_blocks; b += tpr) g1_add<C>(acc, acc, a.row_part + ((size_t)row * a.plan.red_blocks + b) * G1J);
        g1_copy<C>(sp[t], acc);
        __syncthreads();
        for (uint32_t st = tpr / 2; st >= 1; st >>= 1) {
            if (row < rows && sub < st) g1_add<C>(sp[t], sp[t], sp[t + st]);
            __syncthreads();
        }
    }
    const uint32_t job = t >> 5, lane = t & 31;
    g1_set_inf<C>(acc);
    if (job < 2) {
        if (lane == 0) {
            for (int w = (int)W - 1; w >= 0; w--) {
                for (uint32_t k = msm_digit_bits(w, W); k > 0; k--) g1_dbl<C>(acc, acc);
                g1_add<C>(acc, acc, sp[(job * W + w) * tpr]);
            }
            g1_copy<C>(res[job], acc);
        }
    } else if (job == 3) {
        for (uint32_t j = lane; j <= a.n_msgs; j += 32)
            if (!(j == 0 && cx.k_inf)) tab_accumulate<C>(acc, cx, j, sums[j]);
        g1_copy<C>(sf[lane], acc);                           // warp 3 only
        __syncwarp();
        for (int st = 16; st >= 1; st >>= 1) {
            if (lane < (uint32_t)st) g1_add<C>(sf[lane], sf[lane], sf[lane + st]);
            __syncwarp();
        }
        if (lane == 0) g1_copy<C>(res[2], sf[0]);
    }
    __syncthreads();
    if (lane == 0 && job < 2) {
        BBS_A16 uint32_t S[G1J], aff[G1A];
        if (job == 0) g1_copy<C>(S, res[0]);
        else {
            BBS_A16 uint32_t nF[G1J];
            g1_neg<C>(nF, res[2]);
            g1_add<C>(S, res[1], nF);
        }
        const bool fin = g1_to_affine_vt<C>(aff, S);
        g1_compress_affine<C>(a.parts_out + job * C::G1_BYTES, aff, !fin);
        uint32_t* pr = a.pair + job * 3 * FPN;
        bn_copy<2 * C::Fp::N>(pr, aff);
        fe_set_one<F>(pr + 2 * FPN);
        skip[job] = fin ? 0u : 1u;
    }
    __syncthreads();
    if (t == 0) {
        a.flags[0] = ((skip[0] || cx.w_inf) ? FL_SKIP0 : 0u) | (skip[1] ? FL_SKIP1 : 0u);
        a.status[0] = ST_REJECT;
    }
}

// ---- proof batches (bbs_rlc_*proof_verify_batch*) --------------------------------------------------------------
// After the G1 half of proof verification, item i is accepted iff e(Abar_i, W) e(-Bbar_i, BP2) == 1, and its pairing
// record holds exactly (Abar_i, -Bbar_i).  Every item without FL_DONE is checked at once by
//     e( sum r_i Abar_i , W ) * e( sum r_i (-Bbar_i) , BP2 ) == 1
// with the coefficients r_i of rlc_coeff (index = the item's position in the call).  Both sums share the scalar r_i: it is
// value 0 of the item (rows [0, W), base Abar) and value 2 (rows [W, 2W), entry bit 31, base -Bbar) for the unchanged scan
// and scatter kernels; msm_bucket_pair_kernel reads the bases straight from the pairing records.  FL_SKIP0 / FL_SKIP1
// (identity Abar or W, identity Bbar) leave the value out, as the pairing kernels leave the factor out.
struct RlcProofPrepArgs {
    MsmPlan plan;
    const uint32_t* flags;   // the G1 half's per-item flags
    uint32_t* kv;            // n x 3 x 4 words (value 1 stays 0)
    uint32_t* counts;        // rows << c, zeroed by the caller
    uint32_t* live;          // set to 1 when some item reaches the pairing; zeroed by the caller
    uint32_t n;
    BBS_A16 uint32_t seed[8];    // the 32-byte seed as big-endian words
};
template <class C> __global__ void __launch_bounds__(RLC_TPB) rlc_proof_prep_kernel(const RlcProofPrepArgs a) {
    const uint32_t i = blockIdx.x * RLC_TPB + threadIdx.x;
    const uint32_t fl = i < a.n ? a.flags[i] : (uint32_t)FL_DONE;
    const bool live = !(fl & FL_DONE);
    if (__ballot_sync(0xffffffffu, live) && (threadIdx.x & 31) == 0) atomicOr(a.live, 1u);
    if (i >= a.n) return;
    BBS_A16 uint32_t r[8], kv[12];
    for (int k = 0; k < 12; k++) kv[k] = 0;
    if (live) {
        rlc_coeff(r, a.seed, i);
        if (!(fl & FL_SKIP0)) for (int k = 0; k < 4; k++) kv[k] = r[k];
        if (!(fl & FL_SKIP1)) for (int k = 0; k < 4; k++) kv[8 + k] = r[k];
    }
    uint32_t* kd = a.kv + (size_t)i * 12;
    for (int k = 0; k < 12; k++) kd[k] = kv[k];
    if (!live) return;
    const uint32_t c = a.plan.c, W = a.plan.W;
    for (uint32_t s = 0; s < 3; s += 2)
        for (uint32_t w = 0; w < W; w++) {
            const uint32_t d = msm_digit(kd + 4 * s, w, W);
            if (d) atomicAdd(a.counts + ((size_t)msm_row(s, w, W) << c) + d, 1u);
        }
}
// the combined check held: every item that reached the pairing is accepted
template <class C> __global__ void __launch_bounds__(RLC_TPB) rlc_proof_accept_kernel(const uint32_t* flags, uint8_t* status, uint32_t n) {
    const uint32_t i = blockIdx.x * RLC_TPB + threadIdx.x;
    if (i < n && !(flags[i] & FL_DONE)) status[i] = ST_ACCEPT;
}

}  // namespace bbs
#endif  // __CUDACC__
