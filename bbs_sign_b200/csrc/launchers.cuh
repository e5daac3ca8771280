// One launcher per kernel and curve.  Each is explicitly instantiated in its own translation unit
// (tu_*.cu, compiled once per curve) so the library builds in parallel; capi.cu only sees declarations.
#pragma once
#include "kernels.cuh"
#include "pairing_coop.cuh"
#include "rlc.cuh"
#include "rlc_msm.cuh"
#include "selftest.cuh"
#include "launch.cuh"

namespace bbs {

template <class C> int launch_ctx_decode(const CtxDecodeArgs& a, uint32_t n, rt_stream_t s);
template <class C> int launch_ctx_domain(const CtxDomainArgs& a, uint32_t n, rt_stream_t s);
template <class C> int launch_ctx_table(const CtxTableArgs& a, uint32_t n, rt_stream_t s);
template <class C> int launch_ctx_lines(const CtxLinesArgs& a, uint32_t n, rt_stream_t s);
template <class C> int launch_ctx_lines_coop(const CtxLinesCoopArgs& a, uint32_t n, rt_stream_t s);
template <class C> int launch_iss_decode(const IssDecodeArgs& a, uint32_t n, rt_stream_t s);
template <class C> int launch_iss_domain(const IssDomainArgs& a, uint32_t n, rt_stream_t s);
template <class C> int launch_iss_lines(const IssLinesArgs& a, uint32_t n, rt_stream_t s);
template <class C> int launch_iss_lines_coop(const IssLinesCoopArgs& a, uint32_t n, rt_stream_t s);
template <class C> int launch_item_domain(const ItemDomainArgs& a, uint32_t n, rt_stream_t s);
int launch_gen_seed(const GenSeedArgs& a, rt_stream_t s);
template <class C> int launch_gen_point(const GenPointArgs& a, uint32_t n, rt_stream_t s);
template <class C> int launch_h2s(const H2sArgs& a, uint32_t n, rt_stream_t s);
template <class C> int launch_verify_g1(const VerifyG1Args& a, uint32_t n, rt_stream_t s);
template <class C> int launch_pairing(const PairingArgs& a, uint32_t n, rt_stream_t s);
#ifndef BBS_HOSTSIM
// random-linear-combination batch mode (rlc.cuh)
template <class C> int launch_rlc_prep(const RlcPrepArgs& a, uint32_t n_blocks, rt_stream_t s);
int launch_msm_scan(const uint32_t* counts, uint32_t* offsets, uint32_t* cursor, uint32_t nb, rt_stream_t s);
template <class C> int launch_msm_scatter(const MsmScatterArgs& a, rt_stream_t s);
template <class C> int launch_msm_bucket(const MsmBucketArgs& a, rt_stream_t s);
template <class C> int launch_msm_reduce(const MsmReduceArgs& a, rt_stream_t s);
template <class C> int launch_rlc_msm_finish(const RlcMsmFinishArgs& a, rt_stream_t s);
template <class C> int launch_rlc_combine(const RlcCombineArgs& a, rt_stream_t s);
// the proof form of the mode: prep, buckets over the pairing records, acceptance of the undecided items
template <class C> int launch_rlc_proof_prep(const RlcProofPrepArgs& a, rt_stream_t s);
template <class C> int launch_msm_bucket_pair(const MsmBucketArgs& a, rt_stream_t s);
template <class C> int launch_rlc_proof_accept(const uint32_t* flags, uint8_t* status, uint32_t n, rt_stream_t s);
// cooperative pairing kernel; gscratch must hold coop_gscratch_size<C>(n) bytes
template <class C> int launch_pairing_coop(const CoopArgs& a, rt_stream_t s);
template <class C> size_t coop_gscratch_size(size_t n);
#endif
template <class C> int launch_sign(const SignArgs& a, uint32_t n, rt_stream_t s);
template <class C> int launch_sign_per_item(const SignArgs& a, uint32_t n, rt_stream_t s);
template <class C> int launch_proof_g1(const ProofG1Args& a, uint32_t n, rt_stream_t s);
template <class C> int launch_proof_gen(const ProofGenArgs& a, uint32_t n, rt_stream_t s);
template <class C> int launch_proof_gen_per_item(const ProofGenArgs& a, uint32_t n, rt_stream_t s);
template <class C> int launch_field_test(const FieldTestArgs& a, uint32_t n, rt_stream_t s);
template <class C> int launch_g1_mul_test(const G1MulTestArgs& a, uint32_t n, rt_stream_t s);
template <class C> int launch_pair_test_prep(const PairTestPrepArgs& a, uint32_t n, rt_stream_t s);
template <class C> int launch_pair_test(const PairTestArgs& a, uint32_t n, rt_stream_t s);

}  // namespace bbs
