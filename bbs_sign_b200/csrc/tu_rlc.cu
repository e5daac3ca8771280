// Translation unit for the random-linear-combination batch mode (rlc.cuh).  Built once per curve: -DBBS_TU_BLS / -DBBS_TU_BN.
#include "launchers.cuh"

#ifndef BBS_HOSTSIM
namespace bbs {

template <class C> int launch_rlc_prep(const RlcPrepArgs& a, uint32_t n_blocks, int mode, rt_stream_t s) {
    if (n_blocks == 0) return 0;
    if (mode == RLC_PREP_STATUS_HDR) rlc_prep_kernel<C, RLC_PREP_STATUS_HDR><<<n_blocks, RLC_TPB, 0, s>>>(a);
    else if (mode == RLC_PREP_STATUS) rlc_prep_kernel<C, RLC_PREP_STATUS><<<n_blocks, RLC_TPB, 0, s>>>(a);
    else rlc_prep_kernel<C><<<n_blocks, RLC_TPB, 0, s>>>(a);
    RT_CHECK(cudaGetLastError());
    return 0;
}
#if defined(BBS_TU_BLS) || !defined(BBS_TU_BN)
int launch_msm_scan(const uint32_t* counts, uint32_t* offsets, uint32_t* cursor, uint32_t nb, rt_stream_t s) {
    msm_scan_kernel<MSM_SCAN_TPB><<<1, MSM_SCAN_TPB, 0, s>>>(counts, offsets, cursor, nb);
    RT_CHECK(cudaGetLastError());
    return 0;
}
#endif
template <class C> int launch_msm_scatter(const MsmScatterArgs& a, rt_stream_t s) {
    if (a.n == 0) return 0;
    msm_scatter_kernel<C><<<(a.n + 127) / 128, 128, 0, s>>>(a);
    RT_CHECK(cudaGetLastError());
    return 0;
}
template <class C> int launch_msm_bucket(const MsmBucketArgs& a, rt_stream_t s) {
    static int resident = 0;                       // blocks the device holds at once (4 per SM: __launch_bounds__(128, 4))
    if (!resident) {
        int dev = 0, sms = 0;
        RT_CHECK(cudaGetDevice(&dev));
        RT_CHECK(cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev));
        resident = 4 * sms;
    }
    const uint32_t want = (a.nb + 127) / 128;
    msm_bucket_kernel<C><<<want < (uint32_t)resident ? want : (uint32_t)resident, 128, 0, s>>>(a);
    RT_CHECK(cudaGetLastError());
    return 0;
}
template <class C> int launch_msm_bucket_pair(const MsmBucketArgs& a, rt_stream_t s) {
    static int resident = 0;                       // as launch_msm_bucket
    if (!resident) {
        int dev = 0, sms = 0;
        RT_CHECK(cudaGetDevice(&dev));
        RT_CHECK(cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev));
        resident = 4 * sms;
    }
    const uint32_t want = (a.nb + 127) / 128;
    msm_bucket_pair_kernel<C><<<want < (uint32_t)resident ? want : (uint32_t)resident, 128, 0, s>>>(a);
    RT_CHECK(cudaGetLastError());
    return 0;
}
template <class C> int launch_msm_reduce(const MsmReduceArgs& a, rt_stream_t s) {
    msm_reduce_kernel<C><<<dim3(a.plan.red_blocks, a.plan.rows), RLC_TPB, 0, s>>>(a);
    RT_CHECK(cudaGetLastError());
    return 0;
}
template <class C> int launch_rlc_msm_finish(const RlcMsmFinishArgs& a, bool hdr, rt_stream_t s) {
    if (hdr) rlc_msm_finish_kernel<C, true><<<1, RLC_TPB, 0, s>>>(a);
    else rlc_msm_finish_kernel<C><<<1, RLC_TPB, 0, s>>>(a);
    RT_CHECK(cudaGetLastError());
    return 0;
}
template <class C> int launch_rlc_combine(const RlcCombineArgs& a, rt_stream_t s) {
    rlc_combine_kernel<C><<<1, RLC_TPB, 0, s>>>(a);
    RT_CHECK(cudaGetLastError());
    return 0;
}
template <class C> int launch_rlc_proof_prep(const RlcProofPrepArgs& a, rt_stream_t s) {
    if (a.n == 0) return 0;
    rlc_proof_prep_kernel<C><<<(a.n + RLC_TPB - 1) / RLC_TPB, RLC_TPB, 0, s>>>(a);
    RT_CHECK(cudaGetLastError());
    return 0;
}
template <class C> int launch_rlc_proof_accept(const uint32_t* flags, uint8_t* status, uint32_t n, rt_stream_t s) {
    if (n == 0) return 0;
    rlc_proof_accept_kernel<C><<<(n + RLC_TPB - 1) / RLC_TPB, RLC_TPB, 0, s>>>(flags, status, n);
    RT_CHECK(cudaGetLastError());
    return 0;
}

#if defined(BBS_TU_BLS) || !defined(BBS_TU_BN)
template int launch_rlc_prep<Bls>(const RlcPrepArgs&, uint32_t, int, rt_stream_t);
template int launch_msm_scatter<Bls>(const MsmScatterArgs&, rt_stream_t);
template int launch_msm_bucket<Bls>(const MsmBucketArgs&, rt_stream_t);
template int launch_msm_reduce<Bls>(const MsmReduceArgs&, rt_stream_t);
template int launch_rlc_msm_finish<Bls>(const RlcMsmFinishArgs&, bool, rt_stream_t);
template int launch_rlc_combine<Bls>(const RlcCombineArgs&, rt_stream_t);
template int launch_msm_bucket_pair<Bls>(const MsmBucketArgs&, rt_stream_t);
template int launch_rlc_proof_prep<Bls>(const RlcProofPrepArgs&, rt_stream_t);
template int launch_rlc_proof_accept<Bls>(const uint32_t*, uint8_t*, uint32_t, rt_stream_t);
#endif
#if defined(BBS_TU_BN) || !defined(BBS_TU_BLS)
template int launch_rlc_prep<Bn>(const RlcPrepArgs&, uint32_t, int, rt_stream_t);
template int launch_msm_scatter<Bn>(const MsmScatterArgs&, rt_stream_t);
template int launch_msm_bucket<Bn>(const MsmBucketArgs&, rt_stream_t);
template int launch_msm_reduce<Bn>(const MsmReduceArgs&, rt_stream_t);
template int launch_rlc_msm_finish<Bn>(const RlcMsmFinishArgs&, bool, rt_stream_t);
template int launch_rlc_combine<Bn>(const RlcCombineArgs&, rt_stream_t);
template int launch_msm_bucket_pair<Bn>(const MsmBucketArgs&, rt_stream_t);
template int launch_rlc_proof_prep<Bn>(const RlcProofPrepArgs&, rt_stream_t);
template int launch_rlc_proof_accept<Bn>(const uint32_t*, uint8_t*, uint32_t, rt_stream_t);
#endif

}  // namespace bbs
#endif
