// Translation unit for signing with per-item headers (see launchers.cuh).  Built once per curve: -DBBS_TU_BLS / -DBBS_TU_BN;
// with neither macro both curves are instantiated (host-simulation build).  It has its own unit for the reason tu_proofitem.cu
// gives: next to this instance, ptxas allocates the shared kernel of the calls without per-item headers differently.
#define BBS_NO_DEDICATED_SQR      // as tu_sign.cu
#include "launchers.cuh"

#ifndef BBS_SIGN_TPB
#define BBS_SIGN_TPB 128
#endif
#ifndef BBS_SIGN_MINB
#define BBS_SIGN_MINB 4
#endif

namespace bbs {

template <class C> int launch_sign_per_item(const SignArgs& a, uint32_t n, rt_stream_t s) {
#ifdef BBS_HOSTSIM
    return rt_launch<SignArgs, &sign_item<C>, BBS_SIGN_TPB, BBS_SIGN_MINB>(a, n, s);
#else
    if (n == 0) return 0;
    sign_kernel<C, BBS_SIGN_TPB, BBS_SIGN_MINB, true><<<(n + BBS_SIGN_TPB - 1) / BBS_SIGN_TPB, BBS_SIGN_TPB, 0, s>>>(a, n);
    RT_CHECK(cudaGetLastError());
    return 0;
#endif
}

#if defined(BBS_TU_BLS) || !defined(BBS_TU_BN)
template int launch_sign_per_item<Bls>(const SignArgs&, uint32_t, rt_stream_t);
#endif
#if defined(BBS_TU_BN) || !defined(BBS_TU_BLS)
template int launch_sign_per_item<Bn>(const SignArgs&, uint32_t, rt_stream_t);
#endif

}  // namespace bbs
