// Translation unit for the `sign` kernels (see launchers.cuh).  Built once per curve: -DBBS_TU_BLS / -DBBS_TU_BN;
// with neither macro both curves are instantiated (host-simulation build).
#define BBS_NO_DEDICATED_SQR      // see field.cuh FeSqr: this unit's kernels are faster with one multiplication body
#include "launchers.cuh"

// occupancy knobs (threads per block, min resident blocks per SM -> register cap); -D overridable
#ifndef BBS_SIGN_TPB
#define BBS_SIGN_TPB 128
#endif
#ifndef BBS_SIGN_MINB
#define BBS_SIGN_MINB 4
#endif

namespace bbs {

template <class C> int launch_sign(const SignArgs& a, uint32_t n, rt_stream_t s) {
#ifdef BBS_HOSTSIM
    return rt_launch<SignArgs, &sign_item<C>, BBS_SIGN_TPB, BBS_SIGN_MINB>(a, n, s);
#else
    if (n == 0) return 0;
    if (a.item.K) return launch_sign_per_item<C>(a, n, s);        // tu_signitem.cu
    sign_kernel<C, BBS_SIGN_TPB, BBS_SIGN_MINB, false><<<(n + BBS_SIGN_TPB - 1) / BBS_SIGN_TPB, BBS_SIGN_TPB, 0, s>>>(a, n);
    RT_CHECK(cudaGetLastError());
    return 0;
#endif
}

#if defined(BBS_TU_BLS) || !defined(BBS_TU_BN)
template int launch_sign<Bls>(const SignArgs&, uint32_t, rt_stream_t);
#endif
#if defined(BBS_TU_BN) || !defined(BBS_TU_BLS)
template int launch_sign<Bn>(const SignArgs&, uint32_t, rt_stream_t);
#endif

}  // namespace bbs
