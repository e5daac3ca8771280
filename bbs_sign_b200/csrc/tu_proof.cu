// Translation unit for the `proof` kernels (see launchers.cuh).  Built once per curve: -DBBS_TU_BLS / -DBBS_TU_BN;
// with neither macro both curves are instantiated (host-simulation build).
#include "launchers.cuh"

// occupancy knobs (threads per block, min resident blocks per SM -> register cap); -D overridable
#ifndef BBS_PROOF_G1_TPB
#define BBS_PROOF_G1_TPB 128
#endif
#ifndef BBS_PROOF_G1_MINB
#define BBS_PROOF_G1_MINB 4
#endif

namespace bbs {

template <class C> int launch_proof_g1(const ProofG1Args& a, uint32_t n, rt_stream_t s) {
#ifndef BBS_HOSTSIM
    if (a.part_t1 && n) {
        // three tasks per proof (kernels.cuh proof_task_v1 / _f / _v2) and the join; the state bytes of F live behind those of V1
        constexpr int TPB = BBS_PROOF_G1_TPB, MINB = BBS_PROOF_G1_MINB;
        const uint32_t nb = (n + TPB - 1) / TPB;
        uint8_t* fbad = a.part_st + n;
        if (a.item.K || a.ph_off) {
            proof_g1_split_kernel<C, TPB, MINB, true><<<3 * nb, TPB, 0, s>>>(a, n, nb, fbad);
            RT_CHECK(cudaGetLastError());
            proof_g1_join_kernel<C, 128, true><<<(n + 127) / 128, 128, 0, s>>>(a, n, fbad);
        } else {
            proof_g1_split_kernel<C, TPB, MINB, false><<<3 * nb, TPB, 0, s>>>(a, n, nb, fbad);
            RT_CHECK(cudaGetLastError());
            proof_g1_join_kernel<C, 128, false><<<(n + 127) / 128, 128, 0, s>>>(a, n, fbad);
        }
        RT_CHECK(cudaGetLastError());
        return 0;
    }
#else
    if (a.part_t1) {                                    // the task functions of the split path, run in sequence
        uint8_t* fbad = a.part_st + n;
        for (uint32_t i = 0; i < n; i++) { proof_task_v1<C, true>(a, i); proof_task_f<C, true>(a, i, fbad + i); proof_task_v2<C, true>(a, i); }
        for (uint32_t i = 0; i < n; i++) proof_join_item<C, true>(a, i, fbad);
        return 0;
    }
#endif
    return rt_launch<ProofG1Args, &proof_g1_item<C>, BBS_PROOF_G1_TPB, BBS_PROOF_G1_MINB>(a, n, s);
}

template <class C> int launch_proof_gen(const ProofGenArgs& a, uint32_t n, rt_stream_t s) {
    if (a.item.K || a.ph_off) return launch_proof_gen_per_item<C>(a, n, s);     // tu_proofitem.cu
    return rt_launch<ProofGenArgs, &proof_gen_item<C, false>, BBS_PROOF_G1_TPB, BBS_PROOF_G1_MINB>(a, n, s);
}

#if defined(BBS_TU_BLS) || !defined(BBS_TU_BN)
template int launch_proof_gen<Bls>(const ProofGenArgs&, uint32_t, rt_stream_t);
template int launch_proof_g1<Bls>(const ProofG1Args&, uint32_t, rt_stream_t);
#endif
#if defined(BBS_TU_BN) || !defined(BBS_TU_BLS)
template int launch_proof_gen<Bn>(const ProofGenArgs&, uint32_t, rt_stream_t);
template int launch_proof_g1<Bn>(const ProofG1Args&, uint32_t, rt_stream_t);
#endif

}  // namespace bbs
