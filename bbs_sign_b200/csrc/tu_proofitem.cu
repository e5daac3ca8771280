// Translation unit for proof generation with per-item headers / phs (see launchers.cuh).  Built once per curve: -DBBS_TU_BLS /
// -DBBS_TU_BN; with neither macro both curves are instantiated (host-simulation build).  It has its own unit because
// ptxas allocates the non-inlined field helpers (fe_inv) once per unit for all their callers: next to this instance they
// would cost the proof generation of the calls without per-item headers spill slots.
#include "launchers.cuh"

#ifndef BBS_PROOF_G1_TPB
#define BBS_PROOF_G1_TPB 128
#endif
#ifndef BBS_PROOF_G1_MINB
#define BBS_PROOF_G1_MINB 4
#endif

namespace bbs {

template <class C> int launch_proof_gen_per_item(const ProofGenArgs& a, uint32_t n, rt_stream_t s) {
    return rt_launch<ProofGenArgs, &proof_gen_item<C, true>, BBS_PROOF_G1_TPB, BBS_PROOF_G1_MINB>(a, n, s);
}

#if defined(BBS_TU_BLS) || !defined(BBS_TU_BN)
template int launch_proof_gen_per_item<Bls>(const ProofGenArgs&, uint32_t, rt_stream_t);
#endif
#if defined(BBS_TU_BN) || !defined(BBS_TU_BLS)
template int launch_proof_gen_per_item<Bn>(const ProofGenArgs&, uint32_t, rt_stream_t);
#endif

}  // namespace bbs
