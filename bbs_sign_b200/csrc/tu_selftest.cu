// Translation unit for the `selftest` kernels (see launchers.cuh).  Built once per curve: -DBBS_TU_BLS / -DBBS_TU_BN;
// with neither macro both curves are instantiated (host-simulation build).
#include "launchers.cuh"

namespace bbs {

template <class C> int launch_field_test(const FieldTestArgs& a, uint32_t n, rt_stream_t s) {
    return rt_launch<FieldTestArgs, &field_test_item<C>, 128>(a, n, s);
}
template <class C> int launch_g1_mul_test(const G1MulTestArgs& a, uint32_t n, rt_stream_t s) {
    return rt_launch<G1MulTestArgs, &g1_mul_test_item<C>, 128>(a, n, s);
}
template <class C> int launch_g1_test(const G1TestArgs& a, uint32_t n, rt_stream_t s) {
    return rt_launch<G1TestArgs, &g1_test_item<C>, 128>(a, n, s);
}
template <class C> int launch_pair_test_prep(const PairTestPrepArgs& a, uint32_t n, rt_stream_t s) {
    return rt_launch<PairTestPrepArgs, &pair_test_prep_item<C>, 32>(a, n, s);
}
template <class C> int launch_pair_test(const PairTestArgs& a, uint32_t n, rt_stream_t s) {
    return rt_launch<PairTestArgs, &pair_test_item<C>, 128>(a, n, s);
}

#if defined(BBS_TU_BLS) || !defined(BBS_TU_BN)
template int launch_field_test<Bls>(const FieldTestArgs&, uint32_t, rt_stream_t);
template int launch_g1_mul_test<Bls>(const G1MulTestArgs&, uint32_t, rt_stream_t);
template int launch_g1_test<Bls>(const G1TestArgs&, uint32_t, rt_stream_t);
template int launch_pair_test_prep<Bls>(const PairTestPrepArgs&, uint32_t, rt_stream_t);
template int launch_pair_test<Bls>(const PairTestArgs&, uint32_t, rt_stream_t);
#endif
#if defined(BBS_TU_BN) || !defined(BBS_TU_BLS)
template int launch_field_test<Bn>(const FieldTestArgs&, uint32_t, rt_stream_t);
template int launch_g1_mul_test<Bn>(const G1MulTestArgs&, uint32_t, rt_stream_t);
template int launch_g1_test<Bn>(const G1TestArgs&, uint32_t, rt_stream_t);
template int launch_pair_test_prep<Bn>(const PairTestPrepArgs&, uint32_t, rt_stream_t);
template int launch_pair_test<Bn>(const PairTestArgs&, uint32_t, rt_stream_t);
#endif

}  // namespace bbs
