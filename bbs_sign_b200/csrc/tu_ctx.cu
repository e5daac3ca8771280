// Translation unit for the `ctx` kernels (see launchers.cuh).  Built once per curve: -DBBS_TU_BLS / -DBBS_TU_BN;
// with neither macro both curves are instantiated (host-simulation build).
#include "launchers.cuh"

namespace bbs {

template <class C> int launch_ctx_decode(const CtxDecodeArgs& a, uint32_t n, rt_stream_t s) {
    return rt_launch<CtxDecodeArgs, &ctx_decode_item<C>, 32>(a, n, s);
}
template <class C> int launch_ctx_domain(const CtxDomainArgs& a, uint32_t n, rt_stream_t s) {
    return rt_launch<CtxDomainArgs, &ctx_domain_item<C>, 32>(a, n, s);
}
template <class C> int launch_ctx_table(const CtxTableArgs& a, uint32_t n_generators, rt_stream_t s) {
    const TabGeom G(a.tab_bits);
    const uint32_t n_bases = n_generators * (uint32_t)G.windows, n = n_bases * G.entries;
    int rc = rt_launch<CtxTableArgs, &ctx_wbase_item<C>, 32>(a, n_bases, s);
    if (rc) return rc;
#ifdef BBS_HOSTSIM
    return rt_launch<CtxTableArgs, &ctx_table_item<C>, 128>(a, n, s);
#else
    ctx_table_kernel<C, 128><<<(n + 127) / 128, 128, 0, s>>>(a, n);
    RT_CHECK(cudaGetLastError());
    return 0;
#endif
}
template <class C> int launch_ctx_lines(const CtxLinesArgs& a, uint32_t n, rt_stream_t s) {
    return rt_launch<CtxLinesArgs, &ctx_lines_item<C>, 32>(a, n, s);
}

template <class C> int launch_gen_point(const GenPointArgs& a, uint32_t n, rt_stream_t s) {
    return rt_launch<GenPointArgs, &gen_point_item<C>, 32>(a, n, s);
}
#if defined(BBS_TU_BLS) || !defined(BBS_TU_BN)
int launch_gen_seed(const GenSeedArgs& a, rt_stream_t s) { return rt_launch<GenSeedArgs, &gen_seed_item, 32>(a, 1, s); }
template int launch_gen_point<Bls>(const GenPointArgs&, uint32_t, rt_stream_t);
#endif
#if defined(BBS_TU_BN) || !defined(BBS_TU_BLS)
template int launch_gen_point<Bn>(const GenPointArgs&, uint32_t, rt_stream_t);
#endif

template <class C> int launch_ctx_lines_coop(const CtxLinesCoopArgs& a, uint32_t n, rt_stream_t s) {
    return rt_launch<CtxLinesCoopArgs, &ctx_lines_coop_item<C>, 32>(a, n, s);
}
// issuer sets (kernels.cuh): one thread per issuer, resp. per (issuer, line, pair)
template <class C> int launch_iss_decode(const IssDecodeArgs& a, uint32_t n, rt_stream_t s) {
    return rt_launch<IssDecodeArgs, &iss_decode_item<C>, 32>(a, n, s);
}
template <class C> int launch_iss_domain(const IssDomainArgs& a, uint32_t n, rt_stream_t s) {
    return rt_launch<IssDomainArgs, &iss_domain_item<C>, 32>(a, n, s);
}
template <class C> int launch_iss_lines(const IssLinesArgs& a, uint32_t n, rt_stream_t s) {
    return rt_launch<IssLinesArgs, &iss_lines_item<C>, 32>(a, n, s);
}
template <class C> int launch_iss_lines_coop(const IssLinesCoopArgs& a, uint32_t n, rt_stream_t s) {
    return rt_launch<IssLinesCoopArgs, &iss_lines_coop_item<C>, 64>(a, n, s);
}
// per-item headers (kernels.cuh item_domain_kernel): one thread per item
template <class C> int launch_item_domain(const ItemDomainArgs& a, uint32_t n, rt_stream_t s) {
#ifdef BBS_HOSTSIM
    return rt_launch<ItemDomainArgs, &item_domain_item<C>, 128>(a, n, s);
#else
    if (n == 0) return 0;
    item_domain_kernel<C, 128><<<(n + 127) / 128, 128, 0, s>>>(a, n);
    RT_CHECK(cudaGetLastError());
    return 0;
#endif
}

#if defined(BBS_TU_BLS) || !defined(BBS_TU_BN)
template int launch_item_domain<Bls>(const ItemDomainArgs&, uint32_t, rt_stream_t);
template int launch_ctx_lines_coop<Bls>(const CtxLinesCoopArgs&, uint32_t, rt_stream_t);
template int launch_iss_decode<Bls>(const IssDecodeArgs&, uint32_t, rt_stream_t);
template int launch_iss_domain<Bls>(const IssDomainArgs&, uint32_t, rt_stream_t);
template int launch_iss_lines<Bls>(const IssLinesArgs&, uint32_t, rt_stream_t);
template int launch_iss_lines_coop<Bls>(const IssLinesCoopArgs&, uint32_t, rt_stream_t);
template int launch_ctx_decode<Bls>(const CtxDecodeArgs&, uint32_t, rt_stream_t);
template int launch_ctx_domain<Bls>(const CtxDomainArgs&, uint32_t, rt_stream_t);
template int launch_ctx_table<Bls>(const CtxTableArgs&, uint32_t, rt_stream_t);
template int launch_ctx_lines<Bls>(const CtxLinesArgs&, uint32_t, rt_stream_t);
#endif
#if defined(BBS_TU_BN) || !defined(BBS_TU_BLS)
template int launch_item_domain<Bn>(const ItemDomainArgs&, uint32_t, rt_stream_t);
template int launch_ctx_lines_coop<Bn>(const CtxLinesCoopArgs&, uint32_t, rt_stream_t);
template int launch_iss_decode<Bn>(const IssDecodeArgs&, uint32_t, rt_stream_t);
template int launch_iss_domain<Bn>(const IssDomainArgs&, uint32_t, rt_stream_t);
template int launch_iss_lines<Bn>(const IssLinesArgs&, uint32_t, rt_stream_t);
template int launch_iss_lines_coop<Bn>(const IssLinesCoopArgs&, uint32_t, rt_stream_t);
template int launch_ctx_decode<Bn>(const CtxDecodeArgs&, uint32_t, rt_stream_t);
template int launch_ctx_domain<Bn>(const CtxDomainArgs&, uint32_t, rt_stream_t);
template int launch_ctx_table<Bn>(const CtxTableArgs&, uint32_t, rt_stream_t);
template int launch_ctx_lines<Bn>(const CtxLinesArgs&, uint32_t, rt_stream_t);
#endif

}  // namespace bbs
