// launch_estep.cu — instantiations and launchers of the packed E-step kernels (estep.cuh).
#include "launch.h"
#include "estep.cuh"

namespace bamm {

template <typename KF> static int optin(KF kernel, size_t bytes) {
    return cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)bytes) == cudaSuccess ? 0 : -1;
}
// after the n kernels of one launcher call have been enqueued
static int launched(const EStepLaunch& l, int n) {
    *l.launches += (uint64_t)n;
    return cudaGetLastError() == cudaSuccess ? 0 : -1;
}
#define BAMM_G_CASES(X) X(1) X(2) X(3) X(4) X(5) X(6) X(7) X(8) X(9) X(10) X(11) X(12) X(13) X(14) X(15) X(16)

template <int G, bool FAST, bool MULTI>
static int dense_one(const EStepLaunch& l, const EStepArgs& a, bool optin_only) {
    const size_t smem = (size_t)a.gp.table_bytes + (size_t)plain_smem_words(a.plain_words, a.gp.Yn) * 4;
    if (optin_only) return optin(k_estep_packed<G, FAST, MULTI>, smem);
    k_estep_packed<G, FAST, MULTI><<<l.grid, l.block, smem, l.stream>>>(a.pv, a.gp, a.d_tab, a.d_s, a.plain_words, a.d_r, a.d_scal, a.al, a.only_if);
    return launched(l, 1);
}
int launch_estep_dense(const EStepLaunch& l, const EStepArgs& a, bool optin_only) {
    const bool fast = one_shift(a.gp), multi = !(a.gp.pass_first && a.gp.pass_last);
    switch (a.gp.G) {
#define X(g) case g: return fast ? (multi ? dense_one<g, true, true>(l, a, optin_only) : dense_one<g, true, false>(l, a, optin_only)) \
                                 : (multi ? dense_one<g, false, true>(l, a, optin_only) : dense_one<g, false, false>(l, a, optin_only));
        BAMM_G_CASES(X)
#undef X
        default: return -1;
    }
}

template <int G, bool FAST>
static int bound_one(const EStepLaunch& l, const EStepArgs& a, bool optin_only) {
    if (optin_only) return optin(k_ebound<G, FAST>, a.gp.table_bytes) || optin(k_ebound_watch<G, FAST>, a.gp.table_bytes);
    // with bound reuse both kernels are launched; the device flag k_estep_begin set lets exactly one of them do the pass
    k_ebound<G, FAST><<<l.grid, l.block, a.gp.table_bytes, l.stream>>>(a.pv, a.gp, a.d_tab, a.cl);
    if (a.cl.reuse) k_ebound_watch<G, FAST><<<l.grid, l.block, a.gp.table_bytes, l.stream>>>(a.pv, a.gp, a.d_tab, a.cl);
    return launched(l, a.cl.reuse ? 2 : 1);
}
int launch_estep_bound(const EStepLaunch& l, const EStepArgs& a, bool optin_only) {
    const bool fast = one_shift(a.gp);
    switch (a.gp.G) {       // bound plans have few groups (that is their point)
#define X(g) case g: return fast ? bound_one<g, true>(l, a, optin_only) : bound_one<g, false>(l, a, optin_only);
        X(1) X(2) X(3) X(4) X(5) X(6) X(7) X(8)
#undef X
        default: return -1;
    }
}

size_t estep_stage_bytes(int block) { return (size_t)(block / 32) * STAGE_WORDS * sizeof(uint32_t); }

template <int G, bool FAST, bool LEAN>
static int masked_one(const EStepLaunch& l, const EStepArgs& a, bool optin_only) {
    const size_t smem = (size_t)a.gp.table_bytes + (size_t)plain_smem_words(a.plain_words, a.gp.Yn) * 4;
    if (optin_only) return optin(k_emasked<G, FAST, LEAN>, smem);
    k_emasked<G, FAST, LEAN><<<l.grid, l.block, smem, l.stream>>>(a.pv, a.gp, a.d_tab, a.d_s, a.plain_words, a.cl, a.d_seqacc, a.d_partial, a.al);
    return launched(l, 1);
}
int launch_estep_masked(const EStepLaunch& l, const EStepArgs& a, bool optin_only) {
    const bool fast = one_shift(a.gp);
    const bool lean = a.plain_words != 0 && a.d_partial == nullptr && a.gp.pass_first && a.gp.pass_last;      // one pass, plain table in shared memory
    switch (a.gp.G) {
#define X(g) case g: return lean ? (fast ? masked_one<g, true, true>(l, a, optin_only) : masked_one<g, false, true>(l, a, optin_only)) \
                                 : (fast ? masked_one<g, true, false>(l, a, optin_only) : masked_one<g, false, false>(l, a, optin_only));
        BAMM_G_CASES(X)
#undef X
        default: return -1;
    }
}

template <int G, bool FAST, bool MULTI>
static int exact_one(const EStepLaunch& l, const EStepArgs& a, bool optin_only) {
    const size_t smem = (size_t)a.gp.table_bytes + (size_t)plain_smem_words(a.plain_words, a.gp.Yn) * 4 + (a.stage ? estep_stage_bytes(l.block) : 0);
    if (optin_only) return optin(k_eexact<G, FAST, MULTI>, smem);
    k_eexact<G, FAST, MULTI><<<l.grid, l.block, smem, l.stream>>>(a.pv, a.gp, a.d_tab, a.d_s, a.plain_words, a.stage ? 1u : 0u, a.cl, a.d_seqacc,
                                                                   a.d_partial, a.d_scal, a.al);
    return launched(l, 1);
}
int launch_estep_exact(const EStepLaunch& l, const EStepArgs& a, bool optin_only) {
    const bool fast = one_shift(a.gp), multi = !(a.gp.pass_first && a.gp.pass_last);
    switch (a.gp.G) {
#define X(g) case g: return multi ? (fast ? exact_one<g, true, true>(l, a, optin_only) : exact_one<g, false, true>(l, a, optin_only)) \
                                  : (fast ? exact_one<g, true, false>(l, a, optin_only) : exact_one<g, false, false>(l, a, optin_only));
        BAMM_G_CASES(X)
#undef X
        default: return -1;
    }
}

}  // namespace bamm
