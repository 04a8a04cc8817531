// launch_estep.cu — instantiations and launchers of the packed E-step kernels (estep.cuh).
#include "launch.h"
#include "estep.cuh"

namespace bamm {

template <typename KF> static int optin(KF kernel, size_t bytes) {
    return cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)bytes) == cudaSuccess ? 0 : -1;
}
#define BAMM_G_CASES(X) X(1) X(2) X(3) X(4) X(5) X(6) X(7) X(8) X(9) X(10) X(11) X(12) X(13) X(14) X(15) X(16)

template <int G, bool FAST, bool MULTI>
static int dense_one(const EStepLaunch& l, bool optin_only, const PackedView* pv, const GroupPlan& gp, const float* d_tab, const float* d_s,
                     uint32_t plain_words, float* d_r, unsigned long long* d_scal, const ActiveList* al, const uint32_t* only_if) {
    const size_t smem = (size_t)gp.table_bytes + (size_t)plain_smem_words(plain_words, gp.Yn) * 4;
    if (optin_only) return optin(k_estep_packed<G, FAST, MULTI>, smem);
    k_estep_packed<G, FAST, MULTI><<<l.grid, l.block, smem, l.stream>>>(*pv, gp, d_tab, d_s, plain_words, d_r, d_scal, *al, only_if);
    return cudaGetLastError() == cudaSuccess ? 0 : -1;
}
int launch_estep_dense(const EStepLaunch& l, bool optin_only, bool fast, bool multi, const PackedView* pv, const GroupPlan& gp,
                       const float* d_tab, const float* d_s, uint32_t plain_words, float* d_r,
                       unsigned long long* d_scal, const ActiveList* al, const uint32_t* only_if) {
#define ARGS l, optin_only, pv, gp, d_tab, d_s, plain_words, d_r, d_scal, al, only_if
    switch (gp.G) {
#define X(g) case g: return fast ? (multi ? dense_one<g, true, true>(ARGS) : dense_one<g, true, false>(ARGS)) \
                                 : (multi ? dense_one<g, false, true>(ARGS) : dense_one<g, false, false>(ARGS));
        BAMM_G_CASES(X)
#undef X
        default: return -1;
    }
#undef ARGS
}

template <int G, bool FAST>
static int bound_one(const EStepLaunch& l, bool optin_only, const PackedView* pv, const GroupPlan& gp, const float* d_tab, const CandList* cl) {
    if (optin_only) return optin(k_ebound<G, FAST>, gp.table_bytes) || optin(k_ebound_watch<G, FAST>, gp.table_bytes);
    // with bound reuse both kernels are launched; the device flag k_estep_begin set lets exactly one of them do the pass
    k_ebound<G, FAST><<<l.grid, l.block, gp.table_bytes, l.stream>>>(*pv, gp, d_tab, *cl);
    if (cl->reuse) k_ebound_watch<G, FAST><<<l.grid, l.block, gp.table_bytes, l.stream>>>(*pv, gp, d_tab, *cl);
    return cudaGetLastError() == cudaSuccess ? 0 : -1;
}
int launch_estep_bound(const EStepLaunch& l, bool optin_only, bool fast, const PackedView* pv, const GroupPlan& gp, const float* d_tab,
                       const CandList* cl) {
    switch (gp.G) {       // bound plans have few groups (that is their point)
#define X(g) case g: return fast ? bound_one<g, true>(l, optin_only, pv, gp, d_tab, cl) : bound_one<g, false>(l, optin_only, pv, gp, d_tab, cl);
        X(1) X(2) X(3) X(4) X(5) X(6) X(7) X(8)
#undef X
        default: return -1;
    }
}

template <int G, bool FAST>
static int bound_hist_one(const EStepLaunch& l, const PackedView* pv, const GroupPlan& gp, const float* d_tab, unsigned long long* d_hist) {
    if (optin(k_ebound_hist<G, FAST>, gp.table_bytes)) return -1;
    k_ebound_hist<G, FAST><<<l.grid, l.block, gp.table_bytes, l.stream>>>(*pv, gp, d_tab, d_hist);
    return cudaGetLastError() == cudaSuccess ? 0 : -1;
}
int launch_estep_bound_hist(const EStepLaunch& l, bool fast, const PackedView* pv, const GroupPlan& gp, const float* d_tab, unsigned long long* d_hist) {
    switch (gp.G) {
#define X(g) case g: return fast ? bound_hist_one<g, true>(l, pv, gp, d_tab, d_hist) : bound_hist_one<g, false>(l, pv, gp, d_tab, d_hist);
        X(1) X(2) X(3) X(4) X(5) X(6) X(7) X(8)
#undef X
        default: return -1;
    }
}
int estep_bound_hist_bins() { return BOUND_HIST_BINS; }
int estep_bound_hist_zero() { return BOUND_HIST_ZERO; }

size_t estep_stage_bytes(int block) { return (size_t)(block / 32) * STAGE_WORDS * sizeof(uint32_t); }

template <int G, bool FAST, bool LEAN>
static int masked_one(const EStepLaunch& l, bool optin_only, const PackedView* pv, const GroupPlan& gp, const float* d_tab, const float* d_s,
                      uint32_t plain_words, const CandList* cl, ulonglong2* d_seqacc, float* d_partial, const ActiveList* al) {
    const size_t smem = (size_t)gp.table_bytes + (size_t)plain_smem_words(plain_words, gp.Yn) * 4;
    if (optin_only) return optin(k_emasked<G, FAST, LEAN>, smem);
    k_emasked<G, FAST, LEAN><<<l.grid, l.block, smem, l.stream>>>(*pv, gp, d_tab, d_s, plain_words, *cl, d_seqacc, d_partial, *al);
    return cudaGetLastError() == cudaSuccess ? 0 : -1;
}
int launch_estep_masked(const EStepLaunch& l, bool optin_only, bool fast, const PackedView* pv, const GroupPlan& gp, const float* d_tab,
                        const float* d_s, uint32_t plain_words, const CandList* cl, ulonglong2* d_seqacc, float* d_partial,
                        const ActiveList* al) {
#define ARGS l, optin_only, pv, gp, d_tab, d_s, plain_words, cl, d_seqacc, d_partial, al
    const bool lean = plain_words != 0 && d_partial == nullptr && gp.pass_first && gp.pass_last;      // one pass, plain table in shared memory
    switch (gp.G) {
#define X(g) case g: return lean ? (fast ? masked_one<g, true, true>(ARGS) : masked_one<g, false, true>(ARGS)) \
                                 : (fast ? masked_one<g, true, false>(ARGS) : masked_one<g, false, false>(ARGS));
        BAMM_G_CASES(X)
#undef X
        default: return -1;
    }
#undef ARGS
}

template <int G, bool FAST, bool MULTI>
static int exact_one(const EStepLaunch& l, bool optin_only, const PackedView* pv, const GroupPlan& gp, const float* d_tab, const float* d_s,
                     uint32_t plain_words, bool stage, const CandList* cl, const ulonglong2* d_seqacc, float* d_partial, unsigned long long* d_scal, const ActiveList* al) {
    const size_t smem = (size_t)gp.table_bytes + (size_t)plain_smem_words(plain_words, gp.Yn) * 4 + (stage ? estep_stage_bytes(l.block) : 0);
    if (optin_only) return optin(k_eexact<G, FAST, MULTI>, smem);
    k_eexact<G, FAST, MULTI><<<l.grid, l.block, smem, l.stream>>>(*pv, gp, d_tab, d_s, plain_words, stage ? 1u : 0u, *cl, d_seqacc, d_partial, d_scal, *al);
    return cudaGetLastError() == cudaSuccess ? 0 : -1;
}
int launch_estep_exact(const EStepLaunch& l, bool optin_only, bool fast, const PackedView* pv, const GroupPlan& gp, const float* d_tab,
                       const float* d_s, uint32_t plain_words, bool stage, const CandList* cl, const ulonglong2* d_seqacc,
                       float* d_partial, unsigned long long* d_scal, const ActiveList* al) {
#define ARGS l, optin_only, pv, gp, d_tab, d_s, plain_words, stage, cl, d_seqacc, d_partial, d_scal, al
    const bool multi = !(gp.pass_first && gp.pass_last);
    switch (gp.G) {
#define X(g) case g: return multi ? (fast ? exact_one<g, true, true>(ARGS) : exact_one<g, false, true>(ARGS)) \
                                  : (fast ? exact_one<g, true, false>(ARGS) : exact_one<g, false, false>(ARGS));
        BAMM_G_CASES(X)
#undef X
        default: return -1;
    }
#undef ARGS
}

}  // namespace bamm
