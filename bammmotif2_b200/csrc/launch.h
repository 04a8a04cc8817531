// launch.h — host-callable launchers of the heavily templated kernels. Each family lives in its own translation unit
// (launch_estep.cu, launch_mstep.cu, launch_score.cu) so that the library builds in parallel; capi.cu only sees these functions.
#pragma once
#include "common.cuh"

namespace bamm {

struct EStepLaunch {              // geometry + stream of the packed E-step kernels (one CTA per SM)
    int grid, block;
    cudaStream_t stream;
};

// dense E-step (estep.cuh: k_estep_packed<G, FAST, MULTI>). optin_only: set the shared-memory attribute instead of launching.
int launch_estep_dense(const EStepLaunch& l, bool optin_only, bool fast, bool multi, const PackedView* pv, const GroupPlan& gp,
                       const float* d_tab, const float* d_s, uint32_t plain_words, float* d_r,
                       unsigned long long* d_scal, const ActiveList* al, const uint32_t* only_if);
// (d_partial: column passes — the partial products of the earlier passes, one float per masked window / candidate slot; else NULL)
// pruned E-step: windows over the N and truncated windows of every sequence (k_emasked<G, FAST>), bounds (k_ebound<G1, FAST>)
// and exact evaluation of the candidates (k_eexact<G, FAST>)
int launch_estep_masked(const EStepLaunch& l, bool optin_only, bool fast, const PackedView* pv, const GroupPlan& gp, const float* d_tab,
                        const float* d_s, uint32_t plain_words, const CandList* cl, ulonglong2* d_seqacc, float* d_partial,
                        const ActiveList* al);
int launch_estep_bound(const EStepLaunch& l, bool optin_only, bool fast, const PackedView* pv, const GroupPlan& gp, const float* d_tab,
                       const CandList* cl);
int launch_estep_exact(const EStepLaunch& l, bool optin_only, bool fast, const PackedView* pv, const GroupPlan& gp, const float* d_tab,
                       const float* d_s, uint32_t plain_words, bool stage, const CandList* cl, const ulonglong2* d_seqacc,
                       float* d_partial, unsigned long long* d_scal, const ActiveList* al);
// diagnostic (BAMM_DEBUG_BOUND): histogram of log2(bound / threshold) over the windows k_ebound bounds, added to d_hist
// (estep_bound_hist_bins() 64-bit counters, quarter-bit bins, bin estep_bound_hist_zero() starts at bound = threshold)
int launch_estep_bound_hist(const EStepLaunch& l, bool fast, const PackedView* pv, const GroupPlan& gp, const float* d_tab, unsigned long long* d_hist);
int estep_bound_hist_bins();
int estep_bound_hist_zero();
// bytes of the per-warp staging buffers k_eexact appends to its shared memory when `stage` is set
size_t estep_stage_bytes(int block);

// packed M-step (mstep.cuh). mode 0: opt in to `smem` bytes for both kernels of this column count, 1: list kernel, 2: scan kernel
int launch_mstep_packed(int nc, int mode, int grid, size_t smem, cudaStream_t stream, const PackedView* pv, const Plan* pl,
                        const ActiveList* al, uint32_t nregions, int nsplit, MTables mt, unsigned long long* d_part,
                        const float* d_r, const float* d_scale, const uint32_t* only_if);

// ZOOPS-only scoring with column-group pruning (score_zoops.cuh)
int launch_score_zoops(const GroupPlan& gp, bool fast, int sms, cudaStream_t st, const PackedView& pv, const float* d_tab, const float* d_s,
                       float two_eps, float* d_zoops, unsigned long long* d_z, const uint32_t* d_out, size_t plain_bytes);

}  // namespace bamm
