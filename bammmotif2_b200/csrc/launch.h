// launch.h — host-callable launchers of the heavily templated kernels. Each family lives in its own translation unit
// (launch_estep.cu, launch_mstep.cu, launch_score.cu) so that the library builds in parallel; capi.cu only sees these functions.
#pragma once
#include "common.cuh"

namespace bamm {

struct EStepLaunch {              // geometry + stream of the packed E-step kernels (one CTA per SM)
    int grid, block;
    cudaStream_t stream;
    uint64_t* launches;           // every kernel a launcher enqueues is counted here
};

// One pass of the packed E-step: its plan and the buffers its kernels read and write. Each launcher passes on the fields its
// kernel takes; the kernel variant (one-shift extraction, column passes, plain table in shared memory) follows from the plan.
struct EStepArgs {
    GroupPlan gp;                 // plan of the pass (bound plan for the bounds) with q and thr0 filled in
    PackedView pv;
    const float* d_tab;           // tables of the plan
    const float* d_s;             // plain [j][y] table (single columns of masked windows)
    uint32_t plain_words;         // > 0: the plain table rides in shared memory behind the group tables
    bool stage;                   // k_eexact stages the sequence words of every warp in shared memory
    CandList cl;                  // candidates of the pruned E-step
    ActiveList al;
    ulonglong2* d_seqacc;         // per list sequence: normaliser terms of its masked windows (k_emasked -> k_eexact)
    float* d_partial;             // column passes: the partial products of the earlier passes, one float per masked window
                                  // (k_emasked) / candidate slot (k_eexact); NULL for a single pass
    float* d_r;
    unsigned long long* d_scal;   // llh and sum of r, or NULL
    const uint32_t* only_if;      // dense kernel: does work only when this device flag is set (NULL: always)
};

// optin_only: set the shared-memory attribute of the kernels instead of launching them.
// dense E-step (estep.cuh: k_estep_packed<G, FAST, MULTI>)
int launch_estep_dense(const EStepLaunch& l, const EStepArgs& a, bool optin_only);
// pruned E-step: windows over the N and truncated windows of every sequence (k_emasked<G, FAST, LEAN>), bounds (k_ebound<G1, FAST>,
// and k_ebound_watch when the candidate list has bound reuse) and exact evaluation of the candidates (k_eexact<G, FAST, MULTI>)
int launch_estep_masked(const EStepLaunch& l, const EStepArgs& a, bool optin_only);
int launch_estep_bound(const EStepLaunch& l, const EStepArgs& a, bool optin_only);
int launch_estep_exact(const EStepLaunch& l, const EStepArgs& a, bool optin_only);
// bytes of the per-warp staging buffers k_eexact appends to its shared memory when `stage` is set
size_t estep_stage_bytes(int block);

// packed M-step (mstep.cuh). mode 0: opt in to `smem` bytes for both kernels of this column count, 1: list kernel, 2: scan kernel
int launch_mstep_packed(int nc, int mode, int grid, size_t smem, cudaStream_t stream, const PackedView* pv, const Plan* pl,
                        const ActiveList* al, uint32_t nregions, int nsplit, MTables mt, unsigned long long* d_part,
                        const float* d_r, const float* d_scale, const uint32_t* only_if);

// ZOOPS-only scoring with column-group pruning (score_zoops.cuh)
int launch_score_zoops(const GroupPlan& gp, int sms, cudaStream_t st, const PackedView& pv, const float* d_tab, const float* d_s,
                       float two_eps, float* d_zoops, unsigned long long* d_z, const uint32_t* d_out, size_t plain_bytes);

}  // namespace bamm
