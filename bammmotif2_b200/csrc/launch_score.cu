// launch_score.cu — instantiations and launcher of the ZOOPS scoring kernel (score_zoops.cuh).
#include "launch.h"
#include "score_zoops.cuh"

namespace bamm {

template <int G, bool FAST>
static int score_zoops_one(const GroupPlan& gp, int sms, cudaStream_t st, const PackedView& pv, const float* d_tab, const float* d_s, float two_eps,
                           float* d_zoops, unsigned long long* d_z, const uint32_t* d_out, size_t plain_bytes) {
    const size_t smem = (size_t)gp.table_bytes + plain_bytes;
    if (cudaFuncSetAttribute(k_score_zoops_packed<G, FAST>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem) != cudaSuccess) return -1;
    k_score_zoops_packed<G, FAST><<<sms, 1024, smem, st>>>(pv, gp, d_tab, d_s, two_eps, d_zoops, d_z, d_out);
    return cudaGetLastError() == cudaSuccess ? 0 : -1;
}
int launch_score_zoops(const GroupPlan& gp, int sms, cudaStream_t st, const PackedView& pv, const float* d_tab, const float* d_s,
                       float two_eps, float* d_zoops, unsigned long long* d_z, const uint32_t* d_out, size_t plain_bytes) {
    const bool fast = one_shift(gp);
    switch (gp.G) {
#define X(g) case g: return fast ? score_zoops_one<g, true>(gp, sms, st, pv, d_tab, d_s, two_eps, d_zoops, d_z, d_out, plain_bytes) \
                                 : score_zoops_one<g, false>(gp, sms, st, pv, d_tab, d_s, two_eps, d_zoops, d_z, d_out, plain_bytes);
        X(1) X(2) X(3) X(4) X(5) X(6) X(7) X(8) X(9) X(10) X(11) X(12) X(13) X(14) X(15) X(16)
#undef X
        default: return -1;
    }
}

}  // namespace bamm
