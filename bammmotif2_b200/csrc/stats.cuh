// stats.cuh — score statistics behind the scoring path (SURVEY.md §8 row f-1): the sorts of FDR::calculatePR /
// ScoreSeqSet::calcPvalues and the per-window p-value of ScoreSeqSet::calcPvalues on the device.
// The sort is CUB's radix sort (library code, like cuBLAS for a GEMM: not a kernel this repository claims);
// the p-value kernel restates ScoreSeqSet.cpp:98-124 per window.
#pragma once
#include <cub/device/device_radix_sort.cuh>
#include "kernels.cuh"

namespace bamm {

// parameters of the exponential tail of ScoreSeqSet::calcPvalues (ScoreSeqSet.cpp:88-96), made on the host from the sorted
// negatives (mops_tail in capi_score.inl)
struct MopsTail { float S_ntop, lambda, nTop; };

// first index in [lo, hi) with neg[idx] > x (the std::upper_bound of ScoreSeqSet.cpp:98-124), hi when there is none
__device__ __forceinline__ unsigned long long upper_bound_f32(const float* __restrict__ neg, unsigned long long lo,
                                                              unsigned long long hi, float x) {
    while (lo < hi) {
        const unsigned long long mid = (lo + hi) >> 1;
        if (neg[mid] > x) hi = mid; else lo = mid + 1;
    }
    return lo;
}

// reference: src/seq_scoring/ScoreSeqSet.cpp:98-124. neg: ALL negative window scores sorted ascending, ub = upper_bound of Sl.
//   FPl = number of negatives strictly above Sl (upper_bound, :103-104)
//   FPl == negN                      -> p = 1
//   FPl < 10 and |lambda| > eps      -> p = nTop / negN * expf( -(Sl - S_ntop) / lambda )
//   else                             -> p = ( FPl + (S_higher - Sl + eps) / (S_higher - S_lower + eps) ) / negN
// e-value = p * number of positive sequences (:122).
__device__ __forceinline__ float mops_pvalue(const float* __restrict__ neg, unsigned long long negN, unsigned long long ub, float Sl,
                                             const MopsTail& t) {
    const float eps = 1.0e-5;
    const unsigned long long FPl = negN - ub;
    float p;
    if (FPl == negN) p = 1.0f;
    else if (FPl < 10 && fabsf(t.lambda) > eps) p = t.nTop / (float)negN * expf(-(Sl - t.S_ntop) / t.lambda);
    else {
        // FPl == 0 (no negative above Sl) only gets here without a usable tail fit: the reference then reads one element
        // past its vector (ScoreSeqSet.cpp:112); Sl itself stands in for it, which gives p = 1 / negN
        const float SlHigher = neg[negN - FPl - 1], SlLower = FPl ? neg[negN - FPl] : Sl;
        p = ((float)FPl + (SlHigher - Sl + eps) / (SlHigher - SlLower + eps)) / (float)negN;
    }
    return p;
}

__global__ void __launch_bounds__(256)
k_mops_pvalues(const float* __restrict__ neg, unsigned long long negN, const float* __restrict__ pos, unsigned long long npos,
               MopsTail tail, float posN, float* __restrict__ pval, float* __restrict__ eval) {
    for (unsigned long long i = (unsigned long long)blockIdx.x * blockDim.x + threadIdx.x; i < npos; i += (unsigned long long)gridDim.x * blockDim.x) {
        const float Sl = pos[i];
        const float p = mops_pvalue(neg, negN, upper_bound_f32(neg, 0, negN, Sl), Sl, tail);
        pval[i] = p;
        eval[i] = p * posN;
    }
}

}  // namespace bamm
