// mask.cuh — EM::mask, the "advanced EM" of --advanceEM (SURVEY.md §8 row f-4).
// reference: src/refinement/EM.cpp:261-503 (without optimizeQ, whose placement inside the per-sequence loop makes the
// reference's own result depend on stale responsibilities). Three phases:
//   (1) one E-step with the ORDER-0 model over all windows: full W-column products; the window at p = 0 keeps the bare
//       prior (loop bound j < min(W, ij), :300-303); the normaliser is summed in ascending i like the reference does,
//       because phase (2) compares these values with a threshold and must select exactly the same windows;
//   (2) the threshold that keeps the fraction f of all windows with the largest responsibility (:318-345);
//   (3) EM over the kept windows only: full products and full counts (no truncated windows here), prior read at
//       pos_[LW1 - i] (so the window i = 0, when kept, gets prior 0: :417), r[0] divided by the normaliser once more (:422).
// The kernels read the order-K k-mer index array Y (any alphabet); the kept windows form a CSR list per sequence.
#pragma once
#include "kernels.cuh"

namespace bamm {

struct MaskView {
    const uint64_t* seq_off;   // seqset offsets
    const uint32_t* seq_ids;   // subset -> seqset index
    const uint64_t* r_off;     // subset prefix sums of L (nsub+1)
    uint32_t nsub;
};

// phase (1). s0: [A][W] = v[0][y][j] / vbg[0][y]. One warp per sequence.
template <typename YT>
__global__ void __launch_bounds__(256)
k_mask_phase1(const YT* __restrict__ Y, MaskView mv, int W, uint32_t A, const float* __restrict__ s0_g, float q, float* __restrict__ r) {
    __shared__ float s0[6 * BAMM_MAX_MOTIF_WIDTH];
    for (uint32_t i = threadIdx.x; i < A * (uint32_t)W; i += blockDim.x) s0[i] = s0_g[i];
    __syncthreads();
    const int lane = threadIdx.x & 31;
    const uint32_t warp = blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
    const uint32_t nwarps = gridDim.x * (blockDim.x >> 5);
    for (uint32_t li = warp; li < mv.nsub; li += nwarps) {
        const uint32_t n = mv.seq_ids[li];
        const uint64_t base = mv.seq_off[n], L = mv.seq_off[n + 1] - base, LW1 = L - W + 1;
        const YT* __restrict__ yn = Y + base;
        float* __restrict__ rn = r + mv.r_off[li];
        const float pos_i = q / (float)LW1;
        for (uint64_t i = lane; i < LW1; i += 32) {
            const uint64_t p = L - W - i;
            float prod = 1.0f;
            if (p != 0) for (int j = 0; j < W; j++) prod *= s0[((uint32_t)yn[p + j] % A) * W + j];
            rn[i] = prod * pos_i;
        }
        __syncwarp();
        float norm = 1.0f - q;
        if (lane == 0) for (uint64_t i = 0; i < LW1; i++) norm += rn[i];       // ascending i, one thread: the reference's order
        norm = __shfl_sync(FULL, norm, 0);
        for (uint64_t i = lane; i < LW1; i += 32) rn[i] /= norm;
        __syncwarp();
    }
}

// all responsibilities of the windows (i < LW1 of every sequence), densely: input of the descending sort of phase (2)
__global__ void k_mask_gather(MaskView mv, int W, const uint64_t* __restrict__ woff /* [nsub+1] prefix sums of LW1 */,
                              const float* __restrict__ r, float* __restrict__ out) {
    const int lane = threadIdx.x & 31;
    const uint32_t warp = blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
    const uint32_t nwarps = gridDim.x * (blockDim.x >> 5);
    for (uint32_t li = warp; li < mv.nsub; li += nwarps) {
        const uint64_t LW1 = woff[li + 1] - woff[li];
        const float* __restrict__ rn = r + mv.r_off[li];
        for (uint64_t i = lane; i < LW1; i += 32) out[woff[li] + i] = rn[i];
    }
}

// kept windows per sequence: count (FILL = false) or the ascending list of their r indices (FILL = true)
template <bool FILL>
__global__ void k_mask_select(MaskView mv, const uint64_t* __restrict__ woff, const float* __restrict__ r, float cutoff,
                              uint32_t* __restrict__ cnt, const uint64_t* __restrict__ sel_off, uint32_t* __restrict__ sel_i) {
    const int lane = threadIdx.x & 31;
    const uint32_t warp = blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
    const uint32_t nwarps = gridDim.x * (blockDim.x >> 5);
    for (uint32_t li = warp; li < mv.nsub; li += nwarps) {
        const uint64_t LW1 = woff[li + 1] - woff[li];
        const float* __restrict__ rn = r + mv.r_off[li];
        uint32_t c = 0;
        for (uint64_t i0 = 0; i0 < LW1; i0 += 32) {
            const uint64_t i = i0 + lane;
            const bool keep = i < LW1 && rn[i] >= cutoff;
            const uint32_t m = __ballot_sync(FULL, keep);
            if (FILL && keep) sel_i[sel_off[li] + c + __popc(m & ((1u << lane) - 1u))] = (uint32_t)i;
            c += __popc(m);
        }
        if (!FILL && lane == 0) cnt[li] = c;
    }
}

// phase (3) E-step over the kept windows. s: [j][y] table of the current model (global; L2-resident). One warp per sequence.
template <typename YT>
__global__ void __launch_bounds__(256)
k_mask_estep(const YT* __restrict__ Y, MaskView mv, int W, uint32_t Yn, const float* __restrict__ s, float q,
             const uint64_t* __restrict__ sel_off, const uint32_t* __restrict__ sel_i, float* __restrict__ r,
             unsigned long long* __restrict__ scal) {
    const int lane = threadIdx.x & 31;
    const uint32_t warp = blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
    const uint32_t nwarps = gridDim.x * (blockDim.x >> 5);
    long long llh_fx = 0;
    for (uint32_t li = warp; li < mv.nsub; li += nwarps) {
        const uint32_t n = mv.seq_ids[li];
        const uint64_t base = mv.seq_off[n], L = mv.seq_off[n + 1] - base, LW1 = L - W + 1;
        const YT* __restrict__ yn = Y + base;
        float* __restrict__ rn = r + mv.r_off[li];
        const float pos_i = q / (float)LW1;
        const uint64_t x0 = sel_off[li], x1 = sel_off[li + 1];
        for (uint64_t x = x0 + lane; x < x1; x += 32) {
            const uint32_t i = sel_i[x];
            const uint64_t p = L - W - i;
            float prod = 1.0f;
            for (int j = 0; j < W; j++) prod *= __ldg(&s[(uint32_t)j * Yn + (uint32_t)yn[p + j]]);
            rn[i] = prod * (i == 0 ? 0.0f : pos_i);                            // pos_[LW1 - i]: never set for i = 0
        }
        __syncwarp();
        float norm = 1.0f - q;
        if (lane == 0) {
            for (uint64_t x = x0; x < x1; x++) norm += rn[sel_i[x]];           // kept windows in ascending i, one thread
            rn[0] /= norm;                                                      // EM.cpp:422
            llh_fx += __double2ll_rn((double)logf(norm) * SC_SCALE_D);
        }
        norm = __shfl_sync(FULL, norm, 0);
        __syncwarp();
        for (uint64_t x = x0 + lane; x < x1; x += 32) rn[sel_i[x]] /= norm;
        __syncwarp();
    }
    if (lane == 0 && llh_fx) atomicAdd(&scal[0], (unsigned long long)llh_fx);
}

// phase (3) M-step: n[K][y(p+j)][j] += r for every kept window and ALL W columns (EM.cpp:453-461), 2^-40 fixed point into the
// CTA's slice of the partial tables (SMEM: low words in shared memory, as in k_mstep)
template <typename YT, bool SMEM>
__global__ void __launch_bounds__(512)
k_mask_mstep(const YT* __restrict__ Y, MaskView mv, int W, uint32_t Yn, const uint64_t* __restrict__ sel_off,
             const uint32_t* __restrict__ sel_i, const float* __restrict__ r, unsigned long long* __restrict__ part) {
    extern __shared__ uint32_t lo_sh[];
    const uint32_t nbin = (uint32_t)W * Yn;
    unsigned long long* mypart = SMEM ? part + (uint64_t)blockIdx.x * nbin : part;
    if (SMEM) {
        for (uint32_t i = threadIdx.x; i < nbin; i += blockDim.x) lo_sh[i] = 0u;
        __syncthreads();
    }
    const int lane = threadIdx.x & 31;
    const uint32_t warp = blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
    const uint32_t nwarps = gridDim.x * (blockDim.x >> 5);
    for (uint32_t li = warp; li < mv.nsub; li += nwarps) {
        const uint32_t n = mv.seq_ids[li];
        const uint64_t base = mv.seq_off[n], L = mv.seq_off[n + 1] - base;
        const YT* __restrict__ yn = Y + base;
        const float* __restrict__ rn = r + mv.r_off[li];
        for (uint64_t x = sel_off[li] + lane; x < sel_off[li + 1]; x += 32) {
            const uint32_t i = sel_i[x];
            const float rv = rn[i];
            if (!(rv > 0.0f)) continue;
            const unsigned long long X = __float2ull_rn(rv * FX_SCALE_F);
            if (X == 0) continue;
            const uint64_t p = L - W - i;
            const uint32_t xlo = (uint32_t)X, xhi = (uint32_t)(X >> 32);
            for (int j = 0; j < W; j++) {
                const uint32_t bin = (uint32_t)j * Yn + (uint32_t)yn[p + j];
                if (SMEM) {
                    const uint32_t old = atomicAdd(&lo_sh[bin], xlo);
                    const uint32_t h = xhi + ((uint32_t)(old + xlo) < old ? 1u : 0u);
                    if (h) atomicAdd(&mypart[bin], (unsigned long long)h << 32);
                } else {
                    atomicAdd(&mypart[bin], X);
                }
            }
        }
    }
    if (SMEM) {
        __syncthreads();
        for (uint32_t i = threadIdx.x; i < nbin; i += blockDim.x) {
            const uint32_t v = lo_sh[i];
            if (v) atomicAdd(&mypart[i], (unsigned long long)v);
        }
    }
}

}  // namespace bamm

namespace bamm {

// ---- Motif::initFromPWM, the sampling step (src/init/Motif.cpp:236-299; SURVEY.md §8 row f-4) -------------------------------
// Per sequence: posterior of the motif start over the LW1 windows plus "no motif" from the order-0 odds `score` (float, the
// reference's operation order: products in ascending j, normaliser summed for i = 1..LW1 and then the no-motif term), one
// site z drawn from it the way libstdc++'s std::discrete_distribution does (probabilities and cumulative sums in double, last
// sum forced to 1.0, lower_bound of a uniform double that the HOST takes from std::mt19937 in sequence order), and the
// k-mer counts n[k][y][j] += 1 of the sampled site for every order k <= K. Y: index array of order >= max(K,1).
// One warp per sequence; scratch: one row of max(LW1)+1 floats per warp.
template <typename YT>
__global__ void __launch_bounds__(256)
k_pwm_sample_sites(const YT* __restrict__ Y, const uint64_t* __restrict__ seq_off, const uint32_t* __restrict__ ids, uint32_t nsub,
                   int W, int K, uint32_t A, uint32_t asize, const float* __restrict__ score_g /* [asize][W] */, float q,
                   const double* __restrict__ uniforms, float* __restrict__ scratch, uint64_t scratch_stride,
                   int* __restrict__ n_all, const uint32_t* __restrict__ voff /* [K+2] */, unsigned long long* __restrict__ z_out) {
    __shared__ float score[6 * BAMM_MAX_MOTIF_WIDTH];
    for (uint32_t i = threadIdx.x; i < asize * (uint32_t)W; i += blockDim.x) score[i] = score_g[i];
    __syncthreads();
    const int lane = threadIdx.x & 31;
    const uint32_t warp = blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
    const uint32_t nwarps = gridDim.x * (blockDim.x >> 5);
    float* __restrict__ r = scratch + (uint64_t)warp * scratch_stride;
    for (uint32_t li = warp; li < nsub; li += nwarps) {
        const uint32_t n = ids[li];
        const uint64_t base = seq_off[n], L = seq_off[n + 1] - base, LW1 = L - W + 1;
        const YT* __restrict__ yn = Y + base;
        const float pos0 = 1.0f - q, pos1 = q / (float)LW1;
        for (uint64_t i = 1 + lane; i <= LW1; i += 32) {
            float v = 1.0f;
            for (int j = 0; j < W; j++) v *= score[((uint32_t)yn[i - 1 + j] % asize) * W + j];
            r[i] = v * pos1;
        }
        __syncwarp();
        float norm = 0.0f;
        if (lane == 0) {
            for (uint64_t i = 1; i <= LW1; i++) norm += r[i];
            r[0] = pos0;
            norm += r[0];
        }
        norm = __shfl_sync(FULL, norm, 0);
        __syncwarp();
        for (uint64_t i = lane; i <= LW1; i += 32) r[i] /= norm;
        __syncwarp();
        unsigned long long z = 0;
        if (lane == 0) {
            double sum = 0.0;
            for (uint64_t i = 0; i <= LW1; i++) sum += (double)r[i];
            const double p = uniforms[li];
            double run = 0.0;
            z = LW1;                                                        // the last cumulative sum is forced to 1.0
            for (uint64_t i = 0; i < LW1; i++) {
                run += (double)r[i] / sum;
                if (!(run < p)) { z = i; break; }                           // lower_bound: first cumulative sum >= p
            }
        }
        z = __shfl_sync(FULL, z, 0);
        if (z_out && lane == 0) z_out[li] = z;
        if (z > 0) {
            uint32_t Yk1 = A;
            for (int k = 0; k <= K; k++) {
                for (int j = lane; j < W; j += 32) atomicAdd(&n_all[voff[k] + ((uint32_t)yn[z - 1 + j] % Yk1) * W + j], 1);
                Yk1 *= A;
            }
        }
        __syncwarp();
    }
}

}  // namespace bamm
