// kernels.cuh — sm_100a device code of the EM / scoring path.
//
// Data layout in HBM (DESIGN.md §3):
//   Y      : order-K k-mer index per stored position, uint16 (A^(K+1) <= 65536) or uint32, all sequences
//            concatenated in the seqset's order; y = kmer_[i] % A^(K+1) of the reference (Sequence.cpp:35-41).
//   s      : odds table, TRANSPOSED to [j][y] (reference Motif::s_[y][j]) so that the 32 lanes of a warp, which
//            look up the same motif column j for 32 different k-mers, spread over the shared-memory banks by y.
//   r      : posteriors, float per stored position, reference index order (i = L-W-p, zero tail).
//   counts : 64-bit fixed-point (scale 2^40) per (j,y); integer sums are associative, which makes the M-step
//            bit-reproducible for any CTA schedule, any grid size and any number of GPUs.
#pragma once
#pragma once
#include <cuda_runtime.h>
#include <cooperative_groups.h>
#include <stdint.h>
#include "common.cuh"

namespace bamm {

// ---------------------------------------------------------------------------------------------------------
// k-mer index build: y[i] = (sum_{t=0..K} digit(code[i-t]) * A^t) mod A^(K+1), digit(0) = 0 (patched afterwards),
// digit(c) = c-1 otherwise (also for the reverse-complemented N code 78, Alphabet.cpp:51). One warp per sequence.
// reference: src/init/Sequence.cpp:35-41 followed by `% Y_[K+1]` at every consumer (e.g. EM.cpp:170).
template <typename YT>
__global__ void k_build_index(const uint8_t* __restrict__ codes, const uint64_t* __restrict__ off, uint64_t nseq,
                              int A, int K, uint64_t Yn, YT* __restrict__ Y) {
    const int lane = threadIdx.x & 31;
    const uint64_t warp = (uint64_t)blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
    const uint64_t nwarps = (uint64_t)gridDim.x * (blockDim.x >> 5);
    for (uint64_t n = warp; n < nseq; n += nwarps) {
        const uint64_t base = off[n], L = off[n + 1] - base;
        for (uint64_t i = lane; i < L; i += 32) {
            uint64_t y = 0, pw = 1;
            for (int t = 0; t <= K && (uint64_t)t <= i; t++) {
                const uint32_t c = codes[base + i - t];
                y += (uint64_t)(c ? c - 1 : 0) * pw;
                pw *= (uint64_t)A;
            }
            Y[base + i] = (YT)(y % Yn);
        }
    }
}

template <typename YT>
__global__ void k_patch_index(const uint64_t* __restrict__ ppos, const uint64_t* __restrict__ pkmer, uint64_t np,
                              uint64_t Yn, YT* __restrict__ Y) {
    uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i < np) Y[ppos[i]] = (YT)(pkmer[i] % Yn);
}

// top-order k-mer histogram over all positions (reference: BackgroundModel.cpp:26-42; lower orders are folds).
// SMEM: CTA-private 32-bit histogram in shared memory (a CTA sees far fewer than 2^32 positions), flushed with one
// 64-bit global atomic per non-empty bin; otherwise global atomics directly.
template <typename YT, bool SMEM>
__global__ void k_count_kmers(const YT* __restrict__ Y, uint64_t npos, uint32_t Yn, unsigned long long* __restrict__ cnt) {
    extern __shared__ uint32_t hist[];
    if (SMEM) {
        for (uint32_t b = threadIdx.x; b < Yn; b += blockDim.x) hist[b] = 0u;
        __syncthreads();
    }
    uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
    const uint64_t stride = (uint64_t)gridDim.x * blockDim.x;
    for (; i < npos; i += stride) {
        if (SMEM) atomicAdd(&hist[Y[i]], 1u);
        else atomicAdd(&cnt[Y[i]], 1ull);
    }
    if (SMEM) {
        __syncthreads();
        for (uint32_t b = threadIdx.x; b < Yn; b += blockDim.x) if (hist[b]) atomicAdd(&cnt[b], (unsigned long long)hist[b]);
    }
}

// ---------------------------------------------------------------------------------------------------------
// Sliding k-mer window of a warp: lane l holds y[p0+l] and y[p0+32+l]; the k-mer under motif column j of the
// window that starts at p0+l is element l+j of that 64-entry strip (W <= 32; wider motifs: BlockStrip), fetched with one shuffle.
template <typename YT> struct Strip;
template <> struct Strip<uint16_t> {
    uint32_t packed;
    __device__ __forceinline__ void load(const uint16_t* __restrict__ y, uint64_t p, uint64_t L) {
        uint32_t a = (p < L) ? y[p] : 0u, b = (p + 32 < L) ? y[p + 32] : 0u;
        packed = a | (b << 16);
    }
    __device__ __forceinline__ uint32_t get(int lane, int j) const {
        const int src = lane + j;
        const uint32_t t = __shfl_sync(FULL, packed, src & 31);
        return (src < 32) ? (t & 0xffffu) : (t >> 16);
    }
};
template <> struct Strip<uint32_t> {
    uint32_t a, b;
    __device__ __forceinline__ void load(const uint32_t* __restrict__ y, uint64_t p, uint64_t L) {
        a = (p < L) ? y[p] : 0u; b = (p + 32 < L) ? y[p + 32] : 0u;
    }
    __device__ __forceinline__ uint32_t get(int lane, int j) const {
        const int src = lane + j;
        const uint32_t ta = __shfl_sync(FULL, a, src & 31), tb = __shfl_sync(FULL, b, src & 31);
        return (src < 32) ? ta : tb;
    }
};

// Column blocks of a wide motif (DESIGN.md §4.6): columns [32b, min(W, 32b+32)) for b < NB form block b, and the strip holds
// NB+1 segments of 32 k-mer indices, seg[s] = y[p0 + 32s + lane]. Block b reads the pair (seg[b], seg[b+1]) with the shuffle of
// Strip::get, so j still ascends from 0 and every product and sum keeps its order. NB = 1 is the Strip above (W <= 32).
template <typename YT, int NB> struct BlockStrip {
    uint32_t seg[NB + 1];
    __device__ __forceinline__ void load(const YT* __restrict__ y, uint64_t p, uint64_t L) {
#pragma unroll
        for (int s = 0; s <= NB; s++) seg[s] = (p + 32 * s < L) ? (uint32_t)y[p + 32 * s] : 0u;
    }
    // the strip of the windows 32 further on: the segments shift by one, one new segment is loaded
    __device__ __forceinline__ void load_next(const BlockStrip& cur, const YT* __restrict__ y, uint64_t p /* first new window */, uint64_t L) {
#pragma unroll
        for (int s = 0; s < NB; s++) seg[s] = cur.seg[s + 1];
        seg[NB] = (p + 32 * NB < L) ? (uint32_t)y[p + 32 * NB] : 0u;
    }
    __device__ __forceinline__ uint32_t get(int lane, int b, int jj) const {
        const int src = lane + jj;
        const uint32_t ta = __shfl_sync(FULL, seg[b], src & 31), tb = __shfl_sync(FULL, seg[b + 1], src & 31);
        return (src < 32) ? ta : tb;
    }
};
template <typename YT> struct BlockStrip<YT, 1> {
    Strip<YT> st;
    __device__ __forceinline__ void load(const YT* __restrict__ y, uint64_t p, uint64_t L) { st.load(y, p, L); }
    __device__ __forceinline__ void load_next(const BlockStrip&, const YT* __restrict__ y, uint64_t p, uint64_t L) { st.load(y, p, L); }
    __device__ __forceinline__ uint32_t get(int lane, int, int jj) const { return st.get(lane, jj); }
};
// f(b, jj) for the columns j = 32 b + jj, j = 0 .. W-1 in ascending order
template <int NB, typename F>
__device__ __forceinline__ void for_columns(int W, F&& f) {
    if (NB == 1) {
        for (int j = 0; j < W; j++) f(0, j);
    } else {
#pragma unroll
        for (int b = 0; b < NB; b++) {
            const int nc = min(W - 32 * b, 32);
#pragma unroll 8                                // the default unrolling spills in k_score
            for (int jj = 0; jj < nc; jj++) f(b, jj);
        }
    }
}
// column blocks a width needs (1 for W <= 32, 2 up to BAMM_MAX_MOTIF_WIDTH)
static inline int column_blocks(int W) { return W > 32 ? 2 : 1; }

struct SubsetView {
    const uint64_t* seq_off;   // seqset offsets (nseq+1)
    const uint32_t* seq_ids;   // subset -> seqset index, or nullptr for identity
    const uint64_t* r_off;     // subset prefix sums of L (nsub+1)
    uint32_t nsub;
};

// ---------------------------------------------------------------------------------------------------------
// E-step. reference: EM::EStep, src/refinement/EM.cpp:139-200, in the gather form of SURVEY.md §8a-1:
//   r[L-W-p] = ( prod_{j=0..min(W-1, L-W-p)} s[y(p+j)][j] ) * q/LW1 / norm,  norm = (1-q) + sum_p (...)
// The product runs in ascending j from 1.0f like the reference's scatter loop (EM.cpp:167-176), the prior is
// applied with one multiply (EM.cpp:180) and the normalisation is a true IEEE division (EM.cpp:186), so r differs
// from the reference only through the summation order inside norm. One warp per sequence; lanes = window starts.
// Scalars (log likelihood, sum of r for optimize_q) are accumulated per warp as 2^32 fixed point and added to
// the exchange buffer with one 64-bit atomic per warp: integer sums => order-independent result.
// NB: column blocks (column_blocks(W)).
template <typename YT, int NB>
__global__ void __launch_bounds__(512)
k_estep(const YT* __restrict__ Y, SubsetView sv, int W, uint32_t Yn, const float* __restrict__ s_g /* [j][y] */, float q,
        float* __restrict__ r, unsigned long long* __restrict__ scal /* [0]=llh_fx, [1]=rsum_fx */) {
    extern __shared__ float s_sh[];
    for (uint32_t i = threadIdx.x; i < (uint32_t)W * Yn; i += blockDim.x) s_sh[i] = s_g[i];
    __syncthreads();
    const float* s = s_sh;
    const int lane = threadIdx.x & 31;
    const uint32_t warp = blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
    const uint32_t nwarps = gridDim.x * (blockDim.x >> 5);
    long long llh_fx = 0, rsum_fx = 0;
    const float one_minus_q = 1.0f - q;
    // the offsets of the NEXT sequence and the k-mer indices of the NEXT 32 windows are loaded while the current ones are
    // processed: the table gathers of a round depend on its indices, a chain the 16 warps of a CTA do not cover by themselves
    struct Hdr { uint64_t base, L, roff; };
    auto load_hdr = [&](uint64_t i) {
        Hdr h; h.base = 0; h.L = 0; h.roff = 0;
        if (i < sv.nsub) {
            const uint32_t n = sv.seq_ids ? sv.seq_ids[i] : (uint32_t)i;
            h.base = sv.seq_off[n]; h.L = sv.seq_off[n + 1] - h.base; h.roff = sv.r_off[i];
        }
        return h;
    };
    Hdr hd = load_hdr(warp);
    for (uint64_t i = warp; i < sv.nsub; i += nwarps) {
        const Hdr hn = load_hdr(i + nwarps);
        const uint64_t L = hd.L;
        const uint64_t LW1 = L - W + 1;
        const YT* __restrict__ yn = Y + hd.base;
        float* __restrict__ rn = r + hd.roff;
        hd = hn;
        const float pos = q / (float)LW1;
        float sum = 0.0f;
        BlockStrip<YT, NB> st; st.load(yn, lane, L);
        for (uint64_t p0 = 0; p0 < LW1; p0 += 32) {
            const uint64_t p = p0 + lane;
            BlockStrip<YT, NB> nx; nx.load_next(st, yn, p + 32, L);
            const int jmax = (p < LW1) ? (int)min((uint64_t)(W - 1), L - W - p) : -1;
            float prod = 1.0f;
            for_columns<NB>(W, [&](int b, int jj) {
                const int j = 32 * b + jj;
                const uint32_t y = st.get(lane, b, jj);
                if (j <= jmax) prod *= s[(uint32_t)j * Yn + y];
            });
            if (p < LW1) {
                const float val = prod * pos;
                rn[L - W - p] = val;
                sum += val;
            }
            st = nx;
        }
        sum = warp_sum(sum);
        const float norm = one_minus_q + sum;
        __syncwarp();
        for (uint64_t k = lane; k < L; k += 32) rn[k] = (k < LW1) ? __fdiv_rn(rn[k], norm) : 0.0f;
        if (lane == 0) {
            llh_fx += __double2ll_rn((double)logf(norm) * SC_SCALE_D);
            rsum_fx += __double2ll_rn((double)__fdiv_rn(sum, norm) * SC_SCALE_D);
        }
    }
    if (lane == 0) {
        if (llh_fx) atomicAdd(&scal[0], (unsigned long long)llh_fx);
        if (rsum_fx) atomicAdd(&scal[1], (unsigned long long)rsum_fx);
    }
}

// ---------------------------------------------------------------------------------------------------------
// E-step for tables beyond shared memory, row form. The lanes of a warp own 32 consecutive POSITIONS: lane l loads the whole
// table row of its k-mer, s[y(i)][0..W) — W4/4 16-byte loads from the padded [y][W4] copy of the table — and window p takes
// column j from the lane that owns position p+j with one shuffle. A warp then touches 32 rows per 32 windows (3 load
// instructions at W = 12) where gathering one column at a time from the [y][j] table in global memory issues W gathers of 32
// scattered addresses each: the L1 wavefronts, which bound that form (ncu: 92 % of the LSU wavefront peak), drop by W / (W4/4). Same factors multiplied in the same order =>
// the same r, bit for bit. The rows of the next 32 positions and the k-mer indices of the 32 after them are in flight while
// the current round is multiplied.
// A motif wider than 32 columns takes two column passes, PASS 1 over columns [0, 32) and PASS 2 over [32, W), and the product of
// PASS 1 is stored in r: the rows of both blocks for this round and the next would be 4 x 32 floats per lane, beyond the 128
// registers of a 512-thread CTA. PASS 2 continues the product from the stored float, so the factors are multiplied in the same
// order. PASS 0 takes all W <= 32 columns at once. RS: row stride of the padded table in PASS 1 / 2 (PASS 0: W4).
__global__ void k_pad_rows(const float* __restrict__ sT /* [y][W] */, int W, int W4, uint32_t Yn, float* __restrict__ out /* [y][W4] */) {
    const uint32_t total = Yn * (uint32_t)W4;
    for (uint32_t i = blockIdx.x * blockDim.x + threadIdx.x; i < total; i += gridDim.x * blockDim.x) {
        const uint32_t y = i / W4, j = i % W4;
        out[i] = j < (uint32_t)W ? sT[y * (uint32_t)W + j] : 1.0f;
    }
}
// PASS 1 / 2 ask ptxas for one CTA per SM: its occupancy heuristic otherwise caps the PASS 2 instantiations near 64 registers and spills
template <typename YT, int W4, int PASS>
__global__ void __launch_bounds__(512, PASS == 0 ? 0 : 1)
k_estep_rows(const YT* __restrict__ Y, SubsetView sv, int W, const float* __restrict__ rows /* [y][RS] */, int RS, float q,
             float* __restrict__ r, unsigned long long* __restrict__ scal /* [0]=llh_fx, [1]=rsum_fx */) {
    constexpr int C0 = PASS == 2 ? 32 : 0;                                      // first column of this pass
    const int lane = threadIdx.x & 31;
    const uint32_t warp = blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
    const uint32_t nwarps = gridDim.x * (blockDim.x >> 5);
    long long llh_fx = 0, rsum_fx = 0;
    const float one_minus_q = 1.0f - q;
    const int nc = PASS == 1 ? 32 : W - C0;                                     // columns of this pass
    struct Hdr { uint64_t base, L, roff; };
    auto load_hdr = [&](uint64_t i) {
        Hdr h; h.base = 0; h.L = 0; h.roff = 0;
        if (i < sv.nsub) {
            const uint32_t n = sv.seq_ids ? sv.seq_ids[i] : (uint32_t)i;
            h.base = sv.seq_off[n]; h.L = sv.seq_off[n + 1] - h.base; h.roff = sv.r_off[i];
        }
        return h;
    };
    auto load_row = [&](float (&dst)[W4], bool on, uint32_t y) {
        const float4* __restrict__ src = reinterpret_cast<const float4*>(rows + (size_t)y * (PASS == 0 ? W4 : RS) + C0);
#pragma unroll
        for (int qd = 0; qd < W4 / 4; qd++) {
            float4 v = make_float4(1.0f, 1.0f, 1.0f, 1.0f);
            if (on) v = __ldg(src + qd);
            dst[4 * qd] = v.x; dst[4 * qd + 1] = v.y; dst[4 * qd + 2] = v.z; dst[4 * qd + 3] = v.w;
        }
    };
    Hdr hd = load_hdr(warp);
    for (uint64_t i = warp; i < sv.nsub; i += nwarps) {
        const Hdr hn = load_hdr(i + nwarps);
        const uint32_t L = (uint32_t)hd.L, LW1 = L - W + 1;                      // stored lengths are below 2^32
        const YT* __restrict__ yn = Y + hd.base;
        float* __restrict__ rn = r + hd.roff;
        hd = hn;
        const float pos = q / (float)LW1;
        float sum = 0.0f;
        float cur[W4], nxt[W4];
        load_row(cur, (uint32_t)lane + C0 < L, (uint32_t)lane + C0 < L ? (uint32_t)yn[lane + C0] : 0u);
        uint32_t y1 = 32u + C0 + lane < L ? (uint32_t)yn[32 + C0 + lane] : 0u;   // k-mer of this lane's position in the next round
        for (uint32_t p0 = 0; p0 < LW1; p0 += 32) {
            const uint32_t p = p0 + lane;
            load_row(nxt, p + C0 + 32 < L, y1);
            y1 = p + C0 + 64 < L ? (uint32_t)yn[p + C0 + 64] : 0u;
            const int jmax = (p < LW1) ? (int)min((uint32_t)(W - 1), L - W - p) - C0 : -1;    // last column of this pass
            float prod = (PASS == 2 && p < LW1) ? rn[L - W - p] : 1.0f;
#pragma unroll
            for (int j = 0; j < W4; j++) {
                // position p+C0+j belongs to lane (lane+j) mod 32 of this round if lane+j < 32, of the next round otherwise
                if (j >= nc) break;                                                  // padding columns (uniform)
                const float v = __shfl_sync(FULL, lane >= j ? cur[j] : nxt[j], (lane + j) & 31);
                if (j <= jmax) prod *= v;
            }
            if (p < LW1) {
                if (PASS == 1) {
                    rn[L - W - p] = prod;
                } else {
                    const float val = prod * pos;
                    rn[L - W - p] = val;
                    sum += val;
                }
            }
#pragma unroll
            for (int j = 0; j < W4; j++) cur[j] = nxt[j];
        }
        if (PASS == 1) continue;
        sum = warp_sum(sum);
        const float norm = one_minus_q + sum;
        __syncwarp();
        for (uint32_t k = lane; k < L; k += 32) rn[k] = (k < LW1) ? __fdiv_rn(rn[k], norm) : 0.0f;
        if (lane == 0) {
            llh_fx += __double2ll_rn((double)logf(norm) * SC_SCALE_D);
            rsum_fx += __double2ll_rn((double)__fdiv_rn(sum, norm) * SC_SCALE_D);
        }
    }
    if (lane == 0) {
        if (llh_fx) atomicAdd(&scal[0], (unsigned long long)llh_fx);
        if (rsum_fx) atomicAdd(&scal[1], (unsigned long long)rsum_fx);
    }
}

// ---------------------------------------------------------------------------------------------------------
// M-step accumulation. reference: EM::MStep, src/refinement/EM.cpp:230-243, gather form (SURVEY.md §8a-2):
//   n[K][y(p+j)][j] += r[L-W-p]   for every window start p and j <= min(W-1, L-W-p).
// Each r is converted ONCE to 2^40 fixed point (round to nearest) and added with native 32-bit integer shared
// atomics to the low word of a CTA-private table; the returned old value tells whether the low word wrapped,
// and the carry (plus the high word of large r) goes to the CTA's 64-bit partial table in global memory.
// No floating-point atomics anywhere => the sum is exact in fixed point and independent of execution order.
template <typename YT, bool SMEM, int NB /* column blocks, as k_estep */>
__global__ void __launch_bounds__(512)
k_mstep(const YT* __restrict__ Y, SubsetView sv, int W, uint32_t Yn, const float* __restrict__ r,
        unsigned long long* __restrict__ part /* SMEM: [gridDim.x][W*Yn]; else nrep [W*Yn] tables shared by the CTAs */, uint32_t nrep) {
    extern __shared__ uint32_t lo_sh[];
    const uint32_t nbin = (uint32_t)W * Yn;
    // tables too large for shared memory: CTA c adds into copy c % nrep in global memory, so that the few hot bins of a
    // large alphabet (A = 6 data is mostly ACGT) are not one serialised address for the whole grid
    unsigned long long* mypart = part + (uint64_t)(SMEM ? blockIdx.x : blockIdx.x % nrep) * nbin;
    if (SMEM) {
        for (uint32_t i = threadIdx.x; i < nbin; i += blockDim.x) lo_sh[i] = 0u;
        __syncthreads();
    }
    const int lane = threadIdx.x & 31;
    const uint32_t warp = blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
    const uint32_t nwarps = gridDim.x * (blockDim.x >> 5);
    for (uint32_t i = warp; i < sv.nsub; i += nwarps) {
        const uint32_t n = sv.seq_ids ? sv.seq_ids[i] : i;
        const uint64_t base = sv.seq_off[n], L = sv.seq_off[n + 1] - base;
        const uint64_t LW1 = L - W + 1;
        const YT* __restrict__ yn = Y + base;
        const float* __restrict__ rn = r + sv.r_off[i];
        for (uint64_t p0 = 0; p0 < LW1; p0 += 32) {
            const uint64_t p = p0 + lane;
            BlockStrip<YT, NB> st; st.load(yn, p, L);
            int jmax = -1;
            unsigned long long X = 0;
            if (p < LW1) {
                const float rv = rn[L - W - p];
                if (rv > 0.0f) { X = __float2ull_rn(rv * FX_SCALE_F); jmax = (int)min((uint64_t)(W - 1), L - W - p); }
                if (X == 0) jmax = -1;
            }
            const uint32_t xlo = (uint32_t)X, xhi = (uint32_t)(X >> 32);
            for_columns<NB>(W, [&](int b, int jj) {
                const int j = 32 * b + jj;
                const uint32_t y = st.get(lane, b, jj);
                if (j <= jmax) {
                    const uint32_t bin = (uint32_t)j * Yn + y;
                    if (SMEM) {
                        const uint32_t old = atomicAdd(&lo_sh[bin], xlo);
                        const uint32_t h = xhi + ((uint32_t)(old + xlo) < old ? 1u : 0u);
                        if (h) atomicAdd(&mypart[bin], (unsigned long long)h << 32);
                    } else {
                        atomicAdd(&mypart[bin], X);
                    }
                }
            });
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

// The same accumulation when the W * Yn table does not fit shared memory but a few columns do (A = 6 at order 5: one
// column = 187 KB): the grid is cut into nsplit column ranges x ngroups sequence shares, CTA (share g, range c) keeps the low
// words of columns [c nc, c nc + nc) in shared memory and adds into partial table g. r is read once per column range
// (L2 / HBM streaming) instead of paying one 64-bit global atomic per window and column.
constexpr int MC_U = 4;
template <typename YT, bool NC1 /* one column per CTA */>
__global__ void __launch_bounds__(1024)
k_mstep_cols(const YT* __restrict__ Y, SubsetView sv, int W, uint32_t Yn, const float* __restrict__ r,
             unsigned long long* __restrict__ part /* [gridDim.x / nsplit][W*Yn] */, int nsplit, int nc) {
    extern __shared__ uint32_t lo_sh[];
    const int split = blockIdx.x % nsplit, g = blockIdx.x / nsplit, ngroups = gridDim.x / nsplit;
    const int j0 = split * nc, j1 = min(W, j0 + nc);
    if (j0 >= j1) return;
    const uint32_t nb = (uint32_t)(j1 - j0) * Yn;
    for (uint32_t i = threadIdx.x; i < nb; i += blockDim.x) lo_sh[i] = 0u;
    __syncthreads();
    unsigned long long* mypart = part + (uint64_t)g * W * Yn + (uint64_t)j0 * Yn;
    const int lane = threadIdx.x & 31;
    const uint32_t wpc = blockDim.x >> 5;
    // One CTA per SM (the table fills shared memory), so the memory latency has to be covered inside the warp: the offsets of the
    // NEXT sequence are loaded while this one is processed (seq_ids -> seq_off is a chain of two loads), and the loads of the
    // next round of MC_U windows per lane (r and the k-mer index of the first column) are issued before the atomics of this one.
    struct Hdr { uint64_t base, L, roff; };
    auto load_hdr = [&](uint64_t i) {
        Hdr h; h.base = 0; h.L = 0; h.roff = 0;
        if (i < sv.nsub) {
            const uint32_t n = sv.seq_ids ? sv.seq_ids[i] : (uint32_t)i;
            h.base = sv.seq_off[n]; h.L = sv.seq_off[n + 1] - h.base; h.roff = sv.r_off[i];
        }
        return h;
    };
    const uint64_t first = (uint64_t)g * wpc + (threadIdx.x >> 5), stride = (uint64_t)ngroups * wpc;
    const uint32_t lo_base = (uint32_t)__cvta_generic_to_shared(lo_sh);
    Hdr h = load_hdr(first);
    for (uint64_t i = first; i < sv.nsub; i += stride) {
        const Hdr hn = load_hdr(i + stride);
        const uint32_t L = (uint32_t)h.L, LW1 = L - W + 1, lim = L - W;         // stored lengths are below 2^32 (host/SequenceSet.cpp)
        const YT* __restrict__ yn = Y + h.base + j0;                             // k-mer of the first column of window p: yn[p]
        const float* __restrict__ rn = r + h.roff + lim;                         // r of window p: rn[-p] (EM.cpp:173, reversed index)
        float rv[MC_U]; uint32_t yv[MC_U];
#pragma unroll
        for (int u = 0; u < MC_U; u++) {
            const uint32_t p = (uint32_t)lane + 32 * u;
            const bool in = p < LW1;                                             // then p + j0 <= L - W + j0 < L
            rv[u] = in ? *(rn - p) : 0.0f;
            yv[u] = in ? (uint32_t)yn[p] : 0u;
        }
        for (uint32_t p0 = lane; p0 < LW1; p0 += 32 * MC_U) {
            float rnx[MC_U]; uint32_t ynx[MC_U];
#pragma unroll
            for (int u = 0; u < MC_U; u++) {                                   // next round
                const uint32_t p = p0 + 32 * (MC_U + u);
                const bool in = p < LW1;
                rnx[u] = in ? *(rn - p) : 0.0f;
                ynx[u] = in ? (uint32_t)yn[p] : 0u;
            }
            unsigned long long X[MC_U];
#pragma unroll
            for (int u = 0; u < MC_U; u++) X[u] = rv[u] > 0.0f ? __float2ull_rn(rv[u] * FX_SCALE_F) : 0ull;      // 0 for p >= LW1
            if (NC1) {
                // one column per CTA (bin = k-mer): the low-word atomics of the round under predicates, then ONE branch for the
                // rare rest — a carry out of the low word or a posterior >= 2^-8 (high word) goes to the global partial table
                uint32_t hc[MC_U];
                uint32_t any = 0u;
#pragma unroll
                for (int u = 0; u < MC_U; u++) {
                    const uint32_t xlo = (uint32_t)X[u];
                    hc[u] = (uint32_t)(X[u] >> 32);
                    const bool on = X[u] != 0 && p0 + 32 * u + (uint32_t)j0 <= lim;     // j0 <= jmax = min(W-1, L-W-p), EM.cpp:167
                    // predicated shared-memory atomic: no branch region per window
                    uint32_t old = 0u;
                    asm volatile("{ .reg .pred p; setp.ne.u32 p, %3, 0; @p atom.shared.add.u32 %0, [%1], %2; }"
                                 : "+r"(old) : "r"(lo_base + (yv[u] << 2)), "r"(xlo), "r"((uint32_t)on) : "memory");
                    hc[u] = on ? hc[u] + ((uint32_t)(old + xlo) < old ? 1u : 0u) : 0u;
                    any |= hc[u];
                }
                if (any) {
#pragma unroll
                    for (int u = 0; u < MC_U; u++) if (hc[u]) atomicAdd(&mypart[yv[u]], (unsigned long long)hc[u] << 32);
                }
            } else {
                for (int j = j0; j < j1; j++) {
                    uint32_t y[MC_U];
#pragma unroll
                    for (int u = 0; u < MC_U; u++) y[u] = j == j0 ? yv[u] : (p0 + 32 * u + j < L ? (uint32_t)yn[p0 + 32 * u + (j - j0)] : 0u);
#pragma unroll
                    for (int u = 0; u < MC_U; u++) {
                        if (X[u] == 0 || p0 + 32 * u + (uint32_t)j > lim) continue;     // j <= jmax = min(W-1, L-W-p), EM.cpp:167
                        const uint32_t xlo = (uint32_t)X[u], xhi = (uint32_t)(X[u] >> 32);
                        const uint32_t bin = (uint32_t)(j - j0) * Yn + y[u];
                        const uint32_t old = atomicAdd(&lo_sh[bin], xlo);
                        const uint32_t hc = xhi + ((uint32_t)(old + xlo) < old ? 1u : 0u);
                        if (hc) atomicAdd(&mypart[bin], (unsigned long long)hc << 32);
                    }
                }
            }
#pragma unroll
            for (int u = 0; u < MC_U; u++) { rv[u] = rnx[u]; yv[u] = ynx[u]; }
        }
        h = hn;
    }
    __syncthreads();
    for (uint32_t i = threadIdx.x; i < nb; i += blockDim.x) {
        const uint32_t v = lo_sh[i];
        if (v) atomicAdd(&mypart[i], (unsigned long long)v);
    }
}

// Sum of the per-CTA partial tables (integers: any order gives the same bits) into the exchange buffer. A CTA sums 32
// consecutive bins; its RP_SUB warps each take every RP_SUB-th partial table (256-byte coalesced reads, nparts / RP_SUB
// independent loads per thread instead of nparts) and warp 0 adds the RP_SUB partial sums. Launch: RP_THREADS threads,
// reduce_grid(bins) CTAs.
constexpr int RP_SUB = 8, RP_THREADS = 32 * RP_SUB;
static inline unsigned reduce_grid(uint32_t bins) { return (bins + 31u) / 32u; }
__device__ __forceinline__ unsigned long long sum_parts_cta(const unsigned long long* __restrict__ part, uint32_t nparts, uint32_t nbin,
                                                            uint32_t b, unsigned long long (*sh)[32]) {
    const uint32_t sub = threadIdx.x >> 5, lane = threadIdx.x & 31;
    unsigned long long acc = 0;
    if (b < nbin) for (uint32_t c = sub; c < nparts; c += RP_SUB) acc += part[(uint64_t)c * nbin + b];
    sh[sub][lane] = acc;
    __syncthreads();
    if (sub == 0) {
#pragma unroll
        for (int u = 1; u < RP_SUB; u++) acc += sh[u][lane];
    }
    return acc;                                   // complete in warp 0 only
}
__global__ void __launch_bounds__(RP_THREADS)
k_reduce_parts(const unsigned long long* __restrict__ part, uint32_t nparts, uint32_t nbin, unsigned long long* __restrict__ xbuf) {
    __shared__ unsigned long long sh[RP_SUB][32];
    const uint32_t b = blockIdx.x * 32 + (threadIdx.x & 31);
    const unsigned long long acc = sum_parts_cta(part, nparts, nbin, b, sh);
    if (threadIdx.x < 32 && b < nbin) xbuf[b] = acc;
}

// ---------------------------------------------------------------------------------------------------------
// Multi-GPU exchange over NVLink peer memory, fused into the tail of the M-step (SURVEY.md §5, §8e): the reduction of
// the per-CTA partial tables writes this rank's sums straight into slot [rank] of EVERY rank's receive buffer (peer
// stores through CUDA-IPC mapped pointers) and the last CTA to finish publishes the iteration's epoch in every rank's
// flag array. k_peer_sum on each rank then waits for all flags and adds the slots in rank order — the same integers
// on every rank, hence bit-identical models without a collective library call or a host round trip.
// Receive buffers are double-buffered by epoch parity: a rank can run at most one iteration ahead of its peers.
constexpr int MAX_PEERS = 16;
struct PeerPtrs { unsigned long long* slots[MAX_PEERS]; unsigned int* flags[MAX_PEERS]; };

__global__ void __launch_bounds__(RP_THREADS)
k_reduce_push(const unsigned long long* __restrict__ part, uint32_t nparts, uint32_t nbin,
                              const unsigned long long* __restrict__ scal /* 2 scalars of the E-step */,
                              PeerPtrs pp, int rank, int world, uint32_t parity, uint32_t epoch, unsigned int* __restrict__ done) {
    __shared__ unsigned long long sh[RP_SUB][32];
    const uint32_t words = nbin + 2;
    const uint32_t b = blockIdx.x * 32 + (threadIdx.x & 31);
    unsigned long long acc = sum_parts_cta(part, nparts, nbin, b, sh);
    if (threadIdx.x < 32 && b < words) {
        if (b >= nbin) acc = scal[b - nbin];
        const uint64_t at = ((uint64_t)parity * world + rank) * words + b;
        for (int p = 0; p < world; p++) pp.slots[p][at] = acc;
    }
    __threadfence_system();                       // this CTA's peer stores are visible before it counts itself done
    __syncthreads();
    if (threadIdx.x == 0) {
        const unsigned int prev = atomicAdd(done, 1u);
        if (prev == gridDim.x - 1) {              // last CTA: everything of this rank has landed
            *done = 0u;
            __threadfence_system();
            for (int p = 0; p < world; p++) {
                volatile unsigned int* f = pp.flags[p] + rank;
                *f = epoch;
            }
            __threadfence_system();
        }
    }
}

__device__ __forceinline__ unsigned long long global_timer_ns() {
    unsigned long long t;
    asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t));
    return t;
}
// wait_acc: nullptr, or two counters — nanoseconds CTA 0 spent waiting for the slowest rank (summed) and the number of waits
__global__ void k_peer_sum(const unsigned long long* __restrict__ slots /* [2][world][words] local */, const unsigned int* flags /* [world] local */,
                           int world, uint32_t nbin, uint32_t parity, uint32_t epoch, unsigned long long* __restrict__ xbuf,
                           unsigned long long* __restrict__ wait_acc) {
    const uint32_t words = nbin + 2;
    const bool timed = wait_acc != nullptr && blockIdx.x == 0 && threadIdx.x == 0;
    const unsigned long long t0 = timed ? global_timer_ns() : 0ull;
    if (threadIdx.x < (unsigned)world) {
        const volatile unsigned int* f = flags + threadIdx.x;
        while ((int)(*f - epoch) < 0) __nanosleep(200);      // epochs only grow; wrap-safe comparison
    }
    __syncthreads();
    if (timed) { wait_acc[0] += global_timer_ns() - t0; wait_acc[1] += 1ull; }
    __threadfence_system();
    const uint32_t b = blockIdx.x * blockDim.x + threadIdx.x;
    if (b >= words) return;
    unsigned long long acc = 0;
    for (int p = 0; p < world; p++) acc += __ldcv(&slots[((uint64_t)parity * world + p) * words + b]);
    xbuf[b] = acc;
}

// sequence list of a scoring call from the caller's 64-bit subset (NULL = the whole set): narrowed to 32 bits, range-checked
// (an index outside the set raises the flag and is replaced by 0, so the kernels that follow stay inside the set)
__global__ void k_ids_from_u64(const uint64_t* __restrict__ subset, uint64_t n, uint64_t nseq, uint32_t* __restrict__ out, uint32_t* __restrict__ bad) {
    const uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    uint64_t v = subset ? subset[i] : i;
    if (v >= nseq) { *bad = 1u; v = 0; }
    out[i] = (uint32_t)v;
}

// out[i] = i: the sequence list of an EM object over a whole set
__global__ void k_iota_u32(uint32_t* __restrict__ out, uint64_t n) {
    const uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n) out[i] = (uint32_t)i;
}

// ---------------------------------------------------------------------------------------------------------
// Model update, one CTA. reference: fold of the counts EM.cpp:247-254, Motif::updateV Motif.h:95-136,
// convergence term EM.cpp:102-107, Motif::calculateLinearS Motif.cpp:485-494. Every formula keeps the
// reference's operation order (compiled with -fmad=false); only sum|dv| is a tree instead of a serial sum.
struct ModelDims { int A, K, W, K_bg; uint32_t Y[16]; uint32_t voff[16]; uint32_t bgoff[16]; };

// CL = 1: one CTA, phases separated by __syncthreads. CL = 8: one thread-block cluster of 8 CTAs (large tables, orders >= 4
// or the 6-letter alphabet): the same phases over 8 x 1024 threads, separated by the cluster barrier (release / acquire at
// cluster scope makes the other CTAs' global writes visible); sum|dv| goes through per-CTA partials summed in rank order.
template <int CL>
__device__ __forceinline__ void update_sync() {
    if (CL == 1) __syncthreads();
    else cooperative_groups::this_cluster().sync();
}
template <int CL>
__device__ __forceinline__ void update_model_body(ModelDims d, const unsigned long long* __restrict__ xbuf /* [W*Yn] fixed-point counts, [j][y] */,
               float* __restrict__ n_all, float* __restrict__ v_all, float* __restrict__ vK_prev,
               const float* __restrict__ vbg_all, const float* __restrict__ alpha,
               float* __restrict__ s_lin /* [j][y] */, float* __restrict__ s_rows /* [y][j], same values */,
               float* __restrict__ vdiff_out, double* __restrict__ vdiff_part /* [CL], CL > 1 only */) {
    const int W = d.W, K = d.K, A = d.A;
    const uint32_t YK = d.Y[K + 1];
    const uint32_t crank = CL == 1 ? 0u : cooperative_groups::this_cluster().block_rank();
    const uint32_t tid = crank * blockDim.x + threadIdx.x, nt = CL * blockDim.x;
    __shared__ float sumN[64];
    static_assert(BAMM_MAX_MOTIF_WIDTH <= 64, "sumN holds one sum per column");
    __shared__ double red[32];
    // top-order counts: fixed point -> float, [j][y] -> [y][j]
    float* nK = n_all + d.voff[K];
    for (uint32_t i = tid; i < YK * (uint32_t)W; i += nt) {
        const uint32_t y = i / W, j = i % W;
        nK[i] = (float)((double)(long long)xbuf[(uint32_t)j * YK + y] * FX_INV_D);
    }
    update_sync<CL>();
    // fold to lower orders: n[k-1][y2][j] = ((0 + n[k][0*Y_k+y2][j]) + n[k][1*Y_k+y2][j]) + ...  (EM.cpp:247-254)
    for (int k = K; k > 0; k--) {
        const float* nk = n_all + d.voff[k];
        float* nk1 = n_all + d.voff[k - 1];
        const uint32_t Yk = d.Y[k];
        for (uint32_t i = tid; i < Yk * (uint32_t)W; i += nt) {
            const uint32_t y2 = i / W, j = i % W;
            float acc = 0.0f;
            for (int a = 0; a < A; a++) acc += nk[((uint32_t)a * Yk + y2) * W + j];
            nk1[i] = acc;
        }
        update_sync<CL>();
    }
    // order 0 (Motif.h:101-118)
    if (threadIdx.x < (uint32_t)W) {                      // every CTA keeps its own copy of the column sums
        float sN = 0.0f;
        for (int y = 0; y < A; y++) sN += n_all[y * W + threadIdx.x];
        sumN[threadIdx.x] = sN;
    }
    __syncthreads();
    double dsum = 0.0;
    for (uint32_t i = tid; i < (uint32_t)A * W; i += nt) {
        const uint32_t y = i / W, j = i % W;
        const float nv = (n_all[i] + alpha[j] * vbg_all[y]) / (sumN[j] + alpha[j]);
        if (K == 0) { dsum += (double)fabsf(nv - vK_prev[i]); vK_prev[i] = nv; }
        v_all[i] = nv;
    }
    update_sync<CL>();
    // orders 1..K (Motif.h:121-135)
    for (int k = 1; k <= K; k++) {
        float* vk = v_all + d.voff[k];
        const float* vk1 = v_all + d.voff[k - 1];
        const float* nk = n_all + d.voff[k];
        const float* nk1 = n_all + d.voff[k - 1];
        const float* ak = alpha + k * W;
        const uint32_t Yk1 = d.Y[k + 1], Yk = d.Y[k];
        for (uint32_t i = tid; i < Yk1 * (uint32_t)W; i += nt) {
            const uint32_t y = i / W, j = i % W;
            const uint32_t y2 = y % Yk, yk = y / A;
            float nv;
            if ((int)j < k) nv = vk1[y2 * W + j];
            else nv = (nk[i] + ak[j] * vk1[y2 * W + j]) / (nk1[yk * W + j - 1] + ak[j]);
            if (k == K) { dsum += (double)fabsf(nv - vK_prev[i]); vK_prev[i] = nv; }
            vk[i] = nv;
        }
        update_sync<CL>();
    }
    // sum |dv|
    for (int o = 16; o > 0; o >>= 1) dsum += __shfl_xor_sync(FULL, dsum, o);
    if ((threadIdx.x & 31) == 0) red[threadIdx.x >> 5] = dsum;
    __syncthreads();
    if (threadIdx.x == 0) {
        double t = 0.0;
        for (uint32_t w = 0; w < (blockDim.x >> 5); w++) t += red[w];
        if (CL == 1) *vdiff_out = (float)t; else vdiff_part[crank] = t;
    }
    if (CL > 1) {
        update_sync<CL>();
        if (tid == 0) {
            double t = 0.0;
            for (int c = 0; c < CL; c++) t += vdiff_part[c];
            *vdiff_out = (float)t;
        }
    }
    // next E-step's table (Motif.cpp:485-494), transposed to [j][y]
    const float* vK = v_all + d.voff[K];
    const float* vb = vbg_all + d.bgoff[d.K_bg];
    const uint32_t YB = d.Y[d.K_bg + 1];
    for (uint32_t i = tid; i < YK * (uint32_t)W; i += nt) {
        const uint32_t y = i / W, j = i % W;
        const float sv = vK[i] / vb[y % YB];
        s_lin[(uint32_t)j * YK + y] = sv;
        s_rows[i] = sv;
    }
}

__global__ void __launch_bounds__(1024)
k_update_model(ModelDims d, const unsigned long long* __restrict__ xbuf, float* __restrict__ n_all, float* __restrict__ v_all,
               float* __restrict__ vK_prev, const float* __restrict__ vbg_all, const float* __restrict__ alpha,
               float* __restrict__ s_lin, float* __restrict__ s_rows, float* __restrict__ vdiff_out) {
    update_model_body<1>(d, xbuf, n_all, v_all, vK_prev, vbg_all, alpha, s_lin, s_rows, vdiff_out, nullptr);
}
constexpr int UPDATE_CLUSTER = 8;
__global__ void __cluster_dims__(UPDATE_CLUSTER, 1, 1) __launch_bounds__(1024)
k_update_model_cluster(ModelDims d, const unsigned long long* __restrict__ xbuf, float* __restrict__ n_all, float* __restrict__ v_all,
                       float* __restrict__ vK_prev, const float* __restrict__ vbg_all, const float* __restrict__ alpha,
                       float* __restrict__ s_lin, float* __restrict__ s_rows, float* __restrict__ vdiff_out, double* __restrict__ vdiff_part) {
    update_model_body<UPDATE_CLUSTER>(d, xbuf, n_all, v_all, vK_prev, vbg_all, alpha, s_lin, s_rows, vdiff_out, vdiff_part);
}

// s table only (first E-step after set_model)
__global__ void k_make_s(ModelDims d, const float* __restrict__ v_all, const float* __restrict__ vbg_all,
                         float* __restrict__ s_lin, float* __restrict__ s_rows, float* __restrict__ vK_prev) {
    const int W = d.W, K = d.K;
    const uint32_t YK = d.Y[K + 1], YB = d.Y[d.K_bg + 1];
    const float* vK = v_all + d.voff[K];
    const float* vb = vbg_all + d.bgoff[d.K_bg];
    for (uint32_t i = blockIdx.x * blockDim.x + threadIdx.x; i < YK * (uint32_t)W; i += gridDim.x * blockDim.x) {
        const uint32_t y = i / W, j = i % W;
        const float sv = vK[i] / vb[y % YB];
        s_lin[(uint32_t)j * YK + y] = sv;
        s_rows[i] = sv;
        vK_prev[i] = vK[i];
    }
}

// ---------------------------------------------------------------------------------------------------------
// Scoring. reference: ScoreSeqSet::calcLogOdds, src/seq_scoring/ScoreSeqSet.cpp:25-67. Full windows (all W
// columns, :49-54), float sum in ascending j from 0.0f (bit-identical to the reference for the same table),
// per-sequence maximum with the FIRST maximal window winning (strict '>' scan, :59-62).
template <typename YT, bool SMEM, int NB /* column blocks, as k_estep */>
__global__ void __launch_bounds__(512)
k_score(const YT* __restrict__ Y, SubsetView sv, const uint64_t* __restrict__ mops_off, int W, uint32_t Yn,
        const float* __restrict__ s_g, float* __restrict__ zoops, unsigned long long* __restrict__ z,
        float* __restrict__ mops, const uint32_t* __restrict__ out_idx /* list -> output slot, nullptr = identity */) {
    extern __shared__ float s_sh[];
    const float* s = s_g;
    if (SMEM) {
        for (uint32_t i = threadIdx.x; i < (uint32_t)W * Yn; i += blockDim.x) s_sh[i] = s_g[i];
        __syncthreads();
        s = s_sh;
    }
    const int lane = threadIdx.x & 31;
    const uint32_t warp = blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
    const uint32_t nwarps = gridDim.x * (blockDim.x >> 5);
    for (uint32_t i = warp; i < sv.nsub; i += nwarps) {
        const uint32_t n = sv.seq_ids ? sv.seq_ids[i] : i;
        const uint32_t oi = out_idx ? out_idx[i] : i;
        const uint64_t base = sv.seq_off[n], L = sv.seq_off[n + 1] - base;
        const uint64_t LW1 = L - W + 1;
        const YT* __restrict__ yn = Y + base;
        float best = -3.402823466e+38f;   // -FLT_MAX, ScoreSeqSet.cpp:44
        uint64_t bestp = 0;
        for (uint64_t p0 = 0; p0 < LW1; p0 += 32) {
            const uint64_t p = p0 + lane;
            BlockStrip<YT, NB> st; st.load(yn, p, L);
            float sc = 0.0f;
            for_columns<NB>(W, [&](int b, int jj) {
                const uint32_t y = st.get(lane, b, jj);
                sc += s[(uint32_t)(32 * b + jj) * Yn + y];
            });
            if (p < LW1) {
                if (mops) mops[mops_off[oi] + p] = sc;
                if (sc > best) { best = sc; bestp = p; }
            }
        }
        // lanes scanned ascending p with strict '>', so each lane holds its first maximum; combine: larger score
        // wins, equal scores -> smaller position (what the serial scan would have kept).
        for (int o = 16; o > 0; o >>= 1) {
            const float ob = __shfl_xor_sync(FULL, best, o);
            const uint64_t op = __shfl_xor_sync(FULL, bestp, o);
            if (ob > best || (ob == best && op < bestp)) { best = ob; bestp = op; }
        }
        if (lane == 0) { zoops[oi] = best; z[oi] = bestp; }
    }
}

}  // namespace bamm
