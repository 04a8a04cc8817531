// scan.cuh — occurrence scan (BaMMScan; DESIGN.md §4.7): window-parallel log-odds scoring of a subset's window stream, the
// negative side written for a device sort, the positive side fused with the p-value of ScoreSeqSet::calcPvalues and an
// ordered compaction of the windows with p < cutoff (ScoreSeqSet.cpp:245-291).
//
// Windows, not sequences, are the unit of work: subset entry i owns the windows [roff[i], roff[i+1]) of one flat stream
// (L - W + 1 per sequence, subset order, window ascending), and a CTA takes a tile of SCAN_TILE consecutive windows whatever
// sequences they belong to. A record of 10^8 bases spreads over the whole device; a tile of records with L = W holds 2048 of
// them. Only full windows are in the stream, so nothing has to be masked.
#pragma once
#include "../../include/bamm_b200.h"
#include "stats.cuh"

namespace bamm {

constexpr int SCAN_THREADS = 512, SCAN_ROUNDS = 4, SCAN_TILE = SCAN_THREADS * SCAN_ROUNDS;
constexpr int SCAN_SAMPLES = 2048;   // sorted negatives kept in shared memory: the upper levels of every p-value's search

struct ScanWindows {
    const unsigned long long* roff;    // nsub+1 prefix sums of the windows per subset entry
    const unsigned long long* wbase;   // per subset entry: stored position of its window 0 minus roff[i] (mod 2^64), so the
                                       // index-array position of window g of entry i is wbase[i] + g
    unsigned long long nsub;
    unsigned long long first, count;   // the windows [first, first + count) of this launch; tile t starts at first + t * SCAN_TILE
};

// the subset entry of window g, searched in [lo, hi] (every entry owns at least one window: roff is strictly increasing)
__device__ __forceinline__ unsigned long long scan_entry(const unsigned long long* __restrict__ roff, unsigned long long lo,
                                                         unsigned long long hi, unsigned long long g) {
    while (lo < hi) {
        const unsigned long long mid = (lo + hi + 1) >> 1;
        if (roff[mid] <= g) lo = mid; else hi = mid - 1;
    }
    return lo;
}

// the entries of the tile's first and last window, for the per-window searches of the whole CTA
__device__ __forceinline__ void scan_tile_entries(const ScanWindows& sw, unsigned long long g0, unsigned long long* sh) {
    if (threadIdx.x == 0) sh[0] = scan_entry(sw.roff, 0, sw.nsub - 1, g0);
    if (threadIdx.x == 32) {
        const unsigned long long end = sw.first + sw.count, last = (g0 + SCAN_TILE < end ? g0 + SCAN_TILE : end) - 1;
        sh[1] = scan_entry(sw.roff, 0, sw.nsub - 1, last);
    }
    __syncthreads();
}

// Scores every window of the launch: sc[g - first] = sum_{j = 0 .. W-1} s[j][y(g + j)], in ascending j from 0.0f like k_score
// (ScoreSeqSet.cpp:49-54), so the scores are the same bits. Each thread reads its own W indices; the neighbouring threads of a
// warp read neighbouring positions, so every index load is one coalesced request and the tile's indices stay in L1 (no
// shuffles, and no column blocks for W > 32). SMEM: the [j][y] table is copied to shared memory, else read through L2.
// POS: also the p-value of every window against the sorted negatives (mops_pvalue: the formula of k_mops_pvalues), pv[g - first],
// and the number of windows with p < cutoff per tile, tile_hits[t]. The search for the upper bound runs through SCAN_SAMPLES
// evenly spaced negatives in shared memory first and ends in global memory between two neighbouring samples; both searches
// use the predicate neg[idx] > Sl of upper_bound_f32, so the result is the index of the full search.
template <typename YT, bool SMEM, bool POS>
__global__ void __launch_bounds__(SCAN_THREADS)
k_scan_score(const YT* __restrict__ Y, ScanWindows sw, int W, uint32_t Yn, const float* __restrict__ s_g,
             float* __restrict__ sc_out,
             const float* __restrict__ neg, unsigned long long negN, const float* __restrict__ samples, uint32_t nsamp,
             unsigned long long step, MopsTail tail, float cutoff, float* __restrict__ pv_out, uint32_t* __restrict__ tile_hits) {
    extern __shared__ float sh[];
    __shared__ unsigned long long ent[2];
    float* samp = sh;                                        // POS: nsamp floats
    const float* s = s_g;
    if (POS) for (uint32_t i = threadIdx.x; i < nsamp; i += blockDim.x) samp[i] = samples[i];
    if (SMEM) {
        float* t = sh + (POS ? SCAN_SAMPLES : 0);
        for (uint32_t i = threadIdx.x; i < (uint32_t)W * Yn; i += blockDim.x) t[i] = s_g[i];
        s = t;
    }
    const unsigned long long g0 = sw.first + (unsigned long long)blockIdx.x * SCAN_TILE, end = sw.first + sw.count;
    scan_tile_entries(sw, g0, ent);                          // also the barrier of the shared-memory copies
    uint32_t nhit = 0;
#pragma unroll 1
    for (int k = 0; k < SCAN_ROUNDS; k++) {
        const unsigned long long g = g0 + (unsigned long long)k * SCAN_THREADS + threadIdx.x;
        bool hit = false;
        if (g < end) {
            const unsigned long long i = scan_entry(sw.roff, ent[0], ent[1], g);
            const YT* __restrict__ y = Y + (sw.wbase[i] + g);
            float sc = 0.0f;
#pragma unroll 4
            for (int j = 0; j < W; j++) sc += s[(uint32_t)j * Yn + y[j]];
            sc_out[g - sw.first] = sc;
            if (POS) {
                uint32_t c = 0, hi = nsamp;                  // first sample above sc
                while (c < hi) { const uint32_t mid = (c + hi) >> 1; if (samp[mid] > sc) hi = mid; else c = mid + 1; }
                const unsigned long long lo = c ? (unsigned long long)(c - 1) * step + 1 : 0;
                const unsigned long long up = c < nsamp ? (unsigned long long)c * step : negN;
                const float p = mops_pvalue(neg, negN, upper_bound_f32(neg, lo, up, sc), sc, tail);
                pv_out[g - sw.first] = p;
                hit = p < cutoff;
            }
        }
        if (POS) nhit += (uint32_t)__syncthreads_count(hit);
    }
    if (POS && threadIdx.x == 0) tile_hits[blockIdx.x] = nhit;
}

// Writes the hits of every tile with at least one, in window order, at tile_off[t] (exclusive prefix sums of tile_hits) and
// on: hit r of the launch goes to out[r] when r < limit (the caller's remaining capacity). The rank inside a tile comes from
// warp ballots, round after round, so the order is the window order whatever the schedule.
__global__ void __launch_bounds__(SCAN_THREADS)
k_scan_emit(ScanWindows sw, const float* __restrict__ sc, const float* __restrict__ pv, float cutoff, float posN,
            const uint32_t* __restrict__ tile_hits, const unsigned long long* __restrict__ tile_off, unsigned long long limit,
            bamm_hit* __restrict__ out) {
    if (tile_hits[blockIdx.x] == 0 || tile_off[blockIdx.x] >= limit) return;     // uniform over the CTA
    __shared__ unsigned long long ent[2];
    __shared__ uint32_t wcnt[SCAN_ROUNDS][SCAN_THREADS / 32];
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const unsigned long long g0 = sw.first + (unsigned long long)blockIdx.x * SCAN_TILE, end = sw.first + sw.count;
    uint32_t ballots[SCAN_ROUNDS];
#pragma unroll
    for (int k = 0; k < SCAN_ROUNDS; k++) {
        const unsigned long long g = g0 + (unsigned long long)k * SCAN_THREADS + threadIdx.x;
        ballots[k] = __ballot_sync(FULL, g < end && pv[g - sw.first] < cutoff);
        if (lane == 0) wcnt[k][warp] = __popc(ballots[k]);
    }
    scan_tile_entries(sw, g0, ent);
    uint32_t before = 0;                                     // hits of the tile in the rounds before k, running
#pragma unroll
    for (int k = 0; k < SCAN_ROUNDS; k++) {
        uint32_t rank = before;
        for (int w = 0; w < SCAN_THREADS / 32; w++) { const uint32_t c = wcnt[k][w]; if (w < warp) rank += c; before += c; }
        if ((ballots[k] >> lane) & 1u) {
            rank += __popc(ballots[k] & ((1u << lane) - 1u));
            const unsigned long long r = tile_off[blockIdx.x] + rank;
            if (r < limit) {
                const unsigned long long g = g0 + (unsigned long long)k * SCAN_THREADS + threadIdx.x;
                const unsigned long long i = scan_entry(sw.roff, ent[0], ent[1], g);
                const float p = pv[g - sw.first];
                bamm_hit h;
                h.seq = i; h.window = g - sw.roff[i];
                h.score = sc[g - sw.first]; h.p_value = p; h.e_value = p * posN; h.reserved = 0;
                out[r] = h;
            }
        }
    }
}

// every step-th of the nneg sorted negatives, for the shared-memory level of the searches in k_scan_score
__global__ void k_scan_samples(const float* __restrict__ neg, unsigned long long step, uint32_t nsamp, float* __restrict__ samples) {
    for (uint32_t i = blockIdx.x * blockDim.x + threadIdx.x; i < nsamp; i += gridDim.x * blockDim.x) samples[i] = neg[i * step];
}

}  // namespace bamm
