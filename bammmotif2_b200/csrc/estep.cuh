// estep.cuh — packed E-step kernels (4-letter alphabet, 2-bit stream). Included by launch_estep.cu only.
//
// reference: EM::EStep, src/refinement/EM.cpp:139-200 (gather form, SURVEY.md §8a-1). One warp per sequence.
//
// Column groups. Consecutive motif columns are folded into one lookup over the bases they depend on,
//   tab[g][z] = prod_{j in group g} s[j][ y_j(z) ],  so a window costs G shared-memory lookups instead of W; the byte offset of
// group g's entry is a bit field of the 64-bit window word (FAST: every field below bit 32 after the alignment shift: one
// funnel shift + one mask per lookup; otherwise a clamped funnel shift plus a second shift). Windows that cannot use whole
// groups (the last W-1 truncated windows, EM.cpp:167, and windows over the N whose k-mers hold rand() draws,
// Sequence.cpp:38) take a masked evaluation that mixes whole groups with single columns of the plain table.
//
// Two formulations, bit-identical results (same tables, same multiplication order, order-independent normaliser):
//   dense   k_estep_packed: every window exactly (G lookups), r written, active list written. Also the fall-back of the pruned
//           path, the column-pass variant for tables beyond shared memory (MULTI), and what materialises r for bamm_em_get_r.
//   pruned  k_ebound: every window gets an UPPER BOUND of its product from G1 < G lookups (tables over wider base ranges whose
//           leading columns take the maximum of s over the context bases outside the range); only windows whose bound reaches
//           the M-step's threshold 2^-41 (1-q) are listed. k_eexact evaluates the listed windows and the truncated / N windows
//           exactly, normalises, and writes the active list. Windows below the threshold add less than 2^-34 each to the
//           normaliser (>= 1-q) and exactly nothing to the counts; r is not written (bamm_em_get_r runs the dense kernel).
#pragma once
#include <type_traits>
#include "common.cuh"

namespace bamm {

#ifndef BAMM_E_UNROLL
#define BAMM_E_UNROLL 1          // unroll factor of the fast chunk loop
#endif

// ---- normaliser ----------------------------------------------------------------------------------------------------
// sum_p val(p) as integers, so that the dense and the pruned formulation, any lane assignment and any GPU count give the same
// bits: values below 2^20 in units of 2^-33 (a value below 2^-34 adds nothing: at most 1e3 windows * 2^-34 / (1-q) < 1e-7
// relative), values from 2^20 (exact multiples of 2^-3) in units of 2^-8.
struct NormAcc {
    unsigned long long a, b;
    __device__ __forceinline__ void clear() { a = 0ull; b = 0ull; }
    __device__ __forceinline__ void add(float val) {
        const bool big = val >= 1048576.0f;
        const unsigned long long x = __float2ull_rn(val * (big ? 256.0f : 8589934592.0f));
        a += big ? 0ull : x;
        b += big ? x : 0ull;
    }
    // sum over the warp, result in every lane: three 22-bit limbs per counter through the integer warp reduction (REDUX) instead
    // of five rounds of 64-bit shuffles; the counter of large values is zero in almost every warp
    static __device__ __forceinline__ unsigned long long sum_u64(unsigned long long x) {
        const unsigned long long s0 = __reduce_add_sync(FULL, (unsigned)(x & 0x3fffffull));
        const unsigned long long s1 = __reduce_add_sync(FULL, (unsigned)((x >> 22) & 0x3fffffull));
        const unsigned long long s2 = __reduce_add_sync(FULL, (unsigned)(x >> 44));
        return s0 + (s1 << 22) + (s2 << 44);
    }
    __device__ __forceinline__ void warp_reduce() {
        a = sum_u64(a);
        b = __any_sync(FULL, b != 0ull) ? sum_u64(b) : 0ull;
    }
    __device__ __forceinline__ double total() const { return (double)a * (1.0 / 8589934592.0) + (double)b * (1.0 / 256.0); }
};

// end of a sequence: normaliser, its reciprocal for the consumers of the unnormalised posteriors, log likelihood term
// (EM.cpp:183-195) and sum of the posteriors (optimize_q, EM.cpp:505-519)
__device__ __forceinline__ float finish_sequence(NormAcc acc, float one_minus_q, int lane, uint32_t li, float* __restrict__ scale,
                                                 long long& llh_fx, long long& rsum_fx) {
    acc.warp_reduce();
    const double sd = acc.total();
    const float norm = (float)((double)one_minus_q + sd);
    const float rnorm = __frcp_rn(norm);
    if (lane == 0) {
        scale[li] = rnorm;
        llh_fx += __double2ll_rn((double)logf(norm) * SC_SCALE_D);
        rsum_fx += __double2ll_rn((double)((float)sd * rnorm) * SC_SCALE_D);
    }
    return norm;
}

// ---- window evaluation ---------------------------------------------------------------------------------------------
template <int G> struct GroupConsts { uint32_t sh[G], mk[G], ab[G], s2[G]; };
template <int G>
__device__ __forceinline__ void load_consts(GroupConsts<G>& c, const GroupPlan& gp, uint32_t tab_s) {
#pragma unroll
    for (int g = 0; g < G; g++) { c.sh[g] = gp.shift[g]; c.mk[g] = gp.mask4[g]; c.ab[g] = tab_s + gp.base[g]; c.s2[g] = gp.shift2[g]; }
}
template <int G, bool FAST>
__device__ __forceinline__ uint32_t group_offset(const GroupConsts<G>& c, int g, uint32_t whi, uint32_t wlo) {
    if (FAST) return __funnelshift_r(wlo, whi, c.sh[g]) & c.mk[g];
    return (__funnelshift_rc(wlo, whi, c.sh[g]) >> c.s2[g]) & c.mk[g];
}
// full window: product of the G group entries in ascending g, starting from `prod`
template <int G, bool FAST>
__device__ __forceinline__ float groups_prod(const GroupConsts<G>& c, uint32_t whi, uint32_t wlo, float prod) {
#pragma unroll
    for (int g = 0; g < G; g++) prod *= lds_f32(group_offset<G, FAST>(c, g, whi, wlo), c.ab[g]);
    return prod;
}

// floats the padded shared-memory copy of the plain table takes (plain_words = W * Yn source floats, 0 = no copy)
__host__ __device__ __forceinline__ uint32_t plain_smem_words(uint32_t plain_words, uint32_t Yn) { return plain_words ? plain_words + plain_words / Yn : 0u; }

// launch-invariant inputs of the masked evaluation
struct MaskedTabs {
    const float* s_g;         // plain table [j][y], global
    uint32_t plain_s;         // shared-window address of a [j][y] copy in shared memory (rows Yn+1 floats apart: the lanes of a warp
                              // read one k-mer in different columns, or different k-mers in one column), or 0 when there is none
    uint32_t Yn, maskK, passmask;
    int W, K, KD;
};
// window p of a sequence of length L with the structural N at `mid` (-1: none), product over the columns j <= jmax that exist
// (EM.cpp:167) and belong to this column pass. Whole untouched groups come from the group tables (ascending g), then the
// remaining columns in ascending j from the plain table — with the k-mer of the stream, or, where it holds a draw of the N,
// the patched k-mer `yp[j - (mid - p)]` of the sequence. A full window away from the N multiplies exactly what groups_prod
// multiplies; k_emasked multiplies in the same order.
template <int G, bool FAST>
__device__ __forceinline__ float masked_prod(const GroupConsts<G>& c, const GroupPlan& gp, const MaskedTabs& mt, uint32_t whi, uint32_t wlo,
                                             int p, int jmax, int mid, const uint16_t* yp, float prod) {
    const int W = mt.W, K = mt.K;
    const unsigned long long w = ((unsigned long long)whi << 32) | wlo;
    const uint32_t valid = (jmax >= 0 ? (jmax >= 31 ? 0xffffffffu : ((2u << jmax) - 1u)) : 0u) & mt.passmask;
    uint32_t ncols = 0;                     // columns whose k-mer holds a rand() draw of the N
    const bool over_n = jmax >= 0 && mid >= 0 && p <= mid + K && p + W - 1 >= mid;
    if (over_n) {
        const int ja = max(mid - p, 0), jb = min(mid - p + K, W - 1);
        if (jb >= ja) ncols = ((jb >= 31 ? 0xffffffffu : ((2u << jb) - 1u))) & ~((1u << ja) - 1u) & mt.passmask;
    }
    uint32_t cols = valid;
    const uint32_t bad = ~valid | ncols;    // a group is whole and untouched when none of its columns is missing or patched
#pragma unroll
    for (int g = 0; g < G; g++) {
        const uint32_t cm = gp.colmask[g];
        const uint32_t off = group_offset<G, FAST>(c, g, whi, wlo);
        const bool good = (cm & bad) == 0u;
        float v = 1.0f;
        if (good) v = lds_f32(off, c.ab[g]);        // lanes without the group stay off the shared-memory pipe
        prod *= v;
        cols = good ? cols & ~cm : cols;
    }
    // one loop over the columns the groups left, in ascending order: k-mer from the stream or from the patch list, value from the
    // shared-memory copy of the plain table or from the global one (column passes, tables beyond shared memory)
    const int jn = mid - p;
    while (cols) {
        const int j = __ffs(cols) - 1;
        cols &= cols - 1u;
        uint32_t y = field(w, 62 - 2 * mt.KD - 2 * j, mt.maskK);
        if (over_n && (uint32_t)(j - jn) <= (uint32_t)K) y = yp[j - jn];
        prod *= mt.plain_s ? lds_f32(((uint32_t)j * (mt.Yn + 1u) + y) << 2, mt.plain_s) : __ldg(&mt.s_g[(uint32_t)j * mt.Yn + y]);
    }
    return prod;
}

// one region of the active list per warp: windows of full chunks / listed candidates at the front, masked windows at the back.
// Entry (common.cuh, ActiveEntry): word offset of the sequence, p | jmax << 26 | over-the-N << 31, unnormalised value, list index.
struct Emitter {
    ActiveEntry* __restrict__ reg;
    uint32_t cap, lpos, bpos, lt_mask;
    bool on;
    __device__ __forceinline__ void init(const ActiveList& al, uint32_t warp, bool enable) {
        on = enable && al.ent != nullptr;
        reg = on ? al.ent + al.reg_off[warp] : nullptr;
        cap = on ? (uint32_t)(al.reg_off[warp + 1] - al.reg_off[warp]) : 0u;
        lpos = 0; bpos = 0;
        asm("mov.u32 %0, %%lanemask_lt;" : "=r"(lt_mask));
    }
    template <bool BACK>
    __device__ __forceinline__ void put(const ActiveList& al, bool act, uint32_t woff, uint32_t pcode, float val, uint32_t li) {
        if (!on) return;
        const uint32_t m = __ballot_sync(FULL, act);
        if (!m) return;
        const uint32_t cnt = __popc(m);
        if (lpos + bpos + cnt > cap) { on = false; *al.overflow = 1u; return; }
        if (BACK) {
            bpos += cnt;
            if (act) *reinterpret_cast<uint4*>(reg + (cap - bpos) + __popc(m & lt_mask)) = make_uint4(woff, pcode, __float_as_uint(val), li);
        } else {
            if (act) *reinterpret_cast<uint4*>(reg + lpos + __popc(m & lt_mask)) = make_uint4(woff, pcode, __float_as_uint(val), li);
            lpos += cnt;
        }
    }
};
__device__ __forceinline__ uint32_t pcode_of(int p, int jmax, bool over_n) {
    return (uint32_t)p | ((uint32_t)(jmax < 0 ? 0 : jmax) << ACT_JMAX_SHIFT) | (over_n ? 0x80000000u : 0u);
}

// ---- dense E-step --------------------------------------------------------------------------------------------------
// lanes = 32 consecutive window starts. ONE pass: unnormalised posteriors go to r and, when they can reach the M-step's
// threshold, to the warp's region of the active list; the warp reduces the normaliser and stores its reciprocal per sequence.
// Segment schedule per sequence [0,b1) fast | [b1,b2) masked | [b2,b3) fast | [b3,LW1) masked.
// only_if: nullptr, or a device flag — the kernel runs only when it is non-zero (fall-back of the pruned path).
// plain_words: size of the [j][y] table copied to shared memory behind the group tables (0: single columns come from global).
template <int G, bool FAST, bool MULTI>
__global__ void __launch_bounds__(BAMM_E_THREADS, 1)
k_estep_packed(PackedView pv, const __grid_constant__ GroupPlan gp, const float* __restrict__ tab_g, const float* __restrict__ s_g /* [W][Yn] */,
               uint32_t plain_words, float* __restrict__ r, unsigned long long* __restrict__ scal,
               ActiveList al, const uint32_t* __restrict__ only_if) {
    extern __shared__ __align__(16) float tab[];
    __shared__ unsigned long long stage_bar;
    if (only_if != nullptr && *only_if == 0u) return;
    bulk_stage_begin(tab, tab_g, gp.table_bytes, &stage_bar);
    for (uint32_t i = threadIdx.x; i < plain_words; i += blockDim.x) tab[(gp.table_bytes >> 2) + i + i / gp.Yn] = s_g[i];   // rows padded by one float
    bulk_stage_wait(&stage_bar);
    __syncthreads();
    const int lane = threadIdx.x & 31;
    const uint32_t warp = blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
    const uint32_t nwarps = gridDim.x * (blockDim.x >> 5);
    const int W = gp.W, K = gp.K, KD = gp.kd;
    const uint32_t tab_s = (uint32_t)__cvta_generic_to_shared(tab);        // 32-bit shared-window address
    long long llh_fx = 0, rsum_fx = 0;
    const float one_minus_q = 1.0f - gp.q;
    constexpr int E_UNROLL = BAMM_E_UNROLL;
    // a window can only reach the M-step's threshold r >= 2^-41 if val >= 2^-41 (1-q): norm >= 1-q (margin for rounding)
    const float thr0 = gp.thr0;
    GroupConsts<G> gc; load_consts<G>(gc, gp, tab_s);
    MaskedTabs mt; mt.s_g = s_g; mt.plain_s = plain_words ? tab_s + gp.table_bytes : 0u;
    mt.Yn = gp.Yn; mt.maskK = gp.Yn - 1; mt.passmask = MULTI ? gp.passmask : 0xffffffffu; mt.W = W; mt.K = K; mt.KD = KD;
    const bool first = !MULTI || gp.pass_first != 0, last = !MULTI || gp.pass_last != 0;    // CTA-uniform
    Emitter em; em.init(al, warp, last);
    for (uint32_t li = warp; li < pv.nlist; li += nwarps) {
        const uint32_t n = pv.seq_ids[li];
        const PackedSeq sq = pv.seqs[n];
        const int L = (int)sq.L, LW1 = L - W + 1;
        const int mid = (int)sq.mid;                       // -1 when there is no N
        const uint32_t* __restrict__ wseq = pv.words + sq.word_off;
        const uint32_t woff = (uint32_t)sq.word_off;       // the active list exists only for streams below 2^32 words
        const uint16_t* __restrict__ yp = pv.ypatch + (uint64_t)n * (K + 1);
        float* __restrict__ rn = r + pv.r_off[li];
        const float pos = gp.q / (float)LW1;
        // windows that need the masked path: [n0,n1) over the N's patched k-mers (clipped to the tail), [tl,LW1) the truncated
        // tail (p > L-2W+1). Two candidates for the cuts: the exact ranges (fewest masked chunks, but a partial chunk at the
        // end of each fast segment) or rounded outwards to multiples of 32 (every fast chunk full, more windows in masked
        // chunks); a masked chunk costs about SLOW_COST fast chunks.
        const int tl = min(max(L - 2 * W + 2, 0), LW1);
        int b1 = tl, b2 = tl, b3 = tl;
        if (mid >= 0) { b1 = min(max(mid - W + 1, 0), tl); b2 = min(mid + K + 1, tl); }
        {
            constexpr int SLOW_COST = 4;
            const int a1 = b1 & ~31, a3 = tl & ~31, a2 = min((b2 + 31) & ~31, a3);
            const int cost_exact = ((b1 + 31) >> 5) + ((b3 - b2 + 31) >> 5) + SLOW_COST * (((b2 - b1 + 31) >> 5) + ((LW1 - b3 + 31) >> 5));
            const int cost_align = (a1 >> 5) + ((a3 - a2) >> 5) + SLOW_COST * (((a2 - a1) >> 5) + ((LW1 - a3 + 31) >> 5));
            if (cost_align <= cost_exact) { b1 = a1; b2 = a2; b3 = a3; }
        }
        NormAcc acc; acc.clear();
#pragma unroll 1
        for (int seg = 0; seg < 4; seg++) {
            const int p0 = seg == 0 ? 0 : seg == 1 ? b1 : seg == 2 ? b2 : b3;
            const int pe = seg == 0 ? b1 : seg == 1 ? b2 : seg == 2 ? b3 : LW1;
            if (p0 >= pe) continue;
            // this lane's windows start at p0+lane + 32*chunk; its window word starts KD bases earlier. Three stream words are
            // kept and two new ones are fetched per chunk of 32 windows.
            const int bb = p0 + lane - KD;
            const uint32_t* __restrict__ wl = wseq + (bb >> 4);
            const int sft = 2 * (bb & 15);
            uint32_t t0 = wl[0], t1 = wl[1], t2 = wl[2];
            int p = p0 + lane;
            float* __restrict__ rp = rn + (L - W - p);     // r index of this lane's window; moves down 32 per chunk
            if (!(seg & 1)) {
                // fast chunk: G table lookups, no masks; `tail` = the partial last chunk of the segment (lanes p >= pe are off)
                auto fast_chunk = [&](auto tail_tag) {
                    constexpr bool TAILC = decltype(tail_tag)::value;
                    const uint32_t whi = __funnelshift_l(t1, t0, sft), wlo = __funnelshift_l(t2, t1, sft);
                    wl += 2;
                    t0 = t2; t1 = wl[1]; t2 = wl[2];
                    const bool on = !TAILC || p < pe;
                    float prod = 1.0f;
                    if (MULTI && !first && on) prod = *rp;      // product over the columns of the earlier passes
                    prod = groups_prod<G, FAST>(gc, whi, wlo, prod);
                    if (MULTI && !last) { if (on) *rp = prod; }
                    else {
                        const float val = on ? prod * pos : 0.0f;
                        if (on) *rp = val;
                        acc.add(val);
                        em.template put<false>(al, val >= thr0, woff, pcode_of(p, W - 1, false), val, li);
                    }
                    rp -= 32; p += 32;
                };
#pragma unroll E_UNROLL
                for (int c = (pe - p0) >> 5; c > 0; c--) fast_chunk(std::false_type{});
                if ((pe - p0) & 31) fast_chunk(std::true_type{});
            } else {
#pragma unroll 1
                for (int c = (pe - p0 + 31) >> 5; c > 0; c--) {
                    const uint32_t whi = __funnelshift_l(t1, t0, sft), wlo = __funnelshift_l(t2, t1, sft);
                    wl += 2;
                    t0 = t2; t1 = wl[1]; t2 = wl[2];
                    const int jmax = (p < pe) ? min(W - 1, L - W - p) : -1;
                    float prod = 1.0f;
                    if (MULTI && !first && p < pe) prod = *rp;
                    prod = masked_prod<G, FAST>(gc, gp, mt, whi, wlo, p, jmax, mid, yp, prod);
                    float val = 0.0f;
                    if (p < pe) {
                        if (MULTI && !last) *rp = prod;
                        else { val = prod * pos; *rp = val; }
                    }
                    if (!MULTI || last) {
                        acc.add(val);
                        em.template put<true>(al, val >= thr0, woff, pcode_of(p, jmax, mid >= 0 && p <= mid + K && p + W - 1 >= mid), val, li);
                    }
                    rp -= 32; p += 32;
                }
            }
        }
        if (MULTI && !last) continue;
        // r keeps the unnormalised values; the factor is applied by whoever reads them (list / scan M-step,
        // k_normalise_r before r leaves the device). The tail beyond LW1 is zero since allocation.
        finish_sequence(acc, one_minus_q, lane, li, al.scale, llh_fx, rsum_fx);
    }
    if (lane == 0 && scal != nullptr) {
        if (llh_fx) atomicAdd(&scal[0], (unsigned long long)llh_fx);
        if (rsum_fx) atomicAdd(&scal[1], (unsigned long long)rsum_fx);
    }
    if (al.ent != nullptr && last) { al.cnt[warp] = em.lpos; al.cnt_back[warp] = em.bpos; }   // every lane holds the same counts
}

// ---- pruned E-step, part 1: bounds ---------------------------------------------------------------------------------
// gp here is the BOUND plan: G1 groups over base ranges [lo, hi]; an entry of tab[g] holds, as two bfloat16 rounded up, bounds of
// the product of the group's columns for window p and for window p+1, valid for every sequence context outside the range
// (k_make_bound_tables): G1 lookups per TWO windows. Windows in [n0,n1) (over the N) and from tl on (truncated) are
// left to k_eexact, which always evaluates them. The records of the next sequence (list entry two ahead, PackedSeq one ahead)
// and its first stream words are requested while the current one is processed: a warp never waits for a chain of loads.
template <int G1, bool FAST>
__global__ void __launch_bounds__(BAMM_E_THREADS, 1)
k_ebound(PackedView pv, const __grid_constant__ GroupPlan gp, const float* __restrict__ tab_g, CandList cl) {
    extern __shared__ __align__(16) float tab[];
    __shared__ unsigned long long stage_bar;
    volatile uint32_t* flags = cl.flags;
    if (flags[0] != 0u || (cl.reuse != nullptr && cl.reuse[BR_MODE] == 1u)) return;
    const bool build_list = cl.reuse != nullptr && cl.reuse[BR_MODE] == 0u;
    bulk_stage_begin(tab, tab_g, gp.table_bytes, &stage_bar);
    bulk_stage_wait(&stage_bar);
    if (build_list && blockIdx.x == 0)                    // the tables this watch list is built from
        for (uint32_t i = threadIdx.x; i < (gp.table_bytes >> 2); i += blockDim.x) cl.tab_ref[i] = tab[i];
    const int lane = threadIdx.x & 31;
    const uint32_t warp = blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
    const uint32_t nwarps = gridDim.x * (blockDim.x >> 5);
    const int W = gp.W, K = gp.K, KD = gp.kd;
    const uint32_t tab_s = (uint32_t)__cvta_generic_to_shared(tab);
    GroupConsts<G1> gc; load_consts<G1>(gc, gp, tab_s);
    uint32_t* __restrict__ creg = cl.ent + cl.reg_off[warp];
    const uint32_t ccap = (uint32_t)(cl.reg_off[warp + 1] - cl.reg_off[warp]);
    uint32_t cpos = 0;
    bool ok = true;
    // watch list: written in the same order as the candidates, so that filtering it keeps the candidates' order
    bool wok = build_list;
    uint32_t* __restrict__ wreg = wok ? cl.went + cl.wreg_off[warp] : nullptr;
    const uint32_t wcap = wok ? (uint32_t)(cl.wreg_off[warp + 1] - cl.wreg_off[warp]) : 0u;
    uint32_t wpos = 0;
    // a lane owns the windows 2 lane, 2 lane + 1 of every chunk of 64: one entry of a pair table bounds both
    const int lane_word = (2 * lane - KD) >> 4;
    const int sft = 2 * ((2 * lane - KD) & 15);
    uint32_t li = warp;
    if (li < pv.nlist) {
        PackedSeq sq = pv.seqs[pv.seq_ids[li]];
        uint32_t n_next = li + nwarps < pv.nlist ? pv.seq_ids[li + nwarps] : 0u;
        const uint32_t* __restrict__ wl = pv.words + sq.word_off + lane_word;
        uint32_t t0 = wl[0], t1 = wl[1], t2 = wl[2];
        for (;;) {
            if (flags[0] != 0u) break;                       // another warp overflowed: the dense kernel takes over
            const uint32_t li_next = li + nwarps;
            const bool more = li_next < pv.nlist;
            PackedSeq sq_next = sq;
            uint32_t n_nn = 0u;
            if (more) { sq_next = pv.seqs[n_next]; if (li_next + nwarps < pv.nlist) n_nn = pv.seq_ids[li_next + nwarps]; }
            const int L = (int)sq.L, LW1 = L - W + 1, mid = (int)sq.mid;
            // bound * q/LW1 >= thr0  <=>  bound >= thr0 LW1 / q (thr0 already carries the rounding margin of the bound)
            const float thr = gp.thr0 * (float)LW1 / gp.q;
            const float thw = thr * cl.watch_scale;
            const int tl = min(max(L - 2 * W + 2, 0), LW1);
            int n0 = tl, n1 = tl;
            if (mid >= 0) { n0 = min(max(mid - W + 1, 0), tl); n1 = min(mid + K + 1, tl); }
            const uint32_t start = cpos, wstart = wpos;
            const int nch = (tl + 63) >> 6;
            uint32_t u0 = 0, u1 = 0, u2 = 0;
            // The hot loop only records, per lane, WHICH of its windows pass (bit c = window 2 lane + 64 c, bit 16 + c = the
            // window after it, for a block of up to 16 chunks): no vote, no range test, no store per chunk. The windows that
            // are not this kernel's (over the N, truncated tail, past the end) are cleared from the mask afterwards and the
            // survivors written in one go.
            for (int cb = 0; cb < nch && ok; cb += 16) {
                const int ce = min(nch, cb + 16);
                const bool last_block = ce == nch;
                const int c_pf = last_block ? max(ce - 4, cb) : ce;      // chunk before which the next sequence's first words are requested
                uint32_t mine = 0u, watched = 0u, bit = 1u;
                auto chunk = [&]() {
                    const uint32_t whi = __funnelshift_l(t1, t0, sft), wlo = __funnelshift_l(t2, t1, sft);
                    wl += 4;
                    t0 = wl[0]; t1 = wl[1]; t2 = wl[2];
                    float b0 = 1.0f, b1 = 1.0f;
#pragma unroll
                    for (int g = 0; g < G1; g++) {
                        const uint32_t e = __float_as_uint(lds_f32(group_offset<G1, FAST>(gc, g, whi, wlo), gc.ab[g]));
                        const float f0 = __uint_as_float(e << 16), f1 = __uint_as_float(e & 0xffff0000u);
                        b0 = g ? b0 * f0 : f0; b1 = g ? b1 * f1 : f1;
                    }
                    if (b0 >= thr) mine |= bit;
                    if (b1 >= thr) mine |= bit << 16;
                    if (b0 >= thw) watched |= bit;
                    if (b1 >= thw) watched |= bit << 16;
                    bit <<= 1;
                };
#pragma unroll 2
                for (int c = cb; c < c_pf; c++) chunk();
                if (last_block) { const uint32_t* __restrict__ wn = pv.words + sq_next.word_off + lane_word; u0 = wn[0]; u1 = wn[1]; u2 = wn[2]; }
#pragma unroll 2
                for (int c = c_pf; c < ce; c++) chunk();
                // this lane's windows of the block: p = pb + h + 64 c (h = 0, 1; c = 0..15); keep those with p < tl outside [n0, n1)
                const int pb = 2 * lane + 64 * cb;
                uint32_t keep = 0u;
#pragma unroll
                for (int h = 0; h < 2; h++) {
                    const int q0 = pb + h;
                    const int c_tl = tl > q0 ? min((tl - q0 + 63) >> 6, 16) : 0;             // c < c_tl  <=>  p < tl
                    uint32_t k16 = (1u << c_tl) - 1u;
                    if (n1 > n0) {
                        const int ca = n0 > q0 ? min((n0 - q0 + 63) >> 6, 16) : 0, cz = n1 > q0 ? min((n1 - q0 + 63) >> 6, 16) : 0;   // c in [ca, cz)  <=>  n0 <= p < n1
                        k16 &= ~(((1u << cz) - 1u) & ~((1u << ca) - 1u));
                    }
                    keep |= k16 << (16 * h);
                }
                mine &= keep;
                // exclusive prefix of the lanes' counts -> each lane writes its windows behind those of the lower lanes
                const uint32_t mycnt = __popc(mine);
                uint32_t incl = mycnt;
#pragma unroll
                for (int o = 1; o < 32; o <<= 1) { const uint32_t v = __shfl_up_sync(FULL, incl, o); if (lane >= o) incl += v; }
                const uint32_t total = __shfl_sync(FULL, incl, 31);
                if (cpos + total > ccap) { ok = false; break; }
                uint32_t at = cpos + incl - mycnt;
                while (mine) {
                    const int b = __ffs(mine) - 1;
                    mine &= mine - 1u;
                    creg[at++] = (uint32_t)(pb + 64 * (b & 15) + (b >> 4));
                }
                cpos += total;
                if (wok) {                                       // the same for the watch list; when it is full, only it is dropped
                    watched &= keep;
                    const uint32_t wcnt = __popc(watched);
                    uint32_t winc = wcnt;
#pragma unroll
                    for (int o = 1; o < 32; o <<= 1) { const uint32_t v = __shfl_up_sync(FULL, winc, o); if (lane >= o) winc += v; }
                    const uint32_t wtotal = __shfl_sync(FULL, winc, 31);
                    if (wpos + wtotal > wcap) wok = false;
                    else {
                        uint32_t wat = wpos + winc - wcnt;
                        while (watched) {
                            const int b = __ffs(watched) - 1;
                            watched &= watched - 1u;
                            wreg[wat++] = (uint32_t)(pb + 64 * (b & 15) + (b >> 4));
                        }
                        wpos += wtotal;
                    }
                }
            }
            if (nch == 0) { const uint32_t* __restrict__ wn = pv.words + sq_next.word_off + lane_word; u0 = wn[0]; u1 = wn[1]; u2 = wn[2]; }
            if (lane == 0) cl.seq[li] = make_uint2(start, cpos - start);
            if (wok && lane == 0) cl.wseq[li] = make_uint2(wstart, wpos - wstart);
            if (!ok || !more) break;
            li = li_next; sq = sq_next; n_next = n_nn;
            wl = pv.words + sq.word_off + lane_word;
            t0 = u0; t1 = u1; t2 = u2;
        }
    }
    if (!ok && lane == 0) { flags[5] = 1u; __threadfence(); flags[0] = 1u; }
    if (lane == 0 && cpos) atomicAdd(reinterpret_cast<unsigned long long*>(cl.flags + 2), (unsigned long long)cpos);
    if (build_list && lane == 0) {
        if (!wok || !ok) cl.reuse[BR_VALID] = 0u;     // an incomplete list (full watch region, or a warp that stopped early) is not used
        if (!wok) cl.reuse[BR_WFULL] = 1u;
        else if (wpos) atomicAdd(&cl.reuse[BR_WCOUNT], wpos);
    }
}

// ---- pruned E-step, part 1 with reuse: bounds of the watched windows only -------------------------------------------
// Runs instead of k_ebound when k_estep_begin found that no window outside the watch list can reach thr with the current tables.
// Same warp -> sequence walk, same thr, same products (window p's bound is the low half of the entry at p's window word: the
// value k_ebound reads from the low half at p or the high half at p-1), so the candidates come out as the full pass would list
// them, in the same order: the watch list holds them in that order. A region overflows exactly when the full pass's would (its
// warp has more candidates than slots), and then raises the same dense fall-back.
template <int G1, bool FAST>
__global__ void __launch_bounds__(BAMM_E_THREADS, 1)
k_ebound_watch(PackedView pv, const __grid_constant__ GroupPlan gp, const float* __restrict__ tab_g, CandList cl) {
    extern __shared__ __align__(16) float tab[];
    __shared__ unsigned long long stage_bar;
    volatile uint32_t* flags = cl.flags;
    if (flags[0] != 0u || cl.reuse == nullptr || cl.reuse[BR_MODE] != 1u) return;
    bulk_stage_begin(tab, tab_g, gp.table_bytes, &stage_bar);
    bulk_stage_wait(&stage_bar);
    const int lane = threadIdx.x & 31;
    const uint32_t warp = blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
    const uint32_t nwarps = gridDim.x * (blockDim.x >> 5);
    const int W = gp.W, KD = gp.kd;
    const uint32_t tab_s = (uint32_t)__cvta_generic_to_shared(tab);
    GroupConsts<G1> gc; load_consts<G1>(gc, gp, tab_s);
    uint32_t lt_mask;
    asm("mov.u32 %0, %%lanemask_lt;" : "=r"(lt_mask));
    uint32_t* __restrict__ creg = cl.ent + cl.reg_off[warp];
    const uint32_t ccap = (uint32_t)(cl.reg_off[warp + 1] - cl.reg_off[warp]);
    const uint32_t* __restrict__ wreg = cl.went + cl.wreg_off[warp];
    uint32_t cpos = 0;
    bool ok = true;
    uint32_t li = warp;
    if (li < pv.nlist) {
        PackedSeq sq = pv.seqs[pv.seq_ids[li]];
        uint2 ws = cl.wseq[li];
        uint32_t n_next = li + nwarps < pv.nlist ? pv.seq_ids[li + nwarps] : 0u;
        for (;;) {
            if (flags[0] != 0u) break;
            const uint32_t li_next = li + nwarps;
            const bool more = li_next < pv.nlist;
            PackedSeq sq_next = sq;
            uint2 ws_next = ws;
            uint32_t n_nn = 0u;
            if (more) { sq_next = pv.seqs[n_next]; ws_next = cl.wseq[li_next]; if (li_next + nwarps < pv.nlist) n_nn = pv.seq_ids[li_next + nwarps]; }
            const int LW1 = (int)sq.L - W + 1;
            const float thr = gp.thr0 * (float)LW1 / gp.q;
            const uint32_t* __restrict__ wseq = pv.words + sq.word_off;
            const uint32_t* __restrict__ wl = wreg + ws.x;
            const uint32_t start = cpos;
            uint32_t p_next = lane < ws.y ? wl[lane] : 0u;
            for (uint32_t e0 = 0; e0 < ws.y; e0 += 32) {
                const bool on = e0 + lane < ws.y;
                const int p = (int)p_next;
                if (e0 + 32 + lane < ws.y) p_next = wl[e0 + 32 + lane];      // next batch
                uint32_t whi, wlo;
                window_bits(wseq, p - KD, whi, wlo);
                float b0 = 1.0f;
#pragma unroll
                for (int g = 0; g < G1; g++) {
                    const float f0 = __uint_as_float(__float_as_uint(lds_f32(group_offset<G1, FAST>(gc, g, whi, wlo), gc.ab[g])) << 16);
                    b0 = g ? b0 * f0 : f0;
                }
                const bool pass = on && b0 >= thr;
                const uint32_t m = __ballot_sync(FULL, pass);
                const uint32_t cnt = __popc(m);
                if (cpos + cnt > ccap) { ok = false; break; }
                if (pass) creg[cpos + __popc(m & lt_mask)] = (uint32_t)p;
                cpos += cnt;
            }
            if (!ok) break;
            if (lane == 0) cl.seq[li] = make_uint2(start, cpos - start);
            if (!more) break;
            li = li_next; sq = sq_next; ws = ws_next; n_next = n_nn;
        }
    }
    if (!ok && lane == 0) { flags[5] = 1u; __threadfence(); flags[0] = 1u; }
    if (lane == 0 && cpos) atomicAdd(reinterpret_cast<unsigned long long*>(cl.flags + 2), (unsigned long long)cpos);
}

// ---- pruned E-step, part 0: the windows over the N and the truncated tail ----------------------------------------------
// Every sequence has W+K windows over the structural N and W-1 truncated windows (EM.cpp:167); they need the masked evaluation
// and most truncated ones are active, so they are evaluated for all sequences — with the sequences ACROSS the lanes: lane l
// owns sequence 32 i + l and all lanes walk the same window index t. For window t the set of whole groups and of single
// columns is the same in every lane (it only depends on W, K and t), so there is no mask arithmetic and no divergence; the
// window word advances by one base per step in registers. The partial normaliser of every sequence goes to `seqacc`
// (k_eexact starts from it), the windows that reach the threshold to the back of the warp's region of the active list.
// Multiplication order = masked_prod's: whole groups ascending, then the remaining columns ascending.
// Sequences whose ranges are clipped (shorter than 2W-2, N too close to an end) make their warp take the generic route.
// per window index: bit g of good = group g whole; the other columns come from the plain table, in ascending order: the
// unpatched ones below the N's k-mers (lo), the K+1 patched ones, the unpatched ones above (hi)
struct MaskedStep { uint32_t good, lo, hi, pad; };
template <int G, bool FAST, bool LEAN /* one pass with the plain table in shared memory: no partial products, no global table */>
__global__ void __launch_bounds__(BAMM_E_THREADS, 1)
k_emasked(PackedView pv, const __grid_constant__ GroupPlan gp, const float* __restrict__ tab_g, const float* __restrict__ s_g,
          uint32_t plain_words, CandList cl, ulonglong2* __restrict__ seqacc,
          float* __restrict__ partial /* column passes: [nlist][2W+K-1] partial products, else nullptr */, ActiveList al) {
    extern __shared__ __align__(16) float tab[];
    __shared__ unsigned long long stage_bar;
    __shared__ __align__(16) MaskedStep steps[2][48];   // [0]: truncated windows t = p - tl, [1]: windows over the N, t = p - (mid-W+1)
    if (cl.flags[0] != 0u) return;
    bulk_stage_begin(tab, tab_g, gp.table_bytes, &stage_bar);
    for (uint32_t i = threadIdx.x; i < plain_words; i += blockDim.x) tab[(gp.table_bytes >> 2) + i + i / gp.Yn] = s_g[i];   // rows padded by one float
    const int W = gp.W, K = gp.K, KD = gp.kd;
    const int nt_tail = W - 1, nt_n = W + K;
    if (threadIdx.x < 96) {
        const int which = threadIdx.x >= 48, t = threadIdx.x - 48 * which;
        uint32_t valid = 0xffffffffu >> (32 - W), ncols = 0u;
        if (!which) { const int jmax = W - 2 - t; valid = jmax >= 0 ? ((2u << jmax) - 1u) : 0u; }
        else { const int jn = W - 1 - t, ja = max(jn, 0), jb = min(jn + K, W - 1); if (jb >= ja) ncols = ((2u << jb) - 1u) & ~((1u << ja) - 1u); }
        const uint32_t bad = ~valid | ncols;
        uint32_t good = 0u, cols = valid & gp.passmask;             // only the columns of this pass
        for (int g = 0; g < G; g++) if ((gp.colmask[g] & bad) == 0u) { good |= 1u << g; cols &= ~gp.colmask[g]; }
        cols &= ~ncols;                           // the patched columns have their own (unrolled) loop
        const int jn = W - 1 - t;
        const uint32_t below = which && jn > 0 ? ((1u << min(jn, 31)) - 1u) : (which ? 0u : 0xffffffffu);
        steps[which][t].good = good; steps[which][t].lo = cols & below; steps[which][t].hi = cols & ~below; steps[which][t].pad = 0u;
    }
    bulk_stage_wait(&stage_bar);
    __syncthreads();
    const int lane = threadIdx.x & 31;
    const uint32_t warp = blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
    const uint32_t nwarps = gridDim.x * (blockDim.x >> 5);
    const uint32_t tab_s = (uint32_t)__cvta_generic_to_shared(tab);
    const float thr0 = gp.thr0;
    GroupConsts<G> gc; load_consts<G>(gc, gp, tab_s);
    const uint32_t plain_s = tab_s + gp.table_bytes, maskK = gp.Yn - 1u, ystride = gp.Yn + 1u;
    const bool first = LEAN || gp.pass_first != 0, last = LEAN || gp.pass_last != 0;    // column passes: partial products travel through `partial`
    const uint32_t plain_on = LEAN ? plain_s : (plain_words ? plain_s : 0u);
    MaskedTabs mt; mt.s_g = s_g; mt.plain_s = plain_on;
    mt.Yn = gp.Yn; mt.maskK = maskK; mt.passmask = gp.passmask; mt.W = W; mt.K = K; mt.KD = KD;
    const int npart = 2 * W + K - 1;
    Emitter em; em.init(al, warp, last);
    // a warp takes the sequences k_eexact gives it (li = warp mod nwarps), 32 at a time: the two kernels share the warp's region
    for (uint64_t k0 = 0; warp + nwarps * k0 < pv.nlist; k0 += 32) {
        const uint64_t li64 = warp + (uint64_t)nwarps * (k0 + lane);
        const bool have = li64 < pv.nlist;
        const uint32_t li = have ? (uint32_t)li64 : 0u;
        const uint32_t n = have ? pv.seq_ids[li] : 0u;
        PackedSeq sq; sq.word_off = 2; sq.L = (uint32_t)(2 * W + K + 2); sq.mid = 0xffffffffu;
        if (have) sq = pv.seqs[n];
        const int L = (int)sq.L, LW1 = L - W + 1, mid = (int)sq.mid;
        const uint32_t* __restrict__ wseq = pv.words + sq.word_off;
        const uint32_t woff = (uint32_t)sq.word_off;
        const uint16_t* __restrict__ yp = pv.ypatch + (uint64_t)n * (K + 1);
        const float pos = gp.q / (float)LW1;
        const int tl = min(max(L - 2 * W + 2, 0), LW1);
        int n0 = tl, n1 = tl;
        if (mid >= 0) { n0 = min(max(mid - W + 1, 0), tl); n1 = min(mid + K + 1, tl); }
        NormAcc acc; acc.clear();
        const bool regular = !have || (L >= 2 * W - 2 && (mid < 0 || (mid >= W - 1 && mid + K + 1 <= tl)));
        if (__all_sync(FULL, regular)) {
            // the K+1 patched k-mers of this lane's sequence, two per register (a load per use would touch 32 lines)
            uint32_t ypk[6] = {0u, 0u, 0u, 0u, 0u, 0u};
            if (have && mid >= 0) {
#pragma unroll
                for (int d = 0; d < 11; d++) if (d <= K) ypk[d >> 1] |= (uint32_t)yp[d] << (16 * (d & 1));
            }
#pragma unroll 1
            for (int part = 0; part < 2; part++) {
                // part 0: p = tl + t, columns 0 .. W-2-t; part 1: p = mid-W+1 + t, N under column W-1-t
                const int nt = part ? nt_n : nt_tail;
                const bool mine = have && (part == 0 || mid >= 0);
                const int p_first = part ? n0 : tl;
                // window word of p_first (bases from p_first - KD) and the 16 bases behind it, advanced one base per step
                int b0 = (mine ? p_first : 0) - KD;
                uint32_t whi, wlo;
                window_bits(wseq, b0, whi, wlo);
                uint32_t nxt = wseq[(b0 >> 4) + 2] << (2 * (b0 & 15));       // bases b0+32 .. : 16 - (b0 & 15) of them left
                int nleft = 16 - (b0 & 15);
                int nw = (b0 >> 4) + 3;                                       // next stream word
#pragma unroll 1
                for (int t = 0; t < nt; t++) {
                    const MaskedStep st = steps[part][t];
                    const unsigned long long w = ((unsigned long long)whi << 32) | wlo;
                    float* const pp = !LEAN && partial ? partial + (size_t)li * npart + (part ? nt_tail : 0) + t : nullptr;
                    float prod = 1.0f;
                    if (!LEAN && !first && mine) prod = *pp;
#pragma unroll
                    for (int g = 0; g < G; g++)
                        if ((st.good >> g) & 1u) prod *= lds_f32(group_offset<G, FAST>(gc, g, whi, wlo), gc.ab[g]);
                    auto plain_at = [&](int j, uint32_t y) {                 // s[j][y]: shared-memory copy, or the global table
                        return (LEAN || plain_on) ? lds_f32(((uint32_t)j * ystride + y) << 2, plain_s) : __ldg(&s_g[(uint32_t)j * gp.Yn + y]);
                    };
                    auto single = [&](int j) {                               // column j with the k-mer of the stream
                        prod *= plain_at(j, field(w, 62 - 2 * KD - 2 * j, maskK));
                    };
                    for (uint32_t c = st.lo; c; c &= c - 1u) single(__ffs(c) - 1);
                    if (part) {
                        const int jn = W - 1 - t;                             // column of the N: patched k-mer d sits in column jn + d
#pragma unroll
                        for (int d = 0; d < 11; d++) {
                            const int j = jn + d;
                            if (d <= K && j >= 0 && j < W && (LEAN || ((gp.passmask >> j) & 1u))) {          // warp-uniform
                                const uint32_t y = (ypk[d >> 1] >> (16 * (d & 1))) & 0xffffu;
                                prod *= plain_at(j, y);
                            }
                        }
                    }
                    for (uint32_t c = st.hi; c; c &= c - 1u) single(__ffs(c) - 1);
                    if (!LEAN && !last) { if (mine) *pp = prod; }
                    else {
                        const float val = mine ? prod * pos : 0.0f;
                        acc.add(val);
                        em.template put<true>(al, val >= thr0, woff, pcode_of(p_first + t, part ? W - 1 : W - 2 - t, part != 0), val, li);
                    }
                    // next base
                    whi = __funnelshift_l(wlo, whi, 2); wlo = __funnelshift_l(nxt, wlo, 2); nxt <<= 2;
                    if (--nleft == 0) { nxt = wseq[nw++]; nleft = 16; }
                }
            }
        } else {
            // generic route: every lane walks its own list of masked windows, masked_prod per window
            const int nn = n1 - n0, nm = have ? nn + (LW1 - tl) : 0;
            int nm_max = nm;
#pragma unroll
            for (int o = 16; o > 0; o >>= 1) nm_max = max(nm_max, __shfl_xor_sync(FULL, nm_max, o));
#pragma unroll 1
            for (int idx = 0; idx < nm_max; idx++) {
                const bool on = idx < nm;
                const int p = on ? (idx < nn ? n0 + idx : tl + (idx - nn)) : 0;
                uint32_t whi, wlo;
                window_bits(wseq, p - KD, whi, wlo);
                const int jmax = on ? min(W - 1, L - W - p) : -1;
                float* const pp = partial && idx < npart ? partial + (size_t)li * npart + idx : nullptr;
                float prod = 1.0f;
                if (!first && on && pp) prod = *pp;
                prod = masked_prod<G, FAST>(gc, gp, mt, whi, wlo, p, jmax, mid, yp, prod);
                if (!last) { if (on && pp) *pp = prod; }
                else {
                    const float val = on ? prod * pos : 0.0f;
                    acc.add(val);
                    em.template put<true>(al, val >= thr0, woff, pcode_of(p, jmax, mid >= 0 && p <= mid + K && p + W - 1 >= mid), val, li);
                }
            }
        }
        if (have && last) seqacc[li] = make_ulonglong2(acc.a, acc.b);
    }
    if (last) al.cnt_back[warp] = em.bpos;
}

// ---- pruned E-step, part 2: exact evaluation of the listed windows -------------------------------------------------
// gp is the exact plan of the dense kernel. Per sequence: the candidates in batches of 32, then the normaliser terms of the
// windows over the N and of the truncated tail (k_emasked), then the normaliser. The stream words of the sequence (up to
// STAGE_SEQ_WORDS, i.e. about 1500 bases) are staged in a per-warp slice of shared memory with coalesced loads, so a window word is
// three shared-memory reads instead of a gather; longer sequences gather from global memory. The records of the next
// sequence are requested one sequence ahead.
constexpr int STAGE_SEQ_WORDS = 96, STAGE_WORDS = STAGE_SEQ_WORDS;
template <int G, bool FAST, bool MULTI /* column passes: partial products between them */>
__global__ void __launch_bounds__(BAMM_E_THREADS, 1)
k_eexact(PackedView pv, const __grid_constant__ GroupPlan gp, const float* __restrict__ tab_g, const float* __restrict__ s_g,
         uint32_t plain_words, uint32_t stage /* 0: no staging buffer */, CandList cl,
         const ulonglong2* __restrict__ seqacc, float* __restrict__ partial /* column passes: one float per candidate slot, else nullptr */,
         unsigned long long* __restrict__ scal, ActiveList al) {
    extern __shared__ __align__(16) float tab[];
    __shared__ unsigned long long stage_bar;
    if (cl.flags[0] != 0u) return;
    bulk_stage_begin(tab, tab_g, gp.table_bytes, &stage_bar);
    for (uint32_t i = threadIdx.x; i < plain_words; i += blockDim.x) tab[(gp.table_bytes >> 2) + i + i / gp.Yn] = s_g[i];   // rows padded by one float
    bulk_stage_wait(&stage_bar);
    __syncthreads();
    const int lane = threadIdx.x & 31;
    const uint32_t warp = blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
    const uint32_t nwarps = gridDim.x * (blockDim.x >> 5);
    const int W = gp.W, KD = gp.kd;
    const uint32_t tab_s = (uint32_t)__cvta_generic_to_shared(tab);
    long long llh_fx = 0, rsum_fx = 0;
    const float one_minus_q = 1.0f - gp.q;
    const float thr0 = gp.thr0;
    GroupConsts<G> gc; load_consts<G>(gc, gp, tab_s);
    const bool first = !MULTI || gp.pass_first != 0, last = !MULTI || gp.pass_last != 0;   // column passes (tables of all columns beyond shared memory)
    Emitter em; em.init(al, warp, last);
    em.bpos = al.cnt_back[warp];                                        // the back of the region is k_emasked's
    float* const preg = MULTI && partial ? partial + cl.reg_off[warp] : nullptr;
    uint32_t* const stg = reinterpret_cast<uint32_t*>(tab + (gp.table_bytes >> 2) + plain_smem_words(plain_words, gp.Yn)) + (threadIdx.x >> 5) * STAGE_WORDS;
    const uint32_t* __restrict__ creg = cl.ent + cl.reg_off[warp];
    uint32_t li = warp;
    if (li < pv.nlist) {
        uint32_t n = pv.seq_ids[li];
        PackedSeq sq = pv.seqs[n];
        uint2 sc = cl.seq[li];
        uint32_t n_next = li + nwarps < pv.nlist ? pv.seq_ids[li + nwarps] : 0u;
        for (;;) {
            const uint32_t li_next = li + nwarps;
            const bool more = li_next < pv.nlist;
            PackedSeq sq_next = sq;
            uint2 sc_next = sc;
            uint32_t n_nn = 0u;
            if (more) { sq_next = pv.seqs[n_next]; sc_next = cl.seq[li_next]; if (li_next + nwarps < pv.nlist) n_nn = pv.seq_ids[li_next + nwarps]; }
            const int L = (int)sq.L, LW1 = L - W + 1;
            const uint32_t* __restrict__ wseq = pv.words + sq.word_off;
            const uint32_t woff = (uint32_t)sq.word_off;
            const uint32_t* __restrict__ cand = creg + sc.x;
            uint32_t c_first = lane < sc.y ? cand[lane] : 0u;       // first batch of candidates, in flight with the staging loads
            const uint32_t* wsrc = wseq;                            // generic pointer: shared staging or global
            const int last_word = ((L - W - KD) >> 4) + 4;          // staging index of the last word any window of this sequence reads
            if (stage && last_word < STAGE_SEQ_WORDS) {
                __syncwarp();                                       // the previous sequence's readers are done
                const uint32_t* __restrict__ g = wseq - 2;          // two pad words in front: windows that start before the sequence
                for (int k = lane; k <= last_word; k += 32) stg[k] = g[k];
                __syncwarp();
                wsrc = stg + 2;
            }
            const float pos = gp.q / (float)LW1;
            NormAcc acc; acc.clear();
            // Up to two batches are held back until the normaliser is known: a window whose posterior rounds to zero in the
            // M-step's fixed point (val / norm < 2^-41; about a quarter of those above the a-priori threshold, because norm
            // is large wherever the sequence holds a site) is then not listed at all. Longer lists are written as they come.
            const bool defer = sc.y <= 64u;
            float v0 = 0.0f, v1 = 0.0f;
            int q0 = 0, q1 = 0;
#pragma unroll 1
            for (uint32_t e0 = 0; e0 < sc.y; e0 += 32) {
                const bool on = e0 + lane < sc.y;
                const int p = (int)c_first;
                if (e0 + 32 + lane < sc.y) c_first = cand[e0 + 32 + lane];      // next batch
                uint32_t whi, wlo;
                window_bits(wsrc, p - KD, whi, wlo);
                float* const pp = MULTI && preg ? preg + sc.x + e0 + lane : nullptr;
                float prod = 1.0f;
                if (MULTI && !first && on) prod = *pp;
                prod = groups_prod<G, FAST>(gc, whi, wlo, prod);
                if (MULTI && !last) { if (on) *pp = prod; continue; }
                const float val = on ? prod * pos : 0.0f;
                acc.add(val);
                if (!defer) em.template put<false>(al, val >= thr0, woff, pcode_of(p, W - 1, false), val, li);
                else if (e0 == 0u) { v0 = val; q0 = p; }
                else { v1 = val; q1 = p; }
            }
            if (MULTI && !last) { if (!more) break; li = li_next; n = n_next; n_next = n_nn; sq = sq_next; sc = sc_next; continue; }
            if (lane == 0) { const ulonglong2 m = seqacc[li]; acc.a += m.x; acc.b += m.y; }      // the masked windows (k_emasked)
            const float norm = finish_sequence(acc, one_minus_q, lane, li, al.scale, llh_fx, rsum_fx);
            if (defer && sc.y) {
                const float thr = fmaxf(thr0, FX_HALF_UNIT * 0.999f * norm);
                em.template put<false>(al, v0 >= thr, woff, pcode_of(q0, W - 1, false), v0, li);
                if (sc.y > 32u) em.template put<false>(al, v1 >= thr, woff, pcode_of(q1, W - 1, false), v1, li);
            }
            if (!more) break;
            li = li_next; n = n_next; n_next = n_nn; sq = sq_next; sc = sc_next;
        }
    }
    if (MULTI && !last) return;
    if (lane == 0) {
        if (llh_fx) atomicAdd(&scal[0], (unsigned long long)llh_fx);
        if (rsum_fx) atomicAdd(&scal[1], (unsigned long long)rsum_fx);
    }
    al.cnt[warp] = em.lpos;
}

}  // namespace bamm
