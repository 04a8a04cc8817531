// packed.cuh — the fast path for the 4-letter alphabet: sequences as 2-bit packed base streams.
//
// Layout (DESIGN.md §3.2). A "regular" sequence (codes 1..4 everywhere, except optionally the structural N in the
// middle of a both-strand sequence, Sequence.cpp:10-14) is stored as 32-bit words of 16 bases, FIRST base in the
// most significant bits, preceded by two zero pad words (32 bases) and followed by six. The order-K k-mer index of the
// reference, y(i) = sum_t c(i-t) 4^t (Sequence.cpp:35-41), is then literally a bit field of the stream: for a
// window start p the 64-bit word  w = bases p-K .. p-K+31  gives  y(p+j) = (w >> (62-2K-2j)) & (4^(K+1)-1), and the
// zero pad supplies the implicit leading 'A's of k-mers that start before the sequence does. No index array is read.
//
// E-step: column groups. Consecutive motif columns are folded into one lookup over the bases they depend on,
//   tab[g][z] = prod_{j in group g} s[j][ y_j(z) ],  so a window costs G shared-memory lookups instead of W. Windows that
// cannot use whole groups (the last W-1 truncated windows, EM.cpp:167, and windows over the N whose k-mers hold rand()
// draws, Sequence.cpp:38) take a masked path that mixes whole groups with single columns of the plain table. When the
// tables of all W columns do not fit shared memory the kernel runs once per column range ("column passes").
//
// M-step: sparse or dense. r is converted to 2^40 fixed point; every window whose r rounds to 0 contributes exactly
// nothing. The E-step lists the surviving (window, value) pairs per warp; the list kernel scatters them with full
// lanes. When the posteriors are dense (list overflow) a scan kernel walks r instead. Both use unguarded 32-bit shared
// atomics on CTA-private low / high tables, optionally split by motif column over the CTAs.
#pragma once
#include <type_traits>
#include "kernels.cuh"

namespace bamm {

// ---- classification + packing (device side of bamm_seqset_create) --------------------------------------------------
// kind: 0 irregular, 1 regular without N, 2 regular with exactly one 0 code at (L-1)/2, L odd
__global__ void k_classify(const uint8_t* __restrict__ codes, const uint64_t* __restrict__ off, uint64_t nseq,
                           uint8_t* __restrict__ kind) {
    const int lane = threadIdx.x & 31;
    const uint64_t warp = (uint64_t)blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
    const uint64_t nwarps = (uint64_t)gridDim.x * (blockDim.x >> 5);
    for (uint64_t n = warp; n < nseq; n += nwarps) {
        const uint64_t base = off[n], L = off[n + 1] - base;
        const uint64_t mid = (L & 1) ? (L - 1) / 2 : ~0ull;
        int bad = 0, zeros_at_mid = 0;
        auto check = [&](uint64_t i, uint32_t c) {
            if (c == 0) { if (i == mid) zeros_at_mid = 1; else bad = 1; }
            else if (c > 4) bad = 1;
        };
        // unaligned head and tail byte by byte, the aligned interior four codes per load: a word is suspicious when one of
        // its bytes is 0 or above 4 (bit tricks), only then its bytes are looked at one by one
        const uint64_t a0 = (base + 3) & ~3ull, a1 = (base + L) & ~3ull;     // aligned interior [a0, a1) in global offsets
        if (a0 >= a1) {
            for (uint64_t i = lane; i < L; i += 32) check(i, codes[base + i]);
        } else {
            for (uint64_t g = base + lane; g < a0; g += 32) check(g - base, codes[g]);
            for (uint64_t g = a1 + lane; g < base + L; g += 32) check(g - base, codes[g]);
            const uint32_t* __restrict__ w4 = reinterpret_cast<const uint32_t*>(codes + a0);
            const uint64_t nw = (a1 - a0) >> 2;
            for (uint64_t k = lane; k < nw; k += 32) {
                const uint32_t w = w4[k];
                const uint32_t zero = (w - 0x01010101u) & ~w & 0x80808080u;
                const uint32_t big = (((w & 0x7f7f7f7fu) + 0x7b7b7b7bu) | w) & 0x80808080u;
                if (zero | big) {
                    const uint64_t i = a0 - base + (k << 2);
                    check(i, w & 0xffu); check(i + 1, (w >> 8) & 0xffu); check(i + 2, (w >> 16) & 0xffu); check(i + 3, w >> 24);
                }
            }
        }
        bad = __any_sync(FULL, bad);
        zeros_at_mid = __any_sync(FULL, zeros_at_mid);
        if (lane == 0) kind[n] = (bad || L == 0 || L >= PACKED_MAX_L) ? 0 : (zeros_at_mid ? 2 : 1);
    }
}


// patch list contract of bamm_seqset_create: positions inside the set (bit 0 of *bad otherwise) and strictly increasing (bit 1)
__global__ void k_validate_patches(const uint64_t* __restrict__ ppos, uint64_t np, uint64_t npos, uint32_t* __restrict__ bad) {
    const uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= np) return;
    const uint64_t p = ppos[i];
    if (p >= npos) atomicOr(bad, 1u);
    if (i && p <= ppos[i - 1]) atomicOr(bad, 2u);
}

// every patch must sit at mid..mid+10 of a kind-2 sequence; anything else makes its sequence irregular.
// cover[n] counts the patches that landed in the structural region.
__global__ void k_check_patches(const uint64_t* __restrict__ ppos, uint64_t np, const uint64_t* __restrict__ off,
                                uint64_t nseq, uint8_t* __restrict__ kind, uint32_t* __restrict__ cover) {
    const uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= np) return;
    const uint64_t pos = ppos[i];
    uint64_t lo = 0, hi = nseq;                      // last n with off[n] <= pos
    while (hi - lo > 1) { const uint64_t m = (lo + hi) >> 1; if (off[m] <= pos) lo = m; else hi = m; }
    const uint64_t n = lo, L = off[n + 1] - off[n], local = pos - off[n];
    const uint64_t mid = (L - 1) / 2;
    if (kind[n] == 2 && local >= mid && local <= mid + 10) atomicAdd(&cover[n], 1u);
    else kind[n] = 0;                                // benign race: every writer stores 0
}

__global__ void k_finish_kinds(const uint64_t* __restrict__ off, uint64_t nseq, const uint32_t* __restrict__ cover,
                               uint8_t* __restrict__ kind) {
    const uint64_t n = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (n >= nseq) return;
    if (kind[n] == 2) {
        const uint64_t L = off[n + 1] - off[n], mid = (L - 1) / 2;
        const uint64_t need = (L - mid < 11) ? L - mid : 11;      // positions mid..min(mid+10, L-1)
        if (cover[n] != need) kind[n] = 0;                         // the caller did not patch the N: generic path
    }
}

// words of every regular sequence in the packed stream: data words + 2 pad words in front + 6 behind (0 for irregular ones)
__global__ void k_word_counts(const uint64_t* __restrict__ off, uint64_t nseq, const uint8_t* __restrict__ kind, unsigned long long* __restrict__ wc) {
    const uint64_t n = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (n >= nseq) return;
    const uint64_t L = off[n + 1] - off[n];
    wc[n] = kind[n] ? (L + 15) / 16 + 8 : 0ull;
}
// PackedSeq records from the exclusive scan of the word counts
__global__ void k_fill_pseq(const uint64_t* __restrict__ off, uint64_t nseq, const uint8_t* __restrict__ kind,
                            const unsigned long long* __restrict__ wscan, PackedSeq* __restrict__ seqs) {
    const uint64_t n = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (n >= nseq) return;
    PackedSeq q; q.word_off = 0; q.L = 0; q.mid = 0xffffffffu;
    if (kind[n]) {
        const uint64_t L = off[n + 1] - off[n];
        q.word_off = wscan[n] + 2; q.L = (uint32_t)L; q.mid = kind[n] == 2 ? (uint32_t)((L - 1) / 2) : 0xffffffffu;
    }
    seqs[n] = q;
}

// one lane per output word (16 bases)
__global__ void k_pack(const uint8_t* __restrict__ codes, const uint64_t* __restrict__ off, uint64_t nseq,
                       const uint8_t* __restrict__ kind, const PackedSeq* __restrict__ seqs,
                       uint32_t* __restrict__ words) {
    const int lane = threadIdx.x & 31;
    const uint64_t warp = (uint64_t)blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
    const uint64_t nwarps = (uint64_t)gridDim.x * (blockDim.x >> 5);
    for (uint64_t n = warp; n < nseq; n += nwarps) {
        if (kind[n] == 0) continue;
        const uint64_t base = off[n], L = off[n + 1] - base;
        const uint64_t nw = (L + 15) / 16;
        uint32_t* dst = words + seqs[n].word_off;
        if (lane < 2) dst[-1 - lane] = 0u;
        if (lane < 6) dst[nw + lane] = 0u;
        for (uint64_t wi = lane; wi < nw; wi += 32) {
            uint32_t w = 0;
            for (int b = 0; b < 16; b++) {
                const uint64_t i = wi * 16 + b;
                const uint32_t c = (i < L) ? codes[base + i] : 0u;
                w = (w << 2) | (c ? c - 1 : 0u);
            }
            dst[wi] = w;
        }
    }
}

__global__ void k_make_ypatch(const uint64_t* __restrict__ ppos, const uint64_t* __restrict__ pkmer, uint64_t np,
                              const uint64_t* __restrict__ off, uint64_t nseq, const uint8_t* __restrict__ kind,
                              int K, uint64_t Yn, uint16_t* __restrict__ ypatch) {
    const uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= np) return;
    const uint64_t pos = ppos[i];
    uint64_t lo = 0, hi = nseq;
    while (hi - lo > 1) { const uint64_t m = (lo + hi) >> 1; if (off[m] <= pos) lo = m; else hi = m; }
    const uint64_t n = lo;
    if (kind[n] != 2) return;
    const uint64_t L = off[n + 1] - off[n], d = pos - off[n] - (L - 1) / 2;
    if (d <= (uint64_t)K) ypatch[n * (uint64_t)(K + 1) + d] = (uint16_t)(pkmer[i] % Yn);
}

// tab[g][z] = prod_{j in group g} s[j][ y_j(z) ], product in ascending j from 1.0f; z holds bases p+lo .. p+hi
// (newest base in the low digits), y_j = the part of the (K+1)-mer ending at p+j that lies inside the group's bases
// (digits outside do not influence s[j][.], see above).
template <bool LOGSUM>
__device__ __forceinline__ void group_tables_part(const float* __restrict__ s, const GroupPlan& gp, float* __restrict__ tab, uint32_t nblocks) {
    const uint32_t total = gp.table_bytes >> 2;
    const uint32_t maskK = gp.Yn - 1;
    for (uint32_t i = blockIdx.x * blockDim.x + threadIdx.x; i < total; i += nblocks * blockDim.x) {
        int g = 0;
        while (g + 1 < gp.G && i >= (gp.base[g + 1] >> 2)) g++;
        const uint32_t z = i - (gp.base[g] >> 2);
        const int hi = gp.col0[g] + gp.ncol[g] - 1;
        float p = LOGSUM ? 0.0f : 1.0f;
        for (int t = 0; t < gp.ncol[g]; t++) {
            const int j = gp.col0[g] + t;
            const int avail = j - gp.lo[g] + 1;                          // bases of the group up to column j
            uint32_t y = (z >> (2 * (hi - j))) & maskK;
            if (avail < gp.K + 1) y &= (1u << (2 * avail)) - 1u;
            if (LOGSUM) p += s[(uint32_t)j * gp.Yn + y]; else p *= s[(uint32_t)j * gp.Yn + y];
        }
        tab[i] = p;
    }
}
template <bool LOGSUM>
__global__ void k_make_group_tables(const float* __restrict__ s, GroupPlan gp, float* __restrict__ tab) {
    group_tables_part<LOGSUM>(s, gp, tab, gridDim.x);
}

// ---- bound tables of the pruned E-step (estep.cuh, k_ebound) ---------------------------------------------------------
// A bound group covers the bases lo..hi relative to the window start and the columns col0..hi. A column whose context reaches
// left of lo only sees avail = j-lo+1 < K+1 of its bases; its factor is then the maximum of s[j][.] over the missing (older)
// bases, U_avail[j][y mod 4^avail]. The levels are built top-down: level a = maximum over the 4 values of the next older base
// of level a+1 (level K+1 is s itself), one CTA, a barrier per level.
struct BoundLevels { uint32_t off[12]; };     // off[a]: first float of level a (a = 1..K), [j][4^a]
constexpr uint32_t LEV_CAP = 11264;           // floats of the levels kept in shared memory as well (44 KB: all of them up to order 4 at W = 32)
__device__ __forceinline__ void bound_levels_cta(const float* __restrict__ s /* [j][Yn] */, int W, int K, BoundLevels bl, float* __restrict__ U) {
    __shared__ float lev[LEV_CAP];            // the small levels: the next level reads them here instead of waiting for global memory
    for (int a = K; a >= 1; a--) {
        const uint32_t Ya = 1u << (2 * a), Ysrc = Ya << 2;
        const bool src_sh = a < K && bl.off[a + 1] + (uint32_t)W * Ysrc <= LEV_CAP;
        const bool dst_sh = bl.off[a] + (uint32_t)W * Ya <= LEV_CAP;
        const float* src = (a == K) ? s : src_sh ? lev + bl.off[a + 1] : U + bl.off[a + 1];
        float* __restrict__ dst = U + bl.off[a];
        for (uint32_t i = threadIdx.x; i < (uint32_t)W * Ya; i += blockDim.x) {
            const uint32_t j = i >> (2 * a), y = i & (Ya - 1u);
            const float* row = src + (size_t)j * Ysrc;
            const float v = fmaxf(fmaxf(row[y], row[Ya + y]), fmaxf(row[2u * Ya + y], row[3u * Ya + y]));
            dst[i] = v;
            if (dst_sh) lev[bl.off[a] + i] = v;
        }
        __syncthreads();
    }
}
// The tables an EM iteration rebuilds first, in one launch: the exact group tables of a pass on all CTAs but the last, which
// builds the bound levels meanwhile (both only read s).
__global__ void __launch_bounds__(1024)
k_em_tables(const float* __restrict__ s, GroupPlan gp, float* __restrict__ tab, BoundLevels bl, float* __restrict__ U) {
    if (blockIdx.x + 1 == gridDim.x) bound_levels_cta(s, gp.W, gp.K, bl, U);
    else group_tables_part<false>(s, gp, tab, gridDim.x - 1);
}
// f_g(z) = prod_{j in group g} U_avail(j)[j][...] over the group's T bases lo..hi: an upper bound of the product of the group's
// columns for EVERY context left of the group's bases. The table is indexed by T+1 bases (lo..hi+1) and an entry holds TWO
// bounds as bfloat16, rounded UP: low half = f_g of window p (bases lo..hi), high half = f_g of window p+1 (bases lo+1..hi+1),
// so one 32-bit lookup serves two neighbouring windows.
__device__ __forceinline__ uint32_t bf16_up(float x) {      // smallest bfloat16 >= x (x finite, >= 0)
    uint32_t b = __float_as_uint(x);
    if (b & 0xffffu) b = (b | 0xffffu) + 1u;
    return b >> 16;
}
// ref != nullptr (bound reuse): rho[g] = max over the group's bfloat16 values of new / ref, rounded up (+inf where ref is 0 and the new
// value is not; a zero new value bounds nothing and is skipped): one atomicMax of the float bits per warp and group.
__global__ void k_make_bound_tables(const float* __restrict__ s, const float* __restrict__ U, BoundLevels bl, GroupPlan gp, uint32_t* __restrict__ tab,
                                    const uint32_t* __restrict__ ref, uint32_t* __restrict__ rho) {
    const uint32_t total = gp.table_bytes >> 2;
    for (uint32_t i = blockIdx.x * blockDim.x + threadIdx.x; i < total; i += gridDim.x * blockDim.x) {
        int g = 0;
        while (g + 1 < gp.G && i >= (gp.base[g + 1] >> 2)) g++;
        const uint32_t z2 = i - (gp.base[g] >> 2);
        const int hi = gp.col0[g] + gp.ncol[g] - 1, T = hi - gp.lo[g] + 1;
        uint32_t packed = 0u;
        for (int h = 0; h < 2; h++) {
            const uint32_t z = h == 0 ? (z2 >> 2) : (z2 & ((1u << (2 * T)) - 1u));
            float p = 1.0f;
            for (int t = 0; t < gp.ncol[g]; t++) {
                const int j = gp.col0[g] + t;
                const int avail = min(j - gp.lo[g] + 1, gp.K + 1);
                const uint32_t y = (z >> (2 * (hi - j))) & ((1u << (2 * avail)) - 1u);
                p *= (avail == gp.K + 1) ? s[(uint32_t)j * gp.Yn + y] : U[bl.off[avail] + ((uint32_t)j << (2 * avail)) + y];
            }
            packed |= bf16_up(p) << (16 * h);
        }
        tab[i] = packed;
        if (ref) {
            const uint32_t r = ref[i];
            uint32_t x = 0u;
            for (int h = 0; h < 2; h++) {
                const float B = __uint_as_float(h ? packed & 0xffff0000u : packed << 16), R = __uint_as_float(h ? r & 0xffff0000u : r << 16);
                const float q = B == 0.0f ? 0.0f : R == 0.0f ? __int_as_float(0x7f800000) : __fdiv_ru(B, R);
                x = max(x, __float_as_uint(q));             // non-negative floats order as their bits
            }
            const uint32_t peers = __match_any_sync(__activemask(), g);
            x = __reduce_max_sync(peers, x);
            if ((__ffs(peers) - 1) == (int)(threadIdx.x & 31)) atomicMax(&rho[g], x);
        }
    }
}
// start of an E-step: scalars and list-overflow flag cleared; the dense-hold counter of the pruned path ticks down.
// reuse != nullptr: choose between the full bound pass and the watch pass (k_ebound, k_ebound_watch). A window outside the watch
// list has b_ref(p) < thr_ref 2^-m; the bounds now are at most P = prod_g rho_g times the reference ones, so b(p) < thr when
// P thr_ref / thr < 2^m. thr = thr0 LW1 / q with thr0 proportional to 1 - q, so thr_ref / thr = ((1-q_ref)/q_ref) / ((1-q)/q).
// Rounding: b(p) and b_ref(p) are float products of G1 <= 8 factors, each within (1+2^-24)^7 of the exact product, thr within
// a few ulps; the factor 1 + 2^-16 in P covers all of it. Intermediate products that end up subnormal lose relative accuracy,
// but their absolute error (< 2^-149 times the remaining factors, each < 2^64) stays far below thr * 2^-m (> 2^-80 for m <= 32).
// P has to bound the drift of the CURRENT tables, however many E-steps ran since they were built (estep, optimize_q, estep; the
// E-steps of a dense hold): the table factor prod_g rho_g is kept in BR_PTAB and replaced only when tables were built since the
// last E-step (some rho_g != 0; all of them 0 means every bound is 0, and any P is then right). The q ratio is formed afresh.
__global__ void k_estep_begin(unsigned long long* __restrict__ scal, uint32_t* __restrict__ overflow, uint32_t* __restrict__ eflags,
                              uint32_t* __restrict__ reuse, float q, float slack_pow /* 2^m */, int G1, unsigned long long nwin) {
    if (threadIdx.x == 0) {
        scal[0] = 0ull; scal[1] = 0ull;
        if (overflow) *overflow = 0u;
        if (eflags) {
            uint32_t hold = eflags[1];
            if (eflags[5]) {                                      // the last E-step ran over its candidate cap
                const uint32_t len = eflags[4] ? min(2u * eflags[4], DENSE_HOLD_MAX) : DENSE_HOLD_MIN;
                eflags[4] = len; eflags[5] = 0u;
                hold = len;
            } else if (eflags[0] == 0u) eflags[4] = 0u;           // a pruned E-step that fit: the next overflow starts at the short hold
            eflags[0] = hold ? 1u : 0u;
            eflags[1] = hold ? hold - 1u : 0u;
            eflags[2] = 0u; eflags[3] = 0u;
        }
        if (reuse) {
            bool built = false;
            double T = 1.0;
            for (int g = 0; g < G1; g++) { built |= reuse[BR_RHO + g] != 0u; T *= (double)__uint_as_float(reuse[BR_RHO + g]); reuse[BR_RHO + g] = 0u; }
            if (built) reuse[BR_PTAB] = __float_as_uint(__double2float_ru(T));
            const float qr = __uint_as_float(reuse[BR_QREF]);
            const double P = ((1.0 - (double)qr) / (double)qr) / ((1.0 - (double)q) / (double)q) * (1.0 + 1.0 / 65536.0) *
                             (double)__uint_as_float(reuse[BR_PTAB]);
            // a watch window costs about two windows of the full pass (one lookup per window instead of per pair, a list read,
            // dependent loads): a list of more than a quarter of the windows does not pay, and is then rebuilt only every 8th full pass
            const bool dense = eflags[0] != 0u, big = reuse[BR_WFULL] != 0u || 4ull * reuse[BR_WCOUNT] > nwin;
            const bool watch = !dense && reuse[BR_VALID] != 0u && !big && P < (double)slack_pow;
            const bool rebuild = !watch && !dense && !(big && ++reuse[BR_SKIP] % 8u != 0u);
            reuse[BR_MODE] = watch ? 1u : rebuild ? 0u : 2u;
            if (reuse[BR_VALID]) reuse[BR_LAMBDA] = __float_as_uint((float)log2(P));
            if (watch) reuse[BR_WATCH]++;
            else if (!dense) reuse[BR_FULL]++;
            if (rebuild) {                                        // this full pass rebuilds the list (k_ebound clears VALID if it cannot)
                reuse[BR_VALID] = 1u; reuse[BR_QREF] = __float_as_uint(q); reuse[BR_WCOUNT] = 0u; reuse[BR_WFULL] = 0u;
                reuse[BR_PTAB] = __float_as_uint(1.0f);           // tab_ref becomes the current tables
            }
        }
    }
}

// r <- r * scale for every packed-list sequence: run before r leaves the device (bamm_em_get_r). One warp per sequence.
__global__ void k_normalise_r(PackedView pv, int W, const float* __restrict__ scale, float* __restrict__ r) {
    const int lane = threadIdx.x & 31;
    const uint32_t warp = blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
    const uint32_t nwarps = gridDim.x * (blockDim.x >> 5);
    for (uint32_t li = warp; li < pv.nlist; li += nwarps) {
        const int LW1 = (int)pv.seqs[pv.seq_ids[li]].L - W + 1;
        const float f = scale[li];
        float* __restrict__ rn = r + pv.r_off[li];
        for (int k = lane; k < LW1; k += 32) rn[k] *= f;
    }
}

// ---- scoring -------------------------------------------------------------------------------------------------------
// reference: ScoreSeqSet::calcLogOdds, src/seq_scoring/ScoreSeqSet.cpp:25-67. Plain table, sum in ascending j from
// 0.0f: bit-identical to the reference for the same table. Only the k-mer fetch differs from k_score.
__global__ void __launch_bounds__(512)
k_score_packed(PackedView pv, Plan pl, const uint64_t* __restrict__ mops_off, const float* __restrict__ s_g,
               float* __restrict__ zoops, unsigned long long* __restrict__ z, float* __restrict__ mops, const uint32_t* __restrict__ out_idx) {
    extern __shared__ float s_sh[];
    for (uint32_t i = threadIdx.x; i < (uint32_t)pl.W * pl.Yn; i += blockDim.x) s_sh[i] = s_g[i];
    __syncthreads();
    const int lane = threadIdx.x & 31;
    const uint32_t warp = blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
    const uint32_t nwarps = gridDim.x * (blockDim.x >> 5);
    const int W = pl.W, K = pl.K;
    const uint32_t maskK = pl.Yn - 1;
    for (uint32_t li = warp; li < pv.nlist; li += nwarps) {
        const uint32_t n = pv.seq_ids[li];
        const uint32_t oi = out_idx ? out_idx[li] : li;    // position of this sequence in the caller's subset
        const PackedSeq sq = pv.seqs[n];
        const int L = (int)sq.L, LW1 = L - W + 1, mid = (int)sq.mid;
        const uint32_t* __restrict__ wd = pv.words + sq.word_off;
        float best = -3.402823466e+38f;
        int bestp = 0;
        for (int p0 = 0; p0 < LW1; p0 += 32) {
            const int p = p0 + lane;
            const unsigned long long w = window_word(wd, p - K);
            const bool over_n = mid >= 0 && p <= mid + K && p + W - 1 >= mid;
            float sc = 0.0f;
            int sh = 62 - 2 * K;
            uint32_t jb = 0;
            if (__any_sync(FULL, over_n)) {
                for (int j = 0; j < W; j++) {
                    uint32_t y = field(w, sh, maskK);
                    const int d = p + j - mid;
                    if (over_n && d >= 0 && d <= K) y = pv.ypatch[(uint64_t)n * (K + 1) + d];
                    sc += s_sh[jb + y];
                    sh -= 2; jb += pl.Yn;
                }
            } else {
                for (int j = 0; j < W; j++) {
                    sc += s_sh[jb + field(w, sh, maskK)];
                    sh -= 2; jb += pl.Yn;
                }
            }
            if (p < LW1) {
                if (mops) mops[mops_off[oi] + p] = sc;
                if (sc > best) { best = sc; bestp = p; }
            }
        }
        for (int o = 16; o > 0; o >>= 1) {
            const float ob = __shfl_xor_sync(FULL, best, o);
            const int op = __shfl_xor_sync(FULL, bestp, o);
            if (ob > best || (ob == best && op < bestp)) { best = ob; bestp = op; }
        }
        if (lane == 0) { zoops[oi] = best; z[oi] = (unsigned long long)bestp; }
    }
}

}  // namespace bamm
