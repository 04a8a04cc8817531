// common.cuh — types and small device helpers shared by every translation unit of libbamm_b200 (no kernels here: each kernel
// header is included by exactly one .cu file, see build.py).
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>
#include "../../include/bamm_b200.h"       // BAMM_MAX_MOTIF_WIDTH sizes per-column arrays in the kernels

namespace bamm {

constexpr int   FX_SHIFT      = 40;                       // counts: value * 2^40
constexpr float FX_SCALE_F    = 1099511627776.0f;         // 2^40
constexpr double FX_INV_D     = 1.0 / 1099511627776.0;
constexpr double SC_SCALE_D   = 4294967296.0;             // scalars (llh, sum r): value * 2^32
constexpr double SC_INV_D     = 1.0 / 4294967296.0;
constexpr unsigned FULL = 0xffffffffu;
#ifndef BAMM_E_THREADS
#define BAMM_E_THREADS 1024      // threads per CTA of the packed E-step (one CTA per SM: the tables fill shared memory)
#endif

__device__ __forceinline__ float warp_sum(float v) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(FULL, v, o);
    return v;
}

struct PackedSeq {           // per regular sequence
    uint64_t word_off;       // index of the sequence's FIRST DATA word (two zero pad words sit before it)
    uint32_t L;              // stored length
    uint32_t mid;            // position of the structural N, or 0xffffffff
};

struct PackedView {
    const uint32_t* words;             // packed stream, 16 bases per 32-bit word
    const PackedSeq* seqs;             // [nseq] (entries of irregular sequences are unused)
    const uint16_t* ypatch;            // [nseq][K+1] order-K k-mer index at positions mid..mid+K (rand() draws inside)
    const uint32_t* seq_ids;           // list -> seqset index
    const uint64_t* r_off;             // list -> offset of the sequence's r
    uint32_t nlist;
};

// ---- column groups ------------------------------------------------------------------------------------------------
// The W motif columns are cut into G consecutive groups; group g folds its columns into ONE table lookup over the
// bases its columns depend on. Column j reads the (K+1)-mer ending at base p+j, but its value only depends on
// ctx(j)+1 of those bases, ctx(j) = max(min(j,K), K_bg): for j < K the model's v[K][y][j] is a copy of the order-j
// entry (Motif::updateV, Motif.h:126-128) and the background factor uses K_bg+1 bases (Motif.cpp:485-494). The first
// group therefore reaches only K_bg bases left of the window and can be wider for the same table size
// (C3: columns 0-4 in one 4^7 table). A host-side DP picks the cut with the fewest groups that fits shared memory.
constexpr int MAXG = 16;
struct GroupPlan {
    int W, K, G, kd;             // window word = the 32 bases starting at base p-kd (kd may be negative in later column passes)
    uint32_t Yn;                 // 4^(K+1)
    float q;
    uint32_t table_bytes;
    uint32_t shift[MAXG];        // (w >> shift) & mask4 = byte offset of the group's entry
    uint32_t shift2[MAXG];       // general mode: extra shift after the clamped funnel shift
    uint32_t mask4[MAXG];
    uint32_t base[MAXG];         // byte offset of the group's table
    uint32_t colmask[MAXG];      // bit j for every column of the group
    int col0[MAXG], ncol[MAXG], lo[MAXG];   // first column, column count, first base relative to the window start p
    // column passes: when the tables of all W columns do not fit shared memory (orders >= 5 with wide motifs) the E-step
    // runs once per pass over a column range; the partial product of the earlier passes travels through r
    uint32_t passmask;           // bit j for every column of this pass (all W columns in a single-pass plan)
    int pass_first, pass_last;
    float thr0;                  // 2^-41 (1-q) 0.999: smallest unnormalised value that can reach the M-step's threshold (norm >= 1-q)
};
// every group's bit field sits below bit 32 of the window word, so one shift extracts it (the kernels' FAST variant). Group 0
// ends at the lowest column and has the largest shift; the planners place it at <= 30 when they can and at >= 32 otherwise.
inline bool one_shift(const GroupPlan& gp) { return gp.shift[0] < 32; }

// ---- window extraction ---------------------------------------------------------------------------------------------
// 64 bits holding bases b0 .. b0+31 of a sequence (b0 >= -32: the pad words supply leading zeros), as (hi, lo).
__device__ __forceinline__ void window_bits(const uint32_t* wd, int b0, uint32_t& whi, uint32_t& wlo) {
    const int wi = b0 >> 4;                      // floor
    const int s = 2 * (b0 & 15);
    const uint32_t t0 = wd[wi], t1 = wd[wi + 1], t2 = wd[wi + 2];
    whi = __funnelshift_l(t1, t0, s);
    wlo = __funnelshift_l(t2, t1, s);
}
__device__ __forceinline__ unsigned long long window_word(const uint32_t* wd, int b0) {
    uint32_t hi, lo; window_bits(wd, b0, hi, lo);
    return ((unsigned long long)hi << 32) | lo;
}

__device__ __forceinline__ uint32_t field(unsigned long long w, int shift, uint32_t mask) {
    return (uint32_t)(w >> shift) & mask;
}

struct Plan {                 // launch-invariant parameters of the packed M-step / scoring kernels
    int W, K, T, C;
    uint32_t Yn, Zn;          // 4^(K+1)
    float q;
};

// Windows whose posterior survives the M-step's fixed-point rounding, written by the E-step while it normalises:
// one region per E-step warp (no atomics, no ordering requirement: the M-step sums integers).
// Entry: everything the M-step needs without a second dependent load — the word offset of the sequence in the packed stream
// (streams below 2^32 words), the window start p (sequences below 2^26 bases) with the last column of the window
// (jmax, EM.cpp:167) and a flag for windows over the structural N packed above it, the UNNORMALISED posterior, the list index.
struct ActiveEntry { uint32_t woff, pcode; float rv; uint32_t li; };   // 16 bytes: one 128-bit store / load per entry
constexpr int ACT_JMAX_SHIFT = 26;
constexpr uint32_t ACT_P_MASK = (1u << ACT_JMAX_SHIFT) - 1u;
constexpr uint64_t PACKED_MAX_L = 1ull << ACT_JMAX_SHIFT;              // longer sequences take the generic path
struct ActiveList {
    ActiveEntry* ent;         // entries
    float* scale;             // [nlist] 1/normaliser of every list sequence: posterior = rv * scale[li]
    const uint64_t* reg_off;  // [nregions+1] first entry of every region
    uint32_t* cnt;            // [nregions] entries written at the front of the region (full windows of the fast chunks)
    uint32_t* cnt_back;       // [nregions] entries written at the back, downwards (windows of the masked chunks)
    uint32_t* overflow;       // set when a region was too small: the M-step then scans r instead
};
constexpr float FX_HALF_UNIT = 4.547473508864641e-13f;   // 2^-41: smallest r that rounds to a non-zero count

// Candidate windows of the pruned E-step (estep.cuh): window starts whose upper bound reaches the M-step's threshold, written by
// k_ebound (one region per warp, the candidates of a sequence contiguous and ascending), evaluated exactly by k_eexact.
struct CandList {
    uint32_t* ent;            // window starts
    const uint64_t* reg_off;  // [nregions+1] first entry of every region
    uint2* seq;               // [nlist] (first entry inside the region, count) of every list sequence
    uint32_t* flags;          // [0] != 0: this iteration runs the dense E-step (a region overflowed, or the hold below is active)
                              // [1] iterations the dense E-step stays switched on after an overflow; [2..3] 64-bit candidate count (diagnostics)
                              // [4] length of the current hold; [5] != 0: a region overflowed in the last E-step (k_estep_begin turns it into a hold)
    // bound reuse (k_ebound_watch): the full pass also lists the windows whose bound reaches thr * watch_scale (the watch list,
    // same region layout and order as the candidates); while the tables have not moved far enough from those it was built from
    // (tab_ref) to lift any other window to thr, only the listed windows are bounded again. reuse == nullptr: always full passes.
    uint32_t* went;           // watched window starts
    const uint64_t* wreg_off; // [nregions+1] first entry of every watch region
    uint2* wseq;              // [nlist] (first entry inside the region, count)
    uint32_t* reuse;          // BREUSE_WORDS words, see below
    float* tab_ref;           // the bound tables the watch list was built from (copied by CTA 0 of the full pass)
    float watch_scale;        // 2^-m, m = slack in bits
};
// words of CandList::reuse. [BR_MODE] this E-step runs 0: the full pass and rebuilds the watch list, 1: the watch pass, 2: the full
// pass without the list (the last one was too long to pay); [BR_SKIP] full passes that kept a too long list; [BR_WFULL] a watch region filled up in the last list build; [BR_VALID] the watch list matches tab_ref and q_ref;
// [BR_QREF] q of the full pass that built it (float bits); [BR_LAMBDA] log2 of the last drift bound (float bits);
// [BR_FULL], [BR_WATCH] passes of each kind (diagnostics); [BR_WCOUNT] entries of the watch list;
// [BR_PTAB] prod_g rho_g of the current tables against tab_ref, rounded up (float bits; k_estep_begin keeps it across E-steps that
// follow no table build, 1 after a list build);
// [BR_RHO + g] max_e B_g[e] / tab_ref_g[e] of the tables built since the last E-step (float bits, k_make_bound_tables; 0: none built)
constexpr int BR_MODE = 0, BR_VALID = 1, BR_QREF = 2, BR_LAMBDA = 3, BR_FULL = 4, BR_WATCH = 5, BR_WCOUNT = 6, BR_SKIP = 7, BR_WFULL = 8, BR_PTAB = 9,
              BR_RHO = 10, BREUSE_WORDS = BR_RHO + MAXG;
// After an overflow the dense E-step runs for 2 iterations, then the bound pass tries again; every further overflow in a row
// doubles the hold (a model whose posteriors stay diffuse pays log2(iterations) wasted bound passes, one that sharpens after
// the first iterations is back on the pruned path at once); a pruned iteration that fits resets it.
constexpr uint32_t DENSE_HOLD_MIN = 2, DENSE_HOLD_MAX = 64;

struct MTables {                                  // packed M-step
    uint32_t nrep, rstride;                       // table copies per CTA and their stride in words (rstride >= NC * Yn)
    uint32_t hi_global;                           // != 0: no high-word table in shared memory (twice the columns per CTA): the rare
};                                                // high parts / carries go to the CTA's 64-bit partial table with global atomics

// ---- table staging: global -> shared memory with the TMA (1-D bulk copies, no tensor map) --------------------------
// Thread 0 arms an mbarrier with the byte count and issues cp.async.bulk copies of up to 64 KB; every thread of the CTA then
// waits on the barrier's phase. The copy engine moves the tables while the threads do other set-up work (copying the padded
// plain table, building step tables), instead of 50 dependent load / store rounds per thread. bytes: multiple of 16; both
// pointers 16-byte aligned. Call bulk_stage_begin from all threads (it contains a __syncthreads), bulk_stage_wait before the
// first use of the tables. One staging per kernel launch (phase 0 of the barrier).
__device__ __forceinline__ void bulk_stage_begin(void* smem_dst, const void* gmem_src, uint32_t bytes, unsigned long long* mbar) {
    const uint32_t mb = (uint32_t)__cvta_generic_to_shared(mbar);
    if (threadIdx.x == 0) {
        asm volatile("mbarrier.init.shared::cta.b64 [%0], 1;" :: "r"(mb) : "memory");
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    __syncthreads();
    if (threadIdx.x == 0) {
        asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" :: "r"(mb), "r"(bytes) : "memory");
        const uint32_t dst = (uint32_t)__cvta_generic_to_shared(smem_dst);
        const char* src = static_cast<const char*>(gmem_src);
        for (uint32_t off = 0; off < bytes; off += 65536u) {
            const uint32_t n = bytes - off < 65536u ? bytes - off : 65536u;
            asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];"
                         :: "r"(dst + off), "l"(src + off), "r"(n), "r"(mb) : "memory");
        }
    }
}
__device__ __forceinline__ void bulk_stage_wait(unsigned long long* mbar) {
    const uint32_t mb = (uint32_t)__cvta_generic_to_shared(mbar);
    uint32_t done;
    do {
        asm volatile("{ .reg .pred p; mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2; selp.u32 %0, 1, 0, p; }"
                     : "=r"(done) : "r"(mb), "r"(0u) : "memory");
    } while (!done);
}

// shared-memory load at (per-lane byte offset) + (warp-uniform base): one LDS with a uniform-register base operand
__device__ __forceinline__ float lds_f32(uint32_t off, uint32_t ubase) {
    float v;
    asm("ld.shared.f32 %0, [%1];" : "=f"(v) : "r"(off + ubase));
    return v;
}

}  // namespace bamm
