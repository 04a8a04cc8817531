// capi.cu — implementation of include/bamm_b200.h on top of kernels.cuh. Host plumbing only: device memory,
// one CUDA stream per EM object, launches, scalar read-back. No CPU fallback: every compute entry point needs a device.
#include "../../include/bamm_b200.h"
#include "kernels.cuh"
#include "packed.cuh"
#include "launch.h"
#include "negatives.cuh"
#include "stats.cuh"
#include "scan.cuh"
#include <cub/device/device_scan.cuh>
#include "fasta.cuh"
#include "mask.cuh"

#include <math.h>
#include <stdarg.h>
#include <stdio.h>
#include <stdlib.h>
#include <string.h>

#include <algorithm>
#include <map>
#include <mutex>
#include <new>
#include <string>
#include <type_traits>
#include <vector>

using namespace bamm;

// ------------------------------------------------------------------------------------------- errors
static thread_local char g_err[512] = "";
static thread_local float g_score_ms = 0.0f;      // device time of the scoring kernels of the last bamm_score_logodds call on this thread
static int fail(int code, const char* fmt, ...) {
    va_list ap; va_start(ap, fmt); vsnprintf(g_err, sizeof(g_err), fmt, ap); va_end(ap);
    return code;
}
#define CU(call) do { cudaError_t e_ = (call); if (e_ != cudaSuccess) \
    return fail(e_ == cudaErrorMemoryAllocation ? BAMM_E_NOMEM : BAMM_E_CUDA, "%s failed: %s (%s:%d)", #call, cudaGetErrorString(e_), __FILE__, __LINE__); } while (0)
#define REQUIRE(cond, ...) do { if (!(cond)) return fail(BAMM_E_INVALID, __VA_ARGS__); } while (0)

// Device memory comes from the device's default memory pool (cudaMallocAsync) with an unlimited release threshold: buffers a
// finished object gives back stay mapped, so creating the next sequence set / EM object / scoring call does not pay the
// driver's map-and-zero cost again (measured: the same 1-12 GB allocations vary between 3 ms and 150 ms with cudaMalloc
// after a large cudaFree). cudaFree() returns pool memory to the pool. Falls back to cudaMalloc where pools are missing.
static cudaError_t pool_malloc(void** p, size_t bytes) {
    static thread_local int ready_dev = -1;
    static thread_local bool usable = false;
    int dev = 0;
    cudaError_t e = cudaGetDevice(&dev);
    if (e != cudaSuccess) return e;
    if (ready_dev != dev) {
        int supported = 0;
        usable = !getenv("BAMM_NO_MEMPOOL") && cudaDeviceGetAttribute(&supported, cudaDevAttrMemoryPoolsSupported, dev) == cudaSuccess && supported;
        if (usable) {
            cudaMemPool_t pool;
            unsigned long long thr = ~0ull;
            usable = cudaDeviceGetDefaultMemPool(&pool, dev) == cudaSuccess &&
                     cudaMemPoolSetAttribute(pool, cudaMemPoolAttrReleaseThreshold, &thr) == cudaSuccess;
        }
        cudaGetLastError();
        ready_dev = dev;
    }
    if (!usable) return cudaMalloc(p, bytes);
    e = cudaMallocAsync(p, bytes, 0);
    if (e != cudaSuccess) return e;
    return cudaStreamSynchronize(0);                          // the buffer is used from other (non-blocking) streams right away
}
template <typename T> static cudaError_t dev_malloc(T** p, size_t bytes) { return pool_malloc(reinterpret_cast<void**>(p), bytes); }

// BAMM_TRACE=1: wall-clock phases of the set-up calls on stderr (diagnostics of the end-to-end path)
#include <chrono>
struct Trace {
    bool on; const char* what; std::chrono::steady_clock::time_point t0;
    explicit Trace(const char* w) : on(getenv("BAMM_TRACE") != nullptr), what(w), t0(std::chrono::steady_clock::now()) {}
    void mark(const char* phase) {
        if (getenv("BAMM_SYNC_MARKS")) cudaDeviceSynchronize();
        if (!on) return;
        cudaDeviceSynchronize();
        const auto t1 = std::chrono::steady_clock::now();
        fprintf(stderr, "[bamm trace] %s: %s %.2f ms\n", what, phase, std::chrono::duration<double, std::milli>(t1 - t0).count());
        t0 = t1;
    }
};
// Pinned host scalars of the EM objects (log likelihood, sum of posteriors, sum|dv| read back every iteration): slots of one
// process-wide pinned slab — a pinned allocation per object costs milliseconds (FDR creates an EM object per fold).
static std::mutex g_pin_mu;
static unsigned long long* g_pin_slab = nullptr;
static std::vector<int> g_pin_free;
constexpr int PIN_SLOTS = 256, PIN_SLOT_WORDS = 4;
static cudaError_t pinned_scalars_get(unsigned long long** out) {
    {
        std::lock_guard<std::mutex> g(g_pin_mu);
        if (!g_pin_slab) {
            void* p = nullptr;
            if (cudaHostAlloc(&p, (size_t)PIN_SLOTS * PIN_SLOT_WORDS * sizeof(unsigned long long), cudaHostAllocPortable) == cudaSuccess) {
                g_pin_slab = static_cast<unsigned long long*>(p);
                for (int i = PIN_SLOTS - 1; i >= 0; i--) g_pin_free.push_back(i);
            } else cudaGetLastError();
        }
        if (g_pin_slab && !g_pin_free.empty()) {
            *out = g_pin_slab + (size_t)g_pin_free.back() * PIN_SLOT_WORDS;
            g_pin_free.pop_back();
            return cudaSuccess;
        }
    }
    return cudaMallocHost(out, PIN_SLOT_WORDS * sizeof(unsigned long long));
}
static void pinned_scalars_put(unsigned long long* p) {
    if (!p) return;
    {
        std::lock_guard<std::mutex> g(g_pin_mu);
        if (g_pin_slab && p >= g_pin_slab && p < g_pin_slab + (size_t)PIN_SLOTS * PIN_SLOT_WORDS) {
            g_pin_free.push_back((int)((p - g_pin_slab) / PIN_SLOT_WORDS));
            return;
        }
    }
    cudaFreeHost(p);
}
static uint64_t ipow_u64(uint64_t b, int e) { uint64_t r = 1; while (e-- > 0) r *= b; return r; }

// ------------------------------------------------------------------------------------------- objects
struct IndexArray { void* d = nullptr; int bytes = 2; uint64_t Yn = 0; };
// The order-K index array holds uint16_t entries when A^(K+1) <= 65536 and uint32_t otherwise (seqset_index_locked); every
// kernel that reads it is instantiated for both. f is a generic lambda and receives the typed pointer.
template <typename F> static auto with_index(const IndexArray& ia, F&& f) { return ia.bytes == 2 ? f((const uint16_t*)ia.d) : f((const uint32_t*)ia.d); }
template <typename F> static auto with_index_mut(IndexArray& ia, F&& f) { return ia.bytes == 2 ? f((uint16_t*)ia.d) : f((uint32_t*)ia.d); }
// The column blocks of a W-column motif (column_blocks, kernels.cuh) as the compile-time NB of the index-array kernels
template <typename F> static auto with_column_blocks(int W, F&& f) { return column_blocks(W) == 2 ? f(std::integral_constant<int, 2>()) : f(std::integral_constant<int, 1>()); }
// Index-array kernels with the [j][y] table in shared memory run 512-thread CTAs, as many per SM as the opt-in shared memory
// holds (1 KB per CTA reserved), at most 4 (2048 threads, the SM's limit); a table beyond shared memory: 4 CTAs per SM.
struct TableGrid { bool smem; int grid; };
static TableGrid table_grid(size_t table_bytes, int max_optin, int sms) {
    if (table_bytes > (size_t)max_optin) return {false, sms * 4};
    return {true, sms * std::max(1, std::min(4, (int)((size_t)(max_optin + 1024) / (table_bytes + 1024))))};
}

struct bamm_seqset {
    int device = 0;
    int A = 4;
    uint64_t nseq = 0, npos = 0, npatch = 0, maxL = 0, minL = 0;
    uint8_t* d_codes = nullptr;
    uint64_t* d_off = nullptr;
    uint64_t* d_ppos = nullptr;
    uint64_t* d_pkmer = nullptr;
    std::vector<uint64_t> h_off;
    std::map<int, IndexArray> index;   // per order K (built on demand: generic path, get_index, count_kmers)
    std::mutex mu;
    int sm_count = 148;
    // 2-bit packed path (A == 4): per-sequence kind (0 irregular, 1 regular, 2 regular with the structural N)
    std::vector<uint8_t> h_kind;
    uint8_t* d_kind = nullptr;
    PackedSeq* d_pseq = nullptr;
    uint32_t* d_words = nullptr;        // 16 bases per word
    uint64_t nwords = 0, nregular = 0;
    std::map<int, uint16_t*> ypatch;   // per order K: [nseq][K+1] k-mer index at mid..mid+K
    // sets encoded from FASTA text on the device: stored positions of the forward undefined bases, until the patches arrive
    uint64_t* d_zero_pos = nullptr;
    uint64_t n_zero_fwd = 0;
    std::map<int, bamm_seqset*> replicas;   // device -> copy of this set on that device (device groups, capi_group.inl)
    // bamm_seqset_create: the uploads run on their own stream while the host checks the offsets and the first kernels start
    cudaStream_t copy_stream = nullptr;
    cudaEvent_t ev_codes = nullptr, ev_patches = nullptr;
};
static void seqset_copy_done(bamm_seqset* s) {      // waits for the uploads and drops the stream
    if (s->copy_stream) { cudaStreamSynchronize(s->copy_stream); cudaStreamDestroy(s->copy_stream); s->copy_stream = nullptr; }
    if (s->ev_codes) { cudaEventDestroy(s->ev_codes); s->ev_codes = nullptr; }
    if (s->ev_patches) { cudaEventDestroy(s->ev_patches); s->ev_patches = nullptr; }
}

struct bamm_em {
    // device group: a non-empty list makes this object a facade (no device state of its own) over one object per device, each
    // over a contiguous block of the subset; shard_first[d] = first subset position of shard d (capi_group.inl)
    std::vector<bamm_em*> shards;
    std::vector<uint64_t> shard_first;
    bool peer_sums_global = false;   // the scalars in d_xbuf are sums over all ranks (after an exchange), not this rank's own
    bamm_seqset* ss = nullptr;
    int device = 0;
    cudaStream_t stream = nullptr;
    cudaEvent_t ev[4] = {nullptr, nullptr, nullptr, nullptr};
    std::vector<cudaEvent_t> loop_ev;       // LOOP_EV per iteration of the last bamm_em_iterate call (capi_em.inl, launch_iteration)
    int loop_iters = 0;
    bool own_xbuf = true;
    int W = 0, K = 0, K_bg_model = 0, K_bg = 0, A = 4;
    uint32_t Yn = 0;            // A^(K+1)
    uint32_t nbin = 0;          // W * Yn
    uint64_t nsub = 0, rsize = 0, nseq_global = 0;
    uint64_t model_size = 0, bg_size = 0;
    ModelDims dims;
    bool smem_tables = true;    // generic path: tables fit in shared memory
    int grid_e = 0, grid_m = 0, block = 512;
    size_t smem_e = 0, smem_m = 0;
    // the subset is split into a packed list (regular 4-letter sequences) and a generic list (everything else)
    uint32_t ngen = 0, npk = 0;
    uint32_t* d_gen_ids = nullptr;  uint64_t* d_gen_roff = nullptr;
    uint32_t* d_pk_ids = nullptr;   uint64_t* d_pk_roff = nullptr;
    Plan plan;                  // W, K, Yn for the packed M-step / scoring kernels
    std::vector<GroupPlan> gplans;   // column groups of the packed E-step, one plan per column pass (chosen in set_model)
    size_t tab_capacity = 0;    // bytes available for the group tables (= opt-in shared memory)
    float* d_tab = nullptr;     // group tables, concatenated; tab_capacity bytes per pass
    float* d_tab_alt = nullptr; // second buffer: launch_update writes the next tables there and swaps, so the tables of the last
                                // E-step stay available (bamm_em_get_r materialises r from them, bamm_em_get_s returns them)
    size_t tab_passes = 0;      // passes d_tab has room for
    uint32_t plain_words = 0;   // > 0: the plain [j][y] table rides in shared memory behind the group tables (single columns of masked windows)
    // pruned E-step (estep.cuh): bound plan + tables, candidate list, device-side flags
    bool cand_ok = false;       // candidate list allocated (bamm_em_create)
    bool sparse = false;        // the current plans use the pruned path (bamm_em_set_model)
    bool stage = false;         // the exact pass stages the sequence words in shared memory
    GroupPlan bplan;
    BoundLevels blev;
    float* d_btab = nullptr;    // bound tables
    float* d_U = nullptr;       // maxima of s over dropped context bases, per level
    uint32_t* d_cand = nullptr; uint2* d_cand_seq = nullptr; uint64_t* d_creg_off = nullptr;
    uint64_t cand_slots = 0;         // entries of the candidate list
    float* d_cand_part = nullptr;    // column passes: partial product per candidate slot (k_eexact)
    float* d_mask_part = nullptr;    // column passes: partial product per masked window of every sequence (k_emasked)
    ulonglong2* d_seqacc = nullptr;  // per list sequence: normaliser terms of its masked windows (k_emasked -> k_eexact)
    uint32_t* d_eflags = nullptr;   // CandList::flags (8 words)
    // bound reuse (CandList::went ..): watch list, its region offsets and per-sequence records, the tables it was built from,
    // the device-side state (BREUSE_WORDS); d_reuse == nullptr: off (BAMM_NO_BOUND_REUSE, or no memory for the list)
    uint32_t* d_watch = nullptr; uint64_t* d_wreg_off = nullptr; uint2* d_watch_seq = nullptr;
    float* d_btab_ref = nullptr; uint32_t* d_reuse = nullptr;
    int bound_slack = 10;           // m: the watch list holds the windows whose bound reaches thr 2^-m (BAMM_BOUND_SLACK)
    bool r_mat = true;          // d_r holds the posteriors of the last E-step (false after a pruned E-step until bamm_em_get_r)
    const float *d_s_e = nullptr, *d_tab_e = nullptr;   // the tables the last E-step read
    float q_e = 0.3f;           // ... and its prior
    float* d_s_keep = nullptr;  // copy of the s of the last E-step once a second update reuses its buffer (keep_last_estep)
    // active list (windows that survive the M-step's fixed-point rounding), one region per E-step warp
    uint32_t nregions = 0;
    ActiveEntry* d_act = nullptr;
    float* d_scale = nullptr;   // 1/normaliser per packed-list sequence (the packed E-step leaves r unnormalised)
    bool r_scaled = true;       // r already holds normalised values
    uint64_t launches = 0;      // kernels launched by this object (bench.py reports them)
    // NVLink peer exchange (multi-GPU): local receive buffer [2][world][nbin+2] + flags, peers' buffers mapped through CUDA IPC
    int peer_rank = 0, peer_world = 0;
    bool peer_attached = false;
    unsigned char* d_peer_local = nullptr;      // slots, then flags
    void* peer_mapped[MAX_PEERS] = {nullptr};   // cudaIpcOpenMemHandle results (to close)
    PeerPtrs peer_ptrs;
    uint32_t peer_epoch = 0;
    unsigned int* d_peer_done = nullptr;
    unsigned long long* d_peer_wait = nullptr;  // [0] ns spent waiting for the other ranks in k_peer_sum, [1] number of waits
    int m_nc = 0, m_nsplit = 1; // packed M-step: columns per CTA and number of column splits (packed.cuh, "column split")
    MTables m_tab = {1, 0, 0};  // table copies per CTA (orders 0 and 1), their stride in words, high words in global memory
    int grid_pl = 0;            // CTAs of the packed M-step kernels (a multiple of m_nsplit)
    uint32_t *d_act_cnt = nullptr, *d_overflow = nullptr;
    uint64_t* d_reg_off = nullptr;
    uint16_t* d_ypatch = nullptr;   // owned by the seqset
    int grid_pe = 0, block_pe = 1024;
    uint32_t nparts = 1;
    uint32_t gen_nrep = 1;          // generic M-step without shared-memory tables: copies of the global count table
    int gen_nsplit = 0, gen_nc = 0; // ... or column ranges with shared-memory low words (k_mstep_cols), 0 = off
    // device
    float* d_r = nullptr;
    float* d_s = nullptr;         // [j][y]
    float* d_sT = nullptr;        // the same table in the reference's [y][j] order (row gathers of the patched k-mers)
    float *d_s_alt = nullptr, *d_sT_alt = nullptr;   // second buffers, see d_tab_alt
    float* d_rows = nullptr;      // index-array E-step with tables beyond shared memory: [y][W4] rows padded for 16-byte loads
    float* d_v = nullptr;         // all orders
    float* d_vK_prev = nullptr;
    float* d_n = nullptr;         // all orders (float, reference layout)
    float* d_vbg = nullptr;
    float* d_alpha = nullptr;
    unsigned long long* d_part = nullptr;   // per-CTA partial count tables
    unsigned long long* d_xbuf = nullptr;   // [nbin] counts + [2] scalars  (the multi-GPU exchange buffer)
    float* d_vdiff = nullptr;
    double* d_vdiff_part = nullptr;         // per-CTA partial sums of the clustered model update
    // EM::mask workspaces (created by the first bamm_em_mask call)
    uint32_t* d_m_ids = nullptr; uint64_t* d_m_roff = nullptr; uint64_t* d_m_woff = nullptr;
    uint64_t* d_m_seloff = nullptr; uint32_t* d_m_sel = nullptr;
    std::vector<uint32_t> h_ids;            // subset -> seqset index (all sequences of the subset, in order)
    bool whole_set = false;                 // identity subset of an all-regular set: h_ids / h_r_off are made on first use (host_lists)
    // host (pinned)
    unsigned long long* h_scal = nullptr;   // 2 scalars
    float* h_vdiff = nullptr;
    std::vector<uint64_t> h_r_off;
    float q = 0.3f;
    float llh = 0.0f;
    bool model_set = false, r_valid = false;
};

// ------------------------------------------------------------------------------------------- library / device
extern "C" int bamm_version(void) { return 10000 * 0 + 100 * 1 + 0; }
extern "C" const char* bamm_last_error(void) { return g_err; }
extern "C" int bamm_device_count(int* count) {
    REQUIRE(count, "count is NULL");
    cudaError_t e = cudaGetDeviceCount(count);
    if (e != cudaSuccess) { *count = 0; return fail(BAMM_E_CUDA, "cudaGetDeviceCount: %s", cudaGetErrorString(e)); }
    return BAMM_OK;
}
extern "C" int bamm_set_device(int device) { CU(cudaSetDevice(device)); return BAMM_OK; }
extern "C" int bamm_device_info(int* sm_count, int* cc_major, int* cc_minor, uint64_t* total_mem) {
    int dev; CU(cudaGetDevice(&dev));
    cudaDeviceProp p; CU(cudaGetDeviceProperties(&p, dev));
    if (sm_count) *sm_count = p.multiProcessorCount;
    if (cc_major) *cc_major = p.major;
    if (cc_minor) *cc_minor = p.minor;
    if (total_mem) *total_mem = (uint64_t)p.totalGlobalMem;
    return BAMM_OK;
}

// ------------------------------------------------------------------------------------------- seqset
extern "C" void bamm_seqset_destroy(bamm_seqset* s);
// host bookkeeping + device allocation of codes / offsets (codes are filled by the caller: H2D copy or a device kernel)
// upload_codes: host codes to copy (bamm_seqset_create); the copy is started first, on the set's copy stream, and the host
// pass over the offsets runs while the bases travel. ev_codes marks codes + offsets in place.
// own_offsets: the vector `offsets` points into; it is moved into the set instead of copied (10^7 records of a negative set)
static int seqset_new(const uint64_t* offsets, uint64_t nseq, int A, bamm_seqset** out, const uint8_t* upload_codes = nullptr,
                      std::vector<uint64_t>* own_offsets = nullptr) {
    REQUIRE(out, "out is NULL");
    *out = nullptr;
    REQUIRE(offsets, "offsets is NULL");
    REQUIRE(A >= 2 && A <= 6, "alphabet size %d not in [2,6]", A);
    REQUIRE(offsets[0] == 0, "offsets[0] must be 0");
    REQUIRE(nseq < (1ull << 32), "too many sequences");
    if (!upload_codes)
        for (uint64_t n = 0; n < nseq; n++) REQUIRE(offsets[n + 1] >= offsets[n], "offsets not monotone at %llu", (unsigned long long)n);
    const uint64_t npos = offsets[nseq];
    bamm_seqset* s = new (std::nothrow) bamm_seqset();
    if (!s) return fail(BAMM_E_NOMEM, "host allocation failed");
    int dev; cudaError_t e = cudaGetDevice(&dev);
    if (e != cudaSuccess) { delete s; return fail(BAMM_E_CUDA, "no CUDA device: %s", cudaGetErrorString(e)); }
    s->device = dev; s->A = A; s->nseq = nseq; s->npos = npos; s->npatch = 0;
    cudaDeviceGetAttribute(&s->sm_count, cudaDevAttrMultiProcessorCount, dev);
#define CUS(call) do { cudaError_t e2_ = (call); if (e2_ != cudaSuccess) { bamm_seqset_destroy(s); \
    return fail(e2_ == cudaErrorMemoryAllocation ? BAMM_E_NOMEM : BAMM_E_CUDA, "%s failed: %s", #call, cudaGetErrorString(e2_)); } } while (0)
    CUS(dev_malloc(&s->d_codes, npos ? npos : 1));
    CUS(dev_malloc(&s->d_off, (nseq + 1) * sizeof(uint64_t)));
    if (upload_codes) {
        CUS(cudaStreamCreateWithFlags(&s->copy_stream, cudaStreamNonBlocking));
        CUS(cudaEventCreateWithFlags(&s->ev_codes, cudaEventDisableTiming));
        CUS(cudaEventCreateWithFlags(&s->ev_patches, cudaEventDisableTiming));
        CUS(cudaMemcpyAsync(s->d_off, offsets, (nseq + 1) * sizeof(uint64_t), cudaMemcpyHostToDevice, s->copy_stream));
        if (npos) CUS(cudaMemcpyAsync(s->d_codes, upload_codes, npos, cudaMemcpyHostToDevice, s->copy_stream));
        CUS(cudaEventRecord(s->ev_codes, s->copy_stream));
    } else {
        CUS(cudaMemcpy(s->d_off, offsets, (nseq + 1) * sizeof(uint64_t), cudaMemcpyHostToDevice));
    }
    uint64_t maxL = 0, minL = ~0ull, bad = ~0ull;
    for (uint64_t n = 0; n < nseq; n++) {
        if (offsets[n + 1] < offsets[n]) { bad = n; break; }
        uint64_t L = offsets[n + 1] - offsets[n];
        if (L > maxL) maxL = L;
        if (L < minL) minL = L;
    }
    if (bad != ~0ull) { bamm_seqset_destroy(s); return fail(BAMM_E_INVALID, "offsets not monotone at %llu", (unsigned long long)bad); }
    s->maxL = maxL; s->minL = nseq ? minL : 0;
    if (own_offsets) s->h_off.swap(*own_offsets);
    else s->h_off.assign(offsets, offsets + nseq + 1);
    *out = s;
    return BAMM_OK;
}

// classification + 2-bit packing on the device (no host pass over the bases); d_codes and the patch list are in place
// known_regular: the caller vouches that every code is in 1..4 (a set the library sampled itself): no classification pass
// validate_patches: the patch list came from the caller and is checked first (strictly increasing, inside the set)
static int seqset_finish(bamm_seqset* s, bool known_regular = false, bool validate_patches = false) {
    const uint64_t nseq = s->nseq, npatch = s->npatch;
    Trace tr("seqset_finish");
    s->h_kind.assign(nseq, s->A == 4 && known_regular ? 1 : 0);
    const bool classify = s->A == 4 && nseq && !known_regular;
    uint32_t* d_cover0 = nullptr;
    if (classify) {
        CUS(dev_malloc(&s->d_kind, nseq));
        CUS(dev_malloc(&d_cover0, nseq * sizeof(uint32_t)));
    }
    if (s->ev_codes) { cudaError_t ew = cudaStreamWaitEvent(0, s->ev_codes, 0); if (ew != cudaSuccess) { cudaFree(d_cover0); CUS(ew); } }
    if (classify) {       // needs the bases only: runs while the patch list is still on its way
        cudaMemsetAsync(d_cover0, 0, nseq * sizeof(uint32_t), 0);
        k_classify<<<s->sm_count * 8, 256>>>(s->d_codes, s->d_off, nseq, s->d_kind);
    }
    if (s->ev_patches) { cudaError_t ew = cudaStreamWaitEvent(0, s->ev_patches, 0); if (ew != cudaSuccess) { cudaFree(d_cover0); CUS(ew); } }
    if (validate_patches && npatch) {
        uint32_t* d_bad = nullptr; uint32_t bad = 0;
        cudaError_t ev = dev_malloc(&d_bad, sizeof(uint32_t));
        if (ev == cudaSuccess) ev = cudaMemsetAsync(d_bad, 0, sizeof(uint32_t), 0);
        if (ev == cudaSuccess) {
            k_validate_patches<<<(unsigned)((npatch + 255) / 256), 256>>>(s->d_ppos, npatch, s->npos, d_bad);
            ev = cudaMemcpy(&bad, d_bad, sizeof(bad), cudaMemcpyDeviceToHost);
        }
        cudaFree(d_bad);
        if (ev != cudaSuccess || bad) cudaFree(d_cover0);
        CUS(ev);
        if (bad) { bamm_seqset_destroy(s); return fail(BAMM_E_INVALID, bad & 1u ? "patch position out of range" : "patch positions must be strictly increasing"); }
    }
    if (s->A == 4 && nseq && known_regular) {
        CUS(dev_malloc(&s->d_kind, nseq));
        CUS(cudaMemset(s->d_kind, 1, nseq));
    }
    if (s->A == 4 && nseq) {
        uint32_t* d_cover = d_cover0;
        if (!known_regular) {
        if (npatch) k_check_patches<<<(unsigned)((npatch + 255) / 256), 256>>>(s->d_ppos, npatch, s->d_off, nseq, s->d_kind, d_cover);
        k_finish_kinds<<<(unsigned)((nseq + 255) / 256), 256>>>(s->d_off, nseq, d_cover, s->d_kind);
        cudaError_t ec = cudaMemcpy(s->h_kind.data(), s->d_kind, nseq, cudaMemcpyDeviceToHost);
        cudaFree(d_cover);
        CUS(ec);
        }
        tr.mark("classify + kinds D2H");
        // packed-stream layout on the device: word counts -> exclusive scan -> PackedSeq records (no host pass, no upload)
        if (known_regular) s->nregular = nseq;
        else for (uint64_t n = 0; n < nseq; n++) s->nregular += s->h_kind[n] != 0;
        if (s->nregular) {
            unsigned long long* d_wc = nullptr; void* d_tmp = nullptr; size_t tmp_bytes = 0;
            CUS(dev_malloc(&d_wc, (nseq + 1) * 2 * sizeof(unsigned long long)));
            unsigned long long* d_scan = d_wc + nseq + 1;
            CUS(cudaMemset(d_wc + nseq, 0, sizeof(unsigned long long)));            // sentinel: the scan's last entry is the total
            k_word_counts<<<(unsigned)((nseq + 255) / 256), 256>>>(s->d_off, nseq, s->d_kind, d_wc);
            cub::DeviceScan::ExclusiveSum(nullptr, tmp_bytes, d_wc, d_scan, (int)(nseq + 1));
            cudaError_t es = dev_malloc(&d_tmp, tmp_bytes ? tmp_bytes : 16);
            if (es == cudaSuccess) es = cub::DeviceScan::ExclusiveSum(d_tmp, tmp_bytes, d_wc, d_scan, (int)(nseq + 1));
            unsigned long long w = 0;
            if (es == cudaSuccess) es = cudaMemcpy(&w, d_scan + nseq, sizeof(w), cudaMemcpyDeviceToHost);
            if (es == cudaSuccess) es = dev_malloc(&s->d_pseq, nseq * sizeof(PackedSeq));
            if (es == cudaSuccess) {
                k_fill_pseq<<<(unsigned)((nseq + 255) / 256), 256>>>(s->d_off, nseq, s->d_kind, d_scan, s->d_pseq);
                es = cudaGetLastError();
            }
            cudaFree(d_tmp); cudaFree(d_wc);
            CUS(es);
            s->nwords = w;
            tr.mark("layout scan");
            CUS(dev_malloc(&s->d_words, (w + 16) * sizeof(uint32_t)));
            tr.mark("words alloc");    // slack: the rolling fetch of the last sequence runs a few words ahead
            k_pack<<<s->sm_count * 8, 256>>>(s->d_codes, s->d_off, nseq, s->d_kind, s->d_pseq, s->d_words);
            CUS(cudaGetLastError());
            CUS(cudaDeviceSynchronize());
            tr.mark("pack kernel");
        }
    }
    return BAMM_OK;
}

extern "C" int bamm_seqset_create(const uint8_t* codes, const uint64_t* offsets, uint64_t nseq, int A,
                                  const uint64_t* patch_pos, const uint64_t* patch_kmer, uint64_t npatch,
                                  bamm_seqset** out) {
    REQUIRE(out, "out is NULL");
    *out = nullptr;
    REQUIRE(codes && offsets, "codes/offsets is NULL");
    REQUIRE(npatch == 0 || (patch_pos && patch_kmer), "patch arrays are NULL");
    bamm_seqset* s = nullptr;
    Trace tr("seqset_create");
    // uploads on the copy stream: offsets, bases, then the patch list; the host pass over the offsets, the classification of
    // the bases and the patch checks (on the device: 11 entries per both-strand sequence) start as soon as their input is there
    { int rc = seqset_new(offsets, nseq, A, &s, codes); if (rc) return rc; }
    tr.mark("alloc + host checks (uploads in flight)");
    s->npatch = npatch;
    if (npatch) {
        CUS(dev_malloc(&s->d_ppos, npatch * sizeof(uint64_t)));
        CUS(dev_malloc(&s->d_pkmer, npatch * sizeof(uint64_t)));
        CUS(cudaMemcpyAsync(s->d_ppos, patch_pos, npatch * sizeof(uint64_t), cudaMemcpyHostToDevice, s->copy_stream));
        CUS(cudaMemcpyAsync(s->d_pkmer, patch_kmer, npatch * sizeof(uint64_t), cudaMemcpyHostToDevice, s->copy_stream));
    }
    CUS(cudaEventRecord(s->ev_patches, s->copy_stream));
    { int rc = seqset_finish(s, false, true); if (rc) return rc; }
    seqset_copy_done(s);                           // the caller's buffers are free again
    tr.mark("uploads + classify + pack");
    *out = s;
    return BAMM_OK;
}
#undef CUS

extern "C" void bamm_seqset_destroy(bamm_seqset* s) {
    if (!s) return;
    for (auto& kv : s->replicas) bamm_seqset_destroy(kv.second);
    s->replicas.clear();
    cudaSetDevice(s->device);
    for (auto& kv : s->index) cudaFree(kv.second.d);
    for (auto& kv : s->ypatch) cudaFree(kv.second);
    cudaFree(s->d_kind); cudaFree(s->d_pseq); cudaFree(s->d_words); cudaFree(s->d_zero_pos);
    seqset_copy_done(s);
    cudaFree(s->d_codes); cudaFree(s->d_off); cudaFree(s->d_ppos); cudaFree(s->d_pkmer);
    delete s;
}

extern "C" int bamm_seqset_info(const bamm_seqset* s, uint64_t* nseq, uint64_t* npos, int* A) {
    REQUIRE(s, "seqset is NULL");
    if (nseq) *nseq = s->nseq;
    if (npos) *npos = s->npos;
    if (A) *A = s->A;
    return BAMM_OK;
}

static int seqset_index_locked(bamm_seqset* s, int K, IndexArray** out) {
    REQUIRE(K >= 0 && K <= 10, "order K=%d not in [0,10]", K);   // the reference hashes at most 11-mers (Sequence.cpp:36)
    auto it = s->index.find(K);
    if (it != s->index.end()) { if (out) *out = &it->second; return BAMM_OK; }
    const uint64_t Yn = ipow_u64((uint64_t)s->A, K + 1);
    REQUIRE(Yn <= (1ull << 31), "A^(K+1) too large");
    IndexArray ia; ia.Yn = Yn; ia.bytes = (Yn <= 65536) ? 2 : 4;
    CU(cudaSetDevice(s->device));
    CU(dev_malloc(&ia.d, (s->npos ? s->npos : 1) * (uint64_t)ia.bytes));
    const int block = 256;
    const int grid = s->sm_count * 8;
    with_index_mut(ia, [&](auto Y) {
        if (s->nseq) k_build_index<<<grid, block>>>(s->d_codes, s->d_off, s->nseq, s->A, K, Yn, Y);
        if (s->npatch) k_patch_index<<<(int)((s->npatch + 255) / 256), 256>>>(s->d_ppos, s->d_pkmer, s->npatch, Yn, Y);
    });
    cudaError_t e = cudaDeviceSynchronize();
    if (e == cudaSuccess) e = cudaGetLastError();
    if (e != cudaSuccess) { cudaFree(ia.d); return fail(BAMM_E_CUDA, "index build failed: %s", cudaGetErrorString(e)); }
    auto ins = s->index.emplace(K, ia);
    if (out) *out = &ins.first->second;
    return BAMM_OK;
}

extern "C" int bamm_seqset_index(bamm_seqset* s, int K) {
    REQUIRE(s, "seqset is NULL");
    std::lock_guard<std::mutex> g(s->mu);
    return seqset_index_locked(s, K, nullptr);
}

// per-order k-mer index at the K+1 positions after the structural N of every kind-2 sequence
static int seqset_ypatch_locked(bamm_seqset* s, int K, uint16_t** out) {
    auto it = s->ypatch.find(K);
    if (it != s->ypatch.end()) { *out = it->second; return BAMM_OK; }
    const uint64_t Yn = ipow_u64(4, K + 1);
    REQUIRE(Yn <= 65536, "order too high for the packed path");
    uint16_t* d = nullptr;
    CU(cudaSetDevice(s->device));
    const uint64_t bytes = (s->nseq ? s->nseq : 1) * (uint64_t)(K + 1) * sizeof(uint16_t);
    CU(dev_malloc(&d, bytes));
    CU(cudaMemset(d, 0, bytes));
    if (s->npatch) {
        k_make_ypatch<<<(unsigned)((s->npatch + 255) / 256), 256>>>(s->d_ppos, s->d_pkmer, s->npatch, s->d_off, s->nseq, s->d_kind, K, Yn, d);
        cudaError_t e = cudaDeviceSynchronize();
        if (e != cudaSuccess) { cudaFree(d); return fail(BAMM_E_CUDA, "ypatch build failed: %s", cudaGetErrorString(e)); }
    }
    s->ypatch[K] = d;
    *out = d;
    return BAMM_OK;
}

extern "C" int bamm_seqset_get_index(bamm_seqset* s, int K, uint32_t* out) {
    REQUIRE(s && out, "NULL argument");
    IndexArray* ia;
    { std::lock_guard<std::mutex> g(s->mu); int rc = seqset_index_locked(s, K, &ia); if (rc) return rc; }
    CU(cudaSetDevice(s->device));
    if (ia->bytes == 4) { CU(cudaMemcpy(out, ia->d, s->npos * 4, cudaMemcpyDeviceToHost)); return BAMM_OK; }
    std::vector<uint16_t> tmp(s->npos);
    CU(cudaMemcpy(tmp.data(), ia->d, s->npos * 2, cudaMemcpyDeviceToHost));
    for (uint64_t i = 0; i < s->npos; i++) out[i] = tmp[i];
    return BAMM_OK;
}

extern "C" int bamm_seqset_count_kmers(bamm_seqset* s, int K, uint64_t* n_all) {
    REQUIRE(s && n_all, "NULL argument");
    IndexArray* ia;
    { std::lock_guard<std::mutex> g(s->mu); int rc = seqset_index_locked(s, K, &ia); if (rc) return rc; }
    CU(cudaSetDevice(s->device));
    unsigned long long* d_cnt;
    CU(dev_malloc(&d_cnt, ia->Yn * 8));
    CU(cudaMemset(d_cnt, 0, ia->Yn * 8));
    if (s->npos) {
        const uint32_t Yn = (uint32_t)ia->Yn;
        const bool smem = ia->Yn <= 12288 && s->npos / ((uint64_t)s->sm_count * 8) < 0xffffffffull;     // 48 KB of 32-bit bins
        const size_t sh = smem ? (size_t)Yn * 4 : 0;
        const int grid = s->sm_count * 8;
        with_index(*ia, [&](auto Y) {
            using YT = std::decay_t<decltype(*Y)>;
            (smem ? k_count_kmers<YT, true> : k_count_kmers<YT, false>)<<<grid, 256, sh>>>(Y, s->npos, Yn, d_cnt);
        });
    }
    std::vector<uint64_t> top(ia->Yn);
    cudaError_t e = cudaMemcpy(top.data(), d_cnt, ia->Yn * 8, cudaMemcpyDeviceToHost);
    cudaFree(d_cnt);
    if (e != cudaSuccess) return fail(BAMM_E_CUDA, "k-mer count failed: %s", cudaGetErrorString(e));
    // every position contributes once to every order and y_{k-1} = y_k % A^k, so lower orders are folds
    std::vector<uint64_t> off(K + 2, 0);
    for (int k = 0; k <= K; k++) off[k + 1] = off[k] + ipow_u64(s->A, k + 1);
    memset(n_all, 0, off[K + 1] * sizeof(uint64_t));
    memcpy(n_all + off[K], top.data(), ia->Yn * 8);
    for (int k = K; k > 0; k--) {
        const uint64_t Yk = ipow_u64(s->A, k), Yk1 = Yk * s->A;
        for (uint64_t y = 0; y < Yk1; y++) n_all[off[k - 1] + y % Yk] += n_all[off[k] + y];
    }
    return BAMM_OK;
}

// The entry points, by subject (one translation unit; the order matters: later parts use the helpers of earlier ones)
#include "capi_em.inl"
#include "capi_group.inl"
#include "capi_negatives.inl"
#include "capi_score.inl"
#include "capi_fasta.inl"
#include "capi_scan.inl"
