/*
 * bamm_b200.h — C ABI of the B200-native EM-refinement / sequence-scoring path of BaMM!motif v2.
 *
 * The reference (soedinglab/BaMMmotif2) has no FFI: its hot path sits behind the public C++ classes
 * EM, ScoreSeqSet and FDR (SURVEY.md §8b). This header is the boundary a maintainer binds instead of
 * the bodies of those methods; the C++ mirror classes in bammmotif2_b200/host/ do exactly that and
 * INTEGRATION.md shows the binding. Everything is plain pointers and sizes; no torch / C++ types.
 *
 * Conventions
 *   - every function returns 0 (BAMM_OK) or a negative BAMM_E_* code; bamm_last_error() gives the text
 *     (thread-local). The C++ wrappers print it to stderr and exit(1), the reference's error convention
 *     (e.g. src/init/SequenceSet.cpp:144-149).
 *   - model tables are flat float arrays in the reference's index order:
 *       v_all   : for k=0..K, for y<A^(k+1), for j<W        (reference float*** Motif::v_[k][y][j], Motif.h:56)
 *       vbg_all : for k=0..K_bg_model, for y<A^(k+1)        (reference float**  BackgroundModel::v_[k][y])
 *       alpha   : [K+1][W]                                   (reference float**  Motif::A_[k][j])
 *   - r is indexed like EM::r_[n][i] (src/refinement/EM.h:48-52): i = L-W-p for window start p, zero for
 *     i >= L-W+1, L floats per sequence.
 *   - objects are re-entrant across host threads as long as each thread uses its own bamm_em
 *     (FDR::evaluateMotif runs folds concurrently, src/evaluation/FDR.cpp:37-38); a bamm_seqset is
 *     immutable after bamm_seqset_index() and may be shared.
 *   - there is NO CPU fallback: without a CUDA device every compute entry point fails with BAMM_E_CUDA.
 */
#ifndef BAMM_B200_H_
#define BAMM_B200_H_

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define BAMM_OK            0
#define BAMM_E_INVALID    -1   /* bad argument (message says which) */
#define BAMM_E_CUDA       -2   /* CUDA runtime error / no device */
#define BAMM_E_NOMEM      -3   /* device or host allocation failed */
#define BAMM_E_STATE      -4   /* call order violated (e.g. estep before set_model) */

typedef struct bamm_seqset bamm_seqset;   /* sequences resident in HBM: codes + per-order k-mer index arrays */
typedef struct bamm_em     bamm_em;       /* one EM problem: subset of a seqset, model, r, counts, workspaces */

/* ---- library / device ----------------------------------------------------------------------- */
int         bamm_version(void);                    /* 10000*major + 100*minor + patch */
const char* bamm_last_error(void);                 /* text of the last failure on this thread */
/* Limits of the device path (the reference has none of them; calls outside return BAMM_E_INVALID):
 *   motif width W (after --extend) in [1, BAMM_MAX_MOTIF_WIDTH] for EM, scoring and PWM sampling;
 *   model orders K, K_bg in [0, 10] (the reference hashes at most 11-mers, src/init/Sequence.cpp:36).
 * The packed 2-bit kernels (and the plans of bamm_plan_describe / bamm_bound_plan_describe) hold a window and its context in
 * one 32-base word, so they take W <= BAMM_MAX_PACKED_WIDTH. A wider motif always takes the index-array kernels, which walk its
 * columns in blocks of 32 (DESIGN.md §4.6). */
#define BAMM_MAX_MOTIF_WIDTH 63
#define BAMM_MAX_PACKED_WIDTH 32
int         bamm_device_count(int* count);
int         bamm_set_device(int device);           /* device used by objects created afterwards on this thread */
/* The column-group plan of the packed E-step for (W, K, K_bg) under a shared-memory budget, as plain numbers; host
 * arithmetic only, no device needed (the planner replaces the per-position loop bounds of EM::EStep, src/refinement/EM.cpp:149-196,
 * by table lookups; DESIGN.md "column groups"). out: [npass] then per pass {G, kd, fast, table_bytes, first column, end column,
 * is_first, is_last} followed by G x {col0, ncol, lo, shift, shift2, mask4, base, colmask}. npass = 0: no packed plan fits. */
int         bamm_plan_describe(int W, int K, int K_bg_model, int reduced, uint64_t table_budget_bytes, int32_t* out, uint64_t cap,
                               uint64_t* n_used);
/* The bound plan of the pruned E-step (DESIGN.md §4.1): groups of up to 6 bases whose tables, indexed by one base more, hold an
 * upper bound of the group's columns for window p and for window p+1 — what replaces the per-window product of EM::EStep
 * (src/refinement/EM.cpp:167-176) for the 95 % of windows that cannot matter. out: {G, kd, fast, table_bytes} followed by G x
 * {first column, columns, first base, shift, shift2, mask4, base}. G = 0: no plan (W + 1 bases do not fit one window word). */
int         bamm_bound_plan_describe(int W, int K, int K_bg_model, uint64_t table_budget_bytes, int32_t* out, uint64_t cap, uint64_t* n_used);
int         bamm_device_info(int* sm_count, int* cc_major, int* cc_minor, uint64_t* total_mem);
/* Device group: several devices of one box driven by ONE process (the reference parallelises EM::EStep / MStep over the
 * sequences with OpenMP, src/refinement/EM.cpp:148-149, 230; here the sequences are cut into one contiguous block per device).
 * After this call, EM objects created over a sequence set that lives on devices[0] span all devices of the group (large enough
 * subsets only): bamm_em_optimize / bamm_em_iterate / bamm_em_estep / bamm_em_mstep run every block on its device and exchange
 * the count tensor over NVLink peer memory; results are bit-identical to one device. n = 0 or 1 switches the group off.
 * Everything else (sequence sets, scoring, negative sampling, bamm_em_mask) stays on devices[0]. */
int         bamm_set_device_group(const int* devices, int n);
int         bamm_get_device_group(int* devices, int cap, int* n);

/* ---- sequence set  (replaces Sequence::kmer_ / getKmer(), src/init/Sequence.cpp:35-41, Sequence.h:56-58) ---- */
/*
 * codes   : stored codes exactly as Sequence::sequence_ holds them (0 = N, 1..A, 78 for a reverse-complemented N;
 *           both strands already laid out as fwd | 0 | revcomp, src/init/Sequence.cpp:10-14,91-99), all sequences
 *           concatenated.
 * offsets : nseq+1 prefix sums of the stored lengths L_n.
 * patch_* : the positions whose k-mer hash cannot be derived from `codes` because a code-0 base draws
 *           rand() % A per (position, order) pair (Sequence.cpp:38): global position index and the reference's
 *           full 11-mer hash kmer_[i] for it. Sorted by position, at most one entry per position. May be empty.
 */
int bamm_seqset_create(const uint8_t* codes, const uint64_t* offsets, uint64_t nseq, int A,
                       const uint64_t* patch_pos, const uint64_t* patch_kmer, uint64_t npatch,
                       bamm_seqset** out);
/* Builds (once; cached) the order-K index array y[i] = kmer_[i] % A^(K+1) on the device. */
int bamm_seqset_index(bamm_seqset* s, int K);
/* Copies the order-K index array back (npos entries, widened to uint32) — for bit-exact parity checks. */
int bamm_seqset_get_index(bamm_seqset* s, int K, uint32_t* out);
int bamm_seqset_info(const bamm_seqset* s, uint64_t* nseq, uint64_t* npos, int* A);
/* Background k-mer counts n[k][y] for k<=K over all positions (BackgroundModel.cpp:26-42); out: sum_k A^(k+1). */
int bamm_seqset_count_kmers(bamm_seqset* s, int K, uint64_t* n_all);
/* Stored codes / offsets of a set back on the host (npos bytes / nseq+1 entries) - sets created on the device. */
int bamm_seqset_get_codes(bamm_seqset* s, uint8_t* out);
int bamm_seqset_get_offsets(const bamm_seqset* s, uint64_t* out);
/*
 * Negative (background) set sampled ON THE DEVICE  (replaces SeqGenerator::sample_bgseqset_by_fold with genericNeg = false,
 * src/seq_generator/SeqGenerator.cpp:63-206, 285-348; called from src/refinement/mainBaMM.cpp:100-116 and FDR):
 * for every template — the sequences `subset[0..nsub)` of `pos` in that order, or all of them when subset is NULL (the driver
 * filters sequences shorter than the motif before sampling, mainBaMM.cpp:75-83) — `fold` single-stranded records of the same stored length, drawn from the set-wide
 * order-2 k-mer model rescaled by the template's own k-mer counts. The bases are BIT-IDENTICAL to the reference's: the
 * device re-creates the libc rand() stream after srand(seed) (the reference seeds 42, SeqGenerator.cpp:33-34) and jumps to
 * every record's first draw. Returns BAMM_E_STATE in the (about 1 in 10^7 records) case where the reference's own draw
 * sequence would diverge from one-draw-per-base; the caller then samples on the host.
 */
int bamm_seqset_sample_negatives(bamm_seqset* pos, const uint64_t* subset, uint64_t nsub, uint64_t fold, uint32_t seed,
                                 bamm_seqset** out);
/*
 * The same negative set sampled in shards (one process per GPU, every rank holds a contiguous block of the templates): the
 * set-wide k-mer counts are a sum over ranks (bamm_seqset_negative_kmer_counts gives this rank's A + A^2 + A^3 counters, orders
 * 0, 1, 2 concatenated; all-reduce them), and a rank's first record starts at draw `draw_offset` = fold * (stored bases of all
 * templates on earlier ranks). The concatenation of the shards is bit-identical to the set one device samples alone.
 */
int bamm_seqset_negative_kmer_counts(bamm_seqset* pos, const uint64_t* subset, uint64_t nsub, uint64_t* counts);
int bamm_seqset_sample_negatives_shard(bamm_seqset* pos, const uint64_t* subset, uint64_t nsub, uint64_t fold, uint32_t seed,
                                       uint64_t draw_offset, const uint64_t* global_counts, bamm_seqset** out);
/* draws [first, first+count) of rand() after srand(seed), computed on the device (test hook for the generator above) */
int bamm_rand_stream(uint32_t seed, uint64_t first, uint64_t count, int32_t* out);
void bamm_seqset_destroy(bamm_seqset* s);

/* ---- EM  (replaces EM::EStep/MStep/optimize/optimize_q, src/refinement/EM.cpp:62-259,505-519) -------------- */
/*
 * subset : indices into the seqset (NULL = all sequences, in order); the EM object sees exactly these sequences
 *          in this order (FDR training folds, src/evaluation/FDR.cpp:49-57). Every sequence must have L >= W
 *          (the reference filters shorter ones before EM, src/refinement/mainBaMM.cpp:75-83).
 * K_bg_model : order of the background model that will be passed to set_model; K_bg = min(K_bg_model, K) (EM.cpp:23).
 */
int bamm_em_create(bamm_seqset* s, const uint64_t* subset, uint64_t nsub, int W, int K, int K_bg_model,
                   bamm_em** out);
int bamm_em_set_model(bamm_em* em, const float* v_all, const float* vbg_all, const float* alpha, float q);
/* EM::EStep (EM.cpp:139-200): refreshes s = v[K]/vbg, r and the log likelihood. */
int bamm_em_estep(bamm_em* em, float* llh);
/* EM::MStep (EM.cpp:217-259): counts from r, fold to lower orders, Motif::updateV (Motif.h:95-136). */
int bamm_em_mstep(bamm_em* em);
/* EM::optimize_q (EM.cpp:505-519) from the r of the last E-step. */
int bamm_em_optimize_q(bamm_em* em, float* q);
/*
 * EM::optimize (EM.cpp:62-137) with the reference's stop rule: stop when sum|dv[K]| < epsilon, or the log
 * likelihood dropped after iteration 10, or max_iter (reference constants 0.01 / 1000, EM.h:62-63).
 * Traces may be NULL; when given they must hold max_iter floats. optimize_q != 0 re-estimates q during the
 * first five iterations (EM.cpp:99).
 */
int bamm_em_optimize(bamm_em* em, int optimize_q, float epsilon, int max_iter, int* iterations,
                     float* llh_trace, float* vdiff_trace, float* q_trace);
/*
 * EM::mask (src/refinement/EM.cpp:261-503, the "advanced EM" of --advanceEM; SURVEY.md §8 row f-4) without optimizeQ: one
 * order-0 E-step over all windows, the threshold that keeps the fraction f of them with the largest responsibility, then EM
 * over the kept windows with the stop rule of optimize(). The reference's quirks are kept (window p = 0 unscored in the first
 * phase, prior 0 for a kept window i = 0, r[0] divided once more per iteration). Afterwards get_model / get_counts / get_r /
 * llh describe the final state like after bamm_em_optimize. One device only.
 */
int bamm_em_mask(bamm_em* em, float f, float epsilon, int max_iter, int* iterations, float* llh, uint64_t* n_kept,
                 float* r_cutoff);
/* n_iter full iterations (E, M, update) back to back without a host round trip; for throughput runs. */
int bamm_em_iterate(bamm_em* em, int n_iter, float* llh_last, float* vdiff_last);
int bamm_em_get_model(bamm_em* em, float* v_all);              /* current v, all orders */
int bamm_em_get_counts(bamm_em* em, float* n_all);             /* n of the last M-step, all orders (EM::n_) */
int bamm_em_get_s(bamm_em* em, float* s);                      /* s[y][j] of the last E-step (Motif::getS) */
int bamm_em_get_q(bamm_em* em, float* q);
int bamm_em_get_r(bamm_em* em, uint64_t first, uint64_t count, float* out);  /* r of subset sequences [first, first+count), concatenated */
uint64_t bamm_em_r_size(const bamm_em* em);                    /* sum of L over the subset */
/* device time of the last estep / mstep+update call in milliseconds (CUDA events on the EM stream) */
int bamm_em_last_timing(bamm_em* em, float* estep_ms, float* mstep_ms);
/* device times of the last bamm_em_iterate call, summed over its iterations (CUDA events on the EM stream):
 * E-step kernel, M-step accumulation kernel, reduce + model update, and first-launch-to-last-completion. */
int bamm_em_loop_timing(bamm_em* em, int* iters, float* estep_ms, float* maccum_ms, float* update_ms, float* total_ms);
/* the E-step share of bamm_em_loop_timing by kernel of the pruned path (DESIGN.md §4.1): the windows over the N and the
 * truncated windows (k_emasked), the bound pass (k_ebound), the exact pass over the candidates (k_eexact, plus the dense
 * kernel when it ran). Without the pruned path the whole E-step is in exact_ms. */
int bamm_em_loop_timing_estep(bamm_em* em, float* masked_ms, float* bound_ms, float* exact_ms);
/* number of CUDA kernels this object has launched so far (E-step, M-step, reduce, update, table kernels) */
int bamm_em_launch_count(bamm_em* em, uint64_t* kernels);
/* how the last E-step of the packed path ran (diagnostics; synchronises the EM stream). The per-position loop of EM::EStep
 * (src/refinement/EM.cpp:149-196) is evaluated either for every window (dense) or, when the plan allows it, only for the
 * windows whose upper bound can reach the M-step's threshold (pruned; DESIGN.md §4.1). info[0] pruned path enabled for the
 * current model, [1] groups of the exact product, [2] groups of the bound (0: none), [3] the dense kernel ran in the last E-step
 * (always 1 when [0] is 0), [4] candidate windows listed by the bound pass of the last E-step, [5] windows in the active list,
 * [6] column passes of the exact plan, [7] the plain table rides in shared memory (0/1). */
int bamm_em_estep_info(bamm_em* em, uint64_t info[8]);
/* bound reuse of the pruned E-step (DESIGN.md §4.1; diagnostics, synchronises the EM stream): while the bound tables stay close
 * to those of the last full bound pass, only the windows that pass listed within BAMM_BOUND_SLACK bits of the threshold are
 * bounded again. info[0] reuse enabled for this object (0 with BAMM_NO_BOUND_REUSE), [1] full bound passes and [2] watch passes
 * since creation, [3] windows in the watch list, [4] the last E-step took the watch pass (0/1), [5] the watch list is valid.
 * *log2_drift: log2 of the last bound on how far the tables moved since the list was built (the watch pass needs < slack). */
int bamm_em_bound_reuse_info(bamm_em* em, uint64_t info[6], float* log2_drift);
void bamm_em_destroy(bamm_em* em);

/* ---- multi-GPU (sequences sharded over ranks, one process per GPU; SURVEY.md §8e) ---------------------------- */
/*
 * The per-iteration exchange is a SUM over ranks of the integer (fixed-point) count table and two integer
 * scalars (log likelihood, sum of r). The library exposes the device buffer that has to be summed; the host
 * plumbing (torch.distributed / NCCL) all-reduces it in place between the two halves of an iteration:
 *   bamm_em_estep_local + bamm_em_mstep_local  -> buffer holds this rank's partial sums (int64)
 *   <all-reduce SUM int64 over `words` elements at `dev_ptr`>
 *   bamm_em_finish_iteration                   -> fold / updateV / new s on every rank (bit-identical)
 * Integer sums are associative, so the result does not depend on the rank count or the reduction order.
 */
int bamm_em_exchange_buffer(bamm_em* em, void** dev_ptr, uint64_t* words);
/* Makes the EM object use caller-owned device memory (e.g. a torch tensor registered with NCCL) as its exchange buffer. */
int bamm_em_set_exchange_buffer(bamm_em* em, void* dev_ptr, uint64_t words);
int bamm_em_set_global_nseq(bamm_em* em, uint64_t nseq_all_ranks);   /* N in optimize_q's formula */
int bamm_em_estep_local(bamm_em* em);
int bamm_em_mstep_local(bamm_em* em);
/* With optimize_q == 0 and llh == vdiff == NULL the call only enqueues work (no host round trip). */
int bamm_em_finish_iteration(bamm_em* em, int optimize_q, float* llh, float* vdiff);
/*
 * NVLink peer exchange: instead of an external all-reduce, the M-step's reduction kernel writes this rank's sums directly
 * into every rank's receive buffer (CUDA-IPC mapped peer memory) and bamm_em_finish_iteration waits for all ranks on the
 * device. Call bamm_em_peer_alloc on every rank, exchange the 64-byte handles (any transport), pass all of them
 * (world x 64 bytes, rank order) to bamm_em_peer_attach; afterwards the iteration is
 *   bamm_em_estep_local ; bamm_em_mstep_local ; bamm_em_finish_iteration      (no collective call in between)
 * Every rank must run the same number of iterations. Up to 16 ranks on one NVLink domain.
 */
int bamm_em_peer_alloc(bamm_em* em, int rank, int world, void* ipc_handle_out /* 64 bytes */);
int bamm_em_peer_attach(bamm_em* em, const void* ipc_handles /* world * 64 bytes */);
/* time this rank's device spent waiting for the slowest rank before it could sum the exchanged counts (the per-iteration
 * all-reduce of EM::MStep's n, SURVEY.md §8e), summed over the iterations since the last reset, and the number of waits */
int bamm_em_peer_wait(bamm_em* em, int reset, double* total_ms, uint64_t* waits);
/* CUDA stream (cudaStream_t as void*) the EM object launches on, so callers can order collectives after it */
int bamm_em_stream(bamm_em* em, void** stream);

/* ---- scoring  (replaces ScoreSeqSet::calcLogOdds, src/seq_scoring/ScoreSeqSet.cpp:25-67) ------------------- */
/*
 * Scores every window start of every subset sequence with s = log(v[K]+1e-5) - log(vbg) (Motif::calculateLogS,
 * src/init/Motif.cpp:471-483; the table is built on the host with the same libm logf as the reference).
 * zoops[n] = max score, z[n] = first argmax (strict '>' scan, ScoreSeqSet.cpp:59-62), mops (nullable) =
 * all window scores, sum(L_n - W + 1) floats in sequence order.
 */
int bamm_score_logodds(bamm_seqset* s, const uint64_t* subset, uint64_t nsub, int W, int K, int K_bg_model,
                       const float* v_all, const float* vbg_all, float* zoops, uint64_t* z, float* mops);

/* ---- FASTA text -> sequence set on the device  (SURVEY.md §8 row f-3) ------------------------------------------ */
/*
 * Replaces the per-base work of SequenceSet::readFASTA / Sequence::Sequence / appendRevComp (src/init/SequenceSet.cpp:67-225,
 * src/init/Sequence.cpp:4-43, 91-99): the caller finds the lines of the file (headers stay on the host) and passes the raw
 * text; encoding through the alphabet tables (Alphabet.cpp:10-55), the forward | 0 | reverse-complement layout and the base
 * counts (SequenceSet.cpp:99-108) happen on the device. The k-mer hashes around undefined bases depend on libc rand() draws
 * (Sequence.cpp:35-41) and therefore come back from the host as the usual patch list:
 *     bamm_seqset_encode_text    -> set (not yet usable), base counts, number of forward undefined bases
 *     bamm_seqset_forward_zeros  -> their stored positions (unordered); the structural N of both-strand records is implied
 *     bamm_seqset_code_windows   -> the 21 stored codes around any positions (0xff outside [beg,end)), for the host's hashes
 *     bamm_seqset_finish_patches -> patch list in, set classified + packed and ready (destroyed on failure)
 */
typedef struct bamm_fasta_seg {     /* one sequence line of the file */
    uint64_t text_off;              /* first byte in `text` */
    uint32_t len;                   /* bytes of the line = bases (line terminator excluded, a '\r' counts like the reference counts it) */
    uint32_t rec;                   /* record index */
    uint64_t dst;                   /* bases of the record before this line */
} bamm_fasta_seg;
int bamm_seqset_encode_text(const char* text, uint64_t nbytes, const bamm_fasta_seg* segs, uint64_t nseg,
                            const uint64_t* offsets /* nrec+1 stored offsets */, const uint32_t* rec_L0 /* bases per record */,
                            uint64_t nrec, int single_strand, int A, const uint8_t* base2code /* [256] */,
                            const uint8_t* code2comp /* [256] */, uint64_t* base_counts /* [A] out */, uint64_t* n_forward_zeros,
                            bamm_seqset** out);
int bamm_seqset_forward_zeros(bamm_seqset* s, uint64_t* positions);
int bamm_seqset_code_windows(bamm_seqset* s, const uint64_t* pos, const uint64_t* beg, const uint64_t* end, uint64_t n,
                             uint8_t* windows /* [n][21] */);
int bamm_seqset_finish_patches(bamm_seqset* s, const uint64_t* patch_pos, const uint64_t* patch_kmer, uint64_t npatch);

/*
 * The sampling step of Motif::initFromPWM (src/init/Motif.cpp:236-299; SURVEY.md §8 row f-4): for every listed sequence the
 * posterior of the motif start under the order-0 odds `score[y][j] = v[0][y][j] / vbg[0][y]` (y < asize, the PWM's alphabet
 * size; k-mers are reduced modulo asize like the reference does), one site per sequence drawn like std::discrete_distribution
 * draws it from `uniforms[n]` (the caller takes them from std::mt19937 with std::generate_canonical<double,53>, in sequence
 * order), and the integer k-mer counts n[k][y][j] of the sampled sites for all orders k <= K (flat, the model's index order).
 * z_out (nullable): the sampled outcome per sequence, 0 = no motif, z = window start + 1.
 */
int bamm_seqset_sample_pwm_sites(bamm_seqset* s, const uint64_t* subset, uint64_t nsub, int W, int K, int asize,
                                 const float* score, float q, const double* uniforms, int32_t* n_all, uint64_t* z_out);

/* ---- score statistics  (SURVEY.md §8 row f-1) ---------------------------------------------------------------- */
/* Sorts n scores in place (host buffer in and out) with a device radix sort: the std::sort calls of FDR::calculatePR
 * (src/evaluation/FDR.cpp:161-162, 207-208) and ScoreSeqSet::calcPvalues (src/seq_scoring/ScoreSeqSet.cpp:85). */
int bamm_sort_scores(float* scores, uint64_t n, int descending);
/* ScoreSeqSet::calcPvalues (src/seq_scoring/ScoreSeqSet.cpp:70-126): p-value and e-value of every positive window score
 * against ALL negative window scores (sorted on the device; exponential tail for the best scores, linear interpolation
 * between neighbouring negatives otherwise). expf is the device's: results agree with the host's within a few ulp. */
int bamm_mops_pvalues(const float* neg_scores, uint64_t nneg, const float* pos_scores, uint64_t npos, uint64_t n_pos_sequences,
                      float* p_values, float* e_values);

/* device time (CUDA events on the scoring stream) of the scoring kernels of the last bamm_score_logodds call of this thread */
int bamm_score_last_timing(float* kernel_ms);

#ifdef __cplusplus
}
#endif
#endif /* BAMM_B200_H_ */
