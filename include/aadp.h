/* include/aadp.h -- C ABI of the B200-native DP-fill library (libaadp.so).
 *
 * Drop-in boundary for ONE path of christang/alignment-algos: the dynamic-programming matrix
 * fill of dpmatrix.{h,cpp} (forward + reverse, global + local), the optimal tracebacks of
 * optimal.h / optimal_rev.h and the near-optimal cell set the enumerators of ucw.h / cw.h
 * consume -- plus the callers either side of it (SURVEY.md §8f): those two enumerators themselves,
 * sub-rectangle fills with optimal_subali.h for loop closure, and evaluators with tabulated
 * (position-dependent) gap penalties.  The reference has no FFI of its own (it is one C++ template library); the entry
 * points below are what its DPMatrix<S1,S2,Etype>::build() (dpmatrix.h:291-317) binds to when
 * the fill is moved to the GPU -- see INTEGRATION.md for the C++ side of the binding
 * (include/hmap2/dpmatrix.h is that binding, source compatible with the reference class).
 *
 * Conventions
 *   - plain pointers and sizes only; no C++/torch types cross this boundary;
 *   - sequences are residue CODES 0..A-1 without the '^'/'$' sentinels the reference adds
 *     (sequence.cpp:15-16); every matrix-shaped output is (Lq+2) x (Lt+2) row-major, index 0 =
 *     Head, last = Tail, exactly the reference's DPCell matrix (dpmatrix.h:250-259);
 *   - every function returns 0 on success, nonzero on error; aadp_last_error() returns a
 *     thread-local message (the C++ wrapper rethrows it as std::string like dpmatrix.h:361);
 *   - a context owns one device + one stream and is not shared between threads;
 *   - there is NO CPU fallback: without a CUDA device every compute call fails loudly.
 */
#ifndef AADP_H
#define AADP_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

typedef struct aadp_ctx aadp_ctx;

/* alib.h:20-26 (align_t) */
#define AADP_GLOBAL_LOCAL 0
#define AADP_GLOBAL 1
#define AADP_LOCAL_GLOBAL 2
#define AADP_LOCAL 3
#define AADP_SEMI_LOCAL 4

/* dpmatrix.h:23-26 (direction_t); 3 = both */
#define AADP_FWD 1
#define AADP_REV 2

/* aadp_set_scoring flags */
#define AADP_REPRO_REV_BUG 1u /* reproduce dpmatrix.h:868 (opt_j = t1_m1) -- the reference's behaviour */
/* aadp_fill_pair_general only.  In the reference the DPMatrix constructor's align_t alone selects the 0-clamp of the
 * local fills (dpmatrix.h:155, 310) while the evaluator's AliParams alone selects the free end gaps
 * (aasubalib.h:27-77); the two may disagree (e.g. a `global` constructor over semi_local AliParams).  These flags
 * override the clamp that `align_type` would imply. */
#define AADP_CLAMP_ON 2u   /* local (0-clamped) fill whatever align_type says */
#define AADP_CLAMP_OFF 4u  /* non-local fill whatever align_type says */

/* `what` bits of the batch calls */
#define AADP_W_FWD 1u    /* forward fill (build_forw[_local]_dpm_nonlinear_gaps, dpmatrix.h:356,538) */
#define AADP_W_REV 2u    /* reverse fill (build_rev[_local]_dpm_nonlinear_gaps, dpmatrix.h:691,879) */
#define AADP_W_TB 4u     /* keep bit-packed traceback (4 bit/cell) for every filled direction */
#define AADP_W_SCORES 8u /* keep the score matrices (needed by AADP_W_MASK and by local tracebacks) */
#define AADP_W_MASK 16u  /* near-optimal cell set {F+R-sim > thr} (ucw.h:141-180), needs FWD|REV */

/* ---- lifetime ------------------------------------------------------------------------- */
aadp_ctx* aadp_create(int device); /* NULL on failure (see aadp_last_error) */
void aadp_destroy(aadp_ctx* ctx);
const char* aadp_last_error(void);
const char* aadp_version(void);
/* Run all work of this context on an existing CUDA stream (cudaStream_t as void*), e.g. torch's
 * current stream, so that the caller's events bracket the kernels. NULL is the legacy default
 * stream; until this is called the context uses a private non-blocking stream.               */
int aadp_set_stream(aadp_ctx* ctx, void* cuda_stream);
int aadp_synchronize(aadp_ctx* ctx);
/* Tuning / test switches. "packed" (default 1): use the packed int16x2 kernels for every pair that
 * qualifies (Lt <= 512, |score| bound < 7000 units; local alignments unless the run asks for the near-optimal
 * cell set); 0 forces the int32 kernels.
 * "wave" / "wave_min_cells": multi-CTA wavefront for long pairs.  "host_threads": host scheduler
 * threads (0 = min(hardware, 8)).  "exact_float": see aadp_set_scoring.  "general_budget_mcells":
 * scratch budget (10^6 dense cells per direction, default 1000) of one chunk of an exact-float batch.  "general_prune" (default 1):
 * pruned candidate scans in the exact general-gap kernel (identical results; 0 = scan every candidate).
 * "general_threads" (default 256): CTA size limit of that kernel.  "general_records" (default 1): the record-list
 * kernel for affine gaps in exact-float mode (identical results at a cost per cell that does not grow with the
 * reference's scans; 0 = the scan kernel).  "ucw_user_limit" / "cw_user_limit": alignment limits of the
 * enumerators (<= 0 restores the reference's 100000 / 1000000).  "enum_mask_prune" (default 1): the enumeration kernel
 * tests only the deletion candidates that lie in the resident near-optimal set (same delta_ratio; identical results).                                          */
int aadp_set_option(aadp_ctx* ctx, const char* key, int value);

/* ---- scoring: replaces AASubstitutionEval(AliParams&, SubstitutionMatrix&) (aasubalib.h:14-15)
 * sub is A x A row-major, sub[q_code*A + t_code] == SubstitutionMatrix::score (submatrix.h:36-38).
 * gap(len) = gi + ge*(len-1) (aasubalib.h:37-38) with the per-align_type free end gaps of
 * aasubalib.h:27-77.  Two exactness classes, both BIT-EXACT against the reference:
 *   - sub, gi, ge on one dyadic grid (multiples of 2^-s, s<=8; integer matrices trivially are): the
 *     fast O(Lq*Lt) integer kernels (packed int16x2 / int32 / multi-CTA wavefront);
 *   - anything else (e.g. the reference defaults 4.73 / 0.34, alib.cpp:17-18): the exact general-gap
 *     fp32 path: every candidate of the reference's scans (dpmatrix.h:459-480) that can win is evaluated
 *     with the same fp32 operations in the same order and the first maximum in scan order is kept
 *     (record-list kernel for affine gaps, literal scans otherwise).  In this mode batches return per-pair scalars,
 *     aadp_batch_fetch_pair / aadp_batch_optimal recompute the requested pair, and no packed
 *     traceback is kept.  aadp_set_option("exact_float", 1) forces this class for any scoring.      */
int aadp_set_scoring(aadp_ctx* ctx, const float* sub, int A, float gi, float ge, int align_type,
                     uint32_t flags);

/* ---- single pair, dense reference-shaped outputs: replaces the DPMatrix constructor
 * (dpmatrix.h:147-165) + build() (dpmatrix.h:291-317).  direction: AADP_FWD, AADP_REV or 3.
 * Outputs (host pointers, any may be NULL), all (Lq+2)*(Lt+2):
 *   score_*          DPCell::score            prevq_* / prevt_*   DPCell::prev_query_idx / prev_template_idx
 *   nearopt          1 byte per cell, 1 where F+R-sim > threshold (needs direction 3, delta_ratio >= 0)
 *   threshold        min((1-delta_ratio)*opt, opt-0.1f)  (cw.h:86-88)                           */
int aadp_fill_pair(aadp_ctx* ctx, const uint8_t* q, int Lq, const uint8_t* t, int Lt,
                   int direction, float delta_ratio, float* score_fwd, int32_t* prevq_fwd,
                   int32_t* prevt_fwd, float* score_rev, int32_t* prevq_rev, int32_t* prevt_rev,
                   uint8_t* nearopt, float* threshold);

/* ---- sub-rectangle fill: replaces the 9-argument DPMatrix constructor + build_subdpm (dpmatrix.h:169-189,
 * 319-353; used by the loop-closure code of ssss.h:621,710).  The fill runs between the anchors
 * (q1_end, t1_end) and (q2_beg, t2_beg) (matrix indices, 0 = Head, L+1 = Tail); both anchor scores are 0,
 * cells outside the rectangle keep the DPCell defaults (score 0, predecessors -1).  Anchors that are ordinary
 * residues pay gap penalties and the final cell adds its real similarity, exactly as the reference does.
 * Always computed by an exact fp32 kernel (any scoring): the record-list kernel (frec_fill_kernel) by default, the
 * general-gap kernel (general_fill_kernel) with option general_records 0 or beyond the record-list kernel's limits (more
 * than 2048 interior columns, or 32 000 interior rows).  The rectangle alone picks the kernel and sizes its shared
 * memory, not the sequence lengths.
 * direction: AADP_FWD or AADP_REV.  Outputs are (Lq+2)*(Lt+2) host arrays, any may be NULL.               */
int aadp_fill_subpair(aadp_ctx* ctx, const uint8_t* q, int Lq, const uint8_t* t, int Lt, int q1_end,
                      int t1_end, int q2_beg, int t2_beg, int direction, float* score,
                      int32_t* prev_q, int32_t* prev_t);

/* ---- many sub-rectangle fills + their optimal sub-alignments in ONE call (SURVEY.md §8 row f4): the loop-closure
 * pattern of ssss.h:600-633,700-720 -- per loop a 9-argument DPMatrix (dpmatrix.h:169-189, build_subdpm :319-353)
 * followed by Optimal_Subali::enumerate (optimal_subali.h:59-83) -- for a whole list of loops.
 * Item k fills the rectangle rects[4k..4k+3] = (q1_end, t1_end, q2_beg, t2_beg) of query sequence item_q[k] against
 * template sequence item_t[k] (ids into residues/seq_off as in aadp_fill_batch; items may share sequences).  Each
 * item runs on an exact fp32 kernel as in aadp_fill_subpair, in COMPACT storage: only its rectangle lives on the
 * device, in HBM and in shared memory, not the (Lq+2)*(Lt+2) matrix around it, so loops of very long pairs fill too.
 * Items are launched in chunks (option general_budget_mcells); the widest rectangle of a chunk picks its kernel, and
 * every result is the same whatever chunk an item lands in.  direction: AADP_FWD or AADP_REV (REV: scores only).  Host outputs (any may be NULL):
 *   score    nitems: score of the final cell, D[q2_beg][t2_beg] (FWD, = AlignedPairList::score of
 *            optimal_subali.h:68) or D[q1_end][t1_end] (REV)
 *   ali_off  nitems+1: slot k is ali_off[k]..ali_off[k+1] = q2_beg-q1_end+1 aligned pairs (every traceback step lowers
 *            the query index); computed on the host -- call with every other output NULL to size `pairs`
 *   pairs    2*ali_off[nitems] ints (pairs_cap = capacity in aligned pairs): slot k holds n_out[k] (query_idx,
 *            template_idx) pairs front to back, from (q1_end, t1_end) to (q2_beg, t2_beg)
 *   status   0, or 3 where the reference throws "Illegal alignment start pair" (optimal_subali.h:80)          */
int aadp_fill_subpair_batch(aadp_ctx* ctx, const uint8_t* residues, const int64_t* seq_off, int64_t nseq,
                            const int32_t* item_q, const int32_t* item_t, const int32_t* rects, int64_t nitems,
                            int direction, float* score, int64_t* ali_off, int32_t* pairs, int64_t pairs_cap,
                            int32_t* n_out, int32_t* status);

/* ---- ANY Evaluator with a uniform affine gap model: the similarity matrix the reference builds on the host
 * (SimilarityMatrix, simmatrix.h:40-73: sim[i][j] = evaluator.similarity(q,t,i,j), after post_process) is handed
 * over as it is -- (Lq+2)*(Lt+2) floats, row-major -- together with gap(len) = gi + ge*(len-1) and the align
 * type that selects the free end gaps (aasubalib.h:27-77).  This is what DPMatrix<S1,S2,Etype>::build() /
 * build_subdpm() can bind to for every Etype whose gap functions have that form, without describing residues
 * or a substitution table (tests/cxx/refpatch_demo.cpp does exactly that to the UNMODIFIED reference headers).
 * rect: NULL for the whole matrix, or {q1_end, t1_end, q2_beg, t2_beg}.  Exact general-gap fp32 kernel; needs
 * no aadp_set_scoring.                                                                                    */
int aadp_fill_pair_general(aadp_ctx* ctx, const float* sim, int Lq, int Lt, float gi, float ge,
                           int align_type, uint32_t flags, int direction, const int* rect, float* score,
                           int32_t* prev_q, int32_t* prev_t);

/* ---- ANY Evaluator, position-dependent gap penalties included (SURVEY.md §8 row f3): the fill asks an Evaluator
 * (evaluator.h:20-147) for similarity(i,j), deletion(.,.,t1,t2) and insertion(q1,q2,t2-1,t2); the host tabulates
 * the three over every argument combination dpmatrix.h:356-1030 can pass and the exact general-gap kernel runs the
 * reference's own scan over the tables -- bit-exact for hmap_eval.h:63-117 (gi/ge = min over the two template
 * positions) and gn2_eval.h:99-158 (pairwise deletion table, per-position insertion) style models as well.
 * Requirements (all reference evaluators meet them): deletion ignores the query positions; insertion sees the query
 * only through q2-q1 except at the Head/Tail; both are 0 for adjacent positions.  sz1 = Lq+2, sz2 = Lt+2:
 *   sim      sz1*sz2   SimilarityMatrix (simmatrix.h:40-73)
 *   del_tab  sz2*sz2   [t1*sz2 + t2] = deletion(q, q+1, t1, t2) for 0 <= t1 < t2 <= Lt+1 (other entries unused)
 *   ins_tab  (Lq+1)*sz2  [len*sz2 + t2] = insertion(q1, q1+len+1, t2-1, t2), len = 0..Lq, t2 = 1..Lt+1, where
 *            t2 == 1 means q1 = Head (boundary column, dpmatrix.h:421) and t2 == Lt+1 means q1+len+1 = Tail
 *            (final cell, dpmatrix.h:520); any interior q1 for the other columns
 * include/hmap2/dpmatrix.h builds these tables for every Etype without a DeviceScoring mapping.             */
int aadp_fill_pair_tabulated(aadp_ctx* ctx, const float* sim, int Lq, int Lt, const float* del_tab,
                             const float* ins_tab, int is_local, uint32_t flags, int direction, float* score,
                             int32_t* prev_q, int32_t* prev_t);

/* The same for MANY pairs in one call (database search with a profile evaluator): item k has Lq[k] x Lt[k] positions
 * and its three tables at sim + sim_off[k], del_tab + del_off[k], ins_tab + ins_off[k] (offsets in floats, layouts as
 * above).  One CTA per (item, direction), chunked by the dense-scratch budget.  direction: AADP_FWD, AADP_REV or 3.
 * Host outputs (any may be NULL): fwd_score[k] = D[last][last] of the forward fill, rev_score[k] = D[0][0] of the
 * reverse fill, and -- non-local forward fills only -- the optimal alignment of every item traced on the GPU
 * (Optimal::enumerate, optimal.h:47-75): ali_off (n+1, slot k = Lq[k]+2 aligned pairs, computed on the host), pairs
 * (2*ali_off[n] ints), n_out, status (3 = "Illegal alignment start pair").                                      */
int aadp_fill_batch_tabulated(aadp_ctx* ctx, int64_t n, const int32_t* Lq, const int32_t* Lt, const float* sim,
                              const int64_t* sim_off, const float* del_tab, const int64_t* del_off,
                              const float* ins_tab, const int64_t* ins_off, int is_local, uint32_t flags,
                              int direction, float* fwd_score, float* rev_score, int64_t* ali_off, int32_t* pairs,
                              int64_t pairs_cap, int32_t* n_out, int32_t* status);

/* ---- batch of pairs, HOST buffers (the end-to-end call) ------------------------------------
 * residues: all sequences back to back; sequence s is residues[seq_off[s] .. seq_off[s+1]).
 * pair p aligns query pair_q[p] against template pair_t[p].
 * Per-pair host outputs (any may be NULL): fwd_score[p] = D[last][last].score of the forward
 * matrix, rev_score[p] = D[0][0].score of the reverse matrix, threshold[p], nearopt_count[p].
 * Traceback / score matrices / masks stay RESIDENT in HBM inside the context (they are tens of
 * GB for 100k pairs); fetch what is needed with aadp_batch_fetch_*.                           */
int aadp_fill_batch(aadp_ctx* ctx, const uint8_t* residues, const int64_t* seq_off, int64_t nseq,
                    const int32_t* pair_q, const int32_t* pair_t, int64_t npairs, uint32_t what,
                    float delta_ratio, float* fwd_score, float* rev_score, float* threshold,
                    int64_t* nearopt_count);

/* The same call in two halves, for a caller that wants to overlap batches WITHOUT threads: submit does the host
 * scheduling and enqueues every copy and kernel, wait returns when the results are in the caller's buffers (and
 * reports what submit could not know yet, e.g. a residue outside the alphabet).  With two contexts,
 *     submit(A, batch k); submit(B, batch k+1); wait(A); submit(A, batch k+2); wait(B); ...
 * the host schedules one batch while the GPU fills the other.  Between submit and wait only aadp_fill_batch_wait
 * may be called on that context, and the input and output buffers must stay untouched.                              */
int aadp_fill_batch_submit(aadp_ctx* ctx, const uint8_t* residues, const int64_t* seq_off, int64_t nseq,
                    const int32_t* pair_q, const int32_t* pair_t, int64_t npairs, uint32_t what,
                    float delta_ratio, float* fwd_score, float* rev_score, float* threshold,
                    int64_t* nearopt_count);
int aadp_fill_batch_wait(aadp_ctx* ctx);

/* Same work with inputs ALREADY RESIDENT in device memory and per-pair outputs left in device
 * memory (d_* are device pointers; may be NULL like above). Asynchronous on the context stream. */
int aadp_upload_batch(aadp_ctx* ctx, const uint8_t* residues, const int64_t* seq_off, int64_t nseq,
                      const int32_t* pair_q, const int32_t* pair_t, int64_t npairs, uint32_t what);
int aadp_run_batch(aadp_ctx* ctx, uint32_t what, float delta_ratio, float* d_fwd_score,
                   float* d_rev_score, float* d_threshold, int64_t* d_nearopt_count);

/* ---- all queries x all templates, forward score only (database-search / all-vs-all shape) ------
 * Replaces the caller-side double loop `for q: for t: DPMatrix<..>(q, t, eval, forward, type);
 * D[last][last].score` (aa_ali.cpp:74-90 run once per combination).  Sequences are uploaded once and
 * stay resident; each call scores the rectangle q_ids x t_ids (sequence ids, may repeat, may overlap):
 *   scores[i*nt + j] = forward optimum of query q_ids[i] against template t_ids[j].
 * Templates of 1..512 residues whose scores fit the packed int16 domain run on the cross-mode packed
 * kernel (one template profile shared by a group of query couples); every other combination is routed
 * through the general pair-list path (which replaces the resident pair batch of this context).
 * aadp_cross_run is asynchronous on the context stream and writes DEVICE memory (d_scores, nq*nt
 * floats); aadp_cross_scores is the host-buffer convenience call (upload + run + download).          */
int aadp_upload_sequences(aadp_ctx* ctx, const uint8_t* residues, const int64_t* seq_off, int64_t nseq);
int aadp_cross_run(aadp_ctx* ctx, const int32_t* q_ids, int64_t nq, const int32_t* t_ids, int64_t nt,
                   float* d_scores);
int aadp_cross_scores(aadp_ctx* ctx, const uint8_t* residues, const int64_t* seq_off, int64_t nseq,
                      const int32_t* q_ids, int64_t nq, const int32_t* t_ids, int64_t nt, float* scores);
/* Cell updates (sum of Lq*Lt over the rectangle) of the last aadp_cross_run. */
double aadp_last_cross_cell_updates(aadp_ctx* ctx);

/* Bytes of HBM the resident batch products occupy (0 if none). which: AADP_W_TB / _SCORES / _MASK */
int64_t aadp_batch_resident_bytes(aadp_ctx* ctx, uint32_t which);
/* Number of kernels launched by the last batch/pair call (for bench.py's gpu_launches). */
int64_t aadp_last_launch_count(aadp_ctx* ctx);
/* Bytes copied host->device / device->host by the last aadp_fill_batch / aadp_upload_batch call. */
int64_t aadp_last_h2d_bytes(aadp_ctx* ctx);
int64_t aadp_last_d2h_bytes(aadp_ctx* ctx);
/* Cell updates (sum of Lq*Lt per filled direction) of the last batch call. */
double aadp_last_cell_updates(aadp_ctx* ctx);

/* Per-launch device timing (CUDA events on the context stream around every kernel of the batch
 * calls). Off by default; aadp_set_profiling(ctx,1) clears the log and every following run appends
 * to it. aadp_profile_get returns the idx-th logged launch: kernel name, milliseconds and the
 * cell updates that launch processed (0 for helper kernels).                                  */
int aadp_set_profiling(aadp_ctx* ctx, int on);
int aadp_profile_count(aadp_ctx* ctx);
int aadp_profile_get(aadp_ctx* ctx, int idx, char* name, int name_cap, float* ms, double* cells);

/* Dense, reference-shaped view of pair p of the resident batch (same outputs as aadp_fill_pair;
 * requires the batch to have been run with the corresponding AADP_W_* bits).                    */
int aadp_batch_fetch_pair(aadp_ctx* ctx, int64_t p, float* score_fwd, int32_t* prevq_fwd,
                          int32_t* prevt_fwd, float* score_rev, int32_t* prevq_rev,
                          int32_t* prevt_rev, uint8_t* nearopt);

/* Optimal alignment of pair p, walked (on the host) over the packed traceback fetched from HBM: replaces
 * Optimal::enumerate (optimal.h:47-75) for direction AADP_FWD and Optimal_Rev::enumerate
 * (optimal_rev.h:47-78) for AADP_REV. pairs receives 2 ints (query_idx, template_idx) per
 * aligned pair in alignment order, including (0,0) and (last,last). Returns 3 with
 * "Illegal alignment start pair" when the reference would throw (optimal.h:74).  Local alignments: find_max +
 * enumerate_local (optimal.h:76-124, optimal_rev.h:79-131) over the dense view of the pair.       */
int aadp_batch_optimal(aadp_ctx* ctx, int64_t p, int direction, int32_t* pairs, int32_t max_pairs,
                       int32_t* npairs, float* score);

/* Optimal alignments of EVERY pair of the resident batch, traced on the GPU: one thread per pair follows
 * the packed traceback in HBM (Optimal::enumerate, optimal.h:47-75, for AADP_FWD; Optimal_Rev::enumerate,
 * optimal_rev.h:47-78, for AADP_REV).  Needs a batch run with AADP_W_TB.  Local alignments (align type local): one warp
 * per pair runs find_max + enumerate_local (optimal.h:76-124, optimal_rev.h:79-131) over the stored scores instead
 * (needs AADP_W_SCORES as well); status is always 0 there, as the reference never throws in that mode.
 * Exact-float scoring (the reference defaults 4.73 / 0.34) keeps no resident traceback: there the forward, non-local
 * alignments of the whole batch are produced chunk by chunk (dense fill with predecessors, then one walk per pair);
 * the batch only has to be uploaded (any aadp_fill_batch / aadp_upload_batch).
 *   ali_off  host, npairs+1 (out, may be NULL): slot p is ali_off[p]..ali_off[p+1] = Lq+Lt+2 aligned pairs
 *   pairs    host, 2*ali_off[npairs] ints (may be NULL; pairs_cap = its capacity in aligned pairs): slot p holds
 *            n_out[p] (query_idx, template_idx) pairs front to back, including (0,0) and (last,last)
 *   status   host per pair: 0, or 3 where the reference throws "Illegal alignment start pair"           */
int aadp_batch_optimal_all(aadp_ctx* ctx, int direction, int64_t* ali_off, int32_t* pairs, int64_t pairs_cap,
                           int32_t* n_out, int32_t* status);
/* The same, COMPACT: ali_off (npairs+1, required) receives the offsets of the alignments packed one after the other
 * (ali_off[p+1] - ali_off[p] = n_out[p] aligned pairs), and only those pairs are copied back -- for 100 k pairs of the
 * C3 shape 28 MB instead of the 485 MB of the capacity-sized slots.  pairs_cap (in aligned pairs) must hold
 * ali_off[npairs]; the capacity total of aadp_batch_optimal_all is always enough.                               */
int aadp_batch_optimal_all_compact(aadp_ctx* ctx, int direction, int64_t* ali_off, int32_t* pairs, int64_t pairs_cap,
                                   int32_t* n_out, int32_t* status);

/* ---- near-optimal ENUMERATION of listed pairs of the resident batch on the GPU (SURVEY.md §8 row f1): replaces
 * UnconstrainedNearOptimal::enumerate / branch (ucw.h:63-191) up to, not including, its final sortSet.  One warp per
 * listed pair walks the Waterman branching depth first over the RESIDENT forward scores (no dense expansion); the
 * alignments come back in the reference's depth-first slot order with the reference's fp32 scores.  Needs a batch run
 * with AADP_W_FWD and (AADP_W_SCORES or AADP_W_MASK) on the integer (dyadic-grid) kernels; not for local alignments.
 * Host outputs (any may be NULL); K = max_alignments is the output budget per pair:
 *   n_ali      n: alignments emitted for listed pair k (<= K)
 *   status     n: 0; 1 = the pair has more than K alignments (the first K in depth-first order are returned; the
 *              reference itself stops branching at 100000, ucw.h:72,115-126)
 *   scores     n*K: AlignedPairList::score of alignment a of pair k at [k*K + a]
 *   ali_len    n*K: aligned pairs of that alignment, including (0,0) and (last,last)
 *   path_off   n+1 (computed on the host; call with every other output NULL to size `paths`): alignment a of pair k
 *              occupies paths[2*(path_off[k] + a*(Lq+2)) ...], (query_idx, template_idx) front to back; only the
 *              slots a < n_ali[k] are written
 *   threshold  n: min((1-delta_ratio)*opt, opt-0.1f) (ucw.h:81-83)                                                */
int aadp_batch_near_optimal(aadp_ctx* ctx, const int64_t* pair_ids, int64_t n, float delta_ratio,
                            int32_t max_alignments, int32_t* n_ali, int32_t* status, float* scores, int32_t* ali_len,
                            int64_t* path_off, int32_t* paths, int64_t paths_cap, float* threshold);

/* The constrained variant: ConstrainedNearOptimal::enumerate (cw.h:60-284) up to its final sortSet.  Branching is
 * restricted by SuboptFlags (cw.h:62-63, built per template position as nalign.cpp:84 does): after every accepted branch
 * the optimal predecessors are followed (opt_path, cw.h:213-281, here the packed traceback decoded on the fly) until
 * the flag of the template position changes state, and only there the candidates are scanned again.
 *   subopt_flags / flag_off: one byte per template position INCLUDING both sentinels for every listed pair, pair k at
 *   subopt_flags[flag_off[k] .. flag_off[k+1]) (Lt+2 bytes); subopt_flags == NULL means all true.
 * Needs AADP_W_TB in addition to what aadp_batch_near_optimal needs.  Outputs as above.                          */
int aadp_batch_near_optimal_constrained(aadp_ctx* ctx, const int64_t* pair_ids, int64_t n, const uint8_t* subopt_flags,
                                        const int64_t* flag_off, float delta_ratio, int32_t max_alignments,
                                        int32_t* n_ali, int32_t* status, float* scores, int32_t* ali_len,
                                        int64_t* path_off, int32_t* paths, int64_t paths_cap, float* threshold);

/* ---- the PRUNED near-optimal enumerators (SURVEY.md §8 row f2) of ONE pair of the resident batch:
 *   AADP_PRUNE_KSORTED     KSConstrainedNearOptimal::enumerate  (kscw.h:113-351): every branch point ranks its passing
 *                          predecessors by f + r - g and keeps the k_limit best (the best one keeps the budget, the
 *                          others continue with half of it)
 *   AADP_PRUNE_REDUNDANCY  CRConstrainedNearOptimal::enumerate  (crcw.h:134-594): ranked predecessors (at most sort_limit)
 *                          are extended along their optimal sub-paths to the next SuboptFlags region boundary; one that
 *                          shares more than max_overlap of an accepted sub-path is dropped
 * subopt_flags: Lt+2 bytes (sflags.h), NULL = all true.  k_limit / sort_limit / max_overlap / user_limit: the fields of
 * NOaliParams (noalib.cpp:16-22).  The batch must have been run with AADP_W_FWD | AADP_W_TB | AADP_W_SCORES.  Output: the
 * alignments in the reference's slot order BEFORE its final sortSet -- scores[k], ali_len[k], and the aligned pairs of
 * alignment k packed one after the other in `paths` (2 ints per pair, (0,0) first; paths_cap in pairs).  status: 0, or 1
 * when more than max_alignments alignments exist (the first max_alignments are returned).  The walk itself runs on the
 * host over the GPU-filled matrices of the pair (csrc/aadp_pruned.h): it is a short sequential recursion whose width the
 * pruning bounds.  Equal-score cuts are resolved by std::sort / std::partial_sort as in the reference.              */
#define AADP_PRUNE_KSORTED 2
#define AADP_PRUNE_REDUNDANCY 3
int aadp_batch_near_optimal_pruned(aadp_ctx* ctx, int64_t pair_id, int variant, const uint8_t* subopt_flags, float delta_ratio,
                                   uint32_t k_limit, uint32_t sort_limit, float max_overlap, uint32_t user_limit,
                                   int32_t max_alignments, int32_t* n_ali, int32_t* status, float* scores, int32_t* ali_len,
                                   int32_t* paths, int64_t paths_cap, float* threshold);

/* ---- packed traceback format helpers (host side, no GPU needed) ---------------------------
 * Row stride in bytes of the ROW-MAJOR packed traceback (int32 kernels) for template length Lt. */
int64_t aadp_tb_row_bytes(int Lt);
/* Bytes the packed traceback of pair p of the resident batch occupies (either layout).          */
int64_t aadp_batch_tb_bytes(aadp_ctx* ctx, int64_t p);
/* Decode one cell of a packed traceback fetched with aadp_batch_fetch_tb. (i,j) and the result
 * are reference matrix coordinates; direction selects the fwd or rev conventions.              */
int aadp_batch_fetch_tb(aadp_ctx* ctx, int64_t p, int direction, uint8_t* tb, int64_t tb_bytes,
                        int32_t* final_rec /* [6]: score units, kind, k, scale_log2, leading pad columns, layout class (0 = 8-column words, 1 = diagonal-major, 2 = 4-column nibble groups) */);
int aadp_decode_cell(const uint8_t* tb, int Lq, int Lt, int direction, int align_type,
                     uint32_t flags, const int32_t* final_rec, int i, int j, int32_t* prev_q,
                     int32_t* prev_t);

#ifdef __cplusplus
}
#endif
#endif /* AADP_H */
