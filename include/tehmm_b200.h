/*
 * tehmm_b200.h -- C ABI of libtehmm_b200.so, the B200 (sm_100a) replacement for
 * teHmm's multitrack-HMM hot path.
 *
 * The reference has no FFI of its own: its native layer is five Cython modules
 * whose Python-visible `def` functions take NumPy arrays.  The entry points
 * below are what a ctypes/cffi binding for those functions binds (the binding a
 * maintainer would add is shown in INTEGRATION.md).  Plain C: pointers, sizes,
 * scalars.  No torch / NumPy / C++ types appear in any signature.
 *
 * Two layers.
 *
 *  L0 "strict" entry points  (tehmm_strict_*): HOST pointers, float64, one
 *     sequence per call, caller owns every buffer -- a 1:1 replacement for
 *       _hmm._forward            /root/reference/_hmm.pyx:120-158
 *       _hmm._backward           /root/reference/_hmm.pyx:160-198
 *       _hmm._viterbi            /root/reference/_hmm.pyx:201-259
 *       _hmm._log_sum_lneta      /root/reference/_hmm.pyx:62-117
 *       _emission.fastAllLogProbs      /root/reference/_emission.pyx:20-144
 *       _emission.fastAccumulateStats  /root/reference/_emission.pyx:146-234
 *       _emission.fastUpdateCounts     /root/reference/_emission.pyx:236-332
 *     They run CUDA kernels that keep the reference's operation order in fp64
 *     (including every quirk listed in SURVEY.md section 8a / Appendix).
 *
 *  L1 "batched" entry points (tehmm_set_model / tehmm_set_batch / tehmm_run_* ):
 *     DEVICE pointers, many sequences per call, chunked parallel-in-time
 *     scaled-space kernels in fp32 (production) or fp64 (verification).  They
 *     back MultitrackHmm.fit / decode / score / score_samples
 *     (/root/reference/hmm.py:155-277,545-729, basehmm.py:238-541) and
 *     IndependentMultinomialEmissionModel.allLogProbs / accumulateStats
 *     (/root/reference/emission.py:179-241).
 *
 * Error handling: every function returns 0 on success or a negative
 * TEHMM_E* code; tehmm_last_error() returns a thread-local message.  The
 * Python layer maps TEHMM_EINVAL to AssertionError (the reference asserts on
 * bad shapes, _emission.pyx:24-32) and everything else to RuntimeError.
 *
 * Threading: a context is bound to one device and one CUDA stream; calls on one
 * context must be serialised by the caller; distinct contexts may be used from
 * distinct threads (teHmmTrain --reps uses a ThreadPool, teHmmTrain.py:279-292).
 * Nothing here is stored on Python model objects (they are pickled and
 * deep-copied, modelIO.py:26-32, hmm.py:694).
 */
#ifndef TEHMM_B200_H
#define TEHMM_B200_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define TEHMM_ABI_VERSION 1

#define TEHMM_OK 0
#define TEHMM_EINVAL (-1)   /* bad argument / shape (reference: AssertionError) */
#define TEHMM_ECUDA (-2)    /* CUDA runtime error */
#define TEHMM_ENOMEM (-3)   /* host or device allocation failed */
#define TEHMM_ESTATE (-4)   /* call order (no model / no batch / workspace too small) */
#define TEHMM_ELIMIT (-5)   /* shape outside the supported envelope */

/* element type of the batched lattices */
#define TEHMM_F32 0
#define TEHMM_F64 1

/* tehmm_run_backward output selection (bit mask) */
#define TEHMM_BWD_POSTERIORS 1   /* write T x N posteriors                        */
#define TEHMM_BWD_MAP 2          /* write argmax-posterior states + sum of maxima   */
#define TEHMM_BWD_TRANS 4        /* accumulate start / transition expected counts   */
#define TEHMM_BWD_RENORM_EPS 8   /* score_samples tail: += float32 eps, /= row sum  */

#define TEHMM_MAX_STATES 64      /* batched path; strict path has no limit */

typedef struct tehmm_ctx tehmm_ctx;

int tehmm_abi_version(void);
const char *tehmm_last_error(void);
int tehmm_device_count(void);

int tehmm_ctx_create(int device, tehmm_ctx **out);
int tehmm_ctx_destroy(tehmm_ctx *ctx);
/* block until everything enqueued on the context's stream has finished */
int tehmm_ctx_sync(tehmm_ctx *ctx);
/* run on a caller-owned cudaStream_t (e.g. torch's current stream) so that the
 * caller's allocations, copies and events are ordered with the kernels.
 * 0 is the CUDA legacy default stream; UINT64_MAX = back to the context's own
 * (non-blocking) stream */
int tehmm_ctx_set_stream(tehmm_ctx *ctx, uint64_t stream);
/* the context's cudaStream_t as an integer (for event timing by the caller) */
uint64_t tehmm_ctx_stream(tehmm_ctx *ctx);
/* number of kernels this context has launched since creation */
int64_t tehmm_ctx_launch_count(tehmm_ctx *ctx);
/* options: "chunk_tiles" (tiles of 64 steps per chunk, 0 = auto),
 * "warmup" (speculative warm-up steps, 0 = auto), "max_repair" (passes),
 * "tile" (0 = never use the tensor-core tile kernels), "fine_len" (steps per
 * chunk of the fine partition, 0 = auto), "umma" (1 / 2 = forward pass of a
 * single-sequence batch of <= 32 states by the tcgen05 / tensor-memory kernel of
 * csrc/umma.cu with one / two threads per chunk; same results, 0.84 / 0.80 ms per
 * 10 M steps against 0.54 ms for the mma.sync kernel there),
 * "umma64" (default 1: the same kernel, 64 columns, and its backward twin ARE the
 * forward and the backward / posterior / MAP pass of single-sequence batches of
 * 33..64 states; 0 = one chunk per warp; stat "umma_passes" counts the launches
 * of any of them), "xi_tile" (0 = expected transition
 * counts by the one-chunk-per-warp backward kernel instead of the tensor-core
 * xi kernel), "timing" (1 = bracket the first
 * launch of each main kernel with CUDA events on the context's stream), "defer" (see
 * tehmm_ctx_check), "bwd_tmap" (1 = the regular tiles of a single-sequence batch take the
 * tensor-map block kernel in the backward pass; experimental: bit-identical results, not faster),
 * "fallback_after" (ordinary repair passes before the chunks still flagged are resolved exactly by
 * transfer operators and a float64 chain, csrc/fallback.cu; default 2, -1 = never: the plain loop, one
 * pass per link of a chain of failed boundaries; stats "fallbacks", "fallback_chunks", "mix_rho_ppm").
 * stats: "launches", "chunks", "fine_chunks", "repaired_chunks_<pass>",
 * "repair_passes_<pass>", "tile_passes", and with "timing" the mean duration in
 * microseconds (over the launches since "timing" was set, at most 32) of "us_emission", "us_forward", "us_backward",
 * "us_viterbi_dp", "us_traceback", "us_rescore", "us_emission_stats", "us_xi" launch
 * (blocks until that launch has finished; -1 if it never ran). */
int tehmm_ctx_set_option(tehmm_ctx *ctx, const char *name, int64_t value);
int64_t tehmm_ctx_get_stat(tehmm_ctx *ctx, const char *name);
/* Deferred verification.  With option "defer" = 1 the tehmm_run_* calls do not stall the
 * stream after each stage to read how many chunk boundaries failed verification (the
 * speculate / verify / repair scheme that replaces the serial recursions of
 * _hmm.pyx:120-259): the count goes to a pinned slot behind the queued kernels and the
 * call carries on as if nothing had to be repaired.  tehmm_ctx_check waits for the stream
 * and returns in *unverified the number of failed boundaries since the last check: 0 =
 * every result stands (the common case); > 0 = recompute those results with "defer" = 0
 * (tehmm_decode_host does both steps itself).  Stats: "deferred_checks", "deferred_bad". */
int tehmm_ctx_check(tehmm_ctx *ctx, int64_t *unverified);

/* ------------------------------------------------------------------ L0 strict
 * obs is (T,K) row-major, obs_bytes = 1 (uint8), 2 (uint16) or 4 (int32)
 * (the three dtype clones of _emission.pyx).  table is (K,N,S) float64,
 * [track][state][symbol].  ratios is NULL for segRatios=None.              */
int tehmm_strict_all_log_probs(tehmm_ctx *ctx, const void *obs, int obs_bytes,
                               int64_t T, int K, const double *table, int N, int S,
                               double *out /*T*N*/, double normalize,
                               const double *ratios /*T or NULL*/);
int tehmm_strict_forward(tehmm_ctx *ctx, int64_t T, int N, const double *log_start,
                         const double *log_trans, const double *frame,
                         const double *ratios, double *fwd /*T*N out*/);
int tehmm_strict_backward(tehmm_ctx *ctx, int64_t T, int N, const double *log_start,
                          const double *log_trans, const double *frame,
                          const double *ratios, double *bwd /*T*N out*/);
int tehmm_strict_viterbi(tehmm_ctx *ctx, int64_t T, int N, const double *log_start,
                         const double *log_trans, const double *ratios,
                         const double *frame, int64_t *states /*T out*/,
                         double *logprob /*out*/);
int tehmm_strict_log_sum_lneta(tehmm_ctx *ctx, int64_t T, int N, const double *fwd,
                               const double *log_trans, const double *bwd,
                               const double *frame, double logprob,
                               const double *ratios, double *out /*N*N in: zeros, out*/);
int tehmm_strict_accumulate_stats(tehmm_ctx *ctx, const void *obs, int obs_bytes,
                                  int64_t T, int K, double *stats /*K*N*S in-out*/,
                                  int N, int S, const double *post /*T*N*/,
                                  const double *ratios);
int tehmm_strict_update_counts(tehmm_ctx *ctx, const void *obs, int obs_bytes,
                               int64_t T, int K, int64_t start, int64_t end, int state,
                               double *stats /*K*N*S in-out*/, int N, int S,
                               const double *ratios);
/* Supervised counts of every labelled interval in one device pass.  d_obs is a
 * DEVICE (total, K) matrix in the layout of tehmm_set_batch's d_obs (the
 * concatenated tables); no model or batch needs to be set.  Interval i covers
 * the global rows [h_row_start[i], h_row_end[i]) with state h_state[i]; the
 * weight of row r is d_ratios[r] (DEVICE, total entries) or 1.0 when d_ratios
 * is NULL.  h_stats (HOST, K*N*S, in-out) ends bit for bit as after one
 * tehmm_strict_update_counts per interval in the given order: every bin is
 * init + w_1 + w_2 + ... in sequential float64 adds, interval order, positions
 * ascending.  Intervals may overlap (counted again) and come in any order;
 * empty ones are no-ops.  With unit weights and integer initial values the
 * counts are integer histograms (order-free, exact); otherwise every bin is
 * summed as one ordered chain.  The kernel launches do not depend on n.
 * TEHMM_EINVAL, with h_stats untouched, for a row outside [0, total), a state
 * outside [0, N), obs_bytes not 1, 2 or 4, or a counted symbol >= S.         */
int tehmm_supervised_counts(tehmm_ctx *ctx, const void *d_obs, int obs_bytes, int64_t total, int K,
                            int64_t n, const int64_t *h_row_start, const int64_t *h_row_end,
                            const int32_t *h_state, const double *d_ratios /* total, or NULL */,
                            double *h_stats /* K*N*S, in-out */, int N, int S);

/* ----------------------------------------------------------------- L1 batched
 * Model: HOST pointers (small).  log_start (N), log_trans (N,N), table (K,N,S)
 * as stored by the reference (hmm.py:625-666, emission.py:43-44,136-159);
 * track_nsym[k] = number of table columns in use for track k (<= S), or NULL
 * for "all S".  normalize = emission.normalizeFac (emission.py:58-60).      */
int tehmm_set_model(tehmm_ctx *ctx, int N, int K, int S, const double *log_start,
                    const double *log_trans, const double *table, double normalize,
                    const int32_t *track_nsym);

/* Batch: nseq sequences concatenated along time.  d_obs is a DEVICE pointer to
 * (total,K) symbols; h_offsets is a HOST array of nseq+1 row offsets.  The
 * pointer must stay valid until the next tehmm_set_batch.                    */
int tehmm_set_batch(tehmm_ctx *ctx, const void *d_obs, int obs_bytes, int64_t nseq,
                    const int64_t *h_offsets);
int64_t tehmm_batch_total(tehmm_ctx *ctx);  /* total rows */
/* Row stride LD (in elements) of every batched lattice below -- d_elog, d_blin,
 * d_alpha, d_post and the Viterbi workspace are (total, LD) row-major with the
 * states in columns 0..N-1 and zero padding after them.  LD = 32 for N <= 32
 * (one 128-byte line per float32 row, 16-byte aligned for vector and bulk
 * copies), N otherwise.  Valid after tehmm_set_model.                         */
int tehmm_lattice_stride(tehmm_ctx *ctx);
int64_t tehmm_batch_chunks(tehmm_ctx *ctx); /* chunks in the time partition */
/* bytes of d_scratch the tehmm_run_* calls need for the current batch+model */
int64_t tehmm_scratch_bytes(tehmm_ctx *ctx, int prec);

/* Emission gather-and-sum (emission.py:179-198 -> _emission.pyx:50-80).
 * Writes, per row t: M[t] = max_j frame[t][j] (float64) and, when non-NULL,
 *   d_elog[t][j] = frame[t][j] - M[t]            (log space, <= 0)
 *   d_blin[t][j] = exp(frame[t][j] - M[t])       (linear,   <= 1)
 * in the element type `prec`.  d_ratios (DEVICE, float64, total) or NULL.     */
int tehmm_run_emission(tehmm_ctx *ctx, int prec, const double *d_ratios,
                       void *d_elog, void *d_blin, double *d_rowmax);
/* The same for the rows [row0, row1) of the batch only, so that a caller streaming the
 * observations onto the device can run the rows that have arrived.  Pieces must come in
 * increasing order, the first starting at row 0 and the last ending at the batch's
 * total (the fix-up of _emission.pyx:59,73-80 runs then); row0 must be a multiple of
 * 32.  stream: the cudaStream_t to enqueue on, or UINT64_MAX for the context's.
 * Only when tehmm_emission_rows_supported() returns 1 (fp32, N <= 32, merged tables). */
int tehmm_emission_rows_supported(tehmm_ctx *ctx, int prec);
int tehmm_run_emission_rows(tehmm_ctx *ctx, int prec, const double *d_ratios, void *d_elog,
                            void *d_blin, double *d_rowmax, int64_t row0, int64_t row1,
                            uint64_t stream);
/* Reference-layout frame: d_frame[t][j] float64 = what fastAllLogProbs writes */
int tehmm_run_emission_f64(tehmm_ctx *ctx, const double *d_ratios, double *d_frame);

/* Forward (hmm.py:678-713 -> _hmm.pyx:120-158).  d_alpha (total*LD, may be NULL
 * for score-only) receives the per-step max-normalised forward vector;
 * d_logprob (nseq, float64) the sequence log-likelihoods.                    */
int tehmm_run_forward(tehmm_ctx *ctx, int prec, const void *d_blin,
                      const double *d_rowmax, const double *d_ratios, void *d_alpha,
                      double *d_logprob, void *d_scratch);

/* Backward + posterior glue + expected counts (hmm.py:715-729,545-574,
 * basehmm.py:265-272,516-517, _hmm.pyx:62-117,160-198).  flags = TEHMM_BWD_*.
 *   d_post        total*LD, element type prec           (POSTERIORS)
 *   d_map_states  total, uint8;  d_map_score nseq f64   (MAP)
 *   d_start_trans N + N*N float64, ACCUMULATED into     (TRANS)             */
int tehmm_run_backward(tehmm_ctx *ctx, int prec, int flags, const void *d_blin,
                       const void *d_alpha, const double *d_ratios, void *d_post,
                       uint8_t *d_map_states, double *d_map_score,
                       double *d_start_trans, void *d_scratch);

/* Posterior-weighted emission histograms (emission.py:221-241 ->
 * _emission.pyx:171-190): d_obs_stats (K,N,stats_S) float64, ACCUMULATED into.
 * stats_S is the width of the caller's obsStats array (initStats gives
 * max(numSymbolsPerTrack)+1, emission.py:212-214, which differs from the table
 * width S when zeroAsMissingData is off).                                    */
int tehmm_run_emission_stats(tehmm_ctx *ctx, int prec, const void *d_post,
                             const double *d_ratios, double *d_obs_stats,
                             int stats_S, void *d_scratch);

/* Viterbi with traceback (hmm.py:668-676 -> _hmm.pyx:201-259).
 * d_states total uint8 (required), d_states64 total int64 (optional, NULL to
 * skip), d_logprob nseq float64: the reference's viterbi_lattice[T-1, argmax]
 * (_hmm.pyx:252-254).  Where the fp32 production DP runs (<= 32 states, no DP
 * ratios) and d_rowmax (tehmm_run_emission's output; may be NULL) is given, it is
 * the DP's own value -- the row maxima it takes out, summed in float64 across
 * steps, plus rowmax; otherwise, and always with context option "rescore" = 1,
 * a float64 re-score of the returned path against the float64 tables.
 * d_lattice: workspace of tehmm_viterbi_workspace_bytes() for the delta lattice.
 * d_ratios_emission: the ratios the emission was computed with (only used by
 * the re-score); d_ratios_dp: the ratios the DP applies (basehmm.py:327 vs
 * hmm.py:674 use different ones).                                            */
int64_t tehmm_viterbi_workspace_bytes(tehmm_ctx *ctx, int prec);
int tehmm_run_viterbi(tehmm_ctx *ctx, int prec, const void *d_elog, const double *d_rowmax,
                      const double *d_ratios_emission, const double *d_ratios_dp,
                      void *d_lattice, uint8_t *d_states, int64_t *d_states64,
                      double *d_logprob, void *d_scratch);

/* ------------------------------------------------------------- host buffers
 * The whole call MultitrackHmm.decode makes (/root/reference/basehmm.py:361-396
 * -> hmm.py:668-676 -> _hmm.pyx:201-259 for Viterbi; basehmm.py:332-359 for
 * MAP), with HOST buffers on both sides: h_obs_ptrs = nptr pointers to (T_i,K)
 * symbol matrices, pageable or pinned -- nptr = 1: one matrix holding all the
 * sequences back to back; nptr = nseq: one matrix per sequence, as the
 * reference's list of TrackTables (no host-side concatenation) --, h_offsets
 * nseq+1 row offsets, h_states int64[total] out (the dtype
 * the reference returns, _hmm.pyx:210), h_logprob float64[nseq] out (Viterbi:
 * path log-probability; MAP: forward log-likelihood), h_score float64[nseq] out
 * (MAP: sum of the posterior maxima, basehmm.py:357; may be NULL for Viterbi).
 * No segment ratios (tehmm_decode_host_ratios below takes them).  The library owns everything in between: a grow-only
 * device arena, pinned staging rings and a thread pool (TEHMM_HOST_THREADS,
 * default min(16, cores)) that stages pageable input and widens the uint8
 * states that crossed PCIe.  Blocks until the outputs are complete.          */
#define TEHMM_DECODE_VITERBI 0
#define TEHMM_DECODE_MAP 1
#define TEHMM_DECODE_BOTH 2
int tehmm_decode_host(tehmm_ctx *ctx, const void *const *h_obs_ptrs, int64_t nptr, int obs_bytes,
                      int64_t nseq, const int64_t *h_offsets, int algorithm, int prec,
                      int64_t *h_states, double *h_logprob, double *h_score);
/* Both decodings of the same observations in ONE call -- what teHmmEval.py does when asked for the
 * Viterbi path and the posterior decoding of the same tracks (teHmmEval.py:127-160), and what the
 * fwd-bwd + Viterbi sweep of BASELINE.json is: the observations cross PCIe once, one emission pass
 * feeds both stages, and the MAP path travels and is widened while the Viterbi kernels run.
 * Outputs as two tehmm_decode_host calls would give them (bit-identical), plus the forward
 * log-likelihood.                                                                              */
int tehmm_decode_host_both(tehmm_ctx *ctx, const void *const *h_obs_ptrs, int64_t nptr, int obs_bytes,
                           int64_t nseq, const int64_t *h_offsets, int prec,
                           int64_t *h_viterbi_states, double *h_viterbi_logprob,
                           int64_t *h_map_states, double *h_map_score, double *h_forward_logprob);
/* The same two calls for segmented tables (segmentTracks.py, teHmmEval.py --segment): h_ratio_ptrs =
 * nseq host float64 arrays of T_i segment ratios (segment length / effective segment length, pageable
 * or pinned), an entry NULL for a sequence without ratios (segRatios=None); h_ratio_ptrs NULL = no
 * sequence has ratios.  As the reference's decode: the emission never sees the ratios (basehmm.py:327);
 * the Viterbi DP, its traceback and the float64 log-probability of the path do (hmm.py:674), each
 * sequence with its own -- a sequence without ratios gets the plain recursion, not the one at ratio 1
 * (_hmm.pyx:234-237 treats from-state 0 differently whenever ratios are given); the MAP path and the
 * forward log-likelihood ignore them (basehmm.py:261-264: not read).  The ratios travel through the
 * same staging ring as the observations.  A ratio that is not finite and > 0 gives TEHMM_EINVAL before
 * any output is written.  At most 64 states.                                                         */
int tehmm_decode_host_ratios(tehmm_ctx *ctx, const void *const *h_obs_ptrs, int64_t nptr, int obs_bytes,
                             int64_t nseq, const int64_t *h_offsets, const double *const *h_ratio_ptrs,
                             int algorithm, int prec, int64_t *h_states, double *h_logprob, double *h_score);
int tehmm_decode_host_both_ratios(tehmm_ctx *ctx, const void *const *h_obs_ptrs, int64_t nptr, int obs_bytes,
                                  int64_t nseq, const int64_t *h_offsets, const double *const *h_ratio_ptrs,
                                  int prec, int64_t *h_viterbi_states, double *h_viterbi_logprob,
                                  int64_t *h_map_states, double *h_map_score, double *h_forward_logprob);
/* bytes the last tehmm_decode_host moved over PCIe: which = 0 host->device, 1 device->host */
int64_t tehmm_decode_host_bytes(tehmm_ctx *ctx, int which);
/* wall-clock milliseconds of the phases of the last tehmm_decode_host call made with the
 * environment variable TEHMM_HOST_TRACE set ("1": also printed on stderr, "2": recorded only;
 * tracing adds a stream synchronisation per phase, so it is not for timed runs): which = 0 batch
 * set-up, 1 host->device copy + emission, 2 trellis, 3 device->host copy + widening; -1 if not traced */
double tehmm_decode_host_phase_ms(tehmm_ctx *ctx, int which);
/* self-test of the library's host thread pool (no GPU needed): `rounds` back-to-back parallel loops of
 * `threads` tiny tasks; returns the number of rounds in which an index did not run exactly once */
int64_t tehmm_host_pool_selftest(int threads, int64_t rounds);
/* device index / model shape of a context */
int tehmm_ctx_device(tehmm_ctx *ctx);
int tehmm_model_dims(tehmm_ctx *ctx, int *N, int *K, int *S);

/* float64 score of a state path over the rows [lo, hi) of the current batch, in the
 * reference's terms (_hmm.pyx:222-225,232-248: start or transition term + emission
 * per row): d_logprob[s] = sum over the rows of sequence s inside the range.  With
 * [0, total) this is what tehmm_run_viterbi returns; a sub-range is one rank's
 * share when a single long sequence is sharded in time (SURVEY.md section 8e).  */
int tehmm_path_score(tehmm_ctx *ctx, const uint8_t *d_states, const double *d_ratios_emission,
                     const double *d_ratios_dp, int64_t lo, int64_t hi, double *d_logprob,
                     void *d_scratch);

/* Segment ratios on the fast path (csrc/ratios.cu).  In the forward / backward recursions a
 * segment ratio r_t > 1 is a per-row diagonal factor A_jj^(r_t - 1) on the emission
 * (/root/reference/_hmm.pyx:140-149,187-188), so tehmm_fold_ratios rewrites the linear emission
 * lattice ONCE (d_blin and d_rowmax of tehmm_run_emission, in place) and tehmm_run_forward /
 * tehmm_run_backward are then called WITHOUT ratios -- on the tensor-core tile kernels where those
 * apply.  Do not hand the folded lattice to a pass that is also given the ratios.  What the
 * E-step still owes the ratios is the diagonal term of _log_sum_lneta (_hmm.pyx:91-96,107-110):
 * tehmm_ratio_diag_counts adds (1/N) sum_{t > s0, r_t > 1} (r_t - 1) gamma_t[j] to trans[j][j] of
 * d_start_trans (layout of tehmm_run_backward's TRANS output), from the posterior lattice.      */
int tehmm_fold_ratios(tehmm_ctx *ctx, int prec, const double *d_ratios, void *d_blin, double *d_rowmax);
int tehmm_ratio_diag_counts(tehmm_ctx *ctx, int prec, const void *d_post, const double *d_ratios,
                            double *d_start_trans, void *d_scratch);

/* ------------------------------------------------- data formats either side of the trellis
 * (SURVEY.md section 8f ranks 2 and 3; csrc/tracks.cu).  The (T, K) symbol table the HMM reads is
 * built in HBM: d_table is a DEVICE pointer to a row-major (T, K) matrix of elem_bytes-wide
 * integers (1 = uint8, the reference's INTEGER_ARRAY_TYPE; 2, 4), exactly the layout of
 * IntegerTrackTable.data (/root/reference/track.py:552-558) and of tehmm_set_batch's d_obs.
 *
 * tehmm_track_fill: column k := value (IntegerTrackTable.initRow, track.py:590-591).
 * tehmm_rasterize_intervals: the per-base fill of readBedData (/root/reference/trackIO.py:175-203)
 *   for n HOST intervals [h_start, h_end) in genome coordinates, in file order -- where intervals
 *   overlap the later one wins, as in the reference's loop; the first base of an interval (after
 *   clipping to [region_start, region_end)) gets h_val0 (the useDelta value), the others h_val.
 *   Values are already mapped through the track's value map (strings -> categories: host work).
 * tehmm_segment_table: bin/segmentTracks.py:200-277 (segmentTracks / isNewSegment) over nregions
 *   regions (h_region_off: nregions + 1 row offsets into the table, one region per TrackTable):
 *   d_cut[T] := 1 where a segment starts, d_seg_off (capacity T) := those rows, *h_nseg their
 *   number.  h_ignore / h_cut: K flags (args.ignoreList / args.cutList), thresh, maxLen, fixLen as
 *   the script's options, prev_mode = (--comp prev).  *h_passes (optional): scan passes used.
 * tehmm_compress_segments: TrackTable.segment with interpolate (track.py:476-481,515-533,603-620)
 *   followed by compressSegments (track.py:594-601): row s of d_out (nseg x K) := per-track mode of
 *   rows [d_seg_off[s], d_seg_off[s+1]) (last segment: to T) for the tracks flagged in h_use_mode
 *   (smallest among the most frequent values, as scipy.stats.mode), the segment's first row for
 *   the others.  Gaussian tracks (mean of mapped-back values, re-mapped) are host work and not
 *   covered.  uint8 tables.
 * tehmm_run_sum: _track.runSum (/root/reference/_track.pyx:13-25): d_out[i] = number of zeros
 *   in d_mask[0 .. i).                                                                          */
int tehmm_track_fill(tehmm_ctx *ctx, void *d_table, int64_t T, int K, int elem_bytes, int k, int32_t value);
int tehmm_rasterize_intervals(tehmm_ctx *ctx, const int64_t *h_start, const int64_t *h_end,
                              const int32_t *h_val, const int32_t *h_val0, int64_t n,
                              int64_t region_start, int64_t region_end, void *d_table, int K,
                              int elem_bytes, int k);
int tehmm_segment_table(tehmm_ctx *ctx, const void *d_table, int64_t T, int K, int elem_bytes,
                        int64_t nregions, const int64_t *h_region_off, const uint8_t *h_ignore,
                        const uint8_t *h_cut, int thresh, int64_t maxLen, int64_t fixLen, int prev_mode,
                        uint8_t *d_cut, int64_t *d_seg_off, int64_t *h_nseg, int *h_passes);
int tehmm_compress_segments(tehmm_ctx *ctx, const void *d_table, int64_t T, int K, int elem_bytes,
                            const int64_t *d_seg_off, int64_t nseg, const uint8_t *h_use_mode,
                            void *d_out);
int tehmm_run_sum(tehmm_ctx *ctx, const uint8_t *d_mask, int32_t *d_out, int64_t n);
/* BED reading on the host, natively: bedRead (/root/reference/trackIO.py:389-404) and, with
 * need_intersect, what `intersectBed -a file -b interval | sortBed` leaves of it
 * (trackIO.py:138-143: the parts of chrom's intervals inside [start, end), by start; stable).
 * sort (without need_intersect): by (chrom, start) like sortBed (trackIO.py:147-151).
 * valcol: 3 or 4 = the column whose string is the interval's value, 0 = none.  Values come back
 * as indices into the distinct value strings IN ORDER OF FIRST APPEARANCE, the order in which
 * the reference's loop shows them to the track's value map (which numbers categories in that
 * order when it is allowed to grow).                                                          */
typedef struct tehmm_bed tehmm_bed;
int tehmm_bed_open(const char *path, const char *chrom, int64_t start, int64_t end, int need_intersect,
                   int sort, int valcol, tehmm_bed **out);
int64_t tehmm_bed_count(tehmm_bed *bed);
int64_t tehmm_bed_nunique(tehmm_bed *bed);
const char *tehmm_bed_unique(tehmm_bed *bed, int64_t i);
int tehmm_bed_fetch(tehmm_bed *bed, int64_t *starts, int64_t *ends, int32_t *value_index);
void tehmm_bed_close(tehmm_bed *bed);

/* Decode output path: the per-observation BED writer of teHmmEval.py:238-262
 * (statesToBed, bedFile part): for observation i one line
 *   chrom \t curStart \t curStart + len_i \t name(states[i]) \n
 * with curStart = start + sum_{j<i} len_j (+ mask_off[curStart - start] when a
 * mask is given), len_i = seg_len[i] or 1 (seg_len NULL), name = names[state] or
 * the decimal state index (nnames 0).  Lines are NOT merged, as in the reference
 * (teHmmEval.py:241-243).  Written to the file descriptor fd at its current
 * offset (flush the Python file object first).  Host only, no GPU needed.     */
int tehmm_states_to_bed(int fd, const char *chrom, int64_t start, const int64_t *states,
                        int64_t n, const int64_t *seg_len, const int32_t *mask_off,
                        int64_t mask_n, const char *const *names, int nnames);

/* the posterior / emission score files of the same reference function (bin/teHmmEval.py:264-270):
 * same intervals, fourth column = scores[i] printed as Python prints a float64 ("%s") */
int tehmm_scores_to_bed(int fd, const char *chrom, int64_t start, const double *scores,
                        int64_t n, const int64_t *seg_len, const int32_t *mask_off, int64_t mask_n);

/* widen / convert on the device before a D2H copy */
int tehmm_widen_states(tehmm_ctx *ctx, const uint8_t *d_in, int64_t *d_out, int64_t n);
int tehmm_convert_lattice(tehmm_ctx *ctx, int prec, const void *d_in, double *d_out, int64_t n);

#ifdef __cplusplus
}
#endif
#endif /* TEHMM_B200_H */
