/*
 * sapr_b200.h -- C ABI of libsaprb200.so: the B200-native replacement for the
 * arithmetic of frankcholula/sapr's assignment2 HMM hot path.
 *
 * The reference has no FFI: its boundary is the Python surface of
 * assignment2/custom_hmm.py::HMM and the hmmlearn GaussianHMM calls in
 * assignment2/hmmlearn_hmm.py / decoder.py.  Each entry point below names the
 * reference code it replaces (file:line, relative to /root/reference).  The
 * Python classes in sapr_b200/ keep the reference's method names and call these
 * through ctypes (see INTEGRATION.md for the stub a maintainer would add).
 *
 * Conventions
 *  - extern "C", plain pointers and sizes, no torch types.  Every function
 *    returns 0 on success or a negative SAPR_E_* code; sapr_last_error() gives
 *    the message.  Nothing throws, nothing calls exit().
 *  - The caller owns every data buffer.  Unless a parameter is documented as
 *    HOST memory it is a DEVICE pointer on the ctx's device.  The library owns
 *    only the opaque handles and a ctx workspace that grows on first use.
 *  - All work is enqueued on the cudaStream_t given to sapr_ctx_create (pass
 *    torch.cuda.current_stream().cuda_stream); calls are asynchronous.
 *  - Features: float32, frame-major X[sum_T][ldx] (ldx >= D, ldx % 4 == 0 so
 *    rows are 16-byte aligned), utterance u = rows offsets[u] .. offsets[u+1].
 *  - State indexing follows the reference: S = N + 2, state 0 = non-emitting
 *    entry, state S-1 = non-emitting exit (custom_hmm.py:24, :94-116).
 */
#ifndef SAPR_B200_H
#define SAPR_B200_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define SAPR_OK 0
#define SAPR_E_INVALID (-1)   /* bad argument (the reference raises AssertionError / ValueError) */
#define SAPR_E_CUDA (-2)      /* CUDA runtime error */
#define SAPR_E_NOMEM (-3)
#define SAPR_E_RANGE (-4)     /* shape outside what the kernels were built for (N > 31, ...) */
#define SAPR_E_SHORT (-5)     /* utterance shorter than the frames decode must walk (reference: IndexError) */

/* precision of the fused kernels */
#define SAPR_FP32 0           /* production: fp32 emission + per-frame renormalised fp32 recursions */
#define SAPR_FP64 1           /* verification: float64 end to end, same summation order as the oracle */
#define SAPR_FP32_SIMT 2      /* fp32 with the SIMT emission forced (A/B against the tensor-core emission) */

/* emission model */
#define SAPR_EMIT_DIAG 0      /* true diagonal Gaussian (north_star; hmmlearn "diag") */
#define SAPR_EMIT_SAPR 1      /* custom_hmm.py:146-174 as written: Gram row-sum + full covariance (SURVEY D1/D2) */

/* topology */
#define SAPR_TOPO_ENTRY_EXIT 0 /* custom_hmm.py: entry/exit non-emitting, left-to-right (D4, D5, D9) */
#define SAPR_TOPO_DENSE 1      /* hmmlearn: all S states emit, dense S x S transmat + startprob */

typedef struct sapr_ctx sapr_ctx;
typedef struct sapr_models sapr_models;

int sapr_version(void);
int sapr_ctx_create(int device, void *cuda_stream, sapr_ctx **out);
int sapr_ctx_destroy(sapr_ctx *ctx);
const char *sapr_last_error(sapr_ctx *ctx);
/* number of kernels this ctx has launched so far (bench.py's gpu_launches) */
int64_t sapr_launch_count(sapr_ctx *ctx);
int sapr_sync(sapr_ctx *ctx);
/* Per-kernel device timing for bench.py's roofline: when enabled, CUDA events bracket every launch of the
 * dominant kernels on the ctx stream.  sapr_profile_read synchronises, then returns the summed duration (ms)
 * and launch count of kernel class `which` (0 = fused Viterbi, 1 = Viterbi finish/back-trace,
 * 2 = fused E-step forward/backward, 3 = E-step feature statistics, 4 = ergodic tensor-core emission,
 * 5 = ergodic tensor-core forward, 6 = fp32 word near-tie re-decoding, 7 = dense-topology fused Viterbi (its arg-max / back-trace
 * counts as 1), 8 = float64 re-decoding of dense-topology word near-ties, 9 = dense-topology fp32 E-step forward / backward,
 * 10 = its feature statistics, 11 = hmmlearn M-step, 12 = dense-topology fp32 forward of sapr_score_words (its arg-max counts
 * as 1), 13 = float64 re-scoring of its word near-ties) since the last sapr_profile(ctx, 1). */
int sapr_profile(sapr_ctx *ctx, int enable);
int sapr_profile_read(sapr_ctx *ctx, int which, double *ms, int64_t *launches);

/* ---- word-model set: replaces the parameter block of class HMM (custom_hmm.py:10-33)
 * and of GaussianHMM (hmmlearn_hmm.py:27-43), for M models at once ------------------- */
int sapr_models_create(sapr_ctx *ctx, int M, int N, int D, int emission, int topology, sapr_models **out);
int sapr_models_destroy(sapr_models *m);
/* HOST pointers, float64: means[M][S][D]; covars[M][S][D] (DIAG: variances) or [M][S][D][D]
 * (SAPR: full covariance); transmat[M][S][S]; startprob[M][S] (DENSE topology only, else NULL). */
int sapr_models_set(sapr_models *m, const double *means, const double *covars, const double *transmat,
                    const double *startprob);
int sapr_models_get(sapr_models *m, double *means, double *covars, double *transmat, double *startprob);

/* ---- flat start: custom_hmm.py:35-116 (calculate_means, calculate_covariance, and the frame /
 * utterance counts initialize_transitions needs).  out (device, float64) = [sum x (D) | sum x^2 (D) |
 * frames | utterances]; pivot (device float64[D], nullable = 0) is subtracted before squaring. ---- */
int sapr_init_stats(sapr_ctx *ctx, const float *X, int ldx, const int64_t *offsets, int B, int D,
                    const double *pivot, double *out);

/* ---- batched Viterbi: custom_hmm.py:462-514 (decode) for every utterance x model, plus the
 * strict-'>' argmax over models of decoder.py:42-47.  DIAG emission + ENTRY_EXIT topology, fused.
 * DIAG emission + DENSE topology (hmmlearn GaussianHMM.decode per model, S <= 32, else SAPR_E_RANGE: large ergodic models keep
 * sapr_hl_decode): delta_0(j) = ln pi_j + e_0(j), delta_t(j) = max_i (delta_{t-1}(i) + ln A_ij) + e_t(j), a model's score is
 * max_j delta_{T-1}(j) (no exit arc), the back-trace takes the first maximum (lowest index).  best_word is the strict-'>' arg-max
 * (first best wins, -1 when every model scores -inf; best_path then holds model 0's path), best_path holds states 0..S-1.
 * SAPR_FP64 equals sapr_hl_decode per model bit for bit; SAPR_FP32 is the fused fp32 kernel (csrc/viterbi_dense.cu) with the
 * near-tie pass below.  DENSE sets refuse first_frames > 0, all_paths and model_of_utt (SAPR_E_INVALID); max_T must cover the
 * longest utterance.
 * DIAG emission + ENTRY_EXIT topology: N <= 31 (else SAPR_E_RANGE).  One model's packed parameters take (D+3)/4 * N * 64 B in
 * SAPR_FP64 and half that in fp32; the all-models call stages up to 16 of them per CTA, fewer when they do not fit 227 KB, and
 * model_of_utt stages all M (M <= 45 float64 / 90 fp32 models at N = 8, D = 39); a shape that does not fit is SAPR_E_RANGE before
 * any launch.  SAPR_FP32 takes the tensor-core kernels for N = 8, M <= 12, D <= 47 when every emitting state's self-loop is
 * non-zero (the tensor-core image folds ln A[j][j] into the emission; re-checked after every sapr_models_set / sapr_mstep), and
 * the SIMT kernel (as SAPR_FP32_SIMT) otherwise.
 *   model_of_utt  int32[B] or NULL; NULL = score against all M models
 *   max_T         the longest utterance of the batch; it sizes the scratch, and an utterance longer than max_T is decoded
 *                 on its first max_T frames only (never past the scratch)
 *   first_frames  > 0 walks only that many frames (SURVEY D3: the reference walks D frames), 0 = all
 *   best_word     int32[B]      index of the winning model (first best wins ties)
 *   best_score    float64[B]    V[T-1, S-1] of the winner (-inf if the exit state is unreachable)
 *   scores        float64[B*M]  nullable; every model's score
 *   best_path     uint8[sum_T]  nullable; winner's state path at the utterance's frame offset
 *   all_paths     uint8[M*sum_T] nullable; every model's path, model-major                      */
int sapr_viterbi(sapr_ctx *ctx, sapr_models *m, const float *X, int ldx, const int64_t *offsets, int B,
                 int64_t total_frames, int max_T, const int32_t *model_of_utt, int precision,
                 int first_frames, int32_t *best_word, double *best_score, double *scores,
                 uint8_t *best_path, uint8_t *all_paths);
/* fp32 production mode (tensor-core kernels or the DENSE kernel, all models, all_paths == NULL): an utterance whose best and second-best word
 * scores differ by less than 8e-6 |best| -- closer than the fp32 scores resolve -- is re-decoded in float64 inside the same
 * call (word, score, score row and path then are the verification mode's), so the recognised word equals the float64 one
 * except on exact float64 ties (decoder.py:42-47 keeps the first).  n = utterances flagged by the last sapr_viterbi or
 * sapr_score_words call on this context
 * (synchronises the stream); the first 8192 flagged utterances of each 1 GB back-pointer chunk are re-decoded, at any length
 * (utterances whose emissions exceed the shared-memory staging use a global-memory scratch).  ENTRY_EXIT sets have this pass on
 * the tensor-core kernels only; the SIMT fp32 kernel keeps its fp32 words.  SAPR_EXACT_WORDS=0 disables the pass.
 * Stream order: part of an equal-length batch's arg-max / back-trace may run on a context-owned auxiliary stream beside the
 * last launch of the main kernel; it is joined back into the context's stream before the call returns, so work the caller
 * enqueues on that stream afterwards sees every output. */
int sapr_viterbi_flagged(sapr_ctx *ctx, int64_t *n);

/* Parity/debug: the tensor-core emission tile of the fused Viterbi kernel written out, E_out float32
 * [sum_T][*ncols_out], column m*8 + (j-1) = state j of model m (compute_emission_matrix, custom_hmm.py:146-174,
 * for all models at once).  Only for model sets the tensor-core path accepts (N == 8, M <= 12, D < 64). */
int sapr_debug_tc_emission(sapr_ctx *ctx, sapr_models *m, const float *X, int ldx, const int64_t *offsets, int B,
                           int64_t total_frames, int max_T, float *E_out, int *ncols_out);

/* Same call with HOST buffers: features are staged through pinned memory and streamed to the GPU in
 * utterance chunks (copy/compute overlap), results come back to host arrays.  This is the call a
 * reference-side plugin makes when its features live in numpy arrays (decoder.py:51-72).          */
int sapr_viterbi_host(sapr_ctx *ctx, sapr_models *m, const float *X_host, int ldx, const int64_t *offsets_host,
                      int B, int precision, int first_frames, int chunk_utts, int32_t *best_word_host,
                      double *best_score_host, uint8_t *best_path_host);

/* ---- Baum-Welch E-step: custom_hmm.py:417-439 (emission, forward, backward, gamma, xi and the
 * accumulators) + the sums update_B consumes (:372-386), every utterance against model_of_utt[u].
 * DIAG emission + ENTRY_EXIT topology, fused.  order[B] (nullable) lists utterance ids grouped by model.
 *   stats   float64[M * sapr_stats_stride(N, D)], zeroed by the call; per model:
 *           G[S] = sum gamma[:-1] | Xi[S] = sum xi(j,j) | occ[S] | sum gamma (x-mu_old) [S*D] |
 *           sum gamma (x-mu_old)^2 [S*D]
 *   loglik  float64[B]  logsumexp(alpha_scaled[T-1,:]) as the reference reports it (SURVEY D6)
 *   gamma_out float32/float64 [sum_T * N] nullable debug output (emitting states only)
 * Range: N <= 31, D <= 256.  Off the tensor-core path (SAPR_FP64, and SAPR_FP32 outside N = 8, M <= 12, D <= 47 or with a zero
 * emitting self-loop) one CTA stages every model: M * ((D+3)/4 * N * 64 + 16) B in float64, half in fp32, within 227 KB (M <= 45
 * float64 / 90 fp32 at N = 8, D = 39); the statistics kernel keeps 8 * 4 * 2 * N * (D+3)/4*4 B (D <= 116 at N = 31).  A shape
 * outside these is SAPR_E_RANGE before any launch. */
/* DIAG emission + DENSE topology (hmmlearn GaussianHMM.fit's E-step, every model at once): model_of_utt is required (NULL =
 * SAPR_E_INVALID), order as above.  stats float64[M * sapr_hl_stats_len(S, D)], zeroed by the call, per model
 * [start S | trans S*S | post S | obs S*D | obs2 S*D] as sapr_hl_estep gives it; loglik = log P(X_u); gamma_out [sum_T][S]
 * (fp32 in SAPR_FP32, float64 in SAPR_FP64).  SAPR_FP64 runs sapr_hl_estep per model on that model's utterances in batch order,
 * so stats and loglik equal GaussianHMM.fit's E-step for the word bit for bit (any S sapr_hl_estep takes).  SAPR_FP32 is the
 * fused kernel of csrc/estep_dense.cu (S <= 32, and one model's parameters and accumulators within the device's opt-in shared
 * memory per block, about D <= 228 at S = 32 on a B200; else SAPR_E_RANGE; max_T must cover the longest utterance): per-frame
 * log-shifted linear recursions, so utterances far from their model stay finite; an utterance the model cannot produce gets
 * loglik -inf and contributes nothing.  Two identical calls give identical bits.  */
int64_t sapr_stats_stride(int N, int D);
int sapr_estep(sapr_ctx *ctx, sapr_models *m, const float *X, int ldx, const int64_t *offsets, int B,
               int64_t total_frames, int max_T, const int32_t *model_of_utt, const int32_t *order,
               int precision, double *stats, double *loglik, void *gamma_out);

/* ---- M-step: custom_hmm.py:351-400 from the packed statistics (after the cross-GPU all-reduce).
 * floor_var[M] HOST float64: var_floor_factor * mean(diag(global_covariance)) per model.
 * Diagonal statistics: var_j = sum gamma (x-c)^2/occ - (mu_j - c)^2 (equals the diagonal of the
 * reference's second pass around the new mean).  Updates the device parameters in place.         */
int sapr_mstep(sapr_ctx *ctx, sapr_models *m, const double *stats, const double *floor_var_host);

/* ---- per-step functions of class HMM on materialised float64 arrays (one utterance, one model),
 * kept so the reference's own tests can run against the CUDA path. mi = model index. ------------ */
/* compute_emission_matrix, custom_hmm.py:146-174: E[T][S] float64 */
int sapr_emission(sapr_ctx *ctx, sapr_models *m, int mi, const float *X, int ldx, int T, double *E);
/* forward, :176-211: alpha[T][S], scale[1] */
int sapr_forward(sapr_ctx *ctx, sapr_models *m, int mi, const double *E, int T, double *alpha, double *scale);
/* backward, :213-246 */
int sapr_backward(sapr_ctx *ctx, sapr_models *m, int mi, const double *E, int T, const double *scale, double *beta);
/* compute_gamma, :248-257 */
int sapr_gamma(sapr_ctx *ctx, int S, const double *alpha, const double *beta, int T, double *gamma);
/* compute_xi, :259-322: xi[T-1][S][S] */
int sapr_xi(sapr_ctx *ctx, sapr_models *m, int mi, const double *alpha, const double *beta, const double *E,
            int T, double *xi);
/* decode on a materialised emission matrix, :462-514: walks T_eff rows; path int32[T_eff], score[1] */
int sapr_decode_mat(sapr_ctx *ctx, sapr_models *m, int mi, const double *E, int T_eff, double *score, int32_t *path);
/* update_A, :351-364: agg_xi[S][S], agg_gamma[S] (device float64) */
int sapr_update_A(sapr_ctx *ctx, sapr_models *m, int mi, const double *agg_xi, const double *agg_gamma);
/* update_B, :366-400: two-pass full-covariance re-estimation from gamma[sum_T][S]; floor_var scalar */
int sapr_update_B(sapr_ctx *ctx, sapr_models *m, int mi, const float *X, int ldx, int64_t total_frames,
                  const double *gamma, double floor_var);
/* One as-written Baum-Welch E-step for model mi over B utterances (SAPR or DIAG emission, float64,
 * materialised): fills gamma[sum_T][S], agg_gamma[S], agg_xi[S][S], loglik[B].  custom_hmm.py:417-439 */
int sapr_estep_compat(sapr_ctx *ctx, sapr_models *m, int mi, const float *X, int ldx, const int64_t *offsets,
                      int B, int64_t total_frames, double *gamma, double *agg_gamma, double *agg_xi, double *loglik);
/* decode of one utterance against model mi with the model's own emission (SAPR or DIAG), float64:
 * emission over all T frames, Viterbi over T_eff.  decoder.py:43 / custom_hmm.py:462-514          */
int sapr_decode_compat(sapr_ctx *ctx, sapr_models *m, int mi, const float *X, int ldx, int T, int T_eff,
                       double *score, int32_t *path);

/* ---- hmmlearn-style (DENSE topology, all states emit): GaussianHMM.score / decode / fit E-step
 * as used by hmmlearn_hmm.py:103-104 and decoder.py:43.  float64.                                 */
/* lf = log frame probabilities [sum_T][S] workspace-free API: returns per-utterance log-prob.
 * All three accept up to 1024 states (BASELINE cfg 4: N = 256 ergodic; SAPR_E_RANGE beyond): thread per utterance up to
 * 32 states, CTA per utterance above. */
int sapr_hl_score(sapr_ctx *ctx, sapr_models *m, int mi, const float *X, int ldx, const int64_t *offsets, int B,
                  int64_t total_frames, double *logprob);
int sapr_hl_decode(sapr_ctx *ctx, sapr_models *m, int mi, const float *X, int ldx, const int64_t *offsets, int B,
                   int64_t total_frames, double *logprob, int32_t *path);
/* Tensor-core forward (score) for large dense models: S in {64, 128, 192, 256}, D <= 39, fp32 scaled linear-domain
 * recursion; both contractions run on tcgen05 (ergodic_tc.cu): the emission [x', x'^2, 1] . W_e per frame and the
 * [128 utterances x S] . [S x S] transition product per frame.  Arguments as sapr_hl_score (which stays the float64
 * verification mode) except max_T, an upper bound on the utterance length that sizes the emission staging
 * (an utterance longer than max_T scores NaN).  Transition weights are fp16 (2^-12 relative), the state vector fp16 hi/lo:
 * |d logP| <= 5e-6 |logP| + 2e-4 T against the float64 kernel.  Operand range: transition probabilities below 2^-39 and
 * posterior mass below 2^-39 of a frame's total count as zero (normal precision above 2^-29); a sequence whose likelihood
 * is carried only through such tails needs the float64 mode.  Replaces hmmlearn GaussianHMM.score as called at
 * hmmlearn_hmm.py:46-75. */
int sapr_ergodic_score(sapr_ctx *ctx, sapr_models *m, int mi, const float *X, int ldx, const int64_t *offsets, int B,
                       int max_T, double *logprob);
/* Batched GaussianHMM.score for every utterance x model of a DENSE + DIAG set, and recognition by total likelihood: scores[u*M + m]
 * = log P(X_u | model m) (the forward log-likelihood, natural log; an empty utterance scores 0, one no state sequence of the
 * model can produce -inf), best_word[u] the strict-'>' arg-max over the models (first best wins, -1 when every model scores
 * -inf), best_score[u] its score.  Each output is nullable; at least one must be given.
 *   SAPR_FP64  verification: sapr_hl_score per model + a running arg-max, bit for bit with GaussianHMM.score per model (any S
 *              sapr_hl_score takes).
 *   SAPR_FP32  fused fp32 forward of csrc/score_dense.cu (S <= 32, else SAPR_E_RANGE: SAPR_FP64, or sapr_ergodic_score for
 *              64-256 states): per-frame log-shifted linear recursion, so utterances far from a model and transitions below the
 *              fp32 range stay finite.  Utterances whose best and second-best scores differ by less than 8e-6 |best| are
 *              re-scored in float64 in the same call (word, score and score row then are the verification mode's; at most 8192
 *              per call, counted by sapr_viterbi_flagged; SAPR_EXACT_WORDS=0 disables the pass).
 * ENTRY_EXIT or SAPR-emission sets, ldx % 4 != 0 and an unknown precision are refused with SAPR_E_INVALID. */
int sapr_score_words(sapr_ctx *ctx, sapr_models *m, const float *X, int ldx, const int64_t *offsets, int B,
                     int64_t total_frames, int precision, int32_t *best_word, double *best_score, double *scores);
/* stats = [start S | trans S*S | post S | obs S*D | obs2 S*D] float64, zeroed by the call */
int64_t sapr_hl_stats_len(int S, int D);
int sapr_hl_estep(sapr_ctx *ctx, sapr_models *m, int mi, const float *X, int ldx, const int64_t *offsets, int B,
                  int64_t total_frames, double *stats, double *logprob);
/* hmmlearn GaussianHMM._do_mstep ('diag') for every model of a DENSE + DIAG set, from the statistics sapr_estep gives it
 * (per model [start S | trans S*S | post S | obs S*D | obs2 S*D], after any all-reduce).  Updates the device parameters in
 * place and re-derives the fp32 image (sapr_models_prepare).  Bit for bit with the numpy expressions (operation order, no FMA
 * contraction, NaN-propagating maximum, numpy's pairwise row sums); S <= 1024.
 *   priors     DEVICE float64[M * (S + S*S + 3*S*D + 1)], per model
 *              [startprob_prior S | transmat_prior S*S | means_prior S*D | means_weight S*D | covars_prior S*D | covars_weight]
 *   flags_host HOST int32[M]: bit 0 's', 1 't', 2 'm', 3 'c' (GaussianHMM.params); 0 leaves the model untouched       */
int sapr_hl_mstep(sapr_ctx *ctx, sapr_models *m, const double *stats, const double *priors, const int32_t *flags_host);

/* ---- evaluation metrics: assignment2/eval.py:28-38 (sklearn confusion_matrix + accuracy_score over the label indices).
 * truth / pred int32[B] (device), cm int64[M][M + 1] (device, zeroed by the call; column M = no model reachable, pred < 0),
 * correct int64[1] (device). */
int sapr_confusion(sapr_ctx *ctx, const int32_t *truth, const int32_t *pred, int B, int M, int64_t *cm, int64_t *correct);

/* ---- multi-GPU: the one collective of the path.  The reference accumulates gamma / xi / feature sums over all utterances
 * in one process (custom_hmm.py:417-419, :434-439, :372-386); with utterances sharded over one process per GPU the packed
 * statistics block (sapr_stats_stride doubles per model, + per-model log-likelihoods) is summed over the ranks once per
 * Baum-Welch iteration.  NCCL is resolved at run time (dlopen libnccl.so.2).  uid128: 128 bytes from sapr_comm_unique_id on
 * rank 0, handed to the other ranks by the host (any side channel).  sapr_stats_allreduce works in place on a DEVICE buffer
 * and only enqueues on the context's stream. */
typedef struct sapr_comm sapr_comm;
int sapr_comm_unique_id(void *uid128);
int sapr_comm_init_rank(sapr_ctx *ctx, const void *uid128, int rank, int world, sapr_comm **out);
int sapr_stats_allreduce(sapr_ctx *ctx, sapr_comm *comm, double *stats, int64_t n);
int sapr_comm_destroy(sapr_comm *comm);

/* ---- MFCC front-end: assignment2/mfcc_extract.py:10-27 (librosa.feature.mfcc) as one fused
 * kernel: (pre-emphasis) -> framing + window -> DFT power -> mel filterbank -> log/dB -> DCT-II. */
typedef struct {
    int sample_rate;     /* 22050 (reference) / 16000 (BASELINE cfg 5) */
    int n_fft;           /* 2048 / 512 */
    int win_length;      /* 661 / 400 */
    int hop_length;      /* 220 / 160 */
    int n_mels;          /* 128 / 26 */
    int n_mfcc;          /* 13 */
    int center;          /* 1: zero-pad n_fft/2 both sides (librosa center=True, pad_mode="constant") */
    int mel_slaney;      /* 1: Slaney scale + slaney norm (librosa default); 0: HTK scale, unnormalised */
    int log_db;          /* 1: 10*log10(max(S,1e-10)) with top_db clamp; 0: ln(max(S, 1e-10)) */
    float top_db;        /* 80 (librosa); <= 0 disables the clamp */
    float preemph;       /* 0 (reference) / 0.97 (cfg 5) */
    float fmin, fmax;    /* 0, sample_rate/2 */
} sapr_mfcc_params;
/* audio float32[sum_samples], sample_offsets int64[B+1]; feat_offsets int64[B+1] (device, filled by the
 * call: frames = 1 + len/hop when center); feats float32[sum_frames][ld_out] frame-major.           */
int64_t sapr_mfcc_num_frames(const sapr_mfcc_params *p, int64_t n_samples);
int sapr_mfcc(sapr_ctx *ctx, const sapr_mfcc_params *p, const float *audio, const int64_t *sample_offsets_host,
              int B, float *feats, int ld_out, int64_t *feat_offsets_host);

#ifdef __cplusplus
}
#endif
#endif /* SAPR_B200_H */
