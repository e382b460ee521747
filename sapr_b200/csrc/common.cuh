// common.cuh -- context, model storage and math helpers shared by all kernels of libsaprb200.
#pragma once
#include <cuda_runtime.h>
#include <math.h>
#include <stdint.h>
#include <stdio.h>
#include <string.h>

#include <algorithm>
#include <string>
#include <type_traits>
#include <vector>

#include "../../include/sapr_b200.h"

#define SAPR_MAX_N 31 /* emitting states per model (backpointer word = N+1 bits) */
#define SAPR_LOG2PI 1.8378770664093454835606594728112
#define SAPR_LN2 0.69314718055994530941723212145818

struct sapr_ctx {
    int device = 0;
    cudaStream_t stream = nullptr;
    std::string err;
    int64_t launches = 0;
    int sm_count = 148;
    // grow-on-demand device workspace arenas (no cudaMalloc in steady state)
    void *ws[10] = {};               // scratch slots shared by the entry points; slot 8 belongs to the near-tie flag buffers alone
    size_t ws_bytes[10] = {};
    // pinned staging + second stream for the host-buffer entry points
    void *pin[4] = {nullptr, nullptr, nullptr, nullptr};
    size_t pin_bytes[4] = {0, 0, 0, 0};
    cudaStream_t copy_stream = nullptr;
    cudaStream_t aux_stream = nullptr;      // arg-max / back-trace of a batch's full rounds beside its partial round (viterbi_v3.cu)
    cudaEvent_t ev[10] = {};
    // optional per-kernel event timing (bench.py roofline)
    bool profiling = false;
    struct ProfRec { cudaEvent_t a, b; int which; };
    std::vector<ProfRec> prof;       // used records
    std::vector<ProfRec> prof_pool;  // recycled event pairs
    bool flag_valid = false;         // ws[8] holds the flag counters of the last fp32 Viterbi or word-scoring call (sapr_viterbi_flagged)
    int flag_maxT = 0;               // longest utterance of that call (sizes the float64 re-decoding)
};

// RAII bracket: records an event pair around one kernel launch when profiling is on
struct ProfScope {
    sapr_ctx *ctx; sapr_ctx::ProfRec r; bool on; cudaStream_t st;
    ProfScope(sapr_ctx *c, int which, cudaStream_t stream = nullptr) : ctx(c), on(c->profiling), st(stream ? stream : c->stream) {
        if (!on) return;
        if (!c->prof_pool.empty()) { r = c->prof_pool.back(); c->prof_pool.pop_back(); }
        else { cudaEventCreate(&r.a); cudaEventCreate(&r.b); }
        r.which = which;
        cudaEventRecord(r.a, st);
    }
    ~ProfScope() {
        if (!on) return;
        cudaEventRecord(r.b, st);
        ctx->prof.push_back(r);
    }
};

// Device-resident parameters of M word models.
struct sapr_models {
    sapr_ctx *ctx = nullptr;
    int M = 0, N = 0, D = 0, S = 0, emission = 0, topology = 0;
    int Dp = 0;      // D rounded up to a multiple of 4
    int n_emit = 0;  // states that emit: N (ENTRY_EXIT) or S (DENSE)
    // float64 masters
    double *mean = nullptr;   // [M][S][D]
    double *cov = nullptr;    // DIAG: [M][S][D]; SAPR: [M][S][D][D]
    double *A = nullptr;      // [M][S][S]
    double *pi = nullptr;     // [M][S] (DENSE)
    // derived, refreshed by models_prepare() after every set / M-step
    double *logA = nullptr;   // [M][S][S] elementwise log (log 0 = -inf)
    double *logpi = nullptr;  // [M][S]
    // ENTRY_EXIT left-to-right transitions: la[j] = ln A[j][j], lb[j] = ln A[j][j+1] (lb[0] = ln A[0][1]),
    // index j in [0, S): la[S-1] = ln A[S-1][S-1]
    double *la64 = nullptr, *lb64 = nullptr;  // [M][S]
    float *la32 = nullptr, *lb32 = nullptr;
    // DIAG emission packed for the fused kernels, per model: [chunk c][state e][8] = (mu x4, h x4),
    // h = 0.5 / var; cst[e] = -0.5 (D ln 2pi + sum ln var); padded dims have mu = 0, h = 0.
    double *pk64 = nullptr;   // [M][Dp/4][n_emit][8]
    float *pk32 = nullptr;
    double *cst64 = nullptr;  // [M][n_emit]
    float *cst32 = nullptr;
    // SAPR emission: P = inv(cov + 1e-6 I) [M][S][D][D], cstS = -0.5 (D ln 2pi + logdet) [M][S]
    double *P = nullptr;
    double *cstS = nullptr;
    // tensor-core Viterbi image (viterbi_tc.cu): fp16 hi/lo weights in shared-memory layout + (g, s) + transitions
    void *tc_image = nullptr;
    int tc_ctas_per_sm = 1;
    // every emitting state's self-loop is non-zero (refreshed by sapr_models_prepare): the image folds ln A[j][j] into the emission
    // constant, so a zero self-loop would make that state's emission NaN; such sets take the SIMT fp32 kernels
    bool tc_loops_finite = false;
    // DENSE + DIAG sets with S <= 32 (viterbi_dense.cu): pivot p[Dp]; per model [chunk][state][8] = (a x4, b x4) with
    // a = (mu - p) / var, b = -1 / (2 var); cst[S] = -0.5 (D ln 2pi + sum ln var + sum (mu - p)^2 / var); ln pi [S];
    // finite arcs (ln A, source) grouped by destination [S*S] float2 with start[S + 1]; the same arcs (A, destination) grouped
    // by source with starts[S + 1] (the E-step's backward sweep, estep_dense.cu), and log2 A of those source-grouped arcs
    // [S*S] (computed in float64: the backward sweep's log-domain branch, where fp32 A of a transition below 2^-126 is 0)
    float *dn_piv = nullptr, *dn_w = nullptr, *dn_cst = nullptr, *dn_lpi = nullptr, *dn_lg2s = nullptr;
    void *dn_arc = nullptr, *dn_arcs = nullptr;
    int32_t *dn_start = nullptr, *dn_starts = nullptr;
    bool valid = false;
};

#define SAPR_CUDA(ctx, call)                                                                  \
    do {                                                                                      \
        cudaError_t _e = (call);                                                              \
        if (_e != cudaSuccess) {                                                              \
            (ctx)->err = std::string(#call) + ": " + cudaGetErrorString(_e);                  \
            return SAPR_E_CUDA;                                                               \
        }                                                                                     \
    } while (0)

#define SAPR_FAIL(ctx, code, msg) \
    do {                          \
        (ctx)->err = (msg);       \
        return (code);            \
    } while (0)

#define SAPR_LAUNCH_CHECK(ctx)                                                   \
    do {                                                                         \
        (ctx)->launches++;                                                       \
        cudaError_t _e = cudaGetLastError();                                     \
        if (_e != cudaSuccess) {                                                 \
            (ctx)->err = std::string("kernel launch: ") + cudaGetErrorString(_e); \
            return SAPR_E_CUDA;                                                  \
        }                                                                        \
    } while (0)

// fp32 production Viterbi: utterances whose best and second-best word scores are closer than the fp32 scores resolve are
// listed (arg-max kernels) and re-decoded in float64 (sapr_viterbi_redo_flagged), so the recognised word is the float64 one
struct SaprFlag {
    int32_t *list = nullptr;    // [cap] utterance indices
    int32_t *count = nullptr;   // [0] entries of this chunk (may exceed cap: the surplus is not listed), [1] running total of the call
    int32_t *done = nullptr;    // [SAPR_FLAG_CAP] models completed per list entry (k_redo_fused; zero between launches)
    int cap = 0;
    float rel = 0.f;
};
#ifdef __CUDACC__
__device__ __forceinline__ void sapr_flag_word(const SaprFlag &f, int u, double best, double second) {
    if (!f.list || !(best > -INFINITY) || !(second > -INFINITY)) return;
    if (best - second < (double)f.rel * fabs(best)) {
        const int pos = atomicAdd(f.count, 1);
        atomicAdd(f.count + 1, 1);
        if (pos < f.cap) f.list[pos] = u;
    }
}
#endif
#define SAPR_FLAG_CAP 8192
#define SAPR_FLAG_REL 8e-6f
int sapr_viterbi_redo_flagged(sapr_ctx *ctx, sapr_models *m, const float *X, int ldx, const int64_t *offsets, int first_frames,
                              int nu, const SaprFlag &flag, int32_t *best_word, double *best_score, double *scores, uint8_t *best_path);
int sapr_flag_setup(sapr_ctx *ctx, SaprFlag *flag, bool first_chunk);   // workspace slot 8; zeroes the per-chunk counter
int sapr_ws_reserve(sapr_ctx *ctx, int slot, size_t bytes);   // grows ctx->ws[slot]
int sapr_pin_reserve(sapr_ctx *ctx, int slot, size_t bytes);  // grows ctx->pin[slot]
int sapr_models_prepare(sapr_models *m);                      // recompute the derived arrays on device
int sapr_dense_prepare(sapr_models *m);                       // fp32 arrays of the dense Viterbi (viterbi_dense.cu)
int sapr_viterbi_dense(sapr_ctx *ctx, sapr_models *m, const float *X, int ldx, const int64_t *offsets, int B, int64_t total_frames,
                       int max_T, const int32_t *model_of_utt, int precision, int first_frames, int32_t *best_word, double *best_score,
                       double *scores, uint8_t *best_path, uint8_t *all_paths);
// float64 emission matrix E[total_frames][S] of model mi for a batch (DIAG or SAPR emission)
bool sapr_tc_eligible(const sapr_models *m);    // shape only: whether the set has a tensor-core image
bool sapr_tc_usable(const sapr_models *m);      // the image exists and every emitting self-loop is non-zero
size_t sapr_tc_image_bytes(const sapr_models *m, int *nck_out, int *ncols_out);
int sapr_tc_prepare(sapr_models *m);
int sapr_viterbi_tc_launch(sapr_ctx *ctx, sapr_models *m, const float *X, int ldx, const int64_t *offsets, int B,
                           int64_t total_frames, int max_T, int first_frames, int32_t *best_word, double *best_score,
                           double *scores, uint8_t *best_path, uint8_t *all_paths, float *dbgE);
int sapr_estep_tc_launch(sapr_ctx *ctx, sapr_models *m, const float *X, int ldx, const int64_t *offsets, int B, int max_T,
                         const int32_t *order, const int32_t *model_start, float *gamma, float *ustats, double *loglik);
int sapr_estep_dense(sapr_ctx *ctx, sapr_models *m, const float *X, int ldx, const int64_t *offsets, int B, int64_t total_frames,
                     int max_T, const int32_t *model_of_utt, const int32_t *order, int precision, double *stats, double *loglik,
                     void *gamma_out);
int sapr_emission_into(sapr_ctx *ctx, sapr_models *m, int mi, const float *X, int ldx, const int64_t *offsets, int B,
                       int64_t total_frames, double *E);

// ---------------------------------------------------------------------------------------------
// math helpers
// ---------------------------------------------------------------------------------------------
template <typename R> struct Num;
template <> struct Num<float> {
    static __device__ __forceinline__ float ninf() { return -INFINITY; }
};
template <> struct Num<double> {
    static __device__ __forceinline__ double ninf() { return -INFINITY; }
};

// numpy's npy_logaddexp, bit-for-bit control flow (custom_hmm.py:190,198,228,237 call np.logaddexp)
__device__ __forceinline__ double lae(double x, double y) {
    if (x == y) return x + SAPR_LN2;
    double tmp = x - y;
    if (tmp > 0) return x + log1p(exp(-tmp));
    else if (tmp <= 0) return y + log1p(exp(tmp));
    return tmp;
}
// fp32 production form: running max + fast exp/log (max abs error ~2e-7 on the log1p term)
__device__ __forceinline__ float lae(float x, float y) {
    float m = fmaxf(x, y);
    if (m == -INFINITY) return m;
    float d = -fabsf(x - y);
    return m + __logf(1.0f + __expf(d));
}
__device__ __forceinline__ float fexp(float x) { return __expf(x); }
__device__ __forceinline__ double fexp(double x) { return exp(x); }
__device__ __forceinline__ float flog(float x) { return __logf(x); }
__device__ __forceinline__ double flog(double x) { return log(x); }
