// hmmlearn.cu -- DENSE topology (every state emits, S x S transmat, startprob): the arithmetic the
// reference delegates to hmmlearn 0.3.3 GaussianHMM(covariance_type="diag", implementation="log")
// (hmmlearn_hmm.py:27-43, :103-104 fit/score; decoder.py:43 decode).  hmmlearn is not vendored in the
// reference; semantics follow SURVEY.md Appendix B (forward_log / backward_log / compute_log_xi_sum /
// viterbi with max-shifted logsumexp).  float64; one thread per utterance, state vectors in local
// arrays (S <= 32) -- small-N ergodic models are latency bound by nature.  For 32 < S <= 1024 (BASELINE cfg 4: the
// N = 256 ergodic model) score and decode run one CTA per utterance, one thread per state (k_hl_*_cta): same
// arithmetic and summation order, so the two mappings agree bit for bit.  The E-step for such models (k_hl_backward_stats_cta)
// is the float64 verification mode too: CTA per utterance, thread per state; the posterior normaliser is a block tree sum.
// The fp32 tensor-core forward of ergodic_tc.cu is the fast score path; a tensor-core backward / xi accumulation is not built.
#include "common.cuh"

#define HL_MAX_S 32

__device__ __forceinline__ double hl_lse(const double *v, int n) {
    double m = -INFINITY;
    for (int i = 0; i < n; i++) if (v[i] > m) m = v[i];
    if (!(m > -INFINITY)) return -INFINITY;
    double s = 0.0;
    for (int i = 0; i < n; i++) s += exp(v[i] - m);
    return log(s) + m;
}

// forward only: per-utterance log-prob
__global__ void k_hl_forward(const double *__restrict__ lf, const int64_t *__restrict__ offsets, int B, int S,
                             const double *__restrict__ logpi, const double *__restrict__ logA,
                             double *__restrict__ fwd_out, double *__restrict__ logprob) {
    const int u = blockIdx.x * blockDim.x + threadIdx.x;
    if (u >= B) return;
    const int64_t off = offsets[u];
    const int T = (int)(offsets[u + 1] - off);
    double prev[HL_MAX_S], cur[HL_MAX_S], w[HL_MAX_S];
    if (T <= 0) { logprob[u] = 0.0; return; }
    for (int i = 0; i < S; i++) {
        prev[i] = logpi[i] + lf[(size_t)off * S + i];
        if (fwd_out) fwd_out[(size_t)off * S + i] = prev[i];
    }
    for (int t = 1; t < T; t++) {
        for (int j = 0; j < S; j++) {
            for (int i = 0; i < S; i++) w[i] = prev[i] + logA[i * S + j];
            cur[j] = hl_lse(w, S) + lf[(size_t)(off + t) * S + j];
        }
        for (int j = 0; j < S; j++) {
            prev[j] = cur[j];
            if (fwd_out) fwd_out[(size_t)(off + t) * S + j] = cur[j];
        }
    }
    logprob[u] = hl_lse(prev, S);
}

// backward + posteriors + statistics for one utterance per thread; per-utterance partial statistics
// [start S | trans S*S | post S] go to pu, posteriors to post_out[sum_T][S].
__global__ void k_hl_backward_stats(const double *__restrict__ lf, const double *__restrict__ fwd,
                                    const int64_t *__restrict__ offsets, int B, int S,
                                    const double *__restrict__ logA, const double *__restrict__ logprob,
                                    double *__restrict__ bwd_ws, double *__restrict__ post_out, double *__restrict__ pu) {
    const int u = blockIdx.x * blockDim.x + threadIdx.x;
    if (u >= B) return;
    const int64_t off = offsets[u];
    const int T = (int)(offsets[u + 1] - off);
    const int len = S + S * S + S;
    double *p = pu + (size_t)u * len;
    for (int k = 0; k < len; k++) p[k] = 0.0;
    if (T <= 0) return;
    double w[HL_MAX_S];
    double *bw = bwd_ws + (size_t)off * S;
    for (int i = 0; i < S; i++) bw[(size_t)(T - 1) * S + i] = 0.0;
    for (int t = T - 2; t >= 0; t--)
        for (int i = 0; i < S; i++) {
            for (int j = 0; j < S; j++) w[j] = logA[i * S + j] + lf[(size_t)(off + t + 1) * S + j] + bw[(size_t)(t + 1) * S + j];
            bw[(size_t)t * S + i] = hl_lse(w, S);
        }
    // posteriors = exp(log_normalize(fwd + bwd))
    for (int t = 0; t < T; t++) {
        for (int j = 0; j < S; j++) w[j] = fwd[(size_t)(off + t) * S + j] + bw[(size_t)t * S + j];
        const double nrm = hl_lse(w, S);
        for (int j = 0; j < S; j++) {
            const double g = exp(w[j] - nrm);
            post_out[(size_t)(off + t) * S + j] = g;
            if (t == 0) p[j] += g;
            p[S + S * S + j] += g;
        }
    }
    // trans += exp(logsumexp_t(fwd[t,i] + logA[i,j] + lf[t+1,j] + bwd[t+1,j] - logprob))
    if (T > 1) {
        const double lp = logprob[u];
        for (int i = 0; i < S; i++)
            for (int j = 0; j < S; j++) {
                const double la_ = logA[i * S + j];
                if (!(la_ > -INFINITY)) continue;
                double mx = -INFINITY;
                for (int t = 0; t < T - 1; t++) {
                    const double v = fwd[(size_t)(off + t) * S + i] + la_ + lf[(size_t)(off + t + 1) * S + j] + bw[(size_t)(t + 1) * S + j] - lp;
                    if (v > mx) mx = v;
                }
                if (!(mx > -INFINITY)) continue;
                double s = 0.0;
                for (int t = 0; t < T - 1; t++)
                    s += exp(fwd[(size_t)(off + t) * S + i] + la_ + lf[(size_t)(off + t + 1) * S + j] + bw[(size_t)(t + 1) * S + j] - lp - mx);
                p[S + i * S + j] += exp(log(s) + mx);
            }
    }
}

// obs = post^T X, obs2 = post^T X^2: one thread per (state, dim) and frame chunk (HL_OBS_CHUNK frames in order), then a
// fixed-order sum over the chunks -- deterministic, and parallel over frames (one thread per output walking every frame
// serially took seconds at 10^7 frames).  gridDim.y stops at 65535, so a y-block takes chunks blockIdx.y, + gridDim.y, ...
#define HL_OBS_CHUNK 512
#define HL_OBS_MAX_GRID_Y 65535
__global__ void k_hl_obs_partial(const float *__restrict__ X, int ldx, int64_t total_frames, int nchunk, int D, int S,
                                 const double *__restrict__ post, double *__restrict__ part) {
    const int idx = blockIdx.x * blockDim.x + threadIdx.x;
    if (idx >= S * D) return;
    const int j = idx / D, d = idx % D;
    for (int c = blockIdx.y; c < nchunk; c += gridDim.y) {
        const int64_t f0 = (int64_t)c * HL_OBS_CHUNK, f1 = min(f0 + HL_OBS_CHUNK, total_frames);
        double a = 0.0, b = 0.0;
        for (int64_t f = f0; f < f1; f++) {
            const double g = post[f * S + j];
            const double x = (double)X[f * ldx + d];
            a += g * x;
            b += g * x * x;
        }
        part[((size_t)c * 2 + 0) * S * D + idx] = a;
        part[((size_t)c * 2 + 1) * S * D + idx] = b;
    }
}
__global__ void k_hl_obs_reduce(const double *__restrict__ part, int nchunk, int SD, double *__restrict__ obs, double *__restrict__ obs2) {
    const int idx = blockIdx.x * blockDim.x + threadIdx.x;
    if (idx >= SD) return;
    double a = 0.0, b = 0.0;
    for (int c = 0; c < nchunk; c++) { a += part[((size_t)c * 2 + 0) * SD + idx]; b += part[((size_t)c * 2 + 1) * SD + idx]; }
    obs[idx] = a; obs2[idx] = b;
}

__global__ void k_hl_sum_pu(const double *__restrict__ pu, int B, int len, double *__restrict__ out) {
    const int k = blockIdx.x * blockDim.x + threadIdx.x;
    if (k >= len) return;
    double s = 0.0;
    for (int u = 0; u < B; u++) s += pu[(size_t)u * len + k];
    out[k] = s;
}

__global__ void k_hl_viterbi(const double *__restrict__ lf, const int64_t *__restrict__ offsets, int B, int S,
                             const double *__restrict__ logpi, const double *__restrict__ logA,
                             double *__restrict__ delta_ws, double *__restrict__ logprob, int32_t *__restrict__ path) {
    const int u = blockIdx.x * blockDim.x + threadIdx.x;
    if (u >= B) return;
    const int64_t off = offsets[u];
    const int T = (int)(offsets[u + 1] - off);
    if (T <= 0) { logprob[u] = 0.0; return; }
    double *dl = delta_ws + (size_t)off * S;
    for (int i = 0; i < S; i++) dl[i] = logpi[i] + lf[(size_t)off * S + i];
    for (int t = 1; t < T; t++)
        for (int j = 0; j < S; j++) {
            double m = -INFINITY;
            for (int i = 0; i < S; i++) {
                const double v = dl[(size_t)(t - 1) * S + i] + logA[i * S + j];
                if (v > m) m = v;
            }
            dl[(size_t)t * S + j] = m + lf[(size_t)(off + t) * S + j];
        }
    int cur = 0;
    double best = dl[(size_t)(T - 1) * S];
    for (int i = 1; i < S; i++) if (dl[(size_t)(T - 1) * S + i] > best) { best = dl[(size_t)(T - 1) * S + i]; cur = i; }
    path[off + T - 1] = cur;
    for (int t = T - 2; t >= 0; t--) {
        int arg = 0;
        double m = dl[(size_t)t * S] + logA[0 * S + cur];
        for (int i = 1; i < S; i++) {
            const double v = dl[(size_t)t * S + i] + logA[i * S + cur];
            if (v > m) { m = v; arg = i; }
        }
        cur = arg;
        path[off + t] = cur;
    }
    logprob[u] = best;
}

// ---- one CTA per utterance, one thread per destination state (32 < S <= 1024) ----
// __launch_bounds__(HL_MAX_S_CTA) caps these kernels at 64 registers, so a 1024-thread block always fits the register file
#define HL_MAX_S_CTA 1024
__global__ void __launch_bounds__(HL_MAX_S_CTA) k_hl_forward_cta(const double *__restrict__ lf, const int64_t *__restrict__ offsets, int S,
                                 const double *__restrict__ logpi, const double *__restrict__ logA,
                                 double *__restrict__ fwd_out, double *__restrict__ logprob) {
    extern __shared__ double sh_prev[];   // [S]
    const int u = blockIdx.x, j = threadIdx.x;
    const int64_t off = offsets[u];
    const int T = (int)(offsets[u + 1] - off);
    if (T <= 0) { if (j == 0) logprob[u] = 0.0; return; }
    if (j < S) {
        sh_prev[j] = logpi[j] + lf[(size_t)off * S + j];
        if (fwd_out) fwd_out[(size_t)off * S + j] = sh_prev[j];
    }
    __syncthreads();
    for (int t = 1; t < T; t++) {
        double cur = 0.0;
        if (j < S) {
            double m = -INFINITY;
            for (int i = 0; i < S; i++) { const double v = sh_prev[i] + logA[(size_t)i * S + j]; if (v > m) m = v; }
            double r = -INFINITY;
            if (m > -INFINITY) {
                double s = 0.0;
                for (int i = 0; i < S; i++) s += exp(sh_prev[i] + logA[(size_t)i * S + j] - m);
                r = log(s) + m;
            }
            cur = r + lf[(size_t)(off + t) * S + j];
        }
        __syncthreads();
        if (j < S) {
            sh_prev[j] = cur;
            if (fwd_out) fwd_out[(size_t)(off + t) * S + j] = cur;
        }
        __syncthreads();
    }
    if (j == 0) logprob[u] = hl_lse(sh_prev, S);
}

// block-wide max / sum over the first S threads' values (fixed tree order: deterministic)
__device__ __forceinline__ double hl_block_reduce(double v, bool is_max, double *sh_red) {
    const int lane = threadIdx.x & 31, w = threadIdx.x >> 5, nw = blockDim.x >> 5;
    for (int o = 16; o > 0; o >>= 1) {
        const double x = __shfl_xor_sync(0xffffffffu, v, o);
        v = is_max ? fmax(v, x) : v + x;
    }
    __syncthreads();
    if (lane == 0) sh_red[w] = v;
    __syncthreads();
    double r = sh_red[0];
    for (int i = 1; i < nw; i++) r = is_max ? fmax(r, sh_red[i]) : r + sh_red[i];
    return r;
}

// backward + posteriors + statistics, one CTA per utterance at a time (CTA b takes utterances b, b + grid, ...),
// one thread per state; the CTA's partial statistics [start S | trans S*S | post S] accumulate in pc[b] (zeroed here).
// Capped at 64 registers for 1024 threads this kernel spills (32 / 40 bytes of stores / loads a thread), so blocks of up to
// HL_BWD_CTA_NOSPILL threads take an instance bounded at 768 threads: 80 registers, no spills.  Same arithmetic in both.
#define HL_BWD_CTA_NOSPILL 768
template <int MAX_THREADS>
__global__ void __launch_bounds__(MAX_THREADS, 1) k_hl_backward_stats_cta(const double *__restrict__ lf, const double *__restrict__ fwd,
                                        const int64_t *__restrict__ offsets, int B, int S,
                                        const double *__restrict__ logA, const double *__restrict__ logprob,
                                        double *__restrict__ bwd_ws, double *__restrict__ post_out, double *__restrict__ pc) {
    extern __shared__ double sh[];        // [S] next-frame term c_j = lf[t+1][j] + bwd[t+1][j]  |  [32] reduction scratch
    double *sh_c = sh, *sh_red = sh + S;
    const int j = threadIdx.x;
    const int len = S + S * S + S;
    double *p = pc + (size_t)blockIdx.x * len;
    for (int k = j; k < len; k += blockDim.x) p[k] = 0.0;
    __syncthreads();
    for (int u = blockIdx.x; u < B; u += gridDim.x) {
        const int64_t off = offsets[u];
        const int T = (int)(offsets[u + 1] - off);
        if (T <= 0) continue;
        double *bw = bwd_ws + (size_t)off * S;
        if (j < S) bw[(size_t)(T - 1) * S + j] = 0.0;
        for (int t = T - 2; t >= 0; t--) {
            __syncthreads();
            if (j < S) sh_c[j] = lf[(size_t)(off + t + 1) * S + j] + bw[(size_t)(t + 1) * S + j];
            __syncthreads();
            if (j < S) {                                   // thread = source state i
                const double *la = logA + (size_t)j * S;
                double m = -INFINITY;
                for (int k = 0; k < S; k++) { const double v = la[k] + sh_c[k]; if (v > m) m = v; }
                double r = -INFINITY;
                if (m > -INFINITY) {
                    double sm = 0.0;
                    for (int k = 0; k < S; k++) sm += exp(la[k] + sh_c[k] - m);
                    r = log(sm) + m;
                }
                bw[(size_t)t * S + j] = r;
            }
        }
        __syncthreads();
        // posteriors = exp(log_normalize(fwd + bwd))
        double g0 = 0.0, gsum = 0.0;
        for (int t = 0; t < T; t++) {
            const double w = (j < S) ? fwd[(size_t)(off + t) * S + j] + bw[(size_t)t * S + j] : -INFINITY;
            const double mx = hl_block_reduce(w, true, sh_red);
            const double e = (j < S && mx > -INFINITY) ? exp(w - mx) : 0.0;
            const double sm = hl_block_reduce(e, false, sh_red);
            const double g = (j < S && mx > -INFINITY) ? exp(w - (log(sm) + mx)) : 0.0;
            if (j < S) post_out[(size_t)(off + t) * S + j] = g;
            if (t == 0) g0 = g;
            gsum += g;
        }
        if (j < S) { p[j] += g0; p[S + S * S + j] += gsum; }
        // trans[i][j] += exp(logsumexp_t(fwd[t,i] + logA[i,j] + lf[t+1,j] + bwd[t+1,j] - logprob)); thread = destination j
        if (T > 1 && j < S) {
            const double lp = logprob[u];
            for (int i = 0; i < S; i++) {
                const double la_ = logA[(size_t)i * S + j];
                if (!(la_ > -INFINITY)) continue;
                double mx = -INFINITY;
                for (int t = 0; t < T - 1; t++) {
                    const double v = fwd[(size_t)(off + t) * S + i] + la_ + lf[(size_t)(off + t + 1) * S + j] + bw[(size_t)(t + 1) * S + j] - lp;
                    if (v > mx) mx = v;
                }
                if (!(mx > -INFINITY)) continue;
                double sm = 0.0;
                for (int t = 0; t < T - 1; t++)
                    sm += exp(fwd[(size_t)(off + t) * S + i] + la_ + lf[(size_t)(off + t + 1) * S + j] + bw[(size_t)(t + 1) * S + j] - lp - mx);
                p[S + (size_t)i * S + j] += exp(log(sm) + mx);
            }
        }
        __syncthreads();
    }
}

__global__ void __launch_bounds__(HL_MAX_S_CTA) k_hl_viterbi_cta(const double *__restrict__ lf, const int64_t *__restrict__ offsets, int S,
                                 const double *__restrict__ logpi, const double *__restrict__ logA,
                                 double *__restrict__ delta_ws, double *__restrict__ logprob, int32_t *__restrict__ path) {
    const int u = blockIdx.x, j = threadIdx.x;
    const int64_t off = offsets[u];
    const int T = (int)(offsets[u + 1] - off);
    if (T <= 0) { if (j == 0) logprob[u] = 0.0; return; }
    double *dl = delta_ws + (size_t)off * S;
    if (j < S) dl[j] = logpi[j] + lf[(size_t)off * S + j];
    __syncthreads();
    for (int t = 1; t < T; t++) {
        if (j < S) {
            double m = -INFINITY;
            for (int i = 0; i < S; i++) {
                const double v = dl[(size_t)(t - 1) * S + i] + logA[(size_t)i * S + j];
                if (v > m) m = v;
            }
            dl[(size_t)t * S + j] = m + lf[(size_t)(off + t) * S + j];
        }
        __syncthreads();      // global writes of this CTA are visible to it after the barrier
    }
    if (j == 0) {            // terminal arg-max and back-trace: first maximum wins (lowest index)
        int cur = 0;
        double best = dl[(size_t)(T - 1) * S];
        for (int i = 1; i < S; i++) if (dl[(size_t)(T - 1) * S + i] > best) { best = dl[(size_t)(T - 1) * S + i]; cur = i; }
        path[off + T - 1] = cur;
        for (int t = T - 2; t >= 0; t--) {
            int arg = 0;
            double m = dl[(size_t)t * S] + logA[cur];
            for (int i = 1; i < S; i++) {
                const double v = dl[(size_t)t * S + i] + logA[(size_t)i * S + cur];
                if (v > m) { m = v; arg = i; }
            }
            cur = arg;
            path[off + t] = cur;
        }
        logprob[u] = best;
    }
}

#define HL_CHECK(fn)                                                                             \
    if (!ctx || !m || !X || !offsets) return SAPR_E_INVALID;                                     \
    if (!m->valid) SAPR_FAIL(ctx, SAPR_E_INVALID, fn ": model parameters not set");              \
    if (mi < 0 || mi >= m->M) SAPR_FAIL(ctx, SAPR_E_INVALID, fn ": model index out of range");   \
    if (m->topology != SAPR_TOPO_DENSE || m->emission != SAPR_EMIT_DIAG)                         \
        SAPR_FAIL(ctx, SAPR_E_INVALID, fn ": needs DENSE topology + DIAG emission");             \
    if (m->S > HL_MAX_S_CTA) SAPR_FAIL(ctx, SAPR_E_RANGE, fn ": more than 1024 states")

// thread per utterance needs thousands of utterances to fill the GPU; below that (the reference's 30 utterances per word) one
// CTA per utterance with a thread per state is the faster mapping
static bool hl_thread_per_utt(const sapr_ctx *ctx, int S, int B) { return S <= HL_MAX_S && B >= 16 * ctx->sm_count; }

extern "C" int64_t sapr_hl_stats_len(int S, int D) { return (int64_t)S + (int64_t)S * S + S + 2 * (int64_t)S * D; }

extern "C" int sapr_hl_score(sapr_ctx *ctx, sapr_models *m, int mi, const float *X, int ldx, const int64_t *offsets,
                             int B, int64_t total_frames, double *logprob) {
    HL_CHECK("hl_score");
    const int S = m->S;
    int rc = sapr_ws_reserve(ctx, 4, sizeof(double) * (size_t)total_frames * S);
    if (rc) return rc;
    double *lf = (double *)ctx->ws[4];
    if ((rc = sapr_emission_into(ctx, m, mi, X, ldx, offsets, B, total_frames, lf))) return rc;
    if (hl_thread_per_utt(ctx, S, B))
        k_hl_forward<<<(B + 31) / 32, 32, 0, ctx->stream>>>(lf, offsets, B, S, m->logpi + (size_t)mi * S,
                                                            m->logA + (size_t)mi * S * S, nullptr, logprob);
    else
        k_hl_forward_cta<<<B, (S + 31) / 32 * 32, sizeof(double) * S, ctx->stream>>>(lf, offsets, S, m->logpi + (size_t)mi * S,
                                                                                     m->logA + (size_t)mi * S * S, nullptr, logprob);
    SAPR_LAUNCH_CHECK(ctx);
    return SAPR_OK;
}

extern "C" int sapr_hl_decode(sapr_ctx *ctx, sapr_models *m, int mi, const float *X, int ldx, const int64_t *offsets,
                              int B, int64_t total_frames, double *logprob, int32_t *path) {
    HL_CHECK("hl_decode");
    const int S = m->S;
    int rc = sapr_ws_reserve(ctx, 4, sizeof(double) * (size_t)total_frames * S * 2);
    if (rc) return rc;
    double *lf = (double *)ctx->ws[4], *dl = lf + (size_t)total_frames * S;
    if ((rc = sapr_emission_into(ctx, m, mi, X, ldx, offsets, B, total_frames, lf))) return rc;
    if (hl_thread_per_utt(ctx, S, B))
        k_hl_viterbi<<<(B + 31) / 32, 32, 0, ctx->stream>>>(lf, offsets, B, S, m->logpi + (size_t)mi * S,
                                                            m->logA + (size_t)mi * S * S, dl, logprob, path);
    else
        k_hl_viterbi_cta<<<B, (S + 31) / 32 * 32, 0, ctx->stream>>>(lf, offsets, S, m->logpi + (size_t)mi * S,
                                                                    m->logA + (size_t)mi * S * S, dl, logprob, path);
    SAPR_LAUNCH_CHECK(ctx);
    return SAPR_OK;
}

extern "C" int sapr_hl_estep(sapr_ctx *ctx, sapr_models *m, int mi, const float *X, int ldx, const int64_t *offsets,
                             int B, int64_t total_frames, double *stats, double *logprob) {
    HL_CHECK("hl_estep");
    if (!stats || !logprob) return SAPR_E_INVALID;
    const int S = m->S, D = m->D;
    const size_t lat = (size_t)total_frames * S;
    const int len = S + S * S + S;
    // partial statistics: one slot per utterance (S <= 32, thread per utterance) or per CTA (larger S, CTA per utterance)
    const bool tpu = hl_thread_per_utt(ctx, S, B);
    const int nslots = tpu ? B : std::min(B, 2 * ctx->sm_count);
    int rc = sapr_ws_reserve(ctx, 4, sizeof(double) * (4 * lat + (size_t)nslots * len));
    if (rc) return rc;
    double *lf = (double *)ctx->ws[4], *fwd = lf + lat, *bwd = fwd + lat, *post = bwd + lat, *pu = post + lat;
    if ((rc = sapr_emission_into(ctx, m, mi, X, ldx, offsets, B, total_frames, lf))) return rc;
    const double *logpi = m->logpi + (size_t)mi * S, *logA = m->logA + (size_t)mi * S * S;
    if (tpu) {
        k_hl_forward<<<(B + 31) / 32, 32, 0, ctx->stream>>>(lf, offsets, B, S, logpi, logA, fwd, logprob);
        SAPR_LAUNCH_CHECK(ctx);
        k_hl_backward_stats<<<(B + 31) / 32, 32, 0, ctx->stream>>>(lf, fwd, offsets, B, S, logA, logprob, bwd, post, pu);
        SAPR_LAUNCH_CHECK(ctx);
    } else {
        const int threads = (S + 31) / 32 * 32;
        k_hl_forward_cta<<<B, threads, sizeof(double) * S, ctx->stream>>>(lf, offsets, S, logpi, logA, fwd, logprob);
        SAPR_LAUNCH_CHECK(ctx);
        auto *bwd_stats = threads <= HL_BWD_CTA_NOSPILL ? k_hl_backward_stats_cta<HL_BWD_CTA_NOSPILL> : k_hl_backward_stats_cta<HL_MAX_S_CTA>;
        bwd_stats<<<nslots, threads, sizeof(double) * (S + 32), ctx->stream>>>(lf, fwd, offsets, B, S, logA, logprob, bwd, post, pu);
        SAPR_LAUNCH_CHECK(ctx);
    }
    k_hl_sum_pu<<<(len + 63) / 64, 64, 0, ctx->stream>>>(pu, nslots, len, stats);
    SAPR_LAUNCH_CHECK(ctx);
    const int nchunk = (int)((total_frames + HL_OBS_CHUNK - 1) / HL_OBS_CHUNK);
    if ((rc = sapr_ws_reserve(ctx, 5, sizeof(double) * (size_t)std::max(nchunk, 1) * 2 * S * D))) return rc;
    if (nchunk > 0) {
        k_hl_obs_partial<<<dim3((S * D + 63) / 64, std::min(nchunk, HL_OBS_MAX_GRID_Y)), 64, 0, ctx->stream>>>(
            X, ldx, total_frames, nchunk, D, S, post, (double *)ctx->ws[5]);
        SAPR_LAUNCH_CHECK(ctx);
    }
    k_hl_obs_reduce<<<(S * D + 63) / 64, 64, 0, ctx->stream>>>((const double *)ctx->ws[5], nchunk, S * D, stats + len, stats + len + (size_t)S * D);
    SAPR_LAUNCH_CHECK(ctx);
    return SAPR_OK;
}

// ---- hmmlearn 0.3.3 GaussianHMM._do_mstep ('diag'), every model of the set at once, bit for bit with the numpy expression of
// hmmlearn_hmm.py: same operation order, no FMA contraction (__d*_rn), numpy's NaN-propagating maximum and its pairwise sum.
__device__ __forceinline__ double np_maximum(double a, double b) { return (a >= b || a != a) ? a : b; }

// numpy's pairwise_sum of a contiguous float64 row (what sp.sum() and tm.sum(axis=1) run): sequential below 8 elements, eight
// strided accumulators up to 128, above that split at n/2 rounded down to a multiple of 8.  L bounds the recursion: the larger
// half is at most n/2 + 8, so 5 levels take n <= 1024 down to <= 128.
__device__ __forceinline__ double np_block_sum(const double *a, int n) {
    if (n < 8) {
        double r = -0.0;
        for (int i = 0; i < n; i++) r = __dadd_rn(r, a[i]);
        return r;
    }
    double r[8];
    for (int k = 0; k < 8; k++) r[k] = a[k];
    int i = 8;
    for (; i < n - (n % 8); i += 8)
        for (int k = 0; k < 8; k++) r[k] = __dadd_rn(r[k], a[i + k]);
    double s = __dadd_rn(__dadd_rn(__dadd_rn(r[0], r[1]), __dadd_rn(r[2], r[3])), __dadd_rn(__dadd_rn(r[4], r[5]), __dadd_rn(r[6], r[7])));
    for (; i < n; i++) s = __dadd_rn(s, a[i]);
    return s;
}
template <int L> __device__ double np_pairwise_sum(const double *a, int n) {
    if (n <= 128) return np_block_sum(a, n);
    int n2 = n / 2;
    n2 -= n2 % 8;
    return __dadd_rn(np_pairwise_sum<L - 1>(a, n2), np_pairwise_sum<L - 1>(a + n2, n - n2));
}
template <> __device__ double np_pairwise_sum<0>(const double *a, int n) { return np_block_sum(a, n); }
// numpy's sum reduction adds the pairwise sum to its identity 0.0
__device__ __forceinline__ double np_sum(const double *a, int n) { return __dadd_rn(0.0, np_pairwise_sum<5>(a, n)); }

// one CTA per model: thread 0 the start probabilities, a thread per transmat row, a thread per (state, dim) for the mean and the
// variance (the variance reads the new mean from the same thread).  The normalisations work in place: a row's zero mask reads
// the old value of the element it replaces.
__global__ void k_hl_mstep(int S, int D, const double *__restrict__ stats, const double *__restrict__ priors,
                           const int32_t *__restrict__ flags, double *__restrict__ mean, double *__restrict__ cov,
                           double *__restrict__ A, double *__restrict__ pi) {
    const int mi = blockIdx.x;
    const int f = flags[mi];
    if (!f) return;
    const size_t SD = (size_t)S * D;
    const double *start = stats + (size_t)mi * (S + (size_t)S * S + S + 2 * SD), *trans = start + S, *post = trans + (size_t)S * S,
                 *obs = post + S, *obs2 = obs + SD;
    const double *spp = priors + (size_t)mi * (S + (size_t)S * S + 3 * SD + 1), *tmp = spp + S, *mp = tmp + (size_t)S * S,
                 *mw = mp + SD, *cp = mw + SD;
    double *pim = pi + (size_t)mi * S, *Am = A + (size_t)mi * S * S, *mu = mean + (size_t)mi * SD, *var = cov + (size_t)mi * SD;
    if ((f & 1) && threadIdx.x == 0) {                 // 's': sp = max(startprob_prior - 1 + start, 0), masked, / sp.sum()
        for (int j = 0; j < S; j++) {
            const double v = np_maximum(__dadd_rn(__dsub_rn(spp[j], 1.0), start[j]), 0.0);
            pim[j] = (pim[j] == 0.0) ? 0.0 : v;
        }
        const double s = np_sum(pim, S);
        for (int j = 0; j < S; j++) pim[j] = __ddiv_rn(pim[j], s);
    }
    if (f & 2)                                         // 't': the same per row; a row summing to 0 is divided by 1
        for (int i = threadIdx.x; i < S; i += blockDim.x) {
            double *row = Am + (size_t)i * S;
            const double *tr = trans + (size_t)i * S, *tp = tmp + (size_t)i * S;
            for (int j = 0; j < S; j++) {
                const double v = np_maximum(__dadd_rn(__dsub_rn(tp[j], 1.0), tr[j]), 0.0);
                row[j] = (row[j] == 0.0) ? 0.0 : v;
            }
            double rs = np_sum(row, S);
            if (rs == 0.0) rs = 1.0;
            for (int j = 0; j < S; j++) row[j] = __ddiv_rn(row[j], rs);
        }
    if (f & 12) {
        const double cwm = __dsub_rn(cp[SD], 1.0);     // max(covars_weight - 1, 0), Python's max
        const double cw0 = (0.0 > cwm) ? 0.0 : cwm;
        for (size_t k = threadIdx.x; k < SD; k += blockDim.x) {
            const double denom = post[k / D];
            double m = mu[k];
            if (f & 4)                                 // 'm': (mw * mp + obs) / (mw + post)
                m = __ddiv_rn(__dadd_rn(__dmul_rn(mw[k], mp[k]), obs[k]), __dadd_rn(mw[k], denom));
            if (f & 8) {                               // 'c': (cp + c_n) / max(c_d, 1e-5) around the (new) mean
                const double md = __dsub_rn(m, mp[k]);
                const double cn = __dadd_rn(__dsub_rn(__dadd_rn(__dmul_rn(mw[k], __dmul_rn(md, md)), obs2[k]), __dmul_rn(__dmul_rn(2.0, m), obs[k])),
                                            __dmul_rn(__dmul_rn(m, m), denom));
                var[k] = __ddiv_rn(__dadd_rn(cp[k], cn), np_maximum(__dadd_rn(cw0, denom), 1e-5));
            }
            mu[k] = m;
        }
    }
}

extern "C" int sapr_hl_mstep(sapr_ctx *ctx, sapr_models *m, const double *stats, const double *priors, const int32_t *flags_host) {
    if (!ctx || !m || !stats || !priors || !flags_host) return SAPR_E_INVALID;
    if (m->topology != SAPR_TOPO_DENSE || m->emission != SAPR_EMIT_DIAG)
        SAPR_FAIL(ctx, SAPR_E_INVALID, "hl_mstep: needs DENSE topology + DIAG emission");
    if (!m->valid) SAPR_FAIL(ctx, SAPR_E_INVALID, "hl_mstep: model parameters not set");
    if (m->S > HL_MAX_S_CTA) SAPR_FAIL(ctx, SAPR_E_RANGE, "hl_mstep: more than 1024 states");
    int rc = sapr_ws_reserve(ctx, 5, sizeof(int32_t) * m->M);
    if (rc) return rc;
    // a copy from pageable memory has consumed the source when it returns: no stream synchronisation is needed
    SAPR_CUDA(ctx, cudaMemcpyAsync(ctx->ws[5], flags_host, sizeof(int32_t) * m->M, cudaMemcpyHostToDevice, ctx->stream));
    {
        ProfScope ps(ctx, 11);
        k_hl_mstep<<<m->M, 256, 0, ctx->stream>>>(m->S, m->D, stats, priors, (const int32_t *)ctx->ws[5], m->mean, m->cov, m->A, m->pi);
    }
    SAPR_LAUNCH_CHECK(ctx);
    return sapr_models_prepare(m);
}
