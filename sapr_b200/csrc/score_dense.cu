// score_dense.cu -- batched scoring for DENSE-topology word models (hmmlearn GaussianHMM, every state emits, S x S transmat +
// startprob): GaussianHMM.score (the forward log-likelihood log P(X_u | model m), hmmlearn_hmm.py:46-75) for every utterance x
// model, and recognition by total likelihood (the strict-'>' arg-max over the models of model.score(x)).  Semantics are those
// of k_hl_forward (hmmlearn.cu): u_0(j) = ln pi_j + e_0(j), u_t(j) = logsumexp_i (u_{t-1}(i) + ln A_ij) + e_t(j),
// score = logsumexp_j u_{T-1}(j); an empty utterance scores 0.
//
// fp32 production path, k_dense_forward<NMAX> (S <= 32, buckets 8 / 16 / 32): the grid, tile staging and shared-memory fitting
// of k_dense_viterbi (viterbi_dense.cu) -- CTA = a tile of 32 utterances, warp = one model, lane = one utterance, the tile's
// frames staged once for up to 16 models -- and the forward step of k_dense_fb (estep_dense.cu):
//   - emission cq_j + sum_d w_jd (x'_d - m_jd)^2 (df_emit_tile: no cancellation, so a one-frame utterance scores within 1e-6);
//   - u_t(j) = log2 sum_i ahat_{t-1}(i) A_ij + e_t(j) over the finite arcs grouped by destination, a sum below 2^-64 redone in
//     the log domain (de_fwd_step), ahat_t = 2^(u_t - max u_t), the shifts summed in float64 per lane;
//   - score = (sum of shifts + log2 sum_j ahat_{T-1}(j)) ln 2; -inf when the model cannot produce the utterance;
//   - no back-pointers and no per-frame scratch: no max_T, no chunking.
// k_dense_finish (scores-only) takes the arg-max and flags word near-ties; k_dense_rescore re-scores the flagged utterances in
// float64 with the arithmetic of sapr_emission_into + k_hl_forward, so their word, score and score row equal the verification
// mode's bit for bit.
//
// SAPR_FP64 (verification): sapr_hl_score per model + the running arg-max of k_dense_merge (no path).
#include <stdlib.h>

#include "dense_common.cuh"

// emission weights of the forward kernel, per model [chunk][state][8] = (m x4, w x4) with m = mu - p (p = k_dense_prepare's fp32
// pivot), w = -1 / (2 var), and cq[state] = -0.5 (D ln 2pi + sum ln var); padded dims have m = 0, w = 0.  One thread per (model,
// state), from the float64 masters on every call.
__global__ void k_dense_score_prepare(int M, int S, int D, int Dp, const double *__restrict__ mean, const double *__restrict__ var,
                                      const float *__restrict__ piv, float *__restrict__ wq, float *__restrict__ cq) {
    const int k = blockIdx.x * blockDim.x + threadIdx.x;
    if (k >= M * S) return;
    const int m = k / S, j = k % S, nch = Dp / 4;
    const double *mu = mean + (size_t)k * D, *vr = var + (size_t)k * D;
    double ld = 0.0;
    for (int d = 0; d < D; d++) ld += log(vr[d]);
    cq[k] = (float)(-0.5 * (D * SAPR_LOG2PI + ld));
    for (int c = 0; c < nch; c++)
        for (int i = 0; i < 4; i++) {
            const int d = c * 4 + i;
            const size_t o = (((size_t)m * nch + c) * S + j) * 8;
            wq[o + i] = (d < D) ? (float)(mu[d] - (double)piv[d]) : 0.f;
            wq[o + 4 + i] = (d < D) ? (float)(-0.5 / vr[d]) : 0.f;
        }
}

// emission of one staged frame (x' = x - p) in natural-log units: cq_j + sum_d w_jd (x'_d - m_jd)^2.  Every term has the sign of
// the result, so the fp32 sum loses nothing to cancellation: k_dense_viterbi's expanded form c_j + sum_d (a_jd x'_d + b_jd x'_d^2)
// cancels partial sums several times larger than the emission, which costs up to ~3e-6 relative per emission -- too much for a
// one-frame utterance, whose score is that emission.  This form keeps it below ~6e-7 at one more FADD per state and dimension.
template <int NMAX>
__device__ __forceinline__ void df_emit_tile(const float4 *xr, const float *wm, const float *cm, int S, int nch, float (&acc)[NMAX]) {
#pragma unroll
    for (int j = 0; j < NMAX; j++) acc[j] = (j < S) ? cm[j] : 0.f;
    for (int c = 0; c < nch; c++) {
        const float4 x = xr[c];
        const float4 *wc = reinterpret_cast<const float4 *>(wm + (size_t)c * S * 8);
#pragma unroll
        for (int j = 0; j < NMAX; j++) {
            if (j < S) {
                const float4 m = wc[2 * j], w = wc[2 * j + 1];
                const float4 y = make_float4(x.x - m.x, x.y - m.y, x.z - m.z, x.w - m.w);
                float e = acc[j];
                e = fmaf(w.x * y.x, y.x, e);
                e = fmaf(w.y * y.y, y.y, e);
                e = fmaf(w.z * y.z, y.z, e);
                e = fmaf(w.w * y.w, y.w, e);
                acc[j] = e;
            }
        }
    }
}

struct DfSmem {   // byte offsets of the dynamic shared memory of k_dense_forward
    size_t w, cst, lpi, arc, start, A, col, lcol, x, total;
    int xs4;      // float4 stride of an utterance row of the feature stage (odd: conflict-free lane rows)
};
static DfSmem df_smem(int mpc, int S, int nch) {
    DfSmem L;
    size_t o = 0;
    auto take = [&](size_t b) { const size_t r = o; o += (b + 15) / 16 * 16; return r; };
    L.xs4 = nch | 1;
    L.w = take((size_t)mpc * nch * S * 8 * sizeof(float));
    L.cst = take((size_t)mpc * S * sizeof(float));
    L.lpi = take((size_t)mpc * S * sizeof(float));
    L.arc = take((size_t)mpc * S * S * sizeof(float2));
    L.start = take((size_t)mpc * (S + 1) * sizeof(int32_t));
    L.A = take((size_t)mpc * S * S * sizeof(float));
    L.col = take((size_t)mpc * S * 32 * sizeof(float));
    L.lcol = take((size_t)mpc * S * 32 * sizeof(float));
    L.x = take((size_t)DN_TF * 32 * L.xs4 * sizeof(float4));
    L.total = o;
    return L;
}

// blockDim = (32, mpc): lane = utterance of the tile, warp y = model m0 + y; scores[u][m] (natural log)
template <int NMAX>
__global__ void __launch_bounds__(32 * 16, 1)
k_dense_forward(const float *__restrict__ X, int ldx, const int64_t *__restrict__ offsets, int B, int M, int S, int nch,
                const float *__restrict__ piv_g, const float *__restrict__ w_g, const float *__restrict__ cst_g,
                const float *__restrict__ lpi_g, const float2 *__restrict__ arc_g, const int32_t *__restrict__ start_g,
                const float2 *__restrict__ arcs_g, const int32_t *__restrict__ starts_g, DfSmem L, double *__restrict__ scores) {
    extern __shared__ __align__(16) unsigned char s_df[];
    __shared__ int64_t s_off[32];
    __shared__ int s_T[32];
    const int lane = threadIdx.x, warp = threadIdx.y, nthr = 32 * blockDim.y, tid = warp * 32 + lane;
    const int m0 = blockIdx.y * blockDim.y, nm = min((int)blockDim.y, M - m0);
    float *sw = reinterpret_cast<float *>(s_df + L.w);
    float *scst = reinterpret_cast<float *>(s_df + L.cst);
    float *slpi = reinterpret_cast<float *>(s_df + L.lpi);
    float2 *sarc = reinterpret_cast<float2 *>(s_df + L.arc);
    int32_t *sstart = reinterpret_cast<int32_t *>(s_df + L.start);
    float *sA = reinterpret_cast<float *>(s_df + L.A);
    float *scol = reinterpret_cast<float *>(s_df + L.col);
    float *slcol = reinterpret_cast<float *>(s_df + L.lcol);
    float4 *sx = reinterpret_cast<float4 *>(s_df + L.x);
    {   // this group's models: weights, constants, ln pi, arc lists by destination, the linear transition matrix
        const size_t nwt = (size_t)nm * nch * S * 8;
        for (size_t i = tid; i < nwt; i += nthr) sw[i] = w_g[(size_t)m0 * nch * S * 8 + i];
        for (int i = tid; i < nm * S; i += nthr) { scst[i] = cst_g[(size_t)m0 * S + i]; slpi[i] = lpi_g[(size_t)m0 * S + i]; }
        for (int i = tid; i < nm * S * S; i += nthr) { sarc[i] = arc_g[(size_t)m0 * S * S + i]; sA[i] = 0.f; }
        for (int i = tid; i < nm * (S + 1); i += nthr) sstart[i] = start_g[(size_t)m0 * (S + 1) + i];
    }
    const int ul = blockIdx.x * 32 + lane;
    int Te = 0;
    int64_t off = 0;
    if (ul < B) {
        off = offsets[ul];
        Te = (int)(offsets[ul + 1] - off);
    }
    if (warp == 0) { s_off[lane] = off; s_T[lane] = Te; }
    int Tmax = Te;
    for (int o = 16; o > 0; o >>= 1) Tmax = max(Tmax, __shfl_xor_sync(0xffffffffu, Tmax, o));
    __syncthreads();
    for (int r = tid; r < nm * S; r += nthr) {             // A_ij from the arcs grouped by source (k_dense_fb's sA)
        const int mm = r / S, i = r % S;
        const size_t mg = (size_t)m0 + mm;
        for (int k = starts_g[mg * (S + 1) + i]; k < starts_g[mg * (S + 1) + i + 1]; k++) {
            const float2 a = arcs_g[mg * S * S + k];
            sA[(size_t)mm * S * S + i * S + (int)a.y] = a.x;
        }
    }

    const bool active = warp < nm;
    const int mw = active ? warp : 0;
    const float *wm = sw + (size_t)mw * nch * S * 8;
    const float *cm = scst + mw * S, *pm = slpi + mw * S;
    const float2 *am = sarc + (size_t)mw * S * S;
    const int32_t *stm = sstart + mw * (S + 1);
    const float *Am = sA + (size_t)mw * S * S;
    float *col = scol + (size_t)mw * S * 32 + lane;       // ahat(j) of this lane at col[j * 32]
    float *lcol = slcol + (size_t)mw * S * 32 + lane;     // log2 ahat(j)
    const float NINF = -INFINITY;
    double C = 0.0;
    bool alive = Te > 0;
    for (int t0 = 0; t0 < Tmax; t0 += DN_TF) {
        __syncthreads();                                   // the previous stage is consumed (the first: sA is built)
        dn_stage(X, ldx, piv_g, s_off, s_T, t0, nch, L.xs4, sx, tid, nthr);
        __syncthreads();
        if (!active) continue;
        const int nf = min(DN_TF, Tmax - t0);
        for (int f = 0; f < nf; f++) {
            const int t = t0 + f;
            if (t >= Te || !alive) continue;
            float e[NMAX];
            df_emit_tile<NMAX>(sx + (size_t)(f * 32 + lane) * L.xs4, wm, cm, S, nch, e);
#pragma unroll
            for (int j = 0; j < NMAX; j++) e[j] *= DE_LOG2E;
            if (t == 0) {
#pragma unroll
                for (int j = 0; j < NMAX; j++) if (j < S) e[j] += __fmul_rn(pm[j], DE_LOG2E);   // ln pi in log2 units, rounded as k_dense_fb stages it
            } else {
                de_fwd_step<NMAX>(col, lcol, Am, am, stm, S, e);
            }
            float c = NINF;
#pragma unroll
            for (int j = 0; j < NMAX; j++) if (j < S) c = fmaxf(c, e[j]);
            if (!(c > NINF)) { alive = false; continue; }
#pragma unroll
            for (int j = 0; j < NMAX; j++) {
                if (j < S) {
                    const float la = e[j] - c;
                    lcol[j * 32] = la;
                    col[j * 32] = de_ex2(la);
                }
            }
            C += (double)c;
        }
    }
    if (active && ul < B) {
        double ll = Te > 0 ? -INFINITY : 0.0;             // an empty utterance scores 0, as k_hl_forward gives it
        if (alive) {
            float z = 0.f;
            for (int j = 0; j < S; j++) z += col[j * 32];
            ll = (C + log2((double)z)) * SAPR_LN2;
        }
        scores[(size_t)ul * M + m0 + mw] = ll;
    }
}

// ------------------------------------------------------------------------------------------------
// float64 re-scoring of the flagged utterances: one 32-thread block per (list entry, model), lane j = state j.  The emission is
// sapr_emission_into's expression (dn_emit64), the recursion k_hl_forward's (max, then the sum of exp over ascending sources,
// log(s) + max), so the entry's word, score and score row equal the verification mode's bit for bit.  The block that completes
// an entry's last model (counter per entry, reset to zero by it) takes the arg-max.
__global__ void __launch_bounds__(32) k_dense_rescore(const float *__restrict__ X, int ldx, const int64_t *__restrict__ offsets,
                                                      const int32_t *__restrict__ utt_list, const int32_t *__restrict__ utt_count,
                                                      int cap, int M, int S, int D, const double *__restrict__ mean,
                                                      const double *__restrict__ var, const double *__restrict__ logpi,
                                                      const double *__restrict__ logA, double *sc, int32_t *done,
                                                      int32_t *__restrict__ best_word, double *__restrict__ best_score,
                                                      double *__restrict__ scores_out) {
    const int j = threadIdx.x, jj = j < S ? j : 0;
    const int n = min(*utt_count, cap);
    for (int w = blockIdx.x; w < n * M; w += gridDim.x) {
        const int pos = w / M, mi = w % M;
        const int u = utt_list[pos];
        const int64_t off = offsets[u];
        const int T = (int)(offsets[u + 1] - off);
        const double *lpi = logpi + (size_t)mi * S, *lA = logA + (size_t)mi * S * S;
        const double *mu = mean + ((size_t)mi * S + jj) * D, *vr = var + ((size_t)mi * S + jj) * D;
        double a = -INFINITY;
        for (int t = 0; t < T; t++) {
            const double e = dn_emit64(X + (off + t) * ldx, mu, vr, D);
            if (t == 0) {
                a = lpi[jj] + e;
            } else {
                double mx = -INFINITY;
                for (int i = 0; i < S; i++) {
                    const double v = __shfl_sync(0xffffffffu, a, i) + lA[i * S + jj];
                    if (v > mx) mx = v;
                }
                double s = 0.0;
                for (int i = 0; i < S; i++) {
                    const double v = __shfl_sync(0xffffffffu, a, i) + lA[i * S + jj];
                    if (mx > -INFINITY) s += exp(v - mx);
                }
                a = ((mx > -INFINITY) ? log(s) + mx : -INFINITY) + e;
            }
        }
        double ll = 0.0;                                                 // T = 0 scores 0
        if (T > 0) {                                                     // hl_lse over the states
            double mx = -INFINITY;
            for (int i = 0; i < S; i++) {
                const double v = __shfl_sync(0xffffffffu, a, i);
                if (v > mx) mx = v;
            }
            double s = 0.0;
            for (int i = 0; i < S; i++) {
                const double v = __shfl_sync(0xffffffffu, a, i);
                if (mx > -INFINITY) s += exp(v - mx);
            }
            ll = (mx > -INFINITY) ? log(s) + mx : -INFINITY;
        }
        if (j == 0) sc[(size_t)pos * M + mi] = ll;
        __threadfence();
        __syncwarp();
        int last = 0;
        if (j == 0) last = atomicAdd(&done[pos], 1) == M - 1;
        last = __shfl_sync(0xffffffffu, last, 0);
        if (!last) continue;
        __threadfence();
        if (j != 0) continue;
        done[pos] = 0;                                                   // ready for the next call
        double bs = -INFINITY;
        int bslot = -1;
        for (int s = 0; s < M; s++) {
            const double val = __ldcg(sc + (size_t)pos * M + s);        // written by other blocks: read at the L2
            if (scores_out) scores_out[(size_t)u * M + s] = val;
            if (val > bs) { bs = val; bslot = s; }
        }
        if (best_word) best_word[u] = bslot;
        if (best_score) best_score[u] = bs;
    }
}

static int score_fp64(sapr_ctx *ctx, sapr_models *m, const float *X, int ldx, const int64_t *offsets, int B, int64_t total_frames,
                      int32_t *best_word, double *best_score, double *scores) {
    const size_t a = ((size_t)B * sizeof(double) + 255) / 256 * 256;
    int rc = sapr_ws_reserve(ctx, 9, 2 * a + (size_t)B * sizeof(int32_t));
    if (rc) return rc;
    double *lp = (double *)ctx->ws[9], *run_bs = (double *)((char *)ctx->ws[9] + a);
    int32_t *run_bw = (int32_t *)((char *)ctx->ws[9] + 2 * a);
    for (int mi = 0; mi < m->M; mi++) {
        if ((rc = sapr_hl_score(ctx, m, mi, X, ldx, offsets, B, total_frames, lp))) return rc;
        k_dense_merge<<<(B + 127) / 128, 128, 0, ctx->stream>>>(offsets, B, mi, m->M, lp, nullptr, run_bs, run_bw, best_word,
                                                                best_score, scores, nullptr);
        SAPR_LAUNCH_CHECK(ctx);
    }
    return SAPR_OK;
}

template <int NMAX>
static int score_fp32(sapr_ctx *ctx, sapr_models *m, const float *X, int ldx, const int64_t *offsets, int B, int32_t *best_word,
                      double *best_score, double *scores) {
    const int M = m->M, S = m->S, nch = m->Dp / 4;
    int mpc = std::min(M, 16);
    DfSmem L = df_smem(mpc, S, nch);
    while (mpc > 1 && L.total > 200 * 1024) L = df_smem(--mpc, S, nch);
    if (L.total > 200 * 1024) SAPR_FAIL(ctx, SAPR_E_RANGE, "score_words: model set does not fit in shared memory");
    auto kern = k_dense_forward<NMAX>;
    SAPR_CUDA(ctx, cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)L.total));
    int rc;
    if ((rc = sapr_ws_reserve(ctx, 1, (size_t)B * M * sizeof(double)))) return rc;
    double *sc_ws = (double *)ctx->ws[1];
    const size_t wqn = (size_t)M * nch * S * 8;
    if ((rc = sapr_ws_reserve(ctx, 2, sizeof(float) * (wqn + (size_t)M * S)))) return rc;
    float *wq = (float *)ctx->ws[2], *cq = wq + wqn;
    k_dense_score_prepare<<<(M * S + 127) / 128, 128, 0, ctx->stream>>>(M, S, m->D, m->Dp, m->mean, m->cov, m->dn_piv, wq, cq);
    SAPR_LAUNCH_CHECK(ctx);
    const char *ex_env = getenv("SAPR_EXACT_WORDS");
    const bool exact = !ex_env || ex_env[0] != '0';
    SaprFlag flag;
    if (exact) {
        if ((rc = sapr_flag_setup(ctx, &flag, true))) return rc;
    }
    {
        ProfScope ps(ctx, 12);
        dim3 block(32, mpc), grid((B + 31) / 32, (M + mpc - 1) / mpc);
        kern<<<grid, block, L.total, ctx->stream>>>(X, ldx, offsets, B, M, S, nch, m->dn_piv, wq, cq, m->dn_lpi,
                                                    (const float2 *)m->dn_arc, m->dn_start, (const float2 *)m->dn_arcs,
                                                    m->dn_starts, L, sc_ws);
    }
    SAPR_LAUNCH_CHECK(ctx);
    {
        ProfScope ps(ctx, 1);
        k_dense_finish<<<(B + 127) / 128, 128, 0, ctx->stream>>>(offsets, 0, B, M, 3, 1, nullptr, 0, 0, sc_ws, nullptr, best_word,
                                                                 best_score, scores, nullptr, exact ? flag : SaprFlag());
    }
    SAPR_LAUNCH_CHECK(ctx);
    if (exact) {
        if ((rc = sapr_ws_reserve(ctx, 4, (size_t)flag.cap * M * sizeof(double)))) return rc;
        ProfScope ps(ctx, 13);
        k_dense_rescore<<<8 * ctx->sm_count, 32, 0, ctx->stream>>>(X, ldx, offsets, flag.list, flag.count, flag.cap, M, S, m->D,
                                                                   m->mean, m->cov, m->logpi, m->logA, (double *)ctx->ws[4],
                                                                   flag.done, best_word, best_score, scores);
        SAPR_LAUNCH_CHECK(ctx);
    }
    return SAPR_OK;
}

extern "C" int sapr_score_words(sapr_ctx *ctx, sapr_models *m, const float *X, int ldx, const int64_t *offsets, int B,
                                int64_t total_frames, int precision, int32_t *best_word, double *best_score, double *scores) {
    if (!ctx || !m || !X || !offsets) return SAPR_E_INVALID;
    if (!m->valid) SAPR_FAIL(ctx, SAPR_E_INVALID, "score_words: model parameters not set");
    if (m->topology != SAPR_TOPO_DENSE || m->emission != SAPR_EMIT_DIAG)
        SAPR_FAIL(ctx, SAPR_E_INVALID, "score_words: needs a DENSE + DIAG model set (hmmlearn GaussianHMM); the entry/exit models' "
                                       "forward has the reference's own conventions");
    if (!best_word && !best_score && !scores) SAPR_FAIL(ctx, SAPR_E_INVALID, "score_words: no output given");
    if (ldx % 4 || ldx < m->Dp) SAPR_FAIL(ctx, SAPR_E_INVALID, "score_words: ldx must be a multiple of 4 and >= D padded");
    if (precision != SAPR_FP32 && precision != SAPR_FP64) SAPR_FAIL(ctx, SAPR_E_INVALID, "score_words: bad precision");
    if (precision == SAPR_FP32 && (m->S > 32 || !m->dn_w))
        SAPR_FAIL(ctx, SAPR_E_RANGE, "score_words: SAPR_FP32 takes up to 32 states (SAPR_FP64 runs sapr_hl_score per model; "
                                     "sapr_ergodic_score is the fp32 forward for 64-256 states)");
    ctx->flag_valid = false;
    if (B <= 0) return SAPR_OK;
    if (precision == SAPR_FP64) return score_fp64(ctx, m, X, ldx, offsets, B, total_frames, best_word, best_score, scores);
    if (m->S <= 8) return score_fp32<8>(ctx, m, X, ldx, offsets, B, best_word, best_score, scores);
    if (m->S <= 16) return score_fp32<16>(ctx, m, X, ldx, offsets, B, best_word, best_score, scores);
    return score_fp32<32>(ctx, m, X, ldx, offsets, B, best_word, best_score, scores);
}
