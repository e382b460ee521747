// viterbi_dense.cu -- batched Viterbi for DENSE-topology word models (hmmlearn GaussianHMM, every state emits,
// S x S transmat + startprob): decoder.py:42-47 with model.decode = GaussianHMM.decode for every utterance x model, and the
// strict-'>' arg-max over the models.  Semantics are those of k_hl_viterbi (hmmlearn.cu): delta_0(j) = ln pi_j + e_0(j),
// delta_t(j) = max_i (delta_{t-1}(i) + ln A_ij) + e_t(j), score = max_j delta_{T-1}(j), first maximum (lowest index) at every
// step of the back-trace.
//
// fp32 production path, k_dense_viterbi<NMAX>: CTA = a tile of 32 utterances, warp = one model, lane = one utterance.
//   - the tile's frames are staged once in shared memory (pivot-centred, x' = x - p) and every model warp of the CTA reads them:
//     HBM sees each feature once per model group (one group up to 16 models);
//   - emission per state c_j + sum_d (a_jd x'_d + b_jd x'_d^2) with a = (mu - p) / var, b = -1/(2 var): two FMAs per dimension,
//     parameters are warp-uniform shared-memory broadcasts;
//   - transitions are a per-model list of the finite arcs grouped by destination (built by sapr_models_prepare): a model trained
//     from the reference's left-to-right initialisation keeps its zero pattern (the M-step maps zeros to zeros) and costs 2S - 2
//     arcs per frame, a fully dense matrix S^2;
//   - the state vector is renormalised every frame (max subtracted, the offset carried in float64 per lane);
//   - back-pointers: ceil(log2 NMAX) bits per state and frame for every model, [model][frame][word][utterance] so a warp store
//     is one coalesced line (DESIGN §4 has the measured cost against a scores-only launch).
// k_dense_finish takes the arg-max over the models (strict >, first best wins, -1 when every model scores -inf), flags word
// near-ties (sapr_flag_word) and traces the winner's path; k_dense_redo re-decodes the flagged utterances in float64 with the
// arithmetic of sapr_emission_into + k_hl_viterbi, so their outputs equal the verification mode's bit for bit.
//
// SAPR_FP64 (verification): sapr_hl_decode per model + a running arg-max kernel.
#include <stdlib.h>

#include "dense_common.cuh"

template <int NMAX> struct DnBits {
    static constexpr int NB = NMAX <= 8 ? 3 : (NMAX <= 16 ? 4 : 5);   // bits per state
    static constexpr int PER = 32 / NB;                                 // states per back-pointer word
    static constexpr int NW = (NMAX + PER - 1) / PER;
};
static int dn_nb(int S) { return S <= 8 ? 3 : (S <= 16 ? 4 : 5); }

// ------------------------------------------------------------------------------------------------
// derived parameters (sapr_models_prepare): pivot, fp32 emission weights, ln pi, arc lists (by destination with ln A for the
// Viterbi, by source with A and log2 A for the E-step's backward sweep, csrc/estep_dense.cu).  One block.
__global__ void k_dense_prepare(int M, int S, int D, int Dp, const double *__restrict__ mean, const double *__restrict__ var,
                                const double *__restrict__ A, const double *__restrict__ pi, float *__restrict__ piv,
                                float *__restrict__ w, float *__restrict__ cst, float *__restrict__ lpi, float2 *__restrict__ arc,
                                int32_t *__restrict__ start, float2 *__restrict__ arcs, float *__restrict__ lg2s,
                                int32_t *__restrict__ starts) {
    __shared__ double s_p[1024];
    const int nch = Dp / 4;
    for (int d = threadIdx.x; d < Dp; d += blockDim.x) {
        double s = 0.0;
        if (d < D)
            for (int k = 0; k < M * S; k++) s += mean[(size_t)k * D + d];
        s_p[d] = (d < D) ? s / (M * S) : 0.0;
        piv[d] = (float)s_p[d];
    }
    __syncthreads();
    for (int k = threadIdx.x; k < M * S; k += blockDim.x) {   // (model, state)
        const int m = k / S, j = k % S;
        const double *mu = mean + (size_t)k * D, *vr = var + (size_t)k * D;
        double ld = 0.0, q = 0.0;
        for (int d = 0; d < D; d++) {
            ld += log(vr[d]);
            const double dm = mu[d] - (double)(float)s_p[d];
            q += dm * dm / vr[d];
        }
        cst[k] = (float)(-0.5 * (D * SAPR_LOG2PI + ld + q));
        lpi[k] = (float)log(pi[k]);
        for (int c = 0; c < nch; c++)
            for (int i = 0; i < 4; i++) {
                const int d = c * 4 + i;
                const size_t o = (((size_t)m * nch + c) * S + j) * 8;
                w[o + i] = (d < D) ? (float)((mu[d] - (double)(float)s_p[d]) / vr[d]) : 0.f;
                w[o + 4 + i] = (d < D) ? (float)(-0.5 / vr[d]) : 0.f;
            }
    }
    for (int m = threadIdx.x; m < M; m += blockDim.x) {       // finite arcs grouped by destination, sources ascending
        const double *Am = A + (size_t)m * S * S;
        int n = 0;
        for (int j = 0; j < S; j++) {
            start[(size_t)m * (S + 1) + j] = n;
            for (int i = 0; i < S; i++) {
                const double la = log(Am[(size_t)i * S + j]);
                if (la > -INFINITY) arc[(size_t)m * S * S + n++] = make_float2((float)la, (float)i);
            }
        }
        start[(size_t)m * (S + 1) + S] = n;
        n = 0;
        for (int i = 0; i < S; i++) {                          // the same arcs grouped by source, destinations ascending
            starts[(size_t)m * (S + 1) + i] = n;
            for (int j = 0; j < S; j++) {
                const double a = Am[(size_t)i * S + j];
                if (log(a) > -INFINITY) {
                    lg2s[(size_t)m * S * S + n] = (float)log2(a);   // finite in fp32 where (float)a is 0 or a denormal
                    arcs[(size_t)m * S * S + n++] = make_float2((float)a, (float)j);
                }
            }
        }
        starts[(size_t)m * (S + 1) + S] = n;
    }
}

int sapr_dense_prepare(sapr_models *m) {
    sapr_ctx *ctx = m->ctx;
    k_dense_prepare<<<1, 256, 0, ctx->stream>>>(m->M, m->S, m->D, m->Dp, m->mean, m->cov, m->A, m->pi, m->dn_piv, m->dn_w,
                                                m->dn_cst, m->dn_lpi, (float2 *)m->dn_arc, m->dn_start,
                                                (float2 *)m->dn_arcs, m->dn_lg2s, m->dn_starts);
    SAPR_LAUNCH_CHECK(ctx);
    return SAPR_OK;
}

// ------------------------------------------------------------------------------------------------
struct DnSmem {   // byte offsets of the dynamic shared memory of k_dense_viterbi
    size_t w, cst, lpi, arc, start, delta, x, total;
    int xs4;      // float4 stride of an utterance row of the feature stage (odd: conflict-free lane rows)
};
static DnSmem dn_smem(int mpc, int S, int nch) {
    DnSmem L;
    size_t o = 0;
    auto take = [&](size_t b) { const size_t r = o; o += (b + 15) / 16 * 16; return r; };
    L.xs4 = nch | 1;
    L.w = take((size_t)mpc * nch * S * 8 * sizeof(float));
    L.cst = take((size_t)mpc * S * sizeof(float));
    L.lpi = take((size_t)mpc * S * sizeof(float));
    L.arc = take((size_t)mpc * S * S * sizeof(float2));
    L.start = take((size_t)mpc * (S + 1) * sizeof(int32_t));
    L.delta = take((size_t)mpc * S * 32 * sizeof(float));
    L.x = take((size_t)DN_TF * 32 * L.xs4 * sizeof(float4));
    L.total = o;
    return L;
}

// blockDim = (32, mpc): lane = utterance of the tile, warp y = model m0 + y
template <int NMAX>
__global__ void __launch_bounds__(32 * 16, 1)
k_dense_viterbi(const float *__restrict__ X, int ldx, const int64_t *__restrict__ offsets, int u0, int nu, int M, int S, int nch,
                const float *__restrict__ piv_g, const float *__restrict__ w_g, const float *__restrict__ cst_g,
                const float *__restrict__ lpi_g, const float2 *__restrict__ arc_g, const int32_t *__restrict__ start_g, DnSmem L,
                uint32_t *__restrict__ bp, int64_t Bpad, int maxT, int nw, double *__restrict__ scores, uint8_t *__restrict__ last_state) {
    using BB = DnBits<NMAX>;
    extern __shared__ __align__(16) unsigned char s_dn[];
    __shared__ int64_t s_off[32];
    __shared__ int s_T[32];
    const int lane = threadIdx.x, warp = threadIdx.y, nthr = 32 * blockDim.y, tid = warp * 32 + lane;
    const int m0 = blockIdx.y * blockDim.y, nm = min((int)blockDim.y, M - m0);
    float *sw = reinterpret_cast<float *>(s_dn + L.w);
    float *scst = reinterpret_cast<float *>(s_dn + L.cst);
    float *slpi = reinterpret_cast<float *>(s_dn + L.lpi);
    float2 *sarc = reinterpret_cast<float2 *>(s_dn + L.arc);
    int32_t *sstart = reinterpret_cast<int32_t *>(s_dn + L.start);
    float *sdel = reinterpret_cast<float *>(s_dn + L.delta);
    float4 *sx = reinterpret_cast<float4 *>(s_dn + L.x);
    {   // this group's models: weights, constants, ln pi, arc lists
        const size_t nwt = (size_t)nm * nch * S * 8;
        for (size_t i = tid; i < nwt; i += nthr) sw[i] = w_g[(size_t)m0 * nch * S * 8 + i];
        for (int i = tid; i < nm * S; i += nthr) { scst[i] = cst_g[(size_t)m0 * S + i]; slpi[i] = lpi_g[(size_t)m0 * S + i]; }
        for (int i = tid; i < nm * S * S; i += nthr) sarc[i] = arc_g[(size_t)m0 * S * S + i];
        for (int i = tid; i < nm * (S + 1); i += nthr) sstart[i] = start_g[(size_t)m0 * (S + 1) + i];
    }
    const int ul = blockIdx.x * 32 + lane;
    int Te = 0;
    int64_t off = 0;
    if (ul < nu) {
        off = offsets[u0 + ul];
        Te = min((int)(offsets[u0 + ul + 1] - off), maxT);
    }
    if (warp == 0) { s_off[lane] = off; s_T[lane] = Te; }
    int Tmax = Te;
    for (int o = 16; o > 0; o >>= 1) Tmax = max(Tmax, __shfl_xor_sync(0xffffffffu, Tmax, o));
    __syncthreads();

    const bool active = warp < nm;
    const int mw = active ? warp : 0;
    const float *wm = sw + (size_t)mw * nch * S * 8;
    const float *cm = scst + mw * S, *pm = slpi + mw * S;
    const float2 *am = sarc + (size_t)mw * S * S;
    const int32_t *stm = sstart + mw * (S + 1);
    float *dl = sdel + (size_t)mw * S * 32 + lane;     // delta[j] of this lane at dl[j * 32]
    const int slot = m0 + mw;
    const float NINF = -INFINITY;
    double base = 0.0, fsc = -INFINITY;
    int flast = 0;
    for (int t0 = 0; t0 < Tmax; t0 += DN_TF) {
        __syncthreads();                                   // the previous stage is consumed
        dn_stage(X, ldx, piv_g, s_off, s_T, t0, nch, L.xs4, sx, tid, nthr);
        __syncthreads();
        if (!active) continue;
        const int nf = min(DN_TF, Tmax - t0);
        for (int f = 0; f < nf; f++) {
            const int t = t0 + f;
            float acc[NMAX];
            dn_emit_tile<NMAX>(sx + (size_t)(f * 32 + lane) * L.xs4, wm, cm, S, nch, acc);
            uint32_t bits[BB::NW];
#pragma unroll
            for (int w = 0; w < BB::NW; w++) bits[w] = 0u;
            if (t == 0) {
#pragma unroll
                for (int j = 0; j < NMAX; j++) if (j < S) acc[j] += pm[j];
            } else {
#pragma unroll
                for (int j = 0; j < NMAX; j++) {
                    if (j < S) {
                        float best = NINF;
                        int arg = 0;
                        const int k1 = stm[j + 1];
                        for (int k = stm[j]; k < k1; k++) {     // first maximum over ascending sources (strict >)
                            const float2 a = am[k];
                            const int i = (int)a.y;
                            const float v = dl[i * 32] + a.x;
                            if (v > best) { best = v; arg = i; }
                        }
                        acc[j] += best;
                        bits[j / BB::PER] |= (uint32_t)arg << (BB::NB * (j % BB::PER));
                    }
                }
            }
            if (t < Te) {
                float mx = NINF;
                int am_ = 0;
#pragma unroll
                for (int j = 0; j < NMAX; j++) if (j < S && acc[j] > mx) { mx = acc[j]; am_ = j; }
                if (t == Te - 1) { fsc = (mx > NINF) ? base + (double)mx : (double)NINF; flast = am_; }
                if (mx > NINF && mx < INFINITY) {
#pragma unroll
                    for (int j = 0; j < NMAX; j++) if (j < S) acc[j] -= mx;
                    base += (double)mx;
                }
#pragma unroll
                for (int j = 0; j < NMAX; j++) if (j < S) dl[j * 32] = acc[j];
                if (bp && t > 0) {
#pragma unroll
                    for (int w = 0; w < BB::NW; w++)
                        if (w < nw) bp[(((size_t)slot * maxT + t) * nw + w) * Bpad + ul] = bits[w];
                }
            }
        }
    }
    if (active && ul < nu) {
        scores[(size_t)ul * M + slot] = fsc;
        last_state[(size_t)ul * M + slot] = (uint8_t)flast;
    }
}

// arg-max over the models (strict >, first best wins, decoder.py:42-47) + near-tie flag + the winner's back-trace
__global__ void k_dense_finish(const int64_t *__restrict__ offsets, int u0, int nu, int M, int nb, int nw,
                               const uint32_t *__restrict__ bp, int64_t Bpad, int maxT, const double *__restrict__ scores,
                               const uint8_t *__restrict__ last_state, int32_t *__restrict__ best_word,
                               double *__restrict__ best_score, double *__restrict__ scores_out, uint8_t *__restrict__ best_path,
                               SaprFlag flag) {
    const int ul = blockIdx.x * blockDim.x + threadIdx.x;
    if (ul >= nu) return;
    const int u = u0 + ul;
    double bs = -INFINITY, second = -INFINITY;
    int bslot = -1;
    for (int s = 0; s < M; s++) {
        const double sc = scores[(size_t)ul * M + s];
        if (scores_out) scores_out[(size_t)u * M + s] = sc;
        if (sc > bs) { second = bs; bs = sc; bslot = s; }
        else if (sc > second) second = sc;
    }
    if (best_word) best_word[u] = bslot;
    if (best_score) best_score[u] = bs;
    sapr_flag_word(flag, u, bs, second);
    if (!best_path) return;
    const int wslot = bslot < 0 ? 0 : bslot;       // no reachable model: model 0's path, as the verification mode gives
    const int64_t off = offsets[u];
    const int Te = min((int)(offsets[u + 1] - off), maxT);
    const int per = 32 / nb;
    const uint32_t mask = (1u << nb) - 1u;
    int cur = last_state[(size_t)ul * M + wslot];
    for (int t = Te - 1; t >= 0; t--) {
        best_path[off + t] = (uint8_t)cur;
        if (t == 0) break;
        const uint32_t word = bp[(((size_t)wslot * maxT + t) * nw + cur / per) * Bpad + ul];
        cur = (int)((word >> (nb * (cur % per))) & mask);
    }
}

// ------------------------------------------------------------------------------------------------
// float64 re-decoding of the flagged utterances: one 32-thread block per (list entry, model), lane j = state j.  The emission
// is k_emission_diag_mat's expression (compat.cu, called by sapr_emission_into), the recursion, the terminal arg-max and the
// back-trace are k_hl_viterbi's, so the entry's word, score, score row and path equal the verification mode's bit for bit.
// The block that completes an entry's last model (counter per entry, reset to zero by it) takes the arg-max and traces the
// winner from the delta scratch dl[entry][model][maxT][S].
__global__ void __launch_bounds__(32) k_dense_redo(const float *__restrict__ X, int ldx, const int64_t *__restrict__ offsets,
                                                   const int32_t *__restrict__ utt_list, const int32_t *__restrict__ utt_count, int cap,
                                                   int M, int S, int D, int maxT, const double *__restrict__ mean,
                                                   const double *__restrict__ var, const double *__restrict__ logpi,
                                                   const double *__restrict__ logA, double *dls, double *sc, int32_t *done,
                                                   int32_t *__restrict__ best_word, double *__restrict__ best_score,
                                                   double *__restrict__ scores_out, uint8_t *__restrict__ best_path) {
    const int j = threadIdx.x;
    const int n = min(*utt_count, cap);
    for (int w = blockIdx.x; w < n * M; w += gridDim.x) {
        const int pos = w / M, mi = w % M;
        const int u = utt_list[pos];
        const int64_t off = offsets[u];
        const int T = min((int)(offsets[u + 1] - off), maxT);
        double *dl = dls + ((size_t)pos * M + mi) * maxT * S;
        const double *lpi = logpi + (size_t)mi * S, *lA = logA + (size_t)mi * S * S;
        const double *mu = mean + ((size_t)mi * S + (j < S ? j : 0)) * D, *vr = var + ((size_t)mi * S + (j < S ? j : 0)) * D;
        double dv = -INFINITY;
        for (int t = 0; t < T; t++) {
            const double e = dn_emit64(X + (off + t) * ldx, mu, vr, D);
            if (t == 0) {
                dv = lpi[j < S ? j : 0] + e;
            } else {
                double mm = -INFINITY;
                for (int i = 0; i < S; i++) {
                    const double v = __shfl_sync(0xffffffffu, dv, i) + lA[i * S + (j < S ? j : 0)];
                    if (v > mm) mm = v;
                }
                dv = mm + e;
            }
            if (j < S) dl[(size_t)t * S + j] = dv;
        }
        double best = __shfl_sync(0xffffffffu, dv, 0);
        for (int i = 1; i < S; i++) {
            const double v = __shfl_sync(0xffffffffu, dv, i);
            if (v > best) best = v;
        }
        if (j == 0) sc[(size_t)pos * M + mi] = best;
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
        if (!best_path) continue;
        const int wslot = bslot < 0 ? 0 : bslot;
        const double *wd = dls + ((size_t)pos * M + wslot) * maxT * S;
        const double *wA = logA + (size_t)wslot * S * S;
        int cur = 0;
        double bv = __ldcg(wd + (size_t)(T - 1) * S);
        for (int i = 1; i < S; i++) {
            const double v = __ldcg(wd + (size_t)(T - 1) * S + i);
            if (v > bv) { bv = v; cur = i; }
        }
        best_path[off + T - 1] = (uint8_t)cur;
        for (int t = T - 2; t >= 0; t--) {
            int arg = 0;
            double mm = __ldcg(wd + (size_t)t * S) + wA[cur];
            for (int i = 1; i < S; i++) {
                const double v = __ldcg(wd + (size_t)t * S + i) + wA[i * S + cur];
                if (v > mm) { mm = v; arg = i; }
            }
            cur = arg;
            best_path[off + t] = (uint8_t)cur;
        }
    }
}

// verification mode: running arg-max over the models of sapr_hl_decode's per-model results (model 0's path is kept when no
// model scores, as the fp32 path does)
__global__ void k_dense_merge(const int64_t *__restrict__ offsets, int B, int mi, int M, const double *__restrict__ lp,
                              const int32_t *__restrict__ path, double *__restrict__ run_bs, int32_t *__restrict__ run_bw,
                              int32_t *__restrict__ best_word, double *__restrict__ best_score, double *__restrict__ scores_out,
                              uint8_t *__restrict__ best_path) {
    const int u = blockIdx.x * blockDim.x + threadIdx.x;
    if (u >= B) return;
    const double sc = lp[u];
    if (scores_out) scores_out[(size_t)u * M + mi] = sc;
    double bs = mi == 0 ? -INFINITY : run_bs[u];
    int bw = mi == 0 ? -1 : run_bw[u];
    const bool take = sc > bs;
    if (take) { bs = sc; bw = mi; }
    run_bs[u] = bs; run_bw[u] = bw;
    if (best_word) best_word[u] = bw;
    if (best_score) best_score[u] = bs;
    if (best_path && (take || mi == 0))
        for (int64_t f = offsets[u]; f < offsets[u + 1]; f++) best_path[f] = (uint8_t)path[f];
}

static int dense_fp64(sapr_ctx *ctx, sapr_models *m, const float *X, int ldx, const int64_t *offsets, int B, int64_t total_frames,
                      int32_t *best_word, double *best_score, double *scores, uint8_t *best_path) {
    const size_t a = ((size_t)B * sizeof(double) + 255) / 256 * 256, b = ((size_t)B * sizeof(int32_t) + 255) / 256 * 256;
    int rc = sapr_ws_reserve(ctx, 9, 2 * a + b + sizeof(int32_t) * (size_t)std::max<int64_t>(total_frames, 1));
    if (rc) return rc;
    double *lp = (double *)ctx->ws[9], *run_bs = (double *)((char *)ctx->ws[9] + a);
    int32_t *run_bw = (int32_t *)((char *)ctx->ws[9] + 2 * a), *path = (int32_t *)((char *)ctx->ws[9] + 2 * a + b);
    for (int mi = 0; mi < m->M; mi++) {
        if ((rc = sapr_hl_decode(ctx, m, mi, X, ldx, offsets, B, total_frames, lp, path))) return rc;
        k_dense_merge<<<(B + 127) / 128, 128, 0, ctx->stream>>>(offsets, B, mi, m->M, lp, path, run_bs, run_bw, best_word, best_score,
                                                                scores, best_path);
        SAPR_LAUNCH_CHECK(ctx);
    }
    return SAPR_OK;
}

template <int NMAX>
static int dense_fp32(sapr_ctx *ctx, sapr_models *m, const float *X, int ldx, const int64_t *offsets, int B, int max_T,
                      int32_t *best_word, double *best_score, double *scores, uint8_t *best_path) {
    const int M = m->M, S = m->S, nch = m->Dp / 4, nb = dn_nb(S), nw = (S + 32 / nb - 1) / (32 / nb);
    int mpc = std::min(M, 16);
    DnSmem L = dn_smem(mpc, S, nch);
    while (mpc > 1 && L.total > 200 * 1024) L = dn_smem(--mpc, S, nch);
    if (L.total > 200 * 1024) SAPR_FAIL(ctx, SAPR_E_RANGE, "viterbi (dense): model set does not fit in shared memory");
    auto kern = k_dense_viterbi<NMAX>;
    SAPR_CUDA(ctx, cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)L.total));
    // back-pointer scratch per chunk <= 1 GB (scores-only calls need none)
    const int64_t per_utt = (int64_t)M * max_T * nw * sizeof(uint32_t);
    int chunk = best_path ? (int)std::min<int64_t>(B, std::max<int64_t>(32, ((int64_t)1 << 30) / per_utt)) : B;
    chunk = (chunk + 31) / 32 * 32;
    const int64_t Bpad = chunk;
    int rc;
    if (best_path && (rc = sapr_ws_reserve(ctx, 0, (size_t)per_utt * Bpad))) return rc;
    const size_t scb = ((size_t)chunk * M * sizeof(double) + 255) / 256 * 256;
    if ((rc = sapr_ws_reserve(ctx, 1, scb + (size_t)chunk * M))) return rc;
    uint32_t *bp = best_path ? (uint32_t *)ctx->ws[0] : nullptr;
    double *sc_ws = (double *)ctx->ws[1];
    uint8_t *last = (uint8_t *)ctx->ws[1] + scb;
    const char *ex_env = getenv("SAPR_EXACT_WORDS");
    const bool exact = !ex_env || ex_env[0] != '0';
    SaprFlag flag;
    for (int u0 = 0; u0 < B; u0 += chunk) {
        const int nu = std::min(chunk, B - u0);
        if (exact) {
            if ((rc = sapr_flag_setup(ctx, &flag, u0 == 0))) return rc;
            // the re-decoding keeps every state's float64 delta of every model and frame: <= 256 MB of scratch
            const int64_t per = (int64_t)M * max_T * S * (int64_t)sizeof(double);
            flag.cap = (int)std::max<int64_t>(32, std::min<int64_t>(flag.cap, ((int64_t)256 << 20) / per));
        }
        {
            ProfScope ps(ctx, 7);
            dim3 block(32, mpc), grid((nu + 31) / 32, (M + mpc - 1) / mpc);
            kern<<<grid, block, L.total, ctx->stream>>>(X, ldx, offsets, u0, nu, M, S, nch, m->dn_piv, m->dn_w, m->dn_cst, m->dn_lpi,
                                                        (const float2 *)m->dn_arc, m->dn_start, L, bp, Bpad, max_T, nw, sc_ws, last);
        }
        SAPR_LAUNCH_CHECK(ctx);
        {
            ProfScope ps(ctx, 1);
            k_dense_finish<<<(nu + 127) / 128, 128, 0, ctx->stream>>>(offsets, u0, nu, M, nb, nw, bp, Bpad, max_T, sc_ws, last, best_word,
                                                                      best_score, scores, best_path, exact ? flag : SaprFlag());
        }
        SAPR_LAUNCH_CHECK(ctx);
        if (exact) {
            const size_t dlb = ((size_t)flag.cap * M * max_T * S * sizeof(double) + 255) / 256 * 256;
            if ((rc = sapr_ws_reserve(ctx, 4, dlb + (size_t)flag.cap * M * sizeof(double)))) return rc;
            double *dls = (double *)ctx->ws[4], *rsc = (double *)((char *)ctx->ws[4] + dlb);
            ProfScope ps(ctx, 8);
            k_dense_redo<<<8 * ctx->sm_count, 32, 0, ctx->stream>>>(X, ldx, offsets, flag.list, flag.count, flag.cap, M, S, m->D, max_T,
                                                                    m->mean, m->cov, m->logpi, m->logA, dls, rsc, flag.done, best_word,
                                                                    best_score, scores, best_path);
            SAPR_LAUNCH_CHECK(ctx);
        }
    }
    return SAPR_OK;
}

// sapr_viterbi for DENSE model sets (dispatched on the topology before anything else)
int sapr_viterbi_dense(sapr_ctx *ctx, sapr_models *m, const float *X, int ldx, const int64_t *offsets, int B, int64_t total_frames,
                       int max_T, const int32_t *model_of_utt, int precision, int first_frames, int32_t *best_word, double *best_score,
                       double *scores, uint8_t *best_path, uint8_t *all_paths) {
    if (m->emission != SAPR_EMIT_DIAG) SAPR_FAIL(ctx, SAPR_E_INVALID, "viterbi (dense): needs DIAG emission");
    if (first_frames > 0) SAPR_FAIL(ctx, SAPR_E_INVALID, "viterbi (dense): first_frames > 0 is the custom models' as-written mode");
    if (all_paths) SAPR_FAIL(ctx, SAPR_E_INVALID, "viterbi (dense): all_paths is not supported");
    if (model_of_utt) SAPR_FAIL(ctx, SAPR_E_INVALID, "viterbi (dense): model_of_utt is not supported");
    if (m->S > 32 || !m->dn_w) SAPR_FAIL(ctx, SAPR_E_RANGE, "viterbi (dense): S > 32 states (use sapr_hl_decode per model)");
    if (ldx % 4 || ldx < m->Dp) SAPR_FAIL(ctx, SAPR_E_INVALID, "viterbi: ldx must be a multiple of 4 and >= D padded");
    if (B <= 0) return SAPR_OK;
    if (max_T <= 0) SAPR_FAIL(ctx, SAPR_E_INVALID, "viterbi: max_T must be positive");
    ctx->flag_valid = false;
    if (precision == SAPR_FP64) return dense_fp64(ctx, m, X, ldx, offsets, B, total_frames, best_word, best_score, scores, best_path);
    if (precision != SAPR_FP32 && precision != SAPR_FP32_SIMT) SAPR_FAIL(ctx, SAPR_E_INVALID, "viterbi: bad precision");
    if (m->S <= 8) return dense_fp32<8>(ctx, m, X, ldx, offsets, B, max_T, best_word, best_score, scores, best_path);
    if (m->S <= 16) return dense_fp32<16>(ctx, m, X, ldx, offsets, B, max_T, best_word, best_score, scores, best_path);
    return dense_fp32<32>(ctx, m, X, ldx, offsets, B, max_T, best_word, best_score, scores, best_path);
}
