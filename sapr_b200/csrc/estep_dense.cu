// estep_dense.cu -- Baum-Welch E-step for DENSE-topology word models (hmmlearn GaussianHMM, every state emits, S x S transmat +
// startprob), every utterance against model_of_utt[u]: the statistics GaussianHMM.fit's E-step accumulates for one word
// (hmmlearn_hmm.py:103 -> sapr_hl_estep), for all words of a vocabulary in one call.
//
// fp32 production path (S <= 32, buckets 8 / 16 / 32):
//   k_dense_fb<NMAX>: CTA = one warp = a tile of up to 32 utterances of ONE model (tiles padded per model), lane = utterance.
//     - emission per state c_j + sum_d (a_jd x'_d + b_jd x'_d^2) on the pivot-centred fp32 image of k_dense_prepare
//       (viterbi_dense.cu), in log2 units;
//     - forward: u_t(j) = log2 sum_i ahat_{t-1}(i) A_ij + e_t(j) over the finite arcs grouped by destination,
//       ahat_t(j) = 2^(u_t(j) - c_t) with c_t = max_j u_t(j) (the state of largest mass is always 1), sum_t c_t in float64.
//       log2 ahat_t is stored to a scratch [tile][frame][state][lane] (one coalesced line per warp store; no underflow);
//     - backward, from the emission of frame t+1 recomputed: w(j) = e_{t+1}(j) + log2 bhat_{t+1}(j),
//       q(j) = 2^(w(j) - max w), r(i) = sum_j A_ij q(j) over the arcs grouped by source, log2 bhat_t(i) = log2 r(i);
//       a linear sum below 2^-64 (a left-to-right chain cannot re-enter a state whose mass fell below the fp32 range) is
//       redone in the log domain for that state, with log2 A_ij from float64 (k_dense_prepare), so no reachable state is lost,
//       utterances far from the model stay finite and an arc below the fp32 range keeps its share of beta and xi;
//       gamma_t(i) ~ 2^(log2 ahat_t(i) + log2 bhat_t(i)), normalised per frame by its own sum, and
//       xi_t(i, j) = gamma_t(i) A_ij q(j) / r(i) (so sum_j xi_t(i, j) = gamma_t(i));
//     - start / trans / post accumulate in fp32 per lane (trans in shared memory, one column per lane), then in float64 per
//       tile (fixed lane order); gamma goes to [sum_T][S] fp32.
//   k_dense_obs: CTA = tile, thread = (state, dim): sum gamma (x - mu_j) and sum gamma (x - mu_j)^2 pivoted at the state's
//     current mean (fp32 per utterance, float64 across utterances), so the variance does not cancel away.
//   k_dense_stats_reduce: fixed-order float64 sum of the tile partials per model, and the conversion of the pivoted moments to
//     hmmlearn's raw sum gamma x and sum gamma x^2.  Two identical calls give bit-identical statistics.
//   An utterance the model cannot produce (every state unreachable at some frame) gets loglik -inf and contributes nothing.
//
// SAPR_FP64 (verification): sapr_hl_estep per model on the model's utterances as a contiguous sub-batch (batch order, offsets
// rebased to 0), so stats and loglik equal GaussianHMM.fit's E-step for that word bit for bit.
#include <vector>

#include "dense_common.cuh"

// estep.cu: grouping of utterances by model
__global__ void k_model_start(const int32_t *__restrict__ model_of_utt, const int32_t *__restrict__ order, int B, int M,
                              int32_t *__restrict__ model_start);
__global__ void k_group_by_model(const int32_t *__restrict__ model_of_utt, int B, int M, int32_t *__restrict__ order);

// tiles of up to 32 utterances of one model: tile_start[m] = sum over m' < m of ceil(n_m' / 32)
__global__ void k_dense_tiles(const int32_t *__restrict__ model_start, int M, int32_t *__restrict__ tile_start) {
    if (threadIdx.x || blockIdx.x) return;
    int n = 0;
    for (int m = 0; m < M; m++) {
        tile_start[m] = n;
        n += (model_start[m + 1] - model_start[m] + 31) / 32;
    }
    tile_start[M] = n;
}

__device__ __forceinline__ int de_tile_model(const int32_t *__restrict__ tile_start, int M, int tile) {
    int lo = 0, hi = M - 1;   // last m with tile_start[m] <= tile (empty models share their successor's start)
    while (lo < hi) {
        const int mid = (lo + hi + 1) >> 1;
        if (tile_start[mid] <= tile) lo = mid; else hi = mid - 1;
    }
    return lo;
}

struct DeSmem {   // byte offsets of the dynamic shared memory of k_dense_fb
    size_t w, cst, lpi, piv, A, arcd, startd, arcs, lg2s, starts, col, lcol, acc, total;
};
static DeSmem de_smem(int S, int nch) {
    DeSmem L;
    size_t o = 0;
    auto take = [&](size_t b) { const size_t r = o; o += (b + 15) / 16 * 16; return r; };
    L.w = take((size_t)nch * S * 8 * sizeof(float));
    L.cst = take((size_t)S * sizeof(float));
    L.lpi = take((size_t)S * sizeof(float));
    L.piv = take((size_t)nch * sizeof(float4));
    L.A = take((size_t)S * S * sizeof(float));
    L.arcd = take((size_t)S * S * sizeof(float2));
    L.startd = take((size_t)(S + 1) * sizeof(int32_t));
    L.arcs = take((size_t)S * S * sizeof(float2));
    L.lg2s = take((size_t)S * S * sizeof(float));
    L.starts = take((size_t)(S + 1) * sizeof(int32_t));
    L.col = take((size_t)S * 32 * sizeof(float));
    L.lcol = take((size_t)S * 32 * sizeof(float));
    L.acc = take((size_t)(2 * S + S * S) * 32 * sizeof(float));   // per lane: start [S] | post [S] | xi per source-ordered arc
    L.total = o;
    return L;
}

// one warp per CTA: tile k0 + blockIdx.x.  part[tile][plen] receives [start S | trans S*S | post S] (float64).
template <int NMAX>
__global__ void __launch_bounds__(32)
k_dense_fb(const float *__restrict__ X, int ldx, const int64_t *__restrict__ offsets, const int32_t *__restrict__ order,
           const int32_t *__restrict__ model_start, const int32_t *__restrict__ tile_start, int M, int S, int nch, int k0,
           const float *__restrict__ piv_g, const float *__restrict__ w_g, const float *__restrict__ cst_g,
           const float *__restrict__ lpi_g, const float2 *__restrict__ arcd_g, const int32_t *__restrict__ startd_g,
           const float2 *__restrict__ arcs_g, const float *__restrict__ lg2s_g, const int32_t *__restrict__ starts_g, DeSmem L,
           float *__restrict__ scr, int maxT, float *__restrict__ gamma, double *__restrict__ part, int64_t plen,
           double *__restrict__ loglik) {
    const int tile = k0 + blockIdx.x;
    if (tile >= tile_start[M]) return;
    const int m = de_tile_model(tile_start, M, tile), lane = threadIdx.x;
    extern __shared__ __align__(16) unsigned char s_de[];
    float *sw = reinterpret_cast<float *>(s_de + L.w);
    float *scst = reinterpret_cast<float *>(s_de + L.cst);
    float *slpi = reinterpret_cast<float *>(s_de + L.lpi);
    float4 *spiv = reinterpret_cast<float4 *>(s_de + L.piv);
    float *sA = reinterpret_cast<float *>(s_de + L.A);
    float2 *sarcd = reinterpret_cast<float2 *>(s_de + L.arcd);
    int32_t *sstartd = reinterpret_cast<int32_t *>(s_de + L.startd);
    float2 *sarcs = reinterpret_cast<float2 *>(s_de + L.arcs);
    float *slg2s = reinterpret_cast<float *>(s_de + L.lg2s);                      // log2 A of sarcs[k], from float64
    int32_t *sstarts = reinterpret_cast<int32_t *>(s_de + L.starts);
    float *col = reinterpret_cast<float *>(s_de + L.col) + lane;                 // col[j * 32]: this lane's state vector
    float *lcol = reinterpret_cast<float *>(s_de + L.lcol) + lane;               // the same in log2 units
    float *acc = reinterpret_cast<float *>(s_de + L.acc);
    const int nacc = 2 * S + S * S;
    for (int i = lane; i < nch * S * 8; i += 32) sw[i] = w_g[(size_t)m * nch * S * 8 + i];
    for (int i = lane; i < S; i += 32) { scst[i] = cst_g[(size_t)m * S + i]; slpi[i] = lpi_g[(size_t)m * S + i] * DE_LOG2E; }
    for (int i = lane; i < nch; i += 32) spiv[i] = reinterpret_cast<const float4 *>(piv_g)[i];
    for (int i = lane; i < S * S; i += 32) {
        sA[i] = 0.f; sarcd[i] = arcd_g[(size_t)m * S * S + i]; sarcs[i] = arcs_g[(size_t)m * S * S + i];
        slg2s[i] = lg2s_g[(size_t)m * S * S + i];
    }
    for (int i = lane; i <= S; i += 32) { sstartd[i] = startd_g[(size_t)m * (S + 1) + i]; sstarts[i] = starts_g[(size_t)m * (S + 1) + i]; }
    for (int i = lane; i < nacc * 32; i += 32) acc[i] = 0.f;
    __syncwarp();
    for (int i = lane; i < S; i += 32)
        for (int k = sstarts[i]; k < sstarts[i + 1]; k++) sA[i * S + (int)sarcs[k].y] = sarcs[k].x;
    __syncwarp();

    const int p = model_start[m] + (tile - tile_start[m]) * 32 + lane;
    int T = 0, u = -1;
    int64_t off = 0;
    if (p < model_start[m + 1]) {
        u = order[p];
        off = offsets[u];
        T = (int)std::min<int64_t>(offsets[u + 1] - off, (int64_t)maxT);
    }
    const float *wm = sw, *cm = scst;
    float *sc = scr + (size_t)blockIdx.x * maxT * S * 32 + lane;                 // log2 ahat_t(j) at sc[(t * S + j) * 32]
    float *sacc = acc + lane;
    float *xi = sacc + 2 * S * 32;
    const float NINF = -INFINITY;

    // ---- forward ----
    double C = 0.0;
    bool alive = T > 0;
    for (int t = 0; t < T && alive; t++) {
        float e[NMAX];
        de_emit<NMAX>(X + (size_t)(off + t) * ldx, spiv, wm, cm, S, nch, e);
        if (t == 0) {
#pragma unroll
            for (int j = 0; j < NMAX; j++) if (j < S) e[j] += slpi[j];
        } else {
            de_fwd_step<NMAX>(col, lcol, sA, sarcd, sstartd, S, e);
        }
        float c = NINF;
#pragma unroll
        for (int j = 0; j < NMAX; j++) if (j < S) c = fmaxf(c, e[j]);
        if (!(c > NINF)) { alive = false; break; }
#pragma unroll
        for (int j = 0; j < NMAX; j++) {
            if (j < S) {
                const float la = e[j] - c;
                sc[((size_t)t * S + j) * 32] = la;
                lcol[j * 32] = la;
                col[j * 32] = de_ex2(la);
            }
        }
        C += (double)c;
    }
    if (u >= 0) {
        double ll = T > 0 ? -INFINITY : 0.0;            // an empty utterance scores 0, as k_hl_forward gives it
        if (alive) {
            float z = 0.f;
            for (int j = 0; j < S; j++) z += col[j * 32];
            ll = (C + log2((double)z)) * SAPR_LN2;
        }
        loglik[u] = ll;
    }

    // ---- backward + posteriors + statistics ----
    float lb[NMAX];
#pragma unroll
    for (int j = 0; j < NMAX; j++) lb[j] = 0.f;
    uint32_t redo = 0u;                                    // states i whose r(i) of this frame was taken in the log domain
    for (int t = T - 1; t >= 0; t--) {
        float *grow = gamma + (size_t)(off + t) * S;
        if (!alive) {                                      // the model cannot produce this utterance: no contribution
            for (int j = 0; j < S; j++) grow[j] = 0.f;
            continue;
        }
        float a[NMAX], e[NMAX];
#pragma unroll
        for (int j = 0; j < NMAX; j++) a[j] = (j < S) ? sc[((size_t)t * S + j) * 32] : NINF;
        const bool last = t == T - 1;
        if (!last) {
            de_emit<NMAX>(X + (size_t)(off + t + 1) * ldx, spiv, wm, cm, S, nch, e);
            float mq = NINF;
#pragma unroll
            for (int j = 0; j < NMAX; j++) if (j < S) { e[j] += lb[j]; mq = fmaxf(mq, e[j]); }
#pragma unroll
            for (int j = 0; j < NMAX; j++) if (j < S) { lcol[j * 32] = e[j] - mq; col[j * 32] = de_ex2(e[j] - mq); }   // q(j)
            redo = 0u;
#pragma unroll
            for (int i = 0; i < NMAX; i++) {
                if (i < S) {
                    float r = 0.f;
                    const int k0 = sstarts[i], k1 = sstarts[i + 1];
                    for (int k = k0; k < k1; k++) {
                        const float2 arc = sarcs[k];
                        r = fmaf(arc.x, col[(int)arc.y * 32], r);
                    }
                    if (r >= 0x1p-64f) {
                        lb[i] = de_lg2(r);                  // log2 bhat_t(i) = log2 r(i)
                    } else {                                // the successors' mass is (near) underflow: log domain
                        float mx = NINF;
                        for (int k = k0; k < k1; k++) mx = fmaxf(mx, slg2s[k] + lcol[(int)sarcs[k].y * 32]);
                        float s2 = 0.f;
                        if (mx > NINF)
                            for (int k = k0; k < k1; k++) s2 += de_ex2(slg2s[k] + lcol[(int)sarcs[k].y * 32] - mx);
                        lb[i] = (mx > NINF) ? mx + de_lg2(s2) : NINF;
                        redo |= 1u << i;
                    }
                    a[i] += lb[i];
                }
            }
        }
        float mg = NINF;
#pragma unroll
        for (int j = 0; j < NMAX; j++) if (j < S) mg = fmaxf(mg, a[j]);
        if (!(mg > NINF)) {                                 // forward and backward mass do not meet in fp32: frame skipped
            for (int j = 0; j < S; j++) grow[j] = 0.f;
            continue;
        }
        float z = 0.f;
#pragma unroll
        for (int j = 0; j < NMAX; j++) if (j < S) { a[j] = de_ex2(a[j] - mg); z += a[j]; }
        const float iz = 1.f / z;
#pragma unroll
        for (int i = 0; i < NMAX; i++) {
            if (i < S) {
                const float g = a[i] * iz;
                grow[i] = g;
                sacc[(S + i) * 32] += g;
                if (t == 0) sacc[i * 32] += g;
                if (!last && g > 0.f) {
                    const int k0 = sstarts[i], k1 = sstarts[i + 1];
                    if (!(redo >> i & 1u)) {
                        const float f = g * de_ex2(-lb[i]);    // gamma_t(i) / r(i)
                        for (int k = k0; k < k1; k++) {
                            const float2 arc = sarcs[k];
                            xi[k * 32] = fmaf(f * arc.x, col[(int)arc.y * 32], xi[k * 32]);
                        }
                    } else {                                   // A_ij q(j) / r(i) in the log domain
                        for (int k = k0; k < k1; k++)
                            xi[k * 32] += g * de_ex2(slg2s[k] + lcol[(int)sarcs[k].y * 32] - lb[i]);
                    }
                }
            }
        }
    }
    __syncwarp();
    // float64 tile sums over the lanes (fixed order)
    double *pt = part + (size_t)tile * plen;
    for (int k = lane; k < S; k += 32) {
        double s0 = 0.0, s1 = 0.0;
        for (int l = 0; l < 32; l++) { s0 += (double)acc[k * 32 + l]; s1 += (double)acc[(S + k) * 32 + l]; }
        pt[k] = s0;
        pt[S + S * S + k] = s1;
    }
    for (int k = lane; k < S * S; k += 32) pt[S + k] = 0.0;
    __syncwarp();
    for (int i = lane; i < S; i += 32)
        for (int k = sstarts[i]; k < sstarts[i + 1]; k++) {
            double s = 0.0;
            for (int l = 0; l < 32; l++) s += (double)acc[(2 * S + k) * 32 + l];
            pt[S + i * S + (int)sarcs[k].y] = s;
        }
}

// pivoted feature moments of a tile: thread = (state j, dim d), sum gamma (x - mu_j) and sum gamma (x - mu_j)^2 over the tile's
// frames (fp32 within an utterance, float64 across them); written to part[tile][S + S*S + S ...]
__global__ void k_dense_obs(const float *__restrict__ X, int ldx, const int64_t *__restrict__ offsets, const int32_t *__restrict__ order,
                            const int32_t *__restrict__ model_start, const int32_t *__restrict__ tile_start, int M, int S, int D,
                            int maxT, const double *__restrict__ mean, const float *__restrict__ gamma, double *__restrict__ part,
                            int64_t plen) {
    const int tile = blockIdx.x;
    if (tile >= tile_start[M]) return;
    const int m = de_tile_model(tile_start, M, tile);
    const int p0 = model_start[m] + (tile - tile_start[m]) * 32, n = min(32, model_start[m + 1] - p0);
    double *pt = part + (size_t)tile * plen + S + S * S + S;
    for (int o = threadIdx.x; o < S * D; o += blockDim.x) {
        const int j = o / D, d = o % D;
        const float mu = (float)mean[((size_t)m * S + j) * D + d];
        double s1 = 0.0, s2 = 0.0;
        for (int l = 0; l < n; l++) {
            const int u = order[p0 + l];
            const int64_t off = offsets[u];
            const int T = (int)std::min<int64_t>(offsets[u + 1] - off, (int64_t)maxT);
            float a = 0.f, b = 0.f;
            for (int t = 0; t < T; t++) {
                const float g = gamma[(size_t)(off + t) * S + j];
                const float x = X[(size_t)(off + t) * ldx + d] - mu;
                const float gx = g * x;
                a += gx;
                b = fmaf(gx, x, b);
            }
            s1 += (double)a; s2 += (double)b;
        }
        pt[o] = s1;
        pt[(size_t)S * D + o] = s2;
    }
}

// stats[m] = fixed-order sum of the model's tile partials; obs / obs2 converted from the pivoted moments:
// sum gamma x = P1 + p post, sum gamma x^2 = P2 + 2 p P1 + p^2 post (p = the fp32 pivot k_dense_obs used)
__global__ void k_dense_stats_reduce(const int32_t *__restrict__ tile_start, int S, int D, const double *__restrict__ mean,
                                     const double *__restrict__ part, int64_t plen, double *__restrict__ stats) {
    const int m = blockIdx.y, k = blockIdx.x * blockDim.x + threadIdx.x;
    if (k >= plen) return;
    const int t0 = tile_start[m], t1 = tile_start[m + 1];
    const int base = S + S * S + S;
    if (k < base) {
        double s = 0.0;
        for (int t = t0; t < t1; t++) s += part[(size_t)t * plen + k];
        stats[(size_t)m * plen + k] = s;
        return;
    }
    const int o = (k - base) % (S * D), j = o / D, d = o % D;
    double post = 0.0, p1 = 0.0, p2 = 0.0;
    for (int t = t0; t < t1; t++) {
        const double *pt = part + (size_t)t * plen;
        post += pt[S + S * S + j];
        p1 += pt[base + o];
        p2 += pt[base + (size_t)S * D + o];
    }
    const double p = (double)(float)mean[((size_t)m * S + j) * D + d];
    stats[(size_t)m * plen + k] = (k - base < S * D) ? p1 + p * post : p2 + 2.0 * p * p1 + p * p * post;
}

template <int NMAX>
static int dense_estep_fp32(sapr_ctx *ctx, sapr_models *m, const float *X, int ldx, const int64_t *offsets, int B,
                            int64_t total_frames, int max_T, const int32_t *order, const int32_t *model_start,
                            const int32_t *tile_start, double *stats, double *loglik, float *gamma) {
    const int M = m->M, S = m->S, D = m->D, nch = m->Dp / 4;
    const int64_t plen = sapr_hl_stats_len(S, D);
    const int ntile_max = (B + 31) / 32 + M;
    int rc;
    if (!gamma) {
        if ((rc = sapr_ws_reserve(ctx, 3, sizeof(float) * (size_t)total_frames * S))) return rc;
        gamma = (float *)ctx->ws[3];
    }
    if ((rc = sapr_ws_reserve(ctx, 1, sizeof(double) * (size_t)ntile_max * plen))) return rc;
    double *part = (double *)ctx->ws[1];
    // log2 ahat scratch, chunked over tiles so it stays <= ~1 GB
    const size_t per_tile = (size_t)max_T * S * 32 * sizeof(float);
    const int chunk = (int)std::max<int64_t>(1, std::min<int64_t>(ntile_max, ((int64_t)1 << 30) / (int64_t)per_tile));
    if ((rc = sapr_ws_reserve(ctx, 0, per_tile * chunk))) return rc;
    const DeSmem L = de_smem(S, nch);
    auto kern = k_dense_fb<NMAX>;
    SAPR_CUDA(ctx, cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)L.total));
    for (int k0 = 0; k0 < ntile_max; k0 += chunk) {
        const int nk = std::min(chunk, ntile_max - k0);
        ProfScope ps(ctx, 9);
        kern<<<nk, 32, L.total, ctx->stream>>>(X, ldx, offsets, order, model_start, tile_start, M, S, nch, k0, m->dn_piv, m->dn_w,
                                               m->dn_cst, m->dn_lpi, (const float2 *)m->dn_arc, m->dn_start,
                                               (const float2 *)m->dn_arcs, m->dn_lg2s, m->dn_starts, L, (float *)ctx->ws[0], max_T,
                                               gamma, part, plen, loglik);
        SAPR_LAUNCH_CHECK(ctx);
    }
    {
        ProfScope ps(ctx, 10);
        k_dense_obs<<<ntile_max, std::min(256, (S * D + 31) / 32 * 32), 0, ctx->stream>>>(X, ldx, offsets, order, model_start, tile_start,
                                                                                        M, S, D, max_T, m->mean, gamma, part, plen);
    }
    SAPR_LAUNCH_CHECK(ctx);
    k_dense_stats_reduce<<<dim3((unsigned)((plen + 127) / 128), M), 128, 0, ctx->stream>>>(tile_start, S, D, m->mean, part, plen, stats);
    SAPR_LAUNCH_CHECK(ctx);
    return SAPR_OK;
}

// ------------------------------------------------------------------------------------------------
// verification mode helpers: rows of a frame-major array gathered into / scattered from a contiguous sub-batch
__global__ void k_rows_gather(const float *__restrict__ src, int ld, const int64_t *__restrict__ rows, int64_t n, float *__restrict__ dst) {
    const int64_t r = blockIdx.x;
    if (r >= n) return;
    for (int c = threadIdx.x; c < ld; c += blockDim.x) dst[r * ld + c] = src[rows[r] * ld + c];
}
__global__ void k_rows_scatter(const double *__restrict__ src, int ld, const int64_t *__restrict__ rows, int64_t n, double *__restrict__ dst) {
    const int64_t r = blockIdx.x;
    if (r >= n) return;
    for (int c = threadIdx.x; c < ld; c += blockDim.x) dst[rows[r] * ld + c] = src[r * ld + c];
}

static int dense_estep_fp64(sapr_ctx *ctx, sapr_models *m, const float *X, int ldx, const int64_t *offsets, int B,
                            const int32_t *model_of_utt, double *stats, double *loglik, double *gamma) {
    const int M = m->M, S = m->S;
    const int64_t plen = sapr_hl_stats_len(S, m->D);
    std::vector<int32_t> mou(B);
    std::vector<int64_t> off(B + 1);
    SAPR_CUDA(ctx, cudaMemcpyAsync(mou.data(), model_of_utt, sizeof(int32_t) * B, cudaMemcpyDeviceToHost, ctx->stream));
    SAPR_CUDA(ctx, cudaMemcpyAsync(off.data(), offsets, sizeof(int64_t) * (B + 1), cudaMemcpyDeviceToHost, ctx->stream));
    SAPR_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
    std::vector<std::vector<int32_t>> utts(M);
    for (int u = 0; u < B; u++) {
        if (mou[u] < 0 || mou[u] >= M) SAPR_FAIL(ctx, SAPR_E_INVALID, "estep (dense): model_of_utt out of range");
        utts[mou[u]].push_back(u);
    }
    // per model: rebased offsets [n + 1] | utterance ids [n] | source frame rows [frames] (int64, one upload); a model whose
    // utterances are consecutive in the batch is read in place and needs no rows
    std::vector<int64_t> idx;
    std::vector<size_t> at(M);
    int64_t max_frames = 0;
    for (int mi = 0; mi < M; mi++) {
        at[mi] = idx.size();
        const size_t n = utts[mi].size();
        int64_t f = 0;
        idx.push_back(0);
        for (int u : utts[mi]) idx.push_back(f += off[u + 1] - off[u]);
        for (int u : utts[mi]) idx.push_back(u);
        if (n && (size_t)(utts[mi][n - 1] - utts[mi][0]) == n - 1) continue;
        for (int u : utts[mi])
            for (int64_t r = off[u]; r < off[u + 1]; r++) idx.push_back(r);
        max_frames = std::max(max_frames, f);
    }
    // slots 0-3: sapr_hl_estep and its callees reserve 4 and 5, the SAPR emission 7, the near-tie flags 8
    int rc;
    if ((rc = sapr_ws_reserve(ctx, 2, sizeof(int64_t) * idx.size()))) return rc;
    if ((rc = sapr_ws_reserve(ctx, 0, sizeof(float) * (size_t)std::max<int64_t>(max_frames, 1) * ldx))) return rc;
    if ((rc = sapr_ws_reserve(ctx, 1, sizeof(double) * (size_t)B))) return rc;
    int64_t *didx = (int64_t *)ctx->ws[2];
    SAPR_CUDA(ctx, cudaMemcpyAsync(didx, idx.data(), sizeof(int64_t) * idx.size(), cudaMemcpyHostToDevice, ctx->stream));
    SAPR_CUDA(ctx, cudaStreamSynchronize(ctx->stream));   // idx is pageable host memory
    for (int mi = 0; mi < M; mi++) {
        const int n = (int)utts[mi].size();
        if (n == 0) continue;
        const int u0 = utts[mi][0];
        const bool contiguous = utts[mi][n - 1] - u0 == n - 1;
        const int64_t *d_off = didx + at[mi], *d_ids = d_off + n + 1, *d_rows = d_ids + n;
        const int64_t frames = idx[at[mi] + n];
        const float *Xs = X + (size_t)off[u0] * ldx;
        double *ll = loglik + u0;
        if (!contiguous) {
            if (frames > 0) {
                k_rows_gather<<<(unsigned)frames, 128, 0, ctx->stream>>>(X, ldx, d_rows, frames, (float *)ctx->ws[0]);
                SAPR_LAUNCH_CHECK(ctx);
            }
            Xs = (const float *)ctx->ws[0];
            ll = (double *)ctx->ws[1];
        }
        if ((rc = sapr_hl_estep(ctx, m, mi, Xs, ldx, d_off, n, frames, stats + (size_t)mi * plen, ll))) return rc;
        if (!contiguous) {
            k_rows_scatter<<<n, 32, 0, ctx->stream>>>(ll, 1, d_ids, n, loglik);
            SAPR_LAUNCH_CHECK(ctx);
        }
        if (gamma && frames > 0) {
            // sapr_hl_estep leaves the posteriors in its workspace: ws[4] = [lf | fwd | bwd | post] x frames x S (hmmlearn.cu)
            const double *post = (const double *)ctx->ws[4] + 3 * (size_t)frames * S;
            if (contiguous)
                SAPR_CUDA(ctx, cudaMemcpyAsync(gamma + (size_t)off[u0] * S, post, sizeof(double) * frames * S, cudaMemcpyDeviceToDevice,
                                               ctx->stream));
            else {
                k_rows_scatter<<<(unsigned)frames, 32, 0, ctx->stream>>>(post, S, d_rows, frames, gamma);
                SAPR_LAUNCH_CHECK(ctx);
            }
        }
    }
    return SAPR_OK;
}

// sapr_estep for DENSE model sets (dispatched on the topology before anything else)
int sapr_estep_dense(sapr_ctx *ctx, sapr_models *m, const float *X, int ldx, const int64_t *offsets, int B, int64_t total_frames,
                     int max_T, const int32_t *model_of_utt, const int32_t *order_in, int precision, double *stats, double *loglik,
                     void *gamma_out) {
    if (m->emission != SAPR_EMIT_DIAG) SAPR_FAIL(ctx, SAPR_E_INVALID, "estep (dense): needs DIAG emission");
    if (ldx % 4 || ldx < m->Dp) SAPR_FAIL(ctx, SAPR_E_INVALID, "estep: ldx must be a multiple of 4 and >= D padded");
    if (precision != SAPR_FP64 && precision != SAPR_FP32) SAPR_FAIL(ctx, SAPR_E_INVALID, "estep (dense): bad precision");
    if (precision == SAPR_FP32 && (m->S > 32 || !m->dn_w))
        SAPR_FAIL(ctx, SAPR_E_RANGE, "estep (dense): S > 32 states in SAPR_FP32 (SAPR_FP64 runs sapr_hl_estep per model)");
    if (precision == SAPR_FP32) {   // one model's parameters, arc lists and per-lane accumulators in one CTA's shared memory
        int smem_max = 0;
        SAPR_CUDA(ctx, cudaDeviceGetAttribute(&smem_max, cudaDevAttrMaxSharedMemoryPerBlockOptin, ctx->device));
        if (de_smem(m->S, m->Dp / 4).total > (size_t)smem_max)
            SAPR_FAIL(ctx, SAPR_E_RANGE, "estep (dense): S and D too large for SAPR_FP32's shared memory (SAPR_FP64 runs "
                                         "sapr_hl_estep per model)");
    }
    if (precision == SAPR_FP64 && m->S > 1024) SAPR_FAIL(ctx, SAPR_E_RANGE, "estep (dense): more than 1024 states");
    const int M = m->M;
    SAPR_CUDA(ctx, cudaMemsetAsync(stats, 0, sizeof(double) * (size_t)M * sapr_hl_stats_len(m->S, m->D), ctx->stream));
    if (B <= 0) return SAPR_OK;
    if (precision == SAPR_FP64) return dense_estep_fp64(ctx, m, X, ldx, offsets, B, model_of_utt, stats, loglik, (double *)gamma_out);
    if (max_T <= 0) SAPR_FAIL(ctx, SAPR_E_INVALID, "estep: max_T must be positive");
    int rc;
    if ((rc = sapr_ws_reserve(ctx, 2, sizeof(int32_t) * ((size_t)B + 2 * M + 4)))) return rc;
    int32_t *order_ws = (int32_t *)ctx->ws[2], *model_start = order_ws + B, *tile_start = model_start + M + 1;
    const int32_t *order = order_in;
    if (!order) {
        k_group_by_model<<<1, 1024, 0, ctx->stream>>>(model_of_utt, B, M, order_ws);
        SAPR_LAUNCH_CHECK(ctx);
        order = order_ws;
    }
    k_model_start<<<(M + 1 + 63) / 64, 64, 0, ctx->stream>>>(model_of_utt, order, B, M, model_start);
    SAPR_LAUNCH_CHECK(ctx);
    k_dense_tiles<<<1, 32, 0, ctx->stream>>>(model_start, M, tile_start);
    SAPR_LAUNCH_CHECK(ctx);
#define GO(NM) \
    return dense_estep_fp32<NM>(ctx, m, X, ldx, offsets, B, total_frames, max_T, order, model_start, tile_start, stats, loglik, (float *)gamma_out)
    if (m->S <= 8) GO(8);
    if (m->S <= 16) GO(16);
    GO(32);
#undef GO
}
