// dense_common.cuh -- device code shared by the fp32 kernels of DENSE-topology word models (hmmlearn GaussianHMM, every state
// emits): the tile staging and emission of k_dense_viterbi (viterbi_dense.cu) and k_dense_forward (score_dense.cu), the
// per-utterance emission and the forward step of k_dense_fb (estep_dense.cu, also k_dense_forward's), and the float64 emission
// of the near-tie re-decoding / re-scoring kernels.  Everything is inlined into the kernels that include it.
#pragma once
#include "common.cuh"

#define DN_TF 16   // frames of the tile staged per round
#define DE_LOG2E 1.4426950408889634f

__device__ __forceinline__ float de_ex2(float x) {
    float r;
    asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(r) : "f"(x));
    return r;
}
__device__ __forceinline__ float de_lg2(float x) {
    float r;
    asm("lg2.approx.ftz.f32 %0, %1;" : "=f"(r) : "f"(x));
    return r;
}

// ---- tile kernels (CTA = 32 utterances, lane = utterance, warp = model) ----
// frames t0 .. t0 + DN_TF - 1 of the tile's utterances, pivot-centred (x' = x - p), into sx[(f * 32 + r) * xs4 + c]; rows past
// an utterance's end are left as they were
__device__ __forceinline__ void dn_stage(const float *__restrict__ X, int ldx, const float *__restrict__ piv_g,
                                         const int64_t *s_off, const int *s_T, int t0, int nch, int xs4, float4 *sx, int tid,
                                         int nthr) {
    for (int idx = tid; idx < DN_TF * 32 * nch; idx += nthr) {
        const int c = idx % nch, r = (idx / nch) & 31, f = idx / (32 * nch), t = t0 + f;
        if (t < s_T[r]) {
            float4 v = __ldg(reinterpret_cast<const float4 *>(X + (size_t)(s_off[r] + t) * ldx) + c);
            const float4 p = __ldg(reinterpret_cast<const float4 *>(piv_g) + c);
            v.x -= p.x; v.y -= p.y; v.z -= p.z; v.w -= p.w;
            sx[(f * 32 + r) * xs4 + c] = v;
        }
    }
}

// emission of one staged frame in natural-log units for the first S states: c_j + sum_d (a_jd x'_d + b_jd x'_d^2), the
// parameters warp-uniform shared-memory broadcasts ([chunk][state][8] = (a x4, b x4))
template <int NMAX>
__device__ __forceinline__ void dn_emit_tile(const float4 *xr, const float *wm, const float *cm, int S, int nch, float (&acc)[NMAX]) {
#pragma unroll
    for (int j = 0; j < NMAX; j++) acc[j] = (j < S) ? cm[j] : 0.f;
    for (int c = 0; c < nch; c++) {
        const float4 x = xr[c];
        const float4 x2 = make_float4(x.x * x.x, x.y * x.y, x.z * x.z, x.w * x.w);
        const float4 *wc = reinterpret_cast<const float4 *>(wm + (size_t)c * S * 8);
#pragma unroll
        for (int j = 0; j < NMAX; j++) {
            if (j < S) {
                const float4 a = wc[2 * j], b = wc[2 * j + 1];
                float e = acc[j];
                e = fmaf(a.x, x.x, e); e = fmaf(b.x, x2.x, e);
                e = fmaf(a.y, x.y, e); e = fmaf(b.y, x2.y, e);
                e = fmaf(a.z, x.z, e); e = fmaf(b.z, x2.z, e);
                e = fmaf(a.w, x.w, e); e = fmaf(b.w, x2.w, e);
                acc[j] = e;
            }
        }
    }
}

// ---- per-utterance form (k_dense_fb): the same emission read from HBM, in log2 units ----
template <int NMAX>
__device__ __forceinline__ void de_emit(const float *__restrict__ xrow, const float4 *__restrict__ piv, const float *__restrict__ w,
                                        const float *__restrict__ cst, int S, int nch, float (&e)[NMAX]) {
#pragma unroll
    for (int j = 0; j < NMAX; j++) e[j] = (j < S) ? cst[j] : 0.f;
    for (int c = 0; c < nch; c++) {
        float4 x = __ldg(reinterpret_cast<const float4 *>(xrow) + c);
        const float4 p = piv[c];
        x.x -= p.x; x.y -= p.y; x.z -= p.z; x.w -= p.w;
        const float4 x2 = make_float4(x.x * x.x, x.y * x.y, x.z * x.z, x.w * x.w);
        const float4 *wc = reinterpret_cast<const float4 *>(w + (size_t)c * S * 8);
#pragma unroll
        for (int j = 0; j < NMAX; j++) {
            if (j < S) {
                const float4 a = wc[2 * j], b = wc[2 * j + 1];
                float v = e[j];
                v = fmaf(a.x, x.x, v); v = fmaf(b.x, x2.x, v);
                v = fmaf(a.y, x.y, v); v = fmaf(b.y, x2.y, v);
                v = fmaf(a.z, x.z, v); v = fmaf(b.z, x2.z, v);
                v = fmaf(a.w, x.w, v); v = fmaf(b.w, x2.w, v);
                e[j] = v;
            }
        }
    }
#pragma unroll
    for (int j = 0; j < NMAX; j++) e[j] *= DE_LOG2E;
}

// forward step t >= 1 in log2 units: e(j) += log2 sum_i ahat_{t-1}(i) A_ij over the finite arcs grouped by destination
// (sources ascending).  col[i * 32] = ahat_{t-1}(i) of this lane, lcol[i * 32] its log2, sA[i * S + j] = A_ij, arcd = (ln A_ij,
// source i) with startd[S + 1].  A sum below 2^-64 (the predecessors' mass is near the fp32 underflow) is redone in the log
// domain, so a state reachable only through such mass, or through transitions below the fp32 range, stays finite; e(j) = -inf
// when no predecessor has mass.
template <int NMAX>
__device__ __forceinline__ void de_fwd_step(const float *col, const float *lcol, const float *sA, const float2 *arcd,
                                            const int32_t *startd, int S, float (&e)[NMAX]) {
    const float NINF = -INFINITY;
#pragma unroll
    for (int j = 0; j < NMAX; j++) {
        if (j < S) {
            float s = 0.f;
            const int k0 = startd[j], k1 = startd[j + 1];
            for (int k = k0; k < k1; k++) {
                const int i = (int)arcd[k].y;
                s = fmaf(col[i * 32], sA[i * S + j], s);
            }
            if (s >= 0x1p-64f) {
                e[j] += de_lg2(s);
            } else {                                // the predecessors' mass is (near) underflow: log domain
                float mx = NINF;
                for (int k = k0; k < k1; k++) mx = fmaxf(mx, lcol[(int)arcd[k].y * 32] + arcd[k].x * DE_LOG2E);
                float s2 = 0.f;
                if (mx > NINF)
                    for (int k = k0; k < k1; k++) s2 += de_ex2(lcol[(int)arcd[k].y * 32] + arcd[k].x * DE_LOG2E - mx);
                e[j] = (mx > NINF) ? e[j] + mx + de_lg2(s2) : NINF;
            }
        }
    }
}

// ---- float64 ----
// log N(x; mu, diag(var)) with k_emission_diag_mat's expression (compat.cu, called by sapr_emission_into), so the near-tie
// re-decoding and re-scoring kernels reproduce the verification mode's emission bit for bit
__device__ __forceinline__ double dn_emit64(const float *__restrict__ x, const double *__restrict__ mu, const double *__restrict__ vr, int D) {
    double ld = 0.0, q = 0.0;
    for (int d = 0; d < D; d++) {
        ld += log(vr[d]);
        const double df = (double)x[d] - mu[d];
        q += df * df / vr[d];
    }
    return -0.5 * (D * SAPR_LOG2PI + ld + q);
}

// viterbi_dense.cu: the scores-only arg-max / near-tie flag and the verification mode's running arg-max, shared with the scoring
__global__ void k_dense_finish(const int64_t *__restrict__ offsets, int u0, int nu, int M, int nb, int nw,
                               const uint32_t *__restrict__ bp, int64_t Bpad, int maxT, const double *__restrict__ scores,
                               const uint8_t *__restrict__ last_state, int32_t *__restrict__ best_word,
                               double *__restrict__ best_score, double *__restrict__ scores_out, uint8_t *__restrict__ best_path,
                               SaprFlag flag);
__global__ void k_dense_merge(const int64_t *__restrict__ offsets, int B, int mi, int M, const double *__restrict__ lp,
                              const int32_t *__restrict__ path, double *__restrict__ run_bs, int32_t *__restrict__ run_bw,
                              int32_t *__restrict__ best_word, double *__restrict__ best_score, double *__restrict__ scores_out,
                              uint8_t *__restrict__ best_path);
