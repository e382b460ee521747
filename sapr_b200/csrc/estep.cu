// estep.cu -- Baum-Welch E-step with fused diagonal-Gaussian emission, and the M-step.
//
// Replaces custom_hmm.py:417-439 (compute_emission_matrix, forward, backward, compute_gamma,
// compute_xi and the accumulators of baum_welch) plus the sums update_B consumes (:372-386), for
// every utterance against its own word model, and update_A / update_B (:351-400).
//
// k_estep_fused   one thread per utterance: log-space forward with a running max (alpha is kept
//                 relative to a per-frame offset accumulated in float64, so fp32 never sees the
//                 -1e4 magnitudes of a 200-frame likelihood), then the backward sweep producing
//                 gamma_t(j) and xi_t(j,j) on the fly.  Only sum_t xi_t(j,j) and sum_t gamma_t(j)
//                 are ever consumed (custom_hmm.py:359-361), so no S x S tensor exists.
// k_stats_diag    sum gamma (x - c) and sum gamma (x - c)^2 per (model, state, dim), pivot c = the
//                 model's current mean (every rank has it, so ONE all-reduce suffices); fp32 inside
//                 one utterance, float64 across utterances, fixed-order reduction across CTAs.
// k_stats_reduce  deterministic reduction of the per-tile partials into the packed stats block.
// k_mstep_diag    A_ii = Xi/G, means, variances with the reference's floor.
#include <stdlib.h>

#include "common.cuh"

template <typename R> struct alignas(16) Vec4e { R x, y, z, w; };

template <typename R> __host__ __device__ inline size_t model_stride(size_t per_model) {
    return per_model + 16 / sizeof(R);   // +16 B: models land in different banks when lanes differ
}

template <typename R, int NMAX>
__device__ __forceinline__ void emit_diag_e(const float *__restrict__ xrow, int nchunk, int N,
                                            const R *__restrict__ spk_model, const R *cst, R *e) {
    R acc[NMAX];
#pragma unroll
    for (int j = 0; j < NMAX; j++) acc[j] = R(0);
    const float4 *xr = reinterpret_cast<const float4 *>(xrow);
    for (int c = 0; c < nchunk; c++) {
        float4 xv = __ldg(xr + c);
        const R *p = spk_model + (size_t)c * N * 8;
#pragma unroll
        for (int j = 0; j < NMAX; j++) {
            if (j < N) {
                Vec4e<R> mu = *reinterpret_cast<const Vec4e<R> *>(p + j * 8);
                Vec4e<R> h = *reinterpret_cast<const Vec4e<R> *>(p + j * 8 + 4);
                R d0 = R(xv.x) - mu.x, d1 = R(xv.y) - mu.y, d2 = R(xv.z) - mu.z, d3 = R(xv.w) - mu.w;
                R a = acc[j];
                a = fma(d0 * d0, h.x, a);
                a = fma(d1 * d1, h.y, a);
                a = fma(d2 * d2, h.z, a);
                a = fma(d3 * d3, h.w, a);
                acc[j] = a;
            }
        }
    }
#pragma unroll
    for (int j = 0; j < NMAX; j++) e[j] = (j < N) ? cst[j] - acc[j] : R(0);
}

// scratch layout per block of 32 pairs: [t][j][lane] (coalesced), two planes: alpha-hat and e.
template <typename R, int NMAX, bool RENORM>
__global__ void __launch_bounds__(128)
k_estep_fused(const float *__restrict__ X, int ldx, const int64_t *__restrict__ offsets, int p0, int np, int M, int N,
              int nchunk, const R *__restrict__ pk, const R *__restrict__ cst_g, const R *__restrict__ la_g,
              const R *__restrict__ lb_g, const int32_t *__restrict__ model_of_utt, const int32_t *__restrict__ order,
              R *__restrict__ scr_alpha, R *__restrict__ scr_e, int maxT, R *__restrict__ gamma_out,
              R *__restrict__ ustats, double *__restrict__ loglik) {
    extern __shared__ __align__(16) unsigned char smem_raw[];
    R *spk = reinterpret_cast<R *>(smem_raw);
    const int S = N + 2;
    const size_t per_model = (size_t)nchunk * N * 8;
    const size_t mstride = model_stride<R>(per_model);
    for (int mm = 0; mm < M; mm++)
        for (size_t i = threadIdx.x; i < per_model; i += blockDim.x) spk[mm * mstride + i] = pk[mm * per_model + i];
    __syncthreads();
    const int pl = blockIdx.x * blockDim.x + threadIdx.x;   // pair index within the chunk
    if (pl >= np) return;
    const int p = p0 + pl;
    const int u = order ? order[p] : p;
    const int m = model_of_utt[u];
    const R *spk_model = spk + (size_t)m * mstride;
    R cst[NMAX], la[NMAX + 2], lb[NMAX + 2];
#pragma unroll
    for (int j = 0; j < NMAX; j++) cst[j] = (j < N) ? cst_g[(size_t)m * N + j] : R(0);
#pragma unroll
    for (int j = 0; j < NMAX + 2; j++) {
        la[j] = (j < S) ? la_g[(size_t)m * S + j] : R(0);
        lb[j] = (j < S) ? lb_g[(size_t)m * S + j] : R(0);
    }
    const R lbN = lb_g[(size_t)m * S + N];   // ln A[N, exit]
    const int64_t off = offsets[u];
    const int T = min((int)(offsets[u + 1] - off), maxT);      // the lattice scratch holds maxT frames per utterance
    const R NINF = Num<R>::ninf();
    const int lane = pl & 31;
    const size_t blk = (size_t)(pl >> 5) * maxT * N * 32;
    R *sa = scr_alpha + blk + lane;
    R *se = scr_e + blk + lane;

    // ---------------- forward (custom_hmm.py:176-211) ----------------
    R a[NMAX], e[NMAX];
    R ax = NINF;          // alpha[t, exit]
    double base = 0.0;    // alpha[t, j] = a[j] + base
    double amax = 0.0;    // running max of alpha over all cells; alpha[0,0] = 0 (:184)
    bool anan = false;
    if (T > 0) {
        emit_diag_e<R, NMAX>(X + (size_t)off * ldx, nchunk, N, spk_model, cst, e);
#pragma unroll
        for (int j = 0; j < NMAX; j++) a[j] = NINF;
        a[0] = lb[0] + e[0];
        if (a[0] != a[0]) anan = true; else amax = fmax(amax, (double)a[0]);
#pragma unroll
        for (int j = 0; j < NMAX; j++) if (j < N) { sa[(size_t)j * 32] = a[j]; se[(size_t)j * 32] = e[j]; }
    }
    for (int t = 1; t < T; t++) {
        emit_diag_e<R, NMAX>(X + (size_t)(off + t) * ldx, nchunk, N, spk_model, cst, e);
        R aN = NINF;                                   // alpha[t-1, N] without dynamic register indexing
#pragma unroll
        for (int j = 0; j < NMAX; j++) if (j == N - 1) aN = a[j];
        R nx = aN + lbN;                               // alpha[t, exit] = alpha[t-1, N] + ln A[N, exit]
#pragma unroll
        for (int j = NMAX - 1; j >= 1; j--)
            if (j < N) a[j] = lae(a[j - 1] + lb[j], a[j] + la[j + 1]) + e[j];
        {
            R ent = (t == 1) ? (R)(R(0) - (R)base) + lb[0] : NINF;   // alpha[t-1, 0] is 0 at t == 1 only
            a[0] = lae(ent, a[0] + la[1]) + e[0];
        }
        ax = nx;
        R mx = ax;
        bool nn = (ax != ax);
#pragma unroll
        for (int j = 0; j < NMAX; j++) if (j < N) { mx = fmax(mx, a[j]); nn = nn || (a[j] != a[j]); }
        if (nn) anan = true;
        if (mx > NINF) amax = fmax(amax, (double)mx + base);
        if (RENORM && mx > NINF && mx < R(INFINITY)) {
#pragma unroll
            for (int j = 0; j < NMAX; j++) if (j < N) a[j] -= mx;
            ax -= mx;
            base += (double)mx;
        }
        const size_t row = (size_t)t * N * 32;
#pragma unroll
        for (int j = 0; j < NMAX; j++) if (j < N) { sa[row + (size_t)j * 32] = a[j]; se[row + (size_t)j * 32] = e[j]; }
    }
    // reported log-likelihood (SURVEY D6): logaddexp.reduce(alpha[T-1, :]) - max(alpha)
    bool xi_live = true;
    double xi_lsum = 0.0;      // ln of the reference's per-frame sum of un-normalised xi, before the scale term (see below)
    if (T > 0) {
        R r = (T == 1) ? R(0) : NINF;                  // alpha[T-1, entry]
#pragma unroll
        for (int j = 0; j < NMAX; j++) if (j < N) r = lae(r, a[j]);
        r = lae(r, ax);
        double scale = anan ? (double)NAN : amax;
        loglik[u] = ((double)r + base) - scale;
        // SURVEY D10: the reference's un-normalised xi (custom_hmm.py:270-316) is exp(alpha + ln a + e + beta - logsumexp(alpha[T-1]));
        // summed over the arcs of a frame that is P(O, path ends in exit) / sum(alpha[T-1]) = exp(ax - r) for every frame, so when
        // ax - r < ln(2^-1075) every arc underflows to 0 in float64, the `if np.sum(xi[t]) > 0` guard (:319) skips the
        // normalisation and the utterance adds nothing to the transition statistics.
        xi_live = !((double)ax - (double)r < -745.13);
        xi_lsum = (double)ax - (double)r;
    }

    // ---------------- backward + gamma + xi (custom_hmm.py:213-322) ----------------
    R gG[NMAX], gO[NMAX], gX[NMAX];
#pragma unroll
    for (int j = 0; j < NMAX; j++) { gG[j] = R(0); gO[j] = R(0); gX[j] = R(0); }
    R b[NMAX];           // beta-hat[t+1, j]
#pragma unroll
    for (int j = 0; j < NMAX; j++) b[j] = NINF;
    R bx = R(0);         // beta[T-1, exit] = 0
    // t = T-1: gamma row is one-hot on the exit state (emitting gammas are exactly 0) unless alpha[T-1, exit]
    // is -inf, in which case the reference produces NaN for the whole row (:252-255).
    if (T > 0) {
        // T == 1 or alpha[T-1, exit] == -inf: every cell of the row is -inf -> NaN row
        const R g_last = (T > 1 && ax > NINF) ? R(0) : R(NAN);
        R *go = gamma_out ? gamma_out + (size_t)(off + T - 1) * N : nullptr;
#pragma unroll
        for (int j = 0; j < NMAX; j++) if (j < N) { if (go) go[j] = g_last; gO[j] += g_last; }
    }
    for (int t = T - 2; t >= 0; t--) {
        const size_t rown = (size_t)(t + 1) * N * 32, row = (size_t)t * N * 32;
        R w[NMAX + 1], at[NMAX];
#pragma unroll
        for (int j = 0; j < NMAX; j++) {
            if (j < N) { w[j] = se[rown + (size_t)j * 32] + b[j]; at[j] = sa[row + (size_t)j * 32]; }
            else { w[j] = NINF; at[j] = NINF; }
        }
        w[NMAX] = NINF;
        // beta[t, i] (:219-242); self[i] = ln A_ii + e_{t+1}(i) + beta_{t+1}(i)
        R self[NMAX], nb[NMAX];
#pragma unroll
        for (int j = 0; j < NMAX; j++) {
            if (j < N) {
                self[j] = la[j + 1] + w[j];
                R adv = (j < N - 1) ? lb[j + 1] + w[j + 1] : lbN + bx;
                nb[j] = lae(self[j], adv);
            } else { self[j] = NINF; nb[j] = NINF; }
        }
        R b0 = lb[0] + w[0];                          // beta[t, entry]
        // normaliser: logaddexp over all states of alpha+beta; entry contributes at t == 0 only,
        // exit never for t < T-1 (beta[t, exit] = -inf)
        R lg[NMAX];
        R nrm = (t == 0) ? (R)(R(0) + b0) : NINF;
#pragma unroll
        for (int j = 0; j < NMAX; j++) if (j < N) { lg[j] = at[j] + nb[j]; nrm = lae(nrm, lg[j]); }
        // xi normaliser (:319-320): sum over the arcs (0,1), (i,i), (i,i+1)_{i<N}; the (N,exit) arc is 0
        R xn = (t == 0) ? (R)(R(0) + b0) : NINF;
#pragma unroll
        for (int j = 0; j < NMAX; j++)
            if (j < N) xn = lae(xn, (j < N - 1) ? lg[j] : at[j] + self[j]);
        R *go = gamma_out ? gamma_out + (size_t)(off + t) * N : nullptr;
        // float64: the reference's un-normalised xi of an arc is its normalised value times exp(L), L = ax - r less the forward
        // scale max(alpha) on the frames whose beta it shifts (custom_hmm.py:241-246, :270-320).  For L below ~ -700 the arcs are
        // subnormal or flushed to 0 in its arithmetic and the per-frame normalisation divides those rounded values, so they are
        // formed the same way here; above, every arc is exact to 1e-16 and the log-domain ratio is used.
        const double L = xi_lsum - ((t + 1 < T - 1) ? amax : 0.0);
        const bool sub_xi = sizeof(R) == 8 && L < -700.0 && !anan && xn > NINF;
        double xsum = 0.0;
        if (sub_xi) {
            const double sh = L - (double)xn;
            if (t == 0) xsum += exp((double)b0 + sh);
#pragma unroll
            for (int j = 0; j < NMAX; j++)
                if (j < N) {
                    xsum += exp((double)(at[j] + self[j]) + sh);
                    if (j < N - 1) xsum += exp((double)(at[j] + lb[j + 1] + w[j + 1]) + sh);
                }
        }
#pragma unroll
        for (int j = 0; j < NMAX; j++) {
            if (j < N) {
                R g = fexp(lg[j] - nrm);               // all -inf row -> NaN like the reference
                gG[j] += g; gO[j] += g;
                if (go) go[j] = g;
                R xs = at[j] + self[j];
                if (sub_xi) {
                    if (xsum > 0.0) gX[j] += (R)(exp((double)xs + (L - (double)xn)) / xsum);     // the `sum > 0` guard (:319)
                } else if (xi_live && xn > NINF && xs > NINF) gX[j] += fexp(xs - xn);
            }
        }
        // next beta, renormalised (offsets cancel in gamma / xi, so they are not kept)
        R mx = NINF;
#pragma unroll
        for (int j = 0; j < NMAX; j++) if (j < N) { b[j] = nb[j]; mx = fmax(mx, nb[j]); }
        bx = NINF;
        if (RENORM && mx > NINF && mx < R(INFINITY)) {
#pragma unroll
            for (int j = 0; j < NMAX; j++) if (j < N) b[j] -= mx;
        }
    }
    R *us = ustats + (size_t)pl * 3 * N;
#pragma unroll
    for (int j = 0; j < NMAX; j++) if (j < N) { us[j] = gG[j]; us[N + j] = gX[j]; us[2 * N + j] = gO[j]; }
}

// ----------------------------------------------------------------------------------------------
// grouping of utterances by model: order[] (stable) and model_start[M+1]
__global__ void k_model_start(const int32_t *__restrict__ model_of_utt, const int32_t *__restrict__ order, int B, int M,
                              int32_t *__restrict__ model_start) {
    int m = blockIdx.x * blockDim.x + threadIdx.x;
    if (m > M) return;
    int lo = 0, hi = B;   // first p with model(order[p]) >= m
    while (lo < hi) {
        int mid = (lo + hi) >> 1;
        if (model_of_utt[order[mid]] >= m) hi = mid; else lo = mid + 1;
    }
    model_start[m] = lo;
}

// single-CTA stable counting sort (fallback when the caller gives no order[])
__global__ void k_group_by_model(const int32_t *__restrict__ model_of_utt, int B, int M, int32_t *__restrict__ order) {
    __shared__ int s_scan[1024];
    __shared__ int s_base;
    if (threadIdx.x == 0) s_base = 0;
    __syncthreads();
    for (int m = 0; m < M; m++) {
        for (int b0 = 0; b0 < B; b0 += blockDim.x) {
            int u = b0 + threadIdx.x;
            int f = (u < B && model_of_utt[u] == m) ? 1 : 0;
            s_scan[threadIdx.x] = f;
            __syncthreads();
            for (int d = 1; d < (int)blockDim.x; d <<= 1) {
                int v = (threadIdx.x >= (unsigned)d) ? s_scan[threadIdx.x - d] : 0;
                __syncthreads();
                s_scan[threadIdx.x] += v;
                __syncthreads();
            }
            if (f) order[s_base + s_scan[threadIdx.x] - 1] = u;
            __syncthreads();
            if (threadIdx.x == blockDim.x - 1) s_base += s_scan[threadIdx.x];
            __syncthreads();
        }
    }
}

// ----------------------------------------------------------------------------------------------
#define STATS_SLOTS 4  /* frame slots per feature dim */

__device__ __forceinline__ int find_tile(const int32_t *model_start, int M, int upc, int tile, int *tile_in_model) {
    int acc = 0;
    for (int m = 0; m < M; m++) {
        int cnt = model_start[m + 1] - model_start[m];
        int nt = (cnt + upc - 1) / upc;
        if (tile < acc + nt) { *tile_in_model = tile - acc; return m; }
        acc += nt;
    }
    return -1;
}

// blockDim = (Dp or fewer dims, STATS_SLOTS).  partial[tile][2][N][Dp] float64.
template <typename R, int NMAX>
__global__ void k_stats_diag(const float *__restrict__ X, int ldx, const int64_t *__restrict__ offsets,
                             const int32_t *__restrict__ order, const int32_t *__restrict__ model_start, int M, int N,
                             int D, int Dp, int S, int upc, const double *__restrict__ mean,
                             const R *__restrict__ gamma, double *__restrict__ partial) {
    __shared__ int s_m, s_tim;
    if (threadIdx.x == 0 && threadIdx.y == 0) s_m = find_tile(model_start, M, upc, blockIdx.x, &s_tim);
    __syncthreads();
    const int m = s_m;
    const int slot = threadIdx.y;
    double *out = partial + (size_t)blockIdx.x * 2 * N * Dp;
    extern __shared__ double s_red[];   // [STATS_SLOTS][2][N][Dp]
    // blockDim.x may be below Dp (the NMAX 16 / 31 instances use too many registers for Dp x STATS_SLOTS threads): dims in rounds
    for (int d0 = 0; d0 < Dp; d0 += blockDim.x) {
        const int d = d0 + threadIdx.x;
        const bool live = d < Dp;
        double a1[NMAX], a2[NMAX];
#pragma unroll
        for (int j = 0; j < NMAX; j++) { a1[j] = 0.0; a2[j] = 0.0; }
        if (m >= 0) {
            R c[NMAX];
#pragma unroll
            for (int j = 0; j < NMAX; j++) c[j] = (j < N && d < D) ? (R)mean[((size_t)m * S + j + 1) * D + d] : R(0);
            const int pbeg = model_start[m] + s_tim * upc;
            const int pend = min(pbeg + upc, model_start[m + 1]);
            for (int p = pbeg; p < pend; p++) {
                const int u = order[p];
                const int64_t off = offsets[u];
                const int T = (int)(offsets[u + 1] - off);
                R f1[NMAX], f2[NMAX];
#pragma unroll
                for (int j = 0; j < NMAX; j++) { f1[j] = R(0); f2[j] = R(0); }
                for (int t = slot; t < T; t += STATS_SLOTS) {
                    const R x = (d < D) ? (R)__ldg(X + (size_t)(off + t) * ldx + d) : R(0);
                    const R *g = gamma + (size_t)(off + t) * N;
#pragma unroll
                    for (int j = 0; j < NMAX; j++) {
                        if (j < N) {
                            R gj = __ldg(g + j);
                            R xc = x - c[j];
                            R gx = gj * xc;
                            f1[j] += gx;
                            f2[j] = fma(gx, xc, f2[j]);
                        }
                    }
                }
#pragma unroll
                for (int j = 0; j < NMAX; j++) { a1[j] += (double)f1[j]; a2[j] += (double)f2[j]; }
            }
        }
        // fixed-order reduction over the frame slots
#pragma unroll
        for (int j = 0; j < NMAX; j++)
            if (j < N && live) {
                s_red[((size_t)(slot * 2 + 0) * N + j) * Dp + d] = a1[j];
                s_red[((size_t)(slot * 2 + 1) * N + j) * Dp + d] = a2[j];
            }
        __syncthreads();
        if (slot == 0 && live) {
            for (int k = 0; k < 2; k++)
                for (int j = 0; j < N; j++) {
                    double s = 0.0;
                    for (int sl = 0; sl < STATS_SLOTS; sl++) s += s_red[((size_t)(sl * 2 + k) * N + j) * Dp + d];
                    out[((size_t)k * N + j) * Dp + d] = s;
                }
        }
        __syncthreads();
    }
}

// Production form of k_stats_diag for N == 8, fp32 gamma: blockDim = (Dp/2 dim pairs, 16 frame slots).
// A thread owns two feature dims and every 16th frame of the tile's utterances: per frame one 8-byte feature load
// (a warp reads whole 160-byte rows), gamma_t broadcast from two 16-byte loads, then per state
//   S1_j += gamma_j x';  S2_j += gamma_j x'^2;  G_j += gamma_j     (x' = x - g, g = mean of the model's state means;
//                                                                    two FFMA2 per state, packed over the two dims)
// fp32 inside a tile (a thread sees at most a few thousand frames; the raw moments are centred on g, so the relative
// error of the variance stays below 1e-4 even for states 8 sigma away from g), float64 across tiles; at the end of
// the tile the raw moments are re-pivoted in float64 to the model's current state means c_j (what the packed
// statistics block holds):
//   sum gamma (x-c) = S1 - (c-g) G,   sum gamma (x-c)^2 = S2 - 2 (c-g) S1 + (c-g)^2 G
// and reduced over the frame slots in a fixed order.
#define STATS2_SLOTS 32
#define STATS2_MAXUPC 256
__device__ __forceinline__ float2 st_fma2(float2 a, float2 b, float2 c) {
    unsigned long long d;
    asm("fma.rn.f32x2 %0, %1, %2, %3;" : "=l"(d) : "l"(*reinterpret_cast<unsigned long long *>(&a)),
        "l"(*reinterpret_cast<unsigned long long *>(&b)), "l"(*reinterpret_cast<unsigned long long *>(&c)));
    return *reinterpret_cast<float2 *>(&d);
}
__device__ __forceinline__ float2 st_mul2(float2 a, float2 b) {
    unsigned long long d;
    asm("mul.f32x2 %0, %1, %2;" : "=l"(d) : "l"(*reinterpret_cast<unsigned long long *>(&a)),
        "l"(*reinterpret_cast<unsigned long long *>(&b)));
    return *reinterpret_cast<float2 *>(&d);
}
__device__ __forceinline__ float2 st_sub2(float2 a, float2 b) {
    unsigned long long d;
    asm("sub.f32x2 %0, %1, %2;" : "=l"(d) : "l"(*reinterpret_cast<unsigned long long *>(&a)),
        "l"(*reinterpret_cast<unsigned long long *>(&b)));
    return *reinterpret_cast<float2 *>(&d);
}

// Shared-memory staged.  All utterances of a tile belong to one model, so the tile's frames are ONE stream: a
// dedicated producer warp bulk-copies it, STATS2_CF frames per stage (256: at 128 the per-stage hand-shakes cost 15 %) (a stage may span utterance boundaries: one copy
// of feature rows + one of gamma rows per piece; both are contiguous in HBM), into a STATS2_STAGES-deep ring.
// Consumer thread = (dim quad, state half, frame slot): 4 dims x 4 states x 2 moments = 32 packed accumulators, per
// frame one LDS.128 of features, one of gamma, and 20 FFMA2/FMUL2.  When D < Dp the first padding dim carries the
// constant 1, so its first-moment column is sum_t gamma (the occupancy the re-pivot needs) at no extra cost.
// blockDim.x = (Dp / 4) * 2 * STATS2_SLOTS consumers + 32 (producer warp).
#define STATS2_CF 256
#define STATS2_STAGES 4
__device__ __forceinline__ uint32_t st_smem(const void *p) { return (uint32_t)__cvta_generic_to_shared(p); }
__device__ __forceinline__ void st_wait(uint32_t bar, uint32_t parity) {
    asm volatile(
        "{\n\t.reg .pred p;\n\t.reg .u32 n;\n\tmov.u32 n, 0;\n\t"
        "LW:\n\tmbarrier.try_wait.parity.shared::cta.b64 p, [%0], %1, 2000;\n\t@p bra LD;\n\t"
        "add.u32 n, n, 1;\n\tsetp.gt.u32 p, n, 8000000;\n\t@p trap;\n\tbra LW;\n\tLD:\n\t}"
        ::"r"(bar), "r"(parity) : "memory");
}

__global__ void __launch_bounds__(672, 1)
k_stats_diag8(const float *__restrict__ X, int ldx, const int64_t *__restrict__ offsets, const int32_t *__restrict__ order,
              const int32_t *__restrict__ model_start, int M, int D, int Dp, int S, int upc, const double *__restrict__ mean,
              const float *__restrict__ gamma, double *__restrict__ partial) {
    constexpr int N = 8, NH = 4;
    __shared__ int s_m, s_tim, s_ftot;
    __shared__ int64_t s_off[STATS2_MAXUPC];
    __shared__ int s_T[STATS2_MAXUPC];
    __shared__ __align__(8) uint64_t s_bar[2 * STATS2_STAGES];
    const int ndq = Dp / 4, ncons = ndq * 2 * STATS2_SLOTS, tid = threadIdx.x;
    const bool consumer = tid < ncons;
    // a warp covers ~3 adjacent frame slots of ONE state half, so a half without posterior mass in those frames can be skipped as a warp
    const int dq = tid % ndq, slot = (tid / ndq) % STATS2_SLOTS, sh = tid / (ndq * STATS2_SLOTS), d0 = 4 * dq;
    const bool ones = Dp > D;                                    // dim D (padding) carries the constant 1
    extern __shared__ __align__(16) unsigned char s_dyn[];
    // the ring; at the end of the tile it is reused for the per-slot partials S1, S2 [STATS2_SLOTS][2][N][Dp], G [STATS2_SLOTS][N]
    float *s_acc = reinterpret_cast<float *>(s_dyn);
    float *s_g = s_acc + (size_t)STATS2_SLOTS * 2 * N * Dp;
    const uint32_t rowbytes = (uint32_t)ldx * 4u;
    const uint32_t stage_bytes = STATS2_CF * (rowbytes + 32u);
    unsigned char *s_stage = s_dyn;                                          // per stage: X rows, then gamma rows
    const uint32_t bar_full = st_smem(s_bar), bar_empty = bar_full + 8 * STATS2_STAGES;
    if (tid == 0) {
        s_m = find_tile(model_start, M, upc, blockIdx.x, &s_tim);
        for (int i = 0; i < STATS2_STAGES; i++) {
            asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(bar_full + 8 * i), "r"(1));
            asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(bar_empty + 8 * i), "r"(ncons / 32));
        }
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    __syncthreads();
    const int m = s_m;
    float2 s1[NH][2], s2[NH][2], gs[NH / 2];
#pragma unroll
    for (int j = 0; j < NH; j++)
#pragma unroll
        for (int h = 0; h < 2; h++) { s1[j][h] = make_float2(0.f, 0.f); s2[j][h] = make_float2(0.f, 0.f); }
#pragma unroll
    for (int j = 0; j < NH / 2; j++) gs[j] = make_float2(0.f, 0.f);
    int nutt = 0;
    if (m >= 0) {
        const int pbeg = model_start[m] + s_tim * upc;
        nutt = min(pbeg + upc, model_start[m + 1]) - pbeg;
        for (int i = tid; i < nutt; i += blockDim.x) {      // the tile's utterance table: frame offset and length
            const int u = order[pbeg + i];
            const int64_t o = offsets[u];
            s_off[i] = o; s_T[i] = max((int)(offsets[u + 1] - o), 0);
        }
    }
    __syncthreads();
    if (tid == 0) {
        int ft = 0;
        for (int i = 0; i < nutt; i++) ft += s_T[i];
        s_ftot = ft;
    }
    __syncthreads();
    const int ftot = s_ftot;
    const int nstage = (ftot + STATS2_CF - 1) / STATS2_CF;
    if (m >= 0 && nstage > 0) {
        if (!consumer) {
            // ---------------- producer warp: lane 0 walks the tile's frame stream ----------------
            if ((tid & 31) == 0) {
                int ppi = 0, pc0 = 0;
                while (ppi < nutt && s_T[ppi] <= 0) ppi++;
                for (int k = 0; k < nstage; k++) {
                    const uint32_t st = (uint32_t)k % STATS2_STAGES, ph = ((uint32_t)k / STATS2_STAGES) & 1u;
                    const int n = min(STATS2_CF, ftot - k * STATS2_CF);
                    st_wait(bar_empty + 8 * st, ph ^ 1u);
                    const uint32_t dst = st_smem(s_stage) + st * stage_bytes;
                    asm volatile("{\n\t.reg .b64 t;\n\tmbarrier.arrive.expect_tx.shared::cta.b64 t, [%0], %1;\n\t}"
                                 ::"r"(bar_full + 8 * st), "r"((uint32_t)n * (rowbytes + 32u)) : "memory");
                    int filled = 0;
                    while (filled < n) {
                        const int piece = min(s_T[ppi] - pc0, n - filled);
                        const size_t row = (size_t)(s_off[ppi] + pc0);
                        asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];"
                                     ::"r"(dst + (uint32_t)filled * rowbytes), "l"(X + row * ldx), "r"((uint32_t)piece * rowbytes),
                                     "r"(bar_full + 8 * st) : "memory");
                        asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];"
                                     ::"r"(dst + STATS2_CF * rowbytes + (uint32_t)filled * 32u), "l"(gamma + row * N),
                                     "r"((uint32_t)piece * 32u), "r"(bar_full + 8 * st) : "memory");
                        filled += piece; pc0 += piece;
                        while (ppi < nutt && pc0 >= s_T[ppi]) { pc0 = 0; ppi++; }
                    }
                }
            }
        } else {
            // pivot g: mean of the model's state means, rounded to fp32 (the same value is used in the float64 re-pivot)
            float gp[4], kk[4];
#pragma unroll
            for (int q = 0; q < 4; q++) {
                double gx = 0.0;
                if (d0 + q < D)
                    for (int j = 0; j < N; j++) gx += mean[((size_t)m * S + j + 1) * D + d0 + q];
                kk[q] = (d0 + q < D) ? 1.f : 0.f;
                gp[q] = -(float)(gx / N) * kk[q];
                if (ones && d0 + q == D) gp[q] = 1.f;                        // x' = x * 0 + 1
            }
            const float2 kk01 = make_float2(kk[0], kk[1]), kk23 = make_float2(kk[2], kk[3]);
            const float2 ng01 = make_float2(gp[0], gp[1]), ng23 = make_float2(gp[2], gp[3]);
            int dense_left = 0;                     // stages this warp still runs without the sparsity test
            for (int k = 0; k < nstage; k++) {
                const uint32_t st = (uint32_t)k % STATS2_STAGES, ph = ((uint32_t)k / STATS2_STAGES) & 1u;
                const int n = min(STATS2_CF, ftot - k * STATS2_CF);
                st_wait(bar_full + 8 * st, ph);
                const unsigned char *sx = s_stage + st * stage_bytes + 16 * dq;
                const unsigned char *sg = s_stage + st * stage_bytes + STATS2_CF * rowbytes + 16 * sh;
                // Posteriors of a left-to-right model are sparse: most frames have exactly zero mass in one half of the states.
                // A zero gamma contributes exactly nothing, so when every lane of the warp sees an all-zero half the frame is
                // skipped (bit-identical sums).  The test costs 4 instructions; a warp that found nothing to skip in a stage
                // runs the next seven stages without the test (dense posteriors, e.g. right after a flat start).
                auto frame = [&](int fi, bool probe) -> bool {
                    const float4 g0 = *reinterpret_cast<const float4 *>(sg + fi * 32);
                    if (probe) {
                        const uint32_t any = (__float_as_uint(g0.x) | __float_as_uint(g0.y) | __float_as_uint(g0.z) | __float_as_uint(g0.w)) << 1;
                        if (__all_sync(0xffffffffu, any == 0u)) return true;
                    }
                    const float4 xr = *reinterpret_cast<const float4 *>(sx + (size_t)fi * rowbytes);
                    const float2 x01 = st_fma2(make_float2(xr.x, xr.y), kk01, ng01);      // x' = x - g (0 for padded dims)
                    const float2 x23 = st_fma2(make_float2(xr.z, xr.w), kk23, ng23);
                    const float2 q01 = st_mul2(x01, x01), q23 = st_mul2(x23, x23);
                    const float gj[NH] = {g0.x, g0.y, g0.z, g0.w};
#pragma unroll
                    for (int j = 0; j < NH; j++) {
                        const float2 gg = make_float2(gj[j], gj[j]);
                        s1[j][0] = st_fma2(gg, x01, s1[j][0]); s1[j][1] = st_fma2(gg, x23, s1[j][1]);
                        s2[j][0] = st_fma2(gg, q01, s2[j][0]); s2[j][1] = st_fma2(gg, q23, s2[j][1]);
                    }
                    if (!ones) { gs[0].x += g0.x; gs[0].y += g0.y; gs[1].x += g0.z; gs[1].y += g0.w; }
                    return false;
                };
                if (n == STATS2_CF) {
                    const bool probe = dense_left == 0;
                    bool skipped = false;
#pragma unroll
                    for (int i = 0; i < STATS2_CF / STATS2_SLOTS; i++) skipped |= frame(slot + i * STATS2_SLOTS, probe);
                    if (probe) { if (!skipped) dense_left = 7; } else dense_left--;
                } else {
                    for (int fi = slot; fi < n; fi += STATS2_SLOTS) frame(fi, false);
                }
                __syncwarp();
                if ((tid & 31) == 0)
                    asm volatile("{\n\t.reg .b64 t;\n\tmbarrier.arrive.shared::cta.b64 t, [%0];\n\t}" ::"r"(bar_empty + 8 * st) : "memory");
            }
        }
    }
    __syncthreads();            // every chunk consumed: the ring is free, reuse it for the per-slot partials
    if (consumer) {
        float *mine = s_acc + (size_t)slot * 2 * N * Dp + d0;       // element (k, j, q) at mine[(k * N + j) * Dp + q]
#pragma unroll
        for (int j = 0; j < NH; j++) {
            const int js = NH * sh + j;
            *reinterpret_cast<float4 *>(mine + (0 * N + js) * Dp) = make_float4(s1[j][0].x, s1[j][0].y, s1[j][1].x, s1[j][1].y);
            *reinterpret_cast<float4 *>(mine + (1 * N + js) * Dp) = make_float4(s2[j][0].x, s2[j][0].y, s2[j][1].x, s2[j][1].y);
            if (ones) {
                if (D >= d0 && D < d0 + 4) {
                    const int q = D - d0;
                    s_g[slot * N + js] = (q == 0) ? s1[j][0].x : (q == 1) ? s1[j][0].y : (q == 2) ? s1[j][1].x : s1[j][1].y;
                }
            } else if (dq == 0) {
                s_g[slot * N + js] = (j & 1) ? gs[j >> 1].y : gs[j >> 1].x;
            }
        }
    }
    __syncthreads();
    // fixed-order reduction over the frame slots and float64 re-pivot to the state means: one thread per output element
    double *out = partial + (size_t)blockIdx.x * 2 * N * Dp;
    const int nsd = N * Dp;
    for (int i = tid; i < nsd; i += blockDim.x) {
        const int j = i / Dp, d = i % Dp;
        double S1 = 0.0, S2 = 0.0, G = 0.0;
        for (int sl = 0; sl < STATS2_SLOTS; sl++) {
            const float *b = s_acc + (size_t)sl * 2 * nsd;
            S1 += (double)b[i]; S2 += (double)b[nsd + i]; G += (double)s_g[sl * N + j];
        }
        double r1 = 0.0, r2 = 0.0;
        if (m >= 0 && d < D) {
            double gm = 0.0;
            for (int jj = 0; jj < N; jj++) gm += mean[((size_t)m * S + jj + 1) * D + d];
            const double gd = (double)(float)(gm / N);
            const double dc = mean[((size_t)m * S + j + 1) * D + d] - gd;
            r1 = S1 - dc * G;
            r2 = S2 - 2.0 * dc * S1 + dc * dc * G;
        }
        out[i] = r1; out[nsd + i] = r2;
    }
}

// fixed-order sum of the tile partials: one thread per (model, k, state, dim)
__global__ void k_reduce_partials(const int32_t *__restrict__ model_start, int M, int N, int D, int Dp, int S, int upc,
                                  const double *__restrict__ partial, double *__restrict__ stats, int64_t stride) {
    const int idx = blockIdx.x * blockDim.x + threadIdx.x;
    const int per_model = 2 * N * D;
    if (idx >= M * per_model) return;
    const int m = idx / per_model, i = idx % per_model;
    const int k = i / (N * D), r = i % (N * D), j = r / D, d = r % D;
    int tile0 = 0;
    for (int q = 0; q < m; q++) tile0 += (model_start[q + 1] - model_start[q] + upc - 1) / upc;
    const int ntile = (model_start[m + 1] - model_start[m] + upc - 1) / upc;
    const double *src = partial + ((size_t)k * N + j) * Dp + d;
    const size_t tstride = (size_t)2 * N * Dp;
    double s0 = 0.0, s1 = 0.0, s2 = 0.0, s3 = 0.0;
    int t = 0;
    for (; t + 3 < ntile; t += 4) {
        s0 += src[(size_t)(tile0 + t) * tstride];
        s1 += src[(size_t)(tile0 + t + 1) * tstride];
        s2 += src[(size_t)(tile0 + t + 2) * tstride];
        s3 += src[(size_t)(tile0 + t + 3) * tstride];
    }
    for (; t < ntile; t++) s0 += src[(size_t)(tile0 + t) * tstride];
    stats[(size_t)m * stride + (size_t)3 * S + (size_t)k * S * D + (size_t)(j + 1) * D + d] = (s0 + s1) + (s2 + s3);
}

// per-utterance (G, Xi, occ) triples of one chunk of pairs, added into stats in a fixed order:
// grid = (3N, M), 256 threads, tree reduction.
template <typename R>
__global__ void k_reduce_triples(const int32_t *__restrict__ model_start, int N, int S, const R *__restrict__ ustats,
                                 int p0, int np, double *__restrict__ stats, int64_t stride) {
    const int m = blockIdx.y, q = blockIdx.x;
    __shared__ double s_acc[256];
    const int pb = max(model_start[m], p0), pe = min(model_start[m + 1], p0 + np);
    double s = 0.0;
    for (int p = pb + threadIdx.x; p < pe; p += blockDim.x) s += (double)ustats[(size_t)(p - p0) * 3 * N + q];
    s_acc[threadIdx.x] = s;
    __syncthreads();
    for (int w = blockDim.x / 2; w > 0; w >>= 1) {
        if ((int)threadIdx.x < w) s_acc[threadIdx.x] += s_acc[threadIdx.x + w];
        __syncthreads();
    }
    if (threadIdx.x == 0) {
        const int k = q / N, j = q % N;
        stats[(size_t)m * stride + (size_t)k * S + j + 1] += s_acc[0];
    }
}

extern "C" int64_t sapr_stats_stride(int N, int D) {
    const int64_t S = N + 2;
    return 3 * S + 2 * S * D;
}

template <typename R, int NMAX>
static int launch_estep(sapr_ctx *ctx, sapr_models *m, const float *X, int ldx, const int64_t *offsets, int B,
                        int64_t total_frames, int max_T, const int32_t *model_of_utt, const int32_t *order_in,
                        double *stats, double *loglik, void *gamma_out) {
    const int N = m->N, M = m->M, D = m->D, Dp = m->Dp, S = m->S, nchunk = Dp / 4;
    const int64_t stride = sapr_stats_stride(N, D);
    int rc;
    // shapes whose shared memory does not fit are refused before the first launch
    const bool use_tc = std::is_same<R, float>::value && sapr_tc_usable(m);
    const size_t smem = (size_t)M * model_stride<R>((size_t)nchunk * N * 8) * sizeof(R);
    if (!use_tc && smem > 227 * 1024)
        SAPR_FAIL(ctx, SAPR_E_RANGE, "estep: the model set does not fit in shared memory (the E-step stages every model)");
    const int upc = std::max(8, std::min(256, B / (4 * ctx->sm_count)));
    const int ncons = (Dp / 4) * 2 * STATS2_SLOTS;
    const size_t ssm2 = std::max(sizeof(float) * STATS2_SLOTS * (2 * N * Dp + N), (size_t)STATS2_STAGES * STATS2_CF * (ldx * 4 + 32));
    const bool use_stats8 = std::is_same<R, float>::value && N == 8 && ssm2 <= 227 * 1024 && ncons <= 640 && ncons % 32 == 0 &&
                            upc <= STATS2_MAXUPC;
    const size_t ssm = sizeof(double) * STATS_SLOTS * 2 * N * Dp;
    if (!use_stats8 && ssm > 227 * 1024)
        SAPR_FAIL(ctx, SAPR_E_RANGE, "estep: the feature statistics of N states x D dims do not fit in shared memory");
    // grouping
    if ((rc = sapr_ws_reserve(ctx, 2, sizeof(int32_t) * ((size_t)B + M + 2)))) return rc;
    int32_t *order_ws = (int32_t *)ctx->ws[2];
    int32_t *model_start = order_ws + B;
    const int32_t *order = order_in;
    if (!order) {
        k_group_by_model<<<1, 1024, 0, ctx->stream>>>(model_of_utt, B, M, order_ws);
        SAPR_LAUNCH_CHECK(ctx);
        order = order_ws;
    }
    k_model_start<<<(M + 1 + 63) / 64, 64, 0, ctx->stream>>>(model_of_utt, order, B, M, model_start);
    SAPR_LAUNCH_CHECK(ctx);
    // gamma workspace (or the caller's debug buffer)
    R *gamma = (R *)gamma_out;
    if (!gamma) {
        if ((rc = sapr_ws_reserve(ctx, 3, sizeof(R) * (size_t)total_frames * N))) return rc;
        gamma = (R *)ctx->ws[3];
    }
    const int ntile_max = (B + upc - 1) / upc + M;
    if ((rc = sapr_ws_reserve(ctx, 4, sizeof(double) * (size_t)ntile_max * 2 * N * Dp))) return rc;
    double *partial = (double *)ctx->ws[4];
    if (use_tc) {
        // production fp32 path: emission on the tensor cores, forward and backward sweep of a tile in one persistent CTA
        if ((rc = sapr_ws_reserve(ctx, 1, sizeof(float) * (size_t)B * 3 * N))) return rc;
        if ((rc = sapr_estep_tc_launch(ctx, m, X, ldx, offsets, B, max_T, order, model_start, (float *)gamma,
                                       (float *)ctx->ws[1], loglik)))
            return rc;
        k_reduce_triples<float><<<dim3(3 * N, M), 256, 0, ctx->stream>>>(model_start, N, S, (const float *)ctx->ws[1], 0, B,
                                                                         stats, stride);
        SAPR_LAUNCH_CHECK(ctx);
    } else {
    // forward/backward lattice scratch, chunked over pairs so it stays bounded (<= ~1 GB)
    const size_t per_pair = (size_t)max_T * N * sizeof(R) * 2;
    int chunk = (int)std::min<int64_t>(B, std::max<int64_t>(128, ((int64_t)1 << 30) / (int64_t)per_pair));
    chunk = (chunk + 127) / 128 * 128;
    if ((rc = sapr_ws_reserve(ctx, 0, per_pair * chunk))) return rc;
    if ((rc = sapr_ws_reserve(ctx, 1, sizeof(R) * (size_t)chunk * 3 * N))) return rc;
    R *scr_alpha = (R *)ctx->ws[0];
    R *scr_e = scr_alpha + (size_t)chunk * max_T * N;
    R *ustats = (R *)ctx->ws[1];

    const R *pk = std::is_same<R, float>::value ? (const R *)m->pk32 : (const R *)m->pk64;
    const R *cst = std::is_same<R, float>::value ? (const R *)m->cst32 : (const R *)m->cst64;
    const R *la = std::is_same<R, float>::value ? (const R *)m->la32 : (const R *)m->la64;
    const R *lb = std::is_same<R, float>::value ? (const R *)m->lb32 : (const R *)m->lb64;
    auto kern = k_estep_fused<R, NMAX, std::is_same<R, float>::value>;
    SAPR_CUDA(ctx, cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    for (int p0 = 0; p0 < B; p0 += chunk) {
        const int np = std::min(chunk, B - p0);
        {
            ProfScope ps(ctx, 2);
            kern<<<(np + 127) / 128, 128, smem, ctx->stream>>>(X, ldx, offsets, p0, np, M, N, nchunk, pk, cst, la, lb,
                                                               model_of_utt, order, scr_alpha, scr_e, max_T, gamma,
                                                               ustats, loglik);
        }
        SAPR_LAUNCH_CHECK(ctx);
        // the small per-utterance triples are folded into stats chunk by chunk (fixed order)
        k_reduce_triples<R><<<dim3(3 * N, M), 256, 0, ctx->stream>>>(model_start, N, S, ustats, p0, np, stats, stride);
        SAPR_LAUNCH_CHECK(ctx);
    }
    }
    // feature statistics over the whole batch
    const int ntiles = ntile_max;
    if (use_stats8) {
        dim3 sb2(ncons + 32);                          // + the producer warp
        SAPR_CUDA(ctx, cudaFuncSetAttribute(k_stats_diag8, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)ssm2));
        {
            ProfScope ps(ctx, 3);
            k_stats_diag8<<<ntiles, sb2, ssm2, ctx->stream>>>(X, ldx, offsets, order, model_start, M, D, Dp, S, upc, m->mean,
                                                              (const float *)gamma, partial);
        }
        SAPR_LAUNCH_CHECK(ctx);
        k_reduce_partials<<<(M * 2 * N * D + 127) / 128, 128, 0, ctx->stream>>>(model_start, M, N, D, Dp, S, upc, partial,
                                                                                stats, stride);
        SAPR_LAUNCH_CHECK(ctx);
        return SAPR_OK;
    }
    auto skern = k_stats_diag<R, NMAX>;
    cudaFuncAttributes fa;
    SAPR_CUDA(ctx, cudaFuncGetAttributes(&fa, skern));
    const int bx = Dp * STATS_SLOTS <= fa.maxThreadsPerBlock ? Dp : fa.maxThreadsPerBlock / STATS_SLOTS / 32 * 32;
    dim3 sb(bx, STATS_SLOTS);
    SAPR_CUDA(ctx, cudaFuncSetAttribute(skern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)ssm));
    {
        ProfScope ps(ctx, 3);
        skern<<<ntiles, sb, ssm, ctx->stream>>>(X, ldx, offsets, order, model_start, M, N, D, Dp, S, upc, m->mean, gamma,
                                                partial);
    }
    SAPR_LAUNCH_CHECK(ctx);
    k_reduce_partials<<<(M * 2 * N * D + 127) / 128, 128, 0, ctx->stream>>>(model_start, M, N, D, Dp, S, upc, partial,
                                                                            stats, stride);
    SAPR_LAUNCH_CHECK(ctx);
    return SAPR_OK;
}

extern "C" int sapr_estep(sapr_ctx *ctx, sapr_models *m, const float *X, int ldx, const int64_t *offsets, int B,
                          int64_t total_frames, int max_T, const int32_t *model_of_utt, const int32_t *order,
                          int precision, double *stats, double *loglik, void *gamma_out) {
    if (!ctx || !m || !X || !offsets || !model_of_utt || !stats || !loglik) return SAPR_E_INVALID;
    if (!m->valid) SAPR_FAIL(ctx, SAPR_E_INVALID, "estep: model parameters not set");
    if (m->topology == SAPR_TOPO_DENSE)
        return sapr_estep_dense(ctx, m, X, ldx, offsets, B, total_frames, max_T, model_of_utt, order, precision, stats, loglik, gamma_out);
    if (m->emission != SAPR_EMIT_DIAG || m->topology != SAPR_TOPO_ENTRY_EXIT)
        SAPR_FAIL(ctx, SAPR_E_INVALID, "estep: fused kernel needs DIAG emission + ENTRY_EXIT topology");
    if (ldx % 4 || ldx < m->Dp) SAPR_FAIL(ctx, SAPR_E_INVALID, "estep: ldx must be a multiple of 4 and >= D padded");
    if (m->Dp * STATS_SLOTS > 1024) SAPR_FAIL(ctx, SAPR_E_RANGE, "estep: D > 256 not supported");
    SAPR_CUDA(ctx, cudaMemsetAsync(stats, 0, sizeof(double) * (size_t)m->M * sapr_stats_stride(m->N, m->D), ctx->stream));
    if (B <= 0) return SAPR_OK;
#define GO(R, NM) \
    return launch_estep<R, NM>(ctx, m, X, ldx, offsets, B, total_frames, max_T, model_of_utt, order, stats, loglik, gamma_out)
    if (precision == SAPR_FP32) {
        if (m->N <= 8) GO(float, 8);
        if (m->N <= 16) GO(float, 16);
        if (m->N <= 31) GO(float, 31);
    } else {
        if (m->N <= 8) GO(double, 8);
        if (m->N <= 16) GO(double, 16);
        if (m->N <= 31) GO(double, 31);
    }
#undef GO
    SAPR_FAIL(ctx, SAPR_E_RANGE, "estep: N > 31 emitting states not supported");
}

// ----------------------------------------------------------------------------------------------
// M-step (custom_hmm.py:351-400) on the packed statistics; one thread per (model, state, dim).
__global__ void k_mstep_diag(int M, int N, int D, int S, const double *__restrict__ stats, int64_t stride,
                             const double *__restrict__ floor_var, double *__restrict__ mean, double *__restrict__ var,
                             double *__restrict__ A) {
    const int idx = blockIdx.x * blockDim.x + threadIdx.x;
    const int total = M * S * D;
    if (idx < total) {
        const int d = idx % D, j = (idx / D) % S, m = idx / (D * S);
        const double *st = stats + (size_t)m * stride;
        double nm = 0.0, nv = 0.0;
        if (j >= 1 && j <= N) {
            const double occ = st[2 * S + j];
            if (occ > 0) {
                const double c = mean[idx];
                const double s1 = st[3 * S + (size_t)j * D + d], s2 = st[3 * S + (size_t)S * D + (size_t)j * D + d];
                const double dm = s1 / occ;
                nm = c + dm;
                double v = s2 / occ - dm * dm;          // = sum gamma (x - mu_new)^2 / occ
                const double fl = floor_var[m];
                nv = (v != v) ? v : (v > fl ? v : fl);   // np.maximum keeps NaN (:397)
            }
        }
        // defer the mean write until every thread of this (m, j) row has read its pivot: each thread only
        // touches its own element, so writing in place is safe.
        mean[idx] = nm;
        var[idx] = nv;
    }
    if (idx < M * S) {   // transitions (:351-364)
        const int j = idx % S, m = idx / S;
        const double *st = stats + (size_t)m * stride;
        double *Am = A + (size_t)m * S * S;
        if (j == 0) Am[0 * S + 1] = 1.0;
        else if (j == S - 1) Am[(size_t)j * S + j] = 1.0;
        else if (st[j] > 0) {
            const double aii = st[S + j] / st[j];
            Am[(size_t)j * S + j] = aii;
            Am[(size_t)j * S + j + 1] = 1.0 - aii;
        }
    }
}

extern "C" int sapr_mstep(sapr_ctx *ctx, sapr_models *m, const double *stats, const double *floor_var_host) {
    if (!ctx || !m || !stats || !floor_var_host) return SAPR_E_INVALID;
    if (m->emission != SAPR_EMIT_DIAG || m->topology != SAPR_TOPO_ENTRY_EXIT)
        SAPR_FAIL(ctx, SAPR_E_INVALID, "mstep: needs DIAG emission + ENTRY_EXIT topology");
    int rc = sapr_ws_reserve(ctx, 5, sizeof(double) * m->M);
    if (rc) return rc;
    SAPR_CUDA(ctx, cudaMemcpyAsync(ctx->ws[5], floor_var_host, sizeof(double) * m->M, cudaMemcpyHostToDevice, ctx->stream));
    SAPR_CUDA(ctx, cudaStreamSynchronize(ctx->stream));   // floor_var_host is pageable caller memory
    const int total = m->M * m->S * m->D;
    k_mstep_diag<<<(total + 255) / 256, 256, 0, ctx->stream>>>(m->M, m->N, m->D, m->S, stats, sapr_stats_stride(m->N, m->D),
                                                               (const double *)ctx->ws[5], m->mean, m->cov, m->A);
    SAPR_LAUNCH_CHECK(ctx);
    return sapr_models_prepare(m);
}
