// estep_tc.cu -- Baum-Welch E-step (forward, backward, gamma, xi sums) with the emission on the tensor cores.
//
// Replaces custom_hmm.py:417-439 (compute_emission_matrix, forward, backward, compute_gamma, compute_xi and the
// accumulators of baum_welch) for every utterance against its own word model, fp32 production mode.  Same machine
// mapping as viterbi_tc.cu: a tile is 128 utterances at the same frame index, the diagonal-Gaussian log-density of
// one frame is the contraction [x', x'^2, 1] . W on tcgen05 (A operand written into TMEM by the threads that own
// the rows, W in shared memory, fp32 accumulators in TMEM), raw features arrive through a cp.async.bulk ring.
//
// Differences from the Viterbi kernel:
//   * utterances are visited in model order (order[] grouped by word, every model's group padded to a multiple of
//     32 rows), so the 32 rows of a TMEM lane quadrant share ONE model and a tile spans one (rarely up to four)
//     adjacent models.  Per model of the tile the MMA is N = 16: accumulator columns 0-7 take the products with the
//     W_hi plane, columns 8-15 the products with the W_lo plane (the B descriptor's 8-row-group stride is the plane
//     distance), so two passes (A_lo, then A_hi) of nck/2 K-steps replace the three of the Viterbi kernel and the
//     large hi*hi sum sees only nck/2 truncating accumulations after the small lo*hi one;
//   * the tensor-core pipeline (bulk copies -> converters -> MMA) runs the FORWARD sweep only.  The recursion thread
//     of a row stores alpha-hat AND the emissions e'_t(j) = E[t,j] + ln A[j,j] of its frames to a per-(CTA, recursion
//     group) scratch ([frame][16][row], 8 KB per frame); the BACKWARD sweep (beta / gamma / xi) is a thread-private
//     loop over that scratch: no second feature read, no second conversion, no barriers.  Only sum_t gamma,
//     sum_t xi(j,j), gamma_t (for the feature statistics) and the log-likelihood leave the CTA;
//   * two recursion warpgroups alternate tiles: while group A sweeps tile k backward, the pipeline and group B are
//     already in the forward sweep of tile k+1, so the converters / MMA warp never idle behind a backward sweep;
//   * warp roles: warps 0-7 = the two recursion groups (one thread per utterance: the left-to-right chain of 8
//     states is register resident, log-sum-exp in the forward sweep, max-normalised linear sums in the backward
//     sweep), warps 8-15 standardise / square / split the features into the A operand (two groups, each converting
//     every second frame into its own A stage), warp 16 issues the MMAs, warps 17-19 issue the bulk copies.  20 warps
//     = 5 per scheduler keep 96 registers per thread: with 24 warps (three converter groups) the cap is 80, the
//     backward sweep's one-frame-ahead scratch loads spill and stall on their own spill stores (measured), and
//     setmaxnreg does not raise the allocator's cap.
#include "tc_common.cuh"

#define ET_REC_WGS 2
#define ET_REC_WARPS 4                                    /* per recursion group: warps 0-3, 4-7 */
#define ET_CONV_GROUPS 2
#define ET_CONV_WARP0 (4 * ET_REC_WGS)                     /* 8 */
#define ET_CONV_WARPS (4 * ET_CONV_GROUPS)                 /* warps 8 .. 15 */
#define ET_MMA_WARP (ET_CONV_WARP0 + ET_CONV_WARPS)        /* 16 */
#define ET_LOAD_WARP0 (ET_MMA_WARP + 1)                    /* 17 .. 19 */
#define ET_LOADERS 3
#define ET_THREADS (32 * (ET_LOAD_WARP0 + ET_LOADERS))     /* 640 */
#define ET_PF 3                                             /* backward sweep: L1 prefetch distance in frames */
#define ET_ACC_W 64                                        /* accumulator stage: up to 4 models x 16 columns */

struct EtParams {
    const float *X; int ldx; const int64_t *offsets; int B;
    const int32_t *order; const int32_t *model_start;       // utterance ids grouped by model; [M+1] group starts
    int M, D, nck, ncols;
    const __half *wimg; const float *sb; const float4 *trp;
    float *scratch; int maxT;                                // alpha-hat | e': [grid][2][maxT][16][128]
    float *gamma;                                            // [sum_T][8]
    float *ustats;                                           // [B][24] by position in order[]: G | Xi | occ
    double *loglik;                                          // [B] by utterance id
    int Fshift, nst_shift; uint32_t rstride;
    int pf;                                                  // backward sweep: L1 prefetch distance in frames
    long long *trace;                                        // [ET_TRACE_ROLES][ET_TRACE_FRAMES][ET_TRACE_EVENTS] or null
};

struct EtSmem { uint32_t w, raw, tr, sb, pad, bar, total; };
__host__ __device__ inline EtSmem et_smem_layout(int M, int nck, int ncols, int nst, uint32_t rstride) {
    EtSmem L;
    L.w = 0;
    L.raw = (uint32_t)2 * (ncols / 8) * nck * 128;
    L.tr = L.raw + (uint32_t)nst * TC_ROWS * rstride;
    L.sb = L.tr + (uint32_t)M * TC_TRQ * 16;
    L.pad = (L.sb + (uint32_t)8 * nck * 4 + 15u) & ~15u;        // int pad_start[16], cnt[16]
    L.bar = L.pad + 32 * 4;
    L.total = L.bar + (2 * TC_MAX_STAGES + 12) * 8 + 16;
    return L;
}

// log(exp(x) + exp(y)), fp32 production form
// branch-free (a select, not a jump), so the eight independent chains of a frame interleave in one warp:
// ex2 / lg2 on the special-function unit, |x - y| = inf gives exp(-inf) = 0, both -inf gives NaN which the select drops
__device__ __forceinline__ float lae32(float x, float y) {
    const float m = fmaxf(x, y);
    float t, r;
    asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(t) : "f"(-1.4426950408889634f * fabsf(x - y)));
    asm("lg2.approx.ftz.f32 %0, %1;" : "=f"(r) : "f"(1.0f + t));
    r = fmaf(r, 0.6931471805599453f, m);
    return (m == -INFINITY) ? m : r;
}
__device__ __forceinline__ float fexp32(float x) {      // exp(x), x <= 0 or -inf
    float t;
    asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(t) : "f"(1.4426950408889634f * x));
    return t;
}

// TRACE: CTA 0 records clock64() at its pipeline events (tuning aid, SAPR_ET_TRACE=file)
#define ET_TRACE_FRAMES 64
#define ET_TRACE_F0 440                           /* third tile of CTA 0: steady state, a backward sweep runs alongside */
#define ET_TRACE_EVENTS 4
#define ET_TRACE_ROLES 4
template <bool TRACE, int NKS>
__global__ void __launch_bounds__(ET_THREADS, 1) k_estep_tc(const EtParams p) {
    extern __shared__ __align__(128) unsigned char smem[];
    const int nck = p.nck, ncols = p.ncols, M = p.M;
    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
    const int F = 1 << p.Fshift, nst = 1 << p.nst_shift;
    const uint32_t rowbytes = (uint32_t)p.ldx * 4u, rstride = p.rstride, stage_bytes = TC_ROWS * rstride;
    const EtSmem L = et_smem_layout(M, nck, ncols, nst, rstride);
    const uint32_t w_plane = (uint32_t)(ncols / 8) * nck * 128;
    unsigned char *sW = smem + L.w;
    unsigned char *sRaw = smem + L.raw;
    const float4 *sTr = reinterpret_cast<const float4 *>(smem + L.tr);
    const float4 *sS = reinterpret_cast<const float4 *>(smem + L.sb);
    int *sPad = reinterpret_cast<int *>(smem + L.pad);          // pad_start[0..M], then cnt[0..M-1] at +16
    uint64_t *sBar = reinterpret_cast<uint64_t *>(smem + L.bar);
    uint32_t *sTmem = reinterpret_cast<uint32_t *>(sBar + 2 * TC_MAX_STAGES + 12);
    const uint32_t barRaw_full = smem_u32(sBar), barRaw_empty = barRaw_full + 8 * TC_MAX_STAGES;
    const uint32_t barA_full = barRaw_empty + 8 * TC_MAX_STAGES, barA_free = barA_full + 24;   // [<= 3], [<= 3]
    const uint32_t barAcc_full = barA_free + 24, barAcc_empty = barAcc_full + 16;               // [2], [2]
    const uint32_t barTurn = barAcc_empty + 16;                                                 // [2]: forward-sweep hand-over between the recursion groups

    {
        const uint4 *src = reinterpret_cast<const uint4 *>(p.wimg);
        uint4 *dst = reinterpret_cast<uint4 *>(sW);
        for (uint32_t i = tid; i < 2 * w_plane / 16; i += ET_THREADS) dst[i] = src[i];
        float4 *dtr = reinterpret_cast<float4 *>(smem + L.tr);
        for (int i = tid; i < M * TC_TRQ; i += ET_THREADS) dtr[i] = p.trp[i];
        float *dsb = reinterpret_cast<float *>(smem + L.sb);
        for (int i = tid; i < 8 * nck; i += ET_THREADS) dsb[i] = p.sb[i];
    }
    if (tid == 0) {
        int acc = 0;
        for (int m = 0; m < M; m++) {
            const int cnt = p.model_start[m + 1] - p.model_start[m];
            sPad[m] = acc; sPad[16 + m] = cnt;
            acc += (cnt + 31) / 32 * 32;
        }
        sPad[M] = acc;
        for (int s = 0; s < nst; s++) {
            mbar_init(barRaw_full + 8 * s, 32 * ET_LOADERS);
            mbar_init(barRaw_empty + 8 * s, ET_CONV_WARPS);
        }
        for (int s = 0; s < ET_CONV_GROUPS; s++) { mbar_init(barA_full + 8 * s, 4); mbar_init(barA_free + 8 * s, 1); }   // one converter group per A stage
        for (int s = 0; s < 2; s++) { mbar_init(barAcc_full + 8 * s, 1); mbar_init(barAcc_empty + 8 * s, ET_REC_WARPS); mbar_init(barTurn + 8 * s, ET_REC_WARPS); }
        fence_barrier_init();
    }
    const uint32_t a_cols = 8u * nck;
    uint32_t tcols = 32;
    while (tcols < 2u * ET_ACC_W + (uint32_t)ET_CONV_GROUPS * a_cols) tcols <<= 1;
    if (warp == ET_MMA_WARP) tmem_alloc(smem_u32(sTmem), tcols);
    fence_proxy_async();
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    const uint32_t tmem_base = *sTmem;
    const uint32_t tmem_acc = tmem_base, tmem_a = tmem_base + 2u * ET_ACC_W;   // 2 accumulator stages, then the A stages

    const int total_pad = sPad[M];
    const int ntiles = (total_pad + TC_ROWS - 1) / TC_ROWS;

    // padded row -> (model, utterance id or -1, frames)
    auto row_info = [&](int prow, int &m, int &pos, int64_t &off) -> int {
        m = 0; pos = -1; off = 0;
        if (prow >= total_pad) { m = M - 1; return 0; }
        while (m + 1 < M && prow >= sPad[m + 1]) m++;
        const int idx = prow - sPad[m];
        if (idx >= sPad[16 + m]) return 0;
        pos = p.model_start[m] + idx;
        const int u = p.order[pos];
        off = p.offsets[u];
        return min((int)(p.offsets[u + 1] - off), p.maxT);      // the scratch holds maxT frames per row
    };
    auto tile_frames = [&](int tile) -> int {
        int Tt = 0;
        for (int r = lane; r < TC_ROWS; r += 32) {
            int m, pos; int64_t o;
            Tt = max(Tt, row_info(tile * TC_ROWS + r, m, pos, o));
        }
        for (int o = 16; o > 0; o >>= 1) Tt = max(Tt, __shfl_xor_sync(0xffffffffu, Tt, o));
        return Tt;
    };
    // first model of a tile and how many adjacent models it spans (1 .. 4: every group is padded to 32 rows)
    auto tile_models = [&](int tile, int &mf) -> int {
        int ml;
        const int r0 = tile * TC_ROWS, r1 = min(r0 + TC_ROWS, total_pad) - 1;
        mf = 0;
        while (mf + 1 < M && r0 >= sPad[mf + 1]) mf++;
        ml = mf;
        while (ml + 1 < M && r1 >= sPad[ml + 1]) ml++;
        return ml - mf + 1;
    };

    uint32_t f = 0, sg = 0;
    auto trace = [&](int role, uint32_t frame, int ev) {
        if (TRACE && blockIdx.x == 0 && lane == 0 && frame >= ET_TRACE_F0 && frame < ET_TRACE_F0 + ET_TRACE_FRAMES)
            p.trace[((size_t)role * ET_TRACE_FRAMES + (frame - ET_TRACE_F0)) * ET_TRACE_EVENTS + ev] = clock64();
    };

    if (warp >= ET_LOAD_WARP0) {
        // ===================== bulk-copy producers: the forward sweep of every tile =====================
        constexpr int RPL = (TC_ROWS + ET_LOADERS - 1) / ET_LOADERS;
        constexpr int RPT = (RPL + 31) / 32;
        const int lw = warp - ET_LOAD_WARP0;
        const int rlo = lw * RPL, rhi = min(rlo + RPL, TC_ROWS);
        for (int tile = blockIdx.x; tile < ntiles; tile += gridDim.x) {
            const int Tt = tile_frames(tile);
            const int nsg = (Tt + F - 1) >> p.Fshift;
            int Te[RPT]; int64_t off[RPT];
#pragma unroll
            for (int i = 0; i < RPT; i++) {
                const int rr = rlo + lane + 32 * i;
                int m, pos;
                Te[i] = (rr < rhi) ? row_info(tile * TC_ROWS + rr, m, pos, off[i]) : 0;
                if (rr >= rhi) off[i] = 0;
            }
            for (int k = 0; k < nsg; k++, sg++) {
                const uint32_t slot = sg & (uint32_t)(nst - 1), ph = (sg >> p.nst_shift) & 1u;
                const uint32_t bar = barRaw_full + 8 * slot;
                int nf[RPT], tot = 0;
#pragma unroll
                for (int i = 0; i < RPT; i++) { nf[i] = min(max(Te[i] - k * F, 0), F); tot += nf[i]; }
                if (lw == 0) trace(3, sg * 4 + ET_TRACE_F0, 0);
                mbar_wait(barRaw_empty + 8 * slot, ph ^ 1u);
                if (lw == 0) trace(3, sg * 4 + ET_TRACE_F0, 1);
                mbar_arrive_tx(bar, (uint32_t)tot * rowbytes);
#pragma unroll
                for (int i = 0; i < RPT; i++)
                    if (nf[i] > 0)
                        bulk_g2s(smem_u32(sRaw) + slot * stage_bytes + (uint32_t)(rlo + lane + 32 * i) * rstride,
                                 p.X + (size_t)(off[i] + k * F) * p.ldx, (uint32_t)nf[i] * rowbytes, bar);
                if (lw == 0) trace(3, sg * 4 + ET_TRACE_F0, 2);
            }
        }
    } else if (warp == ET_MMA_WARP) {
        // ===================== MMA issuer =====================
        const uint32_t sW_hi = smem_u32(sW);
        const uint32_t sboW = (uint32_t)nck * 128u;
        const int nks = nck / 2;
        const uint32_t idesc = (1u << 4) | ((uint32_t)(16 >> 3) << 17) | ((uint32_t)(TC_ROWS >> 4) << 24);   // M = 128, N = 16
        uint32_t a3 = 0, aph = 0;
        for (int tile = blockIdx.x; tile < ntiles; tile += gridDim.x) {
            const int Tt = tile_frames(tile);
            int mf;
            const int nm = tile_models(tile, mf);
            // B = [W_hi rows of model m | W_lo rows of model m]: the second 8-row group lies one plane further
            const uint64_t dW0 = make_desc(sW_hi + (uint32_t)mf * sboW, 128, w_plane);
            for (int t = 0; t < Tt; t++, f++) {
                const uint32_t s = f & 1, ph = (f >> 1) & 1;
                trace(0, f, 0);
                mbar_wait(barA_full + 8 * a3, aph);
                trace(0, f, 1);
                mbar_wait(barAcc_empty + 8 * s, ph ^ 1u);
                trace(0, f, 2);
                tc_fence_after();
                if (elect_one()) {
                    const uint32_t a_hi = tmem_a + a3 * a_cols, a_lo = a_hi + 8u;
                    uint32_t d_tmem = tmem_acc + s * (uint32_t)ET_ACC_W;
                    uint64_t dW = dW0;
                    for (int mi = 0; mi < nm; mi++, d_tmem += 16u, dW += (uint64_t)(sboW >> 4)) {
                        if (NKS > 0) {
#pragma unroll
                            for (int ks = 0; ks < NKS; ks++) umma_f16_ts(d_tmem, a_lo + ks * 16, dW + (uint64_t)(16 * ks), idesc, ks > 0);   // lo * [W_hi | W_lo]
#pragma unroll
                            for (int ks = 0; ks < NKS; ks++) umma_f16_ts(d_tmem, a_hi + ks * 16, dW + (uint64_t)(16 * ks), idesc, 1);        // hi * [W_hi | W_lo]
                        } else {
                            uint64_t dd = dW;
                            uint32_t a = a_lo;
                            for (int ks = 0; ks < nks; ks++, a += 16, dd += 16) umma_f16_ts(d_tmem, a, dd, idesc, ks > 0);
                            a = a_hi; dd = dW;
                            for (int ks = 0; ks < nks; ks++, a += 16, dd += 16) umma_f16_ts(d_tmem, a, dd, idesc, 1);
                        }
                    }
                    umma_commit(barAcc_full + 8 * s);
                    umma_commit(barA_free + 8 * a3);
                }
                __syncwarp();
                trace(0, f, 3);
                if (++a3 == ET_CONV_GROUPS) { a3 = 0; aph ^= 1u; }
            }
        }
    } else {
        const int q = warp & 3, r = q * 32 + lane;
        const uint32_t lane_sel = (uint32_t)(q * 32) << 16;
        auto lds4 = [](uint32_t a) -> float4 {
            float4 v;
            asm volatile("ld.shared.v4.f32 {%0, %1, %2, %3}, [%4];" : "=f"(v.x), "=f"(v.y), "=f"(v.z), "=f"(v.w) : "r"(a));
            return v;
        };
        if (warp >= ET_CONV_WARP0) {
            // ===================== converters: features -> A operand in TMEM =====================
            // Frame-parallel: converter group gi owns A stage gi and converts every ET_CONV_GROUPS-th frame (all feature
            // chunks of its row).  One conversion is a ~1000-cycle dependent chain (LDS -> FFMA2 -> F2FP -> ... ->
            // tcgen05.st -> wait), so frames in flight -- not more threads per frame -- is what raises the frame rate.
            const uint32_t gi = (uint32_t)((warp - ET_CONV_WARP0) >> 2);
            const int npairs = nck / 2;
            const uint32_t ta = tmem_a + lane_sel + gi * a_cols;
            const uint32_t raw0 = smem_u32(sRaw) + (uint32_t)r * rstride;
            const uint32_t sbS = smem_u32(sS), sbB = sbS + 16u * nck;
            const int nrd4 = p.ldx / 4;
            uint32_t cph = 0;
            auto split4 = [&](const float4 x, const float4 sc, const float4 of, uint32_t *hi, uint32_t *lo) {
                const float2 a01 = fma2(make_float2(x.x, x.y), make_float2(sc.x, sc.y), make_float2(of.x, of.y));
                const float2 a23 = fma2(make_float2(x.z, x.w), make_float2(sc.z, sc.w), make_float2(of.z, of.w));
                const float2 q01 = mul2(a01, a01), q23 = mul2(a23, a23);
                hi[0] = pack_h2(a01); hi[1] = pack_h2(a23); hi[2] = pack_h2(q01); hi[3] = pack_h2(q23);
                lo[0] = pack_h2(sub2(a01, unpack_h2(hi[0]))); lo[1] = pack_h2(sub2(a23, unpack_h2(hi[1])));
                lo[2] = pack_h2(sub2(q01, unpack_h2(hi[2]))); lo[3] = pack_h2(sub2(q23, unpack_h2(hi[3])));
            };
            uint32_t fm3 = 0;                              // f % ET_CONV_GROUPS, kept incrementally
            for (int tile = blockIdx.x; tile < ntiles; tile += gridDim.x) {
                const int Tt = tile_frames(tile);
                int m, pos; int64_t off;
                const int Te = row_info(tile * TC_ROWS + r, m, pos, off);
                bool waited = false;                   // raw_full of the current stage already observed by this warp
                for (int tau = 0; tau < Tt; tau++, f++) {
                    const int fi = tau & (F - 1);
                    const uint32_t slot = sg & (uint32_t)(nst - 1);
                    if (fm3 == gi) {
                        if (warp == ET_CONV_WARP0) trace(1, f, 0);
                        if (!waited) { mbar_wait(barRaw_full + 8 * slot, (sg >> p.nst_shift) & 1u); waited = true; }
                        if (warp == ET_CONV_WARP0) trace(1, f, 1);
                        const bool ok = tau < Te;
                        const uint32_t rowp = raw0 + slot * stage_bytes + (uint32_t)(ok ? fi : 0) * rowbytes;
                        // A stage free?  (the MMAs that read it ET_CONV_GROUPS frames ago have completed)
                        mbar_wait(barA_free + 8 * gi, cph ^ 1u);
                        if (warp == ET_CONV_WARP0) trace(1, f, 2);
                        tc_fence_after();
#pragma unroll 2
                        for (int c = 0; c < npairs; c++) {
                            float4 x0 = make_float4(0.f, 0.f, 0.f, 0.f), x1 = x0;
                            if (ok && 2 * c < nrd4) x0 = lds4(rowp + 32u * c);
                            if (ok && 2 * c + 1 < nrd4) x1 = lds4(rowp + 32u * c + 16u);
                            uint32_t v[16];
                            split4(x0, lds4(sbS + 32u * c), lds4(sbB + 32u * c), v, v + 8);
                            split4(x1, lds4(sbS + 32u * c + 16u), lds4(sbB + 32u * c + 16u), v + 4, v + 12);
                            tmem_st16(ta + 16u * c, v);
                        }
                        tmem_st_wait();
                        tc_fence_before();
                        __syncwarp();
                        if (lane == 0) mbar_arrive(barA_full + 8 * gi);
                        cph ^= 1u;
                        if (warp == ET_CONV_WARP0) trace(1, f, 3);
                    }
                    if (fi == F - 1 || tau == Tt - 1) {      // leaving this stage: every converter warp releases it once
                        __syncwarp();
                        if (lane == 0) mbar_arrive(barRaw_empty + 8 * slot);
                        sg++; waited = false;
                    }
                    if (++fm3 == ET_CONV_GROUPS) fm3 = 0;
                }
            }
        } else {
            // ===================== recursions: one thread per utterance, two groups alternating tiles =====================
            const int wg = warp >> 2;
            float *scr = p.scratch + (size_t)(blockIdx.x * ET_REC_WGS + wg) * p.maxT * 16 * TC_ROWS + r;      // [t][alpha-hat 0-7 | e' 8-15][row]
            int kt = 0;
            for (int tile = blockIdx.x; tile < ntiles; tile += gridDim.x, kt++) {
                const int Tt = tile_frames(tile);
                if ((kt & 1) != wg) { f += (uint32_t)Tt; continue; }         // the other group's tile
                // The accumulator barriers carry one parity bit: a group may only start waiting on them once the other group
                // has consumed the last frame of the previous tile (its hand-over arrival), or a stale phase would pass.
                if (kt > 0) mbar_wait(barTurn + 8 * wg, (uint32_t)(((kt - 1) >> 1) & 1));
                int mf;
                tile_models(tile, mf);
                int m, pos; int64_t off;
                const int T = row_info(tile * TC_ROWS + r, m, pos, off);
                const int u = pos >= 0 ? p.order[pos] : 0;
                const uint32_t acc_col = tmem_acc + lane_sel + (uint32_t)(m - mf) * 16u;   // warp-uniform: one model per quadrant
                // transition constants of this thread's model stay in shared memory and are re-read every frame: holding the
                // 25 of them in registers made the recursion spill (local-memory round trips inside a serial chain)
                const uint32_t trM = smem_u32(sTr) + (uint32_t)m * (TC_TRQ * 16u);
                const float lb0 = sTr[m * TC_TRQ + 2].y;

                // e'_t(j) = E[t, j] + ln A[j, j] of this thread's model, frame counter fr: the W_hi and the W_lo products
                // arrive in separate accumulator columns
                auto fetch = [&](uint32_t fr, float (&e)[8]) {
                    const uint32_t s = fr & 1u;
                    if (warp == 0) trace(2, fr, 0);
                    mbar_wait(barAcc_full + 8 * s, (fr >> 1) & 1u);
                    if (warp == 0) trace(2, fr, 1);
                    tc_fence_after();
                    uint32_t ev[16];
                    tmem_ld16(acc_col + s * (uint32_t)ET_ACC_W, ev);
                    tmem_ld_wait();
                    tc_fence_before();
                    __syncwarp();
                    if (lane == 0) mbar_arrive(barAcc_empty + 8 * s);
                    if (warp == 0) trace(2, fr, 2);
#pragma unroll
                    for (int j = 0; j < 8; j++) e[j] = __uint_as_float(ev[j]) + __uint_as_float(ev[8 + j]);
                };

                // ---------------- forward (custom_hmm.py:176-211), U_j = alpha-hat_j + ln A[j,j] ----------------
                float U[8], ax = -INFINITY, base = 0.f;
                float best_mx = 0.f, best_base = 0.f;        // max over all alpha cells = best_mx + best_base; alpha[0,0] = 0
                double ll = 0.0;
                bool exit_ok = false, xi_live = true;
#pragma unroll
                for (int j = 0; j < 8; j++) U[j] = -INFINITY;
                for (int t = 0; t < Tt; t++, f++) {
                    float e[8];
                    fetch(f, e);
                    if (t < T) {
                        const float4 c03 = lds4(trM), c47 = lds4(trM + 16u), st03 = lds4(trM + 48u), st47 = lds4(trM + 64u);
                        const float cadv[8] = {0.f, c03.x, c03.y, c03.z, c03.w, c47.x, c47.y, c47.z};   // into state j from j-1 (U form)
                        const float stay[8] = {st03.x, st03.y, st03.z, st03.w, st47.x, st47.y, st47.z, st47.w};
                        float *sp = scr + (size_t)t * 16 * TC_ROWS;
#pragma unroll
                        for (int j = 0; j < 8; j++) sp[(8 + j) * TC_ROWS] = e[j];
                        if (t == 0) {
                            U[0] = lb0 + e[0];
                        } else {
                            const float nx = U[7] + c47.w;                    // alpha[t, exit] = alpha[t-1, N] + ln A[N, exit]
#pragma unroll
                            for (int j = 7; j >= 1; j--) U[j] = lae32(U[j - 1] + cadv[j], U[j]) + e[j];
                            const float ent = (t == 1) ? lb0 - base : -INFINITY;     // alpha[t-1, entry] is 0 at t == 1 only
                            U[0] = lae32(ent, U[0]) + e[0];
                            ax = nx;
                        }
                        float a[8];
#pragma unroll
                        for (int j = 0; j < 8; j++) a[j] = U[j] - stay[j];
                        float mx = fmaxf(fmaxf(a[0], a[1]), ax);
                        mx = fmaxf(fmaxf(a[2], a[3]), mx);
                        mx = fmaxf(fmaxf(a[4], a[5]), mx);
                        mx = fmaxf(fmaxf(a[6], a[7]), mx);
                        if (mx + base > best_mx + best_base) { best_mx = mx; best_base = base; }
                        if (t == T - 1) {      // reported log-likelihood (SURVEY D6): logaddexp.reduce(alpha[T-1, :]) - max(alpha)
                            float rr = (T == 1) ? 0.f - base : -INFINITY;
#pragma unroll
                            for (int j = 0; j < 8; j++) rr = lae32(rr, a[j]);
                            rr = lae32(rr, ax);
                            ll = ((double)rr + (double)base) - ((double)best_mx + (double)best_base);
                            exit_ok = (T > 1) && (ax > -INFINITY);
                            xi_live = !(ax - rr < -745.13f);      // SURVEY D10 (see k_estep_fused): the reference's float64 xi underflows for the whole utterance
                        }
                        // renormalise with an integer shift (exactly representable running offset)
                        const float sh = (t == 0) ? 0.f : rintf(fminf(fmaxf(mx, -4194304.f), 4194304.f));   // frame 0 stays unshifted (alpha[0, entry] = 0)
#pragma unroll
                        for (int j = 0; j < 8; j++) { U[j] -= sh; a[j] -= sh; }
                        ax -= sh; base += sh;
#pragma unroll
                        for (int j = 0; j < 8; j++) sp[j * TC_ROWS] = a[j];
                    }
                }
                __syncwarp();
                if (lane == 0) mbar_arrive(barTurn + 8 * (wg ^ 1));              // forward sweep done: the other group's turn
                if (pos >= 0 && T > 0) p.loglik[u] = ll;

                // ---------------- backward + gamma + xi sums (custom_hmm.py:213-322): thread-private over the scratch ----------------
                float gG[8], gX[8], b[8], en[8];
                float glast = 0.f;                                 // gamma[T-1, j] of the emitting states (0 or NaN): occ = G + it
#pragma unroll
                for (int j = 0; j < 8; j++) { gG[j] = 0.f; gX[j] = 0.f; b[j] = -INFINITY; en[j] = 0.f; }
                float bx = 0.f;                                    // beta[T-1, exit] = 0
                float atn[8];                                      // alpha-hat of the next backward frame, loaded one frame ahead
#pragma unroll
                for (int j = 0; j < 8; j++) atn[j] = 0.f;
                if (T >= 2) {
                    const float *sp = scr + (size_t)(T - 2) * 16 * TC_ROWS;
#pragma unroll
                    for (int j = 0; j < 8; j++) atn[j] = sp[j * TC_ROWS];
                }
                for (int t = T - 1; t >= 0; t--) {
                    // The scratch rows of this tile left L2 long ago (1.6 MB per group, 296 groups): one iteration does not
                    // cover a DRAM round trip and registers for a deeper prefetch are not there, so the lines of frame
                    // t - ET_PF are pulled into L1 now (one 128-byte line per state and warp) and the loads below hit there.
                    if (t >= p.pf) {
                        const float *pp = scr + (size_t)(t - p.pf) * 16 * TC_ROWS;
#pragma unroll
                        for (int j = 0; j < 16; j++) asm volatile("prefetch.global.L1 [%0];" ::"l"(pp + j * TC_ROWS));
                    }
                    float e[8];                                    // e'_t: consumed at the end of this iteration (as e'_{t+1} of the next)
                    {
                        const float *sp = scr + (size_t)t * 16 * TC_ROWS;
#pragma unroll
                        for (int j = 0; j < 8; j++) e[j] = sp[(8 + j) * TC_ROWS];
                    }
                    float *go = p.gamma + (size_t)(off + t) * 8;
                    if (t == T - 1) {
                        // gamma[T-1] is one-hot on the exit state unless alpha[T-1, exit] = -inf (then the row is NaN)
                        const float gl = exit_ok ? 0.f : NAN;
                        *reinterpret_cast<float4 *>(go) = make_float4(gl, gl, gl, gl);
                        *reinterpret_cast<float4 *>(go + 4) = make_float4(gl, gl, gl, gl);
                        glast = gl;
                    } else {
                        const float4 bd03 = lds4(trM + 80u), bd47 = lds4(trM + 96u);
                        const float badv[7] = {bd03.x, bd03.y, bd03.z, bd03.w, bd47.x, bd47.y, bd47.z};
                        float at[8], self[8], nb[8];
#pragma unroll
                        for (int j = 0; j < 8; j++) { at[j] = atn[j]; self[j] = en[j] + b[j]; }   // ln A_jj + e_{t+1}(j) + beta_{t+1}(j)
                        if (t >= 1) {
                            const float *sp = scr + (size_t)(t - 1) * 16 * TC_ROWS;
#pragma unroll
                            for (int j = 0; j < 8; j++) atn[j] = sp[j * TC_ROWS];
                        }
#pragma unroll
                        for (int j = 0; j < 7; j++) nb[j] = lae32(self[j], badv[j] + self[j + 1]);
                        nb[7] = lae32(self[7], bd47.w + bx);                         // ln A[N, exit] + beta[t+1, exit]
                        const float b0 = sTr[m * TC_TRQ + 7].x + self[0];            // beta[t, entry] = ln A01 - ln A11 + self_1
                        float lg[8];
#pragma unroll
                        for (int j = 0; j < 8; j++) lg[j] = at[j] + nb[j];
                        const float xs7 = at[7] + self[7];
                        float mxl = fmaxf(fmaxf(lg[0], lg[1]), lg[2]);
                        mxl = fmaxf(fmaxf(lg[3], lg[4]), mxl);
                        mxl = fmaxf(fmaxf(lg[5], lg[6]), mxl);
                        mxl = fmaxf(lg[7], mxl);
                        const float ent = (t == 0) ? b0 : -INFINITY;                 // alpha[0, entry] = 0
                        mxl = fmaxf(mxl, ent);
                        float pj[8], sum = 0.f;
#pragma unroll
                        for (int j = 0; j < 8; j++) { pj[j] = fexp32(lg[j] - mxl); sum += pj[j]; }
                        const float pe = fexp32(ent - mxl);
                        // xi normaliser (:319-320): arcs (0,1), (i,i), (i,i+1) for i < N; the (N, exit) arc contributes 0
                        const float q7 = fexp32(xs7 - mxl);
                        const float xsum = (sum - pj[7]) + q7 + pe;
                        sum += pe;
                        const float inv = 1.0f / sum;                                // all -inf row -> NaN like the reference
                        const float xinv = (xi_live && mxl > -INFINITY && xsum > 0.f) ? 1.0f / xsum : 0.f;
                        float gm[8];
#pragma unroll
                        for (int j = 0; j < 8; j++) {
                            gm[j] = pj[j] * inv;
                            gG[j] += gm[j];
                            const float xq = (mxl > -INFINITY) ? fexp32((at[j] + self[j]) - mxl) : 0.f;
                            gX[j] += xq * xinv;
                        }
                        *reinterpret_cast<float4 *>(go) = make_float4(gm[0], gm[1], gm[2], gm[3]);
                        *reinterpret_cast<float4 *>(go + 4) = make_float4(gm[4], gm[5], gm[6], gm[7]);
                        float mb = fmaxf(fmaxf(nb[0], nb[1]), nb[2]);
                        mb = fmaxf(fmaxf(nb[3], nb[4]), mb);
                        mb = fmaxf(fmaxf(nb[5], nb[6]), mb);
                        mb = fmaxf(nb[7], mb);
                        const bool fin = mb > -INFINITY && mb < INFINITY;
#pragma unroll
                        for (int j = 0; j < 8; j++) b[j] = fin ? nb[j] - mb : nb[j];
                        bx = -INFINITY;
                    }
#pragma unroll
                    for (int j = 0; j < 8; j++) en[j] = e[j];
                }
                if (pos >= 0) {
                    float *us = p.ustats + (size_t)pos * 24;
#pragma unroll
                    for (int j = 0; j < 8; j++) { us[j] = gG[j]; us[8 + j] = gX[j]; us[16 + j] = gG[j] + glast; }
                }
            }
        }
    }
    tc_fence_before();
    __syncthreads();
    if (warp == ET_MMA_WARP) tmem_dealloc(tmem_base, tcols);
}

// ------------------------------------------------------------------------------------------------
size_t sapr_tc_image_bytes(const sapr_models *m, int *nck_out, int *ncols_out);

// launcher: fills gamma [sum_T][8] (fp32), ustats [B][24] by position in order[], loglik[B]
int sapr_estep_tc_launch(sapr_ctx *ctx, sapr_models *m, const float *X, int ldx, const int64_t *offsets, int B, int max_T,
                         const int32_t *order, const int32_t *model_start, float *gamma, float *ustats, double *loglik) {
    int nck, ncols;
    sapr_tc_image_bytes(m, &nck, &ncols);
    auto al256 = [](size_t x) { return (x + 255) / 256 * 256; };
    const size_t w = al256((size_t)2 * (ncols / 8) * nck * 64 * sizeof(__half));
    const size_t g = al256((size_t)8 * nck * sizeof(float));
    const int M = m->M;
    const uint32_t rowbytes = (uint32_t)ldx * 4u;
    const size_t budget = 225 * 1024;
    int Fshift = 3, nst = 2, nst_shift = 1;
    uint32_t rstride = 0;
    EtSmem L;
    for (;; Fshift--) {
        const uint32_t F = 1u << Fshift;
        rstride = F * rowbytes + 16u;
        if (((rstride >> 4) & 1u) == 0) rstride += 16u;
        L = et_smem_layout(M, nck, ncols, nst, rstride);
        if (L.total <= budget) break;
        if (Fshift == 0) SAPR_FAIL(ctx, SAPR_E_RANGE, "estep (tensor core): feature rows too wide for the shared-memory ring");
    }
    if (Fshift <= 1 && et_smem_layout(M, nck, ncols, 4, rstride).total <= budget) { nst = 4; nst_shift = 2; }
    L = et_smem_layout(M, nck, ncols, nst, rstride);
    const int grid = std::min((B + 31 * M + TC_ROWS - 1) / TC_ROWS, ctx->sm_count);
    int rc = sapr_ws_reserve(ctx, 7, (size_t)grid * ET_REC_WGS * max_T * 16 * TC_ROWS * sizeof(float));
    if (rc) return rc;
    EtParams prm;
    prm.X = X; prm.ldx = ldx; prm.offsets = offsets; prm.B = B; prm.order = order; prm.model_start = model_start;
    prm.M = M; prm.D = m->D; prm.nck = nck; prm.ncols = ncols;
    prm.wimg = (const __half *)m->tc_image;
    prm.sb = (const float *)((const char *)m->tc_image + w);
    prm.trp = (const float4 *)((const char *)m->tc_image + w + g);
    prm.scratch = (float *)ctx->ws[7]; prm.maxT = max_T;
    prm.gamma = gamma; prm.ustats = ustats; prm.loglik = loglik;
    prm.Fshift = Fshift; prm.nst_shift = nst_shift; prm.rstride = rstride;
    prm.pf = ET_PF;
    prm.trace = nullptr;
    const char *trace_path = getenv("SAPR_ET_TRACE");
    if (trace_path) {       // tuning aid: one traced launch, timestamps to a text file
        const size_t nrec = (size_t)ET_TRACE_ROLES * ET_TRACE_FRAMES * ET_TRACE_EVENTS;
        long long *dtr = nullptr;
        SAPR_CUDA(ctx, cudaMalloc(&dtr, nrec * sizeof(long long)));
        SAPR_CUDA(ctx, cudaMemsetAsync(dtr, 0, nrec * sizeof(long long), ctx->stream));
        prm.trace = dtr;
        SAPR_CUDA(ctx, cudaFuncSetAttribute(k_estep_tc<true, 0>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)L.total));
        k_estep_tc<true, 0><<<grid, ET_THREADS, L.total, ctx->stream>>>(prm);
        SAPR_LAUNCH_CHECK(ctx);
        std::vector<long long> h(nrec);
        cudaMemcpyAsync(h.data(), dtr, nrec * sizeof(long long), cudaMemcpyDeviceToHost, ctx->stream);
        cudaStreamSynchronize(ctx->stream);
        cudaFree(dtr);
        if (FILE *fp = fopen(trace_path, "w")) {
            for (int ro = 0; ro < ET_TRACE_ROLES; ro++)
                for (int fr = 0; fr < ET_TRACE_FRAMES; fr++) {
                    fprintf(fp, "%d %d", ro, fr + ET_TRACE_F0);
                    for (int e = 0; e < ET_TRACE_EVENTS; e++) fprintf(fp, " %lld", h[((size_t)ro * ET_TRACE_FRAMES + fr) * ET_TRACE_EVENTS + e]);
                    fprintf(fp, "\n");
                }
            fclose(fp);
        }
        prm.trace = nullptr;
    }
    auto kern = (nck == 10) ? k_estep_tc<false, 5> : (nck == 4) ? k_estep_tc<false, 2> : k_estep_tc<false, 0>;
    SAPR_CUDA(ctx, cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)L.total));
    {
        ProfScope ps(ctx, 2);
        kern<<<grid, ET_THREADS, L.total, ctx->stream>>>(prm);
    }
    SAPR_LAUNCH_CHECK(ctx);
    return SAPR_OK;
}
