// viterbi_v3.cu -- the cfg-2 headline kernel: batched Viterbi of EQUAL-LENGTH utterances against M <= 12 eight-state word models,
// emission on tcgen05 (same operand images as viterbi_tc.cu), re-cut for instruction count.
//
// Contract: custom_hmm.py:462-514 for every (utterance, model) + decoder.py:42-47, as k_viterbi_tc.  What changed against
// k_viterbi_tc / k_viterbi_tma (which stay for ragged batches, the debug emission dump and all_paths):
//   * Transition constants are gone from the recursion.  With U_j = V_j + ln A[j,j] the step is
//         U'_j = max(U_{j-1} + c_j, U_j) + e_j,      c_j = ln A[j-1,j] - ln A[j-1,j-1],  e_j = E_j + ln A[j,j] (tensor core)
//     and the substitution W_j = U_j - (c_2 + .. + c_j) turns it into  W'_j = max(W_{j-1}, W_j) + e_j : no per-state adds, no
//     constants to hold or load.  The sum of the c's (and the exit arc) is added to the final score only (kx, float64).
//     A model with a zero-probability forward arc has kx = -inf: its score is -inf, as in the reference (no path reaches the
//     exit), and its recursion values are never used.
//   * One 32-bit back-pointer word per (thread, frame) for all of the thread's models (8 "stayed" sign bits per model: exit,
//     states 8..2; state 1 has a predecessor at t == 1 only and borrows the exit slot there), gathered by ONE chained
//     funnel shift per state -- no masks, no inversion, one store per frame instead of one per model.
//   * Four A-operand stages + two accumulator stages = all 512 TMEM columns, frames are processed in blocks of four with
//     every stage index, barrier address and phase a compile-time constant; the raw-feature ring is two stages of four
//     frames filled by TMA tensor-map loads from one thread.  Tiles are padded to a multiple of four frames (zero-filled by
//     the tensor map), so each tile starts at stage 0.
//   * 18 warps (16 workers, MMA issuer, TMA producer): 112 registers per thread, the standardisation constants of a
//     thread's feature chunks live in registers.
#include "tc_common.cuh"

#define V3_THREADS (TC_WORKERS + 64)
#define V3_FB 4                       /* frames per block = frames per raw-ring stage = A-operand stages */

struct V3Params {
    int u0, nu, M, nck, ncols, Tt, Tpad, ntiles;
    const __half *wimg; const float *sb; const float4 *trp;
    uint32_t *bp; uint32_t Bpad;        // back-pointer words [group][Tpad][Bpad]
    double *scores;                     // [nu][M]
    int mod0[TC_GROUPS], nmod[TC_GROUPS], pair0[TC_GROUPS], npair[TC_GROUPS];
    uint32_t rw;                        // bytes per row of the raw ring: (nck + 1) * 16
    long long *trace;                   // [V4_TRACE_ROLES][V4_TRACE_FRAMES][4] clock64 stamps of CTA 0 or null (SAPR_V_TRACE=file)
    int split_col;                      // HALF kernels: accumulator columns of model groups 0-1 (a multiple of 16)
    int hmod0[2][4], hnmod[2][4], hplane[2][4], hshift[2][4], hroles[2];      // HALF kernels: per half and warp group: first model, models (0-2), decision-word plane and byte, active groups
};

struct V3Smem { uint32_t w, raw, tr, sb, bar, total; };
__host__ __device__ inline V3Smem v3_smem_layout(int M, int nck, int ncols, uint32_t rw) {
    V3Smem L;
    L.w = 0;
    L.raw = ((uint32_t)2 * (ncols / 8) * nck * 128 + 127u) & ~127u;
    L.tr = L.raw + 2u * V3_FB * TC_ROWS * rw;
    L.sb = L.tr + (uint32_t)M * TC_TRQ * 16;
    L.bar = (L.sb + (uint32_t)8 * nck * 4 + 15u) & ~15u;
    L.total = L.bar + 12 * 8 + 16;      // raw_full[2], raw_empty[2], A_full[4], acc_full[2]
    return L;
}

__device__ __forceinline__ float4 v3_lds4(uint32_t a) {
    float4 v;
    asm volatile("ld.shared.v4.f32 {%0, %1, %2, %3}, [%4];" : "=f"(v.x), "=f"(v.y), "=f"(v.z), "=f"(v.w) : "r"(a));
    return v;
}
// 4 feature dims: standardise, square, fp16 hi / lo split.  hi = (x'01, x'23, x'^2 01, x'^2 23), lo likewise
__device__ __forceinline__ void v3_split4(const float4 x, const float4 sc, const float4 of, uint32_t *hi, uint32_t *lo) {
    const float2 a01 = fma2(make_float2(x.x, x.y), make_float2(sc.x, sc.y), make_float2(of.x, of.y));
    const float2 a23 = fma2(make_float2(x.z, x.w), make_float2(sc.z, sc.w), make_float2(of.z, of.w));
    const float2 q01 = mul2(a01, a01), q23 = mul2(a23, a23);
    hi[0] = pack_h2(a01); hi[1] = pack_h2(a23); hi[2] = pack_h2(q01); hi[3] = pack_h2(q23);
    lo[0] = pack_h2(residual_h2(a01, hi[0])); lo[1] = pack_h2(residual_h2(a23, hi[1]));
    lo[2] = pack_h2(residual_h2(q01, hi[2])); lo[3] = pack_h2(residual_h2(q23, hi[3]));
}

// one frame of one model in W space; appends 8 "stayed" sign bits to sb: exit first, then states 8 .. 2 (state 2 ends up lowest).
// The predecessor wins ties (sign(+0) = 0 = advanced; custom_hmm.py:488-497 tries j-1 first and replaces on strict > only).
__device__ __forceinline__ void v3_step(float (&W)[8], float &Wx, const float aex, const uint32_t (&ev)[8], uint32_t &sb) {
    const float xs = Wx + aex;                                   // exit self-loop (custom_hmm.py:481-485; D9)
    sb = __funnelshift_l(__float_as_uint(W[7] - xs), sb, 1);
    Wx = fmaxf(W[7], xs);
#pragma unroll
    for (int j = 7; j >= 1; j--) {
        sb = __funnelshift_l(__float_as_uint(W[j - 1] - W[j]), sb, 1);
        W[j] = fmaxf(W[j - 1], W[j]);
    }
#pragma unroll
    for (int j = 0; j < 8; j += 2) {
        const float2 s = add2(make_float2(W[j], W[j + 1]), make_float2(__uint_as_float(ev[j]), __uint_as_float(ev[j + 1])));
        W[j] = s.x; W[j + 1] = s.y;
    }
}
// frame 1: the entry state is still alive (custom_hmm.py:477-480: prev_states = [1, 0], the self-loop wins ties); the exit is
// closed, its slot carries "entry taken"
__device__ __forceinline__ void v3_step_entry(float (&W)[8], float &Wx, const float b0, const uint32_t (&ev)[8], uint32_t &sb) {
    sb = __funnelshift_l(__float_as_uint(W[0] - b0), sb, 1);     // 1 = the entry arc is strictly better
    Wx = -INFINITY;
#pragma unroll
    for (int j = 7; j >= 1; j--) {
        sb = __funnelshift_l(__float_as_uint(W[j - 1] - W[j]), sb, 1);
        W[j] = fmaxf(W[j - 1], W[j]);
    }
    W[0] = fmaxf(W[0], b0);
#pragma unroll
    for (int j = 0; j < 8; j++) W[j] += __uint_as_float(ev[j]);
}
// renormalise by an integer-valued shift (accumulates exactly in fp32 for |offset| < 2^24)
__device__ __forceinline__ void v3_renorm(float (&W)[8], float &Wx, float &base) {
    float mx = fmaxf(fmaxf(W[0], W[1]), Wx);
    mx = fmaxf(fmaxf(W[2], W[3]), mx);
    mx = fmaxf(fmaxf(W[4], W[5]), mx);
    mx = fmaxf(fmaxf(W[6], W[7]), mx);
    mx = rintf(fminf(fmaxf(mx, -4194304.f), 4194304.f));
    const float2 m2 = make_float2(mx, mx);
#pragma unroll
    for (int j = 0; j < 8; j += 2) {
        const float2 s = sub2(make_float2(W[j], W[j + 1]), m2);
        W[j] = s.x; W[j + 1] = s.y;
    }
    Wx -= mx;
    base += mx;
}

template <int NKS>
__global__ void __launch_bounds__(V3_THREADS, 1) k_viterbi_v3(const V3Params p, const __grid_constant__ CUtensorMap tmap) {
    extern __shared__ __align__(128) unsigned char smem[];
    const int nck = p.nck, ncols = p.ncols, M = p.M;
    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
    const uint32_t rw = p.rw, frame_bytes = TC_ROWS * rw, stage_bytes = V3_FB * frame_bytes;
    const V3Smem L = v3_smem_layout(M, nck, ncols, rw);
    const uint32_t w_plane = (uint32_t)(ncols / 8) * nck * 128;
    unsigned char *sW = smem + L.w;
    const uint32_t sRaw = smem_u32(smem + L.raw);
    const float4 *sTr = reinterpret_cast<const float4 *>(smem + L.tr);
    uint64_t *sBar = reinterpret_cast<uint64_t *>(smem + L.bar);
    uint32_t *sTmem = reinterpret_cast<uint32_t *>(sBar + 12);
    const uint32_t barRawFull = smem_u32(sBar), barRawEmpty = barRawFull + 16, barAFull = barRawFull + 32, barAccFull = barRawFull + 64;

    {
        const uint4 *src = reinterpret_cast<const uint4 *>(p.wimg);
        uint4 *dst = reinterpret_cast<uint4 *>(sW);
        for (uint32_t i = tid; i < 2 * w_plane / 16; i += V3_THREADS) dst[i] = src[i];
        float4 *dtr = reinterpret_cast<float4 *>(smem + L.tr);
        for (int i = tid; i < M * TC_TRQ; i += V3_THREADS) dtr[i] = p.trp[i];
        float *dsb = reinterpret_cast<float *>(smem + L.sb);
        for (int i = tid; i < 8 * nck; i += V3_THREADS) dsb[i] = p.sb[i];
    }
    if (tid == 0) {
        for (int s = 0; s < 2; s++) { mbar_init(barRawFull + 8 * s, 1); mbar_init(barRawEmpty + 8 * s, TC_WORKER_WARPS); }
        for (int s = 0; s < 4; s++) mbar_init(barAFull + 8 * s, TC_WORKER_WARPS);
        for (int s = 0; s < 2; s++) mbar_init(barAccFull + 8 * s, 1);
        fence_barrier_init();
    }
    const uint32_t a_cols = 8u * nck;                       // TMEM columns of one A stage: per K step [hi 8 | lo 8]
    if (warp == TC_WORKER_WARPS) tmem_alloc(smem_u32(sTmem), 512);
    fence_proxy_async();
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    const uint32_t tmem_base = *sTmem;
    const uint32_t tmem_acc = tmem_base, tmem_a = tmem_base + 2u * ncols;
    const int Tt = p.Tt, Tpad = p.Tpad;
    const int my_tiles = (p.ntiles - (int)blockIdx.x + (int)gridDim.x - 1) / (int)gridDim.x;     // tiles this CTA walks

    if (warp == TC_WORKER_WARPS + 1) {
        // ===================== TMA producer: one thread, one stage = four frames of a tile =====================
        if (lane == 0) {
            tma_prefetch_desc(&tmap);
            uint32_t G = 0;
            for (int tile = blockIdx.x; tile < p.ntiles; tile += gridDim.x) {
                const int urow = p.u0 + tile * TC_ROWS;
                for (int t0 = 0; t0 < Tpad; t0 += V3_FB, G++) {
                    const uint32_t s = G & 1u, ph = (G >> 1) & 1u;
                    const uint32_t bar = barRawFull + 8 * s;
                    mbar_wait(barRawEmpty + 8 * s, ph ^ 1u);
                    mbar_arrive_tx(bar, stage_bytes);
                    const uint32_t dst = sRaw + s * stage_bytes;
#pragma unroll
                    for (int fi = 0; fi < V3_FB; fi++) tma_load_3d(dst + (uint32_t)fi * frame_bytes, &tmap, 0, t0 + fi, urow, bar);
                }
            }
        }
    } else if (warp == TC_WORKER_WARPS) {
        // ===================== MMA issuer =====================
        const uint32_t idesc = (1u << 4) | ((uint32_t)(ncols >> 3) << 17) | ((uint32_t)(TC_ROWS >> 4) << 24);
        const uint32_t sW_hi = smem_u32(sW), sW_lo = sW_hi + w_plane;
        const uint32_t sboW = (uint32_t)nck * 128u;
        const uint64_t dW_hi = make_desc(sW_hi, 128, sboW), dW_lo = make_desc(sW_lo, 128, sboW);
        const int nks = nck / 2;
        const int nblk = my_tiles * (Tpad / V3_FB);
        uint32_t aph = 0;
        for (int b = 0; b < nblk; b++, aph ^= 1u) {
#pragma unroll
            for (int i = 0; i < V3_FB; i++) {
                mbar_wait(barAFull + 8 * i, aph);
                tc_fence_after();
                if (elect_one()) {
                    const uint32_t d_tmem = tmem_acc + (uint32_t)(i & 1) * (uint32_t)ncols;
                    const uint32_t a_hi = tmem_a + (uint32_t)i * a_cols, a_lo = a_hi + 8u;
                    // the two correction products first: the large hi * W_hi partial sums see the fewest truncating steps
                    if (NKS > 0) {
#pragma unroll
                        for (int ks = 0; ks < NKS; ks++) umma_f16_ts(d_tmem, a_lo + ks * 16, dW_hi + (uint64_t)(16 * ks), idesc, ks > 0);
#pragma unroll
                        for (int ks = 0; ks < NKS; ks++) umma_f16_ts(d_tmem, a_hi + ks * 16, dW_lo + (uint64_t)(16 * ks), idesc, 1);
#pragma unroll
                        for (int ks = 0; ks < NKS; ks++) umma_f16_ts(d_tmem, a_hi + ks * 16, dW_hi + (uint64_t)(16 * ks), idesc, 1);
                    } else {
                        for (int ks = 0; ks < nks; ks++) umma_f16_ts(d_tmem, a_lo + ks * 16, dW_hi + (uint64_t)(16 * ks), idesc, ks > 0);
                        for (int ks = 0; ks < nks; ks++) umma_f16_ts(d_tmem, a_hi + ks * 16, dW_lo + (uint64_t)(16 * ks), idesc, 1);
                        for (int ks = 0; ks < nks; ks++) umma_f16_ts(d_tmem, a_hi + ks * 16, dW_hi + (uint64_t)(16 * ks), idesc, 1);
                    }
                    umma_commit(barAccFull + 8 * (i & 1));
                }
                __syncwarp();
            }
        }
    } else {
        // ===================== workers: thread = (row, group) =====================
        const int q = warp & 3, g = warp >> 2, r = q * 32 + lane;
        const int mbeg = p.mod0[g], pr0 = p.pair0[g];
        const uint32_t lane_sel = (uint32_t)(q * 32) << 16;
        const uint32_t ta0 = tmem_a + lane_sel + 16u * pr0;
        const uint32_t acc0 = tmem_acc + lane_sel + (uint32_t)mbeg * 8u;
        const uint32_t raw0 = sRaw + (uint32_t)r * rw + 32u * pr0;
        const uint32_t sbS = smem_u32(smem + L.sb) + 32u * pr0, sbB = sbS + 16u * nck;

        auto run = [&](auto NPc, auto MCc) {
            constexpr int NP = decltype(NPc)::value, MC = decltype(MCc)::value;
            float aex[MC];
#pragma unroll
            for (int k = 0; k < MC; k++) aex[k] = sTr[(mbeg + k) * TC_TRQ + 2].x;
            uint32_t cG = 0;                                 // raw-ring stage counter of the conversions (stage = cG & 1, phase = cG >> 1)
            // frame (4 G + FI) of the ring -> A stage FI (compile time); waits for / releases the ring stage at its ends
            auto convert = [&](auto FIc) {
                constexpr int FI = decltype(FIc)::value;
                const uint32_t s = cG & 1u;
                if (FI == 0) mbar_wait(barRawFull + 8 * s, (cG >> 1) & 1u);
                const uint32_t src = raw0 + s * stage_bytes + (uint32_t)FI * frame_bytes;
                const uint32_t ta = ta0 + (uint32_t)FI * a_cols;
#pragma unroll
                for (int c = 0; c < 2 * NP; c++) {          // chunk c of this thread: 4 TMEM columns of the hi half, 4 of the lo half of its K step
                    uint32_t hi[4], lo[4];
                    v3_split4(v3_lds4(src + 16u * c), v3_lds4(sbS + 16u * c), v3_lds4(sbB + 16u * c), hi, lo);
                    const uint32_t tc = ta + 16u * (c >> 1) + 4u * (c & 1);
                    tmem_st4(tc, hi[0], hi[1], hi[2], hi[3]);
                    tmem_st4(tc + 8u, lo[0], lo[1], lo[2], lo[3]);
                }
                tmem_st_wait();
                tc_fence_before();
                __syncwarp();
                if (lane == 0) {
                    mbar_arrive(barAFull + 8 * FI);
                    if (FI == V3_FB - 1) mbar_arrive(barRawEmpty + 8 * s);
                }
                if (FI == V3_FB - 1) cG++;
            };
            constexpr std::integral_constant<int, 0> F0{};
            constexpr std::integral_constant<int, 1> F1{};
            constexpr std::integral_constant<int, 2> F2{};
            constexpr std::integral_constant<int, 3> F3{};

            if (my_tiles > 0) { convert(F0); convert(F1); }
            int tiles_left = my_tiles;
            for (int tile = blockIdx.x; tile < p.ntiles; tile += gridDim.x) {
                tiles_left--;
                const int ul = tile * TC_ROWS + r;
                float W[MC][8], Wx[MC], base[MC];
#pragma unroll
                for (int k = 0; k < MC; k++) {
                    Wx[k] = -INFINITY; base[k] = 0.f;
#pragma unroll
                    for (int j = 0; j < 8; j++) W[k][j] = -INFINITY;
                }
                uint32_t bpo = (uint32_t)g * (uint32_t)Tpad * p.Bpad + (uint32_t)ul;
                uint32_t sb = 0;
                // recursion of frame t0 + I from accumulator stage I & 1 (phase (I >> 1) & 1: tiles start at a multiple of four
                // frames); GEN = first / last block of a tile (run-time frame tests), else straight-line
                auto recurse = [&](auto Ic, auto GENc, int t0) {
                    constexpr int I = decltype(Ic)::value;
                    constexpr bool GEN = decltype(GENc)::value;
                    mbar_wait(barAccFull + 8 * (I & 1), (I >> 1) & 1);
                    tc_fence_after();
                    const uint32_t tacc = acc0 + (uint32_t)(I & 1) * (uint32_t)ncols;
                    const int t = t0 + I;
                    if (!GEN) {
                        // accumulator columns of model k - 1 are in flight while model k is stepped
                        uint32_t ev[2][8];
                        tmem_ld8(tacc + 8u * (MC - 1), ev[(MC - 1) & 1]);
#pragma unroll
                        for (int k = MC - 1; k >= 0; k--) {
                            tmem_ld_wait();
                            if (k > 0) tmem_ld8(tacc + 8u * (k - 1), ev[(k - 1) & 1]);
                            v3_step(W[k], Wx[k], aex[k], ev[k & 1], sb);
                        }
                        tc_fence_before();
                        p.bp[bpo] = sb;
                        bpo += p.Bpad;
                        return;
                    }
                    uint32_t ev[MC][8];
#pragma unroll
                    for (int k = 0; k < MC; k++) tmem_ld8(tacc + 8u * k, ev[k]);
                    tmem_ld_wait();
                    tc_fence_before();
                    if (t < Tt) {
                        if (t == 0) {
#pragma unroll
                            for (int k = 0; k < MC; k++) W[k][0] = sTr[(mbeg + k) * TC_TRQ + 2].y + __uint_as_float(ev[k][0]);   // ln A[0,1] + E[0,1] + ln A[1,1]
                        } else if (t == 1) {
#pragma unroll
                            for (int k = MC - 1; k >= 0; k--) v3_step_entry(W[k], Wx[k], sTr[(mbeg + k) * TC_TRQ + 2].y, ev[k], sb);
                        } else {
#pragma unroll
                            for (int k = MC - 1; k >= 0; k--) v3_step(W[k], Wx[k], aex[k], ev[k], sb);
                        }
                        p.bp[bpo] = sb;
                    }
                    bpo += p.Bpad;
                };
                constexpr std::integral_constant<bool, false> LEAN{};
                constexpr std::integral_constant<bool, true> GENERIC{};
                for (int t0 = 0; t0 < Tpad; t0 += V3_FB) {
                    const bool first = t0 == 0, last = t0 + V3_FB >= Tpad;
                    if (!first && !last) {
                        recurse(F0, LEAN, t0); convert(F2);
                        recurse(F1, LEAN, t0); convert(F3);
                        recurse(F2, LEAN, t0); convert(F0);
                        recurse(F3, LEAN, t0); convert(F1);
                    } else {
                        const bool more = !last || tiles_left > 0;     // frames t0 + 4, t0 + 5 exist (this tile or the CTA's next one)
                        recurse(F0, GENERIC, t0); convert(F2);
                        recurse(F1, GENERIC, t0); convert(F3);
                        recurse(F2, GENERIC, t0); if (more) convert(F0);
                        recurse(F3, GENERIC, t0); if (more) convert(F1);
                    }
                    if ((t0 & 4) != 0) {
#pragma unroll
                        for (int k = 0; k < MC; k++) v3_renorm(W[k], Wx[k], base[k]);
                    }
                }
                if (ul < p.nu) {
#pragma unroll
                    for (int k = 0; k < MC; k++) {
                        const float4 cm = sTr[(mbeg + k) * TC_TRQ + 2];
                        const double sc = (Wx[k] > -INFINITY) ? ((double)Wx[k] + (double)base[k]) + ((double)cm.z + (double)cm.w) : -INFINITY;
                        p.scores[(size_t)ul * M + mbeg + k] = sc;
                    }
                }
            }
        };
        const int npr = p.npair[g], mcnt = p.nmod[g];
        if (npr == 2 && mcnt == 2) run(std::integral_constant<int, 2>{}, std::integral_constant<int, 2>{});
        else if (npr == 1 && mcnt == 3) run(std::integral_constant<int, 1>{}, std::integral_constant<int, 3>{});
        else if (npr == 2 && mcnt == 3) run(std::integral_constant<int, 2>{}, std::integral_constant<int, 3>{});
        else if (npr == 1 && mcnt == 2) run(std::integral_constant<int, 1>{}, std::integral_constant<int, 2>{});
        else __trap();      // the launcher only picks this kernel for the splits above
    }
    tc_fence_before();
    __syncthreads();
    if (warp == TC_WORKER_WARPS) tmem_dealloc(tmem_base, 512);
}

// ------------------------------------------------------------------------------------------------
// k_viterbi_v4: the same arithmetic with the two halves of a worker's frame -- feature conversion and recursion -- on SEPARATE
// warps, so that neither waits for the other's barriers and an SM sub-partition has 6 resident instruction streams instead of 4:
//   warps  0-7   conversion: thread = (row, half of the feature chunks); raw ring -> standardise / square / fp16 hi-lo ->
//                A-operand stage in TMEM (A_full); stages are handed back by tcgen05.commit (A_empty)
//   warps  8-23  recursion: thread = (row, model group); steps its models on the columns already in registers while the next
//                frame's columns are fetched behind each model (rolling fetch), then hands that stage back (acc_empty)
//   warp  24     MMA issuer: A_full + acc_empty -> 15 x tcgen05.mma -> commit to acc_full and A_empty
//   warp  25     TMA producer
// (the scheduler favours high warp ids: the conversions, which run stages ahead anyway, get the low ones.)
// Four A stages + two accumulator stages (512 TMEM columns) as in k_viterbi_v3, frames in blocks of four with static stage
// indices.  setmaxnreg moves registers from the conversion warps (56) to the recursion warps (80).
#define V4_REC_WARPS 16
#define V4_CONV_WARPS 8
#define V4_REC_WARP0 V4_CONV_WARPS
#define V4_MMA_WARP (V4_REC_WARPS + V4_CONV_WARPS)
#define V4_TMA_WARP (V4_MMA_WARP + 1)
#define V4_THREADS (32 * (V4_TMA_WARP + 1))
#define V4_TRACE_ROLES 5
#define V4_TRACE_FRAMES 256

struct V4Smem { uint32_t w, raw, tr, sb, bar, total; };
__host__ __device__ inline V4Smem v4_smem_layout(int M, int nck, int ncols, uint32_t rw) {
    V4Smem L;
    L.w = 0;
    L.raw = ((uint32_t)2 * (ncols / 8) * nck * 128 + 127u) & ~127u;
    L.tr = L.raw + 2u * V3_FB * TC_ROWS * rw;
    L.sb = L.tr + (uint32_t)M * TC_TRQ * 16;
    L.bar = (L.sb + (uint32_t)8 * nck * 4 + 15u) & ~15u;
    L.total = L.bar + 24 * 8 + 16;      // raw_full[2], raw_empty[2], A_full[4], A_empty[4], acc_full[2][2], acc_empty[2][2] (stage, column half)
    return L;
}

// waits for two barriers with one poll loop (a check of a completed barrier costs ~150 cycles: the two overlap)
__device__ __forceinline__ void mbar_wait2(uint32_t bar_a, uint32_t par_a, uint32_t bar_b, uint32_t par_b) {
    asm volatile(
        "{\n\t.reg .pred p, q;\n\t.reg .u32 n;\n\t"
        "mov.u32 n, 0;\n\t"
        "LAB_WAIT:\n\t"
        "mbarrier.try_wait.parity.shared::cta.b64 p, [%0], %1;\n\t"
        "mbarrier.try_wait.parity.shared::cta.b64 q, [%2], %3;\n\t"
        "and.pred p, p, q;\n\t"
        "@p bra DONE;\n\t"
        "add.u32 n, n, 1;\n\t"
        "setp.gt.u32 q, n, 64000000;\n\t"
        "@q trap;\n\t"
        "bra LAB_WAIT;\n\t"
        "DONE:\n\t}"
        ::"r"(bar_a), "r"(par_a), "r"(bar_b), "r"(par_b) : "memory");
}

// HALF: the partial round of a batch, TWO CTAs per tile.  Each issues the product of one column half (model groups 0-1 | 2-3,
// with that half's acc_full / acc_empty barriers) and deals the half's models to all four recursion warp groups (at most two
// models per thread, V3Params::h*); both convert the tile's features.
template <int NKS, bool TRACE = false, bool HALF = false>      // nck = 2 * NKS feature chunks
__global__ void __launch_bounds__(V4_THREADS, 1) k_viterbi_v4(const V3Params p, const __grid_constant__ CUtensorMap tmap) {
    extern __shared__ __align__(128) unsigned char smem[];
    constexpr int nck = 2 * NKS;
    const int ncols = p.ncols, M = p.M;
    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
    const uint32_t rw = p.rw, frame_bytes = TC_ROWS * rw, stage_bytes = V3_FB * frame_bytes;
    const V4Smem L = v4_smem_layout(M, nck, ncols, rw);
    const uint32_t w_plane = (uint32_t)(ncols / 8) * nck * 128;
    unsigned char *sW = smem + L.w;
    const uint32_t sRaw = smem_u32(smem + L.raw);
    const float4 *sTr = reinterpret_cast<const float4 *>(smem + L.tr);
    uint64_t *sBar = reinterpret_cast<uint64_t *>(smem + L.bar);
    uint32_t *sTmem = reinterpret_cast<uint32_t *>(sBar + 24);
    const uint32_t barRawFull = smem_u32(sBar), barRawEmpty = barRawFull + 16, barAFull = barRawFull + 32, barAEmpty = barRawFull + 64;
    const uint32_t barAccFull = barRawFull + 96, barAccEmpty = barRawFull + 128;      // + 16 * stage + 8 * half
    const int half = HALF ? (int)(blockIdx.x & 1u) : 0;

    {
        const uint4 *src = reinterpret_cast<const uint4 *>(p.wimg);
        uint4 *dst = reinterpret_cast<uint4 *>(sW);
        for (uint32_t i = tid; i < 2 * w_plane / 16; i += V4_THREADS) dst[i] = src[i];
        float4 *dtr = reinterpret_cast<float4 *>(smem + L.tr);
        for (int i = tid; i < M * TC_TRQ; i += V4_THREADS) dtr[i] = p.trp[i];
        float *dsb = reinterpret_cast<float *>(smem + L.sb);
        for (int i = tid; i < 8 * nck; i += V4_THREADS) dsb[i] = p.sb[i];
    }
    if (tid == 0) {
        for (int s = 0; s < 2; s++) { mbar_init(barRawFull + 8 * s, 1); mbar_init(barRawEmpty + 8 * s, V4_CONV_WARPS); }
        for (int s = 0; s < 4; s++) { mbar_init(barAFull + 8 * s, V4_CONV_WARPS); mbar_init(barAEmpty + 8 * s, 1); }
        for (int s = 0; s < 4; s++) { mbar_init(barAccFull + 8 * s, 1); mbar_init(barAccEmpty + 8 * s, HALF ? 4 * p.hroles[half] : V4_REC_WARPS); }
        fence_barrier_init();
    }
    constexpr uint32_t a_cols = 8u * nck;
    if (warp == V4_MMA_WARP) tmem_alloc(smem_u32(sTmem), 512);
    fence_proxy_async();
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    const uint32_t tmem_base = *sTmem;
    const uint32_t tmem_acc = tmem_base, tmem_a = tmem_base + 2u * ncols;
    const int Tt = p.Tt, Tpad = p.Tpad;
    const int cta = HALF ? (int)(blockIdx.x >> 1) : (int)blockIdx.x, ncta = HALF ? (int)(gridDim.x >> 1) : (int)gridDim.x;
    const int my_tiles = (p.ntiles - cta + ncta - 1) / ncta;
    const int nblk = my_tiles * (Tpad / V3_FB);          // four-frame blocks this CTA walks
    auto trace = [&](int role, int frame, int ev) {
        if (TRACE && blockIdx.x == 0 && lane == 0 && frame < V4_TRACE_FRAMES) p.trace[((size_t)role * V4_TRACE_FRAMES + frame) * 4 + ev] = clock64();
    };

    if (warp == V4_TMA_WARP) {
        // ===================== TMA producer =====================
        if (lane == 0) {
            tma_prefetch_desc(&tmap);
            uint32_t G = 0;
            for (int tile = cta; tile < p.ntiles; tile += ncta) {
                const int urow = p.u0 + tile * TC_ROWS;
                for (int t0 = 0; t0 < Tpad; t0 += V3_FB, G++) {
                    const uint32_t s = G & 1u, ph = (G >> 1) & 1u;
                    const uint32_t bar = barRawFull + 8 * s;
                    mbar_wait(barRawEmpty + 8 * s, ph ^ 1u);
                    trace(1, (int)G, 0);
                    mbar_arrive_tx(bar, stage_bytes);
                    const uint32_t dst = sRaw + s * stage_bytes;
#pragma unroll
                    for (int fi = 0; fi < V3_FB; fi++) tma_load_3d(dst + (uint32_t)fi * frame_bytes, &tmap, 0, t0 + fi, urow, bar);
                    trace(1, (int)G, 1);
                    if (TRACE && blockIdx.x == 0) { mbar_wait(bar, ph); trace(1, (int)G, 2); }
                }
            }
        }
    } else if (warp == V4_MMA_WARP) {
        // ===================== MMA issuer =====================
        const uint32_t idesc = (1u << 4) | ((uint32_t)(ncols >> 3) << 17) | ((uint32_t)(TC_ROWS >> 4) << 24);
        const uint32_t sW_hi = smem_u32(sW), sW_lo = sW_hi + w_plane;
        const uint32_t sboW = (uint32_t)nck * 128u;
        const uint64_t dW_hi = make_desc(sW_hi, 128, sboW), dW_lo = make_desc(sW_lo, 128, sboW);
        const uint32_t colA = (uint32_t)p.split_col;                                       // columns of model groups 0-1
        const uint32_t idescA = (1u << 4) | ((colA >> 3) << 17) | ((uint32_t)(TC_ROWS >> 4) << 24);
        const uint32_t idescB = (1u << 4) | ((((uint32_t)ncols - colA) >> 3) << 17) | ((uint32_t)(TC_ROWS >> 4) << 24);
        const uint64_t wofs = (uint64_t)(((colA >> 3) * sboW) >> 4);                           // descriptor address units of 16 bytes
        uint32_t aph = 0;
        for (int b = 0; b < nblk; b++, aph ^= 1u) {
#pragma unroll
            for (int i = 0; i < V3_FB; i++) {
                trace(0, 4 * b + i, 0);
                if (TRACE && blockIdx.x == 0 && lane == 0 && 4 * b + i < V4_TRACE_FRAMES) {      // wall clock (ns) beside the cycle stamp: the SM frequency under this kernel
                    unsigned long long ns;
                    asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(ns));
                    p.trace[((size_t)0 * V4_TRACE_FRAMES + 4 * b + i) * 4 + 1] = (long long)ns;
                }
                mbar_wait2(barAFull + 8 * i, aph, barAccEmpty + 16 * (i & 1) + 8 * half, ((i >> 1) & 1) ^ 1);
                trace(0, 4 * b + i, 2);
                tc_fence_after();
                const uint32_t d_tmem = tmem_acc + (uint32_t)(i & 1) * (uint32_t)ncols;
                const uint32_t a_hi = tmem_a + (uint32_t)i * a_cols, a_lo = a_hi + 8u;
                if (!HALF) {
                    if (elect_one()) {
                        // the two correction products first: the large hi * W_hi partial sums see the fewest truncating steps
#pragma unroll
                        for (int ks = 0; ks < NKS; ks++) umma_f16_ts(d_tmem, a_lo + ks * 16, dW_hi + (uint64_t)(16 * ks), idesc, ks > 0);
#pragma unroll
                        for (int ks = 0; ks < NKS; ks++) umma_f16_ts(d_tmem, a_hi + ks * 16, dW_lo + (uint64_t)(16 * ks), idesc, 1);
#pragma unroll
                        for (int ks = 0; ks < NKS; ks++) umma_f16_ts(d_tmem, a_hi + ks * 16, dW_hi + (uint64_t)(16 * ks), idesc, 1);
                        umma_commit(barAccFull + 16 * (i & 1));
                        umma_commit(barAEmpty + 8 * i);
                    }
                } else if (elect_one()) {
                    const uint32_t dh = d_tmem + (half ? colA : 0u);
                    const uint32_t idh = half ? idescB : idescA;
                    const uint64_t wh = dW_hi + (half ? wofs : 0ull), wl = dW_lo + (half ? wofs : 0ull);
#pragma unroll
                    for (int ks = 0; ks < NKS; ks++) umma_f16_ts(dh, a_lo + ks * 16, wh + (uint64_t)(16 * ks), idh, ks > 0);
#pragma unroll
                    for (int ks = 0; ks < NKS; ks++) umma_f16_ts(dh, a_hi + ks * 16, wl + (uint64_t)(16 * ks), idh, 1);
#pragma unroll
                    for (int ks = 0; ks < NKS; ks++) umma_f16_ts(dh, a_hi + ks * 16, wh + (uint64_t)(16 * ks), idh, 1);
                    umma_commit(barAccFull + 16 * (i & 1) + 8 * half);
                    umma_commit(barAEmpty + 8 * i);
                }
                __syncwarp();
                trace(0, 4 * b + i, 3);
            }
        }
    } else if (warp < V4_REC_WARP0) {
        // ===================== conversion: thread = (row, chunk half) =====================
        asm volatile("setmaxnreg.dec.sync.aligned.u32 56;");          // registers move from the conversion to the recursion warps
        const int cw = warp, q = cw & 3, h = cw >> 2, r = q * 32 + lane;
        const uint32_t c0 = (uint32_t)(h * NKS);                       // first chunk of this half
        // per-thread addresses pinned in registers: left alone, the compiler re-derives them from %tid and the parameter block
        // in every frame (special-register and indexed constant loads in front of the dependent TMEM / shared accesses)
        const uint32_t raw0 = pin_reg(sRaw + (uint32_t)r * rw + 16u * c0);
        const uint32_t ta0 = pin_reg(tmem_a + ((uint32_t)(q * 32) << 16));
        const uint32_t sbS = pin_reg(smem_u32(smem + L.sb) + 16u * c0), sbB = sbS + 16u * nck;
        const uint32_t lane0 = pin_reg(lane == 0 ? 1u : 0u);
        const uint32_t sbytes = pin_reg(stage_bytes), fbytes = pin_reg(frame_bytes);
        uint32_t G = 0, eph = 1;                                       // ring stage counter; A_empty phase to wait for
        for (int b = 0; b < nblk; b++, G++, eph ^= 1u) {
            const uint32_t s = G & 1u;
            if (cw == 0) trace(2, 4 * b, 0);
            mbar_wait(barRawFull + 8 * s, (G >> 1) & 1u);
#pragma unroll
            for (int fi = 0; fi < V3_FB; fi++) {
                if (cw == 0) trace(2, 4 * b + fi, fi == 0 ? 1 : 0);
                const uint32_t src = raw0 + s * sbytes + (uint32_t)fi * fbytes;
                float4 x[NKS];
#pragma unroll
                for (int c = 0; c < NKS; c++) x[c] = v3_lds4(src + 16u * c);
                mbar_wait(barAEmpty + 8 * fi, eph);
                if (cw == 0) trace(2, 4 * b + fi, 2);
                tc_fence_after();
                const uint32_t ta = ta0 + (uint32_t)fi * a_cols;
#pragma unroll
                for (int c = 0; c < NKS; c++) {
                    uint32_t hi[4], lo[4];
                    v3_split4(x[c], v3_lds4(sbS + 16u * c), v3_lds4(sbB + 16u * c), hi, lo);
                    const uint32_t cg = c0 + (uint32_t)c;
                    const uint32_t tc = ta + 16u * (cg >> 1) + 4u * (cg & 1u);      // chunk cg: 4 columns of the hi half, 4 of the lo half of its K step
                    tmem_st4(tc, hi[0], hi[1], hi[2], hi[3]);
                    tmem_st4(tc + 8u, lo[0], lo[1], lo[2], lo[3]);
                }
                tmem_st_wait();
                tc_fence_before();
                __syncwarp();
                if (lane0) {
                    mbar_arrive(barAFull + 8 * fi);
                    if (fi == V3_FB - 1) mbar_arrive(barRawEmpty + 8 * s);
                }
                if (cw == 0) trace(2, 4 * b + fi, 3);
            }
        }
    } else {
        // ===================== recursion: thread = (row, model group) =====================
        asm volatile("setmaxnreg.inc.sync.aligned.u32 80;");
        const int rwp = warp - V4_REC_WARP0, q = rwp & 3, g = rwp >> 2, r = q * 32 + lane;
        const int mbeg = HALF ? p.hmod0[half][g] : p.mod0[g];
        const uint32_t acc0 = pin_reg(tmem_acc + ((uint32_t)(q * 32) << 16) + (uint32_t)mbeg * 8u);
        const uint32_t acc1 = pin_reg(acc0 + (uint32_t)ncols);
        const uint32_t lane0 = pin_reg(lane == 0 ? 1u : 0u);
        const uint32_t hb = 8u * (uint32_t)half;            // this CTA's column half
        const uint32_t bFull = pin_reg(barAccFull + hb), bEmpty = pin_reg(barAccEmpty + hb);
        const uint32_t bstride = pin_reg(p.Bpad);
        uint32_t *const bpp = p.bp;
        auto run = [&](auto MCc) {
            constexpr int MC = decltype(MCc)::value;
            float aex[MC];
#pragma unroll
            for (int k = 0; k < MC; k++) aex[k] = sTr[(mbeg + k) * TC_TRQ + 2].x;
            // Rolling accumulator fetch: ev[k] holds model k's columns of the frame about to be stepped; as soon as a model has
            // consumed its eight values, the same registers receive that model's columns of the NEXT frame, so the TMEM load
            // latency, the wait and the hand-back of the stage (acc_empty) run under the arithmetic of the current frame.
            uint32_t ev[MC][8];
            if (my_tiles > 0) {
                mbar_wait(bFull, 0);
                tc_fence_after();
#pragma unroll
                for (int k = 0; k < MC; k++) tmem_ld8(acc0 + 8u * k, ev[k]);
                tmem_ld_wait();
                tc_fence_before();
                __syncwarp();
                if (lane0) mbar_arrive(bEmpty);
            }
            int tiles_left = my_tiles;
            for (int tile = cta; tile < p.ntiles; tile += ncta) {
                tiles_left--;
                const int ul = tile * TC_ROWS + r;
                float W[MC][8], Wx[MC], base[MC];
#pragma unroll
                for (int k = 0; k < MC; k++) {
                    Wx[k] = -INFINITY; base[k] = 0.f;
#pragma unroll
                    for (int j = 0; j < 8; j++) W[k][j] = -INFINITY;
                }
                // decision words: plane = the model group of the one-CTA layout; a column-half CTA's thread owns one or two of
                // the word's bytes (same layout, narrower stores), so the arg-max / back-trace kernel does not change
                uint32_t bpo = (uint32_t)(HALF ? p.hplane[half][g] : g) * (uint32_t)Tpad * p.Bpad + (uint32_t)ul;
                const uint32_t bsh = HALF ? (uint32_t)p.hshift[half][g] : 0u;
                auto store_bp = [&](uint32_t v) {
                    if (HALF && MC < 3) {
                        uint8_t *b = reinterpret_cast<uint8_t *>(bpp + bpo) + bsh;
                        if (MC == 2) *reinterpret_cast<uint16_t *>(b) = (uint16_t)v;
                        else *b = (uint8_t)v;
                    } else
                        bpp[bpo] = v;
                };
                uint32_t sb = 0;
                const int trole = rwp == 0 ? 3 : rwp == 15 ? 4 : -1;
                const int fbase = ((tile - cta) / ncta) * Tpad;
                // frame t0 + I: its columns are in ev; frame t0 + I + 1 (stage (I + 1) & 1, phase ((I + 1) >> 1) & 1 -- tiles start at a
                // multiple of four frames) is fetched behind it unless this is the CTA's last frame
                auto recurse = [&](auto Ic, auto GENc, int t0, bool more) {
                    constexpr int I = decltype(Ic)::value;
                    constexpr bool GEN = decltype(GENc)::value;
                    constexpr int NS = (I + 1) & 1;
                    const uint32_t nacc = NS ? acc1 : acc0;
                    if (TRACE && trole >= 0) trace(trole, fbase + t0 + I, 0);
                    if (!GEN || more) {
                        mbar_wait(bFull + 16 * NS, ((I + 1) >> 1) & 1);
                        tc_fence_after();
                    }
                    if (TRACE && trole >= 0) trace(trole, fbase + t0 + I, 1);
                    const int t = t0 + I;
                    if (!GEN) {
                        // one sign-bit chain per model (independent instruction streams), merged bytewise
                        uint32_t sbk[MC];
#pragma unroll
                        for (int k = 0; k < MC; k++) {
                            sbk[k] = 0;
                            v3_step(W[k], Wx[k], aex[k], ev[k], sbk[k]);
                            tmem_ld8(nacc + 8u * k, ev[k]);
                        }
                        sb = sbk[0];
                        if (MC == 2) sb = __byte_perm(sbk[0], sbk[1], 0x3340);
                        if (MC == 3) sb = __byte_perm(__byte_perm(sbk[0], sbk[1], 0x3340), sbk[2], 0x3410);
                        store_bp(sb);
                    } else {
                        if (t < Tt) {
                            if (t == 0) {
#pragma unroll
                                for (int k = 0; k < MC; k++) W[k][0] = sTr[(mbeg + k) * TC_TRQ + 2].y + __uint_as_float(ev[k][0]);   // ln A[0,1] + E[0,1] + ln A[1,1]
                            } else if (t == 1) {
#pragma unroll
                                for (int k = MC - 1; k >= 0; k--) v3_step_entry(W[k], Wx[k], sTr[(mbeg + k) * TC_TRQ + 2].y, ev[k], sb);
                            } else {
#pragma unroll
                                for (int k = MC - 1; k >= 0; k--) v3_step(W[k], Wx[k], aex[k], ev[k], sb);
                            }
                            store_bp(sb);
                        }
                        if (more) {
#pragma unroll
                            for (int k = 0; k < MC; k++) tmem_ld8(nacc + 8u * k, ev[k]);
                        }
                    }
                    bpo += bstride;
                    if (TRACE && trole >= 0) trace(trole, fbase + t0 + I, 2);
                    if (!GEN || more) {
                        tmem_ld_wait();
                        tc_fence_before();
                        __syncwarp();
                        if (lane0) mbar_arrive(bEmpty + 16 * NS);            // the next frame's columns are in registers: its stage is free
                    }
                    if (TRACE && trole >= 0) trace(trole, fbase + t0 + I, 3);
                };
                constexpr std::integral_constant<bool, false> LEAN{};
                constexpr std::integral_constant<bool, true> GENERIC{};
                constexpr std::integral_constant<int, 0> F0{};
                constexpr std::integral_constant<int, 1> F1{};
                constexpr std::integral_constant<int, 2> F2{};
                constexpr std::integral_constant<int, 3> F3{};
                for (int t0 = 0; t0 < Tpad; t0 += V3_FB) {
                    // straight-line block unless it holds frames 0 / 1, frames past the utterance, or the CTA's very last frame
                    if (t0 != 0 && (t0 + V3_FB < Tpad || (Tt == Tpad && tiles_left > 0))) {
                        recurse(F0, LEAN, t0, true); recurse(F1, LEAN, t0, true); recurse(F2, LEAN, t0, true); recurse(F3, LEAN, t0, true);
                    } else {
                        const bool more = t0 + V3_FB < Tpad || tiles_left > 0;      // a frame follows the block's last one
                        recurse(F0, GENERIC, t0, true); recurse(F1, GENERIC, t0, true); recurse(F2, GENERIC, t0, true); recurse(F3, GENERIC, t0, more);
                    }
                    if ((t0 & 12) == 12) {      // every 16 frames: values drift by ~ -55 per frame, fp32 keeps 1e-4 absolute at 900
#pragma unroll
                        for (int k = 0; k < MC; k++) v3_renorm(W[k], Wx[k], base[k]);
                    }
                }
                if (ul < p.nu) {
#pragma unroll
                    for (int k = 0; k < MC; k++) {
                        const float4 cm = sTr[(mbeg + k) * TC_TRQ + 2];
                        const double sc = (Wx[k] > -INFINITY) ? ((double)Wx[k] + (double)base[k]) + ((double)cm.z + (double)cm.w) : -INFINITY;
                        p.scores[(size_t)ul * M + mbeg + k] = sc;
                    }
                }
            }
        };
        const int mcnt = HALF ? p.hnmod[half][g] : p.nmod[g];
        if (HALF && mcnt == 0) { }
        else if (mcnt == 3) run(std::integral_constant<int, 3>{});
        else if (mcnt == 2) run(std::integral_constant<int, 2>{});
        else if (mcnt == 1) run(std::integral_constant<int, 1>{});
        else __trap();
    }
    tc_fence_before();
    __syncthreads();
    if (warp == V4_MMA_WARP) tmem_dealloc(tmem_base, 512);
}

// ------------------------------------------------------------------------------------------------
// arg-max over models (strict >, first model wins: decoder.py:42-47) + back-trace of the winner from the packed words
struct V3Map { int grp[16], shift[16]; };
__device__ __forceinline__ uint32_t ldg_nc_u32(const void *p) {
    uint32_t v;
    asm volatile("ld.global.nc.u32 %0, [%1];" : "=r"(v) : "l"(p));
    return v;
}
__device__ __forceinline__ void hold8(uint32_t *v) {
    asm volatile("" : "+r"(v[0]), "+r"(v[1]), "+r"(v[2]), "+r"(v[3]), "+r"(v[4]), "+r"(v[5]), "+r"(v[6]), "+r"(v[7]));
}
__global__ void __launch_bounds__(128)
k_viterbi_finish_v3(const int64_t *__restrict__ offsets, int u0, int nu, int M, int Tt, int Tpad, const uint32_t *__restrict__ bp,
                    uint32_t Bpad, const V3Map map, const double *__restrict__ scores, int32_t *__restrict__ best_word,
                    double *__restrict__ best_score, double *__restrict__ scores_out, uint8_t *__restrict__ best_path, const SaprFlag flag) {
    constexpr int CH = 32;
    const int ul = blockIdx.x * blockDim.x + threadIdx.x;
    const bool live = ul < nu;
    const int u = u0 + ul;
    double bs = -INFINITY;
    int bslot = -1;
    int64_t off = 0;
    if (live) {
        off = offsets[u];
        double second = -INFINITY;
        for (int s = 0; s < M; s++) {
            const double sc = scores[(size_t)ul * M + s];
            if (scores_out) scores_out[(size_t)u * M + s] = sc;
            if (sc > bs) { second = bs; bs = sc; bslot = s; }
            else if (sc > second) second = sc;
        }
        if (best_word) best_word[u] = bslot;
        if (best_score) best_score[u] = bs;
        sapr_flag_word(flag, u, bs, second);      // word near-tie in fp32: re-decoded in float64 by the launcher
    }
    if (!best_path) return;
    const int wslot = bslot < 0 ? 0 : bslot;
    const bool reachable = live && bslot >= 0;
    const uint32_t *bpp = bp + (size_t)map.grp[wslot] * Tpad * Bpad + (live ? ul : 0);      // loads are unconditional: idle lanes read column 0
    const int sh = map.shift[wslot];
    const int Te = live ? Tt : 0;
    // every utterance has Tt frames: lane = utterance, 32 frames per chunk.  The chunk's words are fetched with 32 independent
    // loads (pointer walks by a fixed stride) one chunk AHEAD of the chunk being traced, the traced states are packed four per
    // register and written with 8-byte stores when the utterance's path is 8-byte aligned (byte stores otherwise).  The winner's
    // model group differs from lane to lane, so a lane's 4-byte word costs a 32-byte sector (3.2 KB per utterance).
    // The trace itself is the latency of a small launch (one dependent chain of Tt steps per thread), so a step is three
    // dependent instructions and no branch: frame t's decisions become a "stay" mask indexed by the CURRENT state c
    // (bit 0: the entry state stays; bit 1: state 1 stays except over the entry arc at t == 1, which sits in the exit slot;
    // bits 2..9: the kernel's sign bits, set = stayed), and c <- c - 1 + ((mask >> c) & 1).
    const uint8_t *bpb = reinterpret_cast<const uint8_t *>(bpp);
    const size_t fstride = (size_t)Bpad * sizeof(uint32_t);
    uint8_t *out = best_path + off;
    const bool al8 = ((reinterpret_cast<uintptr_t>(out) & 7) == 0);
    // volatile loads + an empty asm that "modifies" the 32 values: all loads of a chunk are issued before the first one is
    // consumed (left alone, the compiler interleaves load and use and the chunk costs ~25 memory round trips instead of one)
    const int tlast = Tpad - 1;
    auto fetch = [&](int t0, uint32_t (&mask)[CH]) {
#pragma unroll
        for (int j = 0; j < CH; j++) mask[j] = ldg_nc_u32(bpb + (size_t)min(t0 + j, tlast) * fstride);
#pragma unroll
        for (int j = 0; j < CH; j += 8) hold8(&mask[j]);
#pragma unroll
        for (int j = 0; j < CH; j++) {
            const int t = t0 + j;
            const uint32_t b = (reachable && t >= 1 && t < Te) ? (mask[j] >> sh) & 0xFFu : 0xFFu;
            mask[j] = (b << 2) | (t == 1 ? ((b >> 6) & 2u) ^ 2u : 2u) | 1u;
        }
    };
    uint32_t cur = 9;
    auto walk = [&](int t0, const uint32_t (&mask)[CH]) {
        uint32_t pk[CH / 4];
#pragma unroll
        for (int k = 0; k < CH / 4; k++) pk[k] = 0;
#pragma unroll
        for (int j = CH - 1; j >= 0; j--) {
            // an unreachable winner (every score -inf) keeps the exit state in its last frame and 0 before (custom_hmm.py:470)
            const uint32_t rec = reachable ? cur : (t0 + j == Te - 1 ? 9u : 0u);
            pk[j >> 2] |= rec << (8 * (j & 3));
            cur = cur - 1u + ((mask[j] >> cur) & 1u);
        }
        if (live) {
            const int nb = min(CH, Te - t0);                                      // bytes of this chunk
            if (al8 && (t0 & 7) == 0 && nb == CH) {
#pragma unroll
                for (int k = 0; k < CH / 8; k++) *reinterpret_cast<uint2 *>(out + t0 + 8 * k) = make_uint2(pk[2 * k], pk[2 * k + 1]);
            } else {
#pragma unroll
                for (int j = 0; j < CH; j++)
                    if (j < nb) out[t0 + j] = (uint8_t)(pk[j >> 2] >> (8 * (j & 3)));
            }
        }
    };
    uint32_t ma[CH];
    for (int t0 = (Tt - 1) / CH * CH; t0 >= 0; t0 -= CH) {
        fetch(t0, ma);
        walk(t0, ma);
    }
}

// ------------------------------------------------------------------------------------------------
// returns SAPR_OK and sets *taken when the batch / model set has the shape this kernel is cut for
int sapr_viterbi_v3_launch(sapr_ctx *ctx, sapr_models *m, const float *X, int ldx, const int64_t *offsets, int B, int max_T,
                           int first_frames, int32_t *best_word, double *best_score, double *scores, uint8_t *best_path,
                           bool *taken) {
    *taken = false;
    int nck, ncols;
    sapr_tc_image_bytes(m, &nck, &ncols);
    const int M = m->M;
    const int Tt = (first_frames > 0 && first_frames < max_T) ? first_frames : max_T;
    if (Tt < 2 || ((uintptr_t)X & 15u) || nck % 2) return SAPR_OK;
    V3Params prm;
    const bool use_v4 = (nck == 10 || nck == 4) && M >= TC_GROUPS;
    const int npairs = nck / 2;
    if (use_v4) {      // models over the four recursion groups, as evenly as they go
        int ma = 0;
        for (int g = 0; g < TC_GROUPS; g++) {
            prm.mod0[g] = ma; prm.nmod[g] = M / TC_GROUPS + (g < M % TC_GROUPS ? 1 : 0); ma += prm.nmod[g];
            prm.pair0[g] = 0; prm.npair[g] = 0;
        }
    } else {
    // work split over the four worker groups: chunk pairs to the low groups, models to the high groups
    if (npairs > 2 * TC_GROUPS || npairs < TC_GROUPS) return SAPR_OK;
    {
        int pc[TC_GROUPS], mcn[TC_GROUPS];
        const int MG = (M + TC_GROUPS - 1) / TC_GROUPS;
        for (int g = 0; g < TC_GROUPS; g++) { pc[g] = npairs / TC_GROUPS + (g < npairs % TC_GROUPS ? 1 : 0); mcn[g] = 0; }
        for (int mi = 0; mi < M; mi++) {
            int best = TC_GROUPS - 1;
            for (int g = TC_GROUPS - 1; g >= 0; g--)
                if (mcn[g] < MG && (mcn[best] >= MG || pc[g] + mcn[g] < pc[best] + mcn[best])) best = g;
            mcn[best]++;
        }
        int pa = 0, ma = 0;
        for (int g = 0; g < TC_GROUPS; g++) {
            prm.pair0[g] = pa; prm.npair[g] = pc[g]; pa += pc[g];
            prm.mod0[g] = ma; prm.nmod[g] = mcn[g]; ma += mcn[g];
            const bool ok = (pc[g] == 2 && mcn[g] == 2) || (pc[g] == 1 && mcn[g] == 3) || (pc[g] == 2 && mcn[g] == 3) || (pc[g] == 1 && mcn[g] == 2);
            if (!ok) return SAPR_OK;
        }
    }
    }
    const uint32_t rw = (uint32_t)(nck + 1) * 16u;
    V3Smem L = v3_smem_layout(M, nck, ncols, rw);
    if (use_v4) L.total = v4_smem_layout(M, nck, ncols, rw).total;
    if (L.total > 227 * 1024 || 2 * ncols + 4 * 8 * nck > 512) return SAPR_OK;
    const int Tpad = (Tt + V3_FB - 1) / V3_FB * V3_FB;
    const int64_t per_utt = (int64_t)TC_GROUPS * Tpad * sizeof(uint32_t);
    int chunk = (int)std::min<int64_t>(B, std::max<int64_t>(TC_ROWS, ((int64_t)1024 << 20) / per_utt));
    if (const char *ce = getenv("SAPR_V_CHUNK")) chunk = std::max(1, std::min(chunk, atoi(ce)));     // tests: force the multi-chunk path
    chunk = (chunk + TC_ROWS - 1) / TC_ROWS * TC_ROWS;
    int rc;
    if ((rc = sapr_ws_reserve(ctx, 0, (size_t)per_utt * chunk))) return rc;
    if ((rc = sapr_ws_reserve(ctx, 1, (size_t)chunk * M * sizeof(double)))) return rc;
    CUtensorMap tmap;
    {
        const uint64_t dim[3] = {(uint64_t)ldx, (uint64_t)max_T, (uint64_t)B};
        const uint64_t str[2] = {(uint64_t)ldx * 4u, (uint64_t)max_T * ldx * 4u};
        const uint32_t box[3] = {rw / 4u, 1u, (uint32_t)TC_ROWS};
        if ((rc = sapr_tmap_f32_3d(ctx, &tmap, X, dim, str, box))) return rc;
    }
    auto al256 = [](size_t x) { return (x + 255) / 256 * 256; };
    const size_t w = al256((size_t)2 * (ncols / 8) * nck * 64 * sizeof(__half));
    const size_t gsz = al256((size_t)8 * nck * sizeof(float));
    V3Map map;
    for (int g = 0; g < TC_GROUPS; g++)
        for (int k = 0; k < prm.nmod[g]; k++) { map.grp[prm.mod0[g] + k] = g; map.shift[prm.mod0[g] + k] = 8 * k; }
    auto kern = use_v4 ? (nck == 10 ? k_viterbi_v4<5> : k_viterbi_v4<2>)
                       : (nck == 10) ? k_viterbi_v3<5> : (nck == 4) ? k_viterbi_v3<2> : k_viterbi_v3<0>;
    const int nthreads = use_v4 ? V4_THREADS : V3_THREADS;
    // column halves for the partial round: model groups 0-1 | 2-3 split the accumulator at a multiple of 16 columns
    prm.split_col = 8 * prm.mod0[2];
    const bool can_half = use_v4 && prm.split_col >= 16 && prm.split_col % 16 == 0 && ncols - prm.split_col >= 16 && (ncols - prm.split_col) % 16 == 0;
    auto kern_half = !can_half ? nullptr : nck == 10 ? k_viterbi_v4<5, false, true> : k_viterbi_v4<2, false, true>;
    if (kern_half) SAPR_CUDA(ctx, cudaFuncSetAttribute(kern_half, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)L.total));
    if (can_half) {
        // a half's two model groups (1-3 models each) are dealt to the four recursion warp groups of its CTA: 3 -> 2 + 1, 2 -> 1 + 1,
        // 1 -> 1 + idle; a warp group keeps the bytes its models have in the group's decision word
        for (int h = 0; h < 2; h++) {
            prm.hroles[h] = 0;
            for (int k = 0; k < 2; k++) {
                const int g = 2 * h + k, n = prm.nmod[g], first = n == 3 ? 2 : n >= 1 ? 1 : 0;
                const int cnt[2] = {first, n - first};
                for (int r = 0; r < 2; r++) {
                    const int role = 2 * k + r;
                    prm.hmod0[h][role] = prm.mod0[g] + (r ? first : 0);
                    prm.hnmod[h][role] = cnt[r];
                    prm.hplane[h][role] = g;
                    prm.hshift[h][role] = r ? first : 0;
                    prm.hroles[h] += cnt[r] > 0;
                }
            }
        }
    }
    SAPR_CUDA(ctx, cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)L.total));
    const char *ex_env = getenv("SAPR_EXACT_WORDS");
    const bool exact = !ex_env || ex_env[0] != '0';
    SaprFlag flag;
    ctx->flag_maxT = max_T;
    for (int u0 = 0; u0 < B; u0 += chunk) {
        const int nu = std::min(chunk, B - u0);
        if (exact && (rc = sapr_flag_setup(ctx, &flag, u0 == 0))) return rc;
        prm.u0 = u0; prm.nu = nu; prm.M = M; prm.nck = nck; prm.ncols = ncols; prm.Tt = Tt; prm.Tpad = Tpad;
        prm.ntiles = (nu + TC_ROWS - 1) / TC_ROWS;
        prm.wimg = (const __half *)m->tc_image;
        prm.sb = (const float *)((const char *)m->tc_image + w);
        prm.trp = (const float4 *)((const char *)m->tc_image + w + gsz);
        prm.bp = (uint32_t *)ctx->ws[0]; prm.Bpad = (uint32_t)chunk; prm.scores = (double *)ctx->ws[1]; prm.rw = rw;
        prm.trace = nullptr;
        const char *trace_path = getenv("SAPR_V_TRACE");
        if (trace_path && use_v4 && nck == 10 && u0 == 0) {      // tuning aid: one traced launch, stamps to a text file
            const size_t nrec = (size_t)V4_TRACE_ROLES * V4_TRACE_FRAMES * 4;
            long long *dtr = nullptr;
            SAPR_CUDA(ctx, cudaMalloc(&dtr, nrec * sizeof(long long)));
            SAPR_CUDA(ctx, cudaMemsetAsync(dtr, 0, nrec * sizeof(long long), ctx->stream));
            prm.trace = dtr;
            auto tk = k_viterbi_v4<5, true>;
            SAPR_CUDA(ctx, cudaFuncSetAttribute(tk, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)L.total));
            tk<<<std::min(prm.ntiles, ctx->sm_count), nthreads, L.total, ctx->stream>>>(prm, tmap);
            std::vector<long long> h(nrec);
            cudaMemcpyAsync(h.data(), dtr, nrec * sizeof(long long), cudaMemcpyDeviceToHost, ctx->stream);
            cudaStreamSynchronize(ctx->stream);
            cudaFree(dtr);
            if (FILE *fp = fopen(trace_path, "w")) {
                for (int ro = 0; ro < V4_TRACE_ROLES; ro++)
                    for (int fr = 0; fr < V4_TRACE_FRAMES; fr++)
                        fprintf(fp, "%d %d %lld %lld %lld %lld\n", ro, fr, h[((size_t)ro * V4_TRACE_FRAMES + fr) * 4], h[((size_t)ro * V4_TRACE_FRAMES + fr) * 4 + 1],
                                h[((size_t)ro * V4_TRACE_FRAMES + fr) * 4 + 2], h[((size_t)ro * V4_TRACE_FRAMES + fr) * 4 + 3]);
                fclose(fp);
            }
            prm.trace = nullptr;
        }
        // A batch whose tile count is not a multiple of the SM count goes in two launches: the full rounds, then the partial
        // round.  The arg-max / back-trace of the first part runs on the auxiliary stream beside the partial round (which leaves
        // most SMs idle), so only the small second part's back-trace is left after the last main launch.  SAPR_V_TAIL=0: one launch.
        const int rounds = prm.ntiles / ctx->sm_count;
        const char *tl_env = getenv("SAPR_V_TAIL");
        const bool tail = rounds >= 1 && prm.ntiles % ctx->sm_count != 0 && best_path && (!tl_env || tl_env[0] != '0');
        const int nuA = tail ? rounds * ctx->sm_count * TC_ROWS : nu;      // utterances of the first launch
        uint32_t *const bp0 = prm.bp;
        double *const sc0 = prm.scores;
        {
            ProfScope ps(ctx, 0);
            prm.nu = nuA; prm.ntiles = (nuA + TC_ROWS - 1) / TC_ROWS;
            kern<<<std::min(prm.ntiles, ctx->sm_count), nthreads, L.total, ctx->stream>>>(prm, tmap);
            if (tail) {
                SAPR_CUDA(ctx, cudaEventRecord(ctx->ev[8], ctx->stream));
                prm.u0 = u0 + nuA; prm.nu = nu - nuA; prm.ntiles = (nu - nuA + TC_ROWS - 1) / TC_ROWS;
                prm.bp = bp0 + nuA; prm.scores = sc0 + (size_t)nuA * M;
                if (kern_half && 2 * prm.ntiles <= ctx->sm_count) {
                    // the partial round leaves most SMs idle: two CTAs per tile, each with the products and the recursion warps of
                    // one column half (model groups 0-1 | 2-3); both convert the tile's features
                    kern_half<<<2 * prm.ntiles, nthreads, L.total, ctx->stream>>>(prm, tmap);
                } else
                    kern<<<std::min(prm.ntiles, ctx->sm_count), nthreads, L.total, ctx->stream>>>(prm, tmap);
                prm.u0 = u0; prm.bp = bp0; prm.scores = sc0;
                ctx->launches++;
            }
        }
        SAPR_LAUNCH_CHECK(ctx);
        // arg-max / back-trace; with word exactness on, the same kernels list the word near-ties (best - second below the fp32
        // error bound) and ONE more launch re-decodes the listed utterances in float64 and overwrites their results
        const SaprFlag fl = exact ? flag : SaprFlag();
        if (tail) {
            SAPR_CUDA(ctx, cudaStreamWaitEvent(ctx->aux_stream, ctx->ev[8], 0));
            k_viterbi_finish_v3<<<(nuA + 127) / 128, 128, 0, ctx->aux_stream>>>(offsets, u0, nuA, M, Tt, Tpad, bp0, prm.Bpad, map, sc0, best_word,
                                                                                 best_score, scores, best_path, fl);
            SAPR_LAUNCH_CHECK(ctx);
            SAPR_CUDA(ctx, cudaEventRecord(ctx->ev[9], ctx->aux_stream));
        }
        const int uB = tail ? nuA : 0;      // utterances whose arg-max / back-trace is still to do
        {
            ProfScope ps(ctx, 1);
            k_viterbi_finish_v3<<<(nu - uB + 127) / 128, 128, 0, ctx->stream>>>(offsets, u0 + uB, nu - uB, M, Tt, Tpad, bp0 + uB, prm.Bpad, map,
                                                                               sc0 + (size_t)uB * M, best_word, best_score, scores, best_path, fl);
        }
        SAPR_LAUNCH_CHECK(ctx);
        if (tail) SAPR_CUDA(ctx, cudaStreamWaitEvent(ctx->stream, ctx->ev[9], 0));
        if (exact && (rc = sapr_viterbi_redo_flagged(ctx, m, X, ldx, offsets, first_frames, nu, flag, best_word, best_score, scores, best_path))) return rc;
    }
    *taken = true;
    return SAPR_OK;
}
