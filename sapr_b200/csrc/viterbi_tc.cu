// viterbi_tc.cu -- batched Viterbi with the diagonal-Gaussian emission on the 5th-gen tensor cores.
//
// Same contract as k_viterbi_fused (custom_hmm.py:462-514 x all models + decoder.py:42-47), different
// machine mapping.  The emission of one frame against all M*8 states is the dense contraction
//      E[r, n] = sum_k A[r, k] * W[n, k],   A[r, :] = [x', x'^2, 1] of utterance r at frame t,
// where x' = x * s + b is the feature standardised by a per-dimension centre/scale derived from the model
// set (keeps the expanded quadratic well conditioned) and W[n, :] = [2 mu' h', -h', c - sum mu'^2 h' + ln a_nn].
// One MMA tile = 128 utterances AT THE SAME FRAME INDEX: tcgen05.mma writes row r to TMEM lane r, and
// tcgen05.ld.32x32b hands the threads of row r exactly the emissions of THEIR utterance -- no transposition
// between the tensor-core tile and the register-resident left-to-right recursion.
//
// Data movement (per CTA = one SM, persistent over 128-utterance tiles):
//   HBM --cp.async.bulk (one copy per utterance: F consecutive frames, contiguous)--> shared-memory ring
//   shared --LDS.128 (row r, conflict-free padded stride)--> registers: standardise, square, fp16 hi/lo split
//   registers --tcgen05.st--> TMEM: the A operand lives in tensor memory (row r = lane r), never in shared memory
//   tcgen05.mma (A from TMEM, W from shared memory, fp32 accumulators in TMEM, double buffered)
//   TMEM --tcgen05.ld--> registers: max-product recursion, 1-bit back-pointers --> HBM scratch
//
// Precision: operands are fp16 hi/lo splits (x' = hi + lo to 22 bits, likewise W); the three products
// hi*Whi + lo*Whi + hi*Wlo are one K = 3*Kh accumulation chain in fp32 TMEM (Kh = 80 for D = 39).
//
// CTA = 20 warps: warps 0-15 are workers (thread = (row r, group g): converts a quarter of row r's next frame
// into the A operand, then runs the recursion for a quarter of the models), warp 16 issues the MMAs, warps 17-19
// issue the bulk copies.  Pipeline per frame f (stage = f & 1): workers write A[f+1] -> mbarrier A_full ->
// MMA warp issues 3*nck/2 tcgen05.mma into accumulator (f+1)&1 -> tcgen05.commit -> mbarrier acc_full ->
// workers tcgen05.ld, recursion, mbarrier acc_empty.  The MMAs of frame f+1 overlap the recursion of frame f.
#include "tc_common.cuh"

// ------------------------------------------------------------------------------------------------
// model-set preparation: standardisation (s, b) and the fp16 hi/lo weight image in its shared-memory layout
//   wimg[2][ncols/8][nck][8][8] halves (hi plane, lo plane); n = m*8 + state.  A chunk is 4 feature dims =
//   8 K elements ordered [x'_0 .. x'_3, x'^2_0 .. x'^2_3] (so a packed pair of one kind is one TMEM column).
//   Dim index D is the constant slot: x' = 1 there; its x' weight carries the constant and its (otherwise
//   unused) x'^2 weight the part of the constant the fp16 hi/lo pair of the first cannot represent.
//   sb[2][4*nck] float (scale s, offset b: x' = x*s + b);  trp[M][TC_TRQ = 8] float4 transition block:
//     [0] = (c1, c2, c3, c4)  [1] = (c5, c6, c7, cx)   c_j = ln A[j-1,j] - ln A[j-1,j-1] (advance minus stay),
//                                                      cx = ln A[N,exit] - ln A[N,N]
//     [2] = (ln A[exit,exit], ln A[0,1], kx_hi, kx_lo)   [3], [4] = stay_1 .. stay_8 = ln A[j,j] (folded into W's constant)
//     [5], [6] = (badv_1 .. badv_7, ln A[N,exit])   [7] = (ln A[0,1] - ln A[1,1], 0, 0, 0)   (E-step backward sweep)
__global__ void k_prepare_tc(int M, int S, int D, int nck, int ncols, const double *__restrict__ mean,
                             const double *__restrict__ var, const double *__restrict__ la, const double *__restrict__ lb,
                             __half *__restrict__ wimg, float *__restrict__ sb, float4 *__restrict__ trp) {
    extern __shared__ double s_gs[];   // [2][4*nck]: effective centre g, scale s
    const int N = S - 2, nd = 4 * nck;
    // one warp per feature dim, lanes stride over the (model, state) pairs, fixed-order shuffle tree; every CTA recomputes
    // these cheap constants and block 0 writes them (one thread per dim walking all states made this kernel 0.18 ms)
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31, nwarp = blockDim.x >> 5;
    auto wsum = [](double v) {
        for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
        return v;
    };
    for (int d = warp; d < nd; d += nwarp) {
        double g = 0.0, sc = 0.0;
        float sf = 0.f, bf = 0.f;
        if (d < D) {
            double sm = 0.0;
            for (int q = lane; q < M * N; q += 32) sm += mean[((size_t)(q / N) * S + (q % N) + 1) * D + d];
            g = wsum(sm) / (M * N);
            double v = 0.0;
            for (int q = lane; q < M * N; q += 32) {
                const size_t o = ((size_t)(q / N) * S + (q % N) + 1) * D + d;
                const double df = mean[o] - g;
                v += var[o] + df * df;
            }
            v = wsum(v) / (M * N);
            sc = (v > 0 && v < 1e300) ? 4.0 / sqrt(v) : 1.0;
            sf = (float)sc; bf = (float)(-g * sc);
            sc = (double)sf; g = -(double)bf / sc;   // the kernel standardises in fp32 with exactly (sf, bf)
        } else if (d == D) {
            sf = 0.f; bf = 1.f;                       // constant slot: x' = 1
        }
        if (lane == 0) {
            s_gs[d] = g; s_gs[nd + d] = sc;
            if (blockIdx.x == 0) { sb[d] = sf; sb[nd + d] = bf; }
        }
    }
    __syncthreads();
    const size_t plane = (size_t)(ncols / 8) * nck * 64;
    for (int idx = blockIdx.x * blockDim.x + threadIdx.x; idx < ncols * nd; idx += gridDim.x * blockDim.x) {
        const int n = idx / nd, d = idx % nd;
        const int m = n / 8, j = (n % 8) + 1;
        double wx = 0.0, wx2 = 0.0;
        if (m < M && j <= N) {
            const double *mu = mean + ((size_t)m * S + j) * D, *vr = var + ((size_t)m * S + j) * D;
            if (d < D) {
                const double g = s_gs[d], sc = s_gs[nd + d];
                const double hp = 0.5 / vr[d] / (sc * sc), mp = (mu[d] - g) * sc;
                wx = 2.0 * mp * hp; wx2 = -hp;
            } else if (d == D) {   // constant slot: A carries x' = 1 and x'^2 = 1 here
                double ld = 0.0, c2 = 0.0;
                for (int q = 0; q < D; q++) {
                    const double g = s_gs[q], sc = s_gs[nd + q];
                    const double hp = 0.5 / vr[q] / (sc * sc), mp = (mu[q] - g) * sc;
                    ld += log(vr[q]); c2 += mp * mp * hp;
                }
                const double cst = -0.5 * (D * SAPR_LOG2PI + ld) - c2 + la[(size_t)m * S + j];   // + ln A[j,j]
                const __half ch = __double2half(cst);
                const double r1 = cst - (double)__half2float(ch);
                const __half cl = __double2half(r1);
                wx = cst; wx2 = r1 - (double)__half2float(cl);   // third-order piece of the constant
            }
        }
        // element (n, k) of the image: group n/8, chunk d/4, row n%8, elem (d%4) for x', 4 + (d%4) for x'^2
        const size_t o = ((size_t)(n / 8) * nck + d / 4) * 64 + (size_t)(n % 8) * 8 + (d % 4);
        const __half hx = __double2half(wx), hx2 = __double2half(wx2);
        wimg[o] = hx; wimg[o + 4] = hx2;
        wimg[plane + o] = __double2half(wx - (double)__half2float(hx));
        wimg[plane + o + 4] = __double2half(wx2 - (double)__half2float(hx2));
    }
    for (int m = threadIdx.x; m < M && blockIdx.x == 0; m += blockDim.x) {
        const double *a = la + (size_t)m * S, *b = lb + (size_t)m * S;
        float v[20];
        for (int j = 1; j <= 7; j++) v[j - 1] = (j + 1 <= N) ? (float)(b[j] - a[j]) : -INFINITY;   // c_{j+1}: into state j+1
        v[7] = (float)(b[N] - a[N]);                                                              // cx (N == 8)
        v[8] = (float)a[S - 1]; v[9] = (float)b[0];
        {   // kx = sum of the advance-minus-stay constants along the chain incl. the exit arc (k_viterbi_v3 adds it to the final
            // score only), as a float pair; -inf when a forward arc has probability zero
            double kx = 0.0;
            for (int j = 1; j <= N; j++) kx += b[j] - a[j];
            v[10] = (float)kx;
            const double rest = kx - (double)v[10];
            v[11] = (rest == rest && rest - rest == 0.0) ? (float)rest : 0.f;
        }
        for (int j = 1; j <= 8; j++) v[11 + j] = (j <= N) ? (float)a[j] : 0.f;
        // E-step extras: badv_j = ln A[j,j+1] - ln A[j+1,j+1] (advance arc of state j on top of self[j+1]), ln A[N,exit],
        // ln A[0,1] - ln A[1,1]
        float w[12];
        for (int j = 1; j <= 7; j++) w[j - 1] = (j + 1 <= N) ? (float)(b[j] - a[j + 1]) : -INFINITY;
        w[7] = (float)b[N]; w[8] = (float)(b[0] - a[1]); w[9] = 0.f; w[10] = 0.f; w[11] = 0.f;
        for (int q = 0; q < 5; q++) trp[(size_t)m * TC_TRQ + q] = make_float4(v[4 * q], v[4 * q + 1], v[4 * q + 2], v[4 * q + 3]);
        for (int q = 0; q < 3; q++) trp[(size_t)m * TC_TRQ + 5 + q] = make_float4(w[4 * q], w[4 * q + 1], w[4 * q + 2], w[4 * q + 3]);
    }
}

// ------------------------------------------------------------------------------------------------
struct TcParams {
    const float *X; int ldx; const int64_t *offsets; int u0, nu, M, D, nck, ncols, first_frames;
    const __half *wimg; const float *sb; const float4 *trp;
    uint16_t *bp; int64_t Bpad; int maxT; double *scores; float *dbgE;   // dbgE: [sum_T][ncols] or null
    long long *trace;           // [TC_TRACE_ROLES][TC_TRACE_FRAMES][TC_TRACE_EVENTS] or null
    int Fshift, nst_shift;      // raw ring: 2^Fshift frames per stage, 2^nst_shift stages
    int mod0[TC_GROUPS], nmod[TC_GROUPS], pair0[TC_GROUPS], npair[TC_GROUPS];   // per worker group: models, chunk pairs
    uint32_t rstride;           // bytes per row per stage (F * row bytes + pad, an odd multiple of 16)
};

struct TcSmem {   // byte offsets into dynamic shared memory
    uint32_t w, raw, tr, sb, base, bar, total;
};
__host__ __device__ inline TcSmem tc_smem_layout(int M, int nck, int ncols, int nst, uint32_t rstride) {
    TcSmem L;
    L.w = 0;
    L.raw = (uint32_t)2 * (ncols / 8) * nck * 128;
    L.tr = L.raw + (uint32_t)nst * TC_ROWS * rstride;
    L.sb = L.tr + (uint32_t)M * TC_TRQ * 16;
    L.base = 0;
    L.bar = (L.sb + (uint32_t)8 * nck * 4 + 15u) & ~15u;
    L.total = L.bar + (2 * TC_MAX_STAGES + 6) * 8 + 16;
    return L;
}

// one frame of the max-product recursion of one model (custom_hmm.py:476-503) on U_j = V[t, j] + ln A[j, j]:
//   U_j <- max(U_{j-1} + c_j, U_j) + e'_j,  e'_j = E[t, j] + ln A[j, j] straight from the tensor core.
// Returns the 9 "advanced" bits (bit j-1 = state j took its predecessor j-1, bit 8 = the exit state took state N;
// the first candidate wins ties, :488-497).  EARLY = frames 1..8: entry state alive at t == 1, exit closed for t < N.
template <bool EARLY>
__device__ __forceinline__ uint32_t vit_step(float2 (&U)[4], float &Ux, const float4 c03, const float4 c47, const float a_exit,
                                             const float b0, const uint32_t (&ev)[8], int t) {
    const float2 P01 = add2(U[0], make_float2(c03.x, c03.y));   // advance candidates P_j = U_j + c_{j+1}
    const float2 P23 = add2(U[1], make_float2(c03.z, c03.w));
    const float2 P45 = add2(U[2], make_float2(c47.x, c47.y));
    const float2 P67 = add2(U[3], make_float2(c47.z, c47.w));   // P67.y feeds the exit state
    const float xs = Ux + a_exit;                               // exit self-loop
    uint32_t sb;                                                // "stayed" bits, exit first
    float nx;
    if (!EARLY || t >= 8) {                                     // exit opens at t >= N (custom_hmm.py:481-485)
        sb = __float_as_uint(P67.y - xs) >> 31;
        nx = fmaxf(P67.y, xs);
    } else {
        sb = 1; nx = -INFINITY;
    }
    sb = __funnelshift_l(__float_as_uint(P67.x - U[3].y), sb, 1);   // state 8
    sb = __funnelshift_l(__float_as_uint(P45.y - U[3].x), sb, 1);
    sb = __funnelshift_l(__float_as_uint(P45.x - U[2].y), sb, 1);
    sb = __funnelshift_l(__float_as_uint(P23.y - U[2].x), sb, 1);
    sb = __funnelshift_l(__float_as_uint(P23.x - U[1].y), sb, 1);
    sb = __funnelshift_l(__float_as_uint(P01.y - U[1].x), sb, 1);
    sb = __funnelshift_l(__float_as_uint(P01.x - U[0].y), sb, 1);   // state 2
    float n0;
    if (EARLY) {                                                    // state 1: the entry state is alive at t == 1 only
        const float ent = (t == 1) ? b0 : -INFINITY;
        sb = __funnelshift_l(__float_as_uint(ent - U[0].x), sb, 1);
        n0 = fmaxf(ent, U[0].x);
    } else {
        sb = (sb << 1) | 1u;
        n0 = U[0].x;
    }
    const float2 n01 = make_float2(n0, fmaxf(P01.x, U[0].y));
    const float2 n23 = make_float2(fmaxf(P01.y, U[1].x), fmaxf(P23.x, U[1].y));
    const float2 n45 = make_float2(fmaxf(P23.y, U[2].x), fmaxf(P45.x, U[2].y));
    const float2 n67 = make_float2(fmaxf(P45.y, U[3].x), fmaxf(P67.x, U[3].y));
    U[0] = add2(n01, make_float2(__uint_as_float(ev[0]), __uint_as_float(ev[1])));
    U[1] = add2(n23, make_float2(__uint_as_float(ev[2]), __uint_as_float(ev[3])));
    U[2] = add2(n45, make_float2(__uint_as_float(ev[4]), __uint_as_float(ev[5])));
    U[3] = add2(n67, make_float2(__uint_as_float(ev[6]), __uint_as_float(ev[7])));
    Ux = nx;
    return (~sb) & 0x1FFu;
}

// renormalise (fp32 stays at O(1) magnitudes).  The shift is the maximum rounded to an integer, so the running offset
// is an integer-valued float that accumulates exactly (|offset| < 2^24) -- no float64 in the hot loop.
__device__ __forceinline__ void vit_renorm(float2 (&U)[4], float &Ux, float &base) {
    float mx = fmaxf(fmaxf(U[0].x, U[0].y), Ux);
    mx = fmaxf(fmaxf(U[1].x, U[1].y), mx);
    mx = fmaxf(fmaxf(U[2].x, U[2].y), mx);
    mx = fmaxf(fmaxf(U[3].x, U[3].y), mx);
    mx = rintf(fminf(fmaxf(mx, -4194304.f), 4194304.f));      // -inf (nothing reachable yet) shifts by a finite amount
    const float2 m2 = make_float2(mx, mx);
    U[0] = sub2(U[0], m2);
    U[1] = sub2(U[1], m2);
    U[2] = sub2(U[2], m2);
    U[3] = sub2(U[3], m2);
    Ux -= mx;
    base += mx;
}

// TRACE: CTA 0 records clock64() at its pipeline events for the first TC_TRACE_FRAMES frames (tuning aid, SAPR_TC_TRACE=file)
#define TC_TRACE_FRAMES 96
#define TC_TRACE_EVENTS 6
#define TC_TRACE_ROLES 5
template <int MG, int NKS, bool DBG, bool TRACE = false>
__global__ void __launch_bounds__(TC_THREADS, 1) k_viterbi_tc(const TcParams p) {
    extern __shared__ __align__(128) unsigned char smem[];
    const int nck = p.nck, ncols = p.ncols, M = p.M;
    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
    const int F = 1 << p.Fshift, nst = 1 << p.nst_shift;
    const uint32_t rowbytes = (uint32_t)p.ldx * 4u, rstride = p.rstride, stage_bytes = TC_ROWS * rstride;
    const TcSmem L = tc_smem_layout(M, nck, ncols, nst, rstride);
    const uint32_t w_plane = (uint32_t)(ncols / 8) * nck * 128;            // bytes per W plane
    unsigned char *sW = smem + L.w;
    unsigned char *sRaw = smem + L.raw;
    const float4 *sTr = reinterpret_cast<const float4 *>(smem + L.tr);     // [M][5]
    const float4 *sS = reinterpret_cast<const float4 *>(smem + L.sb);      // [nck] scales, then [nck] offsets
    uint64_t *sBar = reinterpret_cast<uint64_t *>(smem + L.bar);
    uint32_t *sTmem = reinterpret_cast<uint32_t *>(sBar + 2 * TC_MAX_STAGES + 6);
    const uint32_t barRaw_full = smem_u32(sBar), barRaw_empty = barRaw_full + 8 * TC_MAX_STAGES;
    const uint32_t barA_full = barRaw_empty + 8 * TC_MAX_STAGES, barAcc_full = barA_full + 24;   // A_full[3], acc_full[2]

    {   // stage the constant images
        const uint4 *src = reinterpret_cast<const uint4 *>(p.wimg);
        uint4 *dst = reinterpret_cast<uint4 *>(sW);
        for (uint32_t i = tid; i < 2 * w_plane / 16; i += TC_THREADS) dst[i] = src[i];
        float4 *dtr = reinterpret_cast<float4 *>(smem + L.tr);
        for (int i = tid; i < M * TC_TRQ; i += TC_THREADS) dtr[i] = p.trp[i];
        float *dsb = reinterpret_cast<float *>(smem + L.sb);
        for (int i = tid; i < 8 * nck; i += TC_THREADS) dsb[i] = p.sb[i];
    }
    if (tid == 0) {
        for (int s = 0; s < nst; s++) {
            mbar_init(barRaw_full + 8 * s, 32 * TC_LOADERS);
            mbar_init(barRaw_empty + 8 * s, TC_WORKER_WARPS);
        }
        for (int s = 0; s < 3; s++) mbar_init(barA_full + 8 * s, TC_WORKER_WARPS);
        for (int s = 0; s < 2; s++) mbar_init(barAcc_full + 8 * s, 1);
        fence_barrier_init();
    }
    // TMEM: two accumulator buffers of ncols columns, three A-operand buffers of 8*nck columns (per K step: hi 8 | lo 8)
    const uint32_t a_cols = 8u * nck;
    uint32_t tcols = 32;
    while (tcols < 2u * ncols + 3u * a_cols) tcols <<= 1;
    if (warp == TC_WORKER_WARPS) tmem_alloc(smem_u32(sTmem), tcols);
    fence_proxy_async();            // W image written with generic stores, read by the tensor core
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    const uint32_t tmem_base = *sTmem;
    const uint32_t tmem_acc = tmem_base, tmem_a = tmem_base + 2u * ncols;

    const int ntiles = (p.nu + TC_ROWS - 1) / TC_ROWS;
    uint32_t f = 0;                 // running frame counter of this CTA (A / accumulator stage and phase)
    uint32_t sg = 0;                // running raw-stage counter of this CTA (ring slot and phase)

    // frames a row walks; every role derives the tile length (max over the 128 rows) with one warp reduction
    auto row_frames = [&](int ul, int64_t &off) -> int {
        off = 0;
        if (ul >= p.nu) return 0;
        off = p.offsets[p.u0 + ul];
        const int T = min((int)(p.offsets[p.u0 + ul + 1] - off), p.maxT);     // the scratch is sized by the caller's max_T: never walk past it
        return (p.first_frames > 0 && p.first_frames < T) ? p.first_frames : T;
    };
    auto tile_frames = [&](int tile) -> int {
        int Tt = 0;
        for (int r = lane; r < TC_ROWS; r += 32) {
            int64_t o;
            Tt = max(Tt, row_frames(tile * TC_ROWS + r, o));
        }
        for (int o = 16; o > 0; o >>= 1) Tt = max(Tt, __shfl_xor_sync(0xffffffffu, Tt, o));
        return Tt;
    };

    auto trace = [&](int role, uint32_t frame, int ev) {
        if (TRACE && blockIdx.x == 0 && lane == 0 && frame < TC_TRACE_FRAMES)
            p.trace[((size_t)role * TC_TRACE_FRAMES + frame) * TC_TRACE_EVENTS + ev] = clock64();
    };
    if (warp >= TC_WORKER_WARPS) {
    if (warp > TC_WORKER_WARPS) {
        // ===================== bulk-copy producers =====================
        // loader warp lw owns rows [lw*RPL, (lw+1)*RPL) of the tile; a lane issues at most two copies per stage
        constexpr int RPL = (TC_ROWS + TC_LOADERS - 1) / TC_LOADERS;
        const int lw = warp - TC_WORKER_WARPS - 1;
        const int rlo = lw * RPL, rhi = min(rlo + RPL, TC_ROWS);
        const int r0 = rlo + lane, r1 = rlo + lane + 32;
        const uint32_t dst0 = smem_u32(sRaw) + (uint32_t)r0 * rstride, dst1 = smem_u32(sRaw) + (uint32_t)r1 * rstride;
        const uint32_t stage_adv = (uint32_t)F * rowbytes;
        for (int tile = blockIdx.x; tile < ntiles; tile += gridDim.x) {
            const int Tt = tile_frames(tile);
            const int nsg = (Tt + F - 1) >> p.Fshift;
            int64_t o0 = 0, o1 = 0;
            const int Te0 = (r0 < rhi) ? row_frames(tile * TC_ROWS + r0, o0) : 0;
            const int Te1 = (r1 < rhi) ? row_frames(tile * TC_ROWS + r1, o1) : 0;
            const char *src0 = reinterpret_cast<const char *>(p.X + (size_t)o0 * p.ldx);
            const char *src1 = reinterpret_cast<const char *>(p.X + (size_t)o1 * p.ldx);
            int rem0 = Te0, rem1 = Te1;                      // frames not yet requested
            for (int k = 0; k < nsg; k++, sg++) {
                const uint32_t slot = sg & (uint32_t)(nst - 1), ph = (sg >> p.nst_shift) & 1u;
                const uint32_t nb0 = (uint32_t)min(max(rem0, 0), F) * rowbytes, nb1 = (uint32_t)min(max(rem1, 0), F) * rowbytes;
                const uint32_t bar = barRaw_full + 8 * slot;
                mbar_wait(barRaw_empty + 8 * slot, ph ^ 1u);
                if (lw == 0) trace(1, sg, 0);
                mbar_arrive_tx(bar, nb0 + nb1);
                if (nb0) bulk_g2s(dst0 + slot * stage_bytes, src0, nb0, bar);
                if (nb1) bulk_g2s(dst1 + slot * stage_bytes, src1, nb1, bar);
                src0 += stage_adv; src1 += stage_adv; rem0 -= F; rem1 -= F;
                if (lw == 0) trace(1, sg, 1);
                if (TRACE && lw == 0) { mbar_wait(bar, ph); trace(1, sg, 2); }
            }
        }
    } else if (warp == TC_WORKER_WARPS) {
        // ===================== MMA issuer =====================
        const uint32_t idesc = (1u << 4) | ((uint32_t)(ncols >> 3) << 17) | ((uint32_t)(TC_ROWS >> 4) << 24);
        const uint32_t sW_hi = smem_u32(sW), sW_lo = sW_hi + w_plane;
        const uint32_t sboW = (uint32_t)nck * 128u;
        const uint64_t dW_hi = make_desc(sW_hi, 128, sboW), dW_lo = make_desc(sW_lo, 128, sboW);
        const int nks = nck / 2;
        uint32_t a3 = 0, aph = 0;      // A-operand stage (frame counter mod 3) and its barrier phase
        for (int tile = blockIdx.x; tile < ntiles; tile += gridDim.x) {
            const int Tt = tile_frames(tile);
            for (int t = 0; t < Tt; t++, f++) {
                const uint32_t s = f & 1, ph = (f >> 1) & 1;
                trace(0, f, 0);
                mbar_wait(barA_full + 8 * a3, aph);
                trace(0, f, 1);
                tc_fence_after();
                if (elect_one()) {      // one elected lane, provably uniform operands: no per-lane issue loop around UTCHMMA
                    const uint32_t d_tmem = tmem_acc + s * (uint32_t)ncols;
                    const uint32_t a_hi = tmem_a + a3 * a_cols, a_lo = a_hi + 8u;   // K step ks: hi at +16 ks, lo at +16 ks + 8
                    // the two small correction products first: the tensor core truncates the fp32 accumulator on
                    // every step, so the large hi * W_hi partial sums should see as few steps as possible.
                    // One K = 16 step advances A by 8 TMEM columns and the W descriptor by 256 B (16 in its address field).
                    if (NKS > 0) {
#pragma unroll
                        for (int ks = 0; ks < NKS; ks++) umma_f16_ts(d_tmem, a_lo + ks * 16, dW_hi + (uint64_t)(16 * ks), idesc, ks > 0);
#pragma unroll
                        for (int ks = 0; ks < NKS; ks++) umma_f16_ts(d_tmem, a_hi + ks * 16, dW_lo + (uint64_t)(16 * ks), idesc, 1);
#pragma unroll
                        for (int ks = 0; ks < NKS; ks++) umma_f16_ts(d_tmem, a_hi + ks * 16, dW_hi + (uint64_t)(16 * ks), idesc, 1);
                    } else {
                        uint64_t dh = dW_hi, dl = dW_lo;
                        uint32_t a = a_lo;
                        for (int ks = 0; ks < nks; ks++, a += 16, dh += 16) umma_f16_ts(d_tmem, a, dh, idesc, ks > 0);   // lo * W_hi
                        a = a_hi;
                        for (int ks = 0; ks < nks; ks++, a += 16, dl += 16) umma_f16_ts(d_tmem, a, dl, idesc, 1);        // hi * W_lo
                        a = a_hi; dh = dW_hi;
                        for (int ks = 0; ks < nks; ks++, a += 16, dh += 16) umma_f16_ts(d_tmem, a, dh, idesc, 1);        // hi * W_hi
                    }
                    umma_commit(barAcc_full + 8 * s);
                }
                __syncwarp();
                if (++a3 == 3) { a3 = 0; aph ^= 1u; }
                trace(0, f, 2);
                if (TRACE) { mbar_wait(barAcc_full + 8 * s, ph); trace(0, f, 3); }
            }
        }
    }
    } else {
        // ===================== workers =====================
        const int q = warp & 3;                      // TMEM lane quadrant this warp may access
        const int g = warp >> 2;                     // group: which models / which feature chunk pairs
        const int r = q * 32 + lane;                 // row of the tile = TMEM lane
        const int mbeg = p.mod0[g], mcnt = p.nmod[g];                 // this thread's models
        const int pr0 = p.pair0[g], npr = p.npair[g];                 // this thread's chunk pairs (8 feature dims each)
        const int trole = (warp == 0) ? 2 : (warp == 6) ? 3 : (warp == 15) ? 4 : -1;   // traced worker warps
        // Phase mixing: groups 0-1 convert frame t+1 and then recurse frame t; groups 2-3 recurse frame t first and
        // convert frame t+2 (one more A stage ahead).  At any time half of an SM sub-partition's warps are in the
        // fma-heavy conversion and half in the alu-heavy recursion.
        const bool rec_first = g >= 2;
        uint32_t c3 = 0;              // A stage of the next frame this warp converts (frame counter mod 3)
        const uint32_t lane_sel = (uint32_t)(q * 32) << 16;
        // per-thread addresses, pinned in registers
        const uint32_t ta0 = pin_reg(tmem_a + lane_sel + 16u * pr0);               // A operand, stage 0 (stage 1: + a_cols)
        const uint32_t acc0 = pin_reg(tmem_acc + lane_sel + (uint32_t)mbeg * 8u);  // accumulators, stage 0 (stage 1: + ncols)
        const uint32_t raw0 = pin_reg(smem_u32(sRaw) + (uint32_t)r * rstride + 32u * pr0);
        const uint32_t trS = pin_reg(smem_u32(sTr) + (uint32_t)mbeg * (TC_TRQ * 16u));
        const uint32_t sbS = pin_reg(smem_u32(sS) + 32u * pr0);
        const uint32_t sbB = sbS + 16u * nck;
        const size_t bp_model = (size_t)p.maxT * p.Bpad;                 // elements between consecutive models
        const size_t bp_frame = (size_t)p.Bpad;
        // float4 index (within the row) from which a pair's chunks lie outside the feature row (never read)
        const int nrd4 = p.ldx / 4 - 2 * pr0;

        auto lds4 = [](uint32_t a) -> float4 {
            float4 v;
            asm volatile("ld.shared.v4.f32 {%0, %1, %2, %3}, [%4];" : "=f"(v.x), "=f"(v.y), "=f"(v.z), "=f"(v.w) : "r"(a));
            return v;
        };
        // 4 feature dims: standardise, square, split into fp16 hi / lo.  out[0..3] = hi (x'01, x'23, x'^2 01, x'^2 23), out2 = lo
        auto split4 = [&](const float4 x, const float4 sc, const float4 of, uint32_t *hi, uint32_t *lo) {
            const float2 a01 = fma2(make_float2(x.x, x.y), make_float2(sc.x, sc.y), make_float2(of.x, of.y));
            const float2 a23 = fma2(make_float2(x.z, x.w), make_float2(sc.z, sc.w), make_float2(of.z, of.w));
            const float2 q01 = mul2(a01, a01), q23 = mul2(a23, a23);
            hi[0] = pack_h2(a01); hi[1] = pack_h2(a23); hi[2] = pack_h2(q01); hi[3] = pack_h2(q23);
            lo[0] = pack_h2(sub2(a01, unpack_h2(hi[0]))); lo[1] = pack_h2(sub2(a23, unpack_h2(hi[1])));
            lo[2] = pack_h2(sub2(q01, unpack_h2(hi[2]))); lo[3] = pack_h2(sub2(q23, unpack_h2(hi[3])));
        };

        // NPc / MCc: compile-time pair and model counts of this group (0 = run-time counts, generic model sets)
        auto run = [&](auto NPc, auto MCc) {
            constexpr int NPT = decltype(NPc)::value, MCT = decltype(MCc)::value;
            constexpr int NPMAX = NPT > 0 ? NPT : 2, MCMAX = MCT > 0 ? MCT : MG;
            const int np = NPT > 0 ? NPT : npr, mc = MCT > 0 ? MCT : mcnt;
            const uint32_t recf = pin_reg(rec_first ? 1u : 0u);
            // accumulator stage / phase of the frame being recursed (frame counter f): toggled, not recomputed
            uint32_t as = f & 1u, aph = (f >> 1) & 1u;
            for (int tile = blockIdx.x; tile < ntiles; tile += gridDim.x) {
                // tile length, and whether every row is live with exactly that length (equal-length batches: the
                // per-row activity tests then drop out of the frame loops)
                int Tt = 0, Tmin = 0x7fffffff;
                for (int rr = lane; rr < TC_ROWS; rr += 32) {
                    int64_t o;
                    const int Tr = row_frames(tile * TC_ROWS + rr, o);
                    Tt = max(Tt, Tr); Tmin = min(Tmin, Tr);
                }
                for (int o = 16; o > 0; o >>= 1) {
                    Tt = max(Tt, __shfl_xor_sync(0xffffffffu, Tt, o));
                    Tmin = min(Tmin, __shfl_xor_sync(0xffffffffu, Tmin, o));
                }
                const bool uniform = Tmin == Tt;
                const int ul = tile * TC_ROWS + r;
                int64_t off;
                const int Te = row_frames(ul, off);
                const bool live = ul < p.nu;

                float2 U[MCMAX][4];
                float Ux[MCMAX], base[MCMAX];
                uint16_t *bpt = p.bp + (size_t)mbeg * bp_model + ul;       // back-pointer word of (first model, frame t, this row)
#pragma unroll
                for (int k = 0; k < MCMAX; k++) {
                    Ux[k] = -INFINITY; base[k] = 0.f;
#pragma unroll
                    for (int j = 0; j < 4; j++) U[k][j] = make_float2(-INFINITY, -INFINITY);
                }

                // conversion cursor: frames are converted strictly in order, so the ring position is kept incrementally
                int cfi = 0, ct = 0;                                        // frame inside the stage, frame of the tile
                uint32_t cslot = sg & (uint32_t)(nst - 1), crph = (sg >> p.nst_shift) & 1u;
                uint32_t crow = raw0 + cslot * stage_bytes;
                // frame ct of this tile -> standardise, square, split, store into A-operand stage c3 (= frame counter mod 3)
                auto convert = [&](auto UNIc, uint32_t fr) {
                    constexpr bool UNI = decltype(UNIc)::value;
                    if (TRACE && trole >= 0) trace(trole, fr, 0);
                    if (cfi == 0) mbar_wait(barRaw_full + 8 * cslot, crph);
                    if (TRACE && trole >= 0) trace(trole, fr, 1);
                    const bool ok = UNI || ct < Te;              // Te == 0 for rows beyond the batch
                    const uint32_t ta = ta0 + c3 * a_cols;
#pragma unroll
                    for (int c = 0; c < NPMAX; c++) {
                        if (c < np) {
                            float4 x0 = make_float4(0.f, 0.f, 0.f, 0.f), x1 = x0;
                            if (ok && 2 * c < nrd4) x0 = lds4(crow + 32u * c);
                            if (ok && 2 * c + 1 < nrd4) x1 = lds4(crow + 32u * c + 16u);
                            uint32_t v[16];      // [hi chunk 0 | hi chunk 1 | lo chunk 0 | lo chunk 1] = 16 consecutive TMEM columns
                            split4(x0, lds4(sbS + 32u * c), lds4(sbB + 32u * c), v, v + 8);
                            split4(x1, lds4(sbS + 32u * c + 16u), lds4(sbB + 32u * c + 16u), v + 4, v + 12);
                            tmem_st16(ta + 16u * c, v);
                        }
                    }
                    tmem_st_wait();
                    tc_fence_before();
                    __syncwarp();
                    const bool last = (cfi == F - 1) || (ct == Tt - 1);
                    if (lane == 0) {
                        mbar_arrive(barA_full + 8 * c3);
                        if (last) mbar_arrive(barRaw_empty + 8 * cslot);
                    }
                    if (++c3 == 3) c3 = 0;
                    ct++;
                    if (last) {                                   // next stage of the ring
                        cfi = 0; sg++;
                        if (++cslot == (uint32_t)nst) { cslot = 0; crph ^= 1u; }
                        crow = raw0 + cslot * stage_bytes;
                    } else {
                        cfi++; crow += rowbytes;
                    }
                    if (TRACE && trole >= 0) trace(trole, fr, 2);
                };
                // accumulators of the current frame ready?  (their release needs no barrier: a warp signals A_full(f + 2) only
                // after its last tcgen05.ld of frame f, and the MMAs of frame f + 2 wait for every warp's A_full(f + 2))
                auto acc_ready = [&]() -> uint32_t {
                    if (TRACE && trole >= 0) trace(trole, f, 3);
                    mbar_wait(barAcc_full + 8 * as, aph);
                    if (TRACE && trole >= 0) trace(trole, f, 4);
                    tc_fence_after();
                    return acc0 + as * (uint32_t)ncols;
                };
                auto acc_next = [&]() { aph ^= as; as ^= 1u; };       // phase flips when the stage wraps from 1 to 0
                auto dbg_dump = [&](int k, int t, const uint32_t (&ev)[8]) {
                    const float4 st0 = lds4(trS + (TC_TRQ * 16u) * k + 48u), st1 = lds4(trS + (TC_TRQ * 16u) * k + 64u);
                    const float st[8] = {st0.x, st0.y, st0.z, st0.w, st1.x, st1.y, st1.z, st1.w};
#pragma unroll
                    for (int j = 0; j < 8; j++)
                        p.dbgE[(size_t)(off + t) * ncols + (mbeg + k) * 8 + j] = __uint_as_float(ev[j]) - st[j];
                };
                constexpr std::integral_constant<bool, false> RAGGED{};
                constexpr std::integral_constant<bool, true> UNIFORM{};

                if (Tt > 0) convert(RAGGED, f);
                if (recf && Tt > 1) convert(RAGGED, f + 1);
                const int Tearly = min(Tt, 9);
                int t = 0;
                // ---- frames 0 .. 8: entry state, closed exit (generic step) ----
                for (; t < Tearly; t++, f++) {
                    if (!recf && t + 1 < Tt) convert(RAGGED, f + 1);
                    const uint32_t tacc = acc_ready();
                    acc_next();
                    const bool act = t < Te;
#pragma unroll
                    for (int k = 0; k < MCMAX; k++) {
                        if (k < mc) {
                            uint32_t ev[8];
                            tmem_ld8(tacc + 8u * k, ev);
                            tmem_ld_wait();
                            if (DBG && p.dbgE && act) dbg_dump(k, t, ev);
                            if (act) {
                                const float4 cm = lds4(trS + (TC_TRQ * 16u) * k + 32u);
                                if (t == 0) {
                                    U[k][0].x = cm.y + __uint_as_float(ev[0]);   // U_1 = ln A01 + E[0,1] + ln A11
                                } else {
                                    const float4 c03 = lds4(trS + (TC_TRQ * 16u) * k), c47 = lds4(trS + (TC_TRQ * 16u) * k + 16u);
                                    const uint32_t bits = vit_step<true>(U[k], Ux[k], c03, c47, cm.x, cm.y, ev, t);
                                    bpt[(size_t)k * bp_model] = (uint16_t)bits;
                                    if ((t & 3) == 0) vit_renorm(U[k], Ux[k], base[k]);
                                }
                            }
                        }
                    }
                    tc_fence_before();
                    if (TRACE && trole >= 0) trace(trole, f, 5);
                    bpt += bp_frame;
                    if (recf && t + 2 < Tt) convert(RAGGED, f + 2);
                }
                // ---- steady state: no entry arc, exit open ----
                auto steady = [&](auto UNIc) {
                    constexpr bool UNI = decltype(UNIc)::value;
                    for (; t < Tt; t++, f++) {
                        if (!recf && t + 1 < Tt) convert(UNIc, f + 1);
                        const uint32_t tacc = acc_ready();
                        acc_next();
                        const bool act = UNI || t < Te;
                        const bool rn = (t & 3) == 0;
#pragma unroll
                        for (int k = 0; k < MCMAX; k++) {
                            if (k < mc) {
                                uint32_t ev[8];
                                tmem_ld8(tacc + 8u * k, ev);
                                tmem_ld_wait();
                                if (DBG && p.dbgE && act) dbg_dump(k, t, ev);
                                if (act) {
                                    const float4 c03 = lds4(trS + (TC_TRQ * 16u) * k), c47 = lds4(trS + (TC_TRQ * 16u) * k + 16u), cm = lds4(trS + (TC_TRQ * 16u) * k + 32u);
                                    const uint32_t bits = vit_step<false>(U[k], Ux[k], c03, c47, cm.x, cm.y, ev, t);
                                    bpt[(size_t)k * bp_model] = (uint16_t)bits;
                                    if (rn) vit_renorm(U[k], Ux[k], base[k]);
                                }
                            }
                        }
                        tc_fence_before();
                        if (TRACE && trole >= 0) trace(trole, f, 5);
                        bpt += bp_frame;
                        if (recf && t + 2 < Tt) convert(UNIc, f + 2);
                    }
                };
                if (uniform) steady(UNIFORM); else steady(RAGGED);
                if (live) {
#pragma unroll
                    for (int k = 0; k < MCMAX; k++)
                        if (k < mc) {
                            const double sc = (Te > 0 && Ux[k] > -INFINITY) ? (double)Ux[k] + (double)base[k] : -INFINITY;
                            p.scores[(size_t)ul * M + mbeg + k] = sc;
                        }
                }
            }
        };
        // the cfg-2 split (M = 11, D = 39): group 0 = 2 chunk pairs + 2 models, groups 1-3 = 1 pair + 3 models
        if (MG == 3 && npr == 2 && mcnt == 2) run(std::integral_constant<int, 2>{}, std::integral_constant<int, 2>{});
        else if (MG == 3 && npr == 1 && mcnt == 3) run(std::integral_constant<int, 1>{}, std::integral_constant<int, 3>{});
        else run(std::integral_constant<int, 0>{}, std::integral_constant<int, 0>{});
    }
    tc_fence_before();
    __syncthreads();
    if (warp == TC_WORKER_WARPS) tmem_dealloc(tmem_base, tcols);
}

// ------------------------------------------------------------------------------------------------
// k_viterbi_tma: the same pipeline for EQUAL-LENGTH batches stored contiguously (total_frames == B * T, the shape of
// BASELINE cfg 2): the raw-feature ring is filled by TMA tensor-map tile loads -- one cp.async.bulk.tensor.3d per frame of
// a tile (box = [row width] x 1 frame x 128 utterances) issued by ONE thread -- instead of 128 per-row bulk copies per
// stage from three polling copy warps (which were 12 % of the issued instructions of k_viterbi_tc).  The box is one
// 16-byte chunk wider than the K extent of the A operand, so rows land at an odd multiple of 16 bytes (conflict-free
// LDS.128 with one row per lane) and the columns past the feature row arrive as zeros; utterances past the end of the
// batch arrive as zero rows, so the worker loops carry no per-row activity tests.  18 warps (16 workers, MMA, TMA) leave
// 112 registers per thread: the standardisation constants of a thread's feature chunks and the transition constants of
// its models stay in registers for the specialised splits.  The lo halves of the fp16 split come from one mixed-precision
// FMA per element (FHFMA: x - (fp32)hi) instead of unpack + subtract.
#define TM_THREADS (TC_WORKERS + 64)
#ifndef TM_TR_IN_REGS
#define TM_TR_IN_REGS 0
#endif
#ifndef TM_SB_IN_REGS
#define TM_SB_IN_REGS 0
#endif
struct TmSmem { uint32_t w, raw, tr, sb, bar, total; };
__host__ __device__ inline TmSmem tm_smem_layout(int M, int nck, int ncols, int nst, int F, uint32_t rw) {
    TmSmem L;
    L.w = 0;
    L.raw = ((uint32_t)2 * (ncols / 8) * nck * 128 + 127u) & ~127u;
    L.tr = L.raw + (uint32_t)nst * F * TC_ROWS * rw;
    L.sb = L.tr + (uint32_t)M * TC_TRQ * 16;
    L.bar = (L.sb + (uint32_t)8 * nck * 4 + 15u) & ~15u;
    L.total = L.bar + (2 * TC_MAX_STAGES + 6) * 8 + 16;
    return L;
}

template <int MG, int NKS>
__global__ void __launch_bounds__(TM_THREADS, 1) k_viterbi_tma(const TcParams p, const __grid_constant__ CUtensorMap tmap) {
    extern __shared__ __align__(128) unsigned char smem[];
    const int nck = p.nck, ncols = p.ncols, M = p.M;
    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
    const int F = 1 << p.Fshift, nst = 1 << p.nst_shift;
    const uint32_t rw = p.rstride;                                   // bytes per row in the ring: (nck + 1) * 16
    const uint32_t frame_bytes = TC_ROWS * rw, stage_bytes = (uint32_t)F * frame_bytes;
    const TmSmem L = tm_smem_layout(M, nck, ncols, nst, F, rw);
    const uint32_t w_plane = (uint32_t)(ncols / 8) * nck * 128;
    unsigned char *sW = smem + L.w;
    unsigned char *sRaw = smem + L.raw;
    const float4 *sTr = reinterpret_cast<const float4 *>(smem + L.tr);
    const float4 *sS = reinterpret_cast<const float4 *>(smem + L.sb);
    uint64_t *sBar = reinterpret_cast<uint64_t *>(smem + L.bar);
    uint32_t *sTmem = reinterpret_cast<uint32_t *>(sBar + 2 * TC_MAX_STAGES + 6);
    const uint32_t barRaw_full = smem_u32(sBar), barRaw_empty = barRaw_full + 8 * TC_MAX_STAGES;
    const uint32_t barA_full = barRaw_empty + 8 * TC_MAX_STAGES, barAcc_full = barA_full + 24;

    {
        const uint4 *src = reinterpret_cast<const uint4 *>(p.wimg);
        uint4 *dst = reinterpret_cast<uint4 *>(sW);
        for (uint32_t i = tid; i < 2 * w_plane / 16; i += TM_THREADS) dst[i] = src[i];
        float4 *dtr = reinterpret_cast<float4 *>(smem + L.tr);
        for (int i = tid; i < M * TC_TRQ; i += TM_THREADS) dtr[i] = p.trp[i];
        float *dsb = reinterpret_cast<float *>(smem + L.sb);
        for (int i = tid; i < 8 * nck; i += TM_THREADS) dsb[i] = p.sb[i];
    }
    if (tid == 0) {
        for (int s = 0; s < nst; s++) {
            mbar_init(barRaw_full + 8 * s, 1);
            mbar_init(barRaw_empty + 8 * s, TC_WORKER_WARPS);
        }
        for (int s = 0; s < 3; s++) mbar_init(barA_full + 8 * s, TC_WORKER_WARPS);
        for (int s = 0; s < 2; s++) mbar_init(barAcc_full + 8 * s, 1);
        fence_barrier_init();
    }
    const uint32_t a_cols = 8u * nck;
    uint32_t tcols = 32;
    while (tcols < 2u * ncols + 3u * a_cols) tcols <<= 1;
    if (warp == TC_WORKER_WARPS) tmem_alloc(smem_u32(sTmem), tcols);
    fence_proxy_async();
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    const uint32_t tmem_base = *sTmem;
    const uint32_t tmem_acc = tmem_base, tmem_a = tmem_base + 2u * ncols;

    const int ntiles = (p.nu + TC_ROWS - 1) / TC_ROWS;
    const int Tt = p.maxT;               // frames walked: the same for every utterance
    uint32_t f = 0, sg = 0;

    if (warp == TC_WORKER_WARPS + 1) {
        // ===================== TMA producer: one thread =====================
        if (lane == 0) {
            tma_prefetch_desc(&tmap);
            const int nsg = (Tt + F - 1) >> p.Fshift;
            for (int tile = blockIdx.x; tile < ntiles; tile += gridDim.x) {
                const int urow = p.u0 + tile * TC_ROWS;
                for (int k = 0; k < nsg; k++, sg++) {
                    const uint32_t slot = sg & (uint32_t)(nst - 1), ph = (sg >> p.nst_shift) & 1u;
                    const uint32_t bar = barRaw_full + 8 * slot;
                    const int nf = min(F, Tt - k * F);
                    mbar_wait(barRaw_empty + 8 * slot, ph ^ 1u);
                    mbar_arrive_tx(bar, (uint32_t)nf * frame_bytes);
                    const uint32_t dst = smem_u32(sRaw) + slot * stage_bytes;
                    for (int fi = 0; fi < nf; fi++) tma_load_3d(dst + (uint32_t)fi * frame_bytes, &tmap, 0, k * F + fi, urow, bar);
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
        uint32_t a3 = 0, aph = 0;
        const int nfr = Tt * ((ntiles - (int)blockIdx.x + (int)gridDim.x - 1) / (int)gridDim.x);   // frames this CTA walks
        for (int i = 0; i < nfr; i++, f++) {
            const uint32_t s = f & 1;
            mbar_wait(barA_full + 8 * a3, aph);
            tc_fence_after();
            if (elect_one()) {
                const uint32_t d_tmem = tmem_acc + s * (uint32_t)ncols;
                const uint32_t a_hi = tmem_a + a3 * a_cols, a_lo = a_hi + 8u;
                if (NKS > 0) {
#pragma unroll
                    for (int ks = 0; ks < NKS; ks++) umma_f16_ts(d_tmem, a_lo + ks * 16, dW_hi + (uint64_t)(16 * ks), idesc, ks > 0);
#pragma unroll
                    for (int ks = 0; ks < NKS; ks++) umma_f16_ts(d_tmem, a_hi + ks * 16, dW_lo + (uint64_t)(16 * ks), idesc, 1);
#pragma unroll
                    for (int ks = 0; ks < NKS; ks++) umma_f16_ts(d_tmem, a_hi + ks * 16, dW_hi + (uint64_t)(16 * ks), idesc, 1);
                } else {
                    uint64_t dh = dW_hi, dl = dW_lo;
                    uint32_t a = a_lo;
                    for (int ks = 0; ks < nks; ks++, a += 16, dh += 16) umma_f16_ts(d_tmem, a, dh, idesc, ks > 0);
                    a = a_hi;
                    for (int ks = 0; ks < nks; ks++, a += 16, dl += 16) umma_f16_ts(d_tmem, a, dl, idesc, 1);
                    a = a_hi; dh = dW_hi;
                    for (int ks = 0; ks < nks; ks++, a += 16, dh += 16) umma_f16_ts(d_tmem, a, dh, idesc, 1);
                }
                umma_commit(barAcc_full + 8 * s);
            }
            __syncwarp();
            if (++a3 == 3) { a3 = 0; aph ^= 1u; }
        }
    } else {
        // ===================== workers =====================
        const int q = warp & 3, g = warp >> 2, r = q * 32 + lane;
        const int mbeg = p.mod0[g], mcnt = p.nmod[g];
        const int pr0 = p.pair0[g], npr = p.npair[g];
        const bool rec_first = g >= 2;
        uint32_t c3 = 0;
        const uint32_t lane_sel = (uint32_t)(q * 32) << 16;
        const uint32_t ta0 = pin_reg(tmem_a + lane_sel + 16u * pr0);
        const uint32_t acc0 = pin_reg(tmem_acc + lane_sel + (uint32_t)mbeg * 8u);
        const uint32_t raw0 = pin_reg(smem_u32(sRaw) + (uint32_t)r * rw + 32u * pr0);
        const uint32_t trS = smem_u32(sTr) + (uint32_t)mbeg * (TC_TRQ * 16u);
        const uint32_t sbS = smem_u32(sS) + 32u * pr0;
        const uint32_t sbB = sbS + 16u * nck;
        // back-pointer scratch addressed with 32-bit element offsets (the scratch is bounded to 1 GB by the launcher)
        const uint32_t bp_model = (uint32_t)p.maxT * (uint32_t)p.Bpad;
        const uint32_t bp_frame = (uint32_t)p.Bpad;

        auto lds4 = [](uint32_t a) -> float4 {
            float4 v;
            asm volatile("ld.shared.v4.f32 {%0, %1, %2, %3}, [%4];" : "=f"(v.x), "=f"(v.y), "=f"(v.z), "=f"(v.w) : "r"(a));
            return v;
        };
        auto split4 = [&](const float4 x, const float4 sc, const float4 of, uint32_t *hi, uint32_t *lo) {
            const float2 a01 = fma2(make_float2(x.x, x.y), make_float2(sc.x, sc.y), make_float2(of.x, of.y));
            const float2 a23 = fma2(make_float2(x.z, x.w), make_float2(sc.z, sc.w), make_float2(of.z, of.w));
            const float2 q01 = mul2(a01, a01), q23 = mul2(a23, a23);
            hi[0] = pack_h2(a01); hi[1] = pack_h2(a23); hi[2] = pack_h2(q01); hi[3] = pack_h2(q23);
            lo[0] = pack_h2(residual_h2(a01, hi[0])); lo[1] = pack_h2(residual_h2(a23, hi[1]));
            lo[2] = pack_h2(residual_h2(q01, hi[2])); lo[3] = pack_h2(residual_h2(q23, hi[3]));
        };

        auto run = [&](auto NPc, auto MCc) {
            constexpr int NPT = decltype(NPc)::value, MCT = decltype(MCc)::value;
            constexpr bool SPEC = NPT > 0 && TM_TR_IN_REGS;      // specialised split: transition constants live in registers
            constexpr int NPMAX = NPT > 0 ? NPT : 2, MCMAX = MCT > 0 ? MCT : MG;
            const int np = NPT > 0 ? NPT : npr, mc = MCT > 0 ? MCT : mcnt;
            const uint32_t recf = pin_reg(rec_first ? 1u : 0u);
            uint32_t as = 0, aph = 0;
            // register-resident constants (specialised splits only)
            constexpr bool SBREG = SPEC && TM_SB_IN_REGS;     // standardisation constants in registers, too
            float4 rsc[SBREG ? 2 * NPMAX : 1], rof[SBREG ? 2 * NPMAX : 1];
            float4 rc03[SPEC ? MCMAX : 1];
            if (SBREG) {
#pragma unroll
                for (int c = 0; c < 2 * NPMAX; c++) { rsc[c] = lds4(sbS + 16u * c); rof[c] = lds4(sbB + 16u * c); }
            }
            if (SPEC) {
#pragma unroll
                for (int k = 0; k < MCMAX; k++) {
                    rc03[k] = lds4(trS + (TC_TRQ * 16u) * k);
                }
            }
            for (int tile = blockIdx.x; tile < ntiles; tile += gridDim.x) {
                const int ul = tile * TC_ROWS + r;
                const bool live = ul < p.nu;
                float2 U[MCMAX][4];
                float Ux[MCMAX], base[MCMAX];
                uint32_t bpo = (uint32_t)mbeg * bp_model + (uint32_t)ul;
#pragma unroll
                for (int k = 0; k < MCMAX; k++) {
                    Ux[k] = -INFINITY; base[k] = 0.f;
#pragma unroll
                    for (int j = 0; j < 4; j++) U[k][j] = make_float2(-INFINITY, -INFINITY);
                }
                int cfi = 0, ct = 0;
                uint32_t cslot = sg & (uint32_t)(nst - 1), crph = (sg >> p.nst_shift) & 1u;
                uint32_t crow = raw0 + cslot * stage_bytes;
                auto convert = [&]() {
                    if (cfi == 0) mbar_wait(barRaw_full + 8 * cslot, crph);
                    const uint32_t ta = ta0 + c3 * a_cols;
#pragma unroll
                    for (int c = 0; c < NPMAX; c++) {
                        if (c < np) {
                            const float4 x0 = lds4(crow + 32u * c), x1 = lds4(crow + 32u * c + 16u);
                            uint32_t v[16];
                            if (SBREG) {
                                split4(x0, rsc[2 * c], rof[2 * c], v, v + 8);
                                split4(x1, rsc[2 * c + 1], rof[2 * c + 1], v + 4, v + 12);
                            } else {
                                split4(x0, lds4(sbS + 32u * c), lds4(sbB + 32u * c), v, v + 8);
                                split4(x1, lds4(sbS + 32u * c + 16u), lds4(sbB + 32u * c + 16u), v + 4, v + 12);
                            }
                            tmem_st16(ta + 16u * c, v);
                        }
                    }
                    tmem_st_wait();
                    tc_fence_before();
                    __syncwarp();
                    const bool last = (cfi == F - 1) || (ct == Tt - 1);
                    if (lane == 0) {
                        mbar_arrive(barA_full + 8 * c3);
                        if (last) mbar_arrive(barRaw_empty + 8 * cslot);
                    }
                    if (++c3 == 3) c3 = 0;
                    ct++;
                    if (last) {
                        cfi = 0; sg++;
                        if (++cslot == (uint32_t)nst) { cslot = 0; crph ^= 1u; }
                        crow = raw0 + cslot * stage_bytes;
                    } else {
                        cfi++; crow += frame_bytes;
                    }
                };
                auto acc_ready = [&]() -> uint32_t {
                    mbar_wait(barAcc_full + 8 * as, aph);
                    tc_fence_after();
                    return acc0 + as * (uint32_t)ncols;
                };
                auto acc_next = [&]() { aph ^= as; as ^= 1u; };

                if (Tt > 0) convert();
                if (recf && Tt > 1) convert();
                const int Tearly = min(Tt, 9);
                int t = 0;
                for (; t < Tearly; t++) {
                    if (!recf && t + 1 < Tt) convert();
                    const uint32_t tacc = acc_ready();
                    acc_next();
#pragma unroll
                    for (int k = 0; k < MCMAX; k++) {
                        if (k < mc) {
                            uint32_t ev[8];
                            tmem_ld8(tacc + 8u * k, ev);
                            tmem_ld_wait();
                            const float4 cm = lds4(trS + (TC_TRQ * 16u) * k + 32u);
                            if (t == 0) {
                                U[k][0].x = cm.y + __uint_as_float(ev[0]);
                            } else {
                                const float4 c03 = lds4(trS + (TC_TRQ * 16u) * k), c47 = lds4(trS + (TC_TRQ * 16u) * k + 16u);
                                const uint32_t bits = vit_step<true>(U[k], Ux[k], c03, c47, cm.x, cm.y, ev, t);
                                p.bp[bpo + (uint32_t)k * bp_model] = (uint16_t)bits;
                                if ((t & 3) == 0) vit_renorm(U[k], Ux[k], base[k]);
                            }
                        }
                    }
                    tc_fence_before();
                    bpo += bp_frame;
                    if (recf && t + 2 < Tt) convert();
                }
                for (; t < Tt; t++) {
                    if (!recf && t + 1 < Tt) convert();
                    const uint32_t tacc = acc_ready();
                    acc_next();
                    const bool rn = (t & 7) == 0;
#pragma unroll
                    for (int k = 0; k < MCMAX; k++) {
                        if (k < mc) {
                            uint32_t ev[8];
                            tmem_ld8(tacc + 8u * k, ev);
                            tmem_ld_wait();
                            uint32_t bits;
                            if (SPEC) {
                                float aex;
                                asm volatile("ld.shared.f32 %0, [%1];" : "=f"(aex) : "r"(trS + (TC_TRQ * 16u) * k + 32u));
                                bits = vit_step<false>(U[k], Ux[k], rc03[k], lds4(trS + (TC_TRQ * 16u) * k + 16u), aex, 0.f, ev, t);
                            } else {
                                const float4 c03 = lds4(trS + (TC_TRQ * 16u) * k), c47 = lds4(trS + (TC_TRQ * 16u) * k + 16u), cm = lds4(trS + (TC_TRQ * 16u) * k + 32u);
                                bits = vit_step<false>(U[k], Ux[k], c03, c47, cm.x, cm.y, ev, t);
                            }
                            p.bp[bpo + (uint32_t)k * bp_model] = (uint16_t)bits;
                            if (rn) vit_renorm(U[k], Ux[k], base[k]);
                        }
                    }
                    tc_fence_before();
                    bpo += bp_frame;
                    if (recf && t + 2 < Tt) convert();
                }
                if (live) {
#pragma unroll
                    for (int k = 0; k < MCMAX; k++)
                        if (k < mc) {
                            const double sc = (Tt > 0 && Ux[k] > -INFINITY) ? (double)Ux[k] + (double)base[k] : -INFINITY;
                            p.scores[(size_t)ul * M + mbeg + k] = sc;
                        }
                }
            }
        };
        if (MG == 3 && npr == 2 && mcnt == 2) run(std::integral_constant<int, 2>{}, std::integral_constant<int, 2>{});
        else if (MG == 3 && npr == 1 && mcnt == 3) run(std::integral_constant<int, 1>{}, std::integral_constant<int, 3>{});
        else run(std::integral_constant<int, 0>{}, std::integral_constant<int, 0>{});
    }
    tc_fence_before();
    __syncthreads();
    if (warp == TC_WORKER_WARPS) tmem_dealloc(tmem_base, tcols);
}

// ------------------------------------------------------------------------------------------------
bool sapr_tc_eligible(const sapr_models *m) {
    return m->emission == SAPR_EMIT_DIAG && m->topology == SAPR_TOPO_ENTRY_EXIT && m->N == 8 && m->M <= 12 &&
           m->D + 1 <= 48;
}

bool sapr_tc_usable(const sapr_models *m) { return m->tc_image && sapr_tc_eligible(m) && m->tc_loops_finite; }

static void tc_geometry(const sapr_models *m, int *nck_out, int *ncols_out) {
    int nck = (m->D + 1 + 3) / 4;
    nck = (nck + 1) / 2 * 2;
    const int ncols = (m->M * 8 + 15) / 16 * 16;
    if (nck_out) *nck_out = nck;
    if (ncols_out) *ncols_out = ncols;
}

static inline size_t al256(size_t x) { return (x + 255) / 256 * 256; }

size_t sapr_tc_image_bytes(const sapr_models *m, int *nck_out, int *ncols_out) {
    int nck, ncols;
    tc_geometry(m, &nck, &ncols);
    if (nck_out) *nck_out = nck;
    if (ncols_out) *ncols_out = ncols;
    return al256((size_t)2 * (ncols / 8) * nck * 64 * sizeof(__half)) + al256((size_t)8 * nck * sizeof(float)) +
           al256((size_t)m->M * TC_TRQ * sizeof(float4));
}

int sapr_tc_prepare(sapr_models *m) {
    sapr_ctx *ctx = m->ctx;
    int nck, ncols;
    tc_geometry(m, &nck, &ncols);
    const size_t w = al256((size_t)2 * (ncols / 8) * nck * 64 * sizeof(__half));
    const size_t g = al256((size_t)8 * nck * sizeof(float));
    __half *wimg = (__half *)m->tc_image;
    float *sb = (float *)((char *)m->tc_image + w);
    float4 *trp = (float4 *)((char *)m->tc_image + w + g);
    k_prepare_tc<<<std::max(1, std::min(32, (ncols * 4 * nck + 255) / 256)), 256, sizeof(double) * 2 * 4 * nck, ctx->stream>>>(m->M, m->S, m->D, nck, ncols, m->mean, m->cov, m->la64,
                                                                         m->lb64, wimg, sb, trp);
    SAPR_LAUNCH_CHECK(ctx);
    return SAPR_OK;
}

// argmax + back-trace launcher shared with the SIMT path (viterbi.cu)
int sapr_viterbi_finish_u16(sapr_ctx *ctx, const int64_t *offsets, int u0, int nu, int N, int nslots, int first_frames,
                            const uint16_t *bp, int64_t Bpad, int maxT, const double *scores, int32_t *best_word,
                            double *best_score, double *scores_out, int M, uint8_t *best_path, uint8_t *all_paths,
                            int64_t total_frames, const SaprFlag *flag);

int sapr_viterbi_v3_launch(sapr_ctx *ctx, sapr_models *m, const float *X, int ldx, const int64_t *offsets, int B, int max_T,
                           int first_frames, int32_t *best_word, double *best_score, double *scores, uint8_t *best_path,
                           bool *taken);

int sapr_viterbi_tc_launch(sapr_ctx *ctx, sapr_models *m, const float *X, int ldx, const int64_t *offsets, int B,
                           int64_t total_frames, int max_T, int first_frames, int32_t *best_word, double *best_score,
                           double *scores, uint8_t *best_path, uint8_t *all_paths, float *dbgE) {
    int nck, ncols;
    tc_geometry(m, &nck, &ncols);
    const size_t w = al256((size_t)2 * (ncols / 8) * nck * 64 * sizeof(__half));
    const size_t g = al256((size_t)8 * nck * sizeof(float));
    const int M = m->M;
    const int Tm = (first_frames > 0 && first_frames < max_T) ? first_frames : max_T;
    int64_t per_utt = (int64_t)M * (Tm > 0 ? Tm : 1) * sizeof(uint16_t);
    int chunk = (int)std::min<int64_t>(B, std::max<int64_t>(TC_ROWS, ((int64_t)1024 << 20) / per_utt));
    chunk = (chunk + TC_ROWS - 1) / TC_ROWS * TC_ROWS;
    const int64_t Bpad = chunk;
    int rc = sapr_ws_reserve(ctx, 0, (size_t)per_utt * Bpad);
    if (rc) return rc;
    if ((rc = sapr_ws_reserve(ctx, 1, (size_t)chunk * M * sizeof(double)))) return rc;
    uint16_t *bp = (uint16_t *)ctx->ws[0];
    double *sc_ws = (double *)ctx->ws[1];

    // raw-feature ring: largest power-of-two frames per stage (<= 8) such that two stages fit beside the W image
    const uint32_t rowbytes = (uint32_t)ldx * 4u;
    const size_t budget = 225 * 1024;
    int Fshift = 3, nst = 2, nst_shift = 1;
    uint32_t rstride = 0;
    TcSmem L;
    for (;; Fshift--) {
        const uint32_t F = 1u << Fshift;
        rstride = F * rowbytes + 16u;
        if (((rstride >> 4) & 1u) == 0) rstride += 16u;     // odd multiple of 16 B: conflict-free LDS.128 across rows
        L = tc_smem_layout(M, nck, ncols, nst, rstride);
        if (L.total <= budget) break;
        if (Fshift == 0) SAPR_FAIL(ctx, SAPR_E_RANGE, "viterbi (tensor core): feature rows too wide for the shared-memory ring");
    }
    if (Fshift <= 1 && tc_smem_layout(M, nck, ncols, 4, rstride).total <= budget) { nst = 4; nst_shift = 2; }
    L = tc_smem_layout(M, nck, ncols, nst, rstride);
    const size_t smem = L.total;
    const int MG = (M + TC_GROUPS - 1) / TC_GROUPS;
    // equal-length contiguous batch, best path only: the re-cut kernel (viterbi_v3.cu) when the shape fits it
    if (!dbgE && !all_paths && Tm > 0 && total_frames == (int64_t)B * max_T && !getenv("SAPR_TC_TRACE")) {
        bool taken = false;
        if ((rc = sapr_viterbi_v3_launch(ctx, m, X, ldx, offsets, B, max_T, first_frames, best_word, best_score, scores, best_path, &taken)))
            return rc;
        if (taken) return SAPR_OK;
    }
    // equal-length contiguous batch (every utterance has max_T frames): TMA tensor-map loads, k_viterbi_tma
    const char *tma_env = getenv("SAPR_TMA");
    bool use_tma = !dbgE && Tm > 0 && total_frames == (int64_t)B * max_T && (!tma_env || tma_env[0] != '0') &&
                   ((uintptr_t)X & 15u) == 0 && !getenv("SAPR_TC_TRACE");
    const uint32_t tm_rw = (uint32_t)(nck + 1) * 16u;                 // ring row: K extent of the A operand + one chunk (odd multiple of 16 B)
    int tm_Fshift = 3;
    TmSmem TL = tm_smem_layout(M, nck, ncols, 2, 1 << tm_Fshift, tm_rw);
    while (use_tma && TL.total > budget) {
        if (tm_Fshift == 0) { use_tma = false; break; }
        tm_Fshift--;
        TL = tm_smem_layout(M, nck, ncols, 2, 1 << tm_Fshift, tm_rw);
    }
    CUtensorMap tmap;
    if (use_tma) {
        const uint64_t dim[3] = {(uint64_t)ldx, (uint64_t)max_T, (uint64_t)B};
        const uint64_t str[2] = {(uint64_t)ldx * 4u, (uint64_t)max_T * ldx * 4u};
        const uint32_t box[3] = {tm_rw / 4u, 1u, (uint32_t)TC_ROWS};
        if ((rc = sapr_tmap_f32_3d(ctx, &tmap, X, dim, str, box))) return rc;
    }
    auto launch_tma = [&](auto kern, const TcParams &prm, int grid) -> int {
        SAPR_CUDA(ctx, cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)TL.total));
        {
            ProfScope ps(ctx, 0);
            kern<<<grid, TM_THREADS, TL.total, ctx->stream>>>(prm, tmap);
        }
        SAPR_LAUNCH_CHECK(ctx);
        return SAPR_OK;
    };
    auto launch = [&](auto kern, const TcParams &prm, int grid) -> int {
        SAPR_CUDA(ctx, cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
        {
            ProfScope ps(ctx, 0);
            kern<<<grid, TC_THREADS, smem, ctx->stream>>>(prm);
        }
        SAPR_LAUNCH_CHECK(ctx);
        return SAPR_OK;
    };
    // word exactness: near-ties of the fp32 word scores are listed by the arg-max kernel and re-decoded in float64
    const char *ex_env = getenv("SAPR_EXACT_WORDS");
    const bool exact = !dbgE && !all_paths && (!ex_env || ex_env[0] != '0');
    SaprFlag flag;
    ctx->flag_maxT = max_T;
    for (int u0 = 0; u0 < B; u0 += chunk) {
        const int nu = std::min(chunk, B - u0);
        if (exact && (rc = sapr_flag_setup(ctx, &flag, u0 == 0))) return rc;
        TcParams prm;
        prm.X = X; prm.ldx = ldx; prm.offsets = offsets; prm.u0 = u0; prm.nu = nu; prm.M = M; prm.D = m->D; prm.nck = nck;
        prm.ncols = ncols; prm.first_frames = first_frames; prm.wimg = (const __half *)m->tc_image;
        prm.sb = (const float *)((const char *)m->tc_image + w); prm.trp = (const float4 *)((const char *)m->tc_image + w + g);
        prm.bp = bp; prm.Bpad = Bpad; prm.maxT = Tm; prm.scores = sc_ws; prm.dbgE = dbgE;
        prm.Fshift = Fshift; prm.nst_shift = nst_shift; prm.rstride = rstride; prm.trace = nullptr;
        {   // split chunk pairs and models over the 4 worker groups so that 30 * chunks + 60 * models is balanced:
            // pairs go to the low groups first, models to the high groups first
            const int npairs = nck / 2;
            int pc[TC_GROUPS], mcn[TC_GROUPS];
            for (int gI = 0; gI < TC_GROUPS; gI++) { pc[gI] = npairs / TC_GROUPS + (gI < npairs % TC_GROUPS ? 1 : 0); mcn[gI] = 0; }
            for (int mI = 0; mI < M; mI++) {      // next model to the group with the least work so far (ties: highest group)
                int best = TC_GROUPS - 1;
                for (int gI = TC_GROUPS - 1; gI >= 0; gI--)
                    if (mcn[gI] < MG && (mcn[best] >= MG || 60 * pc[gI] + 60 * mcn[gI] < 60 * pc[best] + 60 * mcn[best])) best = gI;
                mcn[best]++;
            }
            int pa = 0, ma = 0;
            for (int gI = 0; gI < TC_GROUPS; gI++) {
                prm.pair0[gI] = pa; prm.npair[gI] = pc[gI]; pa += pc[gI];
                prm.mod0[gI] = ma; prm.nmod[gI] = mcn[gI]; ma += mcn[gI];
            }
        }
        const char *trace_path = getenv("SAPR_TC_TRACE");
        if (trace_path && MG == 3 && !dbgE && u0 == 0) {      // tuning aid: one traced launch, timestamps to a text file
            const size_t nrec = (size_t)TC_TRACE_ROLES * TC_TRACE_FRAMES * TC_TRACE_EVENTS;
            long long *dtr = nullptr;
            SAPR_CUDA(ctx, cudaMalloc(&dtr, nrec * sizeof(long long)));
            SAPR_CUDA(ctx, cudaMemsetAsync(dtr, 0, nrec * sizeof(long long), ctx->stream));
            prm.trace = dtr;
            const int ntl = (nu + TC_ROWS - 1) / TC_ROWS;
            rc = (nck == 10) ? launch(k_viterbi_tc<3, 5, false, true>, prm, std::min(ntl, ctx->sm_count))
                             : launch(k_viterbi_tc<3, 0, false, true>, prm, std::min(ntl, ctx->sm_count));
            std::vector<long long> h(nrec);
            cudaMemcpyAsync(h.data(), dtr, nrec * sizeof(long long), cudaMemcpyDeviceToHost, ctx->stream);
            cudaStreamSynchronize(ctx->stream);
            cudaFree(dtr);
            if (FILE *fp = fopen(trace_path, "w")) {
                for (int ro = 0; ro < TC_TRACE_ROLES; ro++)
                    for (int fr = 0; fr < TC_TRACE_FRAMES; fr++) {
                        fprintf(fp, "%d %d", ro, fr);
                        for (int e = 0; e < TC_TRACE_EVENTS; e++) fprintf(fp, " %lld", h[((size_t)ro * TC_TRACE_FRAMES + fr) * TC_TRACE_EVENTS + e]);
                        fprintf(fp, "\n");
                    }
                fclose(fp);
            }
            prm.trace = nullptr;
            if (rc) return rc;
        }
        const int ntiles = (nu + TC_ROWS - 1) / TC_ROWS;
        const int grid = std::min(ntiles, ctx->sm_count);
        if (use_tma) {
            prm.Fshift = tm_Fshift; prm.nst_shift = 1; prm.rstride = tm_rw;
            if (MG <= 1) rc = launch_tma(k_viterbi_tma<1, 0>, prm, grid);
            else if (MG <= 2) rc = launch_tma(k_viterbi_tma<2, 0>, prm, grid);
            else if (nck == 10) rc = launch_tma(k_viterbi_tma<3, 5>, prm, grid);
            else if (nck == 4) rc = launch_tma(k_viterbi_tma<3, 2>, prm, grid);
            else rc = launch_tma(k_viterbi_tma<3, 0>, prm, grid);
        } else
        if (dbgE) rc = launch(k_viterbi_tc<3, 0, true>, prm, grid);
        else if (MG <= 1) rc = launch(k_viterbi_tc<1, 0, false>, prm, grid);
        else if (MG <= 2) rc = launch(k_viterbi_tc<2, 0, false>, prm, grid);
        else if (nck == 10) rc = launch(k_viterbi_tc<3, 5, false>, prm, grid);     // D = 36..39 (cfg 2/3)
        else if (nck == 4) rc = launch(k_viterbi_tc<3, 2, false>, prm, grid);      // D = 12..15 (cfg 1)
        else rc = launch(k_viterbi_tc<3, 0, false>, prm, grid);
        if (rc) return rc;
        if ((rc = sapr_viterbi_finish_u16(ctx, offsets, u0, nu, m->N, M, first_frames, bp, Bpad, Tm, sc_ws, best_word, best_score,
                                          scores, M, best_path, all_paths, total_frames, exact ? &flag : nullptr)))
            return rc;
        if (exact && (rc = sapr_viterbi_redo_flagged(ctx, m, X, ldx, offsets, first_frames, nu, flag, best_word, best_score, scores, best_path)))
            return rc;
    }
    return SAPR_OK;
}
