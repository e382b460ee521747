// viterbi.cu -- batched max-product decoding with fused diagonal-Gaussian emission.
//
// Replaces custom_hmm.py:462-514 (HMM.decode) for every (utterance, model) pair and the
// strict-'>' argmax over word models of decoder.py:42-47.
//
// Mapping: one thread per (utterance, model); a warp holds 32 utterances of the SAME model so the
// model's packed (mu, 0.5/var) rows are shared-memory broadcasts, the N state scores and the exit
// score live in registers, and the left-to-right transition needs no shuffles at all.  Features are
// read once per CTA from HBM (the M model-warps of a CTA walk the same 32 utterances in lock step, so
// M-1 of the M reads hit L1).  Back-pointers are one bit per (frame, state) -- "advanced from j-1" vs
// "stayed in j" -- packed in one word per frame and kept in an L2-resident scratch laid out
// [model][frame][utterance] so each warp store is one coalesced line.
#include <stdlib.h>

#include "common.cuh"

template <typename R> struct alignas(16) Vec4 { R x, y, z, w; };

template <typename R, int NMAX>
__device__ __forceinline__ void emit_diag(const float *__restrict__ xrow, int nchunk, int N,
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
                Vec4<R> mu = *reinterpret_cast<const Vec4<R> *>(p + j * 8);
                Vec4<R> h = *reinterpret_cast<const Vec4<R> *>(p + j * 8 + 4);
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

// blockDim = (32 utterances, models-per-CTA).  all-models mode: slot = model; own-model mode
// (model_of_utt != NULL): one slot, the model differs per lane.
template <typename R, typename BP, int NMAX, bool RENORM>
__global__ void __launch_bounds__(32 * 16)
k_viterbi_fused(const float *__restrict__ X, int ldx, const int64_t *__restrict__ offsets, int u0, int nu, int M,
                int N, int nchunk, const R *__restrict__ pk, const R *__restrict__ cst_g, const R *__restrict__ la_g,
                const R *__restrict__ lb_g, const int32_t *__restrict__ model_of_utt, int first_frames,
                BP *__restrict__ bp, int64_t Bpad, int maxT, int nslots, double *__restrict__ scores) {
    extern __shared__ __align__(16) unsigned char smem_raw[];
    R *spk = reinterpret_cast<R *>(smem_raw);
    const int S = N + 2;
    const size_t per_model = (size_t)nchunk * N * 8;
    const bool own = (model_of_utt != nullptr);
    const int m0 = own ? 0 : blockIdx.y * blockDim.y;
    const int nm = own ? M : min((int)blockDim.y, M - m0);
    {   // stage the packed emission parameters of this CTA's models
        const int tid = threadIdx.y * 32 + threadIdx.x, nt = blockDim.x * blockDim.y;
        const R *src = pk + (size_t)m0 * per_model;
        for (size_t i = tid; i < (size_t)nm * per_model; i += nt) spk[i] = src[i];
    }
    __syncthreads();
    const int ul = blockIdx.x * 32 + threadIdx.x;   // utterance within this chunk
    const int slot = own ? 0 : m0 + threadIdx.y;
    if (ul >= nu || slot >= nslots || (own && threadIdx.y > 0)) return;
    const int u = u0 + ul;
    const int m = own ? model_of_utt[u] : slot;
    const R *spk_model = spk + (size_t)(m - m0) * per_model;

    R cst[NMAX], la[NMAX + 2], lb[NMAX + 2];
#pragma unroll
    for (int j = 0; j < NMAX; j++) cst[j] = (j < N) ? cst_g[(size_t)m * N + j] : R(0);
#pragma unroll
    for (int j = 0; j < NMAX + 2; j++) {
        la[j] = (j < S) ? la_g[(size_t)m * S + j] : R(0);
        lb[j] = (j < S) ? lb_g[(size_t)m * S + j] : R(0);
    }
    const R lbN = lb_g[(size_t)m * S + N], laX = la_g[(size_t)m * S + S - 1];   // ln A[N, exit], ln A[exit, exit]
    const int64_t off = offsets[u];
    const int T = (int)(offsets[u + 1] - off);
    const int Te = min((first_frames > 0 && first_frames < T) ? first_frames : T, maxT);   // the scratch holds maxT frames
    const R NINF = Num<R>::ninf();

    R V[NMAX + 1];   // V[j] = state j+1 (emitting), j < N;  exit kept separately
    R e[NMAX];
#pragma unroll
    for (int j = 0; j <= NMAX; j++) V[j] = NINF;
    R Vx = NINF;
    double base = 0.0;
    auto emit = [&](int t) { emit_diag<R, NMAX>(X + (size_t)(off + t) * ldx, nchunk, N, spk_model, cst, e); };
    if (Te > 0) {
        emit(0);
        V[0] = lb[0] + e[0];   // V[0,1] = ln A01 + E[0,1]   (custom_hmm.py:473)
    }
    BP *bpp = bp + ((size_t)slot * maxT) * Bpad + ul;
    for (int t = 1; t < Te; t++) {
        emit(t);
        unsigned bits = 0;
        // exit state first (reads the old V[N-1]); open only for t >= N (custom_hmm.py:481-485)
        R nx = NINF;
        if (t >= N) {
            R best = NINF;
            R vN = NINF;   // V of the last emitting state, selected without dynamic register indexing
#pragma unroll
            for (int j = 0; j < NMAX; j++) if (j == N - 1) vN = V[j];
            R c_adv = vN + lbN, c_stay = Vx + laX;
            if (c_adv > best) { best = c_adv; bits |= (1u << N); }
            if (c_stay > best) { best = c_stay; bits &= ~(1u << N); }
            nx = best;
        }
        // emitting states, high to low so V[j-1] is still the previous frame's value
#pragma unroll
        for (int j = NMAX - 1; j >= 1; j--) {
            if (j < N) {
                R best = NINF;
                R c_adv = V[j - 1] + lb[j], c_stay = V[j] + la[j + 1];
                bool adv = false;
                if (c_adv > best) { best = c_adv; adv = true; }     // first candidate: j-1 (:488)
                if (c_stay > best) { best = c_stay; adv = false; }
                if (adv) bits |= (1u << j);
                V[j] = (best > NINF) ? best + e[j] : NINF;
            }
        }
        {   // state 1: candidates [1] then, at t == 1 only, the entry state (:477-480)
            R best = NINF;
            R c_stay = V[0] + la[1];
            bool adv = false;
            if (c_stay > best) best = c_stay;
            if (t == 1) {
                R c_ent = R(0) + lb[0];   // V[0,0] = 0
                if (c_ent > best) { best = c_ent; adv = true; }
            }
            if (adv) bits |= 1u;
            V[0] = (best > NINF) ? best + e[0] : NINF;
        }
        Vx = nx;
        if (RENORM) {
            R mx = Vx;
#pragma unroll
            for (int j = 0; j < NMAX; j++) if (j < N) mx = fmax(mx, V[j]);
            if (mx > NINF && mx < R(INFINITY)) {
#pragma unroll
                for (int j = 0; j < NMAX; j++) if (j < N) V[j] -= mx;
                Vx -= mx;
                base += (double)mx;
            }
        }
        bpp[(size_t)t * Bpad] = (BP)bits;
    }
    double sc = (Vx > NINF || Vx != Vx) ? (double)Vx + base : (double)NINF;
    if (Te <= 0) sc = (double)NINF;
    scores[(size_t)ul * nslots + slot] = sc;
}

// argmax over models (strict '>' keeps the first best, decoder.py:44) + back-trace (custom_hmm.py:505-512)
template <typename BP>
__global__ void k_viterbi_finish(const int64_t *__restrict__ offsets, int u0, int nu, int N, int nslots,
                                 const int32_t *__restrict__ model_of_utt, int first_frames,
                                 const BP *__restrict__ bp, int64_t Bpad, int maxT,
                                 const double *__restrict__ scores, int32_t *__restrict__ best_word,
                                 double *__restrict__ best_score, double *__restrict__ scores_out, int M,
                                 uint8_t *__restrict__ best_path, uint8_t *__restrict__ all_paths,
                                 int64_t total_frames) {
    const int ul = blockIdx.x * blockDim.x + threadIdx.x;
    if (ul >= nu) return;
    const int u = u0 + ul;
    const int S = N + 2;
    const int64_t off = offsets[u];
    const int T = (int)(offsets[u + 1] - off);
    const int Te = min((first_frames > 0 && first_frames < T) ? first_frames : T, maxT);
    double bs = -INFINITY;
    int bslot = -1;
    for (int s = 0; s < nslots; s++) {
        double sc = scores[(size_t)ul * nslots + s];
        if (scores_out) scores_out[(size_t)u * nslots + s] = sc;
        if (sc > bs) { bs = sc; bslot = s; }
    }
    if (best_word) best_word[u] = (bslot < 0) ? -1 : (model_of_utt ? model_of_utt[u] : bslot);
    if (best_score) best_score[u] = bs;
    const int wslot = bslot < 0 ? 0 : bslot;
    for (int s = 0; s < nslots; s++) {
        uint8_t *out = all_paths ? all_paths + (size_t)s * total_frames + off : nullptr;
        uint8_t *out2 = (best_path && s == wslot) ? best_path + off : nullptr;
        if (!out) { out = out2; out2 = nullptr; }
        if (!out) continue;
        const bool reachable = scores[(size_t)ul * nslots + s] != -INFINITY;
        const BP *bpp = bp + ((size_t)s * maxT) * Bpad + ul;
        int cur = S - 1;
        for (int t = Te - 1; t >= 0; t--) {
            out[t] = (uint8_t)cur;
            if (out2) out2[t] = (uint8_t)cur;
            if (!reachable) { cur = 0; continue; }     // unreachable cell: backpointer stays 0 (:470)
            if (t == 0) break;
            unsigned bits = (unsigned)bpp[(size_t)t * Bpad];
            if (cur == S - 1) cur = ((bits >> N) & 1u) ? N : S - 1;
            else if (cur >= 1) cur = ((bits >> (cur - 1)) & 1u) ? cur - 1 : cur;
        }
    }
}

__device__ __forceinline__ unsigned ldg_nc_bp(const uint32_t *p) {
    unsigned v;
    asm volatile("ld.global.nc.u32 %0, [%1];" : "=r"(v) : "l"(p));
    return v;
}
__device__ __forceinline__ unsigned ldg_nc_bp(const uint16_t *p) {
    unsigned short v;
    asm volatile("ld.global.nc.u16 %0, [%1];" : "=h"(v) : "l"(p));
    return v;
}

// Fast path of the above for the production call (winner's path only): a warp owns 32 utterances (lane = utterance).
// Back-pointer words of a 32-frame chunk are fetched with 32 independent loads per lane (the address does not depend
// on the state being traced), the traced states are staged in shared memory and written out row by row so every
// store instruction covers 32 consecutive bytes of one utterance's path.
template <typename BP>
__global__ void __launch_bounds__(128)
k_viterbi_finish_fast(const int64_t *__restrict__ offsets, int u0, int nu, int N, int nslots,
                      const int32_t *__restrict__ model_of_utt, int first_frames, const BP *__restrict__ bp, int64_t Bpad,
                      int maxT, const double *__restrict__ scores, int32_t *__restrict__ best_word,
                      double *__restrict__ best_score, double *__restrict__ scores_out, uint8_t *__restrict__ best_path,
                      const int32_t *__restrict__ utt_list = nullptr, const int32_t *__restrict__ utt_count = nullptr,
                      SaprFlag flag = SaprFlag()) {
    constexpr int CH = 32;
    __shared__ uint8_t sp[4][32][CH + 4];
    const int lane = threadIdx.x & 31, w = threadIdx.x >> 5;
    const int ul = blockIdx.x * blockDim.x + threadIdx.x;
    const bool live = ul < (utt_list ? min(*utt_count, nu) : nu);
    const int u = live ? (utt_list ? utt_list[ul] : u0 + ul) : 0;
    const int S = N + 2;
    int64_t off = 0;
    int Te = 0;
    double bs = -INFINITY;
    int bslot = -1;
    if (live) {
        off = offsets[u];
        const int T = (int)(offsets[u + 1] - off);
        Te = min((first_frames > 0 && first_frames < T) ? first_frames : T, maxT);
        double second = -INFINITY;
        for (int s = 0; s < nslots; s++) {
            const double sc = scores[(size_t)ul * nslots + s];
            if (scores_out) scores_out[(size_t)u * nslots + s] = sc;
            if (sc > bs) { second = bs; bs = sc; bslot = s; }
            else if (sc > second) second = sc;
        }
        if (best_word) best_word[u] = (bslot < 0) ? -1 : (model_of_utt ? model_of_utt[u] : bslot);
        if (best_score) best_score[u] = bs;
        sapr_flag_word(flag, u, bs, second);
    }
    if (!best_path) return;
    const int wslot = bslot < 0 ? 0 : bslot;
    const bool reachable = live && scores[(size_t)ul * nslots + wslot] != -INFINITY;
    const BP *bpp = bp + ((size_t)wslot * maxT) * Bpad + (live ? ul : 0);      // loads are unconditional: idle lanes read column 0
    int Tm = Te;
    for (int o = 16; o > 0; o >>= 1) Tm = max(Tm, __shfl_xor_sync(0xffffffffu, Tm, o));
    int cur = S - 1;
    for (int t0 = (Tm - 1) / CH * CH; t0 >= 0; t0 -= CH) {
        // volatile loads + an empty asm that "modifies" the values: every load of the chunk is issued before the first is consumed
        unsigned bits[CH];
#pragma unroll
        for (int j = 0; j < CH; j++) bits[j] = ldg_nc_bp(bpp + (size_t)min(t0 + j, maxT - 1) * Bpad);
#pragma unroll
        for (int j = 0; j < CH; j += 8)
            asm volatile("" : "+r"(bits[j]), "+r"(bits[j + 1]), "+r"(bits[j + 2]), "+r"(bits[j + 3]), "+r"(bits[j + 4]), "+r"(bits[j + 5]),
                         "+r"(bits[j + 6]), "+r"(bits[j + 7]));
#pragma unroll
        for (int j = 0; j < CH; j++) {
            const int t = t0 + j;
            bits[j] = (reachable && t >= 1 && t < Te) ? bits[j] : 0u;
        }
        // one dependent shift / and / subtract per frame, no branch (the trace is the latency of a small launch): bits[] is 0 for
        // frames outside [1, Te), bit c - 1 = state c advanced (exit (S-1) -> N uses bit N), so shifted left by one the entry
        // state's bit is 0 and it stays.  An unreachable winner keeps the exit state in its last frame and 0 before (:470).
#pragma unroll
        for (int j = CH - 1; j >= 0; j--) {
            sp[w][lane][j] = (uint8_t)(reachable ? cur : (t0 + j == Te - 1 ? S - 1 : 0));
            cur -= (int)(((bits[j] << 1) >> cur) & 1u);
        }
        __syncwarp();
        for (int row = 0; row < 32; row++) {
            const int Te_r = __shfl_sync(0xffffffffu, Te, row);
            const int64_t off_r = __shfl_sync(0xffffffffu, off, row);
            if (t0 + lane < Te_r) best_path[off_r + t0 + lane] = sp[w][row][lane];
        }
        __syncwarp();
    }
}

int sapr_viterbi_finish_u16(sapr_ctx *ctx, const int64_t *offsets, int u0, int nu, int N, int nslots, int first_frames,
                            const uint16_t *bp, int64_t Bpad, int maxT, const double *scores, int32_t *best_word,
                            double *best_score, double *scores_out, int M, uint8_t *best_path, uint8_t *all_paths,
                            int64_t total_frames, const SaprFlag *flag) {
    {
        ProfScope ps(ctx, 1);
        if (!all_paths)
            k_viterbi_finish_fast<uint16_t><<<(nu + 127) / 128, 128, 0, ctx->stream>>>(offsets, u0, nu, N, nslots, nullptr, first_frames,
                                                                                       bp, Bpad, maxT, scores, best_word, best_score,
                                                                                       scores_out, best_path, nullptr, nullptr,
                                                                                       flag ? *flag : SaprFlag());
        else
            k_viterbi_finish<uint16_t><<<(nu + 127) / 128, 128, 0, ctx->stream>>>(offsets, u0, nu, N, nslots, nullptr, first_frames, bp,
                                                                                  Bpad, maxT, scores, best_word, best_score,
                                                                                  scores_out, M, best_path, all_paths, total_frames);
    }
    SAPR_LAUNCH_CHECK(ctx);
    return SAPR_OK;
}

template <typename R, typename BP, int NMAX>
static int launch_viterbi(sapr_ctx *ctx, sapr_models *m, const float *X, int ldx, const int64_t *offsets, int B,
                          int64_t total_frames, int max_T, const int32_t *model_of_utt, int first_frames,
                          int32_t *best_word, double *best_score, double *scores, uint8_t *best_path,
                          uint8_t *all_paths) {
    const bool own = model_of_utt != nullptr;
    const int nslots = own ? 1 : m->M;
    const int nchunk = m->Dp / 4;
    const int Tm = (first_frames > 0 && first_frames < max_T) ? first_frames : max_T;
    // chunk the batch so the back-pointer scratch stays <= ~192 MB
    int64_t per_utt = (int64_t)nslots * (Tm > 0 ? Tm : 1) * sizeof(BP);
    int chunk = (int)std::min<int64_t>(B, std::max<int64_t>(32, ((int64_t)192 << 20) / per_utt));
    chunk = (chunk + 31) / 32 * 32;
    const int64_t Bpad = chunk;
    int rc = sapr_ws_reserve(ctx, 0, (size_t)per_utt * Bpad);
    if (rc) return rc;
    rc = sapr_ws_reserve(ctx, 1, (size_t)chunk * nslots * sizeof(double));
    if (rc) return rc;
    BP *bp = (BP *)ctx->ws[0];
    double *sc_ws = (double *)ctx->ws[1];
    const int mpc = own ? 1 : std::min(m->M, 16);
    const int nm_stage = own ? m->M : mpc;
    size_t smem = (size_t)nm_stage * nchunk * m->N * 8 * sizeof(R);
    auto kern = k_viterbi_fused<R, BP, NMAX, std::is_same<R, float>::value>;
    if (smem > 227 * 1024) SAPR_FAIL(ctx, SAPR_E_RANGE, "viterbi: model set does not fit in shared memory");
    SAPR_CUDA(ctx, cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    const R *pk = std::is_same<R, float>::value ? (const R *)m->pk32 : (const R *)m->pk64;
    const R *cst = std::is_same<R, float>::value ? (const R *)m->cst32 : (const R *)m->cst64;
    const R *la = std::is_same<R, float>::value ? (const R *)m->la32 : (const R *)m->la64;
    const R *lb = std::is_same<R, float>::value ? (const R *)m->lb32 : (const R *)m->lb64;
    for (int u0 = 0; u0 < B; u0 += chunk) {
        const int nu = std::min(chunk, B - u0);
        dim3 block(32, mpc), grid((nu + 31) / 32, own ? 1 : (m->M + mpc - 1) / mpc);
        {
            ProfScope ps(ctx, 0);
            kern<<<grid, block, smem, ctx->stream>>>(X, ldx, offsets, u0, nu, m->M, m->N, nchunk, pk, cst, la, lb,
                                                     model_of_utt, first_frames, bp, Bpad, Tm, nslots, sc_ws);
        }
        SAPR_LAUNCH_CHECK(ctx);
        {
            ProfScope ps(ctx, 1);
            if (!all_paths)
                k_viterbi_finish_fast<BP><<<(nu + 127) / 128, 128, 0, ctx->stream>>>(
                    offsets, u0, nu, m->N, nslots, model_of_utt, first_frames, bp, Bpad, Tm, sc_ws, best_word, best_score,
                    scores, best_path);
            else
                k_viterbi_finish<BP><<<(nu + 127) / 128, 128, 0, ctx->stream>>>(
                    offsets, u0, nu, m->N, nslots, model_of_utt, first_frames, bp, Bpad, Tm, sc_ws, best_word, best_score,
                    scores, m->M, best_path, all_paths, total_frames);
        }
        SAPR_LAUNCH_CHECK(ctx);
    }
    return SAPR_OK;
}

// ------------------------------------------------------------------------------------------------
// word exactness of the fp32 production path: flag buffers and the float64 re-decoding of the flagged utterances.
// k_redo_fused, ONE launch behind the fp32 arg-max / back-trace (the list is usually a handful of utterances, so what counts is
// the latency of one list entry: every dependent launch and every dependent memory round trip is on the critical path of
// the whole Viterbi call).  One 256-thread block per (list entry, model):
//   1. emissions: the utterance's features and the model's packed parameters are staged in shared memory with one round of
//      independent loads; one thread per (frame, state) with the fma order of emit_diag<double>; results stay in shared memory
//   2. recursion: warp 0, lane j < N = emitting state j + 1, lane N = exit state; the candidates, their order and the strict
//      comparisons are those of k_viterbi_fused<double> (custom_hmm.py:475-503), so scores and back-pointer words are
//      bit-identical to the verification mode's
//   3. the block that completes an entry's last model (a counter per entry) takes the arg-max over the models and traces the
//      winner's path, overwriting the entry's word, score, score row and path.
__global__ void __launch_bounds__(256) k_redo_fused(const float *__restrict__ X, int ldx, const int64_t *__restrict__ offsets,
                                                    const int32_t *__restrict__ utt_list, const int32_t *__restrict__ utt_count, int cap, int M, int N,
                                                    int nchunk, int maxT, int xs, int first_frames, const double *__restrict__ pk,
                                                    const double *__restrict__ cst_g, const double *__restrict__ la_g, const double *__restrict__ lb_g,
                                                    uint16_t *bp, int64_t Bpad, double *sc, int32_t *done, int32_t *__restrict__ best_word,
                                                    double *__restrict__ best_score, double *__restrict__ scores_out, uint8_t *__restrict__ best_path) {
    extern __shared__ __align__(16) unsigned char s_rd[];
    double *se = reinterpret_cast<double *>(s_rd);                                              // [maxT][8] + a zero slot
    double2 *sp = reinterpret_cast<double2 *>(s_rd + ((size_t)maxT * 8 + 8) * sizeof(double));   // [nchunk][4 fields][8]
    unsigned char *s_x = reinterpret_cast<unsigned char *>(sp) + (size_t)nchunk * 8 * 64;
    float4 *sx = reinterpret_cast<float4 *>(s_x);                                               // [xs frames][nchunk]
    uint16_t *sw = reinterpret_cast<uint16_t *>(s_x);                                           // step 3 reuses the feature slab
    uint8_t *spath = reinterpret_cast<uint8_t *>(sw + maxT);
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5, S = N + 2;
    const double NINF = -INFINITY;
    const int n = min(*utt_count, cap);
    for (int w = blockIdx.x; w < n * M; w += gridDim.x) {
        const int pos = w / M, m = w % M;
        const int u = utt_list[pos];
        const int64_t off = offsets[u];
        const int T = (int)(offsets[u + 1] - off);
        const int Te = min((first_frames > 0 && first_frames < T) ? first_frames : T, maxT);
        __syncthreads();                                  // the previous item is done with the shared memory
        // ---- 1. emissions ----
        // packed parameters [chunk][state][mean01, mean23, weight01, weight23] -> [chunk][field][state]: the eight states of a warp
        // read consecutive 16-byte words (state-major rows 64 bytes apart put states 0, 2, 4, 6 on the same banks)
        const double2 *pm2 = reinterpret_cast<const double2 *>(pk + (size_t)m * nchunk * N * 8);
        for (int idx = tid; idx < nchunk * N * 4; idx += 256) {
            const int q = idx & 3, cj = idx >> 2, c = cj / N, jj = cj - c * N;
            sp[(c * 4 + q) * 8 + jj] = __ldg(pm2 + idx);
        }
        if (tid == 0) se[(size_t)maxT * 8] = 0.0;
        for (int s0 = 0; s0 < Te; s0 += xs) {
            if (s0) __syncthreads();
            const int nf = min(xs, Te - s0);
            for (int idx = tid; idx < nf * nchunk; idx += 256)
                sx[idx] = __ldg(reinterpret_cast<const float4 *>(X + (size_t)(off + s0 + idx / nchunk) * ldx) + idx % nchunk);
            __syncthreads();
            for (int item = tid; item < nf * 8; item += 256) {
                const int t_l = item >> 3, j = item & 7;
                double ev = 0.0;
                if (j < N) {
                    double acc = 0.0;
                    for (int c = 0; c < nchunk; c++) {
                        const float4 xv = sx[t_l * nchunk + c];
                        const double2 *p = sp + (size_t)c * 32 + j;
                        const double2 m01 = p[0], m23 = p[8], w01 = p[16], w23 = p[24];
                        const double d0 = (double)xv.x - m01.x, d1 = (double)xv.y - m01.y, d2 = (double)xv.z - m23.x, d3 = (double)xv.w - m23.y;
                        acc = fma(d0 * d0, w01.x, acc);
                        acc = fma(d1 * d1, w01.y, acc);
                        acc = fma(d2 * d2, w23.x, acc);
                        acc = fma(d3 * d3, w23.y, acc);
                    }
                    ev = cst_g[(size_t)m * N + j] - acc;
                }
                se[(size_t)(s0 + t_l) * 8 + j] = ev;
            }
        }
        __syncthreads();
        if (warp != 0) continue;
        // ---- 2. recursion ----
        double c_in = NINF, c_self = NINF;     // advance arc into this lane's state, its self-loop
        if (lane >= 1 && lane < N) { c_in = lb_g[(size_t)m * S + lane]; c_self = la_g[(size_t)m * S + lane + 1]; }
        else if (lane == 0) { c_in = lb_g[(size_t)m * S]; c_self = la_g[(size_t)m * S + 1]; }         // entry arc, self-loop of state 1
        else if (lane == N) { c_in = lb_g[(size_t)m * S + N]; c_self = la_g[(size_t)m * S + S - 1]; }  // ln A[N, exit], ln A[exit, exit]
        double v = NINF;
        if (lane == 0 && Te > 0) v = c_in + se[0];                                   // V[0, 1] = ln A01 + E[0, 1]
        uint16_t *bpp = bp + ((size_t)m * maxT) * Bpad + pos;
        const int le = lane < 8 ? lane : 0;
        // one instruction stream for all lanes: a = the candidate tried first, b = the second one (replaces on strict > only).
        // States 2..N and the exit try the predecessor first (custom_hmm.py:488: prev_states = [j-1, j]); state 1 tries its
        // self-loop first and the entry state (alive at t == 1 only) second (:477-480).
        const bool adv_first = lane >= 1;
        const bool emits = lane < N;
        if (Te > 1) {      // frame 1: the only one where the entry arc is alive
            const int t = 1;
            const double e = emits ? se[t * 8 + le] : 0.0;
            double up = __shfl_up_sync(0xffffffffu, v, 1);
            if (lane == 0) up = 0.0;                                    // V[0, entry] = 0
            const bool open = lane < N || (lane == N && t >= N);        // the exit state opens at t >= N (:481-485)
            const double c_adv = open ? up + c_in : NINF, c_stay = open ? v + c_self : NINF;
            const double a = adv_first ? c_adv : c_stay, b2 = adv_first ? c_stay : c_adv;
            double best = (a > NINF) ? a : NINF;
            const bool took_b = b2 > best;
            best = took_b ? b2 : best;
            const bool adv = adv_first ? (!took_b && a > NINF) : took_b;
            v = emits ? ((best > NINF) ? best + e : NINF) : best;
            const unsigned bits = __ballot_sync(0xffffffffu, adv && lane <= N);
            if (lane == 0) bpp[(size_t)t * Bpad] = (uint16_t)bits;
        }
        // Frames >= 2, one warp and one dependent chain: the per-lane special cases are folded into the lane's constants so every
        // lane runs the same few instructions.  State 1 has no live predecessor (arc constant -inf: its "advance" candidate is
        // -inf and never taken, which is what trying the self-loop first gives); the exit state's two arcs are -inf until
        // t >= N; lanes past the exit are -inf throughout.  The comparisons and their order are the ones above: advance first,
        // stay replaces it on strict > only; best > -inf <=> one of the two comparisons held.
        {
            const double *pe = emits ? se + le : se + (size_t)maxT * 8;          // non-emitting lanes add the zero slot
            const int estep = emits ? 8 : 0;
            uint16_t *q = bpp + 2 * Bpad;
            auto frames = [&](int t_from, int t_to, const double cin, const double cself) {
#pragma unroll 4
                for (int t = t_from; t < t_to; t++, q += Bpad) {
                    const double e = pe[t * estep];
                    const double up = __shfl_up_sync(0xffffffffu, v, 1);
                    const double c_adv = up + cin, c_stay = v + cself;
                    const bool p1 = c_adv > NINF;
                    const double best0 = p1 ? c_adv : NINF;
                    const bool p2 = c_stay > best0;
                    const double best = p2 ? c_stay : best0;
                    v = (p1 || p2) ? best + e : NINF;
                    const unsigned bits = __ballot_sync(0xffffffffu, p1 && !p2);
                    if (lane == 0) *q = (uint16_t)bits;
                }
            };
            const double cin2 = lane == 0 ? NINF : c_in;
            const int t_open = min(max(N, 2), Te);
            frames(2, t_open, lane == N ? NINF : cin2, lane == N ? NINF : c_self);
            frames(t_open, Te, cin2, c_self);
        }
        if (lane == N) sc[(size_t)pos * M + m] = (Te > 0 && (v > NINF || v != v)) ? v : NINF;
        // ---- 3. the entry's last model: arg-max (strict >, first model wins, NaN never wins: decoder.py:42-47) + back-trace ----
        __threadfence();
        __syncwarp();
        int last = 0;
        if (lane == 0) last = atomicAdd(&done[pos], 1) == M - 1;
        last = __shfl_sync(0xffffffffu, last, 0);
        if (!last) continue;
        __threadfence();
        if (lane == 0) done[pos] = 0;                                        // ready for the next call
        double bs = NINF;
        int bslot = 0x7fffffff;
        for (int s0 = lane; s0 < M; s0 += 32) {
            const double val = __ldcg(sc + (size_t)pos * M + s0);            // written by other blocks: read at the L2
            if (scores_out) scores_out[(size_t)u * M + s0] = val;
            if (val > bs) { bs = val; bslot = s0; }
        }
        for (int o = 16; o > 0; o >>= 1) {
            const double ov = __shfl_xor_sync(0xffffffffu, bs, o);
            const int os = __shfl_xor_sync(0xffffffffu, bslot, o);
            if (ov > bs || (ov == bs && os < bslot)) { bs = ov; bslot = os; }
        }
        if (bslot == 0x7fffffff) bslot = -1;                                 // every score -inf (or NaN)
        if (lane == 0) {
            if (best_word) best_word[u] = bslot;
            if (best_score) best_score[u] = bs;
        }
        if (!best_path) continue;
        const int wslot = bslot < 0 ? 0 : bslot;
        const bool reachable = __ldcg(sc + (size_t)pos * M + wslot) != NINF;
        const uint16_t *wp = bp + ((size_t)wslot * maxT) * Bpad + pos;
        for (int t = lane; t < Te; t += 32) sw[t] = (reachable && t >= 1) ? __ldcg(wp + (size_t)t * Bpad) : (uint16_t)0;
        __syncwarp();
        if (lane == 0) {
            int cur = S - 1;
            // bit c - 1 of a word = state c advanced (exit -> N uses bit N); shifted left by one the entry state's bit is 0 and it stays.
            // An unreachable winner keeps the exit state in its last frame and 0 before (custom_hmm.py:470).
#pragma unroll 8
            for (int t = Te - 1; t >= 0; t--) {
                spath[t] = (uint8_t)(reachable ? cur : (t == Te - 1 ? S - 1 : 0));
                cur -= (int)((((unsigned)sw[t] << 1) >> cur) & 1u);
            }
        }
        __syncwarp();
        for (int t = lane; t < Te; t += 32) best_path[off + t] = spath[t];
    }
}

int sapr_flag_setup(sapr_ctx *ctx, SaprFlag *flag, bool first_chunk) {
    const size_t need = sizeof(int32_t) * (2 * SAPR_FLAG_CAP + 4);      // count, list, per-entry completion counters
    const bool fresh = ctx->ws_bytes[8] < need;      // slot 8 has no other user: the counters survive between calls
    int rc = sapr_ws_reserve(ctx, 8, need);
    if (rc) return rc;
    int32_t *base = (int32_t *)ctx->ws[8];
    if (fresh) SAPR_CUDA(ctx, cudaMemsetAsync(base, 0, need, ctx->stream));      // the counters are left at zero by every launch
    flag->done = base + 4 + SAPR_FLAG_CAP;
    // list capacity: the re-decoding scratch (float64 emissions of every model and frame) stays below 256 MB
    const int64_t per = (int64_t)std::max(ctx->flag_M, 1) * std::max(ctx->flag_maxT, 1) * 8 * (int64_t)sizeof(double);
    flag->count = base; flag->list = base + 4; flag->rel = SAPR_FLAG_REL;
    flag->cap = (int)std::max<int64_t>(32, std::min<int64_t>(SAPR_FLAG_CAP, ((int64_t)256 << 20) / per));
    SAPR_CUDA(ctx, cudaMemsetAsync(base, 0, sizeof(int32_t) * (first_chunk ? 2 : 1), ctx->stream));
    ctx->flag_valid = true;
    return SAPR_OK;
}

// float64 re-decoding of the listed utterances on the context's stream, behind the fp32 arg-max / back-trace whose word, score,
// score row and path it overwrites; the kernel reads the list length on the device (no host round trip)
int sapr_viterbi_redo_flagged(sapr_ctx *ctx, sapr_models *m, const float *X, int ldx, const int64_t *offsets, int first_frames,
                              const SaprFlag &flag, int32_t *best_word, double *best_score, double *scores, uint8_t *best_path) {
    if (m->N > 8) return SAPR_OK;
    const int maxT = ctx->flag_maxT;
    const int Tm = (first_frames > 0 && first_frames < maxT) ? first_frames : maxT;
    const int Tq = Tm > 0 ? Tm : 1, nchunk = m->Dp / 4;
    const int xs = std::min(Tq, 256);
    const size_t x_bytes = std::max((size_t)xs * nchunk * 16, ((size_t)Tq * 3 + 31) / 16 * 16);
    const size_t smem = ((size_t)Tq * 8 + 8) * sizeof(double) + (size_t)nchunk * 8 * 64 + x_bytes;
    if (smem > 220 * 1024) return SAPR_OK;      // utterances too long for the shared-memory emission staging: no re-decoding
    const size_t bp_bytes = ((size_t)m->M * Tq * flag.cap * sizeof(uint16_t) + 255) / 256 * 256;
    const size_t sc_bytes = ((size_t)flag.cap * m->M * sizeof(double) + 255) / 256 * 256;
    int rc = sapr_ws_reserve(ctx, 4, bp_bytes + sc_bytes);
    if (rc) return rc;
    uint16_t *bp = (uint16_t *)ctx->ws[4];
    double *sc = (double *)((char *)ctx->ws[4] + bp_bytes);
    SAPR_CUDA(ctx, cudaFuncSetAttribute(k_redo_fused, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    const int per_sm = (int)std::max<size_t>(1, std::min<size_t>(4, (200 * 1024) / smem));
    ProfScope ps(ctx, 6);
    k_redo_fused<<<per_sm * ctx->sm_count, 256, smem, ctx->stream>>>(X, ldx, offsets, flag.list, flag.count, flag.cap, m->M, m->N, nchunk, Tq, xs,
                                                                     first_frames, m->pk64, m->cst64, m->la64, m->lb64, bp, (int64_t)flag.cap, sc,
                                                                     flag.done, best_word, best_score, scores, best_path);
    SAPR_LAUNCH_CHECK(ctx);
    return SAPR_OK;
}

extern "C" int sapr_viterbi_flagged(sapr_ctx *ctx, int64_t *n) {
    if (!ctx || !n) return SAPR_E_INVALID;
    *n = 0;
    if (!ctx->flag_valid || !ctx->ws[8]) return SAPR_OK;
    int32_t h[2] = {0, 0};
    SAPR_CUDA(ctx, cudaMemcpyAsync(h, ctx->ws[8], sizeof(h), cudaMemcpyDeviceToHost, ctx->stream));
    SAPR_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
    *n = h[1];
    return SAPR_OK;
}

// debug / parity entry: the tensor-core emission tile written out as E[sum_T][ncols] float32
// (ncols = M*8 rounded up to 16; column m*8 + j-1 = state j of model m) -- compute_emission_matrix, custom_hmm.py:146-174
extern "C" int sapr_debug_tc_emission(sapr_ctx *ctx, sapr_models *m, const float *X, int ldx, const int64_t *offsets, int B,
                                      int64_t total_frames, int max_T, float *E_out, int *ncols_out) {
    if (!ctx || !m || !X || !offsets || !E_out) return SAPR_E_INVALID;
    if (!m->valid || !m->tc_image || !sapr_tc_eligible(m)) SAPR_FAIL(ctx, SAPR_E_RANGE, "tc emission: model set not eligible");
    int ncols = 0;
    sapr_tc_image_bytes(m, nullptr, &ncols);
    if (ncols_out) *ncols_out = ncols;
    return sapr_viterbi_tc_launch(ctx, m, X, ldx, offsets, B, total_frames, max_T, 0, nullptr, nullptr, nullptr, nullptr, nullptr,
                                  E_out);
}

extern "C" int sapr_viterbi(sapr_ctx *ctx, sapr_models *m, const float *X, int ldx, const int64_t *offsets, int B,
                            int64_t total_frames, int max_T, const int32_t *model_of_utt, int precision,
                            int first_frames, int32_t *best_word, double *best_score, double *scores,
                            uint8_t *best_path, uint8_t *all_paths) {
    if (!ctx || !m || !X || !offsets) return SAPR_E_INVALID;
    if (!m->valid) SAPR_FAIL(ctx, SAPR_E_INVALID, "viterbi: model parameters not set");
    if (m->topology == SAPR_TOPO_DENSE)
        return sapr_viterbi_dense(ctx, m, X, ldx, offsets, B, total_frames, max_T, model_of_utt, precision, first_frames, best_word,
                                  best_score, scores, best_path, all_paths);
    if (m->emission != SAPR_EMIT_DIAG || m->topology != SAPR_TOPO_ENTRY_EXIT)
        SAPR_FAIL(ctx, SAPR_E_INVALID, "viterbi: fused kernel needs DIAG emission + ENTRY_EXIT topology");
    if (ldx % 4 || ldx < m->Dp) SAPR_FAIL(ctx, SAPR_E_INVALID, "viterbi: ldx must be a multiple of 4 and >= D padded");
    if (B <= 0) return SAPR_OK;
    if (max_T <= 0) SAPR_FAIL(ctx, SAPR_E_INVALID, "viterbi: max_T must be positive");
    ctx->flag_valid = false;
#define GO(R, BP, NM)                                                                                       \
    return launch_viterbi<R, BP, NM>(ctx, m, X, ldx, offsets, B, total_frames, max_T, model_of_utt,        \
                                     first_frames, best_word, best_score, scores, best_path, all_paths)
    if (precision == SAPR_FP32 && !model_of_utt && m->tc_image && sapr_tc_eligible(m))
        return sapr_viterbi_tc_launch(ctx, m, X, ldx, offsets, B, total_frames, max_T, first_frames, best_word, best_score,
                                      scores, best_path, all_paths, nullptr);
    if (precision == SAPR_FP32 || precision == SAPR_FP32_SIMT) {
        if (m->N <= 8) GO(float, uint16_t, 8);
        if (m->N <= 15) GO(float, uint16_t, 15);
        if (m->N <= 31) GO(float, uint32_t, 31);
    } else {
        if (m->N <= 8) GO(double, uint16_t, 8);
        if (m->N <= 15) GO(double, uint16_t, 15);
        if (m->N <= 31) GO(double, uint32_t, 31);
    }
#undef GO
    SAPR_FAIL(ctx, SAPR_E_RANGE, "viterbi: N > 31 emitting states not supported by the left-to-right kernel");
}
