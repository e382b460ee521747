// api.cu -- context / model-set lifetime, workspace, and the derived-parameter kernels.
#include "common.cuh"

extern "C" int sapr_version(void) { return 103; }

extern "C" int sapr_ctx_create(int device, void *cuda_stream, sapr_ctx **out) {
    if (!out) return SAPR_E_INVALID;
    *out = nullptr;
    int ndev = 0;
    if (cudaGetDeviceCount(&ndev) != cudaSuccess || ndev <= 0) return SAPR_E_CUDA;   // no GPU: fail loudly
    if (device < 0 || device >= ndev) return SAPR_E_INVALID;
    if (cudaSetDevice(device) != cudaSuccess) return SAPR_E_CUDA;
    sapr_ctx *c = new sapr_ctx();
    c->device = device;
    c->stream = (cudaStream_t)cuda_stream;
    cudaDeviceProp prop;
    if (cudaGetDeviceProperties(&prop, device) == cudaSuccess) c->sm_count = prop.multiProcessorCount;
    if (cudaStreamCreateWithFlags(&c->copy_stream, cudaStreamNonBlocking) != cudaSuccess) { delete c; return SAPR_E_CUDA; }
    if (cudaStreamCreateWithFlags(&c->aux_stream, cudaStreamNonBlocking) != cudaSuccess) { delete c; return SAPR_E_CUDA; }
    for (int i = 0; i < 10; i++)
        if (cudaEventCreateWithFlags(&c->ev[i], cudaEventDisableTiming) != cudaSuccess) { delete c; return SAPR_E_CUDA; }
    *out = c;
    return SAPR_OK;
}

extern "C" int sapr_ctx_destroy(sapr_ctx *ctx) {
    if (!ctx) return SAPR_OK;
    cudaSetDevice(ctx->device);
    cudaStreamSynchronize(ctx->stream);
    for (int i = 0; i < 10; i++) if (ctx->ws[i]) cudaFree(ctx->ws[i]);
    for (int i = 0; i < 4; i++) if (ctx->pin[i]) cudaFreeHost(ctx->pin[i]);
    for (int i = 0; i < 10; i++) if (ctx->ev[i]) cudaEventDestroy(ctx->ev[i]);
    for (auto &r : ctx->prof) { cudaEventDestroy(r.a); cudaEventDestroy(r.b); }
    for (auto &r : ctx->prof_pool) { cudaEventDestroy(r.a); cudaEventDestroy(r.b); }
    if (ctx->copy_stream) cudaStreamDestroy(ctx->copy_stream);
    if (ctx->aux_stream) { cudaStreamSynchronize(ctx->aux_stream); cudaStreamDestroy(ctx->aux_stream); }
    delete ctx;
    return SAPR_OK;
}

extern "C" const char *sapr_last_error(sapr_ctx *ctx) { return ctx ? ctx->err.c_str() : "null ctx"; }
extern "C" int64_t sapr_launch_count(sapr_ctx *ctx) { return ctx ? ctx->launches : 0; }
extern "C" int sapr_sync(sapr_ctx *ctx) {
    if (!ctx) return SAPR_E_INVALID;
    SAPR_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
    return SAPR_OK;
}

extern "C" int sapr_profile(sapr_ctx *ctx, int enable) {
    if (!ctx) return SAPR_E_INVALID;
    SAPR_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
    for (auto &r : ctx->prof) ctx->prof_pool.push_back(r);
    ctx->prof.clear();
    ctx->profiling = enable != 0;
    return SAPR_OK;
}

extern "C" int sapr_profile_read(sapr_ctx *ctx, int which, double *ms, int64_t *launches) {
    if (!ctx || !ms || !launches) return SAPR_E_INVALID;
    SAPR_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
    double tot = 0.0;
    int64_t n = 0;
    for (auto &r : ctx->prof)
        if (r.which == which) {
            float t = 0.f;
            SAPR_CUDA(ctx, cudaEventElapsedTime(&t, r.a, r.b));
            tot += t; n++;
        }
    *ms = tot; *launches = n;
    return SAPR_OK;
}

int sapr_ws_reserve(sapr_ctx *ctx, int slot, size_t bytes) {
    if (bytes <= ctx->ws_bytes[slot]) return SAPR_OK;
    // the old buffer may still be in use by queued kernels: drain the stream before releasing it
    SAPR_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
    if (ctx->ws[slot]) { cudaFree(ctx->ws[slot]); ctx->ws[slot] = nullptr; ctx->ws_bytes[slot] = 0; }
    size_t want = bytes + (bytes >> 3) + 256;
    cudaError_t e = cudaMalloc(&ctx->ws[slot], want);
    if (e != cudaSuccess) {
        cudaGetLastError();
        want = bytes;
        e = cudaMalloc(&ctx->ws[slot], want);
        if (e != cudaSuccess) { cudaGetLastError(); SAPR_FAIL(ctx, SAPR_E_NOMEM, "workspace allocation failed"); }
    }
    ctx->ws_bytes[slot] = want;
    return SAPR_OK;
}

int sapr_pin_reserve(sapr_ctx *ctx, int slot, size_t bytes) {
    if (bytes <= ctx->pin_bytes[slot]) return SAPR_OK;
    SAPR_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
    SAPR_CUDA(ctx, cudaStreamSynchronize(ctx->copy_stream));
    if (ctx->pin[slot]) { cudaFreeHost(ctx->pin[slot]); ctx->pin[slot] = nullptr; ctx->pin_bytes[slot] = 0; }
    if (cudaMallocHost(&ctx->pin[slot], bytes) != cudaSuccess) { cudaGetLastError(); SAPR_FAIL(ctx, SAPR_E_NOMEM, "pinned allocation failed"); }
    ctx->pin_bytes[slot] = bytes;
    return SAPR_OK;
}

// ----------------------------------------------------------------------------------------------
template <typename T> static int dalloc(sapr_ctx *ctx, T **p, size_t n) {
    SAPR_CUDA(ctx, cudaMalloc((void **)p, sizeof(T) * (n ? n : 1)));
    SAPR_CUDA(ctx, cudaMemsetAsync(*p, 0, sizeof(T) * (n ? n : 1), ctx->stream));
    return SAPR_OK;
}

extern "C" int sapr_models_create(sapr_ctx *ctx, int M, int N, int D, int emission, int topology, sapr_models **out) {
    if (!ctx || !out) return SAPR_E_INVALID;
    *out = nullptr;
    if (M <= 0 || N <= 0 || D <= 0) SAPR_FAIL(ctx, SAPR_E_INVALID, "models_create: M, N, D must be positive");
    if (emission != SAPR_EMIT_DIAG && emission != SAPR_EMIT_SAPR) SAPR_FAIL(ctx, SAPR_E_INVALID, "models_create: bad emission");
    if (topology != SAPR_TOPO_ENTRY_EXIT && topology != SAPR_TOPO_DENSE) SAPR_FAIL(ctx, SAPR_E_INVALID, "models_create: bad topology");
    if (emission == SAPR_EMIT_SAPR && D > 64) SAPR_FAIL(ctx, SAPR_E_RANGE, "models_create: SAPR emission supports D <= 64");
    sapr_models *m = new sapr_models();
    m->ctx = ctx; m->M = M; m->N = N; m->D = D; m->emission = emission; m->topology = topology;
    // ENTRY_EXIT: N emitting states + entry + exit.  DENSE: the caller passes the total number of
    // (all-emitting) states as N, so S = N (hmmlearn_hmm.py:28 uses n_components = num_states + 2).
    m->S = (topology == SAPR_TOPO_ENTRY_EXIT) ? N + 2 : N;
    m->n_emit = (topology == SAPR_TOPO_ENTRY_EXIT) ? N : m->S;
    m->Dp = (D + 3) / 4 * 4;
    const size_t S = m->S, ne = m->n_emit, nch = m->Dp / 4;
    const size_t covn = (emission == SAPR_EMIT_DIAG) ? (size_t)M * S * D : (size_t)M * S * D * D;
    int rc = 0;
    rc |= dalloc(ctx, &m->mean, (size_t)M * S * D);
    rc |= dalloc(ctx, &m->cov, covn);
    rc |= dalloc(ctx, &m->A, (size_t)M * S * S);
    rc |= dalloc(ctx, &m->pi, (size_t)M * S);
    rc |= dalloc(ctx, &m->logA, (size_t)M * S * S);
    rc |= dalloc(ctx, &m->logpi, (size_t)M * S);
    rc |= dalloc(ctx, &m->la64, (size_t)M * S);
    rc |= dalloc(ctx, &m->lb64, (size_t)M * S);
    rc |= dalloc(ctx, &m->la32, (size_t)M * S);
    rc |= dalloc(ctx, &m->lb32, (size_t)M * S);
    if (emission == SAPR_EMIT_DIAG) {
        rc |= dalloc(ctx, &m->pk64, (size_t)M * nch * ne * 8);
        rc |= dalloc(ctx, &m->pk32, (size_t)M * nch * ne * 8);
        rc |= dalloc(ctx, &m->cst64, (size_t)M * ne);
        rc |= dalloc(ctx, &m->cst32, (size_t)M * ne);
    } else {
        rc |= dalloc(ctx, &m->P, (size_t)M * S * D * D);
        rc |= dalloc(ctx, &m->cstS, (size_t)M * S);
    }
    if (!rc && emission == SAPR_EMIT_DIAG && topology == SAPR_TOPO_DENSE && S <= 32 && m->Dp <= 1024) {
        float2 *arc = nullptr, *arcs = nullptr;
        rc |= dalloc(ctx, &m->dn_piv, (size_t)m->Dp);
        rc |= dalloc(ctx, &m->dn_w, (size_t)M * nch * S * 8);
        rc |= dalloc(ctx, &m->dn_cst, (size_t)M * S);
        rc |= dalloc(ctx, &m->dn_lpi, (size_t)M * S);
        rc |= dalloc(ctx, &arc, (size_t)M * S * S);
        rc |= dalloc(ctx, &m->dn_start, (size_t)M * (S + 1));
        rc |= dalloc(ctx, &arcs, (size_t)M * S * S);
        rc |= dalloc(ctx, &m->dn_starts, (size_t)M * (S + 1));
        m->dn_arc = arc; m->dn_arcs = arcs;
    }
    if (!rc && sapr_tc_eligible(m)) {
        unsigned char *img = nullptr;
        rc |= dalloc(ctx, &img, sapr_tc_image_bytes(m, nullptr, nullptr));
        m->tc_image = img;
    }
    if (rc) { sapr_models_destroy(m); return SAPR_E_CUDA; }
    *out = m;
    return SAPR_OK;
}

extern "C" int sapr_models_destroy(sapr_models *m) {
    if (!m) return SAPR_OK;
    cudaStreamSynchronize(m->ctx->stream);
    void *ptrs[] = {m->mean, m->cov, m->A, m->pi, m->logA, m->logpi, m->la64, m->lb64, m->la32, m->lb32,
                    m->pk64, m->pk32, m->cst64, m->cst32, m->P, m->cstS, m->tc_image, m->dn_piv, m->dn_w, m->dn_cst,
                    m->dn_lpi, m->dn_arc, m->dn_start, m->dn_arcs, m->dn_starts};
    for (void *p : ptrs) if (p) cudaFree(p);
    delete m;
    return SAPR_OK;
}

extern "C" int sapr_models_set(sapr_models *m, const double *means, const double *covars, const double *transmat,
                               const double *startprob) {
    if (!m || !means || !covars || !transmat) return SAPR_E_INVALID;
    sapr_ctx *ctx = m->ctx;
    const size_t S = m->S, D = m->D, M = m->M;
    const size_t covn = (m->emission == SAPR_EMIT_DIAG) ? M * S * D : M * S * D * D;
    SAPR_CUDA(ctx, cudaMemcpyAsync(m->mean, means, sizeof(double) * M * S * D, cudaMemcpyHostToDevice, ctx->stream));
    SAPR_CUDA(ctx, cudaMemcpyAsync(m->cov, covars, sizeof(double) * covn, cudaMemcpyHostToDevice, ctx->stream));
    SAPR_CUDA(ctx, cudaMemcpyAsync(m->A, transmat, sizeof(double) * M * S * S, cudaMemcpyHostToDevice, ctx->stream));
    if (m->topology == SAPR_TOPO_DENSE) {
        if (!startprob) SAPR_FAIL(ctx, SAPR_E_INVALID, "models_set: DENSE topology needs startprob");
        SAPR_CUDA(ctx, cudaMemcpyAsync(m->pi, startprob, sizeof(double) * M * S, cudaMemcpyHostToDevice, ctx->stream));
    }
    SAPR_CUDA(ctx, cudaStreamSynchronize(ctx->stream));   // host buffers are pageable caller memory
    return sapr_models_prepare(m);
}

extern "C" int sapr_models_get(sapr_models *m, double *means, double *covars, double *transmat, double *startprob) {
    if (!m) return SAPR_E_INVALID;
    sapr_ctx *ctx = m->ctx;
    const size_t S = m->S, D = m->D, M = m->M;
    const size_t covn = (m->emission == SAPR_EMIT_DIAG) ? M * S * D : M * S * D * D;
    if (means) SAPR_CUDA(ctx, cudaMemcpyAsync(means, m->mean, sizeof(double) * M * S * D, cudaMemcpyDeviceToHost, ctx->stream));
    if (covars) SAPR_CUDA(ctx, cudaMemcpyAsync(covars, m->cov, sizeof(double) * covn, cudaMemcpyDeviceToHost, ctx->stream));
    if (transmat) SAPR_CUDA(ctx, cudaMemcpyAsync(transmat, m->A, sizeof(double) * M * S * S, cudaMemcpyDeviceToHost, ctx->stream));
    if (startprob) SAPR_CUDA(ctx, cudaMemcpyAsync(startprob, m->pi, sizeof(double) * M * S, cudaMemcpyDeviceToHost, ctx->stream));
    SAPR_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
    return SAPR_OK;
}

// ----------------------------------------------------------------------------------------------
// derived parameters
__global__ void k_prepare_trans(int M, int S, const double *__restrict__ A, const double *__restrict__ pi,
                                double *__restrict__ logA, double *__restrict__ logpi, double *__restrict__ la64,
                                double *__restrict__ lb64, float *__restrict__ la32, float *__restrict__ lb32) {
    const int idx = blockIdx.x * blockDim.x + threadIdx.x;
    if (idx < M * S * S) logA[idx] = log(A[idx]);
    if (idx < M * S) {
        const int m = idx / S, j = idx % S;
        logpi[idx] = log(pi[idx]);
        const double *Am = A + (size_t)m * S * S;
        const double a = log(Am[(size_t)j * S + j]);
        const double b = (j + 1 < S) ? log(Am[(size_t)j * S + j + 1]) : -INFINITY;
        la64[idx] = a; lb64[idx] = b; la32[idx] = (float)a; lb32[idx] = (float)b;
    }
}

// one thread per (model, emitting state): constant + packed (mu, 0.5/var) chunks
__global__ void k_prepare_diag(int M, int S, int D, int Dp, int n_emit, int first_state, const double *__restrict__ mean,
                               const double *__restrict__ var, double *__restrict__ pk64, float *__restrict__ pk32,
                               double *__restrict__ cst64, float *__restrict__ cst32) {
    const int idx = blockIdx.x * blockDim.x + threadIdx.x;
    if (idx >= M * n_emit) return;
    const int m = idx / n_emit, e = idx % n_emit, j = e + first_state;
    const double *mu = mean + ((size_t)m * S + j) * D;
    const double *vr = var + ((size_t)m * S + j) * D;
    double ld = 0.0;
    for (int d = 0; d < D; d++) ld += log(vr[d]);
    const double c = -0.5 * (D * SAPR_LOG2PI + ld);
    cst64[idx] = c; cst32[idx] = (float)c;
    const int nch = Dp / 4;
    for (int ch = 0; ch < nch; ch++) {
        const size_t o = (((size_t)m * nch + ch) * n_emit + e) * 8;
        for (int k = 0; k < 4; k++) {
            const int d = ch * 4 + k;
            const double mv = (d < D) ? mu[d] : 0.0;
            const double hv = (d < D) ? 0.5 / vr[d] : 0.0;
            pk64[o + k] = mv; pk64[o + 4 + k] = hv;
            pk32[o + k] = (float)mv; pk32[o + 4 + k] = (float)hv;
        }
    }
}

// custom_hmm.py:160-165 -- P = inv(cov + 1e-6 I), logdet via LU with partial pivoting (what LAPACK
// getrf does behind np.linalg.inv / slogdet).  One thread per (model, emitting state); D <= 64.
__global__ void k_prepare_sapr(int M, int S, int D, const double *__restrict__ cov, double *__restrict__ lu_ws,
                               double *__restrict__ P, double *__restrict__ cstS) {
    const int idx = blockIdx.x * blockDim.x + threadIdx.x;
    if (idx >= M * S) return;
    const int j = idx % S;
    if (j == 0 || j == S - 1) { cstS[idx] = -INFINITY; return; }
    const double *c = cov + (size_t)idx * D * D;
    double *a = lu_ws + (size_t)idx * D * D;
    double *inv = P + (size_t)idx * D * D;
    int piv[64];
    double col[64];
    for (int r = 0; r < D; r++)
        for (int q = 0; q < D; q++) a[r * D + q] = c[r * D + q] + (r == q ? 1e-6 : 0.0);
    double logabsdet = 0.0;
    for (int k = 0; k < D; k++) {
        int p = k;
        double best = fabs(a[k * D + k]);
        for (int i = k + 1; i < D; i++) {
            double v = fabs(a[i * D + k]);
            if (v > best) { best = v; p = i; }
        }
        piv[k] = p;
        if (p != k)
            for (int q = 0; q < D; q++) { double t = a[k * D + q]; a[k * D + q] = a[p * D + q]; a[p * D + q] = t; }
        const double dd = a[k * D + k];
        logabsdet += log(fabs(dd));
        for (int i = k + 1; i < D; i++) {
            a[i * D + k] /= dd;
            const double l = a[i * D + k];
            for (int q = k + 1; q < D; q++) a[i * D + q] -= l * a[k * D + q];
        }
    }
    for (int cc = 0; cc < D; cc++) {
        for (int i = 0; i < D; i++) col[i] = (i == cc) ? 1.0 : 0.0;
        for (int k = 0; k < D; k++)
            if (piv[k] != k) { double t = col[k]; col[k] = col[piv[k]]; col[piv[k]] = t; }
        for (int i = 0; i < D; i++)
            for (int q = 0; q < i; q++) col[i] -= a[i * D + q] * col[q];
        for (int i = D - 1; i >= 0; i--) {
            for (int q = i + 1; q < D; q++) col[i] -= a[i * D + q] * col[q];
            col[i] /= a[i * D + i];
        }
        for (int i = 0; i < D; i++) inv[i * D + cc] = col[i];
    }
    cstS[idx] = -0.5 * (D * SAPR_LOG2PI + logabsdet);
}

int sapr_models_prepare(sapr_models *m) {
    sapr_ctx *ctx = m->ctx;
    const int M = m->M, S = m->S, D = m->D;
    const int nt = M * S * S;
    k_prepare_trans<<<(nt + 127) / 128, 128, 0, ctx->stream>>>(M, S, m->A, m->pi, m->logA, m->logpi, m->la64, m->lb64,
                                                              m->la32, m->lb32);
    SAPR_LAUNCH_CHECK(ctx);
    if (m->emission == SAPR_EMIT_DIAG) {
        const int first = (m->topology == SAPR_TOPO_ENTRY_EXIT) ? 1 : 0;
        k_prepare_diag<<<(M * m->n_emit + 63) / 64, 64, 0, ctx->stream>>>(M, S, D, m->Dp, m->n_emit, first, m->mean,
                                                                          m->cov, m->pk64, m->pk32, m->cst64, m->cst32);
        SAPR_LAUNCH_CHECK(ctx);
        if (m->tc_image) {
            int rc = sapr_tc_prepare(m);
            if (rc) return rc;
        }
        if (m->dn_w) {
            int rc = sapr_dense_prepare(m);
            if (rc) return rc;
        }
    } else {
        int rc = sapr_ws_reserve(ctx, 6, sizeof(double) * (size_t)M * S * D * D);
        if (rc) return rc;
        k_prepare_sapr<<<(M * S + 31) / 32, 32, 0, ctx->stream>>>(M, S, D, m->cov, (double *)ctx->ws[6], m->P, m->cstS);
        SAPR_LAUNCH_CHECK(ctx);
    }
    m->valid = true;
    return SAPR_OK;
}

// ----------------------------------------------------------------------------------------------
// flat start sums (custom_hmm.py:70-92): out = [sum (x-p) (D) | sum (x-p)^2 (D) | frames | utterances]
__global__ void k_init_stats(const float *__restrict__ X, int ldx, int64_t total_frames, int D,
                             const double *__restrict__ pivot, double *__restrict__ partial) {
    // grid.x CTAs, blockDim = (Dpad32, rows): each thread strides over frames for one dim
    const int d = threadIdx.x;
    const int64_t stride = (int64_t)gridDim.x * blockDim.y;
    double s1 = 0.0, s2 = 0.0;
    const double p = (pivot && d < D) ? pivot[d] : 0.0;
    if (d < D)
        for (int64_t f = (int64_t)blockIdx.x * blockDim.y + threadIdx.y; f < total_frames; f += stride) {
            const double x = (double)X[f * ldx + d] - p;
            s1 += x; s2 += x * x;
        }
    extern __shared__ double s_part[];   // [rows][2][Dx]
    const int Dx = blockDim.x;
    s_part[(threadIdx.y * 2 + 0) * Dx + d] = s1;
    s_part[(threadIdx.y * 2 + 1) * Dx + d] = s2;
    __syncthreads();
    if (threadIdx.y == 0 && d < D) {
        double a = 0.0, b = 0.0;
        for (int r = 0; r < (int)blockDim.y; r++) { a += s_part[(r * 2 + 0) * Dx + d]; b += s_part[(r * 2 + 1) * Dx + d]; }
        partial[((size_t)blockIdx.x * 2 + 0) * D + d] = a;
        partial[((size_t)blockIdx.x * 2 + 1) * D + d] = b;
    }
}

__global__ void k_init_stats_final(const double *__restrict__ partial, int nblk, int D, int64_t total_frames, int B,
                                   double *__restrict__ out) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i < 2 * D) {
        const int k = i / D, d = i % D;
        double s = 0.0;
        for (int b = 0; b < nblk; b++) s += partial[((size_t)b * 2 + k) * D + d];
        out[i] = s;
    }
    if (i == 0) { out[2 * D] = (double)total_frames; out[2 * D + 1] = (double)B; }
}

extern "C" int sapr_init_stats(sapr_ctx *ctx, const float *X, int ldx, const int64_t *offsets, int B, int D,
                               const double *pivot, double *out) {
    if (!ctx || !X || !offsets || !out || B <= 0 || D <= 0) return SAPR_E_INVALID;
    if (D > 1024) SAPR_FAIL(ctx, SAPR_E_RANGE, "init_stats: D > 1024");
    int64_t total = 0;
    SAPR_CUDA(ctx, cudaMemcpyAsync(&total, offsets + B, sizeof(int64_t), cudaMemcpyDeviceToHost, ctx->stream));
    SAPR_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
    const int Dx = (D + 31) / 32 * 32;
    const int rows = std::max(1, 256 / Dx);
    int nblk = (int)std::min<int64_t>(4 * ctx->sm_count, (total + rows - 1) / rows);
    if (nblk < 1) nblk = 1;
    int rc = sapr_ws_reserve(ctx, 5, sizeof(double) * (size_t)nblk * 2 * D);
    if (rc) return rc;
    dim3 blk(Dx, rows);
    k_init_stats<<<nblk, blk, sizeof(double) * rows * 2 * Dx, ctx->stream>>>(X, ldx, total, D, pivot, (double *)ctx->ws[5]);
    SAPR_LAUNCH_CHECK(ctx);
    k_init_stats_final<<<(2 * D + 127) / 128, 128, 0, ctx->stream>>>((const double *)ctx->ws[5], nblk, D, total, B, out);
    SAPR_LAUNCH_CHECK(ctx);
    return SAPR_OK;
}

// ----------------------------------------------------------------------------------------------
// evaluation metrics on the device (assignment2/eval.py:28-38: confusion_matrix + accuracy_score over the label indices):
// cm[t][p] counts (true word t, predicted word p); an utterance with no reachable model (predicted -1) goes to column M.
__global__ void k_confusion(const int32_t *__restrict__ truth, const int32_t *__restrict__ pred, int B, int M,
                            unsigned long long *__restrict__ cm, unsigned long long *__restrict__ correct) {
    extern __shared__ unsigned int s_cm[];          // [M][M + 1] per CTA, flushed with one atomic per cell
    const int cells = M * (M + 1);
    for (int i = threadIdx.x; i < cells + 1; i += blockDim.x) s_cm[i] = 0;
    __syncthreads();
    for (int u = blockIdx.x * blockDim.x + threadIdx.x; u < B; u += gridDim.x * blockDim.x) {
        const int t = truth[u];
        int q = pred[u];
        if (t < 0 || t >= M) continue;
        if (q < 0 || q >= M) q = M;
        atomicAdd(&s_cm[t * (M + 1) + q], 1u);
        if (q == t) atomicAdd(&s_cm[cells], 1u);
    }
    __syncthreads();
    for (int i = threadIdx.x; i < cells; i += blockDim.x)
        if (s_cm[i]) atomicAdd(&cm[i], (unsigned long long)s_cm[i]);
    if (threadIdx.x == 0 && s_cm[cells]) atomicAdd(correct, (unsigned long long)s_cm[cells]);
}

extern "C" int sapr_confusion(sapr_ctx *ctx, const int32_t *truth, const int32_t *pred, int B, int M, int64_t *cm, int64_t *correct) {
    if (!ctx || !truth || !pred || !cm || !correct || M <= 0 || B < 0) return SAPR_E_INVALID;
    if ((size_t)(M * (M + 1) + 1) * sizeof(unsigned int) > 48 * 1024) SAPR_FAIL(ctx, SAPR_E_RANGE, "confusion: vocabulary too large (M <= 109)");
    SAPR_CUDA(ctx, cudaMemsetAsync(cm, 0, sizeof(int64_t) * (size_t)M * (M + 1), ctx->stream));
    SAPR_CUDA(ctx, cudaMemsetAsync(correct, 0, sizeof(int64_t), ctx->stream));
    if (B == 0) return SAPR_OK;
    const int grid = std::max(1, std::min(ctx->sm_count, (B + 255) / 256));
    k_confusion<<<grid, 256, (size_t)(M * (M + 1) + 1) * sizeof(unsigned int), ctx->stream>>>(truth, pred, B, M, (unsigned long long *)cm,
                                                                                              (unsigned long long *)correct);
    SAPR_LAUNCH_CHECK(ctx);
    return SAPR_OK;
}
