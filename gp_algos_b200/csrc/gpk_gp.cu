// gpk_gp.cu -- C ABI (include/gpk.h), part 2: the fused GpPredictor pipelines
//   gpk_gp_fit            gp/regression/GpPredictor.scala:104-124 + :144-149
//   gpk_gp_nll_grad       gp/regression/GpPredictor.scala:60-80
//   gpk_gp_model_* / gpk_gp_predict   GpPredictor.scala:24-58 and the GP-UKF call pattern (GPUnscentedKalmanFilter.scala:77-147)
//   *_batched             B independent GPs of one shape per call (MLE restarts, one GP per state dimension)
// One code path serves single and batched problems: every kernel below takes a batch count, so B problems of size n
// cost the same number of launches as one.  K, L, L^-1, K^-1 never leave the device.
#include "gpk_internal.cuh"

#include <stdlib.h>

#include <new>

namespace {

// Per-problem working set of the fused pipelines.
struct Work {
    int N, B;          // padded size, problems resident at once
    double *A, *Li, *T, *ypad, *z, *alpha, *scratch;
    size_t sT, sScratch;  // per-problem strides (doubles) of T and scratch
    ProblemParams* pp_dev;
    int* info_dev;
};

size_t per_problem_doubles(int N, int D, size_t* sT, size_t* sScr) {
    *sT = gpk_chol_scratch_doubles(N);
    const size_t trmv = gpk_trmv_scratch_doubles(N);
    const size_t grad = gpk_grad_scratch_doubles(N, D);
    *sScr = trmv > grad ? trmv : grad;
    return (size_t)2 * N * N + *sT + (size_t)3 * N + *sScr;
}

int make_work(gpk_handle h, int n, int D, int Bwant, Work* w) {
    const int N = gpk_pad(n);
    size_t sT, sScr;
    const size_t per = per_problem_doubles(N, D, &sT, &sScr) * sizeof(double);
    int B = Bwant;
    if ((size_t)B * per > batch_budget_bytes()) B = (int)(batch_budget_bytes() / per);
    if (B < 1) B = 1;
    ARENA_OR_FAIL(A, double*, h, ARENA_A, (size_t)B * N * N * sizeof(double));
    ARENA_OR_FAIL(Li, double*, h, ARENA_B, (size_t)B * N * N * sizeof(double));
    ARENA_OR_FAIL(T, double*, h, ARENA_T, (size_t)B * sT * sizeof(double));
    ARENA_OR_FAIL(m, double*, h, ARENA_MISC, (size_t)B * ((size_t)3 * N + sScr) * sizeof(double));
    ARENA_OR_FAIL(pp_dev, ProblemParams*, h, ARENA_PP, (size_t)B * sizeof(ProblemParams));
    ARENA_OR_FAIL(info_dev, int*, h, ARENA_INFO, (size_t)B * sizeof(int));
    w->N = N; w->B = B; w->sT = sT; w->sScratch = sScr;
    w->A = A; w->Li = Li; w->T = T; w->pp_dev = pp_dev; w->info_dev = info_dev;
    w->ypad = m;
    w->z = m + (size_t)B * N;
    w->alpha = m + (size_t)2 * B * N;
    w->scratch = m + (size_t)3 * B * N;
    return GPK_OK;
}

// host staging of per-problem hyper-parameters; returns the by-value params of problem 0 in *first
int stage_params(gpk_handle h, const double* thetas, int D, int has_s, double s, int B, ProblemParams* dev, ProblemParams* first) {
    const size_t bytes = (size_t)B * sizeof(ProblemParams);
    if (h->pp_host_bytes < bytes) {
        free(h->pp_host);
        h->pp_host = malloc(bytes);
        h->pp_host_bytes = h->pp_host ? bytes : 0;
        if (!h->pp_host) return gpk_set_error(h, GPK_ENOMEM, "host allocation failed");
    }
    ProblemParams* hp = (ProblemParams*)h->pp_host;
    for (int b = 0; b < B; ++b) {
        int rc = gpk_make_problem_params(h, thetas + (size_t)b * gpk_theta_len(h, D), D, has_s, s, &hp[b]);
        if (rc) return rc;
    }
    *first = hp[0];
    if (B > 1) {
        // pageable source: the runtime stages the bytes before returning, so pp_host may be reused by the next call
        GPK_CUDA(h, cudaMemcpyAsync(dev, hp, bytes, cudaMemcpyHostToDevice, h->stream));
    }
    return GPK_OK;
}

// K -> L^-1 (and L when keep_L), alpha, ll for `B` resident problems.  X, y on the device.
int fit_core(gpk_handle h, const Work& w, int B, const double* dX, int n, int D, int64_t ldx, int64_t strideX, const double* dy,
             const ProblemParams& pp0, int keep_L, double* Li, double* alpha, double* ll_dev, int64_t ll_stride, int* info_dev,
             double* Kinv = nullptr, cudaEvent_t* kinv_done = nullptr, bool params_on_device = false) {
    const ProblemParams* ppd = (B > 1 || params_on_device) ? w.pp_dev : nullptr;
    int rc = gpk_cov_sym_lower_padded(h, dX, n, ldx, pp0.cp, w.A, w.N, B, strideX, ppd);
    if (rc) return rc;
    // Kinv != nullptr: the look-ahead driver also accumulates K^-1 = L^-t L^-1 while it factors (one large problem only)
    rc = Kinv ? gpk_potrf_inv_pipelined(h, w.A, Li, Kinv, w.T, w.N, keep_L, info_dev, kinv_done)
              : gpk_potrf_inv(h, w.A, Li, w.T, w.N, keep_L, info_dev, B);
    if (rc) return rc;
    rc = gpk_pad_vector(h, w.ypad, w.N, dy, n, B);
    if (rc) return rc;
    rc = gpk_trmv_lower(h, Li, w.N, w.ypad, w.z, w.scratch, B);       // z = L^-1 y      (GpPredictor.scala:121)
    if (rc) return rc;
    rc = gpk_trmv_lower_t(h, Li, w.N, w.z, alpha, B);                  // alpha = L^-t z  (GpPredictor.scala:122)
    if (rc) return rc;
    return gpk_loglik(h, w.A, w.N, n, w.ypad, alpha, ll_dev, B, ll_stride);  // GpPredictor.scala:144-149
}

// params_on_device (B == 1 only): the caller has already written the problem's ProblemParams to w.pp_dev on the handle's
// stream and *pp_single holds the same record; every kernel reads the device copy (graph replay, see the top of this file).
int nll_grad_core(gpk_handle h, int B, const double* dX, int n, int D, int64_t ldx, int64_t strideX, const double* dy,
                  const double* thetas, int has_s, double s, int nparams, double* out_dev, int* info_dev,
                  const ProblemParams* pp_single = nullptr) {
    Work w;
    int rc = make_work(h, n, D, B, &w);
    if (rc) return rc;
    const int64_t so = nparams + 1;
    const bool on_dev = pp_single != nullptr;
    for (int b0 = 0; b0 < B; b0 += w.B) {
        const int bc = (B - b0 < w.B) ? B - b0 : w.B;
        ProblemParams pp0;
        if (on_dev) pp0 = *pp_single;
        else rc = stage_params(h, thetas + (size_t)b0 * gpk_theta_len(h, D), D, has_s, s, bc, w.pp_dev, &pp0);
        if (rc) return rc;
        const double* X = dX + b0 * strideX;
        int* info = info_dev ? info_dev + b0 : (B == 1 ? h->d_info : w.info_dev);
        double* Kinv = nullptr;
        if (nparams > 0 && gpk_use_pipelined(w.N, bc)) {
            ARENA_OR_FAIL(dKinv, double*, h, ARENA_KINV, (size_t)w.N * w.N * sizeof(double));
            Kinv = dKinv;
        }
        cudaEvent_t kinv_done = nullptr;
        rc = fit_core(h, w, bc, X, n, D, ldx, strideX, dy + (size_t)b0 * n, pp0, 0, w.Li, w.alpha, out_dev + b0 * so, so, info, Kinv,
                      &kinv_done, on_dev);
        if (rc) return rc;
        if (kinv_done) GPK_CUDA(h, cudaStreamWaitEvent(h->stream, kinv_done, 0));   // alpha / ll above overlapped the last K^-1 row
        if (nparams > 0) {
            if (!Kinv) {
                rc = gpk_lauum_lower(h, w.Li, w.A, w.N, bc);  // K^-1 = L^-t L^-1 (GpPredictor.scala:67), lower tiles, into A
                if (rc) return rc;
            }
            rc = gpk_grad_trace(h, Kinv ? Kinv : w.A, w.N, X, n, ldx, w.alpha, pp0, nparams, out_dev + b0 * so + 1, w.scratch, bc, strideX,
                                (bc > 1 || on_dev) ? w.pp_dev : nullptr, so);
            if (rc) return rc;
        }
    }
    return GPK_OK;
}

__global__ void store_params_kernel(const ProblemParams pp, ProblemParams* __restrict__ dst) {
    if (threadIdx.x == 0) *dst = pp;
}

// The single-problem evaluation through the graph cache (gpk_graph.cu).  Hyper-parameters reach the kernels through a
// ProblemParams record in device memory that a one-thread kernel rewrites in front of every replay.
int nll_grad_single(gpk_handle h, const double* dX, int n, int D, int64_t ldx, const double* dy, const double* theta, int has_s,
                    double s, int nparams, double* out_dev, int* info_dev) {
    if (!h->graph_mode) return nll_grad_core(h, 1, dX, n, D, ldx, 0, dy, theta, has_s, s, nparams, out_dev, info_dev);
    ProblemParams pp;
    int rc = gpk_make_problem_params(h, theta, D, has_s, s, &pp);
    if (rc) return rc;
    Work w;
    rc = make_work(h, n, D, 1, &w);     // sizes every arena now, so that the workspace epoch the cache compares is final
    if (rc) return rc;
    if (nparams > 0 && gpk_use_pipelined(w.N, 1)) {
        ARENA_OR_FAIL(Kinv, double*, h, ARENA_KINV, (size_t)w.N * w.N * sizeof(double));
    }
    GraphKey key;
    memset(&key, 0, sizeof(key));
    key.p[0] = dX; key.p[1] = dy; key.p[2] = out_dev; key.p[3] = info_dev;
    key.i[0] = n; key.i[1] = D; key.i[2] = nparams; key.i[3] = ldx; key.i[4] = h->kernel_family;
    store_params_kernel<<<1, 32, 0, h->stream>>>(pp, w.pp_dev);
    GPK_LAUNCH_CHECK(h);
    auto body = [&]() { return nll_grad_core(h, 1, dX, n, D, ldx, 0, dy, theta, has_s, s, nparams, out_dev, info_dev, &pp); };
    // captured on the second call: an optimiser's objective is called 25-60 times per fit, a benchmark loop more often
    static int after = -1;
    if (after < 0) { const char* e = getenv("GPK_GRAPH_AFTER_EVAL"); after = e ? atoi(e) : 1; if (after < 1) after = 1; }
    return gpk_graph_run(h, GPK_SLOT_EVAL, key, after, body, "evaluation");
}


// GPOptimizer.scala:93-103: for candidate c and input dimension d (one CTA each)
//   G_id   = ((x_d - x_id) * 1/l_d^2) * (-k(x, x_i))                       KernelRequisites.scala:99-107, afterFirstArg
//   dmean  = sum_i G_id alpha_i                                            testTrainDerMtx * alphaVec
//   dvar   = 0 - 2 sum_i G_id u_i,  u = L^-t (L^-1 k*)                     derAfterVarFirst(x,x) = 0; (L^-1 G)^t v = G^t L^-t v
//   grad   = dmean + dvar * k / (2 sqrt(sigma))
__global__ void __launch_bounds__(256) ucb_grad_kernel(const double* __restrict__ KsT, const double* __restrict__ U, int N, int n,
                                                       const double* __restrict__ X, int ldx, const double* __restrict__ Xs, int ms,
                                                       const double* __restrict__ alpha, const double* __restrict__ colsq,
                                                       const double* __restrict__ mean, CovParams cp, double kparam,
                                                       double* __restrict__ grad, double* __restrict__ ucb, double* __restrict__ var) {
    __shared__ double sa[256], sb[256];
    const int c = blockIdx.x, d = blockIdx.y;
    const double xd = Xs[c + (int64_t)d * ms], inv = cp.inv_ls2[d];
    const double* ks = KsT + (int64_t)c * N;
    const double* u = U + (int64_t)c * N;
    const double* xcol = X + (int64_t)d * ldx;
    double a = 0.0, b = 0.0;
    for (int i = threadIdx.x; i < n; i += 256) {
        const double g = ((xd - xcol[i]) * inv) * (-ks[i]);
        a += g * alpha[i];
        b += g * u[i];
    }
    sa[threadIdx.x] = a; sb[threadIdx.x] = b;
    __syncthreads();
    for (int s = 128; s > 0; s >>= 1) {
        if (threadIdx.x < s) { sa[threadIdx.x] += sa[threadIdx.x + s]; sb[threadIdx.x] += sb[threadIdx.x + s]; }
        __syncthreads();
    }
    if (threadIdx.x == 0) {
        const double sigma = gpk_prior_var(cp) - colsq[c];       // k(x,x) - v^t v
        const double coeff = kparam / (2 * sqrt(sigma));
        grad[c + (int64_t)d * ms] = sa[0] + (0.0 - 2.0 * sb[0]) * coeff;
        if (d == 0) { ucb[c] = mean[c] + kparam * sqrt(sigma); var[c] = sigma; }
    }
}

}  // namespace

namespace {

int upload_model_x(gpk_handle h, gpk_model m, const double* X, int64_t ldx) {   // host n x D (ld ldx) -> device (ld m->ldx)
    GPK_CUDA(h, cudaMemcpy2DAsync(m->X, (size_t)m->ldx * sizeof(double), X, (size_t)ldx * sizeof(double), (size_t)m->n * sizeof(double),
                                  (size_t)m->D, cudaMemcpyHostToDevice, h->stream));
    return GPK_OK;
}

// The three device buffers of a model of padded size N: X (N x D), Li (N x N), alpha (N) -- all three or none
int model_buffers(gpk_handle h, int N, int D, double** X, double** Li, double** alpha) {
    *X = *Li = *alpha = nullptr;
    if (cudaMalloc((void**)X, (size_t)N * D * sizeof(double)) == cudaSuccess &&
        cudaMalloc((void**)Li, (size_t)N * N * sizeof(double)) == cudaSuccess &&
        cudaMalloc((void**)alpha, (size_t)N * sizeof(double)) == cudaSuccess)
        return GPK_OK;
    cudaGetLastError();
    cudaFree(*X); cudaFree(*Li); cudaFree(*alpha);
    *X = *Li = *alpha = nullptr;
    return gpk_set_error(h, GPK_ENOMEM, "allocation of a model of padded size %d failed", N);
}

// A new resident model of n training rows whose buffers `fill` writes; a failure destroys the half-built model here.
template <class F>
int model_make(gpk_handle h, int n, int D, const double* theta, gpk_model* out, F&& fill) {
    GPK_CUDA(h, cudaSetDevice(h->device));
    gpk_model m = new (std::nothrow) gpk_model_s();
    if (!m) return GPK_ENOMEM;
    memset(m, 0, sizeof(*m));
    m->n = n; m->N = gpk_pad(n); m->D = D; m->ldx = m->N;
    memcpy(m->theta, theta, sizeof(double) * gpk_theta_len(h, D));
    int rc = model_buffers(h, m->N, D, &m->X, &m->Li, &m->alpha);
    if (!rc) rc = fill(m);
    if (rc) { gpk_gp_model_destroy(h, m); return rc; }
    *out = m;
    return GPK_OK;
}

// Bordered update of a resident model by one training point (gpk_gp_model_append).  With k = k(X, x), l = L^-1 k,
// d^2 = k(x,x) - l.l, w = L^-t l = K^-1 k and zeta = (y - k.alpha) / d   (l . L^-1 y_old = k . alpha):
//   L_new^-1 = [ L^-1 0 ; -w^t/d  1/d ],   alpha_new = [ alpha - w zeta/d ; zeta/d ].
// dots = { l.l, k.alpha }.  A non-positive d^2 sets *info = n+1 (the failing leading minor) and changes nothing.
__global__ void __launch_bounds__(256) model_append_kernel(double* __restrict__ Li, int N, int n, double* __restrict__ alpha,
                                                           double* __restrict__ X, int ldx, int D, const double* __restrict__ xnew,
                                                           const double* __restrict__ w, const double* __restrict__ dots, double kss,
                                                           double ynew, int* __restrict__ info, double* __restrict__ out) {
    const int i = blockIdx.x * 256 + threadIdx.x;
    const double d2 = kss - dots[0];
    if (!(d2 > 0.0)) {
        if (i == 0) *info = n + 1;
        return;
    }
    const double d = sqrt(d2), zeta = (ynew - dots[1]) / d;
    if (i < n) {
        const double u = -w[i] / d;
        Li[n + (int64_t)i * N] = u;
        alpha[i] += u * zeta;
    } else if (i == n) {
        Li[n + (int64_t)n * N] = 1.0 / d;
        alpha[n] = zeta / d;
        for (int c = 0; c < D; ++c) X[n + (int64_t)c * ldx] = xnew[c];
        out[0] = d; out[1] = zeta;
    }
}

// new (N2 x N2) inverse factor from the old (N x N) one: old block copied, identity on the new diagonal, zeros in the new rows
__global__ void __launch_bounds__(256) model_grow_kernel(const double* __restrict__ Lo, int N, double* __restrict__ Ln, int N2) {
    const int64_t idx = (int64_t)blockIdx.x * 256 + threadIdx.x;
    if (idx >= (int64_t)N2 * N2) return;
    const int r = (int)(idx % N2), c = (int)(idx / N2);
    double v = 0.0;
    if (r < N && c < N) v = Lo[r + (int64_t)c * N];
    else if (r == c) v = 1.0;
    Ln[idx] = v;
}

}  // namespace

int gpk_posterior(gpk_handle h, const double* dX, int n, int64_t ldx, const double* dXs, int ms, const double* Li,
                  const double* alpha, int N, const CovParams& cp, double* KsT, double* mean, double* V, int nv, double* vsq,
                  int batch, int64_t strideX, int64_t strideXs, const ProblemParams* pp_dev) {
    const int M = gpk_pad(ms);
    const int64_t sK = (int64_t)N * M;
    int rc = gpk_cov_cross(h, dX, n, ldx, dXs, ms, ms, cp, KsT, N, N, M, batch, strideX, strideXs, sK, pp_dev);  // GpPredictor.scala:53
    if (rc) return rc;
    rc = gpk_colwise_dot(h, KsT, N, N, ms, alpha, mean, 0, batch, sK, N, M);                                       // :54
    if (rc || !V) return rc;
    rc = gpk_trmm_lower(h, Li, N, KsT, V, gpk_pad(nv), batch);                                                     // :55
    if (rc || !vsq) return rc;
    return gpk_colwise_dot(h, V, N, N, nv, nullptr, vsq, 1, batch, sK, 0, M);                                      // :56, diagonal
}

size_t batch_budget_bytes() {
    static size_t v = 0;
    if (!v) {
        const char* e = getenv("GPK_BATCH_GB");
        v = (size_t)((e ? atof(e) : 48.0) * (1ull << 30));
    }
    return v;
}

// A stack of nx host matrices (n x D, ld ldx, matrix b at X + b*stride) to the device, compact and back to back (matrix b at
// dst + b*n*D): one copy when the stack already is laid out so (Breeze matrices back to back)
int upload_stack(gpk_handle h, double* dst, const double* X, int nx, int n, int D, int64_t ldx, int64_t stride) {
    if (ldx == n && (nx == 1 || stride == (int64_t)n * D)) {
        GPK_CUDA(h, cudaMemcpyAsync(dst, X, (size_t)nx * n * D * sizeof(double), cudaMemcpyHostToDevice, h->stream));
        return GPK_OK;
    }
    int rc = GPK_OK;
    for (int b = 0; b < nx && !rc; ++b) rc = gpk_upload_matrix(h, dst + (size_t)b * n * D, X + b * stride, n, D, ldx);
    return rc;
}

// The results of a batched call come back through the handle's pinned staging (grown on demand, never per call): res_bytes
// of results at dres (0: none) followed on the device by the B per-problem info words, staged at h->res_pinned in one copy
// and one synchronisation.  info (optional) receives the info words.  The call's first failure goes to h->last_info and
// sets *failed, which stays set across the chunks of one call: GPK_ENOTPD from then on.
int fetch_batch_results(gpk_handle h, const void* dres, size_t res_bytes, int B, int* info, bool* failed) {
    const size_t bytes = res_bytes + (size_t)B * sizeof(int);
    if (h->res_pinned_bytes < bytes) {
        if (h->res_pinned) cudaFreeHost(h->res_pinned);
        h->res_pinned = nullptr; h->res_pinned_bytes = 0;
        if (cudaMallocHost(&h->res_pinned, bytes) != cudaSuccess) { cudaGetLastError(); return gpk_set_error(h, GPK_ENOMEM, "pinned host allocation failed"); }
        h->res_pinned_bytes = bytes;
    }
    GPK_CUDA(h, cudaMemcpyAsync(h->res_pinned, dres, bytes, cudaMemcpyDeviceToHost, h->stream));
    GPK_CUDA(h, cudaStreamSynchronize(h->stream));
    const int* hinfo = (const int*)((const char*)h->res_pinned + res_bytes);
    for (int b = 0; b < B; ++b) {
        if (info) info[b] = hinfo[b];
        if (hinfo[b] && !*failed) { *failed = true; h->last_info = hinfo[b]; }
    }
    if (*failed) return gpk_set_error(h, GPK_ENOTPD, "at least one problem of the batch is not positive definite (see info[])");
    return GPK_OK;
}

extern "C" {

// ------------------------------------------------------------------------------------------------
// log marginal likelihood + gradient
// ------------------------------------------------------------------------------------------------
int gpk_gp_nll_grad_dev(gpk_handle h, const double* dX, int n, int D, int64_t ldx, const double* dy, const double* theta,
                        int has_s, double s, int nparams, double* out_dev, int* info_dev) {
    int rc = gpk_check_args(h, "gpk_gp_nll_grad_dev", true, n, 1, ldx, D, nparams);
    if (rc) return rc;
    return nll_grad_single(h, dX, n, D, ldx, dy, theta, has_s, s, nparams, out_dev, info_dev);
}

int gpk_gp_nll_grad(gpk_handle h, const double* X, int n, int D, int64_t ldx, const double* y, const double* theta,
                    int has_s, double s, int nparams, double* ll, double* grad) {
    int rc = gpk_check_args(h, "gpk_gp_nll_grad", true, n, 1, ldx, D, nparams);
    if (rc) return rc;
    GPK_CUDA(h, cudaSetDevice(h->device));
    ARENA_OR_FAIL(dX, double*, h, ARENA_X, ((size_t)n * D + n + 256) * sizeof(double));
    double* dy = dX + (size_t)n * D;
    double* dout = dy + n;
    rc = gpk_upload_matrix(h, dX, X, n, D, ldx);
    if (rc) return rc;
    GPK_CUDA(h, cudaMemcpyAsync(dy, y, (size_t)n * sizeof(double), cudaMemcpyHostToDevice, h->stream));
    rc = nll_grad_single(h, dX, n, D, n, dy, theta, has_s, s, nparams, dout, nullptr);
    if (rc) return rc;
    GPK_CUDA(h, cudaMemcpyAsync(h->h_pinned, dout, (size_t)(nparams + 1) * sizeof(double), cudaMemcpyDeviceToHost, h->stream));
    rc = gpk_finish_info(h);
    if (rc) return rc;
    *ll = h->h_pinned[0];
    for (int p = 0; p < nparams; ++p) grad[p] = h->h_pinned[1 + p];
    return GPK_OK;
}

int gpk_gp_nll_grad_batched_dev(gpk_handle h, int B, const double* dX, int n, int D, int64_t ldx, int64_t strideX,
                                const double* dy, const double* thetas, int has_s, double s, int nparams, double* out_dev,
                                int* info_dev) {
    int rc = gpk_check_args(h, "gpk_gp_nll_grad_batched_dev", B > 0 && info_dev, n, 1, ldx, D, nparams);
    if (rc) return rc;
    return nll_grad_core(h, B, dX, n, D, ldx, strideX, dy, thetas, has_s, s, nparams, out_dev, info_dev);
}

int gpk_gp_nll_grad_batched(gpk_handle h, int B, const double* X, int n, int D, int64_t ldx, int64_t strideX, const double* y,
                            const double* thetas, int has_s, double s, int nparams, double* ll, double* grad, int* info) {
    int rc = gpk_check_args(h, "gpk_gp_nll_grad_batched", B > 0, n, 1, ldx, D, nparams);
    if (rc) return rc;
    if (strideX != 0 && strideX < (int64_t)ldx * (D - 1) + n)
        return gpk_set_error(h, GPK_EINVAL, "gpk_gp_nll_grad_batched: strideX overlaps consecutive problems");
    GPK_CUDA(h, cudaSetDevice(h->device));
    const int nx = strideX ? B : 1;
    const size_t so = (size_t)nparams + 1;
    ARENA_OR_FAIL(dX, double*, h, ARENA_X, ((size_t)nx * n * D + (size_t)B * n + B * so + 256) * sizeof(double) + (size_t)B * sizeof(int));
    double* dy = dX + (size_t)nx * n * D;
    double* dout = dy + (size_t)B * n;
    int* dinfo = (int*)(dout + B * so);
    rc = upload_stack(h, dX, X, nx, n, D, ldx, strideX);
    if (rc) return rc;
    GPK_CUDA(h, cudaMemcpyAsync(dy, y, (size_t)B * n * sizeof(double), cudaMemcpyHostToDevice, h->stream));
    rc = nll_grad_core(h, B, dX, n, D, n, strideX ? (int64_t)n * D : 0, dy, thetas, has_s, s, nparams, dout, dinfo);
    if (rc) return rc;
    bool failed = false;
    rc = fetch_batch_results(h, dout, B * so * sizeof(double), B, info, &failed);   // dinfo follows dout
    if (rc && rc != GPK_ENOTPD) return rc;
    const double* hout = (const double*)h->res_pinned;
    for (int b = 0; b < B; ++b) {
        ll[b] = hout[b * so];
        for (int p = 0; p < nparams; ++p) grad[(size_t)b * nparams + p] = hout[b * so + 1 + p];
    }
    return rc;
}

// ------------------------------------------------------------------------------------------------
// fit
// ------------------------------------------------------------------------------------------------
int gpk_gp_fit(gpk_handle h, const double* X, int n, int D, int64_t ldx, const double* y, const double* theta, int has_s,
               double s, double* L, int64_t ldl, double* alpha, double* ll) {
    int rc = gpk_check_args(h, "gpk_gp_fit", !L || ldl >= n, n, 1, ldx, D, 0);
    if (rc) return rc;
    GPK_CUDA(h, cudaSetDevice(h->device));
    ARENA_OR_FAIL(dX, double*, h, ARENA_X, ((size_t)n * D + n + 256) * sizeof(double));
    double* dy = dX + (size_t)n * D;
    double* dout = dy + n;
    rc = gpk_upload_matrix(h, dX, X, n, D, ldx);
    if (rc) return rc;
    GPK_CUDA(h, cudaMemcpyAsync(dy, y, (size_t)n * sizeof(double), cudaMemcpyHostToDevice, h->stream));
    Work w;
    rc = make_work(h, n, D, 1, &w);
    if (rc) return rc;
    ProblemParams pp;
    rc = gpk_make_problem_params(h, theta, D, has_s, s, &pp);
    if (rc) return rc;
    rc = fit_core(h, w, 1, dX, n, D, n, 0, dy, pp, L != nullptr, w.Li, w.alpha, dout, 1, h->d_info);
    if (rc) return rc;
    GPK_CUDA(h, cudaMemcpyAsync(h->h_pinned, dout, sizeof(double), cudaMemcpyDeviceToHost, h->stream));
    rc = gpk_finish_info(h);
    if (rc) return rc;
    if (ll) *ll = h->h_pinned[0];
    if (alpha) GPK_CUDA(h, cudaMemcpyAsync(alpha, w.alpha, (size_t)n * sizeof(double), cudaMemcpyDeviceToHost, h->stream));
    if (L) {
        rc = gpk_download_tri(h, L, ldl, w.A, w.N, n, 0);
        if (rc) return rc;
    }
    return gpk_synchronize(h);
}

// ------------------------------------------------------------------------------------------------
// resident model + prediction
// ------------------------------------------------------------------------------------------------
int gpk_gp_model_destroy(gpk_handle h, gpk_model m) {
    if (!m) return GPK_OK;
    if (h) { cudaSetDevice(h->device); cudaStreamSynchronize(h->stream); }
    cudaFree(m->X); cudaFree(m->Li); cudaFree(m->alpha);
    delete m;
    return GPK_OK;
}

int gpk_gp_model_fit(gpk_handle h, const double* X, int n, int D, int64_t ldx, const double* y, const double* theta,
                     int has_s, double s, gpk_model* out, double* ll) {
    int rc = gpk_check_args(h, "gpk_gp_model_fit", out != nullptr, n, 1, ldx, D, 0);
    if (rc) return rc;
    return model_make(h, n, D, theta, out, [&](gpk_model m) -> int {
        ARENA_OR_FAIL(dy, double*, h, ARENA_X, ((size_t)n + 256) * sizeof(double));
        double* dout = dy + n;
        int rc = upload_model_x(h, m, X, ldx);
        if (rc) return rc;
        GPK_CUDA(h, cudaMemcpyAsync(dy, y, (size_t)n * sizeof(double), cudaMemcpyHostToDevice, h->stream));
        Work w;
        rc = make_work(h, n, D, 1, &w);
        if (!rc) rc = gpk_make_problem_params(h, theta, D, has_s, s, &m->pp);
        // factor straight into the model's resident buffers
        if (!rc) rc = fit_core(h, w, 1, m->X, n, D, m->ldx, 0, dy, m->pp, 0, m->Li, m->alpha, dout, 1, h->d_info);
        if (rc) return rc;
        GPK_CUDA(h, cudaMemcpyAsync(h->h_pinned, dout, sizeof(double), cudaMemcpyDeviceToHost, h->stream));
        rc = gpk_finish_info(h);
        if (rc) return rc;
        // predictions never include the Option sigmaNoise in the kernel (GpPredictor.scala:31,36 use newKernelFunc only)
        m->pp.cp.extra_diag = 0.0;
        m->has_s = has_s ? 1 : 0; m->s = has_s ? s : 0.0;     // remembered for gpk_gp_model_append
        if (ll) *ll = h->h_pinned[0];
        return GPK_OK;
    });
}

int gpk_gp_model_from_factor(gpk_handle h, const double* X, int n, int D, int64_t ldx, const double* L, int64_t ldl,
                             const double* alpha, const double* theta, gpk_model* out) {
    int rc = gpk_check_args(h, "gpk_gp_model_from_factor", out && ldl >= n, n, 1, ldx, D, 0);
    if (rc) return rc;
    return model_make(h, n, D, theta, out, [&](gpk_model m) -> int {
        const int N = m->N;
        int rc = gpk_make_problem_params(h, theta, D, 0, 0.0, &m->pp);
        if (rc) return rc;
        ARENA_OR_FAIL(dA, double*, h, ARENA_A, (size_t)N * N * sizeof(double));
        ARENA_OR_FAIL(dT, double*, h, ARENA_T, gpk_chol_scratch_doubles(N) * sizeof(double));
        rc = upload_model_x(h, m, X, ldx);
        if (!rc) rc = gpk_upload_padded(h, dA, N, L, n, ldl, GPK_PAD_LOWER);
        if (!rc) rc = gpk_trtri_lower(h, dA, m->Li, dT, N);
        if (rc) return rc;
        GPK_CUDA(h, cudaMemsetAsync(m->alpha, 0, (size_t)N * sizeof(double), h->stream));
        GPK_CUDA(h, cudaMemcpyAsync(m->alpha, alpha, (size_t)n * sizeof(double), cudaMemcpyHostToDevice, h->stream));
        m->has_s = -1;                                     // unknown: the caller's factor may or may not include a sigmaNoise
        return gpk_synchronize(h);
    });
}

// gp/optimization/GPOptimizer.scala:48-71: every outer GP-UCB iteration appends ONE evaluated point to the training set and
// the reference refits from scratch (preComputeComponents, O(n^3), :51).  With the hyper-parameters unchanged the new factor
// is the old one bordered by one row, so the resident (L^-1, alpha) are updated in O(n^2): two triangular mat-vecs.
int gpk_gp_model_append(gpk_handle h, gpk_model m, const double* x_new, double y_new, int has_s, double s, double* ll_delta) {
    if (!h || !m || !x_new) return gpk_set_error(h, GPK_EINVAL, "gpk_gp_model_append: bad arguments");
    // the bordered row must carry the same Option sigmaNoise the factor was built with (GpPredictor.scala:116-117); a model
    // adopted from a caller's factor (gpk_gp_model_from_factor) has none recorded and takes the caller's word
    if (m->has_s >= 0 && ((has_s ? 1 : 0) != m->has_s || (has_s && s != m->s)))
        return gpk_set_error(h, GPK_EINVAL, "gpk_gp_model_append: sigmaNoise differs from the one the model was fitted with");
    GPK_CUDA(h, cudaSetDevice(h->device));
    const int D = m->D;
    if (m->n == m->N) {   // no padding row left: move to a factor that is one tile larger
        const int N2 = m->N + GPK_TILE;
        double *Xn, *Ln, *an;
        int rc = model_buffers(h, N2, D, &Xn, &Ln, &an);
        if (rc) return rc;
        model_grow_kernel<<<(unsigned)(((int64_t)N2 * N2 + 255) / 256), 256, 0, h->stream>>>(m->Li, m->N, Ln, N2);
        GPK_LAUNCH_CHECK(h);
        GPK_CUDA(h, cudaMemsetAsync(an, 0, (size_t)N2 * sizeof(double), h->stream));
        GPK_CUDA(h, cudaMemcpyAsync(an, m->alpha, (size_t)m->n * sizeof(double), cudaMemcpyDeviceToDevice, h->stream));
        GPK_CUDA(h, cudaMemcpy2DAsync(Xn, (size_t)N2 * sizeof(double), m->X, (size_t)m->ldx * sizeof(double), (size_t)m->n * sizeof(double),
                                      (size_t)D, cudaMemcpyDeviceToDevice, h->stream));
        GPK_CUDA(h, cudaStreamSynchronize(h->stream));
        cudaFree(m->Li); cudaFree(m->alpha); cudaFree(m->X);
        m->Li = Ln; m->alpha = an; m->X = Xn; m->N = N2; m->ldx = N2;
    }
    const int n = m->n, N = m->N;
    // x (D), k (N), l (N), w (N), dots (2), out (2), trmv scratch
    ARENA_OR_FAIL(buf, double*, h, ARENA_IO2, ((size_t)3 * N + D + 8 + gpk_trmv_scratch_doubles(N)) * sizeof(double));
    double* dx = buf;
    double* dk = dx + ((D + 1) & ~1);
    double* dl = dk + N;
    double* dw = dl + N;
    double* ddots = dw + N;
    double* dres = ddots + 2;
    double* scratch = dres + 2;
    for (int c = 0; c < D; ++c) h->h_pinned[64 + c] = x_new[c];
    GPK_CUDA(h, cudaMemcpyAsync(dx, h->h_pinned + 64, (size_t)D * sizeof(double), cudaMemcpyHostToDevice, h->stream));
    GPK_CUDA(h, cudaMemsetAsync(h->d_info, 0, sizeof(int), h->stream));
    int rc = gpk_cov_cross(h, m->X, n, m->ldx, dx, 1, 1, m->pp.cp, dk, N, N, 1);      // k = k(X, x), zero in the padding
    if (rc) return rc;
    rc = gpk_trmv_lower(h, m->Li, N, dk, dl, scratch);                                  // l = L^-1 k
    if (rc) return rc;
    rc = gpk_colwise_dot(h, dl, N, N, 1, nullptr, ddots, 1);                            // l.l
    if (rc) return rc;
    rc = gpk_colwise_dot(h, dk, N, N, 1, m->alpha, ddots + 1, 0);                       // k.alpha
    if (rc) return rc;
    rc = gpk_trmv_lower_t(h, m->Li, N, dl, dw);                                         // w = L^-t l
    if (rc) return rc;
    // k(x,x) and the Option sigmaNoise of the fit (GpPredictor.scala:116-117)
    const double kss = gpk_prior_var(m->pp.cp) + (has_s ? s : 0.0);
    model_append_kernel<<<(n + 256) / 256, 256, 0, h->stream>>>(m->Li, N, n, m->alpha, m->X, m->ldx, D, dx, dw, ddots, kss, y_new,
                                                                h->d_info, dres);
    GPK_LAUNCH_CHECK(h);
    GPK_CUDA(h, cudaMemcpyAsync(h->h_pinned, dres, 2 * sizeof(double), cudaMemcpyDeviceToHost, h->stream));
    rc = gpk_finish_info(h);
    if (rc) return rc;
    m->n = n + 1;
    // log-likelihood of the enlarged set minus that of the old one: -zeta^2/2 - log d - log(2 pi)/2  (GpPredictor.scala:144-149)
    if (ll_delta) *ll_delta = -0.5 * h->h_pinned[1] * h->h_pinned[1] - log(h->h_pinned[0]) - 0.9189385332046727;
    return GPK_OK;
}

int gpk_gp_model_size(gpk_handle h, gpk_model m) { return m ? m->n : gpk_set_error(h, GPK_EINVAL, "null model"); }

int gpk_gp_model_get_alpha(gpk_handle h, gpk_model m, double* alpha) {
    if (!h || !m || !alpha) return gpk_set_error(h, GPK_EINVAL, "gpk_gp_model_get_alpha: bad arguments");
    GPK_CUDA(h, cudaSetDevice(h->device));
    GPK_CUDA(h, cudaMemcpyAsync(alpha, m->alpha, (size_t)m->n * sizeof(double), cudaMemcpyDeviceToHost, h->stream));
    return gpk_synchronize(h);
}

int gpk_gp_model_predict(gpk_handle h, gpk_model m, const double* Xs, int ms, int64_t ldxs, int want_full_cov, double* mean,
                         double* sigma, int64_t lds, double* V, int64_t ldv) {
    if (!h || !m || ms <= 0 || ldxs < ms || (V && ldv < m->n) || (want_full_cov && sigma && lds < ms))
        return gpk_set_error(h, GPK_EINVAL, "gpk_gp_model_predict: bad dimensions");
    GPK_CUDA(h, cudaSetDevice(h->device));
    const int n = m->n, N = m->N, D = m->D, M = gpk_pad(ms);
    const CovParams& cp = m->pp.cp;
    ARENA_OR_FAIL(dXs, double*, h, ARENA_X, (size_t)ms * D * sizeof(double));
    // KsT (N x M), V (N x M), Sig (M x M), mean (M), var (M)
    ARENA_OR_FAIL(buf, double*, h, ARENA_IO2, ((size_t)2 * N * M + (size_t)M * M + 2 * M) * sizeof(double));
    double* dKsT = buf;
    double* dV = dKsT + (size_t)N * M;
    double* dSig = dV + (size_t)N * M;
    double* dMean = dSig + (size_t)M * M;
    double* dVar = dMean + M;
    int rc = gpk_upload_matrix(h, dXs, Xs, ms, D, ldxs);
    if (rc) return rc;
    // V is skipped when only the mean is wanted (the GP-UKF transition / observation functions, GPUnscentedKalmanFilter.scala:77-90,
    // read nothing else); the full covariance needs no column sums
    rc = gpk_posterior(h, m->X, n, m->ldx, dXs, ms, m->Li, m->alpha, N, cp, dKsT, dMean, (sigma || V) ? dV : nullptr, ms,
                       (sigma && !want_full_cov) ? dVar : nullptr);
    if (rc) return rc;
    if (mean) GPK_CUDA(h, cudaMemcpyAsync(mean, dMean, (size_t)ms * sizeof(double), cudaMemcpyDeviceToHost, h->stream));
    if (sigma) {
        if (want_full_cov) {
            // sigma = k(X*,X*) (+ sn^2 on the diagonal, MatrixUtils.scala:63) - V^t V   (GpPredictor.scala:56)
            GPK_CUDA(h, cudaMemsetAsync(dSig, 0, (size_t)M * M * sizeof(double), h->stream));
            rc = gpk_cov_sym_full(h, dXs, ms, ms, cp, dSig, M);
            if (rc) return rc;
            GemmDesc g = gemm_desc();
            g.P = dV; g.ldp = N; g.p_kcontig = 1;
            g.Q = dV; g.ldq = N; g.q_kcontig = 1;
            g.D = dSig; g.ldd = M; g.Cin = dSig; g.ldc = M; g.R = M; g.S = M; g.K = N; g.alpha = -1.0; g.beta = 1.0;
            rc = gpk_gemm(h, g);
            if (rc) return rc;
            GPK_CUDA(h, cudaMemcpy2DAsync(sigma, (size_t)lds * sizeof(double), dSig, (size_t)M * sizeof(double),
                                          (size_t)ms * sizeof(double), (size_t)ms, cudaMemcpyDeviceToHost, h->stream));
        } else {
            GPK_CUDA(h, cudaMemcpyAsync(sigma, dVar, (size_t)ms * sizeof(double), cudaMemcpyDeviceToHost, h->stream));
        }
    }
    if (V) GPK_CUDA(h, cudaMemcpy2DAsync(V, (size_t)ldv * sizeof(double), dV, (size_t)N * sizeof(double), (size_t)n * sizeof(double),
                                         (size_t)ms, cudaMemcpyDeviceToHost, h->stream));
    rc = gpk_synchronize(h);
    if (rc) return rc;
    if (sigma && !want_full_cov)
        for (int i = 0; i < ms; ++i) sigma[i] = gpk_prior_var(cp) - sigma[i];
    return GPK_OK;
}

// gp/optimization/GPOptimizer.scala:82-109 maximizeUCB: the objective handed to the gradient optimiser, for ms candidate
// points at once against a resident model (the reference calls computePosterior + two n x D derivative matrices + an
// n x n x D product per candidate, and re-inverts L once per restart, GPOptimizer.scala:85).
int gpk_gp_model_ucb(gpk_handle h, gpk_model m, const double* Xs, int ms, int64_t ldxs, double k_param, double* ucb, double* grad,
                     int64_t ldg, double* mean, double* var) {
    if (!h || !m || !Xs || !ucb || ms <= 0 || ldxs < ms || (grad && ldg < ms))
        return gpk_set_error(h, GPK_EINVAL, "gpk_gp_model_ucb: bad dimensions");
    if (m->pp.cp.kind != GPK_KERNEL_SE_ARD)   // Co2Kernel.gradient is `???` (Co2Prediction.scala:62-64)
        return gpk_set_error(h, GPK_EINVAL, "scala.NotImplementedError: the kernel has no gradient with respect to its inputs");
    GPK_CUDA(h, cudaSetDevice(h->device));
    const int n = m->n, N = m->N, D = m->D, M = gpk_pad(ms);
    const CovParams& cp = m->pp.cp;
    ARENA_OR_FAIL(dXs, double*, h, ARENA_X, (size_t)ms * D * sizeof(double));
    // KsT, V, U (N x M each), mean, colsq, ucb, var (M each), grad (ms x D)
    ARENA_OR_FAIL(buf, double*, h, ARENA_IO2, ((size_t)3 * N * M + 4 * M + (size_t)ms * D) * sizeof(double));
    double* dKsT = buf;
    double* dV = dKsT + (size_t)N * M;
    double* dU = dV + (size_t)N * M;
    double* dMean = dU + (size_t)N * M;
    double* dSq = dMean + M;
    double* dUcb = dSq + M;
    double* dVar = dUcb + M;
    double* dGrad = dVar + M;
    int rc = gpk_upload_matrix(h, dXs, Xs, ms, D, ldxs);
    if (rc) return rc;
    rc = gpk_posterior(h, m->X, n, m->ldx, dXs, ms, m->Li, m->alpha, N, cp, dKsT, dMean, dV, ms, dSq);
    if (rc) return rc;
    GemmDesc g = gemm_desc();                                                    // U = L^-t V: U(i,c) = sum_{k>=i} Li(k,i) V(k,c)
    g.P = dV; g.ldp = N; g.p_kcontig = 1;
    g.Q = m->Li; g.ldq = N; g.q_kcontig = 1;
    g.D = dU; g.ldd = N; g.R = M; g.S = N; g.K = N; g.kb_s = 1;
    rc = gpk_gemm(h, g);
    if (rc) return rc;
    ucb_grad_kernel<<<dim3(ms, D), 256, 0, h->stream>>>(dKsT, dU, N, n, m->X, m->ldx, dXs, ms, m->alpha, dSq, dMean, cp, k_param, dGrad, dUcb,
                                                        dVar);
    GPK_LAUNCH_CHECK(h);
    GPK_CUDA(h, cudaMemcpyAsync(ucb, dUcb, (size_t)ms * sizeof(double), cudaMemcpyDeviceToHost, h->stream));
    if (mean) GPK_CUDA(h, cudaMemcpyAsync(mean, dMean, (size_t)ms * sizeof(double), cudaMemcpyDeviceToHost, h->stream));
    if (var) GPK_CUDA(h, cudaMemcpyAsync(var, dVar, (size_t)ms * sizeof(double), cudaMemcpyDeviceToHost, h->stream));
    if (grad) GPK_CUDA(h, cudaMemcpy2DAsync(grad, (size_t)ldg * sizeof(double), dGrad, (size_t)ms * sizeof(double),
                                            (size_t)ms * sizeof(double), (size_t)D, cudaMemcpyDeviceToHost, h->stream));
    return gpk_synchronize(h);
}

// Posterior means of SEVERAL resident models at the same test rows in one call / one synchronisation: the GP-UKF step
// (GPUnscentedKalmanFilter.scala:77-90: one GP per state / observation dimension, each asked for its mean at every sigma
// point).  mean[j*ms + i] = mean of model j at row i.  Models may differ in training set, targets and hyper-parameters.
int gpk_gp_models_mean(gpk_handle h, const gpk_model* models, int nmodels, const double* Xs, int ms, int64_t ldxs, double* mean) {
    return gpk_gp_models_mean_var(h, models, nmodels, Xs, ms, ldxs, mean, nullptr);
}

// GPUnscentedKalmanFilter.scala:77-90 + :138-147 in one call: means AND variances (diagonal of computePosterior's sigma,
// including noiseVar^2, MatrixUtils.scala:63) of nmodels resident models at the same ms test rows.
int gpk_gp_models_mean_var(gpk_handle h, const gpk_model* models, int nmodels, const double* Xs, int ms, int64_t ldxs,
                           double* mean, double* var) {
    if (!h || !models || nmodels <= 0 || !Xs || ms <= 0 || ldxs < ms || !mean)
        return gpk_set_error(h, GPK_EINVAL, "gpk_gp_models_mean_var: bad arguments");
    GPK_CUDA(h, cudaSetDevice(h->device));
    const int D = models[0]->D, M = gpk_pad(ms);
    int Nmax = 0;
    for (int j = 0; j < nmodels; ++j) {
        if (!models[j] || models[j]->D != D) return gpk_set_error(h, GPK_EINVAL, "gpk_gp_models_mean_var: models disagree on D");
        if (models[j]->N > Nmax) Nmax = models[j]->N;
    }
    ARENA_OR_FAIL(dXs, double*, h, ARENA_X, (size_t)ms * D * sizeof(double));
    // KsT (Nmax x M), mean (nmodels x M); with var also V (Nmax x M), vsq (nmodels x M)
    const size_t nKm = (size_t)Nmax * M + (size_t)nmodels * M;
    ARENA_OR_FAIL(buf, double*, h, ARENA_IO2, (var ? 2 : 1) * nKm * sizeof(double));
    double* dKsT = buf;
    double* dMean = dKsT + (size_t)Nmax * M;
    double* dV = var ? buf + nKm : nullptr;
    double* dVsq = var ? dV + (size_t)Nmax * M : nullptr;
    int rc = gpk_upload_matrix(h, dXs, Xs, ms, D, ldxs);
    if (rc) return rc;
    for (int j = 0; j < nmodels; ++j) {
        gpk_model m = models[j];
        rc = gpk_posterior(h, m->X, m->n, m->ldx, dXs, ms, m->Li, m->alpha, m->N, m->pp.cp, dKsT, dMean + (size_t)j * M, dV, ms,
                           var ? dVsq + (size_t)j * M : nullptr);
        if (rc) return rc;
    }
    GPK_CUDA(h, cudaMemcpy2DAsync(mean, (size_t)ms * sizeof(double), dMean, (size_t)M * sizeof(double), (size_t)ms * sizeof(double),
                                  (size_t)nmodels, cudaMemcpyDeviceToHost, h->stream));
    if (var)
        GPK_CUDA(h, cudaMemcpy2DAsync(var, (size_t)ms * sizeof(double), dVsq, (size_t)M * sizeof(double), (size_t)ms * sizeof(double),
                                      (size_t)nmodels, cudaMemcpyDeviceToHost, h->stream));
    rc = gpk_synchronize(h);
    if (rc) return rc;
    if (var)
        for (int j = 0; j < nmodels; ++j)
            for (int i = 0; i < ms; ++i) var[(size_t)j * ms + i] = gpk_prior_var(models[j]->pp.cp) - var[(size_t)j * ms + i];
    return GPK_OK;
}

int gpk_gp_predict(gpk_handle h, const double* X, int n, int D, int64_t ldx, const double* y, const double* Xs, int ms,
                   int64_t ldxs, const double* theta, int has_s, double s, double* mean, double* sigma, int64_t lds, double* ll) {
    int rc = gpk_check_args(h, "gpk_gp_predict", ms > 0 && ldxs >= ms && (!sigma || lds >= ms), n, 1, ldx, D, 0);
    if (rc) return rc;
    gpk_model m = nullptr;
    rc = gpk_gp_model_fit(h, X, n, D, ldx, y, theta, has_s, s, &m, ll);
    if (rc) return rc;
    rc = gpk_gp_model_predict(h, m, Xs, ms, ldxs, 1, mean, sigma, lds, nullptr, 0);
    gpk_gp_model_destroy(h, m);
    if (rc) return rc;
    if (has_s && sigma)  // GpPredictor.scala:37-39: + sigmaNoise * I
        for (int i = 0; i < ms; ++i) sigma[i + (int64_t)i * lds] += s;
    return GPK_OK;
}

// B independent GPs: fit each (its own theta_b, y_b; X shared when strideX == 0) and evaluate the posterior mean and
// variance at ms test rows each -- the GP-UKF sigma-point pattern (GPUnscentedKalmanFilter.scala:77-88,138-147).
int gpk_gp_predict_batched(gpk_handle h, int B, const double* X, int n, int D, int64_t ldx, int64_t strideX, const double* y,
                           const double* thetas, const double* Xs, int ms, int64_t ldxs, int64_t strideXs, int has_s, double s,
                           double* mean, double* var, double* ll, int* info) {
    int rc = gpk_check_args(h, "gpk_gp_predict_batched", B > 0 && ms > 0 && ldxs >= ms, n, 1, ldx, D, 0);
    if (rc) return rc;
    GPK_CUDA(h, cudaSetDevice(h->device));
    const int N = gpk_pad(n), M = gpk_pad(ms);
    Work w;
    rc = make_work(h, n, D, B, &w);
    if (rc) return rc;
    const int Bc = w.B;
    const int nx = strideX ? Bc : 1, nxs = strideXs ? Bc : 1;
    ARENA_OR_FAIL(dX, double*, h, ARENA_X, ((size_t)nx * n * D + (size_t)nxs * ms * D + (size_t)Bc * n + Bc + 256) * sizeof(double));
    double* dXs = dX + (size_t)nx * n * D;
    double* dy = dXs + (size_t)nxs * ms * D;
    double* dll = dy + (size_t)Bc * n;
    ARENA_OR_FAIL(buf, double*, h, ARENA_IO2, (size_t)Bc * ((size_t)2 * N * M + 2 * M) * sizeof(double));
    double* dKsT = buf;
    double* dV = dKsT + (size_t)Bc * N * M;
    double* dMean = dV + (size_t)Bc * N * M;
    double* dVar = dMean + (size_t)Bc * M;
    bool failed = false;
    for (int b0 = 0; b0 < B; b0 += Bc) {
        const int bc = (B - b0 < Bc) ? B - b0 : Bc;
        ProblemParams pp0;
        rc = stage_params(h, thetas + (size_t)b0 * gpk_theta_len(h, D), D, has_s, s, bc, w.pp_dev, &pp0);
        if (!rc) rc = upload_stack(h, dX, X + b0 * strideX, strideX ? bc : 1, n, D, ldx, strideX);
        if (!rc) rc = upload_stack(h, dXs, Xs + b0 * strideXs, strideXs ? bc : 1, ms, D, ldxs, strideXs);
        if (rc) return rc;
        GPK_CUDA(h, cudaMemcpyAsync(dy, y + (size_t)b0 * n, (size_t)bc * n * sizeof(double), cudaMemcpyHostToDevice, h->stream));
        const int64_t sX = strideX ? (int64_t)n * D : 0, sXs = strideXs ? (int64_t)ms * D : 0;
        rc = fit_core(h, w, bc, dX, n, D, n, sX, dy, pp0, 0, w.Li, w.alpha, dll, 1, w.info_dev);
        if (rc) return rc;
        // predictions use the kernel without the Option sigmaNoise: extra_diag does not enter cross-covariances
        rc = gpk_posterior(h, dX, n, n, dXs, ms, w.Li, w.alpha, N, pp0.cp, dKsT, dMean, dV, ms, dVar, bc, sX, sXs,
                           bc > 1 ? w.pp_dev : nullptr);
        if (rc) return rc;
        GPK_CUDA(h, cudaMemcpy2DAsync(mean + (size_t)b0 * ms, (size_t)ms * sizeof(double), dMean, (size_t)M * sizeof(double),
                                      (size_t)ms * sizeof(double), (size_t)bc, cudaMemcpyDeviceToHost, h->stream));
        GPK_CUDA(h, cudaMemcpy2DAsync(var + (size_t)b0 * ms, (size_t)ms * sizeof(double), dVar, (size_t)M * sizeof(double),
                                      (size_t)ms * sizeof(double), (size_t)bc, cudaMemcpyDeviceToHost, h->stream));
        if (ll) GPK_CUDA(h, cudaMemcpyAsync(ll + b0, dll, (size_t)bc * sizeof(double), cudaMemcpyDeviceToHost, h->stream));
        rc = fetch_batch_results(h, w.info_dev, 0, bc, info ? info + b0 : nullptr, &failed);
        if (rc && rc != GPK_ENOTPD) return rc;
        const ProblemParams* hp = (const ProblemParams*)h->pp_host;   // the chunk's records, as stage_params built them
        for (int b = 0; b < bc; ++b)
            for (int i = 0; i < ms; ++i) var[(size_t)(b0 + b) * ms + i] = gpk_prior_var(hp[b].cp) - var[(size_t)(b0 + b) * ms + i];
    }
    return rc;
}

}  // extern "C"
