// gpk_debug.cu -- development aids (include/gpk.h): each entry point issues exactly one internal routine of the evaluation
// (covariance build, gradient trace, triangular mat-vecs, column dots, log-likelihood) on device pointers with that routine's
// own arguments, so tests/test_gpu_eval_kernels.py can compare it with a host reference kernel by kernel.  No kernels here.
#include "gpk_internal.cuh"

#include <vector>

namespace {

// Per-problem hyper-parameters of `batch` problems: *first gets problem 0 (by value, as the single-problem paths pass it);
// for batch > 1 all records are copied to ARENA_PP and *dev points at them (the staging of the batched pipelines).
int stage_debug_params(gpk_handle h, const double* thetas, int D, int has_s, double s, int batch, ProblemParams* first,
                       const ProblemParams** dev) {
    std::vector<ProblemParams> hp((size_t)batch);
    for (int b = 0; b < batch; ++b) {
        int rc = gpk_make_problem_params(h, thetas + (size_t)b * gpk_theta_len(h, D), D, has_s, s, &hp[b]);
        if (rc) return rc;
    }
    *first = hp[0];
    *dev = nullptr;
    if (batch > 1) {
        ARENA_OR_FAIL(pp, ProblemParams*, h, ARENA_PP, (size_t)batch * sizeof(ProblemParams));
        // pageable source: the runtime has staged the bytes when the call returns, so hp may go out of scope
        GPK_CUDA(h, cudaMemcpyAsync(pp, hp.data(), (size_t)batch * sizeof(ProblemParams), cudaMemcpyHostToDevice, h->stream));
        *dev = pp;
    }
    return GPK_OK;
}

}  // namespace

extern "C" {

int gpk_debug_cov(gpk_handle h, int mode, const double* dX1, int m, int64_t ldx1, const double* dX2, int n, int64_t ldx2, int D,
                  const double* thetas_host, int has_sigma_noise, double sigma_noise, double* dK, int64_t ldk, int mp, int np,
                  int batch, int64_t strideX1, int64_t strideX2, int64_t strideK) {
    const bool ok = mode >= GPK_DEBUG_COV_SYM_FULL && mode <= GPK_DEBUG_COV_CROSS && batch >= 1 && m >= 0 && ldx1 >= m &&
                    (mode != GPK_DEBUG_COV_SYM_FULL || (batch == 1 && ldk >= m)) &&
                    (mode != GPK_DEBUG_COV_SYM_LOWER_PAD || (mp >= m && mp % GPK_TILE == 0)) &&
                    (mode != GPK_DEBUG_COV_CROSS || (ldk >= (mp > m ? mp : m) && n >= 0 && ldx2 >= n));
    int rc = gpk_check_args(h, "gpk_debug_cov", ok, 0, 0, 0, D, 0);
    if (rc) return rc;
    ProblemParams pp0;
    const ProblemParams* ppd;
    rc = stage_debug_params(h, thetas_host, D, has_sigma_noise, sigma_noise, batch, &pp0, &ppd);
    if (rc) return rc;
    if (mode == GPK_DEBUG_COV_SYM_FULL) return gpk_cov_sym_full(h, dX1, m, ldx1, pp0.cp, dK, ldk);
    if (mode == GPK_DEBUG_COV_SYM_LOWER_PAD) return gpk_cov_sym_lower_padded(h, dX1, m, ldx1, pp0.cp, dK, mp, batch, strideX1, ppd);
    return gpk_cov_cross(h, dX1, m, ldx1, dX2, n, ldx2, pp0.cp, dK, ldk, mp, np, batch, strideX1, strideX2, strideK, ppd);
}

int gpk_debug_grad_trace(gpk_handle h, const double* dKinv, int N, const double* dX, int n, int D, int64_t ldx,
                         const double* dalpha, const double* thetas_host, int nparams, double* dg, int batch, int64_t strideX,
                         int64_t strideOut) {
    int rc = gpk_check_args(h, "gpk_debug_grad_trace", batch >= 1 && N % GPK_TILE == 0 && N >= n, n, 1, ldx, D, nparams);
    if (rc) return rc;
    ProblemParams pp0;
    const ProblemParams* ppd;
    rc = stage_debug_params(h, thetas_host, D, 0, 0.0, batch, &pp0, &ppd);
    if (rc) return rc;
    ARENA_OR_FAIL(scratch, double*, h, ARENA_MISC, (size_t)batch * gpk_grad_scratch_doubles(N, D) * sizeof(double));
    return gpk_grad_trace(h, dKinv, N, dX, n, ldx, dalpha, pp0, nparams, dg, scratch, batch, strideX, ppd, strideOut);
}

int gpk_debug_trmv(gpk_handle h, int transposed, const double* dLi, int N, const double* dx, double* dout, int batch) {
    if (!h) return GPK_EINVAL;
    if (N <= 0 || N % GPK_TILE || batch < 1) return gpk_set_error(h, GPK_EINVAL, "gpk_debug_trmv: bad arguments N=%d batch=%d", N, batch);
    if (transposed) return gpk_trmv_lower_t(h, dLi, N, dx, dout, batch);
    ARENA_OR_FAIL(scratch, double*, h, ARENA_MISC, (size_t)batch * gpk_trmv_scratch_doubles(N) * sizeof(double));
    return gpk_trmv_lower(h, dLi, N, dx, dout, scratch, batch);
}

int gpk_debug_colwise_dot(gpk_handle h, const double* dM, int64_t ld, int rows, int cols, const double* dv, double* dout,
                          int square, int batch, int64_t strideM, int64_t strideV, int64_t strideOut) {
    if (!h) return GPK_EINVAL;
    if (rows < 0 || ld < rows || batch < 1 || (!square && !dv))
        return gpk_set_error(h, GPK_EINVAL, "gpk_debug_colwise_dot: bad arguments");
    return gpk_colwise_dot(h, dM, ld, rows, cols, dv, dout, square, batch, strideM, strideV, strideOut);
}

int gpk_debug_loglik(gpk_handle h, const double* dA, int N, int n, const double* dy, const double* dalpha, double* dout,
                     int batch, int64_t strideOut) {
    if (!h) return GPK_EINVAL;
    if (n < 0 || N < n || batch < 1) return gpk_set_error(h, GPK_EINVAL, "gpk_debug_loglik: bad arguments");
    return gpk_loglik(h, dA, N, n, dy, dalpha, dout, batch, strideOut);
}

}  // extern "C"
