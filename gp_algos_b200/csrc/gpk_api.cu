// gpk_api.cu -- C ABI (include/gpk.h), part 1: handle lifetime and the fine-grained MatrixUtils-level entry points
// (covariance, cholesky, triangular solve / inverse on caller-supplied matrices).  The fused GpPredictor pipelines
// live in gpk_gp.cu.  Everything numeric runs in CUDA kernels; there is no CPU fallback -- a missing device is an error.
#include "gpk_internal.cuh"

#include <stdarg.h>
#include <stdlib.h>

#include <new>

// ------------------------------------------------------------------------------------------------
// handle
// ------------------------------------------------------------------------------------------------
int gpk_set_error(gpk_handle h, int status, const char* fmt, ...) {
    if (h) {
        va_list ap;
        va_start(ap, fmt);
        vsnprintf(h->err, sizeof(h->err), fmt, ap);
        va_end(ap);
    }
    return status;
}

int gpk_check_args(gpk_handle h, const char* fn, bool ok, int n, int n_min, int64_t ldx, int D, int nparams) {
    const char* bad = !h ? "null handle"
                    : (!ok || n < n_min || ldx < n) ? "bad arguments"
                    : (D < 1 || D > GPK_MAX_D) ? "feature dimension out of range"
                    : (nparams < 0 || nparams > gpk_theta_len(h, D)) ? "nparams out of range"
                    : nullptr;
    if (!bad) return GPK_OK;
    return gpk_set_error(h, GPK_EINVAL, "%s: %s (n=%d, ldx=%lld, D=%d of 1..%d, nparams=%d)", fn, bad, n, (long long)ldx, D,
                         GPK_MAX_D, nparams);
}

void* gpk_arena(gpk_handle h, int which, size_t bytes) {
    if (bytes <= h->arena_bytes[which] && h->arena[which]) return h->arena[which];
    if (h->cap) {  // stream capture in progress: allocation would synchronise; the capturing caller falls back to eager launches
        gpk_set_error(h, GPK_ENOMEM, "arena %d would have to grow during graph capture", which);
        return nullptr;
    }
    if (h->arena[which]) {
        cudaStreamSynchronize(h->stream);
        for (int i = 0; i < GPK_NSIDE; ++i) cudaStreamSynchronize(h->side[i]);
        for (int i = 0; i < GPK_NPIPE; ++i) cudaStreamSynchronize(h->pipe[i]);
        for (int i = 0; i < GPK_NGROUP - 1; ++i) cudaStreamSynchronize(h->grp[i]);
        cudaFree(h->arena[which]);
        h->arena[which] = nullptr;
        h->arena_bytes[which] = 0;
    }
    bytes = (bytes + 255) & ~(size_t)255;
    void* p = nullptr;
    if (cudaMalloc(&p, bytes) != cudaSuccess) {
        cudaGetLastError();
        gpk_set_error(h, GPK_ENOMEM, "cudaMalloc of %zu bytes failed (arena %d)", bytes, which);
        return nullptr;
    }
    h->arena[which] = p;
    h->arena_bytes[which] = bytes;
    h->arena_epoch++;
    return p;
}

int gpk_upload_matrix(gpk_handle h, double* dst, const double* src, int rows, int cols, int64_t ld) {
    if (rows <= 0 || cols <= 0) return GPK_OK;
    GPK_CUDA(h, cudaMemcpy2DAsync(dst, (size_t)rows * sizeof(double), src, (size_t)ld * sizeof(double),
                                  (size_t)rows * sizeof(double), (size_t)cols, cudaMemcpyHostToDevice, h->stream));
    return GPK_OK;
}
int gpk_download_matrix(gpk_handle h, double* dst, int64_t ld, const double* src, int rows, int cols) {
    if (rows <= 0 || cols <= 0) return GPK_OK;
    GPK_CUDA(h, cudaMemcpy2DAsync(dst, (size_t)ld * sizeof(double), src, (size_t)rows * sizeof(double),
                                  (size_t)rows * sizeof(double), (size_t)cols, cudaMemcpyDeviceToHost, h->stream));
    return GPK_OK;
}

int gpk_upload_padded(gpk_handle h, double* dst, int N, const double* src, int n, int64_t lds, int form, int* d_notsym) {
    ARENA_OR_FAIL(dIn, double*, h, ARENA_IO, (size_t)n * n * sizeof(double));
    int rc = gpk_upload_matrix(h, dIn, src, n, n, lds);
    return rc ? rc : gpk_load_padded(h, dst, N, dIn, n, n, form, d_notsym);
}
int gpk_download_tri(gpk_handle h, double* dst, int64_t ldd, const double* src, int N, int n, int transpose) {
    ARENA_OR_FAIL(dOut, double*, h, ARENA_IO, (size_t)n * n * sizeof(double));
    int rc = gpk_store_tri(h, dOut, n, src, N, n, transpose);
    return rc ? rc : gpk_download_matrix(h, dst, ldd, dOut, n, n);
}

// after a single factorisation: fetch info, map to status
int gpk_finish_info(gpk_handle h) {
    int info = 0;
    GPK_CUDA(h, cudaMemcpyAsync(&info, h->d_info, sizeof(int), cudaMemcpyDeviceToHost, h->stream));
    GPK_CUDA(h, cudaStreamSynchronize(h->stream));
    h->last_info = info;
    if (info != 0) return gpk_set_error(h, GPK_ENOTPD, "matrix not positive definite: leading minor %d", info);
    return GPK_OK;
}

extern "C" {

const char* gpk_version(void) { return "gpk 0.2 (sm_100a, FP64 DMMA)"; }

int gpk_create(gpk_handle* out, int device, void* stream) {
    if (!out) return GPK_EINVAL;
    *out = nullptr;
    int count = 0;
    if (cudaGetDeviceCount(&count) != cudaSuccess || count <= 0 || device < 0 || device >= count) return GPK_ECUDA;
    if (cudaSetDevice(device) != cudaSuccess) return GPK_ECUDA;
    gpk_handle h = new (std::nothrow) gpk_handle_s();
    if (!h) return GPK_ENOMEM;
    memset(h, 0, sizeof(*h));
    h->device = device;
    if (stream) {
        h->stream = (cudaStream_t)stream;
        h->own_stream = false;
    } else {
        // own main stream at the highest priority: its (critical-path) CTAs are scheduled before the side streams'
        int least = 0, greatest = 0;
        cudaDeviceGetStreamPriorityRange(&least, &greatest);
        if (cudaStreamCreateWithPriority(&h->stream, cudaStreamNonBlocking, greatest) != cudaSuccess) { delete h; return GPK_ECUDA; }
        h->own_stream = true;
    }
    h->main_stream = h->stream;
    if (cudaDeviceGetAttribute(&h->num_sms, cudaDevAttrMultiProcessorCount, device) != cudaSuccess || h->num_sms <= 0) h->num_sms = 148;
    if (cudaMallocHost((void**)&h->h_pinned, 4096 * sizeof(double)) != cudaSuccess ||
        cudaMalloc((void**)&h->d_info, 4 * sizeof(int)) != cudaSuccess) {
        delete h;
        return GPK_ENOMEM;
    }
    cudaMemset(h->d_info, 0, 4 * sizeof(int));
    // side streams (off-critical-path GEMMs that are joined inside a recursion node) run one priority step above the
    // pipelined driver's bulk streams, which take the lowest priority
    int least = 0, greatest = 0, mainprio = 0;
    cudaDeviceGetStreamPriorityRange(&least, &greatest);
    cudaStreamGetPriority(h->stream, &mainprio);
    // numerically lower = more urgent; [greatest, least] is e.g. [-5, 0]
    // below the main stream: side (fork/join of the recursion, near-critical panels) two levels above pipe (lowest) when the
    // device has that many levels, else one level or none
    const bool wide = least - 2 > greatest && mainprio < least - 2;
    const int sideprio = wide ? least - 2 : ((mainprio < least && least - 1 >= greatest) ? least - 1 : least);
    h->prio_main = mainprio; h->prio_side = sideprio; h->prio_pipe = least;
    const char* gm = getenv("GPK_GRAPH");
    const char* tr = getenv("GPK_TRACE");
    h->graph_mode = (tr && atoi(tr) > 0) ? 0 : (gm ? atoi(gm) : 1);   // the trace timeline needs eager launches
    for (int i = 0; i < GPK_NSIDE; ++i)
        if (cudaStreamCreateWithPriority(&h->side[i], cudaStreamNonBlocking, sideprio) != cudaSuccess) { delete h; return GPK_ECUDA; }
    for (int i = 0; i < GPK_NPIPE; ++i)
        if (cudaStreamCreateWithPriority(&h->pipe[i], cudaStreamNonBlocking, least) != cudaSuccess) { delete h; return GPK_ECUDA; }
    for (int i = 0; i < GPK_NGROUP - 1; ++i)
        if (cudaStreamCreateWithPriority(&h->grp[i], cudaStreamNonBlocking, mainprio) != cudaSuccess) { delete h; return GPK_ECUDA; }
    for (int i = 0; i < GPK_NEVENTS; ++i)
        if (cudaEventCreateWithFlags(&h->evpool[i], cudaEventDisableTiming) != cudaSuccess) { delete h; return GPK_ECUDA; }
    *out = h;
    return GPK_OK;
}

int gpk_destroy(gpk_handle h) {
    if (!h) return GPK_OK;
    cudaSetDevice(h->device);
    cudaStreamSynchronize(h->stream);
    gpk_graph_drop_all(h);
    for (int i = 0; i < GPK_NSIDE; ++i)
        if (h->side[i]) { cudaStreamSynchronize(h->side[i]); cudaStreamDestroy(h->side[i]); }
    for (int i = 0; i < GPK_NPIPE; ++i)
        if (h->pipe[i]) { cudaStreamSynchronize(h->pipe[i]); cudaStreamDestroy(h->pipe[i]); }
    for (int i = 0; i < GPK_NGROUP - 1; ++i)
        if (h->grp[i]) { cudaStreamSynchronize(h->grp[i]); cudaStreamDestroy(h->grp[i]); }
    for (int i = 0; i < GPK_NARENA; ++i)
        if (h->arena[i]) cudaFree(h->arena[i]);
    if (h->h_pinned) cudaFreeHost(h->h_pinned);
    if (h->res_pinned) cudaFreeHost(h->res_pinned);
    if (h->d_info) cudaFree(h->d_info);
    for (int i = 0; i < GPK_NEVENTS; ++i)
        if (h->evpool[i]) cudaEventDestroy(h->evpool[i]);
    if (h->own_stream) cudaStreamDestroy(h->stream);
    free(h->pp_host);
    delete h;
    return GPK_OK;
}

const char* gpk_last_error(gpk_handle h) { return h ? h->err : "null handle"; }
int gpk_last_info(gpk_handle h) { return h ? h->last_info : 0; }
int64_t gpk_launch_count(gpk_handle h) { return h ? h->launches : 0; }
int gpk_set_kernel_family(gpk_handle h, int family) {
    if (!h || (family != GPK_KERNEL_SE_ARD && family != GPK_KERNEL_CO2)) return gpk_set_error(h, GPK_EINVAL, "unknown kernel family %d", family);
    h->kernel_family = family;
    return GPK_OK;
}
int gpk_get_kernel_family(gpk_handle h) { return h ? h->kernel_family : GPK_EINVAL; }
int gpk_theta_length(gpk_handle h, int D) { return h ? gpk_theta_len(h, D) : GPK_EINVAL; }
int gpk_set_graph_mode(gpk_handle h, int on) {
    if (!h) return GPK_EINVAL;
    h->graph_mode = on < 0 ? 0 : (on > 2 ? 2 : on);
    if (!on) { cudaStreamSynchronize(h->stream); gpk_graph_drop_all(h); }
    return GPK_OK;
}

int gpk_synchronize(gpk_handle h) {
    GPK_CUDA(h, cudaStreamSynchronize(h->stream));
    return GPK_OK;
}

// ------------------------------------------------------------------------------------------------
// covariance
// ------------------------------------------------------------------------------------------------
int gpk_cov_se_ard_dev(gpk_handle h, const double* dX, int n, int D, int64_t ldx, const double* theta, double* dK, int64_t ldk) {
    int rc = gpk_check_args(h, "gpk_cov_se_ard_dev", ldk >= n, n, 0, ldx, D, 0);
    if (rc) return rc;
    CovParams cp;
    rc = gpk_make_cov_params(h, theta, D, 0, 0.0, &cp);
    if (rc) return rc;
    return gpk_cov_sym_full(h, dX, n, ldx, cp, dK, ldk);
}

int gpk_cov_se_ard(gpk_handle h, const double* X, int n, int D, int64_t ldx, const double* theta, double* K, int64_t ldk) {
    int rc = gpk_check_args(h, "gpk_cov_se_ard", ldk >= n, n, 0, ldx, D, 0);
    if (rc || n == 0) return rc;
    GPK_CUDA(h, cudaSetDevice(h->device));
    ARENA_OR_FAIL(dX, double*, h, ARENA_X, (size_t)n * D * sizeof(double));
    ARENA_OR_FAIL(dK, double*, h, ARENA_IO, (size_t)n * n * sizeof(double));
    rc = gpk_upload_matrix(h, dX, X, n, D, ldx);
    if (rc) return rc;
    rc = gpk_cov_se_ard_dev(h, dX, n, D, n, theta, dK, n);
    if (rc) return rc;
    rc = gpk_download_matrix(h, K, ldk, dK, n, n);
    if (rc) return rc;
    return gpk_synchronize(h);
}

int gpk_cov_cross_se_ard_dev(gpk_handle h, const double* dX1, int m, int64_t ldx1, const double* dX2, int n, int64_t ldx2,
                             int D, const double* theta, double* dK, int64_t ldk) {
    int rc = gpk_check_args(h, "gpk_cov_cross_se_ard_dev", m >= 0 && ldx1 >= m && ldk >= m, n, 0, ldx2, D, 0);
    if (rc) return rc;
    CovParams cp;
    rc = gpk_make_cov_params(h, theta, D, 0, 0.0, &cp);
    if (rc) return rc;
    return gpk_cov_cross(h, dX1, m, ldx1, dX2, n, ldx2, cp, dK, ldk, m, n);
}

int gpk_cov_cross_se_ard(gpk_handle h, const double* X1, int m, int64_t ldx1, const double* X2, int n, int64_t ldx2, int D,
                         const double* theta, double* K, int64_t ldk) {
    int rc = gpk_check_args(h, "gpk_cov_cross_se_ard", m >= 0 && ldx1 >= m && ldk >= m, n, 0, ldx2, D, 0);
    if (rc || m == 0 || n == 0) return rc;
    GPK_CUDA(h, cudaSetDevice(h->device));
    ARENA_OR_FAIL(dX, double*, h, ARENA_X, (size_t)(m + n) * D * sizeof(double));
    ARENA_OR_FAIL(dK, double*, h, ARENA_IO, (size_t)m * n * sizeof(double));
    double* dX2 = dX + (size_t)m * D;
    rc = gpk_upload_matrix(h, dX, X1, m, D, ldx1);
    if (rc) return rc;
    rc = gpk_upload_matrix(h, dX2, X2, n, D, ldx2);
    if (rc) return rc;
    rc = gpk_cov_cross_se_ard_dev(h, dX, m, m, dX2, n, n, D, theta, dK, m);
    if (rc) return rc;
    rc = gpk_download_matrix(h, K, ldk, dK, m, n);
    if (rc) return rc;
    return gpk_synchronize(h);
}

int gpk_cov_deriv_se_ard(gpk_handle h, int param_num, const double* X, int n, int D, int64_t ldx, const double* theta,
                         double* dKout, int64_t ldk) {
    int rc = gpk_check_args(h, "gpk_cov_deriv_se_ard", ldk >= n, n, 0, ldx, D, 0);
    if (rc) return rc;
    if (param_num < 1 || param_num > gpk_theta_len(h, D))
        return gpk_set_error(h, GPK_EINVAL, "scala.MatchError: hyper-parameter %d outside 1..%d", param_num, gpk_theta_len(h, D));
    if (n == 0) return GPK_OK;
    GPK_CUDA(h, cudaSetDevice(h->device));
    ARENA_OR_FAIL(dX, double*, h, ARENA_X, (size_t)n * D * sizeof(double));
    ARENA_OR_FAIL(dK, double*, h, ARENA_IO, (size_t)n * n * sizeof(double));
    CovParams cp;
    rc = gpk_make_cov_params(h, theta, D, 0, 0.0, &cp);
    if (rc) return rc;
    rc = gpk_upload_matrix(h, dX, X, n, D, ldx);
    if (rc) return rc;
    rc = gpk_cov_deriv(h, param_num, dX, n, n, cp, theta[0], theta[D + 1], theta + 1, dK, n);
    if (rc) return rc;
    rc = gpk_download_matrix(h, dKout, ldk, dK, n, n);
    if (rc) return rc;
    return gpk_synchronize(h);
}

// ------------------------------------------------------------------------------------------------
// cholesky / triangular solves / triangular inverse on caller-supplied matrices
// ------------------------------------------------------------------------------------------------
int gpk_potrf_lower(gpk_handle h, const double* A, int n, int64_t lda, double* L, int64_t ldl, int check_symmetric) {
    if (!h || n < 0 || lda < n || ldl < n) return gpk_set_error(h, GPK_EINVAL, "gpk_potrf_lower: bad dimensions");
    if (n == 0) return GPK_OK;
    GPK_CUDA(h, cudaSetDevice(h->device));
    const int N = gpk_pad(n);
    ARENA_OR_FAIL(dA, double*, h, ARENA_A, (size_t)N * N * sizeof(double));
    ARENA_OR_FAIL(dLi, double*, h, ARENA_B, (size_t)N * N * sizeof(double));
    ARENA_OR_FAIL(dT, double*, h, ARENA_T, gpk_chol_scratch_doubles(N) * sizeof(double));
    int* d_notsym = h->d_info + 1;
    GPK_CUDA(h, cudaMemsetAsync(d_notsym, 0, sizeof(int), h->stream));
    int rc = gpk_upload_padded(h, dA, N, A, n, lda, GPK_PAD_SYM, check_symmetric ? d_notsym : nullptr);
    if (rc) return rc;
    if (check_symmetric) {
        int ns = 0;
        GPK_CUDA(h, cudaMemcpyAsync(&ns, d_notsym, sizeof(int), cudaMemcpyDeviceToHost, h->stream));
        GPK_CUDA(h, cudaStreamSynchronize(h->stream));
        if (ns) return gpk_set_error(h, GPK_ENOTSYM, "matrix is not symmetric");
    }
    rc = gpk_potrf_factor(h, dA, dLi, dT, N, h->d_info);     // L only: n^3/3 flops (no L^-1, no K^-1)
    if (rc) return rc;
    rc = gpk_finish_info(h);
    if (rc) return rc;
    rc = gpk_download_tri(h, L, ldl, dA, N, n, 0);
    if (rc) return rc;
    return gpk_synchronize(h);
}

int gpk_trtri(gpk_handle h, int is_upper, const double* T, int n, int64_t ldt, double* Tinv, int64_t ldi) {
    if (!h || n < 0 || ldt < n || ldi < n) return gpk_set_error(h, GPK_EINVAL, "gpk_trtri: bad dimensions");
    if (n == 0) return GPK_OK;
    GPK_CUDA(h, cudaSetDevice(h->device));
    const int N = gpk_pad(n);
    ARENA_OR_FAIL(dA, double*, h, ARENA_A, (size_t)N * N * sizeof(double));
    ARENA_OR_FAIL(dLi, double*, h, ARENA_B, (size_t)N * N * sizeof(double));
    ARENA_OR_FAIL(dT, double*, h, ARENA_T, gpk_chol_scratch_doubles(N) * sizeof(double));
    // an upper-triangular U is handled through its transpose: (U^t)^-1 = (U^-1)^t
    int rc = gpk_upload_padded(h, dA, N, T, n, ldt, is_upper ? GPK_PAD_UPPER : GPK_PAD_LOWER);
    if (rc) return rc;
    rc = gpk_trtri_lower(h, dA, dLi, dT, N);
    if (rc) return rc;
    rc = gpk_download_tri(h, Tinv, ldi, dLi, N, n, is_upper ? 1 : 0);
    if (rc) return rc;
    return gpk_synchronize(h);
}

// Blocked substitution on the padded lower-triangular Lw (N x N, ld N) with the inverses of its 128 x 128 diagonal blocks
// (Di: block k at Di + k*128*128, ld 128).  O(n^2) work per right-hand side, nothing n x n is inverted:
//   forward  (X = Lw^-1 B):  X1 = solve(L11, B1);  B2 -= L21 X1;    X2 = solve(L22, B2)
//   backward (X = Lw^-t B):  X2 = solve(L22^t, B2); B1 -= L21^t X2;  X1 = solve(L11^t, B1)
// with the 128-row base case X_k = Di_k B_k (or Di_k^t B_k).  B is overwritten; X is a second buffer of the same shape.
// M > 0: B, X are N x M (ld N) and every step is a DMMA GEMM; M == 0: one vector, every step is an HBM-bound mat-vec.
}  // extern "C"
namespace {
int trsm_rec(gpk_handle h, const double* Lw, const double* Di, int N, int backward, double* B, double* X, int M, int r0, int len) {
    if (len == GPK_TILE) {
        const double* Dk = Di + (size_t)(r0 / GPK_TILE) * GPK_TILE * GPK_TILE;
        if (M == 0) return gpk_gemv(h, backward, GPK_TILE, GPK_TILE, 1.0, Dk, GPK_TILE, B + r0, 0.0, X + r0);
        GemmDesc g = gemm_desc();
        g.P = B + r0; g.ldp = N; g.p_kcontig = 1;              // P(r,k) = B_k(k, r)
        g.Q = Dk; g.ldq = GPK_TILE;
        g.D = X + r0; g.ldd = N; g.R = M; g.S = GPK_TILE; g.K = GPK_TILE;
        if (!backward) { g.q_kcontig = 0; g.ke_s = 1; }        // Q(s,k) = Di_k(s,k), zero for k > s
        else           { g.q_kcontig = 1; g.kb_s = 1; }        // Q(s,k) = Di_k(k,s), zero for k < s
        return gpk_gemm(h, g);
    }
    const int n1 = (len / GPK_TILE / 2) * GPK_TILE, n2 = len - n1;
    const double* L21 = Lw + (r0 + n1) + (int64_t)r0 * N;
    int rc;
    if (!backward) {
        rc = trsm_rec(h, Lw, Di, N, 0, B, X, M, r0, n1);
        if (rc) return rc;
        if (M == 0) rc = gpk_gemv(h, 0, n2, n1, -1.0, L21, N, X + r0, 1.0, B + r0 + n1);
        else {
            GemmDesc g = gemm_desc();
            g.P = X + r0; g.ldp = N; g.p_kcontig = 1;          // P(r,k) = X1(k, r)
            g.Q = L21; g.ldq = N; g.q_kcontig = 0;             // Q(s,k) = L21(s, k)
            g.D = B + r0 + n1; g.ldd = N; g.Cin = g.D; g.ldc = N;
            g.R = M; g.S = n2; g.K = n1; g.alpha = -1.0; g.beta = 1.0;
            rc = gpk_gemm(h, g);
        }
        if (rc) return rc;
        return trsm_rec(h, Lw, Di, N, 0, B, X, M, r0 + n1, n2);
    }
    rc = trsm_rec(h, Lw, Di, N, 1, B, X, M, r0 + n1, n2);
    if (rc) return rc;
    if (M == 0) rc = gpk_gemv(h, 1, n2, n1, -1.0, L21, N, X + r0 + n1, 1.0, B + r0);
    else {
        GemmDesc g = gemm_desc();
        g.P = X + r0 + n1; g.ldp = N; g.p_kcontig = 1;         // P(r,k) = X2(k, r)
        g.Q = L21; g.ldq = N; g.q_kcontig = 1;                 // Q(s,k) = L21(k, s)
        g.D = B + r0; g.ldd = N; g.Cin = g.D; g.ldc = N;
        g.R = M; g.S = n1; g.K = n2; g.alpha = -1.0; g.beta = 1.0;
        rc = gpk_gemm(h, g);
    }
    if (rc) return rc;
    return trsm_rec(h, Lw, Di, N, 1, B, X, M, r0, n1);
}
}  // namespace

// Lw: padded lower factor on the device.  Inverts its diagonal 128-blocks into Di (one launch) and substitutes.
int gpk_trsm_padded(gpk_handle h, const double* Lw, double* Di, int N, int backward, double* B, double* X, int M, int nvec) {
    int rc = gpk_base_potrf_trtri(h, const_cast<double*>(Lw), N, Di, GPK_TILE, h->d_info + 2, 0, 1, N / GPK_TILE,
                                  (int64_t)GPK_TILE * (N + 1), (int64_t)GPK_TILE * GPK_TILE, 0, GPK_TILE);
    if (rc) return rc;
    if (M > 0) return trsm_rec(h, Lw, Di, N, backward, B, X, M, 0, N);
    for (int c = 0; c < nvec && !rc; ++c) rc = trsm_rec(h, Lw, Di, N, backward, B + (size_t)c * N, X + (size_t)c * N, 0, 0, N);
    return rc;
}

extern "C" {

int gpk_trsm(gpk_handle h, int upper, int transposed, const double* T, int n, int64_t ldt, const double* B, int nrhs,
             int64_t ldb, double* Xout, int64_t ldx) {
    if (!h || n < 0 || nrhs < 0 || ldt < n || ldb < n || ldx < n) return gpk_set_error(h, GPK_EINVAL, "gpk_trsm: bad dimensions");
    if (n == 0 || nrhs == 0) return GPK_OK;
    GPK_CUDA(h, cudaSetDevice(h->device));
    // The stored matrix is lower triangular iff (upper XOR transposed) == 0.
    const int stored_upper = (upper != 0) != (transposed != 0);
    // a handful of right-hand sides go column by column through the mat-vec path (no padding to a 128-column GEMM operand)
    const bool vec = nrhs <= 4;
    const int N = gpk_pad(n), M = vec ? nrhs : gpk_pad(nrhs);
    ARENA_OR_FAIL(dA, double*, h, ARENA_A, (size_t)N * N * sizeof(double));
    ARENA_OR_FAIL(dDi, double*, h, ARENA_T, (size_t)N * GPK_TILE * sizeof(double));
    ARENA_OR_FAIL(dB, double*, h, ARENA_IO2, (size_t)2 * N * M * sizeof(double));
    double* dX = dB + (size_t)N * M;
    // dA = lower-triangular Lw (= stored or stored^t)
    int rc = gpk_upload_padded(h, dA, N, T, n, ldt, stored_upper ? GPK_PAD_UPPER : GPK_PAD_LOWER);
    if (rc) return rc;
    GPK_CUDA(h, cudaMemsetAsync(dB, 0, (size_t)2 * N * M * sizeof(double), h->stream));
    GPK_CUDA(h, cudaMemcpy2DAsync(dB, (size_t)N * sizeof(double), B, (size_t)ldb * sizeof(double), (size_t)n * sizeof(double),
                                  (size_t)nrhs, cudaMemcpyHostToDevice, h->stream));
    // effective operand E: lower (forwardSolve) -> E = Lw, X = Lw^-1 B;  upper (backSolve) -> E = Lw^t, X = Lw^-t B
    rc = gpk_trsm_padded(h, dA, dDi, N, upper ? 1 : 0, dB, dX, vec ? 0 : M, nrhs);
    if (rc) return rc;
    GPK_CUDA(h, cudaMemcpy2DAsync(Xout, (size_t)ldx * sizeof(double), dX, (size_t)N * sizeof(double), (size_t)n * sizeof(double),
                                  (size_t)nrhs, cudaMemcpyDeviceToHost, h->stream));
    return gpk_synchronize(h);
}

// Cholesky of a device-resident matrix, in place: on exit the lower triangle of dA holds L and the strict upper triangle is
// zero (Breeze `cholesky` semantics, GpPredictor.scala:120).  Asynchronous on the handle's stream; info_dev (device int, may
// be null -> gpk_last_info after gpk_synchronize is NOT updated) receives 0 or the failing leading minor.
int gpk_potrf_lower_dev(gpk_handle h, double* dA, int n, int64_t lda, int* info_dev) {
    if (!h || !dA || n <= 0 || lda < n) return gpk_set_error(h, GPK_EINVAL, "gpk_potrf_lower_dev: bad dimensions");
    const int N = gpk_pad(n);
    ARENA_OR_FAIL(dLi, double*, h, ARENA_B, (size_t)N * N * sizeof(double));
    ARENA_OR_FAIL(dT, double*, h, ARENA_T, gpk_chol_scratch_doubles(N) * sizeof(double));
    int* info = info_dev ? info_dev : h->d_info;
    const bool in_place = N == n && lda == n && !((uintptr_t)dA & 15);
    double* dW = dA;
    if (!in_place) {
        ARENA_OR_FAIL(dWork, double*, h, ARENA_A, (size_t)N * N * sizeof(double));
        dW = dWork;
    }
    // ~40 launches per block column, most of them small and dependent: a caller that factors the same buffer again (a solver in a
    // loop) replays the launch sequence from a graph, like the evaluation and the EP sweep -- up to N = 4096, where the launch gaps
    // dominate (2.74 -> 2.45 ms at n = 4096; at n = 8192 replay is SLOWER, 8.77 -> 9.27 ms: profiles/r02_potrf_nb.log)
    auto body = [&]() {
        int rc = GPK_OK;
        if (!in_place) rc = gpk_load_padded(h, dW, N, dA, n, lda, GPK_PAD_SYM);
        if (!rc) rc = gpk_potrf_factor(h, dW, dLi, dT, N, info);
        if (!rc) rc = in_place ? gpk_store_tri(h, dA, n, dA, N, n, 0)     // zero the strict upper triangle (element-wise, in place)
                               : gpk_store_tri(h, dA, lda, dW, N, n, 0);
        return rc;
    };
    if (!h->graph_mode || N < 1024 || N > 4096) return body();
    GraphKey key;
    memset(&key, 0, sizeof(key));
    key.p[0] = dA; key.p[1] = dW; key.p[2] = dLi; key.p[3] = dT; key.p[4] = info;
    key.i[0] = n; key.i[1] = N; key.i[2] = lda;
    return gpk_graph_run(h, GPK_SLOT_POTRF, key, 1, body, "Cholesky factorisation");
}

int gpk_syrk_lower_dev(gpk_handle h, const double* dP, int64_t ldp, double* dC, int64_t ldc, int n, int k) {
    if (!h || n <= 0 || k <= 0) return gpk_set_error(h, GPK_EINVAL, "gpk_syrk_lower_dev: bad dimensions");
    GemmDesc g = gemm_desc();
    g.P = dP; g.ldp = ldp; g.Q = dP; g.ldq = ldp;
    g.D = dC; g.ldd = ldc; g.Cin = dC; g.ldc = ldc;
    g.R = n; g.S = n; g.K = k; g.alpha = -1.0; g.beta = 1.0; g.tri_out = 1;
    return gpk_gemm(h, g);
}

}  // extern "C"

// ------------------------------------------------------------------------------------------------
// device-level building blocks of the multi-GPU block-column Cholesky (BASELINE.json config 5; orchestrated one
// process per GPU in gp_algos_b200/distributed.py with NCCL panel broadcasts)
// ------------------------------------------------------------------------------------------------
extern "C" {

int gpk_potrf_inv_block_dev(gpk_handle h, double* dA, double* dLi, int N, int* info_dev) {
    if (!h || N <= 0 || N % GPK_TILE) return gpk_set_error(h, GPK_EINVAL, "gpk_potrf_inv_block_dev: N must be a multiple of 128");
    ARENA_OR_FAIL(dT, double*, h, ARENA_T, gpk_chol_scratch_doubles(N) * sizeof(double));
    return gpk_potrf_inv(h, dA, dLi, dT, N, /*keep_L=*/1, info_dev ? info_dev : h->d_info, 1);
}

int gpk_gemm_nt_dev(gpk_handle h, int m, int p, int k, double alpha, const double* dP, int64_t ldp, const double* dQ,
                    int64_t ldq, double beta, double* dC, int64_t ldc, int q_lower_tri) {
    if (!h || m < 0 || p < 0 || k < 0) return gpk_set_error(h, GPK_EINVAL, "gpk_gemm_nt_dev: bad dimensions");
    if (m == 0 || p == 0) return GPK_OK;
    // C(i,c) = alpha sum_k P(i,k) Q(c,k) + beta C(i,c);  D = C^t: r = c, s = i
    GemmDesc g = gemm_desc();
    g.P = dQ; g.ldp = ldq; g.p_kcontig = 0;
    g.Q = dP; g.ldq = ldp; g.q_kcontig = 0;
    g.D = dC; g.ldd = ldc;
    if (beta != 0.0) { g.Cin = dC; g.ldc = ldc; }
    g.R = p; g.S = m; g.K = k; g.alpha = alpha; g.beta = beta;
    if (q_lower_tri) { g.ke_r = 1; g.heavy_last = 1; }   // Q(c,k) = 0 for k > c
    return gpk_gemm(h, g);
}

int gpk_gemv_dev(gpk_handle h, int trans, int m, int ncols, double alpha, const double* dM, int64_t ld, const double* dx,
                 double beta, double* dy) {
    if (!h || m < 0 || ncols < 0 || ld < m) return gpk_set_error(h, GPK_EINVAL, "gpk_gemv_dev: bad dimensions");
    return gpk_gemv(h, trans, m, ncols, alpha, dM, ld, dx, beta, dy);
}

int gpk_add_diag_dev(gpk_handle h, double* dA, int64_t ld, int n, double value) {
    if (!h || !dA || n < 0 || ld < n) return gpk_set_error(h, GPK_EINVAL, "gpk_add_diag_dev: bad arguments");
    return gpk_add_diag(h, dA, ld, n, value);
}

int gpk_sum_log_diag_dev(gpk_handle h, const double* dA, int64_t ld, int n, double* out_dev, int accumulate) {
    if (!h || !dA || !out_dev || n < 0 || ld < n) return gpk_set_error(h, GPK_EINVAL, "gpk_sum_log_diag_dev: bad arguments");
    return gpk_sum_log_diag(h, dA, ld, n, out_dev, accumulate);
}

}  // extern "C"
