/*
 * gpk.h -- C ABI of libgpk: the B200-native (sm_100a) dense FP64 Gaussian-process linear algebra
 * that replaces the hot path of astroHaoPeng/gp_algos.  No torch types, no C++ types: plain pointers
 * and sizes, so the same entry points can be bound from Scala/JVM (JNA / JNI / Java FFM), Python
 * (ctypes) or C.  See INTEGRATION.md for the reference-side bindings.
 *
 * Conventions (SURVEY.md 8(b)):
 *   - every matrix is COLUMN-MAJOR FP64 with an explicit leading dimension (Breeze DenseMatrix
 *     layout: element (r,c) at base[r + c*ld]); vectors are contiguous.
 *   - theta is the reference's hyper-parameter packing [signalVar, lengthScale_1..D, noiseVar]
 *     (utils/KernelRequisites.scala:39-58), length D+2.  signalVar/noiseVar are std-dev-like and
 *     squared inside the kernel (KernelRequisites.scala:66-72).
 *   - functions without a suffix take HOST pointers, copy in/out and return when results are on
 *     the host (synchronous, like the Scala functions they replace).  Functions ending in `_dev`
 *     take DEVICE pointers, enqueue on the handle's stream and return without synchronising
 *     (scalars are written to device memory the caller provides).
 *   - all functions return 0 on success or a negative gpk_status; gpk_last_error(h) gives text.
 *     There is NO CPU fallback anywhere in this library.
 *
 * Reference paths below are relative to /root/reference/src/main/scala/.
 */
#ifndef GPK_H
#define GPK_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

typedef struct gpk_handle_s* gpk_handle;

enum gpk_status {
    GPK_OK = 0,
    GPK_EINVAL = -1,   /* IllegalArgumentException (require(...) at GpPredictor.scala:108, MatrixUtils.scala:125) */
    GPK_ENOTSYM = -2,  /* breeze MatrixNotSymmetricException from `cholesky` */
    GPK_ENOTPD = -3,   /* breeze NotConvergedException from `cholesky`; gpk_last_info(h) = failing minor (1-based) */
    GPK_ECUDA = -4,    /* CUDA runtime error */
    GPK_ENOMEM = -5    /* device allocation failed */
};

/* ---- lifetime -------------------------------------------------------------------------------- */
/* One handle = one device + one stream + a grow-only device workspace. Not re-entrant; use one
 * handle per host thread / per GPU.  `stream` may be NULL (the handle creates its own) or a
 * cudaStream_t owned by the caller (e.g. torch.cuda.current_stream().cuda_stream). */
int gpk_create(gpk_handle* out, int device, void* stream);
int gpk_destroy(gpk_handle h);
const char* gpk_last_error(gpk_handle h);
int gpk_last_info(gpk_handle h);
int gpk_synchronize(gpk_handle h);
/* number of kernel launches issued through this handle since creation (bench.py "gpu_launches") */
int64_t gpk_launch_count(gpk_handle h);
const char* gpk_version(void);
/* Development aid, not part of the drop-in surface: runs the 128 x 128 diagonal-block kernel (factor + triangular inverse, the
 * serial spine of every factorisation) once on a synthetic SPD block and returns 17 clock64() stamps, one per phase
 * (tools/base_timing.py prints them; profiles/r02_base_timing.log). */
int gpk_debug_base_timing(gpk_handle h, long long* stamps_host);
/* Development aid: clock64() stamps of the EP site kernel on one synthetic 64-site block (tools/ep_site_timing.py).
 * chain 1: ep_sites_block_w (the reference kernel the tests compare against); chain >= 10: ep_sites_block_p (the default
 * kernel); any other chain: GPK_EINVAL.
 * stamps_host must hold 14 * 64 + 1 = 897 entries: [0..319] five stamps per site of the (scalar) warp, [320] duration in ns of
 * one unstamped launch of the default kernel, [321..576] barrier arrival of four other warps per site, [577..896] phases of
 * tile warp 0 (the last two groups for chain >= 10 only). */
int gpk_debug_ep_site_timing(gpk_handle h, int chain, long long* stamps_host);
/* Development aids, not part of the drop-in surface (tests/test_gpu_ep_kernels.py): each issues exactly one routine of the EP
 * sweep (csrc/gpk_ep.cu) on device pointers, asynchronously on the handle's stream, and returns its status.
 * gpk_debug_ep_scalar: one scalar primitive of the site kernels per element, c_erfcx staged in shared memory as the site kernel
 *   stages it.  Per element i:
 *     RCP, EXP_NEG_SQ, ERFCX_TAB, RATIO, RATIO_FAST   in[i] -> out[i]   (rcp_nr, exp_neg_sq, erfcx_tab, dnorm_over_pnorm,
 *                                                                        dnorm_over_pnorm_fast)
 *     RSQRT        in[i] -> out[2i] = rsqrt_nr, out[2i+1] = libdevice rsqrt
 *     SITE_FAST    in[5i..] = (sii, mui, t_old, n_old, y) -> out[9i..] = (c, g, mu_hat, sig_hat, rs, ct, cn, tau, nu) of
 *                  ep_site_fast, tau and nu finished as ep_sites_block_p finishes them
 *     SITE_SCALAR  in[5i..] as above -> out[6i..] = (ct, cn, c, g, dtau, nu) of ep_site_scalar
 * gpk_debug_ep_sites: one launch of the site kernel (variant 5: ep_sites_block_p, 4: ep_sites_block_w) on the 64 x 64 block Dg
 *   (column-major; the leading bsz x bsz is read) for the sites i0 .. i0+bsz-1 of mu, tau, nu, cav_tau, cav_nu and y; writes
 *   blk = (c[64], g[64]) and W = (I + A)^-1 (64 x 64 column-major).
 * gpk_debug_ep_apply: one launch of ep_apply_gemm for block b (bsz sites) of an n-site sweep: Sigma0 N x N (lower triangle
 *   outside tile (b, b)), Dg the N/64 diagonal 64 x 64 blocks, U and P N x 64 (ld N), mu N.
 * gpk_debug_ep_site_loop: the site loop of one sweep (site kernel, apply and delayed flush of every block; variant from
 *   GPK_EP_SITES) from Sigma0 (N x N lower, N = n rounded up to a multiple of 128) and the n-vectors tau, nu, mu, y; writes the
 *   n-vectors tau, nu, mu, cav_tau, cav_nu after the sweep.
 * gpk_debug_ep_refactor: the posterior re-factorisation from K (n x n, ld n) and the n-vectors tau, nu: L = chol(I + S^1/2 K S^1/2)
 *   and Sigma = K - V^t V (N x N, ld N, lower tiles), mu = Sigma nu (n); waits for the result and returns GPK_ENOTPD if B
 *   is not positive definite. */
enum { GPK_DEBUG_EP_RCP = 0, GPK_DEBUG_EP_RSQRT = 1, GPK_DEBUG_EP_EXP_NEG_SQ = 2, GPK_DEBUG_EP_ERFCX_TAB = 3, GPK_DEBUG_EP_RATIO = 4,
       GPK_DEBUG_EP_RATIO_FAST = 5, GPK_DEBUG_EP_SITE_FAST = 6, GPK_DEBUG_EP_SITE_SCALAR = 7 };
int gpk_debug_ep_scalar(gpk_handle h, int what, const double* d_in, int count, double* d_out);
int gpk_debug_ep_sites(gpk_handle h, int variant, const double* dDg, int i0, int bsz, const double* dmu, double* dtau, double* dnu,
                       double* dcav_tau, double* dcav_nu, const int* dy, double* dblk, double* dW);
int gpk_debug_ep_apply(gpk_handle h, const double* dSigma0, int N, int n, int b, int bsz, const double* dblk, const double* dW,
                       double* dU, double* dP, double* dmu, double* dDg);
int gpk_debug_ep_site_loop(gpk_handle h, const double* dSigma0, int n, const double* dtau, const double* dnu, const double* dmu,
                           const int* dy, double* dtau_out, double* dnu_out, double* dmu_out, double* dcav_tau_out,
                           double* dcav_nu_out);
int gpk_debug_ep_refactor(gpk_handle h, const double* dK, int n, const double* dtau, const double* dnu, double* dL, double* dSigma,
                          double* dmu);
/* Development aid, not part of the drop-in surface (tests/test_gpu_gemm.py): issues exactly one internal DMMA GEMM with the
 * descriptor given field by field and returns its status (GPK_EINVAL, without a launch, for R or S not a multiple of 64, K not
 * a multiple of 16, an odd leading dimension or a pointer that is not 16-byte aligned).  Device pointers; for every 64 x 64
 * tile selected by GPK_GEMM_TRI_OUT and each batch entry b (operands at base + b*stride):
 *   D(r,s) = alpha * sum_{k in [kbeg,kend)} P(r,k) Q(s,k) + beta * Cin(r,s),  D(r,s) at D[s + r*ldd]
 *   P(r,k) at P[k + r*ldp] if p_kcontig else P[r + k*ldp];  Q(s,k) likewise with q_kcontig
 *   kbeg = max(KB_R ? r0 : 0, KB_S ? s0 : 0),  kend = min(K, KE_R ? r0 + 64 : K, KE_S ? s0 + 64 : K)
 * with (r0, s0) the tile's first row / column.  TRI_OUT: only tiles with s0 >= r0; HEAVY_LAST: tiles in reverse launch
 * order.  Cin may be NULL (no beta term) or equal to D. */
enum { GPK_GEMM_TRI_OUT = 1, GPK_GEMM_KB_R = 2, GPK_GEMM_KB_S = 4, GPK_GEMM_KE_R = 8, GPK_GEMM_KE_S = 16, GPK_GEMM_HEAVY_LAST = 32 };
int gpk_debug_gemm(gpk_handle h, const double* P, int64_t ldp, int64_t strideP, const double* Q, int64_t ldq, int64_t strideQ,
                   double* D, int64_t ldd, int64_t strideD, const double* Cin, int64_t ldc, int64_t strideC, int R, int S, int K,
                   int batch, double alpha, double beta, int p_kcontig, int q_kcontig, int flags);
/* Development aids, not part of the drop-in surface (tests/test_gpu_eval_kernels.py): each runs one internal routine of the
 * evaluation once, on device pointers, asynchronously on the handle's stream, and returns its status.  Hyper-parameters are
 * HOST arrays of `batch` theta vectors of the handle's kernel family, back to back; problem b reads X at + b*strideX.
 * gpk_debug_cov: the covariance build of the handle's family.
 *   SYM_FULL       K (m x m, ld ldk) = k(X1, X1) + (sn^2 + sigma_noise) I, lower 64-tiles computed and mirrored; batch 1.
 *   SYM_LOWER_PAD  K (mp x mp, ld mp, problem b at + b*mp*mp; mp a multiple of 128 and >= m): every 64-tile whose 128-block
 *                  is on or below the diagonal, with identity padding beyond m; the 128-blocks above it are not written.
 *   CROSS          K (ld ldk, at + b*strideK) = k(X1, X2) without noise, zero-filled up to (mp, np); nothing beyond.
 * gpk_debug_grad_trace: g[b*strideOut + p] = 1/2 sum_{i,j<n} (alpha_i alpha_j - Kinv_ij) dk_p(x_i, x_j) for p < nparams, reading
 *   the lower 64-tiles of Kinv (N x N at + b*N*N; NULL: alpha alpha^t alone) and alpha (at + b*N).
 * gpk_debug_trmv: out = Li x (transposed == 0) or Li^t x, Li N x N lower (at + b*N*N), x and out at + b*N.
 * gpk_debug_colwise_dot: out[b*strideOut + c] = sum_{r<rows} M[b*strideM + r + c*ld] * (square ? M[..] : v[b*strideV + r]).
 * gpk_debug_loglik: out[b*strideOut] = -1/2 y.alpha - sum_{i<n} log A_ii - n/2 log(2 pi), A N x N at + b*N*N, y, alpha at + b*N. */
enum { GPK_DEBUG_COV_SYM_FULL = 0, GPK_DEBUG_COV_SYM_LOWER_PAD = 1, GPK_DEBUG_COV_CROSS = 2 };
int gpk_debug_cov(gpk_handle h, int mode, const double* dX1, int m, int64_t ldx1, const double* dX2, int n, int64_t ldx2, int D,
                  const double* thetas_host, int has_sigma_noise, double sigma_noise, double* dK, int64_t ldk, int mp, int np,
                  int batch, int64_t strideX1, int64_t strideX2, int64_t strideK);
int gpk_debug_grad_trace(gpk_handle h, const double* dKinv, int N, const double* dX, int n, int D, int64_t ldx,
                         const double* dalpha, const double* thetas_host, int nparams, double* dg, int batch, int64_t strideX,
                         int64_t strideOut);
int gpk_debug_trmv(gpk_handle h, int transposed, const double* dLi, int N, const double* dx, double* dout, int batch);
int gpk_debug_colwise_dot(gpk_handle h, const double* dM, int64_t ld, int rows, int cols, const double* dv, double* dout,
                          int square, int batch, int64_t strideM, int64_t strideV, int64_t strideOut);
int gpk_debug_loglik(gpk_handle h, const double* dA, int N, int n, const double* dy, const double* dalpha, double* dout,
                     int batch, int64_t strideOut);
/* Launch sequences that callers repeat verbatim are captured into CUDA graphs and replayed: the single-problem
 * gpk_gp_nll_grad[_dev] evaluation (an optimiser's objective, GpPredictor.scala:126-142; same buffers and shape, new
 * hyper-parameters through device memory) from its second call on, the device-resident factor-only Cholesky up to n = 4096
 * when the same buffers are factored again, and -- only with GPK_GRAPH_AFTER_EP=k in the environment, after k eager sweeps of one
 * size -- the EP sweep (EpParameterEstimator.scala:37-67; measured slower than eager launches since the round-2 rework).  on = 0: eager launches only; 1 (default,
 * or the GPK_GRAPH environment variable): as described; 2: capture at the first repetition of anything.  Results are
 * bit-identical in every mode.  The batched EP evaluation (gpk_ep_nll_grad_batched) always launches eagerly. */
int gpk_set_graph_mode(gpk_handle h, int on);

/* ---- kernel family -------------------------------------------------------------------------------
 * The reference's GpPredictor works on any utils.KernelRequisites.KernelFunc; two of them are closed-form and are lowered
 * to the device.  The family is a property of the handle and applies to every later call that takes (D, theta):
 *   GPK_KERNEL_SE_ARD  GaussianRbfKernel, utils/KernelRequisites.scala:62-114: theta = [signalVar, lengthScale_1..D, noiseVar]
 *   GPK_KERNEL_CO2     Co2Kernel, gp/regression/Co2Prediction.scala:29-137: 1-D inputs (D must be 1), theta = hp1..hp11,
 *                      k = hp1^2 exp(-r^2/(2 hp2^2)) + hp3^2 exp(-r^2/(2 hp4^2) - 2 sin^2(pi r)/hp5^2)
 *                        + hp6^2 (1 + r^2/(2 hp8 hp7^2))^-hp8 + hp9^2 exp(-r^2/(2 hp10^2)) + hp11^2 [i == j]
 *                      with the derivatives of :66-137; `gradient` is `???` in the reference -> gpk_gp_model_ucb: GPK_EINVAL.
 * A resident model (gpk_model) keeps the family it was fitted with.  The Scala shim selects the family by pattern-matching
 * on the KernelFunc class; other kernels (PMKKernel) stay on the Scala path. */
enum gpk_kernel_family { GPK_KERNEL_SE_ARD = 0, GPK_KERNEL_CO2 = 1 };
int gpk_set_kernel_family(gpk_handle h, int family);
int gpk_get_kernel_family(gpk_handle h);
/* number of hyper-parameters (length of theta) of the handle's family for D-dimensional inputs: D + 2, or 11 */
int gpk_theta_length(gpk_handle h, int D);

/* ---- fine-grained MatrixUtils replacements ---------------------------------------------------- */
/* utils/MatrixUtils.scala:57-70  buildKernelMatrix(kernel, data): symmetric n x n,
 * K(i,j) = sf^2 exp(-1/2 sum_d (x_id-x_jd)^2/l_d^2) + sn^2 [i==j]; lower triangle computed, mirrored. */
int gpk_cov_se_ard(gpk_handle h, const double* X, int n, int D, int64_t ldx, const double* theta,
                   double* K, int64_t ldk);
int gpk_cov_se_ard_dev(gpk_handle h, const double* dX, int n, int D, int64_t ldx, const double* theta_host,
                       double* dK, int64_t ldk);
/* utils/MatrixUtils.scala:44-55,86-97  buildKernelMatrix(kernel, in1, in2): m x n, never adds noise. */
int gpk_cov_cross_se_ard(gpk_handle h, const double* X1, int m, int64_t ldx1, const double* X2, int n,
                         int64_t ldx2, int D, const double* theta, double* K, int64_t ldk);
int gpk_cov_cross_se_ard_dev(gpk_handle h, const double* dX1, int m, int64_t ldx1, const double* dX2, int n,
                             int64_t ldx2, int D, const double* theta_host, double* dK, int64_t ldk);
/* utils/MatrixUtils.scala:72-84 with f = derAfterHyperParam(param_num) (KernelRequisites.scala:76-86;
 * param_num is 1-based like the reference).  Provided for API completeness/tests: the fused
 * gradient (gpk_gp_nll_grad) never materialises these matrices. */
int gpk_cov_deriv_se_ard(gpk_handle h, int param_num, const double* X, int n, int D, int64_t ldx,
                         const double* theta, double* dK, int64_t ldk);

/* breeze `cholesky` at GpPredictor.scala:120 / EpParameterEstimator.scala:58 (LAPACK dpotrf 'L'):
 * A n x n symmetric -> L lower with strict upper zeroed.  check_symmetric != 0 reproduces Breeze's
 * exact-symmetry test (GPK_ENOTSYM).  GPK_ENOTPD + gpk_last_info on a non-positive pivot. */
int gpk_potrf_lower(gpk_handle h, const double* A, int n, int64_t lda, double* L, int64_t ldl,
                    int check_symmetric);
/* Same factorisation of a DEVICE-resident matrix, in place and asynchronous on the handle's stream: on exit the
 * lower triangle of dA holds L and the strict upper triangle is zero.  *info_dev (device int, may be NULL) = 0 or the
 * failing leading minor.  n^3/3 flops: only the 128..512-wide diagonal blocks are inverted (the panels below them are
 * solved as DMMA GEMMs with those inverses); no n x n inverse is formed.  In place without a copy when n is a multiple
 * of 128, lda == n and dA is 16-byte aligned.  bench.py's "cholesky" record times this call. */
int gpk_potrf_lower_dev(gpk_handle h, double* dA, int n, int64_t lda, int* info_dev);
/* utils/MatrixUtils.scala:17-35,115-133  forwardSolve / backSolve, vector or matrix right-hand side.
 * `T` is the triangular matrix as stored (n x n, column-major); transposed != 0 means the operand is
 * T^t (the `L.t` view of GpPredictor.scala:122).  upper != 0 selects backSolve semantics (the
 * EFFECTIVE operand is upper triangular), otherwise forwardSolve (effective operand lower).
 * Blocked substitution, O(n^2) work per right-hand side: the 128 x 128 diagonal blocks are inverted (one launch), the
 * off-diagonal updates are HBM-bound mat-vecs (nrhs <= 4) or DMMA GEMMs (the right-hand sides padded to a multiple of
 * 128 columns); no n x n inverse is formed.  Numerics: each diagonal block is applied through its explicit inverse, so
 * the residual is bounded by O(n eps cond(T_kk)) per block rather than LAPACK dtrsv's O(n eps); on the path's matrices
 * (Cholesky factors of K + sn^2 I, cond(K) <= 1e8) the solves agree with the reference's row-oriented substitution to
 * 1e-9 relative (tests/test_gpu_matrix_utils.py). */
int gpk_trsm(gpk_handle h, int upper, int transposed, const double* T, int n, int64_t ldt,
             const double* B, int nrhs, int64_t ldb, double* Xout, int64_t ldx);
/* utils/MatrixUtils.scala:106-113  invTriangular(matrix, isUpper): dense n x n inverse. */
int gpk_trtri(gpk_handle h, int is_upper, const double* T, int n, int64_t ldt, double* Tinv, int64_t ldi);

/* The Cholesky trailing update on its own (device pointers, asynchronous): C(lower 128-tiles) -= P * P^t with
 * C n x n (ldc) and P n x k (ldp) column-major, n a multiple of 128, k a multiple of 16, 16-byte aligned,
 * even leading dimensions.  This is the DMMA kernel that carries ~all flops of gpk_potrf_lower; bench.py
 * times it in isolation for the FP64 tensor roofline. */
int gpk_syrk_lower_dev(gpk_handle h, const double* dP, int64_t ldp, double* dC, int64_t ldc, int n, int k);

/* ---- fused GpPredictor replacements ----------------------------------------------------------- */
/* gp/regression/GpPredictor.scala:104-124 preComputeComponents + :144-149 logLikelihood.
 * has_sigma_noise/sigma_noise mirror Option[Double]; it is added UN-squared to the diagonal
 * (GpPredictor.scala:116-117).  Outputs: L (n x n, may be NULL), alpha (n), ll (1). */
int gpk_gp_fit(gpk_handle h, const double* X, int n, int D, int64_t ldx, const double* y,
               const double* theta, int has_sigma_noise, double sigma_noise, double* L, int64_t ldl,
               double* alpha, double* ll);
/* Numerics of the fused pipelines (gpk_gp_fit, gpk_gp_nll_grad, gpk_gp_model_*, the batched calls): the factorisation builds
 * L^-1 alongside L (blocked, DMMA), and alpha = L^-t (L^-1 y), V = L^-1 K*^t, K^-1 = L^-t L^-1 are PRODUCTS with that explicit
 * inverse, not substitutions.  Forward error of alpha is therefore bounded by O(n eps cond(L)^2) = O(n eps cond(K)) -- the same
 * order as substitution's bound for the SOLUTION, but without substitution's small-residual guarantee: ||K alpha - y|| / ||y|| is
 * O(n eps cond(K)) rather than O(n eps).  Measured: 2e-12 at n = 65536 (cond ~ 2e6), parity with the reference's row-oriented
 * substitution 1e-9 relative on the BASELINE configs and 1e-7 on the Boston set (cond(K) = 1e8), which is the stated
 * tolerance scaling 1e-9 max(1, cond / 1e5) of the tests.  Callers that need dtrsv-grade residuals use gpk_trsm (blocked
 * substitution on 128-block inverses) on the returned L. */
/* gp/regression/GpPredictor.scala:60-80 logLikelihoodWithDerivatives: ll and g[nparams],
 * g_p = 1/2 tr((alpha alpha^t - K^-1) dK/dtheta_{p+1}).  K, L, L^-1, K^-1 never leave the device
 * and dK/dtheta is never materialised. */
int gpk_gp_nll_grad(gpk_handle h, const double* X, int n, int D, int64_t ldx, const double* y,
                    const double* theta, int has_sigma_noise, double sigma_noise, int nparams,
                    double* ll, double* grad);
/* Same with X (n x D, ld ldx) and y resident on the device; out_dev[0] = ll, out_dev[1..nparams] = g.
 * Asynchronous on the handle's stream; *info_dev (int, device) receives 0 or the failing minor. */
int gpk_gp_nll_grad_dev(gpk_handle h, const double* dX, int n, int D, int64_t ldx, const double* dy,
                        const double* theta_host, int has_sigma_noise, double sigma_noise, int nparams,
                        double* out_dev, int* info_dev);

/* Resident fitted model (GP-UKF / GP-UCB call pattern, GPUnscentedKalmanFilter.scala:77-88,123-147):
 * fit once, keep X, L^-1 and alpha on the device, predict many times. */
typedef struct gpk_model_s* gpk_model;
int gpk_gp_model_fit(gpk_handle h, const double* X, int n, int D, int64_t ldx, const double* y,
                     const double* theta, int has_sigma_noise, double sigma_noise, gpk_model* out, double* ll);
/* Adopt an existing factor (computePosterior(trainingData,testData,l,alphaVec,kernelFunc),
 * GpPredictor.scala:50-58, is handed L and alpha by its caller). */
int gpk_gp_model_from_factor(gpk_handle h, const double* X, int n, int D, int64_t ldx, const double* L,
                             int64_t ldl, const double* alpha, const double* theta, gpk_model* out);
int gpk_gp_model_destroy(gpk_handle h, gpk_model m);
/* alphaVec = L^t \\ (L \\ targets) of the resident model (GpPredictor.scala:121-122), n doubles. */
int gpk_gp_model_get_alpha(gpk_handle h, gpk_model m, double* alpha);
/* gp/optimization/GPOptimizer.scala:48-71: each GP-UCB iteration adds ONE evaluated point (x_new: D doubles, y_new) to the
 * training set and the reference refits from scratch (preComputeComponents, :51).  This updates the resident L^-1 and alpha
 * by the bordered row instead (O(n^2)); afterwards the model equals gpk_gp_model_fit on the enlarged set with the same
 * hyper-parameters and the same Option sigmaNoise; a (has_sigma_noise, sigma_noise) pair that differs from the one the model
 * was fitted with is rejected with GPK_EINVAL (the bordered factor would be inconsistent).  ll_delta (may be NULL) =
 * logLikelihood(new set) - logLikelihood(old set).
 * GPK_ENOTPD (gpk_last_info = n+1) when the enlarged matrix is not positive definite; the model is then unchanged. */
int gpk_gp_model_append(gpk_handle h, gpk_model m, const double* x_new, double y_new, int has_sigma_noise,
                        double sigma_noise, double* ll_delta);
/* number of training points of the resident model */
int gpk_gp_model_size(gpk_handle h, gpk_model m);
/* gp/regression/GpPredictor.scala:45-58 computePosterior: mean (m), sigma (m x m full if
 * want_full_cov, else only the diagonal in sigma[0..m-1]), V = L^-1 K*^t (n x m, may be NULL).
 * The sigma diagonal includes noiseVar^2 (MatrixUtils.scala:63 via GpPredictor.scala:56). */
int gpk_gp_model_predict(gpk_handle h, gpk_model m, const double* Xs, int ms, int64_t ldxs,
                         int want_full_cov, double* mean, double* sigma, int64_t lds, double* V, int64_t ldv);
/* Posterior means of nmodels resident models at the same ms test rows, one call and one synchronisation:
 * mean[j*ms + i].  The GP-UKF step (GPUnscentedKalmanFilter.scala:77-90) asks one GP per state / observation dimension
 * for its mean at every sigma point; the reference does that with (2d+1) x dims computePosterior calls. */
int gpk_gp_models_mean(gpk_handle h, const gpk_model* models, int nmodels, const double* Xs, int ms, int64_t ldxs,
                       double* mean);
/* The same for means AND variances: var[j*ms + i] = diagonal of computePosterior's sigma of model j at row i (includes
 * noiseVar^2, MatrixUtils.scala:63) -- the quantity GPUnscentedKalmanFilter.computeNoiseMatrix (:138-147) reads for the Q / R
 * noise matrices, one computePosterior call per model in the reference.  var may be NULL. */
int gpk_gp_models_mean_var(gpk_handle h, const gpk_model* models, int nmodels, const double* Xs, int ms, int64_t ldxs,
                           double* mean, double* var);
/* The GP-UKF filter run, device-resident (SURVEY.md 8(f) row 4): dynamicalsystems/filtering/UnscentedKalmanFilter.scala:24-80
 * (inferHiddenState) with :82-118 (unscentedTransform, parameters alpha / beta / kappa) over the GP state-space model of
 * GPUnscentedKalmanFilter.scala:63-103: transition x -> x + [mean_j(x)]_j over the d `sys_models` (one GP per state dimension,
 * trained on z_t -> z_{t+1} - z_t), observation x -> [mean_j(x)]_j over the p `obs_models`, qNoise / rNoise = diag of the
 * models' posterior variances at the previous hidden mean / the predicted mean.  Every model takes the d-dimensional state as
 * input.  B independent series are filtered by the same launches and nothing crosses the host between time steps.
 *   y            observations, series b: p x T column-major (Breeze DenseMatrix) at y + b*p*T
 *   init_mean    d per series; init_cov: d x d column-major per series
 *   hidden_means d x T column-major per series (column 0 = init_mean); hidden_covs: T matrices of d x d per series
 *   ll           per series: sum_t log N(y_t; predicted observation mean, S_t) as KalmanFilter.marginalLogLikelihood computes it
 *                (log of the density, -inf once the density underflows); may be NULL / compute_ll == 0.
 * d, p <= 16.  GPK_ENOTPD when a covariance loses positive definiteness (breeze cholesky would throw NotConvergedException);
 * gpk_last_info = 1 + t*B + b of the first such (time step, series). */
int gpk_gpukf_filter(gpk_handle h, const gpk_model* sys_models, int d, const gpk_model* obs_models, int p, int B, int T,
                     const double* y, const double* init_mean, const double* init_cov, double alpha, double beta, double kappa,
                     int compute_ll, double* hidden_means, double* hidden_covs, double* ll);
/* gp/optimization/GPOptimizer.scala:82-109 maximizeUCB's objective for ms candidate points (rows of Xs) at once:
 * ucb[i] = mean_i + k_param sqrt(sigma_i) and grad[i + d*ldg] = d ucb_i / d x_d
 *        = (dKs/dx) alpha + (0 - 2 (L^-1 dKs^t/dx)^t v) k_param / (2 sqrt(sigma_i)), Ks = k(x, X), v = L^-1 Ks^t
 *          (KernelRequisites.scala:99-107),
 * with mean/sigma from computePosterior (sigma includes noiseVar^2).  mean, var, grad may be NULL. */
int gpk_gp_model_ucb(gpk_handle h, gpk_model m, const double* Xs, int ms, int64_t ldxs, double k_param, double* ucb,
                     double* grad, int64_t ldg, double* mean, double* var);
/* gp/regression/GpPredictor.scala:24-43 predict: fit + computePosterior (+ sigma_noise * I) + ll. */
int gpk_gp_predict(gpk_handle h, const double* X, int n, int D, int64_t ldx, const double* y,
                   const double* Xs, int ms, int64_t ldxs, const double* theta, int has_sigma_noise,
                   double sigma_noise, double* mean, double* sigma, int64_t lds, double* ll);

/* ---- batched independent GPs (BASELINE.json config 4) ---------------------------------------------
 * B problems of one shape (n, D) per call: MLE restarts (GpPredictor.scala:126-142 evaluated from several
 * start points), one GP per state / observation dimension (GPUnscentedKalmanFilter.scala:123-136), GP-UCB
 * restarts (GPOptimizer.scala:54-61).  Problem b uses X + b*strideX (strideX == 0: every problem shares X, the
 * GP-UKF case), y + b*n and thetas + b*(D+2).  Results: ll[b], grad[b*nparams + p], info[b] (0, or the failing
 * leading minor of problem b; may be NULL).  Returns GPK_ENOTPD if any problem failed; the others are valid.
 * Problems never interact, so any partition of the batch over handles / GPUs gives identical results. */
int gpk_gp_nll_grad_batched(gpk_handle h, int B, const double* X, int n, int D, int64_t ldx, int64_t strideX,
                            const double* y, const double* thetas, int has_sigma_noise, double sigma_noise,
                            int nparams, double* ll, double* grad, int* info);
/* Device-resident variant: out_dev[b*(nparams+1)] = ll_b followed by nparams gradients; info_dev[b]; thetas on
 * the HOST.  Asynchronous on the handle's stream. */
int gpk_gp_nll_grad_batched_dev(gpk_handle h, int B, const double* dX, int n, int D, int64_t ldx, int64_t strideX,
                                const double* dy, const double* thetas_host, int has_sigma_noise, double sigma_noise,
                                int nparams, double* out_dev, int* info_dev);
/* Fit B GPs and evaluate each at its own ms test rows (Xs + b*strideXs; strideXs == 0: shared test rows):
 * mean[b*ms + i], var[b*ms + i] = diag of computePosterior's sigma (includes noiseVar^2), ll[b] (may be NULL).
 * This is the GP-UKF sigma-point pattern (GPUnscentedKalmanFilter.scala:77-88,138-147) with m = 2d+1 rows. */
int gpk_gp_predict_batched(gpk_handle h, int B, const double* X, int n, int D, int64_t ldx, int64_t strideX,
                           const double* y, const double* thetas, const double* Xs, int ms, int64_t ldxs,
                           int64_t strideXs, int has_sigma_noise, double sigma_noise, double* mean, double* var,
                           double* ll, int* info);

/* ---- device-level building blocks of the multi-GPU block-column Cholesky (BASELINE.json config 5) -------------
 * Orchestrated one process per GPU by gp_algos_b200/distributed.py (torch.distributed / NCCL panel broadcasts).
 * All pointers are DEVICE pointers, calls are asynchronous on the handle's stream; N, m, p multiples of 128, k a
 * multiple of 16, 16-byte aligned bases, even leading dimensions. */
/* dA (N x N, ld N, symmetric, lower used) -> L in place (lower), dLi = L^-1 (N x N, ld N); *info_dev = failing minor or 0 */
int gpk_potrf_inv_block_dev(gpk_handle h, double* dA, double* dLi, int N, int* info_dev);
/* C (m x p) = alpha * P (m x k) * Q (p x k)^t + beta * C, column-major; q_lower_tri != 0: Q is lower triangular (k <= c) */
int gpk_gemm_nt_dev(gpk_handle h, int m, int p, int k, double alpha, const double* dP, int64_t ldp, const double* dQ,
                    int64_t ldq, double beta, double* dC, int64_t ldc, int q_lower_tri);
/* y = alpha * op(M) x + beta * y, M m x ncols column-major; trans != 0: op(M) = M^t (y has ncols entries) */
int gpk_gemv_dev(gpk_handle h, int trans, int m, int ncols, double alpha, const double* dM, int64_t ld, const double* dx,
                 double beta, double* dy);

/* dA[i + i*ld] += value for i < n (the noiseVar^2 [sameIndex] term of KernelRequisites.scala:69 on a diagonal block) */
int gpk_add_diag_dev(gpk_handle h, double* dA, int64_t ld, int n, double value);
/* out_dev[0] (+)= sum_{i<n} log dA[i + i*ld]: the sum_i log L_ii term of GpPredictor.scala:147 for one diagonal block */
int gpk_sum_log_diag_dev(gpk_handle h, const double* dA, int64_t ld, int n, double* out_dev, int accumulate);

/* ---- one large GP on all GPUs of the node, behind the C ABI (BASELINE.json config 5; SURVEY.md 8(b)) -------------------------
 * Single process, no launcher: a JVM binds these like every other symbol.  gpk_mg_create opens `ndev` devices (devices == NULL:
 * 0..ndev-1; ndev <= 0: all) with one libgpk handle, two bulk lanes and a put stream each and maps peer memory
 * (cudaDeviceEnablePeerAccess: NVLink / NVSwitch on a B200 node).  gpk_mg_potrf_solve is GpPredictor.preComputeComponents +
 * logLikelihood (GpPredictor.scala:104-124,144-149) for one training set: K is built block column by block column on the
 * owning device from the replicated X (never communicated), factored right-looking with look-ahead 1 on a round-robin block-
 * column layout (width gpk_mg_set_block; default 0 = automatic, 256..1024 by n and the device count), each step's panel PUT into every peer's buffer by cudaMemcpy2DAsync over
 * the peer mapping (no collective, event-ordered), alpha by a forward solve that rides along and a back solve over the owners.
 * Outputs: alpha[n], ll, *info = 0 or the failing leading minor (GPK_ENOTPD).  Results on 1, 2, 4, 8 devices agree to rounding
 * (the summation order of the trailing updates does not depend on the device count).
 * The multi-PROCESS arrangement of the same algorithm (one process per GPU, 2-D block-cyclic, NCCL panel broadcasts) is
 * gp_algos_b200/distributed.py over the *_dev building blocks above. */
typedef struct gpk_mg_s* gpk_mg;
int gpk_mg_create(gpk_mg* out, int ndev, const int* devices);
int gpk_mg_destroy(gpk_mg mg);
const char* gpk_mg_last_error(gpk_mg mg);
int gpk_mg_device_count(gpk_mg mg);
int gpk_mg_set_block(gpk_mg mg, int nb);
int gpk_mg_potrf_solve(gpk_mg mg, const double* X, int n, int D, int64_t ldx, const double* y, const double* theta,
                       int has_sigma_noise, double sigma_noise, double* alpha, double* ll, int* info);
/* device time (CUDA events on device 0 around build + factor + solves) and bytes put to peers of the last solve */
double gpk_mg_last_seconds(gpk_mg mg);
int64_t gpk_mg_last_put_bytes(gpk_mg mg);

/* ---- EP binary GP classification (BASELINE.json config 3) ------------------------------------------
 * gp/classification/EpParameterEstimator.scala:29-69 estimateSiteParams (+ :71-96 epMarginalLikelihood, :98-109
 * marginalMoments, :187-202 AvgBasedStopCriterion).  K: n x n symmetric kernel matrix (the reference is handed a
 * prebuilt K too), targets in {-1,+1} (DenseVector[Int]).  Stop rule: fixed_sweeps > 0 runs exactly that many sweeps,
 * otherwise sweeps continue until abs(avgBetweenSiteParams) < eps (at least one sweep, at most max_sweeps).
 * keep_linebreak_quirk != 0 reproduces the reference AS COMPILED: the statement at EpParameterEstimator.scala:91 ends
 * at the newline, so the "fourth and first" term of log Z is dropped; 0 includes it (R&W eq. 3.65).
 * Outputs (any may be NULL): tau, nu, mu[n], L (n x n lower factor of I + S^1/2 K S^1/2), cav_tau, cav_nu[n], logZ,
 * sweeps.  The site loop runs as blocked delayed updates on the device (see csrc/gpk_ep.cu). */
int gpk_ep_fit(gpk_handle h, const double* K, int n, int64_t ldk, const int* targets, double eps, int fixed_sweeps,
               int max_sweeps, int keep_linebreak_quirk, double* tau, double* nu, double* mu, double* L, int64_t ldl,
               double* cav_tau, double* cav_nu, double* logZ, int* sweeps);
/* gp/classification/GpClassifier.scala:24-47 classify with learnParams = (siteParams, L): K n x n, Ks m x n
 * (test-train), kss_diag[m] = diagonal of the test kernel matrix (only the diagonal is read, :44).
 * prob[m] = Phi(fmean / sqrt(1 + fvar)); fmean / fvar optional. */
int gpk_ep_classify(gpk_handle h, const double* K, int n, int64_t ldk, const double* Ks, int m, int64_t ldks,
                    const double* kss_diag, const double* tau, const double* nu, const double* L, int64_t ldl,
                    double* prob, double* fmean, double* fvar);

/* gp/classification/MarginalLikelihoodEvaluator.scala:33-45 logLikelihood(trainInput, targets, hyperParams) -> (logZ,
 * gradient): K = buildKernelMatrix(kernel(theta), X) is built on the device, EP runs to the stop rule (arguments as
 * gpk_ep_fit), then the hyper-parameter gradient of :47-66 AS COMPILED: the statement at :58 ends at the newline, so
 * rMatrix = b b^t and grad[p] = 1/2 b^t (dK/dtheta_{p+1}) b with b = nu - (S^1/2 L)^-1 L^-t S^1/2 K nu (:53-57; the
 * inner forward solve of Rasmussen & Williams Alg. 5.2 is absent in the reference and therefore here).  dK/dtheta is
 * never materialised.  Outputs: logZ, grad[nparams], tau/nu[n] (may be NULL), sweeps (may be NULL). */
int gpk_ep_nll_grad(gpk_handle h, const double* X, int n, int D, int64_t ldx, const double* theta, const int* targets,
                    double eps, int fixed_sweeps, int max_sweeps, int keep_linebreak_quirk, int nparams, double* logZ,
                    double* grad, double* tau, double* nu, int* sweeps);
/* B evaluations of MarginalLikelihoodEvaluator.logLikelihood (MarginalLikelihoodEvaluator.scala:33-66) of one size n in one
 * call: the hyper-parameter mesh (MeshHyperParamsLogLikelihoodEvaluator.scala:12-45) and optimiser restarts
 * (HyperParamsOptimization.scala:31-136) evaluate many points on one training set.  Problem b: X + b*strideX (strideX == 0:
 * every problem shares X), targets + b*strideT (strideT == 0: shared labels), thetas + b*gpk_theta_length(h, D), the
 * handle's kernel family.  Stop rule, quirk and nparams exactly as gpk_ep_nll_grad, applied to EACH problem on its own:
 * each problem stops at its own sweep.  Outputs: logZ[b], grad[b*nparams + p], tau / nu[b*n + i] (may be NULL),
 * sweeps[b], info[b] (0 or the failing leading minor of I + S^1/2 K S^1/2; may be NULL).  GPK_ENOTPD if any problem
 * failed (its logZ and gradient are NaN); the others are valid.  nparams == 0: no gradient (logLikelihoodWithoutGrad,
 * :24-31).  The sweeps of all problems run together (one site-kernel CTA per problem, every other launch batched); a
 * problem's results do not depend on the other problems of the call or on its position.  Eager launches only:
 * gpk_set_graph_mode does not apply.  A batch larger than GPK_BATCH_GB (see gpk_gp_nll_grad_batched) runs chunk by chunk. */
int gpk_ep_nll_grad_batched(gpk_handle h, int B, const double* X, int n, int D, int64_t ldx, int64_t strideX,
                            const double* thetas, const int* targets, int64_t strideT, double eps, int fixed_sweeps,
                            int max_sweeps, int keep_linebreak_quirk, int nparams, double* logZ, double* grad,
                            double* tau, double* nu, int* sweeps, int* info);
/* MarginalLikelihoodEvaluator.scala:47-66 logLikelihoodDerivativesAfterHyperParams(HyperParameterOptimInput(siteParams,
 * lowerTriangular, kernelMatrix, trainInput), kernelFun): the gradient alone from a finished EP run.  K may be NULL
 * (rebuilt from X and theta). */
int gpk_ep_grad_from_factor(gpk_handle h, const double* X, int n, int D, int64_t ldx, const double* theta, const double* K,
                            int64_t ldk, const double* tau, const double* nu, const double* L, int64_t ldl, int nparams,
                            double* grad);

#ifdef __cplusplus
}
#endif
#endif /* GPK_H */
