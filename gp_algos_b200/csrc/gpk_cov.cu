// gpk_cov.cu -- squared-exponential / ARD covariance construction.
// Replaces utils/MatrixUtils.scala:44-97 (buildKernelMatrix / buildMatrixWithFunc) evaluated with
// utils/KernelRequisites.scala:62-114 (GaussianRbfKernel): one closure call + >=4 heap allocations per
// element in the reference, a single fused pass here.
//
// k(x,x') = sf^2 * exp(-0.5 * sum_d ((x_d - x'_d) * (1/(l_d*l_d))) * (x_d - x'_d)) + sn^2 [i==j]
// The distance uses the reference's direct-difference form and association (KernelRequisites.scala:109-113)
// with un-fused multiplies/adds (__dmul_rn/__dadd_rn) so the exponent argument is bit-identical to
// the JVM's; only exp() itself (<= 1 ulp in both libraries) can differ.
//
// HBM-write-bound kernel: 8 bytes written per element, X (n x D) is read once per 64x64 tile through
// shared memory.  One CTA = 256 threads = one 64x64 tile; a thread owns 2 consecutive rows x 8 columns,
// so a warp writes 512 contiguous bytes per column (16-byte vector stores).  The symmetric variant
// computes tiles on/below the diagonal only and mirrors them through a padded shared-memory transpose,
// like the reference's "lower loop and mirror" (MatrixUtils.scala:60-67), which also guarantees exact symmetry.
#include "gpk_internal.cuh"

#include <stdarg.h>

namespace {

constexpr int CT = 64;       // tile edge
constexpr int DC = 8;        // feature-dimension chunk staged in shared memory
constexpr int TLD = CT + 1;  // transpose buffer stride

enum { MODE_SYM_FULL = 0, MODE_SYM_LOWER_PAD = 1, MODE_CROSS = 2 };

struct CovArgs {
    const double* X1; int64_t ldx1; int m;  // row points
    const double* X2; int64_t ldx2; int n;  // column points
    double* K; int64_t ldk;
    int mp, np;  // padded extents written (>= m, n)
    int64_t strideX1, strideX2, strideK;  // per-problem strides (blockIdx.z)
    const ProblemParams* pp;               // device array of per-problem hyper-parameters, or nullptr -> cp
    CovParams cp;
};

__device__ __forceinline__ void store2(double* p, double a, double b, bool ok0, bool ok1) {
    if (ok0 && ok1 && ((reinterpret_cast<uintptr_t>(p) & 15) == 0)) {
        *reinterpret_cast<double2*>(p) = make_double2(a, b);
    } else {
        if (ok0) p[0] = a;
        if (ok1) p[1] = b;
    }
}

// KIND = gpk_kernel_family: GPK_KERNEL_SE_ARD accumulates the scaled squared distance over the feature dimensions;
// GPK_KERNEL_CO2 (1-D inputs) keeps the plain difference and evaluates Co2Prediction.scala:38-56 on it.
template <int MODE, int KIND>
__global__ void __launch_bounds__(256) cov_se_ard_kernel(const CovArgs a0) {
    // per-problem view (blockIdx.z); hyper-parameters by value (single problem) or from the device array (batched)
    struct View { const double* X1; const double* X2; double* K; int64_t ldx1, ldx2, ldk; int m, n, mp, np; const CovParams& cp; };
    const int64_t bz = blockIdx.z;
    const View a = {a0.X1 + bz * a0.strideX1, a0.X2 + bz * a0.strideX2, a0.K + bz * a0.strideK, a0.ldx1, a0.ldx2, a0.ldk,
                    a0.m, a0.n, a0.mp, a0.np, a0.pp ? a0.pp[bz].cp : a0.cp};
    __shared__ double xi[DC][CT];
    __shared__ double xj[DC][CT];
    __shared__ double tbuf[(MODE == MODE_SYM_FULL) ? CT * TLD : 1];

    const int bi = blockIdx.x, bj = blockIdx.y;
    if (MODE == MODE_SYM_FULL && bj > bi) return;
    if (MODE == MODE_SYM_LOWER_PAD && (bj >> 1) > (bi >> 1)) return;  // keep whole 128x128 diagonal blocks
    const int i0 = bi * CT, j0 = bj * CT;
    const int tid = threadIdx.x, tx = tid & 31, ty = tid >> 5;
    const int D = a.cp.D;

    double r[2][8];
#pragma unroll
    for (int q = 0; q < 2; ++q)
#pragma unroll
        for (int b = 0; b < 8; ++b) r[q][b] = 0.0;

    for (int d0 = 0; d0 < D; d0 += DC) {
        const int dc = min(DC, D - d0);
        __syncthreads();
        for (int e = tid; e < dc * CT; e += 256) {
            const int d = e / CT, l = e % CT;
            const int gi = i0 + l, gj = j0 + l;
            xi[d][l] = (gi < a.m) ? a.X1[gi + (int64_t)(d0 + d) * a.ldx1] : 0.0;
            xj[d][l] = (gj < a.n) ? a.X2[gj + (int64_t)(d0 + d) * a.ldx2] : 0.0;
        }
        __syncthreads();
        for (int d = 0; d < dc; ++d) {
            const double inv = a.cp.inv_ls2[d0 + d];
            const double x0 = xi[d][2 * tx], x1 = xi[d][2 * tx + 1];
#pragma unroll
            for (int b = 0; b < 8; ++b) {
                const double xv = xj[d][ty + 8 * b];
                const double f0 = __dsub_rn(x0, xv), f1 = __dsub_rn(x1, xv);
                if (KIND == GPK_KERNEL_CO2) {
                    r[0][b] = f0; r[1][b] = f1;     // D == 1: the difference itself
                } else {
                    r[0][b] = __dadd_rn(r[0][b], __dmul_rn(__dmul_rn(f0, inv), f0));
                    r[1][b] = __dadd_rn(r[1][b], __dmul_rn(__dmul_rn(f1, inv), f1));
                }
            }
        }
    }

    const int gi0 = i0 + 2 * tx;
#pragma unroll
    for (int b = 0; b < 8; ++b) {
        const int gj = j0 + ty + 8 * b;
        double v[2];
#pragma unroll
        for (int q = 0; q < 2; ++q) {
            const int gi = gi0 + q;
            double val;
            if (KIND == GPK_KERNEL_CO2) {
                Co2Terms t;
                val = co2_value(a.cp.inv_ls2, r[q][b], t);
            } else {
                val = __dmul_rn(a.cp.sf2, exp(__dmul_rn(-0.5, r[q][b])));
            }
            if (MODE != MODE_CROSS && gi == gj) {
                val = __dadd_rn(val, a.cp.sn2);
                if (a.cp.extra_diag != 0.0) val = __dadd_rn(val, a.cp.extra_diag);
            }
            if (gi >= a.m || gj >= a.n) val = (MODE == MODE_SYM_LOWER_PAD && gi == gj) ? 1.0 : 0.0;
            v[q] = val;
        }
        store2(a.K + gi0 + (int64_t)gj * a.ldk, v[0], v[1], gi0 < a.mp && gj < a.np, gi0 + 1 < a.mp && gj < a.np);
        if (MODE == MODE_SYM_FULL) {
            tbuf[(2 * tx) * TLD + ty + 8 * b] = v[0];
            tbuf[(2 * tx + 1) * TLD + ty + 8 * b] = v[1];
        }
    }
    if (MODE == MODE_SYM_FULL && bi != bj) {
        __syncthreads();
        // mirrored tile: element (row = j0 + jl, col = i0 + il) = tbuf[il][jl]
        const int jl0 = 2 * tx;
#pragma unroll
        for (int b = 0; b < 8; ++b) {
            const int il = ty + 8 * b;
            const int grow = j0 + jl0, gcol = i0 + il;
            store2(a.K + grow + (int64_t)gcol * a.ldk, tbuf[il * TLD + jl0], tbuf[il * TLD + jl0 + 1],
                   grow < a.n && gcol < a.m, grow + 1 < a.n && gcol < a.m);
        }
    }
}

// utils/KernelRequisites.scala:76-86 derAfterHyperParam, materialised (API completeness only).
__global__ void cov_deriv_kernel(int param_num, const double* X, int n, int64_t ldx, CovParams cp, double sf, double sn,
                                 double ls_d, double* dK, int64_t ldk) {
    const int i = blockIdx.y * blockDim.x + threadIdx.x;
    const int j = blockIdx.x;
    if (i >= n || j >= n) return;
    const int D = cp.D;
    if (cp.kind == GPK_KERNEL_CO2) {   // Co2Prediction.scala:66-137
        Co2Terms t;
        double dk[GPK_CO2_NPARAMS];
        co2_value(cp.inv_ls2, __dsub_rn(X[i], X[j]), t);
        co2_derivs(cp.inv_ls2, t, dk);
        dk[10] = (i == j) ? 2 * cp.inv_ls2[10] : 0.0;
        dK[i + (int64_t)j * ldk] = dk[param_num - 1];
        return;
    }
    double r = 0.0;
    for (int d = 0; d < D; ++d) {
        const double f = __dsub_rn(X[i + (int64_t)d * ldx], X[j + (int64_t)d * ldx]);
        r = __dadd_rn(r, __dmul_rn(__dmul_rn(f, cp.inv_ls2[d]), f));
    }
    double v;
    if (param_num == 1) {
        v = 2 * sf * exp(-0.5 * r);
    } else if (param_num < D + 2) {
        const int d = param_num - 2;
        const double f = X[i + (int64_t)d * ldx] - X[j + (int64_t)d * ldx];
        v = __dmul_rn(__dmul_rn(__dmul_rn(sf * sf, exp(-0.5 * r)), f * f), pow(ls_d, -3.0));
    } else {
        v = (i == j) ? 2 * sn : 0.0;
    }
    dK[i + (int64_t)j * ldk] = v;
}

}  // namespace

int gpk_make_problem_params(gpk_handle h, const double* theta, int D, int has_sigma_noise, double sigma_noise, ProblemParams* out) {
    int rc = gpk_make_cov_params(h, theta, D, has_sigma_noise, sigma_noise, &out->cp);
    if (rc) return rc;
    if (out->cp.kind == GPK_KERNEL_CO2) {   // the trace kernel accumulates the full derivative: only the 1/2 of the trace is left
        memset(out->gscale, 0, sizeof(out->gscale));
        for (int p = 0; p < GPK_CO2_NPARAMS; ++p) out->gscale[p] = 0.5;
        return GPK_OK;
    }
    const double sf = theta[0], sn = theta[D + 1];
    memset(out->gscale, 0, sizeof(out->gscale));
    out->gscale[0] = sf;                                          // 1/2 * 2 sf
    for (int d = 0; d < D; ++d) {
        const double l = theta[1 + d];
        out->gscale[1 + d] = 0.5 * (sf * sf) / (l * l * l);       // 1/2 * sf^2 / l_d^3
    }
    out->gscale[D + 1] = sn;                                      // 1/2 * 2 sn
    return GPK_OK;
}

int gpk_make_cov_params(gpk_handle h, const double* theta, int D, int has_sigma_noise, double sigma_noise, CovParams* out) {
    memset(out, 0, sizeof(*out));
    out->D = D;
    out->kind = h ? h->kernel_family : GPK_KERNEL_SE_ARD;
    if (out->kind == GPK_KERNEL_CO2) {
        // require(obj1.length == 1 && obj2.length == 1, "This kernel is applicable only for 1D objects") Co2Prediction.scala:39
        if (D != 1) return gpk_set_error(h, GPK_EINVAL, "requirement failed: This kernel is applicable only for 1D objects");
        double* par = out->inv_ls2;
        for (int p = 0; p < GPK_CO2_NPARAMS; ++p) par[p] = theta[p];
        par[11] = pow(theta[1], -3); par[12] = pow(theta[3], -3); par[13] = pow(theta[4], -3); par[14] = pow(theta[6], -3);
        par[15] = pow(theta[9], -3);
        // k(x,x): every exp / pow factor is exactly 1, summed in the order of Co2Prediction.scala:55
        out->sf2 = ((theta[0] * theta[0] + theta[2] * theta[2]) + theta[5] * theta[5]) + theta[8] * theta[8];
        out->sn2 = theta[10] * theta[10];
        out->extra_diag = has_sigma_noise ? sigma_noise : 0.0;
        return GPK_OK;
    }
    out->sf2 = theta[0] * theta[0];
    out->sn2 = theta[D + 1] * theta[D + 1];
    out->extra_diag = has_sigma_noise ? sigma_noise : 0.0;
    for (int d = 0; d < D; ++d) out->inv_ls2[d] = 1.0 / (theta[1 + d] * theta[1 + d]);
    return GPK_OK;
}

int gpk_cov_sym_full(gpk_handle h, const double* dX, int n, int64_t ldx, const CovParams& cp, double* dK, int64_t ldk) {
    if (n <= 0) return GPK_OK;
    CovArgs a;
    a.X1 = dX; a.ldx1 = ldx; a.m = n; a.X2 = dX; a.ldx2 = ldx; a.n = n; a.K = dK; a.ldk = ldk; a.mp = n; a.np = n; a.cp = cp;
    a.strideX1 = a.strideX2 = a.strideK = 0; a.pp = nullptr;
    const int t = (n + CT - 1) / CT;
    if (cp.kind == GPK_KERNEL_CO2) cov_se_ard_kernel<MODE_SYM_FULL, GPK_KERNEL_CO2><<<dim3(t, t), 256, 0, h->stream>>>(a);
    else cov_se_ard_kernel<MODE_SYM_FULL, GPK_KERNEL_SE_ARD><<<dim3(t, t), 256, 0, h->stream>>>(a);
    GPK_LAUNCH_CHECK(h);
    return GPK_OK;
}

int gpk_cov_sym_lower_padded(gpk_handle h, const double* dX, int n, int64_t ldx, const CovParams& cp, double* dK, int N,
                             int batch, int64_t strideX, const ProblemParams* pp_dev) {
    CovArgs a;
    a.X1 = dX; a.ldx1 = ldx; a.m = n; a.X2 = dX; a.ldx2 = ldx; a.n = n; a.K = dK; a.ldk = N; a.mp = N; a.np = N; a.cp = cp;
    a.strideX1 = a.strideX2 = strideX; a.strideK = (int64_t)N * N; a.pp = pp_dev;
    const int t = N / CT;
    if (cp.kind == GPK_KERNEL_CO2) cov_se_ard_kernel<MODE_SYM_LOWER_PAD, GPK_KERNEL_CO2><<<dim3(t, t, batch), 256, 0, h->stream>>>(a);
    else cov_se_ard_kernel<MODE_SYM_LOWER_PAD, GPK_KERNEL_SE_ARD><<<dim3(t, t, batch), 256, 0, h->stream>>>(a);
    GPK_LAUNCH_CHECK(h);
    return GPK_OK;
}

int gpk_cov_cross(gpk_handle h, const double* dX1, int m, int64_t ldx1, const double* dX2, int n, int64_t ldx2,
                  const CovParams& cp, double* dK, int64_t ldk, int mp, int np, int batch, int64_t strideX1, int64_t strideX2,
                  int64_t strideK, const ProblemParams* pp_dev) {
    if (mp < m) mp = m;
    if (np < n) np = n;
    if (mp <= 0 || np <= 0) return GPK_OK;
    CovArgs a;
    a.X1 = dX1; a.ldx1 = ldx1; a.m = m; a.X2 = dX2; a.ldx2 = ldx2; a.n = n; a.K = dK; a.ldk = ldk; a.mp = mp; a.np = np; a.cp = cp;
    a.strideX1 = strideX1; a.strideX2 = strideX2; a.strideK = strideK; a.pp = pp_dev;
    const dim3 grid((mp + CT - 1) / CT, (np + CT - 1) / CT, batch);
    if (cp.kind == GPK_KERNEL_CO2) cov_se_ard_kernel<MODE_CROSS, GPK_KERNEL_CO2><<<grid, 256, 0, h->stream>>>(a);
    else cov_se_ard_kernel<MODE_CROSS, GPK_KERNEL_SE_ARD><<<grid, 256, 0, h->stream>>>(a);
    GPK_LAUNCH_CHECK(h);
    return GPK_OK;
}

int gpk_cov_deriv(gpk_handle h, int param_num, const double* dX, int n, int64_t ldx, const CovParams& cp, double sf,
                  double sn, const double* ls_host, double* dK, int64_t ldk) {
    if (n <= 0) return GPK_OK;
    const double ls_d = (param_num >= 2 && param_num < cp.D + 2) ? ls_host[param_num - 2] : 1.0;
    cov_deriv_kernel<<<dim3(n, (n + 127) / 128), 128, 0, h->stream>>>(param_num, dX, n, ldx, cp, sf, sn, ls_d, dK, ldk);
    GPK_LAUNCH_CHECK(h);
    return GPK_OK;
}
