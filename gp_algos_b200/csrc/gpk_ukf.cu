// gpk_ukf.cu -- the GP-UKF filter step, device-resident and batched over independent filters (SURVEY.md 8(f) row 4).
//
// Reference: dynamicalsystems/filtering/UnscentedKalmanFilter.scala:24-80 (inferHiddenState) and :82-118 (unscentedTransform)
// driven by the GP state-space model of GPUnscentedKalmanFilter.scala:63-103: transition x -> x + [mean_j(x)]_j over one GP per
// state dimension, observation x -> [mean_j(x)]_j over one GP per observation dimension, Q / R = diag of the GPs' posterior
// variances at the previous hidden mean / the predicted mean (:95-102,138-147).  The reference makes (2d+1)(d+p) + (d+p)
// computePosterior calls per time step, each an O(n^2) scalar triangular solve, and runs the d x d algebra on the JVM.
//
// Here one call filters B independent series for T steps without touching the host: per step
//   ukf_sigma1      chol(P_{t-1}) and the 2d+1 sigma points of every filter                      (one warp per filter)
//   GP evaluation   for each of the d transition GPs: k(X, points) (tiled cross-covariance), means = K* alpha for all
//                   B(2d+1) points, variances for the B central points through V = L^-1 K*^t (DMMA GEMM)
//   ukf_predict     transformed points, predicted mean / covariance + Q, its Cholesky, the second set of sigma points
//   GP evaluation   the p observation GPs at the second sigma points (+ variances at the central points -> R)
//   ukf_update      innovation covariance S, cross covariance, gain K = C S^-1, new mean / covariance, log-likelihood term.
// Sigma points of all filters form ONE test matrix (row i B + b = sigma point i of filter b), so the GP work of a step is
// (d + p) x 4 launches however many filters run.
#include "gpk_internal.cuh"

#include <math.h>

namespace {

constexpr int UD = 16;   // largest state / observation dimension

struct UkfDims { int d, p, B, M, Mp, Bp, T; };   // M = (2d+1) B sigma points per transform, Mp / Bp = padded to 128

// lower Cholesky of the dim x dim matrix a (column-major, ld dim) in place; returns 0 or the failing minor (1-based)
__device__ int small_chol(double* a, int dim) {
    for (int j = 0; j < dim; ++j) {
        double s = a[j + j * dim];
        for (int k = 0; k < j; ++k) s -= a[j + k * dim] * a[j + k * dim];
        if (!(s > 0.0)) return j + 1;
        const double l = sqrt(s);
        a[j + j * dim] = l;
        for (int i = j + 1; i < dim; ++i) {
            double v = a[i + j * dim];
            for (int k = 0; k < j; ++k) v -= a[i + k * dim] * a[j + k * dim];
            a[i + j * dim] = v / l;
        }
        for (int i = 0; i < j; ++i) a[i + j * dim] = 0.0;
    }
    return 0;
}

// sigma points of N(mean, L L^t): row 0 = mean, rows 1..d = mean + c L[:,col], rows d+1..2d = mean - c L[:,col]
// (UnscentedKalmanFilter.scala:88-94); written for filter b into SP (M x d, ld M) at rows i B + b
__device__ void write_sigma_points(const double* mean, const double* L, int d, double c, double* SP, int M, int B, int b) {
    for (int j = 0; j < d; ++j) SP[b + (int64_t)j * M] = mean[j];
    for (int col = 0; col < d; ++col)
        for (int j = 0; j < d; ++j) {
            const double sc = L[j + col * d] * c;
            SP[(col + 1) * B + b + (int64_t)j * M] = mean[j] + sc;
            SP[(col + 1 + d) * B + b + (int64_t)j * M] = mean[j] - sc;
        }
}

// Unscented-transform moments of the transformed points tp (row i of filter b at tp[i B + b + j ldt]), out dimension q
// (UnscentedKalmanFilter.scala:96-113: the non-central points are weighted by w_i_c in the MEAN too, SURVEY.md 8(c)(7))
__device__ void ut_moments(const double* tp, int64_t ldt, int B, int b, int npts, int q, double w0m, double w0c, double wic,
                           double* mean, double* cov) {
    for (int j = 0; j < q; ++j) {
        double m = tp[b + j * ldt] * w0m;
        for (int i = 1; i < npts; ++i) m = m + tp[i * B + b + j * ldt] * wic;
        mean[j] = m;
    }
    for (int c = 0; c < q; ++c)
        for (int r = 0; r < q; ++r) {
            double s = ((tp[b + r * ldt] - mean[r]) * (tp[b + c * ldt] - mean[c])) * w0c;
            for (int i = 1; i < npts; ++i) s = s + ((tp[i * B + b + r * ldt] - mean[r]) * (tp[i * B + b + c * ldt] - mean[c])) * wic;
            cov[r + c * q] = s;
        }
}

struct UkfState {      // device arrays, one entry per filter
    double* mean;      // d x B        current hidden mean
    double* cov;       // d x d x B    current hidden covariance
    double* pmean;     // d x B        predicted mean (first transform)
    double* pcov;      // d x d x B    predicted covariance + Q
    double* zT;        // M x d        transformed sigma points of the first transform (row i B + b)
    double* ll;        // B
    int* info;         // [0] = 0, or 1 + (t * B + b) of the first non-positive-definite covariance
};

// step 1 of time t: sigma points of N(mean, cov) of every filter.  One thread per filter (the d x d algebra is <= 16^3 flops).
__global__ void ukf_sigma1(UkfDims dm, UkfState st, double c, int t, double* SP) {
    const int b = blockIdx.x * blockDim.x + threadIdx.x;
    if (b >= dm.B) return;
    double L[UD * UD];
    const int d = dm.d;
    for (int e = 0; e < d * d; ++e) L[e] = st.cov[(int64_t)b * d * d + e];
    if (small_chol(L, d)) atomicCAS(st.info, 0, 1 + t * dm.B + b);
    write_sigma_points(st.mean + (int64_t)b * d, L, d, c, SP, dm.M, dm.B, b);
}

// step 2: zT = SP + GP means (GPUnscentedKalmanFilter.scala:77-83), predicted moments, Q = diag(kss_j - |v_j|^2) (:95-98,138-147),
// second set of sigma points.  gmean: Mp per model; vsq: Bp per model; kss[j] = k(x,x) incl. the i == j noise term.
__global__ void ukf_predict(UkfDims dm, UkfState st, double c, double w0m, double w0c, double wic, int t, const double* SP,
                            const double* gmean, const double* vsq, const double* kss, double* SP2) {
    const int b = blockIdx.x * blockDim.x + threadIdx.x;
    if (b >= dm.B) return;
    const int d = dm.d, npts = 2 * d + 1;
    for (int i = 0; i < npts; ++i)
        for (int j = 0; j < d; ++j) {
            const int r = i * dm.B + b;
            st.zT[r + (int64_t)j * dm.M] = SP[r + (int64_t)j * dm.M] + gmean[r + (int64_t)j * dm.Mp];
        }
    double mean[UD], cov[UD * UD];
    ut_moments(st.zT, dm.M, dm.B, b, npts, d, w0m, w0c, wic, mean, cov);
    for (int j = 0; j < d; ++j) cov[j + j * d] = cov[j + j * d] + (kss[j] - vsq[b + (int64_t)j * dm.Bp]);     // sigma + qNoise (:43-45)
    for (int j = 0; j < d; ++j) st.pmean[(int64_t)b * d + j] = mean[j];
    for (int e = 0; e < d * d; ++e) st.pcov[(int64_t)b * d * d + e] = cov[e];
    if (small_chol(cov, d)) atomicCAS(st.info, 0, 1 + t * dm.B + b);
    write_sigma_points(mean, cov, d, c, SP2, dm.M, dm.B, b);
}

// step 3: observation moments + R, cross covariance, gain, update (UnscentedKalmanFilter.scala:46-74)
__global__ void ukf_update(UkfDims dm, UkfState st, double w0m, double w0c, double wic, int t, const double* gmean,
                           const double* vsq, const double* kss, const double* y, int compute_ll, double* out_means,
                           double* out_covs) {
    const int b = blockIdx.x * blockDim.x + threadIdx.x;
    if (b >= dm.B) return;
    const int d = dm.d, p = dm.p, npts = 2 * d + 1;
    double my[UD], S[UD * UD], Si[UD * UD], zy[UD * UD], K[UD * UD], KS[UD * UD];
    ut_moments(gmean, dm.Mp, dm.B, b, npts, p, w0m, w0c, wic, my, S);                      // yT = GP means (:84-90)
    for (int j = 0; j < p; ++j) S[j + j * p] = S[j + j * p] + (kss[j] - vsq[b + (int64_t)j * dm.Bp]);  // + rNoise (:50-51)
    const double* mz = st.pmean + (int64_t)b * d;
    const double* cz = st.pcov + (int64_t)b * d * d;
    for (int c = 0; c < p; ++c)                                                            // z-y covariance (:54-62)
        for (int r = 0; r < d; ++r) {
            double s = ((st.zT[b + (int64_t)r * dm.M] - mz[r]) * (gmean[b + (int64_t)c * dm.Mp] - my[c])) * w0c;
            for (int i = 1; i < npts; ++i)
                s = s + ((st.zT[i * dm.B + b + (int64_t)r * dm.M] - mz[r]) * (gmean[i * dm.B + b + (int64_t)c * dm.Mp] - my[c])) * wic;
            zy[r + c * d] = s;
        }
    // inv(S) by Gauss-Jordan with partial pivoting (breeze inv = LAPACK dgetrf + dgetri, :64); det for the density
    double A[UD * UD];
    for (int e = 0; e < p * p; ++e) { A[e] = S[e]; Si[e] = 0.0; }
    for (int j = 0; j < p; ++j) Si[j + j * p] = 1.0;
    double det = 1.0;
    for (int col = 0; col < p; ++col) {
        int piv = col;
        for (int r = col + 1; r < p; ++r) if (fabs(A[r + col * p]) > fabs(A[piv + col * p])) piv = r;
        if (piv != col) {
            for (int c = 0; c < p; ++c) {
                double tmp = A[col + c * p]; A[col + c * p] = A[piv + c * p]; A[piv + c * p] = tmp;
                tmp = Si[col + c * p]; Si[col + c * p] = Si[piv + c * p]; Si[piv + c * p] = tmp;
            }
            det = -det;
        }
        const double pv = A[col + col * p];
        det *= pv;
        const double rp = 1.0 / pv;
        for (int c = 0; c < p; ++c) { A[col + c * p] *= rp; Si[col + c * p] *= rp; }
        for (int r = 0; r < p; ++r) {
            if (r == col) continue;
            const double f = A[r + col * p];
            if (f == 0.0) continue;
            for (int c = 0; c < p; ++c) { A[r + c * p] -= f * A[col + c * p]; Si[r + c * p] -= f * Si[col + c * p]; }
        }
    }
    for (int c = 0; c < p; ++c)                                                            // K = zy S^-1 (:65)
        for (int r = 0; r < d; ++r) {
            double s = 0.0;
            for (int k = 0; k < p; ++k) s += zy[r + k * d] * Si[k + c * p];
            K[r + c * d] = s;
        }
    const double* yt = y + ((int64_t)b * dm.T + t) * p;
    double innov[UD];
    for (int j = 0; j < p; ++j) innov[j] = yt[j] - my[j];
    double* nm = st.mean + (int64_t)b * d;
    for (int r = 0; r < d; ++r) {                                                          // :66-67
        double s = 0.0;
        for (int k = 0; k < p; ++k) s += K[r + k * d] * innov[k];
        nm[r] = mz[r] + s;
        out_means[((int64_t)b * dm.T + t) * d + r] = nm[r];
    }
    for (int c = 0; c < p; ++c)                                                            // (K S) K^t (:68-69)
        for (int r = 0; r < d; ++r) {
            double s = 0.0;
            for (int k = 0; k < p; ++k) s += K[r + k * d] * S[k + c * p];
            KS[r + c * d] = s;
        }
    double* nc = st.cov + (int64_t)b * d * d;
    for (int c = 0; c < d; ++c)
        for (int r = 0; r < d; ++r) {
            double s = 0.0;
            for (int k = 0; k < p; ++k) s += KS[r + k * d] * K[c + k * d];
            nc[r + c * d] = cz[r + c * d] - s;
            out_covs[(((int64_t)b * dm.T + t) * d + c) * d + r] = nc[r + c * d];
        }
    if (compute_ll) {                                                                      // KalmanFilter.marginalLogLikelihood -> StatsUtils.scala:47-58
        double quad = 0.0;
        for (int r = 0; r < p; ++r) {
            double s = 0.0;
            for (int k = 0; k < p; ++k) s += Si[r + k * p] * innov[k];
            quad += innov[r] * s;
        }
        const double dens = pow(2.0 * 3.14159265358979323846, -0.5 * p) * pow(det, -0.5) * exp(-0.5 * quad);
        st.ll[b] += (dens > 0.0) ? log(dens) : -INFINITY;                                  // log(density): -inf when the density underflows
    }
}

__global__ void ukf_init(UkfDims dm, UkfState st, const double* init_mean, const double* init_cov, double* out_means, double* out_covs) {
    const int b = blockIdx.x * blockDim.x + threadIdx.x;
    if (b >= dm.B) return;
    const int d = dm.d;
    for (int j = 0; j < d; ++j) {
        st.mean[(int64_t)b * d + j] = init_mean[(int64_t)b * d + j];
        out_means[(int64_t)b * dm.T * d + j] = init_mean[(int64_t)b * d + j];
    }
    for (int e = 0; e < d * d; ++e) {
        st.cov[(int64_t)b * d * d + e] = init_cov[(int64_t)b * d * d + e];
        out_covs[(int64_t)b * dm.T * d * d + e] = init_cov[(int64_t)b * d * d + e];
    }
    st.ll[b] = 0.0;
    if (b == 0) st.info[0] = 0;
}

}  // namespace

extern "C" {

int gpk_gpukf_filter(gpk_handle h, const gpk_model* sys_models, int d, const gpk_model* obs_models, int p, int B, int T,
                     const double* y, const double* init_mean, const double* init_cov, double alpha, double beta, double kappa,
                     int compute_ll, double* hidden_means, double* hidden_covs, double* ll) {
    if (!h || !sys_models || !obs_models || !y || !init_mean || !init_cov || !hidden_means || !hidden_covs)
        return gpk_set_error(h, GPK_EINVAL, "gpk_gpukf_filter: null argument");
    if (d < 1 || d > UD || p < 1 || p > UD || B < 1 || T < 1)
        return gpk_set_error(h, GPK_EINVAL, "gpk_gpukf_filter: need 1 <= d, p <= %d, B >= 1, T >= 1", UD);
    int Nmax = 0;
    for (int j = 0; j < d + p; ++j) {
        gpk_model m = j < d ? sys_models[j] : obs_models[j - d];
        if (!m || m->D != d) return gpk_set_error(h, GPK_EINVAL, "gpk_gpukf_filter: every GP must take the d-dimensional hidden state as input");
        if (m->N > Nmax) Nmax = m->N;
    }
    GPK_CUDA(h, cudaSetDevice(h->device));
    UkfDims dm;
    dm.d = d; dm.p = p; dm.B = B; dm.T = T; dm.M = (2 * d + 1) * B; dm.Mp = gpk_pad(dm.M); dm.Bp = gpk_pad(B);
    const int q = d > p ? d : p;
    // device workspace: SP, SP2, zT (M x d each); means (q x Mp), vsq (q x Bp), kss (d + p); KsT (Nmax x Mp), V (Nmax x Bp);
    // filter state; inputs (y, init) and outputs (means, covs)
    const size_t nSP = (size_t)dm.M * d, nState = (size_t)B * (2 * d + 2 * d * d + 1) + 8;
    const size_t nIn = (size_t)B * T * p + (size_t)B * d + (size_t)B * d * d;
    const size_t nOut = (size_t)B * T * d + (size_t)B * T * d * d;
    const size_t total = 3 * nSP + (size_t)q * dm.Mp + (size_t)q * dm.Bp + (size_t)(d + p) + (size_t)Nmax * dm.Mp + (size_t)Nmax * dm.Bp +
                         nState + nIn + nOut + 64;
    double* w = (double*)gpk_arena(h, ARENA_IO3, total * sizeof(double));
    if (!w) return GPK_ENOMEM;
    double* SP = w; double* SP2 = SP + nSP; double* zT = SP2 + nSP;
    double* gmean = zT + nSP; double* vsq = gmean + (size_t)q * dm.Mp; double* kss = vsq + (size_t)q * dm.Bp;
    double* KsT = kss + (d + p); double* V = KsT + (size_t)Nmax * dm.Mp;
    UkfState st;
    st.mean = V + (size_t)Nmax * dm.Bp; st.cov = st.mean + (size_t)B * d; st.pmean = st.cov + (size_t)B * d * d;
    st.pcov = st.pmean + (size_t)B * d; st.zT = zT; st.ll = st.pcov + (size_t)B * d * d; st.info = (int*)(st.ll + B);
    double* dY = st.ll + B + 8; double* dM0 = dY + (size_t)B * T * p; double* dC0 = dM0 + (size_t)B * d;
    double* dOutM = dC0 + (size_t)B * d * d; double* dOutC = dOutM + (size_t)B * T * d;
    GPK_CUDA(h, cudaMemcpyAsync(dY, y, (size_t)B * T * p * sizeof(double), cudaMemcpyHostToDevice, h->stream));
    GPK_CUDA(h, cudaMemcpyAsync(dM0, init_mean, (size_t)B * d * sizeof(double), cudaMemcpyHostToDevice, h->stream));
    GPK_CUDA(h, cudaMemcpyAsync(dC0, init_cov, (size_t)B * d * d * sizeof(double), cudaMemcpyHostToDevice, h->stream));
    for (int j = 0; j < d + p; ++j) {
        gpk_model m = j < d ? sys_models[j] : obs_models[j - d];
        h->h_pinned[128 + j] = gpk_prior_var(m->pp.cp);
    }
    GPK_CUDA(h, cudaMemcpyAsync(kss, h->h_pinned + 128, (size_t)(d + p) * sizeof(double), cudaMemcpyHostToDevice, h->stream));
    // weights (UnscentedKalmanFilter.scala:87,96-97)
    const double lambda = alpha * alpha * (d + kappa) - d;
    const double c = sqrt(d + lambda);
    const double w0m = lambda / (d + lambda), w0c = (lambda / (d + lambda)) + (1 - alpha * alpha + beta), wic = 1 / (2 * (d + lambda));
    const int nb = (B + 63) / 64;
    ukf_init<<<nb, 64, 0, h->stream>>>(dm, st, dM0, dC0, dOutM, dOutC);
    GPK_LAUNCH_CHECK(h);
    for (int t = 1; t < T; ++t) {
        ukf_sigma1<<<nb, 64, 0, h->stream>>>(dm, st, c, t, SP);
        GPK_LAUNCH_CHECK(h);
        // means at every sigma point, |L^-1 k*|^2 at the B central ones (rows 0 .. B-1)
        for (int j = 0; j < d; ++j) {
            const gpk_model m = sys_models[j];
            int rc = gpk_posterior(h, m->X, m->n, m->ldx, SP, dm.M, m->Li, m->alpha, m->N, m->pp.cp, KsT, gmean + (size_t)j * dm.Mp, V,
                                   B, vsq + (size_t)j * dm.Bp);
            if (rc) return rc;
        }
        ukf_predict<<<nb, 64, 0, h->stream>>>(dm, st, c, w0m, w0c, wic, t, SP, gmean, vsq, kss, SP2);
        GPK_LAUNCH_CHECK(h);
        for (int j = 0; j < p; ++j) {
            const gpk_model m = obs_models[j];
            int rc = gpk_posterior(h, m->X, m->n, m->ldx, SP2, dm.M, m->Li, m->alpha, m->N, m->pp.cp, KsT, gmean + (size_t)j * dm.Mp, V,
                                   B, vsq + (size_t)j * dm.Bp);
            if (rc) return rc;
        }
        ukf_update<<<nb, 64, 0, h->stream>>>(dm, st, w0m, w0c, wic, t, gmean, vsq, kss + d, dY, compute_ll, dOutM, dOutC);
        GPK_LAUNCH_CHECK(h);
    }
    GPK_CUDA(h, cudaMemcpyAsync(hidden_means, dOutM, (size_t)B * T * d * sizeof(double), cudaMemcpyDeviceToHost, h->stream));
    GPK_CUDA(h, cudaMemcpyAsync(hidden_covs, dOutC, (size_t)B * T * d * d * sizeof(double), cudaMemcpyDeviceToHost, h->stream));
    if (ll) GPK_CUDA(h, cudaMemcpyAsync(ll, st.ll, (size_t)B * sizeof(double), cudaMemcpyDeviceToHost, h->stream));
    int info = 0;
    GPK_CUDA(h, cudaMemcpyAsync(&info, st.info, sizeof(int), cudaMemcpyDeviceToHost, h->stream));
    GPK_CUDA(h, cudaStreamSynchronize(h->stream));
    if (info) {
        h->last_info = info;
        return gpk_set_error(h, GPK_ENOTPD, "GP-UKF: covariance of filter %d is not positive definite at time step %d", (info - 1) % B, (info - 1) / B);
    }
    return GPK_OK;
}

}  // extern "C"
