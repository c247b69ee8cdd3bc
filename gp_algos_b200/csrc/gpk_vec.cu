// gpk_vec.cu -- O(n^2) / O(n) pieces of the path: triangular matrix-vector products (the alpha = L^-t (L^-1 y)
// solves of GpPredictor.scala:121-122, done with the explicit inverse that gpk_chol.cu produces), the
// log-marginal-likelihood reduction (GpPredictor.scala:144-149), padding / triangle copies at the ABI.
// All reductions are order-deterministic (no floating-point atomics).  Every kernel is batched over independent
// problems through a grid dimension (matrix b at base + b*N*N, vector b at base + b*N).
#include "gpk_internal.cuh"

namespace {

constexpr int KCH = 256;   // k-chunk of the split-k lower matvec (short chunks: ~2000 CTAs at n = 8192 keep enough loads in flight)

// partial[b][chunk][r] = sum_{k in chunk, k < rowblock_end} Li_b[r + k*N] * y_b[k]
__global__ void __launch_bounds__(128) trmv_lower_partial(const double* __restrict__ Li, int N, const double* __restrict__ y,
                                                          double* __restrict__ partial, int nch) {
    const int rb = blockIdx.x, ch = blockIdx.y;
    const int64_t b = blockIdx.z;
    const int k0 = ch * KCH;
    const int rend = (rb + 1) * GPK_TILE;
    if (k0 >= rend) return;
    Li += b * (int64_t)N * N;
    y += b * N;
    partial += b * (int64_t)nch * N;
    const int k1 = min(k0 + KCH, rend);
    const int r = rb * GPK_TILE + threadIdx.x;
    const double* col = Li + r + (int64_t)k0 * N;
    double a0 = 0, a1 = 0, a2 = 0, a3 = 0;
    int k = k0;
    for (; k + 7 < k1; k += 8) {
        const double m0 = col[0], m1 = col[N], m2 = col[2 * (int64_t)N], m3 = col[3 * (int64_t)N];
        const double m4 = col[4 * (int64_t)N], m5 = col[5 * (int64_t)N], m6 = col[6 * (int64_t)N], m7 = col[7 * (int64_t)N];
        a0 += m0 * y[k];     a1 += m1 * y[k + 1]; a2 += m2 * y[k + 2]; a3 += m3 * y[k + 3];
        a0 += m4 * y[k + 4]; a1 += m5 * y[k + 5]; a2 += m6 * y[k + 6]; a3 += m7 * y[k + 7];
        col += 8 * (int64_t)N;
    }
    for (; k < k1; ++k) { a0 += col[0] * y[k]; col += N; }
    partial[(int64_t)ch * N + r] = (a0 + a1) + (a2 + a3);
}

__global__ void trmv_lower_finish(const double* __restrict__ partial, int N, double* __restrict__ z, int nch) {
    const int r = blockIdx.x * blockDim.x + threadIdx.x;
    const int64_t b = blockIdx.y;
    if (r >= N) return;
    partial += b * (int64_t)nch * N;
    const int rend = (r / GPK_TILE + 1) * GPK_TILE;
    double acc = 0.0;
    for (int ch = 0; ch * KCH < rend; ++ch) acc += partial[(int64_t)ch * N + r];
    z[b * N + r] = acc;
}

// out[c] = sum_{r >= rstart(c)} M[r + c*ld] * v[r]; one warp per column.  tri != 0: rstart = 128-block of c.
__global__ void __launch_bounds__(256) colwise_dot(const double* __restrict__ M, int64_t ld, int rows, int cols,
                                                   const double* __restrict__ v, double* __restrict__ out, int tri, int square,
                                                   int64_t strideM, int64_t strideV, int64_t strideOut) {
    const int c = blockIdx.x * 8 + (threadIdx.x >> 5);
    if (c >= cols) return;
    const int64_t b = blockIdx.y;
    M += b * strideM;
    if (v) v += b * strideV;
    out += b * strideOut;
    const int lane = threadIdx.x & 31;
    const int rs = tri ? (c / GPK_TILE) * GPK_TILE : 0;
    const double* col = M + (int64_t)c * ld;
    double a0 = 0, a1 = 0;
    int r = rs + lane;
    for (; r + 32 < rows; r += 64) {
        const double m0 = col[r], m1 = col[r + 32];
        a0 += m0 * (square ? m0 : v[r]);
        a1 += m1 * (square ? m1 : v[r + 32]);
    }
    if (r < rows) { const double m0 = col[r]; a0 += m0 * (square ? m0 : v[r]); }
    double a = a0 + a1;
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) a += __shfl_xor_sync(0xffffffffu, a, o);
    if (lane == 0) out[c] = a;
}

__global__ void __launch_bounds__(256) loglik_kernel(const double* __restrict__ A, int N, int n, const double* __restrict__ y,
                                                     const double* __restrict__ alpha, double* __restrict__ out,
                                                     int64_t strideOut) {
    __shared__ double sd[256], sl[256];
    const int64_t b = blockIdx.x;
    A += b * (int64_t)N * N;
    y += b * N;
    alpha += b * N;
    double d = 0.0, l = 0.0;
    for (int i = threadIdx.x; i < n; i += 256) {
        d += y[i] * alpha[i];
        l += log(A[i + (int64_t)i * N]);
    }
    sd[threadIdx.x] = d; sl[threadIdx.x] = l;
    __syncthreads();
    for (int s = 128; s > 0; s >>= 1) {
        if (threadIdx.x < s) { sd[threadIdx.x] += sd[threadIdx.x + s]; sl[threadIdx.x] += sl[threadIdx.x + s]; }
        __syncthreads();
    }
    if (threadIdx.x == 0) out[b * strideOut] = -0.5 * sd[0] - sl[0] - 0.5 * n * log(2.0 * 3.14159265358979323846);
}

// y = alpha * M x + beta * y, M m x ncols column-major.  Split over column chunks (grid.y) so that a tall panel
// (m = 32768, ncols = 1024) keeps ~8 MB of loads in flight; partial sums go to scratch and are added in chunk order
// (deterministic, no floating-point atomics).  One thread per row, coalesced over rows.
__global__ void __launch_bounds__(128) gemv_n_partial(int m, int ncols, int cchunk, const double* __restrict__ M, int64_t ld,
                                                      const double* __restrict__ x, double* __restrict__ partial) {
    const int r = blockIdx.x * 128 + threadIdx.x;
    if (r >= m) return;
    const int c0 = blockIdx.y * cchunk, c1 = min(c0 + cchunk, ncols);
    const double* p = M + r + (int64_t)c0 * ld;
    double a0 = 0, a1 = 0, a2 = 0, a3 = 0;
    int c = c0;
    for (; c + 3 < c1; c += 4) {
        a0 += p[0] * x[c];
        a1 += p[ld] * x[c + 1];
        a2 += p[2 * ld] * x[c + 2];
        a3 += p[3 * ld] * x[c + 3];
        p += 4 * ld;
    }
    for (; c < c1; ++c) { a0 += p[0] * x[c]; p += ld; }
    partial[(int64_t)blockIdx.y * m + r] = (a0 + a1) + (a2 + a3);
}
__global__ void gemv_n_finish(int m, int nchunks, double alpha, const double* __restrict__ partial, double beta,
                              double* __restrict__ y) {
    const int r = blockIdx.x * blockDim.x + threadIdx.x;
    if (r >= m) return;
    double acc = 0.0;
    for (int ch = 0; ch < nchunks; ++ch) acc += partial[(int64_t)ch * m + r];
    y[r] = (beta == 0.0) ? alpha * acc : alpha * acc + beta * y[r];
}
// A[i + i*ld] += v for i < n
__global__ void add_diag_kernel(double* A, int64_t ld, int n, double v) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n) A[i + (int64_t)i * ld] += v;
}
// out[0] (+)= sum_{i<n} log A[i + i*ld]   (one CTA, fixed summation order)
__global__ void __launch_bounds__(256) sum_log_diag_kernel(const double* __restrict__ A, int64_t ld, int n, double* out,
                                                           int accumulate) {
    __shared__ double sl[256];
    double l = 0.0;
    for (int i = threadIdx.x; i < n; i += 256) l += log(A[i + (int64_t)i * ld]);
    sl[threadIdx.x] = l;
    __syncthreads();
    for (int s = 128; s > 0; s >>= 1) {
        if (threadIdx.x < s) sl[threadIdx.x] += sl[threadIdx.x + s];
        __syncthreads();
    }
    if (threadIdx.x == 0) out[0] = accumulate ? out[0] + sl[0] : sl[0];
}
// y[c] = alpha * sum_r M[r + c*ld] x[r] + beta * y[c]: one warp per column
__global__ void __launch_bounds__(256) gemv_t_kernel(int m, int ncols, double alpha, const double* __restrict__ M, int64_t ld,
                                                     const double* __restrict__ x, double beta, double* __restrict__ y) {
    const int c = blockIdx.x * 8 + (threadIdx.x >> 5);
    if (c >= ncols) return;
    const int lane = threadIdx.x & 31;
    const double* col = M + (int64_t)c * ld;
    double a0 = 0, a1 = 0;
    int r = lane;
    for (; r + 32 < m; r += 64) { a0 += col[r] * x[r]; a1 += col[r + 32] * x[r + 32]; }
    if (r < m) a0 += col[r] * x[r];
    double a = a0 + a1;
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) a += __shfl_xor_sync(0xffffffffu, a, o);
    if (lane == 0) y[c] = (beta == 0.0) ? alpha * a : alpha * a + beta * y[c];
}

__global__ void pad_vector_kernel(double* dst, int N, const double* src, int n) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    const int64_t b = blockIdx.y;
    if (i < N) dst[b * N + i] = (i < n) ? src[b * n + i] : 0.0;
}

// dst (N x N): lower triangle (and full diagonal 128-blocks) of the symmetric src, identity padding.
__global__ void load_sym_padded_kernel(double* dst, int N, const double* src, int n, int64_t lds, int* notsym) {
    const int r = blockIdx.y * blockDim.x + threadIdx.x, c = blockIdx.x;
    if (r >= N) return;
    double v;
    if (r < n && c < n) {
        v = src[r + (int64_t)c * lds];
        if (notsym != nullptr && r > c && v != src[c + (int64_t)r * lds]) *notsym = 1;
    } else {
        v = (r == c) ? 1.0 : 0.0;
    }
    dst[r + (int64_t)c * N] = v;
}

// triangular load: dst (N x N) lower-triangular with identity padding; transpose_in: src holds the upper factor
__global__ void load_tri_padded_kernel(double* dst, int N, const double* src, int n, int64_t lds, int transpose_in) {
    const int r = blockIdx.y * blockDim.x + threadIdx.x, c = blockIdx.x;
    if (r >= N) return;
    double v = 0.0;
    if (r < n && c < n) {
        if (r >= c) v = transpose_in ? src[c + (int64_t)r * lds] : src[r + (int64_t)c * lds];
    } else if (r == c) {
        v = 1.0;
    }
    dst[r + (int64_t)c * N] = v;
}

// dst (n x n, ld) = tri(src): lower triangle of src (transpose == 0) or its transpose into the upper triangle
__global__ void store_tri_kernel(double* dst, int64_t ldd, const double* src, int N, int n, int transpose) {
    const int r = blockIdx.y * blockDim.x + threadIdx.x, c = blockIdx.x;
    if (r >= n || c >= n) return;
    double v = 0.0;
    if (!transpose) { if (r >= c) v = src[r + (int64_t)c * N]; }
    else            { if (c >= r) v = src[c + (int64_t)r * N]; }
    dst[r + (int64_t)c * ldd] = v;
}

}  // namespace

int gpk_trmv_lower(gpk_handle h, const double* Li, int N, const double* y, double* z, double* scratch, int batch) {
    const int nch = (N + KCH - 1) / KCH;
    dim3 grid(N / GPK_TILE, nch, batch);
    trmv_lower_partial<<<grid, 128, 0, h->stream>>>(Li, N, y, scratch, nch);
    GPK_LAUNCH_CHECK(h);
    trmv_lower_finish<<<dim3((N + 255) / 256, batch), 256, 0, h->stream>>>(scratch, N, z, nch);
    GPK_LAUNCH_CHECK(h);
    return GPK_OK;
}

int gpk_trmv_lower_t(gpk_handle h, const double* Li, int N, const double* z, double* a, int batch) {
    colwise_dot<<<dim3((N + 7) / 8, batch), 256, 0, h->stream>>>(Li, N, N, N, z, a, 1, 0, (int64_t)N * N, N, N);
    GPK_LAUNCH_CHECK(h);
    return GPK_OK;
}

size_t gpk_trmv_scratch_doubles(int N) { return (size_t)((N + KCH - 1) / KCH) * N; }

int gpk_colwise_dot(gpk_handle h, const double* M, int64_t ld, int rows, int cols, const double* v, double* out, int square,
                    int batch, int64_t strideM, int64_t strideV, int64_t strideOut) {
    if (cols <= 0) return GPK_OK;
    colwise_dot<<<dim3((cols + 7) / 8, batch), 256, 0, h->stream>>>(M, ld, rows, cols, v, out, 0, square, strideM, strideV, strideOut);
    GPK_LAUNCH_CHECK(h);
    return GPK_OK;
}

int gpk_gemv(gpk_handle h, int trans, int m, int ncols, double alpha, const double* M, int64_t ld, const double* x, double beta,
             double* y) {
    const int ny = trans ? ncols : m;
    if (ny <= 0) return GPK_OK;
    if ((trans ? m : ncols) <= 0) {   // empty product: y = beta * y (y = 0 for beta == 0, whatever y held)
        gemv_n_finish<<<(ny + 255) / 256, 256, 0, h->stream>>>(ny, 0, alpha, nullptr, beta, y);
        GPK_LAUNCH_CHECK(h);
        return GPK_OK;
    }
    if (!trans) {
        const int rblocks = (m + 127) / 128;
        int nch = (4 * 148 + rblocks - 1) / rblocks;               // ~4 CTAs per SM in total
        nch = max(1, min(nch, (ncols + 63) / 64));                 // at least 64 columns per chunk
        const int cchunk = ((ncols + nch - 1) / nch + 3) & ~3;
        nch = (ncols + cchunk - 1) / cchunk;
        double* partial = (double*)gpk_arena(h, ARENA_GEMV, (size_t)nch * m * sizeof(double));
        if (!partial) return GPK_ENOMEM;
        gemv_n_partial<<<dim3(rblocks, nch), 128, 0, h->stream>>>(m, ncols, cchunk, M, ld, x, partial);
        GPK_LAUNCH_CHECK(h);
        gemv_n_finish<<<(m + 255) / 256, 256, 0, h->stream>>>(m, nch, alpha, partial, beta, y);
    } else {
        gemv_t_kernel<<<(ncols + 7) / 8, 256, 0, h->stream>>>(m, ncols, alpha, M, ld, x, beta, y);
    }
    GPK_LAUNCH_CHECK(h);
    return GPK_OK;
}

int gpk_add_diag(gpk_handle h, double* A, int64_t ld, int n, double v) {
    if (n <= 0) return GPK_OK;
    add_diag_kernel<<<(n + 255) / 256, 256, 0, h->stream>>>(A, ld, n, v);
    GPK_LAUNCH_CHECK(h);
    return GPK_OK;
}

int gpk_sum_log_diag(gpk_handle h, const double* A, int64_t ld, int n, double* out, int accumulate) {
    sum_log_diag_kernel<<<1, 256, 0, h->stream>>>(A, ld, n, out, accumulate);
    GPK_LAUNCH_CHECK(h);
    return GPK_OK;
}

int gpk_loglik(gpk_handle h, const double* A, int N, int n, const double* y, const double* alpha, double* out, int batch,
               int64_t strideOut) {
    loglik_kernel<<<batch, 256, 0, h->stream>>>(A, N, n, y, alpha, out, strideOut);
    GPK_LAUNCH_CHECK(h);
    return GPK_OK;
}

int gpk_copy2d(gpk_handle h, double* dst, int64_t ldd, const double* src, int64_t lds, int rows, int cols) {
    if (rows <= 0 || cols <= 0) return GPK_OK;
    GPK_CUDA(h, cudaMemcpy2DAsync(dst, ldd * sizeof(double), src, lds * sizeof(double), (size_t)rows * sizeof(double),
                                  (size_t)cols, cudaMemcpyDeviceToDevice, h->stream));
    return GPK_OK;
}

int gpk_pad_vector(gpk_handle h, double* dst, int N, const double* src, int n, int batch) {
    pad_vector_kernel<<<dim3((N + 255) / 256, batch), 256, 0, h->stream>>>(dst, N, src, n);
    GPK_LAUNCH_CHECK(h);
    return GPK_OK;
}

int gpk_load_sym_padded(gpk_handle h, double* dst, int N, const double* src, int n, int64_t lds, int* d_notsym) {
    load_sym_padded_kernel<<<dim3(N, (N + 127) / 128), 128, 0, h->stream>>>(dst, N, src, n, lds, d_notsym);
    GPK_LAUNCH_CHECK(h);
    return GPK_OK;
}

int gpk_load_tri_padded(gpk_handle h, double* dst, int N, const double* src, int n, int64_t lds, int transpose_in) {
    load_tri_padded_kernel<<<dim3(N, (N + 127) / 128), 128, 0, h->stream>>>(dst, N, src, n, lds, transpose_in);
    GPK_LAUNCH_CHECK(h);
    return GPK_OK;
}

int gpk_store_tri(gpk_handle h, double* dst, int64_t ldd, const double* src, int N, int n, int transpose) {
    if (n <= 0) return GPK_OK;
    store_tri_kernel<<<dim3(n, (n + 127) / 128), 128, 0, h->stream>>>(dst, ldd, src, N, n, transpose);
    GPK_LAUNCH_CHECK(h);
    return GPK_OK;
}

int gpk_store_lower(gpk_handle h, double* dst, int64_t ldd, const double* src, int N, int n) {
    return gpk_store_tri(h, dst, ldd, src, N, n, 0);
}
