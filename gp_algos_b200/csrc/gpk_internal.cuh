// gpk_internal.cuh -- shared declarations of libgpk's translation units (not part of the C ABI).
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>
#include <stdio.h>
#include <string.h>

#include <functional>

#include "../../include/gpk.h"

#define GPK_TILE 128
#define GPK_NPIPE 3
#define GPK_NSIDE 16     // side streams (one per recursion depth, cyclic; the second batch group starts at 4; the last one is
                         // also the panel stream of the factor-only look-ahead driver)
#define GPK_NGROUP 4     // grp[] has GPK_NGROUP - 1 main-priority streams: grp[0] runs the second batch group of the batched
                         // factorisation, grp[0..2] the narrow flushes of the EP sweep
#define GPK_NEVENTS 256  // fork/join event pool (cyclic)  // every internal matrix dimension / leading dimension is a multiple of this

struct gpk_handle_s {
    int device;
    cudaStream_t stream;       // the stream launches go to (temporarily swapped to a side / pipe stream by the drivers)
    cudaStream_t main_stream;  // the handle's own stream: never swapped
    int num_sms;
    bool own_stream;
    cudaStream_t side[GPK_NSIDE];
    cudaStream_t grp[GPK_NGROUP - 1];   // same priority as the main stream
    cudaStream_t pipe[GPK_NPIPE];   // lowest-priority streams of the pipelined factorisation (trailing updates; inverse rows; K^-1)
    cudaEvent_t evpool[GPK_NEVENTS];
    unsigned ev_next;
    // grow-only device arenas (A: factor / K^-1, B: L^-1, T: GEMM scratch, misc: small vectors)
    void* arena[16];
    size_t arena_bytes[16];
    double* h_pinned;  // 4096 doubles of pinned host scratch
    void* res_pinned;          // grow-only pinned staging for the results of batched calls
    size_t res_pinned_bytes;
    int* d_info;       // device int: first failing minor of the last factorisation
    int last_info;
    int64_t launches;
    unsigned func_cfg;  // bitmask: kernels whose dynamic-smem attribute has been set on this device
    void* pp_host;           // host staging for per-problem hyper-parameters (batched calls)
    size_t pp_host_bytes;
    // CUDA-graph replay of the single-problem evaluation (gpk_gp.cu: the evaluation is ~350 launches on 8 streams; an
    // optimiser calls it over and over with the same buffers and new hyper-parameters)
    int graph_mode;               // 0 off, 1 capture on the second call with one signature and replay from then on
    unsigned arena_epoch;         // bumped whenever an arena is (re)allocated: a cached graph holds arena pointers
    struct gpk_graph_slot* slots[3];   // cached graphs (gpk_graph.cu): GPK_SLOT_EVAL, GPK_SLOT_EP_SWEEP, GPK_SLOT_POTRF
    struct gpk_capture_log* cap;  // non-null while capturing: every kernel node with the priority of the stream it came from
    int prio_main, prio_side, prio_pipe;
    int kernel_family;            // gpk_kernel_family: how (D, theta) arguments are interpreted
    char err[512];
};
// fork / join helpers of the multi-stream schedules
struct StreamSwap {  // run the enclosed launches on another stream of the same handle
    gpk_handle h; cudaStream_t saved;
    StreamSwap(gpk_handle h_, cudaStream_t s) : h(h_), saved(h_->stream) { h->stream = s; }
    ~StreamSwap() { h->stream = saved; }
};
static inline cudaEvent_t next_event(gpk_handle h) { return h->evpool[h->ev_next++ % GPK_NEVENTS]; }
// ---- graph replay (gpk_graph.cu) ----
#define GPK_NSLOTS 3
enum { GPK_SLOT_EVAL = 0, GPK_SLOT_EP_SWEEP = 1, GPK_SLOT_POTRF = 2 };
struct GraphKey { const void* p[6]; int64_t i[6]; };   // zero-initialise, then fill: compared bytewise
void gpk_capture_note(gpk_handle h);
void gpk_graph_drop_all(gpk_handle h);                  // forget every cached graph (handle teardown, graph mode off)
// Runs `body` (a launch sequence on h->stream that forks/joins the handle's other streams and synchronises nothing) eagerly on
// the first call with `key`, captures it on the second and replays the instantiated graph afterwards.
int gpk_graph_run_impl(gpk_handle h, int slot, const GraphKey& key, int eager_calls, int (*body)(void*), void* ctx, const char* what);
template <class F>
int gpk_graph_run(gpk_handle h, int slot, const GraphKey& key, int eager_calls, F& body, const char* what) {
    return gpk_graph_run_impl(h, slot, key, eager_calls, [](void* c) { return (*static_cast<F*>(c))(); }, &body, what);
}

enum { ARENA_A = 0, ARENA_B = 1, ARENA_T = 2, ARENA_MISC = 3, ARENA_X = 4, ARENA_IO = 5, ARENA_IO2 = 6, ARENA_IO3 = 7, ARENA_PP = 8, ARENA_INFO = 9, ARENA_GEMV = 10, ARENA_KINV = 11, GPK_NARENA = 12 };

int gpk_set_error(gpk_handle h, int status, const char* fmt, ...);
// returns device pointer to at least `bytes` bytes in arena `which` (contents undefined after growth)
void* gpk_arena(gpk_handle h, int which, size_t bytes);
int gpk_upload_matrix(gpk_handle h, double* dst, const double* src, int rows, int cols, int64_t ld);   // host (ld) -> device (ld = rows)
int gpk_download_matrix(gpk_handle h, double* dst, int64_t ld, const double* src, int rows, int cols);  // device (ld = rows) -> host (ld)
int gpk_finish_info(gpk_handle h);  // sync, read h->d_info[0], map to GPK_ENOTPD

#define GPK_CUDA(h, call)                                                                         \
    do {                                                                                          \
        cudaError_t e__ = (call);                                                                 \
        if (e__ != cudaSuccess)                                                                   \
            return gpk_set_error((h), e__ == cudaErrorMemoryAllocation ? GPK_ENOMEM : GPK_ECUDA,  \
                                 "%s failed: %s (%s:%d)", #call, cudaGetErrorString(e__), __FILE__, __LINE__); \
    } while (0)

#define GPK_LAUNCH_CHECK(h)                                                                       \
    do {                                                                                          \
        (h)->launches++;                                                                          \
        if ((h)->cap) gpk_capture_note(h);                                                        \
        cudaError_t e__ = cudaGetLastError();                                                     \
        if (e__ != cudaSuccess)                                                                   \
            return gpk_set_error((h), GPK_ECUDA, "kernel launch failed: %s (%s:%d)",              \
                                 cudaGetErrorString(e__), __FILE__, __LINE__);                    \
    } while (0)

static inline int gpk_pad(int n) { return (n + GPK_TILE - 1) / GPK_TILE * GPK_TILE; }

// ---------------------------------------------------------------------------------------------
// DMMA GEMM (gpk_gemm.cu).  Computes, for every 64x64 tile (first row r0, first column s0) selected by `tri_out`,
//     D(r,s) = alpha * sum_{k in [kbeg,kend)} P(r,k) * Q(s,k) + beta * Cin(r,s)
// with D(r,s) stored at D[s + r*ldd] (s contiguous).  For a column-major C (M x N) this is D = C^t:
// r is C's column index, s is C's row index.  Cin may be null (no beta term, Cin never read) or alias D.
//   p_kcontig: P(r,k) at P[k + r*ldp]   else P[r + k*ldp]
//   q_kcontig: Q(s,k) at Q[k + s*ldq]   else Q[s + k*ldq]
// k-range per tile (tile-granular exploitation of triangular operands):
//   kbeg = max(kb_r ? r0 : 0, kb_s ? s0 : 0);  kend = min(K, ke_r ? r0+64 : K, ke_s ? s0+64 : K)
// so a triangular operand must hold real zeros inside its diagonal 64-tile; beyond that tile nothing is read.
// tri_out: only tiles with s0 >= r0 are computed (lower triangle of the column-major C); the other tiles of D are not written.
// R, S multiples of 64; K multiple of 16; pointers 16-byte aligned; ld's even (gpk_gemm returns GPK_EINVAL otherwise).
// ---------------------------------------------------------------------------------------------
struct GemmDesc {
    const double* P; int64_t ldp; int64_t strideP;
    const double* Q; int64_t ldq; int64_t strideQ;
    double* D; int64_t ldd; int64_t strideD;
    const double* Cin; int64_t ldc; int64_t strideC;
    int R, S, K;
    int batch;
    double alpha, beta;
    int p_kcontig, q_kcontig;
    int tri_out;
    int kb_r, kb_s, ke_r, ke_s;
    int heavy_last;  // reverse tile order (heavy tiles are at high indices)
};
static inline GemmDesc gemm_desc() {
    GemmDesc g;
    memset(&g, 0, sizeof(g));
    g.batch = 1; g.alpha = 1.0; g.beta = 0.0;
    return g;
}
int gpk_gemm(gpk_handle h, const GemmDesc& g);

// ---------------------------------------------------------------------------------------------
// Batching convention (C4: many independent GPs of the same shape, SURVEY.md 8(e)): every internal routine takes a
// trailing `batch` count.  Problem b uses matrix b at base + b*N*N, vector b at base + b*N, X at dX + b*strideX
// (strideX == 0: all problems share X, the GP-UKF case), y at dy + b*n, and hyper-parameters pp_dev[b].  With
// batch == 1 and pp_dev == nullptr the hyper-parameters travel by value in the kernel arguments.
// ---------------------------------------------------------------------------------------------
#define GPK_MAX_D 64
#define GPK_CO2_NPARAMS 11
struct CovParams {
    int D;
    int kind;            // gpk_kernel_family
    double sf2;          // SE-ARD: signalVar*signalVar.          Co2: k(x,x) without noise = hp1^2 + hp3^2 + hp6^2 + hp9^2
    double sn2;          // SE-ARD: noiseVar*noiseVar.            Co2: hp11^2
    double extra_diag;   // Option sigmaNoise (un-squared), 0 when None
    double inv_ls2[GPK_MAX_D];  // SE-ARD: 1/(ls*ls).             Co2: hp1..hp11, then pow(hp2,-3), pow(hp4,-3), pow(hp5,-3), pow(hp7,-3), pow(hp10,-3)
};
// k(x, x) with the i == j noise term (MatrixUtils.scala:63): the prior variance a posterior variance is taken from
static inline __host__ __device__ double gpk_prior_var(const CovParams& cp) { return cp.sf2 + cp.sn2; }
static inline int gpk_theta_len(const gpk_handle_s* h, int D) { return h->kernel_family == GPK_KERNEL_CO2 ? GPK_CO2_NPARAMS : D + 2; }

#ifdef __CUDACC__
// gp/regression/Co2Prediction.scala:38-56 (apply) and :66-137 (derAfterHyperParam) on one pair of 1-D inputs, xd = x1 - x2.
// Products and sums keep the Scala evaluation order; intrinsics keep nvcc from contracting a*b+c into an fma where the JVM
// rounds twice.  par = CovParams::inv_ls2 of the Co2 family.
struct Co2Terms { double sq, s, e1, k2, p1, pw, k4; };
__device__ __forceinline__ double co2_value(const double* __restrict__ par, double xd, Co2Terms& t) {
    const double hp1 = par[0], hp2 = par[1], hp3 = par[2], hp4 = par[3], hp5 = par[4], hp6 = par[5], hp7 = par[6], hp8 = par[7],
                 hp9 = par[8], hp10 = par[9];
    t.sq = __dmul_rn(xd, xd);
    t.e1 = exp(-t.sq / __dmul_rn(__dmul_rn(2.0, hp2), hp2));
    t.s = sin(__dmul_rn(3.14159265358979323846, xd));
    const double a2 = -t.sq / __dmul_rn(__dmul_rn(2.0, hp4), hp4);
    const double b2 = __dmul_rn(__dmul_rn(2.0, t.s), t.s) / __dmul_rn(hp5, hp5);
    t.k2 = __dmul_rn(__dmul_rn(hp3, hp3), exp(__dsub_rn(a2, b2)));
    t.p1 = __dadd_rn(1.0, t.sq / __dmul_rn(__dmul_rn(__dmul_rn(2.0, hp8), hp7), hp7));
    t.pw = pow(t.p1, -hp8);
    t.k4 = __dmul_rn(__dmul_rn(hp9, hp9), exp(-t.sq / __dmul_rn(__dmul_rn(2.0, hp10), hp10)));
    const double k1 = __dmul_rn(__dmul_rn(hp1, hp1), t.e1), k3 = __dmul_rn(__dmul_rn(hp6, hp6), t.pw);
    return __dadd_rn(__dadd_rn(__dadd_rn(k1, t.k2), k3), t.k4);
}
// dk/dhp_p for p = 1..10 (0-based slot p-1) from the shared sub-expressions; p = 11 is 2 hp11 [i == j] and handled by the callers
__device__ __forceinline__ void co2_derivs(const double* __restrict__ par, const Co2Terms& t, double* __restrict__ dk) {
    const double hp1 = par[0], hp3 = par[2], hp6 = par[5], hp7 = par[6], hp8 = par[7], hp9 = par[8];
    dk[0] = __dmul_rn(__dmul_rn(2.0, hp1), t.e1);
    dk[1] = __dmul_rn(__dmul_rn(__dmul_rn(__dmul_rn(hp1, hp1), t.e1), t.sq), par[11]);
    dk[2] = __dmul_rn(2.0, t.k2) / hp3;
    dk[3] = __dmul_rn(__dmul_rn(t.k2, t.sq), par[12]);
    dk[4] = __dmul_rn(__dmul_rn(__dmul_rn(__dmul_rn(t.k2, 4.0), t.s), t.s), par[13]);
    dk[5] = __dmul_rn(__dmul_rn(2.0, hp6), t.pw);
    dk[6] = __dmul_rn(__dmul_rn(__dmul_rn(__dmul_rn(hp6, hp6), pow(t.p1, __dsub_rn(-hp8, 1.0))), t.sq), par[14]);
    const double lg = log(t.p1);
    const double first = exp(__dmul_rn(-hp8, lg));
    const double den = __dmul_rn(__dmul_rn(__dmul_rn(__dmul_rn(__dmul_rn(2.0, hp7), hp7), hp8), hp8), t.p1);
    const double second = __dadd_rn(-lg, __dmul_rn(hp8, t.sq) / den);
    dk[7] = __dmul_rn(__dmul_rn(__dmul_rn(hp6, hp6), first), second);
    dk[8] = __dmul_rn(2.0, t.k4) / hp9;
    dk[9] = __dmul_rn(__dmul_rn(t.k4, t.sq), par[15]);
}
#endif
struct ProblemParams {
    CovParams cp;
    double gscale[GPK_MAX_D + 2];  // 1/2 * {2 sf, sf^2 / l_d^3 ..., 2 sn}: factors of the gradient trace
};
int gpk_make_cov_params(gpk_handle h, const double* theta, int D, int has_sigma_noise, double sigma_noise, CovParams* out);
int gpk_make_problem_params(gpk_handle h, const double* theta, int D, int has_sigma_noise, double sigma_noise, ProblemParams* out);

// a device-resident fitted GP (gpk_gp.cu creates / destroys it; gpk_ukf.cu reads it)
struct gpk_model_s {
    int n, N, D;
    int ldx;        // rows allocated for X (>= n; == N so that gpk_gp_model_append has room)
    double* X;      // n x D, ld ldx
    double* Li;     // N x N
    double* alpha;  // N
    double theta[GPK_MAX_D + 2];
    ProblemParams pp;
    int has_s;      // Option sigmaNoise the model was fitted with (GpPredictor.scala:116-117) ...
    double s;       // ... replayed by gpk_gp_model_append
};

// computePosterior (GpPredictor.scala:45-58) up to the prior variance, for `batch` GPs of padded size N at ms test rows
// (gpk_gp.cu).  Problem b: X at dX + b*strideX (n rows, ld ldx), X* at dXs + b*strideXs (ld ms), Li (N x N) at + b*N*N,
// alpha (N) at + b*N, hyper-parameters cp (batch == 1) or pp_dev[b].  With M = gpk_pad(ms) it writes, at + b*N*M resp. + b*M:
//   KsT   N x M (ld N)   k(X, X*) with zero padding
//   mean  M              K* alpha
//   V     N x M (ld N)   Li KsT over the first gpk_pad(nv) columns only, so with batch == 1 N x gpk_pad(nv) suffices
//                        (nv <= ms; nv == ms when batch > 1); skipped when null
//   vsq   M              column sums of squares of V over the first nv columns; needs V; skipped when null
int gpk_posterior(gpk_handle h, const double* dX, int n, int64_t ldx, const double* dXs, int ms, const double* Li,
                  const double* alpha, int N, const CovParams& cp, double* KsT, double* mean, double* V, int nv, double* vsq,
                  int batch = 1, int64_t strideX = 0, int64_t strideXs = 0, const ProblemParams* pp_dev = nullptr);

// ---------------------------------------------------------------------------------------------
// covariance (gpk_cov.cu)
// ---------------------------------------------------------------------------------------------
// full symmetric n x n (mirrored) into K (ld ldk)
int gpk_cov_sym_full(gpk_handle h, const double* dX, int n, int64_t ldx, const CovParams& cp, double* dK, int64_t ldk);
// lower tiles only of the padded N x N matrix (N = gpk_pad(n)); padding = identity
int gpk_cov_sym_lower_padded(gpk_handle h, const double* dX, int n, int64_t ldx, const CovParams& cp, double* dK, int N,
                             int batch = 1, int64_t strideX = 0, const ProblemParams* pp_dev = nullptr);
// rectangular m x n, no noise; rows>=m / cols>=n up to (mp, np) are zero-filled when mp/np > m/n
int gpk_cov_cross(gpk_handle h, const double* dX1, int m, int64_t ldx1, const double* dX2, int n, int64_t ldx2,
                  const CovParams& cp, double* dK, int64_t ldk, int mp, int np, int batch = 1, int64_t strideX1 = 0,
                  int64_t strideX2 = 0, int64_t strideK = 0, const ProblemParams* pp_dev = nullptr);
int gpk_cov_deriv(gpk_handle h, int param_num, const double* dX, int n, int64_t ldx, const CovParams& cp,
                  double sf, double sn, const double* ls_host, double* dK, int64_t ldk);

// ---------------------------------------------------------------------------------------------
// factorisation (gpk_chol.cu): A (N x N, ld N, lower, padded) -> L in place (lower part; when
// keep_L is 0 the off-diagonal blocks of A are left in an unspecified state, only diag(L) and the
// diagonal 128-blocks are valid), Li = L^-1 (N x N, ld N, lower; upper parts of diagonal blocks zeroed;
// blocks above the diagonal untouched).  T: scratch of at least gpk_chol_scratch_doubles(N) per problem.
// info_dev[b] receives 0 or the failing leading minor (1-based) of problem b.
// ---------------------------------------------------------------------------------------------
// base case (gpk_base.cu): `batch` 128x128 blocks at A + i*strideA; mode 0 = factor + invert, mode 1 = invert a given
// lower factor.  Block i reports into info[i*info_stride] with column offset col_offset + i*coloff_stride.
int gpk_base_potrf_trtri(gpk_handle h, double* A, int64_t lda, double* Li, int64_t ldi, int* info, int col_offset, int mode,
                         int batch, int64_t strideA, int64_t strideLi, int info_stride, int coloff_stride);
size_t gpk_chol_scratch_doubles(int N);
int gpk_potrf_inv(gpk_handle h, double* A, double* Li, double* T, int N, int keep_L, int* info_dev, int batch = 1);
// Look-ahead driver for one large problem (see gpk_chol.cu): same results as gpk_potrf_inv; when Kinv != nullptr it also
// accumulates K^-1 = Li^t Li (lower tiles) into Kinv (N x N, ld N, a buffer distinct from A and Li).
bool gpk_use_pipelined(int N, int batch);
// kinv_done != nullptr: returns without waiting for the K^-1 accumulation; the caller must cudaStreamWaitEvent(*kinv_done)
// (when non-null) on its stream before reading Kinv.
int gpk_potrf_inv_pipelined(gpk_handle h, double* A, double* Li, double* Kinv, double* T, int N, int keep_L, int* info_dev,
                            cudaEvent_t* kinv_done = nullptr);
// A -> L in place and V = L^-1 B (B, V: N x M, ld N; B destroyed); Li: N x N staging (holds L^-1 only when N is small)
// on_rows (optional): called on the host, in order, once per block row of V -- rows [row0, row0 + rows) are final when `ready` fires
// (the event is recorded on one of the handle's internal streams); lets a consumer of V start before the factorisation is done.
typedef std::function<int(int row0, int rows, cudaEvent_t ready)> GpkRowsHook;
int gpk_potrf_factor_solve(gpk_handle h, double* A, double* Li, double* T, int N, int* info_dev, double* B, double* V, int M,
                           const GpkRowsHook* on_rows = nullptr);
// L only (plus the inverses of the diagonal blocks, left in Li's diagonal blocks): n^3/3 flops.  Li: N x N staging.
int gpk_potrf_factor(gpk_handle h, double* A, double* Li, double* T, int N, int* info_dev);
// X = Lw^-1 B (backward == 0) or Lw^-t B (backward != 0) by blocked substitution on the padded lower factor Lw (N x N, ld N).
// Di: N x 128 scratch for the inverses of the diagonal blocks.  M > 0: B, X are N x M (ld N, M a multiple of 128);
// M == 0: one vector.  B is overwritten.
int gpk_trsm_padded(gpk_handle h, const double* Lw, double* Di, int N, int backward, double* B, double* X, int M);
// L^-1 for a given lower-triangular L (N x N padded, ld N)
int gpk_trtri_lower(gpk_handle h, const double* L, double* Li, double* T, int N);
// Kinv (lower triangle incl. diagonal tiles in full) = Li^t Li
int gpk_lauum_lower(gpk_handle h, const double* Li, double* Kinv, int N, int batch = 1);
// V = Li B for `batch` problems: B, V are N x M (ld N, M a multiple of 64) at + b*N*M, Li at + b*N*N.  Li is read up to the
// diagonal 64-tile of each row tile only (zero above the diagonal inside it, as gpk_potrf_inv leaves it); the blocks above
// may hold anything -- a resident model's are uninitialised memory.
int gpk_trmm_lower(gpk_handle h, const double* Li, int N, const double* B, double* V, int M, int batch = 1);

// ---------------------------------------------------------------------------------------------
// vectors / reductions / gradient (gpk_vec.cu, gpk_grad.cu)
// ---------------------------------------------------------------------------------------------
// z = Li * y (lower-triangular matvec, N padded; y has N entries with zeros in the padding); scratch: gpk_trmv_scratch_doubles(N) per problem
size_t gpk_trmv_scratch_doubles(int N);
int gpk_trmv_lower(gpk_handle h, const double* Li, int N, const double* y, double* z, double* scratch, int batch = 1);
// a = Li^t * z
int gpk_trmv_lower_t(gpk_handle h, const double* Li, int N, const double* z, double* a, int batch = 1);
// out[c] = sum_r M[r + c*ld] * v[r]  (square != 0: sum_r M[r + c*ld]^2), one warp per column
int gpk_colwise_dot(gpk_handle h, const double* M, int64_t ld, int rows, int cols, const double* v, double* out, int square,
                    int batch = 1, int64_t strideM = 0, int64_t strideV = 0, int64_t strideOut = 0);
// y = alpha * op(M) x + beta * y for a column-major m x ncols matrix (trans: y has ncols entries)
int gpk_gemv(gpk_handle h, int trans, int m, int ncols, double alpha, const double* M, int64_t ld, const double* x, double beta,
             double* y);
int gpk_add_diag(gpk_handle h, double* A, int64_t ld, int n, double v);                                       // A_ii += v
int gpk_sum_log_diag(gpk_handle h, const double* A, int64_t ld, int n, double* out, int accumulate);         // sum_i log A_ii
// out[b*strideOut] = -0.5*y.alpha - sum_{i<n} log(diag_i(A)) - 0.5*n*log(2 pi)   (GpPredictor.scala:144-149)
int gpk_loglik(gpk_handle h, const double* A, int N, int n, const double* y, const double* alpha, double* out, int batch = 1,
               int64_t strideOut = 0);
// g[b*strideOut + p] = 0.5 * sum_{i,j<n} (alpha_i alpha_j - Kinv_ij) * dk_p(x_i,x_j,i==j)  for p < nparams
int gpk_grad_trace(gpk_handle h, const double* Kinv, int N, const double* dX, int n, int64_t ldx, const double* alpha,
                   const ProblemParams& pp, int nparams, double* g_out, double* scratch, int batch = 1, int64_t strideX = 0,
                   const ProblemParams* pp_dev = nullptr, int64_t strideOut = 0);
size_t gpk_grad_scratch_doubles(int N, int D);

// misc elementwise helpers (gpk_vec.cu)
int gpk_copy2d(gpk_handle h, double* dst, int64_t ldd, const double* src, int64_t lds, int rows, int cols);
// dst[b*N + i] = i < n ? src[b*n + i] : 0
int gpk_pad_vector(gpk_handle h, double* dst, int N, const double* src, int n, int batch = 1);
// dst (N x N padded, lower + identity padding) from src (n x n, ld lds); optionally checks symmetry -> d_flag
int gpk_load_sym_padded(gpk_handle h, double* dst, int N, const double* src, int n, int64_t lds, int* d_notsym);
// dst (n x n, ld) = lower triangle of src (N x N) with zeros above the diagonal
int gpk_store_lower(gpk_handle h, double* dst, int64_t ldd, const double* src, int N, int n);
int gpk_store_tri(gpk_handle h, double* dst, int64_t ldd, const double* src, int N, int n, int transpose);
int gpk_load_tri_padded(gpk_handle h, double* dst, int N, const double* src, int n, int64_t lds, int transpose_in);
