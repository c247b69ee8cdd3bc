// gpk_chol.cu -- FP64 Cholesky factor AND its triangular inverse, built together.
// Replaces breeze `cholesky` -> LAPACK dpotrf('L') (GpPredictor.scala:120, EpParameterEstimator.scala:58),
// utils/MatrixUtils.scala:106-113 invTriangular (n dense forward solves, n^3/2 scalar MACs in the
// reference) and the `lInversed.t * lInversed` dgemm (GpPredictor.scala:67).
//
// Algorithm (recursive, everything O(n^3) is a DMMA GEMM from gpk_gemm.cu):
//   potrf_inv(A, Li, n):                      A = [A11 . ; A21 A22],  Li = [Li11 . ; Li21 Li22]
//     potrf_inv(A11, Li11)                    L11, L11^-1
//     L21 = A21 * Li11^t                      (TRSM as a GEMM with the already-known inverse; k <= r0+127)
//     A22 -= L21 * L21^t                      (SYRK, lower tiles only)          <- the trailing update
//     potrf_inv(A22, Li22)
//     Li21 = -Li22 * (L21 * Li11)             (two triangular-aware GEMMs)
//   base case n = 128: one CTA factors the block in shared memory and inverts it in place (gpk_base.cu).
// Total n^3/3 (factor) + n^3/3 (inverse) flops; the K^-1 = Li^t Li product (another n^3/3, lower only)
// is a single GEMM launch (gpk_lauum_lower).  Because L^-1 is a by-product, every triangular solve of
// the path (alpha, V = L^-1 K*^t) becomes a matrix product as well.
//
// Batched mode (`batch` independent problems of the same N, matrices N*N apart): every launch of the recursion
// covers all problems through the GEMM's / base kernel's batch dimension, so 512 problems of n = 1024 cost the
// same 45 launches as one.
#include "gpk_internal.cuh"

#include <stdlib.h>

namespace {

constexpr int NB = GPK_TILE;  // 128

struct Ctx {
    gpk_handle h;
    int64_t ld;            // leading dimension of A and Li (== N)
    int keep_L;
    int* info;             // device, one int per problem
    int batch;
    int64_t sM;            // matrix stride between problems (N*N)
    int64_t sT;            // scratch stride between problems
    int side_base;         // first side stream of this batch group
};

int side_min() {
    static int v = -1;
    if (v < 0) { const char* e = getenv("GPK_SIDE_MIN"); v = e ? atoi(e) : 256; }
    return v;
}

int pipe_nb() {      // block-column width of the pipelined driver
    static int v = -1;
    if (v < 0) { const char* e = getenv("GPK_PIPE_NB"); v = e ? atoi(e) : 512; if (v < NB || v % NB) v = 512; }   // measured at n = 8192: 384 20.4, 512 19.1, 640 19.5, 768 19.7, 1024 19.3 ms
    return v;
}
int pipe_min() {     // smallest padded N that takes the pipelined driver (0 disables it)
    static int v = -1;
    if (v < 0) { const char* e = getenv("GPK_PIPE_MIN"); v = e ? atoi(e) : 4096; }
    return v;
}

// block-column width of the factor-only driver.  Measured on B200 (profiles/r02_potrf_nb.log): n = 4096: 2.89 / 3.29 ms at
// 256 / 512; n = 8192: 10.47 / 9.04 / 8.90 / 9.14 ms at 128 / 256 / 384 / 512; n = 16384: 52.3 / 49.0 ms at 256 / 512 -- the spine
// (one diagonal block after the other) favours narrow blocks, the bulk GEMMs (K = width) wide ones.  GPK_POTRF_NB overrides.
int potrf_nb_override() {   // GPK_POTRF_NB when it is a valid width, else 0
    static int v = -1;
    if (v < 0) { const char* e = getenv("GPK_POTRF_NB"); v = e ? atoi(e) : 0; if (v < NB || v % NB) v = 0; }
    return v;
}
int potrf_nb(int N) {
    if (const int f = potrf_nb_override()) return f;
    return N <= 4096 ? 256 : (N <= 12288 ? 384 : 512);
}
int potrf_nb_max() { const int f = potrf_nb(1 << 30); return f > 512 ? f : 512; }

void set_batch(GemmDesc& g, const Ctx& c, int64_t sP, int64_t sQ, int64_t sD, int64_t sC) {
    g.batch = c.batch; g.strideP = sP; g.strideQ = sQ; g.strideD = sD; g.strideC = sC;
}

// T (n2 x n1, ld n2) = L21 * Li11 :  C(m,c) = sum_{k>=c} L21(m,k) Li11(k,c)
int gemm_T(const Ctx& c, const double* L21, int64_t sL21, const double* Li11, double* T, int n1, int n2) {
    GemmDesc g = gemm_desc();
    g.P = Li11; g.ldp = c.ld; g.p_kcontig = 1;    // P(r,k) = Li11(k,r)
    g.Q = L21; g.ldq = c.ld; g.q_kcontig = 0;     // Q(s,k) = L21(s,k)
    g.D = T; g.ldd = n2;
    g.R = n1; g.S = n2; g.K = n1; g.kb_r = 1;
    set_batch(g, c, c.sM, sL21, c.sT, 0);
    return gpk_gemm(c.h, g);
}
// Li21 (n2 x n1) = -Li22 * T :  C(m,c) = -sum_{k<=m} Li22(m,k) T(k,c)
int gemm_Li21(const Ctx& c, const double* T, const double* Li22, double* Li21, int n1, int n2) {
    GemmDesc g = gemm_desc();
    g.P = T; g.ldp = n2; g.p_kcontig = 1;         // P(r,k) = T(k,r)
    g.Q = Li22; g.ldq = c.ld; g.q_kcontig = 0;    // Q(s,k) = Li22(s,k)
    g.D = Li21; g.ldd = c.ld;
    g.R = n1; g.S = n2; g.K = n2; g.ke_s = 1; g.alpha = -1.0; g.heavy_last = 1;
    set_batch(g, c, c.sT, c.sM, c.sM, 0);
    return gpk_gemm(c.h, g);
}

// Schedule: everything on the handle's stream except T = L21 * Li11, which is not needed until the very end of the
// node.  For nodes >= side_min() it is forked to a (low-priority) side stream, one per recursion depth, right after
// L21 exists, and joined before Li21 = -Li22 * T.  Each depth has its own T region because a node's T is live across
// its whole second sub-tree.
int potrf_inv_rec(const Ctx& c, double* A, double* Li, double* T, int n, int col_offset, int depth) {
    gpk_handle h = c.h;
    if (n == NB)
        return gpk_base_potrf_trtri(h, A, c.ld, Li, c.ld, c.info, col_offset, 0, c.batch, c.sM, c.sM, 1, 0);
    const int n1 = (n / NB / 2) * NB, n2 = n - n1;
    double* A21 = A + n1;
    double* A22 = A + n1 + (int64_t)n1 * c.ld;
    double* Li21 = Li + n1;
    double* Li22 = Li + n1 + (int64_t)n1 * c.ld;
    double* Tchild = T + (size_t)n1 * n2;
    int rc = potrf_inv_rec(c, A, Li, Tchild, n1, col_offset, depth + 1);
    if (rc) return rc;
    // L21 = A21 * Li11^t, staged in Li21's (still free) slot: C(m,c) = sum_{k<=c} A21(m,k) Li11(c,k)
    GemmDesc g = gemm_desc();
    g.P = Li; g.ldp = c.ld; g.p_kcontig = 0;      // P(r,k) = Li11(r,k)
    g.Q = A21; g.ldq = c.ld; g.q_kcontig = 0;     // Q(s,k) = A21(s,k)
    g.D = Li21; g.ldd = c.ld;
    g.R = n1; g.S = n2; g.K = n1; g.ke_r = 1; g.heavy_last = 1;
    set_batch(g, c, c.sM, c.sM, c.sM, 0);
    rc = gpk_gemm(h, g);
    if (rc) return rc;
    const bool fork = n >= side_min();
    cudaEvent_t ev_done = nullptr;
    if (fork) {
        cudaStream_t side = h->side[(c.side_base + depth) % GPK_NSIDE];
        cudaEvent_t ev_l21 = next_event(h);
        ev_done = next_event(h);
        GPK_CUDA(h, cudaEventRecord(ev_l21, h->stream));
        GPK_CUDA(h, cudaStreamWaitEvent(side, ev_l21, 0));
        {
            StreamSwap sw(h, side);
            rc = gemm_T(c, Li21, c.sM, Li, T, n1, n2);
        }
        if (rc) return rc;
        GPK_CUDA(h, cudaEventRecord(ev_done, side));
    }
    // A22 -= L21 * L21^t (lower tiles)
    g = gemm_desc();
    g.P = Li21; g.ldp = c.ld; g.Q = Li21; g.ldq = c.ld;
    g.D = A22; g.ldd = c.ld; g.Cin = A22; g.ldc = c.ld;
    g.R = n2; g.S = n2; g.K = n1; g.alpha = -1.0; g.beta = 1.0; g.tri_out = 1;
    set_batch(g, c, c.sM, c.sM, c.sM, c.sM);
    rc = gpk_gemm(h, g);
    if (rc) return rc;
    if (c.keep_L) {
        for (int b = 0; b < c.batch && !rc; ++b)
            rc = gpk_copy2d(h, A21 + b * c.sM, c.ld, Li21 + b * c.sM, c.ld, n2, n1);
        if (rc) return rc;
    }
    rc = potrf_inv_rec(c, A22, Li22, Tchild, n2, col_offset + n1, depth + 1);
    if (rc) return rc;
    if (fork) {
        GPK_CUDA(h, cudaStreamWaitEvent(h->stream, ev_done, 0));
    } else {
        rc = gemm_T(c, Li21, c.sM, Li, T, n1, n2);  // L21 is still staged in Li21's slot
        if (rc) return rc;
    }
    // overwrites the staging slot; T has fully consumed it (stream order / ev_done)
    return gemm_Li21(c, T, Li22, Li21, n1, n2);
}

int trtri_rec(const Ctx& c, const double* L, double* Li, double* T, int n) {
    const int n1 = (n / NB / 2) * NB, n2 = n - n1;
    if (n == NB) return GPK_OK;  // diagonal blocks were inverted by one batched launch up front
    int rc = trtri_rec(c, L, Li, T, n1);
    if (rc) return rc;
    rc = trtri_rec(c, L + n1 + (int64_t)n1 * c.ld, Li + n1 + (int64_t)n1 * c.ld, T, n2);
    if (rc) return rc;
    rc = gemm_T(c, L + n1, c.sM, Li, T, n1, n2);
    if (rc) return rc;
    return gemm_Li21(c, T, Li + n1 + (int64_t)n1 * c.ld, Li + n1, n1, n2);
}

size_t rec_scratch_doubles(int N) {
    // sum over recursion depths of n1*n2 <= (N/2+64)^2 * (1 + 1/4 + 1/16 + ...) plus slack for uneven splits
    const size_t half = (size_t)(N / 2 + NB);
    return half * half * 3 / 2 + (size_t)N * NB;
}

// GPK_TRACE=1: timed events at the milestones of the look-ahead drivers, printed (ms since its start) after a device sync.
// Debug aid only (it serialises the call with the host); off by default.
struct Trace {
    struct Mark { cudaEvent_t ev; char what[24]; };
    bool on; cudaEvent_t t0; Mark m[512]; int n;
    Trace() : on(false), t0(nullptr), n(0) { const char* e = getenv("GPK_TRACE"); on = e && atoi(e) > 0; }
    void start(cudaStream_t s) { if (!on) return; cudaEventCreate(&t0); cudaEventRecord(t0, s); }
    void mark(cudaStream_t s, const char* tag, int k) {
        if (!on || n >= 512) return;
        cudaEventCreate(&m[n].ev); cudaEventRecord(m[n].ev, s); snprintf(m[n].what, sizeof(m[n].what), "%s%d", tag, k); ++n;
    }
    void dump() {
        if (!on) return;
        cudaDeviceSynchronize();
        for (int i = 0; i < n; ++i) { float ms = 0; cudaEventElapsedTime(&ms, t0, m[i].ev); fprintf(stderr, "[gpk trace] %-10s %8.3f ms\n", m[i].what, ms); cudaEventDestroy(m[i].ev); }
        cudaEventDestroy(t0);
    }
};

// A[r0.., bj..bj+sj) -= Lst[r0.., bk..) Lst[bj.., bk..)^t with L staged in Li's slots; nrows rows from r0; tri: the block starts
// on the diagonal (r0 == bj) and only its lower tiles are wanted
int stage_update(gpk_handle h, double* A, const double* Li, int N, int bk, int sk, int bj, int sj, int r0, int nrows, int tri) {
    if (nrows <= 0 || sj <= 0) return GPK_OK;
    GemmDesc g = gemm_desc();
    g.P = Li + bj + (int64_t)bk * N; g.ldp = N;
    g.Q = Li + r0 + (int64_t)bk * N; g.ldq = N;
    g.D = A + r0 + (int64_t)bj * N; g.ldd = N; g.Cin = g.D; g.ldc = N;
    g.R = sj; g.S = nrows; g.K = sk; g.alpha = -1.0; g.beta = 1.0; g.tri_out = tri;
    return gpk_gemm(h, g);
}

// rows [r0, r1) of panel k: Lst = A L_kk^-T into Li's slots, then (keep_L) copied back into A
int stage_panel(gpk_handle h, double* A, double* Li, int N, int bk, int sk, int r0, int r1, int keep_L) {
    if (r1 <= r0) return GPK_OK;
    GemmDesc g = gemm_desc();
    g.P = Li + bk + (int64_t)bk * N; g.ldp = N; g.p_kcontig = 0;
    g.Q = A + r0 + (int64_t)bk * N; g.ldq = N; g.q_kcontig = 0;
    g.D = Li + r0 + (int64_t)bk * N; g.ldd = N;
    g.R = sk; g.S = r1 - r0; g.K = sk; g.ke_r = 1; g.heavy_last = 1;
    int rc = gpk_gemm(h, g);
    if (rc || !keep_L) return rc;
    return gpk_copy2d(h, A + r0 + (int64_t)bk * N, N, Li + r0 + (int64_t)bk * N, N, r1 - r0, sk);
}

// ------------------------------------------------------------------------------------------------------------------
// Factor-only look-ahead driver (gpk_potrf_factor / gpk_potrf_factor_solve).  Without the inverse rows and the K^-1
// accumulation of gpk_potrf_inv_pipelined (below) there are only n^3/3 flops of bulk work to hide the serial spine behind,
// so the spine itself is cut to what the NEXT diagonal block needs: per step k the handle's stream runs
//     F_k            L_kk, L_kk^-1                      (recursion on the nb x nb diagonal block)
//     Pc_k           L_{k+1,k} = A_{k+1,k} L_kk^-T      (ONE block row of the panel)
//     Uc_k           A_{k+1,k+1} -= L_{k+1,k} L_{k+1,k}^t   (ONE diagonal block)
// and nothing else; a medium-priority stream S1 solves the rest of the panel (Pr_k) and finishes block column k+1 (Ur_k),
// the low-priority stream S updates block column k+2 first (the next step's Uc / Ur wait for it) and then everything to the
// right of it.  Optional right-hand sides ride along on a fourth stream (forward substitution V = L^-1 B).
// Hazards: every region of A is written by one stream at a time -- Uc_k / Ur_k wait for S's column-first launch of step k-1,
// Pc_{k+1} waits for Ur_k, Pr_{k+1} follows Ur_k in stream order, S's launches are in order.
// ------------------------------------------------------------------------------------------------------------------
int potrf_factor_pipelined(gpk_handle h, double* A, double* Li, double* T, int N, int* info_dev, double* rhsB, double* rhsV,
                           int rhsM, const GpkRowsHook* on_rows = nullptr) {
    // with right-hand sides riding along the gaps of the spine are filled anyway: wider blocks (fewer, longer spine steps) win
    // from N = 4096 on (EP re-factorisation, n = 4096: 5.90 / 5.59 / 5.60 ms at 256 / 384 / 512, profiles/r02_ep_timing.log)
    const int nbk = (rhsB && N >= 4096 && N >= 2 * 512 && !potrf_nb_override()) ? 512 : potrf_nb(N);
    const int nt = (N + nbk - 1) / nbk;
    auto bs = [&](int k) { return k * nbk < N ? k * nbk : N; };
    GPK_CUDA(h, cudaMemsetAsync(info_dev, 0, sizeof(int), h->stream));
    Ctx c{h, N, 1, info_dev, 1, (int64_t)N * N, 0, 0};
    cudaStream_t M = h->stream, S = h->pipe[0], S1 = h->side[GPK_NSIDE - 1], R = h->pipe[1];
    cudaEvent_t ev0 = next_event(h);
    GPK_CUDA(h, cudaEventRecord(ev0, M));
    GPK_CUDA(h, cudaStreamWaitEvent(S, ev0, 0));
    GPK_CUDA(h, cudaStreamWaitEvent(S1, ev0, 0));
    if (rhsB) GPK_CUDA(h, cudaStreamWaitEvent(R, ev0, 0));
    cudaEvent_t evUr_prev = nullptr;                 // S1 finished block column k (rows below block row k) of update k-1
    cudaEvent_t evG_next = nullptr;                  // S's column-first launch of step k-1: block column k+1 has updates <= k-1
    int rc;
    Trace tr;
    tr.start(M);
    for (int k = 0; k < nt; ++k) {
        const int bk = bs(k), sk = bs(k + 1) - bk;
        rc = potrf_inv_rec(c, A + bk + (int64_t)bk * N, Li + bk + (int64_t)bk * N, T, sk, bk, 0);                   // F_k
        if (rc) return rc;
        cudaEvent_t evF = next_event(h);
        GPK_CUDA(h, cudaEventRecord(evF, M));
        tr.mark(M, "M:F", k);
        cudaEvent_t evPc = nullptr, evPr = nullptr, evG_this = nullptr;
        if (k + 1 < nt) {
            const int b1 = bs(k + 1), b2 = bs(k + 2), s1 = b2 - b1;
            if (evUr_prev) GPK_CUDA(h, cudaStreamWaitEvent(M, evUr_prev, 0));
            rc = stage_panel(h, A, Li, N, bk, sk, b1, b2, 1);                                                        // Pc_k
            if (rc) return rc;
            evPc = next_event(h);
            GPK_CUDA(h, cudaEventRecord(evPc, M));
            if (evG_next) GPK_CUDA(h, cudaStreamWaitEvent(M, evG_next, 0));
            tr.mark(M, "M:Pc", k);
            rc = stage_update(h, A, Li, N, bk, sk, b1, s1, b1, s1, 1);                                               // Uc_k
            if (rc) return rc;
            tr.mark(M, "M:Uc", k);
            evUr_prev = nullptr;
            if (k + 2 < nt) {
                {
                    GPK_CUDA(h, cudaStreamWaitEvent(S1, evF, 0));
                    StreamSwap sw(h, S1);
                    rc = stage_panel(h, A, Li, N, bk, sk, b2, N, 1);                                                 // Pr_k
                    if (rc) return rc;
                    evPr = next_event(h);
                    GPK_CUDA(h, cudaEventRecord(evPr, S1));
                    GPK_CUDA(h, cudaStreamWaitEvent(S1, evPc, 0));
                    if (evG_next) GPK_CUDA(h, cudaStreamWaitEvent(S1, evG_next, 0));
                    rc = stage_update(h, A, Li, N, bk, sk, b1, s1, b2, N - b2, 0);                                   // Ur_k
                    if (rc) return rc;
                    evUr_prev = next_event(h);
                    GPK_CUDA(h, cudaEventRecord(evUr_prev, S1));
                    tr.mark(S1, "S1:Ur", k);
                }
                {
                    GPK_CUDA(h, cudaStreamWaitEvent(S, evPc, 0));
                    GPK_CUDA(h, cudaStreamWaitEvent(S, evPr, 0));
                    StreamSwap sw(h, S);
                    const int b3 = bs(k + 3);
                    rc = stage_update(h, A, Li, N, bk, sk, b2, b3 - b2, b2, N - b2, 1);                              // U_k(:, k+2)
                    if (rc) return rc;
                    evG_this = next_event(h);
                    GPK_CUDA(h, cudaEventRecord(evG_this, S));
                    tr.mark(S, "S:G", k);
                    if (k + 3 < nt) {
                        rc = stage_update(h, A, Li, N, bk, sk, b3, N - b3, b3, N - b3, 1);                           // U_k(k+3:, k+3:)
                        if (rc) return rc;
                    }
                    tr.mark(S, "S:bulk", k);
                }
            }
            evG_next = evG_this;
        }
        if (rhsB) {
            // right-hand sides riding along: V_k = L_kk^-1 B_k ;  B_i -= L_ik V_k for i > k
            GPK_CUDA(h, cudaStreamWaitEvent(R, evF, 0));
            StreamSwap swr(h, R);
            GemmDesc g = gemm_desc();
            g.P = rhsB + bk; g.ldp = N; g.p_kcontig = 1;                        // P(r,q) = B(bk+q, r)
            g.Q = Li + bk + (int64_t)bk * N; g.ldq = N; g.q_kcontig = 0;        // Q(s,q) = Li_kk(s,q), zero for q > s
            g.D = rhsV + bk; g.ldd = N; g.R = rhsM; g.S = sk; g.K = sk; g.ke_s = 1; g.heavy_last = 1;
            rc = gpk_gemm(h, g);
            if (rc) return rc;
            if (on_rows) {                                   // rows [bk, bk + sk) of V are final: the caller's consumer may start
                cudaEvent_t evV = next_event(h);
                GPK_CUDA(h, cudaEventRecord(evV, R));
                rc = (*on_rows)(bk, sk, evV);
                if (rc) return rc;
            }
            if (k + 1 < nt) {
                const int b1 = bs(k + 1);
                GPK_CUDA(h, cudaStreamWaitEvent(R, evPc, 0));
                if (evPr) GPK_CUDA(h, cudaStreamWaitEvent(R, evPr, 0));
                g = gemm_desc();
                g.P = rhsV + bk; g.ldp = N; g.p_kcontig = 1;                    // P(r,q) = V(bk+q, r)
                g.Q = Li + b1 + (int64_t)bk * N; g.ldq = N; g.q_kcontig = 0;    // Q(s,q) = L(b1+s, bk+q)
                g.D = rhsB + b1; g.ldd = N; g.Cin = g.D; g.ldc = N;
                g.R = rhsM; g.S = N - b1; g.K = sk; g.alpha = -1.0; g.beta = 1.0;
                rc = gpk_gemm(h, g);
                if (rc) return rc;
            }
        }
    }
    cudaEvent_t e1 = next_event(h), e2 = next_event(h);
    GPK_CUDA(h, cudaEventRecord(e1, S));
    GPK_CUDA(h, cudaStreamWaitEvent(M, e1, 0));
    GPK_CUDA(h, cudaEventRecord(e2, S1));
    GPK_CUDA(h, cudaStreamWaitEvent(M, e2, 0));
    if (rhsB) {
        cudaEvent_t e3 = next_event(h);
        GPK_CUDA(h, cudaEventRecord(e3, R));
        GPK_CUDA(h, cudaStreamWaitEvent(M, e3, 0));
    }
    tr.dump();
    return GPK_OK;
}

}  // namespace

size_t gpk_chol_scratch_doubles(int N) {
    const size_t rec = rec_scratch_doubles(N);
    const size_t pipe = rec_scratch_doubles(pipe_nb()) + (size_t)pipe_nb() * N;   // diagonal-block scratch + one row panel
    const size_t fact = rec_scratch_doubles(potrf_nb_max());
    const size_t m = rec > pipe ? rec : pipe;
    return m > fact ? m : fact;
}

// ------------------------------------------------------------------------------------------------------------------
// Pipelined (look-ahead) driver for one large problem.  The recursion leaves most SMs idle while it walks the bottom of
// the tree (128-blocks: one CTA; 256..1024 nodes: a handful of 64x64 tiles) -- ~7 ms of the 23 ms evaluation at n = 8192
// (profiles/r01_launches_v3_eval.csv).  Here the matrix is cut into block columns of nbk = pipe_nb() (512) and four streams
// run concurrently:
//   M  (the handle's stream, high priority) -- the serial spine: for k = 0..nt-1
//          F_k  L_kk, L_kk^-1 = potrf_inv_rec(A_kk)                       (the recursion, on a 512 block)
//          P_k  L_ik = A_ik L_kk^-T for all i > k, staged in Li's (i,k) slots (free until row i is inverted)
//          U_k(:,k+1)  block column k+1 -= L_:k L_{k+1,k}^T               (look-ahead: F_{k+1} can start at once)
//   S  (low priority) -- the rest of trailing update k: block column k+2 first (M's next look-ahead needs it), then
//          the lower triangle of columns >= k+3 in one SYRK launch;
//   S2 (low priority) -- as soon as F_i is done, row i of the inverse
//          T_i = L_{i,0:i} Li_{0:i,0:i};  Li_{i,0:i} = -Li_ii T_i          (L row i is dead once F_i has run)
//   S3 (low priority, only when K^-1 is wanted) -- as soon as S2 has row i of the inverse, its contribution to
//      K^-1 = Li^t Li (GpPredictor.scala:67):
//          Kinv[i,0:i] = Li_ii^t Li_{i,0:i}; Kinv[i,i] = Li_ii^t Li_ii; Kinv[0:i,0:i] += Li_{i,0:i}^t Li_{i,0:i}.
// Same n^3 flops as the recursive path, same GEMM kernel; only the order changes, so the spine hides behind ~14 ms of
// full-GPU GEMM work.  Hazards are argued in DESIGN.md section 4 (each block column's updates finish before its F).
// ------------------------------------------------------------------------------------------------------------------
int gpk_potrf_inv_pipelined(gpk_handle h, double* A, double* Li, double* Kinv, double* T, int N, int keep_L, int* info_dev,
                            cudaEvent_t* kinv_done) {
    const int nbk = pipe_nb();
    const int nt = (N + nbk - 1) / nbk;
    auto bs = [&](int k) { return k * nbk < N ? k * nbk : N; };
    GPK_CUDA(h, cudaMemsetAsync(info_dev, 0, sizeof(int), h->stream));
    Ctx c{h, N, keep_L, info_dev, 1, (int64_t)N * N, 0, 0};
    double* Tdiag = T;
    double* Trow = T + rec_scratch_doubles(nbk);
    cudaStream_t M = h->stream, S = h->pipe[0], S2 = h->pipe[1], S3 = h->pipe[2];
    cudaEvent_t ev = next_event(h);
    GPK_CUDA(h, cudaEventRecord(ev, M));            // K is built (and earlier users of the buffers are done) before S/S2 start
    GPK_CUDA(h, cudaStreamWaitEvent(S, ev, 0));
    GPK_CUDA(h, cudaStreamWaitEvent(S2, ev, 0));
    if (Kinv) GPK_CUDA(h, cudaStreamWaitEvent(S3, ev, 0));   // (a stream that is forked must also be joined: graph capture insists)
    cudaEvent_t evGcol_prev = nullptr;              // S finished block column k+1 of trailing update k-1
    cudaEvent_t evLi = nullptr;                     // S2 finished the last row of L^-1
    int rc;
    Trace tr;
    tr.start(M);
    for (int k = 0; k < nt; ++k) {
        const int bk = bs(k), sk = bs(k + 1) - bk;
        rc = potrf_inv_rec(c, A + bk + (int64_t)bk * N, Li + bk + (int64_t)bk * N, Tdiag, sk, bk, 0);              // F_k
        if (rc) return rc;
        cudaEvent_t evF = next_event(h);
        GPK_CUDA(h, cudaEventRecord(evF, M));
        tr.mark(M, "M:F", k);
        if (k + 1 < nt) {
            const int b1 = bs(k + 1), s1 = bs(k + 2) - b1;
            rc = stage_panel(h, A, Li, N, bk, sk, b1, N, keep_L);                                                    // P_k
            if (rc) return rc;
            cudaEvent_t evE = next_event(h);
            GPK_CUDA(h, cudaEventRecord(evE, M));
            if (evGcol_prev) GPK_CUDA(h, cudaStreamWaitEvent(M, evGcol_prev, 0));
            tr.mark(M, "M:P", k);
            rc = stage_update(h, A, Li, N, bk, sk, b1, s1, b1, N - b1, 1);                                           // U_k(:,k+1)
            if (rc) return rc;
            tr.mark(M, "M:Ucol", k);
            evGcol_prev = nullptr;
            if (k + 2 < nt) {
                GPK_CUDA(h, cudaStreamWaitEvent(S, evE, 0));
                StreamSwap sw(h, S);
                const int b2 = bs(k + 2), s2 = bs(k + 3) - b2;
                rc = stage_update(h, A, Li, N, bk, sk, b2, s2, b2, N - b2, 1);                                       // U_k(:,k+2)
                if (rc) return rc;
                evGcol_prev = next_event(h);
                GPK_CUDA(h, cudaEventRecord(evGcol_prev, S));
                if (k + 3 < nt) {
                    const int b3 = bs(k + 3);
                    rc = stage_update(h, A, Li, N, bk, sk, b3, N - b3, b3, N - b3, 1);                               // U_k(k+3:, k+3:)
                    if (rc) return rc;
                }
                tr.mark(S, "S:U", k);
            }
        }
        GPK_CUDA(h, cudaStreamWaitEvent(S2, evF, 0));
        StreamSwap sw(h, S2);
        const double* Likk = Li + bk + (int64_t)bk * N;
        if (k > 0) {
            rc = gemm_T(c, Li + bk, 0, Li, Trow, bk, sk);                         // T_k = L_{k,0:k} Li_{0:k,0:k}   (sk x bk, ld sk)
            if (rc) return rc;
            rc = gemm_Li21(c, Trow, Likk, Li + bk, bk, sk);                       // Li_{k,0:k} = -Li_kk T_k
            if (rc) return rc;
        }
        tr.mark(S2, "S2:R", k);
        if (k == nt - 1) {                                                        // L^-1 is complete
            evLi = next_event(h);
            GPK_CUDA(h, cudaEventRecord(evLi, S2));
        }
        if (Kinv) {
            // the K^-1 contribution of row k only needs row k of L^-1: it runs on its own stream so that the row chain on S2
            // (which every later row waits for) is not queued behind these larger GEMMs
            cudaEvent_t evR = next_event(h);
            GPK_CUDA(h, cudaEventRecord(evR, S2));
            GPK_CUDA(h, cudaStreamWaitEvent(S3, evR, 0));
            StreamSwap sw3(h, S3);
            GemmDesc g;
            if (k > 0) {
                g = gemm_desc();                                                  // Kinv[k,0:k] = Li_kk^t Li_{k,0:k}
                g.P = Li + bk; g.ldp = N; g.p_kcontig = 1;                        // P(r,q) = Li(bk+q, r)
                g.Q = Likk; g.ldq = N; g.q_kcontig = 1;                           // Q(s,q) = Li_kk(q, s), zero for q < s
                g.D = Kinv + bk; g.ldd = N; g.R = bk; g.S = sk; g.K = sk; g.kb_s = 1;
                rc = gpk_gemm(h, g);
                if (rc) return rc;
            }
            g = gemm_desc();                                                      // Kinv[k,k] = Li_kk^t Li_kk (lower)
            g.P = Likk; g.ldp = N; g.p_kcontig = 1;
            g.Q = Likk; g.ldq = N; g.q_kcontig = 1;
            g.D = Kinv + bk + (int64_t)bk * N; g.ldd = N; g.R = sk; g.S = sk; g.K = sk; g.kb_r = 1; g.kb_s = 1; g.tri_out = 1;
            rc = gpk_gemm(h, g);
            if (rc) return rc;
            if (k > 0) {
                g = gemm_desc();                                                  // Kinv[0:k,0:k] += Li_{k,0:k}^t Li_{k,0:k} (lower)
                g.P = Li + bk; g.ldp = N; g.p_kcontig = 1;
                g.Q = Li + bk; g.ldq = N; g.q_kcontig = 1;
                g.D = Kinv; g.ldd = N; g.Cin = Kinv; g.ldc = N; g.R = bk; g.S = bk; g.K = sk; g.beta = 1.0; g.tri_out = 1;
                rc = gpk_gemm(h, g);
                if (rc) return rc;
            }
        }
    }
    tr.mark(S3, "S3:Q", nt - 1);
    tr.dump();
    // join: the caller's stream continues once L and L^-1 are complete.  With kinv_done != nullptr the K^-1 accumulation of
    // the last row (the largest) keeps running on S3 and the caller waits for *kinv_done only where it reads K^-1, so
    // alpha = L^-t L^-1 y and the log-likelihood overlap it.
    cudaEvent_t e1 = next_event(h), e2 = next_event(h);
    GPK_CUDA(h, cudaEventRecord(e1, S));
    GPK_CUDA(h, cudaStreamWaitEvent(M, e1, 0));
    GPK_CUDA(h, cudaEventRecord(e2, Kinv ? S3 : S2));   // no K^-1 requested: S3 was never forked, join the row chain
    if (kinv_done && Kinv) {
        GPK_CUDA(h, cudaStreamWaitEvent(M, evLi, 0));
        *kinv_done = e2;
    } else {
        GPK_CUDA(h, cudaStreamWaitEvent(M, e2, 0));
        if (kinv_done) *kinv_done = nullptr;
    }
    return GPK_OK;
}

// Factor only (LAPACK dpotrf 'L': GpPredictor.scala:120, EpParameterEstimator.scala:58 when the caller wants nothing but L): the
// look-ahead driver without the inverse rows and the K^-1 accumulation -- n^3/3 flops instead of n^3.  Only the diagonal
// blocks are inverted (the panels are solved as GEMMs with them).  Li is still an N x N staging area.
int gpk_potrf_factor(gpk_handle h, double* A, double* Li, double* T, int N, int* info_dev) {
    if (N >= 2 * potrf_nb(N)) return potrf_factor_pipelined(h, A, Li, T, N, info_dev, nullptr, nullptr, 0);
    return gpk_potrf_inv(h, A, Li, T, N, 1, info_dev, 1);
}

// Factor + multi-right-hand-side forward solve: A -> L (in place), V = L^-1 B for B, V: N x M (ld N, M a multiple of 128); B is
// destroyed.  EP's posterior re-factorisation (EpParameterEstimator.scala:58-59: cholesky, then forwardSolve with n right-hand
// sides) is this call.  Large N: the look-ahead driver with the right-hand sides riding along (no L^-1 is ever formed:
// n^3/3 + n^2 M flops); small N: L^-1 by the recursion and one GEMM.
int gpk_potrf_factor_solve(gpk_handle h, double* A, double* Li, double* T, int N, int* info_dev, double* B, double* V, int M,
                           const GpkRowsHook* on_rows) {
    if (N >= 2 * potrf_nb(N))
        return potrf_factor_pipelined(h, A, Li, T, N, info_dev, B, V, M, on_rows);
    int rc = gpk_potrf_inv(h, A, Li, T, N, 1, info_dev, 1);
    if (rc) return rc;
    rc = gpk_trmm_lower(h, Li, N, B, V, M);
    if (rc || !on_rows) return rc;
    cudaEvent_t evV = next_event(h);                                // all rows at once
    GPK_CUDA(h, cudaEventRecord(evV, h->stream));
    return (*on_rows)(0, N, evV);
}

bool gpk_use_pipelined(int N, int batch) { return batch == 1 && pipe_min() > 0 && N >= pipe_min() && N >= 2 * pipe_nb(); }

int gpk_potrf_inv(gpk_handle h, double* A, double* Li, double* T, int N, int keep_L, int* info_dev, int batch, bool lookahead) {
    if (lookahead && gpk_use_pipelined(N, batch)) return gpk_potrf_inv_pipelined(h, A, Li, nullptr, T, N, keep_L, info_dev, nullptr);
    GPK_CUDA(h, cudaMemsetAsync(info_dev, 0, sizeof(int) * (size_t)batch, h->stream));
    const int64_t sM = (int64_t)N * N, sT = (int64_t)gpk_chol_scratch_doubles(N);
    if (batch < 8) {
        Ctx c{h, N, keep_L, info_dev, batch, sM, sT, 0};
        return potrf_inv_rec(c, A, Li, T, N, 0, 0);
    }
    // Batch groups: from 8 problems on the batch is cut in two halves that walk the recursion on two streams.  The base-case
    // launches (one CTA per problem, latency-bound, ~40 us each, 8 per factorisation at n = 1024) and the partial last waves of
    // the small GEMMs of one half are filled by the other half's launches.  Measured on B200 (profiles/r02_c4_groups.log),
    // n = 1024: 64 problems 3.53 / 3.42 / 3.74 ms and 512 problems 24.33 / 23.94 / 24.02 ms with 1 / 2 / 4 groups.
    // Group 1 (problems [b1, batch), on grp[0], side streams from 4) is enqueued first; group 0 (problems [0, b1)) runs on
    // the handle's own stream, whose launches need no join.
    const int b1 = (batch + 1) / 2;
    cudaEvent_t ev0 = next_event(h);
    GPK_CUDA(h, cudaEventRecord(ev0, h->stream));
    GPK_CUDA(h, cudaStreamWaitEvent(h->grp[0], ev0, 0));
    int rc;
    {
        StreamSwap sw(h, h->grp[0]);
        Ctx c{h, N, keep_L, info_dev + b1, batch - b1, sM, sT, 4};
        rc = potrf_inv_rec(c, A + b1 * sM, Li + b1 * sM, T + b1 * sT, N, 0, 0);
    }
    if (rc) return rc;
    cudaEvent_t done = next_event(h);
    GPK_CUDA(h, cudaEventRecord(done, h->grp[0]));
    Ctx c{h, N, keep_L, info_dev, b1, sM, sT, 0};
    rc = potrf_inv_rec(c, A, Li, T, N, 0, 0);
    if (rc) return rc;
    GPK_CUDA(h, cudaStreamWaitEvent(h->stream, done, 0));
    return GPK_OK;
}

int gpk_trtri_lower(gpk_handle h, const double* L, double* Li, double* T, int N) {
    // const_cast: mode 1 never writes A.  One launch inverts all N/128 diagonal blocks.
    int rc = gpk_base_potrf_trtri(h, const_cast<double*>(L), N, Li, N, h->d_info, 0, 1, N / NB, (int64_t)NB * (N + 1),
                                  (int64_t)NB * (N + 1), 0, NB);
    if (rc) return rc;
    Ctx c{h, N, 0, h->d_info, 1, (int64_t)N * N, (int64_t)gpk_chol_scratch_doubles(N), 0};
    return trtri_rec(c, L, Li, T, N);
}

int gpk_lauum_lower(gpk_handle h, const double* Li, double* Kinv, int N, int batch) {
    // Kinv(m,c) = sum_{k >= max(m,c)} Li(k,m) Li(k,c), lower tiles (m >= c)
    GemmDesc g = gemm_desc();
    g.P = Li; g.ldp = N; g.p_kcontig = 1;  // P(r,k) = Li(k,r)
    g.Q = Li; g.ldq = N; g.q_kcontig = 1;  // Q(s,k) = Li(k,s)
    g.D = Kinv; g.ldd = N;
    g.R = N; g.S = N; g.K = N; g.kb_r = 1; g.kb_s = 1; g.tri_out = 1;
    g.batch = batch; g.strideP = g.strideQ = g.strideD = (int64_t)N * N;
    return gpk_gemm(h, g);
}

int gpk_trmm_lower(gpk_handle h, const double* Li, int N, const double* B, double* V, int M, int batch) {
    // V(m,c) = sum_{k <= m} Li(m,k) B(k,c)
    GemmDesc g = gemm_desc();
    g.P = B; g.ldp = N; g.p_kcontig = 1;   // P(r,k) = B(k,r)
    g.Q = Li; g.ldq = N; g.q_kcontig = 0;  // Q(s,k) = Li(s,k)
    g.D = V; g.ldd = N;
    g.R = M; g.S = N; g.K = N; g.ke_s = 1; g.heavy_last = 1;
    g.batch = batch; g.strideP = g.strideD = (int64_t)N * M; g.strideQ = (int64_t)N * N;
    return gpk_gemm(h, g);
}
