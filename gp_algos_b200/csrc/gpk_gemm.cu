// gpk_gemm.cu -- FP64 tensor-core (DMMA.8x8x4) tile GEMM used by every O(n^3) step of the path:
// Cholesky trailing update (SYRK), L21 = A21 L11^-T, the blocked triangular inverse, K^-1 = L^-T L^-1
// (reference: GpPredictor.scala:66-67,120; EpParameterEstimator.scala:58-60) and the predictive
// V = L^-1 K*^t (GpPredictor.scala:34,55).
//
// sm_100a has no tcgen05 kind for f64 (ptxas rejects .kind::f64), so the FP64 tensor path is the
// warp-level mma.sync.m8n8k4.f64 -> SASS DMMA.8x8x4.  Measured on B200 (profiles/r01_fp64_microbench.txt):
// DMMA and DFMA both peak at 37.1 TFLOP/s; DMMA needs 4x fewer shared-memory operand bytes per flop, which is what lets
// a small CTA tile run pipe-bound.
//
// One layout (SmallTile): 64 x 64 x 16 CTA tile, 128 threads = 4 warps as 2 (r) x 2 (s), each warp owning a 32 x 32
// sub-tile = 4 x 4 DMMA accumulators; 3 CTAs per SM (60 KB of shared memory each), which beat every larger tile shape
// (profiles/r01_tile_configs.txt).  Operands are staged global -> shared with 16-byte cp.async (LDGSTS) through a 3-stage
// ring; shared rows are padded by 4 doubles so that the 8-byte fragment reads of a half-warp (4 k x 4 rows) hit 16 distinct
// bank pairs.  The main loop carries running global pointers and cycling stage counters and issues the next refill behind
// the first DMMA group of each k-step.  Measured: 32.5 TFLOP/s on the SYRK of n = k = 4096 (91.7 % of cuBLAS Dgemm), DMMA
// pipe 95 % of active cycles (profiles/r01_ncu_summary_v3.txt).
#include "gpk_internal.cuh"

namespace {

constexpr int TK = 16;
constexpr int LDK = TK + 4;  // row stride (doubles) of a [x][k] stage   (k-contiguous source)
constexpr int GROUP_S = 8;   // raster: blocks walk bands of 8 s-tiles so a wave shares operand panels in L2

__device__ __forceinline__ void cp_async16(double* smem, const double* gmem) {
    unsigned s = (unsigned)__cvta_generic_to_shared(smem);
    asm volatile("cp.async.cg.shared.global [%0], [%1], 16;\n" ::"r"(s), "l"(gmem));
}
__device__ __forceinline__ void cp_async_commit() { asm volatile("cp.async.commit_group;\n" ::); }
template <int N>
__device__ __forceinline__ void cp_async_wait() {
    asm volatile("cp.async.wait_group %0;\n" ::"n"(N));
}
__device__ __forceinline__ void dmma(double& c0, double& c1, double a, double b) {
    asm("mma.sync.aligned.m8n8k4.row.col.f64.f64.f64.f64 {%0,%1}, {%2}, {%3}, {%0,%1};\n"
        : "+d"(c0), "+d"(c1)
        : "d"(a), "d"(b));
}

// Tile configuration: WR x WS warps, each owning a (BI*8) x (BJ*8) sub-tile.
template <int WR_, int WS_, int BI_, int BJ_, int STAGES_, int MINB_>
struct TileCfg {
    static constexpr int WR = WR_, WS = WS_, BI = BI_, BJ = BJ_, STAGES = STAGES_;
    static constexpr int TR = WR * BI * 8, TS = WS * BJ * 8, NT = 32 * WR * WS;
    static constexpr int LDRP = TR + 4, LDRQ = TS + 4;  // row stride of a [k][x] stage (x-contiguous source), %16 == 4
    static constexpr int P_STAGE = (TR * LDK > TK * LDRP) ? TR * LDK : TK * LDRP;
    static constexpr int Q_STAGE = (TS * LDK > TK * LDRQ) ? TS * LDK : TK * LDRQ;
    static constexpr size_t SMEM = (size_t)STAGES * (P_STAGE + Q_STAGE) * sizeof(double);
    static constexpr int MIN_BLOCKS = MINB_;
};
using SmallTile = TileCfg<2, 2, 4, 4, 3, 3>;   // 3 stages x 20 KB = 60 KB -> 3 CTAs (12 warps) per SM

// One CTA tile: acc += sum over nk k-chunks (of TK) starting at kbeg of P(r0.., k) Q(s0.., k).  Called by every thread of the
// CTA; returns with all cp.async groups drained (a caller that reuses the shared-memory ring needs a barrier first).
template <bool PK, bool QK, class Cfg>
__device__ __forceinline__ void tile_mainloop(const GemmDesc& g, const double* __restrict__ P, const double* __restrict__ Q, int r0,
                                              int s0, int kbeg, int nk, double* smem, double (&acc)[Cfg::BI][Cfg::BJ][2]) {
    constexpr int TR = Cfg::TR, TS = Cfg::TS, NT = Cfg::NT, BI = Cfg::BI, BJ = Cfg::BJ;
    constexpr int LDRP = Cfg::LDRP, LDRQ = Cfg::LDRQ, STAGES = Cfg::STAGES;
    const int tid = threadIdx.x;
    double* Ps = smem;
    double* Qs = smem + STAGES * Cfg::P_STAGE;
    const int warp = tid >> 5, lane = tid & 31;
    const int gid = lane >> 2, tig = lane & 3;
    const int wr0 = (warp / Cfg::WS) * (BI * 8), ws0 = (warp % Cfg::WS) * (BJ * 8);

    // Per-thread copy descriptors: running global pointers (advanced by one k-chunk per issue) and fixed offsets inside a
    // stage, so the steady-state loop carries no 64-bit address arithmetic and no `% STAGES`.
    constexpr int PPT = TR * TK / 2 / NT, QPT = TS * TK / 2 / NT;
    const double* pg[PPT];
    const double* qg[QPT];
    int pso[PPT], qso[QPT];
#pragma unroll
    for (int i = 0; i < PPT; ++i) {
        const int c = tid + i * NT;
        if (!PK) { const int k = c / (TR / 2), x = (c % (TR / 2)) * 2; pso[i] = k * LDRP + x; pg[i] = P + (int64_t)(kbeg + k) * g.ldp + (r0 + x); }
        else     { const int x = c >> 3, k = (c & 7) * 2;              pso[i] = x * LDK + k;  pg[i] = P + (int64_t)(r0 + x) * g.ldp + (kbeg + k); }
    }
#pragma unroll
    for (int i = 0; i < QPT; ++i) {
        const int c = tid + i * NT;
        if (!QK) { const int k = c / (TS / 2), x = (c % (TS / 2)) * 2; qso[i] = k * LDRQ + x; qg[i] = Q + (int64_t)(kbeg + k) * g.ldq + (s0 + x); }
        else     { const int x = c >> 3, k = (c & 7) * 2;              qso[i] = x * LDK + k;  qg[i] = Q + (int64_t)(s0 + x) * g.ldq + (kbeg + k); }
    }
    const int64_t pstep = PK ? (int64_t)TK : (int64_t)TK * g.ldp;
    const int64_t qstep = QK ? (int64_t)TK : (int64_t)TK * g.ldq;
    auto issue = [&](int stage) {
        double* pst = Ps + stage * Cfg::P_STAGE;
        double* qst = Qs + stage * Cfg::Q_STAGE;
#pragma unroll
        for (int i = 0; i < PPT; ++i) { cp_async16(pst + pso[i], pg[i]); pg[i] += pstep; }
#pragma unroll
        for (int i = 0; i < QPT; ++i) { cp_async16(qst + qso[i], qg[i]); qg[i] += qstep; }
    };

#pragma unroll
    for (int s = 0; s < STAGES - 1; ++s) {
        if (s < nk) issue(s);
        cp_async_commit();
    }

    int cstage = 0, lstage = STAGES - 1;   // stage computed on / stage loaded into, both cycle through 0..STAGES-1
    for (int kc = 0; kc < nk; ++kc) {
        cp_async_wait<STAGES - 2>();
        __syncthreads();
        const double* ps = Ps + cstage * Cfg::P_STAGE;
        const double* qs = Qs + cstage * Cfg::Q_STAGE;
        const double* pf = PK ? ps + (wr0 + gid) * LDK + tig : ps + tig * LDRP + wr0 + gid;
        const double* qf = QK ? qs + (ws0 + gid) * LDK + tig : qs + tig * LDRQ + ws0 + gid;
#pragma unroll
        for (int kk = 0; kk < TK; kk += 4) {
            double a[BI], bb[BJ];
#pragma unroll
            for (int i = 0; i < BI; ++i) a[i] = PK ? pf[i * 8 * LDK + kk] : pf[kk * LDRP + i * 8];
#pragma unroll
            for (int j = 0; j < BJ; ++j) bb[j] = QK ? qf[j * 8 * LDK + kk] : qf[kk * LDRQ + j * 8];
#pragma unroll
            for (int i = 0; i < BI; ++i)
#pragma unroll
                for (int j = 0; j < BJ; ++j) dmma(acc[i][j][0], acc[i][j][1], a[i], bb[j]);
            if (kk == 0) {
                // refill the stage that was consumed in the previous iteration (every warp is past the barrier above, so
                // nobody reads it any more); issued behind the first DMMA group so the copies overlap the math
                if (kc + STAGES - 1 < nk) issue(lstage);
                cp_async_commit();
            }
        }
        cstage = (cstage + 1 == STAGES) ? 0 : cstage + 1;
        lstage = (lstage + 1 == STAGES) ? 0 : lstage + 1;
    }
    cp_async_wait<0>();
}

// D tile = alpha acc + beta Cin
template <class Cfg>
__device__ __forceinline__ void tile_epilogue(const GemmDesc& g, double* __restrict__ D, const double* Cin, int r0, int s0,
                                              const double (&acc)[Cfg::BI][Cfg::BJ][2]) {
    constexpr int BI = Cfg::BI, BJ = Cfg::BJ;
    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
    const int gid = lane >> 2, tig = lane & 3;
    const int wr0 = (warp / Cfg::WS) * (BI * 8), ws0 = (warp % Cfg::WS) * (BJ * 8);
    const double alpha = g.alpha, beta = g.beta;
#pragma unroll
    for (int i = 0; i < BI; ++i) {
        const int64_t r = r0 + wr0 + 8 * i + gid;
#pragma unroll
        for (int j = 0; j < BJ; ++j) {
            const int s = s0 + ws0 + 8 * j + 2 * tig;
            double2 v = make_double2(alpha * acc[i][j][0], alpha * acc[i][j][1]);
            if (Cin != nullptr) {
                const double2 c = *reinterpret_cast<const double2*>(Cin + r * g.ldc + s);
                v.x += beta * c.x;
                v.y += beta * c.y;
            }
            *reinterpret_cast<double2*>(D + r * g.ldd + s) = v;
        }
    }
}

template <bool PK, bool QK, class Cfg>
__global__ void __launch_bounds__(Cfg::NT, Cfg::MIN_BLOCKS) gemm_f64_dmma_kernel(const GemmDesc g) {
    constexpr int TR = Cfg::TR, TS = Cfg::TS, BI = Cfg::BI, BJ = Cfg::BJ;
    extern __shared__ __align__(16) double smem[];
    const int tilesS = g.S / TS, tilesR = g.R / TR;
    int bid = blockIdx.x;
    if (g.heavy_last) bid = gridDim.x - 1 - bid;
    const int group = bid / (GROUP_S * tilesR);
    const int first_s = group * GROUP_S;
    const int gs = min(GROUP_S, tilesS - first_s);
    const int within = bid - group * GROUP_S * tilesR;
    const int tr = within / gs, ts = first_s + within % gs;
    const int r0 = tr * TR, s0 = ts * TS;
    if (g.tri_out && s0 + TS <= r0) return;
    int kbeg = 0, kend = g.K;
    if (g.kb_r) kbeg = max(kbeg, r0);
    if (g.kb_s) kbeg = max(kbeg, s0);
    if (g.ke_r) kend = min(kend, r0 + TR);
    if (g.ke_s) kend = min(kend, s0 + TS);
    const int nk = (kend - kbeg) / TK;

    const int64_t b = blockIdx.y;
    const double* __restrict__ P = g.P + b * g.strideP;
    const double* __restrict__ Q = g.Q + b * g.strideQ;
    double* __restrict__ D = g.D + b * g.strideD;
    const double* Cin = g.Cin ? g.Cin + b * g.strideC : nullptr;

    double acc[BI][BJ][2];
#pragma unroll
    for (int i = 0; i < BI; ++i)
#pragma unroll
        for (int j = 0; j < BJ; ++j) acc[i][j][0] = acc[i][j][1] = 0.0;
    tile_mainloop<PK, QK, Cfg>(g, P, Q, r0, s0, kbeg, nk, smem, acc);
    tile_epilogue<Cfg>(g, D, Cin, r0, s0, acc);
}

template <bool PK, bool QK, class Cfg>
int launch(gpk_handle h, const GemmDesc& g) {
    const unsigned bit = 1u << (12 + (PK ? 2 : 0) + (QK ? 1 : 0));
    if (!(h->func_cfg & bit)) {
        GPK_CUDA(h, cudaFuncSetAttribute(gemm_f64_dmma_kernel<PK, QK, Cfg>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                         (int)Cfg::SMEM));
        h->func_cfg |= bit;
    }
    dim3 grid((unsigned)((g.R / Cfg::TR) * (g.S / Cfg::TS)), (unsigned)g.batch);
    gemm_f64_dmma_kernel<PK, QK, Cfg><<<grid, Cfg::NT, Cfg::SMEM, h->stream>>>(g);
    GPK_LAUNCH_CHECK(h);
    return GPK_OK;
}

template <class Cfg>
int dispatch(gpk_handle h, const GemmDesc& g) {
    if (g.p_kcontig) return g.q_kcontig ? launch<true, true, Cfg>(h, g) : launch<true, false, Cfg>(h, g);
    return g.q_kcontig ? launch<false, true, Cfg>(h, g) : launch<false, false, Cfg>(h, g);
}

}  // namespace

int gpk_gemm(gpk_handle h, const GemmDesc& g) {
    if (g.R <= 0 || g.S <= 0 || g.batch <= 0) return GPK_OK;
    if (g.R % 64 || g.S % 64 || g.K % TK || (g.ldp & 1) || (g.ldq & 1) || (g.ldd & 1) ||
        ((uintptr_t)g.P & 15) || ((uintptr_t)g.Q & 15) || ((uintptr_t)g.D & 15) || (g.Cin && (((uintptr_t)g.Cin & 15) || (g.ldc & 1))))
        return gpk_set_error(h, GPK_EINVAL, "gpk_gemm: unaligned problem R=%d S=%d K=%d", g.R, g.S, g.K);
    return dispatch<SmallTile>(h, g);
}

extern "C" int gpk_debug_gemm(gpk_handle h, const double* P, int64_t ldp, int64_t strideP, const double* Q, int64_t ldq,
                              int64_t strideQ, double* D, int64_t ldd, int64_t strideD, const double* Cin, int64_t ldc,
                              int64_t strideC, int R, int S, int K, int batch, double alpha, double beta, int p_kcontig,
                              int q_kcontig, int flags) {
    if (!h) return GPK_EINVAL;
    if (flags & ~0x3f) return gpk_set_error(h, GPK_EINVAL, "gpk_debug_gemm: unknown flag bits 0x%x", flags);
    GemmDesc g = gemm_desc();
    g.P = P; g.ldp = ldp; g.strideP = strideP;
    g.Q = Q; g.ldq = ldq; g.strideQ = strideQ;
    g.D = D; g.ldd = ldd; g.strideD = strideD;
    g.Cin = Cin; g.ldc = ldc; g.strideC = strideC;
    g.R = R; g.S = S; g.K = K; g.batch = batch; g.alpha = alpha; g.beta = beta;
    g.p_kcontig = p_kcontig != 0; g.q_kcontig = q_kcontig != 0;
    g.tri_out = (flags & GPK_GEMM_TRI_OUT) != 0;
    g.kb_r = (flags & GPK_GEMM_KB_R) != 0;
    g.kb_s = (flags & GPK_GEMM_KB_S) != 0;
    g.ke_r = (flags & GPK_GEMM_KE_R) != 0;
    g.ke_s = (flags & GPK_GEMM_KE_S) != 0;
    g.heavy_last = (flags & GPK_GEMM_HEAVY_LAST) != 0;
    return gpk_gemm(h, g);
}
