"""GPU parity (through the C ABI) for the MatrixUtils-level entry points.  Mirrors the reference's
src/test/scala/utils/MatrixUtilsTest.scala and widens it with ragged sizes and error behaviour."""
import os

import numpy as np
import pytest

import gp_algos_b200 as gp
from gp_algos_b200 import MatrixUtils as MU
from oracle import gp_oracle as orc

pytestmark = pytest.mark.gpu
G = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")
EPS = 0.001  # MatrixUtilsTest.scala:22


def _kernel(th):
    return gp.GaussianRbfKernel(gp.GaussianRbfParams(th[0], th[1:-1], th[-1]))


def ulp_close(a, b, k=4):
    return np.all(np.abs(a - b) <= k * np.spacing(np.maximum(np.abs(a), np.abs(b))))


# ---- the reference's own test cases (3x3) ------------------------------------------------------------
def test_reference_3x3_solves_and_golden():
    g = np.load(os.path.join(G, "mu_3x3.npz"))
    x = MU.forwardSolve(g["lower"], g["rhs_l"])
    assert np.all(np.abs(x - g["np_fwd_vec"]) < EPS) and np.allclose(x, g["fwd_vec"], rtol=1e-12)
    x = MU.backSolve(g["upper"], g["rhs_u"])
    assert np.all(np.abs(x - g["np_back_vec"]) < EPS) and np.allclose(x, g["back_vec"], rtol=1e-12)
    Xm = MU.forwardSolve(g["lower"], g["rhs_m"])
    assert Xm.shape == (3, 2) and np.allclose(Xm, g["fwd_mat"], rtol=1e-12)
    Xm = MU.backSolve(g["upper"], g["rhs_m"])
    assert Xm.shape == (3, 2) and np.allclose(Xm, g["back_mat"], rtol=1e-12)


def test_reference_3x3_kernel_matrix_unit_diagonal_and_cholesky():
    g = np.load(os.path.join(G, "mu_3x3.npz"))
    K = MU.buildKernelMatrix(_kernel(g["theta"]), g["input"])
    assert K.shape == (3, 3)
    assert all(K[i, i] == 1.0 for i in range(3))        # MatrixUtilsTest.scala:99 (exact)
    assert ulp_close(K, g["K"])
    L = MU.cholesky(K)                                   # MatrixUtilsTest.scala:100 "does not throw"
    assert np.allclose(L, g["L"], rtol=1e-12, atol=1e-15)
    Li = MU.invTriangular(L, isUpper=False)              # MatrixUtilsTest.scala:104-114
    assert np.all(np.abs(Li.T @ Li - g["Kinv_np"]) < EPS)
    assert np.allclose(Li, g["Linv"], rtol=1e-11, atol=1e-14)


# ---- covariance: ragged sizes, ARD, exact symmetry -----------------------------------------------------
@pytest.mark.parametrize("n,D", [(1, 1), (2, 3), (63, 2), (64, 8), (65, 8), (129, 5), (257, 1), (1000, 1), (1030, 17), (2048, 8)])
def test_cov_matches_oracle(n, D):
    rng = np.random.default_rng(n * 31 + D)
    X = rng.standard_normal((n, D)) * 3.0 + 50.0  # un-normalised features: direct-difference form must hold up
    th = orc.pack_theta(1.7, rng.uniform(0.5, 3.0, size=D), 0.3)
    K = MU.buildKernelMatrix(_kernel(th), X)
    Ko = orc.lit_build_kernel_matrix(X, th) if n <= 300 else orc.fast_build_kernel_matrix(X, th)
    assert K.shape == (n, n)
    assert np.array_equal(K, K.T)                        # lower-loop-and-mirror => exactly symmetric
    assert ulp_close(K, Ko, 4)
    assert np.array_equal(np.diag(K), np.full(n, 1.7 * 1.7 * 1.0 + 0.3 * 0.3))
    m = min(n, 37)
    Xs = rng.standard_normal((m, D)) * 3.0 + 50.0
    Kc = MU.buildKernelMatrix(_kernel(th), Xs, X)        # MatrixUtils.scala:44-55: m x n, never noise
    assert Kc.shape == (m, n)
    assert ulp_close(Kc, orc.fast_build_kernel_matrix(Xs, th, X), 4)
    Kc2 = MU.buildKernelMatrix(_kernel(th), X[:m], X)
    assert np.all(np.abs(np.diag(Kc2[:, :m]) - 1.7 * 1.7) < 1e-15)  # sameIndex=false even for identical points


def test_cov_deriv_matrices():
    rng = np.random.default_rng(5)
    X = rng.uniform(0, 1, size=(150, 4))
    th = orc.pack_theta(1.2, rng.uniform(0.4, 1.0, size=4), 0.25)
    for p in range(1, 7):
        dK = MU.buildKernelDerMatrix(_kernel(th), X, p)
        dKo = orc.lit_build_der_matrix(p, X, th)
        assert np.allclose(dK, dKo, rtol=1e-14, atol=1e-300), p
    with pytest.raises(LookupError):  # scala.MatchError
        MU.buildKernelDerMatrix(_kernel(th), X, 7)


# ---- cholesky ------------------------------------------------------------------------------------------
@pytest.mark.parametrize("n", [1, 2, 127, 128, 129, 255, 384, 640, 1000, 1500, 4300])   # 4300 -> N = 4352: pipelined driver with keep_L
def test_cholesky_backward_error_and_parity(n):
    import scipy.linalg as sla
    X, y, th = orc.make_c2(n=n, D=8, seed=n)
    K = orc.fast_build_kernel_matrix(X, th)
    L = MU.cholesky(K)
    assert np.all(np.triu(L, 1) == 0.0)                  # strict upper zeroed like breeze cholesky
    eps = np.finfo(np.float64).eps
    assert np.linalg.norm(L @ L.T - K) <= 8 * n * eps * np.linalg.norm(K)   # SURVEY.md 8(d) gate
    Lo = sla.cholesky(K, lower=True)
    cond = np.linalg.cond(K)
    assert np.linalg.norm(L - Lo) <= 1e-9 * max(cond / 1e5, 1.0) * np.linalg.norm(Lo)
    if n <= 384:
        assert np.allclose(L, orc.lit_cholesky(K), rtol=1e-9, atol=1e-13)


def test_cholesky_error_behaviour():
    with pytest.raises(gp.MatrixNotSymmetricError):
        MU.cholesky(np.array([[1., 2.], [3., 4.]]))
    with pytest.raises(gp.NotPositiveDefiniteError) as e:
        MU.cholesky(np.array([[1., 2.], [2., 1.]]))
    assert e.value.minor == 2                            # same failing minor as LAPACK info
    A = np.eye(300); A[200, 200] = -1.0
    with pytest.raises(gp.NotPositiveDefiniteError) as e:
        MU.cholesky(A)
    assert e.value.minor == 201
    assert np.allclose(MU.cholesky(np.eye(5) * 4.0), np.eye(5) * 2.0)  # handle stays usable after an error
    # same through the look-ahead (pipelined) driver, which takes over at padded N >= 4096: the failing minor sits in
    # the 6th block column and every stream must drain cleanly
    B = np.eye(4500); B[2900, 2900] = -3.0
    with pytest.raises(gp.NotPositiveDefiniteError) as e:
        MU.cholesky(B)
    assert e.value.minor == 2901
    assert np.allclose(MU.cholesky(np.eye(4200) * 9.0), np.eye(4200) * 3.0)


# ---- triangular solves / inverse -------------------------------------------------------------------------
@pytest.mark.parametrize("n,m", [(5, 1), (130, 3), (300, 140), (777, 17)])
def test_triangular_solves_match_oracle(n, m):
    import scipy.linalg as sla
    rng = np.random.default_rng(n)
    X, y, th = orc.make_c2(n=n, D=8, seed=n + 1)
    L = sla.cholesky(orc.fast_build_kernel_matrix(X, th), lower=True)
    b = rng.standard_normal(n); B = rng.standard_normal((n, m))
    ref = orc.lit_forward_solve if n <= 300 else (lambda T, r, trans=False: sla.solve_triangular(T, r, lower=True))
    assert np.allclose(MU.forwardSolve(L, b), ref(L, b), rtol=1e-9, atol=1e-12)
    assert np.allclose(MU.forwardSolve(L, B), ref(L, B), rtol=1e-9, atol=1e-12)
    # backSolve(R = L.t, b) -- GpPredictor.scala:122
    xb = MU.backSolve(L, b, transposed=True)
    xo = orc.lit_back_solve(L, b, trans=True) if n <= 300 else sla.solve_triangular(L, b, lower=True, trans="T")
    assert np.allclose(xb, xo, rtol=1e-9, atol=1e-12)
    U = np.ascontiguousarray(L.T)
    assert np.allclose(MU.backSolve(U, B), sla.solve_triangular(U, B, lower=False), rtol=1e-9, atol=1e-12)
    assert np.allclose(MU.forwardSolve(U, b, transposed=True), sla.solve_triangular(L, b, lower=True), rtol=1e-9, atol=1e-12)
    # a row-major operand is passed as the column-major storage of its transpose (no host re-striding): same bits either way
    Lf, Lc = np.asfortranarray(L), np.ascontiguousarray(L)
    assert np.array_equal(MU.forwardSolve(Lf, B), MU.forwardSolve(Lc, B))
    assert np.array_equal(MU.backSolve(Lf, b, transposed=True), MU.backSolve(Lc, b, transposed=True))


@pytest.mark.parametrize("n", [4, 128, 200, 515])
def test_inv_triangular(n):
    import scipy.linalg as sla
    X, y, th = orc.make_c2(n=n, D=8, seed=n + 7)
    L = sla.cholesky(orc.fast_build_kernel_matrix(X, th), lower=True)
    Li = MU.invTriangular(L, isUpper=False)
    assert np.all(np.triu(Li, 1) == 0.0)
    ref = orc.lit_inv_triangular(L) if n <= 200 else np.linalg.inv(L)
    assert np.allclose(Li, ref, rtol=1e-9, atol=1e-12)
    Ui = MU.invTriangular(np.ascontiguousarray(L.T), isUpper=True)
    assert np.all(np.tril(Ui, -1) == 0.0)
    assert np.allclose(Ui, ref.T, rtol=1e-9, atol=1e-12)


# ---- device-resident factor-only Cholesky (gpk_potrf_lower_dev) and large solves ---------------------------
@pytest.mark.parametrize("n,lda", [(1024, 1024), (1000, 1100), (2304, 2304), (130, 130)])
def test_potrf_lower_dev_in_place(n, lda):
    import scipy.linalg as sla
    import torch
    from gp_algos_b200 import _lib
    X, y, th = orc.make_c2(n=n, D=8, seed=n + 3)
    K = orc.fast_build_kernel_matrix(X, th)
    buf = np.full((n, lda), 7.0)                        # column-major n x n block inside an lda-strided buffer: buf[c, r]
    buf[:, :n] = K.T
    d = torch.from_numpy(buf.reshape(-1).copy()).cuda()
    info = torch.zeros(1, dtype=torch.int32, device="cuda")
    h = _lib.default_handle()
    h.check(h.lib.gpk_potrf_lower_dev(h.h, d.data_ptr(), n, lda, info.data_ptr()))
    h.synchronize()
    assert int(info.item()) == 0
    out = d.cpu().numpy().reshape(n, lda)
    L = out[:, :n].T
    assert np.all(np.triu(L, 1) == 0.0)
    assert np.all(out[:, n:] == 7.0)                     # nothing outside the n x n block is touched
    Lo = sla.cholesky(K, lower=True)
    assert np.linalg.norm(L @ L.T - K) <= 8 * n * np.finfo(float).eps * np.linalg.norm(K)
    assert np.linalg.norm(L - Lo) <= 1e-9 * max(np.linalg.cond(K) / 1e5, 1.0) * np.linalg.norm(Lo)
    assert np.array_equal(L, MU.cholesky(K))             # host and device entry points run the same kernels
    # not positive definite: the failing leading minor arrives in *info_dev
    Kb = K.copy(); Kb[n // 2, n // 2] = -1.0
    buf[:, :n] = Kb.T
    d = torch.from_numpy(buf.reshape(-1).copy()).cuda()
    h.check(h.lib.gpk_potrf_lower_dev(h.h, d.data_ptr(), n, lda, info.data_ptr()))
    h.synchronize()
    assert int(info.item()) == n // 2 + 1


@pytest.mark.parametrize("n,m", [(2500, 1), (2500, 2), (1300, 129)])
def test_triangular_solves_blocked_substitution_large(n, m):
    """The blocked O(n^2)-per-right-hand-side substitution at sizes with many diagonal blocks, vector and matrix paths."""
    import scipy.linalg as sla
    rng = np.random.default_rng(n + m)
    X, y, th = orc.make_c2(n=n, D=8, seed=n + 11)
    L = sla.cholesky(orc.fast_build_kernel_matrix(X, th), lower=True)
    B = rng.standard_normal((n, m)) if m > 1 else rng.standard_normal(n)
    for got, want in ((MU.forwardSolve(L, B), sla.solve_triangular(L, B, lower=True)),
                      (MU.backSolve(L, B, transposed=True), sla.solve_triangular(L, B, lower=True, trans="T")),
                      (MU.backSolve(np.ascontiguousarray(L.T), B), sla.solve_triangular(L, B, lower=True, trans="T"))):
        assert got.shape == want.shape
        assert np.allclose(got, want, rtol=1e-9, atol=1e-9 * np.abs(want).max())


@pytest.mark.parametrize("n,lda", [(2048, 2048), (1500, 1504)])
def test_potrf_lower_dev_graph_replay(n, lda):
    """The same buffers factored again: eager first, captured into a CUDA graph at the second call, replayed afterwards
    (N <= 4096) -- the three must agree bit for bit, and a not-positive-definite input must still report its leading minor."""
    import torch
    from gp_algos_b200 import _lib
    X, y, th = orc.make_c2(n=n, D=8, seed=n + 17)
    K = orc.fast_build_kernel_matrix(X, th)
    buf = np.zeros((n, lda)); buf[:, :n] = K.T
    src = torch.from_numpy(buf.reshape(-1).copy()).cuda()
    d = torch.empty_like(src)
    info = torch.zeros(1, dtype=torch.int32, device="cuda")
    h = _lib.Handle(0, torch.cuda.current_stream().cuda_stream)
    outs = []
    for rep in range(4):
        d.copy_(src)
        h.check(h.lib.gpk_potrf_lower_dev(h.h, d.data_ptr(), n, lda, info.data_ptr()))
        h.synchronize()
        assert int(info.item()) == 0
        outs.append(d.cpu().numpy().copy())
    for o in outs[1:]:
        assert np.array_equal(o, outs[0])
    L = outs[0].reshape(n, lda)[:, :n].T
    assert np.linalg.norm(L @ L.T - K) <= 8 * n * np.finfo(float).eps * np.linalg.norm(K)
    Kb = K.copy(); Kb[n // 3, n // 3] = -1.0
    buf[:, :n] = Kb.T
    d.copy_(torch.from_numpy(buf.reshape(-1).copy()).cuda())
    h.check(h.lib.gpk_potrf_lower_dev(h.h, d.data_ptr(), n, lda, info.data_ptr()))      # replayed graph, other data
    h.synchronize()
    assert int(info.item()) == n // 3 + 1
