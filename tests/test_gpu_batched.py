"""GPU parity for the batched independent-GP entry points (BASELINE.json config 4) through the C ABI."""
import os
import subprocess
import sys

import numpy as np
import pytest

import gp_algos_b200 as gp
from gp_algos_b200 import batched
from oracle import gp_oracle as orc

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
G = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")
RTOL = 1e-9


def _grad_ok(g, go):
    floor = RTOL * np.abs(go).max()
    return np.all(np.abs(g - go) <= RTOL * np.maximum(np.abs(go), floor))


def test_golden_c4_small_batched():
    g = np.load(os.path.join(G, "c4_small.npz"))
    B = int(g["B"])
    X = np.stack([g[f"X{b}"] for b in range(B)]); ys = np.stack([g[f"y{b}"] for b in range(B)])
    th = np.stack([g[f"theta{b}"] for b in range(B)]); Xs = np.stack([g[f"Xs{b}"] for b in range(B)])
    ll, grad, info = batched.log_likelihood_with_derivatives_batched(X, ys, th)
    assert np.all(info == 0)
    for b in range(B):
        assert abs(ll[b] - float(g[f"ll{b}"])) <= RTOL * abs(float(g[f"ll{b}"]))
        assert _grad_ok(grad[b], g[f"grad{b}"])
    mean, var, ll2, info = batched.predict_batched(X, ys, th, Xs)
    assert np.all(info == 0)
    for b in range(B):
        assert np.all(np.abs(mean[b] - g[f"mean{b}"]) <= RTOL * np.abs(g[f"mean{b}"]).max())
        assert np.all(np.abs(var[b] - g[f"var{b}"]) <= RTOL * np.abs(g[f"var{b}"]))
        assert abs(ll2[b] - float(g[f"ll{b}"])) <= RTOL * abs(float(g[f"ll{b}"]))


def test_batched_equals_single_calls_and_shared_x():
    """GP-UKF flavour: one X shared by every output dimension (GPUnscentedKalmanFilter.scala:123-136)."""
    B, n, D, m = 5, 300, 4, 9
    rng = np.random.default_rng(4)
    X = rng.uniform(0, 1, size=(n, D)); Xs = rng.uniform(0, 1, size=(m, D))
    ys = np.stack([np.sin(X @ rng.standard_normal(D)) + 0.1 * rng.standard_normal(n) for _ in range(B)])
    th = np.stack([orc.pack_theta(10 ** rng.uniform(-0.3, 0.3), 10 ** rng.uniform(-0.5, 0.2, size=D), 0.1) for _ in range(B)])
    ll, grad, info = batched.log_likelihood_with_derivatives_batched(X, ys, th)
    mean, var, ll2, _ = batched.predict_batched(X, ys, th, Xs)
    for b in range(B):
        p = gp.GpPredictor(gp.GaussianRbfKernel(gp.GaussianRbfParams(th[b, 0], th[b, 1:-1], th[b, -1])))
        l1, g1 = p.logLikelihoodWithDerivatives(gp.PredictionTrainingInput(X, None, ys[b]), th[b], D + 2)
        assert l1 == ll[b] and np.array_equal(g1, grad[b])           # same kernels, same order: bit-identical
        llo, go = orc.lit_loglik_with_derivs(X, ys[b], th[b])
        assert abs(ll[b] - llo) <= RTOL * abs(llo) and _grad_ok(grad[b], go)
        Lo, ao = orc.lit_precompute(X, ys[b], th[b])
        mo, So, _ = orc.lit_compute_posterior(X, Xs, Lo, ao, th[b])
        assert np.all(np.abs(mean[b] - mo) <= RTOL * np.abs(mo).max())
        assert np.all(np.abs(var[b] - np.diag(So)) <= RTOL * np.abs(np.diag(So)))
    # partitioning the batch (what each GPU rank does) does not change any result
    lo, hi = batched.shard_bounds(B, 1, 2)
    ll_s, grad_s, _ = batched.log_likelihood_with_derivatives_batched(X, ys[lo:hi], th[lo:hi])
    assert np.array_equal(ll_s, ll[lo:hi]) and np.array_equal(grad_s, grad[lo:hi])


def test_batched_failure_is_isolated_per_problem():
    B, n, D = 4, 200, 2
    rng = np.random.default_rng(9)
    X = np.stack([rng.uniform(0, 1, size=(n, D)) for _ in range(B)])
    X[2, 50] = X[2, 10]                                   # duplicate point in problem 2 ...
    ys = rng.standard_normal((B, n))
    th = np.tile(orc.pack_theta(1.0, [0.5, 0.5], 0.1), (B, 1))
    th[2, -1] = 0.0                                        # ... with zero noise: K_2 is singular
    ll, grad, info = batched.log_likelihood_with_derivatives_batched(X, ys, th)
    assert info[2] != 0 and np.all(info[[0, 1, 3]] == 0)
    for b in (0, 1, 3):
        llo, go = orc.lit_loglik_with_derivs(X[b], ys[b], th[b])
        assert abs(ll[b] - llo) <= RTOL * abs(llo) and _grad_ok(grad[b], go)


def test_c4_shape_subset_full_n():
    """Problems of the real C4 shape (n = 1024, D = 8, m = 17), a 24-problem subset against the LAPACK-backed oracle."""
    B = 24
    probs = [orc.make_c4_problem(b) for b in range(B)]
    X = np.stack([p[0] for p in probs]); ys = np.stack([p[1] for p in probs])
    Xs = np.stack([p[2] for p in probs]); th = np.stack([p[3] for p in probs])
    ll, grad, info = batched.log_likelihood_with_derivatives_batched(X, ys, th)
    mean, var, _, _ = batched.predict_batched(X, ys, th, Xs)
    assert np.all(info == 0)
    for b in range(0, B, 5):
        llo, go = orc.fast_loglik_with_derivs(X[b], ys[b], th[b])
        assert abs(ll[b] - llo) <= RTOL * abs(llo) and _grad_ok(grad[b], go)
        Lo, ao = orc.fast_precompute(X[b], ys[b], th[b])
        mo, vo, _ = orc.fast_compute_posterior(X[b], Xs[b], Lo, ao, th[b], full_cov=False)
        assert np.all(np.abs(mean[b] - mo) <= RTOL * np.abs(mo).max())
        assert np.all(np.abs(var[b] - vo) <= RTOL * np.abs(vo))


def test_c4_config_full_size_sampled_parity_and_partition_invariance():
    """BASELINE.json config 4 at full size (512 problems of n = 1024, D = 8): three sampled problems against the LAPACK-backed
    oracle, every problem finite, and the size-independent property that any partition of the batch gives identical results."""
    B = 512
    probs = [orc.make_c4_problem(b) for b in range(B)]
    X = np.stack([p[0] for p in probs]); ys = np.stack([p[1] for p in probs]); th = np.stack([p[3] for p in probs])
    ll, grad, info = batched.log_likelihood_with_derivatives_batched(X, ys, th)
    assert np.all(info == 0) and np.all(np.isfinite(ll)) and np.all(np.isfinite(grad))
    for b in (0, 255, 511):
        llo, go = orc.fast_loglik_with_derivs(X[b], ys[b], th[b])
        assert abs(ll[b] - llo) <= RTOL * abs(llo)
        assert _grad_ok(grad[b], go)
    lo, hi = batched.shard_bounds(B, 5, 8)                                   # the shard rank 5 of 8 would evaluate
    ll_s, grad_s, _ = batched.log_likelihood_with_derivatives_batched(X[lo:hi], ys[lo:hi], th[lo:hi])
    assert np.array_equal(ll_s, ll[lo:hi]) and np.array_equal(grad_s, grad[lo:hi])


def test_multistart_hyperparameter_fit_in_lockstep():
    """batched.obtain_optimal_hyper_params_multistart: R restarts of GpPredictor.obtainOptimalHyperParams (GpPredictor.scala:126-142)
    advanced in lockstep, one batched objective call per round.  Every returned (theta, ll) is a point of the single-problem
    objective and not worse than its start."""
    X, y, th = orc.make_c2(n=300, D=3, seed=21)
    rng = np.random.default_rng(3)
    starts = th * 10 ** rng.uniform(-0.3, 0.3, size=(5, th.size))
    thetas, lls = batched.obtain_optimal_hyper_params_multistart(X, y, starts, maxIter=8)
    assert thetas.shape == starts.shape and lls.shape == (5,)
    for r in range(5):
        ll_r, _ = orc.fast_loglik_with_derivs(X, y, thetas[r], None, 0)
        ll_0, _ = orc.fast_loglik_with_derivs(X, y, starts[r], None, 0)
        assert abs(ll_r - lls[r]) <= 1e-9 * abs(ll_r) and lls[r] >= ll_0 - 1e-9 * abs(ll_0)
    # against R sequential single-start fits (GpPredictor.obtainOptimalHyperParams, GpPredictor.scala:126-142): the lockstep
    # optimiser is not Breeze's (Armijo backtracking, its own stop rule), so only the outcome is compared: given enough
    # iterations the best restart reaches the best sequential fit's likelihood to 0.1 %
    thetas, lls = batched.obtain_optimal_hyper_params_multistart(X, y, starts, maxIter=40)
    import gp_algos_b200 as gp
    best_seq = -np.inf
    for r in range(5):
        kf = gp.GaussianRbfKernel(gp.GaussianRbfParams(starts[r][0], starts[r][1:-1], starts[r][-1]))
        pred = gp.GpPredictor(kf)
        hp = pred.obtainOptimalHyperParams(X, None, y, True)
        best_seq = max(best_seq, pred.logLikelihoodWithDerivatives(gp.PredictionTrainingInput(X, None, y), hp, 0)[0])
    assert lls.max() >= best_seq - 1e-3 * abs(best_seq)


def test_multistart_restart_that_is_never_positive_definite_reports_minus_infinity():
    X, y, th = orc.make_c2(n=200, D=3, seed=22)
    X[1] = X[0]                                                   # duplicate row + zero noise: K is singular at this start
    bad = th.copy(); bad[-1] = 0.0
    thetas, lls = batched.obtain_optimal_hyper_params_multistart(X, y, np.stack([th, bad]), maxIter=3)
    assert np.isfinite(lls[0]) and lls[1] == -np.inf and np.array_equal(thetas[1], bad)


def test_full_batch_is_bit_reproducible_over_many_runs():
    """512 x (n = 1024) through two concurrent batch groups, 25 times: every run must reproduce the first bit for bit.  Guards
    the 128-block base kernel against read/write races that only show when kernels of two streams run side by side -- round 1
    had one (the panel's diagonal block was read from the rows their owner threads overwrite): about one run in seven came back
    with ONE problem's log-likelihood and gradient off by 1e-4 .. 1e-1, invisible to tests that compare a few problems."""
    import torch
    from gp_algos_b200 import _lib
    B, n, D = 512, 1024, 8
    probs = [orc.make_c4_problem(b) for b in range(B)]
    X = np.stack([p[0] for p in probs]); ys = np.stack([p[1] for p in probs]); th = np.ascontiguousarray(np.stack([p[3] for p in probs]))
    h = _lib.default_handle()
    dX = torch.from_numpy(np.ascontiguousarray(np.transpose(X, (0, 2, 1)))).cuda(); dy = torch.from_numpy(ys).cuda()
    out = torch.zeros(B * (D + 3), dtype=torch.float64, device="cuda"); info = torch.zeros(B, dtype=torch.int32, device="cuda")
    first = None
    for rep in range(25):
        h.check(h.lib.gpk_gp_nll_grad_batched_dev(h.h, B, dX.data_ptr(), n, D, n, n * D, dy.data_ptr(), _lib.ptr(th), 0, 0.0, D + 2,
                                                  out.data_ptr(), info.data_ptr()))
        h.synchronize()
        res = out.cpu().numpy().copy()
        assert int(info.abs().sum().item()) == 0
        if first is None:
            first = res
        else:
            assert np.array_equal(res, first), f"run {rep} differs from run 0 in problems {np.unique(np.argwhere(res != first) // (D + 3))[:5]}"


# GPK_BATCH_GB = 0.032 GiB holds 5 problems of n = 300 (N = 384, D = 4): about 5.95 MiB each (L, L^-1, the Cholesky scratch and
# the vectors of make_work, csrc/gpk_gp.cu), so the 19 problems run in chunks of 5, 5, 5 and 4.  n stays far below 4096, where a
# chunk of one problem would take the look-ahead driver.
CHUNK_ENV = {"GPK_BATCH_GB": "0.032"}


def _chunk_results(path):
    """Runs in the child and in the parent: both batched entry points on 19 problems with their own X and X*."""
    from gp_algos_b200 import _lib
    B, n, D, m = 19, 300, 4, 9
    rng = np.random.default_rng(31)
    X = rng.uniform(0, 1, size=(B, n, D)); Xs = rng.uniform(0, 1, size=(B, m, D))
    ys = np.stack([np.sin(X[b] @ rng.standard_normal(D)) + 0.1 * rng.standard_normal(n) for b in range(B)])
    th = np.stack([orc.pack_theta(10 ** rng.uniform(-0.3, 0.3), 10 ** rng.uniform(-0.5, 0.2, size=D), 0.1) for _ in range(B)])
    h = _lib.default_handle()
    l0 = h.launch_count()
    mean, var, ll, info = batched.predict_batched(X, ys, th, Xs)
    launches = h.launch_count() - l0
    ll_g, grad, info_g = batched.log_likelihood_with_derivatives_batched(X, ys, th)
    np.savez(path, mean=mean, var=var, ll=ll, info=info, ll_g=ll_g, grad=grad, info_g=info_g, launches=launches)


def test_chunked_batch_equals_one_chunk(tmp_path):
    """A batch larger than GPK_BATCH_GB runs chunk by chunk.  The budget is read once per process, so the chunked run is a child.
    Every problem is computed on its own, so the chunks must reproduce the one-chunk run bit for bit."""
    code = ("import sys; sys.path.insert(0, sys.argv[1]); from tests.test_gpu_batched import _chunk_results; "
            "_chunk_results(sys.argv[2])")
    r = subprocess.run([sys.executable, "-c", code, ROOT, str(tmp_path / "chunked.npz")], env=dict(os.environ, **CHUNK_ENV),
                       capture_output=True, text=True, timeout=600)
    assert r.returncode == 0, f"child with {CHUNK_ENV} failed:\n{r.stderr[-4000:]}"
    _chunk_results(tmp_path / "whole.npz")
    got, want = np.load(tmp_path / "chunked.npz"), np.load(tmp_path / "whole.npz")
    assert got["launches"] > want["launches"], "GPK_BATCH_GB did not split the batch"
    assert np.all(want["info"] == 0) and np.all(want["info_g"] == 0)
    for k in ("mean", "var", "ll", "info", "ll_g", "grad", "info_g"):
        assert np.array_equal(got[k], want[k]), f"{k}: chunked run differs from the one-chunk run"
