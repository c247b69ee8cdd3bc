"""GPU tests of the batched EP evaluation (gpk_ep_nll_grad_batched, ep_classification.log_likelihood_batched): every problem of a
batch must give what one gpk_ep_nll_grad call gives on it (same sweep count, logZ / gradient / tau / nu to 1e-9), bit for bit the
same whatever else shares the call, and stop at its own sweep."""
import ctypes as C
import os
import subprocess
import sys

import numpy as np
import pytest

import gp_algos_b200 as gp
from gp_algos_b200 import _lib
from oracle import gp_oracle as orc

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
RTOL = 1e-9


def close(a, b, rtol=RTOL):
    a, b = np.asarray(a), np.asarray(b)
    return np.all(np.abs(a - b) <= rtol * np.maximum(np.abs(b), np.abs(b).max() * 1e-6))


def _stop(stop):
    if isinstance(stop, gp.FixedSweeps):
        return 0.0, stop.sweeps, stop.sweeps
    return stop.eps, 0, stop.max_sweeps


def batched_raw(X, t, thetas, stop, nparams=None, outputs=True, h=None):
    """gpk_ep_nll_grad_batched through ctypes with every output.  X: (n, D) or (B, n, D); t: (n,) or (B, n)."""
    h = h or _lib.default_handle()
    thetas = np.ascontiguousarray(thetas, dtype=np.float64)
    B, P = thetas.shape
    X = np.asarray(X, dtype=np.float64)
    n, D = X.shape[-2:]
    Xb = np.asfortranarray(X) if X.ndim == 2 else np.ascontiguousarray(np.transpose(X, (0, 2, 1)))
    t = np.ascontiguousarray(t, dtype=np.int32)
    nparams = P if nparams is None else nparams
    eps, fixed, mx = _stop(stop)
    logz = np.empty(B); grad = np.zeros((B, max(nparams, 1))); tau = np.empty((B, n)); nu = np.empty((B, n))
    sw = np.zeros(B, dtype=np.int32); info = np.zeros(B, dtype=np.int32)
    o = _lib.ptr if outputs else (lambda a: None)
    rc = h.lib.gpk_ep_nll_grad_batched(h.h, B, _lib.ptr(Xb), n, D, n, 0 if X.ndim == 2 else n * D, _lib.ptr(thetas), _lib.ptr(t),
                                       0 if t.ndim == 1 else n, eps, fixed, mx, 1, nparams, _lib.ptr(logz), _lib.ptr(grad),
                                       o(tau), o(nu), _lib.ptr(sw), o(info))
    h.check(rc)
    return dict(logZ=logz, grad=grad[:, :nparams], tau=tau, nu=nu, sweeps=sw, info=info)


def single(X, t, theta, stop, nparams=None, h=None):
    """one gpk_ep_nll_grad call"""
    h = h or _lib.default_handle()
    X = np.asfortranarray(X, dtype=np.float64); t = np.ascontiguousarray(t, dtype=np.int32)
    theta = np.ascontiguousarray(theta, dtype=np.float64)
    n, D = X.shape
    nparams = len(theta) if nparams is None else nparams
    eps, fixed, mx = _stop(stop)
    grad = np.zeros(max(nparams, 1)); tau = np.empty(n); nu = np.empty(n)
    logz = C.c_double(); sw = C.c_int()
    h.check(h.lib.gpk_ep_nll_grad(h.h, _lib.ptr(X), n, D, n, _lib.ptr(theta), t.ctypes.data_as(C.c_void_p), eps, fixed, mx, 1,
                                  nparams, C.addressof(logz), _lib.ptr(grad), _lib.ptr(tau), _lib.ptr(nu), C.addressof(sw)))
    return dict(logZ=logz.value, grad=grad[:nparams], tau=tau, nu=nu, sweeps=sw.value)


def thetas_of(pairs, D=4, sn=0.1):
    return np.stack([orc.pack_theta(sf, [ls] * D, sn) for sf, ls in pairs])


# (signalVar, lengthScale) per size.  With eps = 0.01 the CPU oracle's avgBetweenSiteParams passes eps by at least a factor 1.5
# on either side of every stop (sweep counts in the comments), so no criterion is borderline.
THETAS = {65: [(1.0, 0.7), (1.0, 1.5), (4.0, 1.5)],           # 4, 5, 5 sweeps
          130: [(0.5, 1.5), (2.0, 0.7), (4.0, 1.5)],          # 5, 6, 6
          300: [(0.5, 0.7), (1.0, 0.7), (1.0, 1.5)],          # 5, 6, 7
          1000: [(0.5, 0.7), (1.0, 1.5), (2.0, 0.7)]}
EPS = gp.AvgBasedStopCriterion(0.01)


def data(n, D=4):
    return orc.make_c3(n=n, D=D, seed=100 + n)[:2]


@pytest.mark.parametrize("n", [65, 130, 300, 1000])     # last blocks of 1, 2, 44 and 40 sites
def test_parity_with_single_calls(n):
    X, t = data(n)
    th = thetas_of(THETAS[n])
    got = batched_raw(X, t, th, EPS)
    assert np.all(got["info"] == 0)
    for b in range(len(th)):
        want = single(X, t, th[b], EPS)
        assert got["sweeps"][b] == want["sweeps"]
        assert abs(got["logZ"][b] - want["logZ"]) <= RTOL * abs(want["logZ"])
        assert close(got["grad"][b], want["grad"])
        assert close(got["tau"][b], want["tau"]) and close(got["nu"][b], want["nu"])
        if n <= 130:
            lz_o, g_o, o = orc.lit_ep_loglik_with_derivs(X, t, th[b], eps=0.01)
            assert got["sweeps"][b] == o["sweeps"]
            assert abs(got["logZ"][b] - lz_o) <= RTOL * abs(lz_o)
            assert close(got["grad"][b], g_o)
            assert close(got["tau"][b], o["tau"]) and close(got["nu"][b], o["nu"])


def test_batch_invariance():
    """A problem's outputs do not depend on what else shares the call or on its position (one group of batched launches below
    eight problems, two from eight on)."""
    n = 300
    X, t = data(n)
    rng = np.random.default_rng(7)
    th = thetas_of([(10 ** rng.uniform(-0.3, 0.5), 10 ** rng.uniform(-0.2, 0.2)) for _ in range(9)])
    alone = batched_raw(X, t, th[3:4], EPS)
    seven = batched_raw(X, t, th[:7], EPS)
    nine_rev = batched_raw(X, t, th[::-1], EPS)                        # problem 3 at position 5 of 9
    for got, pos in ((seven, 3), (nine_rev, 5)):
        for k in ("logZ", "grad", "tau", "nu", "sweeps"):
            assert np.array_equal(got[k][pos], alone[k][0]), k
    for k in ("logZ", "grad", "tau", "nu", "sweeps"):
        assert np.array_equal(seven[k], nine_rev[k][::-1][:7]), k


def test_each_problem_stops_at_its_own_sweep():
    n = 300
    X, t = data(n)
    th = thetas_of(THETAS[n])
    got = batched_raw(X, t, th, EPS)
    want = [single(X, t, th[b], EPS)["sweeps"] for b in range(len(th))]
    assert list(got["sweeps"]) == want
    assert len(set(want)) >= 2
    capped = gp.AvgBasedStopCriterion(0.01, max_sweeps=6)
    got = batched_raw(X, t, th, capped)
    assert list(got["sweeps"]) == [min(s, 6) for s in want]
    for b in range(len(th)):
        s = single(X, t, th[b], capped)
        assert got["sweeps"][b] == s["sweeps"]
        assert abs(got["logZ"][b] - s["logZ"]) <= RTOL * abs(s["logZ"])
    fixed = batched_raw(X, t, th, gp.FixedSweeps(2))
    assert list(fixed["sweeps"]) == [2] * len(th)


def test_inputs_per_problem_shared_and_optional_outputs():
    n, B = 200, 4
    sets = [orc.make_c3(n=n, D=3, seed=40 + b)[:2] for b in range(B)]
    Xs = np.stack([s[0] for s in sets]); ts = np.stack([s[1] for s in sets])
    th = thetas_of([(1.0, 0.8), (2.0, 1.2), (0.7, 1.0), (1.5, 0.6)], D=3)
    stop = gp.FixedSweeps(3)
    for X, t in ((Xs, ts), (Xs, ts[0]), (Xs[0], ts)):                  # strideX, strideT non-zero / zero
        got = batched_raw(X, t, th, stop)
        for b in range(B):
            want = single(X if X.ndim == 2 else X[b], t if t.ndim == 1 else t[b], th[b], stop)
            assert abs(got["logZ"][b] - want["logZ"]) <= RTOL * abs(want["logZ"])
            assert close(got["grad"][b], want["grad"]) and close(got["tau"][b], want["tau"])
    full = batched_raw(Xs, ts, th, stop)
    none = batched_raw(Xs, ts, th, stop, nparams=0, outputs=False)     # no gradient; tau, nu, info NULL
    assert np.array_equal(none["logZ"], full["logZ"]) and np.array_equal(none["sweeps"], full["sweeps"])
    two = batched_raw(Xs, ts, th, stop, nparams=2)
    assert np.array_equal(two["grad"], full["grad"][:, :2])
    logz, grad, sweeps, info = gp.log_likelihood_batched(Xs, ts, th, stop)
    assert np.array_equal(logz, full["logZ"]) and np.array_equal(grad, full["grad"]) and np.all(info == 0)


# GPK_BATCH_GB = 0.032 GiB holds at most four problems of n = 300 (N = 384): the six N x N matrices of a slot of EpBatch
# (csrc/gpk_ep.cu) alone are 6.75 MiB, so the 9 problems run in at least three chunks.
CHUNK_ENV = {"GPK_BATCH_GB": "0.032"}


def _chunk_results(path):
    """Runs in the child and in the parent."""
    from tests.test_gpu_ep_batched import batched_raw, data, EPS
    rng = np.random.default_rng(11)
    th = np.stack([orc.pack_theta(10 ** rng.uniform(-0.3, 0.5), [10 ** rng.uniform(-0.2, 0.2)] * 4, 0.1) for _ in range(9)])
    X, t = data(300)
    h = _lib.default_handle()
    l0 = h.launch_count()
    r = batched_raw(X, t, th, EPS)
    np.savez(path, launches=h.launch_count() - l0, **r)


def test_chunked_batch_equals_one_chunk(tmp_path):
    code = ("import sys; sys.path.insert(0, sys.argv[1]); from tests.test_gpu_ep_batched import _chunk_results; "
            "_chunk_results(sys.argv[2])")
    r = subprocess.run([sys.executable, "-c", code, ROOT, str(tmp_path / "chunked.npz")], env=dict(os.environ, **CHUNK_ENV),
                       capture_output=True, text=True, timeout=600)
    assert r.returncode == 0, f"child with {CHUNK_ENV} failed:\n{r.stderr[-4000:]}"
    _chunk_results(tmp_path / "whole.npz")
    got, want = np.load(tmp_path / "chunked.npz"), np.load(tmp_path / "whole.npz")
    assert got["launches"] > want["launches"], "GPK_BATCH_GB did not split the batch"
    assert np.all(want["info"] == 0)
    for k in ("logZ", "grad", "tau", "nu", "sweeps", "info"):
        assert np.array_equal(got[k], want[k]), f"{k}: chunked run differs from the one-chunk run"


def test_argument_errors_before_any_launch():
    h = _lib.default_handle()
    n, D, B = 64, 2, 2
    X = np.asfortranarray(np.random.default_rng(0).standard_normal((n, D))); t = np.ones(n, dtype=np.int32)
    th = np.ascontiguousarray(thetas_of([(1.0, 1.0)] * B, D=D))
    out = np.empty(B); g = np.empty(B * (D + 2)); sw = np.zeros(B, dtype=np.int32)
    p = _lib.ptr

    def call(B=B, Xp=p(X), n=n, D=D, ldx=n, sX=0, thp=p(th), tp=p(t), sT=0, nparams=D + 2, lz=p(out), gp_=p(g), swp=p(sw)):
        return h.lib.gpk_ep_nll_grad_batched(h.h, B, Xp, n, D, ldx, sX, thp, tp, sT, 0.01, 0, 10, 1, nparams, lz, gp_, None, None,
                                             swp, None)

    l0 = h.launch_count()
    bad = [dict(B=0), dict(n=0), dict(ldx=n - 1), dict(D=0), dict(D=65), dict(nparams=D + 3), dict(nparams=-1),
           dict(Xp=None), dict(thp=None), dict(tp=None), dict(lz=None), dict(gp_=None), dict(swp=None), dict(sX=-1), dict(sT=-1),
           dict(sX=n * D - 1), dict(sT=n - 1)]
    for kw in bad:
        assert call(**kw) == _lib.GPK_EINVAL, kw
    assert h.launch_count() == l0
    assert call(nparams=0, gp_=None) == _lib.GPK_OK          # no gradient: grad may be NULL


def test_multistart_never_ends_below_its_start():
    n = 200
    X, t = orc.make_c3(n=n, D=2, seed=77)[:2]
    init = thetas_of([(0.5, 0.5), (1.0, 1.0), (3.0, 2.0)], D=2)
    stop = gp.AvgBasedStopCriterion(0.01)
    pts, vals = gp.obtain_optimal_ep_hyper_params_multistart(X, t, init, stop, maxIter=4)
    assert pts.shape == init.shape and np.all(np.isfinite(vals))
    for r in range(len(init)):
        start, end = single(X, t, init[r], stop)["logZ"], single(X, t, pts[r], stop)["logZ"]
        assert end >= start - 1e-9 * abs(start)
        assert abs(end - vals[r]) <= 1e-9 * abs(vals[r])
