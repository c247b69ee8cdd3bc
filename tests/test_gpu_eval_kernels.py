"""GPU: the kernels of the evaluation besides the factorisation, one routine at a time, against plain high-precision
references (tests/eval_refs.py, NumPy longdouble; never the oracle), plus the device-resident entry points against their host
counterparts.

- covariance build (csrc/gpk_cov.cu, gpk_debug_cov): SE-ARD values within 3 ulp of sf^2 exp(-r/2) with r in float64 in the
  kernel's unfused association; the mode contracts (SYM_FULL symmetric with an exact diagonal, LOWER_PAD's whole diagonal
  128-blocks and identity padding, CROSS's zero fill) with sentinels where nothing may be written and NaN padding rows of X
  that must not be read; batches with per-problem theta equal to single calls bit for bit; the Co2 family and both
  families' derivative matrices against the true derivatives;
- gradient trace (csrc/gpk_grad.cu, gpk_debug_grad_trace): against 1/2 sum_ij W_ij dk_p over the full square, with NaN in the
  strictly upper triangle of K^-1, beyond n and in alpha's padding, within a rounding bound derived from the reduction depth;
- vector kernels (csrc/gpk_vec.cu): trmv / trmv^t / colwise_dot exact on small integers, NaN wherever they must not read;
  loglik against longdouble;
- gpk_gp_nll_grad_dev / _batched_dev / gpk_cov_*_dev with ldx > n against the host entry points bit for bit.
"""
import contextlib
import math

import numpy as np
import pytest

from oracle import gp_oracle as orc
from tests import eval_refs as R

pytestmark = pytest.mark.gpu

U = 2.0 ** -53
LD = np.longdouble
SENT = -777.25                      # sentinel: elements a routine must not write
NAN = float("nan")
SYM_FULL, LOWER_PAD, CROSS = 0, 1, 2
KERNEL_CO2 = 1


@pytest.fixture(scope="module")
def h():
    from gp_algos_b200 import _lib
    hd = _lib.Handle(0)
    yield hd
    hd.close()


def _dev(a):
    import torch
    return torch.from_numpy(np.ascontiguousarray(a)).cuda()


def _host(t):
    return t.cpu().numpy()


def _run(h, fn):
    """Run `fn` on the handle's stream after every pending torch upload, wait for it and raise on a bad status."""
    import torch
    torch.cuda.synchronize()
    rc = fn()
    h.check(rc)
    h.synchronize()


def _ptr(t):
    return None if t is None else t.data_ptr()


def _thp(a):
    from gp_algos_b200 import _lib
    return _lib.ptr(a)


def _pad128(n):
    return (n + 127) // 128 * 128


def _xbuf(Xs, ldx, stride=None):
    """Column-major X (ld ldx) of each problem in Xs at b * stride, NaN in the padding rows and between problems."""
    n, D = Xs[0].shape
    stride = ldx * D if stride is None else stride
    buf = np.full(len(Xs) * stride + 7, NAN)
    for b, X in enumerate(Xs):
        buf[b * stride:b * stride + ldx * D].reshape(D, ldx)[:, :n] = X.T
    return buf


def _colmajor(buf, ld, rows, cols, off=0):
    """View (rows x cols) of a column-major matrix with leading dimension ld at buf[off]."""
    return buf[off:off + ld * cols].reshape(cols, ld)[:, :rows].T


def _se_theta(rng, D, sf=1.3, sn=0.4):
    return np.concatenate([[sf], rng.uniform(0.7, 1.4, D) * math.sqrt(D / 8.0), [sn]])


def _cov(h, mode, X1, m, ldx1, thetas, Kbuf, ldk, mp=0, np_=0, X2=None, n=0, ldx2=0, has_s=0, s=0.0, batch=1,
         sX1=0, sX2=0, sK=0, D=None):
    th = np.ascontiguousarray(thetas, dtype=np.float64).ravel()
    D = (len(th) // batch - 2) if D is None else D
    _run(h, lambda: h.lib.gpk_debug_cov(h.h, mode, X1.data_ptr(), m, ldx1, _ptr(X2), n, ldx2, D, _thp(th), has_s, s,
                                        Kbuf.data_ptr(), ldk, mp, np_, batch, sX1, sX2, sK))
    return _host(Kbuf)


# =========================================================================================================================
# covariance build
# =========================================================================================================================
def _ulps(dev, ref_ld):
    """|dev - ref| in units of the last place of ref rounded to float64."""
    return np.abs(dev.astype(LD) - ref_ld) / np.spacing(np.abs(ref_ld.astype(np.float64))).astype(LD)


# The kernel computes r exactly as se_ard_r64 does, -r/2 exactly, exp within 1 ulp (CUDA math library) and one rounded
# product with sf^2: at most 1 ulp (exp, up to 2u relative) + 0.5 ulp (product) + 0.5 ulp (rounding the reference) in
# units of a result's ulp >= u |result|, i.e. < 3 ulp.  A contracted FMA in the distance changes r by an ulp of r and
# the value by ~r/2 ulp, which the r ~ 5..60 of these inputs exposes.
MAX_ULP = 3


@pytest.mark.parametrize("D", [1, 7, 8, 9, 16, 17, 64])
def test_se_ard_values_within_3_ulp(h, D):
    rng = np.random.default_rng(100 + D)
    for n in (1, 63, 64, 65, 127, 128, 129, 1000):
        X = rng.standard_normal((n, D))
        th = _se_theta(rng, D)
        ldx, ldk = n + 5, n + 3
        dX = _dev(_xbuf([X], ldx))
        K = _colmajor(_cov(h, SYM_FULL, dX, n, ldx, th, _dev(np.full(ldk * n, SENT)), ldk), ldk, ldk, n)
        ref = R.se_ard_value_from_r(R.se_ard_r64(X, X, R.se_ard_inv_ls2(th)), th)
        off = ~np.eye(n, dtype=bool)
        if n > 1:
            worst = _ulps(K[:n][off], ref[off]).max()
            assert worst <= MAX_ULP, (n, D, float(worst))
        assert np.all(K[n:] == SENT), (n, D)                       # rows n..ldk-1 of every column: never written
        # cross against other points
        m2 = max(1, n // 2 + 1)
        X2 = rng.standard_normal((m2, D))
        Kc = _colmajor(_cov(h, CROSS, dX, n, ldx, th, _dev(np.full(ldk * m2, SENT)), ldk, mp=n, np_=m2,
                            X2=_dev(_xbuf([X2], m2 + 2)), n=m2, ldx2=m2 + 2), ldk, ldk, m2)
        refc = R.se_ard_value_from_r(R.se_ard_r64(X, X2, R.se_ard_inv_ls2(th)), th)
        worst = _ulps(Kc[:n], refc).max()
        assert worst <= MAX_ULP, ("cross", n, D, float(worst))
        assert np.all(Kc[n:] == SENT)


def _tile_written_lower_pad(N):
    b = np.arange(N) // 64
    return (b[None, :] >> 1) <= (b[:, None] >> 1)                     # [row, col]: (bj >> 1) <= (bi >> 1)


def _mode_contracts(h, rng, n, D, thetas_fn, co2=False):
    th = thetas_fn()
    th0 = th.copy()
    s = 0.0625
    if co2:
        th0[10] = 0.0
        X = np.sort(rng.uniform(1960.0, 1963.0, n))[:, None]
    else:
        th0[-1] = 0.0
        X = rng.standard_normal((n, D))
    ldx = n + 3
    dX = _dev(_xbuf([X], ldx))
    # SYM_FULL with noise and sigmaNoise: bitwise symmetric, diagonal exactly (sf^2 + sn^2) + s
    Kf = _colmajor(_cov(h, SYM_FULL, dX, n, ldx, th, _dev(np.full(n * n, SENT)), n, has_s=1, s=s, D=D), n, n, n).copy()
    assert np.array_equal(Kf, Kf.T)
    sf2 = R.co2_value_diag(th) if co2 else th[0] * th[0]
    sn2 = th[10] * th[10] if co2 else th[-1] * th[-1]
    assert np.all(np.diag(Kf) == (sf2 + sn2) + s)
    # LOWER_PAD: every 64-tile of a 128-block on or below the diagonal, identity padding, bitwise SYM_FULL; sentinel above
    N = _pad128(n)
    Kp = _colmajor(_cov(h, LOWER_PAD, dX, n, ldx, th, _dev(np.full(N * N, SENT)), N, mp=N, has_s=1, s=s, D=D), N, N, N)
    written = _tile_written_lower_pad(N)
    assert np.all(Kp[~written] == SENT), "LOWER_PAD wrote a 128-block above the diagonal"
    assert np.array_equal(Kp[:n, :n][written[:n, :n]], Kf[written[:n, :n]]), "LOWER_PAD differs from SYM_FULL"
    pad = written.copy()
    pad[:n, :n] = False
    assert np.array_equal(Kp[pad], np.eye(N)[pad]), "LOWER_PAD padding is not the identity"
    # CROSS(X, X): zero fill up to (mp, np), nothing beyond; equals SYM_FULL without noise bitwise
    Kf0 = _colmajor(_cov(h, SYM_FULL, dX, n, ldx, th0, _dev(np.full(n * n, SENT)), n, D=D), n, n, n)
    mp, np_ = n + 7, n + 9
    ldk = mp + 3
    Kc = _colmajor(_cov(h, CROSS, dX, n, ldx, th, _dev(np.full(ldk * (np_ + 2), SENT)), ldk, mp=mp, np_=np_, X2=dX, n=n,
                        ldx2=ldx, D=D), ldk, ldk, np_ + 2)
    assert np.array_equal(Kc[:n, :n], Kf0)
    zero = np.zeros((ldk, np_ + 2), dtype=bool)
    zero[:mp, :np_] = True
    zero[:n, :n] = False
    assert np.all(Kc[zero] == 0.0)
    assert np.all(Kc[mp:] == SENT) and np.all(Kc[:, np_:] == SENT)


@pytest.mark.parametrize("n,D", [(1, 1), (63, 9), (65, 8), (129, 17), (300, 64)])
def test_cov_mode_contracts_se_ard(h, n, D):
    rng = np.random.default_rng(n * 7 + D)
    _mode_contracts(h, rng, n, D, lambda: _se_theta(rng, D))


@pytest.mark.parametrize("n", [1, 65, 200])
def test_cov_mode_contracts_co2(h, n):
    rng = np.random.default_rng(n)
    with h.kernel_family(KERNEL_CO2):
        _mode_contracts(h, rng, n, 1, lambda: orc.CO2_SHIPPED_HP.copy(), co2=True)


def _thetas3(rng, D, co2):
    if co2:
        return np.stack([orc.CO2_SHIPPED_HP * rng.uniform(0.8, 1.25, 11) for _ in range(3)])
    return np.stack([_se_theta(rng, D, sf=rng.uniform(0.8, 1.6), sn=rng.uniform(0.1, 0.5)) for _ in range(3)])


@pytest.mark.parametrize("co2", [False, True])
@pytest.mark.parametrize("shared_x", [True, False])
def test_cov_batch_equals_single_calls(h, co2, shared_x):
    rng = np.random.default_rng(31 + co2 + 2 * shared_x)
    n, D = (130, 1) if co2 else (130, 9)
    ths = _thetas3(rng, D, co2)
    Xs = [np.sort(rng.uniform(1960.0, 1970.0, n))[:, None] if co2 else rng.standard_normal((n, D)) for _ in range(3)]
    ldx = n + 3
    sX = 0 if shared_x else ldx * D + 13
    dXb = _dev(_xbuf(Xs[:1] if shared_x else Xs, ldx, None if shared_x else sX))
    N = _pad128(n)
    m2 = 77
    X2s = [rng.uniform(1960.0, 1970.0, (m2, 1)) if co2 else rng.standard_normal((m2, D)) for _ in range(3)]
    ldx2 = m2 + 1
    sX2 = 0 if shared_x else ldx2 * D + 5
    dX2b = _dev(_xbuf(X2s[:1] if shared_x else X2s, ldx2, None if shared_x else sX2))
    mp, np_ = n + 2, m2 + 3
    ldk = mp + 1
    sK = ldk * (np_ + 1) + 9
    ctx = h.kernel_family(KERNEL_CO2) if co2 else contextlib.nullcontext()
    with ctx:
        Kb = _cov(h, LOWER_PAD, dXb, n, ldx, ths, _dev(np.full(3 * N * N, SENT)), N, mp=N, batch=3, sX1=sX, D=D)
        Cb = _cov(h, CROSS, dXb, n, ldx, ths, _dev(np.full(3 * sK + 4, SENT)), ldk, mp=mp, np_=np_, X2=dX2b, n=m2, ldx2=ldx2,
                  batch=3, sX1=sX, sX2=sX2, sK=sK, D=D)
        for b in range(3):
            Xb = Xs[0] if shared_x else Xs[b]
            X2 = X2s[0] if shared_x else X2s[b]
            K1 = _cov(h, LOWER_PAD, _dev(_xbuf([Xb], ldx)), n, ldx, ths[b], _dev(np.full(N * N, SENT)), N, mp=N, D=D)
            assert np.array_equal(Kb[b * N * N:(b + 1) * N * N], K1), b
            C1 = _cov(h, CROSS, _dev(_xbuf([Xb], ldx)), n, ldx, ths[b], _dev(np.full(sK, SENT)), ldk, mp=mp, np_=np_,
                      X2=_dev(_xbuf([X2], ldx2)), n=m2, ldx2=ldx2, D=D)
            assert np.array_equal(Cb[b * sK:(b + 1) * sK], C1), b
        assert np.all(Cb[3 * sK:] == SENT)


def _co2_points(rng, n):
    return np.sort(rng.uniform(1960.0, 1964.0, n))


def test_co2_values(h):
    rng = np.random.default_rng(41)
    hp = orc.CO2_SHIPPED_HP.copy()
    for n in (1, 64, 129, 400):
        x = _co2_points(rng, n)
        with h.kernel_family(KERNEL_CO2):
            K = _colmajor(_cov(h, SYM_FULL, _dev(x), n, n, hp, _dev(np.full(n * n, SENT)), n, D=1), n, n, n)
        k, _, _, cond = R.co2_parts(x[:, None] - x[None, :], hp)
        k = k + np.eye(n) * LD(hp[10] * hp[10])
        # ~20 rounded operations, each amplified by at most the conditioning of the terms (all terms of k are positive)
        assert np.all(np.abs(K.astype(LD) - k) <= 32 * U * cond * k), n


def _deriv_matrix(h, p, X, th):
    n, D = X.shape
    out = np.zeros((n, n), order="F")
    Xf = np.asfortranarray(X)
    h.check(h.lib.gpk_cov_deriv_se_ard(h.h, p, _thp(Xf), n, D, n, _thp(th), _thp(out), n))
    return out


def test_co2_derivative_matrices_are_the_true_derivatives(h):
    """All ten dk/dhp of co2_derivs (and dk/dhp11) against the analytic derivatives that tests/test_eval_refs.py checks
    against mpmath.diff at 50 digits."""
    rng = np.random.default_rng(43)
    hp = orc.CO2_SHIPPED_HP.copy()
    n = 150
    x = _co2_points(rng, n)
    _, dk, mag, cond = R.co2_parts(x[:, None] - x[None, :], hp)
    with h.kernel_family(KERNEL_CO2):
        for p in range(1, 12):
            dK = _deriv_matrix(h, p, x[:, None], hp)
            if p == 11:
                assert np.array_equal(dK, np.eye(n) * 2 * hp[10])
                continue
            err = np.abs(dK.astype(LD) - dk[p - 1])
            assert np.all(err <= 64 * U * cond * mag[p - 1]), (p, float((err / (cond * mag[p - 1] + 1e-300)).max() / U))


@pytest.mark.parametrize("D", [1, 9])
def test_se_ard_derivative_matrices_are_the_true_derivatives(h, D):
    rng = np.random.default_rng(47 + D)
    n = 140
    X = rng.standard_normal((n, D))
    th = _se_theta(rng, D)
    dk, r = R.se_ard_dk(X, X, th, np.eye(n, dtype=bool))
    cond = 16 + r / 2 * (D + 4)
    for p in range(1, D + 3):
        dK = _deriv_matrix(h, p, X, th)
        err = np.abs(dK.astype(LD) - dk[p - 1])
        assert np.all(err <= cond * U * np.abs(dk[p - 1])), p


# =========================================================================================================================
# gradient trace
# =========================================================================================================================
def _kinv_sym(i, j):
    """A symmetric matrix with entries in [-1, -0.25] that is not low rank (so W = alpha alpha^t - Kinv >= 0 for alpha > 0)."""
    a, b = np.minimum(i, j).astype(np.float64), np.maximum(i, j).astype(np.float64)
    return -(0.25 + 0.75 * np.modf(a * 0.6180339887 + b * 0.4142135623 + ((a * b) % 97) * 0.0131)[0])


def _kinv_device(n, N, batch=1):
    """batch x (N x N) column-major: the lower triangle of _kinv_sym (scaled by b + 1 for problem b), NaN in the strictly
    upper triangle (so in every strictly upper 64-tile) and in rows / columns >= n."""
    i = np.arange(N)[:, None]
    j = np.arange(N)[None, :]
    full = _kinv_sym(i[:n], j[:, :n])
    out = np.full((batch, N, N), NAN)            # out[b, col, row]
    low = (i[:n] >= j[:, :n])
    for b in range(batch):
        m = np.where(low, full * (b + 1), NAN)
        out[b, :n, :n] = m.T
    return out.ravel(), full


def _grad_bound(n, D, s0, s1, co2):
    """u * ((c + S) * s0 + c' * s1): S = summation depth (16 terms per thread, 5 shuffle levels, 8 warp partials, then
    ceil(nblocks / 256) per finish thread and 8 tree levels), c = roundings per term (W: 2, e: 2, products: 3, (x_i - x_j)^2:
    3, gscale: 6) with 64 for the Co2 derivatives, c' = the exponent's conditioning: r/2 times (D + 4) roundings of r
    (SE-ARD), or ~64 roundings of the Co2 arguments."""
    nt = (n + 63) // 64
    nblocks = nt * (nt + 1) // 2
    S = 16 + 5 + 8 + math.ceil(nblocks / 256) + 8
    c, c1 = (64, 64) if co2 else (16, D + 4)
    return U * ((c + S) * s0 + c1 * s1), nblocks


def _grad(h, n, D, thetas, nparams, dX, ldx, Xs_host, alphas, kinv="neg", batch=1, strideX=0, strideOut=None, co2=False,
          check=True):
    N = _pad128(n)
    so = (nparams + 1) if strideOut is None else strideOut
    abuf = np.full(batch * N, NAN)
    for b in range(batch):
        abuf[b * N:b * N + n] = alphas[b]
    if kinv == "neg":
        kb, full = _kinv_device(n, N, batch)
        dK = _dev(kb)
    elif kinv == "zero":
        dK, full = _dev(np.zeros(batch * N * N)), None
    else:
        dK, full = None, None
    out = _dev(np.full(batch * so + 3, SENT))
    th = np.ascontiguousarray(thetas, dtype=np.float64).ravel()
    dA = _dev(abuf)
    _run(h, lambda: h.lib.gpk_debug_grad_trace(h.h, _ptr(dK), N, dX.data_ptr(), n, D, ldx, dA.data_ptr(), _thp(th), nparams,
                                               out.data_ptr(), batch, strideX, so))
    g = _host(out)
    for b in range(batch):
        assert np.all(g[b * so + nparams:(b + 1) * so] == SENT), "wrote beyond nparams"
    assert np.all(g[batch * so:] == SENT)
    if check:
        ths = np.asarray(thetas, dtype=np.float64).reshape(batch, -1)
        for b in range(batch):
            Kfull = None if full is None or kinv != "neg" else full * (b + 1)
            ref, s0, s1 = R.grad_trace_ref(Xs_host[b], alphas[b], Kfull, ths[b], nparams, co2=co2)
            bound, nblocks = _grad_bound(n, D, s0, s1, co2)
            gb = g[b * so:b * so + nparams]
            assert np.all(np.abs(gb - ref) <= bound), (n, D, b, gb, ref, np.abs(gb - ref) / np.maximum(bound, 1e-300))
            if kinv == "neg":
                # W >= 0: every signal / length-scale term is >= 0, so one dropped or doubled tile moves g by ~g / nblocks
                pos = list(range(min(nparams, D + 1 if n > 1 else 1)))    # n = 1: the length-scale terms are 0
                if not co2:
                    assert np.all(bound[pos] < 0.01 * ref[pos] / nblocks)
    return g


GRAD_CASES = [(1, 1), (2, 8), (63, 9), (64, 17), (65, 64), (129, 8), (129, 9), (1100, 17), (2050, 8), (8192, 1)]


@pytest.mark.parametrize("n,D", GRAD_CASES)
def test_grad_trace_against_full_square_reference(h, n, D):
    rng = np.random.default_rng(1000 + n + D)
    X = rng.uniform(0.0, 1.0, (n, D))
    th = np.concatenate([[1.1], rng.uniform(0.8, 1.2, D) * (0.5 * math.sqrt(D) + 0.3), [0.3]])
    alpha = rng.uniform(0.5, 1.5, n)
    ldx = n + 3
    _grad(h, n, D, th, D + 2, _dev(_xbuf([X], ldx)), ldx, [X], [alpha])


def test_grad_trace_fewer_parameters_and_null_kinv(h):
    rng = np.random.default_rng(7)
    n, D = 1100, 8
    X = rng.uniform(0.0, 1.0, (n, D))
    th = np.concatenate([[0.9], rng.uniform(0.8, 1.2, D) * 1.7, [0.2]])
    alpha = rng.standard_normal(n)
    ldx = n + 1
    dX = _dev(_xbuf([X], ldx))
    _grad(h, n, D, th, 5, dX, ldx, [X], [alpha])                     # nparams < D + 2
    g_null = _grad(h, n, D, th, D + 2, dX, ldx, [X], [alpha], kinv="null")
    g_zero = _grad(h, n, D, th, D + 2, dX, ldx, [X], [alpha], kinv="zero", check=False)
    assert np.array_equal(g_null, g_zero), "Kinv = NULL differs from Kinv = 0"


@pytest.mark.parametrize("co2", [False, True])
def test_grad_trace_batched_per_problem_theta(h, co2):
    rng = np.random.default_rng(11 + co2)
    n, D = (129, 1) if co2 else (129, 9)
    ths = _thetas3(rng, D, co2)
    if co2:
        Xs = [_co2_points(rng, n)[:, None] for _ in range(3)]
    else:
        Xs = [rng.uniform(0.0, 1.0, (n, D)) for _ in range(3)]
    alphas = [rng.uniform(0.5, 1.5, n) for _ in range(3)]
    ldx = n + 2
    sX = ldx * D + 3
    nparams = 11 if co2 else D + 2
    with (h.kernel_family(KERNEL_CO2) if co2 else contextlib.nullcontext()):
        _grad(h, n, D, ths, nparams, _dev(_xbuf(Xs, ldx, sX)), ldx, Xs, alphas, batch=3, strideX=sX, strideOut=nparams + 1,
              co2=co2)


@pytest.mark.parametrize("n", [1, 65, 300])
def test_grad_trace_co2_family(h, n):
    rng = np.random.default_rng(500 + n)
    hp = orc.CO2_SHIPPED_HP.copy()
    x = _co2_points(rng, n)[:, None]
    alpha = rng.uniform(0.5, 1.5, n)
    with h.kernel_family(KERNEL_CO2):
        _grad(h, n, 1, hp, 11, _dev(_xbuf([x], n + 1)), n + 1, [x], [alpha], co2=True)


def test_grad_trace_tile_decode_at_large_t(h):
    """n = 65536: 524800 tiles, the largest linear tile ids of the sqrt(8t + 1) decode.  alpha is non-zero only at tile edges,
    so the reference is a sum over ~20 x 20 pairs and no n x n buffer is needed (Kinv = NULL)."""
    rng = np.random.default_rng(65536)
    n, D = 65536, 2
    X = rng.uniform(0.0, 1.0, (n, D))
    th = np.array([1.2, 0.9, 1.1, 0.3])
    idx = np.array([0, 1, 63, 64, 127, 128, 4095, 4096, 20000, 32767, 32768, 40063, 40064, 65407, 65408, 65471, 65472,
                    65534, 65535])
    alpha = np.zeros(n)
    alpha[idx] = rng.uniform(0.5, 1.5, len(idx))
    N = n
    abuf = alpha.copy()
    dX = _dev(_xbuf([X], n))
    out = _dev(np.full(D + 3, SENT))
    dA = _dev(abuf)
    _run(h, lambda: h.lib.gpk_debug_grad_trace(h.h, None, N, dX.data_ptr(), n, D, n, dA.data_ptr(), _thp(th), D + 2,
                                               out.data_ptr(), 1, 0, D + 2))
    g = _host(out)
    ref, s0, s1 = R.grad_trace_ref(X, alpha, None, th, D + 2, rows=idx)
    bound, _ = _grad_bound(n, D, s0, s1, False)
    assert np.all(np.abs(g[:D + 2] - ref) <= bound), (g, ref)
    assert np.all(g[D + 2:] == SENT)


# =========================================================================================================================
# vector kernels (exact on small integers)
# =========================================================================================================================
def _li_int(rng, N):
    """Lower-triangular integer Li (|v| <= 8): exact zeros above the diagonal inside the diagonal 128-blocks, NaN in the
    strictly upper 128-blocks.  Returns (device layout, N x N column-major as [col, row]; the matrix as [row, col] with zeros
    above the diagonal, whose float64 products with small-integer vectors are exact in any summation order)."""
    L = np.tril(rng.integers(-8, 9, (N, N)).astype(np.float64))
    stored = L.copy()
    blk = np.arange(N) // 128
    stored[blk[:, None] < blk[None, :]] = NAN
    return stored.T.copy(), L


@pytest.mark.parametrize("N", [128, 256, 384, 640, 1280, 8192])
@pytest.mark.parametrize("transposed", [0, 1])
def test_trmv_exact(h, N, transposed):
    rng = np.random.default_rng(N + transposed)
    batch = 3 if N in (384, 1280) else 1
    Ls, xs, bufs = [], [], []
    for _ in range(batch):
        st, L = _li_int(rng, N)
        bufs.append(st.ravel())
        Ls.append(L)
        xs.append(rng.integers(-8, 9, N).astype(np.float64))
    dL = _dev(np.concatenate(bufs))
    dx = _dev(np.concatenate(xs))
    out = _dev(np.full(batch * N + 5, SENT))
    _run(h, lambda: h.lib.gpk_debug_trmv(h.h, transposed, dL.data_ptr(), N, dx.data_ptr(), out.data_ptr(), batch))
    o = _host(out)
    for b in range(batch):
        ref = (Ls[b].T if transposed else Ls[b]) @ xs[b]
        assert np.array_equal(o[b * N:(b + 1) * N], ref), (N, b)
    assert np.all(o[batch * N:] == SENT)


@pytest.mark.parametrize("square", [0, 1])
def test_colwise_dot_exact(h, square):
    rng = np.random.default_rng(17 + square)
    for rows in (1, 31, 32, 33, 63, 65, 127, 1001):
        for cols in (1, 7, 9, 33):
            batch = 3
            ld = rows + 3
            sM, sV, sO = ld * cols + 5, rows + 2, cols + 4
            Mbuf = np.full(batch * sM, NAN)
            vbuf = np.full(batch * sV, NAN)
            Ms, vs = [], []
            for b in range(batch):
                M = rng.integers(-8, 9, (rows, cols))
                v = rng.integers(-8, 9, rows)
                _colmajor(Mbuf, ld, rows, cols, b * sM)[...] = M
                vbuf[b * sV:b * sV + rows] = v
                Ms.append(M)
                vs.append(v)
            dM, dv = _dev(Mbuf), _dev(vbuf)
            out = _dev(np.full(batch * sO, SENT))
            _run(h, lambda: h.lib.gpk_debug_colwise_dot(h.h, dM.data_ptr(), ld, rows, cols, None if square else dv.data_ptr(),
                                                        out.data_ptr(), square, batch, sM, sV, sO))
            o = _host(out)
            for b in range(batch):
                ref = (Ms[b] * Ms[b]).sum(0) if square else vs[b] @ Ms[b]
                assert np.array_equal(o[b * sO:b * sO + cols], ref.astype(np.float64)), (rows, cols, b)
                assert np.all(o[b * sO + cols:(b + 1) * sO] == SENT)


@pytest.mark.parametrize("n", [1, 100, 256, 300, 1000])
def test_loglik_against_longdouble(h, n):
    rng = np.random.default_rng(n + 3)
    N = _pad128(n)
    batch = 3
    sO = 2
    A = np.full((batch, N, N), NAN)
    ys, als = np.full((batch, N), NAN), np.full((batch, N), NAN)
    for b in range(batch):
        A[b, np.arange(n), np.arange(n)] = rng.uniform(0.5, 3.0, n)
        ys[b, :n] = rng.standard_normal(n)
        als[b, :n] = rng.standard_normal(n)
    dA, dy, da = _dev(A.ravel()), _dev(ys.ravel()), _dev(als.ravel())
    out = _dev(np.full(batch * sO + 1, SENT))
    _run(h, lambda: h.lib.gpk_debug_loglik(h.h, dA.data_ptr(), N, n, dy.data_ptr(), da.data_ptr(), out.data_ptr(), batch, sO))
    o = _host(out)
    for b in range(batch):
        d = np.diag(A[b])[:n].astype(LD)
        yl, al = ys[b, :n].astype(LD), als[b, :n].astype(LD)
        ref = -np.sum(yl * al) / 2 - np.sum(np.log(d)) - LD(n) / 2 * np.log(2 * R.PI)
        mag = np.sum(np.abs(yl * al)) / 2 + np.sum(np.abs(np.log(d))) + LD(n) / 2 * np.log(2 * R.PI)
        depth = math.ceil(n / 256) + 8 + 8                            # per-thread terms, tree, log / product / final terms
        assert abs(LD(o[b * sO]) - ref) <= depth * U * mag, (n, b)
        assert o[b * sO + 1] == SENT
    assert o[batch * sO] == SENT


# =========================================================================================================================
# device-resident entry points
# =========================================================================================================================
@pytest.mark.parametrize("n", [300, 4200])
@pytest.mark.parametrize("has_s", [0, 1])
def test_nll_grad_dev_strided_x(h, n, has_s):
    """ldx = n + 37 with NaN padding rows, eager and through the graph cache (the capturing call and a replay): the numbers
    of the host entry point bit for bit, and the oracle's at 1e-9."""
    import ctypes as C
    import torch
    from gp_algos_b200 import _lib
    X, y, th = orc.make_c2(n=n, D=8)
    s = 0.01 if has_s else 0.0
    P = 10
    ldx = n + 37
    dX = _dev(_xbuf([X], ldx))
    dy = _dev(y)
    hd = _lib.Handle(0)
    hh = _lib.Handle(0)
    try:
        hh.set_graph_mode(0)
        Xf = np.asfortranarray(X)
        ll_h = C.c_double()
        g_h = np.zeros(P)
        hh.check(hh.lib.gpk_gp_nll_grad(hh.h, _thp(Xf), n, 8, n, _thp(y), _thp(th), has_s, s, P, C.byref(ll_h), _thp(g_h)))
        host = np.concatenate([[ll_h.value], g_h])
        runs = []
        out = _dev(np.full(P + 2, SENT))                      # the same buffers on every call: the graph cache's key
        info = torch.full((1,), -1, dtype=torch.int32, device="cuda")
        for mode, calls in ((0, 1), (1, 3)):                  # mode 1: eager, capture, replay
            hd.set_graph_mode(mode)
            for _ in range(calls):
                out.fill_(SENT)
                info.fill_(-1)
                _run(hd, lambda: hd.lib.gpk_gp_nll_grad_dev(hd.h, dX.data_ptr(), n, 8, ldx, dy.data_ptr(), _thp(th), has_s, s,
                                                            P, out.data_ptr(), info.data_ptr()))
                assert int(info.item()) == 0
                o = _host(out)
                assert o[P + 1] == SENT
                runs.append(o[:P + 1])
        for k, o in enumerate(runs):
            assert np.array_equal(o, host), (k, o, host)
    finally:
        hd.close()
        hh.close()
    sig = s if has_s else None
    if n <= 512:
        ll_o, g_o = orc.lit_loglik_with_derivs(X, y, th, sigma_noise=sig)
    else:
        ll_o, g_o = orc.fast_loglik_with_derivs(X, y, th, sigma_noise=sig)
    assert abs(host[0] - ll_o) <= 1e-9 * abs(ll_o)
    floor = 1e-9 * np.abs(g_o).max()
    assert np.all(np.abs(host[1:] - g_o) <= 1e-9 * np.maximum(np.abs(g_o), floor)), (host[1:], g_o)


def test_nll_grad_batched_dev_strided_x(h):
    import torch
    B, n, D, P = 3, 300, 8, 10
    rng = np.random.default_rng(77)
    Xs = [orc.make_c2(n=n, D=D, seed=10 + b)[0] for b in range(B)]
    ys = np.concatenate([orc.make_c2(n=n, D=D, seed=10 + b)[1] for b in range(B)])
    ths = np.stack([orc.pack_theta(rng.uniform(0.8, 1.2), rng.uniform(0.5, 0.9, D), rng.uniform(0.05, 0.2))
                    for _ in range(B)])
    ldx = n + 5
    sX = ldx * D + 11
    xb = _xbuf(Xs, ldx, sX)
    xh = np.where(np.isnan(xb), 0.0, xb)                      # the host call copies padding too: keep it finite there
    out = _dev(np.full(B * (P + 1) + 2, SENT))
    info = torch.full((B,), -1, dtype=torch.int32, device="cuda")
    dX, dy = _dev(xb), _dev(ys)
    _run(h, lambda: h.lib.gpk_gp_nll_grad_batched_dev(h.h, B, dX.data_ptr(), n, D, ldx, sX, dy.data_ptr(), _thp(ths), 0, 0.0, P,
                                                      out.data_ptr(), info.data_ptr()))
    assert np.all(_host(info) == 0)
    o = _host(out)
    assert np.all(o[B * (P + 1):] == SENT)
    ll, g, inf = np.zeros(B), np.zeros(B * P), np.zeros(B, dtype=np.int32)
    h.check(h.lib.gpk_gp_nll_grad_batched(h.h, B, _thp(xh), n, D, ldx, sX, _thp(ys), _thp(ths), 0, 0.0, P, _thp(ll), _thp(g),
                                          _thp(inf)))
    for b in range(B):
        assert o[b * (P + 1)] == ll[b]
        assert np.array_equal(o[b * (P + 1) + 1:(b + 1) * (P + 1)], g[b * P:(b + 1) * P]), b


def test_cov_dev_entry_points_equal_host(h):
    rng = np.random.default_rng(91)
    n, m, D = 203, 71, 5
    X, X2 = rng.standard_normal((n, D)), rng.standard_normal((m, D))
    th = _se_theta(rng, D)
    ldx, ldx2, ldk = n + 3, m + 2, n + 4
    dX, dX2 = _dev(_xbuf([X], ldx)), _dev(_xbuf([X2], ldx2))
    K = np.zeros((n, n), order="F")
    h.check(h.lib.gpk_cov_se_ard(h.h, _thp(np.asfortranarray(X)), n, D, n, _thp(th), _thp(K), n))
    dK = _dev(np.full(ldk * n, SENT))
    _run(h, lambda: h.lib.gpk_cov_se_ard_dev(h.h, dX.data_ptr(), n, D, ldx, _thp(th), dK.data_ptr(), ldk))
    Kd = _colmajor(_host(dK), ldk, ldk, n)
    assert np.array_equal(Kd[:n], K) and np.all(Kd[n:] == SENT)
    Kc = np.zeros((n, m), order="F")
    h.check(h.lib.gpk_cov_cross_se_ard(h.h, _thp(np.asfortranarray(X)), n, n, _thp(np.asfortranarray(X2)), m, m, D, _thp(th),
                                       _thp(Kc), n))
    dKc = _dev(np.full(ldk * m, SENT))
    _run(h, lambda: h.lib.gpk_cov_cross_se_ard_dev(h.h, dX.data_ptr(), n, ldx, dX2.data_ptr(), m, ldx2, D, _thp(th),
                                                   dKc.data_ptr(), ldk))
    Kcd = _colmajor(_host(dKc), ldk, ldk, m)
    assert np.array_equal(Kcd[:n], Kc) and np.all(Kcd[n:] == SENT)
