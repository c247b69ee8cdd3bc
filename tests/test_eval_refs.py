"""CPU: the longdouble references of tests/eval_refs.py (used by tests/test_gpu_eval_kernels.py) against mpmath at 50 digits
and against the oracle, so that they are known to be right before any GPU run."""
import mpmath
import numpy as np
import pytest

from oracle import gp_oracle as orc
from tests import eval_refs as R

U = 2.0 ** -53


def _mp(v):
    """Exact mpf of a longdouble."""
    num, den = np.longdouble(v).as_integer_ratio()
    return mpmath.mpf(num) / den


def _se_theta(rng, D):
    return np.concatenate([[1.3], rng.uniform(0.7, 1.4, D) * np.sqrt(max(D, 1) / 8.0) + 0.2, [0.4]])


def _mp_se_k(x1, x2, th):
    D = len(th) - 2
    r = mpmath.fsum(((mpmath.mpf(x1[d]) - mpmath.mpf(x2[d])) / th[1 + d]) ** 2 for d in range(D))
    return th[0] ** 2 * mpmath.exp(-r / 2)


def _mp_co2_k(xd, hp):
    h1, h2, h3, h4, h5, h6, h7, h8, h9, h10 = hp[:10]
    sq = xd * xd
    s = mpmath.sin(mpmath.pi * xd)
    return (h1 ** 2 * mpmath.exp(-sq / (2 * h2 ** 2))
            + h3 ** 2 * mpmath.exp(-sq / (2 * h4 ** 2) - 2 * s * s / h5 ** 2)
            + h6 ** 2 * (1 + sq / (2 * h8 * h7 ** 2)) ** (-h8)
            + h9 ** 2 * mpmath.exp(-sq / (2 * h10 ** 2)))


@pytest.mark.parametrize("D", [1, 3, 9])
def test_se_ard_value_and_derivatives_against_mpmath(D):
    rng = np.random.default_rng(10 + D)
    X = rng.standard_normal((6, D))
    th = _se_theta(rng, D)
    r64 = R.se_ard_r64(X, X, R.se_ard_inv_ls2(th))
    val = R.se_ard_value_from_r(r64, th)
    dk, _ = R.se_ard_dk(X, X, th, np.eye(6, dtype=bool))
    with mpmath.workdps(50):
        for i in range(6):
            for j in range(6):
                ref = mpmath.mpf(float(th[0]) * float(th[0])) * mpmath.exp(-mpmath.mpf(r64[i, j]) / 2)
                assert abs(_mp(val[i, j]) - ref) <= 1e-18 * abs(ref)
                thm = [mpmath.mpf(v) for v in th]
                for p in range(D + 1):
                    def k_of(t, p=p):
                        th2 = list(thm)
                        th2[p] = t
                        return _mp_se_k(X[i], X[j], th2)
                    ref_d = mpmath.diff(k_of, thm[p])
                    assert abs(_mp(dk[p][i, j]) - ref_d) <= 1e-17 * max(abs(ref_d), 1e-30), (p, i, j)
                # noise: d(sn^2 [i == j]) / dsn
                assert float(dk[D + 1][i, j]) == (2 * th[-1] if i == j else 0.0)


def test_co2_value_and_derivatives_against_mpmath():
    hp = orc.CO2_SHIPPED_HP.copy()
    rng = np.random.default_rng(3)
    xd = np.concatenate([[0.0, 1e-3, 0.5, 1.0, 2.25], rng.uniform(-3, 3, 7)])
    k, dk, _, _ = R.co2_parts(xd, hp)
    with mpmath.workdps(50):
        hpm = [mpmath.mpf(v) for v in hp]
        for t, x in enumerate(xd):
            xm = mpmath.mpf(x)
            ref = _mp_co2_k(xm, hpm)
            assert abs(_mp(k[t]) - ref) <= 1e-17 * abs(ref)
            for p in range(10):
                def k_of(v, p=p):
                    h2 = list(hpm)
                    h2[p] = v
                    return _mp_co2_k(xm, h2)
                ref_d = mpmath.diff(k_of, hpm[p])
                # floor: the longdouble cancellation in dk/dhp8 at small xd (-log p1 + ...) leaves ~eps_ld * k absolute
                assert abs(_mp(dk[p][t]) - ref_d) <= 1e-16 * abs(ref_d) + 1e-18 * abs(ref), (p, x)


def test_se_ard_value_against_oracle_kernel_matrix():
    rng = np.random.default_rng(5)
    X, X2 = rng.standard_normal((30, 4)), rng.standard_normal((11, 4))
    th = _se_theta(rng, 4)
    K = R.se_ard_value_from_r(R.se_ard_r64(X, X, R.se_ard_inv_ls2(th)), th).astype(np.float64)
    K[np.diag_indices(30)] += th[-1] ** 2
    Ko = orc.lit_build_kernel_matrix(X, th)
    assert np.all(np.abs(K - Ko) <= 4 * U * np.abs(Ko))
    Kc = R.se_ard_value_from_r(R.se_ard_r64(X, X2, R.se_ard_inv_ls2(th)), th).astype(np.float64)
    Kco = orc.lit_build_kernel_matrix(X, th, X2)
    assert np.all(np.abs(Kc - Kco) <= 4 * U * np.abs(Kco))
    dk, r = R.se_ard_dk(X, X, th, np.eye(30, dtype=bool))
    cond = 16 + r.astype(np.float64) / 2 * (4 + 4)      # the oracle's exp(-r/2) inherits r's rounding, (D + 4) u relative
    for p in range(6):
        dko = orc.lit_build_der_matrix(p + 1, X, th)
        assert np.all(np.abs(dk[p].astype(np.float64) - dko) <= cond * U * np.abs(dko)), p


def test_co2_against_oracle_k_and_dk():
    hp = orc.CO2_SHIPPED_HP.copy()
    rng = np.random.default_rng(6)
    x = np.sort(rng.uniform(1960.0, 1963.0, 9))
    xd = x[:, None] - x[None, :]
    k, dk, _, cond = R.co2_parts(xd, hp)
    for i in range(9):
        for j in range(9):
            ko = orc.co2_k(x[i], x[j], hp)
            assert abs(float(k[i, j]) - ko) <= 64 * U * float(cond[i, j]) * abs(ko)
            for p in range(10):
                do = orc.co2_dk(p + 1, x[i], x[j], hp)
                assert abs(float(dk[p][i, j]) - do) <= 64 * U * float(cond[i, j]) * max(abs(do), 1e-3 * abs(ko)), (p, i, j)
            assert orc.co2_dk(11, x[i], x[j], hp, i == j) == (2 * hp[10] if i == j else 0.0)


@pytest.mark.parametrize("co2", [False, True])
def test_gradient_reference_against_oracle(co2):
    """grad_trace_ref with alpha = K^-1 y and K^-1 from the same K is the literal gradient (GpPredictor.scala:60-80)."""
    rng = np.random.default_rng(8)
    n = 48
    if co2:
        X, y, th = orc.make_co2_like(n=n)
        y = y - y.mean()
        with orc.co2_kernel():
            K = orc.lit_build_kernel_matrix(X, th)
            _, g_o = orc.lit_loglik_with_derivs(X, y, th)
    else:
        X = rng.standard_normal((n, 3))
        th = _se_theta(rng, 3)
        y = rng.standard_normal(n)
        K = orc.lit_build_kernel_matrix(X, th)
        _, g_o = orc.lit_loglik_with_derivs(X, y, th)
    Kinv = np.linalg.inv(K)
    Kinv = (Kinv + Kinv.T) / 2
    g, s0, _ = R.grad_trace_ref(X, Kinv @ y, Kinv, th, len(th), co2=co2)
    assert np.all(np.abs(g - g_o) <= 1e-8 * np.maximum(np.abs(g_o), np.abs(g_o).max())), (g, g_o)
