"""CPU: the references of tests/ep_refs.py (used by tests/test_gpu_ep_kernels.py) against mpmath at 50 digits and against the
oracle's literal EP sweep; their error bounds against a plain float64 run of the same formulas."""
import numpy as np
import pytest

from oracle import gp_oracle as orc
from tests import ep_refs as R

mp = pytest.importorskip("mpmath")
LD = np.longdouble


def _site_inputs(rng, m):
    """First-sweep and later-sweep states: sii in [1e-6, 1e3], den = 1 - t_old sii down to 1e-6, y = +-1."""
    sii = 10.0 ** rng.uniform(-6, 3, m)
    den = np.where(rng.random(m) < 0.3, 1.0, 10.0 ** rng.uniform(-6, 0, m))
    t_old = (1 - den) / sii
    mui = rng.normal(0, 1, m) * np.sqrt(sii) * 3
    n_old = rng.normal(0, 1, m) * t_old
    y = rng.choice([-1.0, 1.0], m)
    return sii, mui, t_old, n_old, y


def _site_mp(sii, mui, t_old, n_old, y):
    """The site update as written, at 50 digits."""
    with mp.workdps(50):
        sii, mui, t_old, n_old, y = (mp.mpf(float(v)) for v in (sii, mui, t_old, n_old, y))
        ct = 1 / sii - t_old
        cn = mui / sii - n_old
        cmu, csig = cn / ct, 1 / ct
        temp = mp.sqrt(1 + csig)
        z = y * cmu / temp
        r = mp.npdf(z) / mp.ncdf(z)
        mu_hat = cmu + y * csig * r / temp
        sig_hat = csig - csig * csig * r * (z + r) / (1 + csig)
        dtau = 1 / sig_hat - ct - t_old
        nu = mu_hat / sig_hat - cn
        c = 1 / (1 / dtau + sii)
        dnu = nu - n_old
        g = dnu - c * (mui + dnu * sii)
        return dict(ct=ct, cn=cn, tau=t_old + dtau, nu=nu, c=c, g=g, sig_hat=sig_hat, mu_hat=mu_hat)


def test_site_update_matches_mpmath():
    rng = np.random.default_rng(11)
    sii, mui, t_old, n_old, y = _site_inputs(rng, 300)
    ld = R.site_update(sii, mui, t_old, n_old, y)
    for i in range(len(sii)):
        ref = _site_mp(sii[i], mui[i], t_old[i], n_old[i], y[i])
        for k, v in ref.items():
            # longdouble: u_ld = 2^-64, magnified by the condition of the site update (bounded by the float64 bound / u)
            b = R.site_bound(sii[i:i + 1], mui[i:i + 1], t_old[i:i + 1], n_old[i:i + 1], y[i:i + 1], False)
            bk = {"tau": "dtau"}.get(k, k)
            tol = float(b[bk][0]) * 2.0 ** -11
            assert abs(float(ld[k][i] - R._from_mp(v))) <= tol + 1e-300, (k, i, float(ld[k][i]), float(v), tol)


def test_site_bound_covers_a_float64_run_of_the_formulas():
    """The literal formulas evaluated in float64 (phi/Phi rounded to float64, inside the modelled libdevice error) stay inside
    the bound of ep_site_scalar, output by output."""
    rng = np.random.default_rng(12)
    sii, mui, t_old, n_old, y = _site_inputs(rng, 400)
    ld = R.site_update(sii, mui, t_old, n_old, y)
    f64 = R.site_update(sii, mui, t_old, n_old, y, dtype=np.float64)
    b = R.site_bound(sii, mui, t_old, n_old, y, False)
    for k, bk in (("ct", "ct"), ("cn", "cn"), ("c", "c"), ("g", "g"), ("dtau", "dtau"), ("nu", "nu")):
        err = np.abs(f64[k].astype(LD) - ld[k])
        assert np.all(err <= b[bk]), (k, float(np.max(err / b[bk])))


def test_ratio_and_erfcx_match_mpmath():
    for z in (-40.0, -11.3, -1.0, 0.0, 1e-300, 0.5, 11.3, 40.0):
        with mp.workdps(50):
            ref = mp.npdf(mp.mpf(z)) / mp.ncdf(mp.mpf(z))
        assert abs(float(R.ratio([z])[0] / R._from_mp(ref) - 1)) < 1e-18
    assert abs(float(R._from_mp(R.erfcx_mp(3.0))) - float(mp.exp(9) * mp.erfc(3))) < 1e-15


@pytest.mark.parametrize("n", [65, 130])
def test_site_loop_matches_literal_oracle_first_sweep(n):
    X, t, th = orc.make_c3(n=n, D=2, seed=n)
    K = orc.lit_build_kernel_matrix(X, th)
    o = orc.lit_ep_estimate(K, t, fixed_sweeps=1)
    z = np.zeros(n)
    ld = R.site_loop(K, z, z, z, t)
    assert np.max(np.abs(ld["tau"].astype(float) - o["tau"]) / np.abs(o["tau"]).max()) <= 1e-12
    assert np.max(np.abs(ld["nu"].astype(float) - o["nu"]) / np.abs(o["nu"]).max()) <= 1e-12
    assert np.max(np.abs(ld["cav_tau"].astype(float) - o["cav_tau"]) / np.abs(o["cav_tau"]).max()) <= 1e-12


def test_site_loop_rank1_mean_equals_full_product():
    """mu += s g keeps mu = Sigma nu (the reference's full product at :54) when the sweep starts consistent."""
    rng = np.random.default_rng(3)
    n = 40
    x = np.sort(rng.uniform(0, 4, n))
    K = np.exp(-0.5 * (x[:, None] - x[None, :]) ** 2) + 1e-3 * np.eye(n)
    y = rng.choice([-1, 1], n)
    z = np.zeros(n)
    s1 = R.site_loop(K, z, z, z, y)
    rf = R.refactor(K, s1["tau"], s1["nu"])
    s2 = R.site_loop(rf["Sigma"], s1["tau"], s1["nu"], rf["mu"], y)
    full = s2["Sigma"] @ s2["nu"]
    assert np.max(np.abs(s2["mu"] - full)) <= 1e-15 * np.max(np.abs(full))


def test_refactor_matches_mpmath():
    rng = np.random.default_rng(5)
    n = 12
    x = np.sort(rng.uniform(0, 3, n))
    K = np.exp(-0.5 * (x[:, None] - x[None, :]) ** 2) + 1e-2 * np.eye(n)
    tau = rng.uniform(0.05, 2.0, n)
    nu = rng.normal(0, 1, n)
    ld = R.refactor(K, tau, nu)
    with mp.workdps(50):
        Km = mp.matrix(K.tolist())
        S = mp.diag([mp.mpf(float(v)) for v in tau])
        Sigma = mp.inverse(mp.inverse(Km) + S)
        st = mp.diag([mp.sqrt(mp.mpf(float(v))) for v in tau])
        L = mp.cholesky(mp.eye(n) + st * Km * st)
        mu = Sigma * mp.matrix([float(v) for v in nu])
    Sm = np.array([[float(Sigma[i, j]) for j in range(n)] for i in range(n)])
    Lm = np.array([[float(L[i, j]) for j in range(n)] for i in range(n)])
    mum = np.array([float(mu[i]) for i in range(n)])
    assert np.max(np.abs(ld["Sigma"].astype(float) - Sm)) <= 1e-15 * np.abs(K).max()
    assert np.max(np.abs(ld["L"].astype(float) - Lm)) <= 1e-15 * np.abs(Lm).max()
    assert np.max(np.abs(ld["mu"].astype(float) - mum)) <= 1e-15 * np.abs(mum).max() * 10
    f64 = R.refactor(K, tau, nu, dtype=np.float64)
    b = R.refactor_bounds(ld, f64, K, nu)
    assert np.all(np.abs(f64["Sigma"] - ld["Sigma"]) <= b["Sigma"])
