"""Plain high-precision references of the EP sweep's kernels (csrc/gpk_ep.cu) for tests/test_gpu_ep_kernels.py: the scalar site
update, the sequential site loop with a full rank-1 downdate of Sigma per site, and the posterior re-factorisation.  NumPy
`longdouble` (64-bit significand), phi/Phi from mpmath; never the oracle.  tests/test_ep_refs.py checks them against mpmath at 50
digits and against the oracle on the CPU.

Error bounds (all constants fixed from the derivations below, not from observed kernel errors):
- scalar site update: a first-order running error analysis of the kernel's own sequence of operations (`site_bound`): every
  value carries |error| <= e, and each operation adds the propagated input errors (|d result / d input| e_input) and its own
  rounding, u |result| for + - * / sqrt and the correctly rounded reciprocals, 2u for rsqrt.  That is a term-magnitude sum: for
  c = (sii - sig_hat) / sii^2 it is u (sii + |sig_hat|) / sii^2 plus e(sig_hat) / sii^2, for tau = t_old + (1/sig_hat - 1/sii)
  it is u (1/sig_hat + 1/sii + |t_old|) plus the propagated error of sig_hat.  phi/Phi carries a relative error of 3e-14 on
  the table route (the table's 1.8e-14 with the evaluation's rounding, as the CPU test of the table allows) and (2 z^2 + 8) u
  on the libdevice routes (exp(-z^2/2) and erfc(-z/sqrt2) see the rounding of their argument magnified by z^2; a few ulp
  of their own).  The bound used is SITE_FACTOR = 2 times the first-order sum: the factor covers the second-order terms and
  the libdevice functions' last ulp.
- products: gamma_k (|X| |W|) with gamma_k = k u / (1 - k u).
- site loop and re-factorisation: the accumulated rounding of a recurrence has no closed-form bound here.  The bound is
  LOOP_FACTOR = 16 times the error of the same recurrence run in plain float64 against the longdouble run, plus a floor of
  64 n u scale (scale: the quantity's term-magnitude sum), plus, for a site output, the site update's own bound.
"""
import numpy as np

LD = np.longdouble
U = 2.0 ** -53
SITE_FACTOR = 2
LOOP_FACTOR = 16
FLOOR = 64
RATIO_TABLE_REL = 3e-14
SQRT_2_OVER_PI = LD("0.797884560802865355879892119868763737")


def gamma(k):
    return k * U / (1 - k * U)


# ---------------------------------------------------------------------------------------------------------------------------
# phi(z) / Phi(z) in high precision
# ---------------------------------------------------------------------------------------------------------------------------
def _to_mp(x):
    import mpmath as mp
    x = LD(x)
    hi = float(x)
    return mp.mpf(hi) + mp.mpf(float(x - LD(hi)))      # exact: a longdouble is the sum of two doubles


def _from_mp(v):
    import mpmath as mp
    return LD(mp.nstr(v, 24, min_fixed=1, max_fixed=0))     # through the decimal string: no float64 underflow on the way


def ratio_mp(z, dps=40):
    """phi(z) / Phi(z) as an mpmath number (z a float or longdouble, taken exactly)."""
    import mpmath as mp
    with mp.workdps(dps):
        zz = _to_mp(z)
        return mp.npdf(zz) / mp.ncdf(zz)


def ratio(z, dtype=LD):
    """phi/Phi elementwise, rounded to dtype (longdouble or float64) from 40 digits."""
    z = np.asarray(z)
    out = np.array([_from_mp(ratio_mp(v)) for v in z.ravel()], dtype=LD).reshape(z.shape)
    return out.astype(dtype)


def erfcx_mp(x, dps=40):
    import mpmath as mp
    with mp.workdps(dps):
        xx = _to_mp(x)
        return mp.exp(xx * xx) * mp.erfc(xx)


# ---------------------------------------------------------------------------------------------------------------------------
# the site update of EpParameterEstimator.scala:41-55, as written
# ---------------------------------------------------------------------------------------------------------------------------
def site_update(sii, mui, t_old, n_old, y, dtype=LD):
    """The site update as written (EpParameterEstimator.scala:45-53, marginalMoments :98-109) in `dtype`, phi/Phi from 40 digits.
    Returns a dict of arrays: ct, cn, z, ratio, mu_hat, sig_hat, dtau, tau, nu, c, g."""
    sii, mui, t_old, n_old, y = (np.asarray(v, dtype=dtype) for v in (sii, mui, t_old, n_old, y))
    one = dtype(1)
    ct = one / sii - t_old                                        # :45
    cn = mui / sii - n_old                                        # :46
    cmu, csig = cn / ct, one / ct                                 # marginalMoments(cav_nu / cav_tau, 1 / cav_tau, y)
    temp = np.sqrt(1 + csig)
    z = (y * cmu) / temp
    r = ratio(z, dtype)
    mu_hat = cmu + (y * csig * r) / temp
    sig_hat = csig - ((csig * csig * r) * (z + r)) / (1 + csig)
    dtau = one / sig_hat - ct - t_old                             # :49
    tau = t_old + dtau                                            # :50
    nu = mu_hat / sig_hat - cn                                    # :51
    with np.errstate(divide="ignore"):
        c = one / (one / dtau + sii)                              # :53
    dnu = nu - n_old
    g = dnu - c * (mui + dnu * sii)                               # mu = Sigma nu after the rank-1 change (:54)
    return dict(ct=ct, cn=cn, z=z, ratio=r, mu_hat=mu_hat, sig_hat=sig_hat, dtau=dtau, tau=tau, nu=nu, c=c, g=g)


def site_update_mp(sii, mui, t_old, n_old, y, dps=40):
    """The site update as written at `dps` digits, rounded to longdouble (same keys as site_update).  For later-sweep states
    with den = 1 - t_old sii near 0 the longdouble evaluation of 1/sii - t_old loses log10(1/den) digits; this one does not."""
    import mpmath as mp
    keys = ("ct", "cn", "z", "ratio", "mu_hat", "sig_hat", "dtau", "tau", "nu", "c", "g")
    out = {k: [] for k in keys}
    with mp.workdps(dps):
        for a in zip(*(np.asarray(v, dtype=np.float64).ravel() for v in (sii, mui, t_old, n_old, y))):
            si, mi, to, no, yy = (mp.mpf(float(v)) for v in a)
            ct = 1 / si - to
            cn = mi / si - no
            cmu, csig = cn / ct, 1 / ct
            temp = mp.sqrt(1 + csig)
            z = yy * cmu / temp
            r = mp.npdf(z) / mp.ncdf(z)
            mu_hat = cmu + yy * csig * r / temp
            sig_hat = csig - csig * csig * r * (z + r) / (1 + csig)
            dtau = 1 / sig_hat - ct - to
            nu = mu_hat / sig_hat - cn
            c = dtau / (1 + dtau * si)
            dnu = nu - no
            g = dnu - c * (mi + dnu * si)
            for k, v in zip(keys, (ct, cn, z, r, mu_hat, sig_hat, dtau, to + dtau, nu, c, g)):
                out[k].append(_from_mp(v))
    return {k: np.array(v, dtype=LD) for k, v in out.items()}


class _E:
    """A value (longdouble, exact to the reference's precision) with a first-order bound of the kernel's error in it."""

    def __init__(self, v, e=None):
        self.v = np.asarray(v, dtype=LD)
        self.e = np.zeros_like(self.v) if e is None else np.asarray(e, dtype=LD)

    def _r(self, v, e, k=1):
        return _E(v, e + k * U * np.abs(v))

    def __add__(self, o):
        o = _c(o); return self._r(self.v + o.v, self.e + o.e)

    def __sub__(self, o):
        o = _c(o); return self._r(self.v - o.v, self.e + o.e)

    def __rsub__(self, o):
        return _c(o) - self

    def __mul__(self, o):
        o = _c(o); return self._r(self.v * o.v, np.abs(o.v) * self.e + np.abs(self.v) * o.e)

    __radd__ = __add__
    __rmul__ = __mul__

    def __truediv__(self, o):
        o = _c(o); v = self.v / o.v
        return self._r(v, self.e / np.abs(o.v) + np.abs(v) * o.e / np.abs(o.v))

    def __rtruediv__(self, o):
        return _c(o) / self


def _c(x):
    return x if isinstance(x, _E) else _E(x)


def _fma(a, b, c):
    a, b, c = _c(a), _c(b), _c(c)
    v = a.v * b.v + c.v
    return _E(v, np.abs(b.v) * a.e + np.abs(a.v) * b.e + c.e + U * np.abs(v))


def _rsqrt(a):
    v = 1 / np.sqrt(a.v)
    return _E(v, np.abs(v) * a.e / (2 * np.abs(a.v)) + 2 * U * np.abs(v))


def _sqrt(a):
    v = np.sqrt(a.v)
    return _E(v, a.e / (2 * v) + U * v)


def _ratio(z, rel):
    r = ratio(z.v)
    return _E(r, np.abs(r * (z.v + r)) * z.e + rel * np.abs(r))     # d ratio / dz = -ratio (z + ratio)


def ratio_rel_err(z, fast):
    """Relative error of the kernel's phi/Phi at z: the table route (|z| < 8 sqrt2) or the libdevice routes."""
    z = np.abs(np.asarray(z, dtype=LD))
    lib = (2 * z * z + 8) * U
    return np.where(z < 8 * np.sqrt(LD(2)), RATIO_TABLE_REL, lib) if fast else lib


def site_bound(sii, mui, t_old, n_old, y, fast, e_sii=None, e_mui=None):
    """SITE_FACTOR x the first-order error bound of the kernel's scalar site update at these inputs (exact, or sii and mui
    carrying the error bounds e_sii, e_mui).
    fast: ep_site_fast + the finish of ep_sites_block_p -> dict(c, g, mu_hat, sig_hat, ct, cn, tau, nu);
    else: ep_site_scalar -> dict(ct, cn, c, g, dtau, nu, mu_hat, sig_hat)."""
    sii, mui, t_old, n_old, y = (_E(np.asarray(v, dtype=LD)) for v in (sii, mui, t_old, n_old, y))
    if e_sii is not None:
        sii, mui = _E(sii.v, e_sii), _E(mui.v, e_mui)
    if fast:
        den = _fma(-t_old.v, sii, 1)
        num = _fma(-n_old.v, sii, mui)
        r, rs = 1 / den, 1 / sii
        wq = _rsqrt(den + sii)
        rt = _sqrt(den) * wq
        csig, cmu = sii * r, num * r
        ct, cn = den * rs, num * rs
        z = (y * cmu) * rt
        a1 = (csig * rt) * (csig * rt)
        b1 = (y * csig) * rt
        q = _ratio(z, ratio_rel_err(z.v, True))
        mu_hat = _fma(b1, q, cmu)
        sig_hat = _fma(_E(-a1.v, a1.e), q * (z + q), csig)
        c = (sii - sig_hat) * (rs * rs)
        g = (mu_hat - mui) * rs
        rsig = 1 / sig_hat
        tau = t_old + (rsig - rs)
        nu = mu_hat * rsig - cn
        out = dict(c=c, g=g, mu_hat=mu_hat, sig_hat=sig_hat, ct=ct, cn=cn, tau=tau, nu=nu)
    else:
        rsii = 1 / sii
        ct = rsii - t_old
        cn = mui * rsii - n_old
        csig = 1 / ct
        cmu = cn * csig
        rt = _rsqrt(1 + csig)
        z = (y * cmu) * rt
        q = _ratio(z, ratio_rel_err(z.v, False))
        mu_hat = cmu + (y * csig) * (q * rt)
        sig_hat = csig - ((csig * csig) * q) * ((z + q) * (rt * rt))
        rsig = 1 / sig_hat
        dtau = rsig - ct - t_old
        nu = mu_hat * rsig - cn
        c = dtau / (1 + dtau * sii)
        dnu = nu - n_old
        g = dnu - c * (mui + dnu * sii)
        out = dict(ct=ct, cn=cn, c=c, g=g, dtau=dtau, nu=nu, mu_hat=mu_hat, sig_hat=sig_hat)
    return {k: SITE_FACTOR * v.e for k, v in out.items()}


# ---------------------------------------------------------------------------------------------------------------------------
# the sequential site loop: one sweep, full rank-1 downdate of Sigma per site (EpParameterEstimator.scala:44-55)
# ---------------------------------------------------------------------------------------------------------------------------
def site_loop(Sigma, tau, nu, mu, y, dtype=LD, keep_columns=False):
    """One sweep over all sites of the n x n Sigma (symmetric) in `dtype`.  mu is kept as Sigma nu by the rank-1 form of
    :54, mu += s g (equal to the full product when the input mu = Sigma nu).  Returns a dict: tau, nu, mu, cav_tau, cav_nu, c, g,
    the per-site inputs sii, mui, t_old, n_old, the term-magnitude sums mu_scale = |mu_0| + sum_k |s_k g_k| (after the sweep),
    sii_scale = |Sigma_ii| + sum_{k<i} |c_k| s_k[i]^2 and mui_scale (the same sums at site i) and, with
    keep_columns, S (column k: the update vector s_k = Sigma[:, k] at site k)."""
    S = np.array(Sigma, dtype=dtype)
    n = S.shape[0]
    tau, nu, mu = (np.array(v, dtype=dtype) for v in (tau, nu, mu))
    yv = np.asarray(y, dtype=dtype)
    out = {k: np.zeros(n, dtype=dtype) for k in ("cav_tau", "cav_nu", "c", "g", "sii", "mui", "t_old", "n_old")}
    mu_scale = np.abs(mu).astype(LD)
    dg_scale = np.abs(np.diag(S)).astype(LD)
    out["sii_scale"], out["mui_scale"] = np.zeros(n, dtype=LD), np.zeros(n, dtype=LD)
    cols = np.zeros((n, n), dtype=dtype) if keep_columns else None
    for i in range(n):
        sii, mui = S[i, i], mu[i]
        out["sii"][i], out["mui"][i], out["t_old"][i], out["n_old"][i] = sii, mui, tau[i], nu[i]
        out["sii_scale"][i], out["mui_scale"][i] = dg_scale[i], mu_scale[i]
        r = site_update(sii, mui, tau[i], nu[i], yv[i], dtype)
        out["cav_tau"][i], out["cav_nu"][i], out["c"][i], out["g"][i] = r["ct"], r["cn"], r["c"], r["g"]
        tau[i], nu[i] = r["tau"], r["nu"]
        s = S[:, i].copy()
        if keep_columns:
            cols[:, i] = s
        S -= np.outer(s, s) * r["c"]
        mu += s * r["g"]
        mu_scale += np.abs(s * r["g"]).astype(LD)
        dg_scale += (np.abs(r["c"]) * s * s).astype(LD)
    out.update(tau=tau, nu=nu, mu=mu, mu_scale=mu_scale, Sigma=S)
    if keep_columns:
        out["S"] = cols
    return out


def loop_bound(ld, f64, y, n, fast):
    """Per-output bounds of a site loop (dicts of site_loop in longdouble and float64): LOOP_FACTOR |f64 - ld| plus the site
    update's own bound (fast: ep_sites_block_p's, else ep_sites_block_w's) at the reference's inputs sii, mui, which carry the
    floor FLOOR n u (sii_scale, mui_scale) of the downdates that formed them; mu: LOOP_FACTOR |f64 - ld| + FLOOR n u mu_scale."""
    e_sii, e_mui = FLOOR * n * U * ld["sii_scale"], FLOOR * n * U * ld["mui_scale"]
    sb = site_bound(ld["sii"], ld["mui"], ld["t_old"], ld["n_old"], np.asarray(y, dtype=LD), fast, e_sii, e_mui)
    own = dict(tau=sb["tau"] if fast else sb["dtau"] + U * np.abs(ld["tau"]), nu=sb["nu"], cav_tau=sb["ct"], cav_nu=sb["cn"],
               c=sb["c"], g=sb["g"], mu=FLOOR * n * U * ld["mu_scale"])
    return {k: LOOP_FACTOR * np.abs(f64[k].astype(LD) - ld[k]) + own[k] for k in own}


# ---------------------------------------------------------------------------------------------------------------------------
# the posterior re-factorisation (EpParameterEstimator.scala:56-61)
# ---------------------------------------------------------------------------------------------------------------------------
def cholesky(A):
    """Lower Cholesky factor in A's dtype (right-looking, column by column)."""
    A = np.array(A)
    n = A.shape[0]
    L = np.zeros_like(A)
    for k in range(n):
        d = np.sqrt(A[k, k])
        L[k, k] = d
        L[k + 1:, k] = A[k + 1:, k] / d
        A[k + 1:, k + 1:] -= np.outer(L[k + 1:, k], L[k + 1:, k])
    return L


def forward_solve(L, B):
    X = np.array(B)
    for i in range(L.shape[0]):
        X[i] = (X[i] - L[i, :i] @ X[:i]) / L[i, i]
    return X


def refactor(K, tau, nu, dtype=LD):
    """B = I + S^1/2 K S^1/2 = L L^t, V = L^-1 S^1/2 K, Sigma = K - V^t V, mu = Sigma nu, in dtype.  float64 goes through LAPACK
    (numpy), longdouble through the loops above.  Returns dict(L, Sigma, mu, V)."""
    K = np.asarray(K, dtype=dtype)
    st = np.sqrt(np.asarray(tau, dtype=dtype))
    B = np.eye(K.shape[0], dtype=dtype) + (st[:, None] * st[None, :]) * K
    SK = st[:, None] * K
    if dtype == np.float64:
        import scipy.linalg as sl
        L = np.linalg.cholesky(B)
        V = sl.solve_triangular(L, SK, lower=True)
    else:
        L = cholesky(B)
        V = forward_solve(L, SK)
    Sigma = K - V.T @ V
    mu = Sigma @ np.asarray(nu, dtype=dtype)
    return dict(L=L, Sigma=Sigma, mu=mu, V=V)


def refactor_bounds(ld, f64, K, nu):
    """LOOP_FACTOR |f64 - ld| + FLOOR n u scale; scales: sqrt(B_ii) for row i of L, |K| + |V|^t |V| for Sigma, and that times
    |nu| for mu."""
    n = K.shape[0]
    aV = np.abs(ld["V"])
    sS = np.abs(K.astype(LD)) + aV.T @ aV
    sL = np.sqrt(np.diag(ld["L"] @ ld["L"].T))[:, None] * np.ones((1, n), dtype=LD)
    smu = sS @ np.abs(np.asarray(nu, dtype=LD))
    return dict(L=LOOP_FACTOR * np.abs(f64["L"] - ld["L"]) + FLOOR * n * U * sL,
                Sigma=LOOP_FACTOR * np.abs(f64["Sigma"] - ld["Sigma"]) + FLOOR * n * U * sS,
                mu=LOOP_FACTOR * np.abs(f64["mu"] - ld["mu"]) + FLOOR * n * U * smu)
