"""GPU: the kernels of the EP sweep (csrc/gpk_ep.cu), one routine at a time, against plain high-precision references
(tests/ep_refs.py: NumPy longdouble and mpmath; never the oracle), within the bounds derived there.

- scalar primitives of the site kernels (gpk_debug_ep_scalar): rcp_nr correctly rounded, rsqrt_nr against libdevice rsqrt,
  exp_neg_sq, the erfcx table and phi/Phi at the table's interval ends, the rounding ties of its index and the switch to
  libdevice, and both scalar site updates;
- the site kernels ep_sites_block_p (5) and ep_sites_block_w (4) on one block (gpk_debug_ep_sites): site parameters, c, g and
  W = (I + A)^-1 against the sequential site loop, with NaN wherever they must not read and sentinels where they must not write;
- the apply kernel (gpk_debug_ep_apply): U = X W, P = U diag(c) bit for bit, mu += U g, Dg[jb] -= P U^t for jb > b only;
- the site loop of a whole sweep with the paired flush on four streams (gpk_debug_ep_site_loop), every row of every output;
- the re-factorisation (gpk_debug_ep_refactor) on its small, pipelined and nb = 512 paths.
"""
import math
from fractions import Fraction

import numpy as np
import pytest

from tests import ep_refs as R

pytestmark = pytest.mark.gpu

U = 2.0 ** -53
LD = np.longdouble
EB = 64
SENT = -777.25
NAN = float("nan")
RCP, RSQRT, EXP_NEG_SQ, ERFCX_TAB, RATIO, RATIO_FAST, SITE_FAST, SITE_SCALAR = range(8)


@pytest.fixture(scope="module")
def h():
    from gp_algos_b200 import _lib
    hd = _lib.Handle(0)
    yield hd
    hd.close()


def _dev(a, dtype=None):
    import torch
    return torch.from_numpy(np.ascontiguousarray(a, dtype=dtype)).cuda()


def _host(t):
    return t.cpu().numpy()


def _run(h, fn):
    import torch
    torch.cuda.synchronize()
    h.check(fn())
    h.synchronize()


def _pad128(n):
    return (n + 127) // 128 * 128


def _scalar(h, what, x, per_in=1, per_out=1):
    x = np.ascontiguousarray(x, dtype=np.float64).ravel()
    count = len(x) // per_in
    out, dx = _dev(np.full(count * per_out, SENT)), _dev(x)
    _run(h, lambda: h.lib.gpk_debug_ep_scalar(h.h, what, dx.data_ptr(), count, out.data_ptr()))
    return _host(out).reshape(count, per_out) if per_out > 1 else _host(out)


def _within(got, ref, bound, what, inputs=None):
    """|got - ref| <= bound elementwise (got finite); the message names the worst element relative to its bound."""
    err = np.abs(np.asarray(got).astype(LD) - ref)
    ok = np.isfinite(got) & (err <= bound)
    if not np.all(ok):
        r = np.where(ok, 0, err / np.maximum(bound, LD(1e-300)))
        i = int(np.argmax(np.where(np.isnan(r), np.inf, r)))
        raise AssertionError(f"{what}: {np.count_nonzero(~ok)} of {ok.size} outside the bound; worst index {i}: got "
                             f"{float(np.ravel(got)[i])!r}, ref {float(np.ravel(ref)[i])!r}, bound {float(np.ravel(bound)[i]):.3g}"
                             + ("" if inputs is None else f", inputs {inputs[i]}"))


def _neighbours(v):
    v = np.asarray(v, dtype=np.float64)
    return np.concatenate([v, np.nextafter(v, np.inf), np.nextafter(v, -np.inf)])


# =========================================================================================================================
# scalar primitives
# =========================================================================================================================
def test_rcp_nr_is_correctly_rounded(h):
    rng = np.random.default_rng(1)
    pw = 2.0 ** np.arange(-1021, 1022)
    x = np.concatenate([2.0 ** rng.uniform(-1021, 1021.9, 20000), _neighbours(pw)])
    x = x[(x >= 2.0 ** -1022) & (x < 2.0 ** 1022)]                   # positive normal with a normal reciprocal
    got = _scalar(h, RCP, x)
    ref = np.array([float(Fraction(1) / Fraction(v)) for v in x])    # int / int true division: correctly rounded
    # x = 2^k (1 - 2^-53), the last double below a power of two: 1/x = 2^-k (1 + 2^-53 + 2^-106) lies 2^-106 above the midpoint
    # of two doubles, and the last Newton step fma(y, 1 - x y, y) from y = 2^-k lands on the midpoint and rounds to even,
    # one ulp below the correctly rounded 2^-k (1 + 2^-52).  Everywhere else rcp_nr is correctly rounded.
    below_pow2 = np.nextafter(2.0 ** np.round(np.log2(x)), 0) == x
    bad = np.flatnonzero((got != ref) & ~below_pow2)
    assert bad.size == 0, (bad.size, x[bad[:4]], got[bad[:4]], ref[bad[:4]])
    e = below_pow2
    assert np.all((got[e] == ref[e]) | (got[e] == np.nextafter(ref[e], 0))), "more than one ulp from 1/x below a power of two"


def test_rsqrt_nr_equals_libdevice_rsqrt(h):
    rng = np.random.default_rng(2)
    x = np.concatenate([2.0 ** rng.uniform(-1000, 1000, 20000), 10.0 ** rng.uniform(-6, 6, 20000),
                        _neighbours(2.0 ** np.arange(-1000, 1001)), _neighbours(4.0 ** np.arange(-500, 501))])
    out = _scalar(h, RSQRT, x, 1, 2)
    nr, lib = out[:, 0], out[:, 1]
    ulps = np.abs(nr.view(np.int64) - lib.view(np.int64))
    assert ulps.max() == 0, f"rsqrt_nr differs from libdevice rsqrt in {np.count_nonzero(ulps)} of {len(x)} inputs, " \
                            f"by up to {ulps.max()} ulp (x = {x[np.argmax(ulps)]!r})"


def _mp_rel(got, ref_mp):
    """|got / ref - 1| in longdouble for mpmath references."""
    return np.array([abs(float((LD(g) - R._from_mp(r)) / R._from_mp(r))) for g, r in zip(got, ref_mp)])


def test_exp_neg_sq_within_bound(h):
    import mpmath as mp
    rng = np.random.default_rng(3)
    k = np.arange(0, 93)
    edges = np.sqrt(k * math.log(2.0))                                 # exp(-ax^2) = 2^-k: the exponent of the result changes
    x = np.concatenate([[0.0, np.nextafter(8.0, 0)], rng.uniform(0, 8, 4000), _neighbours(edges)])
    x = x[(x >= 0) & (x < 8)]
    got = _scalar(h, EXP_NEG_SQ, x)
    with mp.workdps(40):
        ref = [mp.exp(-mp.mpf(v) ** 2) for v in x]
    rel = _mp_rel(got, ref)
    # the polynomial's 4.4e-16 (header) + 2u for the reduction and the evaluation's last rounding
    assert rel.max() <= 4.4e-16 + 2 * U, (x[np.argmax(rel)], rel.max())


def _table_points():
    k = np.arange(0, 65) / 8.0
    ends = np.concatenate([k[:-1], np.nextafter(k[1:], 0)])            # both ends of every interval [i/8, (i+1)/8)
    return np.unique(np.concatenate([ends, _neighbours(k), [0.0, 8.0, np.nextafter(8.0, 0), 5e-324, 1e-300]]))


def test_erfcx_tab_at_interval_ends_ties_and_switch(h):
    import mpmath as mp
    x = _table_points()
    x = x[x >= 0]
    x = np.concatenate([x, np.linspace(8, 28.3, 200)])                 # libdevice route, |z| out to 40
    got = _scalar(h, ERFCX_TAB, x)
    ref = [R.erfcx_mp(v) for v in x]
    rel = _mp_rel(got, ref)
    # table: 4.4e-16 fit + the evaluation's rounding (6e-16 in the CPU test's float64 evaluation) + 2u; libdevice erfcx: 4u
    tol = np.where(x < 8, 6e-16 + 2 * U, 4 * U)
    assert np.all(rel <= tol), (x[np.argmax(rel / tol)], (rel / tol).max())


def _z_for_x(ax):
    """z values with fl(z * -1/sqrt2) = +-ax exactly (so that the kernel's |x| is the table point), both signs of z."""
    c = -0.70710678118654752440
    out = []
    for a in ax:
        for xt in (a, -a):
            z0 = xt / c
            cand = [z0]
            up, dn = z0, z0
            for _ in range(4):
                up, dn = np.nextafter(up, np.inf), np.nextafter(dn, -np.inf)
                cand += [up, dn]
            hit = [z for z in cand if z * c == xt]
            if hit:
                out.append(hit[0])
    return np.array(out)


@pytest.mark.parametrize("what", [RATIO_FAST, RATIO])
def test_dnorm_over_pnorm_within_bound(h, what):
    x = _table_points()
    zt = _z_for_x(x)
    assert len(zt) >= 1.5 * len(x)                                     # most table points hit exactly, from both sides
    z = np.concatenate([zt, [0.0, -0.0, 5e-324, -5e-324, 1e-300, -1e-300],
                        np.linspace(-40, 40, 801), np.linspace(-11.4, -11.2, 41), np.linspace(11.2, 11.4, 41)])
    got = _scalar(h, what, z)
    ref = R.ratio(z)
    # relative bound, plus 4 subnormal ulps where phi/Phi underflows (z > 37.5: exp(-z^2/2) is subnormal)
    _within(got, ref, R.ratio_rel_err(z, True) * np.abs(ref) + LD(4 * 5e-324), "phi/Phi", z)


def _site_cases(rng, m=3000):
    """First sweeps (t_old = 0), later sweeps with den = 1 - t_old sii down to 1e-6, sii in [1e-6, 1e3], y = +-1, |z| out to
    about 30 (beyond the table's 11.3)."""
    sii = 10.0 ** rng.uniform(-6, 3, m)
    first = rng.random(m) < 0.3
    den = np.where(first, 1.0, 10.0 ** rng.uniform(-6, 0, m))
    t_old = np.where(first, 0.0, (1 - den) / sii)
    zt = np.where(rng.random(m) < 0.2, rng.uniform(-30, 30, m), rng.normal(0, 2, m))     # target |z|
    # z = y cmu / sqrt(1 + csig), cmu = (mui - n_old sii) / den, csig = sii / den
    n_old = np.where(first, 0.0, rng.normal(0, 1, m) * t_old)
    y = rng.choice([-1.0, 1.0], m)
    mui = zt * np.sqrt(1 + sii / den) * den * y + n_old * sii
    return sii, mui, t_old, n_old, y


@pytest.mark.parametrize("fast", [True, False])
def test_site_updates_within_bound(h, fast):
    rng = np.random.default_rng(4)
    sii, mui, t_old, n_old, y = _site_cases(rng)
    inp = np.stack([sii, mui, t_old, n_old, y], axis=1)
    ref = R.site_update_mp(sii, mui, t_old, n_old, y)
    assert np.max(np.abs(ref["z"].astype(float))) > 20
    bnd = R.site_bound(sii, mui, t_old, n_old, y, fast)
    if fast:
        out = _scalar(h, SITE_FAST, inp, 5, 9)
        names = ["c", "g", "mu_hat", "sig_hat", "rs", "ct", "cn", "tau", "nu"]
        assert np.array_equal(out[:, 4], np.array([float(Fraction(1) / Fraction(v)) for v in sii]))    # rs = rcp_nr(sii)
    else:
        out = _scalar(h, SITE_SCALAR, inp, 5, 6)
        names = ["ct", "cn", "c", "g", "dtau", "nu"]
    for j, k in enumerate(names):
        if k != "rs":
            _within(out[:, j], ref[k], bnd[k], k, inp)


# =========================================================================================================================
# site kernels on one block
# =========================================================================================================================
def _se_block(n, signal=1.0, seed=0, jitter=1e-3, span=None):
    """SE kernel (length scale 1) on n sorted points: neighbours ~0.08 apart (rho > 0.99), or spread over [0, span] (every pair
    correlated: exp(-span^2 / 2) at the ends)."""
    rng = np.random.default_rng(seed)
    x = np.sort(rng.uniform(0, 0.08 * n if span is None else span, n))
    return signal ** 2 * np.exp(-0.5 * (x[:, None] - x[None, :]) ** 2) + jitter * np.eye(n)


def _targets(n, seed=0):
    rng = np.random.default_rng(seed + 1)
    return rng.choice(np.array([-1, 1], dtype=np.int32), n)


def _state(K, y, later):
    """(Sigma, tau, nu, mu) in float64: the first sweep's (K, 0, 0, 0) or the state after the reference's own first sweep and
    re-factorisation (Sigma = (K^-1 + S)^-1, mu = Sigma nu), Sigma symmetric from its lower triangle."""
    n = K.shape[0]
    z = np.zeros(n)
    if not later:
        return K.copy(), z, z, z
    s1 = R.site_loop(K, z, z, z, y)
    rf = R.refactor(K, s1["tau"], s1["nu"])
    S = np.tril(rf["Sigma"].astype(np.float64))
    S = S + np.tril(S, -1).T
    return S, s1["tau"].astype(np.float64), s1["nu"].astype(np.float64), rf["mu"].astype(np.float64)


_BLOCK_STATES = {"first": (1.0, False), "later": (1.0, True), "signal40": (40.0, False)}


@pytest.fixture(scope="module")
def block_refs():
    cache = {}

    def get(state, bsz):
        key = (state, bsz)
        if key not in cache:
            if state not in cache:
                signal, later = _BLOCK_STATES[state]
                y = _targets(EB, 5)
                cache[state] = _state(_se_block(EB, signal, 5), y, later) + (y,)
            S, tau, nu, mu, y = cache[state]
            S, tau, nu, mu, y = S[:bsz, :bsz], tau[:bsz], nu[:bsz], mu[:bsz], y[:bsz]
            ld = R.site_loop(S, tau, nu, mu, y, keep_columns=True)
            f64 = R.site_loop(S, tau, nu, mu, y, dtype=np.float64, keep_columns=True)
            cache[key] = (S, tau, nu, mu, y, ld, f64)
        return cache[key]
    return get


def _w_of(c, cols):
    """W = (I + A)^-1 with a_lk = c_l s_l[k] (l < k) in the dtype of c."""
    n = len(c)
    A = np.triu(c[:, None] * cols.T, 1)
    I = np.eye(n, dtype=A.dtype)
    return np.linalg.inv(I + A) if A.dtype == np.float64 else _inv_unit_upper(I + A), A


def _inv_unit_upper(T):
    n = T.shape[0]
    W = np.eye(n, dtype=T.dtype)
    for k in range(n):
        for j in range(k):
            W[j, k] = -(W[j, j:k] @ T[j:k, k])
    return W


@pytest.mark.parametrize("variant", [5, 4])
@pytest.mark.parametrize("state", ["first", "later", "signal40"])
@pytest.mark.parametrize("bsz", [1, 2, 3, 8, 9, 31, 32, 33, 63, 64])
def test_site_kernel_one_block(h, block_refs, variant, state, bsz):
    S, tau, nu, mu, y, ld, f64 = block_refs(state, bsz)
    bound = R.loop_bound(ld, f64, y, bsz, variant == 5)
    Dg = np.full((EB, EB), NAN)
    Dg[:bsz, :bsz] = S
    Wl, Al = _w_of(ld["c"], ld["S"])
    W64, _ = _w_of(f64["c"], f64["S"])
    IA = np.abs(np.eye(bsz, dtype=LD) + Al)
    wb = R.LOOP_FACTOR * np.abs(W64 - Wl) + R.FLOOR * bsz * U * (np.abs(Wl) @ IA @ np.abs(Wl))
    for i0 in (0, 64, 192):
        L = i0 + EB + 64
        vec = lambda v: _dev(np.concatenate([np.full(i0, NAN), v, np.full(L - i0 - bsz, NAN)]))
        dmu, dtau, dnu = vec(mu), vec(tau), vec(nu)
        dct, dcn = _dev(np.full(L, SENT)), _dev(np.full(L, SENT))
        yy = np.full(L, 7, dtype=np.int32); yy[i0:i0 + bsz] = y
        dy = _dev(yy)
        dblk, dW, dDg = _dev(np.full(2 * EB, SENT)), _dev(np.full(EB * EB, SENT)), _dev(Dg.T.copy())
        _run(h, lambda: h.lib.gpk_debug_ep_sites(h.h, variant, dDg.data_ptr(), i0, bsz, dmu.data_ptr(), dtau.data_ptr(),
                                                 dnu.data_ptr(), dct.data_ptr(), dcn.data_ptr(), dy.data_ptr(), dblk.data_ptr(),
                                                 dW.data_ptr()))
        t, nv, ct, cn, blk = _host(dtau), _host(dnu), _host(dct), _host(dcn), _host(dblk)
        W = _host(dW).reshape(EB, EB).T                                  # column-major
        got = dict(tau=t[i0:i0 + bsz], nu=nv[i0:i0 + bsz], cav_tau=ct[i0:i0 + bsz], cav_nu=cn[i0:i0 + bsz],
                   c=blk[:bsz], g=blk[EB:EB + bsz])
        for k, v in got.items():
            _within(v, ld[k], bound[k], (k, i0))
        out = np.r_[0:i0, i0 + bsz:L]
        assert np.all(np.isnan(t[out])) and np.all(np.isnan(nv[out])), "tau / nu written outside the block"
        assert np.all(ct[out] == SENT) and np.all(cn[out] == SENT), "cavities written outside the block"
        assert np.all(blk[bsz:EB] == 0) and np.all(blk[EB + bsz:] == 0)
        assert np.all(np.diag(W) == 1) and np.all(np.tril(W, -1) == 0)
        Wo = W.copy(); Wo[:bsz, :bsz] = np.eye(bsz)
        assert np.array_equal(Wo, np.eye(EB)), "W is not the identity outside the block"
        Wk = W[:bsz, :bsz]
        assert np.all(np.abs(Wk.astype(LD) - Wl) <= wb), ("W", i0, float(np.max(np.abs(Wk - Wl.astype(float)) / wb.astype(float))))
        # W (I + A) = I with the kernel's own coefficients c (update vectors of the reference)
        # (the kernel's update vectors differ from the reference's by the loop's rounding: the |W| |c_kernel - c_ref| |s| term)
        Ak = np.triu(blk[:bsz].astype(LD)[:, None] * ld["S"].T, 1)
        dA = np.triu(np.abs(blk[:bsz].astype(LD) - ld["c"])[:, None] * np.abs(ld["S"].T), 1) + np.abs(Ak) * bound["c"][:, None] / \
            np.maximum(np.abs(ld["c"]), LD(1e-300))[:, None]
        res = Wk.astype(LD) @ (np.eye(bsz, dtype=LD) + Ak) - np.eye(bsz, dtype=LD)
        aW = np.abs(Wk).astype(LD)
        _within(res, np.zeros_like(res), R.FLOOR * bsz * U * (aW @ np.abs(np.eye(bsz, dtype=LD) + Ak)) + aW @ dA, ("W (I + A) - I", i0))


# =========================================================================================================================
# apply kernel
# =========================================================================================================================
@pytest.mark.parametrize("n,b", [(256, 0), (256, 1), (256, 3), (300, 0), (300, 1), (300, 4), (129, 2), (65, 1)])
def test_apply_kernel(h, n, b):
    rng = np.random.default_rng(n * 10 + b)
    N = _pad128(n)
    nblk = (n + EB - 1) // EB
    i0 = b * EB
    bsz = min(EB, n - i0)
    K = _se_block(N, 1.0, n)
    Sig = np.tril(K)
    Sig[np.triu_indices(N, 1)] = NAN
    Sig[i0:i0 + EB, i0:i0 + EB] = NAN                                   # tile (b, b) comes from Dg[b]
    Dg = rng.standard_normal((N // EB, EB, EB))
    Dg = Dg + Dg.transpose(0, 2, 1)
    c = np.zeros(EB); g = np.zeros(EB)
    c[:bsz] = rng.uniform(0.1, 1.0, bsz); g[:bsz] = rng.standard_normal(bsz)
    W = np.eye(EB)
    W[:bsz, :bsz] += np.triu(rng.standard_normal((bsz, bsz)) * 0.3, 1)
    mu = np.full(N, SENT); mu[:n] = rng.standard_normal(n)
    dSig = _dev(Sig.T.copy().ravel())
    dDg = _dev(Dg.transpose(0, 2, 1).copy().ravel())                   # column-major blocks
    dblk, dW = _dev(np.concatenate([c, g])), _dev(W.T.copy().ravel())
    dU, dP, dmu = _dev(np.full(N * EB, SENT)), _dev(np.full(N * EB, SENT)), _dev(mu)
    _run(h, lambda: h.lib.gpk_debug_ep_apply(h.h, dSig.data_ptr(), N, n, b, bsz, dblk.data_ptr(), dW.data_ptr(), dU.data_ptr(),
                                             dP.data_ptr(), dmu.data_ptr(), dDg.data_ptr()))
    Uk = _host(dU).reshape(EB, N).T
    Pk = _host(dP).reshape(EB, N).T
    mk = _host(dmu)
    Dk = _host(dDg).reshape(N // EB, EB, EB).transpose(0, 2, 1)
    # X = Sigma0[:, block b] through the lower triangle, the block's own rows from Dg[b]
    Kf = np.tril(K) + np.tril(K, -1).T
    X = Kf[:, i0:i0 + EB].copy()
    X[i0:i0 + EB] = Dg[b]
    X[n:] = 0; X[:, bsz:] = 0
    ref = X.astype(LD) @ W.astype(LD)
    assert np.all(np.abs(Uk.astype(LD) - ref) <= R.gamma(EB) * (np.abs(X) @ np.abs(W))), "U != X W"
    assert np.all(Uk[n:] == 0) and np.all(Uk[:, bsz:] == 0) and np.all(Pk[n:] == 0) and np.all(Pk[:, bsz:] == 0)
    assert np.array_equal(Pk, Uk * c[None, :]), "P != fl(U c)"
    mref = mu[:n].astype(LD) + Uk[:n].astype(LD) @ g.astype(LD)
    assert np.all(np.abs(mk[:n] - mref) <= R.gamma(EB + 1) * (np.abs(mu[:n]) + np.abs(Uk[:n]) @ np.abs(g)))
    assert np.all(mk[n:] == SENT), "mu written beyond n"
    for jb in range(N // EB):
        if jb <= b:
            assert np.array_equal(Dk[jb], Dg[jb]), f"Dg[{jb}] changed (jb <= b)"
        else:
            Pj, Uj = Pk[jb * EB:(jb + 1) * EB], Uk[jb * EB:(jb + 1) * EB]
            dref = Dg[jb].astype(LD) - Pj.astype(LD) @ Uj.T.astype(LD)
            tol = R.gamma(EB + 1) * (np.abs(Dg[jb]) + np.abs(Pj) @ np.abs(Uj).T)
            assert np.all(np.abs(Dk[jb] - dref) <= tol), f"Dg[{jb}] != Dg - P U^t"
    assert nblk <= N // EB


# =========================================================================================================================
# site loop of one sweep (site kernel, apply, paired flush on four streams)
# =========================================================================================================================
LOOP_NS = [1, 37, 64, 65, 127, 128, 129, 192, 193, 256, 300, 320, 385, 449, 700]


@pytest.fixture(scope="module")
def loop_refs():
    cache = {}

    def get(n, later):
        if (n, later) not in cache:
            K = _se_block(n, 1.0, 100 + n, span=3.0)                  # every block moves every later site
            y = _targets(n, 100 + n)
            S, tau, nu, mu = _state(K, y, later)
            ld = R.site_loop(S, tau, nu, mu, y)
            f64 = R.site_loop(S, tau, nu, mu, y, dtype=np.float64)
            cache[(n, later)] = (S, tau, nu, mu, y, ld, f64)
        return cache[(n, later)]
    return get


@pytest.mark.parametrize("variant", ["5", "4"])
@pytest.mark.parametrize("later", [False, True])
@pytest.mark.parametrize("n", LOOP_NS)
def test_site_loop_paired_flush(h, loop_refs, monkeypatch, variant, later, n):
    monkeypatch.setenv("GPK_EP_SITES", variant)
    S, tau, nu, mu, y, ld, f64 = loop_refs(n, later)
    N = _pad128(n)
    Sig = np.full((N, N), NAN)
    Sig[:n, :n] = np.tril(S)
    Sig[np.triu_indices(N, 1)] = NAN
    dS = _dev(Sig.T.copy().ravel())
    ins = [_dev(v) for v in (tau, nu, mu)] + [_dev(y.astype(np.int32))]

    def run():
        outs = [_dev(np.full(n, SENT)) for _ in range(5)]
        _run(h, lambda: h.lib.gpk_debug_ep_site_loop(h.h, dS.data_ptr(), n, *[t.data_ptr() for t in ins],
                                                     *[t.data_ptr() for t in outs]))
        return [_host(t) for t in outs]
    got = run()
    bound = R.loop_bound(ld, f64, y, n, variant == "5")
    for k, v in zip(("tau", "nu", "mu", "cav_tau", "cav_nu"), got):
        _within(v, ld[k], bound[k], k)
    again = run()
    assert all(np.array_equal(a, b) for a, b in zip(got, again)), "second identical call not bit-identical"


# =========================================================================================================================
# re-factorisation
# =========================================================================================================================
@pytest.mark.parametrize("n", [40, 300, 520, 1100, 4096])
def test_refactor(h, n):
    import torch
    rng = np.random.default_rng(n)
    K = _se_block(n, 1.0, 200 + n, jitter=1e-2)
    tau = rng.uniform(0.05, 1.0, n)
    nu = rng.standard_normal(n)
    N = _pad128(n)
    dL, dS, dmu = _dev(np.full(N * N, SENT)), _dev(np.full(N * N, SENT)), _dev(np.full(n, SENT))
    dK, dtau, dnu = _dev(K.T.copy().ravel()), _dev(tau), _dev(nu)         # (kept alive until the call has run)
    _run(h, lambda: h.lib.gpk_debug_ep_refactor(h.h, dK.data_ptr(), n, dtau.data_ptr(), dnu.data_ptr(), dL.data_ptr(),
                                                dS.data_ptr(), dmu.data_ptr()))
    L = _host(dL).reshape(N, N).T[:n, :n]
    Sg = _host(dS).reshape(N, N).T[:n, :n]
    mu = _host(dmu)
    low = np.tril_indices(n)
    if n <= 1100:
        ld = R.refactor(K, tau, nu)
        f64 = R.refactor(K, tau, nu, dtype=np.float64)
        b = R.refactor_bounds(ld, f64, K, nu)
        for name, v in (("L", L), ("Sigma", Sg)):
            _within(v[low], ld[name][low], b[name][low], name)
        _within(mu, ld["mu"], b["mu"], "mu")
    else:
        Sf = np.tril(Sg) + np.tril(Sg, -1).T
        Kt, St = torch.from_numpy(K).cuda(), torch.from_numpy(Sf).cuda()
        tt = torch.from_numpy(tau).cuda()
        res = St + Kt @ (tt[:, None] * St) - Kt
        mag = St.abs() + Kt.abs() @ (tt[:, None] * St.abs()) + Kt.abs()
        assert bool((res.abs() <= R.FLOOR * n * U * mag).all()), "(I + K S) Sigma != K"
        # L: B = L L^t
        Lt = torch.from_numpy(np.tril(L)).cuda()
        st = tt.sqrt()
        B = torch.eye(n, dtype=torch.float64, device="cuda") + st[:, None] * Kt * st[None, :]
        # (|L| |L|^t)_ij <= sqrt(B_ii B_jj): the per-element form of the Cholesky backward error, immune to underflow
        dB = B.diagonal().sqrt()
        assert bool(((Lt @ Lt.T - B).abs() <= R.FLOOR * n * U * (dB[:, None] * dB[None, :])).all()), "L L^t != B"
        mref = St @ torch.from_numpy(nu).cuda()
        mmag = St.abs() @ torch.from_numpy(np.abs(nu)).cuda()
        assert bool(((torch.from_numpy(mu).cuda() - mref).abs() <= R.FLOOR * n * U * mmag).all()), "mu != Sigma nu"
