"""Plain high-precision references of the evaluation's kernels (covariance build, gradient trace) for
tests/test_gpu_eval_kernels.py.  NumPy `longdouble` (64-bit significand: 2^11 times the precision of a double); never the
oracle.  tests/test_eval_refs.py checks them against mpmath at 50 digits and against the oracle on the CPU."""
import numpy as np

LD = np.longdouble
PI = LD("3.14159265358979323846264338327950288")
CO2_NPARAMS = 11


# ---------------------------------------------------------------------------------------------------------------------------
# SE-ARD: k = sf^2 exp(-r/2) + sn^2 [i == j],  r = sum_d (x_d - x'_d)^2 / l_d^2,  theta = [sf, l_1..l_D, sn]
# ---------------------------------------------------------------------------------------------------------------------------
def se_ard_inv_ls2(theta):
    """1 / (l_d * l_d) in float64, as the host computes the kernel's arguments."""
    ls = np.asarray(theta[1:-1], dtype=np.float64)
    return 1.0 / (ls * ls)


def se_ard_r64(X1, X2, inv_ls2):
    """r_ij in float64 with cov_se_ard_kernel's association: ((x1_id - x2_jd) * inv_d) * (x1_id - x2_jd), unfused, summed in
    order over d (NumPy rounds every operation on its own)."""
    r = np.zeros((X1.shape[0], X2.shape[0]))
    for d in range(X1.shape[1]):
        f = X1[:, d, None] - X2[None, :, d]
        r = r + (f * inv_ls2[d]) * f
    return r


def se_ard_value_from_r(r64, theta):
    """sf^2 exp(-r/2) for a given float64 r, with sf^2 rounded to float64 as the kernel's argument is."""
    sf2 = LD(float(theta[0]) * float(theta[0]))
    return sf2 * np.exp(-r64.astype(LD) / 2)


def se_ard_terms(X1, X2, theta):
    """Exact-input terms in longdouble: (r, e = exp(-r/2), [f_d^2]) for every pair (rows of X1) x (rows of X2)."""
    A, B = np.asarray(X1, dtype=LD), np.asarray(X2, dtype=LD)
    ls = np.asarray(theta[1:-1], dtype=LD)
    f2 = [(A[:, d, None] - B[None, :, d]) ** 2 for d in range(A.shape[1])]
    r = sum(f2[d] / (ls[d] * ls[d]) for d in range(len(f2)))
    return r, np.exp(-r / 2), f2


def se_ard_dk(X1, X2, theta, same_index):
    """The true derivatives dk/dtheta_p (p = 0..D+1) as longdouble arrays: 2 sf e, sf^2 e f_d^2 / l_d^3, 2 sn [i == j]."""
    D = len(theta) - 2
    sf, ls, sn = LD(theta[0]), np.asarray(theta[1:-1], dtype=LD), LD(theta[-1])
    r, e, f2 = se_ard_terms(X1, X2, theta)
    out = [2 * sf * e] + [sf * sf * e * f2[d] / ls[d] ** 3 for d in range(D)]
    out.append(np.where(same_index, 2 * sn, LD(0)))
    return out, r


# ---------------------------------------------------------------------------------------------------------------------------
# Co2Kernel (Co2Prediction.scala:38-56), 1-D inputs, hp = hp1..hp11, on the float64 difference xd = x1 - x2
# ---------------------------------------------------------------------------------------------------------------------------
def co2_parts(xd, hp):
    """Value terms, true derivatives dk/dhp_1..10 and the magnitudes an FP64 evaluation is conditioned by, in longdouble.
    Returns (k without noise, [dk_1..dk_10], [|dk_p| as evaluated], cond): cond = 1 + the sum of the exponent / power
    arguments + the sensitivity to rounding pi * xd (4 pi |xd| / hp5^2), so that a double evaluation of k or dk_p has error
    O(u) * cond * k resp. * |dk_p| as evaluated.  The latter differs from |dk_p| in two places.  dk/dhp5 = k2 4 s^2 / hp5^3
    with s = sin(pi xd): the rounding of pi * xd (u pi |xd| absolute) is relative to s, which vanishes at integer xd (whole
    years of the Mauna Loa data), so it is k2 4 (s^2 + 2 |s| pi |xd|) / hp5^3.  dk/dhp8 = k3 (-log p1 + sq / (...)): the two
    terms cancel at small xd and log p1 carries the rounding of p1 = 1 + ... (an absolute u), so it is
    k3 (1 + log p1 + sq / (...))."""
    x = np.asarray(xd, dtype=LD)
    h = [LD(v) for v in hp]
    h1, h2, h3, h4, h5, h6, h7, h8, h9, h10 = h[:10]
    sq = x * x
    a1 = sq / (2 * h2 * h2)
    e1 = np.exp(-a1)
    s = np.sin(PI * x)
    a2 = sq / (2 * h4 * h4) + 2 * s * s / (h5 * h5)
    k2 = h3 * h3 * np.exp(-a2)
    p1 = 1 + sq / (2 * h8 * h7 * h7)
    lg = np.log(p1)
    pw = np.exp(-h8 * lg)
    k3 = h6 * h6 * pw
    a4 = sq / (2 * h10 * h10)
    k4 = h9 * h9 * np.exp(-a4)
    k = h1 * h1 * e1 + k2 + k3 + k4
    dk = [2 * h1 * e1,
          h1 * h1 * e1 * sq / h2 ** 3,
          2 * k2 / h3,
          k2 * sq / h4 ** 3,
          k2 * 4 * s * s / h5 ** 3,
          2 * h6 * pw,
          h6 * h6 * pw / p1 * sq / h7 ** 3,
          k3 * (-lg + sq / (2 * h7 * h7 * h8 * p1)),
          2 * k4 / h9,
          k4 * sq / h10 ** 3]
    mag = [np.abs(v) for v in dk]
    mag[4] = k2 * 4 * (s * s + 2 * np.abs(s) * PI * np.abs(x)) / h5 ** 3
    mag[7] = k3 * (1 + lg + sq / (2 * h7 * h7 * h8 * p1))
    cond = 1 + a1 + a2 + h8 * lg + a4 + 4 * PI * np.abs(x) / (h5 * h5)
    return k, dk, mag, cond


def co2_value_diag(hp):
    """k(x, x) without noise as the host rounds it: ((hp1^2 + hp3^2) + hp6^2) + hp9^2 in float64."""
    hp = [float(v) for v in hp]
    return ((hp[0] * hp[0] + hp[2] * hp[2]) + hp[5] * hp[5]) + hp[8] * hp[8]


# ---------------------------------------------------------------------------------------------------------------------------
# gradient trace: g_p = 1/2 sum_{i,j<n} W_ij dk_p(x_i, x_j, i == j),  W = alpha alpha^t - Kinv, over the full square
# ---------------------------------------------------------------------------------------------------------------------------
def grad_trace_ref(X, alpha, Kinv, theta, nparams, co2=False, rows=None, block=512):
    """Returns (g, s0, s1) as float64 arrays of length nparams, summed in longdouble:
        g  = 1/2 sum_ij W_ij dk_p
        s0 = 1/2 sum_ij (|alpha_i alpha_j| + |Kinv_ij|) |dk_p|
        s1 = 1/2 sum_ij (|alpha_i alpha_j| + |Kinv_ij|) |dk_p| c_ij,  c_ij = r_ij / 2 (SE-ARD) or the Co2 conditioning - 1
    (|dk_p| as evaluated, see co2_parts).
    Kinv: full symmetric n x n float64 array, or None (W = alpha alpha^t).  rows: restrict i and j to these indices (alpha
    must vanish elsewhere and Kinv be None)."""
    X = np.asarray(X, dtype=np.float64)
    idx = np.arange(X.shape[0]) if rows is None else np.asarray(rows)
    a = np.asarray(alpha, dtype=np.float64)[idx]
    g, s0, s1 = (np.zeros(nparams, dtype=LD) for _ in range(3))
    for b0 in range(0, len(idx), block):
        bi = idx[b0:b0 + block]
        ab = a[b0:b0 + block]
        aa = ab[:, None].astype(LD) * a[None, :].astype(LD)
        mag = np.abs(aa)
        W = aa
        if Kinv is not None:
            Kb = Kinv[np.ix_(bi, idx)].astype(LD)
            W = aa - Kb
            mag = mag + np.abs(Kb)
        same = bi[:, None] == idx[None, :]
        if co2:
            xd = X[bi, 0][:, None] - X[idx, 0][None, :]          # the kernel's float64 difference
            _, dk, mag_dk, cond = co2_parts(xd, theta)
            dk = dk + [np.where(same, 2 * LD(theta[10]), LD(0))]
            mag_dk = mag_dk + [np.abs(dk[10])]
            c = cond - 1
        else:
            dk, r = se_ard_dk(X[bi], X[idx], theta, same)
            mag_dk = [np.abs(v) for v in dk]
            c = r / 2
        for p in range(nparams):
            g[p] += np.sum(W * dk[p])
            t = mag * mag_dk[p]
            s0[p] += np.sum(t)
            s1[p] += np.sum(t * c)
    return (g / 2).astype(np.float64), (s0 / 2).astype(np.float64), (s1 / 2).astype(np.float64)
