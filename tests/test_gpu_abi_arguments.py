"""GPU: malformed arguments at the C ABI (include/gpk.h).  Every host-buffer entry point is called with a small table of
malformed arguments: D = 0 and D = 65, a leading dimension below its row count, n <= 0 where the entry point rejects it,
nparams out of range, a null pointer the entry point checks, and overlapping problems in a batched call.  Each call must
return GPK_EINVAL, launch nothing, leave every output buffer holding its sentinel and set a message of its own.

Every buffer passed is valid and large enough for what a call could read before rejecting (X has room for 65 columns), and
each case runs on a fresh handle, so no arena is sized yet when it starts."""
import ctypes as C

import numpy as np
import pytest

from gp_algos_b200 import _lib

pytestmark = pytest.mark.gpu

SENT, ISENT, PSENT = -777.25, -7777, 0xDEAD0
n, m, D, B = 40, 7, 3, 3
P = D + 2                      # theta length of the SE-ARD family
BIG = 1 << 16                  # doubles in every host input: > B * (n + 8) * 65

_rng = np.random.default_rng(5)
INP = _rng.random(BIG) + 0.5   # X, y, theta, K, L, tau, nu, Ks, kss: every double input reads from here
TGT = np.ones(1024, dtype=np.int32)


def p(a):
    return None if a is None else _lib.ptr(a)


class Outs:
    """Output buffers holding sentinels: doubles, ints and a gpk_model slot."""

    def __init__(self):
        self.d = {}
        self.i = {}
        self.model = C.c_void_p(PSENT)

    def __getattr__(self, name):
        if name.startswith("i_"):
            return p(self.i.setdefault(name, np.full(1024, ISENT, dtype=np.int32)))
        return p(self.d.setdefault(name, np.full(BIG, SENT)))

    def untouched(self):
        return (all(np.all(a == SENT) for a in self.d.values()) and all(np.all(a == ISENT) for a in self.i.values())
                and self.model.value == PSENT)


def fit_model(lib, h):
    """A valid resident model of n rows (its launches happen before the case is measured)."""
    X = np.asfortranarray(_rng.standard_normal((n, D)))
    y = _rng.standard_normal(n)
    th = np.array([1.0] + [0.8] * D + [0.1])
    mdl = C.c_void_p()
    assert lib.gpk_gp_model_fit(h, p(X), n, D, n, p(y), p(th), 0, 0.0, C.byref(mdl), None) == _lib.GPK_OK
    return mdl


def dev(count, fill=0.0):
    import torch
    return torch.full((count,), fill, dtype=torch.float64, device="cuda")


# entry point -> (call(lib, h, args, outs, ctx), default args, malformed cases)
X = p(INP)
ENTRIES = {
    "gpk_cov_se_ard": (
        lambda L, h, a, o, c: L.gpk_cov_se_ard(h, X, a["n"], a["D"], a["ldx"], X, o.K, a["ldk"]),
        dict(n=n, D=D, ldx=n, ldk=n),
        [dict(D=0), dict(D=65), dict(ldx=n - 1), dict(ldk=n - 1), dict(n=-1)]),
    "gpk_cov_cross_se_ard": (
        lambda L, h, a, o, c: L.gpk_cov_cross_se_ard(h, X, a["m"], a["ldx1"], X, a["n"], a["ldx2"], a["D"], X, o.K, a["ldk"]),
        dict(n=n, m=m, D=D, ldx1=m, ldx2=n, ldk=m),
        [dict(D=0), dict(D=65), dict(ldx1=m - 1), dict(ldx2=n - 1), dict(ldk=m - 1), dict(m=-1), dict(n=-1)]),
    "gpk_cov_deriv_se_ard": (
        lambda L, h, a, o, c: L.gpk_cov_deriv_se_ard(h, a["param"], X, a["n"], a["D"], a["ldx"], X, o.K, a["ldk"]),
        dict(param=1, n=n, D=D, ldx=n, ldk=n),
        [dict(D=0), dict(D=65), dict(ldx=n - 1), dict(ldk=n - 1), dict(n=-1), dict(param=0), dict(param=P + 1)]),
    "gpk_potrf_lower": (
        lambda L, h, a, o, c: L.gpk_potrf_lower(h, X, a["n"], a["lda"], o.L, a["ldl"], 1),
        dict(n=n, lda=n, ldl=n),
        [dict(lda=n - 1), dict(ldl=n - 1), dict(n=-1)]),
    "gpk_trtri": (
        lambda L, h, a, o, c: L.gpk_trtri(h, 0, X, a["n"], a["ldt"], o.Ti, a["ldi"]),
        dict(n=n, ldt=n, ldi=n),
        [dict(ldt=n - 1), dict(ldi=n - 1), dict(n=-1)]),
    "gpk_trsm": (
        lambda L, h, a, o, c: L.gpk_trsm(h, 0, 0, X, a["n"], a["ldt"], X, a["nrhs"], a["ldb"], o.X, a["ldx"]),
        dict(n=n, ldt=n, nrhs=2, ldb=n, ldx=n),
        [dict(ldt=n - 1), dict(ldb=n - 1), dict(ldx=n - 1), dict(n=-1), dict(nrhs=-1)]),
    "gpk_gp_nll_grad": (
        lambda L, h, a, o, c: L.gpk_gp_nll_grad(h, X, a["n"], a["D"], a["ldx"], X, X, 0, 0.0, a["np"], o.ll, o.grad),
        dict(n=n, D=D, ldx=n, np=P),
        [dict(D=0), dict(D=65), dict(ldx=n - 1), dict(n=0), dict(np=-1), dict(np=P + 1)]),
    "gpk_gp_nll_grad_dev": (
        lambda L, h, a, o, c: L.gpk_gp_nll_grad_dev(h, c["dX"], a["n"], a["D"], a["ldx"], c["dX"], X, 0, 0.0, a["np"],
                                                    c["dout"], None),
        dict(n=n, D=D, ldx=n, np=P),
        [dict(D=0), dict(D=65), dict(ldx=n - 1), dict(n=0), dict(np=-1), dict(np=P + 1)]),
    "gpk_gp_nll_grad_batched": (
        lambda L, h, a, o, c: L.gpk_gp_nll_grad_batched(h, a["B"], X, a["n"], a["D"], a["ldx"], a["sX"], X, X, 0, 0.0, a["np"],
                                                        o.ll, o.grad, o.i_info),
        dict(B=B, n=n, D=D, ldx=n, sX=n * D, np=P),
        [dict(D=0), dict(D=65), dict(ldx=n - 1), dict(n=0), dict(np=-1), dict(np=P + 1), dict(B=0),
         dict(sX=n * D - 1), dict(ldx=n + 2, sX=(n + 2) * (D - 1) + n - 1)]),
    "gpk_gp_nll_grad_batched_dev": (
        lambda L, h, a, o, c: L.gpk_gp_nll_grad_batched_dev(h, a["B"], c["dX"], a["n"], a["D"], a["ldx"], n * D, c["dX"], X, 0,
                                                            0.0, a["np"], c["dout"], c["dinfo"] if a["info"] else None),
        dict(B=B, n=n, D=D, ldx=n, np=P, info=True),
        [dict(info=False), dict(D=0), dict(D=65), dict(ldx=n - 1), dict(n=0), dict(np=-1), dict(np=P + 1), dict(B=0)]),
    "gpk_gp_fit": (
        lambda L, h, a, o, c: L.gpk_gp_fit(h, X, a["n"], a["D"], a["ldx"], X, X, 0, 0.0, o.L, a["ldl"], o.alpha, o.ll),
        dict(n=n, D=D, ldx=n, ldl=n),
        [dict(D=0), dict(D=65), dict(ldx=n - 1), dict(ldl=n - 1), dict(n=0)]),
    "gpk_gp_model_fit": (
        lambda L, h, a, o, c: L.gpk_gp_model_fit(h, X, a["n"], a["D"], a["ldx"], X, X, 0, 0.0,
                                                 C.byref(o.model) if a["out"] else None, o.ll),
        dict(n=n, D=D, ldx=n, out=True),
        [dict(D=0), dict(D=65), dict(ldx=n - 1), dict(n=0), dict(out=False)]),
    "gpk_gp_model_from_factor": (
        lambda L, h, a, o, c: L.gpk_gp_model_from_factor(h, X, a["n"], a["D"], a["ldx"], X, a["ldl"], X, X,
                                                         C.byref(o.model) if a["out"] else None),
        dict(n=n, D=D, ldx=n, ldl=n, out=True),
        [dict(D=0), dict(D=65), dict(ldx=n - 1), dict(ldl=n - 1), dict(n=0), dict(out=False)]),
    "gpk_gp_predict": (
        lambda L, h, a, o, c: L.gpk_gp_predict(h, X, a["n"], a["D"], a["ldx"], X, X, a["m"], a["ldxs"], X, 0, 0.0, o.mean,
                                               o.sigma, a["lds"], o.ll),
        dict(n=n, m=m, D=D, ldx=n, ldxs=m, lds=m),
        [dict(D=0), dict(D=65), dict(ldx=n - 1), dict(n=0), dict(ldxs=m - 1), dict(m=0), dict(lds=m - 1)]),
    "gpk_gp_predict_batched": (
        lambda L, h, a, o, c: L.gpk_gp_predict_batched(h, a["B"], X, a["n"], a["D"], a["ldx"], n * D, X, X, X, a["m"], a["ldxs"],
                                                       m * D, 0, 0.0, o.mean, o.var, o.ll, o.i_info),
        dict(B=B, n=n, m=m, D=D, ldx=n, ldxs=m),
        [dict(D=0), dict(D=65), dict(ldx=n - 1), dict(ldxs=m - 1), dict(n=0), dict(m=0), dict(B=0)]),
    "gpk_gp_model_predict": (
        lambda L, h, a, o, c: L.gpk_gp_model_predict(h, c["model"] if a["model"] else None, X, a["m"], a["ldxs"], 1, o.mean,
                                                     o.sigma, a["lds"], o.V, a["ldv"]),
        dict(m=m, ldxs=m, lds=m, ldv=n, model=True),
        [dict(ldxs=m - 1), dict(m=0), dict(lds=m - 1), dict(ldv=n - 1), dict(model=False)]),
    "gpk_gp_model_ucb": (
        lambda L, h, a, o, c: L.gpk_gp_model_ucb(h, c["model"], X if a["Xs"] else None, a["m"], a["ldxs"], 2.0,
                                                 o.ucb if a["ucb"] else None, o.grad, a["ldg"], o.mean, o.var),
        dict(m=m, ldxs=m, ldg=m, Xs=True, ucb=True),
        [dict(ucb=False), dict(Xs=False), dict(ldxs=m - 1), dict(m=0), dict(ldg=m - 1)]),
    "gpk_gp_models_mean": (
        lambda L, h, a, o, c: L.gpk_gp_models_mean(h, c["models"], a["k"], X if a["Xs"] else None, a["m"], a["ldxs"], o.mean),
        dict(k=1, m=m, ldxs=m, Xs=True),
        [dict(k=0), dict(Xs=False), dict(ldxs=m - 1), dict(m=0)]),
    "gpk_gp_models_mean_var": (
        lambda L, h, a, o, c: L.gpk_gp_models_mean_var(h, c["models"], a["k"], X, a["m"], a["ldxs"],
                                                       o.mean if a["mean"] else None, o.var),
        dict(k=1, m=m, ldxs=m, mean=True),
        [dict(k=0), dict(mean=False), dict(ldxs=m - 1), dict(m=0)]),
    "gpk_gp_model_append": (
        lambda L, h, a, o, c: L.gpk_gp_model_append(h, c["model"] if a["model"] else None, X if a["x"] else None, 0.5, 0, 0.0,
                                                    o.dll),
        dict(model=True, x=True),
        [dict(x=False), dict(model=False)]),
    "gpk_ep_fit": (
        lambda L, h, a, o, c: L.gpk_ep_fit(h, X, a["n"], a["ldk"], p(TGT) if a["t"] else None, 1e-6, 0, 10, 0, o.tau, o.nu, o.mu,
                                           o.L, a["ldl"], o.ct, o.cn, o.logZ, o.i_sweeps),
        dict(n=n, ldk=n, ldl=n, t=True),
        [dict(t=False), dict(ldk=n - 1), dict(ldl=n - 1), dict(n=0)]),
    "gpk_ep_nll_grad": (
        lambda L, h, a, o, c: L.gpk_ep_nll_grad(h, X, a["n"], a["D"], a["ldx"], X, p(TGT) if a["t"] else None, 1e-6, 0, 10, 0,
                                                a["np"], o.logZ, o.grad, o.tau, o.nu, o.i_sweeps),
        dict(n=n, D=D, ldx=n, np=P, t=True),
        [dict(D=0), dict(D=65), dict(ldx=n - 1), dict(n=0), dict(np=-1), dict(np=P + 1), dict(t=False)]),
    "gpk_ep_grad_from_factor": (
        lambda L, h, a, o, c: L.gpk_ep_grad_from_factor(h, X, a["n"], a["D"], a["ldx"], X, X, a["ldk"], X if a["tau"] else None,
                                                        X, X, a["ldl"], a["np"], o.grad),
        dict(n=n, D=D, ldx=n, ldk=n, ldl=n, np=P, tau=True),
        [dict(D=0), dict(D=65), dict(ldx=n - 1), dict(ldk=n - 1), dict(ldl=n - 1), dict(n=0), dict(np=-1), dict(np=P + 1),
         dict(tau=False)]),
    "gpk_ep_classify": (
        lambda L, h, a, o, c: L.gpk_ep_classify(h, X, a["n"], a["ldk"], X, a["m"], a["ldks"], X, X, X, X, a["ldl"], o.prob,
                                                o.fmean, o.fvar),
        dict(n=n, m=m, ldk=n, ldks=m, ldl=n),
        [dict(ldk=n - 1), dict(ldks=m - 1), dict(ldl=n - 1), dict(n=0), dict(m=0)]),
}

ON_MODEL = {"gpk_gp_model_predict", "gpk_gp_model_ucb", "gpk_gp_models_mean", "gpk_gp_models_mean_var", "gpk_gp_model_append"}
CASES = [(name, i) for name, (_, _, cases) in ENTRIES.items() for i in range(len(cases))]


def case_id(c):
    name, i = c
    return f"{name}-" + "-".join(f"{k}={v}" for k, v in ENTRIES[name][2][i].items())


@pytest.mark.parametrize("case", CASES, ids=[case_id(c) for c in CASES])
def test_malformed_call_is_rejected_without_effect(case):
    name, i = case
    call, defaults, cases = ENTRIES[name]
    args = dict(defaults, **cases[i])
    handle = _lib.Handle()
    L, h = handle.lib, handle.h
    ctx = {}
    if name in ON_MODEL:
        ctx["model"] = fit_model(L, h)
        ctx["models"] = C.cast((C.c_void_p * 1)(ctx["model"].value), C.c_void_p)
    if name.endswith("_dev"):
        ctx["tensors"] = [dev(BIG, 0.5), dev(BIG, SENT), dev(1024, 0.0)]
        ctx["dX"], ctx["dout"], ctx["dinfo"] = (t.data_ptr() for t in ctx["tensors"])
    try:
        handle.synchronize()
        # a different entry point fails first: the case must replace its message
        assert L.gpk_set_kernel_family(h, 99) == _lib.GPK_EINVAL
        before = L.gpk_last_error(h)
        l0 = handle.launch_count()
        o = Outs()
        rc = call(L, h, args, o, ctx)
        launches = handle.launch_count() - l0
        msg = L.gpk_last_error(h)
        assert rc == _lib.GPK_EINVAL, (rc, msg)
        assert launches == 0
        assert o.untouched()
        if "dout" in ctx:
            assert bool((ctx["tensors"][1] == SENT).all())
        assert msg != before and msg, msg
    finally:
        if "model" in ctx:
            L.gpk_gp_model_destroy(h, ctx["model"])
        handle.close()
