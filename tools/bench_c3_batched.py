"""Batched EP evaluation (gpk_ep_nll_grad_batched) against a loop of single gpk_ep_nll_grad calls on the same inputs, in one
process, the two routes alternating.  C3 data (synthetic.make_c3, X shared by every problem) with theta on a signalVar x
lengthScale grid around the C3 point: what a hyper-parameter mesh or a set of optimiser restarts evaluates.  Two workloads,
B = 64 problems of n = 1024 (the sizes a hyper-parameter search runs, where one EP run leaves the GPU mostly idle) and B = 8 of
n = 4096 (where one run already keeps the tensor pipe busy), each with FixedSweeps(5) and with the shipped eps = 0.01.
Prints one JSON line per workload and stop rule: problems/s and ms per problem-sweep of both routes, the speed-up, the largest
relative difference between the routes, and the GPU's name and power limit."""
import ctypes as C
import json
import os
import subprocess
import sys
import time

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import numpy as np  # noqa: E402
import gp_algos_b200 as gp  # noqa: E402
from gp_algos_b200 import _lib, synthetic  # noqa: E402

REPS = int(os.environ.get("C3B_REPS", 3))
WORKLOADS = [(64, 1024), (8, 4096)]


def gpu_info():
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader", "-i", "0"],
                             capture_output=True, text=True, timeout=60).stdout.strip()
        name, power = [s.strip() for s in out.split(",")]
        return name, power
    except Exception:
        return "unknown", "unknown"


def grid_thetas(B, D):
    """B points: signalVar x lengthScale factors 2^[-1, 1] around the C3 point (1, 1, .., 0)."""
    k_ls = 8 if B >= 64 else 2
    k_sf = B // k_ls
    pts = [(sf, ls) for sf in 2.0 ** np.linspace(-1, 1, k_sf) for ls in 2.0 ** np.linspace(-1, 1, k_ls)]
    return np.stack([synthetic.pack_theta(sf, [ls] * D, 0.0) for sf, ls in pts[:B]])


def stop_args(stop):
    return (0.0, stop.sweeps, stop.sweeps) if isinstance(stop, gp.FixedSweeps) else (stop.eps, 0, stop.max_sweeps)


def loop_route(h, X, t, th, stop):
    Xf = np.asfortranarray(X); tt = np.ascontiguousarray(t, dtype=np.int32)
    n, D = X.shape
    eps, fixed, mx = stop_args(stop)
    logz = np.empty(len(th)); grad = np.empty_like(th); sweeps = np.empty(len(th), dtype=np.int32)
    for b in range(len(th)):
        lz = C.c_double(); sw = C.c_int()
        g = np.empty(th.shape[1])
        h.check(h.lib.gpk_ep_nll_grad(h.h, _lib.ptr(Xf), n, D, n, _lib.ptr(np.ascontiguousarray(th[b])), tt.ctypes.data_as(C.c_void_p),
                                      eps, fixed, mx, 1, th.shape[1], C.addressof(lz), _lib.ptr(g), None, None, C.addressof(sw)))
        logz[b], grad[b], sweeps[b] = lz.value, g, sw.value
    return logz, grad, sweeps


def batched_route(h, X, t, th, stop):
    logz, grad, sweeps, info = gp.log_likelihood_batched(X, t, th, stop, handle=h)
    assert np.all(info == 0)
    return logz, grad, sweeps


def rel(a, b):
    a, b = np.asarray(a), np.asarray(b)
    return float(np.max(np.abs(a - b) / np.maximum(np.abs(b), 1e-6 * np.abs(b).max())))


def main():
    name, power = gpu_info()
    h = _lib.default_handle()
    for B, n in WORKLOADS:
        X, t, _ = synthetic.make_c3(n=n)
        th = grid_thetas(B, X.shape[1])
        for stop in (gp.FixedSweeps(5), gp.AvgBasedStopCriterion(0.01)):
            routes = {"batched": batched_route, "loop": loop_route}
            res, times = {}, {k: [] for k in routes}
            for k, f in routes.items():                    # warm-up: module loads, arenas, attributes
                res[k] = f(h, X, t, th, stop)
            for _ in range(REPS):
                for k, f in routes.items():
                    t0 = time.perf_counter()
                    f(h, X, t, th, stop)                       # ends with the results on the host
                    times[k].append(time.perf_counter() - t0)
            sweeps = int(res["loop"][2].sum())
            assert np.array_equal(res["batched"][2], res["loop"][2]), "sweep counts differ between the routes"
            rec = {"workload": f"B={B} x n={n}", "stop": "fixed5" if isinstance(stop, gp.FixedSweeps) else "eps0.01",
                   "problem_sweeps": sweeps, "sweeps_min_max": [int(res["loop"][2].min()), int(res["loop"][2].max())]}
            for k in routes:
                tm = float(np.median(times[k]))
                rec[k] = {"seconds_median": tm, "seconds_all": times[k], "problems_per_s": B / tm, "ms_per_problem_sweep": 1e3 * tm / sweeps}
            rec["speedup_batched_over_loop"] = rec["loop"]["seconds_median"] / rec["batched"]["seconds_median"]
            rec["max_rel_diff"] = {"logZ": rel(res["batched"][0], res["loop"][0]), "grad": rel(res["batched"][1], res["loop"][1])}
            rec["gpu"] = name
            rec["power_limit"] = power
            print(json.dumps(rec), flush=True)


if __name__ == "__main__":
    main()
