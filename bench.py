#!/usr/bin/env python
"""bench.py -- headline benchmark of the B200-native dense-GP path (BASELINE.json metric):
"MLE objective+gradient evals/sec at n=8192 D=8 (FP64); Cholesky TFLOP/s vs peak".

One "step" = one evaluation of GpPredictor.logLikelihoodWithDerivatives (gp/regression/GpPredictor.scala:60-80)
with nParams = D+2 = 10 on the synthetic C2 workload of SURVEY.md 8(d) (seed 2, X ~ U(0,1)^{8192x8}).

  python bench.py [--gpus N] [--steps K] [--warmup W] [--impl reference] [--dump-outputs DIR]

* value  : evals/s with X, y resident in HBM (gpk_gp_nll_grad_dev), CUDA-event timed, max over ranks.
* e2e    : same metric through the public host API (GpPredictor.logLikelihoodWithDerivatives) with pinned
           HOST buffers: H2D of X,y and D2H of (ll, g) inside the timed region.
* N > 1  : MLE restarts are independent evaluations (SURVEY.md 8(e)): each rank evaluates its own restart
           (different theta, same data), no data-path collective; value = N evals / max-over-ranks time.
* roofline: the Cholesky trailing update (SYRK on DMMA) timed alone against a live cuBLAS Dgemm peak.
* cpu_baseline / --impl reference: the oracle's LAPACK-backed port on the box's host cores (the Scala
  reference needs a JVM, absent here -- see DESIGN.md).
* --dump-outputs DIR: after the timed steps, what the last timed step returned, as DIR/ll.npy (N,) and DIR/grad.npy
  (N, nparams) in float64, one row per rank.  The inputs are seeded, so two builds run with the same arguments can be
  compared output for output.
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
# more hardware work queues than the default 8: libgpk's drivers use up to ~20 streams per handle (see gp_algos_b200/__init__.py);
# must be in the environment before the CUDA context exists
os.environ.setdefault("CUDA_DEVICE_MAX_CONNECTIONS", "32")

N_TRAIN, DIM = 8192, 8
NPARAMS = DIM + 2
METRIC = "MLE objective+gradient evals/sec at n=8192 D=8 (FP64)"
UNIT = "evals/s"


def parse():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="gpk", choices=["gpk", "reference"])
    ap.add_argument("--n", type=int, default=N_TRAIN, help="(debug only) problem size; the reported config is n=8192")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-sharded", action="store_true", help="skip the C4 / C5 sharded record (debug)")
    ap.add_argument("--dump-outputs", metavar="DIR", help="write the last timed step's (ll, grad) to DIR/ll.npy, DIR/grad.npy")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "gpk":
        ap.error("--dump-outputs writes the outputs of the gpk path only")
    return args


def config(n, n_gpus):
    return {"workload": f"C2: GP regression MLE objective+gradient, ARD-SE kernel, n={n}, D={DIM}, P={NPARAMS}, FP64, "
                        f"synthetic seed 2 (SURVEY.md 8(d))",
            "n": n, "D": DIM, "nparams": NPARAMS,
            "parallelism": "1 GPU" if n_gpus == 1 else f"{n_gpus} independent MLE restarts, one per GPU, no collective",
            "l2": "working set (K, L^-1: 2 x 512 MiB) exceeds the 126 MB L2; no explicit flush",
            "launches": ("eager launches (GPK_GRAPH=0)" if os.environ.get("GPK_GRAPH", "1") == "0" else
                         "CUDA-graph replay: per step one parameter kernel + one graph launch; gpu_launches counts the graph's "
                         "kernel nodes (398 per evaluation), captured during warm-up")}


# ------------------------------------------------------------------------------------------------------
# CPU arm (oracle port)
# ------------------------------------------------------------------------------------------------------
def cpu_eval_time(n, reps=1):
    from oracle import gp_oracle as orc
    X, y, theta = orc.make_c2(n=n, D=DIM)
    best = 1e30
    for _ in range(reps):
        t0 = time.perf_counter()
        orc.fast_loglik_with_derivs(X, y, theta, None, NPARAMS)
        best = min(best, time.perf_counter() - t0)
    return best


def cpu_literal_time(n=768):
    from oracle import gp_oracle as orc
    X, y, theta = orc.make_c2(n=n, D=DIM)
    t0 = time.perf_counter()
    orc.lit_loglik_with_derivs(X, y, theta, None, NPARAMS)
    return time.perf_counter() - t0


def blas_threads_all():
    """Give the CPU arm every host core, whatever the launcher exported: torch.distributed.run sets OMP_NUM_THREADS=1 for
    its workers, which throttled the round-1 reference arm at N >= 2 to one BLAS thread.  Returns the thread count in use."""
    cores = os.cpu_count() or 1
    try:
        from threadpoolctl import threadpool_limits, threadpool_info
        import numpy  # noqa: F401  (loads OpenBLAS so that threadpoolctl sees it)
        import scipy.linalg  # noqa: F401
        threadpool_limits(limits=cores)
        used = [p.get("num_threads", 1) for p in threadpool_info() if p.get("user_api") == "blas"]
        return max(used) if used else cores
    except Exception:
        return cores


def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    cores = blas_threads_all()
    n = args.n
    for _ in range(min(args.warmup, 1)):  # one warm-up eval is enough to page in BLAS (each takes seconds)
        cpu_eval_time(n)
    t0 = time.perf_counter()
    for _ in range(args.steps):
        cpu_eval_time(n)
    dt = (time.perf_counter() - t0) / args.steps
    v = 1.0 / dt
    sample = (f"each step = one full n={n} evaluation through the oracle's LAPACK-backed port (OpenBLAS dpotrf+dpotri, "
              f"fused O(n^2 P) gradient on a {cores}-thread pool, {cores} BLAS threads); the Scala reference as written does ~23x more flops "
              f"single-threaded")
    print(json.dumps({
        "impl": "reference", "metric": METRIC, "value": v, "unit": UNIT, "n_gpus": args.gpus, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": dt * 1e3, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
        "dtype": "f64", "data": "synthetic", "config": config(n, args.gpus),
        "cpu_baseline": {"value": v, "unit": UNIT, "cores": cores, "kind": "port", "sample": sample},
        "e2e": {"value": v, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
    }))


# ------------------------------------------------------------------------------------------------------
# GPU arm
# ------------------------------------------------------------------------------------------------------
class ClockSampler:
    Q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        self.index, self.rows, self.proc = index, [], None

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.index), f"--query-gpu={self.Q}",
                                          "--format=csv,noheader,nounits", "-lms", "100"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            threading.Thread(target=self._read, daemon=True).start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append([c.strip() for c in line.split(",")])

    def stop(self):
        if self.proc:
            self.proc.terminate()
        sm, reasons, mx = [], set(), None
        for r in self.rows:
            try:
                sm.append(float(r[0])); mx = float(r[1])
                for name, val in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), r[3:7]):
                    if val.lower().startswith("active"):
                        reasons.add(name)
            except Exception:
                pass
        sm.sort()
        return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": mx, "reasons": sorted(reasons), "samples": len(sm)}



# ------------------------------------------------------------------------------------------------------
# second half of the metric: "Cholesky TFLOP/s vs peak" -- gpk_potrf_lower_dev alone at n = 8192
# ------------------------------------------------------------------------------------------------------
def bench_cholesky(h, dX, n, theta, peak_tflops, reps=5):
    """Factor-only Cholesky (breeze `cholesky` -> dpotrf 'L', GpPredictor.scala:120) of the C2 kernel matrix, resident in HBM.
    K is rebuilt before every repetition (outside the timed region); algorithmic flops n^3/3."""
    import numpy as np
    import torch
    from gp_algos_b200 import _lib
    K0 = torch.empty(n * n, dtype=torch.float64, device="cuda")
    A = torch.empty_like(K0)
    info = torch.zeros(1, dtype=torch.int32, device="cuda")
    th = np.ascontiguousarray(theta)
    h.check(h.lib.gpk_cov_se_ard_dev(h.h, dX.data_ptr(), n, DIM, n, _lib.ptr(th), K0.data_ptr(), n))
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    times = []
    for rep in range(reps + 2):
        A.copy_(K0)
        torch.cuda.synchronize()
        e0.record()
        h.check(h.lib.gpk_potrf_lower_dev(h.h, A.data_ptr(), n, n, info.data_ptr()))
        e1.record()
        torch.cuda.synchronize()
        if rep >= 2:
            times.append(e0.elapsed_time(e1))
    assert int(info.item()) == 0, "factorisation failed"
    # check: ||L (L^t v) - K v|| / ||K v|| for a random v (three HBM-bound mat-vecs through libgpk)
    v = torch.from_numpy(np.random.default_rng(7).standard_normal(n)).cuda()
    t1, t2, t3 = (torch.empty(n, dtype=torch.float64, device="cuda") for _ in range(3))
    h.check(h.lib.gpk_gemv_dev(h.h, 1, n, n, 1.0, A.data_ptr(), n, v.data_ptr(), 0.0, t1.data_ptr()))
    h.check(h.lib.gpk_gemv_dev(h.h, 0, n, n, 1.0, A.data_ptr(), n, t1.data_ptr(), 0.0, t2.data_ptr()))
    h.check(h.lib.gpk_gemv_dev(h.h, 0, n, n, 1.0, K0.data_ptr(), n, v.data_ptr(), 0.0, t3.data_ptr()))
    torch.cuda.synchronize()
    resid = float(torch.linalg.norm(t2 - t3) / torch.linalg.norm(t3))
    ms = min(times)
    tf = float(n) ** 3 / 3 / ms * 1e-9
    return {"n": n, "ms": ms, "ms_all": times, "tflops": tf, "frac": tf / peak_tflops if peak_tflops else None,
            "flops": float(n) ** 3 / 3, "what": "gpk_potrf_lower_dev: factor only, K resident in HBM, in place; best of "
            f"{reps} after 2 warm-ups; frac = tflops / live cuBLAS Dgemm peak", "resid_LLt_v_vs_K_v": resid}


# ------------------------------------------------------------------------------------------------------
# the sharded configs (SURVEY.md 8(e)): C4 = 512 independent GPs split over the ranks, no collective;
# C5 = one GP of n = 65536 on a 2-D block-cyclic grid with NCCL panel broadcasts
# ------------------------------------------------------------------------------------------------------
C4_B, C4_N, C4_M = 512, 1024, 17


def _max_over_ranks(dist, vals):
    import torch
    t = torch.tensor(list(vals), dtype=torch.float64, device="cuda")
    if dist is not None:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    return [float(v) for v in t.tolist()]


def bench_c4(h, dist, rank, world, reps=5):
    """512 x (n = 1024, D = 8) objective+gradient evaluations (MLE-restart flavour, GPOptimizer.scala:54-61 /
    GPUnscentedKalmanFilter.scala:123-136), problems [lo, hi) = batched.shard_bounds on each rank.  Strong scaling: the total
    work is fixed.  Device-timed with the shard resident in HBM, and end to end from host buffers."""
    import numpy as np
    import torch
    from gp_algos_b200 import _lib, batched, synthetic
    lo, hi = batched.shard_bounds(C4_B, rank, world)
    # rank 0 also times the whole batch alone (the in-run 1-GPU figure the speed-up is quoted against)
    need = range(C4_B) if rank == 0 else range(lo, hi)
    probs = {b: synthetic.make_c4_problem(b, n=C4_N, D=DIM, m=C4_M) for b in need}

    def stack(idx):
        X = np.stack([probs[b][0] for b in idx]); ys = np.stack([probs[b][1] for b in idx]); th = np.stack([probs[b][3] for b in idx])
        return X, ys, np.ascontiguousarray(th)

    def timed(idx):
        X, ys, th = stack(idx)
        nb = len(idx)
        dX = torch.from_numpy(np.ascontiguousarray(np.transpose(X, (0, 2, 1)))).cuda()
        dy = torch.from_numpy(ys).cuda()
        out = torch.zeros(nb * (NPARAMS + 1), dtype=torch.float64, device="cuda")
        info = torch.zeros(nb, dtype=torch.int32, device="cuda")

        def step():
            h.check(h.lib.gpk_gp_nll_grad_batched_dev(h.h, nb, dX.data_ptr(), C4_N, DIM, C4_N, C4_N * DIM, dy.data_ptr(), _lib.ptr(th),
                                                      0, 0.0, NPARAMS, out.data_ptr(), info.data_ptr()))
        for _ in range(3):
            step()
        torch.cuda.synchronize()
        return step, info, out, (X, ys, th)

    step, info, out, host = timed(list(range(lo, hi)))
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    if dist is not None:
        dist.barrier()
    torch.cuda.synchronize()
    l0 = h.launch_count()
    e0.record()
    for _ in range(reps):
        step()
    e1.record()
    torch.cuda.synchronize()
    ms = e0.elapsed_time(e1) / reps
    launches = (h.launch_count() - l0) // reps
    assert int(info.abs().sum().item()) == 0, "a C4 problem failed to factor"
    # end to end: PINNED host buffers in the reference's (Breeze, column-major) layout in, (ll, grad) out through the public
    # batched API; H2D of X, y and D2H of the results inside the timed region
    X, ys, th = host
    Xp = torch.from_numpy(np.ascontiguousarray(np.transpose(X, (0, 2, 1)))).pin_memory()     # (B, D, n): column-major stack
    yp = torch.from_numpy(ys.copy()).pin_memory()
    X, ys = Xp.numpy().transpose(0, 2, 1), yp.numpy()
    batched.log_likelihood_with_derivatives_batched(X, ys, th, handle=h)
    if dist is not None:
        dist.barrier()
    t0 = time.perf_counter()
    ll, g, _ = batched.log_likelihood_with_derivatives_batched(X, ys, th, handle=h)
    t_e2e = time.perf_counter() - t0
    dev = out.cpu().numpy().reshape(hi - lo, NPARAMS + 1)
    assert np.allclose(dev[:, 0], ll, rtol=1e-12, atol=0) and np.allclose(dev[:, 1:], g, rtol=1e-12, atol=0)
    ms, t_e2e = _max_over_ranks(dist, [ms, t_e2e])
    rec = {"workload": f"C4: {C4_B} independent GPs, n={C4_N}, D={DIM}, objective+gradient (P={NPARAMS}); problems split over "
                       f"{world} GPU(s) by batched.shard_bounds, no data-path collective", "scaling": "strong",
           "problems_per_s": C4_B / (ms * 1e-3), "ms": ms, "eff_tflops": C4_B * float(C4_N) ** 3 / (ms * 1e-3) * 1e-12,
           "e2e_problems_per_s": C4_B / t_e2e, "e2e_ms": t_e2e * 1e3, "problems_on_rank0": hi - lo,
           "e2e_h2d_bytes_rank0": int((hi - lo) * (C4_N * DIM + C4_N) * 8), "e2e_d2h_bytes_rank0": int((hi - lo) * ((NPARAMS + 1) * 8 + 4)),
           "launches_per_batch_rank0": int(launches), "timing": "CUDA events on each rank's stream, max over ranks"}
    del step, out, info
    if world > 1:
        ms1 = None
        if rank == 0:
            step1, info1, out1, _ = timed(list(range(C4_B)))
            e0.record()
            for _ in range(reps):
                step1()
            e1.record()
            torch.cuda.synchronize()
            ms1 = e0.elapsed_time(e1) / reps
            # the shard's results are bit-identical to the same problems evaluated inside the full batch
            full = out1.cpu().numpy().reshape(C4_B, NPARAMS + 1)
            rec["shard_equals_full_batch"] = bool(np.array_equal(full[lo:hi], dev))
            rec["one_gpu_ms_in_run"] = ms1
            rec["speedup_vs_one_gpu_in_run"] = ms1 / ms
        dist.barrier()
    return rec


def bench_c5(dist, rank, world, local, cpu_group=None, n=65536, nb=None, reps=2):
    """One GP of n = 65536, D = 8 (seed 5): K build + 2-D block-cyclic FP64 Cholesky + both solves + log-likelihood
    (GpPredictor.scala:104-124,144-149) through DistributedGp.fit.  Strong scaling.  CUDA events per rank, max over ranks."""
    import numpy as np
    import torch
    from gp_algos_b200 import synthetic
    from gp_algos_b200.distributed import DistributedGp, choose_grid
    X, y, theta = synthetic.make_c2(n=n, D=DIM, seed=5)
    grid = choose_grid(world)
    if nb is None:
        nb = 512 if world >= 8 else 1024      # narrower blocks shorten the serial factor -> panel -> broadcast chain (0.438 vs 0.450 s on 8)
    solver = DistributedGp(grid=grid, nb=nb, device=local)
    times, fit = [], None
    for _ in range(reps):
        fit = solver.fit(X, y, theta)
        times.append(_max_over_ranks(dist, [fit.seconds])[0])
    res = solver.residual(y, fit.alphaVec)
    best = min(times)
    rec = {"workload": f"C5: one GP, n={n}, D={DIM}, K build + block-cyclic Cholesky (nb={nb}) + alpha solves + log-likelihood",
           "scaling": "strong", "grid": f"{grid[0]}x{grid[1]}", "seconds": best, "seconds_all": times,
           "potrf_tflops_total": float(n) ** 3 / 3 / best * 1e-12, "potrf_tflops_per_gpu": float(n) ** 3 / 3 / best * 1e-12 / world,
           "residual_Kalpha_minus_y_over_y": res, "ll": fit.logLikelihood,
           "bytes_broadcast_received_per_rank": int(getattr(solver, "bcast_bytes", 0) // max(reps, 1)),
           "collectives": "none (1 GPU)" if world == 1 else "NCCL broadcast of L_kk^-1 and the panel pieces per step, one nb-vector "
                          "all-reduce per back-solve step, two scalar all-reduces",
           "timing": "CUDA events around build + factor + solves on each rank, max over ranks, best of %d" % reps}
    # ---- the same solve through the C ABI (gpk_mg_create / gpk_mg_potrf_solve): ONE process drives all `world` GPUs with
    # peer-to-peer panel puts; rank 0 runs it while the other ranks wait on a CPU (gloo) barrier, their GPUs idle
    try:
        cabi = {"what": "gpk_mg_potrf_solve: single process, round-robin block columns, cudaMemcpy2DAsync peer puts (no NCCL)",
                "ndev": world, "nb": "automatic (gpk_mg_set_block(0): 1024 up to 4 devices, 512 on 8 at this n)"}
        alpha_c = torch.zeros(n, dtype=torch.float64, device="cuda")
        if rank == 0:
            from gp_algos_b200.multi_gpu import MultiGpuGp
            mg = MultiGpuGp(world)                  # block width: the library's automatic choice
            runs = [mg.fit(X, y, theta) for _ in range(reps)]
            mg.close()
            f = min(runs, key=lambda r: r.seconds)
            cabi.update({"seconds": f.seconds, "seconds_all": [r.seconds for r in runs],
                         "potrf_tflops_per_gpu": float(n) ** 3 / 3 / f.seconds * 1e-12 / world, "ll": f.logLikelihood,
                         "ll_rel_diff_vs_nccl_path": abs(f.logLikelihood - fit.logLikelihood) / abs(fit.logLikelihood),
                         "bytes_put_to_peers": f.put_bytes})
            alpha_c.copy_(torch.from_numpy(f.alphaVec))
        if dist is not None:
            dist.barrier(group=cpu_group)          # CPU-side wait: no NCCL kernel spins on the idle GPUs meanwhile
            dist.broadcast(alpha_c, src=0)
        cabi["residual_Kalpha_minus_y_over_y"] = solver.residual(y, alpha_c.cpu().numpy())
        rec["c_abi"] = cabi
    except Exception as e:
        rec["c_abi"] = {"error": f"{type(e).__name__}: {e}"[:400]}
    del solver
    torch.cuda.empty_cache()
    return rec


def nccl_parity(dist, rank, world, local, g0, n=5000, nb=256):
    """N >= 2 only: the NCCL data plane against the same solver on a 1 x 1 grid (rank 0 alone), in this run, because the
    2-GPU pytest cannot run on a 1-GPU test box.  ll to 1e-11, alpha to 1e-9, K alpha = y to 1e-10."""
    import numpy as np
    import torch
    from gp_algos_b200 import synthetic
    from gp_algos_b200.distributed import DistributedGp, choose_grid
    X, y, theta = synthetic.make_c2(n=n, D=DIM, seed=5)
    grid = choose_grid(world)
    solver = DistributedGp(grid=grid, nb=nb, device=local)
    fit = solver.fit(X, y, theta)
    res = solver.residual(y, fit.alphaVec)
    rec = {"n": n, "nb": nb, "grid": f"{grid[0]}x{grid[1]}", "residual_Kalpha_minus_y_over_y": res}
    ok = torch.zeros(1, dtype=torch.float64, device="cuda")
    if rank == 0:
        single = DistributedGp(grid=(1, 1), nb=nb, device=local, group=g0)
        fit1 = single.fit(X, y, theta)
        rec["ll_rel_diff_vs_1x1"] = abs(fit.logLikelihood - fit1.logLikelihood) / abs(fit1.logLikelihood)
        rec["alpha_max_rel_diff_vs_1x1"] = float(np.abs(fit.alphaVec - fit1.alphaVec).max() / np.abs(fit1.alphaVec).max())
        rec["passed"] = bool(rec["ll_rel_diff_vs_1x1"] <= 1e-11 and rec["alpha_max_rel_diff_vs_1x1"] <= 1e-9 and res < 1e-10)
        ok[0] = 1.0 if rec["passed"] else 0.0
    dist.broadcast(ok, src=0)
    rec["passed"] = bool(ok.item() == 1.0)
    return rec


def run_sharded(h, dist, rank, world, local):
    rec = {}
    g0 = dist.new_group(ranks=[0]) if dist is not None else None     # rank 0 alone: the in-run single-GPU references
    cpu_group = dist.new_group(backend="gloo") if dist is not None else None
    for name, fn in (("c4", lambda: bench_c4(h, dist, rank, world)),
                     ("c5", lambda: bench_c5(dist, rank, world, local, cpu_group)),
                     ("nccl_parity", (lambda: nccl_parity(dist, rank, world, local, g0)) if world > 1 else None)):
        if fn is None:
            continue
        try:
            rec[name] = fn()
        except Exception as e:  # keep the headline line; a failed sharded leg is reported, not hidden
            rec[name] = {"error": f"{type(e).__name__}: {e}"[:400]}
    return rec


def syrk_traffic(nn, kk):
    """roofline.traffic: dram__bytes_read.sum + dram__bytes_write.sum per launch of the SYRK kernel at this shape, taken from
    the committed `ncu --set full` capture summary (profiles/syrk_traffic.json, written by tools/ncu_traffic.py from the
    .ncu-rep); DRAM traffic cannot be measured outside a profiler, so it is null when no capture of this shape is recorded."""
    try:
        with open(os.path.join(ROOT, "profiles", "syrk_traffic.json")) as f:
            t = json.load(f)
        if (t.get("n"), t.get("k")) == (nn, kk):
            return {"traffic": float(t["dram_bytes_per_launch"]), "traffic_source": t.get("source"),
                    "algorithmic_bytes": 8.0 * (nn * (nn + 128) / 2 * 2 + nn * kk)}
    except Exception:
        pass
    return {"traffic": None}


def dump_outputs(path, res):
    """res: (ranks, 1 + nparams) rows of gpk_gp_nll_grad_dev's output (ll, grad) -> path/ll.npy, path/grad.npy (float64)."""
    import numpy as np
    os.makedirs(path, exist_ok=True)
    np.save(os.path.join(path, "ll.npy"), np.ascontiguousarray(res[:, 0], dtype=np.float64))
    np.save(os.path.join(path, "grad.npy"), np.ascontiguousarray(res[:, 1:], dtype=np.float64))


def run_gpk(args):
    import numpy as np
    import torch
    import ctypes as C
    import gp_algos_b200 as gp
    from gp_algos_b200 import _lib, synthetic   # oracle/ is imported by the cpu_baseline / --impl reference legs only

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device (libgpk has no CPU fallback)")
    torch.cuda.set_device(local)
    dist = None
    if world > 1:
        import torch.distributed as dist
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    n = args.n
    X, y, theta0 = synthetic.make_c2(n=n, D=DIM)
    # each rank = one MLE restart: same data, its own hyper-parameter point
    rng = np.random.default_rng(100 + rank)
    theta = theta0.copy()
    if rank > 0:
        theta[0] *= 10 ** rng.uniform(-0.1, 0.1)
        theta[1:-1] *= 10 ** rng.uniform(-0.1, 0.1, size=DIM)
    # a real (non-default) torch stream shared with libgpk so torch.cuda.Event brackets the library's launches
    tstream = torch.cuda.Stream(priority=-1)  # above libgpk's low-priority side streams
    torch.cuda.set_stream(tstream)
    h = _lib.Handle(local, tstream.cuda_stream)
    dX = torch.from_numpy(np.asfortranarray(X).T.copy()).cuda()  # (D, n) row-major == n x D column-major, ld n
    dy = torch.from_numpy(y).cuda()
    dout = torch.zeros(NPARAMS + 1, dtype=torch.float64, device="cuda")
    dinfo = torch.zeros(1, dtype=torch.int32, device="cuda")
    th_c = np.ascontiguousarray(theta)

    def step_dev():
        h.check(h.lib.gpk_gp_nll_grad_dev(h.h, dX.data_ptr(), n, DIM, n, dy.data_ptr(), _lib.ptr(th_c), 0, 0.0, NPARAMS,
                                          dout.data_ptr(), dinfo.data_ptr()))

    def barrier():
        if dist is not None:
            dist.barrier()
        torch.cuda.synchronize()

    for _ in range(max(args.warmup, 3)):
        step_dev()
    barrier()
    sampler = ClockSampler(local)
    if rank == 0:
        sampler.start()
    l0 = h.launch_count()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    barrier()
    e0.record()
    for _ in range(args.steps):
        step_dev()
    e1.record()
    barrier()
    ms = e0.elapsed_time(e1)
    launches = h.launch_count() - l0
    if dist is not None:
        t = torch.tensor([ms], dtype=torch.float64, device="cuda")
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        ms = float(t.item())
    clocks = sampler.stop() if rank == 0 else None
    assert int(dinfo.item()) == 0, "factorisation failed"
    res_dev = dout.cpu().numpy().copy()
    if args.dump_outputs:
        rows = [dout]
        if dist is not None:
            rows = [torch.empty_like(dout) for _ in range(world)]
            dist.all_gather(rows, dout)
        if rank == 0:
            dump_outputs(args.dump_outputs, torch.stack(rows).cpu().numpy())

    # ---- e2e: public host API, pinned host buffers, H2D + D2H inside the timed region -----------------
    Xp = torch.from_numpy(np.asfortranarray(X).T.copy()).pin_memory()
    yp = torch.from_numpy(y.copy()).pin_memory()
    Xh = Xp.numpy().T  # n x D column-major view over pinned memory
    yh = yp.numpy()
    kf = gp.GaussianRbfKernel(gp.GaussianRbfParams(theta[0], theta[1:-1], theta[-1]))
    pred = gp.GpPredictor(kf, handle=h)
    inp = gp.PredictionTrainingInput(Xh, None, yh)
    for _ in range(2):
        ll, g = pred.logLikelihoodWithDerivatives(inp, theta, NPARAMS)
    barrier()
    t0 = time.perf_counter()
    for _ in range(args.steps):
        ll, g = pred.logLikelihoodWithDerivatives(inp, theta, NPARAMS)
    torch.cuda.synchronize()
    e2e_s = time.perf_counter() - t0
    if dist is not None:
        t = torch.tensor([e2e_s], dtype=torch.float64, device="cuda")
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        e2e_s = float(t.item())
    assert abs(ll - res_dev[0]) <= 1e-12 * abs(ll) and np.allclose(g, res_dev[1:], rtol=1e-12, atol=0)

    # ---- roofline: the Cholesky trailing update (SYRK, DMMA) alone; peak = live cuBLAS Dgemm ----------
    roofline = None
    if rank == 0:
        nn, kk = n // 2, n // 2
        P = torch.randn(kk, nn, dtype=torch.float64, device="cuda")  # n x k column-major
        Cm = torch.zeros(nn, nn, dtype=torch.float64, device="cuda")
        for _ in range(2):
            h.check(h.lib.gpk_syrk_lower_dev(h.h, P.data_ptr(), nn, Cm.data_ptr(), nn, nn, kk))
        reps = 5
        s0, s1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        torch.cuda.synchronize(); s0.record()
        for _ in range(reps):
            h.check(h.lib.gpk_syrk_lower_dev(h.h, P.data_ptr(), nn, Cm.data_ptr(), nn, nn, kk))
        s1.record(); torch.cuda.synchronize()
        syrk_ms = s0.elapsed_time(s1) / reps
        syrk_flops = float(nn) * nn * kk  # algorithmic: lower triangle only, 2 * (n^2/2) * k
        A = torch.randn(n, n, dtype=torch.float64, device="cuda"); B = torch.randn(n, n, dtype=torch.float64, device="cuda")
        Co = torch.empty_like(A)
        for _ in range(2):
            torch.matmul(A, B, out=Co)
        best = 1e30
        for _ in range(5):
            s0.record(); torch.matmul(A, B, out=Co); s1.record(); torch.cuda.synchronize()
            best = min(best, s0.elapsed_time(s1))
        peak = 2.0 * n ** 3 / best * 1e-9
        ach = syrk_flops / syrk_ms * 1e-9
        roofline = {"kernel": "gemm_f64_dmma_kernel<false,false,SmallTile 64x64> as the Cholesky trailing update (SYRK lower, "
                              f"n={nn}, k={kk})", "bound": "tensor", "achieved": ach, "peak": peak, "unit": "TFLOP/s",
                    "frac": ach / peak,
                    **syrk_traffic(nn, kk),
                    "peak_source": f"cuBLAS Dgemm {n}^3 measured live in this run (MEASURED_PEAKS.json has no FP64 entry; "
                                   "DMMA pipe ceiling 37.1 TFLOP/s, profiles/r01_fp64_microbench.txt)",
                    "eval_flops": float(n) ** 3, "eval_tflops": float(n) ** 3 / (ms / args.steps) * 1e-9,
                    "eval_frac_of_peak": float(n) ** 3 / (ms / args.steps) * 1e-9 / peak}
        del A, B, Co, P, Cm

    cholesky = None
    if rank == 0:
        try:
            cholesky = bench_cholesky(h, dX, n, theta, roofline["peak"])
        except Exception as e:
            cholesky = {"error": f"{type(e).__name__}: {e}"[:400]}
    sharded = None
    if not args.no_sharded:
        sharded = run_sharded(h, dist, rank, world, local)

    if rank == 0:
        cpu = None
        if not args.no_cpu_baseline and world == 1:
            cores = blas_threads_all()
            t_cpu = cpu_eval_time(n)
            t_lit = cpu_literal_time(768)
            cpu = {"value": 1.0 / t_cpu, "unit": UNIT, "cores": cores, "kind": "port",
                   "sample": f"one full n={n} evaluation, oracle LAPACK-backed port (OpenBLAS dpotrf + dpotri with {cores} threads, fused "
                             f"gradient on a {cores}-thread pool): {t_cpu:.2f} s",
                   "literal_port_n768_s": t_lit,
                   "literal_port_extrapolated_n8192_s": t_lit * (8192 / 768) ** 3,
                   "literal_note": "line-by-line C restatement of the Scala path, 1 thread, timed at n=768 and scaled by n^3"}
        out = {
            "metric": METRIC, "value": world * args.steps / (ms * 1e-3), "unit": UNIT, "n_gpus": world, "steps": args.steps,
            "warmup": max(args.warmup, 3), "ms_per_step": ms / args.steps, "higher_is_better": True, "scaling": "weak",
            "vs_baseline": None, "dtype": "f64", "data": "synthetic", "config": config(n, world),
            "e2e": {"value": world * args.steps / e2e_s, "unit": UNIT, "h2d_bytes_per_step": (n * DIM + n) * 8,
                    "d2h_bytes_per_step": (NPARAMS + 1) * 8 + 4},
            "gpu_launches": int(launches), "clocks": clocks, "roofline": roofline, "cholesky": cholesky, "sharded": sharded,
            "cpu_baseline": cpu,
            "result": {"ll": float(res_dev[0]), "grad_inf_norm": float(np.abs(res_dev[1:]).max())},
        }
        print(json.dumps(out))
    if dist is not None:
        dist.destroy_process_group()


def main():
    args = parse()
    if args.impl == "reference":
        run_reference(args)
    else:
        run_gpk(args)


if __name__ == "__main__":
    main()
