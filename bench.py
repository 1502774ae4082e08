#!/usr/bin/env python
"""bench.py -- candidate-fits/sec of the cross-validated grid search (BASELINE.json metric).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--workload c2] [--impl ours|reference] [--dump-outputs DIR]
    python -m torch.distributed.run --nproc-per-node N ... bench.py --gpus N ...      (N > 1)

A "step" is one pass of the hot path over the whole workload: every (candidate, fold) fit+score task of
BASELINE config 2 -- GridSearchCV(SVC rbf) on synthetic 10000x512 fp32, C x gamma 8x8, cv=5 = 320 fits per
GPU.  At N > 1 GPUs every rank holds the dataset and evaluates its own 64 candidates of a grid refined
on the same ranges (N*64 candidates dealt to the ranks by predicted cost): weak scaling, no data-path collective, one
all-gather of the score blocks per step (the counterpart of RDD.collect()).  The N=4 grid is BASELINE config 4's
16x16 grid: its scores are asserted equal to the committed scikit-learn golden inside the run.

value  : fits/s with the dataset resident in HBM (gs_set_data done before the timed region); device time
         from CUDA events recorded on the engine's stream around each gs_svc call, max over ranks.
e2e    : the same metric through the public API -- GridSearchCV(...).fit(X, y) with HOST numpy buffers
         every step (H2D of X/y/folds and D2H of the score arrays inside the timed region), refit=False.
roofline: the dominant kernel (batched SMO): algorithmic HBM bytes (2 gathered float32 K rows of the
         sub-problem per SMO iteration, SURVEY.md 8d) / CUDA-event duration of the solve phase; `gram_roofline` is
         the Gram build north_star names (algorithmic bytes / its event time).
secondary: BASELINE configs 4 (SVC 16x16), 3 (LogisticRegression random 256) and 5 (Ridge 512 alphas) measured in
         the same run, STRONG-scaled over the N ranks (candidates dealt, one score all-gather): fits/s, e2e, parity
         against the committed scikit-learn goldens, and a roofline each (tensor-pipe fraction of the tcgen05
         contraction kernel against a TF32 peak measured here with cuBLAS for configs 3 and 5).
cpu_baseline / --impl reference: scikit-learn's own GridSearchCV (the reference's CPU path, joblib) with ONE
         (candidate, fold) task per host core per step: `cores` candidates whose predicted cost is nearest the grid
         mean, one fold -- every core is busy for the whole step and the sample's mean cost is the grid's.
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

GOLDEN = {"c2": "c2_svc_rbf_8x8", "c4": "c4_svc_rbf_16x16", "c3": "c3_logreg_random256", "c5": "c5_ridge_512",
          "c2_small": "c2_small", "c2_mid": "c2_mid", "c3_small": "c3_small", "c5_small": "c5_small"}


# ----------------------------------------------------------------------------- helpers ----------
def measured_peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        d = json.load(open(p))
        return float(d["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
    return 6650.0, "fallback (B200_PROFILING.md)"


class ClockSampler:
    """nvidia-smi clocks / throttle reasons sampled DURING the timed region (B200_PROFILING.md recipe)."""
    Q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, index=0):
        self.index, self.rows, self.proc = index, [], None

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.index), "--query-gpu=" + self.Q,
                                          "--format=csv,noheader,nounits", "-lms", "100"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.t = threading.Thread(target=self._read, daemon=True)
            self.t.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append([x.strip() for x in line.split(",")])

    def stop(self):
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except Exception:
            self.proc.kill()
        sm = [float(r[0]) for r in self.rows if len(r) >= 7 and r[0].replace(".", "").isdigit()]
        mx = [float(r[1]) for r in self.rows if len(r) >= 7 and r[1].replace(".", "").isdigit()]
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        reasons = [n for i, n in enumerate(names) if any(len(r) >= 7 and r[3 + i].lower().startswith("active") for r in self.rows)]
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": reasons, "samples": len(sm)}


def scaled_workload(key, n_gpus):
    """Weak scaling: 64 candidates per GPU on the ranges of config 2 (N=1 is config 2 itself; N=4 is the
    16x16 grid of config 4)."""
    from spark_sklearn_b200 import workloads as W
    w = W.make_workload(key)
    if key == "c2" and n_gpus > 1:
        nc, ng = {2: (8, 16), 4: (16, 16), 8: (16, 32)}.get(n_gpus, (8, 8 * n_gpus))
        w["param_grid"] = {"C": np.logspace(-1, 2.5, nc), "gamma": np.geomspace(1 / 4096, 1 / 256, ng)}
        w["name"] = "c2_weak_%dx%d" % (nc, ng)
        if (nc, ng) == (16, 16):
            w["golden"] = GOLDEN["c4"]                       # the N=4 weak-scaling grid IS config 4
    w.setdefault("golden", GOLDEN.get(key))
    return w


def effective_cores():
    """Host cores this process may actually use: min(affinity, cgroup cpu.max quota)."""
    n = len(os.sched_getaffinity(0)) if hasattr(os, "sched_getaffinity") else (os.cpu_count() or 1)
    try:
        quota, period = open("/sys/fs/cgroup/cpu.max").read().split()
        if quota != "max":
            n = min(n, max(1, int(round(int(quota) / int(period)))))
    except Exception:
        pass
    return n


def predicted_cost(w, cands):
    """Relative cost of one fold-fit per candidate, for picking the CPU sample only (plain Python, none of the library):
    SVC rbf: the SMO iteration count rises like (C gamma d)^0.95 and saturates ~ 1/(gamma d); other estimators: flat."""
    d = w["X"].shape[1]
    out = np.ones(len(cands))
    if w["estimator"] == "SVC":
        for i, c in enumerate(cands):
            g = c.get("gamma", w["est_params"].get("gamma"))
            if isinstance(g, (int, float)) and g > 0 and c.get("kernel", w["est_params"].get("kernel", "rbf")) == "rbf":
                gd = float(g) * d
                out[i] = min(4.0 + 10.3 * (float(c["C"]) * gd) ** 0.95, 9.0 + 7.3 / gd)
    return out


def measured_cost(w, cands):
    """Per-candidate cost from the committed golden of the workload when there is one (scikit-learn's own n_iter_ per fit,
    tests/golden/*.npz `diag`), else the closed-form prediction: the better the costs, the more evenly the sampled tasks end."""
    g = load_golden(w.get("golden"))
    if g is not None and "diag" in g and g["diag"].shape[0] == len(cands) and w["estimator"] == "SVC":
        return g["diag"][:, :, 0].mean(1).astype(float), "golden n_iter_"
    return predicted_cost(w, cands), "closed-form prediction"


def cpu_sample(w, cands, cores, cost_fraction=1.0):
    """`cores` candidates whose cost is nearest cost_fraction x the grid mean (ties: lower index), so that one step gives every
    host core exactly one (candidate, fold) task of about equal cost: all cores busy, tasks end together.  cost_fraction < 1
    (many steps asked for: bounded run time) picks cheaper-than-average tasks, which OVERSTATES the CPU's fits/s on the grid."""
    cost, src = measured_cost(w, cands)
    order = np.argsort(np.abs(cost - cost_fraction * cost.mean()), kind="stable")
    idx = sorted(int(i) for i in order[:min(cores, len(cands))])
    return idx, float(cost[idx].mean() / cost.mean()), src


def run_reference_step(w, cand_idx, fold, cores):
    """The reference's CPU implementation of the path: sklearn GridSearchCV -> joblib -> _fit_and_score
    (what spark_sklearn maps over Spark executors, base_search.py:74-90), n_jobs = all host cores, refit=False.
    One fold of the workload's CV and len(cand_idx) candidates = len(cand_idx) concurrent fit+score tasks."""
    from sklearn.base import is_classifier
    from sklearn.model_selection import GridSearchCV, check_cv
    from spark_sklearn_b200 import workloads as W
    cands = W.candidates(w)
    est = W.make_estimator(w)
    splits = list(check_cv(w["cv"], w["y"], classifier=is_classifier(est)).split(w["X"], w["y"]))
    grid = [{k: [v] for k, v in cands[i].items()} for i in cand_idx]
    s = GridSearchCV(est, grid, cv=[splits[fold % len(splits)]], return_train_score=True, refit=False, n_jobs=cores)
    t0 = time.perf_counter()
    s.fit(w["X"], w["y"])
    dt = time.perf_counter() - t0
    busy = float(np.sum(s.cv_results_["mean_fit_time"]) + np.sum(s.cv_results_["mean_score_time"]))
    return dt, len(cand_idx), busy, s.cv_results_["split0_test_score"]


def cpu_reference(w, cands, cores, steps, warmup):
    # bounded run: about 9 minutes for the whole --steps/--warmup run; a mean-cost config-2 task takes ~50 s on the GPU box's cores
    t_step = min(60.0, max(8.0, 540.0 / max(steps + warmup, 1)))
    frac = min(1.0, t_step / 50.0) if w["estimator"] == "SVC" and w["X"].shape[0] >= 8000 else 1.0
    idx, rel, src = cpu_sample(w, cands, cores, frac)
    for k in range(warmup):
        run_reference_step(w, idx, k, cores)
    tot = busy = 0.0
    fits = 0
    last = None
    for k in range(steps):
        dt, nf, b, last = run_reference_step(w, idx, warmup + k, cores)
        tot += dt; busy += b; fits += nf
    desc = ("%d of %d candidates (cost by %s nearest %.2f x the grid mean: sample mean / grid mean = %.2f%s) x 1 fold per step = "
            "%d concurrent fit+score tasks on %d cores" % (
                len(idx), len(cands), src, frac, rel,
                "" if frac >= 1.0 else "; cheaper-than-average tasks keep the run bounded and OVERSTATE the CPU's fits/s", len(idx), cores))
    return {"value": fits / tot, "unit": "fits/s", "cores": cores, "kind": "reference", "sample": desc,
            "seconds": tot, "cores_busy": busy / (tot * cores), "sample_cost_over_grid_mean": rel,
            "what": "scikit-learn %s GridSearchCV(n_jobs=%d, refit=False): the reference's own CPU path "
                    "(spark_sklearn is not importable here: no pyspark/JVM)" % (__import__("sklearn").__version__, cores)}, idx, last


def load_golden(name):
    p = os.path.join(ROOT, "tests", "golden", "%s.npz" % name) if name else None
    return np.load(p) if p and os.path.exists(p) else None


def parity_block(w, test_scores):
    g = load_golden(w.get("golden"))
    if g is None or g["test_scores"].shape != test_scores.shape:
        return None
    dm = float(np.max(np.abs(test_scores.mean(1) - g["test_scores"].mean(1))))
    return {"golden": "tests/golden/%s.npz (scikit-learn %s)" % (w["golden"], str(g["sklearn_version"]) if "sklearn_version" in g else "?"),
            "max_abs_diff_mean_test_score": dm, "split_scores_equal": bool(np.array_equal(test_scores, g["test_scores"]))}


def dump_outputs(path, key, m):
    """The split scores the last timed step returned ([candidates][splits] float64) as <path>/<key>_{test,train}_scores.npy.
    fit_time / score_time, the other arrays of that step, are wall-clock timings and would differ on every run."""
    os.makedirs(path, exist_ok=True)
    for part in ("test", "train"):
        np.save(os.path.join(path, "%s_%s_scores.npy" % (key, part)), np.asarray(m[part], np.float64))


def tf32_peak_tflops():
    """cuBLAS TF32 GEMM throughput on this GPU (the denominator for the tcgen05 kind::tf32 contraction kernel)."""
    import torch
    old = torch.backends.cuda.matmul.allow_tf32
    torch.backends.cuda.matmul.allow_tf32 = True
    try:
        n = 8192
        a = torch.randn(n, n, device="cuda"); b = torch.randn(n, n, device="cuda")
        for _ in range(3):
            a @ b
        best = 1e9
        for _ in range(8):
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record(); a @ b; e1.record(); torch.cuda.synchronize()
            best = min(best, e0.elapsed_time(e1))
        return 2.0 * n ** 3 / (best * 1e-3) / 1e12
    finally:
        torch.backends.cuda.matmul.allow_tf32 = old


# ----------------------------------------------------------------------------- one workload on the GPUs ----
class Runner:
    """Resident-data and end-to-end measurement of one workload over the ranks of this job."""

    def __init__(self, w, rank, world, local_rank, dist):
        from sklearn.base import is_classifier
        from sklearn.model_selection import check_cv
        from spark_sklearn_b200 import workloads as WL
        from spark_sklearn_b200.base_search import _dist as D
        from spark_sklearn_b200.estimators import adapter_for, fold_ids_from_splits
        self.w, self.rank, self.world, self.dist, self.D = w, rank, world, dist, D
        self.est = WL.make_estimator(w)
        self.cands = WL.candidates(w)
        X, y = w["X"], w["y"]
        self.splits = list(check_cv(w["cv"], y, classifier=is_classifier(self.est)).split(X, y))
        fold_id = fold_ids_from_splits(self.splits, len(y))
        self.plan = adapter_for(self.est).plan(self.est, self.cands, X, y, fold_id, len(self.splits))   # gs_set_data happens here
        self.parts = D.assign_for_plan(self.plan, len(self.cands), world)                               # same dealing as GridSearchCV.fit
        self.my = self.parts[rank]
        self.fits = len(self.cands) * len(self.splits)

    def barrier(self):
        import torch
        if self.dist is not None:
            self.dist.barrier()
        torch.cuda.synchronize()

    def resident_step(self):
        local = self.plan.evaluate(self.my, return_train=True)
        out = self.D.allgather_candidates(local, self.my, len(self.cands), len(self.splits), self.world, self.parts,
                                          device=self.plan.engine.device)
        return out, self.plan.profile()

    def e2e_step(self):
        from spark_sklearn_b200 import GridSearchCV, RandomizedSearchCV
        w = self.w
        if w["search"] == "grid":
            s = GridSearchCV(None, self.est, w["param_grid"], cv=w["cv"], refit=False)
        else:
            s = RandomizedSearchCV(None, self.est, w["param_distributions"], n_iter=w["n_iter"], cv=w["cv"], refit=False,
                                   random_state=w["random_state"])
        s.fit(w["X"], w["y"])
        return s

    def measure(self, steps, warmup, sampler=None):
        """-> dict of sums over the timed steps (device ms from the engine's CUDA events, profile counters), max/sum over ranks."""
        import torch
        for _ in range(warmup):
            self.resident_step()
        self.barrier()
        if sampler is not None:
            sampler.start()
        acc = {}
        t0 = time.perf_counter()
        for _ in range(steps):
            out, prof = self.resident_step()
            for k, v in prof.items():
                acc[k] = acc.get(k, 0.0) + float(v)
        self.barrier()
        wall = time.perf_counter() - t0
        clocks = sampler.stop() if sampler is not None else None
        for _ in range(min(warmup, 2)):
            self.e2e_step()
        self.barrier()
        t0 = time.perf_counter()
        for _ in range(steps):
            s = self.e2e_step()
        self.barrier()
        e2e_wall = time.perf_counter() - t0
        e2e_prof = s.device_profile_
        keys_max = ["ms_total", "ms_solve", "ms_gram", "ms_kernel_matrix", "ms_score", "ms_tensor"]
        keys_sum = ["launches", "smo_iterations", "solve_bytes", "gram_flops", "gram_bytes", "tensor_flops"]
        tm = torch.tensor([acc.get(k, 0.0) for k in keys_max] + [wall, e2e_wall], dtype=torch.float64, device="cuda")
        ts = torch.tensor([acc.get(k, 0.0) for k in keys_sum], dtype=torch.float64, device="cuda")
        if self.dist is not None:
            self.dist.all_reduce(tm, op=self.dist.ReduceOp.MAX)
            self.dist.all_reduce(ts, op=self.dist.ReduceOp.SUM)
        tavg = torch.tensor([acc.get(k, 0.0) for k in keys_max], dtype=torch.float64, device="cuda")
        if self.dist is not None:
            self.dist.all_reduce(tavg, op=self.dist.ReduceOp.SUM)
        r = dict(zip(keys_max + ["wall", "e2e_wall"], [float(x) for x in tm.cpu()]))
        r.update(zip(keys_sum, [float(x) for x in ts.cpu()]))
        r["phase_mean"] = dict(zip(keys_max, [float(x) / max(self.world, 1) for x in tavg.cpu()]))
        r.update(test=out["test"], train=out["train"], e2e_prof=e2e_prof, clocks=clocks, steps=steps)
        return r


def secondary_entry(key, rank, world, local_rank, dist, steps, peaks, dump_dir=None):
    """One BASELINE config, strong-scaled over the ranks: value, e2e, parity vs golden, roofline of its dominant kernel."""
    from spark_sklearn_b200 import workloads as WL
    w = WL.make_workload(key)
    w["golden"] = GOLDEN.get(key)
    run = Runner(w, rank, world, local_rank, dist)
    m = run.measure(steps, 2)
    if rank != 0:
        return None
    if dump_dir:
        dump_outputs(dump_dir, key, m)
    fits, K = run.fits, steps
    ent = {"workload": "%s: %s(%s), %dx%d, %d candidates x cv=%d = %d fits" % (
               w["name"], "GridSearchCV" if w["search"] == "grid" else "RandomizedSearchCV", w["estimator"],
               w["X"].shape[0], w["X"].shape[1], len(run.cands), len(run.splits), fits),
           "n_gpus": world, "scaling": "strong", "steps": K,
           "value": K * fits / (m["ms_total"] * 1e-3), "unit": "fits/s", "ms_per_step": m["ms_total"] / K,
           "e2e": {"value": K * fits / m["e2e_wall"], "unit": "fits/s", "h2d_bytes_per_step": int(m["e2e_prof"].get("h2d_bytes", 0)),
                   "d2h_bytes_per_step": int(m["e2e_prof"].get("d2h_bytes", 0))},
           "gpu_launches": int(m["launches"]), "parity": parity_block(w, m["test"])}
    hbm, tf32 = peaks
    if w["estimator"] == "SVC":
        ach = m["solve_bytes"] / max(world, 1) / (m["ms_solve"] * 1e-3) / 1e9 if m["ms_solve"] > 0 else 0.0
        ent["roofline"] = {"kernel": "batched SMO (smo_lean_kernel / smo_colown_kernel)", "bound": "hbm", "achieved": ach, "peak": hbm,
                           "unit": "GB/s", "frac": ach / hbm, "traffic": None,
                           "note": "per-rank algorithmic bytes (n_iter * 2 rows * l * 4 B) / solve-phase event time (max over ranks)"}
    else:
        ach = m["tensor_flops"] / max(world, 1) / (m["ms_tensor"] * 1e-3) / 1e12 if m["ms_tensor"] > 0 else 0.0
        ent["roofline"] = {"kernel": "gemm_nt_tf32x3_kernel (tcgen05 kind::tf32, TMA operands, 3xTF32 split)", "bound": "tensor",
                           "achieved": ach, "peak": tf32, "unit": "TFLOP/s", "frac": ach / tf32 if tf32 else None, "traffic": None,
                           "tensor_ms_per_step": m["ms_tensor"] / K, "share_of_step": m["ms_tensor"] / m["ms_total"] if m["ms_total"] else None,
                           "note": "executed TF32 tensor flops (3 MMAs per fp32-faithful product) of all contraction launches of a step / "
                                   "their CUDA-event time; peak = cuBLAS TF32 8192^3 measured in this run"}
    run.plan.close()
    return ent


# ----------------------------------------------------------------------------- main -------------
def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--workload", default="c2")
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-secondary", action="store_true")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="after the timed steps, write the split scores of every measured workload's last step to "
                         "DIR/<workload>_{test,train}_scores.npy (float64; the inputs are seeded, so runs and builds compare)")
    a = ap.parse_args()
    if a.steps < 1:
        ap.error("--steps must be at least 1")
    if a.dump_outputs and a.impl != "ours":
        ap.error("--dump-outputs writes the outputs of --impl ours")
    # stdout carries exactly ONE line (the JSON): libraries that print there (NCCL's version banner, joblib) go to stderr
    sys.stdout.flush()
    real_stdout = os.fdopen(os.dup(1), "w")
    os.dup2(2, 1)
    sys.stdout = sys.stderr

    def emit(obj):
        real_stdout.write(json.dumps(obj) + "\n")
        real_stdout.flush()

    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    cores = effective_cores()
    W_ = max(a.warmup, 0)

    w = scaled_workload(a.workload, max(a.gpus, world))
    from spark_sklearn_b200 import workloads as WL
    cands = WL.candidates(w)
    n_splits = w["cv"]
    cfg = {"workload": "%s: GridSearchCV(%s %s), synthetic %dx%d fp32, %d candidates x cv=%d"
                       % (w["name"], w["estimator"], w["est_params"], w["X"].shape[0], w["X"].shape[1], len(cands), n_splits),
           "n_candidates": len(cands), "n_splits": n_splits, "fits_per_step": len(cands) * n_splits,
           "parallelism": "candidates dealt by predicted cost over %d GPU(s), dataset replicated, one score all-gather" % max(world, 1),
           "l2": "inputs larger than L2 (float64 Gram 0.8 GB + float32 kernel matrices 0.4 GB each)", "refit": False}

    # ---------------- reference arm: the CPU path on the host cores (rank 0 only) ----------------
    if a.impl == "reference":
        if rank != 0:
            return
        cb, idx, _ = cpu_reference(w, cands, cores, a.steps, W_)
        v = cb["value"]
        emit(({
            "impl": "reference", "metric": "candidate-fits/sec", "value": v, "unit": "fits/s", "n_gpus": a.gpus,
            "steps": a.steps, "warmup": W_, "ms_per_step": 1e3 * cb["seconds"] / max(a.steps, 1), "higher_is_better": True,
            "scaling": "weak", "vs_baseline": None, "dtype": "f64", "data": "synthetic", "config": cfg,
            "cpu_baseline": cb,
            "e2e": {"value": v, "unit": "fits/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
            "gpu_launches": 0}))
        return

    # ---------------- our arm -----------------------------------------------------------------------
    import torch
    # the contract measures N GPUs = N torchrun ranks with one GPU each: a plain fit() must not fan out over the other
    # visible GPUs of the node (the in-process scheduler is measured separately below, `in_process`)
    os.environ["B200GS_DEVICES"] = "1"
    dist = None
    if world > 1:
        import torch.distributed as dist
        torch.cuda.set_device(local_rank)
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))
    run = Runner(w, rank, world, local_rank, dist)
    sampler = ClockSampler(local_rank) if rank == 0 else None
    m = run.measure(a.steps, W_, sampler)
    test_scores = m["test"]
    fits = run.fits
    if a.dump_outputs and rank == 0:
        dump_outputs(a.dump_outputs, a.workload, m)

    peak, peak_src = measured_peaks()
    secondary = None
    if not a.no_secondary and a.workload == "c2":
        tf32 = tf32_peak_tflops() if rank == 0 else 0.0
        secondary = {}
        for key in ("c4", "c3", "c5"):
            ent = secondary_entry(key, rank, world, local_rank, dist, a.steps, (peak, tf32), a.dump_outputs)
            if rank == 0:
                secondary[key] = ent
        if rank == 0:
            secondary["tf32_peak_tflops"] = tf32
            secondary["note"] = ("BASELINE configs 4 / 3 / 5 in this same run, STRONG-scaled over the %d rank(s); efficiency at N "
                                 "= value(N) / (N * value(1)) of the same entry" % world)

    if rank != 0:
        if dist is not None:
            dist.destroy_process_group()
        return

    K = max(a.steps, 1)
    # roofline of the dominant kernel: batched SMO, HBM-bound by design (row gathers)
    per_launch_bytes = m["solve_bytes"] / K / max(world, 1)
    per_launch_s = m["ms_solve"] / K * 1e-3
    achieved = per_launch_bytes / per_launch_s / 1e9 if per_launch_s > 0 else 0.0
    traffic, traffic_src = None, None
    tp = os.path.join(ROOT, "profiles", "traffic.json")      # DRAM bytes of the SMO launches of one step, from an ncu capture
    if os.path.exists(tp) and world <= 1:
        t = json.load(open(tp)).get(a.workload)
        if t:
            traffic, traffic_src = float(t["dram_bytes_per_step"]), t["source"]
    roofline = {"kernel": "smo_lean_kernel (one CTA per sub-problem, two per SM) + smo_colown_kernel (thread-block cluster per critical-path "
                          "sub-problem), launched concurrently: batched exact-trajectory C-SVC SMO", "bound": "hbm",
                "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak, "peak_source": peak_src,
                "traffic": traffic, "traffic_source": traffic_src,
                "algorithmic_bytes_per_launch": per_launch_bytes,
                "note": "algorithmic bytes = sum over sub-problems of n_iter * 2 rows * l * 4 B (SURVEY.md 8d) per step (both SMO "
                        "launches); time = the solve phase of the step from CUDA events on the engine stream"}
    gram_s = m["ms_gram"] / K * 1e-3
    gram_ach = (m["gram_bytes"] / K / max(world, 1)) / gram_s / 1e9 if gram_s > 0 else 0.0
    gram_roofline = {"kernel": "gram_f64_kernel (X X^T in float64, shared by every candidate, fold and pair)", "bound": "hbm",
                     "achieved": gram_ach, "peak": peak, "unit": "GB/s", "frac": gram_ach / peak,
                     "ms_per_step": m["ms_gram"] / K, "share_of_step": m["ms_gram"] / m["ms_total"] if m["ms_total"] else None,
                     "note": "north_star's Gram-build roofline: algorithmic bytes (read X once, write S once) / event time; the float64-exact "
                             "Gram runs on the FP64 pipe (%.1f TFLOP/s), far from the HBM floor, and is ~1%% of the step"
                             % (m["gram_flops"] / K / max(world, 1) / gram_s / 1e12 if gram_s > 0 else 0.0)}
    result = {
        "metric": "candidate-fits/sec", "value": K * fits / (m["ms_total"] * 1e-3), "unit": "fits/s", "n_gpus": max(world, 1),
        "steps": a.steps, "warmup": W_, "ms_per_step": m["ms_total"] / K, "higher_is_better": True,
        "scaling": "weak", "vs_baseline": None, "dtype": "f64", "data": "synthetic", "config": cfg,
        "wall_ms_per_step": 1e3 * m["wall"] / K,
        "e2e": {"value": K * fits / m["e2e_wall"], "unit": "fits/s",
                "h2d_bytes_per_step": int(m["e2e_prof"].get("h2d_bytes", 0)), "d2h_bytes_per_step": int(m["e2e_prof"].get("d2h_bytes", 0)),
                "api": "spark_sklearn_b200.GridSearchCV(sc=None, ..., refit=False).fit(X, y) with host numpy arrays"},
        "gpu_launches": int(m["launches"]), "smo_iterations_per_step": m["smo_iterations"] / K,
        # device ms per step of the phases of a search (CUDA events on the engine stream): slowest rank / mean over the ranks
        "phases_ms": {k[3:]: {"max": m[k] / K, "mean": m["phase_mean"][k] / K}
                      for k in ("ms_total", "ms_gram", "ms_kernel_matrix", "ms_solve", "ms_score")},
        "roofline": roofline, "gram_roofline": gram_roofline, "clocks": m["clocks"],
        "best_mean_test_score": float(np.max(np.mean(test_scores, 1))),
        "parity": parity_block(w, test_scores),
    }
    if result["parity"] is not None and w["estimator"] == "SVC":
        # the bar of BASELINE.json (1e-4 on mean_test_score) enforced inside the measured run; observed: bit-identical splits
        assert result["parity"]["max_abs_diff_mean_test_score"] <= 1e-4, result["parity"]
    if secondary is not None:
        result["secondary"] = secondary
    if world == 1:
        from spark_sklearn_b200.engine import device_count
        nd = device_count()
        if nd > 1:                                               # north_star's single in-process scheduler: ONE fit() over every GPU of the node
            from spark_sklearn_b200 import GridSearchCV
            os.environ["B200GS_DEVICES"] = "all"
            est = WL.make_estimator(w)
            for _ in range(2):
                s_ = GridSearchCV(None, est, w["param_grid"], cv=w["cv"], refit=False).fit(w["X"], w["y"])
            t0 = time.perf_counter()
            s_ = GridSearchCV(None, est, w["param_grid"], cv=w["cv"], refit=False).fit(w["X"], w["y"])
            dt = time.perf_counter() - t0
            os.environ["B200GS_DEVICES"] = "1"
            got = np.stack([s_.cv_results_["split%d_test_score" % k] for k in range(n_splits)], 1)
            result["in_process"] = {"devices": len(s_.devices_), "e2e_value": fits / dt, "unit": "fits/s", "strong_scaling": True,
                                    "scores_equal_single_gpu": bool(np.array_equal(got, test_scores)),
                                    "what": "one GridSearchCV.fit() without torch.distributed: a handle and a host thread per GPU"}
    if not a.no_cpu_baseline and world == 1:
        cb, idx, cpu_split0 = cpu_reference(w, cands, cores, 1, 0)
        cb["max_abs_diff_split0_test_score_vs_gpu"] = float(np.max(np.abs(cpu_split0 - test_scores[idx, 0])))
        result["cpu_baseline"] = cb
    emit(result)
    if dist is not None:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
