#!/usr/bin/env python
"""Per-chain HMC step sizes and their dual-averaging adaptation (pyb_hmc_adapt_begin / _end, pyb_hmc_set_step_sizes):
cost, benefit and the default path, one JSON line per case appended to --out.

* Cost: device ms per iteration of the scalar path against per-chain step sizes all set to epsilon (the same chains,
  bit for bit), the two engines alternated iteration by iteration in one process; C3 (1024 chains, 60000 x 784
  synthetic MNIST-shaped data, 784-256-10, L = 20) and C1 (16 384 chains, make_moons 2-50-2, N = 1600, L = 30).
  Iterations are neither burn-in nor sampling, so no sample arena is involved.
* Benefit: C1 at the reference's own settings (epsilon = 0.005, m = 0.5, L = 30, prior sigma = 1): the reference's 10
  burn-in iterations, then --benefit-iters sampling iterations, once without adaptation and once after --adapt-iters
  adaptation iterations (target 0.8).  Reported: the accept rate of the sampling iterations, min / median / max of the
  per-chain step sizes, and the median / max R-hat of the tracked predictive on a 100 x 100 grid.
* Default path (--parent DIR, a checkout of the parent commit with its library built): `bench.py` at C3 (headline
  only) run alternately from DIR and from this tree, --bench-runs times each; the `value` of every run.

The GPU's name, power limit and SM clocks are read in the same run and written into every line.
Usage: python tools/bench_hmc_adapt.py [--c3-iters 12] [--c1-iters 40] [--adapt-iters 500] [--benefit-iters 200]
                                       [--parent DIR] [--bench-runs 3] [--out FILE]
"""
import argparse
import json
import os
import subprocess
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
from bayesian_inference_for_nn_b200 import _lib, keras_json  # noqa: E402
from bayesian_inference_for_nn_b200.engine import Engine  # noqa: E402


def gpu_info():
    q = "name,power.limit,clocks.sm,clocks.max.sm"
    r = subprocess.run(["nvidia-smi", "--query-gpu=" + q, "--format=csv,noheader", "-i", "0"], capture_output=True,
                       text=True)
    vals = [v.strip() for v in r.stdout.strip().split(",")] if r.returncode == 0 else []
    return dict(zip(q.split(","), vals)) if len(vals) == 4 else {"nvidia_smi": "unavailable"}


def moons(n, seed=0, noise=0.2):
    rng = np.random.default_rng(seed)
    n0 = n // 2
    t0, t1 = rng.uniform(0, np.pi, n0), rng.uniform(0, np.pi, n - n0)
    x = np.concatenate([np.stack([np.cos(t0), np.sin(t0)], 1), np.stack([1 - np.cos(t1), 0.5 - np.sin(t1)], 1)])
    y = np.concatenate([np.zeros(n0, np.int32), np.ones(n - n0, np.int32)])
    return (x + rng.normal(0, noise, x.shape)).astype(np.float32), y


def c3_problem():
    rng = np.random.default_rng(0)
    X = rng.random((60000, 784), dtype=np.float32)
    y = rng.integers(0, 10, 60000).astype(np.int32)
    spec = keras_json.parse_model_json(keras_json.make_sequential_json(784, [256, 10], ["relu", "softmax"]))
    return spec, X, y, dict(S=1024, eps=2e-5, m=1.0, L=20)


def c1_problem():
    X, y = moons(1600)
    spec = keras_json.parse_model_json(keras_json.make_sequential_json(2, [50, 2], ["relu", "softmax"]))
    return spec, X, y, dict(S=16384, eps=0.005, m=0.5, L=30)


def engine(problem, per_chain=False, keep=True):
    spec, X, y, hp = problem
    eng = Engine(spec, seed=1)
    eng.set_dataset(X, y, _lib.LOSS_SPARSE_CE)
    eng.set_prior([0.0], [1.0], _lib.PRIOR_SCALAR)
    if not keep:
        eng.set_option("hmc_keep_samples", 0)
    eng.hmc_init(hp["S"], hp["eps"], hp["m"], hp["L"])
    if per_chain:
        eng.hmc_set_step_sizes(np.full(hp["S"], hp["eps"]))
    return eng


def cost(problem, iters, warmup):
    scalar, per_chain = engine(problem), engine(problem, per_chain=True)
    for e in (scalar, per_chain):
        e.hmc_run(warmup, burning=False, sampling=False)
    ms = {"scalar": [], "per_chain": []}
    for _ in range(iters):
        ms["scalar"].append(scalar.hmc_run(1, burning=False, sampling=False)["device_ms"])
        ms["per_chain"].append(per_chain.hmc_run(1, burning=False, sampling=False)["device_ms"])
    same = all(np.array_equal(u, v) for u, v in zip(scalar.hmc_state(), per_chain.hmc_state()))
    path = scalar.info("path_used")
    scalar.close()
    per_chain.close()
    med = {k: float(np.median(v)) for k, v in ms.items()}
    return {"ms_per_iteration_median_scalar": med["scalar"], "ms_per_iteration_median_per_chain": med["per_chain"],
            "ms_per_iteration_min_scalar": float(np.min(ms["scalar"])),
            "ms_per_iteration_min_per_chain": float(np.min(ms["per_chain"])),
            "overhead_median": med["per_chain"] / med["scalar"] - 1.0, "timed_iterations_each": iters,
            "warmup": warmup, "states_bit_identical": bool(same), "path_used": path}


def benefit(n_adapt, n_samp):
    problem = c1_problem()
    g = np.stack(np.meshgrid(np.linspace(-2, 3, 100), np.linspace(-1.5, 2, 100)), -1).reshape(-1, 2).astype(np.float32)
    out = {}
    for label, n in (("no_adaptation", 0), ("adapted", n_adapt)):
        eng = engine(problem, keep=False)
        eng.hmc_track_predictive(g)
        eng.hmc_run(10, burning=True, sampling=False)          # the reference's burn-in
        adapt_ms = 0.0
        if n:
            eng.hmc_adapt_begin(0.8)
            adapt_ms = eng.hmc_run(n, burning=False, sampling=False)["device_ms"]
            eng.hmc_adapt_end()
        d = eng.hmc_run(n_samp, burning=False, sampling=True)
        sums, s2, T = eng.hmc_predictive_sums()
        rhat = eng.hmc_predictive_finish(sums, s2, eng.S, T)["rhat"]
        st = eng.hmc_step_sizes()
        ok = np.isfinite(rhat)
        out[label] = {"adapt_iterations": n, "adapt_device_ms": adapt_ms, "sampling_iterations": n_samp,
                      "sampling_accept_rate": d["accept_rate"], "sampling_device_ms": d["device_ms"],
                      "step_min": float(st.min()), "step_median": float(np.median(st)), "step_max": float(st.max()),
                      "rhat_median": float(np.median(rhat[ok])) if ok.any() else None,
                      "rhat_max": float(rhat[ok].max()) if ok.any() else None,
                      "rhat_undefined_elements": int((~ok).sum()), "n_draws_per_chain": T}
        eng.close()
    return out


def default_path(parent, runs):
    cmd = ["--gpus", "1", "--steps", "3", "--warmup", "3", "--no-cpu-baseline", "--no-extras", "--no-e2e"]
    vals = {"parent": [], "branch": []}
    parent = os.path.abspath(parent)
    for _ in range(runs):
        for label, root in (("parent", parent), ("branch", ROOT)):
            r = subprocess.run([sys.executable, os.path.join(root, "bench.py")] + cmd, cwd=root, capture_output=True,
                               text=True)
            lines = [l for l in r.stdout.splitlines() if l.startswith("{")]
            if r.returncode != 0 or not lines:
                raise RuntimeError("bench.py failed in %s:\n%s\n%s" % (root, r.stdout[-2000:], r.stderr[-2000:]))
            vals[label].append(json.loads(lines[-1])["value"])
    return {"bench_args": " ".join(cmd), "value_parent": vals["parent"], "value_branch": vals["branch"],
            "median_parent": float(np.median(vals["parent"])), "median_branch": float(np.median(vals["branch"])),
            "runs_each": runs, "order": "parent, branch alternated"}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--c3-iters", type=int, default=12)
    ap.add_argument("--c1-iters", type=int, default=40)
    ap.add_argument("--warmup", type=int, default=2)
    ap.add_argument("--adapt-iters", type=int, default=500)
    ap.add_argument("--benefit-iters", type=int, default=200)
    ap.add_argument("--parent", default=None, help="checkout of the parent commit with its library built")
    ap.add_argument("--bench-runs", type=int, default=3)
    ap.add_argument("--out", default=os.path.join("profiles", "r4_hmc_adapt.jsonl"))
    args = ap.parse_args()
    if _lib.device_count() == 0:
        sys.exit("no GPU: nothing measured")
    info = gpu_info()
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)

    def emit(rec):
        rec.update(gpu=info)
        line = json.dumps(rec)
        print(line, flush=True)
        with open(args.out, "a") as f:
            f.write(line + "\n")

    emit(dict(case="cost C3: scalar step vs per-chain step sizes = epsilon (1024 chains, 784-256-10, L=20)",
              **cost(c3_problem(), args.c3_iters, args.warmup)))
    emit(dict(case="cost C1: scalar step vs per-chain step sizes = epsilon (16384 chains, moons 2-50-2, L=30)",
              **cost(c1_problem(), args.c1_iters, args.warmup)))
    emit(dict(case="benefit C1 (16384 chains, eps=0.005, m=0.5, L=30, sigma=1, 100x100 grid): no adaptation vs "
                   "dual averaging to 0.8", **benefit(args.adapt_iters, args.benefit_iters)))
    if args.parent:
        emit(dict(case="default path: bench.py C3 headline, parent commit vs this tree", **default_path(args.parent,
                                                                                                     args.bench_runs)))


if __name__ == "__main__":
    main()
