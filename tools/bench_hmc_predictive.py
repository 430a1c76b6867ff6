#!/usr/bin/env python
"""Cost of the streamed HMC predictive (pyb_hmc_track_predictive), one JSON line per case appended to --out.

* C3 (1024 chains, 60000 x 784 synthetic MNIST-shaped data, 784-256-10, L = 20, 10 000 tracked test rows): device ms
  per sampling iteration without and with tracking, the two engines alternated iteration by iteration in one process.
  Both keep their samples; warm-up + timed iterations stay inside one sample arena (<= 40 iterations at this size),
  so no arena is flushed to the host during the comparison.
* C3 with hmc_keep_samples = 0 and tracking for --flat-iters iterations: host wall time of every iteration (max /
  median) and the growth of the process RSS — what a long run costs when only the predictive is kept.
* C1 (16 384 chains, make_moons 2-50-2, N = 1600, L = 30) with a 100 x 100 grid as the tracked inputs, alternated as C3.

The GPU's name, power limit and SM clocks are read in the same run and written into every line.
Usage: python tools/bench_hmc_predictive.py [--iters 20] [--warmup 2] [--flat-iters 200] [--out FILE]
"""
import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from bayesian_inference_for_nn_b200 import _lib, keras_json  # noqa: E402
from bayesian_inference_for_nn_b200.engine import Engine  # noqa: E402


def gpu_info():
    q = "name,power.limit,clocks.sm,clocks.max.sm"
    r = subprocess.run(["nvidia-smi", "--query-gpu=" + q, "--format=csv,noheader", "-i", "0"], capture_output=True,
                       text=True)
    vals = [v.strip() for v in r.stdout.strip().split(",")] if r.returncode == 0 else []
    return dict(zip(q.split(","), vals)) if len(vals) == 4 else {"nvidia_smi": "unavailable"}


def rss_mb():
    with open("/proc/self/status") as f:
        for line in f:
            if line.startswith("VmRSS:"):
                return int(line.split()[1]) / 1024.0
    return float("nan")


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
    xt = rng.random((10000, 784), dtype=np.float32)
    yt = rng.integers(0, 10, 10000).astype(np.int32)
    spec = keras_json.parse_model_json(keras_json.make_sequential_json(784, [256, 10], ["relu", "softmax"]))
    return spec, X, y, xt, yt, dict(S=1024, eps=2e-5, m=1.0, L=20)


def c1_problem():
    X, y = moons(1600)
    g = np.stack(np.meshgrid(np.linspace(-2, 3, 100), np.linspace(-1.5, 2, 100)), -1).reshape(-1, 2).astype(np.float32)
    yt = (g[:, 1] < 0.25).astype(np.int32)
    spec = keras_json.parse_model_json(keras_json.make_sequential_json(2, [50, 2], ["relu", "softmax"]))
    return spec, X, y, g, yt, dict(S=16384, eps=0.005, m=0.5, L=30)


def engine(problem, track, keep=True):
    spec, X, y, xt, yt, hp = problem
    eng = Engine(spec, seed=1)
    eng.set_dataset(X, y, _lib.LOSS_SPARSE_CE)
    eng.set_prior([0.0], [1.0], _lib.PRIOR_SCALAR)
    if not keep:
        eng.set_option("hmc_keep_samples", 0)
    eng.hmc_init(hp["S"], hp["eps"], hp["m"], hp["L"])
    if track:
        eng.hmc_track_predictive(xt, yt)
    return eng


def alternate(problem, iters, warmup):
    off, on = engine(problem, False), engine(problem, True)
    for e in (off, on):
        e.hmc_run(warmup, burning=False, sampling=True)
    ms = {"off": [], "on": []}
    for _ in range(iters):
        ms["off"].append(off.hmc_run(1, burning=False, sampling=True)["device_ms"])
        ms["on"].append(on.hmc_run(1, burning=False, sampling=True)["device_ms"])
    path = on.info("path_used")
    on.hmc_predictive_sums()                          # the read-out works at this size
    off.close()
    on.close()
    med = {k: float(np.median(v)) for k, v in ms.items()}
    return {"ms_per_iteration_median_off": med["off"], "ms_per_iteration_median_on": med["on"],
            "ms_per_iteration_mean_off": float(np.mean(ms["off"])), "ms_per_iteration_mean_on": float(np.mean(ms["on"])),
            "overhead_median": med["on"] / med["off"] - 1.0, "timed_iterations_each": iters, "warmup": warmup,
            "path_used": path}


def flat(problem, iters, warmup):
    eng = engine(problem, True, keep=False)
    eng.hmc_run(warmup, burning=False, sampling=True)
    rss0 = rss_mb()
    wall = []
    for _ in range(iters):
        t0 = time.perf_counter()
        eng.hmc_run(1, burning=False, sampling=True)
        wall.append(time.perf_counter() - t0)
    rss1 = rss_mb()
    rows = eng.info("hmc_arena_rows")
    eng.close()
    w = np.asarray(wall) * 1e3
    return {"iterations": iters, "wall_ms_median": float(np.median(w)), "wall_ms_max": float(w.max()),
            "max_over_median": float(w.max() / np.median(w)), "rss_mb_start": rss0, "rss_mb_end": rss1,
            "rss_growth_mb": rss1 - rss0, "hmc_arena_rows": rows}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--iters", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=2)
    ap.add_argument("--flat-iters", type=int, default=200)
    ap.add_argument("--out", default=os.path.join("profiles", "r3_hmc_predictive.jsonl"))
    args = ap.parse_args()
    if args.iters + args.warmup > 38:
        ap.error("--iters + --warmup must stay within one sample arena (<= 38 at C3)")
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

    c3 = c3_problem()
    emit(dict(case="C3 tracking off vs on (1024 chains, 784-256-10, L=20, Nt=10000)", **alternate(c3, args.iters, args.warmup)))
    emit(dict(case="C3 hmc_keep_samples=0 with tracking", **flat(c3, args.flat_iters, args.warmup)))
    emit(dict(case="C1 tracking off vs on (16384 chains, moons 2-50-2, L=30, 100x100 grid)",
              **alternate(c1_problem(), args.iters, args.warmup)))


if __name__ == "__main__":
    main()
