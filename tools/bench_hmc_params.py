#!/usr/bin/env python
"""Cost of the streamed per-parameter moments (pyb_hmc_track_params), one JSON line per case appended to --out.

* C3 (1024 chains, 60000 x 784 synthetic MNIST-shaped data, 784-256-10, L = 20) and C1 (16 384 chains, make_moons
  2-50-2, N = 1600, L = 30): device ms per sampling iteration without and with the tracking, two engines alternated
  iteration by iteration in one process, and the device bytes the tracking holds (pyb_get_info "hmc_param_bytes").
  Neither engine keeps samples (hmc_keep_samples = 0), so no sample arena is flushed to the host inside the comparison.

The GPU's name, power limit and SM clocks are read in the same run and written into every line.
Usage: python tools/bench_hmc_params.py [--iters 20] [--warmup 2] [--out FILE]
"""
import argparse
import json
import os
import subprocess
import sys

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


def engine(problem, n_planned):
    spec, X, y, hp = problem
    eng = Engine(spec, seed=1)
    eng.set_dataset(X, y, _lib.LOSS_SPARSE_CE)
    eng.set_prior([0.0], [1.0], _lib.PRIOR_SCALAR)
    eng.set_option("hmc_keep_samples", 0)
    eng.hmc_init(hp["S"], hp["eps"], hp["m"], hp["L"])
    if n_planned:
        eng.hmc_track_params(n_planned)
    return eng


def alternate(problem, iters, warmup):
    n_planned = warmup + iters + 1
    off, on = engine(problem, 0), engine(problem, n_planned)
    nbytes = on.info("hmc_param_bytes")
    for e in (off, on):
        e.hmc_run(warmup, burning=False, sampling=True)
    ms = {"off": [], "on": []}
    for _ in range(iters):
        ms["off"].append(off.hmc_run(1, burning=False, sampling=True)["device_ms"])
        ms["on"].append(on.hmc_run(1, burning=False, sampling=True)["device_ms"])
    path = on.info("path_used")
    sums, T = on.hmc_param_sums()                     # the read-out and the finish work at this size
    r = on.hmc_param_finish(sums, on.S, T, n_planned)
    off.close()
    on.close()
    med = {k: float(np.median(v)) for k, v in ms.items()}
    return {"ms_per_iteration_median_off": med["off"], "ms_per_iteration_median_on": med["on"],
            "ms_per_iteration_mean_off": float(np.mean(ms["off"])), "ms_per_iteration_mean_on": float(np.mean(ms["on"])),
            "overhead_median": med["on"] / med["off"] - 1.0, "timed_iterations_each": iters, "warmup": warmup,
            "hmc_param_bytes": nbytes, "n_draws": T, "ess_median": float(np.nanmedian(r["ess"])),
            "path_used": path}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--iters", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=2)
    ap.add_argument("--out", default=os.path.join("profiles", "r6_hmc_params.jsonl"))
    args = ap.parse_args()
    if args.iters < 2 or args.warmup < 0:
        ap.error("--iters must be >= 2 and --warmup >= 0")
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

    emit(dict(case="C3 parameter tracking off vs on (1024 chains, 784-256-10, L=20)",
              **alternate(c3_problem(), args.iters, args.warmup)))
    emit(dict(case="C1 parameter tracking off vs on (16384 chains, moons 2-50-2, L=30)",
              **alternate(c1_problem(), args.iters, args.warmup)))


if __name__ == "__main__":
    main()
