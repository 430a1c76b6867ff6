#!/usr/bin/env python
"""Parallel tempering (pyb_hmc_set_temperatures, option "hmc_swap"): cost and benefit, one JSON line per case appended
to --out.

* Cost: device ms per iteration at equal total chain count, three engines alternated iteration by iteration in one
  process: untempered chains, a ladder with "hmc_swap" = 0 (the tempered potential alone) and the same ladder with swaps
  (the swap round on top).  C3: 1024 untempered chains against 256 groups x 4 rungs (60000 x 784 synthetic
  MNIST-shaped data, 784-256-10, L = 20); C1: 16 384 untempered chains against 4096 groups x 4 rungs (make_moons
  2-50-2, N = 1600, L = 30).  Iterations are neither burn-in nor sampling, so no sample arena is involved.
* Benefit: the 1-1-1 tanh regression of tests/test_gpu_hmc_tempering.py, whose posterior is exactly symmetric under
  (w1, b1, w2) -> -(w1, b1, w2), every chain started in the w2 > 0 mode; 512 chains untempered against 64 groups x 8
  rungs (geometric ladder 1 .. 1e-3), both after 300 dual-averaging iterations, then --benefit-iters sampling
  iterations.  Reported: the frequency-weighted fraction of cold draws with w2 > 0 (1/2 when the chains visit both
  modes evenly), the per-pair swap acceptance, and the median / max R-hat of the tracked predictive across the cold
  chains on 64 inputs.

The GPU's name, power limit and SM clocks are read in the same run and written into every line.
Usage: python tools/bench_hmc_tempering.py [--c3-iters 12] [--c1-iters 40] [--benefit-iters 1000] [--out FILE]
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
from bayesian_inference_for_nn_b200.tempering import geometric_ladder  # noqa: E402

LADDER4 = [1.0, 0.7, 0.45, 0.2]


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


def engine(problem, ladder=None, swap=True):
    spec, X, y, hp = problem
    eng = Engine(spec, seed=1)
    eng.set_dataset(X, y, _lib.LOSS_SPARSE_CE)
    eng.set_prior([0.0], [1.0], _lib.PRIOR_SCALAR)
    if not swap:
        eng.set_option("hmc_swap", 0)
    eng.hmc_init(hp["S"], hp["eps"], hp["m"], hp["L"])
    if ladder is not None:
        eng.hmc_set_temperatures(ladder)
    return eng


def cost(problem, iters, warmup):
    engs = {"untempered": engine(problem), "ladder_no_swap": engine(problem, LADDER4, swap=False),
            "ladder_swap": engine(problem, LADDER4)}
    for e in engs.values():
        e.hmc_run(warmup, burning=False, sampling=False)
    ms = {k: [] for k in engs}
    for _ in range(iters):
        for k, e in engs.items():
            ms[k].append(e.hmc_run(1, burning=False, sampling=False)["device_ms"])
    st = engs["ladder_swap"].hmc_tempering_stats()
    path = engs["untempered"].info("path_used")
    for e in engs.values():
        e.close()
    med = {k: float(np.median(v)) for k, v in ms.items()}
    out = {"ms_per_iteration_median_" + k: v for k, v in med.items()}
    out.update({"ms_per_iteration_min_" + k: float(np.min(v)) for k, v in ms.items()})
    out.update(overhead_tempered_potential=med["ladder_no_swap"] / med["untempered"] - 1.0,
               overhead_swap_round=med["ladder_swap"] / med["ladder_no_swap"] - 1.0,
               overhead_total=med["ladder_swap"] / med["untempered"] - 1.0, ladder=LADDER4,
               last_iteration_swaps_accepted=st["swap_accepted"].tolist(),
               last_iteration_swaps_attempted=st["swap_attempted"].tolist(), timed_iterations_each=iters, warmup=warmup,
               order="untempered, ladder_no_swap, ladder_swap alternated", path_used=path)
    return out


def benefit(n_samp, n_adapt=300):
    rng = np.random.default_rng(2)
    X = rng.uniform(-2, 2, (50, 1)).astype(np.float32)
    y = (2.0 * np.tanh(1.5 * X) + rng.normal(0, 0.1, X.shape)).astype(np.float32)
    xt = np.linspace(-2.5, 2.5, 64, dtype=np.float32).reshape(-1, 1)
    spec = keras_json.parse_model_json(keras_json.make_sequential_json(1, [1, 1], ["tanh", "linear"]))
    out = {}
    ladder = geometric_ladder(8, 1e-3)
    for label, lad in (("untempered_512_chains", None), ("tempered_64_groups_x_8", ladder)):
        eng = Engine(spec, seed=5)
        eng.set_dataset(X, y, _lib.LOSS_MSE)
        eng.set_prior([0.0], [1.0], _lib.PRIOR_SCALAR)
        S = 512
        eng.hmc_init(S, 0.01, 1.0, 10, semantics=_lib.HMC_CANONICAL, q0=np.tile(np.array([1.5, 0, 2.0, 0], np.float32), (S, 1)))
        if lad is not None:
            eng.hmc_set_temperatures(lad)
        eng.hmc_track_predictive(xt)
        eng.hmc_adapt_begin(0.7)
        eng.hmc_run(n_adapt, burning=False, sampling=False)
        eng.hmc_adapt_end()
        d = eng.hmc_run(n_samp, burning=False, sampling=True)
        s, f, _ = eng.hmc_samples()
        frac = float(np.sum(f * (s[:, 2] > 0)) / np.sum(f))
        sums, s2, T = eng.hmc_predictive_sums()
        G = S // (1 if lad is None else len(lad))
        rhat = eng.hmc_predictive_finish(sums, s2, G, T)["rhat"]
        ok = np.isfinite(rhat)
        rec = {"w2_positive_fraction": frac, "cold_chains": G, "sampling_iterations": n_samp,
               "sampling_device_ms": d["device_ms"], "rhat_median": float(np.median(rhat[ok])) if ok.any() else None,
               "rhat_max": float(rhat[ok].max()) if ok.any() else None}
        if lad is not None:
            st = eng.hmc_tempering_stats()
            rec.update(ladder=lad, swap_accept_last_call=(st["swap_accepted"] / np.maximum(1, st["swap_attempted"])).tolist(),
                       rung_accept_last_call=(st["rung_accepted"] / np.maximum(1, st["rung_total"])).tolist())
        out[label] = rec
        eng.close()
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--c3-iters", type=int, default=12)
    ap.add_argument("--c1-iters", type=int, default=40)
    ap.add_argument("--warmup", type=int, default=2)
    ap.add_argument("--benefit-iters", type=int, default=1000)
    ap.add_argument("--out", default=os.path.join("profiles", "r5_hmc_tempering.jsonl"))
    ap.add_argument("--skip-c3", action="store_true")
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

    emit(dict(case="benefit: 1-1-1 tanh sign-symmetric posterior, 512 chains untempered vs 64 groups x 8 rungs",
              **benefit(args.benefit_iters)))
    emit(dict(case="cost C1: 16384 untempered chains vs 4096 groups x 4 rungs, hmc_swap 0 / 1 (moons 2-50-2, L=30)",
              **cost(c1_problem(), args.c1_iters, args.warmup)))
    if not args.skip_c3:
        emit(dict(case="cost C3: 1024 untempered chains vs 256 groups x 4 rungs, hmc_swap 0 / 1 (784-256-10, L=20)",
                  **cost(c3_problem(), args.c3_iters, args.warmup)))


if __name__ == "__main__":
    main()
