#!/usr/bin/env python
"""bench.py — posterior grad-evals/s (chains x leapfrog steps) of the HMC hot path on B200.

Workload (BASELINE.json configs[2], the config the metric and the >=1024-chain target are quoted
on; it fits one GPU): HMC, 1024 chains per GPU, synthetic MNIST-shaped data 60000x784 (U[0,1),
labels U{0..9}), 784-256-10 MLP, L=20, Gaussian prior N(0,1), reference leapfrog semantics.
One "step" = one HMC sampling iteration of every local chain: momentum draw, L full-dataset
log-posterior forward/backward evaluations at the L new positions (the evaluation at the start position is
carried from the previous iteration - its end point if accepted, its start if rejected - with bit-identical
results, tests/test_gpu_parity.py::test_carried_evaluation_is_bit_identical_to_re_evaluation; the reference
re-evaluates it, HMC.py:80,82), both Hamiltonians, Metropolis accept, sample bookkeeping.
The metric counts S*L grad-evals per step (BASELINE.md §2); `evals_executed_per_step_per_chain` in the
config is what the library actually ran (L; L+1 in the e2e leg, whose re-uploaded dataset drops the carry).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl reference] [--dump-outputs DIR]

`--dump-outputs DIR` writes, after the timed steps, what the last of them handed its caller (see dump_outputs) as
DIR/<name>.npy, so that two builds run with the same arguments (hence the same seeded inputs) can be compared output
for output.

N>1 is launched by torchrun (one rank per GPU).  Chains shard across ranks with no data-path
collective (weak scaling: 1024 chains per GPU); torch.distributed is used only for the barrier and
the max-over-ranks of the device time.  `--impl reference` times the reference's own loop shape on
the host cores (oracle port: ONE chain, eager per-position evaluation, HMC.py:74-104).
"""
import argparse
import json
import os
import statistics
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

D_IN, HIDDEN, N_CLS = 784, 256, 10
FLOPS_PER_GRADEVAL = 2.0 * (D_IN * HIDDEN + HIDDEN * N_CLS) + 2.0 * (D_IN * HIDDEN + 2 * HIDDEN * N_CLS)  # per row


def parse_args():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=3)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    # development overrides (the defaults ARE the named config; a line with overrides says so)
    ap.add_argument("--chains", type=int, default=int(os.environ.get("PYB_BENCH_CHAINS", 1024)))
    ap.add_argument("--rows", type=int, default=int(os.environ.get("PYB_BENCH_ROWS", 60000)))
    ap.add_argument("--leapfrog", type=int, default=int(os.environ.get("PYB_BENCH_L", 20)))
    ap.add_argument("--eps", type=float, default=2e-5)
    ap.add_argument("--path", default=os.environ.get("PYB_BENCH_PATH", "auto"))
    ap.add_argument("--opt", action="append", default=[], help="development: library option key=value (e.g. tc_fuse=0)")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--no-extras", action="store_true", help="skip the C1 / C2 / C4 / C5 / strong-scaling sub-records")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="write what the last timed step returned as DIR/<name>.npy (rank 0's chains)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "b200":
        ap.error("--dump-outputs applies to the b200 implementation")
    return args


def synth(rows, seed=0):
    rng = np.random.default_rng(seed)
    X = rng.random((rows, D_IN), dtype=np.float32)
    y = rng.integers(0, N_CLS, rows).astype(np.int32)
    return X, y


DUMP_STATE_BYTES = 16 << 20           # per state array; the whole dump stays far below 64 MB


def dump_outputs(eng, out_dir):
    """Write what the last HMC step returns to its caller as float32 DIR/<name>.npy: the per-chain energies, log
    acceptance, decision and loss of that step (hmc_last) and the chains' positions q and momenta p (hmc_state).
    q and p are chains x parameters (833 MB each at the default config), so only a fixed, seeded set of parameter
    columns of them is written: every chain, at most DUMP_STATE_BYTES per array."""
    os.makedirs(out_dir, exist_ok=True)
    q, p = eng.hmc_state()
    S, P = q.shape
    n = max(1, min(P, DUMP_STATE_BYTES // (4 * S)))
    cols = np.sort(np.random.default_rng(0).choice(P, n, replace=False))
    arrays = dict(eng.hmc_last(), q_sampled=q[:, cols], p_sampled=p[:, cols])
    for name, a in arrays.items():
        np.save(os.path.join(out_dir, name + ".npy"), np.ascontiguousarray(a, dtype=np.float32))


def measured_peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        try:
            j = json.load(open(p))
            return {"bf16_sustained": float(j["bf16_tflops_sustained"]), "bf16_burst": float(j["bf16_tflops"]),
                    "hbm": float(j["hbm_gbs"]), "source": "measured"}
        except Exception:
            pass
    return {"bf16_sustained": 1400.0, "bf16_burst": 1590.0, "hbm": 6650.0, "source": "fallback"}


def ncu_traffic(split):
    """dram__bytes_read+write per tensor-core launch (mean over the fused forward, dW2 and dW1 launches of one 148-chain
    batch) from the committed `ncu` captures (profiles/r2_traffic.json: int8 slices; r1_traffic.json: bf16x3); None when
    no capture is committed."""
    try:
        if split:
            return json.load(open(os.path.join(ROOT, "profiles", "r2_traffic.json")))["int8_slices"]["dram_bytes_per_launch_mean"]
        return json.load(open(os.path.join(ROOT, "profiles", "r1_traffic.json")))["tc_gemm_bf16x3"]["dram_bytes_per_launch_mean"]
    except Exception:
        return None


class ClockSampler:
    """nvidia-smi clocks/throttle reasons sampled DURING the timed region."""
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index):
        self.gpu, self.proc, self.lines = gpu_index, None, []

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.gpu), "--query-gpu=" + self.Q,
                                          "--format=csv,noheader,nounits", "-lms", "200"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            threading.Thread(target=lambda: [self.lines.append(l) for l in self.proc.stdout], daemon=True).start()
        except Exception:
            self.proc = None

    def stop(self):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        try:
            self.proc.wait(timeout=5)
        except Exception:
            self.proc.kill()
        sm, mx, reasons = [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for l in self.lines:
            f = [v.strip() for v in l.split(",")]
            if len(f) < 9:
                continue
            try:
                sm.append(float(f[1]))
                mx.append(float(f[2]))
            except ValueError:
                continue
            for n, v in zip(names, f[5:9]):
                if v.lower().startswith("active"):
                    reasons.add(n)
        return {"sm_mhz": statistics.median(sm) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "samples": len(sm), "reasons": sorted(reasons)}


def cpu_reference_run(args, steps, warmup, rows):
    """The reference's loop shape on the host cores: one chain, L+2 gradient + 2 potential
    evaluations per iteration (oracle.reference_style_hmc_iteration follows HMC.py:74-104)."""
    sys.path.insert(0, os.path.join(ROOT, "oracle"))
    import pyesian_oracle as O
    X, y = synth(rows)
    spec = O.MLPSpec(D_IN, [HIDDEN, N_CLS], ["relu", "softmax"])
    mu, sg = O.expand_prior(spec, 0.0, 1.0)
    prob = O.Problem(spec, X, y, O.LOSS_SPARSE_CE, mu, sg)
    rng = np.random.default_rng(0)
    q = np.zeros((1, spec.n_params), np.float32)
    with host_blas_threads() as threads:
        for _ in range(warmup):
            q, _, _ = O.reference_style_hmc_iteration(prob, q, rng, args.eps, 1.0, args.leapfrog)
        t0 = time.perf_counter()
        for _ in range(steps):
            q, _, _ = O.reference_style_hmc_iteration(prob, q, rng, args.eps, 1.0, args.leapfrog)
        dt = time.perf_counter() - t0
    return args.leapfrog * steps / dt, dt, threads[0]


class host_blas_threads:
    """Give NumPy's BLAS every core this process may run on for the CPU legs — torchrun exports OMP_NUM_THREADS=1 to its
    workers, which would time the reference arm on ONE thread at N > 1 — and report the thread count actually in use."""

    def __enter__(self):
        self.used = [1]
        try:
            want = len(os.sched_getaffinity(0))
        except AttributeError:
            want = os.cpu_count() or 1
        try:
            import threadpoolctl
            self._ctl = threadpoolctl.threadpool_limits(limits=want, user_api="blas")
            blas = [m for m in threadpoolctl.threadpool_info() if m.get("user_api") == "blas"]
            self.used[0] = max([int(m.get("num_threads", 1)) for m in blas] or [1])
        except Exception:            # no threadpoolctl: whatever the environment configured
            self._ctl = None
            self.used[0] = int(os.environ.get("OMP_NUM_THREADS", 0)) or want
        return self.used

    def __exit__(self, *exc):
        if self._ctl is not None:
            self._ctl.restore_original_limits()
        return False


def run_reference(args):
    rank = int(os.environ.get("RANK", 0))
    if rank != 0:
        return
    # bounded sample: each step is ONE reference-style iteration of ONE chain on the full dataset
    val, dt, cores = cpu_reference_run(args, args.steps, min(args.warmup, 1), args.rows)
    line = {
        "impl": "reference", "metric": "posterior_grad_evals_per_s", "value": val, "unit": "grad-evals/s",
        "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup, "ms_per_step": 1e3 * dt / max(1, args.steps),
        "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": workload_config(args, 1),
        "cpu_baseline": {"value": val, "unit": "grad-evals/s", "cores": cores, "kind": "port",
                         "sample": "1 chain x %d iterations (L=%d, %d rows x 784, 784-256-10), numpy fp32 BLAS on all "
                                   "host cores; reference loop shape HMC.py:74-104 (TensorFlow is not installable here)"
                                   % (args.steps, args.leapfrog, args.rows)},
        "e2e": {"value": val, "unit": "grad-evals/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
    }
    print(json.dumps(line), flush=True)


def named_default(args):
    return bool(args.chains == 1024 and args.rows == 60000 and args.leapfrog == 20 and not args.opt)


def workload_config(args, world, evals_per_step=None):
    return {"workload": "C3 HMC 784-256-10 MLP, %d chains/GPU, %d rows x 784 synthetic MNIST-shaped, L=%d, "
                        "reference leapfrog semantics, Gaussian prior N(0,1)" % (args.chains, args.rows, args.leapfrog),
            "chains_per_gpu": args.chains, "chains_total": args.chains * world, "rows": args.rows, "L": args.leapfrog,
            "epsilon": args.eps, "evals_executed_per_step_per_chain": evals_per_step if evals_per_step is not None else args.leapfrog + 1,
            "parallelism": "chains sharded x%d, no data-path collective" % world,
            "l2_policy": "inputs exceed L2 (X hi/lo 188 MB + per-chain operands >> 126 MB)",
            "named_config": named_default(args)}


FP32_SIMT_PEAK_TFLOPS = 148 * 128 * 2 * 1.965e9 / 1e12      # 74.4: 148 SMs x 128 FMA lanes x 2 x 1.965 GHz (nominal)


def moons(n, seed=0, noise=0.2):
    rng = np.random.default_rng(seed)
    n0 = n // 2
    t0, t1 = rng.uniform(0, np.pi, n0), rng.uniform(0, np.pi, n - n0)
    x = np.concatenate([np.stack([np.cos(t0), np.sin(t0)], 1), np.stack([1 - np.cos(t1), 0.5 - np.sin(t1)], 1)])
    y = np.concatenate([np.zeros(n0, np.int32), np.ones(n - n0, np.int32)])
    return (x + rng.normal(0, noise, x.shape)).astype(np.float32), y


def run_extras(args, rank, local_rank, world, dist, X, y, peaks):
    """The other named configurations of BASELINE.json (C1, C2, C4, C5) and the strong-scaling point of the headline, each
    a few hundred milliseconds of device time after the timed HMC region: sub-records of the one JSON line (`extra`).
    Every record is device-timed (max over ranks where the work is sharded); a failure is recorded, never raised."""
    from bayesian_inference_for_nn_b200 import _lib, keras_json
    from bayesian_inference_for_nn_b200.engine import Engine
    out = {}

    def maxr(v):
        if dist is None:
            return v
        import torch
        t = torch.tensor([v], dtype=torch.float64, device="cuda")
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item())

    def mlp(D, H, C):
        return keras_json.parse_model_json(keras_json.make_sequential_json(D, [H, C], ["relu", "softmax"]))

    def guarded(name, fn):
        try:
            out[name] = fn()
        except Exception as e:                                   # noqa: BLE001  (a sub-record must not cost the headline)
            out[name] = {"error": "%s: %s" % (type(e).__name__, e)}
        if dist is not None:
            dist.barrier()

    # ---- C1: HMC on make_moons (1600 rows, 2-50-2, L = 30, eps = 0.005, m = 0.5), 16 384 chains per GPU (weak)
    def c1():
        Xm, ym = moons(1600)
        S, L, iters = 16384, 30, 5
        eng = Engine(mlp(2, 50, 2), device=local_rank, seed=1)
        eng.set_dataset(Xm, ym, _lib.LOSS_SPARSE_CE)
        eng.set_prior([0.0], [1.0], _lib.PRIOR_SCALAR)
        eng.hmc_init(S, 0.005, 0.5, L, chain_offset=rank * S)
        eng.hmc_run(3, burning=True, sampling=False)
        d = eng.hmc_run(iters, burning=False, sampling=False)
        ms = maxr(d["device_ms"])
        eng.close()
        rate = world * S * L * iters / (ms / 1e3)
        tf = rate * 1.6e6 / 1e12
        return {"workload": "C1 HMC make_moons 1600x2, 2-50-2, L=30, %d chains/GPU" % S, "value": rate, "unit": "grad-evals/s",
                "ms": ms / iters, "scaling": "weak",
                "roofline": {"bound": "fp32-simt", "achieved": tf, "peak": FP32_SIMT_PEAK_TFLOPS * world, "unit": "TFLOP/s",
                             "frac": tf / (FP32_SIMT_PEAK_TFLOPS * world), "hbm_algorithmic_gbs": rate * 23232 / 1e9,
                             "hbm_frac": rate * 23232 / 1e9 / (peaks["hbm"] * world)}}

    # ---- C2: SVGD on make_moons, 64 particles, full batch (rank 0; 64 particles do not shard usefully)
    def c2():
        if rank != 0:
            return None
        Xm, ym = moons(1600)
        res = {"workload": "C2 SVGD make_moons 1600x2, 2-50-2, 64 particles, full batch (one GPU)"}
        for sem, name in ((_lib.SVGD_CANONICAL_MEDIAN, "canonical_median"), (_lib.SVGD_REFERENCE_LIVE, "reference_live")):
            eng = Engine(mlp(2, 50, 2), device=local_rank, seed=1)
            eng.set_dataset(Xm, ym, _lib.LOSS_SPARSE_CE)
            eng.set_prior([0.0], [1.0], _lib.PRIOR_SCALAR)
            eng.svgd_init(64, 1e-3, sem)
            for _ in range(3):
                eng.svgd_step(None)
            ms = 0.0
            for _ in range(20):
                eng.svgd_step(None)
                ms += eng.info("last_device_ms")
            eng.close()
            res[name] = {"value": 20 / (ms / 1e3), "unit": "steps/s", "ms": ms / 20,
                         "particle_grad_evals_per_s": 64 * 20 / (ms / 1e3)}
        gf = 0.107 * res["canonical_median"]["value"] / 1e3
        res["roofline"] = {"bound": "latency / fp32-simt", "achieved": gf, "peak": FP32_SIMT_PEAK_TFLOPS, "unit": "TFLOP/s",
                           "frac": gf / FP32_SIMT_PEAK_TFLOPS}
        return res

    # ---- C4: SVGD at the SVGD_mnist shape, 4096 particles in total sharded over the ranks (784-128-10, minibatch 1024)
    def c4():
        S_total, B, steps = 4096, 1024, 5
        rng = np.random.default_rng(0)
        idx = [rng.permutation(X.shape[0])[:B].astype(np.int32) for _ in range(steps + 2)]
        eng = Engine(mlp(784, 128, 10), device=local_rank, seed=1)
        eng.set_dataset(X, y, _lib.LOSS_SPARSE_CE)
        eng.set_prior([0.0], [1.0], _lib.PRIOR_SCALAR)
        Sl = S_total // world
        if world > 1:
            import torch
            uid = torch.zeros(128, dtype=torch.uint8, device="cuda")
            if rank == 0:
                uid.copy_(torch.frombuffer(bytearray(_lib.nccl_unique_id()), dtype=torch.uint8))
            dist.broadcast(uid, 0)
            eng.svgd_set_comm(rank, world, bytes(uid.cpu().numpy().tobytes()))
        eng.svgd_init(Sl, 0.01, _lib.SVGD_CANONICAL_MEDIAN, offset=rank * Sl)
        ms, loss = [], None
        for k, ix in enumerate(idx):
            loss = eng.svgd_step(ix)
            if k >= 2:
                ms.append(eng.info("last_device_ms"))
        t = maxr(float(np.mean(ms)))
        p2p = bool(world > 1 and int(eng.info("svgd_p2p")))
        eng.close()
        P = 784 * 128 + 128 + 128 * 10 + 10
        flops = S_total * 6.0 * B * (784 * 128 + 128 * 10) + 4.0 * S_total * S_total * P
        tf = flops / (t / 1e3) / 1e12
        return {"workload": "C4 SVGD 784-128-10, %d particles sharded x%d, minibatch 1024 of %d, median-heuristic RBF"
                            % (S_total, world, X.shape[0]), "value": 1e3 / t, "unit": "steps/s", "ms": t, "scaling": "strong",
                "particle_grad_evals_per_s": S_total * 1e3 / t, "mean_loss": float(loss),
                "exchange": ("none (one GPU)" if world == 1 else "peer-memory stores of the library's kernels + NCCL barriers / Gram "
                             "all-reduce" if p2p else "NCCL send/recv + Gram all-reduce"),
                "roofline": {"bound": "tensor (NVLink exchange at N > 1)", "achieved": tf, "peak": peaks["bf16_sustained"] * world,
                             "unit": "TFLOP/s", "frac": tf / (peaks["bf16_sustained"] * world)}}

    # ---- C5: posterior predictive, 1000 weight samples x 10000 x 784 test rows, 784-256-10 (rank 0)
    def c5():
        if rank != 0:
            return None
        import torch
        n, Nt = 1000, 10000
        g = torch.Generator(device="cuda").manual_seed(0)
        Wd = torch.randn((n, 784 * 256 + 256 + 256 * 10 + 10), generator=g, device="cuda") * 0.05
        xd = torch.rand((Nt, 784), generator=g, device="cuda")
        torch.cuda.synchronize()
        eng = Engine(mlp(784, 256, 10), device=local_rank)
        eng.predict(Wd, xd)
        eng.predict(Wd, xd)
        ms = eng.info("last_device_ms")
        eng.close()
        flops = 2.0 * Nt * (784 * 256 + 256 * 10) * n
        tf = flops / (ms / 1e3) / 1e12
        return {"workload": "C5 predictive 1000 weight samples x 10000x784, 784-256-10, mean / variance on the device, samples "
                            "and inputs resident in HBM (one GPU)", "value": n / (ms / 1e3), "unit": "samples/s", "ms": ms,
                "rows_x_samples_per_s": n * Nt / (ms / 1e3),
                "roofline": {"bound": "tensor", "achieved": tf, "peak": peaks["bf16_sustained"], "unit": "TFLOP/s",
                             "frac": tf / peaks["bf16_sustained"]}}

    # ---- the headline at FIXED total work: 1024 chains over all ranks (128 per GPU at 8: less than one 148-SM wave)
    def strong():
        S = max(1, 1024 // world)
        eng = Engine(mlp(D_IN, HIDDEN, N_CLS), device=local_rank, seed=1234)
        eng.set_dataset(X, y, _lib.LOSS_SPARSE_CE)
        eng.set_prior([0.0], [1.0], _lib.PRIOR_SCALAR)
        eng.hmc_init(S, args.eps, 1.0, args.leapfrog, _lib.HMC_REFERENCE, chain_offset=rank * S)
        eng.hmc_run(2, burning=True, sampling=False)
        eng.hmc_run(1, burning=False, sampling=True)
        d = eng.hmc_run(1, burning=False, sampling=True)
        ms = maxr(d["device_ms"])
        eng.close()
        rate = S * world * args.leapfrog / (ms / 1e3)
        tf = rate * FLOPS_PER_GRADEVAL * args.rows / 1e12
        return {"workload": "C3 HMC, 1024 chains in TOTAL over %d GPU(s) (%d per GPU)" % (world, S), "value": rate,
                "unit": "grad-evals/s", "ms": ms, "scaling": "strong",
                "roofline": {"bound": "tensor", "achieved": tf, "peak": peaks["bf16_sustained"] * world, "unit": "TFLOP/s",
                             "frac": tf / (peaks["bf16_sustained"] * world)}}

    guarded("c1_hmc_moons", c1)
    guarded("c2_svgd_moons", c2)
    guarded("c4_svgd_mnist", c4)
    guarded("c5_predictive", c5)
    if world > 1:
        guarded("strong_scaling_1024", strong)
    return out


def main():
    args = parse_args()
    if args.impl == "reference":
        return run_reference(args)
    rank = int(os.environ.get("RANK", 0))
    local_rank = int(os.environ.get("LOCAL_RANK", 0))
    world = int(os.environ.get("WORLD_SIZE", 1))
    dist = None
    if world > 1:
        # stdout carries ONE JSON line: NCCL's own prints go to stderr.  NCCL honours NCCL_DEBUG_FILE only above the
        # VERSION level (at VERSION it prints "NCCL version ..." to stdout), and WARN prints the same version line
        os.environ.setdefault("NCCL_DEBUG_FILE", "/dev/stderr")
        if os.environ.get("NCCL_DEBUG", "").upper() == "VERSION":
            os.environ["NCCL_DEBUG"] = "WARN"
        import torch
        import torch.distributed as dist
        torch.cuda.set_device(local_rank)
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))

    from bayesian_inference_for_nn_b200 import _lib, keras_json
    from bayesian_inference_for_nn_b200.engine import Engine

    def barrier():
        if dist is not None:
            dist.barrier()

    def max_over_ranks(v):
        if dist is None:
            return v
        import torch
        t = torch.tensor([v], dtype=torch.float64, device="cuda")
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item())

    def sum_over_ranks(v):
        if dist is None:
            return v
        import torch
        t = torch.tensor([v], dtype=torch.float64, device="cuda")
        dist.all_reduce(t, op=dist.ReduceOp.SUM)
        return float(t.item())

    S, L = args.chains, args.leapfrog
    X, y = synth(args.rows)
    spec = keras_json.parse_model_json(keras_json.make_sequential_json(D_IN, [HIDDEN, N_CLS], ["relu", "softmax"]))
    eng = Engine(spec, device=local_rank, seed=1234)
    paths = {"auto": _lib.PATH_AUTO, "generic": _lib.PATH_GENERIC, "fused": _lib.PATH_FUSED_SMALL,
             "tensor": _lib.PATH_TENSOR}
    eng.set_option("path", paths[args.path])
    for kv in args.opt:
        k, v = kv.split("=")
        eng.set_option(k, float(v))
    eng.set_dataset(X, y, _lib.LOSS_SPARSE_CE)          # inputs resident in HBM before the timed region
    eng.set_prior([0.0], [1.0], _lib.PRIOR_SCALAR)
    eng.hmc_init(S, args.eps, 1.0, L, _lib.HMC_REFERENCE, chain_offset=rank * S)
    eng.hmc_run(2, burning=True, sampling=False)         # leave the all-zero start (relu'(0)=0 there)

    for _ in range(args.warmup):
        eng.hmc_run(1, burning=False, sampling=True)
    eng.set_option("profile", 1)
    sampler = ClockSampler(local_rank)
    barrier()
    if rank == 0:
        sampler.start()
    t0 = time.perf_counter()
    d = eng.hmc_run(args.steps, burning=False, sampling=True)   # EXACTLY K steps, device-timed inside
    wall = time.perf_counter() - t0
    barrier()
    clocks = sampler.stop() if rank == 0 else None
    dev_ms = max_over_ranks(d["device_ms"])
    wall_s = max_over_ranks(wall)
    launches = d["kernel_launches"]
    prof_ms, prof_flops, prof_n = eng.info("prof_ms"), eng.info("prof_flops"), eng.info("prof_launches")
    eng.set_option("profile", 0)
    path_used = int(eng.info("path_used"))
    total_evals = sum_over_ranks(S * L * args.steps)
    value = total_evals / (dev_ms / 1e3)
    accept_rate = d["accept_rate"]
    if args.dump_outputs and rank == 0:                   # before the e2e leg moves the chains on
        dump_outputs(eng, args.dump_outputs)

    # ---- e2e: same steps through the public C ABI with HOST buffers (H2D of the step's inputs from
    # pinned memory + D2H of the step's result inside the timed region)
    e2e = None
    if not args.no_e2e:
        try:
            import torch
            Xp = torch.from_numpy(X).pin_memory().numpy()
            yp = torch.from_numpy(y).pin_memory().numpy()
        except Exception:
            Xp, yp = X, y
        barrier()
        t0 = time.perf_counter()
        d2h = 0
        for _ in range(args.steps):
            eng.set_dataset(Xp, yp, _lib.LOSS_SPARSE_CE)
            eng.hmc_run(1, burning=False, sampling=True)
            last = eng.hmc_last()
            d2h = sum(v.nbytes for v in last.values())
        e2e_s = max_over_ranks(time.perf_counter() - t0)
        e2e = {"value": total_evals / e2e_s, "unit": "grad-evals/s", "h2d_bytes_per_step": int(Xp.nbytes + yp.nbytes),
               "d2h_bytes_per_step": int(d2h)}

    split = int(eng.info("tc_split")) if path_used == 3 else 0
    peaks = measured_peaks()
    eng.close()                                            # the sub-records below bring their own engines
    extra = None
    if not args.no_extras and named_default(args):
        extra = run_extras(args, rank, local_rank, world, dist, X, y, peaks)
    if rank != 0:
        if dist is not None:
            dist.destroy_process_group()
        return

    algo_flops_per_eval = FLOPS_PER_GRADEVAL * args.rows
    # roofline for the dominant kernel family (the fwd/bwd GEMMs): algorithmic flops they cover /
    # their summed CUDA-event time on the launching stream
    roof = None
    if prof_ms > 0:
        achieved = prof_flops / (prof_ms / 1e3) / 1e12
        # MMA passes per algorithmic product in bf16-rate equivalents: bf16x3 = 3 kind::f16 MMAs; int8 slices = 3 kind::i8
        # MMAs at twice the kind::f16 rate = 1.5 (forward only on slices: the dW1 GEMM still pays 3)
        passes = {0: 3.0, 1: 2.25, 2: 1.5}[split]
        roof = {"bound": "tensor", "achieved": achieved, "peak": peaks["bf16_sustained"], "unit": "TFLOP/s",
                "frac": achieved / peaks["bf16_sustained"], "traffic": ncu_traffic(split),
                "issued_mma_tflops_bf16_equivalent": passes * achieved,
                "issued_mma_frac": passes * achieved / peaks["bf16_sustained"],
                "peak_source": "%s bf16 dense sustained (cuBLAS; MEASURED_PEAKS.json holds no int8 figure: kind::i8 issues at "
                               "twice the kind::f16 rate, so against an int8 peak every fraction here halves)" % peaks["source"],
                "kernel": {1: "k_sgemm (fp32 SIMT)", 2: "fused small",
                           3: ("tc_g1_layer2_fused<.., I8> + tc_gemm_pair_dw1_i8 (tcgen05 kind::i8) + tc_gemm_bf16x3 (dW2)" if split
                               else "tc_gemm bf16x3 (tcgen05 kind::f16)")}.get(path_used, "?"),
                "launches": int(prof_n), "avg_launch_ms": prof_ms / max(1, prof_n),
                "kernel_share_of_step": prof_ms / d["device_ms"],
                "whole_step_algorithmic_tflops": value / max(1, world) * algo_flops_per_eval / 1e12,
                "note": ("fp32-grade products on two int8 fixed-point slices per operand (hi*hi + hi*lo + lo*hi, exact int32 "
                         "accumulation): 1.5 bf16-pass equivalents and 2 operand bytes per element instead of 3 and 4; ncu "
                         "(profiles/r2_*): the dW1 GEMM runs the tensor pipe 89 % active, the fused forward kernel is bound by "
                         "the instruction issue of its layer-2 epilogue (tensor pipe 34 %), the dW2 GEMM by HBM (84 %), see "
                         "DESIGN.md section 4") if split else
                        ("fp32-grade products cost 3 bf16 MMA passes (hi*hi + lo*hi + hi*lo): algorithmic frac <= 1/3 of the "
                         "bf16 peak, issued_mma_frac is the tensor-pipe view; ncu (profiles/): the dW1 GEMM runs the tensor "
                         "pipe 95 % active, the fused layer-1 GEMM + layer-2 kernel is bound by its epilogue, see DESIGN.md "
                         "section 4")}
    cpu = None
    if not args.no_cpu_baseline and world == 1:      # rank 0 at N = 1 only (the reference arm reports it at every N)
        # bounded sample (~10 s of CPU work): 1 chain, 3 timed iterations (+1 warm-up) on the full dataset
        v, dt, cores = cpu_reference_run(args, 3, 1, args.rows)
        cpu = {"value": v, "unit": "grad-evals/s", "cores": cores, "kind": "port",
               "sample": "1 chain x 3 iterations (L=%d, %d rows x 784, 784-256-10); numpy fp32 BLAS on all host cores, "
                         "reference loop shape (HMC.py:74-104: L+2 gradient + 2 potential evaluations per iteration); "
                         "%.1f s" % (L, args.rows, dt)}
    line = {
        "metric": "posterior_grad_evals_per_s", "value": value, "unit": "grad-evals/s", "n_gpus": world,
        "steps": args.steps, "warmup": args.warmup, "ms_per_step": dev_ms / args.steps, "higher_is_better": True,
        "scaling": "weak", "vs_baseline": None,
        "dtype": ("f32" if path_used != 3 else
                  "f32 (bf16x3 split tensor-core products, fp32 accumulate)" if split == 0 else
                  "f32 (tensor-core products on two int8 fixed-point slices per operand, kind::i8, exact int32 accumulate%s; "
                  "f32 everywhere else)" % ("" if split == 2 else "; dW1 GEMM on bf16x3")),
        "data": "synthetic",
        "config": workload_config(args, world, d["grad_evals"] / float(S * args.steps)),
        "wall_ms_per_step": 1e3 * wall_s / args.steps, "accept_rate": accept_rate, "path_used": path_used,
        "gpu_launches": int(launches), "clocks": clocks, "e2e": e2e, "roofline": roof, "cpu_baseline": cpu,
        "extra": extra,
    }
    print(json.dumps(line), flush=True)
    if dist is not None:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
