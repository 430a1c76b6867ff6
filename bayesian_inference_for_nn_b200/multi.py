"""Several GPUs of one box behind ONE optimizer object.

The reference runs a single chain / a Python loop over particles on one device (HMC.py:45-72, SVGD.py:219-228).  Here
``HyperParameters(devices=[0, 1, ...])`` (or ``n_devices=k``) makes ``compile`` create one ``Engine`` per device in this
process, each driven by its own host thread (every C call releases the GIL, so the devices run concurrently):

* HMC chains never interact: device i owns the global chains [lo_i, hi_i) (``sharding.shard_range``) and is initialised
  with ``chain_offset=lo_i``, so the Philox counters — and therefore every trajectory and every sample — are those of the
  one-device run; ``result()`` pools the per-device samples in global chain order.  With a tempering ladder of R rungs
  the unit of sharding is the replica group: device i owns groups [lo_i, hi_i), i.e. chains [R lo_i, R hi_i), and swaps
  stay inside a device.
* SVGD particles: each engine joins one NCCL communicator (``pyb_svgd_set_comm``) and the exchange step runs inside the
  library (svgd.cu); the engines must hold the same number of particles.
"""
from concurrent.futures import ThreadPoolExecutor

import numpy as np

from . import _lib
from .engine import Engine
from .sharding import shard_range


def devices_from(hp_get):
    """``devices`` (list of ordinals) or ``n_devices`` (first k devices) or ``device`` (one) -> list of ordinals"""
    devs = hp_get("devices", None)
    if devs is None:
        n = hp_get("n_devices", None)
        devs = list(range(int(n))) if n is not None else [int(hp_get("device", 0))]
    devs = [int(d) for d in devs]
    if len(devs) == 0 or len(set(devs)) != len(devs):
        raise ValueError("devices must be a non-empty list of distinct device ordinals")
    if len(devs) > 1:                       # (one device: pyb_create reports a bad ordinal / a missing GPU itself)
        have = _lib.device_count()
        if max(devs) >= have:
            raise ValueError("device %d requested, %d visible" % (max(devs), have))
    return devs


class EngineGroup:
    """One Engine per device; ``each(fn)`` runs ``fn(i, engine)`` on every engine concurrently and returns the results in
    device order (an exception in any thread is re-raised here)."""

    def __init__(self, spec, devices, seed=0):
        self.devices = list(devices)
        self.engines = [Engine(spec, device=d, seed=seed) for d in self.devices]
        self._pool = ThreadPoolExecutor(max_workers=len(self.engines)) if len(self.engines) > 1 else None

    def __len__(self):
        return len(self.engines)

    def each(self, fn):
        if self._pool is None:
            return [fn(0, self.engines[0])]
        futs = [self._pool.submit(fn, i, e) for i, e in enumerate(self.engines)]
        return [f.result() for f in futs]

    def close(self):
        for e in self.engines:
            e.close()
        if self._pool is not None:
            self._pool.shutdown(wait=True)
            self._pool = None

    # ---- HMC ------------------------------------------------------------------------------------------------------
    def hmc_init(self, n_chains, eps, m, L, semantics, q0=None, chain_offset=0, ladder=None):
        """n_chains posterior chains; with ``ladder`` (R inverse temperatures) each is a replica group of R engine
        chains, q0 rows (one per posterior chain, or one for all) are replicated over a group's rungs, and
        ``chain_offset`` (the global id of the first engine chain) must be a multiple of R"""
        R = 1 if ladder is None else len(ladder)
        self.R = R
        self.ranges = [shard_range(n_chains, i, len(self)) for i in range(len(self))]
        if any(hi == lo for lo, hi in self.ranges):
            raise ValueError("n_chains must be at least the number of devices")
        q0 = None if q0 is None else np.asarray(q0, np.float32)

        def init(i, e):
            lo, hi = self.ranges[i]
            q = None if q0 is None else (q0[lo:hi] if q0.shape[0] == n_chains else q0)
            if q is not None and R > 1:
                q = np.repeat(q.reshape(-1, q.shape[-1]), R, axis=0) if q.shape[0] == hi - lo else q
            e.hmc_init((hi - lo) * R, eps, m, L, semantics, q0=q, chain_offset=chain_offset + lo * R)
            if R > 1:
                e.hmc_set_temperatures(ladder)
        self.each(init)

    def hmc_run(self, n, burning, sampling):
        ds = self.each(lambda i, e: e.hmc_run(n, burning=burning, sampling=sampling))
        return merge_hmc_diag(ds)

    def hmc_samples(self):
        parts = self.each(lambda i, e: e.hmc_samples())
        return tuple(np.concatenate([p[k] for p in parts]) for k in range(3))

    def hmc_state(self):
        parts = self.each(lambda i, e: e.hmc_state())
        return np.concatenate([p[0] for p in parts]), np.concatenate([p[1] for p in parts])

    def hmc_adapt_begin(self, target):
        self.each(lambda i, e: e.hmc_adapt_begin(target))     # chains adapt on their own: no cross-device step

    def hmc_adapt_end(self):
        self.each(lambda i, e: e.hmc_adapt_end())

    def hmc_step_sizes(self):
        """[n_chains] float64 in global chain order"""
        return np.concatenate(self.each(lambda i, e: e.hmc_step_sizes()))

    def hmc_set_step_sizes(self, eps):
        """one step size per engine chain (n_chains R with a ladder), global chain order"""
        eps = np.asarray(eps, np.float64).reshape(-1)
        R = getattr(self, "R", 1)
        if eps.shape[0] != self.ranges[-1][1] * R:
            raise ValueError("expected %d step sizes, got %d" % (self.ranges[-1][1] * R, eps.shape[0]))
        self.each(lambda i, e: e.hmc_set_step_sizes(eps[self.ranges[i][0] * R:self.ranges[i][1] * R]))

    def hmc_tempering_stats(self):
        """``Engine.hmc_tempering_stats`` of the last ``hmc_run``, summed over the devices"""
        parts = self.each(lambda i, e: e.hmc_tempering_stats())
        return {k: sum(p[k] for p in parts) for k in parts[0]}

    def hmc_track_predictive(self, x, y=None):
        self.each(lambda i, e: e.hmc_track_predictive(x, y))

    def hmc_predictive(self, semantics=None, divisor=None):
        """the streamed predictive over every device's chains: the per-device sums are added on the host in device
        order (they are sums over chains) and finished on engine 0 -> (``hmc_predictive_finish`` dict, n_chains, T)"""
        parts = self.each(lambda i, e: e.hmc_predictive_sums())
        Ts = {p[2] for p in parts}
        if len(Ts) != 1:
            raise RuntimeError("the devices tracked different numbers of draws per chain: %s" % sorted(Ts))
        sums, s2 = parts[0][0].copy(), None if parts[0][1] is None else parts[0][1].copy()
        for p in parts[1:]:
            sums += p[0]
            if s2 is not None:
                s2 += p[1]
        n_chains = sum(e.S // e.R for e in self.engines)       # a ladder tracks its rung-0 chains
        T = Ts.pop()
        return self.engines[0].hmc_predictive_finish(sums, s2, n_chains, T, semantics, divisor), n_chains, T

    def hmc_track_params(self, n_planned, batch=0):
        self.each(lambda i, e: e.hmc_track_params(n_planned, batch))

    def hmc_param_summary(self, n_planned, batch=0):
        """the streamed per-parameter moments over every device's chains: the per-device sums are added on the host in
        device order and finished on engine 0 -> (``hmc_param_finish`` dict, n_chains, T)"""
        parts = self.each(lambda i, e: e.hmc_param_sums())
        Ts = {p[1] for p in parts}
        if len(Ts) != 1:
            raise RuntimeError("the devices tracked different numbers of draws per chain: %s" % sorted(Ts))
        sums = parts[0][0].copy()
        for p in parts[1:]:
            sums += p[0]
        n_chains = sum(e.S // e.R for e in self.engines)       # a ladder tracks its rung-0 chains
        T = Ts.pop()
        return self.engines[0].hmc_param_finish(sums, n_chains, T, n_planned, batch), n_chains, T

    # ---- SVGD -----------------------------------------------------------------------------------------------------
    def svgd_join(self):
        """one NCCL communicator over the group's engines (a no-op for one device)"""
        if len(self) > 1:
            uid = _lib.nccl_unique_id()
            self.each(lambda i, e: e.svgd_set_comm(i, len(self), uid))


def merge_hmc_diag(ds):
    """per-device ``pyb_hmc_run`` diagnostics -> one: counts summed, mean loss weighted by chain-iterations, device time
    the maximum (the devices ran side by side)"""
    if len(ds) == 1:
        return ds[0]
    out = dict(ds[0])
    for k in ("n_accepted", "n_total", "n_nan", "grad_evals", "kernel_launches"):
        out[k] = sum(d[k] for d in ds)
    tot = max(1, out["n_total"])
    out["mean_loss"] = sum(d["mean_loss"] * d["n_total"] for d in ds) / tot
    out["accept_rate"] = out["n_accepted"] / tot
    out["device_ms"] = max(d["device_ms"] for d in ds)
    return out
