"""Thin Python wrapper over one libpyesian_b200 handle (one GPU).

Host arrays are NumPy; device-resident inputs arrive through DLPack (see ``tensors.py``).  Every
method is a single C-ABI call plus argument marshalling — no arithmetic happens here.
"""
from __future__ import annotations

import ctypes as C
from typing import Optional

import numpy as np

from . import _lib
from ._lib import check
from .keras_json import ModelSpec
from .tensors import ingest


def _ptr(a: Optional[np.ndarray]):
    return None if a is None else a.ctypes.data


def _f32(a, shape=None):
    a = np.ascontiguousarray(a, dtype=np.float32)
    if shape is not None and tuple(a.shape) != tuple(shape):
        raise ValueError("expected shape %s, got %s" % (tuple(shape), tuple(a.shape)))
    return a


class DeviceArray:
    """A float32 array owned by the caller and resident in the engine's HBM (pyb_buffer_create).  Anything that takes
    weight samples or inputs (``Engine.predict``) reads it in place.  Freed with the object."""

    def __init__(self, engine: "Engine", ptr: int, shape):
        self._engine, self.ptr, self.shape, self.dtype = engine, ptr, tuple(int(v) for v in shape), np.float32

    def free(self):
        eng = self._engine
        if self.ptr and eng is not None and getattr(eng, "h", None):
            eng.lib.pyb_buffer_destroy(eng.h, self.ptr)
        self.ptr = 0

    def __del__(self):
        try:
            self.free()
        except Exception:
            pass


class Engine:
    def __init__(self, spec: ModelSpec, device: int = 0, seed: int = 0):
        self.lib = _lib.load()
        self.spec = spec
        n = len(spec.dense)
        self._units = (C.c_int32 * n)(*[d.units for d in spec.dense])
        self._acts = (C.c_int32 * n)(*[d.activation for d in spec.dense])
        self._bias = (C.c_int32 * n)(*[1 if d.use_bias else 0 for d in spec.dense])
        desc = _lib.ModelDesc(n, spec.in_dim, self._units, self._acts, self._bias)
        h = C.c_void_p()
        check(self.lib.pyb_create(C.byref(desc), int(device), C.c_uint64(int(seed) & (2 ** 64 - 1)), C.byref(h)))
        self.h = h
        p = C.c_int64()
        check(self.lib.pyb_param_count(self.h, C.byref(p)))
        self.P = p.value
        assert self.P == spec.n_params, (self.P, spec.n_params)
        self.S = 0
        self.N = 0
        self._keep = []

    def close(self):
        if getattr(self, "h", None) is not None and self.h:
            self.lib.pyb_destroy(self.h)
            self.h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    # ---- options / info
    def set_option(self, key: str, value: float):
        check(self.lib.pyb_set_option(self.h, key.encode(), float(value)))

    def info(self, key: str) -> float:
        v = C.c_double()
        check(self.lib.pyb_get_info(self.h, key.encode(), C.byref(v)))
        return v.value

    # ---- inputs
    def set_dataset(self, X, y, loss_kind: int, n_train: int = 0):
        """X [N, in_dim] (NumPy / DLPack / tf.Tensor), y int labels [N] or float [N, out_dim]."""
        Xa, xmem, xptr = ingest(X, np.float32)
        ydt = np.int32 if loss_kind == _lib.LOSS_SPARSE_CE else np.float32
        ya, ymem, yptr = ingest(y, ydt)
        N = int(Xa.shape[0])
        if int(np.prod(Xa.shape[1:])) != self.spec.in_dim:
            raise ValueError("X has %d features per row, the model expects %d" % (int(np.prod(Xa.shape[1:])), self.spec.in_dim))
        if int(ya.shape[0]) != N:
            raise ValueError("X and y disagree on the number of rows")
        if xmem != ymem:   # mixed residency: bring y to where X is by staging through the host
            raise ValueError("X and y must both be host or both be device tensors")
        check(self.lib.pyb_set_dataset(self.h, xptr, N, yptr, int(loss_kind), int(xmem), int(n_train)))
        self.N = N
        self._loss_kind = int(loss_kind)

    def set_prior(self, mean, sigma, form: int):
        m = _f32(np.atleast_1d(mean).reshape(-1))
        s = _f32(np.atleast_1d(sigma).reshape(-1))
        check(self.lib.pyb_set_prior_gaussian(self.h, _ptr(m), _ptr(s), int(form)))

    # ---- HMC
    def hmc_init(self, S, eps, m, L, semantics=_lib.HMC_REFERENCE, q0=None, chain_offset=0):
        q0a = None if q0 is None else _f32(q0, (S, self.P))
        check(self.lib.pyb_hmc_init(self.h, int(S), int(chain_offset), float(eps), float(m), int(L), int(semantics),
                                    _ptr(q0a)))
        self.S = int(S)
        self.R = 1                      # pyb_hmc_init clears any tempering ladder
        self._track = None

    def hmc_inject(self, p=None, u=None):
        pa = None if p is None else _f32(p, (self.S, self.P))
        ua = None if u is None else _f32(u, (self.S,))
        check(self.lib.pyb_hmc_inject(self.h, _ptr(pa), _ptr(ua)))

    def hmc_run(self, n_iters, burning=False, sampling=True):
        d = _lib.HmcDiag()
        check(self.lib.pyb_hmc_run(self.h, int(n_iters), int(bool(burning)), int(bool(sampling)), C.byref(d)))
        return {k: getattr(d, k) for k, _ in _lib.HmcDiag._fields_}

    def hmc_eval(self, q, want_grad=True):
        q = _f32(q)
        S = q.shape[0]
        U = np.empty(S, np.float32)
        loss = np.empty(S, np.float32)
        g = np.empty((S, self.P), np.float32) if want_grad else None
        check(self.lib.pyb_hmc_eval(self.h, _ptr(q), S, _ptr(U), _ptr(loss), _ptr(g)))
        return U, loss, g

    def hmc_state(self):
        q = np.empty((self.S, self.P), np.float32)
        p = np.empty((self.S, self.P), np.float32)
        check(self.lib.pyb_hmc_get_state(self.h, _ptr(q), _ptr(p)))
        return q, p

    def hmc_last(self):
        S = self.S
        f = lambda: np.empty(S, np.float32)
        U0, K0, U1, K1, la, loss = f(), f(), f(), f(), f(), f()
        acc = np.empty(S, np.int32)
        check(self.lib.pyb_hmc_last(self.h, _ptr(U0), _ptr(K0), _ptr(U1), _ptr(K1), _ptr(la), _ptr(acc), _ptr(loss)))
        return dict(U0=U0, K0=K0, U1=U1, K1=K1, log_alpha=la, accept=acc.astype(bool), loss=loss)

    def hmc_reset_samples(self):
        check(self.lib.pyb_hmc_reset_samples(self.h))

    def hmc_samples(self):
        n = C.c_int64()
        check(self.lib.pyb_hmc_sample_count(self.h, C.byref(n)))
        n = n.value
        s = np.empty((n, self.P), np.float32)
        f = np.empty(n, np.int32)
        c = np.empty(n, np.int32)
        if n:
            check(self.lib.pyb_hmc_samples(self.h, _ptr(s), _ptr(f), _ptr(c)))
        return s, f, c

    # ---- per-chain step sizes (pyb_hmc_adapt_begin / _end, pyb_hmc_step_sizes, pyb_hmc_set_step_sizes)
    def hmc_adapt_begin(self, target=0.8):
        """From the next ``hmc_run`` on, adapt every chain's step size by dual averaging towards the acceptance
        probability ``target`` (0 < target < 1); no sampling iteration until ``hmc_adapt_end``."""
        check(self.lib.pyb_hmc_adapt_begin(self.h, float(target)))

    def hmc_adapt_end(self):
        """Freeze every chain's step size at its dual-averaging mean."""
        check(self.lib.pyb_hmc_adapt_end(self.h))

    def hmc_step_sizes(self):
        """-> [S] float64: each chain's step size (epsilon for all while none was set or adapted)."""
        out = np.empty(self.S, np.float64)
        check(self.lib.pyb_hmc_step_sizes(self.h, _ptr(out)))
        return out

    def hmc_set_step_sizes(self, eps):
        """eps [S]: one step size per chain, each finite and > 0."""
        e = np.ascontiguousarray(eps, dtype=np.float64).reshape(-1)
        if e.shape[0] != self.S:
            raise ValueError("expected %d step sizes, got %d" % (self.S, e.shape[0]))
        check(self.lib.pyb_hmc_set_step_sizes(self.h, _ptr(e)))

    # ---- parallel tempering (pyb_hmc_set_temperatures, pyb_hmc_tempering_stats, pyb_hmc_last_swaps)
    def hmc_set_temperatures(self, beta):
        """Run the S chains as S / R replica groups over the ladder ``beta`` (R inverse temperatures, beta[0] = 1,
        strictly decreasing, > 0): chain g R + r is rung r of group g; only rung 0 records draws.  None turns tempering
        off.  Call after ``hmc_init`` and before the first sampling iteration."""
        if beta is None:
            check(self.lib.pyb_hmc_set_temperatures(self.h, None, 0))
            self.R = 1
            return
        b = np.ascontiguousarray(beta, dtype=np.float64).reshape(-1)
        check(self.lib.pyb_hmc_set_temperatures(self.h, _ptr(b), int(b.shape[0])))
        self.R = int(b.shape[0])

    def hmc_tempering_stats(self):
        """counts of the last ``hmc_run`` over this engine's groups: per rung HMC proposals accepted / made
        ([R] int64), per pair (r, r + 1) swaps attempted / accepted ([R - 1] int64)"""
        R = self.R
        out = dict(rung_accepted=np.zeros(R, np.int64), rung_total=np.zeros(R, np.int64),
                   swap_attempted=np.zeros(R - 1, np.int64), swap_accepted=np.zeros(R - 1, np.int64))
        check(self.lib.pyb_hmc_tempering_stats(self.h, _ptr(out["rung_accepted"]), _ptr(out["rung_total"]),
                                               _ptr(out["swap_attempted"]), _ptr(out["swap_accepted"])))
        return out

    def hmc_last_swaps(self):
        """-> (log_r [S] float32, swapped [S] bool): the swap each chain proposed with its upper neighbour in the
        last iteration (NaN / False where none)"""
        lr = np.empty(self.S, np.float32)
        sw = np.empty(self.S, np.int32)
        check(self.lib.pyb_hmc_last_swaps(self.h, _ptr(lr), _ptr(sw)))
        return lr, sw.astype(bool)

    # ---- streamed HMC predictive (pyb_hmc_track_predictive / _sums / _finish)
    def hmc_track_predictive(self, x, y=None):
        """Accumulate the posterior predictive on inputs x [Nt, in_dim...] (NumPy / DLPack / tf.Tensor, copied once) over
        every draw the sampler records from the next sampling iteration on; y [Nt] integer labels enable
        ``hmc_predictive_finish(..., semantics=...)``.  x = None stops tracking."""
        if x is None:
            check(self.lib.pyb_hmc_track_predictive(self.h, None, 0, None))
            self._track = None
            return
        if isinstance(x, (np.ndarray, list, tuple)):
            x = _f32(x)
            x = x.reshape(x.shape[0], -1)
        xa, _, xptr = ingest(x, np.float32)
        if int(np.prod(xa.shape[1:])) != self.spec.in_dim:
            raise ValueError("x has %d features per row, the model expects %d" % (int(np.prod(xa.shape[1:])), self.spec.in_dim))
        Nt = int(xa.shape[0])
        ya = None
        if y is not None:
            ya = np.ascontiguousarray(np.asarray(y).reshape(-1), dtype=np.int32)
            if ya.shape[0] != Nt:
                raise ValueError("x and y disagree on the number of rows")
        check(self.lib.pyb_hmc_track_predictive(self.h, xptr, Nt, _ptr(ya)))
        self._track = (Nt, ya is not None)

    def hmc_predictive_sums(self):
        """-> (sums [4, Nt, C] float64 = A, Q, M, W; S2 [Nt, C, C] or None; draws per chain T)"""
        Nt, labels = self._tracked()
        Cc = self.spec.out_dim
        sums = np.empty((4, Nt, Cc), np.float64)
        s2 = np.empty((Nt, Cc, Cc), np.float64) if labels and Cc > 1 else None
        T = C.c_int64()
        check(self.lib.pyb_hmc_predictive_sums(self.h, _ptr(sums), _ptr(s2), C.byref(T)))
        return sums, s2, T.value

    def hmc_predictive_finish(self, sums, s2, n_chains, n_draws, semantics=None, divisor=None):
        """mean / variance / R-hat [Nt, C] from (summed) ``hmc_predictive_sums``; with ``semantics`` ("reference" |
        "canonical") also the uncertainty matrices (total, aleatoric, epistemic) [Nt, Ce, Ce] as ``predict_uncertainty``
        (``divisor`` defaults to the number of rows)."""
        Nt, _ = self._tracked()
        Cc = self.spec.out_dim
        Ce = 2 if Cc == 1 else Cc
        sums = np.ascontiguousarray(sums, dtype=np.float64)
        if sums.shape != (4, Nt, Cc):
            raise ValueError("sums must be [4, %d, %d]" % (Nt, Cc))
        s2 = None if s2 is None else np.ascontiguousarray(s2, dtype=np.float64)
        mean, var, rhat = (np.empty((Nt, Cc), np.float32) for _ in range(3))
        out = dict(mean=mean, variance=var, rhat=rhat)
        uq = (None, None, None)
        sem = 0
        if semantics is not None:
            sem = {"reference": _lib.UQ_REFERENCE, "canonical": _lib.UQ_CANONICAL}[semantics]
            uq = tuple(np.empty((Nt, Ce, Ce), np.float32) for _ in range(3))
            out.update(total=uq[0], aleatoric=uq[1], epistemic=uq[2])
        check(self.lib.pyb_hmc_predictive_finish(self.h, _ptr(sums), _ptr(s2), int(n_chains), int(n_draws), int(sem),
                                                 float(Nt if divisor is None else divisor), _ptr(mean), _ptr(var),
                                                 _ptr(rhat), _ptr(uq[0]), _ptr(uq[1]), _ptr(uq[2])))
        return out

    def _tracked(self):
        t = getattr(self, "_track", None)
        if t is None:
            raise RuntimeError("no predictive is tracked: call hmc_track_predictive first")
        return t

    # ---- streamed per-parameter moments (pyb_hmc_track_params / pyb_hmc_param_sums / pyb_hmc_param_finish)
    def hmc_track_params(self, n_planned, batch=0):
        """Accumulate the mean, sd, split-R-hat, ESS and MCSE of every parameter over every draw the sampler records
        from the next sampling iteration on, planned for ``n_planned`` draws per chain (it fixes the split halves) with
        batch size ``batch`` (0: floor(sqrt(n_planned))).  n_planned = 0 stops tracking."""
        check(self.lib.pyb_hmc_track_params(self.h, int(n_planned), int(batch)))

    def hmc_param_sums(self):
        """-> (sums [7, P] float64 = A, M, W, Ah, Mh, Wh, V, draws per chain T)"""
        sums = np.empty((7, self.P), np.float64)
        T = C.c_int64()
        check(self.lib.pyb_hmc_param_sums(self.h, _ptr(sums), C.byref(T)))
        return sums, T.value

    def hmc_param_finish(self, sums, n_chains, n_draws, n_planned, batch=0):
        """-> dict of mean, sd, rhat (split), ess, mcse, each [P] float64, from (summed) ``hmc_param_sums``"""
        sums = np.ascontiguousarray(sums, dtype=np.float64)
        if sums.shape != (7, self.P):
            raise ValueError("sums must be [7, %d]" % self.P)
        out = {k: np.empty(self.P, np.float64) for k in ("mean", "sd", "rhat", "ess", "mcse")}
        check(self.lib.pyb_hmc_param_finish(self.h, _ptr(sums), int(n_chains), int(n_draws), int(n_planned), int(batch),
                                            _ptr(out["mean"]), _ptr(out["sd"]), _ptr(out["rhat"]), _ptr(out["ess"]),
                                            _ptr(out["mcse"])))
        return out

    # ---- SVGD
    def svgd_init(self, S, lr, semantics=_lib.SVGD_REFERENCE_LIVE, particles0=None, offset=0):
        p0 = None if particles0 is None else np.ascontiguousarray(particles0, dtype=np.float64)
        if p0 is not None and p0.shape != (S, self.P):
            raise ValueError("particles0 must be [S, P]")
        check(self.lib.pyb_svgd_init(self.h, int(S), int(offset), float(lr), int(semantics), _ptr(p0)))
        self.S = int(S)

    def svgd_set_comm(self, rank: int, world: int, unique_id: bytes = None):
        """Shard particles over `world` ranks (one process per GPU); all ranks pass the same 128-byte id
        obtained once from `_lib.nccl_unique_id()`."""
        _lib.preload_nccl()
        buf = C.create_string_buffer(unique_id, 128) if unique_id is not None else None
        check(self.lib.pyb_svgd_set_comm(self.h, int(rank), int(world), buf))

    def set_comm(self, rank: int, world: int, unique_id: bytes = None, predict_sharded: bool = True):
        """Join `world` ranks (one process per GPU).  With ``predict_sharded`` every later ``predict`` /
        ``predict_uncertainty`` call treats W as this rank's share of the weight samples and returns the moments over
        all ranks' samples (one all-reduce of the [Nt, C] sums); all ranks must make the call."""
        _lib.preload_nccl()
        buf = C.create_string_buffer(unique_id, 128) if unique_id is not None else None
        check(self.lib.pyb_set_comm(self.h, int(rank), int(world), buf))
        self.set_option("predict_sharded", 1.0 if (predict_sharded and world > 1) else 0.0)

    def svgd_step(self, batch_idx=None):
        loss = C.c_double()
        if batch_idx is None:
            check(self.lib.pyb_svgd_step(self.h, None, 0, C.byref(loss)))
        else:
            idx = np.ascontiguousarray(batch_idx, dtype=np.int32)
            check(self.lib.pyb_svgd_step(self.h, _ptr(idx), int(idx.shape[0]), C.byref(loss)))
        return loss.value

    def svgd_set_validation(self, X, y):
        """held-out set for ``svgd_validation_loss`` (uploaded once; labels as in ``set_dataset``)"""
        X = _f32(X)
        X = X.reshape(X.shape[0], -1)
        if getattr(self, "_loss_kind", None) is None:
            raise RuntimeError("set_dataset must be called first (it fixes the loss kind)")
        if self._loss_kind == _lib.LOSS_SPARSE_CE:
            y = np.ascontiguousarray(np.asarray(y).reshape(-1), dtype=np.int32)
        else:
            y = np.ascontiguousarray(y, dtype=np.float32).reshape(X.shape[0], -1)
        if y.shape[0] != X.shape[0] or X.shape[1] != self.spec.in_dim:
            raise ValueError("validation set has the wrong shape")
        check(self.lib.pyb_svgd_set_validation(self.h, _ptr(X), _ptr(y), int(X.shape[0])))

    def svgd_validation_loss(self, per_particle=False):
        mean = C.c_double()
        pp = np.empty(self.S, np.float32) if per_particle else None
        check(self.lib.pyb_svgd_validation_loss(self.h, C.byref(mean), _ptr(pp)))
        return (mean.value, pp) if per_particle else mean.value

    def svgd_phi(self, X, G, semantics):
        X = np.ascontiguousarray(X, dtype=np.float64)
        G = _f32(G, X.shape)
        phi = np.empty(X.shape, np.float32)
        h = C.c_double()
        check(self.lib.pyb_svgd_phi(self.h, _ptr(X), _ptr(G), int(X.shape[0]), int(semantics), _ptr(phi), C.byref(h)))
        return phi, h.value

    def svgd_particles(self):
        out = np.empty((self.S, self.P), np.float64)
        check(self.lib.pyb_svgd_get_particles(self.h, _ptr(out)))
        return out

    # ---- S-batched SGLD / SWAG chains
    def sg_init(self, S, kind, k_dev=0, frequency=1, theta0=None, chain_offset=0):
        t0, rows = None, 0
        if theta0 is not None:
            t0 = _f32(np.atleast_2d(theta0))
            rows = int(t0.shape[0])
            if t0.shape[1] != self.P or rows not in (1, int(S)):
                raise ValueError("theta0 must be [1, P] or [S, P]")
        check(self.lib.pyb_sg_init(self.h, int(S), int(chain_offset), int(kind), int(k_dev), int(frequency), _ptr(t0), rows))
        self.S, self._sg_k = int(S), (int(k_dev) if kind == _lib.SG_SWAG else 0)

    def sg_step(self, lr, batch_idx=None, noise=None):
        """-> (per-chain minibatch losses [S], their mean)."""
        loss = np.empty(self.S, np.float32)
        mean = C.c_double()
        z = None if noise is None else _f32(noise, (self.S, self.P))
        idx = None if batch_idx is None else np.ascontiguousarray(batch_idx, dtype=np.int32)
        check(self.lib.pyb_sg_step(self.h, _ptr(idx), 0 if idx is None else int(idx.shape[0]), float(lr), _ptr(z),
                                   _ptr(loss), C.byref(mean)))
        return loss, mean.value

    def sg_state(self):
        S, P, k = self.S, self.P, self._sg_k
        theta, mean, sq = (np.empty((S, P), np.float32) for _ in range(3))
        dev = np.zeros((S, k, P), np.float32) if k else None
        cols, n = C.c_int32(), C.c_int64()
        check(self.lib.pyb_sg_get(self.h, _ptr(theta), _ptr(mean), _ptr(sq), _ptr(dev), C.byref(cols), C.byref(n)))
        return dict(theta=theta, mean=mean, sq_mean=sq, dev=None if dev is None else dev[:, :cols.value], n=n.value)

    # ---- caller-owned device arrays
    def device_array(self, a) -> DeviceArray:
        """Upload a float32 array once; the result can be passed wherever weight samples / inputs are taken."""
        a = np.ascontiguousarray(a, dtype=np.float32)
        out = C.c_void_p()
        check(self.lib.pyb_buffer_create(self.h, a.ctypes.data, int(a.nbytes), C.byref(out)))
        return DeviceArray(self, out.value, a.shape)

    def gather_rows(self, src: DeviceArray, idx) -> DeviceArray:
        """rows src[idx] as a new device array (the distinct weight vectors of a posterior draw)."""
        idx = np.ascontiguousarray(idx, dtype=np.int64)
        if idx.size == 0 or idx.min() < 0 or idx.max() >= src.shape[0]:
            raise IndexError("row index out of range")
        row_len = int(np.prod(src.shape[1:]))
        out = C.c_void_p()
        check(self.lib.pyb_buffer_create(self.h, None, int(idx.size) * row_len * 4, C.byref(out)))
        dst = DeviceArray(self, out.value, (int(idx.size),) + tuple(src.shape[1:]))
        check(self.lib.pyb_gather_rows(self.h, src.ptr, idx.ctypes.data, int(idx.size), row_len, dst.ptr))
        return dst

    # ---- predictive
    def _predict_args(self, W, x):
        if isinstance(W, (np.ndarray, list, tuple)):
            W = _f32(W)
        Wa, _, wptr = ingest(W, np.float32)
        if len(Wa.shape) != 2 or int(Wa.shape[1]) != self.P:
            raise ValueError("W must be [n, P]")
        if isinstance(x, (np.ndarray, list, tuple)):
            x = _f32(x)
            x = x.reshape(x.shape[0], -1)
        xa, _, xptr = ingest(x, np.float32)
        if int(np.prod(xa.shape[1:])) != self.spec.in_dim:
            raise ValueError("x has %d features per row, the model expects %d" % (int(np.prod(xa.shape[1:])), self.spec.in_dim))
        return (Wa, W, wptr), (xa, x, xptr)

    def predict_uncertainty(self, W, x, y, weights=None, semantics="reference", divisor=None):
        """Metrics.classification_uncertainty on the device (pyb_predict_uncertainty): -> (total, aleatoric, epistemic,
        mean), the first three [Nt, Ce, Ce].  ``semantics``: "reference" (what the reference's code computes: running
        sums over the rows, broadcast epistemic term) or "canonical" (per-row matrices, (p - onehot)(p - onehot)^T).
        ``divisor`` defaults to the number of rows."""
        sem = {"reference": _lib.UQ_REFERENCE, "canonical": _lib.UQ_CANONICAL}[semantics]
        (Wa, _Wk, wptr), (xa, _xk, xptr) = self._predict_args(W, x)
        n, Nt, Cc = int(Wa.shape[0]), int(xa.shape[0]), self.spec.out_dim
        Ce = 2 if Cc == 1 else Cc
        ya = np.ascontiguousarray(np.asarray(y).reshape(-1), dtype=np.int32)
        if ya.shape[0] != Nt:
            raise ValueError("x and y disagree on the number of rows")
        w = None if weights is None else _f32(weights, (n,))
        tot, al, ep = (np.empty((Nt, Ce, Ce), np.float32) for _ in range(3))
        mean = np.empty((Nt, Cc), np.float32)
        check(self.lib.pyb_predict_uncertainty(self.h, wptr, n, _ptr(w), xptr, Nt, _ptr(ya), int(sem),
                                               float(Nt if divisor is None else divisor), _ptr(tot), _ptr(al), _ptr(ep),
                                               _ptr(mean)))
        return tot, al, ep, mean

    def predict(self, W, x, weights=None, want_all=False):
        """W [n, P] weight samples, x [Nt, in_dim...] inputs: NumPy arrays, or device tensors (DLPack / tf.Tensor), which
        the library reads in place instead of uploading."""
        if isinstance(W, (np.ndarray, list, tuple)):
            W = _f32(W)
        Wa, _, wptr = ingest(W, np.float32)
        if len(Wa.shape) != 2 or int(Wa.shape[1]) != self.P:
            raise ValueError("W must be [n, P]")
        if isinstance(x, (np.ndarray, list, tuple)):
            x = _f32(x)
            x = x.reshape(x.shape[0], -1)
        xa, _, xptr = ingest(x, np.float32)
        if int(np.prod(xa.shape[1:])) != self.spec.in_dim:
            raise ValueError("x has %d features per row, the model expects %d" % (int(np.prod(xa.shape[1:])), self.spec.in_dim))
        n, Nt, Cc = int(Wa.shape[0]), int(xa.shape[0]), self.spec.out_dim
        w = None if weights is None else _f32(weights, (n,))
        mean = np.empty((Nt, Cc), np.float32)
        var = np.empty((Nt, Cc), np.float32)
        allo = np.empty((n, Nt, Cc), np.float32) if want_all else None
        check(self.lib.pyb_predict(self.h, wptr, n, _ptr(w), xptr, Nt, _ptr(mean), _ptr(var), _ptr(allo)))
        return mean, var, allo
