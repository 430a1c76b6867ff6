"""GPU tests of the streamed per-parameter moments and diagnostics of the HMC chains (pyb_hmc_track_params,
pyb_hmc_param_sums, pyb_hmc_param_finish): every estimator against a float64 NumPy restatement over the full
trajectories on the fused-small, tensor and generic paths and under a tempering ladder, the pooled moments against the
kept samples, bit-identical sampling with and without tracking, the statistics on posteriors with known answers, the
error codes and lifecycle, the optimizer flow and sharding over two devices."""
import re

import numpy as np
import pytest

pytestmark = pytest.mark.gpu

from Pyesian.datasets import Dataset  # noqa: E402
from Pyesian.distributions import GaussianPrior  # noqa: E402
from Pyesian.optimizers import HMC  # noqa: E402
from Pyesian.optimizers.hyperparameters import HyperParameters  # noqa: E402
from bayesian_inference_for_nn_b200 import _lib, keras_json  # noqa: E402
from bayesian_inference_for_nn_b200.engine import Engine  # noqa: E402

ERR_INVALID, ERR_STATE, ERR_OOM = -1, -3, -5
PATHS = {"moons": _lib.PATH_FUSED_SMALL, "mnist_shaped": _lib.PATH_TENSOR, "deep_tanh": _lib.PATH_GENERIC}
LADDERS = {2: [1.0, 0.5], 3: [1.0, 0.6, 0.3], 4: [1.0, 0.7, 0.45, 0.2]}


# ---- the float64 restatement ----------------------------------------------------------------------------------------
def restate(x, n_planned, b=0):
    """x [S, T, P] float64 draws -> dict of mean, sd, rhat, ess, mcse [P] as the header defines them"""
    S, T, P = x.shape
    h = n_planned // 2
    b = b or int(np.floor(np.sqrt(n_planned)))
    n = S * T
    nan = np.full(P, np.nan)
    out = dict(mean=x.mean((0, 1)), sd=x.reshape(n, P).std(0))

    def classic_rhat(y):
        T_ = y.shape[1]
        W = y.var(1, ddof=1).mean(0)
        V = (T_ - 1) / T_ * W + y.mean(1).var(0, ddof=1)
        with np.errstate(divide="ignore", invalid="ignore"):
            r = np.sqrt(V / W)
        r[~(W > 0)] = np.nan
        return r

    out["rhat"] = classic_rhat(np.concatenate([x[:, :h], x[:, h:2 * h]], 0)) if T >= 2 * h and h >= 2 else nan
    a = T // b
    if T >= 2 and a >= 2:
        lam2 = x.var(1, ddof=1).mean(0)
        Y = x[:, :a * b].reshape(S, a, b, P).mean(2)
        V = ((Y - Y.mean(1, keepdims=True)) ** 2).sum((0, 1))
        sbm = b * V / (S * (a - 1))
        with np.errstate(divide="ignore", invalid="ignore"):
            ess = n * lam2 / sbm
        ess[(lam2 == 0) | (sbm == 0)] = np.nan
        out.update(ess=ess, mcse=np.sqrt(sbm / n))
    else:
        out.update(ess=nan, mcse=nan.copy())
    return out


def test_restatement_of_a_known_series():
    """the restatement itself on a series whose batch means and halves are known by hand"""
    x = np.array([[0, 1, 2, 3, 4, 5, 6, 7, 8], [1, 1, 1, 1, 1, 1, 1, 1, 5]], np.float64)[:, :, None]
    r = restate(x, 8, 3)            # h = 4, b = 3, a = 3
    assert r["mean"][0] == pytest.approx(x.mean())
    Y = np.array([[1, 4, 7], [1, 1, 7 / 3]])
    V = ((Y - Y.mean(1, keepdims=True)) ** 2).sum()
    sbm = 3 * V / (2 * 2)
    lam2 = (x[0].var(ddof=1) + x[1].var(ddof=1)) / 2
    assert r["ess"][0] == pytest.approx(18 * lam2 / sbm)
    assert r["mcse"][0] == pytest.approx(np.sqrt(sbm / 18))
    assert np.isnan(restate(x, 12, 3)["rhat"][0])      # T = 9 < 2h = 12
    assert np.isnan(restate(x, 8, 5)["ess"][0])        # a = 1


# ---- problems -------------------------------------------------------------------------------------------------------
def moons(n, seed=0, noise=0.2):
    rng = np.random.default_rng(seed)
    n0 = n // 2
    t0, t1 = rng.uniform(0, np.pi, n0), rng.uniform(0, np.pi, n - n0)
    x = np.concatenate([np.stack([np.cos(t0), np.sin(t0)], 1), np.stack([1 - np.cos(t1), 0.5 - np.sin(t1)], 1)])
    y = np.concatenate([np.zeros(n0, np.int64), np.ones(n - n0, np.int64)])
    return (x + rng.normal(0, noise, x.shape)).astype(np.float32), y.astype(np.int32)


def _problem(name):
    """-> (model json, X, y, chains, eps, m, L, path) on the fused-small, tensor and generic paths"""
    rng = np.random.default_rng(3)
    if name == "moons":
        X, y = moons(400)
        return keras_json.make_sequential_json(2, [50, 2], ["relu", "softmax"]), X, y, 64, 0.005, 0.5, 10, _lib.PATH_AUTO
    if name == "mnist_shaped":
        X = rng.random((640, 784), dtype=np.float32)
        y = rng.integers(0, 10, 640).astype(np.int32)
        return keras_json.make_sequential_json(784, [256, 10], ["relu", "softmax"]), X, y, 8, 2e-4, 1.0, 5, _lib.PATH_AUTO
    if name == "deep_tanh":
        X = rng.normal(0, 1, (300, 4)).astype(np.float32)
        y = rng.integers(0, 3, 300).astype(np.int32)
        return (keras_json.make_sequential_json(4, [16, 16, 3], ["tanh", "tanh", "softmax"]), X, y, 12, 0.01, 1.0, 5,
                _lib.PATH_GENERIC)
    raise KeyError(name)


def _engine(name, seed=7, R=None, S=None, chain_offset=0, sigma=1.0):
    js, X, y, S0, eps, m, L, path = _problem(name)
    eng = Engine(keras_json.parse_model_json(js), seed=seed)
    eng.set_option("path", path)
    if name == "mnist_shaped":
        eng.set_option("tc_i8", 0)
    eng.set_dataset(X, y, _lib.LOSS_SPARSE_CE)
    eng.set_prior([0.0], [sigma], _lib.PRIOR_SCALAR)
    eng.hmc_init(S or S0, eps, m, L, chain_offset=chain_offset)
    if R is not None:
        eng.hmc_set_temperatures(LADDERS[R])
    return eng


def _trajectories(eng, n):
    """n sampling iterations one call at a time -> the tracked draws [S_cold, n + 1, P] float64"""
    R = eng.R
    xs = [eng.hmc_state()[0][::R]]
    for _ in range(n):
        eng.hmc_run(1, burning=False, sampling=True)
        xs.append(eng.hmc_state()[0][::R])
    return np.stack(xs, 1).astype(np.float64)


def _summary(eng, n_planned, batch=0):
    sums, T = eng.hmc_param_sums()
    return eng.hmc_param_finish(sums, eng.S // eng.R, T, n_planned, batch), T


def _check(got, want, keys=("mean", "sd", "rhat", "ess", "mcse")):
    for k in keys:
        np.testing.assert_allclose(got[k], want[k], rtol=1e-8, atol=1e-14 if k == "mean" else 0, err_msg=k)


# ---- 1 + 2. against float64, and against the kept samples -----------------------------------------------------------
CASES = [("moons", None, 10, 0, 9),          # fused-small; n_planned even, b = 3 does not divide T = 10
         ("moons", 4, 9, 3, 8),              # fused-small under a ladder; n_planned odd, b divides T = 9
         ("mnist_shaped", None, 8, 2, 11),   # tensor; T = 12 > n_planned
         ("deep_tanh", None, 12, 0, 6),      # generic; T = 7 < 2h = 12: split R-hat NaN
         ("deep_tanh", 3, 9, 0, 8),          # generic under a ladder of R = 3 (cold rows only)
         ("moons", None, 16, 4, 4)]          # a = floor(5 / 4) = 1 < 2: ESS and MCSE NaN


@pytest.mark.parametrize("name,R,n_planned,batch,n", CASES)
def test_matches_the_float64_restatement(name, R, n_planned, batch, n):
    eng = _engine(name, R=R)
    eng.hmc_run(2, burning=True, sampling=False)
    eng.hmc_track_params(n_planned, batch)
    x = _trajectories(eng, n)
    assert eng.info("path_used") == PATHS[name]
    got, T = _summary(eng, n_planned, batch)
    assert T == n + 1 == x.shape[1]
    want = restate(x, n_planned, batch)
    _check(got, want)
    h, b = n_planned // 2, batch or int(np.floor(np.sqrt(n_planned)))
    assert np.isnan(got["rhat"]).all() == (T < 2 * h)
    assert np.isnan(got["ess"]).all() == (T // b < 2)
    # the pooled moments are those of the kept samples weighted by their frequencies
    s, f, c = eng.hmc_samples()
    R_ = R or 1
    cold = np.unique(c)
    assert len(cold) == x.shape[0] and (cold % R_ == 0).all()
    for ch in cold:
        assert f[c == ch].sum() == T
    w = f.astype(np.float64)
    mu = (w[:, None] * s).sum(0) / w.sum()
    var = (w[:, None] * (s - mu) ** 2).sum(0) / w.sum()
    np.testing.assert_allclose(got["mean"], mu, rtol=0, atol=1e-6)
    np.testing.assert_allclose(got["sd"] ** 2, var, rtol=0, atol=1e-6)


def test_reset_clears_the_sums():
    eng = _engine("deep_tanh")
    eng.hmc_track_params(6)
    eng.hmc_run(4, burning=False, sampling=True)
    assert eng.hmc_param_sums()[1] == 5
    eng.hmc_reset_samples()
    assert eng.lib.pyb_hmc_param_sums(eng.h, np.zeros((7, eng.P)).ctypes.data, None) == ERR_STATE   # no draw yet
    x = _trajectories(eng, 5)
    got, T = _summary(eng, 6)
    assert T == 6
    _check(got, restate(x, 6))


# ---- 3. tracking changes nothing ------------------------------------------------------------------------------------
@pytest.mark.parametrize("name,R", [("moons", None), ("moons", 2), ("deep_tanh", 3), ("mnist_shaped", None)])
def test_tracking_changes_nothing(name, R):
    xt = _problem(name)[1][:50]
    runs = []
    for params in (False, True):
        eng = _engine(name, R=R)
        eng.hmc_track_predictive(xt)
        eng.hmc_run(2, burning=True, sampling=False)
        if params:
            eng.hmc_track_params(8)
        acc = []
        for _ in range(6):
            eng.hmc_run(1, burning=False, sampling=True)
            acc.append(eng.hmc_last()["accept"])
        runs.append((eng.hmc_state()[0], np.stack(acc), eng.hmc_samples(), eng.hmc_predictive_sums()[0]))
    (q0, a0, s0, p0), (q1, a1, s1, p1) = runs
    np.testing.assert_array_equal(q0, q1)
    np.testing.assert_array_equal(a0, a1)
    for u, v in zip(s0, s1):
        np.testing.assert_array_equal(u, v)
    np.testing.assert_array_equal(p0, p1)


@pytest.mark.parametrize("name,R", [("moons", None), ("deep_tanh", 3), ("mnist_shaped", None)])
def test_one_call_equals_many(name, R):
    n = 7
    one, many = _engine(name, R=R), _engine(name, R=R)
    for e in (one, many):
        e.hmc_run(2, burning=True, sampling=False)
        e.hmc_track_params(n + 1)
    one.hmc_run(n, burning=False, sampling=True)
    for _ in range(n):
        many.hmc_run(1, burning=False, sampling=True)
    (s1, t1), (s2, t2) = one.hmc_param_sums(), many.hmc_param_sums()
    assert t1 == t2 == n + 1
    np.testing.assert_array_equal(s1, s2)


# ---- 4. statistics --------------------------------------------------------------------------------------------------
def _linear_problem():
    rng = np.random.default_rng(11)
    N = 20
    X = rng.normal(0, 1, (N, 2)).astype(np.float32)
    y = (X @ np.array([0.8, -0.5]) + 0.3 + rng.normal(0, 0.5, N)).astype(np.float32).reshape(N, 1)
    return X, y


def test_linear_gaussian_posterior():
    X, y = _linear_problem()
    N = X.shape[0]
    spec = keras_json.parse_model_json(keras_json.make_sequential_json(2, [1], ["linear"]))
    eng = Engine(spec, seed=3)
    eng.set_option("path", _lib.PATH_GENERIC)
    eng.set_option("hmc_keep_samples", 0)
    eng.set_dataset(X, y, _lib.LOSS_MSE)
    eng.set_prior([0.0], [1.0], _lib.PRIOR_SCALAR)
    eng.hmc_init(256, 0.05, 1.0, 10, semantics=_lib.HMC_CANONICAL)
    eng.hmc_run(200, burning=False, sampling=False)
    n = 600
    eng.hmc_track_params(n + 1)
    eng.hmc_run(n, burning=False, sampling=True)
    r, T = _summary(eng, n + 1)
    # closed form: theta = (w1, w2, b), E = n_train mean (A theta - y)^2 = sum (A theta - y)^2 (n_train = N)
    A = np.concatenate([X.astype(np.float64), np.ones((N, 1))], 1)
    cov = np.linalg.inv(np.eye(3) + 2.0 * A.T @ A)
    mu = cov @ (2.0 * A.T @ y[:, 0].astype(np.float64))
    print("mean", r["mean"], "closed", mu, "mcse", r["mcse"], "ess", r["ess"], "rhat", r["rhat"])
    assert (r["ess"] >= 1000).all(), r["ess"]
    assert (np.abs(r["mean"] - mu) < 4 * r["mcse"]).all()
    np.testing.assert_allclose(r["sd"], np.sqrt(np.diag(cov)), rtol=0.05)
    assert (r["rhat"] < 1.05).all(), r["rhat"]


def test_split_rhat_flags_chains_in_different_modes():
    rng = np.random.default_rng(2)
    X = rng.uniform(-2, 2, (50, 1)).astype(np.float32)
    y = (2.0 * np.tanh(1.5 * X) + rng.normal(0, 0.1, X.shape)).astype(np.float32)
    spec = keras_json.parse_model_json(keras_json.make_sequential_json(1, [1, 1], ["tanh", "linear"]))
    eng = Engine(spec, seed=5)
    eng.set_dataset(X, y, _lib.LOSS_MSE)
    eng.set_prior([0.0], [1.0], _lib.PRIOR_SCALAR)
    S = 64
    q0 = np.tile(np.array([1.5, 0.0, 2.0, 0.0], np.float32), (S, 1))     # (w1, b1, w2, b2)
    q0[1::2] *= -1.0                                                     # half the chains in the mirrored mode
    eng.hmc_init(S, 0.01, 1.0, 10, semantics=_lib.HMC_CANONICAL, q0=q0)
    eng.hmc_adapt_begin(0.7)
    eng.hmc_run(300, burning=False, sampling=False)
    eng.hmc_adapt_end()
    eng.hmc_track_params(201)
    eng.hmc_run(200, burning=False, sampling=True)
    r, _ = _summary(eng, 201)
    print("split R-hat", r["rhat"])
    assert r["rhat"][2] > 1.5, r["rhat"]


def test_negative_sigma_nothing_moves():
    """the reference's sigma < 0 prior: every proposal after burn-in is rejected"""
    eng = _engine("moons", S=1, sigma=-1.0)
    eng.hmc_run(3, burning=True, sampling=False)
    q, _ = eng.hmc_state()
    eng.hmc_track_params(20)
    d = eng.hmc_run(19, burning=False, sampling=True)
    assert d["n_accepted"] == 0
    r, T = _summary(eng, 20)
    assert T == 20
    np.testing.assert_allclose(r["mean"], q[0], rtol=1e-12)
    assert (r["sd"] == 0).all()
    assert np.isnan(r["rhat"]).all() and np.isnan(r["ess"]).all()
    assert (r["mcse"] == 0).all()


# ---- 5. errors and lifecycle ----------------------------------------------------------------------------------------
def test_errors_and_lifecycle():
    js, X, y, S, eps, m, L, path = _problem("deep_tanh")
    eng = Engine(keras_json.parse_model_json(js), seed=7)
    eng.set_option("path", path)
    eng.set_dataset(X, y, _lib.LOSS_SPARSE_CE)
    eng.set_prior([0.0], [1.0], _lib.PRIOR_SCALAR)
    lib, h, P = eng.lib, eng.h, eng.P
    sums = np.zeros((7, P))
    outs = [np.zeros(P) for _ in range(5)]
    optr = [o.ctypes.data for o in outs]
    assert lib.pyb_hmc_track_params(h, 10, 0) == ERR_STATE                  # before pyb_hmc_init
    eng.hmc_init(S, eps, m, L)
    assert lib.pyb_hmc_param_sums(h, sums.ctypes.data, None) == ERR_STATE  # not tracking
    for n_planned, batch in [(3, 0), (-1, 0), (10, -1), (10, 6), (9, 5), (4, 3)]:
        assert lib.pyb_hmc_track_params(h, n_planned, batch) == ERR_INVALID, (n_planned, batch)
    assert eng.info("hmc_param_bytes") == 0
    eng.hmc_track_params(10, 5)                                             # two batches of 5
    assert lib.pyb_hmc_param_sums(h, sums.ctypes.data, None) == ERR_STATE  # no draw yet
    nbytes = eng.info("hmc_param_bytes")
    assert nbytes >= 36 * S * P
    eng.hmc_run(2, burning=True, sampling=False)                           # burn-in tracks nothing
    assert lib.pyb_hmc_param_sums(h, sums.ctypes.data, None) == ERR_STATE
    eng.hmc_run(1, burning=False, sampling=True)
    assert lib.pyb_hmc_track_params(h, 10, 0) == ERR_STATE                  # a sampling iteration has run
    s, T = eng.hmc_param_sums()
    assert T == 2
    for args in [(None, S, T, 10, 0), (s.ctypes.data, 0, T, 10, 0), (s.ctypes.data, S, 0, 10, 0),
                 (s.ctypes.data, S, T, 3, 0), (s.ctypes.data, S, T, 10, -1), (s.ctypes.data, S, T, 10, 6)]:
        assert lib.pyb_hmc_param_finish(h, *args, *optr) == ERR_INVALID, args[1:]
    assert lib.pyb_hmc_param_finish(h, s.ctypes.data, S, T, 10, 0, None, None, None, None, None) == 0
    eng.hmc_reset_samples()
    assert lib.pyb_hmc_param_sums(h, sums.ctypes.data, None) == ERR_STATE  # cleared
    eng.hmc_set_temperatures(LADDERS[3])                                    # resized to the S / 3 cold chains
    assert eng.info("hmc_param_bytes") < nbytes
    eng.hmc_run(3, burning=False, sampling=True)
    eng.hmc_track_params(0)                                                 # stops
    assert eng.info("hmc_param_bytes") == 0
    assert lib.pyb_hmc_param_sums(h, sums.ctypes.data, None) == ERR_STATE
    eng.hmc_reset_samples()
    eng.hmc_set_temperatures(None)
    eng.hmc_track_params(5)
    eng.hmc_init(S, eps, m, L)                                              # pyb_hmc_init stops tracking
    assert eng.info("hmc_param_bytes") == 0
    assert lib.pyb_hmc_param_sums(h, sums.ctypes.data, None) == ERR_STATE


def _param_groups(nch, P):
    xb = (P + 255) // 256
    return max(1, min((nch + 31) // 32, (4096 + xb - 1) // xb))


def test_oversized_request_reports_oom():
    """the size check runs before any allocation: a request larger than the free memory names its size"""
    import torch
    spec = keras_json.parse_model_json(keras_json.make_sequential_json(1000, [1000, 1], ["tanh", "linear"]))
    eng = Engine(spec, seed=1)
    P = eng.P
    rng = np.random.default_rng(0)
    eng.set_dataset(rng.normal(size=(16, 1000)).astype(np.float32), rng.normal(size=(16, 1)).astype(np.float32),
                    _lib.LOSS_MSE)
    eng.set_prior([0.0], [1.0], _lib.PRIOR_SCALAR)
    free0, _ = torch.cuda.mem_get_info(0)
    # hmc_init holds ~16 S P bytes (q, p, g, q0); tracking needs ~36 S P: size S so that the request exceeds what is free
    S = int(1.1 * free0 / (52.0 * P)) + 1
    eng.hmc_init(S, 1e-3, 1.0, 1)
    free1, _ = torch.cuda.mem_get_info(0)
    need = S * P * 36.0 + (1 + _param_groups(S, P)) * 48.0 * P
    assert need > free1, (need, free1)
    rc = eng.lib.pyb_hmc_track_params(eng.h, 10, 0)
    msg = eng.lib.pyb_last_error().decode()
    assert rc == ERR_OOM, (rc, msg)
    assert re.search(r"%d chains x %d parameters needs %.2f GB" % (S, P, need / 1e9), msg), msg
    assert eng.info("hmc_param_bytes") == 0
    eng.close()


# ---- 6. the optimizer flow and sharding -----------------------------------------------------------------------------
def _optimizer(devices=None, ladder=(1.0, 0.5, 0.25), n_chains=16, **extra):
    x, y = moons(1000)
    ds = Dataset((x, y), "SparseCategoricalCrossentropy", "Classification", seed=0)
    if devices is not None:
        extra["devices"] = devices
    if ladder is not None:
        extra["inverse_temperatures"] = list(ladder)
    opt = HMC()
    opt.compile(HyperParameters(epsilon=0.005, m=0.5, L=20, n_chains=n_chains, seed=11, keep_samples=False, **extra),
                keras_json.make_sequential_json(2, [50, 2], ["relu", "softmax"]), ds, verbose=False,
                prior=GaussianPrior(0.0, 1.0))
    return opt


def test_optimizer_flow():
    opt = _optimizer()
    with pytest.raises(RuntimeError):
        opt.parameter_summary()
    opt.track_parameters()
    opt.train(30)
    r = opt.parameter_summary()
    assert r.n_draws == 31 and r.n_chains == 16
    P = opt._spec.n_params
    for k in ("mean", "sd", "rhat", "ess", "mcse"):
        assert getattr(r, k).shape == (P,) and getattr(r, k).dtype == np.float64
    assert np.isfinite(r.mean).all() and (r.sd > 0).all() and np.isfinite(r.rhat).all()
    # sampling by step(): n_iterations is required and the tracking starts at once
    opt = _optimizer(ladder=None, n_chains=4)
    opt.track_parameters(n_iterations=5, batch_size=2)
    for _ in range(5):
        opt.step(sampling=True)
    r = opt.parameter_summary()
    assert r.n_draws == 6 and r.n_chains == 4
    with pytest.raises(RuntimeError):
        opt.track_parameters(5)                      # sampling has started
    with pytest.raises(ValueError):
        _optimizer().track_parameters(batch_size=0)


def test_two_gpus_give_the_one_gpu_summary():
    if _lib.device_count() < 2:
        pytest.skip("needs two GPUs")
    runs = []
    for devices in ([0], [0, 1]):
        opt = _optimizer(devices=devices)
        opt.track_parameters()
        opt.train(12)
        runs.append(opt.parameter_summary())
    a, b = runs
    assert a.n_chains == b.n_chains == 16 and a.n_draws == b.n_draws == 13
    for k in ("mean", "sd", "rhat", "ess", "mcse"):
        np.testing.assert_allclose(getattr(b, k), getattr(a, k), rtol=1e-10, atol=0, err_msg=k)
