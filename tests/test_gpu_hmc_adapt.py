"""GPU tests of per-chain HMC step sizes and their dual-averaging adaptation (pyb_hmc_adapt_begin / _end,
pyb_hmc_step_sizes, pyb_hmc_set_step_sizes; Hoffman & Gelman 2014, Algorithm 5): the device's step-size trajectories
against a float64 NumPy restatement driven by the device's own log acceptance ratios, per-chain step sizes against
scalar runs bit for bit on the fused-small, tensor and generic paths, the acceptance rate the adaptation reaches, and
the lifecycle rules."""
import numpy as np
import pytest

pytestmark = pytest.mark.gpu

from Pyesian.datasets import Dataset  # noqa: E402
from Pyesian.distributions import GaussianPrior  # noqa: E402
from Pyesian.optimizers import HMC  # noqa: E402
from Pyesian.optimizers.hyperparameters import HyperParameters  # noqa: E402
from bayesian_inference_for_nn_b200 import _lib, keras_json  # noqa: E402
from bayesian_inference_for_nn_b200.engine import Engine  # noqa: E402

ERR_INVALID, ERR_STATE = -1, -3
PATHS = {"moons": _lib.PATH_FUSED_SMALL, "mnist_shaped": _lib.PATH_TENSOR, "deep_tanh": _lib.PATH_GENERIC}


def moons(n, seed=0, noise=0.2):
    rng = np.random.default_rng(seed)
    n0 = n // 2
    t0, t1 = rng.uniform(0, np.pi, n0), rng.uniform(0, np.pi, n - n0)
    x = np.concatenate([np.stack([np.cos(t0), np.sin(t0)], 1), np.stack([1 - np.cos(t1), 0.5 - np.sin(t1)], 1)])
    y = np.concatenate([np.zeros(n0, np.int64), np.ones(n - n0, np.int64)])
    return (x + rng.normal(0, noise, x.shape)).astype(np.float32), y.astype(np.int32)


def _problem(name):
    """-> (model json, X, y, chains, eps, m, L, path): the shapes of test_gpu_hmc_predictive.py"""
    rng = np.random.default_rng(3)
    if name == "moons":          # fused-small HMC
        X, y = moons(400)
        return keras_json.make_sequential_json(2, [50, 2], ["relu", "softmax"]), X, y, 64, 0.005, 0.5, 10, _lib.PATH_AUTO
    if name == "mnist_shaped":   # tensor path
        X = rng.random((640, 784), dtype=np.float32)
        y = rng.integers(0, 10, 640).astype(np.int32)
        return keras_json.make_sequential_json(784, [256, 10], ["relu", "softmax"]), X, y, 5, 2e-4, 1.0, 5, _lib.PATH_AUTO
    if name == "deep_tanh":      # generic path
        X = rng.normal(0, 1, (300, 4)).astype(np.float32)
        y = rng.integers(0, 3, 300).astype(np.int32)
        return (keras_json.make_sequential_json(4, [16, 16, 3], ["tanh", "tanh", "softmax"]), X, y, 12, 0.01, 1.0, 5,
                _lib.PATH_GENERIC)
    raise KeyError(name)


def _engine(name, seed=7, S=None, eps=None, sigma=1.0, tc_i8=None):
    js, X, y, S0, eps0, m, L, path = _problem(name)
    eng = Engine(keras_json.parse_model_json(js), seed=seed)
    eng.set_option("path", path)
    if tc_i8 is not None:
        eng.set_option("tc_i8", tc_i8)
    eng.set_dataset(X, y, _lib.LOSS_SPARSE_CE)
    eng.set_prior([0.0], [sigma], _lib.PRIOR_SCALAR)
    eng.hmc_init(S or S0, eps0 if eps is None else eps, m, L)
    return eng


def _dual_averaging(step0, log_alphas, target):
    """float64 restatement of the update: step0 [S], log_alphas [T, S] float32 -> (step after every iteration [T, S],
    the frozen exp(log_eps_bar) [S])"""
    mu = np.log(10.0 * np.asarray(step0, np.float64))
    h_bar = np.zeros_like(mu)
    log_eps_bar = np.zeros_like(mu)
    traj = []
    for t, la in enumerate(log_alphas, 1):
        a = np.exp(np.asarray(la, np.float64))
        a = np.where(np.isnan(a), 0.0, np.minimum(1.0, a))
        eta = 1.0 / (t + 10.0)
        h_bar = (1.0 - eta) * h_bar + eta * (target - a)
        log_eps = mu - np.sqrt(t) / 0.05 * h_bar
        w = float(t) ** -0.75
        log_eps_bar = w * log_eps + (1.0 - w) * log_eps_bar
        traj.append(np.exp(log_eps))
    return np.array(traj), np.exp(log_eps_bar)


def _accept_prob(la):
    a = np.exp(np.asarray(la, np.float64))
    return np.where(np.isnan(a), 0.0, np.minimum(1.0, a))


@pytest.mark.parametrize("name", ["moons", "mnist_shaped", "deep_tanh", "moons_nan_prior"])
def test_adaptation_follows_the_float64_restatement(name):
    nan_prior = name == "moons_nan_prior"
    eng = _engine("moons" if nan_prior else name, sigma=-1.0 if nan_prior else 1.0)   # GaussianPrior(0, -1): NaN
    if not nan_prior:
        eng.hmc_run(1, burning=True, sampling=False)
        assert eng.info("path_used") == PATHS[name]
    start = eng.hmc_step_sizes()
    eng.hmc_adapt_begin(0.7)
    las, steps = [], []
    for it in range(30):
        d = eng.hmc_run(1, burning=it < 3, sampling=False)     # the update ignores the burning flag
        last = eng.hmc_last()
        las.append(last["log_alpha"])
        steps.append(eng.hmc_step_sizes())
        if nan_prior:
            assert d["n_nan"] == eng.S and np.isnan(last["log_alpha"]).all()
            if it >= 3:
                assert not last["accept"].any()
    eng.hmc_adapt_end()
    want, frozen = _dual_averaging(start, las, 0.7)
    np.testing.assert_allclose(np.array(steps), want, rtol=1e-12, atol=0)
    np.testing.assert_allclose(eng.hmc_step_sizes(), frozen, rtol=1e-12, atol=0)
    assert np.isfinite(eng.hmc_step_sizes()).all() and (eng.hmc_step_sizes() >= 0).all()
    if nan_prior:       # every proposal after burn-in is rejected, at the adapted step sizes too
        d = eng.hmc_run(3, burning=False, sampling=True)
        assert d["n_accepted"] == 0 and d["n_nan"] == 3 * eng.S
    else:
        assert not np.array_equal(eng.hmc_step_sizes(), start)


def _iterations(eng, n_burn=2, n_samp=3):
    """per-iteration (hmc_last, state) of n_burn burn-in and n_samp sampling iterations, then the samples"""
    out = []
    for i in range(n_burn + n_samp):
        if i == n_burn:
            eng.hmc_reset_samples()
        eng.hmc_run(1, burning=i < n_burn, sampling=i >= n_burn)
        out.append((eng.hmc_last(), eng.hmc_state()))
    return out, eng.hmc_samples()


@pytest.mark.parametrize("name", ["moons", "mnist_shaped", "deep_tanh"])
def test_equal_step_sizes_equal_the_scalar_path(name):
    a = _engine(name)
    b = _engine(name)
    b.hmc_set_step_sizes(np.full(b.S, _problem(name)[4]))
    ra, sa = _iterations(a)
    rb, sb = _iterations(b)
    assert a.info("path_used") == b.info("path_used") == PATHS[name]
    for (la, qa), (lb, qb) in zip(ra, rb):
        for k in ("U0", "K0", "U1", "K1", "log_alpha", "accept", "loss"):
            np.testing.assert_array_equal(la[k], lb[k], err_msg=k)
        for u, v in zip(qa, qb):
            np.testing.assert_array_equal(u, v)
    for u, v in zip(sa, sb):
        np.testing.assert_array_equal(u, v)


@pytest.mark.parametrize("name", ["moons", "mnist_shaped", "deep_tanh"])
def test_each_chain_moves_with_its_own_step_size(name):
    eps0 = _problem(name)[4]
    values = np.array([eps0 * 0.5, eps0, eps0 * 1.7])
    S = 150 if name == "moons" else None          # moons: one CTA per chain here, a cluster per chain elsewhere
    tc_i8 = 0 if name == "mnist_shaped" else None   # the int8 guard looks at all chains together
    mixed = _engine(name, S=S, tc_i8=tc_i8)
    mixed.hmc_set_step_sizes(values[np.arange(mixed.S) % 3])
    rm, (sm, fm, cm) = _iterations(mixed)
    assert mixed.info("path_used") == PATHS[name]
    for k, v in enumerate(values):
        ref = _engine(name, S=S, eps=v, tc_i8=tc_i8)
        rr, (sr, fr, cr) = _iterations(ref)
        sel = np.arange(mixed.S) % 3 == k
        for (lm, qm), (lr, qr) in zip(rm, rr):
            for key in ("U0", "K0", "U1", "K1", "log_alpha", "accept", "loss"):
                np.testing.assert_array_equal(lm[key][sel], lr[key][sel], err_msg=key)
            for u, w in zip(qm, qr):
                np.testing.assert_array_equal(u[sel], w[sel])
        rows_m, rows_r = sel[cm], sel[cr]
        np.testing.assert_array_equal(sm[rows_m], sr[rows_r])
        np.testing.assert_array_equal(fm[rows_m], fr[rows_r])
        np.testing.assert_array_equal(cm[rows_m], cr[rows_r])


def _adapted_accept(name, eps, target, n_adapt, n_samp, S=None):
    eng = _engine(name, seed=21, S=S, eps=eps)
    eng.hmc_run(10, burning=True, sampling=False)          # the reference's burn-in
    eng.hmc_adapt_begin(target)
    eng.hmc_run(n_adapt, burning=False, sampling=False)
    eng.hmc_adapt_end()
    probs = []
    for _ in range(n_samp):
        eng.hmc_run(1, burning=False, sampling=True)
        probs.append(_accept_prob(eng.hmc_last()["log_alpha"]))
    return float(np.mean(probs)), eng.hmc_step_sizes()


@pytest.mark.parametrize("target", [0.8, 0.6])
@pytest.mark.parametrize("eps", [0.05, 1e-4])
def test_adaptation_reaches_the_target(eps, target):
    rate, steps = _adapted_accept("moons", eps, target, 400, 200)
    assert abs(rate - target) <= 0.06, (rate, target, np.median(steps))     # measured on a B200: 0.036 at most
    assert np.isfinite(steps).all() and (steps > 0).all()


def test_adaptation_reaches_the_target_on_the_tensor_path():
    rate, steps = _adapted_accept("mnist_shaped", 2e-4, 0.8, 300, 40, S=8)
    assert abs(rate - 0.8) <= 0.2, (rate, steps)


@pytest.mark.parametrize("name", ["moons", "deep_tanh"])
def test_one_call_equals_many(name):
    a, b = _engine(name), _engine(name)
    for e in (a, b):
        e.hmc_run(2, burning=True, sampling=False)
        e.hmc_adapt_begin(0.8)
    a.hmc_run(50, burning=False, sampling=False)
    for _ in range(50):
        b.hmc_run(1, burning=False, sampling=False)
    np.testing.assert_array_equal(a.hmc_step_sizes(), b.hmc_step_sizes())
    for e in (a, b):
        e.hmc_adapt_end()
    np.testing.assert_array_equal(a.hmc_step_sizes(), b.hmc_step_sizes())
    for u, v in zip(a.hmc_state(), b.hmc_state()):
        np.testing.assert_array_equal(u, v)


def test_lifecycle_and_errors():
    js, X, y, S, eps, m, L, _ = _problem("moons")
    eng = Engine(keras_json.parse_model_json(js), seed=7)
    eng.set_dataset(X, y, _lib.LOSS_SPARSE_CE)
    eng.set_prior([0.0], [1.0], _lib.PRIOR_SCALAR)
    buf = np.full(S, eps)
    lib, h = eng.lib, eng.h
    assert lib.pyb_hmc_adapt_begin(h, 0.8) == ERR_STATE                 # before pyb_hmc_init
    assert lib.pyb_hmc_adapt_end(h) == ERR_STATE
    assert lib.pyb_hmc_step_sizes(h, buf.ctypes.data) == ERR_STATE
    assert lib.pyb_hmc_set_step_sizes(h, buf.ctypes.data) == ERR_STATE
    eng.hmc_init(S, eps, m, L)
    np.testing.assert_array_equal(eng.hmc_step_sizes(), np.full(S, eps))
    eng.hmc_run(2, burning=True, sampling=False)

    def snapshot():
        return eng.hmc_state(), eng.hmc_step_sizes()

    def unchanged(before):
        (q0, p0), s0 = before
        (q1, p1), s1 = snapshot()
        np.testing.assert_array_equal(q0, q1)
        np.testing.assert_array_equal(p0, p1)
        np.testing.assert_array_equal(s0, s1)

    before = snapshot()
    assert lib.pyb_hmc_adapt_end(h) == ERR_STATE                        # not adapting
    for bad in (0.0, 1.0, -0.5, 1.5, float("nan")):
        assert lib.pyb_hmc_adapt_begin(h, bad) == ERR_INVALID
    assert lib.pyb_hmc_adapt_end(h) == ERR_STATE                        # a refused begin starts nothing
    for bad in (0.0, -eps, float("nan"), float("inf")):
        v = np.full(S, eps)
        v[S // 2] = bad
        assert lib.pyb_hmc_set_step_sizes(h, v.ctypes.data) == ERR_INVALID
    with pytest.raises(ValueError):
        eng.hmc_set_step_sizes(np.full(S + 1, eps))
    unchanged(before)

    eng.hmc_set_step_sizes(np.linspace(0.5, 1.5, S) * eps)
    eng.hmc_adapt_begin(0.8)
    before = snapshot()
    assert lib.pyb_hmc_run(h, 1, 0, 1, None) == ERR_STATE              # sampling while adapting
    assert lib.pyb_hmc_adapt_begin(h, 0.8) == ERR_STATE                 # already adapting
    assert lib.pyb_hmc_set_step_sizes(h, buf.ctypes.data) == ERR_STATE
    unchanged(before)
    assert eng.hmc_samples()[0].shape[0] == 0
    eng.hmc_run(3, burning=False, sampling=False)
    eng.hmc_adapt_end()
    eng.hmc_run(2, burning=False, sampling=True)                         # sampling is allowed again
    assert eng.hmc_samples()[0].shape[0] > 0

    # pyb_hmc_init ends adaptation and drops the per-chain step sizes: the run is a fresh scalar run
    eng.hmc_adapt_begin(0.8)
    eng.hmc_init(S, eps, m, L)
    np.testing.assert_array_equal(eng.hmc_step_sizes(), np.full(S, eps))
    assert lib.pyb_hmc_adapt_end(h) == ERR_STATE
    fresh = _engine("moons")
    for e in (eng, fresh):
        e.hmc_run(2, burning=True, sampling=False)
        e.hmc_run(2, burning=False, sampling=True)
    for u, v in zip(eng.hmc_state(), fresh.hmc_state()):
        np.testing.assert_array_equal(u, v)
    for u, v in zip(eng.hmc_samples(), fresh.hmc_samples()):
        np.testing.assert_array_equal(u, v)


def _optimizer(devices=None, n_chains=64, adapt=200, **extra):
    x, y = moons(1000)
    ds = Dataset((x, y), "SparseCategoricalCrossentropy", "Classification", seed=0)
    if devices is not None:
        extra["devices"] = devices
    opt = HMC()
    opt.compile(HyperParameters(epsilon=0.005, m=0.5, L=20, n_chains=n_chains, seed=11, adapt_iterations=adapt, **extra),
                keras_json.make_sequential_json(2, [50, 2], ["relu", "softmax"]), ds, verbose=False,
                prior=GaussianPrior(0.0, 1.0))
    x_test, y_test = next(iter(ds.test_data.batch(ds.test_size)))
    return opt, np.asarray(x_test), np.asarray(y_test)


def test_drop_in_flow_through_the_optimizer():
    opt, x_test, _ = _optimizer()
    np.testing.assert_array_equal(opt.step_sizes, np.full(64, 0.005))     # before train: epsilon everywhere
    opt.track_predictive(x_test)
    opt.train(100)
    steps = opt.step_sizes
    assert steps.shape == (64,) and steps.dtype == np.float64
    assert np.isfinite(steps).all() and (steps > 0).all() and not np.all(steps == 0.005)
    assert abs(opt.accept_rate - 0.8) <= 0.1, opt.accept_rate                # the sampling iterations only
    pr = opt.predictive()
    assert pr.n_chains == 64 and pr.n_draws == 101                          # adaptation records no draw
    bm = opt.result()
    assert sum(bm._distributions[0].frequencies) == 64 * 101
    _, exact = bm.predict(x_test, 0, mode="exact")
    np.testing.assert_allclose(pr.mean, exact, rtol=0, atol=1e-6)
    with pytest.raises(ValueError):
        _optimizer(target_accept=1.0)


def test_two_gpus_give_the_one_gpu_step_sizes():
    if _lib.device_count() < 2:
        pytest.skip("needs two GPUs")
    runs = []
    for devices in ([0], [0, 1]):
        opt, _, _ = _optimizer(devices=devices, n_chains=16, adapt=50)
        opt.train(20)
        d = opt.result()._distributions[0]
        runs.append((opt.step_sizes, d.samples.copy(), list(d.frequencies), opt.accept_rate))
    (e1, s1, f1, a1), (e2, s2, f2, a2) = runs
    np.testing.assert_array_equal(e1, e2)
    np.testing.assert_array_equal(s1, s2)
    assert f1 == f2 and a1 == a2
