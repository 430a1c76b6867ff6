"""GPU tests of the streamed HMC posterior predictive (pyb_hmc_track_predictive / _sums / _finish): the sums
accumulated while the chains run must give what BayesianModel.predict(mode="exact") and
Metrics.classification_uncertainty give over the recorded samples (BayesianModel.py:106-129, Metrics.py:344-375,
HMC.py:92-104), the R-hat of the per-draw outputs, and must leave the chains exactly as they are without tracking."""
import numpy as np
import pytest

pytestmark = pytest.mark.gpu

from Pyesian.datasets import Dataset  # noqa: E402
from Pyesian.distributions import GaussianPrior  # noqa: E402
from Pyesian.optimizers import HMC  # noqa: E402
from Pyesian.optimizers.hyperparameters import HyperParameters  # noqa: E402
from bayesian_inference_for_nn_b200 import _lib, keras_json  # noqa: E402
from bayesian_inference_for_nn_b200.engine import Engine  # noqa: E402

TOL = 2e-5   # uncertainty matrices: the tolerance of test_gpu_metrics.py


def moons(n, seed=0, noise=0.2):
    rng = np.random.default_rng(seed)
    n0 = n // 2
    t0, t1 = rng.uniform(0, np.pi, n0), rng.uniform(0, np.pi, n - n0)
    x = np.concatenate([np.stack([np.cos(t0), np.sin(t0)], 1), np.stack([1 - np.cos(t1), 0.5 - np.sin(t1)], 1)])
    y = np.concatenate([np.zeros(n0, np.int64), np.ones(n - n0, np.int64)])
    return (x + rng.normal(0, noise, x.shape)).astype(np.float32), y.astype(np.int32)


def _problem(name):
    """-> (model json, X, y, loss kind, chains, eps, m, L, path, test inputs, test labels)"""
    rng = np.random.default_rng(3)
    if name == "moons":          # fused-small HMC, generic forward
        X, y = moons(400)
        xt, yt = moons(150, seed=5)
        return (keras_json.make_sequential_json(2, [50, 2], ["relu", "softmax"]), X, y, _lib.LOSS_SPARSE_CE, 64, 0.005,
                0.5, 10, _lib.PATH_AUTO, xt, yt)
    if name == "mnist_shaped":   # tensor path, training and forward
        X = rng.random((640, 784), dtype=np.float32)
        y = rng.integers(0, 10, 640).astype(np.int32)
        xt = rng.random((300, 784), dtype=np.float32)
        return (keras_json.make_sequential_json(784, [256, 10], ["relu", "softmax"]), X, y, _lib.LOSS_SPARSE_CE, 5, 2e-4,
                1.0, 5, _lib.PATH_AUTO, xt, rng.integers(0, 10, 300).astype(np.int32))
    if name == "deep_tanh":      # generic path
        X = rng.normal(0, 1, (300, 4)).astype(np.float32)
        y = rng.integers(0, 3, 300).astype(np.int32)
        xt = rng.normal(0, 1, (200, 4)).astype(np.float32)
        return (keras_json.make_sequential_json(4, [16, 16, 3], ["tanh", "tanh", "softmax"]), X, y, _lib.LOSS_SPARSE_CE,
                12, 0.01, 1.0, 5, _lib.PATH_GENERIC, xt, rng.integers(0, 3, 200).astype(np.int32))
    if name == "regression":     # MSE, one output unit
        X = rng.uniform(-2, 2, (200, 1)).astype(np.float32)
        y = (np.sin(X) + rng.normal(0, 0.1, X.shape)).astype(np.float32)
        xt = np.linspace(-3, 3, 97, dtype=np.float32).reshape(-1, 1)
        return (keras_json.make_sequential_json(1, [8, 1], ["relu", "linear"]), X, y, _lib.LOSS_MSE, 16, 0.002, 1.0, 10,
                _lib.PATH_AUTO, xt, None)
    if name == "sigmoid":        # one-unit output widened to two classes for the uncertainty matrices
        X = rng.normal(0, 1, (300, 3)).astype(np.float32)
        y = (X[:, :1] > 0).astype(np.float32)
        xt = rng.normal(0, 1, (130, 3)).astype(np.float32)
        return (keras_json.make_sequential_json(3, [8, 1], ["tanh", "sigmoid"]), X, y, _lib.LOSS_MSE, 10, 0.01, 1.0, 5,
                _lib.PATH_AUTO, xt, (xt[:, 0] > 0).astype(np.int32))
    raise KeyError(name)


def _engine(name, seed=7, keep=True):
    js, X, y, loss, S, eps, m, L, path, xt, yt = _problem(name)
    eng = Engine(keras_json.parse_model_json(js), seed=seed)
    eng.set_option("path", path)
    eng.set_dataset(X, y, loss)
    eng.set_prior([0.0], [1.0], _lib.PRIOR_SCALAR)
    if not keep:
        eng.set_option("hmc_keep_samples", 0)
    eng.hmc_init(S, eps, m, L)
    return eng, xt, yt


def _run(eng, xt, yt, n_burn=3, n_samp=16, track=True):
    if track:
        eng.hmc_track_predictive(xt, yt)
    eng.hmc_run(n_burn, burning=True, sampling=False)
    eng.hmc_reset_samples()
    eng.hmc_run(n_samp, burning=False, sampling=True)


def _finish(eng, semantics=None, divisor=None):
    sums, s2, T = eng.hmc_predictive_sums()
    return eng.hmc_predictive_finish(sums, s2, eng.S, T, semantics, divisor), sums, s2, T


def _rhat_ref(o):
    """classic Gelman-Rubin over draws o [S, T, ...] in float64"""
    S, T = o.shape[:2]
    m = o.mean(axis=1)
    W = o.var(axis=1, ddof=1).mean(axis=0)
    B = T * m.var(axis=0, ddof=1)
    with np.errstate(divide="ignore", invalid="ignore"):
        r = np.sqrt(((T - 1) / T * W + B / T) / W)
    r[W == 0] = np.nan
    return r


@pytest.mark.parametrize("name", ["moons", "mnist_shaped", "deep_tanh", "regression"])
def test_streamed_equals_exact_over_the_samples(name):
    eng, xt, yt = _engine(name)
    n_samp = 16
    _run(eng, xt, yt, n_samp=n_samp)
    got, _, _, T = _finish(eng)
    samples, freq, chain = eng.hmc_samples()
    assert T == n_samp + 1
    assert all(freq[chain == c].sum() == T for c in range(eng.S))
    mean, var, allo = eng.predict(samples, xt, weights=freq.astype(np.float32), want_all=True)
    np.testing.assert_allclose(got["mean"], mean, rtol=0, atol=1e-6)
    np.testing.assert_allclose(got["variance"], var, rtol=0, atol=1e-6)
    # R-hat against the per-draw outputs: each chain's samples expanded by their frequencies into its draw sequence
    o = np.stack([np.repeat(allo[chain == c].astype(np.float64), freq[chain == c], axis=0) for c in range(eng.S)])
    want = _rhat_ref(o)
    np.testing.assert_array_equal(np.isnan(got["rhat"]), np.isnan(want))
    ok = ~np.isnan(want)
    assert ok.any()
    np.testing.assert_allclose(got["rhat"][ok], want[ok], rtol=1e-5)


@pytest.mark.parametrize("name", ["moons", "mnist_shaped", "deep_tanh", "sigmoid"])
def test_streamed_uncertainty_equals_exact_over_the_samples(name):
    eng, xt, yt = _engine(name)
    _run(eng, xt, yt, n_samp=15)
    samples, freq, _ = eng.hmc_samples()
    for semantics in ("reference", "canonical"):
        got, _, _, _ = _finish(eng, semantics, divisor=40)
        want = eng.predict_uncertainty(samples, xt, yt, weights=freq.astype(np.float32), semantics=semantics, divisor=40)
        for k, ref in zip(("total", "aleatoric", "epistemic"), want[:3]):
            assert got[k].shape == ref.shape
            assert np.abs(got[k] - ref).max() <= TOL * max(1.0, np.abs(ref).max()), (semantics, k)


@pytest.mark.parametrize("name", ["moons", "mnist_shaped"])
def test_tracking_does_not_change_the_chains(name):
    a, xt, yt = _engine(name)
    _run(a, xt, yt, track=False)
    b, _, _ = _engine(name)
    _run(b, xt, yt, track=True)
    for u, v in zip(a.hmc_state(), b.hmc_state()):
        np.testing.assert_array_equal(u, v)
    np.testing.assert_array_equal(a.hmc_last()["accept"], b.hmc_last()["accept"])
    for u, v in zip(a.hmc_samples(), b.hmc_samples()):
        np.testing.assert_array_equal(u, v)
    # one call of n iterations == n calls of one
    c, _, _ = _engine(name)
    c.hmc_track_predictive(xt, yt)
    c.hmc_run(3, burning=True, sampling=False)
    c.hmc_reset_samples()
    for _ in range(16):
        c.hmc_run(1, burning=False, sampling=True)
    for u, v in zip(b.hmc_predictive_sums(), c.hmc_predictive_sums()):
        np.testing.assert_array_equal(u, v)
    # no samples kept: the same chains and sums, no arena, no samples
    d, _, _ = _engine(name, keep=False)
    _run(d, xt, yt)
    for u, v in zip(b.hmc_state(), d.hmc_state()):
        np.testing.assert_array_equal(u, v)
    for u, v in zip(b.hmc_predictive_sums(), d.hmc_predictive_sums()):
        np.testing.assert_array_equal(u, v)
    assert d.hmc_samples()[0].shape[0] == 0
    assert d.info("hmc_arena_rows") == 0 and b.info("hmc_arena_rows") > 0


def test_lifecycle_and_errors():
    eng, xt, yt = _engine("moons")
    with pytest.raises(ValueError):
        eng.hmc_track_predictive(np.zeros((10, 3), np.float32))        # wrong feature count
    with pytest.raises(_lib.PyesianB200Error):
        eng.hmc_track_predictive(xt, np.full(xt.shape[0], 2))           # label out of range
    eng.hmc_track_predictive(xt)                                        # no labels
    eng.hmc_run(3, burning=True, sampling=False)
    with pytest.raises(_lib.PyesianB200Error):
        eng.hmc_predictive_sums()                                       # burn-in adds nothing: no draw yet
    eng.hmc_run(4, burning=False, sampling=True)
    sums, s2, T = eng.hmc_predictive_sums()
    assert T == 5 and s2 is None
    with pytest.raises(_lib.PyesianB200Error):
        eng.hmc_predictive_finish(sums, s2, eng.S, T, "reference")     # uncertainty without labels
    with pytest.raises(_lib.PyesianB200Error):
        eng.hmc_track_predictive(xt, yt)                                # sampling has started
    eng.hmc_reset_samples()                                             # clears the sums
    with pytest.raises(_lib.PyesianB200Error):
        eng.hmc_predictive_sums()
    eng.hmc_run(2, burning=False, sampling=True)
    got, _, _, T = _finish(eng)
    samples, freq, _ = eng.hmc_samples()
    assert T == 3 and freq.sum() == 3 * eng.S
    mean, var, _ = eng.predict(samples, xt, weights=freq.astype(np.float32))
    np.testing.assert_allclose(got["mean"], mean, rtol=0, atol=1e-6)
    # one sampling iteration gives two draws per chain (its start and its end); R-hat over a single chain is undefined
    one, _, _ = _engine("moons")
    one.hmc_track_predictive(xt)
    one.hmc_run(1, burning=False, sampling=False)
    with pytest.raises(_lib.PyesianB200Error):
        one.hmc_predictive_sums()
    one.hmc_run(1, burning=False, sampling=True)
    sums, s2, T = one.hmc_predictive_sums()
    assert T == 2
    assert np.isnan(one.hmc_predictive_finish(sums, s2, 1, T)["rhat"]).all()
    eng.hmc_init(eng.S, 0.005, 0.5, 10)                                 # re-init drops tracking
    eng.hmc_run(1, burning=False, sampling=True)
    buf = np.zeros(4 * xt.shape[0] * 2)
    assert eng.lib.pyb_hmc_predictive_sums(eng.h, buf.ctypes.data, None, None) == -3    # PYB_ERR_STATE
    with pytest.raises(_lib.PyesianB200Error):
        eng.set_option("hmc_keep_samples", 0)                           # not during a sampling phase


def _optimizer(keep=True, devices=None, n_chains=8):
    x, y = moons(1000)
    ds = Dataset((x, y), "SparseCategoricalCrossentropy", "Classification", seed=0)
    extra = {} if keep else {"keep_samples": False}
    if devices is not None:
        extra["devices"] = devices
    opt = HMC()
    opt.compile(HyperParameters(epsilon=0.005, m=0.5, L=20, n_chains=n_chains, seed=11, **extra),
                keras_json.make_sequential_json(2, [50, 2], ["relu", "softmax"]), ds, verbose=False,
                prior=GaussianPrior(0.0, 1.0))
    x_test, y_test = next(iter(ds.test_data.batch(ds.test_size)))
    return opt, np.asarray(x_test), np.asarray(y_test)


def test_drop_in_flow_through_the_optimizer():
    opt, x_test, y_test = _optimizer()
    opt.track_predictive(x_test, y_test)
    opt.train(60)
    with pytest.raises(RuntimeError):
        opt.track_predictive(x_test, y_test)
    pr = opt.predictive()
    assert pr.n_chains == 8 and pr.n_draws == 61
    assert pr.mean.shape == pr.variance.shape == pr.rhat.shape == (x_test.shape[0], 2)
    bm = opt.result()
    _, exact = bm.predict(x_test, 0, mode="exact")
    np.testing.assert_allclose(pr.mean, exact, rtol=0, atol=1e-6)
    np.testing.assert_allclose(pr.variance, bm.last_variance, rtol=0, atol=1e-6)
    for semantics in ("reference", "canonical"):
        got = opt.classification_uncertainty(semantics=semantics)
        want = bm.classification_uncertainty(x_test, y_test, 0, semantics=semantics, mode="exact")
        for g, w in zip(got, want):
            assert np.abs(g - w).max() <= TOL * max(1.0, np.abs(w).max())
    # no samples kept: result() refuses, the predictive still answers (same seed: the same chains)
    opt2, _, _ = _optimizer(keep=False)
    opt2.track_predictive(x_test, y_test)
    opt2.train(60)
    with pytest.raises(RuntimeError, match="predictive"):
        opt2.result()
    pr2 = opt2.predictive()
    np.testing.assert_array_equal(pr2.mean, pr.mean)
    np.testing.assert_array_equal(pr2.rhat, pr.rhat)
    opt3, _, _ = _optimizer()
    with pytest.raises(RuntimeError):
        opt3.predictive()                                   # nothing tracked


def test_two_gpus_give_the_one_gpu_answer():
    if _lib.device_count() < 2:
        pytest.skip("needs two GPUs")
    res = []
    for devices in ([0], [0, 1]):
        opt, x_test, y_test = _optimizer(devices=devices, n_chains=16)
        opt.track_predictive(x_test, y_test)
        opt.train(20)
        parts = opt._engine.each(lambda i, e: e.hmc_predictive_sums())
        res.append((sum(p[0] for p in parts), opt.predictive()))
    (s1, p1), (s2, p2) = res
    np.testing.assert_allclose(s2, s1, rtol=1e-12, atol=1e-12 * np.abs(s1).max())    # the float64 sums
    for a, b in zip(p1[:3], p2[:3]):                                                # finished in float32
        np.testing.assert_allclose(b, a, rtol=1e-6, atol=1e-7)
    assert (p1.n_chains, p1.n_draws) == (p2.n_chains, p2.n_draws)
