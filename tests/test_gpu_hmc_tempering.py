"""GPU tests of parallel tempering (pyb_hmc_set_temperatures, pyb_hmc_tempering_stats, pyb_hmc_last_swaps, option
"hmc_swap"): the cold rung against untempered chains bit for bit, one tempered iteration against a float64
restatement, the swap rule against its Philox restatement, every rung's distribution on a model whose tempered
posteriors are Gaussian in closed form, mode-hopping on a sign-symmetric posterior, the tracked predictive over the cold
draws, sharding by replica groups, the lifecycle rules and the optimizer flow."""
import numpy as np
import pytest

pytestmark = pytest.mark.gpu

import pyesian_oracle as O  # noqa: E402
from Pyesian.datasets import Dataset  # noqa: E402
from Pyesian.distributions import GaussianPrior  # noqa: E402
from Pyesian.optimizers import HMC  # noqa: E402
from Pyesian.optimizers.hyperparameters import HyperParameters  # noqa: E402
from bayesian_inference_for_nn_b200 import _lib, keras_json  # noqa: E402
from bayesian_inference_for_nn_b200.engine import Engine  # noqa: E402

ERR_INVALID, ERR_STATE = -1, -3
PATHS = {"moons": _lib.PATH_FUSED_SMALL, "mnist_shaped": _lib.PATH_TENSOR, "deep_tanh": _lib.PATH_GENERIC}
LADDERS = {2: [1.0, 0.5], 3: [1.0, 0.6, 0.3], 4: [1.0, 0.7, 0.45, 0.2]}


def moons(n, seed=0, noise=0.2):
    rng = np.random.default_rng(seed)
    n0 = n // 2
    t0, t1 = rng.uniform(0, np.pi, n0), rng.uniform(0, np.pi, n - n0)
    x = np.concatenate([np.stack([np.cos(t0), np.sin(t0)], 1), np.stack([1 - np.cos(t1), 0.5 - np.sin(t1)], 1)])
    y = np.concatenate([np.zeros(n0, np.int64), np.ones(n - n0, np.int64)])
    return (x + rng.normal(0, noise, x.shape)).astype(np.float32), y.astype(np.int32)


def _problem(name):
    """-> (model json, X, y, chains, eps, m, L, path): the fused-small, tensor and generic shapes of
    test_gpu_hmc_adapt.py, with chain counts that several ladder lengths divide"""
    rng = np.random.default_rng(3)
    if name == "moons":          # fused-small HMC
        X, y = moons(400)
        return keras_json.make_sequential_json(2, [50, 2], ["relu", "softmax"]), X, y, 64, 0.005, 0.5, 10, _lib.PATH_AUTO
    if name == "mnist_shaped":   # tensor path
        X = rng.random((640, 784), dtype=np.float32)
        y = rng.integers(0, 10, 640).astype(np.int32)
        return keras_json.make_sequential_json(784, [256, 10], ["relu", "softmax"]), X, y, 8, 2e-4, 1.0, 5, _lib.PATH_AUTO
    if name == "deep_tanh":      # generic path
        X = rng.normal(0, 1, (300, 4)).astype(np.float32)
        y = rng.integers(0, 3, 300).astype(np.int32)
        return (keras_json.make_sequential_json(4, [16, 16, 3], ["tanh", "tanh", "softmax"]), X, y, 12, 0.01, 1.0, 5,
                _lib.PATH_GENERIC)
    raise KeyError(name)


def _engine(name, seed=7, S=None, chain_offset=0, ladder=None, swap=True, carry=True, sem=_lib.HMC_REFERENCE):
    js, X, y, S0, eps, m, L, path = _problem(name)
    eng = Engine(keras_json.parse_model_json(js), seed=seed)
    eng.set_option("path", path)
    if name == "mnist_shaped":
        eng.set_option("tc_i8", 0)       # the automatic int8 guard looks at all chains together, hot rungs included
    if not carry:
        eng.set_option("hmc_carry", 0)
    if not swap:
        eng.set_option("hmc_swap", 0)
    eng.set_dataset(X, y, _lib.LOSS_SPARSE_CE)
    eng.set_prior([0.0], [1.0], _lib.PRIOR_SCALAR)
    eng.hmc_init(S or S0, eps, m, L, semantics=sem, chain_offset=chain_offset)
    if ladder is not None:
        eng.hmc_set_temperatures(ladder)
    return eng


def _iterations(eng, n_burn=2, n_samp=3):
    out = []
    for i in range(n_burn + n_samp):
        if i == n_burn:
            eng.hmc_reset_samples()
        eng.hmc_run(1, burning=i < n_burn, sampling=i >= n_burn)
        out.append((eng.hmc_last(), eng.hmc_state()))
    return out, eng.hmc_samples()


# ---- 1. the cold rung of a ladder without swaps is an untempered chain ----------------------------------------------
@pytest.mark.parametrize("name,R,carry", [("moons", 4, True), ("mnist_shaped", 4, True), ("mnist_shaped", 2, False),
                                          ("deep_tanh", 3, True)])
def test_cold_rung_without_swaps_is_the_untempered_chain(name, R, carry):
    plain = _engine(name, carry=carry)
    tempered = _engine(name, carry=carry, ladder=LADDERS[R], swap=False)
    rp, (sp, fp, cp) = _iterations(plain)
    rt, (st, ft, ct) = _iterations(tempered)
    assert plain.info("path_used") == tempered.info("path_used") == PATHS[name]
    cold = np.arange(plain.S) % R == 0
    for (lp, qp), (lt, qt) in zip(rp, rt):
        for k in ("U0", "K0", "U1", "K1", "log_alpha", "accept", "loss"):
            np.testing.assert_array_equal(lp[k][cold], lt[k][cold], err_msg=k)
        for u, v in zip(qp, qt):
            np.testing.assert_array_equal(u[cold], v[cold])
    rows = cold[cp]
    assert (ct % R == 0).all()
    np.testing.assert_array_equal(sp[rows], st)
    np.testing.assert_array_equal(fp[rows], ft)
    np.testing.assert_array_equal(cp[rows], ct)


# ---- 2. one tempered iteration against float64 ----------------------------------------------------------------------
def _tempered_restatement(prob, beta, q, p, u, eps, m, L):
    """float64 tempered leapfrog (reference semantics) from the oracle's loss / prior: U = nlp + beta n_train loss,
    dU/dq = gp + beta n_train g"""
    def pot(x):
        loss, g = O.mean_loss_and_grad(prob.spec, x, prob.X, prob.y, prob.loss_kind, np.float64)
        nlp, gp = O.prior_neg_logp_and_grad(x, prob.mu, prob.sigma, np.float64)
        return nlp + beta * prob.n_train * loss, gp + (beta * prob.n_train)[:, None] * g, loss
    q = q.astype(np.float64)
    p = p.astype(np.float64)
    K0 = (p * p).sum(1) / (2 * m)
    U0, g, loss0 = pot(q)
    p = p - eps / 2 * g
    for _ in range(L):
        q = q + eps / m * p
        U1, g, loss1 = pot(q)
        p = p - eps * g
    p = p - eps / 2 * g
    K1 = (p * p).sum(1) / (2 * m)
    la = ((K0 + U0) - K1) - U1
    return dict(U0=U0, U1=U1, K0=K0, K1=K1, log_alpha=la, accept=u < np.exp(la), loss0=loss0, loss1=loss1)


@pytest.mark.parametrize("name", ["moons", "mnist_shaped", "deep_tanh"])
def test_tempered_iteration_matches_float64(name):
    R = 4
    js, X, y, S, eps, m, L, _ = _problem(name)
    eng = _engine(name, ladder=LADDERS[R], swap=False)
    eng.hmc_run(2, burning=True, sampling=False)
    q, _ = eng.hmc_state()
    rng = np.random.default_rng(5)
    p = rng.normal(0, 1, q.shape).astype(np.float32)
    u = rng.random(S).astype(np.float32)
    eng.hmc_inject(p=p, u=u)
    eng.hmc_run(1, burning=False, sampling=False)
    assert eng.info("path_used") == PATHS[name]
    last = eng.hmc_last()
    spec = keras_json.parse_model_json(js)
    ospec = O.MLPSpec(spec.in_dim, [d.units for d in spec.dense], [d.activation for d in spec.dense])
    P = q.shape[1]
    prob = O.Problem(ospec, X.astype(np.float64), y, O.LOSS_SPARSE_CE, np.zeros(P), np.ones(P))
    beta = np.asarray(LADDERS[R])[np.arange(S) % R]
    want = _tempered_restatement(prob, beta, q, p, u, eps, m, L)
    scale = np.maximum(np.abs(want["U0"]), 1.0)
    np.testing.assert_allclose(last["U0"], want["U0"], rtol=1e-4)
    np.testing.assert_allclose(last["U1"], want["U1"], rtol=1e-3)           # the end point of L leapfrog steps
    assert np.all(np.abs(last["log_alpha"] - want["log_alpha"]) <= 2e-4 * scale), (last["log_alpha"], want["log_alpha"])
    lu = np.log(np.maximum(u.astype(np.float64), 1e-300))
    decisive = np.abs(want["log_alpha"] - lu) > 4e-4 * scale           # twice the log_alpha budget
    np.testing.assert_array_equal(last["accept"][decisive], want["accept"][decisive])
    # the carried evaluation stays untempered: what step() returns is the mean loss
    np.testing.assert_allclose(last["loss"], np.where(last["accept"], want["loss1"], want["loss0"]), rtol=1e-3)


# ---- 3. the swap rule, exactly --------------------------------------------------------------------------------------
@pytest.mark.parametrize("R", [2, 3, 4])
@pytest.mark.parametrize("parity", [0, 1])
def test_swap_rule_and_exchange_exactly(R, parity):
    name = "deep_tanh"
    seed = 13
    a = _engine(name, seed=seed, ladder=LADDERS[R])
    b = _engine(name, seed=seed, ladder=LADDERS[R], swap=False)
    a.set_option("hmc_swap", 0)
    for e in (a, b):
        e.hmc_run(1 + parity, burning=True, sampling=False)     # identical states up to here (no swaps proposed)
    a.set_option("hmc_swap", 1)
    it = 1 + parity                                             # the iteration counter of the swapping iteration
    for e in (a, b):
        e.hmc_run(1, burning=False, sampling=False)
    la, lb = a.hmc_last(), b.hmc_last()
    for k in ("U0", "K0", "U1", "K1", "log_alpha", "accept"):
        np.testing.assert_array_equal(la[k], lb[k], err_msg=k)   # everything before the swap is shared
    S = a.S
    r = np.arange(S) % R
    lower = (r + 1 < R) & (r % 2 == it % 2)
    beta = np.asarray(LADDERS[R])
    n_train = _problem(name)[1].shape[0]
    loss = lb["loss"].astype(np.float64)                         # the pre-swap losses
    want_lr = np.full(S, np.nan)
    idx = np.nonzero(lower)[0]
    want_lr[idx] = (beta[r[idx]] - beta[r[idx] + 1]) * float(n_train) * (loss[idx] - loss[idx + 1])
    uni = O.philox_uniforms(seed, np.arange(S), it, stream=4).astype(np.float64)
    want_sw = np.zeros(S, bool)
    with np.errstate(over="ignore"):
        want_sw[idx] = uni[idx] < np.exp(want_lr[idx])
    log_r, swapped = a.hmc_last_swaps()
    np.testing.assert_array_equal(np.isnan(log_r), ~lower)
    np.testing.assert_allclose(log_r[idx], want_lr[idx].astype(np.float32), rtol=1e-12)
    away = np.abs(np.log(np.maximum(uni[idx], 1e-300)) - want_lr[idx]) > 1e-9 * np.maximum(np.abs(want_lr[idx]), 1.0)
    np.testing.assert_array_equal(swapped[idx][away], want_sw[idx][away])
    assert not swapped[~lower].any()
    perm = np.arange(S)
    for s in idx[swapped[idx]]:
        perm[s], perm[s + 1] = s + 1, s
    qa, _ = a.hmc_state()
    qb, _ = b.hmc_state()
    np.testing.assert_array_equal(qa, qb[perm])
    np.testing.assert_array_equal(la["loss"], lb["loss"][perm])
    st = a.hmc_tempering_stats()
    np.testing.assert_array_equal(st["swap_attempted"], [np.sum(lower & (r == k)) for k in range(R - 1)])
    np.testing.assert_array_equal(st["swap_accepted"], [np.sum(swapped & (r == k)) for k in range(R - 1)])
    np.testing.assert_array_equal(st["rung_total"], np.full(R, S // R))
    np.testing.assert_array_equal(st["rung_accepted"], [np.sum(la["accept"] & (r == k)) for k in range(R)])
    # a swapped state keeps its carried evaluation: the next iteration's U0 of every chain is its own state's
    a.hmc_run(1, burning=False, sampling=False)
    U, lossq, _ = a.hmc_eval(qa.copy(), want_grad=False)
    nt = float(n_train)
    prior = U.astype(np.float64) - nt * lossq
    np.testing.assert_allclose(a.hmc_last()["U0"], prior + beta[r] * nt * lossq, rtol=1e-5)


# ---- 4. every rung samples its tempered posterior -------------------------------------------------------------------
def _linear_problem():
    rng = np.random.default_rng(11)
    N = 20
    X = rng.normal(0, 1, (N, 2)).astype(np.float32)
    y = (X @ np.array([0.8, -0.5]) + 0.3 + rng.normal(0, 0.5, N)).astype(np.float32).reshape(N, 1)
    return X, y


def _batch_means_se(x, n_batches=20):
    """standard error of the mean of the series x [T, ...] by batch means"""
    T = x.shape[0] - x.shape[0] % n_batches
    b = x[:T].reshape(n_batches, T // n_batches, *x.shape[1:]).mean(1)
    return b.std(0, ddof=1) / np.sqrt(n_batches)


def test_every_rung_samples_its_tempered_gaussian():
    X, y = _linear_problem()
    N = X.shape[0]
    ladder = [1.0, 0.5, 0.25, 0.1]
    R, G = len(ladder), 256
    spec = keras_json.parse_model_json(keras_json.make_sequential_json(2, [1], ["linear"]))
    eng = Engine(spec, seed=3)
    eng.set_option("path", _lib.PATH_GENERIC)
    eng.set_dataset(X, y, _lib.LOSS_MSE)
    eng.set_prior([0.0], [1.0], _lib.PRIOR_SCALAR)
    eng.hmc_init(G * R, 0.05, 1.0, 10, semantics=_lib.HMC_CANONICAL)
    eng.hmc_set_temperatures(ladder)
    eng.hmc_run(200, burning=False, sampling=False)
    T = 400
    qs = np.empty((T, G * R, 3), np.float64)
    swaps = np.zeros(R - 1, np.int64)
    for t in range(T):
        eng.hmc_run(1, burning=False, sampling=False)
        qs[t] = eng.hmc_state()[0]
        swaps += eng.hmc_tempering_stats()["swap_accepted"]      # counts of the last call: one round parity
    assert (swaps > 0).all(), swaps
    # closed form: theta = (w1, w2, b), E = n_train mean (A theta - y)^2 = sum (A theta - y)^2 (n_train = N)
    A = np.concatenate([X.astype(np.float64), np.ones((N, 1))], 1)
    yy = y[:, 0].astype(np.float64)
    for r, b in enumerate(ladder):
        prec = np.eye(3) + 2.0 * b * A.T @ A
        cov = np.linalg.inv(prec)
        mean = cov @ (2.0 * b * A.T @ yy)
        q = qs[:, r::R]                                   # [T, G, 3]
        m_t = q.mean(1)                                   # chain-averaged series
        se = _batch_means_se(m_t)
        got = m_t.mean(0)
        assert np.all(np.abs(got - mean) <= 5 * se + 1e-9), (r, got, mean, se)
        v_t = ((q - mean) ** 2).mean(1)
        se_v = _batch_means_se(v_t)
        assert np.all(np.abs(v_t.mean(0) - np.diag(cov)) <= 5 * se_v + 1e-9), (r, v_t.mean(0), np.diag(cov), se_v)


# ---- 5. mode-hopping on a sign-symmetric posterior ------------------------------------------------------------------
def _tanh_problem():
    rng = np.random.default_rng(2)
    X = rng.uniform(-2, 2, (50, 1)).astype(np.float32)
    y = (2.0 * np.tanh(1.5 * X) + rng.normal(0, 0.1, X.shape)).astype(np.float32)
    return X, y


def _w2_positive_fraction(ladder, n_chains, n_adapt=300, n_samp=1000):
    X, y = _tanh_problem()
    spec = keras_json.parse_model_json(keras_json.make_sequential_json(1, [1, 1], ["tanh", "linear"]))
    eng = Engine(spec, seed=5)
    eng.set_dataset(X, y, _lib.LOSS_MSE)
    eng.set_prior([0.0], [1.0], _lib.PRIOR_SCALAR)
    q0 = np.tile(np.array([1.5, 0.0, 2.0, 0.0], np.float32), (n_chains, 1))    # (w1, b1, w2, b2): all in w2 > 0
    eng.hmc_init(n_chains, 0.01, 1.0, 10, semantics=_lib.HMC_CANONICAL, q0=q0)
    if ladder is not None:
        eng.hmc_set_temperatures(ladder)
    eng.hmc_adapt_begin(0.7)
    eng.hmc_run(n_adapt, burning=False, sampling=False)
    eng.hmc_adapt_end()
    eng.hmc_run(n_samp, burning=False, sampling=True)
    s, f, c = eng.hmc_samples()
    frac = float(np.sum(f * (s[:, 2] > 0)) / np.sum(f))
    return frac, eng


def test_tempering_hops_between_the_sign_modes():
    ladder = list(np.geomspace(1.0, 1e-3, 8))
    ladder[0] = 1.0
    frac_plain, _ = _w2_positive_fraction(None, 64 * 8)
    frac_pt, eng = _w2_positive_fraction(ladder, 64 * 8)
    rates = eng.hmc_tempering_stats()
    print("w2>0 fraction: untempered %.4f tempered %.4f; swap acceptance %s" % (
        frac_plain, frac_pt, rates["swap_accepted"] / np.maximum(1, rates["swap_attempted"])))
    # measured on a B200: untempered 1.0000 (no cold draw ever left the starting mode), tempered 0.4806
    assert frac_plain >= 0.99, frac_plain
    assert abs(frac_pt - 0.5) <= 0.06, frac_pt


# ---- 6. the tracked predictive of a tempered run --------------------------------------------------------------------
def test_tracked_predictive_is_the_cold_draws():
    R = 2
    eng = _engine("moons", ladder=LADDERS[R])
    G = eng.S // R
    xt = moons(100, seed=9)[0]
    eng.hmc_track_predictive(xt)
    eng.hmc_run(3, burning=True, sampling=False)
    eng.hmc_run(20, burning=False, sampling=True)
    sums, s2, T = eng.hmc_predictive_sums()
    assert T == 21
    s, f, c = eng.hmc_samples()
    assert (c % R == 0).all() and len(np.unique(c)) == G
    for g in range(G):
        assert f[c == g * R].sum() == T
    res = eng.hmc_predictive_finish(sums, s2, G, T)
    mean, var = eng.predict(s, xt, weights=f)[:2]
    np.testing.assert_allclose(res["mean"], mean, rtol=0, atol=1e-6)
    np.testing.assert_allclose(res["variance"], var, rtol=0, atol=1e-6)
    assert np.isfinite(res["rhat"]).any()


# ---- 7. sharding by replica groups ----------------------------------------------------------------------------------
def test_two_handles_reproduce_one():
    R, S = 4, 160                   # every handle runs one CTA per chain on the fused path (no cluster)
    ladder = LADDERS[R]

    def run(e):
        e.hmc_run(3, burning=True, sampling=False)
        e.hmc_adapt_begin(0.8)
        e.hmc_run(10, burning=False, sampling=False)
        e.hmc_adapt_end()
        e.hmc_reset_samples()
        e.hmc_run(8, burning=False, sampling=True)
        return e.hmc_samples(), e.hmc_tempering_stats(), e.hmc_step_sizes()

    one = _engine("moons", S=S, ladder=ladder)
    (s1, f1, c1), st1, e1 = run(one)
    halves = [_engine("moons", S=S // 2, chain_offset=k * S // 2, ladder=ladder) for k in range(2)]
    parts = [run(e) for e in halves]
    np.testing.assert_array_equal(s1, np.concatenate([p[0][0] for p in parts]))
    np.testing.assert_array_equal(f1, np.concatenate([p[0][1] for p in parts]))
    np.testing.assert_array_equal(c1, np.concatenate([p[0][2] for p in parts]))
    np.testing.assert_array_equal(e1, np.concatenate([p[2] for p in parts]))
    for k in st1:
        np.testing.assert_array_equal(st1[k], parts[0][1][k] + parts[1][1][k], err_msg=k)
    assert st1["swap_accepted"].sum() > 0


def _optimizer(devices=None, n_chains=16, ladder=(1.0, 0.5, 0.25), adapt=50, **extra):
    x, y = moons(1000)
    ds = Dataset((x, y), "SparseCategoricalCrossentropy", "Classification", seed=0)
    if devices is not None:
        extra["devices"] = devices
    if ladder is not None:
        extra["inverse_temperatures"] = list(ladder)
    opt = HMC()
    opt.compile(HyperParameters(epsilon=0.005, m=0.5, L=20, n_chains=n_chains, seed=11, adapt_iterations=adapt, **extra),
                keras_json.make_sequential_json(2, [50, 2], ["relu", "softmax"]), ds, verbose=False,
                prior=GaussianPrior(0.0, 1.0))
    x_test, y_test = next(iter(ds.test_data.batch(ds.test_size)))
    return opt, np.asarray(x_test), np.asarray(y_test)


def test_two_gpus_give_the_one_gpu_run():
    if _lib.device_count() < 2:
        pytest.skip("needs two GPUs")
    runs = []
    for devices in ([0], [0, 1]):
        opt, _, _ = _optimizer(devices=devices, n_chains=16, adapt=20)
        opt.train(10)
        d = opt.result()._distributions[0]
        runs.append((opt.step_sizes, d.samples.copy(), list(d.frequencies), opt.accept_rate, opt.tempering_rates()))
    (e1, s1, f1, a1, t1), (e2, s2, f2, a2, t2) = runs
    np.testing.assert_array_equal(e1, e2)
    np.testing.assert_array_equal(s1, s2)
    assert f1 == f2 and a1 == a2
    for u, v in zip(t1, t2):
        np.testing.assert_array_equal(u, v)


# ---- 8. lifecycle and errors ----------------------------------------------------------------------------------------
def test_lifecycle_and_errors():
    js, X, y, S, eps, m, L, _ = _problem("deep_tanh")      # S = 12
    eng = Engine(keras_json.parse_model_json(js), seed=7)
    eng.set_option("path", _lib.PATH_GENERIC)
    eng.set_dataset(X, y, _lib.LOSS_SPARSE_CE)
    eng.set_prior([0.0], [1.0], _lib.PRIOR_SCALAR)
    lib, h = eng.lib, eng.h
    good = np.array([1.0, 0.5, 0.25], np.float64)
    i64 = np.zeros(4, np.int64)
    lr = np.zeros(S, np.float32)
    sw = np.zeros(S, np.int32)
    assert lib.pyb_hmc_set_temperatures(h, good.ctypes.data, 3) == ERR_STATE          # before pyb_hmc_init
    assert lib.pyb_hmc_tempering_stats(h, None, None, None, None) == ERR_STATE
    assert lib.pyb_hmc_last_swaps(h, None, None) == ERR_STATE
    eng.hmc_init(S, eps, m, L)
    assert lib.pyb_hmc_tempering_stats(h, i64.ctypes.data, None, None, None) == ERR_STATE   # no ladder
    bad = [[0.9, 0.5], [1.0, 1.0], [1.0, 0.5, 0.6], [1.0, 0.0], [1.0, -0.5], [1.0, float("nan")],
           [1.0, float("inf")], [1.0], [1.0, 0.5, 0.4, 0.3, 0.2],                    # R = 1; R = 5 does not divide 12
           list(np.geomspace(1.0, 1e-3, 65))]
    for b in bad:
        a = np.asarray(b, np.float64)
        assert lib.pyb_hmc_set_temperatures(h, a.ctypes.data, len(b)) == ERR_INVALID, b
    assert lib.pyb_hmc_set_temperatures(h, None, 2) == ERR_INVALID
    assert lib.pyb_hmc_set_temperatures(h, good.ctypes.data, 0) == ERR_INVALID
    assert lib.pyb_hmc_tempering_stats(h, None, None, None, None) == ERR_STATE        # refused ladders set nothing
    eng.hmc_init(S, eps, m, L, chain_offset=2)
    assert lib.pyb_hmc_set_temperatures(h, good[:2].ctypes.data, 2) == 0              # 2 | 2
    assert lib.pyb_hmc_set_temperatures(h, good.ctypes.data, 3) == ERR_INVALID        # chain_offset 2 is not a multiple of 3
    eng.hmc_init(S, eps, m, L)
    eng.hmc_set_temperatures(good)
    assert lib.pyb_hmc_last_swaps(h, lr.ctypes.data, sw.ctypes.data) == ERR_STATE     # no iteration under the ladder yet
    eng.hmc_run(2, burning=True, sampling=False)
    eng.hmc_set_temperatures([1.0, 0.3, 0.1])           # burn-in does not lock the ladder
    # adaptation under a ladder: every rung adapts its own step size
    eng.hmc_adapt_begin(0.8)
    eng.hmc_run(30, burning=False, sampling=False)
    eng.hmc_adapt_end()
    steps = eng.hmc_step_sizes().reshape(-1, 3)
    assert np.isfinite(steps).all() and (steps > 0).all() and not np.all(steps == eps)
    eng.hmc_run(1, burning=False, sampling=True)
    assert lib.pyb_hmc_set_temperatures(h, good.ctypes.data, 3) == ERR_STATE           # a sampling iteration has run
    assert lib.pyb_hmc_set_temperatures(h, None, 0) == ERR_STATE
    st = eng.hmc_tempering_stats()
    assert st["rung_total"].tolist() == [S // 3] * 3
    log_r, swapped = eng.hmc_last_swaps()
    assert np.isnan(log_r).sum() == S - (S // 3)        # one proposing chain per group in each round of R = 3
    eng.hmc_reset_samples()
    eng.hmc_set_temperatures(None)                      # allowed again after pyb_hmc_reset_samples; turns tempering off
    assert lib.pyb_hmc_tempering_stats(h, None, None, None, None) == ERR_STATE
    eng.hmc_set_temperatures(good)
    eng.hmc_init(S, eps, m, L)                          # pyb_hmc_init clears the ladder
    assert lib.pyb_hmc_tempering_stats(h, None, None, None, None) == ERR_STATE
    assert lib.pyb_hmc_last_swaps(h, None, None) == ERR_STATE
    fresh = _engine("deep_tanh")
    for e in (eng, fresh):
        e.hmc_run(2, burning=True, sampling=False)
        e.hmc_run(2, burning=False, sampling=True)
    for u, v in zip(eng.hmc_samples(), fresh.hmc_samples()):
        np.testing.assert_array_equal(u, v)


# ---- 9. the optimizer flow ------------------------------------------------------------------------------------------
def test_optimizer_flow():
    opt, x_test, y_test = _optimizer()
    assert opt.step_sizes.shape == (16, 3)
    opt.track_predictive(x_test, y_test)
    opt.train(30)
    rung, swap = opt.tempering_rates()
    assert rung.shape == (3,) and swap.shape == (2,)
    assert ((0 <= rung) & (rung <= 1)).all() and ((0 <= swap) & (swap <= 1)).all() and swap.sum() > 0
    assert opt.accept_rate == pytest.approx(rung[0])
    steps = opt.step_sizes
    assert steps.shape == (16, 3) and np.isfinite(steps).all()
    bm = opt.result()
    assert sum(bm._distributions[0].frequencies) == 16 * 31          # cold draws only
    pr = opt.predictive()
    assert pr.n_chains == 16 and pr.n_draws == 31
    _, exact = bm.predict(x_test, 0, mode="exact")
    np.testing.assert_allclose(pr.mean, exact, rtol=0, atol=1e-6)
    total, _, _ = opt.classification_uncertainty()
    assert total.shape[1:] == (2, 2)
    with pytest.raises(ValueError):
        _optimizer(ladder=(1.0, 1.5))
