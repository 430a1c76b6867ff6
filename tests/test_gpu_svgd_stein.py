"""Every branch of the SVGD Stein update (csrc/svgd.cu) against a float64 reference at its particle, parameter and select
edges: the live sweep in one CTA, as one cooperative launch and as per-particle launches; the canonical update on the
float64 kernels and on the tensor cores; the exact median select in its plain, compacted and fused forms.  Each case
asserts the branch that ran (info "svgd_stein_used") and prints its worst error.

The reference computes d2 from direct differences (in row blocks) and h from np.median of all S^2 entries; phi's
translation-invariant term is formed from the particles centred in float64, so the reference itself carries no
cancellation for particles far from the origin."""
import math

import numpy as np
import pytest

from conftest import rel_err

pytestmark = pytest.mark.gpu

from bayesian_inference_for_nn_b200 import _lib, keras_json  # noqa: E402
from bayesian_inference_for_nn_b200.engine import Engine  # noqa: E402

LIVE_LAUNCHES, LIVE_COOP, LIVE_CTA, CANON_F64, CANON_TENSOR = 0, 1, 2, 3, 4

# nets by parameter count: (in_dim, hidden, classes)
NETS = {17: (2, 3, 2), 62: (3, 10, 2), 63: (4, 3, 12), 64: (1, 2, 20), 65: (6, 7, 2), 252: (2, 50, 2), 257: (2, 64, 1),
        387: (8, 32, 3), 1410: (8, 128, 2), 2212: (64, 32, 4), 12730: (784, 16, 10)}


def net_engine(P, seed=0):
    D, H, Cc = NETS[P]
    js = keras_json.make_sequential_json(D, [H, Cc], ["relu", "softmax" if Cc > 1 else "linear"])
    eng = Engine(keras_json.parse_model_json(js), seed=seed)
    assert eng.P == P
    return eng


def stein_used(eng):
    return int(eng.info("svgd_stein_used"))


# ---- float64 reference ------------------------------------------------------------------------
def ref_d2(X, block=None):
    """squared distances from direct differences, float64, in row blocks of at most ~32 MB"""
    X = np.asarray(X, np.float64)
    S, P = X.shape
    block = block or max(1, (4 << 20) // max(1, S * P))
    d2 = np.empty((S, S))
    for i0 in range(0, S, block):
        diff = X[i0:i0 + block, None, :] - X[None, :, :]
        d2[i0:i0 + block] = np.einsum("ijk,ijk->ij", diff, diff)
    return d2


def ref_h(d2):
    S = d2.shape[0]
    return math.sqrt(0.5 * float(np.median(d2)) / math.log(S + 1))


def ref_phi(X, G, d2=None):
    """canonical phi = (K G + (X rowsum(K) - K X)/h^2)/S with the median bandwidth; (X, h)"""
    X = np.asarray(X, np.float64)
    d2 = ref_d2(X) if d2 is None else d2
    h = ref_h(d2)
    K = np.exp(-d2 / (2.0 * h * h))
    Xc = X - X.mean(0)
    S = X.shape[0]
    return (K @ np.asarray(G, np.float64) + (Xc * K.sum(1)[:, None] - K @ Xc) / (h * h)) / S, h


def particles(rng, S, P, offset=0.0, sigma=0.3):
    """c + sigma N(0,1) with c ~ offset N(0,1) per parameter, rounded to float32 (what the device holds)"""
    c = rng.standard_normal(P) * offset
    return (c + sigma * rng.standard_normal((S, P))).astype(np.float32).astype(np.float64)


# ---- live sweep -------------------------------------------------------------------------------
def live_problem(oracle, P, seed):
    O = oracle
    D, H, Cc = NETS[P]
    rng = np.random.default_rng(seed)
    spec = O.MLPSpec(D, [H, Cc], ["relu", "softmax"])
    X = rng.standard_normal((64, D)).astype(np.float32)
    y = rng.integers(0, Cc, 64).astype(np.int32)
    return spec, X, y, rng


def live_run(X, y, P, p0, lr, idx, cta, fused):
    eng = net_engine(P)
    eng.set_dataset(X, y, _lib.LOSS_SPARSE_CE)
    eng.set_prior([0.0], [1.0], _lib.PRIOR_SCALAR)
    if cta is not None:
        eng.set_option("live_cta", cta)
    if fused is not None:
        eng.set_option("live_fused", fused)
    eng.svgd_init(p0.shape[0], lr, _lib.SVGD_REFERENCE_LIVE, particles0=p0)
    out = []
    for ix in idx:
        loss = eng.svgd_step(ix)
        out.append((loss, eng.svgd_particles(), stein_used(eng)))
    eng.close()
    return out


def live_cases():
    cases = [(6, 17), (6, 252), (6, 1410), (201, 252), (202, 252), (36, 1410), (37, 1410), (1025, 17), ("sm", 17)]
    return [pytest.param(S, P, id="S%s-P%d" % (S, P)) for S, P in cases]


@pytest.mark.parametrize("S,P", live_cases())
def test_live_sweep_variants_match_oracle(oracle, S, P):
    """one step and three steps of every live-sweep variant against oracle.svgd_live_step; cooperative and per-particle
    launches bit-identical (k_live_sweep claims the arithmetic and order of k_live_row / k_live_update), one CTA equal to
    them up to the float64 order of its row sums; AUTO picks one CTA exactly when S*8 + S*P*4 <= 200 KiB"""
    O = oracle
    spec, X, y, rng = live_problem(O, P, seed=P + (S if isinstance(S, int) else 7))
    if S == "sm":
        probe = net_engine(P)
        S = 8 * int(probe.info("sm_count")) + 37               # more particles than co-resident 256-thread blocks
        probe.close()
    lr, n_steps = 1e-3, 3
    p0 = (rng.standard_normal((S, P)) * 0.5).astype(np.float32).astype(np.float64)
    idx = [rng.permutation(64)[:32].astype(np.int32) for _ in range(n_steps)]
    want, am, av = p0.copy(), np.zeros((S, P), np.float32), np.zeros((S, P), np.float32)
    ref = []
    for t, ix in enumerate(idx, 1):
        want, am, av, loss, _ = O.svgd_live_step(spec, want, X[ix], y[ix], O.LOSS_SPARSE_CE, am, av, t, lr)
        ref.append((loss, want.copy()))
    fits = S * 8 + S * P * 4 <= 200 * 1024
    runs = {"auto": live_run(X, y, P, p0, lr, idx, None, None),
            "cooperative": live_run(X, y, P, p0, lr, idx, 0, 1),
            "launches": live_run(X, y, P, p0, lr, idx, 0, 0)}
    expect = {"auto": LIVE_CTA if fits else LIVE_COOP, "cooperative": LIVE_COOP, "launches": LIVE_LAUNCHES}
    for name, run in runs.items():
        worst = 0.0
        for k, ((loss, parts, used), (loss_ref, want_k)) in enumerate(zip(run, ref)):
            assert used == expect[name], (name, used)
            np.testing.assert_allclose(loss, loss_ref, rtol=1e-4)
            err = np.abs(parts - want_k).max()
            worst = max(worst, err / (lr * (k + 1)))
            assert err < 2e-3 * lr * (k + 1) + 1e-6, (name, k, err)
        print("live S=%d P=%d %s: worst |particles - oracle| / (lr * steps) = %.2e" % (S, P, name, worst))
    for (_, a, _), (_, b, _) in zip(runs["cooperative"], runs["launches"]):
        np.testing.assert_array_equal(a, b)
    if fits:
        for (_, a, _), (_, b, _) in zip(runs["auto"], runs["launches"]):
            np.testing.assert_allclose(a, b, rtol=1e-6, atol=1e-9)


# ---- canonical on the float64 kernels ---------------------------------------------------------
F64_S = [2, 3, 7, 8, 9, 15, 16, 17, 127, 128, 129, 255, 260]


@pytest.mark.parametrize("P", [17, 62, 63, 64, 65, 252, 257])
def test_canonical_phi_on_float64_kernels(P):
    """16x16 Gram tiles, 8-row phi groups, 128-column K chunks; 260 >= 256 but not a multiple of 8 stays here"""
    eng = net_engine(P)
    rng = np.random.default_rng(P)
    worst_h = worst_phi = 0.0
    for S in F64_S:
        X = particles(rng, S, P, offset=0.5 if S % 2 else 0.0)
        G = rng.standard_normal((S, P)).astype(np.float32)
        want, h_ref = ref_phi(X, G)
        phi, h = eng.svgd_phi(X, G, _lib.SVGD_CANONICAL_MEDIAN)
        assert stein_used(eng) == CANON_F64, S
        eh, ep = abs(h - h_ref) / h_ref, rel_err(phi, want)
        assert eh < 1e-9 and ep < 1e-5, (S, eh, ep)
        worst_h, worst_phi = max(worst_h, eh), max(worst_phi, ep)
    print("float64 phi P=%d: worst h rel %.2e, phi rel %.2e" % (P, worst_h, worst_phi))
    eng.close()


def canonical_reference_step(oracle, spec, mu, sigma, parts, Xb, yb, am, av, t, lr, n_train):
    """oracle.svgd_canonical_step with phi from ref_phi (direct-difference d2, centred Stein term)"""
    O = oracle
    th = parts.astype(np.float32)
    loss, g = O.mean_loss_and_grad(spec, th, Xb, yb, O.LOSS_SPARSE_CE, np.float32)
    _, gp = O.prior_neg_logp_and_grad(th, mu, sigma, np.float32)
    glogp = -(np.float32(n_train) * g + gp)
    phi, h = ref_phi(th.astype(np.float64), glogp)
    phi32 = phi.astype(np.float32)
    new = np.empty_like(th)
    for i in range(th.shape[0]):
        new[i], am[i], av[i] = O.adam_legacy(th[i], -phi32[i], am[i], av[i], t, lr)
    return new.astype(np.float64), float(loss.mean()), phi, h


def run_training(oracle, S, P, offset, sigma, seed, expect, n_steps=3, lr=1e-3, tol_h=1e-9):
    """three minibatch steps with a per-element prior (mu != 0, sigma varied) against the reference step: the loss to
    1e-4 and svgd_h to tol_h each step; the first step's direction (Adam's first step is lr sign(phi)) exactly where
    |phi_ref| is ten times the path's phi tolerance or more; svgd_h against the reference bandwidth of the particles the
    device stepped from; the bulk of the particles within the bound of
    test_svgd_minibatch_gradients_on_tensor_path and every particle within Adam's own step bound"""
    O = oracle
    D, H, Cc = NETS[P]
    rng = np.random.default_rng(seed)
    spec = O.MLPSpec(D, [H, Cc], ["relu", "softmax"])
    N = 256
    X = rng.standard_normal((N, D)).astype(np.float32)
    y = rng.integers(0, Cc, N).astype(np.int32)
    mu = (0.3 * rng.standard_normal(P)).astype(np.float32)
    sg = rng.uniform(0.5, 2.0, P).astype(np.float32)
    p0 = particles(rng, S, P, offset, sigma)
    idx = [rng.permutation(N)[:64].astype(np.int32) for _ in range(n_steps)]
    eng = net_engine(P)
    eng.set_dataset(X, y, _lib.LOSS_SPARSE_CE)
    eng.set_prior(mu, sg, _lib.PRIOR_PER_ELEMENT)
    eng.svgd_init(S, lr, _lib.SVGD_CANONICAL_MEDIAN, particles0=p0)
    want, am, av = p0.copy(), np.zeros((S, P), np.float32), np.zeros((S, P), np.float32)
    worst = {"loss": 0.0, "h": 0.0}
    dev = p0
    for t, ix in enumerate(idx, 1):
        prev = want.astype(np.float32)
        h_dev = ref_h(ref_d2(dev))              # the bandwidth of the particles the device steps from
        want, loss_ref, phi_ref, h_ref = canonical_reference_step(O, spec, mu, sg, want, X[ix], y[ix], am, av, t, lr, N)
        loss = eng.svgd_step(ix)
        assert stein_used(eng) == expect
        got = eng.svgd_particles()
        el, eh = abs(loss - loss_ref) / abs(loss_ref), abs(eng.info("svgd_h") - h_dev) / h_dev
        if t == 1:
            assert h_dev == h_ref
        assert el < 1e-4 and eh < tol_h, (t, el, eh)
        worst["loss"], worst["h"] = max(worst["loss"], el), max(worst["h"], eh)
        if t == 1:
            sure = np.abs(phi_ref) >= 10 * 1e-4 * np.abs(phi_ref).max()
            moved = np.sign(got.astype(np.float32) - prev)
            bad = int((moved[sure] != np.sign(phi_ref[sure])).sum())
            assert bad == 0, ("first-step directions differ", bad, int(sure.sum()))
        diff = np.abs(got - want)
        assert np.quantile(diff, 0.9995) < 2e-3 * lr * t + 1e-6, (t, np.quantile(diff, 0.9995))
        assert diff.max() <= 2.1 * lr * t
        dev = got
    eng.close()
    return worst


@pytest.mark.parametrize("S", [7, 128, 129, 260])
def test_canonical_training_step_on_float64_kernels(oracle, S):
    w = run_training(oracle, S, 65, 0.5, 0.1, seed=S, expect=CANON_F64)
    print("float64 training S=%d P=65: worst loss rel %.2e, h rel %.2e" % (S, w["loss"], w["h"]))


# ---- exact median select ----------------------------------------------------------------------
def pm_pairs(half):
    """+/- pairs: every parameter sums to 0 over the particles, so centring subtracts exactly 0"""
    return np.concatenate([half, -half])


def set_clusters(S, P, seed):
    rng = np.random.default_rng(seed)
    half = 7.0 + rng.integers(-1, 2, (S // 2, P))                   # |x| <= 8; within-cluster d2 <= 4P, across >= 144P
    X = pm_pairs(half)
    return np.concatenate([X, np.zeros((1, P))]) if S % 2 else X


def set_simplex(S, P):
    """x_i = S e_i: every off-diagonal d2 is 2 S^2; the mean is exactly 1 in the first S parameters, so the centred
    values S - 1 and -1 stay exact in bf16 for S <= 257"""
    X = np.zeros((S, P))
    X[np.arange(S), np.arange(S)] = S
    return X


def set_last_of_group(S, P, seed):
    """small-integer +/- pairs chosen so that the lower middle order statistic is the last of its group of equals and
    the upper middle one is the next integer"""
    for s in range(seed, seed + 400):
        rng = np.random.default_rng(s)
        X = pm_pairs(rng.integers(-3, 4, (S // 2, P)).astype(np.float64))
        d = np.sort(ref_d2(X).ravel())
        n = d.size
        if d[n // 2] == d[n // 2 - 1] + 1:
            return X
    raise AssertionError("no such set in 400 seeds")


def set_line(S):
    """integer points on a line, +/-2^k, k < S/2 <= 20: d2 from 1 to 2^40 (the top byte varies)"""
    v = 2.0 ** np.arange(S // 2)
    X = np.zeros((S, 3))
    X[:, 0] = np.concatenate([v, -v])
    return X


def set_tiny(S):
    """coordinates one float32 ulp apart near 0 (subnormal float32): d2 about 1e-90"""
    ulp = float(np.nextafter(np.float32(0), np.float32(1)))
    v = np.arange(1, S // 2 + 1) * ulp
    X = np.zeros((S, 2))
    X[:, 0] = np.concatenate([v, -v])
    return X


EXACT = [("clusters", 64, 65), ("clusters", 63, 65), ("clusters", 40, 17), ("clusters", 31, 17), ("simplex", 64, 65),
         ("simplex", 63, 65), ("last_of_group", 64, 17), ("last_of_group", 20, 17),
         ("line", 40, 17), ("tiny", 48, 17),
         ("clusters", 256, 65), ("clusters", 264, 387), ("simplex", 256, 387), ("last_of_group", 256, 65)]


def exact_set(kind, S, P):
    X = {"clusters": lambda: set_clusters(S, P, S),
         "simplex": lambda: set_simplex(S, P),
         "last_of_group": lambda: set_last_of_group(S, P, S),
         "line": lambda: np.pad(set_line(S), ((0, 0), (0, P - 3))),
         "tiny": lambda: np.pad(set_tiny(S), ((0, 0), (0, P - 2)))}[kind]()
    assert X.shape == (S, P) and np.all(X.astype(np.float32).astype(np.float64) == X)
    return X


@pytest.mark.parametrize("kind,S,P", [pytest.param(*c, id="%s-S%d-P%d" % c) for c in EXACT])
def test_median_select_is_exact(oracle, kind, S, P):
    """d2 is exact in float64 in any order (and on the tensor path: bf16 holds the values, every partial sum stays below
    2^24), so h from svgd_phi and from a training step must equal the reference's to 1e-14 with every select variant"""
    X = exact_set(kind, S, P)
    d2 = ref_d2(X)
    assert np.median(d2) > 0
    h_ref = ref_h(d2)
    expect = CANON_TENSOR if (S >= 256 and S % 8 == 0 and P >= 64) else CANON_F64
    rng = np.random.default_rng(S)
    G = rng.standard_normal((S, P)).astype(np.float32)
    D, H, Cc = NETS[P]
    Xd = rng.standard_normal((32, D)).astype(np.float32)
    yd = rng.integers(0, Cc, 32).astype(np.int32)
    for compact in (0, 1, 2):
        eng = net_engine(P)
        eng.set_option("select_compact", compact)
        _, h = eng.svgd_phi(X, G, _lib.SVGD_CANONICAL_MEDIAN)
        assert stein_used(eng) == expect
        assert abs(h - h_ref) <= 1e-14 * h_ref, (compact, h, h_ref)
        eng.set_dataset(Xd, yd, _lib.LOSS_SPARSE_CE)
        eng.set_prior([0.0], [1.0], _lib.PRIOR_SCALAR)
        eng.svgd_init(S, 1e-3, _lib.SVGD_CANONICAL_MEDIAN, particles0=X)
        eng.svgd_step(None)
        assert stein_used(eng) == expect
        hs = eng.info("svgd_h")
        assert abs(hs - h_ref) <= 1e-14 * h_ref, (compact, hs, h_ref)
        eng.close()
    print("exact select %s S=%d P=%d: h = %.17g on branch %d" % (kind, S, P, h_ref, expect))


# ---- canonical on the tensor cores ------------------------------------------------------------
# (St, P): a 128-row tile remainder (264, 520, 1032), a partial 256-column tile, mirror blocks that are not multiples of
# 32 (264, 520, 1032), the padded K of P = 65 and the split-K Gram of P = 12 730
TC_SHAPES = [(256, 65), (264, 65), (520, 65), (1032, 65), (256, 387), (264, 387), (384, 387), (512, 387), (520, 387),
             (1032, 387), (256, 2212), (520, 2212), (256, 12730), (264, 12730)]
OFFSETS = [(0.0, 0.3), (1.0, 0.05), (1.0, 0.01), (3.0, 0.01)]


def phi_errors(eng, X, G, ref):
    """(h rel err, phi rel err) of svgd_phi against ref = ref_phi(X, G)"""
    want, h_ref = ref
    phi, h = eng.svgd_phi(X, G, _lib.SVGD_CANONICAL_MEDIAN)
    return abs(h - h_ref) / h_ref, rel_err(phi, want)


@pytest.mark.parametrize("St,P", [pytest.param(*c, id="S%d-P%d" % c) for c in TC_SHAPES])
def test_canonical_phi_on_tensor_cores(St, P):
    """zero-mean and offset particles (c + sigma N, c ~ offset N per parameter), with and without the symmetric Gram:
    h to 1e-5 and phi to 1e-4"""
    eng = net_engine(P)
    rng = np.random.default_rng(St + P)
    offsets = OFFSETS if P <= 2212 else OFFSETS[::3]
    for offset, sigma in offsets:
        X = particles(rng, St, P, offset, sigma)
        G = rng.standard_normal((St, P)).astype(np.float32)
        ref = ref_phi(X, G)
        for sym in (1, 0):
            eng.set_option("tc_gram_sym", sym)
            eh, ep = phi_errors(eng, X, G, ref)
            assert stein_used(eng) == CANON_TENSOR
            print("tensor phi S=%d P=%d offset=%g sigma=%g sym=%d: h rel %.2e, phi rel %.2e" % (St, P, offset, sigma, sym,
                                                                                                  eh, ep))
            assert eh < 1e-5 and ep < 1e-4, (offset, sigma, sym, eh, ep)
    eng.close()


@pytest.mark.parametrize("St,P,expect", [(255, 2212, CANON_F64), (256, 2212, CANON_TENSOR), (260, 2212, CANON_F64),
                                         (264, 2212, CANON_TENSOR), (256, 62, CANON_F64), (256, 65, CANON_TENSOR)])
def test_auto_rule_picks_the_stein_path(St, P, expect):
    eng = net_engine(P)
    rng = np.random.default_rng(St * P)
    X = particles(rng, St, P, 1.0, 0.05)
    G = rng.standard_normal((St, P)).astype(np.float32)
    eh, ep = phi_errors(eng, X, G, ref_phi(X, G))
    assert stein_used(eng) == expect
    tol_h, tol_phi = (1e-9, 1e-5) if expect == CANON_F64 else (1e-5, 1e-4)
    assert eh < tol_h and ep < tol_phi, (eh, ep)
    eng.close()


@pytest.mark.parametrize("offset,sigma", OFFSETS[:2] + OFFSETS[3:])
@pytest.mark.parametrize("St", [256, 264, 520])
def test_canonical_training_step_on_tensor_cores(oracle, St, offset, sigma):
    """C4's one-GPU path (Gram + K Y on the tensor cores, prior folded into the Stein right-hand side, phi finished with
    the Adam step in one pass): P = 387 makes the float4 groups of k_phi_finish_adam straddle particle rows"""
    w = run_training(oracle, St, 387, offset, sigma, seed=St, expect=CANON_TENSOR, tol_h=1e-5)
    print("tensor training S=%d P=387 offset=%g sigma=%g: worst loss rel %.2e, h rel %.2e" % (St, offset, sigma,
                                                                                              w["loss"], w["h"]))
