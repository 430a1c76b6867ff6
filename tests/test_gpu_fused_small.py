"""GPU tests of the small-width fused kernels (fused_small.cuh) against the float64 oracle.

`k_fs_eval` and `k_fs_hmc` are instantiated once per input width D = 1..4, output width C = 1..4 and hidden activation
(relu compiled in, or any activation chosen at run time): 32 kernels each.  They are the default path of every two-layer
net of that size, so every one of them is checked here, at the edges of the kernel's indexing:
- row-pair interleaving with an odd tail row and the pad row of an odd N;
- phase-1 passes of 4 x 256, 2 x 256 and 1 x 256 rows and a partial last pass;
- phase-2 slices (256 / H of them, idle threads when H does not divide 256, one slice for H > 128) and db2;
- the per-unit packing of W1 / b1 / W2;
- cluster spreading over 2 / 4 / 8 CTAs with even-rounded row ranges;
- the Philox momentum tail when P is not a multiple of 4;
- the shared-memory plan and its 200 KiB cut-off.

Every case forces (or, where the choice itself is the subject, asserts) the fused path through `path_used`, so no case
can pass on the generic path.  The gate is the float64 oracle; the generic path only appears in failure messages as a
second opinion.  Common set-up: a per-element prior with non-zero means and varied sigma (an index slip in mu or
inv_var shows), n_train != N (the n_train scaling is checked apart from the 1/N mean), inputs in [-2, 2], labels that
depend on the inputs (the gradients do not cancel to noise), relu nets moved off their kinks, and every gradient compared
block by block (W1, b1, W2, b2), each norm-wise relative.
"""
import numpy as np
import pytest

from conftest import rel_err
from test_gpu_tensor import move_off_relu_kinks

pytestmark = pytest.mark.gpu

from bayesian_inference_for_nn_b200 import _lib, keras_json  # noqa: E402
from bayesian_inference_for_nn_b200.engine import Engine  # noqa: E402

PYB_ERR_UNSUPPORTED = -4
TOL_U, TOL_GRAD, TOL_E, TOL_TRAJ = 1e-5, 1e-4, 1e-4, 1e-3
TOL_CLUSTER = 2e-5          # one CTA per chain against a cluster: the same arithmetic summed in another order
RT_ACTS = ("tanh", "sigmoid", "linear")
MSE_OUTS = ("linear", "sigmoid", "tanh")


def rt_act(D, C):
    """the run-time hidden activation of (D, C): each of tanh, sigmoid and linear appears at every D and every C"""
    return RT_ACTS[(D + C) % 3]


def mse_out(D, C):
    return MSE_OUTS[(D + 2 * C) % 3]


# ---- restatements of the host-side rules of fused_small.cu / fused_small.cuh ---------------------------------------
def fs_smem_bytes(D, C, H, N, ce, P):
    """fused_small.cuh `fs_smem_bytes`: the dynamic shared memory of one CTA, in bytes"""
    n_slices = 256 // H if 256 // H > 0 else 1
    np_ = (N + 1) & ~1
    f = (64 + 4 + np_ * D + N * (1 if ce else C) + np_ * C + 3 * P + H * (D + 1 + C) * n_slices
         + H * ((D + 1 + C + 3) // 4 * 4) + 4 + 2 * ((P + 1) // 2 * 2 + 2) + 2)
    return f * 4 + 16


FS_SMEM_LIMIT = 200 * 1024   # fused_small.cu `fused_small_supported`


def cluster_size(S, N, sm_count):
    """fused_small.cu `fused_small_hmc_iteration`: CTAs per chain (>= 64 rows per CTA, all chains' CTAs on the SMs)"""
    for c in (8, 4, 2):
        if S * c <= sm_count and N // c >= 64:
            return c
    return 1


def n_params(D, C, H):
    return H * (D + 1 + C) + C


def blocks(D, C, H):
    o1 = D * H
    o2 = o1 + H
    o3 = o2 + H * C
    return (("W1", slice(0, o1)), ("b1", slice(o1, o2)), ("W2", slice(o2, o3)), ("b2", slice(o3, o3 + C)))


# ---- problems ------------------------------------------------------------------------------------------------------
class Case:
    """one net, dataset, prior and starting positions; `prob` is the oracle's view of the same problem"""

    def __init__(self, O, D, C, H, N, act, loss, S, seed, out_act=None, n_train=None):
        rng = np.random.default_rng(seed)
        self.D, self.C, self.H, self.N, self.S, self.act = D, C, H, N, S, act
        self.ce = loss == "ce"
        self.out_act = "softmax" if self.ce else (out_act or mse_out(D, C))
        self.kind = _lib.LOSS_SPARSE_CE if self.ce else _lib.LOSS_MSE
        self.spec = O.MLPSpec(D, [H, C], [act, self.out_act])
        self.P = P = self.spec.n_params
        assert P == n_params(D, C, H)
        self.X = rng.uniform(-2.0, 2.0, (N, D)).astype(np.float32)
        A = rng.standard_normal((D, C))
        base = self.X @ A / np.sqrt(D) + 0.3 * rng.standard_normal((N, C))
        if self.ce:
            self.y = np.argmax(base, axis=1).astype(np.int32)
        elif self.out_act == "sigmoid":
            self.y = (0.1 + 0.8 / (1.0 + np.exp(-base))).astype(np.float32)
        elif self.out_act == "tanh":
            self.y = (0.8 * np.tanh(base)).astype(np.float32)
        else:
            self.y = base.astype(np.float32)
        self.mu = rng.uniform(-0.3, 0.3, P).astype(np.float32)
        self.sg = rng.uniform(0.5, 2.0, P).astype(np.float32)
        self.n_train = 3 * N + 7 if n_train is None else n_train
        q = np.empty((S, P), np.float32)
        b = blocks(D, C, H)
        q[:, b[0][1]] = rng.normal(0, 0.5, (S, D * H))
        q[:, b[1][1]] = rng.normal(0, 0.3, (S, H))
        q[:, b[2][1]] = rng.normal(0, 1.0 / np.sqrt(H), (S, H * C))
        q[:, b[3][1]] = rng.normal(0, 0.3, (S, C))
        if act == "relu":
            # each unit's kink inside the data cloud (between its 25 % and 75 % quantiles, give or take): a relu unit that
            # is active on every row, or on none, is a linear unit or no unit at all
            for s in range(S):
                Z = self.X.astype(np.float64) @ q[s, b[0][1]].astype(np.float64).reshape(D, H)
                qt = [np.quantile(Z[:, h], rng.uniform(0.25, 0.75)) for h in range(H)]
                q[s, b[1][1]] = -np.array(qt) + 0.1 * rng.standard_normal(H)
            q = move_off_relu_kinks(q, self.X, D, H, margin=1e-3 if N <= 1100 else 1e-4)
            self.check_relu_mix(q)
        self.q = q
        self.rng = rng
        self.prob = O.Problem(self.spec, self.X, self.y, O.LOSS_SPARSE_CE if self.ce else O.LOSS_MSE, self.mu, self.sg,
                              n_train=self.n_train)

    def check_relu_mix(self, q):
        """the relu units must stay relu units: a real mix of active and inactive (row, unit) pairs in every chain, and
        (with enough rows) most units active on some rows and inactive on others"""
        D, H = self.D, self.H
        for s in range(q.shape[0]):
            Z = self.X.astype(np.float64) @ q[s, :D * H].astype(np.float64).reshape(D, H) + q[s, D * H:D * H + H]
            frac = (Z > 0).mean()
            assert 0.15 < frac < 0.85, ("relu units degenerate", s, frac)
            if self.N >= 31:
                mixed = ((Z > 0).any(0) & (Z <= 0).any(0)).mean()
                assert mixed >= 0.5, ("relu units degenerate", s, mixed)

    def fits(self):
        return fs_smem_bytes(self.D, self.C, self.H, self.N, self.ce, self.P) <= FS_SMEM_LIMIT

    def engine(self, path=_lib.PATH_FUSED_SMALL, cluster=None, seed=0, X=None, y=None):
        js = keras_json.make_sequential_json(self.D, [self.H, self.C], [self.act, self.out_act])
        eng = Engine(keras_json.parse_model_json(js), seed=seed)
        eng.set_option("path", path)
        if cluster is not None:
            eng.set_option("fs_cluster", cluster)
        eng.set_dataset(self.X if X is None else X, self.y if y is None else y, self.kind, n_train=self.n_train)
        eng.set_prior(self.mu, self.sg, _lib.PRIOR_PER_ELEMENT)
        return eng

    def prior_grad32(self, q):
        """the prior part of the device gradient, float32 as the device computes it: (q - mu) * (1 / sigma^2)"""
        iv = np.float32(1.0) / (self.sg * self.sg)
        return (q - self.mu[None]) * iv[None]


def generic_opinion(case, q, got, want):
    """failure-message text: how far the generic path is from the oracle on the same inputs"""
    try:
        eng = case.engine(path=_lib.PATH_GENERIC)
        _, _, g = eng.hmc_eval(q)
        eng.close()
        return "; generic path vs oracle %.2e, fused vs generic %.2e" % (rel_err(g, want), rel_err(got, g))
    except Exception as e:   # the second opinion must never hide the first
        return "; generic path failed: %s" % e


def check_blocks(case, got, want, tol, what, opinion=None):
    """every (chain, parameter block) norm-wise relative: a wrong b2 (C numbers) cannot hide in the norm of W1"""
    for s in range(got.shape[0]):
        for name, sl in blocks(case.D, case.C, case.H):
            e = rel_err(got[s, sl], want[s, sl])
            if not e < tol:
                extra = opinion() if opinion else ""
                pytest.fail("%s: chain %d block %s rel err %.3e >= %.0e%s" % (what, s, name, e, tol, extra))


def check_eval(case, eng, q, O):
    U, loss, g = eng.hmc_eval(q)
    assert int(eng.info("path_used")) == _lib.PATH_FUSED_SMALL
    U64, loss64, g64 = O.potential(case.prob, q, np.float64)
    np.testing.assert_allclose(U, U64, rtol=TOL_U, err_msg="U")
    if case.ce and case.C == 1:
        # a softmax over one class is 1 on every row: loss and data gradient are exactly 0, so the gradient is the prior's
        assert np.all(loss == 0.0), loss
        np.testing.assert_array_equal(g, case.prior_grad32(q))
    else:
        np.testing.assert_allclose(loss, loss64, rtol=TOL_U, err_msg="loss")
    check_blocks(case, g, g64, TOL_GRAD, "gradient", lambda: generic_opinion(case, q, g, g64))
    return U, loss, g


def run_hmc(case, cluster, eps, L, sem, p, u, m=1.0):
    eng = case.engine(cluster=cluster)
    eng.hmc_init(case.S, eps, m, L, sem, q0=case.q)
    eng.hmc_inject(p=p, u=u)
    eng.hmc_run(1, burning=False, sampling=True)
    assert int(eng.info("path_used")) == _lib.PATH_FUSED_SMALL
    used = int(eng.info("fs_cluster_used"))
    q, pp = eng.hmc_state()
    last = eng.hmc_last()
    eng.close()
    return dict(q=q, p=pp, last=last, cluster=used)


def check_hmc_vs_oracle(case, r, want, u):
    last = r["last"]
    for k in ("U0", "K0", "U1", "K1"):
        np.testing.assert_allclose(last[k], want[k], rtol=TOL_E, err_msg=k)
    scale = np.maximum(np.abs(want["U0"]), 1.0)
    assert np.all(np.abs(last["log_alpha"] - want["log_alpha"]) <= 2e-4 * scale), (last["log_alpha"], want["log_alpha"])
    lu = np.log(np.maximum(np.asarray(u, np.float64), 1e-300))
    decisive = np.abs(want["log_alpha"] - lu) > 1e-5 * scale
    np.testing.assert_array_equal(last["accept"][decisive], want["accept"][decisive])
    same = last["accept"] == want["accept"]
    check_blocks(case, r["q"][same], want["q"][same], TOL_TRAJ, "q after the iteration")
    check_blocks(case, r["p"][same], want["pL"][same], TOL_TRAJ, "p_L")


def check_cluster_agrees(case, a, b):
    """a: one CTA per chain, b: the chain spread over a cluster"""
    assert a["cluster"] == 1
    np.testing.assert_array_equal(a["last"]["accept"], b["last"]["accept"])
    for k in ("U0", "K0", "U1", "K1"):
        np.testing.assert_allclose(b["last"][k], a["last"][k], rtol=TOL_CLUSTER, err_msg=k)
    for s in range(case.S):
        assert rel_err(b["q"][s], a["q"][s]) < TOL_CLUSTER, ("q", s, rel_err(b["q"][s], a["q"][s]))
        assert rel_err(b["p"][s], a["p"][s]) < TOL_CLUSTER, ("p", s, rel_err(b["p"][s], a["p"][s]))


@pytest.fixture(scope="session")
def sm_count():
    eng = Engine(keras_json.parse_model_json(keras_json.make_sequential_json(2, [4, 2], ["relu", "softmax"])))
    n = int(eng.info("sm_count"))
    eng.close()
    return n


# ---- 1. all 32 instantiations ---------------------------------------------------------------------------------------
ALL = [pytest.param(D, C, act, loss, id="D%dC%d-%s-%s" % (D, C, act, loss))
       for D in range(1, 5) for C in range(1, 5) for act in ("relu", "rt") for loss in ("ce", "mse")]
N_ALL, H_ALL = 1025, 50      # a 4 x 256 pass, a partial pass and an odd tail row; 5 slices of 50 units, 6 idle threads


def all_case(O, D, C, act, loss, S=3):
    act = "relu" if act == "relu" else rt_act(D, C)
    return Case(O, D, C, H_ALL, N_ALL, act, loss, S, seed=100 * D + 10 * C + (act == "relu") + 2 * (loss == "ce"))


@pytest.mark.parametrize("D,C,act,loss", ALL)
def test_eval_every_instantiation(oracle, D, C, act, loss):
    case = all_case(oracle, D, C, act, loss)
    eng = case.engine()
    check_eval(case, eng, case.q, oracle)
    eng.close()


@pytest.mark.parametrize("D,C,act,loss", ALL)
def test_hmc_iteration_every_instantiation(oracle, sm_count, D, C, act, loss):
    """one iteration with injected momenta and uniforms, on one CTA per chain and on an 8-CTA cluster per chain"""
    O = oracle
    case = all_case(O, D, C, act, loss)
    sem = _lib.HMC_CANONICAL if (act == "rt" and D == C) else _lib.HMC_REFERENCE
    eps, L = 3e-4, 3
    p = case.rng.standard_normal((case.S, case.P)).astype(np.float32)
    u = np.float32([0.2, 0.999, 0.6])
    want = O.hmc_iteration(case.prob, case.q, p, u, eps, 1.0, L, False, sem, np.float64)
    one = run_hmc(case, 0, eps, L, sem, p, u)
    clu = run_hmc(case, 1, eps, L, sem, p, u)
    assert clu["cluster"] == cluster_size(case.S, case.N, sm_count) == 8
    check_hmc_vs_oracle(case, one, want, u)
    check_hmc_vs_oracle(case, clu, want, u)
    check_cluster_agrees(case, one, clu)


# ---- 2. row and unit geometry ---------------------------------------------------------------------------------------
GEO = [(2, 2, "relu", "mse"), (3, 4, "tanh", "ce")]     # MSE with a sigmoid output
N_SWEEP = [1, 2, 31, 255, 256, 257, 511, 512, 513, 767, 1023, 1024, 1025, 1537, 2049, 4097]
H_SWEEP = [1, 3, 50, 64, 128, 129, 200, 256]
GEO_NH = sorted({(n, h) for n in N_SWEEP for h in (50, 129)} | {(n, h) for n in (513, 1024) for h in H_SWEEP})


def geo_case(O, g, N, H, S=2, **kw):
    D, C, act, loss = g
    return Case(O, D, C, H, N, act, loss, S, seed=7 * N + H + D, out_act="sigmoid", **kw)


@pytest.mark.parametrize("N,H", GEO_NH, ids=["N%d-H%d" % nh for nh in GEO_NH])
@pytest.mark.parametrize("g", GEO, ids=["D%dC%d-%s" % g[:3] for g in GEO])
def test_row_and_unit_geometry(oracle, g, N, H):
    case = geo_case(oracle, g, N, H)
    assert case.fits(), "the case must run on the fused path"
    eng = case.engine()
    check_eval(case, eng, case.q, oracle)
    eng.close()


ADD_N = 2049
ADD_SPLITS = [256, 512, 1024, 777]


@pytest.mark.parametrize("H", [50, 129])
@pytest.mark.parametrize("split", ADD_SPLITS)
@pytest.mark.parametrize("g", GEO, ids=["D%dC%d-%s" % g[:3] for g in GEO])
def test_row_additivity(oracle, g, split, H):
    """rows [0, k) and [k, N) in engines of their own add up to the whole dataset: each row's arithmetic is the same
    whatever pass or pair it lands in, so only the summation order differs — far inside the oracle's 1e-4, which lets a
    dropped or doubled row show at any N"""
    case = geo_case(oracle, g, ADD_N, H, n_train=5000)
    parts = [(slice(0, split), split), (slice(split, ADD_N), ADD_N - split), (slice(0, ADD_N), ADD_N)]
    res = []
    for sl, n in parts:
        eng = case.engine(X=case.X[sl].copy(), y=case.y[sl].copy())
        _, loss, g_ = eng.hmc_eval(case.q)
        assert int(eng.info("path_used")) == _lib.PATH_FUSED_SMALL
        eng.close()
        # data part of the gradient (the device adds the float32 prior gradient to n_train * d(mean loss)), as a row sum
        gd = (g_.astype(np.float64) - case.prior_grad32(case.q).astype(np.float64)) * (n / case.n_train)
        res.append((loss.astype(np.float64) * n, gd))
    (la, ga), (lb, gb), (lw, gw) = res
    np.testing.assert_allclose(la + lb, lw, rtol=1e-5)
    check_blocks(case, ga + gb, gw, 1e-5, "row sums of the two parts")


# ---- 3. cluster geometry --------------------------------------------------------------------------------------------
CL_INST = [(2, 3, "relu", "ce"), (4, 3, "sigmoid", "mse")]
CL_S = [(1, 0), (8, 0), (8, 1), (4, 0), (4, 1), (2, 0), (2, 1)]     # (c, d): S = sm_count // c + d; c = 1: S = 1
CL_CASES = [(c, d, n) for c, d in CL_S for n in (127, 129, 255, 257, 511, 513)] + [(1, 0, n) for n in (128, 256, 512)]


def cl_ids():
    return ["S%s-N%d" % ("1" if c == 1 else "sm%d%s" % (c, "+1" if d else ""), n) for c, d, n in CL_CASES]


@pytest.mark.parametrize("c,d,N", CL_CASES, ids=cl_ids())
@pytest.mark.parametrize("inst", CL_INST, ids=["D%dC%d-%s" % i[:3] for i in CL_INST])
def test_cluster_geometry(oracle, sm_count, inst, c, d, N):
    """chain counts on both sides of every switch of the cluster rule and odd row counts around 64 rows per CTA: the
    rounded row ranges, the last rank's odd end and the DSMEM sum against one CTA per chain and the oracle"""
    O = oracle
    S = 1 if c == 1 else sm_count // c + d
    D, C, act, loss = inst
    case = Case(O, D, C, 16, N, act, loss, S, seed=1000 + S + N, out_act="tanh")
    eps, L = 5e-4, 2
    p = case.rng.standard_normal((S, case.P)).astype(np.float32)
    u = case.rng.random(S).astype(np.float32)
    want = O.hmc_iteration(case.prob, case.q, p, u, eps, 1.0, L, False, _lib.HMC_REFERENCE, np.float64)
    one = run_hmc(case, 0, eps, L, _lib.HMC_REFERENCE, p, u)
    clu = run_hmc(case, 1, eps, L, _lib.HMC_REFERENCE, p, u)
    assert clu["cluster"] == cluster_size(S, N, sm_count)
    check_hmc_vs_oracle(case, clu, want, u)
    check_hmc_vs_oracle(case, one, want, u)
    check_cluster_agrees(case, one, clu)


def test_cluster_rule_switches_are_covered(sm_count):
    """the chain counts above reach every cluster size on both sides of each switch"""
    seen = {cluster_size(1 if c == 1 else sm_count // c + d, 513, sm_count) for c, d in CL_S}
    assert seen == {1, 2, 4, 8}
    for c in (8, 4, 2):
        S = sm_count // c
        assert cluster_size(S, 1 << 20, sm_count) == c and cluster_size(S + 1, 1 << 20, sm_count) < c
        assert cluster_size(1, 64 * c, sm_count) == c and cluster_size(1, 64 * c - 1, sm_count) == c // 2


# ---- 4. Philox momentum tail ----------------------------------------------------------------------------------------
RNG_INST = [(2, 2, 50, "relu", "ce"), (2, 2, 51, "relu", "ce"), (1, 4, 49, "tanh", "ce"), (3, 1, 50, "sigmoid", "mse")]


def test_rng_shapes_cover_every_tail():
    assert sorted(n_params(D, C, H) % 4 for D, C, H, _, _ in RNG_INST) == [0, 1, 2, 3]


@pytest.mark.parametrize("cluster", [0, 1], ids=["one_cta", "cluster"])
@pytest.mark.parametrize("sem", [_lib.HMC_REFERENCE, _lib.HMC_CANONICAL], ids=["reference", "canonical"])
@pytest.mark.parametrize("inst", RNG_INST, ids=["P%d" % (n_params(i[0], i[1], i[2]) % 4) for i in RNG_INST])
def test_device_momenta_and_uniforms(oracle, sm_count, inst, sem, cluster):
    """iteration 0 with step size 0 leaves the Philox momenta untouched: they must equal the restatement, the tail
    block of P included; iteration 1 (step sizes spread over the chains so that some proposals are rejected) must take
    its decisions with the restated uniforms"""
    O = oracle
    D, C, H, act, loss = inst
    S, N, m, off, seed = 6, 600, 0.5, 5, 0x1234ABCD5678
    case = Case(O, D, C, H, N, act, loss, S, seed=H + C)
    eng = case.engine(cluster=cluster, seed=seed)
    eng.hmc_init(S, 0.0, m, 1, sem, q0=case.q, chain_offset=off)
    eng.hmc_run(1, burning=True, sampling=False)
    assert int(eng.info("path_used")) == _lib.PATH_FUSED_SMALL
    assert int(eng.info("fs_cluster_used")) == (cluster_size(S, N, sm_count) if cluster else 1)
    q1, p1 = eng.hmc_state()
    np.testing.assert_array_equal(q1, case.q)
    chains = np.arange(off, off + S)
    stdv = np.float32(m) if sem == _lib.HMC_REFERENCE else np.float32(np.sqrt(m))
    want_p = O.philox_normals(seed, chains, 0, O.STREAM_MOMENTUM, case.P) * stdv
    np.testing.assert_allclose(p1, want_p, rtol=2e-5, atol=2e-6)
    steps = np.geomspace(1e-4, 3e-2, S)
    eng.hmc_set_step_sizes(steps)
    eng.hmc_run(1, burning=False, sampling=True)
    last = eng.hmc_last()
    eng.close()
    u = O.philox_uniforms(seed, chains, 1)
    la = last["log_alpha"].astype(np.float64)
    lu = np.log(np.maximum(u.astype(np.float64), 1e-300))
    clear = np.abs(la - lu) > 1e-5 * np.maximum(np.abs(last["U0"]), 1.0)
    with np.errstate(over="ignore"):          # exp of a large log alpha is +inf: always accepted, as on the device
        alpha = np.exp(last["log_alpha"])
    np.testing.assert_array_equal(last["accept"][clear], (u < alpha)[clear])
    p_it1 = O.philox_normals(seed, chains, 1, O.STREAM_MOMENTUM, case.P) * stdv
    want = {k: [] for k in ("U0", "K0", "U1", "K1", "log_alpha", "accept")}
    for s in range(S):
        w = O.hmc_iteration(case.prob, case.q[s:s + 1], p_it1[s:s + 1], u[s:s + 1], float(steps[s]), m, 1, False, sem,
                            np.float64)
        for k in want:
            want[k].append(w[k][0])
    want = {k: np.array(v) for k, v in want.items()}
    assert want["accept"].any() and not want["accept"].all(), "the case must contain accepted AND rejected proposals"
    for k in ("U0", "K0", "U1", "K1"):
        np.testing.assert_allclose(last[k], want[k], rtol=TOL_E, err_msg=k)
    decisive = np.abs(want["log_alpha"] - lu) > 1e-5 * np.maximum(np.abs(want["U0"]), 1.0)
    np.testing.assert_array_equal(last["accept"][decisive], want["accept"][decisive])


# ---- 5. per-chain step sizes off moons ------------------------------------------------------------------------------
@pytest.mark.parametrize("cluster", [0, 1], ids=["one_cta", "cluster"])
def test_per_chain_step_sizes_equal_single_chain_runs(oracle, cluster):
    """(4, 3, tanh): three chains with three step sizes move bit for bit as three one-chain runs with their chain ids"""
    case = Case(oracle, 4, 3, 50, 1025, "tanh", "ce", 3, seed=45)
    steps = np.array([1e-3, 4e-3, 1.1e-2])
    seed, L, n_it = 99, 3, 2

    def run(S, off, q0, st):
        eng = case.engine(cluster=cluster, seed=seed)
        eng.hmc_init(S, 1e-3, 1.0, L, _lib.HMC_REFERENCE, q0=q0, chain_offset=off)
        eng.hmc_set_step_sizes(st)
        eng.hmc_run(n_it, burning=False, sampling=True)
        assert int(eng.info("path_used")) == _lib.PATH_FUSED_SMALL
        used = int(eng.info("fs_cluster_used"))
        out = eng.hmc_state() + (eng.hmc_last(), used)
        eng.close()
        return out

    qa, pa, la, ca = run(3, 0, case.q, steps)
    assert ca == (8 if cluster else 1)
    for s in range(3):
        qs, ps, ls, cs = run(1, s, case.q[s:s + 1], steps[s:s + 1])
        assert cs == ca
        np.testing.assert_array_equal(qs[0], qa[s])
        np.testing.assert_array_equal(ps[0], pa[s])
        for k in ("U0", "K0", "U1", "K1", "log_alpha", "accept", "loss"):
            np.testing.assert_array_equal(ls[k][0], la[k][s], err_msg=k)


# ---- 6. minibatch route ---------------------------------------------------------------------------------------------
SG_INST = [(1, 3, "tanh", "ce"), (3, 1, "relu", "mse"), (4, 4, "sigmoid", "mse")]
SG_N = 600


@pytest.mark.parametrize("B", [1, 127, 257, SG_N - 1])
@pytest.mark.parametrize("inst", SG_INST, ids=["D%dC%d-%s" % i[:3] for i in SG_INST])
def test_sgld_minibatches_on_the_fused_path(oracle, inst, B):
    """SGLD steps with injected noise: the minibatch gradient runs the fused kernel on B gathered rows, fewer than the
    shared-memory plan was sized for"""
    O = oracle
    D, C, act, loss = inst
    S, steps = 3, 3
    case = Case(O, D, C, 50, SG_N, act, loss, S, seed=B + D)
    eng = case.engine()
    eng.sg_init(S, _lib.SG_SGLD, theta0=case.q)
    st = O.sg_init_state(case.q)
    for n in range(steps):
        idx = case.rng.permutation(SG_N)[:B].astype(np.int32)
        z = case.rng.standard_normal((S, case.P)).astype(np.float32)
        lr = 1e-3 / (n + 1)
        want_loss = O.sg_step(case.spec, st, case.X[idx], case.y[idx], case.prob.loss_kind, O.SG_SGLD, lr, z=z)
        got_loss, _ = eng.sg_step(lr, idx, noise=z)
        assert int(eng.info("path_used")) == _lib.PATH_FUSED_SMALL
        np.testing.assert_allclose(got_loss, want_loss, rtol=1e-4)
    got = eng.sg_state()
    eng.close()
    assert got["n"] == steps
    check_blocks(case, got["theta"], st.theta, 2e-5, "theta after %d SGLD steps" % steps)


# ---- 7. limits of fused_small_supported -----------------------------------------------------------------------------
UNSUPPORTED = {"D5": (5, [16, 2], ["relu", "softmax"], None), "C5": (2, [16, 5], ["relu", "softmax"], None),
               "H257": (2, [257, 2], ["relu", "softmax"], None),
               "no_bias": (2, [16, 2], ["relu", "softmax"], [True, False]),
               "three_layers": (2, [16, 8, 2], ["relu", "tanh", "softmax"], None)}


@pytest.mark.parametrize("name", sorted(UNSUPPORTED))
def test_unsupported_shapes_resolve_to_the_generic_path(oracle, name):
    D, units, acts, bias = UNSUPPORTED[name]
    rng = np.random.default_rng(3)
    N = 100
    X = rng.uniform(-2, 2, (N, D)).astype(np.float32)
    y = rng.integers(0, units[-1], N).astype(np.int32)
    spec = oracle.MLPSpec(D, units, acts, bias or [])
    q = (rng.standard_normal((2, spec.n_params)) * 0.3).astype(np.float32)

    def make(path):
        eng = Engine(keras_json.parse_model_json(keras_json.make_sequential_json(D, units, acts, bias)))
        eng.set_option("path", path)
        eng.set_dataset(X, y, _lib.LOSS_SPARSE_CE)
        eng.set_prior([0.1], [0.7], _lib.PRIOR_SCALAR)
        return eng

    eng = make(_lib.PATH_AUTO)
    eng.hmc_eval(q)
    assert int(eng.info("path_used")) == _lib.PATH_GENERIC
    eng.hmc_init(2, 1e-3, 1.0, 2, q0=q)
    eng.hmc_run(1)
    assert int(eng.info("path_used")) == _lib.PATH_GENERIC
    eng.close()
    eng = make(_lib.PATH_FUSED_SMALL)
    with pytest.raises(_lib.PyesianB200Error) as e:
        eng.hmc_eval(q)
    assert e.value.code == PYB_ERR_UNSUPPORTED
    eng.hmc_init(2, 1e-3, 1.0, 2, q0=q)
    with pytest.raises(_lib.PyesianB200Error) as e:
        eng.hmc_run(1)
    assert e.value.code == PYB_ERR_UNSUPPORTED
    eng.close()


LIMIT_INST = {"D4C4-mse": (4, 4, "relu", "mse"), "D1C1-ce": (1, 1, "tanh", "ce")}
LIMIT_H = 50


def largest_fitting_n(D, C, ce):
    P = n_params(D, C, LIMIT_H)
    n = 1
    while fs_smem_bytes(D, C, LIMIT_H, n + 1, ce, P) <= FS_SMEM_LIMIT:
        n += 1
    return n


def test_shared_memory_plan_restatement():
    """the restated plan grows with N, and the limit N of each case leaves no room for one more row"""
    for D, C, _, loss in LIMIT_INST.values():
        ce = loss == "ce"
        n = largest_fitting_n(D, C, ce)
        P = n_params(D, C, LIMIT_H)
        assert fs_smem_bytes(D, C, LIMIT_H, n, ce, P) <= FS_SMEM_LIMIT < fs_smem_bytes(D, C, LIMIT_H, n + 1, ce, P)
        assert n // 8 >= 64        # one chain at the limit is an 8-CTA cluster of ~200 KiB CTAs
    assert largest_fitting_n(1, 1, True) > largest_fitting_n(4, 4, False)


@pytest.mark.parametrize("name", sorted(LIMIT_INST))
def test_shared_memory_limit(oracle, sm_count, name):
    """at the largest N whose plan fits 200 KiB the fused path runs (eval, and HMC with one chain on an 8-CTA cluster
    of ~200 KiB CTAs) and matches the oracle; one row more and AUTO picks the generic path, forcing the fused path fails"""
    O = oracle
    D, C, act, loss = LIMIT_INST[name]
    n_max = largest_fitting_n(D, C, loss == "ce")
    case = Case(O, D, C, LIMIT_H, n_max, act, loss, 1, seed=n_max)
    assert case.fits()
    eng = case.engine()
    check_eval(case, eng, case.q, O)
    eng.close()
    eps, L = 2e-3, 2
    p = case.rng.standard_normal((1, case.P)).astype(np.float32)
    u = np.float32([0.5])
    want = O.hmc_iteration(case.prob, case.q, p, u, eps, 1.0, L, False, _lib.HMC_REFERENCE, np.float64)
    r = run_hmc(case, 1, eps, L, _lib.HMC_REFERENCE, p, u)
    assert r["cluster"] == cluster_size(1, n_max, sm_count) == 8
    check_hmc_vs_oracle(case, r, want, u)
    # one row more
    X = np.concatenate([case.X, case.X[:1]])
    y = np.concatenate([case.y, case.y[:1]])
    eng = case.engine(path=_lib.PATH_AUTO, X=X, y=y)
    eng.hmc_eval(case.q)
    assert int(eng.info("path_used")) == _lib.PATH_GENERIC
    eng.close()
    eng = case.engine(X=X, y=y)
    with pytest.raises(_lib.PyesianB200Error) as e:
        eng.hmc_eval(case.q)
    assert e.value.code == PYB_ERR_UNSUPPORTED
    eng.close()
