"""Multi-GPU tests (need >= 2 B200s on the box; skipped otherwise): SVGD particles sharded over two
ranks with NCCL (particle/gradient all-gather, all-reduced median histograms, sequential live sweep)
must reproduce the single-GPU golden run."""
import os

import numpy as np
import pytest

from conftest import load_golden

pytestmark = pytest.mark.gpu


def _worker(rank, world, uid, sem, out):
    import numpy as np
    from bayesian_inference_for_nn_b200 import _lib, keras_json
    from bayesian_inference_for_nn_b200.engine import Engine
    from conftest import load_golden as lg
    g = lg("svgd_mini")
    S = g["particles0"].shape[0]
    Sl = S // world
    eng = Engine(keras_json.parse_model_json(keras_json.make_sequential_json(2, [50, 2], ["relu", "softmax"])), device=rank)
    eng.set_dataset(g["X"], g["y"], _lib.LOSS_SPARSE_CE)
    eng.set_prior([0.0], [1.0], _lib.PRIOR_SCALAR)
    eng.svgd_set_comm(rank, world, uid)
    eng.svgd_init(Sl, float(g["lr"]), sem, particles0=g["particles0"][rank * Sl:(rank + 1) * Sl], offset=rank * Sl)
    losses = [eng.svgd_step(ix) for ix in g["idx"]]
    out.put((rank, eng.svgd_particles(), losses))
    eng.close()


@pytest.mark.parametrize("sem,key", [(1, "can"), (0, "live")])
def test_svgd_sharded_over_two_gpus_matches_golden(sem, key):
    from bayesian_inference_for_nn_b200 import _lib
    if _lib.device_count() < 2:
        pytest.skip("needs 2 GPUs")
    import multiprocessing as mp
    ctx = mp.get_context("spawn")
    uid = _lib.nccl_unique_id()
    q = ctx.Queue()
    procs = [ctx.Process(target=_worker, args=(r, 2, uid, sem, q)) for r in range(2)]
    for p in procs:
        p.start()
    res = sorted([q.get(timeout=300) for _ in range(2)], key=lambda t: t[0])
    for p in procs:
        p.join(timeout=60)
        assert p.exitcode == 0
    g = load_golden("svgd_mini")
    parts = np.concatenate([r[1] for r in res])
    np.testing.assert_allclose(res[0][2], g[key + "_losses"], rtol=1e-4)       # all-reduced mean loss
    np.testing.assert_allclose(res[1][2], g[key + "_losses"], rtol=1e-4)
    lr, n = float(g["lr"]), len(g["idx"])
    assert np.abs(parts - g[key + "_particles"]).max() < 2e-3 * lr * n + 1e-6


def _predict_worker(rank, world, uid, out):
    import numpy as np
    from bayesian_inference_for_nn_b200 import keras_json
    from bayesian_inference_for_nn_b200.engine import Engine
    from bayesian_inference_for_nn_b200.sharding import shard_weight_samples
    rng = np.random.default_rng(3)
    js = keras_json.make_sequential_json(784, [128, 10], ["relu", "softmax"])
    eng = Engine(keras_json.parse_model_json(js), device=rank)
    W = rng.normal(0, 0.05, (9, eng.P)).astype(np.float32)
    freq = rng.integers(1, 4, 9).astype(np.float32)
    x = rng.uniform(0, 1, (512, 784)).astype(np.float32)
    y = rng.integers(0, 10, 512)
    eng.set_comm(rank, world, uid)
    Wl, fl = shard_weight_samples(W, freq, rank, world)           # 5 + 4 weight samples
    mean, var, allo = eng.predict(Wl, x, weights=fl, want_all=True)
    tot, al, ep, _ = eng.predict_uncertainty(Wl, x, y, weights=fl)
    out.put((rank, mean, var, allo.shape[0], tot))
    eng.close()


def test_predictive_sharded_over_two_gpus_matches_one_gpu():
    """SURVEY 8e row 3: weight samples split over ranks, moment sums all-reduced over NCCL"""
    from bayesian_inference_for_nn_b200 import _lib, keras_json
    from bayesian_inference_for_nn_b200.engine import Engine
    if _lib.device_count() < 2:
        pytest.skip("needs 2 GPUs")
    import multiprocessing as mp
    ctx = mp.get_context("spawn")
    uid = _lib.nccl_unique_id()
    q = ctx.Queue()
    procs = [ctx.Process(target=_predict_worker, args=(r, 2, uid, q)) for r in range(2)]
    for p in procs:
        p.start()
    res = sorted([q.get(timeout=300) for _ in range(2)], key=lambda t: t[0])
    for p in procs:
        p.join(timeout=60)
        assert p.exitcode == 0
    rng = np.random.default_rng(3)
    js = keras_json.make_sequential_json(784, [128, 10], ["relu", "softmax"])
    eng = Engine(keras_json.parse_model_json(js))
    W = rng.normal(0, 0.05, (9, eng.P)).astype(np.float32)
    freq = rng.integers(1, 4, 9).astype(np.float32)
    x = rng.uniform(0, 1, (512, 784)).astype(np.float32)
    y = rng.integers(0, 10, 512)
    mean, var, _ = eng.predict(W, x, weights=freq)
    tot, _, _, _ = eng.predict_uncertainty(W, x, y, weights=freq)
    assert [r[3] for r in res] == [5, 4]                      # per-draw outputs stay local
    for r in res:                                             # both ranks hold the full answer
        np.testing.assert_allclose(r[1], mean, rtol=1e-6, atol=1e-7)
        np.testing.assert_allclose(r[2], var, rtol=1e-4, atol=1e-9)
        np.testing.assert_allclose(r[4], tot, rtol=1e-5, atol=1e-7)


def _wide_setup(offset=0.0):
    rng = np.random.default_rng(11)
    D, H, C, N, B, S, steps = 784, 128, 10, 2048, 512, 512, 3
    X = rng.random((N, D)).astype(np.float32)
    y = rng.integers(0, C, N).astype(np.int32)
    P = D * H + H + H * C + C
    parts = rng.normal(0, 0.05, (S, P))
    if offset:                  # particles close together around a common point far from the origin
        parts += offset * np.random.default_rng(12).standard_normal(P)
    idx = [rng.permutation(N)[:B].astype(np.int32) for _ in range(steps)]
    return D, H, C, X, y, parts, idx


def _wide_run(rank, world, uid, pshard, offset=0.0):
    from bayesian_inference_for_nn_b200 import _lib, keras_json
    from bayesian_inference_for_nn_b200.engine import Engine
    D, H, C, X, y, parts, idx = _wide_setup(offset)
    S = parts.shape[0]
    Sl = S // world
    eng = Engine(keras_json.parse_model_json(keras_json.make_sequential_json(D, [H, C], ["relu", "softmax"])), device=rank)
    eng.set_dataset(X, y, _lib.LOSS_SPARSE_CE)
    eng.set_prior([0.0], [1.0], _lib.PRIOR_SCALAR)
    if world > 1:
        eng.svgd_set_comm(rank, world, uid)
        eng.set_option("svgd_pshard", 1 if pshard else 0)
        eng.set_option("svgd_p2p", 1 if pshard == 1 else 0)
    eng.svgd_init(Sl, 1e-3, _lib.SVGD_CANONICAL_MEDIAN, particles0=parts[rank * Sl:(rank + 1) * Sl], offset=rank * Sl)
    losses, hs = [], []
    for ix in idx:
        losses.append(eng.svgd_step(ix))
        hs.append(eng.info("svgd_h"))
    assert int(eng.info("path_used")) == _lib.PATH_TENSOR
    res = (rank, eng.svgd_particles(), losses, hs, int(eng.info("svgd_p2p")) if world > 1 else 0)
    eng.close()
    return res


def _wide_worker(rank, world, uid, pshard, offset, out):
    out.put(_wide_run(rank, world, uid, pshard, offset))


@pytest.mark.parametrize("pshard,offset", [pytest.param(1, 0.0, id="1"), pytest.param(2, 0.0, id="2"), pytest.param(0, 0.0, id="0"),
                                           pytest.param(1, 1.0, id="1-offset"), pytest.param(0, 1.0, id="0-offset")])
def test_svgd_sharded_on_the_tensor_path_matches_one_gpu(pshard, offset):
    """C4's shape in small (784-128-10, 512 particles, minibatch 512, canonical median-heuristic update): the sharded step
    on the tensor path — pshard = 1: Stein phase sharded over the parameters, the gradient rows and the updated particle
    blocks exchanged by peer-memory stores of the library's own kernels (CUDA IPC between the rank processes), all-reduced
    Gram matrix and radix-select histograms; 2: the same with NCCL send / recv exchanges; 0: row-sharded with particle and
    gradient all-gathers — against the SAME step on one GPU: losses, bandwidth h and particles after three steps.
    offset = 1: the particles sit around a common point far from the origin (each rank centres its own parameter slice
    with pshard = 1, every rank the same gathered particles with pshard = 0)."""
    from bayesian_inference_for_nn_b200 import _lib
    if _lib.device_count() < 2:
        pytest.skip("needs 2 GPUs")
    import multiprocessing as mp
    _, one_parts, one_losses, one_h, _ = _wide_run(0, 1, None, 0, offset)
    ctx = mp.get_context("spawn")
    uid = _lib.nccl_unique_id()
    q = ctx.Queue()
    procs = [ctx.Process(target=_wide_worker, args=(r, 2, uid, pshard, offset, q)) for r in range(2)]
    for p in procs:
        p.start()
    res = sorted([q.get(timeout=300) for _ in range(2)], key=lambda t: t[0])
    for p in procs:
        p.join(timeout=60)
        assert p.exitcode == 0
    parts = np.concatenate([r[1] for r in res])
    for r in res:
        np.testing.assert_allclose(r[2], one_losses, rtol=1e-5)
        np.testing.assert_allclose(r[3], one_h, rtol=1e-6)
    lr, n = 1e-3, len(one_losses)
    diff = np.abs(parts - one_parts)
    # Adam's first steps are lr * phi / (|phi| + 1e-7): sign-like where |phi| ~ 1e-7, so bound the bulk tightly and the
    # worst case by Adam's own bound (the same criterion as test_svgd_minibatch_gradients_on_tensor_path)
    print("sharded (pshard=%d, peer-memory exchange %s) vs one GPU: particle diff quantile(0.9995) %.2e, max %.2e" %
          (pshard, [r[4] for r in res], np.quantile(diff, 0.9995), diff.max()))
    if pshard != 1:
        assert [r[4] for r in res] == [0, 0]
    assert np.quantile(diff, 0.9995) < 2e-3 * lr * n + 1e-6
    assert diff.max() <= 2.1 * lr * n
