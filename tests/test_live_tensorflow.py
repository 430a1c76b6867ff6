"""Optional LIVE cross-check against the real reference (SURVEY 8c, last bullet).

Everything else in tests/ that says "reference-executed" ran the reference's own Python files on a torch-backed
TensorFlow stand-in (tests/golden/tf_shim.py), because tensorflow==2.15 / tensorflow_probability==0.23
(requirements.txt:9,12; HMC.py:6-7) are not dependencies of this project.  Where they are installed and the environment
variable PYESIAN_REFERENCE names a checkout of the reference, these tests run the REAL `Pyesian.optimizers.HMC`
on TensorFlow and hold the device to it with the momenta and uniforms of the reference run injected.  Otherwise they
skip — they never fail for a missing dependency."""
import os
import random
import sys

import numpy as np
import pytest

pytestmark = pytest.mark.gpu

REF = os.environ.get("PYESIAN_REFERENCE", "")


def _real_tensorflow():
    try:
        import tensorflow as tf
        import tensorflow_probability  # noqa: F401
    except Exception as e:  # noqa: BLE001
        pytest.skip("real TensorFlow / TFP not importable here (%s): the stand-in goldens remain the pin" % type(e).__name__)
    if getattr(tf, "__pyb_stand_in__", False) or not hasattr(tf, "raw_ops"):
        pytest.skip("the importable `tensorflow` is the test stand-in, not TensorFlow")
    if not REF or not os.path.isdir(os.path.join(REF, "Pyesian")):
        pytest.skip("no reference checkout: set PYESIAN_REFERENCE to one")
    return tf


def test_hmc_step_against_the_real_reference_on_tensorflow():
    tf = _real_tensorflow()
    sys.path.insert(0, REF)
    for k in [k for k in sys.modules if k == "Pyesian" or k.startswith("Pyesian.")]:
        del sys.modules[k]                      # the repo's import alias of the same name must not shadow the reference
    from Pyesian.datasets import Dataset as RefDataset
    from Pyesian.distributions import GaussianPrior as RefPrior
    from Pyesian.optimizers import HMC as RefHMC
    from Pyesian.optimizers.hyperparameters import HyperParameters as RefHP
    from bayesian_inference_for_nn_b200 import _lib, keras_json
    from bayesian_inference_for_nn_b200.engine import Engine

    rng = np.random.default_rng(0)
    N, D, Hh, C, L, eps, m = 256, 4, 8, 3, 5, 0.01, 0.7
    X = rng.normal(size=(N, D)).astype(np.float32)
    y = rng.integers(0, C, N)
    model = tf.keras.Sequential([tf.keras.layers.Dense(Hh, activation="relu", input_shape=(D,)),
                                 tf.keras.layers.Dense(C, activation="softmax")])
    ds = RefDataset(tf.data.Dataset.from_tensor_slices((X, y)), tf.keras.losses.SparseCategoricalCrossentropy(),
                    "Classification", train_proportion=1.0, test_proportion=0.0, valid_proportion=0.0)
    ref = RefHMC()
    ref.compile(RefHP(epsilon=eps, m=m, L=L), model.to_json(), ds, verbose=False, prior=RefPrior(0.0, 1.0))
    # record what the reference draws: momenta through tf.random.normal, the uniform through random.random
    drawn, real_normal = [], tf.random.normal
    tf.random.normal = lambda *a, **k: (lambda t: (drawn.append(t.numpy().ravel()), t)[1])(real_normal(*a, **k))
    random.seed(3)
    u = random.Random(3).random()
    q_before = np.concatenate([v.numpy().ravel() for v in ref._base_model.trainable_variables])
    ref.step(sampling=True, burning=False)
    tf.random.normal = real_normal
    q_after = np.concatenate([v.numpy().ravel() for v in ref._base_model.trainable_variables])
    p = np.concatenate(drawn).astype(np.float32)
    x_train, y_train = next(iter(ds.train_data.batch(N)))
    eng = Engine(keras_json.parse_model_json(model.to_json()))
    eng.set_dataset(np.asarray(x_train, np.float32), np.asarray(y_train, np.int32), _lib.LOSS_SPARSE_CE)
    eng.set_prior([0.0], [1.0], _lib.PRIOR_SCALAR)
    eng.hmc_init(1, eps, m, L, _lib.HMC_REFERENCE, q0=q_before[None].astype(np.float32))
    eng.hmc_inject(p=p[None], u=np.float32([u]))
    eng.hmc_run(1, burning=False, sampling=True)
    q_dev, _ = eng.hmc_state()
    np.testing.assert_allclose(q_dev[0], q_after, rtol=1e-3, atol=1e-5)
