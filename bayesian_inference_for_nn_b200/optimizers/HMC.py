"""HMC — Hamiltonian Monte Carlo, S chains at once on one B200.

Drop-in for Pyesian/optimizers/HMC.py:13-187.  Same surface: hyper-parameters ``m, L, epsilon``
(:53-55), ``compile(..., prior=GaussianPrior)`` (KeyError without ``prior``, :60), ``step(
save_document_path, sampling, burning)`` (:74), ``train(n)`` = 10 always-accept burn-in iterations +
n sampling iterations with the ``loss`` / ``accept_rate`` progress line (:106-126), ``result()`` ->
``BayesianModel`` holding one ``Sampled`` over all layers (:176-187).  Quirks kept: the
``nb_burn_epoch``/``nb_burn_epochs`` key mismatch (:61-62), save/loss-file arguments of ``train``
ignored (:106-126), chains start at the prior mean (:69-72).

Underneath, every iteration is a handful of kernel launches on the handle's stream with no host
sync (pyb_hmc_run); the reference's single chain becomes ``n_chains`` (optional hyper-parameter,
default 1) independent chains whose accepted states are pooled into the returned ``Sampled``.
Optional knobs (all absent => reference behaviour): ``n_chains``, ``seed`` (absent: a fresh 64-bit seed per
optimizer, kept in ``self.seed``), ``semantics`` ("reference" | "canonical"), ``device``, ``path`` ("auto" | "generic" |
"fused" | "tensor"), ``chain_offset`` (global id of the first local chain when chains are sharded over processes), and
``devices=[0, 1, ...]`` / ``n_devices=k``: the chains are sharded over several GPUs of the box inside this process
(multi.py) and ``result()`` pools them in global chain order — bit-identical to the one-device run;
``keep_samples`` (default True): False keeps no sample at all (``result()`` raises) for runs that only need the
streamed predictive below, whose memory then stays flat however long the chains run.

Step-size adaptation: ``adapt_iterations`` (default 0: off) and ``target_accept`` (default 0.8).  With
``adapt_iterations = n > 0``, ``train(k)`` runs the reference's burn-in unchanged, then n iterations (progress line
"HMC - Adapting") in which every chain tunes its own step size by dual averaging (Hoffman & Gelman 2014, Algorithm 5;
Stan's constants) towards an average acceptance probability of ``target_accept``, starting from ``epsilon``; then the
step sizes are frozen and the k sampling iterations run as before.  Adaptation draws nothing into the samples, and
``accept_rate`` still covers the sampling iterations only.  ``step_sizes`` gives every chain's step size ([n_chains]
float64, global chain order; ``epsilon`` everywhere without adaptation).  Chains adapt independently, so a run sharded
over devices gives the one-device step sizes.

Parallel tempering: ``inverse_temperatures`` (default absent: off), a list of R inverse temperatures starting at 1.0 and
strictly decreasing to > 0.  Every one of the ``n_chains`` posterior chains then runs as a replica group of R chains
(``n_chains R`` engine chains; q0 rows are replicated over a group's rungs), rung r sampling prior x likelihood^beta_r,
and after every iteration neighbouring rungs propose to swap their states (non-reversible even-odd replica exchange,
Syed et al. 2022), so a cold chain stuck in one mode of the posterior gets states from the hotter rungs, which move
between modes easily.  Only the beta = 1 rung is a posterior sample: ``result()``, ``predictive()`` and
``classification_uncertainty()`` see its draws only, and ``accept_rate`` and the progress line report it.
``tempering_rates()`` gives the per-rung HMC acceptance and per-pair swap acceptance of the sampling phase, the numbers
to tune a ladder by (a swap rate near 0 between two rungs asks for a rung between them); ``step_sizes`` is then
[n_chains, R].  The ladder is checked before any device work (``tempering.validate_ladder``).

Streamed predictive: ``track_predictive(x, y=None)`` after ``compile`` and before ``train`` / the first sampling
``step`` makes every recorded draw go through the forward pass on x while the chains run.  ``predictive()`` then gives
what ``result().predict(x, 0, mode="exact")`` and ``last_variance`` give, plus the R-hat of every output across the
chains; ``classification_uncertainty`` what ``result().classification_uncertainty(x, y, 0, mode="exact")`` gives.

Streamed parameter diagnostics: ``track_parameters(n_iterations=None, batch_size=None)`` after ``compile`` folds every
parameter of every recorded draw into sums on the device, so it works with ``keep_samples=False`` too.
``parameter_summary()`` then gives, per parameter in the flat weight order, the posterior mean and sd (what the
frequency-weighted ``result()`` samples give), the split R-hat over half-chains (Gelman et al., BDA3 11.4; it flags a
chain that drifts, which the classic R-hat misses), the batch-means effective sample size (Flegal & Jones 2010) and the
Monte Carlo standard error of the mean, with the number of chains and draws per chain.  ``train(n)`` plans the halves for
its n + 1 draws per chain; without ``train``, ``n_iterations`` (the sampling iterations to come) is required and the
tracking starts at once.  ``batch_size`` defaults to floor(sqrt(draws)).  ESS per gradient evaluation is the number to
tune epsilon, L, ``target_accept`` or a ladder by.
"""
from collections import namedtuple

import numpy as np

from .. import _lib
from ..distributions import Sampled
from ..keras_json import parse_model_json
from ..multi import EngineGroup, devices_from
from ..nn import BayesianModel
from ..tempering import validate_ladder
from ..tensors import to_numpy
from .Optimizer import Optimizer

Predictive = namedtuple("Predictive", ["mean", "variance", "rhat", "n_chains", "n_draws"])
ParameterSummary = namedtuple("ParameterSummary", ["mean", "sd", "rhat", "ess", "mcse", "n_chains", "n_draws"])

_PATHS = {"auto": _lib.PATH_AUTO, "generic": _lib.PATH_GENERIC, "fused": _lib.PATH_FUSED_SMALL,
          "tensor": _lib.PATH_TENSOR}


class HMC(Optimizer):
    def __init__(self):
        super().__init__()
        self._nb_burn_epoch = 10
        self._engine = None
        self._spec = None
        self._epsilon = self._L = self._m = None
        self._total_runs = 0
        self._accepted_runs = 0
        self._current_loss = 0
        self.last_diag = None
        self._sampling_started = False
        self._tracking = False
        self._ptrack = None              # track_parameters: {"batch": b, "n_planned": draws per chain or None}
        self._keep_samples = True
        self._adapt_iterations = 0
        self._target_accept = 0.8
        self._ladder = None
        self._R = 1
        self._temper = None

    def compile_extra_components(self, **kwargs):
        self._m = self._hyperparameters.m
        self._L = self._hyperparameters.L
        self._epsilon = self._hyperparameters.epsilon
        self._spec = parse_model_json(self._model_config)
        prior = kwargs["prior"]
        if "nb_burn_epoch" in kwargs:
            self._nb_burn_epoch = kwargs["nb_burn_epochs"]
        self._n_chains = int(self._hp("n_chains", 1))
        sem = self._hp("semantics", "reference")
        self._semantics = _lib.HMC_CANONICAL if sem in ("canonical", _lib.HMC_CANONICAL) else _lib.HMC_REFERENCE
        # the reference is stochastic by default (unseeded tf.random.normal / random.random, HMC.py:88,171): without an
        # explicit seed every optimizer draws its own, so repeated runs are independent; self.seed reproduces a run
        seed = self._hp("seed", None)
        self.seed = int(np.random.SeedSequence().entropy & ((1 << 63) - 1)) if seed is None else int(seed)
        self._adapt_iterations = int(self._hp("adapt_iterations", 0))
        self._target_accept = float(self._hp("target_accept", 0.8))
        if self._adapt_iterations < 0:
            raise ValueError("adapt_iterations must be >= 0")
        if not 0.0 < self._target_accept < 1.0:
            raise ValueError("target_accept must be in (0, 1)")
        self._ladder = validate_ladder(self._hp("inverse_temperatures", None))
        self._R = 1 if self._ladder is None else len(self._ladder)
        self._temper = None
        self._devices = devices_from(self._hp)
        self._engine = EngineGroup(self._spec, self._devices, seed=self.seed)
        path = self._hp("path", "auto")
        self._keep_samples = bool(self._hp("keep_samples", True))
        x, y = self._dataset.training_arrays()          # ONE full-dataset batch, frozen for the run (HMC.py:63-65)
        lowered = prior.lower(self._spec)

        def setup(i, e):
            e.set_option("path", _PATHS.get(path, path) if isinstance(path, str) else path)
            e.set_dataset(x, y, self._dataset.loss_kind, n_train=self._dataset.train_size)
            e.set_prior(*lowered)
            if not self._keep_samples:
                e.set_option("hmc_keep_samples", 0)
        self._engine.each(setup)
        self._engine.hmc_init(self._n_chains, self._epsilon, self._m, int(self._L), self._semantics,
                              q0=kwargs.get("q0"), chain_offset=int(self._hp("chain_offset", 0)), ladder=self._ladder)

    # ---- one iteration (HMC.py:74-104) -----------------------------------------------------
    def step(self, save_document_path=None, sampling=True, burning=False):
        self._sampling_started |= bool(sampling)
        d = self._engine.hmc_run(1, burning=burning, sampling=sampling)
        self._book(d, sampling)
        return d["mean_loss"]

    def _book(self, d, sampling=False):
        self.last_diag = d
        self._current_loss = d["mean_loss"]
        if self._ladder is None:
            self._total_runs += d["n_total"]
            self._accepted_runs += d["n_accepted"]
            return
        t = self._engine.hmc_tempering_stats()        # the acceptance rate reported is the beta = 1 rung's
        self._total_runs += int(t["rung_total"][0])
        self._accepted_runs += int(t["rung_accepted"][0])
        if sampling:
            if self._temper is None:
                self._temper = {k: np.zeros_like(v) for k, v in t.items()}
            for k, v in t.items():
                self._temper[k] += v

    def _phase(self, n, suffix, sampling, burning):
        """n iterations; with verbose on, the progress line is refreshed ~20 times per phase (each
        refresh is the only host sync), otherwise the whole phase is one C call."""
        chunk = max(1, n // 20) if self._verbose else max(1, n)
        done = 0
        while done < n:
            k = min(chunk, n - done)
            d = self._engine.hmc_run(k, burning=burning, sampling=sampling)
            self._book(d, sampling)
            done += k
            rate = self._accepted_runs / max(1, self._total_runs)
            self._print_progress(done / n, suffix=suffix, loss=d["mean_loss"], accept_rate=rate, bar_length=20)
        self._new_progress_line()

    def train(self, nb_iterations: int, loss_save_document_path: str = None, model_save_frequency: int = None,
              model_save_path: str = None):
        self._accepted_runs = self._total_runs = 0
        self._sampling_started = True
        self._phase(int(self._nb_burn_epoch), "HMC - Burning", sampling=False, burning=True)
        if self._adapt_iterations > 0:
            self._accepted_runs = self._total_runs = 0
            self._engine.hmc_adapt_begin(self._target_accept)
            self._phase(self._adapt_iterations, "HMC - Adapting", sampling=False, burning=False)
            self._engine.hmc_adapt_end()
        self._accepted_runs = self._total_runs = 0
        self._temper = None
        self._engine.each(lambda i, e: e.hmc_reset_samples())
        if self._ptrack is not None:
            self._ptrack["n_planned"] = int(nb_iterations) + 1
            self._engine.hmc_track_params(self._ptrack["n_planned"], self._ptrack["batch"])
        self._phase(int(nb_iterations), "HMC - Sampling", sampling=True, burning=False)

    @property
    def accept_rate(self):
        return self._accepted_runs / max(1, self._total_runs)

    @property
    def step_sizes(self):
        """[n_chains] float64: every chain's step size, in global chain order; [n_chains, R] (one per rung) with a
        tempering ladder"""
        e = self._engine.hmc_step_sizes()
        return e if self._ladder is None else e.reshape(-1, self._R)

    def tempering_rates(self):
        """-> (rung_accept [R], swap_accept [R - 1]) float64 over the sampling iterations so far: each rung's HMC
        acceptance rate and the acceptance rate of the swaps proposed between rungs r and r + 1"""
        if self._ladder is None:
            raise RuntimeError("no tempering ladder: set the inverse_temperatures hyper-parameter")
        t = self._temper
        if t is None:
            raise RuntimeError("no sampling iteration has run yet")
        return (t["rung_accepted"] / np.maximum(1, t["rung_total"]),
                t["swap_accepted"] / np.maximum(1, t["swap_attempted"]))

    # ---- streamed predictive ---------------------------------------------------------------
    def track_predictive(self, x, y=None):
        """Track the posterior predictive on x [Nt, ...] (and, with integer labels y [Nt], the classification
        uncertainty) over every draw the chains record from here on.  Call after ``compile`` and before ``train`` or the
        first sampling ``step``."""
        if self._engine is None:
            raise RuntimeError("compile the optimizer before tracking the predictive")
        if self._sampling_started:
            raise RuntimeError("track_predictive must be called before train() / the first sampling step")
        self._engine.hmc_track_predictive(to_numpy(x, np.float32), None if y is None else to_numpy(y))
        self._tracking = True

    def _tracked(self, semantics=None, divisor=None):
        if not self._tracking:
            raise RuntimeError("no predictive is tracked: call track_predictive(x) before training")
        return self._engine.hmc_predictive(semantics, divisor)

    def predictive(self) -> Predictive:
        """-> (mean, variance, rhat, n_chains, n_draws): the frequency-weighted predictive mean and population variance
        over every recorded draw, each [Nt, C], and the Gelman-Rubin R-hat of every output across the chains (NaN with
        fewer than two chains or draws, or where no chain moved)."""
        r, n_chains, T = self._tracked()
        return Predictive(r["mean"], r["variance"], r["rhat"], n_chains, T)

    def classification_uncertainty(self, divisor=None, semantics="reference"):
        """-> (total, aleatoric, epistemic), each [Nt, C, C], over every recorded draw: what
        ``result().classification_uncertainty(x, y, 0, divisor, semantics, mode="exact")`` returns.  Needs the labels
        given to ``track_predictive``."""
        r, _, _ = self._tracked(semantics, divisor)
        return r["total"], r["aleatoric"], r["epistemic"]

    # ---- streamed parameter diagnostics ----------------------------------------------------
    def track_parameters(self, n_iterations=None, batch_size=None):
        """Track the per-parameter posterior moments and convergence diagnostics over every draw the chains record.
        Call after ``compile`` and before ``train`` or the first sampling ``step``.  ``train(n)`` plans for its n + 1
        draws per chain; for sampling by ``step``, ``n_iterations`` (the sampling iterations to come) is required and
        the tracking starts now.  ``batch_size``: draws per batch of the ESS (default floor(sqrt(draws)))."""
        if self._engine is None:
            raise RuntimeError("compile the optimizer before tracking the parameters")
        if self._sampling_started:
            raise RuntimeError("track_parameters must be called before train() / the first sampling step")
        if batch_size is not None and int(batch_size) < 1:
            raise ValueError("batch_size must be >= 1")
        self._ptrack = {"batch": 0 if batch_size is None else int(batch_size), "n_planned": None}
        if n_iterations is not None:
            self._ptrack["n_planned"] = int(n_iterations) + 1
            self._engine.hmc_track_params(self._ptrack["n_planned"], self._ptrack["batch"])

    def parameter_summary(self) -> ParameterSummary:
        """-> (mean, sd, rhat, ess, mcse, n_chains, n_draws): per parameter ([P] float64, flat weight order) the mean
        and population sd over every recorded draw, the split R-hat, the batch-means effective sample size and the
        Monte Carlo standard error of the mean.  NaN marks a diverged chain, or a diagnostic that the draws do not
        define (too few draws or batches, or chains that never moved)."""
        t = self._ptrack
        if t is None or t["n_planned"] is None:
            raise RuntimeError("no parameters are tracked: call track_parameters() before train(), or "
                               "track_parameters(n_iterations) before sampling by step()")
        r, n_chains, T = self._engine.hmc_param_summary(t["n_planned"], t["batch"])
        return ParameterSummary(r["mean"], r["sd"], r["rhat"], r["ess"], r["mcse"], n_chains, T)

    def result(self) -> BayesianModel:
        if not self._keep_samples:
            raise RuntimeError("this HMC run keeps no samples (keep_samples=False): use predictive() and "
                               "classification_uncertainty() for the posterior predictive")
        samples, freq, _chain = self._engine.hmc_samples()
        if samples.shape[0] == 0:
            q, _ = self._engine.hmc_state()          # no sampling iteration yet: current positions, weight 1
            q = q[::self._R]                          # (the cold rung of every replica group)
            samples, freq = q, np.ones(q.shape[0], np.int32)
        posterior = BayesianModel(self._model_config, device=self._devices[0])
        posterior.apply_distribution(Sampled(samples, freq.tolist()), 0, self._spec.n_keras_layers - 1)
        return posterior
