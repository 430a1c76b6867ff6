/* pyesian_b200.h — C ABI of libpyesian_b200.so
 *
 * B200-native (sm_100a) implementation of ONE hot path of leoelm/Bayesian_inference_for_NN
 * ("Pyesian"): the particle-batched log-posterior forward/backward of a Keras Dense MLP over the
 * whole dataset for S weight samples at once, fused with the HMC leapfrog / Hamiltonian /
 * Metropolis update and the SVGD Stein step, plus the BayesianModel posterior predictive.
 *
 * The reference has no FFI layer of its own (it is pure Python on TensorFlow eager); the entry
 * points below are what a ctypes binding inside the reference's optimizer classes would bind.
 * Each one cites the reference code (path:line under the reference checkout) it replaces.
 *
 * Conventions
 *   - extern "C", plain pointers and sizes, no C++/torch types, no exceptions across the boundary.
 *   - every call returns 0 (PYB_OK) or a negative pyb_status; pyb_last_error() gives the message
 *     (thread-local).
 *   - the library owns all device memory behind the handle; caller-owned buffers are only read
 *     or written for the duration of the call.  `mem` says whether a caller buffer is host or
 *     device memory (device pointers come from DLPack capsules on the Python side).
 *   - device pointers: the library works on its own non-blocking stream, which is ordered against no other stream.  Every
 *     entry point that READS caller-owned device memory (pyb_set_dataset with PYB_MEM_DEVICE, W / x of pyb_predict and
 *     pyb_predict_uncertainty, src / dst of pyb_gather_rows) first waits for the whole device (cudaDeviceSynchronize), so a
 *     tensor produced on any stream just before the call is complete when it is read; results the library WRITES to
 *     caller-owned device memory are complete when the call returns (every call ends with a stream synchronisation).
 *   - sharded runs (pyb_svgd_set_comm / pyb_set_comm): every rank must hold the same number of particles; the first
 *     sharded step checks it (one all-reduce) and fails with PYB_ERR_INVALID instead of hanging in a collective.
 *   - one handle = one GPU; a handle is not thread-safe; there is NO CPU fallback: without a
 *     usable sm_100 device pyb_create fails with PYB_ERR_CUDA.
 *   - flat parameter order everywhere = model.layers order -> (kernel [in,out] C-order, bias)
 *     (HMC.py:178-183, SVGD.py:159-160,230-239, BayesianModel.py:73-77).
 */
#ifndef PYESIAN_B200_H
#define PYESIAN_B200_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define PYB_ABI_VERSION 1

typedef enum {
  PYB_OK = 0,
  PYB_ERR_INVALID = -1,     /* bad argument */
  PYB_ERR_CUDA = -2,        /* CUDA runtime/driver failure, or no sm_100 device */
  PYB_ERR_STATE = -3,       /* call made in the wrong state (e.g. run before init) */
  PYB_ERR_UNSUPPORTED = -4, /* model/loss combination outside the hot path */
  PYB_ERR_OOM = -5          /* device memory */
} pyb_status;

typedef enum { PYB_ACT_LINEAR = 0, PYB_ACT_RELU = 1, PYB_ACT_SOFTMAX = 2, PYB_ACT_TANH = 3,
               PYB_ACT_SIGMOID = 4 } pyb_activation;
typedef enum { PYB_LOSS_SPARSE_CE = 0, PYB_LOSS_MSE = 1 } pyb_loss;
typedef enum { PYB_MEM_HOST = 0, PYB_MEM_DEVICE = 1 } pyb_mem;
typedef enum { PYB_PRIOR_SCALAR = 0, PYB_PRIOR_PER_VARIABLE = 1, PYB_PRIOR_PER_ELEMENT = 2 } pyb_prior_form;
typedef enum { PYB_HMC_REFERENCE = 0, PYB_HMC_CANONICAL = 1 } pyb_hmc_semantics;
typedef enum { PYB_SVGD_REFERENCE_LIVE = 0, PYB_SVGD_CANONICAL_MEDIAN = 1 } pyb_svgd_semantics;
/* which device path evaluates the MLP; AUTO picks by shape */
typedef enum { PYB_PATH_AUTO = 0, PYB_PATH_GENERIC = 1, PYB_PATH_FUSED_SMALL = 2, PYB_PATH_TENSOR = 3 } pyb_path;

typedef enum { PYB_SG_SGLD = 0, PYB_SG_SWAG = 1 } pyb_sg_kind;
typedef enum { PYB_UQ_CANONICAL = 0, PYB_UQ_REFERENCE = 1 } pyb_uq_semantics;

typedef struct pyb_handle pyb_handle;

/* Dense stack parsed from the Keras model JSON (model.to_json(); consumed at HMC.py:56,
 * SVGD.py:222, BayesianModel.py:18).  The JSON parse itself is host logic on the Python side. */
typedef struct {
  int32_t n_layers;
  int32_t in_dim;
  const int32_t* units;      /* [n_layers] */
  const int32_t* activation; /* [n_layers] pyb_activation */
  const int32_t* use_bias;   /* [n_layers] 0/1 */
} pyb_model_desc;

typedef struct {
  double mean_loss;      /* mean over chains of the loss step() would return (HMC.py:96,104) */
  double accept_rate;    /* accepted / total since the phase started (HMC.py:112,122) */
  int64_t n_accepted;    /* over all local chains and iterations of this call */
  int64_t n_total;
  int64_t n_nan;         /* proposals whose Hamiltonian difference was NaN (rejected) */
  int64_t grad_evals;    /* chain x position evaluations actually executed in this call (L per iteration and chain,
                            plus one when the carried evaluation at the start position is not available) */
  double device_ms;      /* CUDA-event time of the call's kernels on the handle's stream */
  int64_t kernel_launches;
} pyb_hmc_diag;

/* ---- library ---- */
int pyb_version(void);
const char* pyb_last_error(void);
int pyb_device_count(int32_t* n_out);

/* ---- handle / model (replaces tf.keras.models.model_from_json + variable creation,
 *      HMC.py:56, SVGD.py:222, BayesianModel.py:18) ---- */
int pyb_create(const pyb_model_desc* desc, int32_t device_id, uint64_t seed, pyb_handle** out);
int pyb_destroy(pyb_handle* h);
int pyb_param_count(const pyb_handle* h, int64_t* n_params_out);
/* knobs: "path" (pyb_path), "workspace_mb", "chain_batch", "profile" (per-launch CUDA-event timing of the
 * tensor-core kernels, read back with "prof_ms"/"prof_flops"/"prof_launches"), and three A/B switches of the tensor
 * path, all default 1: "tc_pair" (CTA-pair cta_group::2 kernels), "tc_fuse" (layer 2, loss and both deltas inside
 * the layer-1 GEMM's epilogue), "tc_dual" (two feature tiles per item in the dW1 GEMM).  Switching them off selects
 * the older kernels that compute the same quantities (used by the tests and by tools/kernel_cycles.sh);
 * "predict_sharded" (default 0, see pyb_set_comm); "hmc_carry" (default 1): the loss and loss gradient at a chain's
 * current position are carried from the previous iteration (its end point if accepted, its start if rejected) instead
 * of being re-evaluated as HMC.py:80,82 do - L instead of L+1 full-data evaluations per iteration, identical results;
 * "hmc_keep_samples" (default 1): every recorded HMC draw is kept for pyb_hmc_samples; 0 keeps none (no sample arena,
 * no host copy, pyb_hmc_sample_count returns 0) for runs that only need the streamed predictive
 * (pyb_hmc_track_predictive); the chains move identically either way.  It cannot change during a sampling phase.
 * "hmc_swap" (default 1): with a tempering ladder set (pyb_hmc_set_temperatures), 0 keeps the ladder but proposes no
 * replica swaps (the rungs then run side by side as independent tempered chains). */
int pyb_set_option(pyb_handle* h, const char* key, double value);
/* read-outs: "path_used", "kernel_launches", "last_device_ms", "workspace_bytes", "tensor_path_ok", "hmc_arena_rows"
 * (rows of the device sample arena, 0 while it has never been sized), "fs_cluster_used" (CTAs per chain of the last
 * small-width HMC launch: 1, 2, 4 or 8; 0 before the first), "hmc_param_bytes" (device bytes held by
 * pyb_hmc_track_params), "svgd_stein_used" (Stein-update branch of the last pyb_svgd_step or canonical pyb_svgd_phi:
 * 0 live sweep as per-particle launches, 1 live sweep as one cooperative launch, 2 live sweep in one CTA, 3 canonical on
 * the float64 kernels, 4 canonical on the tensor cores, 5 canonical on the tensor cores sharded over the parameters;
 * 0 before the first call; the live-formula pyb_svgd_phi leaves it unchanged) */
int pyb_get_info(const pyb_handle* h, const char* key, double* value_out);

/* ---- inputs ---- */
/* Full training batch kept resident in HBM (HMC.py:63-65: ONE full-dataset batch frozen for the
 * run; SVGD.py:220-221 draws minibatches from the same pool).  X [N, in_dim] float32 row-major;
 * y int32 [N] (SPARSE_CE) or float32 [N, out_dim] (MSE).  n_train multiplies the mean loss in the
 * potential (HMC.py:158); pass N (or <=0) for the reference behaviour. */
int pyb_set_dataset(pyb_handle* h, const float* X, int64_t N, const void* y, int32_t loss_kind,
                    int32_t mem, int64_t n_train);
/* GaussianPrior.get_model_priors (GaussianPrior.py:100-121, :28-47): sigma = rho used RAW.
 * SCALAR: 1 value each; PER_VARIABLE: one per trainable variable (kernel, bias, kernel, ...);
 * PER_ELEMENT: n_params values.  Host pointers. */
int pyb_set_prior_gaussian(pyb_handle* h, const float* mean, const float* sigma, int32_t form);

/* ---- HMC (HMC.py:45-72 compile, :74-104 step, :106-126 train, :128-171 helpers) ---- */
/* S local chains whose global ids are chain_offset .. chain_offset+S-1 (RNG counters use the
 * global id, so a sharded run reproduces the unsharded one).  q0 NULL => every chain starts at
 * the prior mean (HMC.py:69-72); else host float32 [S, P]. */
int pyb_hmc_init(pyb_handle* h, int64_t S, int64_t chain_offset, double epsilon, double m, int32_t L,
                 int32_t semantics, const float* q0);
/* test hook: momenta [S,P] and/or uniforms [S] (host) for the NEXT iteration only. */
int pyb_hmc_inject(pyb_handle* h, const float* p, const float* u);
/* n_iters iterations of HMC.step(sampling, burning) for all chains, no host sync inside. */
int pyb_hmc_run(pyb_handle* h, int32_t n_iters, int32_t burning, int32_t sampling, pyb_hmc_diag* diag_out);
/* parity hook: U = -log prior + n_train*mean_loss, the mean loss, and dU/dq for S given
 * positions (HMC._potential_energy HMC.py:149-159 and the gradient _step_p takes :128-136).
 * All host pointers; U/loss/grad may be NULL. */
int pyb_hmc_eval(pyb_handle* h, const float* q, int64_t S, float* U_out, float* loss_out, float* grad_out);
int pyb_hmc_get_state(pyb_handle* h, float* q_out, float* p_out);
/* per-chain values of the LAST iteration (any may be NULL). */
int pyb_hmc_last(pyb_handle* h, float* U0, float* K0, float* U1, float* K1, float* log_alpha,
                 int32_t* accepted, float* loss);
/* samples + frequencies of every chain (HMC.py:75-77,92-104; HMC.result :176-184), chain-major,
 * within a chain in acceptance order. */
int pyb_hmc_reset_samples(pyb_handle* h);
int pyb_hmc_sample_count(pyb_handle* h, int64_t* n_out);
int pyb_hmc_samples(pyb_handle* h, float* samples_out, int32_t* freq_out, int32_t* chain_out);

/* ---- per-chain step sizes and their adaptation (the reference uses one epsilon for its one chain, HMC.py:53-55) ----
 * Every chain may have its own step size e_s; its leapfrog then kicks by (float)e_s and (float)(e_s/2) and drifts by
 * (float)(e_s/m), each rounded once from double, so a chain whose e_s equals epsilon moves exactly as with the scalar.
 * Until step sizes are set or adapted, every chain uses epsilon.  pyb_hmc_init ends any adaptation and drops the
 * per-chain step sizes.  Before pyb_hmc_init all four calls return PYB_ERR_STATE.
 * pyb_hmc_adapt_begin: from the next pyb_hmc_run on, every iteration (burn-in included) updates each chain's step size
 *   by dual averaging (Hoffman & Gelman 2014, Algorithm 5) towards an acceptance probability of target_accept
 *   (0 < target < 1, else PYB_ERR_INVALID; PYB_ERR_STATE if already adapting).  Per chain and adaptation iteration
 *   t = 1, 2, ... with a = min(1, exp(log_alpha)) (NaN: 0), gamma = 0.05, t0 = 10, kappa = 0.75 (Stan's defaults):
 *     h_bar = (1 - 1/(t + t0)) h_bar + (target - a)/(t + t0);  log_eps = mu - sqrt(t)/gamma h_bar;
 *     log_eps_bar = t^-kappa log_eps + (1 - t^-kappa) log_eps_bar;  e_s = exp(log_eps)
 *   starting from mu = log(10 e_s), h_bar = 0, log_eps_bar = 0.  Chains adapt independently: a sharded run adapts as
 *   the unsharded one.  While adapting, pyb_hmc_run with sampling = 1 returns PYB_ERR_STATE (draws taken while the
 *   step sizes move are not draws from the posterior).
 * pyb_hmc_adapt_end: freezes e_s = exp(log_eps_bar) (unchanged if no iteration ran); PYB_ERR_STATE if not adapting.
 * pyb_hmc_step_sizes: eps_out [S] host float64, the current e_s (epsilon for every chain when never set or adapted).
 * pyb_hmc_set_step_sizes: eps [S] host float64, each finite and > 0 (else PYB_ERR_INVALID); PYB_ERR_STATE while
 *   adapting. */
int pyb_hmc_adapt_begin(pyb_handle* h, double target_accept);
int pyb_hmc_adapt_end(pyb_handle* h);
int pyb_hmc_step_sizes(pyb_handle* h, double* eps_out);
int pyb_hmc_set_step_sizes(pyb_handle* h, const double* eps);

/* ---- parallel tempering: HMC chains as ladders of tempered replicas with replica exchange on the device ----
 * Ladder.  R >= 2 inverse temperatures beta_0 = 1 > beta_1 > ... > beta_{R-1} > 0 (R <= 64).  Local chain s = g R + r
 *   is rung r of replica group g: groups are contiguous and group-major, so global chain ids stay chain_offset + s and
 *   every Philox stream keeps its key.  S and chain_offset must be multiples of R, so a shard always holds whole groups.
 * Tempered potential.  Chain s samples prior(q) exp(-beta_r E(q)) with E = n_train mean_loss: in float
 *   U = (Up + prior_const) + (beta_r loss) n_train and dU/dq = beta_r g_data + (q - mu) / sigma^2.  The loss and loss
 *   gradient carried between iterations ("hmc_carry") stay untempered, so a state keeps its evaluation when it moves to
 *   another rung.  With beta = 1 every expression rounds exactly as without a ladder: the cold rung moves bit for bit as
 *   an untempered chain with the same global id (as long as no swap reaches it).
 * Swap move.  After every iteration's accept / restore, one deterministic even-odd round (Syed, Bouchard-Cote,
 *   Deligiannidis & Doucet 2022, non-reversible parallel tempering): in iteration iter the pairs (r, r + 1) with
 *   r = iter (mod 2) of every group propose to exchange their states, accepted iff u < exp(log_r) with
 *     log_r = (beta_r - beta_{r+1}) n_train ((double)loss_r - (double)loss_{r+1})   in double (NaN rejects),
 *     u = the Philox uniform of global chain chain_offset + g R + r, iteration iter, stream 4 (seed).
 *   loss is the untempered mean loss at each chain's current position (pyb_hmc_last's loss).  An accepted swap exchanges
 *   the two chains' positions, their carried loss gradients and losses; momenta are redrawn every iteration, and step
 *   sizes and their dual-averaging state stay with the chain slot (each rung adapts its own).  Swaps run in every
 *   iteration while a ladder is set: burn-in, adaptation and sampling.
 * Draws.  Only rung-0 chains record draws, into the samples and the tracked predictive: the state before the first
 *   sampling iteration, then a new draw whenever the position changed (HMC accept or swap; the draw is the position
 *   after the swap), else the last draw's frequency grows.  pyb_hmc_samples returns them with their global chain ids;
 *   the tracked predictive keeps sums for the S / R cold chains (n_chains of pyb_hmc_predictive_finish = the number of
 *   groups).  pyb_hmc_diag still counts all chains.
 * Sharding.  Groups never straddle handles and swaps never cross them: a sharded run reproduces the unsharded one bit
 *   for bit with no collective.
 * pyb_hmc_set_temperatures: beta [R] host float64; beta = NULL with R = 0 turns tempering off.  PYB_ERR_INVALID for a
 *   ladder outside the rules above; PYB_ERR_STATE before pyb_hmc_init and once a sampling iteration has run since
 *   pyb_hmc_init / pyb_hmc_reset_samples.  pyb_hmc_init clears the ladder.
 * pyb_hmc_tempering_stats: host arrays of R, R, R - 1 and R - 1 entries (any may be NULL): per rung the HMC proposals
 *   accepted and made, per pair (r, r + 1) the swaps attempted and accepted, counted over the last pyb_hmc_run call and
 *   this handle's groups (counts of different handles add up).  PYB_ERR_STATE without a ladder.
 * pyb_hmc_last_swaps: per chain [S] the log ratio of the swap proposed with its upper neighbour in the last iteration
 *   and whether it was taken (NaN and 0 for a chain that proposed none).  PYB_ERR_STATE without a ladder or before an
 *   iteration has run under it. */
int pyb_hmc_set_temperatures(pyb_handle* h, const double* beta, int32_t R);
int pyb_hmc_tempering_stats(pyb_handle* h, int64_t* rung_accepted, int64_t* rung_total, int64_t* swap_attempted,
                            int64_t* swap_accepted);
int pyb_hmc_last_swaps(pyb_handle* h, float* log_r, int32_t* swapped);

/* ---- streamed HMC posterior predictive (BayesianModel.predict BayesianModel.py:106-129 in mode "exact" over the draws
 *      HMC records, HMC.py:92-104; Metrics.classification_uncertainty Metrics.py:344-375) ----
 * The tracked draws of every chain are exactly the draws pyb_hmc_samples returns with their frequencies: the state
 * before the first sampling iteration after pyb_hmc_init / pyb_hmc_reset_samples, then the position after every
 * sampling iteration; burn-in iterations add nothing.  So every chain has the same number T of draws.  Each draw goes
 * through pyb_predict's forward pass on the tracked inputs (NaN -> 0 per element) inside pyb_hmc_run, on the handle's
 * stream, and only moment sums are kept.
 * pyb_hmc_track_predictive: x [Nt, in_dim] float32 host or device (copied once: the caller may free it), y [Nt] int32
 *   host labels or NULL (needed for the uncertainty matrices; < out_dim, or < 2 for a one-unit output).  Must come before
 *   the first sampling iteration (PYB_ERR_STATE otherwise); x = NULL stops tracking and frees its memory.  Device memory:
 *   (8 + 4) S Nt out_dim bytes of per-chain sums, checked up front (PYB_ERR_OOM with the size in the message).
 *   pyb_hmc_reset_samples clears the sums, pyb_hmc_init stops tracking. */
int pyb_hmc_track_predictive(pyb_handle* h, const float* x, int64_t Nt, const int32_t* y);
/* sums_out [4, Nt, out_dim] float64 over this handle's chains: A = sum o, Q = sum o^2, M = sum_s (sum_t o)^2 and
 * W = sum_s sum_t (o - mean_t o)^2 (the within-chain sum of squares, kept exactly: Q - M/T cancels for chains that
 * barely move); s2_out [Nt, out_dim, out_dim] = sum o o^T (labels given and out_dim > 1; may be NULL); n_draws_out = T.
 * All are sums over chains: the sums of handles holding disjoint chains (devices, ranks) add up. */
int pyb_hmc_predictive_sums(pyb_handle* h, double* sums_out, double* s2_out, int64_t* n_draws_out);
/* From sums (of this handle, or of several added together) over n_chains chains with n_draws draws each: mean_out /
 * var_out [Nt, out_dim] as pyb_predict with the samples weighted by their frequencies (population variance);
 * rhat_out [Nt, out_dim] the Gelman-Rubin R-hat of every output element (classic form, not split or rank-normalised;
 * NaN when n_chains < 2, n_draws < 2 or the within-chain variance is 0); total / aleatoric / epistemic [Nt, Ce, Ce] as
 * pyb_predict_uncertainty (uq_semantics, divisor; need the labels and, for out_dim > 1, s2).  Any output may be NULL.
 * Nt and the labels are this handle's tracked ones. */
int pyb_hmc_predictive_finish(pyb_handle* h, const double* sums, const double* s2, int64_t n_chains, int64_t n_draws,
                              int32_t uq_semantics, double divisor, float* mean_out, float* var_out, float* rhat_out,
                              float* total_out, float* aleatoric_out, float* epistemic_out);

/* ---- streamed per-parameter posterior moments and convergence diagnostics of the HMC chains ----
 * The tracked draws are those of the streamed predictive (and of pyb_hmc_samples with their frequencies): the state
 * before the first sampling iteration after pyb_hmc_init / pyb_hmc_reset_samples, then the position after every
 * sampling iteration (after accept / restore and the swap round); with a ladder the S / R rung-0 chains only.  So every
 * tracked chain has the same number T of draws; after n sampling iterations T = n + 1.  Every parameter (flat order of
 * the weight layout) of every draw is folded into sums inside pyb_hmc_run; nothing is mapped: a NaN parameter (a
 * diverged chain) gives NaN results.
 * Definitions, with S chains, T draws x_st each, h = floor(n_planned / 2), the batch size b and a = floor(T / b):
 *   mean = sum x / (S T);  sd = sqrt of the population variance over all S T draws (pyb_predict's weighting).
 *   split-R-hat = the classic R-hat (pyb_hmc_predictive_finish) over the 2 S half-chains [0, h) and [h, 2h) of h draws;
 *     draws from 2h on count in the moments and the ESS only.  NaN when T < 2h, h < 2 or the within-chain variance is 0.
 *   ESS by batch means (Flegal & Jones 2010): lambda^2 = W / (S (T - 1)) with W the within-chain sum of squares;
 *     sigma^2_bm = b V / (S (a - 1)), V = sum_s sum_{k<a} (Ybar_sk - Ybar_s)^2 over the means Ybar_sk of the complete
 *     batches of chain s and their mean Ybar_s (a trailing partial batch is left out);  ess = S T lambda^2 / sigma^2_bm,
 *     NaN when T < 2, a < 2, lambda^2 = 0 or sigma^2_bm = 0, and not capped at S T (antithetic chains exceed it).
 *   mcse = sqrt(sigma^2_bm / (S T))  (NaN when a < 2).
 * pyb_hmc_track_params: track from the next sampling iteration on, planned for n_planned draws per chain (it fixes h;
 *   more draws may follow) with batch size b = batch, or floor(sqrt(n_planned)) for batch = 0.  PYB_ERR_STATE before
 *   pyb_hmc_init and once a sampling iteration has run (until pyb_hmc_reset_samples); PYB_ERR_INVALID for n_planned < 4,
 *   batch < 0 or fewer than two batches in n_planned.  n_planned = 0 stops tracking and frees its memory.  Device
 *   memory: 36 bytes per (tracked chain, parameter) plus 48 P bytes for the pooled sums and 48 P per group of >= 32
 *   chains of the accumulation, checked up front (PYB_ERR_OOM with
 *   the size in the message; read back with pyb_get_info "hmc_param_bytes").  pyb_hmc_reset_samples clears the sums,
 *   pyb_hmc_init stops tracking, and setting or clearing a ladder resizes them to the tracked chains.  The sums are
 *   added in a fixed order: deterministic, and one call of n iterations gives those of n calls of one.
 * pyb_hmc_param_sums: sums_out [7, P] float64 over this handle's chains, in this order: A = sum of all draws,
 *   M = sum_s (sum_t x)^2, W = within-chain sum of squares; the same three over the complete half-chains (Ah, Mh, Wh);
 *   V (above); n_draws_out = T.  All are sums over chains: the sums of handles holding disjoint chains add up.
 *   PYB_ERR_STATE without tracking or before the first tracked draw.
 * pyb_hmc_param_finish: from sums (of this handle, or of several added) over n_chains chains with n_draws draws each and
 *   the n_planned / batch of the tracking: mean_out, sd_out, rhat_out (split), ess_out, mcse_out, each [P] float64 (any
 *   may be NULL).  PYB_ERR_INVALID for a NULL sums, n_chains or n_draws <= 0, and the n_planned / batch rules above. */
int pyb_hmc_track_params(pyb_handle* h, int64_t n_planned, int32_t batch);
int pyb_hmc_param_sums(pyb_handle* h, double* sums_out, int64_t* n_draws_out);
int pyb_hmc_param_finish(pyb_handle* h, const double* sums, int64_t n_chains, int64_t n_draws, int64_t n_planned,
                         int32_t batch, double* mean_out, double* sd_out, double* rhat_out, double* ess_out,
                         double* mcse_out);

/* ---- SVGD (SVGD.py:219-228 compile, :143-157 init, :84-141 step, :54-68 + :183-202 live kernel,
 *      :165-181 median-heuristic kernel, legacy Adam created :226 applied :120) ---- */
/* particles0 NULL => one prior sample per element (Philox); else host float64 [S, P]. */
int pyb_svgd_init(pyb_handle* h, int64_t S, int64_t particle_offset, double lr, int32_t semantics,
                  const double* particles0);
/* One step on the minibatch given by row indices into the resident dataset (host int32 [B]);
 * batch_idx NULL => the full dataset.  loss_out = mean over particles of the minibatch loss. */
int pyb_svgd_step(pyb_handle* h, const int32_t* batch_idx, int64_t B, double* loss_out);
/* parity hook: phi for given particles X [S,P] (float64) and gradients G [S,P] (float32):
 * CANONICAL_MEDIAN: phi=(K G + dxkxy)/S with the median bandwidth, h_out = h.
 * REFERENCE_LIVE : row i = ((sum_k K_ik) G_i + 2 sum_k K_ik (x_i-x_k))/S with gamma=1 (Jacobi
 * evaluation of the formula the live sweep applies row by row). */
int pyb_svgd_phi(pyb_handle* h, const double* X, const float* G, int64_t S, int32_t semantics,
                 float* phi_out, double* h_out);
int pyb_svgd_get_particles(pyb_handle* h, double* particles_out);
/* The validation pass of SVGD.step (SVGD.py:126-129: every particle's loss over the whole validation split, summed
 * / M) without moving the particles: the held-out set (host X [N, in_dim] float32, y as in pyb_set_dataset) is uploaded
 * once, pyb_svgd_validation_loss evaluates the mean loss of every resident particle on it (per_particle_out [S] host,
 * may be NULL) and returns their mean (all-reduced over the ranks of a sharded run). */
int pyb_svgd_set_validation(pyb_handle* h, const float* X, const void* y, int64_t N);
int pyb_svgd_validation_loss(pyb_handle* h, double* mean_loss_out, float* per_particle_out);
/* NCCL plumbing for sharded particles: all ranks pass the same 128-byte ncclUniqueId.
 * Options of the sharded canonical step on the tensor path (all ranks must set them alike): "svgd_pshard" (default 1:
 * Stein phase sharded over the parameters; 0: row-sharded with all-gathers), "svgd_p2p" (default 1: the gradient rows and
 * the updated particle blocks are exchanged by stores of the library's own kernels into peer memory - CUDA IPC between
 * processes of one host, plain peer access inside one process - with one-float NCCL barriers; falls back to ncclSend /
 * ncclRecv when a mapping is refused; 0: always NCCL; read-out "svgd_p2p" tells which one runs), "svgd_gram_sync" and
 * "svgd_halves" (A/B switches of the pipeline, default 0), "svgd_chain_fused" (default 1: the reduction / median /
 * kernel-matrix chain in half the launches), "select_compact" (median radix select of a local set: 0 default, 1 with
 * candidate compaction, 2 with every digit picked inside the next pass), "live_cta" (default 1: the reference-live sweep of a particle
 * set that fits one CTA's shared memory runs in one CTA); read-outs "svgd_phase_ms_0..6" (with "profile" on): CUDA-event
 * split of the last sharded step. */
int pyb_svgd_set_comm(pyb_handle* h, int32_t rank, int32_t world, const void* nccl_unique_id_128);
/* The same communicator under its general name.  With option "predict_sharded" = 1, pyb_predict and
 * pyb_predict_uncertainty treat W as this rank's share of the weight samples (BayesianModel.predict's nb_samples
 * draws split over the ranks) and all-reduce their moment sums: every rank returns the mean / variance / uncertainty
 * matrices over ALL ranks' samples; all_out stays local.  All ranks must make the call. */
int pyb_set_comm(pyb_handle* h, int32_t rank, int32_t world, const void* nccl_unique_id_128);
int pyb_nccl_unique_id(void* out_128);

/* ---- S-batched stochastic-gradient chains: SGLD (SGLD.py:46-95 step, :115-121 schedule on the host, :133-143
 *      compile) and SWAG (SWAG.py:43-94 step, :97-113 compile) on the same minibatch gradient kernels ----
 * S local chains with global ids chain_offset.. (Philox counters use the global id).  theta0 NULL => Keras Dense
 * defaults per chain (glorot_uniform kernels, zero biases: what model_from_json builds, SGLD.py:138); else host
 * float32 [theta0_rows, P] with theta0_rows = 1 (every chain starts from the same weights: SWAG's starting_model,
 * SWAG.py:105-106) or S.  k_dev / frequency: SWAG's deviation-matrix width and moment update period (ignored by SGLD,
 * whose moments are updated every step and whose deviation matrix is never read, SGLD.py:146-161). */
int pyb_sg_init(pyb_handle* h, int64_t S, int64_t chain_offset, int32_t kind, int32_t k_dev, int32_t frequency,
                const float* theta0, int32_t theta0_rows);
/* One step of every chain on the minibatch batch_idx (host int32 [B] row indices into the resident dataset; NULL =>
 * the full dataset).  SGLD: theta -= lr * (g + lr * z) (the reference draws its noise with stddev = lr and multiplies
 * by lr again, SGLD.py:67-68); noise = host float32 [S, P] standard normals injected for this step (test hook) or
 * NULL => Philox.  SWAG: theta -= lr * g.  Then the running moments / deviation column as the reference updates
 * them.  loss_out [S] (host, may be NULL) = each chain's minibatch loss BEFORE the update; mean_loss_out = their mean. */
int pyb_sg_step(pyb_handle* h, const int32_t* batch_idx, int64_t B, double lr, const float* noise, float* loss_out,
                double* mean_loss_out);
/* State read-back (any pointer may be NULL): theta, mean, sq_mean host float32 [S, P]; dev [S, k_dev, P] (column c of
 * chain s contiguous; columns >= *n_cols are zero); n_cols = deviation columns filled; n_steps = steps taken. */
int pyb_sg_get(pyb_handle* h, float* theta, float* mean, float* sq_mean, float* dev, int32_t* n_cols, int64_t* n_steps);

/* ---- posterior predictive (BayesianModel.predict BayesianModel.py:106-129; Plotter.py:244) ----
 * W [n,P] weight samples, weight [n] or NULL (=1), x [Nt,in_dim]; mean/var [Nt,out_dim] with
 * NaN->0 per element and population variance; all_out [n,Nt,out_dim] or NULL.  weight and the outputs are host
 * pointers; W and x may be host OR device pointers (device memory is read in place: weight samples that already
 * live in HBM skip the n*P*4-byte upload). */
int pyb_predict(pyb_handle* h, const float* W, int64_t n, const float* weight, const float* x,
                int64_t Nt, float* mean_out, float* var_out, float* all_out);

/* Metrics.classification_uncertainty (Metrics.py:344-375): for the same n weight samples and inputs, with integer
 * labels y [Nt] (host), per data row the matrices  aleatoric = sum_k w_k (diag(p_k) - p_k p_k^T)  and epistemic, divided
 * by `divisor` (the reference divides by its n_samples ARGUMENT, :368-369).
 *   PYB_UQ_REFERENCE: what the reference's code computes (pinned by goldens produced by the reference method itself,
 *     tests/golden/reference_metrics.npz): its accumulators are never reset between rows, so row r holds the running sum
 *     over rows 0..r (:352-366), and its epistemic term is D D^T with D = reshape(p, (-1,1)) - one_hot(label) BROADCAST
 *     to D_ij = p_i - onehot_j (:362-363), i.e. C p p^T - p 1^T - 1 p^T + 1 1^T, independent of the label.
 *   PYB_UQ_CANONICAL: per-row matrices with epistemic = sum_k w_k (p_k - onehot(y)) (p_k - onehot(y))^T.
 * Outputs are host float32 [Nt, Ce, Ce] with Ce = out_dim, or 2 for a one-unit output widened to [1-p, p] (:357-359);
 * total = epistemic + aleatoric; mean_out [Nt, out_dim] may be NULL.  At most 32 classes. */
int pyb_predict_uncertainty(pyb_handle* h, const float* W, int64_t n, const float* weight, const float* x, int64_t Nt,
                            const int32_t* y, int32_t semantics, double divisor, float* total_out,
                            float* aleatoric_out, float* epistemic_out, float* mean_out);

/* ---- device-resident arrays owned by the caller (posterior samples kept in HBM between predict calls:
 *      BayesianModel.predict re-draws nb_samples weight vectors from the SAME Sampled on every call,
 *      BayesianModel.py:106-129 / Sampled.py:29-32) ----
 * pyb_buffer_create allocates `bytes` on the handle's device and, if host_or_null is given, uploads them;
 * pyb_gather_rows writes dst[k] = src[idx[k]] for rows of row_len floats (src, dst device pointers, idx on the host);
 * buffers outlive nothing: free them with pyb_buffer_destroy before pyb_destroy. */
int pyb_buffer_create(pyb_handle* h, const void* host_or_null, int64_t bytes, void** dev_out);
int pyb_buffer_destroy(pyb_handle* h, void* dev);
int pyb_gather_rows(pyb_handle* h, const float* src, const int64_t* idx, int64_t n, int64_t row_len, float* dst);

/* ---- diagnostic entry points (used by tests/, never by the host classes) ----
 * pyb_debug_tc_gemm: D[M, Nn] = A[M, K] B[Nn, K]^T through the tcgen05 bf16x3 GEMM kernel (host pointers; Nn % 16 == 0,
 *   Nn <= 256, K % 8 == 0): the unit test of the kernel every tensor-path GEMM is built from.
 * pyb_debug_relu_mask: relu'(z1) exactly as the LAST tensor-path evaluation on the resident dataset used it, for one
 *   chain of its chain batch: mask_out [N, H] uint8 on the host.  HMC._step_p (HMC.py:128-136) differentiates through
 *   Keras' relu, whose derivative is discontinuous at 0; two correct float32 implementations disagree about the units
 *   whose pre-activation lies within rounding of zero, so the full-size parity test evaluates the float64 oracle with
 *   the device's own mask (tests/test_gpu_fullsize.py). */
int pyb_debug_tc_gemm(pyb_handle* h, const float* A, const float* B, int32_t M, int32_t Nn, int32_t K, float* D);
int pyb_debug_relu_mask(pyb_handle* h, int64_t chain, uint8_t* mask_out);

#ifdef __cplusplus
}
#endif
#endif /* PYESIAN_B200_H */
