// common.cuh — handle layout, error plumbing, Philox, small device helpers.
// Part of libpyesian_b200.so (see include/pyesian_b200.h for the C ABI and reference citations).
#pragma once
#include <cuda_runtime.h>
#include <cuda.h>
#include <stdint.h>
#include <stdio.h>
#include <string.h>
#include <stdlib.h>
#include <string>
#include <vector>
#include <stdexcept>
#include "../../include/pyesian_b200.h"

#include <nvtx3/nvToolsExt.h>   // header-only NVTX 3: the ranges cost one predictable branch unless a tool (nsys, ncu --nvtx) is attached

namespace pyb {

// RAII NVTX range on the calling host thread: marks the phases of the hot path in profiler timelines
// (fwd/bwd evaluation, kick/drift, accept, Gram, exchange, ...)
struct NvtxRange {
  explicit NvtxRange(const char* name) { nvtxRangePushA(name); }
  ~NvtxRange() { nvtxRangePop(); }
  NvtxRange(const NvtxRange&) = delete;
  NvtxRange& operator=(const NvtxRange&) = delete;
};

// ------------------------------------------------------------------------------------------
// errors: C++ exceptions are used internally and converted to status codes at the ABI boundary
// ------------------------------------------------------------------------------------------
struct Error : std::runtime_error {
  int code;
  Error(int c, const std::string& m) : std::runtime_error(m), code(c) {}
};
void set_last_error(const std::string& m);

#define PYB_CUDA(expr)                                                                     \
  do {                                                                                     \
    cudaError_t _e = (expr);                                                               \
    if (_e != cudaSuccess) {                                                               \
      char _b[512];                                                                        \
      snprintf(_b, sizeof(_b), "%s failed: %s (%s:%d)", #expr, cudaGetErrorString(_e),     \
               __FILE__, __LINE__);                                                        \
      throw pyb::Error(_e == cudaErrorMemoryAllocation ? PYB_ERR_OOM : PYB_ERR_CUDA, _b);  \
    }                                                                                      \
  } while (0)

#define PYB_REQUIRE(cond, code, msg)                       \
  do {                                                     \
    if (!(cond)) throw pyb::Error((code), (msg));          \
  } while (0)

// ------------------------------------------------------------------------------------------
// device buffer (owning)
// ------------------------------------------------------------------------------------------
template <typename T>
struct DevBuf {
  T* p = nullptr;
  size_t n = 0;
  DevBuf() {}
  DevBuf(const DevBuf&) = delete;
  DevBuf& operator=(const DevBuf&) = delete;
  ~DevBuf() { release(); }
  void release() {
    if (p) cudaFree(p);
    p = nullptr;
    n = 0;
  }
  void alloc(size_t count) {
    if (count <= n && p) return;
    release();
    if (count == 0) return;
    PYB_CUDA(cudaMalloc((void**)&p, count * sizeof(T)));
    n = count;
  }
  size_t bytes() const { return n * sizeof(T); }
  void swap(DevBuf& o) {
    T* tp = p; p = o.p; o.p = tp;
    size_t tn = n; n = o.n; o.n = tn;
  }
};

// ------------------------------------------------------------------------------------------
// model layout: the weight-layout packer's device-side view of the Keras Dense stack
// ------------------------------------------------------------------------------------------
constexpr int kMaxLayers = 16;
struct LayerDesc {
  int fan_in, fan_out, act, use_bias;
  int64_t w_off, b_off;  // offsets into the flat [P] parameter vector (b_off = -1: no bias)
};
struct Model {
  int n_layers = 0;
  int in_dim = 0;
  int out_dim = 0;
  int64_t P = 0;
  int max_width = 0;
  LayerDesc layer[kMaxLayers];
};

// ------------------------------------------------------------------------------------------
// Philox4x32-10 (Salmon et al. 2011).  counter = (block, chain, iteration, stream), key = seed.
// ------------------------------------------------------------------------------------------
enum { STREAM_MOMENTUM = 0, STREAM_UNIFORM = 1, STREAM_INIT = 2, STREAM_SGLD = 3, STREAM_SWAP = 4 };

__host__ __device__ inline void philox4x32_10(uint32_t c0, uint32_t c1, uint32_t c2, uint32_t c3,
                                               uint32_t k0, uint32_t k1, uint32_t out[4]) {
#pragma unroll
  for (int r = 0; r < 10; ++r) {
    uint64_t p0 = (uint64_t)0xD2511F53u * c0;
    uint64_t p1 = (uint64_t)0xCD9E8D57u * c2;
    uint32_t hi0 = (uint32_t)(p0 >> 32), lo0 = (uint32_t)p0;
    uint32_t hi1 = (uint32_t)(p1 >> 32), lo1 = (uint32_t)p1;
    uint32_t n0 = hi1 ^ c1 ^ k0, n1 = lo1, n2 = hi0 ^ c3 ^ k1, n3 = lo0;
    c0 = n0; c1 = n1; c2 = n2; c3 = n3;
    k0 += 0x9E3779B9u;
    k1 += 0xBB67AE85u;
  }
  out[0] = c0; out[1] = c1; out[2] = c2; out[3] = c3;
}

// leapfrog coefficients of a step size e: full kick, half kick, drift (HMC.py:128-141), each computed in double and
// rounded to float once, so a chain whose own step size equals epsilon gets the scalar path's coefficients bit for bit
struct StepCoef { float eps, half, drift; };
__host__ __device__ inline StepCoef step_coef(double e, double m) { return {(float)e, (float)(e / 2), (float)(e / m)}; }

#ifdef __CUDACC__
// 4 standard normals from one Philox block (two Box-Muller pairs)
__device__ inline void philox_normal4(uint32_t block, uint32_t chain, uint32_t iter, uint32_t stream,
                                      uint64_t seed, float z[4]) {
  uint32_t r[4];
  philox4x32_10(block, chain, iter, stream, (uint32_t)seed, (uint32_t)(seed >> 32), r);
  const float k = 5.9604644775390625e-08f;  // 2^-24
  float u1a = ((float)(r[0] >> 8) + 1.0f) * k, u2a = (float)(r[1] >> 8) * k;
  float u1b = ((float)(r[2] >> 8) + 1.0f) * k, u2b = (float)(r[3] >> 8) * k;
  float ra = sqrtf(-2.0f * logf(u1a)), rb = sqrtf(-2.0f * logf(u1b));
  float sa, ca, sb, cb;
  sincosf(6.283185307179586f * u2a, &sa, &ca);
  sincosf(6.283185307179586f * u2b, &sb, &cb);
  z[0] = ra * ca; z[1] = ra * sa; z[2] = rb * cb; z[3] = rb * sb;
}
__device__ inline float philox_uniform(uint32_t chain, uint32_t iter, uint32_t stream, uint64_t seed) {
  uint32_t r[4];
  philox4x32_10(0u, chain, iter, stream, (uint32_t)seed, (uint32_t)(seed >> 32), r);
  return (float)(r[0] >> 8) * 5.9604644775390625e-08f;
}

__device__ inline float warp_sum(float v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  return v;
}
__device__ inline double warp_sum(double v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  return v;
}
// block-wide sum; result valid in thread 0 (all threads must call). scratch >= 32 entries.
template <typename T>
__device__ inline T block_sum(T v, T* scratch) {
  int lane = threadIdx.x & 31, w = threadIdx.x >> 5;
  v = warp_sum(v);
  __syncthreads();
  if (lane == 0) scratch[w] = v;
  __syncthreads();
  int nw = (blockDim.x + 31) >> 5;
  T r = (threadIdx.x < nw) ? scratch[threadIdx.x] : T(0);
  if (w == 0) r = warp_sum(r);
  return r;
}

// Dual averaging of one chain's step size (Hoffman & Gelman 2014, Algorithm 5, with Stan's constants), called from
// the Metropolis test of every adaptation iteration t = 1, 2, ... (k_accept, k_fs_hmc).  da = {log_eps, log_eps_bar,
// h_bar, mu}.  The recursion is rounded operation by operation (no contraction into FMAs), as a float64 restatement
// computes it.
constexpr double DA_GAMMA = 0.05, DA_T0 = 10.0, DA_KAPPA = 0.75;
__device__ inline void dual_average(double* da, double* step, float log_alpha, double target, int64_t t) {
  double a = exp((double)log_alpha);
  a = (a != a) ? 0.0 : fmin(1.0, a);          // a NaN Hamiltonian difference counts as a rejection
  const double td = (double)t, eta = 1.0 / (td + DA_T0);
  const double h_bar = __dadd_rn(__dmul_rn(1.0 - eta, da[2]), __dmul_rn(eta, target - a));
  const double log_eps = da[3] - __dmul_rn(sqrt(td) / DA_GAMMA, h_bar);
  const double w = pow(td, -DA_KAPPA);
  da[0] = log_eps;
  da[1] = __dadd_rn(__dmul_rn(w, log_eps), __dmul_rn(1.0 - w, da[1]));
  da[2] = h_bar;
  *step = exp(log_eps);
}

// classic Gelman-Rubin R-hat of element e from sums over S chains with T draws each: A = sum of all draws,
// M = sum_s (sum_t x)^2, Wss = within-chain sum of squares sum_s sum_t (x - m_s)^2:
//   W = Wss / (S (T-1)),  B/T = var_s(m_s) (ddof 1) = (M/T^2 - S mu^2) / (S-1),
//   V = (T-1)/T W + B/T,  R-hat = sqrt(V / W);  NaN when S < 2, T < 2 or W = 0 (or a sum is NaN)
__device__ inline double gelman_rubin(const double* A, const double* M, const double* Wss, int64_t e, double S,
                                      double T) {
  double r = NAN;
  if (S >= 2.0 && T >= 2.0) {
    const double W = Wss[e] / (S * (T - 1.0));
    const double mu = A[e] / (S * T);
    double bt = (M[e] / (T * T) - S * mu * mu) / (S - 1.0);
    if (bt < 0.0) bt = 0.0;
    if (W > 0.0) r = sqrt(((T - 1.0) / T * W + bt) / W);
  }
  return r;
}

__device__ inline float act_apply(float z, int act) {
  switch (act) {
    case PYB_ACT_RELU: return fmaxf(z, 0.0f);
    case PYB_ACT_TANH: return tanhf(z);
    case PYB_ACT_SIGMOID: return 1.0f / (1.0f + expf(-z));
    default: return z;
  }
}
// derivative through the activation OUTPUT (relu'(z) = 1[z>0] <=> 1[a>0])
__device__ inline float act_grad_from_output(float a, int act) {
  switch (act) {
    case PYB_ACT_RELU: return a > 0.0f ? 1.0f : 0.0f;
    case PYB_ACT_TANH: return 1.0f - a * a;
    case PYB_ACT_SIGMOID: return a * (1.0f - a);
    default: return 1.0f;
  }
}
#endif  // __CUDACC__

// ------------------------------------------------------------------------------------------
// handle
// ------------------------------------------------------------------------------------------
struct HmcState {
  bool inited = false;
  int64_t S = 0, chain_offset = 0;
  double eps = 0, m = 1;
  int L = 0, semantics = 0;
  uint64_t iter = 0;  // global iteration counter (RNG counter word)
  DevBuf<float> q, p, g, q0;
  DevBuf<float> gcur;           // loss gradient at the chain's current position (carried between iterations)
  bool have_cur = false;        // gcur / loss0 are valid for the current q
  DevBuf<float> inj_p, inj_u;
  bool have_inj_p = false, have_inj_u = false;
  // per-chain scalars
  DevBuf<float> loss, loss0, Up0, Up1, K0, K1, U0, U1, log_alpha, ret_loss;
  DevBuf<int32_t> accepted;
  DevBuf<double> partial_e, partial_k;  // [S, nblk] reduction scratch
  DevBuf<int32_t> pending_freq, slot_first, slot_acc;
  DevBuf<unsigned long long> counters;  // [0]=n_accepted [1]=n_total [2]=n_nan ; double sums after
  DevBuf<double> loss_sum;      // [1]
  // sample arena
  DevBuf<float> arena;          // [cap, P]
  DevBuf<int32_t> arena_freq, arena_chain, last_idx, arena_count;
  int64_t arena_cap = 0;
  int64_t arena_used_upper = 0;  // host-side upper bound of arena_count
  std::vector<float> host_samples;
  std::vector<int32_t> host_freq, host_chain;
  std::vector<int64_t> host_last_idx;   // per chain: index into host arrays of its last sample (-1: none)
  bool sampling_started = false;  // a sampling iteration has run since pyb_hmc_init / pyb_hmc_reset_samples
  // per-chain step sizes (pyb_hmc_set_step_sizes, pyb_hmc_adapt_begin); unallocated: every chain uses eps
  DevBuf<double> step;          // [S]
  DevBuf<double> da;            // [S, 4] dual-averaging state {log_eps, log_eps_bar, h_bar, mu} while adapting
  bool adapting = false;
  int64_t adapt_t = 0;          // adaptation iterations run since pyb_hmc_adapt_begin
  double adapt_target = 0;
  // parallel tempering (pyb_hmc_set_temperatures): local chain s = g R + r is rung r of replica group g; R = 0: off
  int R = 0;
  std::vector<double> ladder;   // [R] inverse temperatures, ladder[0] = 1
  DevBuf<float> beta;           // [S] (float) inverse temperature of every chain's rung
  DevBuf<double> ladder_d;      // [R] the ladder in double (swap ratios)
  DevBuf<float> swap_logr;      // [S] log ratio of the swap proposed with the upper neighbour (NaN: none)
  DevBuf<int32_t> swapped;      // [S] that swap was taken
  DevBuf<int32_t> moved;        // [S] the position changed in this iteration: HMC accept or swap
  DevBuf<unsigned long long> tcount;   // [4 R]: rung accepted, rung total, swaps attempted, swaps accepted
  DevBuf<float> cold;           // [S / R, P] rung-0 positions gathered for the tracked predictive
  bool swaps_ran = false;       // swap_logr / swapped hold an iteration's values
  // streamed posterior predictive (hmc_predictive.cu): the outputs o of every tracked draw on the tracked inputs
  struct Track {
    bool on = false;
    int64_t Nt = 0, chunk = 0;
    int64_t T = 0;              // draws per chain so far
    int64_t nch = 0;            // tracked chains: S, or the S / R rung-0 chains of a tempering ladder
    DevBuf<float> x;            // [Nt, in_dim] library-owned copy of the inputs
    DevBuf<int32_t> y;          // [Nt] labels (empty: none given)
    DevBuf<float> out;          // [chunk, Nt, C] forward outputs of one chain chunk
    DevBuf<float> shift;        // [S, Nt, C] each chain's first tracked draw
    DevBuf<double> s1c;         // [S, Nt, C] per chain: sum_t (o - shift)
    DevBuf<double> Q, Qd;       // [Nt, C] pooled sum o^2 and sum (o - shift)^2
    DevBuf<double> S2;          // [Nt, C, C] pooled sum o o^T (labels given and C > 1)
    DevBuf<double> part;        // [chain groups, 2, Nt, C] partial sums of one chunk
  } track;
  // streamed per-parameter moments (hmc_params.cu): the same draws as `track`, in weight space
  struct ParamTrack {
    bool on = false;
    int64_t T = 0;              // draws per chain so far
    int64_t nch = 0;            // tracked chains: S, or the S / R rung-0 chains of a tempering ladder
    int64_t n_planned = 0, half = 0, batch = 0;   // h = n_planned / 2 and the batch size b, fixed at the start
    int ngroups = 0;            // chain groups of the accumulation kernel (a function of nch and P)
    DevBuf<float> shift;        // [nch, P] each chain's first draw c
    DevBuf<double> d, hcur, bcur, bsum;   // [nch, P] per chain: sum_t (x - c), the current half's and batch's, sum of batches
    DevBuf<double> pool;        // [kParamPooled, P] pooled over chains (hmc_params.cu)
    DevBuf<double> part;        // [ngroups, kParamPooled, P] one draw's group partials
  } ptrack;
};

struct SvgdState {
  bool inited = false;
  int64_t S = 0, offset = 0;
  double lr = 0;
  int semantics = 0;
  int64_t t = 0;
  DevBuf<float> theta, g, adam_m, adam_v, phi, loss;
  DevBuf<double> d2, K, rowsum;
  DevBuf<unsigned long long> sel, hist, cand;   // radix-select state (2 x {prefix,mask,k}, next-greater, candidate count), 256-bin histogram, compacted candidates
  DevBuf<double> h2, mean_loss, Krow;
  // tensor-core Gram / Stein contraction operands (bf16 hi/lo kept as raw 16-bit words)
  DevBuf<uint16_t> xh, xl, yth, ytl, kh, kl;
  DevBuf<float> gram, ybuf, kf, norms;
  DevBuf<float> Xb;
  DevBuf<int32_t> yb_i, idx;
  DevBuf<float> yb_f;
  // held-out set for the per-step validation loss (SVGD.py:126-129), resident in HBM
  DevBuf<float> val_X, val_yf;
  DevBuf<int32_t> val_yi;
  int64_t val_N = 0;
  // comm
  int rank = 0, world = 1;
  void* nccl_comm = nullptr;
  void* nccl_comm2 = nullptr;   // duplicate for the gradient / particle exchanges (their own stream)
  void* nccl_comm3 = nullptr;   // duplicate for the Gram all-reduce and the median's histograms (side stream)
  DevBuf<float> theta_all, g_all;
  // parameter-sharded Stein phase (canonical mode, tensor path, world > 1): rank r owns columns [r Pw, (r+1) Pw) of ALL
  // particles — theta slice, gathered gradient slice, Adam moments, phi — and the exchange is two all-to-alls of the
  // LOCAL particles' rows (gradients out, updated particles back) plus one all-reduce of the St x St Gram matrix
  double last_h = 0.0;          // bandwidth h of the last step (canonical: sqrt(0.5 median / log(St + 1)); live: gamma = 1)
  bool ps_ready = false, ps_checked = false;
  int64_t ps_Pw = 0;
  DevBuf<float> ps_pack, ps_x, ps_g, ps_m, ps_v, ps_phi, ps_mu, ps_iv;
  DevBuf<double> ps_norms;
  // "profile" option: CUDA events between the phases of the sharded step (gradients | gradient all-to-all | Gram partial |
  // Gram all-reduce | median + kernel | K Y + Adam | particle all-to-all), milliseconds of the last step
  cudaEvent_t ps_ev[8] = {nullptr, nullptr, nullptr, nullptr, nullptr, nullptr, nullptr, nullptr};
  float ps_ms[7] = {0, 0, 0, 0, 0, 0, 0};
  bool ps_timed = false;
  // the two all-gathers run on their own stream: particles while the local gradients are computed, gradients
  // while the Gram matrix is built (SURVEY 8e: the exchange step is comm-bound at 8 GPUs unless overlapped)
  cudaStream_t comm_stream = nullptr;
  cudaEvent_t ev_fork = nullptr, ev_theta = nullptr, ev_grad = nullptr;
  // peer memory (NVLink): the gradient rows are written straight into every rank's gradient slice and the updated
  // particle blocks straight into their owners' particle rows by this library's own kernels; NCCL only carries the
  // one-float barrier after each of them.  Pointers: CUDA IPC between processes, plain peer access inside one process.
  bool p2p_tried = false, p2p_ready = false;
  const float* p2p_src_theta = nullptr; const float* p2p_src_g = nullptr;   // the allocations the tables were built for
  std::vector<void*> p2p_opened;          // cudaIpcOpenMemHandle mappings to close
  DevBuf<float*> p2p_theta, p2p_g;        // [world] device tables: rank q's particle rows / gradient slice
  std::vector<float*> p2p_theta_host;
  DevBuf<float> p2p_token;
  cudaStream_t gram_stream = nullptr;     // parameter-sharded step: reduction / median / kernel-matrix chain beside the gradients
  cudaEvent_t ev_kernel = nullptr, ev_gh[2] = {nullptr, nullptr}, ev_p1 = nullptr, ev_p2 = nullptr, ev_back = nullptr;
};

// S stochastic-gradient chains (sgmc.cu): SGLD / SWAG state per chain
struct SgState {
  bool inited = false;
  int kind = 0, k = 0, freq = 1, cols = 0;
  int64_t S = 0, offset = 0, n = 0;
  DevBuf<float> theta, g, mean, sq, dev, loss;   // dev [S, k, P]: column c of chain s is contiguous
  DevBuf<double> mean_loss;
  DevBuf<float> Xb, yb_f;
  DevBuf<int32_t> yb_i, idx;
};

struct Workspace {
  // generic-path activations for a chain batch: act[l] = [Bc, N, width_l], dz ping-pong
  std::vector<DevBuf<float>*> act;
  DevBuf<float> dz_a, dz_b;
  DevBuf<float> partial;  // split-K partials
  DevBuf<double> loss_partial;
  int64_t Bc = 0, N = 0;
};

}  // namespace pyb

struct pyb_handle {
  int device = 0;
  int sm_count = 148;
  uint64_t seed = 0;
  cudaStream_t stream = nullptr;
  cudaEvent_t ev0 = nullptr, ev1 = nullptr;
  pyb::Model model;
  // dataset
  int64_t N = 0, n_train = 0;
  int loss_kind = 0;
  pyb::DevBuf<float> X, y_f;
  pyb::DevBuf<int32_t> y_i;
  bool have_data = false;
  pyb::DevBuf<float> X_stage, yf_stage;   // incoming copy of a re-submitted dataset: compared on the device with the resident one
  pyb::DevBuf<int32_t> yi_stage, flag;
  int64_t dataset_uploads = 0, dataset_kept = 0;   // pyb_set_dataset calls / calls whose data equalled the resident copy
  // prior (per element) + derived
  pyb::DevBuf<float> mu, sigma, inv_var;
  bool have_prior = false;
  double prior_const = 0;  // sum_i log sigma_i + P/2 log 2pi (NaN when any sigma<0, as tfp's log_prob)
  // options
  int opt_path = PYB_PATH_AUTO;
  int opt_tc_pair = 1;   // 1: use the CTA-pair (cta_group::2) GEMM kernel where it applies
  int opt_tc_dual = 1;   // 1: the hidden-major dW1 GEMM computes two feature tiles per item (shared A stages)
  int opt_tc_h128_pairs = 1;   // 1: 128-unit hidden layers use the dual hidden-major dW1 GEMM with two chains per CTA pair
  int opt_tc_gram_sym = 1;   // 1: Gram matrices (A == B) compute the upper tile triangle only and mirror it
  int opt_fs_cluster = 1;   // 1: the small-width HMC kernel spreads a chain over a CTA cluster when there are few chains
  int opt_live_fused = 1;   // 1: the reference-live SVGD sweep is one cooperative launch on a single GPU
  int opt_hmc_carry = 1;    // 1: loss and gradient at the current position are carried to the next HMC iteration
  int opt_hmc_keep_samples = 1;   // 1: every tracked HMC draw is recorded (arena + host copy); 0: nothing is kept
  int opt_hmc_swap = 1;     // 1: a tempering ladder proposes replica swaps every iteration; 0: the rungs run side by side
  int opt_predict_sharded = 0;   // 1: pyb_predict all-reduces its moment sums over the handle's communicator
  int opt_tc_fuse = 1;   // 1: layer 2 (+ loss, dZ2, dZ1) runs inside the layer-1 GEMM's epilogue where it applies
  int opt_tc_timeline = 0;   // diagnostics: the fused mma kernel records per-CTA cycle sums of its phases (info "tc_timeline_<k>")
  int opt_tc_epi_mma = 0;    // 1: fused int8 forward kernel with the layer-2 epilogue on mma.sync (tc_fused_mma.cuh): parity green, no faster (DESIGN 6b)
  int opt_select_compact = 0;   // median radix select of a local set: 0 eight passes, two kernels each; 1 candidates compacted after two passes (pays only for spread-out distances: in high dimension they concentrate and the candidates are the whole set); 2 eight passes, the digit picked inside the next pass (half the kernels)
  int opt_svgd_chain_fused = 1; // parameter-sharded SVGD: the side chain with fused kernels (12 launches instead of 25)
  int opt_svgd_gram_sync = 0;   // parameter-sharded SVGD: 1 = the Gram all-reduce on the main stream (not beside the gradients)
  int opt_live_cta = 1;      // live SVGD sweep of a small problem (particles fit one CTA's shared memory) in one CTA, no grid barriers
  int opt_svgd_halves = 0;   // parameter-sharded SVGD: gradients in two halves, the first half's exchange behind the second
  int opt_svgd_p2p = 1;      // parameter-sharded SVGD: exchanges by peer-memory stores of our own kernels (0: NCCL send / recv)
  int opt_svgd_pshard = 1;   // sharded canonical SVGD on the tensor path: shard the Stein phase over the parameters (all-to-all + Gram all-reduce)
  // Guard of the automatic choice (tc_i8 = -1).  16-bit FIXED-point slices carry an error relative to the LARGEST operand
  // magnitude; the float64 comparison of tests/test_gpu_i8.py fits err(gradient) ~ 1.3e-5 / rms_rows(1 - p_y) (+ 3e-5 from
  // the W1 slices): inside the 1e-4 budget while the chains still misfit the data (random labels, early and typical
  // posterior states) and outside it for a nearly converged chain, whose deltas are heavy-tailed and whose gradient is a
  // small difference of large terms.  The library therefore watches the per-chain mean loss it hands back at the end of
  // every pyb_hmc_run / pyb_hmc_eval and uses the slices only while min_s loss_s >= opt_i8_min_loss; below it falls back
  // to bf16x3 (and re-evaluates a pyb_hmc_eval call that was answered with slices).  tc_i8 = 1 / 2 bypass the guard.
  bool i8_guard_ok = true;
  double opt_i8_min_loss = 0.35;
  int64_t i8_guard_trips = 0;
  int opt_tc_i8 = -1;    // operand split of the big GEMMs: 0 bf16x3, 1 int8 slices in the forward GEMM, 2 + in the dW1 GEMM, -1 auto (tc_i8.cuh)
  double opt_workspace_mb = 4096;
  int64_t opt_chain_batch = 0;
  int path_used = PYB_PATH_GENERIC;
  int fs_cluster_used = 0;  // CTAs per chain of the last small-width HMC launch (0 before the first)
  int64_t kernel_launches = 0;
  double last_device_ms = 0;
  pyb::Workspace ws;
  pyb::HmcState hmc;
  pyb::SvgdState svgd;
  pyb::SgState sg;
  // live per-kernel timing of the dominant (GEMM) kernels: CUDA events on the launching stream
  bool prof_enabled = false;
  std::vector<cudaEvent_t> prof_events;   // begin/end pairs, resolved by prof_resolve()
  size_t prof_used = 0;
  double prof_ms = 0, prof_flops = 0;
  int64_t prof_launches = 0;
  void* tc = nullptr;     // tensor-core path state (tc_path.cu)
  void* fused = nullptr;  // fused small path state
};

namespace pyb {
inline void count_launch(pyb_handle* h, int n = 1) { h->kernel_launches += n; }
// bracket ONE dominant-kernel launch with events (no-ops unless the "profile" option is on)
inline void prof_begin(pyb_handle* h) {
  if (!h->prof_enabled) return;
  if (h->prof_used + 2 > h->prof_events.size()) {
    cudaEvent_t a, b;
    cudaEventCreate(&a); cudaEventCreate(&b);
    h->prof_events.push_back(a); h->prof_events.push_back(b);
  }
  cudaEventRecord(h->prof_events[h->prof_used], h->stream);
}
inline void prof_end(pyb_handle* h, double flops) {
  // a launch-configuration error ("too many resources requested for launch", a bad cluster shape) is returned by the launch
  // itself and is LOST once a later runtime call succeeds (measured: the evaluation then continues on stale buffers), so
  // every dominant-kernel launch is checked here, right behind it
  PYB_CUDA(cudaGetLastError());
  if (!h->prof_enabled) return;
  cudaEventRecord(h->prof_events[h->prof_used + 1], h->stream);
  h->prof_used += 2;
  h->prof_flops += flops;
  h->prof_launches += 1;
}
// call after a stream sync: fold the recorded pairs into prof_ms
inline void prof_resolve(pyb_handle* h) {
  for (size_t i = 0; i + 1 < h->prof_used; i += 2) {
    float ms = 0.f;
    if (cudaEventElapsedTime(&ms, h->prof_events[i], h->prof_events[i + 1]) == cudaSuccess) h->prof_ms += ms;
  }
  h->prof_used = 0;
}

// generic_mlp.cu
// loss[S] (mean loss over the batch), grad[S,P] = scale * d(mean loss)/d(theta)  (grad may be null)
void generic_eval(pyb_handle* h, const float* theta, int64_t S, const float* X, const int32_t* y_i,
                  const float* y_f, int64_t N, float scale, float* loss_out, float* grad_out);
// forward only: out [S, N, out_dim] (softmax applied when the last activation is softmax)
void generic_forward(pyb_handle* h, const float* theta, int64_t S, const float* X, int64_t N, float* out);
int64_t generic_chain_batch(pyb_handle* h, int64_t S, int64_t N, bool backward);

// dispatcher (api.cu): picks generic / fused-small / tensor path
void eval_loss_grad(pyb_handle* h, const float* theta, int64_t S, float scale, float* loss_out, float* grad_out);
int resolve_path(pyb_handle* h, int64_t S, bool with_grad);
bool fused_small_supported(pyb_handle* h);
void fused_small_hmc_iteration(pyb_handle* h, bool burning);
void fused_small_eval_on(pyb_handle* h, const float* theta, int64_t S, const float* Xb, const int32_t* yb_i,
                         const float* yb_f, int64_t Nb, float scale, float* loss, float* grad);

// tc_path.cu
bool tc_supported_rows(pyb_handle* h, int64_t n_rows);
void tc_eval_batch(pyb_handle* h, const float* Xb, const int32_t* yb_i, const float* yb_f, int64_t Nb, const float* theta,
                   int64_t S, float scale, float* loss_out, float* grad_out);
void tc_forward(pyb_handle* h, const float* theta, int64_t S, const float* x, int64_t N, float* out);
void tc_forward_tracked(pyb_handle* h, const float* theta, int64_t S, const float* x, int64_t N, float* out);
void tc_invalidate_track(pyb_handle* h);
void gather_rows_f32(pyb_handle* h, const float* src, const int64_t* idx_host, int64_t n, int64_t row_len, float* dst);
void tc_split_rows(pyb_handle* h, const float* src, int64_t R, int C, int64_t lds, void* hi, void* lo, int64_t ldd);
void tc_split_transpose(pyb_handle* h, const float* src, int R, int C, int64_t lds, void* hi, void* lo, int64_t ldd);
void tc_gemm_split(pyb_handle* h, const void* a_hi, const void* a_lo, int64_t lda, int64_t a_rows_total, int a_row0, int M,
                   const void* b_hi, const void* b_lo, int64_t ldb, int Nn, int64_t K, float* out, int64_t ldc);
// loss + gradient on an arbitrary device-resident batch (api.cu): tensor path when the shape allows, else generic
void eval_on_batch(pyb_handle* h, const float* theta, int64_t S, const float* Xb, const int32_t* yb_i, const float* yb_f,
                   int64_t Nb, float scale, float* loss_out, float* grad_out);

// sampler.cu
void hmc_init(pyb_handle* h, int64_t S, int64_t chain_offset, double eps, double m, int L, int sem, const float* q0);
void hmc_run(pyb_handle* h, int n_iters, bool burning, bool sampling, pyb_hmc_diag* out);
void hmc_eval(pyb_handle* h, const float* q, int64_t S, float* U, float* loss, float* grad);
void hmc_flush_arena(pyb_handle* h);
void hmc_adapt_begin(pyb_handle* h, double target);
void hmc_adapt_end(pyb_handle* h);
void hmc_step_sizes(pyb_handle* h, double* out);
void hmc_set_step_sizes(pyb_handle* h, const double* eps);
void hmc_set_temperatures(pyb_handle* h, const double* beta, int R);
void hmc_tempering_stats(pyb_handle* h, int64_t* rung_acc, int64_t* rung_tot, int64_t* swap_att, int64_t* swap_acc);
void hmc_last_swaps(pyb_handle* h, float* log_r, int32_t* swapped);

// svgd.cu
void svgd_init(pyb_handle* h, int64_t S, int64_t offset, double lr, int sem, const double* p0);
void svgd_step(pyb_handle* h, const int32_t* idx, int64_t B, double* loss_out);
void svgd_phi(pyb_handle* h, const double* X, const float* G, int64_t S, int sem, float* phi, double* h_out);
void svgd_set_validation(pyb_handle* h, const float* X, const void* y, int64_t N);
void svgd_validation_loss(pyb_handle* h, double* mean_loss_out, float* per_particle_out);

// rows idx[0..B) of the resident dataset gathered into a contiguous minibatch (device index list)
void gather_batch(pyb_handle* h, const int32_t* idx_dev, int64_t B, float* Xb, int32_t* yb_i, float* yb_f);

// sgmc.cu
void sg_init(pyb_handle* h, int64_t S, int64_t chain_offset, int kind, int k_dev, int frequency, const float* theta0,
             int theta0_rows);
void sg_step(pyb_handle* h, const int32_t* idx, int64_t B, double lr, const float* noise, float* loss_out,
             double* mean_loss_out);
void sg_get(pyb_handle* h, float* theta, float* mean, float* sq, float* dev, int32_t* n_cols, int64_t* n_steps);

// nccl_shim.cu (NCCL resolved with dlopen; only sharded SVGD uses it)
void nccl_unique_id(void* out_128);
void* nccl_comm_init(int rank, int world, const void* id_128);
void nccl_comm_destroy(void* comm);
void nccl_all_gather_f32(void* comm, const float* send, float* recv, size_t count_per_rank, cudaStream_t s);
void nccl_all_reduce_u64(void* comm, unsigned long long* buf, size_t count, cudaStream_t s);
void nccl_all_reduce_f64(void* comm, double* buf, size_t count, cudaStream_t s);
void nccl_broadcast_f32(void* comm, float* buf, size_t count, int root, cudaStream_t s);
void nccl_all_reduce_f32(void* comm, float* buf, size_t count, cudaStream_t s);
void nccl_all_to_all_f32(void* comm, const float* send, float* recv, size_t count_per_peer, int world, cudaStream_t s);
void nccl_check_async(void** comm);
void nccl_all_reduce_min_u64(void* comm, unsigned long long* buf, size_t count, cudaStream_t s);
void* nccl_comm_dup(void* comm, int rank);
void svgd_p2p_release(pyb_handle* h);
void nccl_all_to_all_f32_strided(void* comm, const float* send, size_t send_stride, float* recv, size_t recv_stride,
                                 size_t count, int world, cudaStream_t s);
void nccl_exchange_f32(void* comm, const float* send, float* recv, size_t stride, size_t count, const int* send_to, int n_send,
                       const int* recv_from, int n_recv, cudaStream_t s);

// predict.cu
// optional classification-uncertainty request (Metrics.py:344-375): host labels [Nt], host outputs [Nt, Ce, Ce]
struct UncertaintyReq {
  const int32_t* y;
  int cumulative;     // 1: reference semantics (running sum over the rows, broadcast epistemic term); 0: canonical per-row matrices
  double divisor;     // the reference divides by its n_samples ARGUMENT (Metrics.py:368-369)
  float *total, *aleatoric, *epistemic;
};
void predict(pyb_handle* h, const float* W, int64_t n, const float* weight, const float* x, int64_t Nt,
             float* mean, float* var, float* all, const UncertaintyReq* uq = nullptr);
void predictive_finish(pyb_handle* h, const double* s1, const double* s2, const double* S2, double wsum, int64_t Nt,
                       const int32_t* y_dev, const UncertaintyReq* uq, float* mean, float* var);
// S2 += sum_k w_k o_k o_k^T over a chunk of outputs [nb, Nt, C] (w NULL: 1)
void uncert_s2_accum(pyb_handle* h, const float* out, int64_t nb, int64_t Nt, int C, const float* w, double* S2);
bool is_device_ptr(const void* ptr);

// hmc_predictive.cu
void hmc_track_start(pyb_handle* h, const float* x, int64_t Nt, const int32_t* y);
void hmc_track_stop(pyb_handle* h);
void hmc_track_clear(pyb_handle* h);
void hmc_track_draw(pyb_handle* h, const float* q, int64_t n);
void hmc_track_resize(pyb_handle* h);
void hmc_track_sums(pyb_handle* h, double* sums, double* s2, int64_t* n_draws);
void hmc_track_finish(pyb_handle* h, const double* sums, const double* s2, int64_t n_chains, int64_t n_draws,
                      const UncertaintyReq* uq, float* mean, float* var, float* rhat);

// hmc_params.cu
void hmc_params_start(pyb_handle* h, int64_t n_planned, int64_t batch);
void hmc_params_stop(pyb_handle* h);
void hmc_params_clear(pyb_handle* h);
void hmc_params_resize(pyb_handle* h);
void hmc_params_draw(pyb_handle* h);
void hmc_params_sums(pyb_handle* h, double* sums, int64_t* n_draws);
void hmc_params_finish(pyb_handle* h, const double* sums, int64_t n_chains, int64_t n_draws, int64_t n_planned,
                       int64_t batch, double* mean, double* sd, double* rhat, double* ess, double* mcse);
size_t hmc_params_bytes(const pyb_handle* h);
}  // namespace pyb
