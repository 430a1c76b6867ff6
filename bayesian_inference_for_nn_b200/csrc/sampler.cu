// sampler.cu — HMC for S chains at once: momentum draw (Philox), kinetic/potential energy,
// leapfrog kick/drift, Metropolis accept, sample + frequency bookkeeping.  No host sync inside an
// iteration (the reference syncs twice per iteration: HMC.py:91 and the progress print :113-125).
//
// Reference: HMC.step HMC.py:74-104; _step_p :128-136; _step_q :138-141; _potential_energy
// :149-159; _kinetic_energy :161-166; _sample_kinetic_energy :168-171; result :176-187.
#include "common.cuh"
#include <math.h>
#include <string.h>
#include <algorithm>

namespace pyb {

constexpr int EW_THREADS = 256;
constexpr int EW_PER_THREAD = 4;
constexpr int EW_CHUNK = EW_THREADS * EW_PER_THREAD;  // elements of one chain handled by one block

static inline int ew_blocks(int64_t P) { return (int)((P + EW_CHUNK - 1) / EW_CHUNK); }
// chains ride on grid.y/grid.z (grid.y alone stops at 65535)
constexpr int CHAIN_Y = 32768;
static inline dim3 chain_grid(int nblk, int64_t S) {
  return dim3((unsigned)nblk, (unsigned)std::min<int64_t>(S, CHAIN_Y), (unsigned)((S + CHAIN_Y - 1) / CHAIN_Y));
}
__device__ __forceinline__ int64_t chain_index() { return (int64_t)blockIdx.z * gridDim.y + blockIdx.y; }

__global__ void k_init_q(float* q, const float* q0, const float* mu, int64_t P, int64_t S) {
  int64_t s = chain_index();
  if (s >= S) return;
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < P; i += (int64_t)gridDim.x * blockDim.x)
    q[s * P + i] = q0 ? q0[s * P + i] : mu[i];
}

// p = std * N(0,1) (or injected); partial[s][blk] = sum p^2 over the block's chunk
__global__ void __launch_bounds__(EW_THREADS) k_momentum(float* p, const float* inj, int64_t P, float stdv,
                                                          uint64_t seed, uint32_t iter, int64_t chain_offset,
                                                          double* partial, int64_t S) {
  __shared__ double scratch[32];
  int64_t s = chain_index();
  if (s >= S) return;
  int64_t base = (int64_t)blockIdx.x * EW_CHUNK + (int64_t)threadIdx.x * EW_PER_THREAD;
  double acc = 0.0;
  if (base < P) {
    float z[4];
    if (inj) {
#pragma unroll
      for (int j = 0; j < 4; ++j) z[j] = (base + j < P) ? inj[s * P + base + j] : 0.f;
    } else {
      philox_normal4((uint32_t)(base >> 2), (uint32_t)(chain_offset + s), iter, STREAM_MOMENTUM, seed, z);
#pragma unroll
      for (int j = 0; j < 4; ++j) z[j] *= stdv;
    }
#pragma unroll
    for (int j = 0; j < 4; ++j)
      if (base + j < P) {
        p[s * P + base + j] = z[j];
        acc += (double)z[j] * (double)z[j];
      }
  }
  double tot = block_sum<double>(acc, scratch);
  if (threadIdx.x == 0) partial[s * gridDim.x + blockIdx.x] = tot;
}

// out[s] = scale * sum_blk partial[s][blk]   (fixed order => deterministic)
__global__ void k_finish(const double* partial, int nblk, double scale, float* out) {
  __shared__ double scratch[32];
  int64_t s = blockIdx.x;
  double a = 0.0;
  for (int i = threadIdx.x; i < nblk; i += blockDim.x) a += partial[s * nblk + i];
  double tot = block_sum<double>(a, scratch);
  if (threadIdx.x == 0) out[s] = (float)(tot * scale);
}

// Fused leapfrog element pass after one position evaluation:
//   gtot = g + (q-mu)/sigma^2                      (dU/dq, HMC.py:132-135)
//   [energy]   partial_e += 1/2 ((q-mu)/sigma)^2   (prior part of U at the CURRENT q, HMC.py:152-154)
//   [snapshot] q0 = q                              (HMC.py:81)
//   p -= kick1*gtot ; p -= kick2*gtot (kick2==0: skipped; two roundings, as the reference's two
//                                      separate _step_p calls at q_L, HMC.py:86-87)
//   [kinetic]  partial_k += p^2                    (HMC.py:161-166)
//   q += drift*p   (drift==0: skipped)             (HMC.py:138-141)
// The coefficients are the scalars kick1 / kick2 / drift, or, with per-chain step sizes (step != NULL), those of the
// block's chain for the leapfrog position `role`.  With a tempering ladder (beta != NULL) the data gradient g is scaled
// by the chain's inverse temperature first: gtot = beta g + (q-mu)/sigma^2 (beta = 1 rounds exactly as without).
enum KickRole {
  KICK_HALF_DRIFT,   // first half kick + drift (HMC.py:82-83)
  KICK_FULL_DRIFT,   // full kick + drift (:84-85)
  KICK_FULL_HALF,    // L-th full kick + trailing half kick, reference semantics (:85-87)
  KICK_HALF          // trailing half kick, canonical semantics
};
__host__ __device__ inline void kick_coefs(int role, const StepCoef& c, float& kick1, float& kick2, float& drift) {
  kick1 = (role == KICK_HALF_DRIFT || role == KICK_HALF) ? c.half : c.eps;
  kick2 = role == KICK_FULL_HALF ? c.half : 0.f;
  drift = (role == KICK_HALF_DRIFT || role == KICK_FULL_DRIFT) ? c.drift : 0.f;
}
struct KickArgs {
  float* q; float* p; const float* g; float* q0;
  const float* mu; const float* inv_var;
  int64_t P, S;
  float kick1, kick2, drift;
  const double* step; double m; int role;
  const float* beta;
  int snapshot, energy, kinetic;
  double* partial_e; double* partial_k;
};
__global__ void __launch_bounds__(EW_THREADS) k_kick_drift(KickArgs a) {
  __shared__ double scratch[32];
  int64_t s = chain_index();
  if (s >= a.S) return;
  if (a.step) kick_coefs(a.role, step_coef(a.step[s], a.m), a.kick1, a.kick2, a.drift);
  const float b = a.beta ? a.beta[s] : 1.f;
  int64_t base = (int64_t)blockIdx.x * EW_CHUNK + threadIdx.x;
  double e = 0.0, k = 0.0;
#pragma unroll
  for (int j = 0; j < EW_PER_THREAD; ++j) {
    int64_t i = base + (int64_t)j * EW_THREADS;
    if (i < a.P) {
      int64_t o = s * a.P + i;
      float q = a.q[o], p = a.p[o];
      float d = q - a.mu[i];
      float iv = a.inv_var[i];
      float gt = __fmul_rn(b, a.g[o]) + d * iv;
      if (a.energy) e += 0.5 * (double)(d * d * iv);
      if (a.snapshot) a.q0[o] = q;
      p = p - a.kick1 * gt;
      if (a.kick2 != 0.f) p = p - a.kick2 * gt;
      if (a.kinetic) k += (double)p * (double)p;
      a.p[o] = p;
      if (a.drift != 0.f) a.q[o] = q + a.drift * p;
    }
  }
  if (a.energy) {
    double t = block_sum<double>(e, scratch);
    if (threadIdx.x == 0) a.partial_e[s * gridDim.x + blockIdx.x] = t;
  }
  if (a.kinetic) {
    double t = block_sum<double>(k, scratch);
    if (threadIdx.x == 0) a.partial_k[s * gridDim.x + blockIdx.x] = t;
  }
}

// prior energy partial + total gradient (parity hook pyb_hmc_eval)
__global__ void __launch_bounds__(EW_THREADS) k_prior(const float* q, float* g, const float* mu,
                                                       const float* inv_var, int64_t P, double* partial_e, int64_t S) {
  __shared__ double scratch[32];
  int64_t s = chain_index();
  if (s >= S) return;
  int64_t base = (int64_t)blockIdx.x * EW_CHUNK + threadIdx.x;
  double e = 0.0;
#pragma unroll
  for (int j = 0; j < EW_PER_THREAD; ++j) {
    int64_t i = base + (int64_t)j * EW_THREADS;
    if (i < P) {
      int64_t o = s * P + i;
      float d = q[o] - mu[i], iv = inv_var[i];
      e += 0.5 * (double)(d * d * iv);
      if (g) g[o] += d * iv;
    }
  }
  double t = block_sum<double>(e, scratch);
  if (threadIdx.x == 0) partial_e[s * gridDim.x + blockIdx.x] = t;
}

__global__ void k_potential(const float* Up, const float* loss, float prior_const, float n_train, float* U,
                            int64_t S) {
  int64_t s = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (s < S) U[s] = (Up[s] + prior_const) + loss[s] * n_train;
}

// Metropolis test (HMC.py:91): accept iff burning or u < exp(K0+U0-K1-U1); NaN => reject.  With a tempering ladder
// (beta != NULL) the data term of U is the chain's beta times the mean loss times n_train; ret_loss stays untempered.
struct AcceptArgs {
  const float* Up0; const float* Up1; const float* loss0; const float* loss1; const float* K0; const float* K1;
  float prior_const, n_train;
  const float* inj_u;
  uint64_t seed; uint32_t iter; int64_t chain_offset; int64_t S;
  int burning;
  float* U0; float* U1; float* log_alpha; int32_t* accepted; float* ret_loss;
  unsigned long long* counters; double* loss_sum;
  double* da; double* step; double da_target; int64_t da_t;   // da != NULL: adaptation iteration da_t (dual_average)
  const float* beta;
};
__global__ void k_accept(AcceptArgs a) {
  __shared__ double scratch[32];
  int64_t s = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  double ls = 0.0;
  int acc = 0, isnan_ = 0;
  if (s < a.S) {
    float l0 = a.loss0[s], l1 = a.loss1[s];
    if (a.beta) { l0 = __fmul_rn(a.beta[s], l0); l1 = __fmul_rn(a.beta[s], l1); }
    float U0 = (a.Up0[s] + a.prior_const) + l0 * a.n_train;
    float U1 = (a.Up1[s] + a.prior_const) + l1 * a.n_train;
    float la = ((a.K0[s] + U0) - a.K1[s]) - U1;
    float alpha = expf(la);
    float u = a.inj_u ? a.inj_u[s] : philox_uniform((uint32_t)(a.chain_offset + s), a.iter, STREAM_UNIFORM, a.seed);
    acc = a.burning ? 1 : ((u < alpha) ? 1 : 0);
    isnan_ = (la != la) ? 1 : 0;
    a.U0[s] = U0; a.U1[s] = U1; a.log_alpha[s] = la; a.accepted[s] = acc;
    if (a.da) dual_average(a.da + 4 * s, a.step + s, la, a.da_target, a.da_t);
    float rl = acc ? a.loss1[s] : a.loss0[s];
    a.ret_loss[s] = rl;
    ls = (double)rl;
  }
  // integer counters: exact and order-independent
  unsigned m_acc = __ballot_sync(0xffffffffu, acc), m_nan = __ballot_sync(0xffffffffu, isnan_),
           m_all = __ballot_sync(0xffffffffu, s < a.S);
  if ((threadIdx.x & 31) == 0) {
    if (m_acc) atomicAdd(&a.counters[0], (unsigned long long)__popc(m_acc));
    if (m_all) atomicAdd(&a.counters[1], (unsigned long long)__popc(m_all));
    if (m_nan) atomicAdd(&a.counters[2], (unsigned long long)__popc(m_nan));
  }
  double t = block_sum<double>(ls, scratch);
  if (threadIdx.x == 0) atomicAdd(a.loss_sum, t);
}

// Sample bookkeeping (HMC.py:75-77, 92-96, 103): single block; slot order = chain order, so the
// arena layout is deterministic.  first!=0: every chain first records its pre-iteration state
// with frequency 1.  The recording chains are s = k stride, k < S (stride R: the rung-0 chains of a tempering ladder,
// with accepted = "moved": HMC accept or swap).
__global__ void __launch_bounds__(1024) k_record_slots(const int32_t* accepted, int64_t S, int first,
                                                        int32_t* arena_count, int32_t* arena_freq,
                                                        int32_t* arena_chain, int32_t* last_idx,
                                                        int32_t* pending_freq, int32_t* slot_first,
                                                        int32_t* slot_acc, int64_t chain_offset, int64_t stride) {
  __shared__ int tot[1024];
  const int t = threadIdx.x;
  const int64_t cpt = (S + blockDim.x - 1) / blockDim.x;
  const int64_t lo = (int64_t)t * cpt, hi = (lo + cpt < S) ? lo + cpt : S;
  int need = 0;
  for (int64_t k = lo; k < hi; ++k) need += (first ? 1 : 0) + (accepted[k * stride] ? 1 : 0);
  tot[t] = need;
  __syncthreads();
  // Hillis-Steele inclusive scan over the 1024 per-thread totals
  for (int o = 1; o < (int)blockDim.x; o <<= 1) {
    int v = (t >= o) ? tot[t - o] : 0;
    __syncthreads();
    tot[t] += v;
    __syncthreads();
  }
  int slot = *arena_count + tot[t] - need;
  for (int64_t k = lo; k < hi; ++k) {
    const int64_t s = k * stride;
    int sf = -1, sa = -1;
    if (first) {
      sf = slot++;
      arena_freq[sf] = 1;
      arena_chain[sf] = (int32_t)(chain_offset + s);
      last_idx[s] = sf;
    }
    if (accepted[s]) {
      sa = slot++;
      arena_freq[sa] = 1;
      arena_chain[sa] = (int32_t)(chain_offset + s);
      last_idx[s] = sa;
    } else {
      int li = last_idx[s];
      if (li >= 0) arena_freq[li] += 1; else pending_freq[s] += 1;
    }
    slot_first[s] = sf;
    slot_acc[s] = sa;
  }
  __syncthreads();
  if (t == (int)blockDim.x - 1) *arena_count = *arena_count + tot[t];
}

// q = accepted ? q : q0 (HMC.py:97-101) and copy recorded samples into the arena
// gcur != nullptr: the loss gradient at the chain's CURRENT position is carried to the next iteration — an accepted
// chain takes the end-point gradient g (evaluated at q_L), a rejected one keeps the gradient it already has at q0
__global__ void __launch_bounds__(EW_THREADS) k_select_record(float* q, const float* q0, const int32_t* accepted,
                                                               const int32_t* slot_first, const int32_t* slot_acc,
                                                               float* arena, int64_t P, int sampling, int64_t S,
                                                               float* gcur, const float* g) {
  int64_t s = chain_index();
  if (s >= S) return;
  int acc = accepted[s];
  int sf = sampling ? slot_first[s] : -1, sa = sampling ? slot_acc[s] : -1;
  int64_t base = (int64_t)blockIdx.x * EW_CHUNK + threadIdx.x;
#pragma unroll
  for (int j = 0; j < EW_PER_THREAD; ++j) {
    int64_t i = base + (int64_t)j * EW_THREADS;
    if (i < P) {
      int64_t o = s * P + i;
      float old = q0[o];
      float cur = q[o];
      if (sf >= 0) arena[(int64_t)sf * P + i] = old;
      if (!acc) q[o] = old;
      if (sa >= 0) arena[(int64_t)sa * P + i] = cur;
      if (gcur && acc) gcur[o] = g[o];
    }
  }
}

// ------------------------------------------------------------------------------------------
// replica exchange (parallel tempering): one deterministic even-odd swap round per iteration (Syed, Bouchard-Cote,
// Deligiannidis & Doucet 2022).  Chain s = g R + r is rung r of group g; in iteration `iter` the pairs (r, r + 1) with
// r = iter (mod 2) of every group propose to exchange their states, accepted iff u < exp(log_r) with
//   log_r = (beta_r - beta_{r+1}) n_train (loss_r - loss_{r+1})   (double; NaN rejects)
// and u the Philox uniform of the lower chain's global id on STREAM_SWAP.
// ------------------------------------------------------------------------------------------
constexpr int kMaxRungs = 64;

// One thread per chain.  The lower chain of a proposed pair decides for the pair, exchanges the two untempered losses
// ret_loss (with carry on they become the carried losses) and writes both chains' "moved" flags; every chain reports
// the swap it proposed with its upper neighbour (log_r / swapped: NaN / 0 when none).  propose = 0 (option hmc_swap)
// keeps the rungs apart and only counts.  tcount [4 R] += per rung: HMC accepts, chains, swaps attempted / accepted
// (lower rung of the pair).
__global__ void __launch_bounds__(256) k_swap_decide(const double* ladder, int R, int propose, double n_train,
                                                      uint64_t seed, uint32_t iter, int64_t chain_offset, int64_t S,
                                                      const int32_t* accepted, float* ret_loss, float* log_r,
                                                      int32_t* swapped, int32_t* moved, unsigned long long* tcount) {
  __shared__ unsigned cnt[4 * kMaxRungs];
  for (int i = threadIdx.x; i < 4 * R; i += blockDim.x) cnt[i] = 0u;
  __syncthreads();
  const int64_t s = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (s < S) {
    const int r = (int)(s % R), par = (int)(iter & 1u);
    const bool lower = propose && r + 1 < R && (r & 1) == par;
    const bool upper = propose && r >= 1 && ((r - 1) & 1) == par;
    const int acc = accepted[s];
    float lr_out = NAN;
    int sw = 0;
    if (lower) {
      const float l0 = ret_loss[s], l1 = ret_loss[s + 1];
      const double lr = (ladder[r] - ladder[r + 1]) * n_train * ((double)l0 - (double)l1);
      const float u = philox_uniform((uint32_t)(chain_offset + s), iter, STREAM_SWAP, seed);
      sw = ((double)u < exp(lr)) ? 1 : 0;
      lr_out = (float)lr;
      if (sw) { ret_loss[s] = l1; ret_loss[s + 1] = l0; }
      moved[s] = acc | sw;
      moved[s + 1] = accepted[s + 1] | sw;
      atomicAdd(&cnt[2 * R + r], 1u);
      if (sw) atomicAdd(&cnt[3 * R + r], 1u);
    } else if (!upper) {
      moved[s] = acc;
    }
    log_r[s] = lr_out;
    swapped[s] = sw;
    if (acc) atomicAdd(&cnt[r], 1u);
    atomicAdd(&cnt[R + r], 1u);
  }
  __syncthreads();
  for (int i = threadIdx.x; i < 4 * R; i += blockDim.x)
    if (cnt[i]) atomicAdd(&tcount[i], (unsigned long long)cnt[i]);
}

// the accepted swaps: chains s (swapped[s]) and s + 1 exchange their positions and, with carry on, the loss gradients
// carried with them; momenta are redrawn every iteration and step sizes stay with the chain slot
__global__ void __launch_bounds__(EW_THREADS) k_swap_exchange(float* q, float* gcur, const int32_t* swapped, int64_t P,
                                                               int64_t S) {
  const int64_t s = chain_index();
  if (s >= S || !swapped[s]) return;
  const int64_t base = (int64_t)blockIdx.x * EW_CHUNK + threadIdx.x;
#pragma unroll
  for (int j = 0; j < EW_PER_THREAD; ++j) {
    const int64_t i = base + (int64_t)j * EW_THREADS;
    if (i < P) {
      const int64_t a = s * P + i, b = a + P;
      const float qa = q[a], qb = q[b];
      q[a] = qb; q[b] = qa;
      if (gcur) { const float ga = gcur[a], gb = gcur[b]; gcur[a] = gb; gcur[b] = ga; }
    }
  }
}

// arena rows of the rung-0 chains s = k R (k < G): the pre-iteration state q0 in the first sampling iteration, the
// position after the swap when the chain moved
__global__ void __launch_bounds__(EW_THREADS) k_record_cold(const float* q, const float* q0, const int32_t* slot_first,
                                                             const int32_t* slot_acc, float* arena, int64_t P, int64_t R,
                                                             int64_t G) {
  const int64_t k = chain_index();
  if (k >= G) return;
  const int64_t s = k * R;
  const int sf = slot_first[s], sa = slot_acc[s];
  if (sf < 0 && sa < 0) return;
  const int64_t base = (int64_t)blockIdx.x * EW_CHUNK + threadIdx.x;
#pragma unroll
  for (int j = 0; j < EW_PER_THREAD; ++j) {
    const int64_t i = base + (int64_t)j * EW_THREADS;
    if (i < P) {
      if (sf >= 0) arena[(int64_t)sf * P + i] = q0[s * P + i];
      if (sa >= 0) arena[(int64_t)sa * P + i] = q[s * P + i];
    }
  }
}

// ------------------------------------------------------------------------------------------
// host drivers
// ------------------------------------------------------------------------------------------
static void check_ready(pyb_handle* h) {
  PYB_REQUIRE(h->have_data, PYB_ERR_STATE, "pyb_set_dataset must be called first");
  PYB_REQUIRE(h->have_prior, PYB_ERR_STATE, "pyb_set_prior_gaussian must be called first");
}

void hmc_init(pyb_handle* h, int64_t S, int64_t chain_offset, double eps, double m, int L, int sem,
              const float* q0) {
  check_ready(h);
  PYB_REQUIRE(S > 0 && S <= 1048576, PYB_ERR_INVALID, "S must be in [1, 2^20]");
  PYB_REQUIRE(L >= 1, PYB_ERR_INVALID, "L must be >= 1");
  PYB_REQUIRE(m != 0.0, PYB_ERR_INVALID, "m must be non-zero");
  PYB_REQUIRE(sem == PYB_HMC_REFERENCE || sem == PYB_HMC_CANONICAL, PYB_ERR_INVALID, "bad semantics");
  HmcState& st = h->hmc;
  const int64_t P = h->model.P;
  st.S = S; st.chain_offset = chain_offset; st.eps = eps; st.m = m; st.L = L; st.semantics = sem;
  h->i8_guard_ok = (q0 == nullptr);   // the prior-mean start has loss log(C); supplied positions are unknown until evaluated
  st.iter = 0;
  st.q.alloc(S * P); st.p.alloc(S * P); st.g.alloc(S * P); st.q0.alloc(S * P);
  for (DevBuf<float>* b : {&st.loss, &st.loss0, &st.Up0, &st.Up1, &st.K0, &st.K1, &st.U0, &st.U1, &st.log_alpha,
                           &st.ret_loss})
    b->alloc(S);
  st.accepted.alloc(S);
  int nblk = ew_blocks(P);
  st.partial_e.alloc((size_t)S * nblk);
  st.partial_k.alloc((size_t)S * nblk);
  st.pending_freq.alloc(S); st.slot_first.alloc(S); st.slot_acc.alloc(S); st.last_idx.alloc(S);
  st.counters.alloc(4);
  st.loss_sum.alloc(1);
  st.arena_count.alloc(1);
  // sample arena: sized and allocated at the first SAMPLING iteration (hmc_size_arena), when the evaluation workspaces
  // already exist and the free memory is what it will be
  st.arena_cap = 0;
  st.arena.release(); st.arena_freq.release(); st.arena_chain.release();
  PYB_CUDA(cudaMemsetAsync(st.arena_count.p, 0, sizeof(int32_t), h->stream));
  PYB_CUDA(cudaMemsetAsync(st.pending_freq.p, 0, S * sizeof(int32_t), h->stream));
  PYB_CUDA(cudaMemsetAsync(st.last_idx.p, 0xff, S * sizeof(int32_t), h->stream));
  st.arena_used_upper = 0;
  st.host_samples.clear(); st.host_freq.clear(); st.host_chain.clear();
  st.host_last_idx.assign(S, -1);
  st.sampling_started = false;
  st.have_inj_p = st.have_inj_u = false;
  st.have_cur = false;
  st.adapting = false;
  st.adapt_t = 0;
  st.step.release(); st.da.release();
  st.R = 0; st.ladder.clear();        // pyb_hmc_init clears the tempering ladder
  st.beta.release(); st.ladder_d.release(); st.swap_logr.release(); st.swapped.release(); st.moved.release();
  st.tcount.release(); st.cold.release();
  st.swaps_ran = false;
  hmc_track_stop(h);
  hmc_params_stop(h);
  DevBuf<float> tmp;
  const float* q0d = nullptr;
  if (q0) {
    tmp.alloc(S * P);
    PYB_CUDA(cudaMemcpyAsync(tmp.p, q0, S * P * sizeof(float), cudaMemcpyHostToDevice, h->stream));
    q0d = tmp.p;
  }
  k_init_q<<<chain_grid((int)std::min<int64_t>((P + 255) / 256, 1024), S), 256, 0, h->stream>>>(st.q.p, q0d, h->mu.p, P, S);
  count_launch(h);
  PYB_CUDA(cudaStreamSynchronize(h->stream));
  st.inited = true;
}

// Sample arena [cap, P] on the device: 64 sampling iterations' worth of rows for every chain (a one-chain toy run keeps a
// few KB, not gigabytes), never more than a quarter of the memory that is free NOW (the tensor-path workspaces are
// allocated by then) nor 32 GiB, and at least the 2 S rows the first sampling iteration records; flushed to the host when full.
static void hmc_size_arena(pyb_handle* h) {
  HmcState& st = h->hmc;
  const int64_t P = h->model.P, S = st.S;
  size_t free_b = 0, total_b = 0;
  PYB_CUDA(cudaMemGetInfo(&free_b, &total_b));
  const size_t budget = std::min<size_t>(free_b / 4, (size_t)32 << 30);
  int64_t cap = (int64_t)(budget / (sizeof(float) * (size_t)P));
  cap = std::min<int64_t>(cap, 64 * S);
  cap = std::max<int64_t>(cap, 2 * S);
  cap = std::min<int64_t>(cap, 1ll << 30);
  st.arena_cap = cap;
  st.arena.alloc((size_t)cap * P);
  st.arena_freq.alloc(cap); st.arena_chain.alloc(cap);
}

void hmc_flush_arena(pyb_handle* h) {
  HmcState& st = h->hmc;
  const int64_t P = h->model.P, S = st.S;
  PYB_CUDA(cudaStreamSynchronize(h->stream));
  int32_t cnt = 0;
  PYB_CUDA(cudaMemcpy(&cnt, st.arena_count.p, sizeof(int32_t), cudaMemcpyDeviceToHost));
  std::vector<int32_t> pend(S), last(S);
  PYB_CUDA(cudaMemcpy(pend.data(), st.pending_freq.p, S * sizeof(int32_t), cudaMemcpyDeviceToHost));
  PYB_CUDA(cudaMemcpy(last.data(), st.last_idx.p, S * sizeof(int32_t), cudaMemcpyDeviceToHost));
  for (int64_t s = 0; s < S; ++s)
    if (pend[s] && st.host_last_idx[s] >= 0) st.host_freq[st.host_last_idx[s]] += pend[s];
  if (cnt > 0) {
    size_t base = st.host_freq.size();
    st.host_samples.resize((base + cnt) * (size_t)P);
    st.host_freq.resize(base + cnt);
    st.host_chain.resize(base + cnt);
    PYB_CUDA(cudaMemcpy(st.host_samples.data() + base * P, st.arena.p, (size_t)cnt * P * sizeof(float),
                        cudaMemcpyDeviceToHost));
    PYB_CUDA(cudaMemcpy(st.host_freq.data() + base, st.arena_freq.p, cnt * sizeof(int32_t), cudaMemcpyDeviceToHost));
    PYB_CUDA(cudaMemcpy(st.host_chain.data() + base, st.arena_chain.p, cnt * sizeof(int32_t), cudaMemcpyDeviceToHost));
    for (int64_t s = 0; s < S; ++s)
      if (last[s] >= 0) st.host_last_idx[s] = (int64_t)base + last[s];
  }
  PYB_CUDA(cudaMemset(st.arena_count.p, 0, sizeof(int32_t)));
  PYB_CUDA(cudaMemset(st.pending_freq.p, 0, S * sizeof(int32_t)));
  PYB_CUDA(cudaMemset(st.last_idx.p, 0xff, S * sizeof(int32_t)));
  st.arena_used_upper = 0;
}

static void launch_kick(pyb_handle* h, const float* g, KickRole role, bool snapshot, bool energy, bool kinetic,
                        float* Up_out, float* K_out) {
  NvtxRange nv("pyb.hmc.kick_drift");
  HmcState& st = h->hmc;
  const int64_t P = h->model.P;
  int nblk = ew_blocks(P);
  KickArgs a;
  a.q = st.q.p; a.p = st.p.p; a.g = g; a.q0 = st.q0.p; a.mu = h->mu.p; a.inv_var = h->inv_var.p; a.P = P; a.S = st.S;
  kick_coefs(role, step_coef(st.eps, st.m), a.kick1, a.kick2, a.drift);
  a.step = st.step.p; a.m = st.m; a.role = role;
  a.beta = st.R ? st.beta.p : nullptr;
  a.snapshot = snapshot; a.energy = energy; a.kinetic = kinetic;
  a.partial_e = st.partial_e.p; a.partial_k = st.partial_k.p;
  k_kick_drift<<<chain_grid(nblk, st.S), EW_THREADS, 0, h->stream>>>(a);
  count_launch(h);
  if (energy) { k_finish<<<(unsigned)st.S, 128, 0, h->stream>>>(st.partial_e.p, nblk, 1.0, Up_out); count_launch(h); }
  if (kinetic) {
    k_finish<<<(unsigned)st.S, 128, 0, h->stream>>>(st.partial_k.p, nblk, 1.0 / (2.0 * st.m), K_out);
    count_launch(h);
  }
}

// the int8-slice guard (common.cuh): smallest finite per-chain mean loss among `loss_dev[0..S)` against the threshold;
// the stream has been synchronised.  Returns whether the slices may be used from here on.
static bool update_i8_guard(pyb_handle* h, const float* loss_dev, int64_t S) {
  std::vector<float> l((size_t)S);
  PYB_CUDA(cudaMemcpy(l.data(), loss_dev, (size_t)S * sizeof(float), cudaMemcpyDeviceToHost));
  float mn = INFINITY;
  for (float v : l)
    if (isfinite(v)) mn = fminf(mn, v);
  const bool ok = !(mn < (float)h->opt_i8_min_loss);
  if (!ok && h->i8_guard_ok) h->i8_guard_trips += 1;
  h->i8_guard_ok = ok;
  return ok;
}

// one tracked draw of every chain at its current position; a ladder tracks its rung-0 chains (the parameter sums read
// them in place, the predictive gathers them into [G, P])
static void track_current(pyb_handle* h) {
  HmcState& st = h->hmc;
  const int64_t P = h->model.P;
  if (st.ptrack.on) hmc_params_draw(h);
  if (!st.track.on) return;
  if (!st.R) { hmc_track_draw(h, st.q.p, st.S); return; }
  const int64_t G = st.S / st.R;
  PYB_CUDA(cudaMemcpy2DAsync(st.cold.p, P * sizeof(float), st.q.p, st.R * P * sizeof(float), P * sizeof(float), G,
                             cudaMemcpyDeviceToDevice, h->stream));
  hmc_track_draw(h, st.cold.p, G);
}

// the end of a tempered iteration: restore the rejected chains (carrying the gradient of the accepted ones), one swap
// round, then the rung-0 chains record a draw wherever they moved (HMC accept or swap)
static void tempered_tail(pyb_handle* h, bool record, bool first, bool carry) {
  HmcState& st = h->hmc;
  const int64_t P = h->model.P, S = st.S, R = st.R, G = S / R;
  const int nblk = ew_blocks(P);
  k_select_record<<<chain_grid(nblk, S), EW_THREADS, 0, h->stream>>>(st.q.p, st.q0.p, st.accepted.p, st.slot_first.p,
                                                                     st.slot_acc.p, st.arena.p, P, 0, S,
                                                                     carry ? st.gcur.p : nullptr, st.g.p);
  const int propose = h->opt_hmc_swap ? 1 : 0;
  NvtxRange nv("pyb.hmc.swap");
  k_swap_decide<<<(unsigned)((S + 255) / 256), 256, 0, h->stream>>>(st.ladder_d.p, (int)R, propose, (double)h->n_train,
                                                                    h->seed, (uint32_t)st.iter, st.chain_offset, S,
                                                                    st.accepted.p, st.ret_loss.p, st.swap_logr.p,
                                                                    st.swapped.p, st.moved.p, st.tcount.p);
  count_launch(h, 2);
  if (propose) {
    k_swap_exchange<<<chain_grid(nblk, S), EW_THREADS, 0, h->stream>>>(st.q.p, carry ? st.gcur.p : nullptr,
                                                                       st.swapped.p, P, S);
    count_launch(h);
  }
  st.swaps_ran = true;
  if (record) {
    k_record_slots<<<1, 1024, 0, h->stream>>>(st.moved.p, G, first ? 1 : 0, st.arena_count.p, st.arena_freq.p,
                                              st.arena_chain.p, st.last_idx.p, st.pending_freq.p, st.slot_first.p,
                                              st.slot_acc.p, st.chain_offset, R);
    k_record_cold<<<chain_grid(nblk, G), EW_THREADS, 0, h->stream>>>(st.q.p, st.q0.p, st.slot_first.p, st.slot_acc.p,
                                                                     st.arena.p, P, R, G);
    count_launch(h, 2);
  }
}

void hmc_run(pyb_handle* h, int n_iters, bool burning, bool sampling, pyb_hmc_diag* out) {
  HmcState& st = h->hmc;
  PYB_REQUIRE(st.inited, PYB_ERR_STATE, "pyb_hmc_init must be called first");
  PYB_REQUIRE(n_iters >= 0, PYB_ERR_INVALID, "n_iters must be >= 0");
  PYB_REQUIRE(!(sampling && st.adapting), PYB_ERR_STATE,
              "no sampling while the step sizes adapt: call pyb_hmc_adapt_end first");
  const int64_t P = h->model.P, S = st.S;
  const int nblk = ew_blocks(P);
  const float n_train = (float)h->n_train;
  const float stdv = (st.semantics == PYB_HMC_REFERENCE) ? (float)st.m : (float)sqrt(st.m);
  int64_t launches0 = h->kernel_launches;
  PYB_CUDA(cudaMemsetAsync(st.counters.p, 0, 4 * sizeof(unsigned long long), h->stream));
  PYB_CUDA(cudaMemsetAsync(st.loss_sum.p, 0, sizeof(double), h->stream));
  if (st.R) PYB_CUDA(cudaMemsetAsync(st.tcount.p, 0, st.tcount.bytes(), h->stream));
  PYB_CUDA(cudaEventRecord(h->ev0, h->stream));
  const int path = resolve_path(h, S, true);
  int64_t evals = 0;
  if (path == PYB_PATH_FUSED_SMALL) { st.have_cur = false; evals = (int64_t)n_iters * S * (st.L + 1); }
  NvtxRange nv_run("pyb.hmc_run");
  for (int it = 0; it < n_iters; ++it) {
    NvtxRange nv_it("pyb.hmc.iteration");
    bool first = sampling && !st.sampling_started;
    const bool record = sampling && h->opt_hmc_keep_samples;   // keep the draws (arena), not only the tracked sums
    if (record) {
      int64_t need = (st.R ? S / st.R : S) * (first ? 2 : 1);    // a ladder records its rung-0 chains only
      if (!st.arena.p) hmc_size_arena(h);
      if (st.arena_used_upper + need > st.arena_cap) hmc_flush_arena(h);
      st.arena_used_upper += need;
    }
    const bool tracking = st.track.on || st.ptrack.on;
    if (first && tracking) track_current(h);        // the pre-iteration state is the first draw (HMC.py:75-77)
    if (st.adapting) st.adapt_t++;
    dim3 gridp = chain_grid(nblk, S);
    if (path == PYB_PATH_FUSED_SMALL) {
      PYB_REQUIRE(fused_small_supported(h), PYB_ERR_UNSUPPORTED, "fused small path does not support this model shape");
      fused_small_hmc_iteration(h, burning);     // whole iteration (momentum .. Metropolis test) in ONE launch
      h->path_used = path;
    } else {
    // momentum + K0  (HMC.py:78-79)
    nvtxRangePushA("pyb.hmc.momentum");
    k_momentum<<<gridp, EW_THREADS, 0, h->stream>>>(st.p.p, st.have_inj_p ? st.inj_p.p : nullptr, P, stdv, h->seed,
                                                    (uint32_t)st.iter, st.chain_offset, st.partial_k.p, S);
    count_launch(h);
    k_finish<<<(unsigned)S, 128, 0, h->stream>>>(st.partial_k.p, nblk, 1.0 / (2.0 * st.m), st.K0.p);
    count_launch(h);
    nvtxRangePop();
    // U0 and the first half kick share one evaluation at q0  (HMC.py:80-82).  The reference re-evaluates the
    // potential and its gradient at q0 in every iteration (HMC.py:80,82); q0 is where the previous iteration ended —
    // its end point q_L if that was accepted, its own q0 if not — and both were evaluated then, so with "hmc_carry"
    // the loss and the loss gradient at the current position travel with the chain (k_select_record / ret_loss):
    // L evaluations per iteration instead of L + 1, bit-identical results (every kernel is deterministic).
    if (!st.have_cur) {
      st.gcur.alloc(S * P);
      eval_loss_grad(h, st.q.p, S, n_train, st.loss0.p, st.gcur.p);
      evals += S;
    }
    launch_kick(h, st.gcur.p, KICK_HALF_DRIFT, true, true, false, st.Up0.p, nullptr);
    for (int i = 1; i <= st.L; ++i) {
      eval_loss_grad(h, st.q.p, S, n_train, st.loss.p, st.g.p);
      evals += S;
      if (i < st.L) {
        launch_kick(h, st.g.p, KICK_FULL_DRIFT, false, false, false, nullptr, nullptr);
      } else if (st.semantics == PYB_HMC_REFERENCE) {
        // L-th full kick and the trailing half kick, both with the gradient at q_L (HMC.py:85-87)
        launch_kick(h, st.g.p, KICK_FULL_HALF, false, true, true, st.Up1.p, st.K1.p);
      } else {
        launch_kick(h, st.g.p, KICK_HALF, false, true, true, st.Up1.p, st.K1.p);
      }
    }
    NvtxRange nv_acc("pyb.hmc.accept");
    AcceptArgs a;
    a.Up0 = st.Up0.p; a.Up1 = st.Up1.p; a.loss0 = st.loss0.p; a.loss1 = st.loss.p; a.K0 = st.K0.p; a.K1 = st.K1.p;
    a.prior_const = (float)h->prior_const; a.n_train = n_train;
    a.inj_u = st.have_inj_u ? st.inj_u.p : nullptr;
    a.seed = h->seed; a.iter = (uint32_t)st.iter; a.chain_offset = st.chain_offset; a.S = S;
    a.burning = burning ? 1 : 0;
    a.U0 = st.U0.p; a.U1 = st.U1.p; a.log_alpha = st.log_alpha.p; a.accepted = st.accepted.p;
    a.ret_loss = st.ret_loss.p; a.counters = st.counters.p; a.loss_sum = st.loss_sum.p;
    a.da = st.adapting ? st.da.p : nullptr; a.step = st.step.p; a.da_target = st.adapt_target; a.da_t = st.adapt_t;
    a.beta = st.R ? st.beta.p : nullptr;
    k_accept<<<(unsigned)((S + 255) / 256), 256, 0, h->stream>>>(a);
    count_launch(h);
    }
    const bool carry = h->opt_hmc_carry && path != PYB_PATH_FUSED_SMALL;
    if (st.R) {
      tempered_tail(h, record, first, carry);
    } else {
    if (record) {
      k_record_slots<<<1, 1024, 0, h->stream>>>(st.accepted.p, S, first ? 1 : 0, st.arena_count.p, st.arena_freq.p,
                                                st.arena_chain.p, st.last_idx.p, st.pending_freq.p,
                                                st.slot_first.p, st.slot_acc.p, st.chain_offset, 1);
      count_launch(h);
    }
    k_select_record<<<gridp, EW_THREADS, 0, h->stream>>>(st.q.p, st.q0.p, st.accepted.p, st.slot_first.p,
                                                         st.slot_acc.p, st.arena.p, P, record ? 1 : 0, S,
                                                         carry ? st.gcur.p : nullptr, st.g.p);
    count_launch(h);
    }
    if (sampling) st.sampling_started = true;
    if (sampling && tracking) track_current(h);     // the post-accept (post-swap) position (HMC.py:92-104)
    if (carry)     // loss at the new current position = what step() returns: accepted ? loss(q_L) : loss(q0) (HMC.py:96,104)
      PYB_CUDA(cudaMemcpyAsync(st.loss0.p, st.ret_loss.p, S * sizeof(float), cudaMemcpyDeviceToDevice, h->stream));
    st.have_cur = carry;
    st.have_inj_p = st.have_inj_u = false;
    st.iter++;
  }
  PYB_CUDA(cudaEventRecord(h->ev1, h->stream));
  PYB_CUDA(cudaStreamSynchronize(h->stream));
  PYB_CUDA(cudaGetLastError());
  float ms = 0.f;
  PYB_CUDA(cudaEventElapsedTime(&ms, h->ev0, h->ev1));
  h->last_device_ms = ms;
  prof_resolve(h);
  if (n_iters > 0 && path == PYB_PATH_TENSOR && h->opt_tc_i8 < 0)
    update_i8_guard(h, st.have_cur ? st.loss0.p : st.ret_loss.p, S);      // mean loss of every chain at its current position
  if (out) {
    unsigned long long c[4];
    double ls = 0.0;
    PYB_CUDA(cudaMemcpy(c, st.counters.p, sizeof(c), cudaMemcpyDeviceToHost));
    PYB_CUDA(cudaMemcpy(&ls, st.loss_sum.p, sizeof(double), cudaMemcpyDeviceToHost));
    out->n_accepted = (int64_t)c[0];
    out->n_total = (int64_t)c[1];
    out->n_nan = (int64_t)c[2];
    out->accept_rate = c[1] ? (double)c[0] / (double)c[1] : 0.0;
    out->mean_loss = c[1] ? ls / (double)c[1] : 0.0;
    out->grad_evals = evals;
    out->device_ms = ms;
    out->kernel_launches = h->kernel_launches - launches0;
  }
}

void hmc_eval(pyb_handle* h, const float* q, int64_t S, float* U, float* loss, float* grad) {
  check_ready(h);
  PYB_REQUIRE(S > 0, PYB_ERR_INVALID, "S must be > 0");
  const int64_t P = h->model.P;
  DevBuf<float> dq, dg, dloss, dUp, dU;
  DevBuf<double> part;
  dq.alloc(S * P); dloss.alloc(S); dUp.alloc(S); dU.alloc(S);
  if (grad) dg.alloc(S * P);
  int nblk = ew_blocks(P);
  part.alloc((size_t)S * nblk);
  PYB_CUDA(cudaMemcpyAsync(dq.p, q, S * P * sizeof(float), cudaMemcpyHostToDevice, h->stream));
  eval_loss_grad(h, dq.p, S, (float)h->n_train, dloss.p, grad ? dg.p : nullptr);
  if (h->path_used == PYB_PATH_TENSOR && h->opt_tc_i8 < 0 && grad) {
    // automatic operand split: an answer computed on int8 slices for positions whose loss is below the guard's threshold
    // is computed again on bf16x3 (and an answer on bf16x3 re-opens the guard when the losses allow)
    const bool was_ok = h->i8_guard_ok;
    PYB_CUDA(cudaStreamSynchronize(h->stream));
    if (!update_i8_guard(h, dloss.p, S) && was_ok)
      eval_loss_grad(h, dq.p, S, (float)h->n_train, dloss.p, dg.p);
  }
  k_prior<<<chain_grid(nblk, S), EW_THREADS, 0, h->stream>>>(dq.p, grad ? dg.p : nullptr, h->mu.p, h->inv_var.p, P, part.p, S);
  k_finish<<<(unsigned)S, 128, 0, h->stream>>>(part.p, nblk, 1.0, dUp.p);
  k_potential<<<(unsigned)((S + 255) / 256), 256, 0, h->stream>>>(dUp.p, dloss.p, (float)h->prior_const,
                                                                  (float)h->n_train, dU.p, S);
  count_launch(h, 3);
  if (U) PYB_CUDA(cudaMemcpyAsync(U, dU.p, S * sizeof(float), cudaMemcpyDeviceToHost, h->stream));
  if (loss) PYB_CUDA(cudaMemcpyAsync(loss, dloss.p, S * sizeof(float), cudaMemcpyDeviceToHost, h->stream));
  if (grad) PYB_CUDA(cudaMemcpyAsync(grad, dg.p, S * P * sizeof(float), cudaMemcpyDeviceToHost, h->stream));
  PYB_CUDA(cudaStreamSynchronize(h->stream));
  PYB_CUDA(cudaGetLastError());
}

// ------------------------------------------------------------------------------------------
// per-chain step sizes and their dual-averaging adaptation (dual_average, common.cuh)
// ------------------------------------------------------------------------------------------
__global__ void k_adapt_begin(const double* step, double* da, int64_t S) {
  int64_t s = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (s >= S) return;
  da[4 * s + 0] = log(step[s]);
  da[4 * s + 1] = 0.0;
  da[4 * s + 2] = 0.0;
  da[4 * s + 3] = log(10.0 * step[s]);      // mu: the adaptation leans towards larger steps than it starts from
}
__global__ void k_adapt_end(double* step, const double* da, int64_t S) {
  int64_t s = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (s < S) step[s] = exp(da[4 * s + 1]);
}

static void require_inited(const HmcState& st) {
  PYB_REQUIRE(st.inited, PYB_ERR_STATE, "pyb_hmc_init must be called first");
}

// the per-chain array, every chain at epsilon, the first time it is needed
static void ensure_step_array(pyb_handle* h) {
  HmcState& st = h->hmc;
  if (st.step.p) return;
  std::vector<double> e((size_t)st.S, st.eps);
  st.step.alloc(st.S);
  PYB_CUDA(cudaMemcpyAsync(st.step.p, e.data(), st.S * sizeof(double), cudaMemcpyHostToDevice, h->stream));
  PYB_CUDA(cudaStreamSynchronize(h->stream));
}

void hmc_adapt_begin(pyb_handle* h, double target) {
  HmcState& st = h->hmc;
  require_inited(st);
  PYB_REQUIRE(!st.adapting, PYB_ERR_STATE, "the step sizes are already adapting");
  PYB_REQUIRE(target > 0.0 && target < 1.0, PYB_ERR_INVALID, "target_accept must be in (0, 1)");
  st.da.alloc(4 * st.S);
  ensure_step_array(h);
  k_adapt_begin<<<(unsigned)((st.S + 255) / 256), 256, 0, h->stream>>>(st.step.p, st.da.p, st.S);
  count_launch(h);
  PYB_CUDA(cudaStreamSynchronize(h->stream));
  PYB_CUDA(cudaGetLastError());
  st.adapting = true;
  st.adapt_t = 0;
  st.adapt_target = target;
}

void hmc_adapt_end(pyb_handle* h) {
  HmcState& st = h->hmc;
  require_inited(st);
  PYB_REQUIRE(st.adapting, PYB_ERR_STATE, "the step sizes are not adapting: call pyb_hmc_adapt_begin first");
  if (st.adapt_t > 0) {        // without an adaptation iteration the step sizes stay where they started
    k_adapt_end<<<(unsigned)((st.S + 255) / 256), 256, 0, h->stream>>>(st.step.p, st.da.p, st.S);
    count_launch(h);
  }
  PYB_CUDA(cudaStreamSynchronize(h->stream));
  PYB_CUDA(cudaGetLastError());
  st.adapting = false;
  st.da.release();
}

void hmc_step_sizes(pyb_handle* h, double* out) {
  HmcState& st = h->hmc;
  require_inited(st);
  PYB_REQUIRE(out, PYB_ERR_INVALID, "NULL argument");
  if (!st.step.p) {
    std::fill(out, out + st.S, st.eps);
    return;
  }
  PYB_CUDA(cudaStreamSynchronize(h->stream));
  PYB_CUDA(cudaMemcpy(out, st.step.p, st.S * sizeof(double), cudaMemcpyDeviceToHost));
}

void hmc_set_step_sizes(pyb_handle* h, const double* eps) {
  HmcState& st = h->hmc;
  require_inited(st);
  PYB_REQUIRE(!st.adapting, PYB_ERR_STATE, "the step sizes are adapting: call pyb_hmc_adapt_end first");
  PYB_REQUIRE(eps, PYB_ERR_INVALID, "NULL argument");
  for (int64_t s = 0; s < st.S; ++s)
    PYB_REQUIRE(isfinite(eps[s]) && eps[s] > 0.0, PYB_ERR_INVALID, "step sizes must be finite and > 0");
  st.step.alloc(st.S);
  PYB_CUDA(cudaMemcpyAsync(st.step.p, eps, st.S * sizeof(double), cudaMemcpyHostToDevice, h->stream));
  PYB_CUDA(cudaStreamSynchronize(h->stream));
}

// ------------------------------------------------------------------------------------------
// tempering ladder (parallel tempering / replica exchange)
// ------------------------------------------------------------------------------------------
void hmc_set_temperatures(pyb_handle* h, const double* beta, int R) {
  HmcState& st = h->hmc;
  require_inited(st);
  PYB_REQUIRE(!st.sampling_started, PYB_ERR_STATE,
              "the ladder cannot change during a sampling phase (set it after pyb_hmc_init or pyb_hmc_reset_samples)");
  if (R == 0 && !beta) {
    PYB_CUDA(cudaStreamSynchronize(h->stream));
    st.R = 0; st.ladder.clear();
    st.beta.release(); st.ladder_d.release(); st.swap_logr.release(); st.swapped.release(); st.moved.release();
    st.tcount.release(); st.cold.release();
    st.swaps_ran = false;
    hmc_track_resize(h);
    hmc_params_resize(h);
    return;
  }
  PYB_REQUIRE(beta, PYB_ERR_INVALID, "beta is NULL (pass NULL with R = 0 to turn tempering off)");
  PYB_REQUIRE(R >= 2 && R <= kMaxRungs, PYB_ERR_INVALID, "a ladder has 2 to 64 rungs");
  PYB_REQUIRE(beta[0] == 1.0, PYB_ERR_INVALID, "the first inverse temperature must be 1");
  for (int r = 1; r < R; ++r)
    PYB_REQUIRE(isfinite(beta[r]) && beta[r] > 0.0 && beta[r] < beta[r - 1], PYB_ERR_INVALID,
                "inverse temperatures must decrease strictly and stay > 0");
  PYB_REQUIRE(st.S % R == 0, PYB_ERR_INVALID, "the number of local chains must be a multiple of the ladder length");
  PYB_REQUIRE(st.chain_offset % R == 0, PYB_ERR_INVALID, "chain_offset must be a multiple of the ladder length");
  const int64_t S = st.S, P = h->model.P;
  std::vector<float> bs((size_t)S);
  for (int64_t s = 0; s < S; ++s) bs[s] = (float)beta[s % R];
  PYB_CUDA(cudaStreamSynchronize(h->stream));
  st.beta.alloc(S); st.ladder_d.alloc(R); st.swap_logr.alloc(S); st.swapped.alloc(S); st.moved.alloc(S);
  st.tcount.alloc(4 * (size_t)R); st.cold.alloc((size_t)(S / R) * P);
  PYB_CUDA(cudaMemcpy(st.beta.p, bs.data(), S * sizeof(float), cudaMemcpyHostToDevice));
  PYB_CUDA(cudaMemcpy(st.ladder_d.p, beta, R * sizeof(double), cudaMemcpyHostToDevice));
  PYB_CUDA(cudaMemset(st.tcount.p, 0, st.tcount.bytes()));
  st.ladder.assign(beta, beta + R);
  st.R = R;
  st.swaps_ran = false;
  hmc_track_resize(h);
  hmc_params_resize(h);
}

void hmc_tempering_stats(pyb_handle* h, int64_t* rung_acc, int64_t* rung_tot, int64_t* swap_att, int64_t* swap_acc) {
  HmcState& st = h->hmc;
  require_inited(st);
  PYB_REQUIRE(st.R, PYB_ERR_STATE, "no tempering ladder is set: call pyb_hmc_set_temperatures first");
  const int R = st.R;
  std::vector<unsigned long long> c(4 * (size_t)R);
  PYB_CUDA(cudaStreamSynchronize(h->stream));
  PYB_CUDA(cudaMemcpy(c.data(), st.tcount.p, c.size() * sizeof(unsigned long long), cudaMemcpyDeviceToHost));
  for (int r = 0; r < R; ++r) {
    if (rung_acc) rung_acc[r] = (int64_t)c[r];
    if (rung_tot) rung_tot[r] = (int64_t)c[R + r];
    if (r + 1 < R) {
      if (swap_att) swap_att[r] = (int64_t)c[2 * R + r];
      if (swap_acc) swap_acc[r] = (int64_t)c[3 * R + r];
    }
  }
}

void hmc_last_swaps(pyb_handle* h, float* log_r, int32_t* swapped) {
  HmcState& st = h->hmc;
  require_inited(st);
  PYB_REQUIRE(st.R, PYB_ERR_STATE, "no tempering ladder is set: call pyb_hmc_set_temperatures first");
  PYB_REQUIRE(st.swaps_ran, PYB_ERR_STATE, "no iteration has run under this ladder yet");
  PYB_CUDA(cudaStreamSynchronize(h->stream));
  if (log_r) PYB_CUDA(cudaMemcpy(log_r, st.swap_logr.p, st.S * sizeof(float), cudaMemcpyDeviceToHost));
  if (swapped) PYB_CUDA(cudaMemcpy(swapped, st.swapped.p, st.S * sizeof(int32_t), cudaMemcpyDeviceToHost));
}

}  // namespace pyb
