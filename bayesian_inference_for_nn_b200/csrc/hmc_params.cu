// hmc_params.cu — per-parameter posterior moments and convergence diagnostics streamed while the HMC chains run.
// The weight-space sibling of hmc_predictive.cu: the tracked draws are the same (the state before the first sampling
// iteration, then the position after every sampling iteration, after accept / restore and the swap round; the rung-0
// chains of a tempering ladder), and every parameter of every draw is folded into sums, so no draw has to be kept.
//
// Draw t = 0 .. T-1 of chain s is x_st (one parameter).  With h = n_planned / 2 and the batch size b, fixed when the
// tracking starts, each chain keeps its first draw c_s and the shifted sums
//   D_s = sum_t (x - c_s)    over all draws
//   H_s = the running sum over the current half [0, h) or [h, 2h)
//   E_s = the running sum over the current batch [k b, (k+1) b)
//   F_s = sum of E_sk over the batches completed so far
// and the squares are pooled over the chains on every draw:
//   Qd = sum d^2 (all draws), Qh = sum d^2 (draws t < 2h), at the end of every half Ah += h c + H, Mh += (h c + H)^2,
//   Dh2 += H^2, at the end of every batch Eb2 += E^2.
// Shifting by c_s keeps every within-chain term exact for a chain that never moves (its d, H, E are all 0).
// pyb_hmc_param_sums reduces the per-chain sums over the chains in a fixed order into K = 7 sums over chains:
//   0 A  = sum_s (T c + D)                       (sum of all draws)
//   1 M  = sum_s (T c + D)^2
//   2 W  = Qd - sum_s D^2 / T                    (within-chain sum of squares)
//   3 Ah = sum over the 2S half-chains of their sums       (complete halves only)
//   4 Mh = sum over the half-chains of their squared sums
//   5 Wh = Qh - Dh2 / h                          (within-half-chain sum of squares)
//   6 V  = (Eb2 - sum_s F^2 / a) / b^2 = sum_s sum_{k<a} (Ybar_sk - Ybar_s)^2   (a = floor(T / b) complete batches)
// so the sums of several handles add up to those of the whole run; pyb_hmc_param_finish turns them into the mean, sd,
// split-R-hat, batch-means ESS and MCSE (include/pyesian_b200.h gives the definitions).
#include "common.cuh"
#include <math.h>
#include <algorithm>

namespace pyb {

enum { PP_QD, PP_QH, PP_AH, PP_MH, PP_DH2, PP_EB2, kParamPooled };
constexpr int kParamSums = 7;
constexpr int kParamGroupMin = 32;   // chains per group of k_param_accum, at least

// where draw t falls: computed on the host from the draw counter and passed to each launch
struct ParamDraw {
  int first;         // t == 0: the draw is each chain's shift
  int split;         // t < 2h
  int half_start, half_end;      // t == 0 or h / t == h - 1 or 2h - 1
  int batch_start, batch_end;    // t % b == 0 / t % b == b - 1
  int first_batch;   // t == b - 1
  double hlen;
};

// One draw of the nch tracked chains, rows q[k R] of q [*, P] read in place.  Block (x, g) owns 256 consecutive
// parameters of the chains g*per_group .. (g+1)*per_group - 1; every load and store is coalesced over the parameters.
// The group's pooled terms go to part[g] (k_param_pool adds the groups in a fixed order).
__global__ void __launch_bounds__(256) k_param_accum(const float* __restrict__ q, int64_t P, int64_t R, int64_t nch,
                                                      int64_t per_group, ParamDraw f, float* __restrict__ shift,
                                                      double* __restrict__ d, double* __restrict__ hcur,
                                                      double* __restrict__ bcur, double* __restrict__ bsum,
                                                      double* __restrict__ part) {
  const int64_t p = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (p >= P) return;
  const int64_t k0 = (int64_t)blockIdx.y * per_group, k1 = min(k0 + per_group, nch);
  double qd = 0.0, qh = 0.0, ah = 0.0, mh = 0.0, dh2 = 0.0, eb2 = 0.0;
#pragma unroll 4
  for (int64_t k = k0; k < k1; ++k) {
    const int64_t i = k * P + p;
    const float x = q[k * R * P + p];
    float c;
    if (f.first) { c = x; shift[i] = x; }
    else c = shift[i];
    const double dv = (double)x - (double)c;
    d[i] = (f.first ? 0.0 : d[i]) + dv;
    qd += dv * dv;
    if (f.split) {
      qh += dv * dv;
      const double hs = (f.half_start ? 0.0 : hcur[i]) + dv;
      if (f.half_end) {
        const double tot = f.hlen * (double)c + hs;
        ah += tot;
        mh += tot * tot;
        dh2 += hs * hs;
      } else {
        hcur[i] = hs;
      }
    }
    const double bs = (f.batch_start ? 0.0 : bcur[i]) + dv;
    if (f.batch_end) {
      eb2 += bs * bs;
      bsum[i] = (f.first_batch ? 0.0 : bsum[i]) + bs;
    } else {
      bcur[i] = bs;
    }
  }
  double* pg = part + (int64_t)blockIdx.y * kParamPooled * P + p;
  pg[PP_QD * P] = qd;
  if (f.split) pg[PP_QH * P] = qh;
  if (f.half_end) { pg[PP_AH * P] = ah; pg[PP_MH * P] = mh; pg[PP_DH2 * P] = dh2; }
  if (f.batch_end) pg[PP_EB2 * P] = eb2;
}

// pool[j] += sum_g part[g][j] for the pooled terms j in `terms` (bit j), groups in a fixed order
__global__ void k_param_pool(const double* __restrict__ part, int ngroups, int64_t P, unsigned terms,
                             double* __restrict__ pool) {
  const int64_t p = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (p >= P) return;
  for (int j = 0; j < kParamPooled; ++j) {
    if (!((terms >> j) & 1u)) continue;
    double a = 0.0;
    for (int g = 0; g < ngroups; ++g) a += part[((int64_t)g * kParamPooled + j) * P + p];
    pool[(int64_t)j * P + p] += a;
  }
}

// the K = 7 sums over chains of the header comment, chains in a fixed order; a complete batches of b draws
__global__ void k_param_reduce(const float* __restrict__ shift, const double* __restrict__ d,
                               const double* __restrict__ bsum, const double* __restrict__ pool, int64_t nch,
                               int64_t P, double T, double hlen, int64_t a, double b, double* __restrict__ out) {
  const int64_t p = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (p >= P) return;
  double A = 0.0, M = 0.0, dd = 0.0, ff = 0.0;
  for (int64_t s = 0; s < nch; ++s) {
    const int64_t i = s * P + p;
    const double D = d[i];
    const double tot = T * (double)shift[i] + D;
    A += tot;
    M += tot * tot;
    dd += D * D;
    if (a > 0) ff += bsum[i] * bsum[i];
  }
  out[0 * P + p] = A;
  out[1 * P + p] = M;
  out[2 * P + p] = pool[PP_QD * P + p] - dd / T;
  out[3 * P + p] = pool[PP_AH * P + p];
  out[4 * P + p] = pool[PP_MH * P + p];
  out[5 * P + p] = pool[PP_QH * P + p] - pool[PP_DH2 * P + p] / hlen;
  out[6 * P + p] = a > 0 ? (pool[PP_EB2 * P + p] - ff / (double)a) / (b * b) : 0.0;
}

// mean, sd, split-R-hat, ESS and MCSE per parameter from the sums of S chains with T draws each (definitions:
// include/pyesian_b200.h); out [5, P]
__global__ void k_param_finish(const double* __restrict__ sums, int64_t P, double S, double T, double hlen, double b,
                               double a, double* __restrict__ out) {
  const int64_t p = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (p >= P) return;
  const double A = sums[0 * P + p], M = sums[1 * P + p], W = sums[2 * P + p], V = sums[6 * P + p];
  const double n = S * T;
  double between = M / T - A * A / n;             // sum_s T (m_s - mean)^2
  if (between < 0.0) between = 0.0;
  double var = (W + between) / n;
  if (var < 0.0) var = 0.0;
  double rhat = NAN;
  if (T >= 2.0 * hlen) rhat = gelman_rubin(sums + 3 * P, sums + 4 * P, sums + 5 * P, p, 2.0 * S, hlen);
  double ess = NAN, mcse = NAN;
  if (a >= 2.0) {
    const double lam2 = W / (S * (T - 1.0));
    const double sbm = b * (V < 0.0 ? 0.0 : V) / (S * (a - 1.0));
    if (T >= 2.0 && lam2 != 0.0 && sbm != 0.0) ess = n * lam2 / sbm;
    mcse = sqrt(sbm / n);
  }
  out[0 * P + p] = A / n;
  out[1 * P + p] = sqrt(var);
  out[2 * P + p] = rhat;
  out[3 * P + p] = ess;
  out[4 * P + p] = mcse;
}

// floor(sqrt(n)) in integers
static int64_t default_batch(int64_t n) {
  int64_t b = (int64_t)sqrt((double)n);
  while (b > 1 && b * b > n) --b;
  while ((b + 1) * (b + 1) <= n) ++b;
  return std::max<int64_t>(b, 1);
}

// the batch size b for (n_planned, batch), after the checks every entry point shares
static int64_t checked_batch(int64_t n_planned, int64_t batch) {
  PYB_REQUIRE(n_planned >= 4, PYB_ERR_INVALID, "n_planned must be >= 4");
  PYB_REQUIRE(batch >= 0, PYB_ERR_INVALID, "batch must be >= 0 (0: floor(sqrt(n_planned)))");
  const int64_t b = batch ? batch : default_batch(n_planned);
  PYB_REQUIRE(n_planned / b >= 2, PYB_ERR_INVALID, "n_planned must hold at least two batches of the batch size");
  return b;
}

// enough blocks to fill the device at small P, and at least kParamGroupMin chains per group so that the partials
// stay a small fraction of the per-chain traffic at large P
static int param_groups(int64_t nch, int64_t P) {
  const int64_t xb = (P + 255) / 256;
  const int64_t most = (nch + kParamGroupMin - 1) / kParamGroupMin;
  return (int)std::max<int64_t>(1, std::min<int64_t>(most, (4096 + xb - 1) / xb));
}

void hmc_params_stop(pyb_handle* h) {
  HmcState::ParamTrack& t = h->hmc.ptrack;
  t.shift.release();
  for (DevBuf<double>* b : {&t.d, &t.hcur, &t.bcur, &t.bsum, &t.pool, &t.part}) b->release();
  t.on = false;
  t.T = t.nch = t.n_planned = t.half = t.batch = 0;
  t.ngroups = 0;
}

void hmc_params_clear(pyb_handle* h) {
  HmcState::ParamTrack& t = h->hmc.ptrack;
  if (!t.on) return;
  PYB_CUDA(cudaMemsetAsync(t.pool.p, 0, t.pool.bytes(), h->stream));   // the per-chain sums start at draw 0
  t.T = 0;
}

// (re)allocate the tracking for the chains the handle tracks now, checked against the free memory first
static void params_begin(pyb_handle* h, int64_t n_planned, int64_t b) {
  HmcState& st = h->hmc;
  const int64_t P = h->model.P, n = st.R ? st.S / st.R : st.S;   // a ladder tracks its rung-0 chains only
  const int ng = param_groups(n, P);
  hmc_params_stop(h);
  const double need = (double)n * P * (sizeof(float) + 4 * sizeof(double)) +
                      (1.0 + ng) * kParamPooled * P * sizeof(double);
  size_t free_b = 0, total_b = 0;
  PYB_CUDA(cudaMemGetInfo(&free_b, &total_b));
  if (need > (double)free_b) {
    char msg[256];
    snprintf(msg, sizeof(msg),
             "tracking the parameters of %lld chains x %lld parameters needs %.2f GB of device memory, %.2f GB are free",
             (long long)n, (long long)P, need / 1e9, (double)free_b / 1e9);
    throw Error(PYB_ERR_OOM, msg);
  }
  HmcState::ParamTrack& t = st.ptrack;
  t.shift.alloc((size_t)n * P);
  for (DevBuf<double>* buf : {&t.d, &t.hcur, &t.bcur, &t.bsum}) buf->alloc((size_t)n * P);
  t.pool.alloc((size_t)kParamPooled * P);
  t.part.alloc((size_t)ng * kParamPooled * P);
  t.nch = n;
  t.ngroups = ng;
  t.n_planned = n_planned;
  t.half = n_planned / 2;
  t.batch = b;
  t.on = true;
  hmc_params_clear(h);
  PYB_CUDA(cudaStreamSynchronize(h->stream));
}

void hmc_params_start(pyb_handle* h, int64_t n_planned, int64_t batch) {
  HmcState& st = h->hmc;
  PYB_REQUIRE(st.inited, PYB_ERR_STATE, "pyb_hmc_init must be called first");
  PYB_REQUIRE(!st.sampling_started, PYB_ERR_STATE,
              "the parameters must be tracked from the first sampling iteration on: call before it (or after "
              "pyb_hmc_reset_samples)");
  params_begin(h, n_planned, checked_batch(n_planned, batch));
}

// a tempering ladder set or cleared after tracking started (no draw tracked yet): the per-chain sums follow the number
// of tracked chains
void hmc_params_resize(pyb_handle* h) {
  HmcState& st = h->hmc;
  HmcState::ParamTrack& t = st.ptrack;
  if (!t.on) return;
  if (t.nch == (st.R ? st.S / st.R : st.S)) { hmc_params_clear(h); return; }
  params_begin(h, t.n_planned, t.batch);
}

// one draw of every tracked chain at its current position, enqueued on the handle's stream, no host sync
void hmc_params_draw(pyb_handle* h) {
  NvtxRange nv("pyb.hmc.track_params");
  HmcState& st = h->hmc;
  HmcState::ParamTrack& t = st.ptrack;
  const int64_t P = h->model.P, tt = t.T, hl = t.half, b = t.batch;
  ParamDraw f;
  f.first = tt == 0;
  f.split = tt < 2 * hl;
  f.half_start = tt == 0 || tt == hl;
  f.half_end = tt == hl - 1 || tt == 2 * hl - 1;
  f.batch_start = tt % b == 0;
  f.batch_end = tt % b == b - 1;
  f.first_batch = tt == b - 1;
  f.hlen = (double)hl;
  const unsigned terms = (1u << PP_QD) | (f.split ? 1u << PP_QH : 0u) |
                         (f.half_end ? (1u << PP_AH) | (1u << PP_MH) | (1u << PP_DH2) : 0u) |
                         (f.batch_end ? 1u << PP_EB2 : 0u);
  const unsigned xb = (unsigned)((P + 255) / 256);
  const int64_t per_group = (t.nch + t.ngroups - 1) / t.ngroups;
  k_param_accum<<<dim3(xb, (unsigned)t.ngroups), 256, 0, h->stream>>>(st.q.p, P, st.R ? st.R : 1, t.nch, per_group, f,
                                                                      t.shift.p, t.d.p, t.hcur.p, t.bcur.p, t.bsum.p,
                                                                      t.part.p);
  k_param_pool<<<xb, 256, 0, h->stream>>>(t.part.p, t.ngroups, P, terms, t.pool.p);
  count_launch(h, 2);
  t.T += 1;
}

void hmc_params_sums(pyb_handle* h, double* sums, int64_t* n_draws) {
  HmcState::ParamTrack& t = h->hmc.ptrack;
  PYB_REQUIRE(t.on, PYB_ERR_STATE, "no parameters are tracked: call pyb_hmc_track_params first");
  PYB_REQUIRE(t.T > 0, PYB_ERR_STATE, "no draw has been tracked yet: run a sampling iteration first");
  const int64_t P = h->model.P;
  DevBuf<double> out;
  out.alloc((size_t)kParamSums * P);
  k_param_reduce<<<(unsigned)((P + 255) / 256), 256, 0, h->stream>>>(t.shift.p, t.d.p, t.bsum.p, t.pool.p, t.nch, P,
                                                                     (double)t.T, (double)t.half, t.T / t.batch,
                                                                     (double)t.batch, out.p);
  count_launch(h);
  PYB_CUDA(cudaMemcpyAsync(sums, out.p, out.bytes(), cudaMemcpyDeviceToHost, h->stream));
  PYB_CUDA(cudaStreamSynchronize(h->stream));
  PYB_CUDA(cudaGetLastError());
  if (n_draws) *n_draws = t.T;
}

void hmc_params_finish(pyb_handle* h, const double* sums, int64_t n_chains, int64_t n_draws, int64_t n_planned,
                       int64_t batch, double* mean, double* sd, double* rhat, double* ess, double* mcse) {
  PYB_REQUIRE(sums, PYB_ERR_INVALID, "sums is NULL");
  PYB_REQUIRE(n_chains > 0, PYB_ERR_INVALID, "n_chains must be > 0");
  PYB_REQUIRE(n_draws > 0, PYB_ERR_INVALID, "n_draws must be > 0");
  const int64_t b = checked_batch(n_planned, batch), P = h->model.P;
  DevBuf<double> ds, out;
  ds.alloc((size_t)kParamSums * P);
  out.alloc((size_t)5 * P);
  PYB_CUDA(cudaMemcpyAsync(ds.p, sums, ds.bytes(), cudaMemcpyHostToDevice, h->stream));
  k_param_finish<<<(unsigned)((P + 255) / 256), 256, 0, h->stream>>>(ds.p, P, (double)n_chains, (double)n_draws,
                                                                     (double)(n_planned / 2), (double)b,
                                                                     (double)(n_draws / b), out.p);
  count_launch(h);
  double* dst[5] = {mean, sd, rhat, ess, mcse};
  for (int j = 0; j < 5; ++j)
    if (dst[j]) PYB_CUDA(cudaMemcpyAsync(dst[j], out.p + (size_t)j * P, P * sizeof(double), cudaMemcpyDeviceToHost,
                                         h->stream));
  PYB_CUDA(cudaStreamSynchronize(h->stream));
  PYB_CUDA(cudaGetLastError());
}

size_t hmc_params_bytes(const pyb_handle* h) {
  const HmcState::ParamTrack& t = h->hmc.ptrack;
  return t.shift.bytes() + t.d.bytes() + t.hcur.bytes() + t.bcur.bytes() + t.bsum.bytes() + t.pool.bytes() +
         t.part.bytes();
}

}  // namespace pyb
