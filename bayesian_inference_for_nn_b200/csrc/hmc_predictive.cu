// hmc_predictive.cu — the HMC posterior predictive streamed while the chains run.
// BayesianModel.predict(mode="exact") over HMC.result() (BayesianModel.py:106-129 over HMC.py:176-187) is a
// frequency-weighted expectation over exactly the draws the sampler records (HMC.py:92-104); instead of keeping those
// draws (S P 4 bytes per iteration), every recorded position is pushed through the forward pass on the tracked inputs
// once, inside pyb_hmc_run, and only moment sums are kept:
//   A = sum_s sum_t o          Q = sum_s sum_t o^2          M = sum_s (sum_t o)^2
//   W = sum_s sum_t (o - m_s)^2 (within-chain sum of squares)   S2 = sum_s sum_t o o^T (labels given, C > 1)
// All are sums over chains, so the sums of several handles (devices, ranks) add up to those of the whole run.
// W follows from Q - M/T in exact arithmetic, but that difference cancels catastrophically when a chain barely moves
// (with the reference's sigma < 0 prior every proposal after burn-in is rejected and W is exactly 0), so each chain's
// sums are kept relative to its own first tracked draw: D_s = sum_t (o - c_s), Qd = sum (o - c_s)^2, and
// W = Qd - sum_s D_s^2 / T, which is exactly 0 for a chain that never moved.
#include "common.cuh"
#include <math.h>
#include <algorithm>

namespace pyb {

constexpr int kTrackGroup = 32;   // chains per block of k_track_accum

// One tracked draw of the nb chains of a chunk, outputs out [nb, elems].  Block (x, g) owns 256 consecutive elements of
// the chains g*32 .. g*32+31: NaN -> 0 (BayesianModel.py:125), then per chain d = o - c (first = 1: c = o, d = 0) and
// s1c += d; the group's sum o^2 and sum d^2 go to part[g] (k_track_pool adds the groups in a fixed order).
// Every load and store is coalesced over the elements; one pass over out, shift and s1c.
__global__ void __launch_bounds__(256) k_track_accum(const float* __restrict__ out, int64_t nb, int64_t elems, int first,
                                                      float* __restrict__ shift, double* __restrict__ s1c,
                                                      double* __restrict__ part) {
  const int64_t e = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (e >= elems) return;
  const int64_t k0 = (int64_t)blockIdx.y * kTrackGroup, k1 = min(k0 + (int64_t)kTrackGroup, nb);
  double q = 0.0, qd = 0.0;
#pragma unroll 4
  for (int64_t k = k0; k < k1; ++k) {
    const int64_t i = k * elems + e;
    float o = out[i];
    if (o != o) o = 0.f;
    double d = 0.0;
    if (first) shift[i] = o;
    else d = (double)o - (double)shift[i];
    s1c[i] += d;
    q += (double)o * (double)o;
    qd += d * d;
  }
  part[(int64_t)blockIdx.y * 2 * elems + e] = q;
  part[((int64_t)blockIdx.y * 2 + 1) * elems + e] = qd;
}

__global__ void k_track_pool(const double* __restrict__ part, int ngroups, int64_t elems, double* Q, double* Qd) {
  const int64_t e = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (e >= elems) return;
  double a = 0.0, b = 0.0;
  for (int g = 0; g < ngroups; ++g) {
    a += part[(int64_t)g * 2 * elems + e];
    b += part[((int64_t)g * 2 + 1) * elems + e];
  }
  Q[e] += a;
  Qd[e] += b;
}

// chain reduction, fixed chain order: with c the chain's first draw and D its shifted sum, sum_t o = T c + D, so
// A = sum_s (T c + D), M = sum_s (T c + D)^2 and W = Qd - sum_s D^2 / T
__global__ void k_track_reduce(const float* __restrict__ shift, const double* __restrict__ s1c, const double* __restrict__ Qd,
                               int64_t S, int64_t elems, double T, double* A, double* M, double* W) {
  const int64_t e = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (e >= elems) return;
  double a = 0.0, m = 0.0, dd = 0.0;
  for (int64_t s = 0; s < S; ++s) {
    const double D = s1c[s * elems + e];
    const double tot = T * (double)shift[s * elems + e] + D;
    a += tot;
    m += tot * tot;
    dd += D * D;
  }
  A[e] = a;
  M[e] = m;
  W[e] = Qd[e] - dd / T;
}

// classic Gelman-Rubin R-hat (gelman_rubin, common.cuh) per output element from the sums of S chains with T draws each
__global__ void k_track_rhat(const double* __restrict__ A, const double* __restrict__ M, const double* __restrict__ Wss,
                             int64_t elems, double S, double T, float* rhat) {
  const int64_t e = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (e >= elems) return;
  rhat[e] = (float)gelman_rubin(A, M, Wss, e, S, T);
}

static bool track_tensor(pyb_handle* h, int64_t Nt) {   // the forward pyb_predict would use for these inputs
  return tc_supported_rows(h, Nt) && (h->opt_path == PYB_PATH_AUTO || h->opt_path == PYB_PATH_TENSOR);
}

void hmc_track_stop(pyb_handle* h) {
  HmcState::Track& t = h->hmc.track;
  for (DevBuf<float>* b : {&t.x, &t.out, &t.shift}) b->release();
  for (DevBuf<double>* b : {&t.s1c, &t.Q, &t.Qd, &t.S2, &t.part}) b->release();
  t.y.release();
  t.on = false;
  t.Nt = t.chunk = t.T = t.nch = 0;
}

void hmc_track_clear(pyb_handle* h) {
  HmcState::Track& t = h->hmc.track;
  if (!t.on) return;
  PYB_CUDA(cudaMemsetAsync(t.s1c.p, 0, t.s1c.bytes(), h->stream));
  PYB_CUDA(cudaMemsetAsync(t.Q.p, 0, t.Q.bytes(), h->stream));
  PYB_CUDA(cudaMemsetAsync(t.Qd.p, 0, t.Qd.bytes(), h->stream));
  if (t.S2.p) PYB_CUDA(cudaMemsetAsync(t.S2.p, 0, t.S2.bytes(), h->stream));
  t.T = 0;
}

void hmc_track_start(pyb_handle* h, const float* x, int64_t Nt, const int32_t* y) {
  HmcState& st = h->hmc;
  PYB_REQUIRE(st.inited, PYB_ERR_STATE, "pyb_hmc_init must be called first");
  PYB_REQUIRE(!st.sampling_started, PYB_ERR_STATE,
              "the predictive must be tracked from the first sampling iteration on: call before it (or after pyb_hmc_reset_samples)");
  PYB_REQUIRE(Nt > 0, PYB_ERR_INVALID, "Nt must be > 0");
  const Model& m = h->model;
  const int64_t C = m.out_dim, elems = Nt * C, S = st.R ? st.S / st.R : st.S;   // a ladder tracks its rung-0 chains only
  const int Ce = C == 1 ? 2 : (int)C;
  if (y) {
    PYB_REQUIRE(Ce * Ce <= 1024, PYB_ERR_UNSUPPORTED, "classification uncertainty supports at most 32 classes");
    for (int64_t r = 0; r < Nt; ++r) PYB_REQUIRE(y[r] >= 0 && y[r] < Ce, PYB_ERR_INVALID, "label out of range");
  }
  hmc_track_stop(h);
  // chain chunk of one forward pass: bounded as in predict() by the generic workspace and a 512 MiB output buffer
  int64_t chunk = generic_chain_batch(h, S, Nt, false);
  chunk = std::min<int64_t>(chunk, std::max<int64_t>(1, (int64_t)((512ull << 20) / (sizeof(float) * (size_t)elems))));
  const int64_t ngroups = (chunk + kTrackGroup - 1) / kTrackGroup;
  const bool s2 = y && C > 1;
  const double need = (double)S * elems * (sizeof(double) + sizeof(float)) + 2.0 * elems * sizeof(double) +
                      (s2 ? (double)Nt * C * C * sizeof(double) : 0.0) + (double)chunk * elems * sizeof(float) +
                      (double)ngroups * 2 * elems * sizeof(double) + (double)Nt * m.in_dim * sizeof(float) +
                      (double)Nt * sizeof(int32_t);
  size_t free_b = 0, total_b = 0;
  PYB_CUDA(cudaMemGetInfo(&free_b, &total_b));
  if (need > (double)free_b) {
    char msg[256];
    snprintf(msg, sizeof(msg),
             "tracking the predictive of %lld chains on %lld x %lld outputs needs %.2f GB of device memory, %.2f GB are free",
             (long long)S, (long long)Nt, (long long)C, need / 1e9, (double)free_b / 1e9);
    throw Error(PYB_ERR_OOM, msg);
  }
  HmcState::Track& t = st.track;
  // caller-owned device inputs were produced on the caller's stream (header: "device pointers"); the copy is the
  // library's own, so the caller may free them after this call
  const bool x_dev = is_device_ptr(x);
  if (x_dev) PYB_CUDA(cudaDeviceSynchronize());
  t.x.alloc((size_t)Nt * m.in_dim);
  PYB_CUDA(cudaMemcpyAsync(t.x.p, x, (size_t)Nt * m.in_dim * sizeof(float),
                           x_dev ? cudaMemcpyDeviceToDevice : cudaMemcpyHostToDevice, h->stream));
  if (y) {
    t.y.alloc(Nt);
    PYB_CUDA(cudaMemcpyAsync(t.y.p, y, Nt * sizeof(int32_t), cudaMemcpyHostToDevice, h->stream));
  }
  t.out.alloc((size_t)chunk * elems);
  t.shift.alloc((size_t)S * elems);
  t.s1c.alloc((size_t)S * elems);
  t.Q.alloc(elems); t.Qd.alloc(elems);
  if (s2) t.S2.alloc((size_t)Nt * C * C);
  t.part.alloc((size_t)ngroups * 2 * elems);
  t.Nt = Nt;
  t.nch = S;
  t.chunk = chunk;
  t.on = true;
  tc_invalidate_track(h);
  hmc_track_clear(h);
  PYB_CUDA(cudaStreamSynchronize(h->stream));
}

// a tempering ladder set or cleared after tracking started (no draw tracked yet): the per-chain sums follow the number
// of tracked chains
void hmc_track_resize(pyb_handle* h) {
  HmcState& st = h->hmc;
  HmcState::Track& t = st.track;
  if (!t.on) return;
  const int64_t n = st.R ? st.S / st.R : st.S, elems = t.Nt * h->model.out_dim;
  if (n > t.chunk) {             // the chunk was sized for fewer chains: size it again as hmc_track_start would
    int64_t chunk = generic_chain_batch(h, n, t.Nt, false);
    chunk = std::min<int64_t>(chunk, std::max<int64_t>(1, (int64_t)((512ull << 20) / (sizeof(float) * (size_t)elems))));
    t.chunk = std::max(t.chunk, chunk);
    t.out.alloc((size_t)t.chunk * elems);
    t.part.alloc((size_t)((t.chunk + kTrackGroup - 1) / kTrackGroup) * 2 * elems);
  }
  t.shift.alloc((size_t)n * elems);
  t.s1c.alloc((size_t)n * elems);
  t.nch = n;
  hmc_track_clear(h);
}

// one draw per chain of the n positions q [n, P] (st.q, or the gathered rung-0 chains of a ladder), enqueued on the
// handle's stream, no host sync
void hmc_track_draw(pyb_handle* h, const float* q, int64_t n) {
  NvtxRange nv("pyb.hmc.track_predictive");
  HmcState& st = h->hmc;
  HmcState::Track& t = st.track;
  const Model& m = h->model;
  const int64_t P = m.P, C = m.out_dim, Nt = t.Nt, elems = Nt * C, S = n;
  const bool tensor = track_tensor(h, Nt);
  for (int64_t b0 = 0; b0 < S; b0 += t.chunk) {
    const int64_t nb = std::min(t.chunk, S - b0);
    if (tensor) tc_forward_tracked(h, q + b0 * P, nb, t.x.p, Nt, t.out.p);
    else generic_forward(h, q + b0 * P, nb, t.x.p, Nt, t.out.p);
    const int ngroups = (int)((nb + kTrackGroup - 1) / kTrackGroup);
    dim3 g((unsigned)((elems + 255) / 256), (unsigned)ngroups);
    k_track_accum<<<g, 256, 0, h->stream>>>(t.out.p, nb, elems, t.T == 0 ? 1 : 0, t.shift.p + b0 * elems,
                                            t.s1c.p + b0 * elems, t.part.p);
    k_track_pool<<<(unsigned)((elems + 255) / 256), 256, 0, h->stream>>>(t.part.p, ngroups, elems, t.Q.p, t.Qd.p);
    count_launch(h, 2);
    if (t.S2.p) uncert_s2_accum(h, t.out.p, nb, Nt, (int)C, nullptr, t.S2.p);
  }
  t.T += 1;
}

void hmc_track_sums(pyb_handle* h, double* sums, double* s2, int64_t* n_draws) {
  HmcState& st = h->hmc;
  HmcState::Track& t = st.track;
  PYB_REQUIRE(t.on, PYB_ERR_STATE, "no predictive is tracked: call pyb_hmc_track_predictive first");
  PYB_REQUIRE(t.T > 0, PYB_ERR_STATE, "no draw has been tracked yet: run a sampling iteration first");
  PYB_REQUIRE(!s2 || t.S2.p, PYB_ERR_STATE, "S2 is kept only when labels were given and the output has several units");
  const int64_t elems = t.Nt * h->model.out_dim;
  DevBuf<double> amw;
  amw.alloc(3 * (size_t)elems);
  k_track_reduce<<<(unsigned)((elems + 255) / 256), 256, 0, h->stream>>>(t.shift.p, t.s1c.p, t.Qd.p, t.nch, elems,
                                                                         (double)t.T, amw.p, amw.p + elems, amw.p + 2 * elems);
  count_launch(h);
  const size_t eb = elems * sizeof(double);
  PYB_CUDA(cudaMemcpyAsync(sums, amw.p, eb, cudaMemcpyDeviceToHost, h->stream));                 // A
  PYB_CUDA(cudaMemcpyAsync(sums + elems, t.Q.p, eb, cudaMemcpyDeviceToHost, h->stream));          // Q
  PYB_CUDA(cudaMemcpyAsync(sums + 2 * elems, amw.p + elems, 2 * eb, cudaMemcpyDeviceToHost, h->stream));   // M, W
  if (s2) PYB_CUDA(cudaMemcpyAsync(s2, t.S2.p, t.S2.bytes(), cudaMemcpyDeviceToHost, h->stream));
  PYB_CUDA(cudaStreamSynchronize(h->stream));
  PYB_CUDA(cudaGetLastError());
  if (n_draws) *n_draws = t.T;
}

void hmc_track_finish(pyb_handle* h, const double* sums, const double* s2, int64_t n_chains, int64_t n_draws,
                      const UncertaintyReq* uq, float* mean, float* var, float* rhat) {
  HmcState::Track& t = h->hmc.track;
  PYB_REQUIRE(t.on, PYB_ERR_STATE, "no predictive is tracked: call pyb_hmc_track_predictive first");
  PYB_REQUIRE(n_draws > 0, PYB_ERR_STATE, "no draw has been tracked yet: run a sampling iteration first");
  PYB_REQUIRE(n_chains > 0, PYB_ERR_INVALID, "n_chains must be > 0");
  PYB_REQUIRE(sums, PYB_ERR_INVALID, "sums is NULL");
  const int64_t C = h->model.out_dim, Nt = t.Nt, elems = Nt * C;
  if (uq) {
    PYB_REQUIRE(t.y.p, PYB_ERR_STATE, "classification uncertainty needs the labels: pass y to pyb_hmc_track_predictive");
    PYB_REQUIRE(uq->total && uq->aleatoric && uq->epistemic, PYB_ERR_INVALID, "null pointer");
    PYB_REQUIRE(uq->divisor != 0.0, PYB_ERR_INVALID, "divisor must not be 0");
    PYB_REQUIRE(C == 1 || s2, PYB_ERR_INVALID, "classification uncertainty of a multi-unit output needs s2");
  }
  DevBuf<double> ds, ds2;
  DevBuf<float> dr;
  ds.alloc(4 * (size_t)elems);
  PYB_CUDA(cudaMemcpyAsync(ds.p, sums, 4 * elems * sizeof(double), cudaMemcpyHostToDevice, h->stream));
  if (uq && C > 1) {
    ds2.alloc((size_t)Nt * C * C);
    PYB_CUDA(cudaMemcpyAsync(ds2.p, s2, ds2.bytes(), cudaMemcpyHostToDevice, h->stream));
  }
  PYB_CUDA(cudaEventRecord(h->ev0, h->stream));
  if (rhat) {
    dr.alloc(elems);
    k_track_rhat<<<(unsigned)((elems + 255) / 256), 256, 0, h->stream>>>(ds.p, ds.p + 2 * elems, ds.p + 3 * elems, elems,
                                                                       (double)n_chains, (double)n_draws, dr.p);
    count_launch(h);
    PYB_CUDA(cudaMemcpyAsync(rhat, dr.p, elems * sizeof(float), cudaMemcpyDeviceToHost, h->stream));
  }
  // every draw has weight 1: the sums are pyb_predict's s1 / s2 with weights = frequencies, total weight S T
  predictive_finish(h, ds.p, ds.p + elems, ds2.p, (double)n_chains * (double)n_draws, Nt, t.y.p, uq, mean, var);
}

}  // namespace pyb
