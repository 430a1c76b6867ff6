// predict.cu — posterior predictive for n weight samples at once.
// Replaces BayesianModel.predict's Python loop (BayesianModel.py:106-129: n x {assign weights,
// forward, NaN->0, accumulate}) and the np.var the Plotter takes over the per-draw outputs
// (Plotter.py:244).  Weighted form = frequency-weighted exact expectation over the stored samples.
#include "common.cuh"
#include <algorithm>

namespace pyb {

// s1 += w*o ; s2 += w*o*o over the chunk's samples (NaN -> 0), optional copy to all_out
__global__ void k_pred_accum(const float* out, int64_t n_chunk, int64_t elems, const float* w, double* s1, double* s2) {
  int64_t e = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (e >= elems) return;
  double a = 0.0, b = 0.0;
  for (int64_t k = 0; k < n_chunk; ++k) {
    float o = out[k * elems + e];
    if (o != o) o = 0.f;
    double ww = w ? (double)w[k] : 1.0;
    a += ww * (double)o;
    b += ww * (double)o * (double)o;
  }
  s1[e] += a;
  s2[e] += b;
}
__global__ void k_nan_to_zero(float* v, int64_t n) {
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x)
    if (v[i] != v[i]) v[i] = 0.f;
}
__global__ void k_pred_finish(const double* s1, const double* s2, double wsum, int64_t elems, float* mean, float* var) {
  int64_t e = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (e >= elems) return;
  double m = s1[e] / wsum;
  double v = s2[e] / wsum - m * m;
  mean[e] = (float)m;
  var[e] = (float)(v > 0.0 ? v : 0.0);
}

// ---- Metrics.classification_uncertainty (Metrics.py:344-375) --------------------------------------------------
// Per data row r and weight sample k with class probabilities p (NaN -> 0 as BayesianModel.py:125):
//   aleatoric_r += w_k (diag(p) - p p^T)        epistemic_r += w_k (p - onehot(y_r)) (p - onehot(y_r))^T   (canonical)
// Both follow from the first and second moments over the samples, S1 = sum_k w_k p (k_pred_accum already has it) and
// S2 = sum_k w_k p p^T:   aleatoric = diag(S1) - S2,   epistemic = S2 - S1 e^T - e S1^T + W e e^T  (e = onehot, W = sum w);
// the reference's own epistemic term (a broadcast, see k_uncert_rows) is C S2 - S1 1^T - 1 S1^T + W 1 1^T,
// so the only extra pass over the [n, Nt, C] outputs is the S2 accumulation below.  A block owns 128/C data rows and
// stages 32 samples of their class probabilities in shared memory with coalesced loads (every output byte is read from
// HBM exactly once, ~15 KB in flight per block); thread = (row, class i) then keeps row i of that row's C x C block in
// registers and reads its row's C values back as shared-memory broadcasts: float32 products, flushed into float64
// every 32 samples.  (First version: the same register tile fed by direct global loads - 10 of 11 loads redundant,
// 360 GB/s, long-scoreboard bound at 20 % occupancy; profiles/r1_ncu_full_next.txt.)
// A one-unit (sigmoid) output is widened to the two classes [1-p, p] (Metrics.py:357-359); its moments follow from
// s1 = sum w p and s2 = sum w p^2 alone, no extra pass.
template <int C>
__global__ void __launch_bounds__(128) k_uncert_s2(const float* __restrict__ out, int64_t n_chunk, int64_t Nt,
                                                   const float* __restrict__ w, double* __restrict__ S2) {
  constexpr int R = 128 / C, RC = R * C, KT = 32, PER = (KT * RC + 127) / 128;
  __shared__ float tile[KT * RC];
  __shared__ float wt[KT];
  const int tid = threadIdx.x;
  const int64_t r0 = (int64_t)blockIdx.x * R;
  const int nrows = (int)min((int64_t)R, Nt - r0);
  const int nvalid = nrows * C;                 // this block's contiguous floats per sample
  const int lr = tid / C, i = tid % C;          // compute role: row lr of the block, class i
  const bool active = tid < RC && lr < nrows;
  const float* src = out + r0 * C;
  const int64_t stride = Nt * C;
  double acc[C];
#pragma unroll
  for (int j = 0; j < C; ++j) acc[j] = 0.0;
  for (int64_t k0 = 0; k0 < n_chunk; k0 += KT) {
    const int kt = (int)min((int64_t)KT, n_chunk - k0);
    // stage kt samples x nvalid floats, coalesced; all of a thread's loads are issued before the first store
    float v[PER];
#pragma unroll
    for (int q = 0; q < PER; ++q) {
      const int e = tid + q * 128, kk = e / RC, c = e % RC;
      v[q] = (kk < kt && c < nvalid) ? src[(k0 + kk) * stride + c] : 0.f;
    }
#pragma unroll
    for (int q = 0; q < PER; ++q) {
      const int e = tid + q * 128;
      if (e < KT * RC) tile[e] = (v[q] != v[q]) ? 0.f : v[q];
    }
    if (tid < KT) wt[tid] = (tid < kt) ? (w ? w[k0 + tid] : 1.f) : 0.f;
    __syncthreads();
    if (active) {
      float f[C];
#pragma unroll
      for (int j = 0; j < C; ++j) f[j] = 0.f;
#pragma unroll 8
      for (int kk = 0; kk < KT; ++kk) {          // samples beyond kt were staged as zeros with zero weight
        const float* row = tile + kk * RC + lr * C;
        const float wp = wt[kk] * row[i];
#pragma unroll
        for (int j = 0; j < C; ++j) f[j] = fmaf(wp, row[j], f[j]);
      }
#pragma unroll
      for (int j = 0; j < C; ++j) acc[j] += (double)f[j];
    }
    __syncthreads();
  }
  if (active) {
#pragma unroll
    for (int j = 0; j < C; ++j) S2[((r0 + lr) * C + i) * C + j] += acc[j];
  }
}
// any other class count (<= 32): thread = (row, i, j)
__global__ void k_uncert_s2_generic(const float* out, int64_t n_chunk, int64_t Nt, int C, const float* w, double* S2) {
  const int64_t e = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (e >= Nt * C * C) return;
  const int j = (int)(e % C), i = (int)((e / C) % C);
  const int64_t r = e / ((int64_t)C * C);
  double a = 0.0;
  for (int64_t k = 0; k < n_chunk; ++k) {
    const float* o = out + (k * Nt + r) * C;
    float pi = o[i], pj = o[j];
    if (pi != pi) pi = 0.f;
    if (pj != pj) pj = 0.f;
    a += (w ? (double)w[k] : 1.0) * (double)(pi * pj);
  }
  S2[e] += a;
}
// per-row matrices from the moments; s1/s2 are k_pred_accum's sums over out_dim C, S2 the block above (C > 1)
// reference != 0: the epistemic term as the reference's code computes it — its reshape(p, (-1, 1)) - one_hot(label)
// broadcasts to D_ij = p_i - onehot_j (Metrics.py:362-363) and (D D^T)_ik = Ce p_i p_k - p_i - p_k + 1, label-free
__global__ void k_uncert_rows(const double* s1, const double* s2, const double* S2, double wsum, int64_t Nt, int C, int Ce,
                              const int32_t* y, int reference, double* alea, double* epi) {
  const int64_t e = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (e >= Nt * Ce * Ce) return;
  const int j = (int)(e % Ce), i = (int)((e / Ce) % Ce);
  const int64_t r = e / ((int64_t)Ce * Ce);
  double m1i, m1j, m2;
  if (C == 1) {           // classes [1 - p, p]
    const double a = s1[r], b = s2[r];
    m1i = i ? a : wsum - a;
    m1j = j ? a : wsum - a;
    m2 = (i && j) ? b : ((i || j) ? a - b : wsum - 2.0 * a + b);
  } else {
    m1i = s1[r * C + i];
    m1j = s1[r * C + j];
    m2 = S2[e];
  }
  const int label = y[r];
  const double ei = (i == label) ? 1.0 : 0.0, ej = (j == label) ? 1.0 : 0.0;
  alea[e] = (i == j ? m1i : 0.0) - m2;
  epi[e] = reference ? (double)Ce * m2 - m1i - m1j + wsum : m2 - m1i * ej - ei * m1j + wsum * ei * ej;
}
template <int C>
static void launch_uncert_s2(pyb_handle* h, const float* out, int64_t nb, int64_t Nt, const float* w, double* S2) {
  constexpr int R = 128 / C;
  k_uncert_s2<C><<<(unsigned)((Nt + R - 1) / R), 128, 0, h->stream>>>(out, nb, Nt, w, S2);
}
void uncert_s2_accum(pyb_handle* h, const float* out, int64_t nb, int64_t Nt, int C, const float* w, double* S2) {
  switch (C) {
    case 2: launch_uncert_s2<2>(h, out, nb, Nt, w, S2); break;
    case 3: launch_uncert_s2<3>(h, out, nb, Nt, w, S2); break;
    case 4: launch_uncert_s2<4>(h, out, nb, Nt, w, S2); break;
    case 5: launch_uncert_s2<5>(h, out, nb, Nt, w, S2); break;
    case 10: launch_uncert_s2<10>(h, out, nb, Nt, w, S2); break;
    default:
      k_uncert_s2_generic<<<(unsigned)((Nt * C * C + 255) / 256), 256, 0, h->stream>>>(out, nb, Nt, C, w, S2);
  }
  count_launch(h);
}
// The reference never resets its accumulators between rows (Metrics.py:352-366: `aleatoric +=` inside the row loop,
// appended per row), so row r of its result is the running sum over rows 0..r.  Three passes over 32-row segments:
// segment sums, exclusive scan of the segment sums, running prefix written out (fixed order => deterministic).
constexpr int kUqSeg = 32;
__global__ void k_uncert_segsum(const double* acc, int64_t Nt, int CC, double* seg) {
  const int e = threadIdx.x;
  if (e >= CC) return;
  const int64_t r0 = (int64_t)blockIdx.x * kUqSeg, r1 = min(r0 + (int64_t)kUqSeg, Nt);
  double s = 0.0;
  for (int64_t r = r0; r < r1; ++r) s += acc[r * CC + e];
  seg[(int64_t)blockIdx.x * CC + e] = s;
}
__global__ void k_uncert_segscan(const double* __restrict__ seg, double* __restrict__ excl, int64_t nseg, int CC) {
  const int e = threadIdx.x;
  if (e >= CC) return;
  double run = 0.0;                       // out of place, so the loads of the next segments do not wait for the stores
#pragma unroll 8
  for (int64_t s = 0; s < nseg; ++s) {
    excl[s * CC + e] = run;
    run += seg[s * CC + e];
  }
}
__global__ void k_uncert_finish(const double* alea, const double* epi, const double* seg_a, const double* seg_e,
                                int64_t Nt, int CC, int cumulative, double inv_div, float* total, float* alea_out,
                                float* epi_out) {
  const int e = threadIdx.x;
  if (e >= CC) return;
  const int64_t r0 = (int64_t)blockIdx.x * kUqSeg, r1 = min(r0 + (int64_t)kUqSeg, Nt);
  double ra = cumulative ? seg_a[(int64_t)blockIdx.x * CC + e] : 0.0;
  double re = cumulative ? seg_e[(int64_t)blockIdx.x * CC + e] : 0.0;
  for (int64_t r = r0; r < r1; ++r) {
    const double a = alea[r * CC + e], b = epi[r * CC + e];
    if (cumulative) { ra += a; re += b; } else { ra = a; re = b; }
    const float fa = (float)(ra * inv_div), fe = (float)(re * inv_div);
    alea_out[r * CC + e] = fa;
    epi_out[r * CC + e] = fe;
    total[r * CC + e] = fe + fa;     // epistemics + aleatorics in float32, as Metrics.py:370
  }
}

bool is_device_ptr(const void* ptr) {
  cudaPointerAttributes a;
  if (cudaPointerGetAttributes(&a, ptr) != cudaSuccess) { cudaGetLastError(); return false; }
  return a.type == cudaMemoryTypeDevice || a.type == cudaMemoryTypeManaged;
}

// dst[k][:] = src[idx[k]][:]   (device rows of row_len floats; idx arrives from the host)
__global__ void k_gather_rows_f32(const float* src, const int64_t* idx, int64_t row_len, float* dst) {
  const int64_t k = blockIdx.y;
  const float* s = src + idx[k] * row_len;
  float* d = dst + k * row_len;
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < row_len; i += (int64_t)gridDim.x * blockDim.x) d[i] = s[i];
}
void gather_rows_f32(pyb_handle* h, const float* src, const int64_t* idx_host, int64_t n, int64_t row_len, float* dst) {
  DevBuf<int64_t> di;
  di.alloc(n);
  PYB_CUDA(cudaMemcpyAsync(di.p, idx_host, n * sizeof(int64_t), cudaMemcpyHostToDevice, h->stream));
  for (int64_t k0 = 0; k0 < n; k0 += 65535) {
    const int64_t nk = std::min<int64_t>(65535, n - k0);
    dim3 g((unsigned)std::min<int64_t>((row_len + 255) / 256, 256), (unsigned)nk);
    k_gather_rows_f32<<<g, 256, 0, h->stream>>>(src, di.p + k0, row_len, dst + k0 * row_len);
    count_launch(h);
  }
  PYB_CUDA(cudaStreamSynchronize(h->stream));
  PYB_CUDA(cudaGetLastError());
}

// The finishing tail shared by predict() and the streamed HMC predictive (hmc_predictive.cu): mean / population variance
// and, with uq, the classification-uncertainty matrices from the moment sums over the draws — s1 = sum w o, s2 = sum w o^2,
// S2 = sum w o o^T (device [Nt, C, C], C > 1 only), total weight wsum, labels y_dev on the device.  Outputs are host
// pointers (mean / var may be NULL); ends with a stream synchronisation and last_device_ms measured from ev0.
void predictive_finish(pyb_handle* h, const double* s1, const double* s2, const double* S2, double wsum, int64_t Nt,
                       const int32_t* y_dev, const UncertaintyReq* uq, float* mean, float* var) {
  const int64_t C = h->model.out_dim, elems = Nt * C;
  const int Ce = (C == 1) ? 2 : (int)C, CC = Ce * Ce;
  const int64_t nseg = (Nt + kUqSeg - 1) / kUqSeg;
  DevBuf<float> dmean, dvar;
  DevBuf<double> ua, ue, seg_a, seg_e, exc_a, exc_e;
  DevBuf<float> ut, uao, ueo;
  dmean.alloc(elems); dvar.alloc(elems);
  if (uq) {
    ua.alloc(Nt * CC); ue.alloc(Nt * CC); seg_a.alloc(nseg * CC); seg_e.alloc(nseg * CC); exc_a.alloc(nseg * CC); exc_e.alloc(nseg * CC);
    ut.alloc(Nt * CC); uao.alloc(Nt * CC); ueo.alloc(Nt * CC);
  }
  k_pred_finish<<<(unsigned)((elems + 255) / 256), 256, 0, h->stream>>>(s1, s2, wsum, elems, dmean.p, dvar.p);
  count_launch(h);
  if (uq) {
    k_uncert_rows<<<(unsigned)((Nt * CC + 255) / 256), 256, 0, h->stream>>>(s1, s2, S2, wsum, Nt, (int)C, Ce, y_dev,
                                                                           uq->cumulative ? 1 : 0, ua.p, ue.p);
    count_launch(h);
    if (uq->cumulative) {
      k_uncert_segsum<<<(unsigned)nseg, CC, 0, h->stream>>>(ua.p, Nt, CC, seg_a.p);
      k_uncert_segsum<<<(unsigned)nseg, CC, 0, h->stream>>>(ue.p, Nt, CC, seg_e.p);
      k_uncert_segscan<<<1, CC, 0, h->stream>>>(seg_a.p, exc_a.p, nseg, CC);
      k_uncert_segscan<<<1, CC, 0, h->stream>>>(seg_e.p, exc_e.p, nseg, CC);
      count_launch(h, 4);
    }
    k_uncert_finish<<<(unsigned)nseg, CC, 0, h->stream>>>(ua.p, ue.p, exc_a.p, exc_e.p, Nt, CC, uq->cumulative ? 1 : 0,
                                                         1.0 / uq->divisor, ut.p, uao.p, ueo.p);
    count_launch(h);
  }
  PYB_CUDA(cudaEventRecord(h->ev1, h->stream));
  if (uq) {
    PYB_CUDA(cudaMemcpyAsync(uq->total, ut.p, Nt * CC * sizeof(float), cudaMemcpyDeviceToHost, h->stream));
    PYB_CUDA(cudaMemcpyAsync(uq->aleatoric, uao.p, Nt * CC * sizeof(float), cudaMemcpyDeviceToHost, h->stream));
    PYB_CUDA(cudaMemcpyAsync(uq->epistemic, ueo.p, Nt * CC * sizeof(float), cudaMemcpyDeviceToHost, h->stream));
  }
  if (mean) PYB_CUDA(cudaMemcpyAsync(mean, dmean.p, elems * sizeof(float), cudaMemcpyDeviceToHost, h->stream));
  if (var) PYB_CUDA(cudaMemcpyAsync(var, dvar.p, elems * sizeof(float), cudaMemcpyDeviceToHost, h->stream));
  PYB_CUDA(cudaStreamSynchronize(h->stream));
  PYB_CUDA(cudaGetLastError());
  float ms = 0.f;
  PYB_CUDA(cudaEventElapsedTime(&ms, h->ev0, h->ev1));
  h->last_device_ms = ms;
}

void predict(pyb_handle* h, const float* W, int64_t n, const float* weight, const float* x, int64_t Nt,
             float* mean, float* var, float* all, const UncertaintyReq* uq) {
  PYB_REQUIRE(n > 0 && Nt > 0, PYB_ERR_INVALID, "n and Nt must be > 0");
  PYB_REQUIRE(W && x && (uq || (mean && var)), PYB_ERR_INVALID, "null pointer");
  const Model& m = h->model;
  const int64_t P = m.P, C = m.out_dim, elems = Nt * C;
  DevBuf<float> dW, dx, dw, dout;
  DevBuf<double> s1, s2;
  // classification-uncertainty accumulators [Nt, Ce, Ce] (Ce = 2 for a one-unit output)
  const int Ce = (C == 1) ? 2 : (int)C, CC = Ce * Ce;
  DevBuf<double> uS2;
  DevBuf<int32_t> uy;
  if (uq) {
    PYB_REQUIRE(uq->y && uq->total && uq->aleatoric && uq->epistemic, PYB_ERR_INVALID, "null pointer");
    PYB_REQUIRE(CC <= 1024, PYB_ERR_UNSUPPORTED, "classification uncertainty supports at most 32 classes");
    PYB_REQUIRE(uq->divisor != 0.0, PYB_ERR_INVALID, "divisor must not be 0");
    for (int64_t r = 0; r < Nt; ++r)
      PYB_REQUIRE(uq->y[r] >= 0 && uq->y[r] < Ce, PYB_ERR_INVALID, "label out of range");
    uy.alloc(Nt);
    if (C > 1) {
      uS2.alloc(Nt * CC);
      PYB_CUDA(cudaMemsetAsync(uS2.p, 0, Nt * CC * sizeof(double), h->stream));
    }
    PYB_CUDA(cudaMemcpyAsync(uy.p, uq->y, Nt * sizeof(int32_t), cudaMemcpyHostToDevice, h->stream));
  }
  // W and x may be host pointers (copied chunk by chunk) or device pointers (used in place: samples that already
  // live in HBM, e.g. DLPack tensors, skip the n*P*4-byte upload that otherwise dominates the call)
  const bool W_dev = is_device_ptr(W), x_dev = is_device_ptr(x);
  // caller-owned device memory (DLPack tensors) was produced on the CALLER's stream; this library works on its own
  // non-blocking stream, which is ordered against nothing else: wait for the device before reading (header: "device pointers")
  if (W_dev || x_dev) PYB_CUDA(cudaDeviceSynchronize());
  const float* xd = x;
  if (!x_dev) {
    dx.alloc(Nt * m.in_dim);
    PYB_CUDA(cudaMemcpyAsync(dx.p, x, Nt * m.in_dim * sizeof(float), cudaMemcpyHostToDevice, h->stream));
    xd = dx.p;
  }
  double wsum = 0.0;
  if (weight) {
    for (int64_t i = 0; i < n; ++i) wsum += weight[i];
    dw.alloc(n);
    PYB_CUDA(cudaMemcpyAsync(dw.p, weight, n * sizeof(float), cudaMemcpyHostToDevice, h->stream));
  } else {
    wsum = (double)n;
  }
  PYB_REQUIRE(wsum > 0.0, PYB_ERR_INVALID, "weights must sum to a positive value");
  // chunk of samples per pass: bounded by the generic workspace and a 512 MiB output buffer
  int64_t chunk = generic_chain_batch(h, n, Nt, false);
  int64_t out_cap = (int64_t)((512ull << 20) / (sizeof(float) * (size_t)elems));
  if (out_cap < 1) out_cap = 1;
  chunk = std::min(chunk, out_cap);
  if (!W_dev) dW.alloc(chunk * P);
  dout.alloc(chunk * elems);
  s1.alloc(elems); s2.alloc(elems);
  PYB_CUDA(cudaMemsetAsync(s1.p, 0, elems * sizeof(double), h->stream));
  PYB_CUDA(cudaMemsetAsync(s2.p, 0, elems * sizeof(double), h->stream));
  const bool use_tensor = tc_supported_rows(h, Nt) && (h->opt_path == PYB_PATH_AUTO || h->opt_path == PYB_PATH_TENSOR);
  h->path_used = use_tensor ? PYB_PATH_TENSOR : PYB_PATH_GENERIC;
  PYB_CUDA(cudaEventRecord(h->ev0, h->stream));
  for (int64_t i0 = 0; i0 < n; i0 += chunk) {
    int64_t nb = std::min(chunk, n - i0);
    const float* Wd = W + i0 * P;
    if (!W_dev) {
      PYB_CUDA(cudaMemcpyAsync(dW.p, W + i0 * P, nb * P * sizeof(float), cudaMemcpyHostToDevice, h->stream));
      Wd = dW.p;
    }
    if (use_tensor) tc_forward(h, Wd, nb, xd, Nt, dout.p);
    else generic_forward(h, Wd, nb, xd, Nt, dout.p);
    k_pred_accum<<<(unsigned)((elems + 255) / 256), 256, 0, h->stream>>>(dout.p, nb, elems, weight ? dw.p + i0 : nullptr,
                                                                         s1.p, s2.p);
    count_launch(h);
    if (uq && C > 1) uncert_s2_accum(h, dout.p, nb, Nt, (int)C, weight ? dw.p + i0 : nullptr, uS2.p);
    if (all) {
      k_nan_to_zero<<<(unsigned)std::min<int64_t>((nb * elems + 255) / 256, 4096), 256, 0, h->stream>>>(dout.p, nb * elems);
      count_launch(h);
      PYB_CUDA(cudaMemcpyAsync(all + i0 * elems, dout.p, nb * elems * sizeof(float), cudaMemcpyDeviceToHost, h->stream));
    }
  }
  // weight samples sharded over ranks (SURVEY 8e): the only exchange is the all-reduce of the moment sums
  // ([Nt, C] doubles, 0.8 MB each at C5) and of the total weight; per-draw outputs stay with the rank that made them
  if (h->opt_predict_sharded && h->svgd.nccl_comm && h->svgd.world > 1) {
    DevBuf<double> dws;
    dws.alloc(1);
    PYB_CUDA(cudaMemcpyAsync(dws.p, &wsum, sizeof(double), cudaMemcpyHostToDevice, h->stream));
    nccl_all_reduce_f64(h->svgd.nccl_comm, s1.p, (size_t)elems, h->stream);
    nccl_all_reduce_f64(h->svgd.nccl_comm, s2.p, (size_t)elems, h->stream);
    if (uq && C > 1) nccl_all_reduce_f64(h->svgd.nccl_comm, uS2.p, (size_t)(Nt * CC), h->stream);
    nccl_all_reduce_f64(h->svgd.nccl_comm, dws.p, 1, h->stream);
    PYB_CUDA(cudaMemcpyAsync(&wsum, dws.p, sizeof(double), cudaMemcpyDeviceToHost, h->stream));
    PYB_CUDA(cudaStreamSynchronize(h->stream));
  }
  predictive_finish(h, s1.p, s2.p, uS2.p, wsum, Nt, uy.p, uq, mean, var);
}

}  // namespace pyb
