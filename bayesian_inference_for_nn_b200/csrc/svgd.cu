// svgd.cu — SVGD for S particles at once.
//
// REFERENCE_LIVE  (SVGD.step SVGD.py:84-141 + _svgd_gradients :54-68 + rbf_kernel :183-202):
//   sequential Gauss-Seidel sweep; for particle i: g_i = grad of the minibatch MEAN loss (no prior,
//   no N scaling, :110-112), K_ik = exp(-||x_i-x_k||^2) in float64 with gamma = 1,
//   phi_i = ((sum_k K_ik) g_i + 2 sum_k K_ik (x_i - x_k)) / M in float32, legacy-Adam DESCENT on phi.
//   g_i only depends on theta_i, which nobody else modifies before its turn, so all S gradients
//   come from ONE batched evaluation; only the kernel row + Adam are sequential.
// CANONICAL_MEDIAN (SVGD.baseline__kernel SVGD.py:165-181; north_star's formula): Jacobi update,
//   d2 over all pairs, h^2 = 0.5 median(d2)/log(M+1) with the median over all M*M entries (exact
//   radix select, mean of the two middle order statistics), K = exp(-d2/2h^2),
//   phi = (K grad_logp + (-K X + X rowsum K)/h^2)/M, Adam ascent.
//
// Sharding: the kernels take the global particle matrix [S_tot, P] and a local row range, so the
// same code serves one GPU (row range = everything) and the all-gathered multi-GPU layout.
#include "common.cuh"
#include <cuda_bf16.h>
#include <cooperative_groups.h>
#include <math.h>
#include <algorithm>
#include <unistd.h>

namespace pyb {

// the Stein-update branch that ran last (info "svgd_stein_used")
enum SteinBranch { STEIN_LIVE_LAUNCHES = 0, STEIN_LIVE_COOP = 1, STEIN_LIVE_CTA = 2, STEIN_F64 = 3, STEIN_TENSOR = 4, STEIN_PSHARD = 5 };

__global__ void k_svgd_init(float* theta, const double* p0, const float* mu, const float* sigma, int64_t P,
                            uint64_t seed, int64_t offset) {
  int64_t s = blockIdx.y;
  int64_t base = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) * 4;
  if (base >= P) return;
  float z[4];
  if (p0) {
    for (int j = 0; j < 4; ++j) z[j] = (base + j < P) ? (float)p0[s * P + base + j] : 0.f;
  } else {
    philox_normal4((uint32_t)(base >> 2), (uint32_t)(offset + s), 0u, STREAM_INIT, seed, z);
    for (int j = 0; j < 4; ++j)
      if (base + j < P) z[j] = mu[base + j] + sigma[base + j] * z[j];  // one prior draw per element (SVGD.py:150-155)
  }
  for (int j = 0; j < 4; ++j)
    if (base + j < P) theta[s * P + base + j] = z[j];
}

__global__ void k_gather_rows(const float* X, const int32_t* y_i, const float* y_f, const int32_t* idx, int64_t B,
                              int D, int C, float* Xb, int32_t* yb_i, float* yb_f) {
  int64_t b = blockIdx.x;
  int64_t r = idx[b];
  for (int d = threadIdx.x; d < D; d += blockDim.x) Xb[b * D + d] = X[r * D + d];
  if (y_i && threadIdx.x == 0) yb_i[b] = y_i[r];
  if (y_f)
    for (int c = threadIdx.x; c < C; c += blockDim.x) yb_f[b * C + c] = y_f[r * C + c];
}

void gather_batch(pyb_handle* h, const int32_t* idx_dev, int64_t B, float* Xb, int32_t* yb_i, float* yb_f) {
  const Model& m = h->model;
  k_gather_rows<<<(unsigned)B, 128, 0, h->stream>>>(h->X.p, h->loss_kind == PYB_LOSS_SPARSE_CE ? h->y_i.p : nullptr,
                                                    h->loss_kind == PYB_LOSS_MSE ? h->y_f.p : nullptr, idx_dev, B,
                                                    m.in_dim, m.out_dim, Xb, yb_i, yb_f);
  count_launch(h);
}

// ---- live sweep ---------------------------------------------------------------------------
// Krow[k] = exp(-gamma * ||x_i - x_k||^2), float64; one block per k
__global__ void k_live_row(const float* theta, int64_t P, int i, double gamma, double* Krow) {
  __shared__ double scratch[32];
  int k = blockIdx.x;
  const float* xi = theta + (int64_t)i * P;
  const float* xk = theta + (int64_t)k * P;
  double a = 0.0;
  for (int64_t e = threadIdx.x; e < P; e += blockDim.x) {
    double d = (double)xi[e] - (double)xk[e];
    a += d * d;
  }
  double t = block_sum<double>(a, scratch);
  if (threadIdx.x == 0) Krow[k] = exp(-gamma * t);
}

__device__ inline float adam_update(float th, float g, float& m, float& v, float lr_t, float b1, float b2, float eh) {
  m = b1 * m + (1.0f - b1) * g;
  v = b2 * v + (1.0f - b2) * g * g;
  return th - lr_t * m / (sqrtf(v) + eh);
}

// phi_i[e] = (wsum*g_i[e] + 2 gamma sum_k K_ik (x_i[e]-x_k[e])) / M ; Adam descent on particle i
// theta holds ALL S particles (global order); g/am/av/phi_out hold only the local shard: row `il` of them
// belongs to global particle i
__global__ void k_live_update(float* theta, const float* g, float* am, float* av, float* phi_out, int64_t P,
                              int S, int i, int il, double gamma, const double* Krow, float lr_t) {
  __shared__ double Ks[1024];
  int64_t e = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  double xi = (e < P) ? (double)theta[(int64_t)i * P + e] : 0.0;
  double acc = 0.0;
  float wsum = 0.f;
  for (int k0 = 0; k0 < S; k0 += 1024) {
    int n = min(1024, S - k0);
    __syncthreads();
    for (int k = threadIdx.x; k < n; k += blockDim.x) Ks[k] = Krow[k0 + k];
    __syncthreads();
    if (e < P)
      for (int k = 0; k < n; ++k) acc += Ks[k] * (xi - (double)theta[(int64_t)(k0 + k) * P + e]);
    for (int k = 0; k < n; ++k) wsum += (float)Ks[k];
  }
  if (e < P) {
    const int64_t o = (int64_t)i * P + e, ol = (int64_t)il * P + e;
    float gk = (float)(2.0 * gamma * acc);
    float phi = (wsum * g[ol] + gk) / (float)S;
    if (phi_out) phi_out[ol] = phi;
    theta[o] = adam_update(theta[o], phi, am[ol], av[ol], lr_t, 0.9f, 0.999f, 1e-7f);
  }
}

// The whole sequential sweep of one step in ONE cooperative launch (single GPU): for i = 0..S-1 {kernel row of
// particle i against the current state; grid barrier; phi_i and the Adam step of particle i; grid barrier}.
// Same arithmetic, block shape and summation order as k_live_row / k_live_update (bit-identical results); what goes
// away is 2 S kernel launches per step (the reference's own configuration is launch-bound: S = 10..64, P = 252).
__global__ void __launch_bounds__(256) k_live_sweep(float* theta, const float* g, float* am, float* av, float* phi_out,
                                                    int64_t P, int S, double gamma, double* Krow, float lr_t) {
  namespace cg = cooperative_groups;
  cg::grid_group grid = cg::this_grid();
  __shared__ double scratch[32];
  __shared__ double Ks[1024];
  for (int i = 0; i < S; ++i) {
    // ---- K_ik for every k (one block per k, float64)
    const float* xi_row = theta + (int64_t)i * P;
    for (int k = blockIdx.x; k < S; k += gridDim.x) {
      const float* xk = theta + (int64_t)k * P;
      double a = 0.0;
      for (int64_t e = threadIdx.x; e < P; e += blockDim.x) {
        double d = (double)xi_row[e] - (double)xk[e];
        a += d * d;
      }
      double t = block_sum<double>(a, scratch);
      if (threadIdx.x == 0) Krow[k] = exp(-gamma * t);
      __syncthreads();
    }
    grid.sync();
    // ---- phi_i and the update of particle i (one thread per parameter)
    for (int64_t e0 = (int64_t)blockIdx.x * blockDim.x; e0 < P; e0 += (int64_t)gridDim.x * blockDim.x) {
      const int64_t e = e0 + threadIdx.x;
      double xi = (e < P) ? (double)theta[(int64_t)i * P + e] : 0.0;
      double acc = 0.0;
      float wsum = 0.f;
      for (int k0 = 0; k0 < S; k0 += 1024) {
        int n = min(1024, S - k0);
        __syncthreads();
        for (int k = threadIdx.x; k < n; k += blockDim.x) Ks[k] = Krow[k0 + k];
        __syncthreads();
        if (e < P)
          for (int k = 0; k < n; ++k) acc += Ks[k] * (xi - (double)theta[(int64_t)(k0 + k) * P + e]);
        for (int k = 0; k < n; ++k) wsum += (float)Ks[k];
      }
      if (e < P) {
        const int64_t o = (int64_t)i * P + e;
        float gk = (float)(2.0 * gamma * acc);
        float phi = (wsum * g[o] + gk) / (float)S;
        if (phi_out) phi_out[o] = phi;
        theta[o] = adam_update(theta[o], phi, am[o], av[o], lr_t, 0.9f, 0.999f, 1e-7f);
      }
    }
    grid.sync();
  }
}

// The same sweep in ONE CTA with the particles in shared memory, for the reference's own sizes (S = 10..64 particles of
// P = 252 parameters: 64 KB): the 2 S grid barriers of k_live_sweep (a few microseconds each) become __syncthreads.
// Kernel row: one warp per k, float64, lanes over the parameters; update: one thread per parameter, k in order — the
// arithmetic of k_live_update (the row sums are reduced in a different order than block_sum's: float64, ~1e-16).
__global__ void __launch_bounds__(1024) k_live_sweep_cta(float* theta, const float* __restrict__ g, float* am, float* av,
                                                         float* phi_out, int P, int S, double gamma, float lr_t) {
  extern __shared__ __align__(16) unsigned char live_raw[];
  double* Ks = reinterpret_cast<double*>(live_raw);            // [S]
  float* th = reinterpret_cast<float*>(Ks + S);                // [S][P]
  const int t = threadIdx.x, lane = t & 31, w = t >> 5, nw = blockDim.x >> 5;
  for (int idx = t; idx < S * P; idx += blockDim.x) th[idx] = theta[idx];
  __syncthreads();
  for (int i = 0; i < S; ++i) {
    const float* xi_row = th + i * P;
    // this particle's gradient and moments: in flight while the row and the sum over k are computed
    float gq[1] = {0.f}, mq[1] = {0.f}, vq[1] = {0.f};
    if (t < P) { gq[0] = g[i * P + t]; mq[0] = am[i * P + t]; vq[0] = av[i * P + t]; }
    for (int k = w; k < S; k += nw) {
      const float* xk = th + k * P;
      double a = 0.0;
      for (int e = lane; e < P; e += 32) {
        const double d = (double)xi_row[e] - (double)xk[e];
        a += d * d;
      }
      a = warp_sum(a);
      if (lane == 0) Ks[k] = exp(-gamma * a);
    }
    __syncthreads();
    for (int e = t; e < P; e += blockDim.x) {
      const double xi = (double)th[i * P + e];
      double acc = 0.0;
      float wsum = 0.f;
      for (int k = 0; k < S; ++k) {
        const double kk = Ks[k];
        acc += kk * (xi - (double)th[k * P + e]);
        wsum += (float)kk;
      }
      const int o = i * P + e;
      float gv = gq[0], m = mq[0], v = vq[0];
      if (e != t) { gv = g[o]; m = am[o]; v = av[o]; }          // P > 1024: the later columns of this thread
      const float gk = (float)(2.0 * gamma * acc);
      const float phi = (wsum * gv + gk) / (float)S;
      if (phi_out) phi_out[o] = phi;
      th[o] = adam_update(th[o], phi, m, v, lr_t, 0.9f, 0.999f, 1e-7f);
      am[o] = m; av[o] = v;
    }
    __syncthreads();
  }
  for (int idx = t; idx < S * P; idx += blockDim.x) theta[idx] = th[idx];
}

// ---- canonical (Jacobi) -------------------------------------------------------------------
// d2[i][j] for local rows i in [r0, r0+Sl), all j in [0, St): direct difference form in float64
// (what scipy pdist computes), 16x16 output tile per block, P streamed through shared memory.
__global__ void __launch_bounds__(256) k_gram_d2(const float* X, int64_t P, int r0, int Sl, int St, double* d2) {
  __shared__ float xi[16][65], xj[16][65];
  int ti = threadIdx.x >> 4, tj = threadIdx.x & 15;
  int i = blockIdx.y * 16 + ti, j = blockIdx.x * 16 + tj;
  double acc = 0.0;
  for (int64_t e0 = 0; e0 < P; e0 += 64) {
    for (int t = threadIdx.x; t < 16 * 64; t += 256) {
      int r = t >> 6, c = t & 63;
      int gi = blockIdx.y * 16 + r, gj = blockIdx.x * 16 + r;
      xi[r][c] = (gi < Sl && e0 + c < P) ? X[(int64_t)(r0 + gi) * P + e0 + c] : 0.f;
      xj[r][c] = (gj < St && e0 + c < P) ? X[(int64_t)gj * P + e0 + c] : 0.f;
    }
    __syncthreads();
#pragma unroll 8
    for (int c = 0; c < 64; ++c) {
      double d = (double)xi[ti][c] - (double)xj[tj][c];
      acc += d * d;
    }
    __syncthreads();
  }
  if (i < Sl && j < St) d2[(int64_t)i * St + j] = acc;
}

// radix select over the bit patterns of non-negative doubles (monotone as uint64)
struct SelectState { unsigned long long prefix, mask, k; };
__global__ void k_select_hist(const double* v, int64_t n, const SelectState* st, int shift, unsigned long long* hist) {
  __shared__ unsigned int h[256];
  for (int t = threadIdx.x; t < 256; t += blockDim.x) h[t] = 0;
  __syncthreads();
  unsigned long long prefix = st->prefix, mask = st->mask;
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x) {
    unsigned long long b = (unsigned long long)__double_as_longlong(v[i]);
    if ((b & mask) == prefix) atomicAdd(&h[(b >> shift) & 0xff], 1u);
  }
  __syncthreads();
  for (int t = threadIdx.x; t < 256; t += blockDim.x)
    if (h[t]) atomicAdd(&hist[t], (unsigned long long)h[t]);
}
__global__ void k_select_pick(SelectState* st, int shift, unsigned long long* hist) {
  if (threadIdx.x == 0) {
    unsigned long long k = st->k, c = 0;
    int b = 0;
    for (; b < 256; ++b) {
      if (c + hist[b] > k) break;
      c += hist[b];
    }
    if (b > 255) b = 255;
    st->k = k - c;
    if (shift == 0) st[1].k = hist[b];          // all 64 bits fixed: how many elements EQUAL the selected value
    st->prefix |= ((unsigned long long)b) << shift;
    st->mask |= 0xffull << shift;
  }
  __syncthreads();
  for (int t = threadIdx.x; t < 256; t += blockDim.x) hist[t] = 0;
}
// smallest bit pattern strictly above the selected value (the next order statistic when the selected value is the last
// of its group of equals); nxt is initialised to ~0
__global__ void k_next_greater(const double* v, int64_t n, const SelectState* st, unsigned long long* nxt) {
  const unsigned long long sel = st->prefix;
  unsigned long long m = ~0ull;
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x) {
    const unsigned long long b = (unsigned long long)__double_as_longlong(v[i]);
    if (b > sel && b < m) m = b;
  }
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) {
    const unsigned long long t = __shfl_xor_sync(0xffffffffu, m, o);
    m = t < m ? t : m;
  }
  if ((threadIdx.x & 31) == 0 && m != ~0ull) atomicMin(nxt, m);
}
// After the two leading passes the candidates (elements that share the 16 fixed top bits: sign, exponent and four mantissa
// bits — a sixteenth of an octave) are a small fraction of the matrix: they are copied out once, the remaining six passes
// and the next-greater search run over the copy.  Three passes over the matrix instead of ten.  The same scan finds the
// smallest element ABOVE the candidates' bucket (the next order statistic when the selected value is the bucket's largest).
__global__ void k_select_compact(const double* v, int64_t n, const SelectState* st, unsigned long long* cand,
                                 unsigned long long* cnt, unsigned long long* nxt) {
  const unsigned long long prefix = st->prefix, mask = st->mask, top = prefix | ~mask;
  const int lane = threadIdx.x & 31;
  unsigned long long m = ~0ull;
  for (int64_t base = (int64_t)blockIdx.x * blockDim.x; base < n; base += (int64_t)gridDim.x * blockDim.x) {
    const int64_t i = base + threadIdx.x;
    const bool valid = i < n;
    const unsigned long long b = valid ? (unsigned long long)__double_as_longlong(v[i]) : 0ull;
    const bool in = valid && (b & mask) == prefix;
    const unsigned ballot = __ballot_sync(0xffffffffu, in);
    if (ballot) {
      unsigned long long off = 0;
      if (lane == 0) off = atomicAdd(cnt, (unsigned long long)__popc(ballot));
      off = __shfl_sync(0xffffffffu, off, 0);
      if (in) cand[off + __popc(ballot & ((1u << lane) - 1u))] = b;
    }
    if (valid && b > top && b < m) m = b;
  }
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) {
    const unsigned long long t = __shfl_xor_sync(0xffffffffu, m, o);
    m = t < m ? t : m;
  }
  if (lane == 0 && m != ~0ull) atomicMin(nxt, m);
}
__global__ void k_select_hist_keys(const unsigned long long* keys, const unsigned long long* n_ptr, const SelectState* st, int shift,
                                   unsigned long long* hist) {
  __shared__ unsigned int h[256];
  for (int t = threadIdx.x; t < 256; t += blockDim.x) h[t] = 0;
  __syncthreads();
  const unsigned long long prefix = st->prefix, mask = st->mask;
  const int64_t n = (int64_t)n_ptr[0];
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x) {
    const unsigned long long b = keys[i];
    if ((b & mask) == prefix) atomicAdd(&h[(b >> shift) & 0xff], 1u);
  }
  __syncthreads();
  for (int t = threadIdx.x; t < 256; t += blockDim.x)
    if (h[t]) atomicAdd(&hist[t], (unsigned long long)h[t]);
}
__global__ void k_next_greater_keys(const unsigned long long* keys, const unsigned long long* n_ptr, const SelectState* st,
                                    unsigned long long* nxt) {
  const unsigned long long sel = st->prefix;
  const int64_t n = (int64_t)n_ptr[0];
  unsigned long long m = ~0ull;
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x) {
    const unsigned long long b = keys[i];
    if (b > sel && b < m) m = b;
  }
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) {
    const unsigned long long t = __shfl_xor_sync(0xffffffffu, m, o);
    m = t < m ? t : m;
  }
  if ((threadIdx.x & 31) == 0 && m != ~0ull) atomicMin(nxt, m);
}
// ---- the plain eight-pass select with HALF the kernels (in the sharded step it runs beside persistent kernels that own
//      every SM: each of its kernels can only start at one of their boundaries, so the chain's length is its kernel
//      count): every pass picks the previous digit itself, from the previous pass's own histogram ----
// one radix digit of a select state from a 256-bin histogram in shared memory (the arithmetic of k_select_pick)
__device__ __forceinline__ SelectState select_pick_local(SelectState s, const unsigned long long* hs, int shift,
                                                         unsigned long long* group) {
  unsigned long long c = 0;
  int b = 0;
  for (; b < 256; ++b) {
    if (c + hs[b] > s.k) break;
    c += hs[b];
  }
  if (b > 255) b = 255;
  s.k -= c;
  if (group) *group = hs[b];
  s.prefix |= ((unsigned long long)b) << shift;
  s.mask |= 0xffull << shift;
  return s;
}
// every block picks digit `shift_prev` from hist_prev itself (identical everywhere), block 0 records the state
__device__ __forceinline__ SelectState select_advance(const SelectState* st_in, const unsigned long long* hist_prev, int shift_prev,
                                                      SelectState* st_out, unsigned long long* hs, SelectState* cur) {
  for (int t = threadIdx.x; t < 256; t += blockDim.x) hs[t] = hist_prev[t];
  __syncthreads();
  if (threadIdx.x == 0) {
    *cur = select_pick_local(*st_in, hs, shift_prev, nullptr);
    if (blockIdx.x == 0) *st_out = *cur;
  }
  __syncthreads();
  return *cur;
}
// pass `shift` over the whole set with the previous digit picked on the fly
__global__ void k_select_hist_adv(const double* v, int64_t n, const SelectState* st_in, const unsigned long long* hist_prev,
                                  int shift_prev, SelectState* st_out, int shift, unsigned long long* hist) {
  __shared__ unsigned long long hs[256];
  __shared__ SelectState cur;
  __shared__ unsigned int h[256];
  const SelectState s = select_advance(st_in, hist_prev, shift_prev, st_out, hs, &cur);
  for (int t = threadIdx.x; t < 256; t += blockDim.x) h[t] = 0;
  __syncthreads();
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x) {
    const unsigned long long b = (unsigned long long)__double_as_longlong(v[i]);
    if ((b & s.mask) == s.prefix) atomicAdd(&h[(b >> shift) & 0xff], 1u);
  }
  __syncthreads();
  for (int t = threadIdx.x; t < 256; t += blockDim.x)
    if (h[t]) atomicAdd(&hist[t], (unsigned long long)h[t]);
}
// the LAST digit picked on the fly (block 0 records the final state and the size of the selected value's group of equals),
// then the search for the smallest element above the selected value
__global__ void k_next_greater_adv(const double* v, int64_t n, const SelectState* st_in, const unsigned long long* hist_prev,
                                   SelectState* st_final, int want_next, unsigned long long* nxt) {
  __shared__ unsigned long long hs[256];
  __shared__ SelectState cur;
  for (int t = threadIdx.x; t < 256; t += blockDim.x) hs[t] = hist_prev[t];
  __syncthreads();
  if (threadIdx.x == 0) {
    unsigned long long group = 0;
    cur = select_pick_local(*st_in, hs, 0, &group);
    if (blockIdx.x == 0) { st_final[0] = cur; st_final[1].k = group; }
  }
  __syncthreads();
  if (!want_next) return;
  const unsigned long long sel = cur.prefix;
  unsigned long long m = ~0ull;
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x) {
    const unsigned long long b = (unsigned long long)__double_as_longlong(v[i]);
    if (b > sel && b < m) m = b;
  }
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) {
    const unsigned long long t = __shfl_xor_sync(0xffffffffu, m, o);
    m = t < m ? t : m;
  }
  if ((threadIdx.x & 31) == 0 && m != ~0ull) atomicMin(nxt, m);
}
// K = exp(-d2 / (2 h2)) of one row per block: row sum (float64, block_sum's order) and the bf16 hi / lo split of (float)K in
// one pass (k_kernel_rowsum + k_double_to_float + the row split); d2 is left untouched
__global__ void k_kernel_rowsum_split(const double* d2, int St, const double* h2, double* rowsum, __nv_bfloat16* kh,
                                      __nv_bfloat16* kl) {
  __shared__ double scratch[32];
  const int i = blockIdx.x;
  const double inv = 1.0 / (2.0 * h2[0]);
  double a = 0.0;
  for (int j = threadIdx.x; j < St; j += blockDim.x) {
    const double k = exp(-d2[(int64_t)i * St + j] * inv);
    a += k;
    const float kf = (float)k;
    const __nv_bfloat16 hi = __float2bfloat16_rn(kf);
    kh[(int64_t)i * St + j] = hi;
    kl[(int64_t)i * St + j] = __float2bfloat16_rn(kf - __bfloat162float(hi));
  }
  const double t = block_sum<double>(a, scratch);
  if (threadIdx.x == 0) rowsum[i] = t;
}
// a: the select state of order statistic k0 = (n - 1) / 2 (prefix = its bits, k = its index inside its group of equals,
// a[1].k = size of that group); the next order statistic is the same value unless k0 was the last of the group
__global__ void k_bandwidth_next(const SelectState* a, const unsigned long long* nxt, int want_next, int St, double* h2_out) {
  const double lo = __longlong_as_double((long long)a->prefix);
  double hi = lo;
  if (want_next && a->k + 1 >= a[1].k) hi = __longlong_as_double((long long)nxt[0]);
  double med = 0.5 * (lo + hi);
  h2_out[0] = 0.5 * med / log((double)St + 1.0);
  h2_out[1] = med;
}
// K = exp(-d2/(2 h2)) in place; rowsum per local row (one block per row)
__global__ void k_kernel_rowsum(double* d2, int St, const double* h2, double* rowsum) {
  __shared__ double scratch[32];
  int i = blockIdx.x;
  double inv = 1.0 / (2.0 * h2[0]);
  double a = 0.0;
  for (int j = threadIdx.x; j < St; j += blockDim.x) {
    double k = exp(-d2[(int64_t)i * St + j] * inv);
    d2[(int64_t)i * St + j] = k;
    a += k;
  }
  double t = block_sum<double>(a, scratch);
  if (threadIdx.x == 0) rowsum[i] = t;
}

// phi[i][e] = ( sum_j K[i][j] (G[j][e] - X[j][e]/h2) + X[i][e] rowsum[i]/h2 ) / St     (float64 accumulate)
__global__ void __launch_bounds__(256) k_phi_canonical(const double* K, const float* X, const float* G, int64_t P,
                                                        int r0, int Sl, int St, const double* h2,
                                                        const double* rowsum, float* phi) {
  __shared__ double Ks[8][128];
  int64_t e = (int64_t)blockIdx.x * 256 + threadIdx.x;
  int i0 = blockIdx.y * 8;
  double inv_h2 = 1.0 / h2[0];
  double acc[8];
#pragma unroll
  for (int r = 0; r < 8; ++r) acc[r] = 0.0;
  for (int j0 = 0; j0 < St; j0 += 128) {
    int n = min(128, St - j0);
    __syncthreads();
    for (int t = threadIdx.x; t < 8 * 128; t += 256) {
      int r = t >> 7, c = t & 127;
      Ks[r][c] = (i0 + r < Sl && c < n) ? K[(int64_t)(i0 + r) * St + j0 + c] : 0.0;
    }
    __syncthreads();
    if (e < P)
      for (int c = 0; c < n; ++c) {
        int64_t o = (int64_t)(j0 + c) * P + e;
        double y = (double)G[o] - (double)X[o] * inv_h2;
#pragma unroll
        for (int r = 0; r < 8; ++r) acc[r] += Ks[r][c] * y;
      }
  }
  if (e < P)
#pragma unroll
    for (int r = 0; r < 8; ++r)
      if (i0 + r < Sl) {
        double xi = (double)X[(int64_t)(r0 + i0 + r) * P + e];
        phi[(int64_t)(i0 + r) * P + e] = (float)((acc[r] + xi * rowsum[i0 + r] * inv_h2) / (double)St);
      }
}

// live-formula phi evaluated Jacobi-style for every row (parity hook): gamma fixed, float64 kernel
__global__ void k_kernel_fixed_rowsum(double* d2, int St, double gamma, double* rowsum) {
  __shared__ double scratch[32];
  int i = blockIdx.x;
  double a = 0.0;
  for (int j = threadIdx.x; j < St; j += blockDim.x) {
    double k = exp(-gamma * d2[(int64_t)i * St + j]);
    d2[(int64_t)i * St + j] = k;
    a += (double)(float)k;
  }
  double t = block_sum<double>(a, scratch);
  if (threadIdx.x == 0) rowsum[i] = t;
}
__global__ void __launch_bounds__(256) k_phi_live_all(const double* K, const float* X, const float* G, int64_t P,
                                                       int S, double gamma, const double* rowsum, float* phi) {
  int64_t e = (int64_t)blockIdx.x * 256 + threadIdx.x;
  int i = blockIdx.y;
  if (e >= P) return;
  double xi = (double)X[(int64_t)i * P + e], acc = 0.0;
  for (int k = 0; k < S; ++k) acc += K[(int64_t)i * S + k] * (xi - (double)X[(int64_t)k * P + e]);
  float gk = (float)(2.0 * gamma * acc);
  phi[(int64_t)i * P + e] = ((float)rowsum[i] * G[(int64_t)i * P + e] + gk) / (float)S;
}

// ---- tensor-core variant of the canonical update (large S): Gram and K*Y as bf16x3 GEMMs ---------
// The particles enter the Gram matrix, the norms and the Stein term X/h2 as x - c, c = their mean over the St rows: d2 and
// phi are translation-invariant, but d2 = n_i + n_j - 2 G_ij and K (X/h2) - X_i rowsum_i/h2 cancel to O((|c|/spread)^2)
// of the fp32 / bf16x3 rounding when the particles sit close together far from the origin.
// c[p] = mean over the R rows of column p of X [R, C] (row pitch C), summed in float64 in a fixed order; grid ceil(C/32),
// block (32, 8)
__global__ void k_col_mean(const float* __restrict__ X, int R, int64_t C, float* __restrict__ c) {
  __shared__ double part[8][32];
  const int64_t col = (int64_t)blockIdx.x * 32 + threadIdx.x;
  double a = 0.0;
  if (col < C)
    for (int r = threadIdx.y; r < R; r += 8) a += (double)X[(int64_t)r * C + col];
  part[threadIdx.y][threadIdx.x] = a;
  __syncthreads();
  if (threadIdx.y == 0 && col < C) {
    for (int k = 1; k < 8; ++k) a += part[k][threadIdx.x];
    c[col] = (float)(a / (double)R);
  }
}
// squared norms of the centred rows
__global__ void k_row_norms(const float* X, int64_t P, const float* __restrict__ center, double* norms) {
  __shared__ double scratch[32];
  const float* x = X + (int64_t)blockIdx.x * P;
  double a = 0.0;
  for (int64_t e = threadIdx.x; e < P; e += blockDim.x) {
    const double d = (double)(x[e] - center[e]);
    a += d * d;
  }
  double t = block_sum<double>(a, scratch);
  if (threadIdx.x == 0) norms[blockIdx.x] = t;
}
// d2[i][j] = max(n_{r0+i} + n_j - 2 G[i][j], 0); exact zero on the diagonal (pdist has d(x,x) = 0)
// hist56 != nullptr: also the 256-bin histogram of the results' top bytes — the first pass of the median's radix select
__global__ void k_d2_from_gram(const float* G, const double* norms, int r0, int Sl, int St, double* d2,
                               unsigned long long* hist56 = nullptr) {
  __shared__ unsigned int hb[256];
  if (hist56) {
    for (int t = threadIdx.x; t < 256; t += blockDim.x) hb[t] = 0;
    __syncthreads();
  }
  int64_t idx = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (idx < (int64_t)Sl * St) {
    int i = (int)(idx / St), j = (int)(idx - (int64_t)i * St);
    double v = norms[r0 + i] + norms[j] - 2.0 * (double)G[idx];
    v = (j == r0 + i || v < 0.0) ? 0.0 : v;
    d2[idx] = v;
    if (hist56) atomicAdd(&hb[((unsigned long long)__double_as_longlong(v)) >> 56], 1u);
  }
  if (hist56) {
    __syncthreads();
    for (int t = threadIdx.x; t < 256; t += blockDim.x)
      if (hb[t]) atomicAdd(&hist56[t], (unsigned long long)hb[t]);
  }
}
__global__ void k_double_to_float(const double* a, float* b, int64_t n) {
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x)
    b[i] = (float)a[i];
}
// Y = G - X / h2   (row-major [St, P])
__global__ void k_stein_rhs(const float* X, const float* G, const double* h2, int64_t n, float* Y) {
  const float inv = (float)(1.0 / h2[0]);
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x)
    Y[i] = G[i] - X[i] * inv;
}
// phi = (KY + (X_i - c) rowsum_i / h2) / St   in place on the GEMM output (fp32: the GEMM output already is)
__global__ void k_phi_finish(float* phi, const float* X, int64_t P, int r0, int St, const double* h2, const double* rowsum,
                             const float* __restrict__ center) {
  const int i = blockIdx.y;
  const float c = (float)(rowsum[i] / h2[0]), inv = 1.0f / (float)St;
  for (int64_t e = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; e < P; e += (int64_t)gridDim.x * blockDim.x) {
    int64_t o = (int64_t)i * P + e;
    phi[o] = fmaf(X[(int64_t)(r0 + i) * P + e] - center[e], c, phi[o]) * inv;
  }
}
// the same followed by the Adam ascent step on the local particles (theta_local = rows [r0, r0+Sl) of X): one pass
// over phi / theta / m / v instead of two (the training step does not need phi afterwards)
__device__ inline float adam_update(float th, float g, float& m, float& v, float lr_t, float b1, float b2, float eh);
// Flat [Sl*P] indexing: a thread's four elements are one 16-byte access per stream (7 streams: ky, theta, m, v read;
// theta, m, v written) whatever P is; they may straddle two particle rows, so the row constant is looked up per element.
// The Stein term uses the centred particle theta - center[e]; the Adam step is applied to theta itself.
__global__ void __launch_bounds__(256) k_phi_finish_adam(const float* __restrict__ ky, float* __restrict__ theta_local,
                                                         float* __restrict__ am, float* __restrict__ av, int64_t P,
                                                         int64_t total, int St, const double* __restrict__ h2,
                                                         const double* __restrict__ rowsum,
                                                         const float* __restrict__ center, float lr_t) {
  const int64_t base = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) * 4;
  if (base >= total) return;
  const float inv = 1.0f / (float)St;
  const double ih2 = 1.0 / h2[0];
  int64_t i = base / P;
  int64_t e = base - i * P;
  float c = (float)(rowsum[i] * ih2);
  if (base + 4 <= total) {
    const float4 k4 = *reinterpret_cast<const float4*>(ky + base);
    const float4 t4 = *reinterpret_cast<const float4*>(theta_local + base);
    float4 m4 = *reinterpret_cast<const float4*>(am + base);
    float4 v4 = *reinterpret_cast<const float4*>(av + base);
    float kk[4] = {k4.x, k4.y, k4.z, k4.w}, tt[4] = {t4.x, t4.y, t4.z, t4.w};
    float mm[4] = {m4.x, m4.y, m4.z, m4.w}, vv[4] = {v4.x, v4.y, v4.z, v4.w};
#pragma unroll
    for (int j = 0; j < 4; ++j) {
      const float phi = fmaf(tt[j] - center[e], c, kk[j]) * inv;
      tt[j] = adam_update(tt[j], -phi, mm[j], vv[j], lr_t, 0.9f, 0.999f, 1e-7f);
      if (++e == P) { e = 0; ++i; if (j < 3) c = (float)(rowsum[i] * ih2); }
    }
    *reinterpret_cast<float4*>(theta_local + base) = make_float4(tt[0], tt[1], tt[2], tt[3]);
    *reinterpret_cast<float4*>(am + base) = make_float4(mm[0], mm[1], mm[2], mm[3]);
    *reinterpret_cast<float4*>(av + base) = make_float4(vv[0], vv[1], vv[2], vv[3]);
  } else {
    for (int64_t o = base; o < total; ++o) {
      const float th = theta_local[o];
      const float phi = fmaf(th - center[e], c, ky[o]) * inv;
      theta_local[o] = adam_update(th, -phi, am[o], av[o], lr_t, 0.9f, 0.999f, 1e-7f);
      if (++e == P) { e = 0; ++i; if (o + 1 < total) c = (float)(rowsum[i] * ih2); }
    }
  }
}

// Y^T = (G - (X - c)/h2)^T split into bf16 hi/lo [P, St] (K-major operand of the K*Y GEMM) in one pass.
// mu != nullptr: G holds the raw scaled loss gradient and the log-posterior gradient is formed here,
// G_eff = -(G + (X - mu) inv_var) — the separate k_glogp pass (one more read and write of [St, P]) goes away.
// grid (ceil(P/32), ceil(St/64)), block (32, 8): a warp stores 64 particles x 2 bytes = one 128-byte line per parameter
__global__ void k_stein_rhs_split_t(const float* __restrict__ X, const float* __restrict__ G, const double* h2, int St,
                                    int64_t P, uint16_t* __restrict__ hi, uint16_t* __restrict__ lo, int64_t ldd,
                                    const float* __restrict__ mu, const float* __restrict__ inv_var,
                                    const float* __restrict__ center) {
  __shared__ float tile[64][33];
  const float inv = (float)(1.0 / h2[0]);
  const int64_t c0 = (int64_t)blockIdx.x * 32;
  const int r0 = blockIdx.y * 64;
  const int64_t c = c0 + threadIdx.x;
  float m = 0.f, iv = 0.f, cc = 0.f;
  if (mu && c < P) { m = mu[c]; iv = inv_var[c]; }
  if (c < P) cc = center[c];
#pragma unroll
  for (int i = threadIdx.y; i < 64; i += 8) {
    const int r = r0 + i;
    float v = 0.f;
    if (r < St && c < P) {
      const float x = X[(int64_t)r * P + c];
      float g = G[(int64_t)r * P + c];
      if (mu) g = -(g + (x - m) * iv);
      v = g - (x - cc) * inv;
    }
    tile[i][threadIdx.x] = v;
  }
  __syncthreads();
  for (int i = threadIdx.y; i < 32; i += 8) {
    const int64_t cc = c0 + i;
    const int r = r0 + 2 * threadIdx.x;
    if (cc < P && r < St) {
      const float v0 = tile[2 * threadIdx.x][i], v1 = tile[2 * threadIdx.x + 1][i];
      const __nv_bfloat16 h0 = __float2bfloat16_rn(v0), h1 = __float2bfloat16_rn(v1);
      const __nv_bfloat16 l0 = __float2bfloat16_rn(v0 - __bfloat162float(h0));
      const __nv_bfloat16 l1 = __float2bfloat16_rn(v1 - __bfloat162float(h1));
      if (r + 1 < St && ((cc * ldd + r) & 1) == 0) {
        *reinterpret_cast<uint32_t*>(hi + cc * ldd + r) = (uint32_t)__bfloat16_as_ushort(h0) | ((uint32_t)__bfloat16_as_ushort(h1) << 16);
        *reinterpret_cast<uint32_t*>(lo + cc * ldd + r) = (uint32_t)__bfloat16_as_ushort(l0) | ((uint32_t)__bfloat16_as_ushort(l1) << 16);
      } else {
        hi[cc * ldd + r] = __bfloat16_as_ushort(h0);
        lo[cc * ldd + r] = __bfloat16_as_ushort(l0);
        if (r + 1 < St) { hi[cc * ldd + r + 1] = __bfloat16_as_ushort(h1); lo[cc * ldd + r + 1] = __bfloat16_as_ushort(l1); }
      }
    }
  }
}

// glogp = -(g + (theta-mu)/sigma^2)   (g already scaled by n_train)
__global__ void k_glogp(float* g, const float* theta, const float* mu, const float* inv_var, int64_t P) {
  int64_t s = blockIdx.y;
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < P; i += (int64_t)gridDim.x * blockDim.x) {
    int64_t o = s * P + i;
    g[o] = -(g[o] + (theta[o] - mu[i]) * inv_var[i]);
  }
}

__global__ void k_adam_all(float* theta, const float* phi, float* am, float* av, int64_t n, float sign, float lr_t) {
  for (int64_t o = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; o < n; o += (int64_t)gridDim.x * blockDim.x)
    theta[o] = adam_update(theta[o], sign * phi[o], am[o], av[o], lr_t, 0.9f, 0.999f, 1e-7f);
}

__global__ void k_mean_float(const float* v, int64_t n, double* out) {
  __shared__ double scratch[32];
  double a = 0.0;
  for (int64_t i = threadIdx.x; i < n; i += blockDim.x) a += (double)v[i];
  double t = block_sum<double>(a, scratch);
  if (threadIdx.x == 0) out[0] = t / (double)n;
}

// ------------------------------------------------------------------------------------------
static double adam_lr_t(double lr, int64_t t) {
  return lr * sqrt(1.0 - pow(0.999, (double)t)) / (1.0 - pow(0.9, (double)t));
}

// exact median bandwidth of d2 [n] (device, float64) -> h2 (device double[2] = {h2, median})
// exact median over the GLOBAL set of St*St distances; each rank histograms its own rows and the 256-bin
// histograms are all-reduced (2 KB per pass), so every rank picks the same bins
// reduce = false: d2 already IS the global set on every rank (bit-identical after the Gram all-reduce), so the select runs
// without any collective and still picks the same value everywhere
// The select of a LOCAL set with half the kernels: hist56_done = the caller's distance kernel has already filled histogram 0
// with the top bytes (after median_prepare_fused zeroed the buffers).  Eight histograms, three state slots.
static void median_prepare_fused(pyb_handle* h, int64_t n_global) {
  SvgdState& sc = h->svgd;
  sc.sel.alloc(16);
  sc.hist.alloc(256 * 8);
  SelectState init[2];
  init[0].prefix = 0; init[0].mask = 0; init[0].k = (unsigned long long)((n_global - 1) / 2);
  init[1].prefix = 0; init[1].mask = 0; init[1].k = 0;
  PYB_CUDA(cudaMemsetAsync(sc.hist.p, 0, 256 * 8 * sizeof(unsigned long long), h->stream));
  PYB_CUDA(cudaMemsetAsync(sc.sel.p + 6, 0xff, sizeof(unsigned long long), h->stream));   // slot 6: the next-greater minimum
  PYB_CUDA(cudaMemcpyAsync(sc.sel.p, init, sizeof(init), cudaMemcpyHostToDevice, h->stream));
}
static void median_bandwidth_fused(pyb_handle* h, const double* d2, int64_t n, int St, double* h2_dev, bool hist56_done) {
  SvgdState& sc = h->svgd;
  SelectState* st0 = reinterpret_cast<SelectState*>(sc.sel.p);            // initial and, at the end, final state (+ st0[1].k)
  SelectState* alt[2] = {reinterpret_cast<SelectState*>(sc.sel.p + 8), reinterpret_cast<SelectState*>(sc.sel.p + 11)};
  unsigned long long* nxt = sc.sel.p + 6;
  unsigned long long* H = sc.hist.p;
  const int want_next = (n / 2) != ((n - 1) / 2);
  const int blocks = (int)std::min<int64_t>((n + 255) / 256, 4 * (int64_t)h->sm_count);
  if (!hist56_done) k_select_hist<<<blocks, 256, 0, h->stream>>>(d2, n, st0, 56, H);
  const SelectState* in = st0;
  for (int p = 1; p <= 7; ++p) {
    SelectState* out = alt[p & 1];
    k_select_hist_adv<<<blocks, 256, 0, h->stream>>>(d2, n, in, H + (p - 1) * 256, 64 - 8 * p, out, 56 - 8 * p, H + p * 256);
    in = out;
  }
  k_next_greater_adv<<<blocks, 256, 0, h->stream>>>(d2, n, in, H + 7 * 256, st0, want_next, nxt);
  k_bandwidth_next<<<1, 1, 0, h->stream>>>(st0, nxt, want_next, St, h2_dev);
  count_launch(h, hist56_done ? 9 : 10);
}

static void median_bandwidth(pyb_handle* h, const double* d2, int64_t n, int64_t n_global, int St, double* h2_dev,
                             bool reduce = true) {
  SvgdState& sc = h->svgd;
  if (!(sc.world > 1 && reduce) && h->opt_select_compact == 2) {
    median_prepare_fused(h, n_global);
    median_bandwidth_fused(h, d2, n, St, h2_dev, false);
    return;
  }
  sc.sel.alloc(16);
  sc.hist.alloc(256 * 8);
  // ONE radix select for the lower middle order statistic (8 passes, each with a 2 KB histogram all-reduce when the
  // rows are sharded); the upper middle one is the same value or the next greater element (one more pass, one all-reduce
  // MIN) — half the latency-bound small collectives of two independent selects
  SelectState init[2];
  init[0].prefix = 0; init[0].mask = 0; init[0].k = (unsigned long long)((n_global - 1) / 2);
  init[1].prefix = 0; init[1].mask = 0; init[1].k = 0;
  const int want_next = (n_global / 2) != ((n_global - 1) / 2);
  PYB_CUDA(cudaMemcpyAsync(sc.sel.p, init, sizeof(init), cudaMemcpyHostToDevice, h->stream));
  PYB_CUDA(cudaMemsetAsync(sc.hist.p, 0, 256 * sizeof(unsigned long long), h->stream));
  PYB_CUDA(cudaMemsetAsync(sc.sel.p + 6, 0xff, sizeof(unsigned long long), h->stream));     // slot 6: the next-greater minimum
  int blocks = (int)std::min<int64_t>((n + 255) / 256, 4 * (int64_t)h->sm_count);
  if (!(sc.world > 1 && reduce) && n >= 4096 && h->opt_select_compact == 1) {
    // the whole set is here: two passes over it, one compaction, the rest over the candidates (one kernel per step)
    SelectState* st = reinterpret_cast<SelectState*>(sc.sel.p);
    unsigned long long* nxt = sc.sel.p + 6;
    unsigned long long* cnt = sc.sel.p + 7;
    sc.cand.alloc((size_t)n);
    PYB_CUDA(cudaMemsetAsync(cnt, 0, sizeof(unsigned long long), h->stream));
    for (int shift = 56; shift >= 48; shift -= 8) {
      k_select_hist<<<blocks, 256, 0, h->stream>>>(d2, n, st, shift, sc.hist.p);
      k_select_pick<<<1, 256, 0, h->stream>>>(st, shift, sc.hist.p);
    }
    k_select_compact<<<blocks, 256, 0, h->stream>>>(d2, n, st, sc.cand.p, cnt, nxt);
    const int kb = 2 * h->sm_count;
    for (int shift = 40; shift >= 0; shift -= 8) {
      k_select_hist_keys<<<kb, 256, 0, h->stream>>>(sc.cand.p, cnt, st, shift, sc.hist.p);
      k_select_pick<<<1, 256, 0, h->stream>>>(st, shift, sc.hist.p);
    }
    if (want_next) k_next_greater_keys<<<kb, 256, 0, h->stream>>>(sc.cand.p, cnt, st, nxt);
    k_bandwidth_next<<<1, 1, 0, h->stream>>>(st, nxt, want_next, St, h2_dev);
    count_launch(h, 19);
    return;
  }
  for (int shift = 56; shift >= 0; shift -= 8) {
    k_select_hist<<<blocks, 256, 0, h->stream>>>(d2, n, reinterpret_cast<SelectState*>(sc.sel.p), shift, sc.hist.p);
    if (sc.world > 1 && reduce) nccl_all_reduce_u64(sc.nccl_comm, sc.hist.p, 256, h->stream);
    k_select_pick<<<1, 256, 0, h->stream>>>(reinterpret_cast<SelectState*>(sc.sel.p), shift, sc.hist.p);
    count_launch(h, 2);
  }
  if (want_next) {
    k_next_greater<<<blocks, 256, 0, h->stream>>>(d2, n, reinterpret_cast<SelectState*>(sc.sel.p), sc.sel.p + 6);
    if (sc.world > 1 && reduce) nccl_all_reduce_min_u64(sc.nccl_comm, sc.sel.p + 6, 1, h->stream);
    count_launch(h);
  }
  k_bandwidth_next<<<1, 1, 0, h->stream>>>(reinterpret_cast<SelectState*>(sc.sel.p), sc.sel.p + 6, want_next, St, h2_dev);
  count_launch(h);
}

// phi for local rows [r0, r0+Sl) of the global particle matrix X_all [St,P] with gradients G_all
// wait_g: event after which G_all is complete (sharded runs gather it on the comm stream while the Gram is built)
__global__ void k_adam_all(float* theta, const float* phi, float* am, float* av, int64_t n, float sign, float lr_t);
struct AdamFuse { float* theta_local; float* am; float* av; float lr_t; };   // non-null: finish phi AND apply the update
// large particle sets: Gram matrix and the K*Y contraction run on the tensor cores (bf16x3 split);
// small ones keep the direct float64 kernels (bit-for-bit the formulation scipy's pdist uses)
static bool svgd_tensor_ok(const pyb_handle* h, int St) {
  return St >= 256 && h->model.P >= 64 && (St % 8) == 0 && (h->opt_path == PYB_PATH_AUTO || h->opt_path == PYB_PATH_TENSOR);
}
// raw_loss_grad: G_all is the scaled LOSS gradient and the prior term is folded into the Stein right-hand side
// (tensor path only); otherwise G_all already is the log-posterior gradient
static void phi_canonical(pyb_handle* h, const float* X_all, const float* G_all, int r0, int Sl, int St,
                          float* phi_local, double* h_host_out, cudaEvent_t wait_g = nullptr,
                          const AdamFuse* adam = nullptr, bool raw_loss_grad = false) {
  SvgdState& sv = h->svgd;
  SvgdState& sc = h->svgd;
  const int64_t P = h->model.P;
  PYB_REQUIRE(Sl == St || sv.world > 1, PYB_ERR_STATE, "row-sharded phi needs pyb_svgd_set_comm");
  sv.d2.alloc((size_t)Sl * St);
  sv.rowsum.alloc(Sl);
  sc.h2.alloc(2);
  NvtxRange nv("pyb.svgd.phi(gram,median,KY)");
  const bool tensor = svgd_tensor_ok(h, St);
  PYB_REQUIRE(tensor || !raw_loss_grad, PYB_ERR_STATE, "the prior term is only folded on the tensor path");
  const int64_t Ppad = (P + 7) / 8 * 8;
  if (tensor) {
    sv.xh.alloc((size_t)St * Ppad); sv.xl.alloc((size_t)St * Ppad);
    sv.gram.alloc((size_t)Sl * St); sv.norms.alloc(0); sc.Krow.alloc(St); sv.center.alloc(P);
    // every rank holds the same X_all, so every rank computes the same centre
    k_col_mean<<<(unsigned)((P + 31) / 32), dim3(32, 8), 0, h->stream>>>(X_all, St, P, sv.center.p);
    tc_split_rows(h, X_all, St, (int)P, P, sv.xh.p, sv.xl.p, Ppad, sv.center.p);
    tc_gemm_split(h, sv.xh.p, sv.xl.p, Ppad, St, r0, Sl, sv.xh.p, sv.xl.p, Ppad, St, P, sv.gram.p, St);
    k_row_norms<<<St, 256, 0, h->stream>>>(X_all, P, sv.center.p, sc.Krow.p);
    k_d2_from_gram<<<(unsigned)(((int64_t)Sl * St + 255) / 256), 256, 0, h->stream>>>(sv.gram.p, sc.Krow.p, r0, Sl, St, sv.d2.p);
    count_launch(h, 3);
    h->svgd_stein_used = STEIN_TENSOR;
  } else {
    dim3 g1((St + 15) / 16, (Sl + 15) / 16);
    k_gram_d2<<<g1, 256, 0, h->stream>>>(X_all, P, r0, Sl, St, sv.d2.p);
    count_launch(h);
    h->svgd_stein_used = STEIN_F64;
  }
  median_bandwidth(h, sv.d2.p, (int64_t)Sl * St, (int64_t)St * St, St, sc.h2.p);
  k_kernel_rowsum<<<Sl, 256, 0, h->stream>>>(sv.d2.p, St, sc.h2.p, sv.rowsum.p);
  count_launch(h);
  if (wait_g) PYB_CUDA(cudaStreamWaitEvent(h->stream, wait_g, 0));
  if (tensor) {
    // phi = (K Y + X rowsum/h2)/St with Y = G - X/h2: A = K [Sl, St] (K-major), B = Y^T [P, St]
    const int blocks = (int)std::min<int64_t>(((int64_t)St * P + 255) / 256, 16 * (int64_t)h->sm_count);
    sv.kf.alloc((size_t)Sl * St); sv.kh.alloc((size_t)Sl * St); sv.kl.alloc((size_t)Sl * St);
    sv.yth.alloc((size_t)P * St); sv.ytl.alloc((size_t)P * St);
    k_double_to_float<<<blocks, 256, 0, h->stream>>>(sv.d2.p, sv.kf.p, (int64_t)Sl * St);
    tc_split_rows(h, sv.kf.p, Sl, St, St, sv.kh.p, sv.kl.p, St);
    dim3 gt((unsigned)((P + 31) / 32), (unsigned)((St + 63) / 64)), bt(32, 8);
    k_stein_rhs_split_t<<<gt, bt, 0, h->stream>>>(X_all, G_all, sc.h2.p, St, P, sv.yth.p, sv.ytl.p, St,
                                                 raw_loss_grad ? h->mu.p : nullptr, raw_loss_grad ? h->inv_var.p : nullptr,
                                                 sv.center.p);
    tc_gemm_split(h, sv.kh.p, sv.kl.p, St, Sl, 0, Sl, sv.yth.p, sv.ytl.p, St, (int)P, St, phi_local, P);
    dim3 gf((unsigned)std::min<int64_t>((P + 255) / 256, 1024), (unsigned)Sl);
    if (adam)
      k_phi_finish_adam<<<(unsigned)(((int64_t)Sl * P + 1023) / 1024), 256, 0, h->stream>>>(
          phi_local, adam->theta_local, adam->am, adam->av, P, (int64_t)Sl * P, St, sc.h2.p, sv.rowsum.p, sv.center.p,
          adam->lr_t);
    else
      k_phi_finish<<<gf, 256, 0, h->stream>>>(phi_local, X_all, P, r0, St, sc.h2.p, sv.rowsum.p, sv.center.p);
    count_launch(h, 3);
  } else {
    dim3 g2((unsigned)((P + 255) / 256), (Sl + 7) / 8);
    k_phi_canonical<<<g2, 256, 0, h->stream>>>(sv.d2.p, X_all, G_all, P, r0, Sl, St, sc.h2.p, sv.rowsum.p, phi_local);
    count_launch(h);
    if (adam) {
      int blocks = (int)std::min<int64_t>(((int64_t)Sl * P + 255) / 256, 8 * (int64_t)h->sm_count);
      k_adam_all<<<blocks, 256, 0, h->stream>>>(adam->theta_local, phi_local, adam->am, adam->av, (int64_t)Sl * P, -1.0f,
                                                adam->lr_t);
      count_launch(h);
    }
  }
  if (h_host_out) {
    double v[2];
    PYB_CUDA(cudaMemcpyAsync(v, sc.h2.p, sizeof(v), cudaMemcpyDeviceToHost, h->stream));
    PYB_CUDA(cudaStreamSynchronize(h->stream));
    *h_host_out = sqrt(v[0]);
  }
}

void svgd_init(pyb_handle* h, int64_t S, int64_t offset, double lr, int sem, const double* p0) {
  PYB_REQUIRE(h->have_data && h->have_prior, PYB_ERR_STATE, "dataset and prior must be set first");
  PYB_REQUIRE(S > 0 && S <= 65535, PYB_ERR_INVALID, "S must be in [1, 65535]");
  PYB_REQUIRE(sem == PYB_SVGD_REFERENCE_LIVE || sem == PYB_SVGD_CANONICAL_MEDIAN, PYB_ERR_INVALID, "bad semantics");
  SvgdState& sv = h->svgd;
  const int64_t P = h->model.P;
  sv.S = S; sv.offset = offset; sv.lr = lr; sv.semantics = sem; sv.t = 0;
  sv.ps_ready = false; sv.ps_checked = false;
  sv.theta.alloc(S * P); sv.g.alloc(S * P); sv.adam_m.alloc(S * P); sv.adam_v.alloc(S * P); sv.phi.alloc(S * P);
  sv.loss.alloc(S);
  PYB_CUDA(cudaMemsetAsync(sv.adam_m.p, 0, S * P * sizeof(float), h->stream));
  PYB_CUDA(cudaMemsetAsync(sv.adam_v.p, 0, S * P * sizeof(float), h->stream));
  DevBuf<double> tmp;
  if (p0) {
    tmp.alloc(S * P);
    PYB_CUDA(cudaMemcpyAsync(tmp.p, p0, S * P * sizeof(double), cudaMemcpyHostToDevice, h->stream));
  }
  dim3 grid((unsigned)((P + 1023) / 1024), (unsigned)S);
  k_svgd_init<<<grid, 256, 0, h->stream>>>(sv.theta.p, p0 ? tmp.p : nullptr, h->mu.p, h->sigma.p, P, h->seed, offset);
  count_launch(h);
  PYB_CUDA(cudaStreamSynchronize(h->stream));
  PYB_CUDA(cudaGetLastError());
  sv.inited = true;
}

// ------------------------------------------------------------------------------------------
// Parameter-sharded Stein phase (canonical mode on the tensor path, world > 1).
// The row-sharded exchange above gathers every rank's particles AND gradients (2 x St x P floats received per rank and
// step: 2.9 GB at C4 on 8 GPUs, against ~4 ms of compute: 3.3x at 8 GPUs) and every rank splits all St x P elements
// for its GEMM operands.  Here the Stein phase is sharded over the PARAMETERS instead (the Gram matrix and K Y are
// sums / independent column blocks over them):
//   rank r owns columns [r Pw, (r+1) Pw) of all St particles: theta slice xs, Adam moments, phi  (never move)
//   1. local minibatch gradients of the rank's S particles                      [S, P]
//   2. all-to-all of the gradient rows: [S, P] -> gradient slice of all particles [St, Pw]     (S P / R floats per peer)
//   3. partial Gram over the slice on tcgen05, all-reduce of the St x St matrix and of the squared norms
//   4. d2, exact median (all-reduced radix histograms over the rank's rows), K = exp(-d2 / 2h2) — St x St on every rank
//   5. K Y and the Adam ascent step on the slice
//   6. all-to-all back: the updated slice rows of each rank's own particles -> [S, P] for the next gradient evaluation
// Per rank and step: 2 S P (R-1)/R floats sent + the 4 St^2-byte all-reduce: 0.36 GB + 67 MB at C4 on 8 GPUs.
// ------------------------------------------------------------------------------------------
// src [Sl, P] -> dst [R][Sl][Pw]: block q holds columns [q Pw, (q+1) Pw) (zero beyond P)
// grid (ceil(Pw / 256), Sl, R)
__global__ void k_pack_cols(const float* __restrict__ src, int64_t Sl, int64_t P, int64_t Pw, int R, float* __restrict__ dst) {
  const int64_t c = (int64_t)blockIdx.x * blockDim.x + threadIdx.x, i = blockIdx.y, q = blockIdx.z;
  if (c >= Pw) return;
  const int64_t col = q * Pw + c;
  dst[(q * Sl + i) * Pw + c] = col < P ? src[i * P + col] : 0.f;
}
// src [R][Sl][Pw] -> dst [Sl, P]: blocks q0 + blockIdx.z
__global__ void k_unpack_cols(const float* __restrict__ src, int64_t Sl, int64_t P, int64_t Pw, int q0, float* __restrict__ dst) {
  const int64_t c = (int64_t)blockIdx.x * blockDim.x + threadIdx.x, i = blockIdx.y, q = q0 + blockIdx.z;
  const int64_t col = q * Pw + c;
  if (c >= Pw || col >= P) return;
  dst[i * P + col] = src[(q * Sl + i) * Pw + c];
}
__global__ void k_slice_vec(const float* __restrict__ v, int64_t P, int64_t c0, int64_t Pw, float* __restrict__ out) {
  const int64_t c = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (c < Pw) out[c] = (c0 + c < P) ? v[c0 + c] : 0.f;
}

// ---- peer memory: the exchanges of the parameter-sharded step as stores of our own kernels over NVLink ----------------
// rows of `rows` local particles -> the gradient slice of EVERY rank: peers[q][(row0 + i) * Pw + c] = src[i][q * Pw + c]
// (four columns per thread: the source rows have an arbitrary pitch, the slices a pitch of 8 floats — one 16-byte store
// per thread, 512 contiguous bytes per warp on the wire)
__global__ void k_scatter_cols_p2p(const float* __restrict__ src, int64_t P, int64_t Pw, int64_t row0, float* const* __restrict__ peers) {
  const int64_t c = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) * 4, i = blockIdx.y, q = blockIdx.z;
  if (c >= Pw) return;
  const int64_t col = q * Pw + c;
  const float* s = src + i * P + col;
  float4 v;
  v.x = col < P ? s[0] : 0.f;
  v.y = col + 1 < P ? s[1] : 0.f;
  v.z = col + 2 < P ? s[2] : 0.f;
  v.w = col + 3 < P ? s[3] : 0.f;
  *reinterpret_cast<float4*>(peers[q] + (row0 + i) * Pw + c) = v;
}
// one block of the particle slice (the rows of one rank's particles, this rank's parameter columns) -> those particles'
// rows on their owner: dst[i][col0 + c] = block[i][c]
// (V = 2: two columns per thread as one 8-byte store — needs an even P, so that every row of the owner starts 8-byte aligned)
template <int V>
__global__ void k_scatter_block_p2p(const float* __restrict__ block, int64_t P, int64_t Pw, int64_t col0, float* __restrict__ dst) {
  const int64_t c = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) * V, i = blockIdx.y;
  const int64_t col = col0 + c;
  if (c >= Pw || col >= P) return;
  if (V == 2) {
    if (col + 1 < P) {
      *reinterpret_cast<float2*>(dst + i * P + col) = *reinterpret_cast<const float2*>(block + i * Pw + c);
      return;
    }
  }
  dst[i * P + col] = block[i * Pw + c];
}

struct P2pCard {
  long long pid, host;
  int dev, pad;
  unsigned long long theta, g;
  cudaIpcMemHandle_t h_theta, h_g;
};
static_assert(sizeof(P2pCard) % sizeof(float) == 0, "card travels as floats");

void svgd_p2p_release(pyb_handle* h) {
  SvgdState& sv = h->svgd;
  for (void* m : sv.p2p_opened) cudaIpcCloseMemHandle(m);
  sv.p2p_opened.clear();
  sv.p2p_ready = false;
  sv.p2p_tried = false;
}

// collective over the communicator: every rank publishes where its particle rows and its gradient slice live; peers in
// other processes map them through CUDA IPC, peers in this process (one engine per device, multi.py) through plain peer
// access.  All ranks agree on the outcome (all-reduced flag); on any failure the NCCL send / recv exchange stays.
static void svgd_p2p_setup(pyb_handle* h) {
  SvgdState& sv = h->svgd;
  const int R = sv.world;
  svgd_p2p_release(h);
  sv.p2p_tried = true;
  sv.p2p_src_theta = sv.theta.p; sv.p2p_src_g = sv.ps_g.p;
  P2pCard mine = {};
  mine.pid = (long long)getpid();
  char hn[256] = {0};
  gethostname(hn, sizeof(hn) - 1);
  unsigned long long hh = 1469598103934665603ull;
  for (const char* c = hn; *c; ++c) hh = (hh ^ (unsigned char)*c) * 1099511628211ull;
  mine.host = (long long)hh;
  mine.dev = h->device;
  mine.theta = (unsigned long long)(uintptr_t)sv.theta.p; mine.g = (unsigned long long)(uintptr_t)sv.ps_g.p;
  unsigned long long ok = 1;
  if (cudaIpcGetMemHandle(&mine.h_theta, sv.theta.p) != cudaSuccess || cudaIpcGetMemHandle(&mine.h_g, sv.ps_g.p) != cudaSuccess) {
    cudaGetLastError();
    ok = 0;
  }
  const size_t nf = sizeof(P2pCard) / sizeof(float);
  DevBuf<float> send, recv;
  send.alloc(nf); recv.alloc(nf * R);
  std::vector<P2pCard> cards(R);
  PYB_CUDA(cudaMemcpyAsync(send.p, &mine, sizeof(mine), cudaMemcpyHostToDevice, h->stream));
  nccl_all_gather_f32(sv.nccl_comm, send.p, recv.p, nf, h->stream);
  PYB_CUDA(cudaMemcpyAsync(cards.data(), recv.p, sizeof(P2pCard) * R, cudaMemcpyDeviceToHost, h->stream));
  PYB_CUDA(cudaStreamSynchronize(h->stream));
  std::vector<float*> pt(R, nullptr), pg(R, nullptr);
  for (int q = 0; q < R && ok; ++q) {
    const P2pCard& c = cards[q];
    if (q == sv.rank) { pt[q] = sv.theta.p; pg[q] = sv.ps_g.p; continue; }
    if (c.host != mine.host) { ok = 0; break; }
    if (c.pid == mine.pid) {
      int can = 0;
      if (cudaDeviceCanAccessPeer(&can, h->device, c.dev) != cudaSuccess || !can) { cudaGetLastError(); ok = 0; break; }
      const cudaError_t e = cudaDeviceEnablePeerAccess(c.dev, 0);
      if (e != cudaSuccess && e != cudaErrorPeerAccessAlreadyEnabled) { cudaGetLastError(); ok = 0; break; }
      cudaGetLastError();
      pt[q] = (float*)(uintptr_t)c.theta; pg[q] = (float*)(uintptr_t)c.g;
    } else {
      void *mt = nullptr, *mg = nullptr;
      if (cudaIpcOpenMemHandle(&mt, c.h_theta, cudaIpcMemLazyEnablePeerAccess) != cudaSuccess) { cudaGetLastError(); ok = 0; break; }
      sv.p2p_opened.push_back(mt);
      if (cudaIpcOpenMemHandle(&mg, c.h_g, cudaIpcMemLazyEnablePeerAccess) != cudaSuccess) { cudaGetLastError(); ok = 0; break; }
      sv.p2p_opened.push_back(mg);
      pt[q] = (float*)mt; pg[q] = (float*)mg;
    }
  }
  sv.sel.alloc(8);
  PYB_CUDA(cudaMemcpyAsync(sv.sel.p, &ok, sizeof(ok), cudaMemcpyHostToDevice, h->stream));
  nccl_all_reduce_min_u64(sv.nccl_comm, sv.sel.p, 1, h->stream);
  PYB_CUDA(cudaMemcpyAsync(&ok, sv.sel.p, sizeof(ok), cudaMemcpyDeviceToHost, h->stream));
  PYB_CUDA(cudaStreamSynchronize(h->stream));
  nccl_check_async(&sv.nccl_comm);
  if (!ok) {
    for (void* m : sv.p2p_opened) cudaIpcCloseMemHandle(m);
    sv.p2p_opened.clear();
    return;
  }
  sv.p2p_theta.alloc(R); sv.p2p_g.alloc(R); sv.p2p_token.alloc(1);
  sv.p2p_theta_host = pt;
  PYB_CUDA(cudaMemcpyAsync(sv.p2p_theta.p, pt.data(), sizeof(float*) * R, cudaMemcpyHostToDevice, h->stream));
  PYB_CUDA(cudaMemcpyAsync(sv.p2p_g.p, pg.data(), sizeof(float*) * R, cudaMemcpyHostToDevice, h->stream));
  PYB_CUDA(cudaMemsetAsync(sv.p2p_token.p, 0, sizeof(float), h->stream));
  PYB_CUDA(cudaStreamSynchronize(h->stream));
  sv.p2p_ready = true;
}

static void svgd_step_pshard(pyb_handle* h, const float* Xb, const int32_t* yb_i, const float* yb_f, int64_t Nb, float lr_t,
                             float scale) {
  SvgdState& sv = h->svgd;
  const int64_t P = h->model.P, S = sv.S;
  const int R = sv.world, St = (int)(S * R), r0 = (int)(S * sv.rank);
  const int64_t Pw = ((P + R - 1) / R + 7) / 8 * 8;
  const int64_t c0 = (int64_t)sv.rank * Pw;
  const int eb = (int)std::min<int64_t>(((int64_t)St * Pw + 255) / 256, 16 * (int64_t)h->sm_count);
  if (!sv.ps_checked) {
    // every rank must hold the same number of particles (St = S * world, block q of an exchange = rank q's rows)
    sv.sel.alloc(8);
    unsigned long long v[2] = {(unsigned long long)S, (unsigned long long)(S * S)};
    PYB_CUDA(cudaMemcpyAsync(sv.sel.p, v, sizeof(v), cudaMemcpyHostToDevice, h->stream));
    nccl_all_reduce_u64(sv.nccl_comm, sv.sel.p, 2, h->stream);
    PYB_CUDA(cudaMemcpyAsync(v, sv.sel.p, sizeof(v), cudaMemcpyDeviceToHost, h->stream));
    PYB_CUDA(cudaStreamSynchronize(h->stream));
    nccl_check_async(&sv.nccl_comm);
    PYB_REQUIRE(v[0] == (unsigned long long)(S * R) && v[1] == (unsigned long long)(S * S * R), PYB_ERR_INVALID,
                "sharded SVGD needs the same number of particles on every rank");
    sv.ps_checked = true;
  }
  if (!sv.comm_stream) {
    int prio_lo = 0, prio_hi = 0;
    PYB_CUDA(cudaDeviceGetStreamPriorityRange(&prio_lo, &prio_hi));
    PYB_CUDA(cudaStreamCreateWithPriority(&sv.comm_stream, cudaStreamNonBlocking, prio_hi));
    PYB_CUDA(cudaEventCreateWithFlags(&sv.ev_fork, cudaEventDisableTiming));
    PYB_CUDA(cudaEventCreateWithFlags(&sv.ev_theta, cudaEventDisableTiming));
    PYB_CUDA(cudaEventCreateWithFlags(&sv.ev_grad, cudaEventDisableTiming));
  }
  if (!sv.nccl_comm2) sv.nccl_comm2 = nccl_comm_dup(sv.nccl_comm, sv.rank);
  if (!sv.ps_ready || sv.ps_Pw != Pw) {
    sv.ps_Pw = Pw;
    sv.ps_pack.alloc((size_t)St * Pw); sv.ps_x.alloc((size_t)St * Pw); sv.ps_g.alloc((size_t)St * Pw);
    sv.ps_m.alloc((size_t)St * Pw); sv.ps_v.alloc((size_t)St * Pw); sv.ps_phi.alloc((size_t)St * Pw);
    sv.ps_mu.alloc(Pw); sv.ps_iv.alloc(Pw); sv.ps_norms.alloc(St);
    PYB_CUDA(cudaMemsetAsync(sv.ps_m.p, 0, (size_t)St * Pw * sizeof(float), h->stream));
    PYB_CUDA(cudaMemsetAsync(sv.ps_v.p, 0, (size_t)St * Pw * sizeof(float), h->stream));
    PYB_CUDA(cudaMemsetAsync(sv.ps_g.p, 0, (size_t)St * Pw * sizeof(float), h->stream));
    k_slice_vec<<<(unsigned)((Pw + 255) / 256), 256, 0, h->stream>>>(h->mu.p, P, c0, Pw, sv.ps_mu.p);
    k_slice_vec<<<(unsigned)((Pw + 255) / 256), 256, 0, h->stream>>>(h->inv_var.p, P, c0, Pw, sv.ps_iv.p);
    // the particle slice: one exchange at the start, afterwards the slice IS the master copy the update is applied to
    k_pack_cols<<<dim3((unsigned)((Pw + 255) / 256), (unsigned)S, (unsigned)R), 256, 0, h->stream>>>(sv.theta.p, S, P, Pw, R, sv.ps_pack.p);
    nccl_all_to_all_f32(sv.nccl_comm, sv.ps_pack.p, sv.ps_x.p, (size_t)S * Pw, R, h->stream);
    count_launch(h, 3);
    sv.ps_ready = true;
  }
  if (!sv.gram_stream) {
    // the side chain is a string of small dependent kernels beside persistent ones that fill the GPU: at every kernel
    // boundary of the main stream the side kernel must win the SMs, or it waits for the next boundary
    int prio_lo = 0, prio_hi = 0;
    PYB_CUDA(cudaDeviceGetStreamPriorityRange(&prio_lo, &prio_hi));
    PYB_CUDA(cudaStreamCreateWithPriority(&sv.gram_stream, cudaStreamNonBlocking, prio_hi));
    cudaEvent_t* evs[] = {&sv.ev_kernel, &sv.ev_gh[0], &sv.ev_gh[1], &sv.ev_p1, &sv.ev_p2, &sv.ev_back};
    for (cudaEvent_t* e : evs) PYB_CUDA(cudaEventCreateWithFlags(e, cudaEventDisableTiming));
  }
  if (!sv.nccl_comm3) sv.nccl_comm3 = nccl_comm_dup(sv.nccl_comm, sv.rank);
  if (h->opt_svgd_p2p && (!sv.p2p_tried || sv.p2p_src_theta != sv.theta.p || sv.p2p_src_g != sv.ps_g.p)) svgd_p2p_setup(h);
  const bool p2p = h->opt_svgd_p2p && sv.p2p_ready;
  const bool timed = h->prof_enabled;
  auto mark = [&](int k) {
    if (!timed) return;
    if (!sv.ps_ev[k]) PYB_CUDA(cudaEventCreate(&sv.ps_ev[k]));
    PYB_CUDA(cudaEventRecord(sv.ps_ev[k], h->stream));
  };
  sv.ps_timed = timed;
  cudaStream_t main_stream = h->stream;
  mark(0);
  // ---- 1. partial Gram matrix and squared norms over the slice: they need the particle slice only, which is the master
  //         copy since the last step, so they go first and their reduction hides behind the gradients
  nvtxRangePushA("pyb.svgd.gram_partial");
  sv.xh.alloc((size_t)St * Pw); sv.xl.alloc((size_t)St * Pw);
  sv.gram.alloc((size_t)St * St); sv.d2.alloc((size_t)St * St); sv.rowsum.alloc(St); sv.h2.alloc(2);
  sv.kf.alloc((size_t)St * St); sv.kh.alloc((size_t)St * St); sv.kl.alloc((size_t)St * St);
  sv.yth.alloc((size_t)Pw * St); sv.ytl.alloc((size_t)Pw * St); sv.center.alloc(Pw);
  // the rank's own column slice is centred on its own column means: the Gram matrix is a sum over column slices of
  // translation-invariant parts, so no collective is needed
  k_col_mean<<<(unsigned)((Pw + 31) / 32), dim3(32, 8), 0, h->stream>>>(sv.ps_x.p, St, Pw, sv.center.p);
  tc_split_rows(h, sv.ps_x.p, St, (int)Pw, Pw, sv.xh.p, sv.xl.p, Pw, sv.center.p);
  tc_gemm_split(h, sv.xh.p, sv.xl.p, Pw, St, 0, St, sv.xh.p, sv.xl.p, Pw, St, Pw, sv.gram.p, St);
  k_row_norms<<<St, 256, 0, h->stream>>>(sv.ps_x.p, Pw, sv.center.p, sv.ps_norms.p);
  count_launch(h, 2);
  nvtxRangePop();
  mark(1);
  // ---- 2. side stream, third communicator: all-reduce of the Gram matrix, distances, median bandwidth, kernel matrix and
  //         its bf16 hi / lo split (identical on every rank: the all-reduced inputs are) — while the gradients run
  // (option svgd_gram_sync: the 67 MB all-reduce stays on the main stream — a long collective kernel beside persistent
  // kernels with a static tile schedule holds SMs those kernels' last CTAs then wait for)
  if (h->opt_svgd_gram_sync) {
    nccl_all_reduce_f32(sv.nccl_comm3, sv.gram.p, (size_t)St * St, main_stream);
    nccl_all_reduce_f64(sv.nccl_comm3, sv.ps_norms.p, St, main_stream);
  }
  PYB_CUDA(cudaEventRecord(sv.ev_fork, main_stream));
  PYB_CUDA(cudaStreamWaitEvent(sv.gram_stream, sv.ev_fork, 0));
  {
    nvtxRangePushA("pyb.svgd.gram_all_reduce+median_kernel(side stream)");
    void* comm_main = sv.nccl_comm;
    h->stream = sv.gram_stream; sv.nccl_comm = sv.nccl_comm3;       // the helpers below launch on h->stream / sv.nccl_comm
    try {
      if (!h->opt_svgd_gram_sync) {
        nccl_all_reduce_f32(sv.nccl_comm, sv.gram.p, (size_t)St * St, h->stream);
        nccl_all_reduce_f64(sv.nccl_comm, sv.ps_norms.p, St, h->stream);
      }
      // every rank holds the whole (bit-identical) distance matrix: the select runs over all of it without a collective,
      // and the chain is kept to FEW kernels (each one waits for a kernel boundary of the main stream): distances + first
      // histogram, seven passes that pick the previous digit themselves, last pick + next-greater, bandwidth, and one
      // pass for the kernel matrix's row sums and bf16 split — 12 launches where the plain sequence has 25
      const int64_t nn = (int64_t)St * St;
      if (nn <= (64ll << 20) && h->opt_svgd_chain_fused) {
        median_prepare_fused(h, nn);
        k_d2_from_gram<<<(unsigned)((nn + 255) / 256), 256, 0, h->stream>>>(sv.gram.p, sv.ps_norms.p, 0, St, St, sv.d2.p, sv.hist.p);
        median_bandwidth_fused(h, sv.d2.p, nn, St, sv.h2.p, true);
      } else {
        k_d2_from_gram<<<(unsigned)((nn + 255) / 256), 256, 0, h->stream>>>(sv.gram.p, sv.ps_norms.p, 0, St, St, sv.d2.p);
        if (nn <= (64ll << 20))
          median_bandwidth(h, sv.d2.p, nn, nn, St, sv.h2.p, false);
        else
          median_bandwidth(h, sv.d2.p + (int64_t)r0 * St, (int64_t)S * St, nn, St, sv.h2.p);
      }
      k_kernel_rowsum_split<<<St, 256, 0, h->stream>>>(sv.d2.p, St, sv.h2.p, sv.rowsum.p, (__nv_bfloat16*)sv.kh.p,
                                                       (__nv_bfloat16*)sv.kl.p);
      count_launch(h, 3);
    } catch (...) {
      h->stream = main_stream; sv.nccl_comm = comm_main;
      throw;
    }
    h->stream = main_stream; sv.nccl_comm = comm_main;
    PYB_CUDA(cudaEventRecord(sv.ev_kernel, sv.gram_stream));
    nvtxRangePop();
  }
  // ---- 3. local gradients in (up to) two halves of the particles: a half's rows travel to the parameter slices of
  //         every rank (all-to-all on the exchange stream, second communicator) while the next half is computed
  nvtxRangePushA("pyb.svgd.gradients(+all-to-all)");
  const int nh = (h->opt_svgd_halves && S >= 256 && S % 2 == 0) ? 2 : 1;
  const int64_t Sh = S / nh;
  for (int hf = 0; hf < nh; ++hf) {
    eval_on_batch(h, sv.theta.p + hf * Sh * P, Sh, Xb, yb_i, yb_f, Nb, scale, sv.loss.p + hf * Sh, sv.g.p + hf * Sh * P);
    PYB_CUDA(cudaEventRecord(sv.ev_gh[hf], main_stream));
    PYB_CUDA(cudaStreamWaitEvent(sv.comm_stream, sv.ev_gh[hf], 0));
    if (p2p) {
      // one kernel: every gradient row goes straight into the gradient slice of the rank that owns its columns
      k_scatter_cols_p2p<<<dim3((unsigned)((Pw / 4 + 255) / 256), (unsigned)Sh, (unsigned)R), 256, 0, sv.comm_stream>>>(
          sv.g.p + hf * Sh * P, P, Pw, (int64_t)r0 + hf * Sh, sv.p2p_g.p);
    } else {
      float* pk = sv.ps_pack.p + (int64_t)hf * R * Sh * Pw;
      k_pack_cols<<<dim3((unsigned)((Pw + 255) / 256), (unsigned)Sh, (unsigned)R), 256, 0, sv.comm_stream>>>(
          sv.g.p + hf * Sh * P, Sh, P, Pw, R, pk);
      nccl_all_to_all_f32_strided(sv.nccl_comm2, pk, (size_t)Sh * Pw, sv.ps_g.p + hf * Sh * Pw, (size_t)S * Pw, (size_t)Sh * Pw, R,
                                  sv.comm_stream);
    }
    count_launch(h);
  }
  // peer stores are complete when their kernel is; the one-float all-reduce is the barrier that tells every rank so
  if (p2p) nccl_all_reduce_f32(sv.nccl_comm2, sv.p2p_token.p, 1, sv.comm_stream);
  PYB_CUDA(cudaEventRecord(sv.ev_grad, sv.comm_stream));
  nvtxRangePop();
  mark(2);
  PYB_CUDA(cudaStreamWaitEvent(main_stream, sv.ev_kernel, 0));     // kernel matrix, bandwidth, row sums
  mark(3);
  PYB_CUDA(cudaStreamWaitEvent(main_stream, sv.ev_grad, 0));       // the gradient slice of all particles is complete
  mark(4);
  // ---- 4. K Y and the Adam ascent step on the slice, in two groups of particle blocks (block q = rank q's particles):
  //         rank r takes the blocks in the order r+1, r+2, ..., r-1, r, so that the finished blocks of the first group
  //         are on the wire (balanced: everybody sends to its next ranks and receives from its previous ones) while the
  //         second group is multiplied
  nvtxRangePushA("pyb.svgd.stein_update(KY+Adam, blocks leave as they finish)");
  dim3 gt((unsigned)((Pw + 31) / 32), (unsigned)((St + 63) / 64)), bt(32, 8);
  k_stein_rhs_split_t<<<gt, bt, 0, h->stream>>>(sv.ps_x.p, sv.ps_g.p, sv.h2.p, St, Pw, sv.yth.p, sv.ytl.p, St, sv.ps_mu.p,
                                               sv.ps_iv.p, sv.center.p);
  count_launch(h);
  // remote blocks in the first group: what is left for the second (at most two remote blocks and the own one) is all
  // that can stay exposed after the last multiplication
  const int n1 = std::max(R / 2, R - 3);
  int send1[64], recv1[64], send2[64], recv2[64];
  PYB_REQUIRE(R <= 64, PYB_ERR_INVALID, "at most 64 ranks");
  for (int j = 1; j <= n1; ++j) { send1[j - 1] = (sv.rank + j) % R; recv1[j - 1] = (sv.rank - j + R) % R; }
  for (int j = n1 + 1; j < R; ++j) { send2[j - n1 - 1] = (sv.rank + j) % R; recv2[j - n1 - 1] = (sv.rank - j + R) % R; }
  auto update_blocks = [&](int j_lo, int j_hi) {                   // blocks (rank + j) % R for j in [j_lo, j_hi): <= 2 runs of rows
    int j = j_lo;
    while (j < j_hi) {
      const int q0 = (sv.rank + j) % R;
      int len = 1;
      while (j + len < j_hi && q0 + len < R) ++len;                // a run ends where the block index wraps to 0
      const int64_t m0 = (int64_t)q0 * S, mrows = (int64_t)len * S;
      tc_gemm_split(h, sv.kh.p, sv.kl.p, St, St, (int)m0, (int)mrows, sv.yth.p, sv.ytl.p, St, (int)Pw, St, sv.ps_phi.p + m0 * Pw, Pw);
      k_phi_finish_adam<<<(unsigned)((mrows * Pw + 1023) / 1024), 256, 0, h->stream>>>(
          sv.ps_phi.p + m0 * Pw, sv.ps_x.p + m0 * Pw, sv.ps_m.p + m0 * Pw, sv.ps_v.p + m0 * Pw, Pw, mrows * Pw, St, sv.h2.p,
          sv.rowsum.p + m0, sv.center.p, lr_t);
      count_launch(h);
      j += len;
    }
  };
  update_blocks(1, 1 + n1);
  PYB_CUDA(cudaEventRecord(sv.ev_p1, main_stream));
  PYB_CUDA(cudaStreamWaitEvent(sv.comm_stream, sv.ev_p1, 0));
  auto unpack = [&](const float* src, int q, cudaStream_t st) {   // parameter slice q of this rank's rows -> theta
    k_unpack_cols<<<dim3((unsigned)((Pw + 255) / 256), (unsigned)S, 1), 256, 0, st>>>(src, S, P, Pw, q, sv.theta.p);
    count_launch(h);
  };
  auto scatter_block = [&](int q, cudaStream_t st) {            // rank q's updated rows, this rank's columns -> rank q
    if (P % 2 == 0)
      k_scatter_block_p2p<2><<<dim3((unsigned)((Pw / 2 + 255) / 256), (unsigned)S, 1), 256, 0, st>>>(
          sv.ps_x.p + (int64_t)q * S * Pw, P, Pw, c0, sv.p2p_theta_host[q]);
    else
      k_scatter_block_p2p<1><<<dim3((unsigned)((Pw + 255) / 256), (unsigned)S, 1), 256, 0, st>>>(
          sv.ps_x.p + (int64_t)q * S * Pw, P, Pw, c0, sv.p2p_theta_host[q]);
    count_launch(h);
  };
  if (p2p) {
    for (int i = 0; i < n1; ++i) scatter_block(send1[i], sv.comm_stream);
  } else {
    nccl_exchange_f32(sv.nccl_comm2, sv.ps_x.p, sv.ps_pack.p, (size_t)S * Pw, (size_t)S * Pw, send1, n1, recv1, n1, sv.comm_stream);
    for (int i = 0; i < n1; ++i) unpack(sv.ps_pack.p, recv1[i], sv.comm_stream);
  }
  update_blocks(1 + n1, R + 1);                                    // ... r-1 and, last, this rank's own block
  PYB_CUDA(cudaEventRecord(sv.ev_p2, main_stream));
  PYB_CUDA(cudaStreamWaitEvent(sv.comm_stream, sv.ev_p2, 0));
  if (p2p) {
    for (int i = 0; i < R - 1 - n1; ++i) scatter_block(send2[i], sv.comm_stream);
    nccl_all_reduce_f32(sv.nccl_comm2, sv.p2p_token.p, 1, sv.comm_stream);      // barrier: every rank's stores have landed
  } else {
    nccl_exchange_f32(sv.nccl_comm2, sv.ps_x.p, sv.ps_pack.p, (size_t)S * Pw, (size_t)S * Pw, send2, R - 1 - n1, recv2, R - 1 - n1,
                      sv.comm_stream);
    for (int i = 0; i < R - 1 - n1; ++i) unpack(sv.ps_pack.p, recv2[i], sv.comm_stream);
  }
  PYB_CUDA(cudaEventRecord(sv.ev_back, sv.comm_stream));
  nvtxRangePop();
  mark(5);
  // ---- 5. this rank's own rows: its own slice straight from the master copy; the other slices were unpacked on the
  //         exchange stream as they arrived
  NvtxRange nv_back("pyb.svgd.exchange.particles(own slice + wait)");
  unpack(sv.ps_x.p, sv.rank, main_stream);
  mark(6);
  PYB_CUDA(cudaStreamWaitEvent(main_stream, sv.ev_back, 0));
  mark(7);
}

void svgd_step(pyb_handle* h, const int32_t* idx, int64_t B, double* loss_out) {
  NvtxRange nv("pyb.svgd_step");
  SvgdState& sv = h->svgd;
  PYB_REQUIRE(sv.inited, PYB_ERR_STATE, "pyb_svgd_init must be called first");
  SvgdState& sc = h->svgd;
  const Model& m = h->model;
  const int64_t P = m.P, S = sv.S;
  const float* Xb = h->X.p;
  const int32_t* yb_i = h->y_i.p;
  const float* yb_f = h->y_f.p;
  int64_t Nb = h->N;
  PYB_CUDA(cudaEventRecord(h->ev0, h->stream));
  if (idx) {
    PYB_REQUIRE(B > 0, PYB_ERR_INVALID, "B must be > 0 with batch_idx");
    sv.idx.alloc(B);
    sv.Xb.alloc(B * m.in_dim);
    if (h->loss_kind == PYB_LOSS_SPARSE_CE) sv.yb_i.alloc(B); else sv.yb_f.alloc(B * m.out_dim);
    PYB_CUDA(cudaMemcpyAsync(sv.idx.p, idx, B * sizeof(int32_t), cudaMemcpyHostToDevice, h->stream));
    gather_batch(h, sv.idx.p, B, sv.Xb.p, sv.yb_i.p, sv.yb_f.p);
    Xb = sv.Xb.p; yb_i = sv.yb_i.p; yb_f = sv.yb_f.p; Nb = B;
  }
  sv.t += 1;
  const float lr_t = (float)adam_lr_t(sv.lr, sv.t);
  const float scale = (sv.semantics == PYB_SVGD_REFERENCE_LIVE) ? 1.0f : (float)h->n_train;
  const int R = sv.world, St = (int)(S * R), r0 = (int)(S * sv.rank);
  // particles / gradients of every rank (the one exchange step of the path, SURVEY 8e).  Jacobi (canonical) mode:
  // the particle all-gather is issued before the local gradients are computed and the gradient all-gather before
  // the Gram matrix is built, both on the comm stream, so each transfer hides behind the compute that does not
  // need it; the sequential live sweep exchanges inside its own loop.
  const float* theta_all = sv.theta.p;
  const float* g_all = sv.g.p;
  const bool pshard = R > 1 && sv.semantics != PYB_SVGD_REFERENCE_LIVE && svgd_tensor_ok(h, St) && h->opt_svgd_pshard;
  const bool overlap = R > 1 && sv.semantics != PYB_SVGD_REFERENCE_LIVE && !pshard;
  if (R > 1 && !pshard) {
    sv.theta_all.alloc((size_t)St * P);
    sv.g_all.alloc((size_t)St * P);
    theta_all = sv.theta_all.p;
    g_all = sv.g_all.p;
  }
  if (overlap) {
    if (!sv.comm_stream) {
      PYB_CUDA(cudaStreamCreateWithFlags(&sv.comm_stream, cudaStreamNonBlocking));
      PYB_CUDA(cudaEventCreateWithFlags(&sv.ev_fork, cudaEventDisableTiming));
      PYB_CUDA(cudaEventCreateWithFlags(&sv.ev_theta, cudaEventDisableTiming));
      PYB_CUDA(cudaEventCreateWithFlags(&sv.ev_grad, cudaEventDisableTiming));
    }
    PYB_CUDA(cudaEventRecord(sv.ev_fork, h->stream));                 // last step's update of theta is ordered before
    PYB_CUDA(cudaStreamWaitEvent(sv.comm_stream, sv.ev_fork, 0));
    nccl_all_gather_f32(sv.nccl_comm, sv.theta.p, sv.theta_all.p, (size_t)S * P, sv.comm_stream);
    PYB_CUDA(cudaEventRecord(sv.ev_theta, sv.comm_stream));
  }
  if (pshard) {
    svgd_step_pshard(h, Xb, yb_i, yb_f, Nb, lr_t, scale);
    h->svgd_stein_used = STEIN_PSHARD;
  }
  else eval_on_batch(h, sv.theta.p, S, Xb, yb_i, yb_f, Nb, scale, sv.loss.p, sv.g.p);
  const bool fold_prior = sv.semantics != PYB_SVGD_REFERENCE_LIVE && svgd_tensor_ok(h, St);
  if (sv.semantics != PYB_SVGD_REFERENCE_LIVE && !fold_prior && !pshard) {
    dim3 gg((unsigned)std::min<int64_t>((P + 255) / 256, 1024), (unsigned)S);
    k_glogp<<<gg, 256, 0, h->stream>>>(sv.g.p, sv.theta.p, h->mu.p, h->inv_var.p, P);
    count_launch(h);
  }
  if (overlap) {
    PYB_CUDA(cudaEventRecord(sv.ev_fork, h->stream));
    PYB_CUDA(cudaStreamWaitEvent(sv.comm_stream, sv.ev_fork, 0));
    nccl_all_gather_f32(sv.nccl_comm, sv.g.p, sv.g_all.p, (size_t)S * P, sv.comm_stream);
    PYB_CUDA(cudaEventRecord(sv.ev_grad, sv.comm_stream));
    PYB_CUDA(cudaStreamWaitEvent(h->stream, sv.ev_theta, 0));        // the Gram matrix needs every rank's particles
  } else if (R > 1 && !pshard) {
    nccl_all_gather_f32(sv.nccl_comm, sv.theta.p, sv.theta_all.p, (size_t)S * P, h->stream);
    nccl_all_gather_f32(sv.nccl_comm, sv.g.p, sv.g_all.p, (size_t)S * P, h->stream);
  }
  if (sv.semantics == PYB_SVGD_REFERENCE_LIVE) {
    // sequential sweep over ALL particles in global order: rank rr updates its rows (against the current
    // global state) and broadcasts them before the next rank starts
    sc.Krow.alloc(St);
    float* th_all = (R > 1) ? sv.theta_all.p : sv.theta.p;
    bool swept = false;
    const size_t cta_smem = (size_t)St * sizeof(double) + (size_t)St * P * sizeof(float);
    if (R == 1 && h->opt_live_fused && cta_smem <= 200 * 1024 && h->opt_live_cta) {
      // small enough for one CTA's shared memory: no grid barrier at all
      PYB_CUDA(cudaFuncSetAttribute(k_live_sweep_cta, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)cta_smem));
      k_live_sweep_cta<<<1, 1024, cta_smem, h->stream>>>(sv.theta.p, sv.g.p, sv.adam_m.p, sv.adam_v.p, sv.phi.p, (int)P, St, 1.0,
                                                        lr_t);
      count_launch(h);
      swept = true;
      h->svgd_stein_used = STEIN_LIVE_CTA;
    }
    if (R == 1 && h->opt_live_fused && !swept) {
      // one cooperative launch for the whole sweep (falls back to the per-particle launches if it cannot be co-resident)
      int per_sm = 0;
      PYB_CUDA(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, k_live_sweep, 256, 0));
      const int64_t want = std::max<int64_t>(St, (P + 255) / 256);
      const int grid = (int)std::min<int64_t>(want, (int64_t)per_sm * h->sm_count);
      if (grid >= 1) {
        float* th = sv.theta.p; const float* gp = sv.g.p; float* am = sv.adam_m.p; float* av = sv.adam_v.p;
        float* ph = sv.phi.p; int64_t Pp = P; int Sp = St; double gam = 1.0; double* kr = sc.Krow.p; float lrt = lr_t;
        void* args[] = {&th, &gp, &am, &av, &ph, &Pp, &Sp, &gam, &kr, &lrt};
        PYB_CUDA(cudaLaunchCooperativeKernel((void*)k_live_sweep, dim3(grid), dim3(256), args, 0, h->stream));
        count_launch(h);
        swept = true;
        h->svgd_stein_used = STEIN_LIVE_COOP;
      }
    }
    if (!swept) h->svgd_stein_used = STEIN_LIVE_LAUNCHES;
    for (int rr = 0; rr < R && !swept; ++rr) {
      if (rr == sv.rank) {
        for (int i = 0; i < (int)S; ++i) {
          const int gi = r0 + i;
          k_live_row<<<(unsigned)St, 256, 0, h->stream>>>(th_all, P, gi, 1.0, sc.Krow.p);
          k_live_update<<<(unsigned)((P + 255) / 256), 256, 0, h->stream>>>(
              th_all, sv.g.p, sv.adam_m.p, sv.adam_v.p, sv.phi.p, P, St, gi, i, 1.0, sc.Krow.p, lr_t);
          count_launch(h, 2);
        }
      }
      if (R > 1) nccl_broadcast_f32(sv.nccl_comm, th_all + (int64_t)rr * S * P, (size_t)S * P, rr, h->stream);
    }
    if (R > 1)
      PYB_CUDA(cudaMemcpyAsync(sv.theta.p, th_all + (int64_t)r0 * P, (size_t)S * P * sizeof(float), cudaMemcpyDeviceToDevice,
                               h->stream));
  } else if (!pshard) {
    const AdamFuse af = {sv.theta.p, sv.adam_m.p, sv.adam_v.p, lr_t};
    phi_canonical(h, theta_all, g_all, r0, (int)S, St, sv.phi.p, nullptr, overlap ? sv.ev_grad : nullptr, &af, fold_prior);
  }
  sc.mean_loss.alloc(1);
  k_mean_float<<<1, 256, 0, h->stream>>>(sv.loss.p, S, sc.mean_loss.p);
  count_launch(h);
  if (R > 1) nccl_all_reduce_f64(sv.nccl_comm, sc.mean_loss.p, 1, h->stream);
  PYB_CUDA(cudaEventRecord(h->ev1, h->stream));
  double ml = 0.0, h2v[2] = {0.0, 0.0};
  PYB_CUDA(cudaMemcpyAsync(&ml, sc.mean_loss.p, sizeof(double), cudaMemcpyDeviceToHost, h->stream));
  if (sv.semantics != PYB_SVGD_REFERENCE_LIVE)     // the step's median-heuristic bandwidth, for diagnostics (info "svgd_h")
    PYB_CUDA(cudaMemcpyAsync(h2v, sc.h2.p, sizeof(h2v), cudaMemcpyDeviceToHost, h->stream));
  PYB_CUDA(cudaStreamSynchronize(h->stream));
  PYB_CUDA(cudaGetLastError());
  if (R > 1) nccl_check_async(&sv.nccl_comm);
  sv.last_h = sv.semantics != PYB_SVGD_REFERENCE_LIVE ? sqrt(h2v[0]) : 1.0;
  if (pshard && sv.ps_timed)
    for (int k = 0; k < 7; ++k) PYB_CUDA(cudaEventElapsedTime(&sv.ps_ms[k], sv.ps_ev[k], sv.ps_ev[k + 1]));
  float ms = 0.f;
  PYB_CUDA(cudaEventElapsedTime(&ms, h->ev0, h->ev1));
  h->last_device_ms = ms;
  if (loss_out) *loss_out = ml / (double)R;
}

// mean over the particles of the loss on a held-out set (SVGD.py:126-129: the reference runs one forward pass per
// particle over the whole validation split inside every step).  The set is uploaded once and stays in HBM; the
// particles never leave the device.  The gradient buffer is free between steps and serves as the tensor path's scratch.
void svgd_set_validation(pyb_handle* h, const float* X, const void* y, int64_t N) {
  SvgdState& sv = h->svgd;
  const Model& m = h->model;
  PYB_REQUIRE(h->have_data, PYB_ERR_STATE, "pyb_set_dataset fixes the loss kind: call it first");
  PYB_REQUIRE(X && y && N > 0, PYB_ERR_INVALID, "bad validation set");
  sv.val_X.alloc(N * m.in_dim);
  PYB_CUDA(cudaMemcpyAsync(sv.val_X.p, X, N * m.in_dim * sizeof(float), cudaMemcpyHostToDevice, h->stream));
  if (h->loss_kind == PYB_LOSS_SPARSE_CE) {
    const int32_t* yi = (const int32_t*)y;
    for (int64_t i = 0; i < N; ++i) PYB_REQUIRE(yi[i] >= 0 && yi[i] < m.out_dim, PYB_ERR_INVALID, "label out of range");
    sv.val_yi.alloc(N);
    PYB_CUDA(cudaMemcpyAsync(sv.val_yi.p, y, N * sizeof(int32_t), cudaMemcpyHostToDevice, h->stream));
  } else {
    sv.val_yf.alloc(N * m.out_dim);
    PYB_CUDA(cudaMemcpyAsync(sv.val_yf.p, y, N * m.out_dim * sizeof(float), cudaMemcpyHostToDevice, h->stream));
  }
  PYB_CUDA(cudaStreamSynchronize(h->stream));
  sv.val_N = N;
}
void svgd_validation_loss(pyb_handle* h, double* mean_loss_out, float* per_particle_out) {
  SvgdState& sv = h->svgd;
  PYB_REQUIRE(sv.inited, PYB_ERR_STATE, "pyb_svgd_init must be called first");
  PYB_REQUIRE(sv.val_N > 0, PYB_ERR_STATE, "pyb_svgd_set_validation must be called first");
  DevBuf<float> vloss;
  vloss.alloc(sv.S);
  const bool tensor = tc_supported_rows(h, sv.val_N) && (h->opt_path == PYB_PATH_AUTO || h->opt_path == PYB_PATH_TENSOR);
  eval_on_batch(h, sv.theta.p, sv.S, sv.val_X.p, sv.val_yi.p, sv.val_yf.p, sv.val_N, 1.0f, vloss.p,
                tensor ? sv.g.p : nullptr);
  sv.mean_loss.alloc(1);
  k_mean_float<<<1, 256, 0, h->stream>>>(vloss.p, sv.S, sv.mean_loss.p);
  count_launch(h);
  if (sv.world > 1) nccl_all_reduce_f64(sv.nccl_comm, sv.mean_loss.p, 1, h->stream);
  double ml = 0.0;
  PYB_CUDA(cudaMemcpyAsync(&ml, sv.mean_loss.p, sizeof(double), cudaMemcpyDeviceToHost, h->stream));
  if (per_particle_out)
    PYB_CUDA(cudaMemcpyAsync(per_particle_out, vloss.p, sv.S * sizeof(float), cudaMemcpyDeviceToHost, h->stream));
  PYB_CUDA(cudaStreamSynchronize(h->stream));
  PYB_CUDA(cudaGetLastError());
  if (mean_loss_out) *mean_loss_out = ml / (double)sv.world;
}

void svgd_phi(pyb_handle* h, const double* X, const float* G, int64_t S, int sem, float* phi, double* h_out) {
  PYB_REQUIRE(S > 0 && S <= 65535, PYB_ERR_INVALID, "S must be in [1, 65535]");
  const int64_t P = h->model.P;
  SvgdState& sv = h->svgd;
  DevBuf<double> dX64;
  DevBuf<float> dX, dG, dphi;
  dX64.alloc(S * P); dX.alloc(S * P); dG.alloc(S * P); dphi.alloc(S * P);
  PYB_CUDA(cudaMemcpyAsync(dX64.p, X, S * P * sizeof(double), cudaMemcpyHostToDevice, h->stream));
  PYB_CUDA(cudaMemcpyAsync(dG.p, G, S * P * sizeof(float), cudaMemcpyHostToDevice, h->stream));
  dim3 grid((unsigned)((P + 1023) / 1024), (unsigned)S);
  k_svgd_init<<<grid, 256, 0, h->stream>>>(dX.p, dX64.p, nullptr, nullptr, P, 0, 0);  // f64 -> f32 (SVGD.py:62-63,101)
  count_launch(h);
  if (sem == PYB_SVGD_CANONICAL_MEDIAN) {
    phi_canonical(h, dX.p, dG.p, 0, (int)S, (int)S, dphi.p, h_out);
  } else {
    sv.d2.alloc((size_t)S * S);
    sv.rowsum.alloc(S);
    dim3 g1((unsigned)((S + 15) / 16), (unsigned)((S + 15) / 16));
    k_gram_d2<<<g1, 256, 0, h->stream>>>(dX.p, P, 0, (int)S, (int)S, sv.d2.p);
    k_kernel_fixed_rowsum<<<(unsigned)S, 256, 0, h->stream>>>(sv.d2.p, (int)S, 1.0, sv.rowsum.p);
    dim3 g2((unsigned)((P + 255) / 256), (unsigned)S);
    k_phi_live_all<<<g2, 256, 0, h->stream>>>(sv.d2.p, dX.p, dG.p, P, (int)S, 1.0, sv.rowsum.p, dphi.p);
    count_launch(h, 3);
    if (h_out) *h_out = 1.0;
  }
  PYB_CUDA(cudaMemcpyAsync(phi, dphi.p, S * P * sizeof(float), cudaMemcpyDeviceToHost, h->stream));
  PYB_CUDA(cudaStreamSynchronize(h->stream));
  PYB_CUDA(cudaGetLastError());
}

}  // namespace pyb
