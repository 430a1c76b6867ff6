// tc_layer2.cuh — SIMT kernels around the GEMMs: bf16 hi/lo split (+transpose) of fp32 operands, the stand-alone
// layer-2 forward/backward kernel of the unfused path, the forward-only layer 2 of the predictive, and the
// fixed-order reductions of per-block / per-split partial sums.
#pragma once
#include "tc_gemm.cuh"

namespace pyb {

// ------------------------------------------------------------------------------------------
// SIMT helpers around the GEMMs
// ------------------------------------------------------------------------------------------
__device__ __forceinline__ void split_bf16(float x, __nv_bfloat16& hi, __nv_bfloat16& lo) {
  hi = __float2bfloat16_rn(x);
  lo = __float2bfloat16_rn(x - __bfloat162float(hi));
}

// src [R, C] fp32 (row stride lds) -> hi/lo [R, C] bf16 (row stride ldd), same orientation
// center != nullptr: column c is split as src - center[c]
__global__ void k_split_rows(const float* src, int64_t R, int C, int64_t lds, __nv_bfloat16* hi, __nv_bfloat16* lo,
                             int64_t ldd, const float* center = nullptr) {
  const int64_t total = R * C;
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (int64_t)gridDim.x * blockDim.x) {
    int64_t r = i / C;
    int c = (int)(i - r * C);
    __nv_bfloat16 h, l;
    split_bf16(center ? src[r * lds + c] - center[c] : src[r * lds + c], h, l);
    hi[r * ldd + c] = h;
    lo[r * ldd + c] = l;
  }
}
// the same for even C, lds, ldd and 8-byte aligned bases (every row then starts 8-byte aligned in src and 4-byte aligned
// in hi/lo): two elements per thread, 8-byte loads and 4-byte stores
__global__ void k_split_rows2(const float* __restrict__ src, int64_t R, int C2, int64_t lds, __nv_bfloat16* __restrict__ hi,
                              __nv_bfloat16* __restrict__ lo, int64_t ldd, const float* __restrict__ center = nullptr) {
  const int64_t total = R * C2;
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (int64_t)gridDim.x * blockDim.x) {
    const int64_t r = i / C2;
    const int c = 2 * (int)(i - r * C2);
    float2 v = *reinterpret_cast<const float2*>(src + r * lds + c);
    if (center) { v.x -= center[c]; v.y -= center[c + 1]; }
    __nv_bfloat16 h0, l0, h1, l1;
    split_bf16(v.x, h0, l0);
    split_bf16(v.y, h1, l1);
    *reinterpret_cast<__nv_bfloat162*>(hi + r * ldd + c) = __nv_bfloat162(h0, h1);
    *reinterpret_cast<__nv_bfloat162*>(lo + r * ldd + c) = __nv_bfloat162(l0, l1);
  }
}

// src [R, C] fp32 (batch stride sb) -> transposed hi/lo [C(+ones row), Rpad] bf16 per batch element.
// grid (ceil(C/32), ceil(R/32), batch), block (32, 8)
// Row order inside a 128-row block as the fused G1+layer-2 epilogue stores it: the 4 rows {g, g+8, g+16, g+24} of a
// 32-row TMEM quadrant that one thread owns become 4 CONSECUTIVE elements (one 8-byte store).  Any operand that is
// contracted against those arrays over the data rows ([X^T;1] in the dW1 GEMM) must use the same order.
__host__ __device__ __forceinline__ int fused_row_pos(int r) { return (r & ~31) | ((r & 7) << 2) | ((r >> 3) & 3); }

__global__ void k_split_transpose(const float* src, int64_t sb, int R, int C, int64_t lds, __nv_bfloat16* hi,
                                  __nv_bfloat16* lo, int64_t db, int64_t ldd, int perm = 0) {
  __shared__ float t[32][33];
  const float* s = src + (int64_t)blockIdx.z * sb;
  int c0 = blockIdx.x * 32, r0 = blockIdx.y * 32;
  for (int i = threadIdx.y; i < 32; i += 8) {
    int r = r0 + i, c = c0 + threadIdx.x;
    t[i][threadIdx.x] = (r < R && c < C) ? s[(int64_t)r * lds + c] : 0.f;
  }
  __syncthreads();
  for (int i = threadIdx.y; i < 32; i += 8) {
    int c = c0 + i, r = r0 + threadIdx.x;
    if (c < C && r < R) {
      __nv_bfloat16 h, l;
      split_bf16(t[threadIdx.x][i], h, l);
      int64_t o = (int64_t)blockIdx.z * db + (int64_t)c * ldd + (perm ? fused_row_pos(r) : r);
      hi[o] = h;
      lo[o] = l;
    }
  }
}

__global__ void k_fill_ones_perm(__nv_bfloat16* p, int n) {      // p[fused_row_pos(r)] = 1 for r < n
  for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < n; i += gridDim.x * blockDim.x)
    p[fused_row_pos(i)] = __float2bfloat16_rn(1.0f);
}
__global__ void k_fill_bf16(__nv_bfloat16* p, int64_t n, float v) {
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x)
    p[i] = __float2bfloat16_rn(v);
}

// Layer 2 forward/backward.  One thread owns TWO adjacent data rows (packed bf16x2 loads/stores are
// then 128 B per warp); a block walks 256-row tiles of one chain.  a1 = hi + lo is read ONCE: for
// relu the derivative mask is kept as 2 x 256 bits in registers; other activations re-read a1.
constexpr int L2_CMAX = 16;
constexpr int L2_ROWS = 256;    // rows per tile (128 threads x 2)
struct Layer2Params {
  const __nv_bfloat16* a_hi; const __nv_bfloat16* a_lo;     // A1^T [Bc*H][ld]
  __nv_bfloat16* zt_hi; __nv_bfloat16* zt_lo;               // dZ1^T [Bc*H][ld]
  __nv_bfloat16* z2_hi; __nv_bfloat16* z2_lo;               // dZ2^T [Bc*16][ld]
  int k_tiles;                 // 128-row tiles per chain; arrays are blocked [chain][tile][unit][128]
  const float* theta; int64_t P; int64_t w2_off, b2_off;
  int H, C, N, act1, out_act, loss_kind;
  const int32_t* y_i; const float* y_f;
  float scale;                 // n_train (or 1): dZ = scale * d(mean loss)/dz
  double* loss_partial;        // [Bc][n_groups]
  float* b2_partial;           // [Bc][n_groups][16]
  int n_groups, n_tiles;
  float* fwd_out;              // fused forward-only mode: [Bc][N][C] outputs (softmax / output activation applied)
  // int8-slice operands of the fused kernel (tc_fused.cuh, I8 != 0; tc_i8.cuh)
  const float* sx;             // [N] per-row scale of the forward X slices (rows of the centred data)
  const float* cw;             // [Bc][H] s_w / 127^2: column scale of the W1^T slices times the slice unit
  const float* zq;             // [Bc][H] 127 / s_z: quantisation factor of the dZ1^T slices (I8 == 2)
  int8_t* zi_hi; int8_t* zi_lo;   // dZ1^T int8 slices, blocked [chain][tile][H][128]
  int dbg_flags;               // timing experiments only (results are wrong when set): 2 no phase-B stores, 4 no A1 stores, 8 no phase-B mma, 16 no phase-A mma, 32 no softmax
  unsigned long long* dbg;     // optional [grid][8] cycle sums of the kernel's phases (option "tc_timeline"), else null
};
__device__ __forceinline__ float2 unpack_bf16x2(uint32_t v) {
  return make_float2(__uint_as_float(v << 16), __uint_as_float(v & 0xffff0000u));
}
__device__ __forceinline__ uint32_t pack_bf16x2(__nv_bfloat16 a, __nv_bfloat16 b) {
  return (uint32_t)__bfloat16_as_ushort(a) | ((uint32_t)__bfloat16_as_ushort(b) << 16);
}
template <int CP, typename LT>
__device__ __forceinline__ void l2_loss_dz(const Layer2Params& p, int r, bool valid, const float* z, float* dz,
                                           LT& loss_acc, float invN) {
  const int C = p.C;
#pragma unroll
  for (int c = 0; c < CP; ++c) dz[c] = 0.f;
  if (!valid) return;
  if (p.loss_kind == PYB_LOSS_SPARSE_CE) {
    float mx = -INFINITY;
#pragma unroll
    for (int c = 0; c < CP; ++c) if (c < C) mx = fmaxf(mx, z[c]);
    float se = 0.f;
#pragma unroll
    for (int c = 0; c < CP; ++c) if (c < C) se += expf(z[c] - mx);
    const int yi = p.y_i[r];
    float zy = 0.f;
#pragma unroll
    for (int c = 0; c < CP; ++c) if (c == yi) zy = z[c];
    loss_acc += (LT)(logf(se) - (zy - mx));
    const float inv = 1.0f / se;
#pragma unroll
    for (int c = 0; c < CP; ++c)
      if (c < C) dz[c] = (expf(z[c] - mx) * inv - (c == yi ? 1.f : 0.f)) * invN;
  } else {
    float acc = 0.f;
    const float sc = 2.0f * invN / (float)C;
#pragma unroll
    for (int c = 0; c < CP; ++c)
      if (c < C) {
        float a = act_apply(z[c], p.out_act);
        float df = a - p.y_f[(int64_t)r * C + c];
        acc += df * df;
        dz[c] = sc * df * act_grad_from_output(a, p.out_act);
      }
    loss_acc += (LT)(acc / (float)C);
  }
}
// CP = class count padded to a multiple of 4 (register tile of the per-row logits)
template <int CP>
__global__ void __launch_bounds__(128, 4) k_layer2(Layer2Params p) {
  __shared__ __align__(16) float W2s[256 * CP];
  __shared__ float b2s[CP];
  __shared__ uint32_t mask_s[2][8][128];
  __shared__ float redf[4][CP];
  __shared__ double scratch[32];
  const int t = threadIdx.x, b = blockIdx.y;
  const int H = p.H, C = p.C;
  const float* th = p.theta + (int64_t)b * p.P;
  for (int i = t; i < H * CP; i += 128) {
    int h = i / CP, c = i % CP;
    W2s[i] = (c < C) ? th[p.w2_off + (int64_t)h * C + c] : 0.f;
  }
  if (t < CP) b2s[t] = (t < C) ? th[p.b2_off + t] : 0.f;
  __syncthreads();
  // blocked layout, in packed bf16x2 words: ((chain*k_tiles + tile128)*rows_per_block + unit)*64 + pair
  const uint32_t* ah = reinterpret_cast<const uint32_t*>(p.a_hi);
  const uint32_t* al = reinterpret_cast<const uint32_t*>(p.a_lo);
  uint32_t* zh = reinterpret_cast<uint32_t*>(p.zt_hi);
  uint32_t* zl = reinterpret_cast<uint32_t*>(p.zt_lo);
  uint32_t* z2h = reinterpret_cast<uint32_t*>(p.z2_hi);
  uint32_t* z2l = reinterpret_cast<uint32_t*>(p.z2_lo);
  const int64_t ld2 = 64;                  // pitch between hidden units inside a block, in packed pairs
  float accb[CP];
#pragma unroll
  for (int c = 0; c < CP; ++c) accb[c] = 0.f;
  double loss_acc = 0.0;
  const float invN = p.scale / (float)p.N;
  const bool relu = p.act1 == PYB_ACT_RELU;
  const int nhb = (H + 31) >> 5;
  for (int tile = blockIdx.x; tile < p.n_tiles; tile += gridDim.x) {
    const int r0 = tile * L2_ROWS + 2 * t;
    const int64_t tile128 = (int64_t)b * p.k_tiles + tile * 2 + (t >> 6);   // this thread's 128-row block
    const int64_t col = tile128 * H * 64 + (t & 63);                        // word offset of (unit 0, this row pair)
    const int64_t col2 = tile128 * L2_CMAX * 64 + (t & 63);                 // same for the dZ2^T blocks
    const bool v0 = r0 < p.N, v1 = r0 + 1 < p.N;
    // ---- phase A: z2 = a1 W2 + b2 for both rows; relu mask bits go to shared memory
    float z0[CP], z1[CP];
#pragma unroll
    for (int c = 0; c < CP; ++c) { z0[c] = b2s[c]; z1[c] = b2s[c]; }
    for (int hb = 0; hb < nhb; ++hb) {
      uint32_t m0 = 0u, m1 = 0u;
      const uint32_t* ahp = ah + (int64_t)(hb * 32) * ld2 + col;
      const uint32_t* alp = al + (int64_t)(hb * 32) * ld2 + col;
      const int jn = min(32, H - hb * 32);
#pragma unroll 4
      for (int j = 0; j < jn; ++j) {
        const float2 hi = unpack_bf16x2(ahp[(int64_t)j * ld2]);
        const float2 lo = unpack_bf16x2(alp[(int64_t)j * ld2]);
        const float a0 = hi.x + lo.x, a1v = hi.y + lo.y;
        m0 |= (a0 > 0.f ? 1u : 0u) << j;
        m1 |= (a1v > 0.f ? 1u : 0u) << j;
        const float4* w = reinterpret_cast<const float4*>(&W2s[(hb * 32 + j) * CP]);
#pragma unroll
        for (int q4 = 0; q4 < CP / 4; ++q4) {
          const float4 wv = w[q4];
          z0[q4 * 4 + 0] = fmaf(a0, wv.x, z0[q4 * 4 + 0]); z1[q4 * 4 + 0] = fmaf(a1v, wv.x, z1[q4 * 4 + 0]);
          z0[q4 * 4 + 1] = fmaf(a0, wv.y, z0[q4 * 4 + 1]); z1[q4 * 4 + 1] = fmaf(a1v, wv.y, z1[q4 * 4 + 1]);
          z0[q4 * 4 + 2] = fmaf(a0, wv.z, z0[q4 * 4 + 2]); z1[q4 * 4 + 2] = fmaf(a1v, wv.z, z1[q4 * 4 + 2]);
          z0[q4 * 4 + 3] = fmaf(a0, wv.w, z0[q4 * 4 + 3]); z1[q4 * 4 + 3] = fmaf(a1v, wv.w, z1[q4 * 4 + 3]);
        }
      }
      mask_s[0][hb][t] = m0;
      mask_s[1][hb][t] = m1;
    }
    // ---- loss and dZ2 (scaled); dZ2^T stored split for the dW2 GEMM
    float dz0[CP], dz1[CP];
    l2_loss_dz<CP>(p, r0, v0, z0, dz0, loss_acc, invN);
    l2_loss_dz<CP>(p, r0 + 1, v1, z1, dz1, loss_acc, invN);
#pragma unroll
    for (int c = 0; c < CP; ++c) {
      accb[c] += dz0[c] + dz1[c];
      __nv_bfloat16 h0, l0, h1, l1;
      split_bf16(dz0[c], h0, l0);
      split_bf16(dz1[c], h1, l1);
      z2h[(int64_t)c * ld2 + col2] = pack_bf16x2(h0, h1);
      z2l[(int64_t)c * ld2 + col2] = pack_bf16x2(l0, l1);
    }
    // ---- phase A2: dZ1 = (dZ2 W2^T) * act'(a1) -> split bf16, transposed packed store
    for (int hb = 0; hb < nhb; ++hb) {
      const uint32_t m0 = mask_s[0][hb][t], m1 = mask_s[1][hb][t];   // own writes: no barrier needed
      uint32_t* zhp = zh + (int64_t)(hb * 32) * ld2 + col;
      uint32_t* zlp = zl + (int64_t)(hb * 32) * ld2 + col;
      const int jn = min(32, H - hb * 32);
#pragma unroll 4
      for (int j = 0; j < jn; ++j) {
        const int h = hb * 32 + j;
        const float4* w = reinterpret_cast<const float4*>(&W2s[h * CP]);
        float d0 = 0.f, d1 = 0.f;
#pragma unroll
        for (int q4 = 0; q4 < CP / 4; ++q4) {
          const float4 wv = w[q4];
          d0 = fmaf(dz0[q4 * 4 + 0], wv.x, d0); d1 = fmaf(dz1[q4 * 4 + 0], wv.x, d1);
          d0 = fmaf(dz0[q4 * 4 + 1], wv.y, d0); d1 = fmaf(dz1[q4 * 4 + 1], wv.y, d1);
          d0 = fmaf(dz0[q4 * 4 + 2], wv.z, d0); d1 = fmaf(dz1[q4 * 4 + 2], wv.z, d1);
          d0 = fmaf(dz0[q4 * 4 + 3], wv.w, d0); d1 = fmaf(dz1[q4 * 4 + 3], wv.w, d1);
        }
        if (relu) {
          d0 = ((m0 >> j) & 1u) ? d0 : 0.f;
          d1 = ((m1 >> j) & 1u) ? d1 : 0.f;
        } else {
          const float2 hi = unpack_bf16x2(ah[(int64_t)h * ld2 + col]);
          const float2 lo = unpack_bf16x2(al[(int64_t)h * ld2 + col]);
          d0 *= act_grad_from_output(hi.x + lo.x, p.act1);
          d1 *= act_grad_from_output(hi.y + lo.y, p.act1);
        }
        __nv_bfloat16 h0, l0, h1, l1;
        split_bf16(d0, h0, l0);
        split_bf16(d1, h1, l1);
        zhp[(int64_t)j * ld2] = pack_bf16x2(h0, h1);
        zlp[(int64_t)j * ld2] = pack_bf16x2(l0, l1);
      }
    }
  }
  // ---- per-block partials: db2 (sum of dZ2 over the block's rows) and the loss
  const int lane = t & 31, w = t >> 5;
#pragma unroll
  for (int c = 0; c < CP; ++c) {
    float sum = warp_sum(accb[c]);
    if (lane == 0) redf[w][c] = sum;
  }
  __syncthreads();
  if (t < L2_CMAX)
    p.b2_partial[((int64_t)b * p.n_groups + blockIdx.x) * L2_CMAX + t] =
        (t < CP) ? redf[0][t] + redf[1][t] + redf[2][t] + redf[3][t] : 0.f;
  double tot = block_sum<double>(loss_acc, scratch);
  if (t == 0) p.loss_partial[(int64_t)b * p.n_groups + blockIdx.x] = tot;
}


// forward-only layer 2 (posterior predictive): out[b][row][c] = softmax(a1 W2 + b2) or act(.)
struct Layer2FwdParams {
  const __nv_bfloat16* a_hi; const __nv_bfloat16* a_lo; int k_tiles;
  const float* theta; int64_t P; int64_t w2_off, b2_off;
  int H, C, N, out_act, n_tiles;
  float* out;
};
__global__ void __launch_bounds__(128) k_layer2_fwd(Layer2FwdParams p) {
  __shared__ __align__(16) float W2s[256 * L2_CMAX];
  __shared__ float b2s[L2_CMAX];
  const int t = threadIdx.x, b = blockIdx.y, H = p.H, C = p.C;
  const float* th = p.theta + (int64_t)b * p.P;
  for (int i = t; i < H * L2_CMAX; i += 128) {
    int h = i / L2_CMAX, c = i % L2_CMAX;
    W2s[i] = (c < C) ? th[p.w2_off + (int64_t)h * C + c] : 0.f;
  }
  if (t < L2_CMAX) b2s[t] = (t < C) ? th[p.b2_off + t] : 0.f;
  __syncthreads();
  const uint32_t* ah = reinterpret_cast<const uint32_t*>(p.a_hi);
  const uint32_t* al = reinterpret_cast<const uint32_t*>(p.a_lo);
  for (int tile = blockIdx.x; tile < p.n_tiles; tile += gridDim.x) {
    const int r0 = tile * L2_ROWS + 2 * t;
    const int64_t tile128 = (int64_t)b * p.k_tiles + tile * 2 + (t >> 6);
    const int64_t col = tile128 * H * 64 + (t & 63);
    float z0[L2_CMAX], z1[L2_CMAX];
#pragma unroll
    for (int c = 0; c < L2_CMAX; ++c) { z0[c] = b2s[c]; z1[c] = b2s[c]; }
#pragma unroll 4
    for (int h = 0; h < H; ++h) {
      const float2 hi = unpack_bf16x2(ah[(int64_t)h * 64 + col]);
      const float2 lo = unpack_bf16x2(al[(int64_t)h * 64 + col]);
      const float a0 = hi.x + lo.x, a1v = hi.y + lo.y;
      const float4* w = reinterpret_cast<const float4*>(&W2s[h * L2_CMAX]);
#pragma unroll
      for (int q4 = 0; q4 < L2_CMAX / 4; ++q4) {
        const float4 wv = w[q4];
        z0[q4 * 4 + 0] = fmaf(a0, wv.x, z0[q4 * 4 + 0]); z1[q4 * 4 + 0] = fmaf(a1v, wv.x, z1[q4 * 4 + 0]);
        z0[q4 * 4 + 1] = fmaf(a0, wv.y, z0[q4 * 4 + 1]); z1[q4 * 4 + 1] = fmaf(a1v, wv.y, z1[q4 * 4 + 1]);
        z0[q4 * 4 + 2] = fmaf(a0, wv.z, z0[q4 * 4 + 2]); z1[q4 * 4 + 2] = fmaf(a1v, wv.z, z1[q4 * 4 + 2]);
        z0[q4 * 4 + 3] = fmaf(a0, wv.w, z0[q4 * 4 + 3]); z1[q4 * 4 + 3] = fmaf(a1v, wv.w, z1[q4 * 4 + 3]);
      }
    }
#pragma unroll
    for (int rr = 0; rr < 2; ++rr) {
      const int r = r0 + rr;
      if (r >= p.N) continue;
      float* z = rr ? z1 : z0;
      float* o = p.out + ((int64_t)b * p.N + r) * C;
      if (p.out_act == PYB_ACT_SOFTMAX) {
        float mx = -INFINITY;
#pragma unroll
        for (int c = 0; c < L2_CMAX; ++c) if (c < C) mx = fmaxf(mx, z[c]);
        float se = 0.f;
#pragma unroll
        for (int c = 0; c < L2_CMAX; ++c) if (c < C) se += expf(z[c] - mx);
        const float inv = 1.0f / se;
#pragma unroll
        for (int c = 0; c < L2_CMAX; ++c) if (c < C) o[c] = expf(z[c] - mx) * inv;
      } else {
#pragma unroll
        for (int c = 0; c < L2_CMAX; ++c) if (c < C) o[c] = act_apply(z[c], p.out_act);
      }
    }
  }
}

// grad[b][b2_off + c] = sum_g b2_partial[b][g][c]; loss[b] = sum_g loss_partial / N.  Fixed summation order
// (16 interleaved strands per class, combined in order): deterministic for any number of groups.  blockDim = 256.
__global__ void k_layer2_reduce(const float* b2_partial, const double* loss_partial, int n_groups, int C, float* grad,
                                int64_t P, int64_t b2_off, float* loss_out, int N) {
  __shared__ double scratch[32];
  __shared__ float strands[16][L2_CMAX + 1];
  const int b = blockIdx.x, t = threadIdx.x;
  {
    const int c = t & 15, j = t >> 4;                 // class, strand
    float s = 0.f;
    if (c < C)
      for (int g = j; g < n_groups; g += 16) s += b2_partial[((int64_t)b * n_groups + g) * L2_CMAX + c];
    strands[j][c] = s;
  }
  __syncthreads();
  if (t < C) {
    float s = 0.f;
#pragma unroll
    for (int j = 0; j < 16; ++j) s += strands[j][t];
    grad[(int64_t)b * P + b2_off + t] = s;
  }
  double a = 0.0;
  for (int g = t; g < n_groups; g += blockDim.x) a += loss_partial[(int64_t)b * n_groups + g];
  double tot = block_sum<double>(a, scratch);
  if (t == 0 && loss_out) loss_out[b] = (float)(tot / (double)N);
}

// out[b*out_stride + i] = sum_s part[s*split_stride + b*part_stride + i]   (fixed order => deterministic)
__global__ void k_reduce_ksplits(const float* part, int splits, int64_t split_stride, int64_t part_stride, int64_t count,
                                 float* out, int64_t out_stride) {
  const int b = blockIdx.y;
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < count; i += (int64_t)gridDim.x * blockDim.x) {
    float s = 0.f;
    for (int k = 0; k < splits; ++k) s += part[(int64_t)k * split_stride + (int64_t)b * part_stride + i];
    out[(int64_t)b * out_stride + i] = s;
  }
}
// Gram matrix: out[i][j] = out[j][i] for every element whose 256x256 tile lies strictly below the diagonal
// (those tiles were skipped by the GEMM).  grid (n/32, n/32), block (32, 8); tiled through shared memory.
__global__ void k_mirror_lower_tiles(float* out, int n, int64_t ld) {
  __shared__ float t[32][33];
  const int bi = blockIdx.y, bj = blockIdx.x;          // 32x32 block (rows bi, cols bj) of the LOWER part to fill
  if ((bj * 32) / 256 >= (bi * 32) / 256) return;
  for (int r = threadIdx.y; r < 32; r += 8) {           // read the mirrored block (rows bj, cols bi)
    const int i = bj * 32 + r, j = bi * 32 + threadIdx.x;
    t[r][threadIdx.x] = (i < n && j < n) ? out[(int64_t)i * ld + j] : 0.f;
  }
  __syncthreads();
  for (int r = threadIdx.y; r < 32; r += 8) {
    const int i = bi * 32 + r, j = bj * 32 + threadIdx.x;
    if (i < n && j < n) out[(int64_t)i * ld + j] = t[threadIdx.x][r];
  }
}
// one accumulator sees at most TC_SPLIT_CHUNKS chunks (8192 K elements): <= 1536 truncating accumulations
constexpr int TC_SPLIT_CHUNKS = 256;

}  // namespace pyb
