// fused_small.cu — small-width path (BASELINE configs C1/C2: make_moons 2-50-2, 1-D regression
// 1-1-1): ONE CTA per chain, dataset + q/p/grad resident in shared memory, the whole HMC iteration
// (Philox momentum draw, K0, L+1 full-data forward/backward evaluations with the prior, leapfrog
// kicks/drifts, K1/U1, Metropolis test) in ONE launch.  fp32 SIMT, warp-shuffle block reductions.
//
// Reference: HMC.step HMC.py:74-104 (one chain, ~8 eager TF ops per leapfrog step and two host
// syncs per iteration); _potential_energy :149-159; _step_p :128-136; _step_q :138-141.
//
// Evaluation inside the CTA (N rows, D inputs, H hidden, C outputs):
//   phase 1  thread == data row:  z1, a1, z2 -> loss, dZ2 (kept in smem for all rows)
//   phase 2  thread == (hidden unit, row slice): recompute a1 from the unit's own weights (registers),
//            dZ1 = (dZ2 W2^T) act'(a1), accumulate dW1[:,h], db1[h], dW2[h,:] in registers
//            — TWO data rows per step as packed FP32 pairs (fma.rn.f32x2: one issue slot, two FMAs per lane); the
//            pair's inputs and deltas are (D + C) consecutive 8-byte words of the pair-interleaved array sm.xd: one
//            address register, 16-byte shared loads.  Phase 1 runs its rows as packed pairs too.
//   slices are combined in a fixed order (deterministic), db2 by one warp per class.
//
// Few chains (the reference runs ONE, HMC.py:74): a chain is then spread over a thread-block CLUSTER of up to 8
// CTAs.  Each CTA keeps the whole state (q, p: a few hundred floats, updated redundantly and identically) and
// evaluates an eighth of the data rows; after every evaluation the partial gradients and loss meet through
// distributed shared memory (one cluster barrier per evaluation, double-buffered exchange, fixed summation order).
#pragma once
#include "common.cuh"
#include <cooperative_groups.h>
#include <algorithm>

namespace pyb {

constexpr int FS_THREADS = 256;
constexpr int FS_HMAX = 256;

struct FsParams {
  // model / data
  int N, H, act1, out_act, loss_kind;
  int64_t P, w1_off, b1_off, w2_off, b2_off;
  const float* X; const int32_t* y_i; const float* y_f;
  const float* mu; const float* inv_var;
  float n_train;                 // scale of the mean loss in U (HMC.py:158)
  // eval-only mode
  const float* theta; float* loss_out; float* grad_out; float scale;
  // HMC iteration mode
  float* q; float* p; float* q0; const float* inj_p; const float* inj_u;
  float eps, half_eps, drift, stdv, inv2m, prior_const;
  double* step; double m;        // step != NULL: per-chain step sizes replace eps / half_eps / drift
  double* da; double da_target; int64_t da_t;   // da != NULL: adaptation iteration da_t (dual_average)
  const float* beta;             // != NULL: tempering ladder, the chain's inverse temperature scales the data term
  int L, semantics, burning;
  int cluster;                   // CTAs per chain (1, 2, 4 or 8)
  uint64_t seed; uint32_t iter; int64_t chain_offset;
  float* U0; float* U1; float* K0; float* K1; float* log_alpha; float* ret_loss; int32_t* accepted;
  unsigned long long* counters; double* loss_sum;
};

struct FsSmem {
  float* xd;      // [ceil(N / 2)][D + C][2]: rows 2j, 2j + 1 interleaved — inputs x[d], then the deltas dZ2[c] phase 1 leaves
  float* ys;      // labels as float bits (int) or targets [N][C]
  float* qs; float* ps; float* gs;   // [P]
  float* pk;      // [H][FsPk::S] packed per-unit parameters, rows padded to 16 bytes
  float* part;    // [n_slices][H*(D+1+C)]
  float* gx;      // [2][GX] cluster exchange: partial gradient [P] + loss sum (double) of this CTA's rows
  double* red;    // [32]
  float* kc;      // [4] leapfrog coefficients of the chain's step size: full kick, half kick, drift; inverse temperature
};

template <typename T>
__device__ __forceinline__ T fs_block_sum_all(T v, T* scratch) {
  // block-wide sum broadcast to every thread
  int lane = threadIdx.x & 31, w = threadIdx.x >> 5;
  v = warp_sum(v);
  __syncthreads();
  if (lane == 0) scratch[w] = v;
  __syncthreads();
  T r = (lane < (FS_THREADS >> 5)) ? scratch[lane] : T(0);
  r = warp_sum(r);
  return r;
}

// packed FP32 pairs (sm_100: FFMA2 / FADD2 — two lanes' worth of FMA per issue slot), carried in 64-bit registers
typedef unsigned long long fs_f2;
__device__ __forceinline__ fs_f2 fs_pack2(float x, float y) {
  fs_f2 r;
  asm("mov.b64 %0, {%1, %2};" : "=l"(r) : "f"(x), "f"(y));
  return r;
}
__device__ __forceinline__ void fs_unpack2(fs_f2 v, float& x, float& y) {
  asm("mov.b64 {%0, %1}, %2;" : "=f"(x), "=f"(y) : "l"(v));
}
__device__ __forceinline__ fs_f2 fs_fma2(fs_f2 a, fs_f2 b, fs_f2 c) {
  fs_f2 r;
  asm("fma.rn.f32x2 %0, %1, %2, %3;" : "=l"(r) : "l"(a), "l"(b), "l"(c));
  return r;
}
__device__ __forceinline__ fs_f2 fs_mul2(fs_f2 a, fs_f2 b) {
  fs_f2 r;
  asm("mul.rn.f32x2 %0, %1, %2;" : "=l"(r) : "l"(a), "l"(b));
  return r;
}
__device__ __forceinline__ fs_f2 fs_add2(fs_f2 a, fs_f2 b) {
  fs_f2 r;
  asm("add.rn.f32x2 %0, %1, %2;" : "=l"(r) : "l"(a), "l"(b));
  return r;
}

__device__ __forceinline__ uint32_t fs_smem_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }
// NW consecutive 8-byte words from one shared address: 16-byte loads when NW is even (a row pair is then a multiple of
// 16 bytes, so every pair starts 16-byte aligned), 8-byte loads otherwise
template <int NW>
__device__ __forceinline__ void fs_lds_pairs(uint32_t a, fs_f2 (&v)[NW]) {
  if (NW % 2 == 0) {
#pragma unroll
    for (int i = 0; i + 1 < NW; i += 2)
      asm volatile("ld.shared.v2.b64 {%0, %1}, [%2];" : "=l"(v[i]), "=l"(v[i + 1]) : "r"(a + 8u * (uint32_t)i) : "memory");
  } else {
#pragma unroll
    for (int i = 0; i < NW; ++i) asm volatile("ld.shared.b64 %0, [%1];" : "=l"(v[i]) : "r"(a + 8u * (uint32_t)i) : "memory");
  }
}
// position of (row r, input d) / (row r, delta c) in the pair-interleaved array
template <int D, int C>
__device__ __forceinline__ int fs_xi(int r, int d) { return (r >> 1) * (2 * (D + C)) + 2 * d + (r & 1); }
template <int D, int C>
__device__ __forceinline__ int fs_dzi(int r, int c) { return (r >> 1) * (2 * (D + C)) + 2 * (D + c) + (r & 1); }
// per-unit parameter rows {W1[0..D)[h], b1[h], W2[h][0..C)} padded to 16-byte multiples: 16-byte shared loads
template <int D, int C>
struct FsPk { static constexpr int W = D + 1 + C, S = (W + 3) & ~3; };
template <int D, int C>
__device__ __forceinline__ void fs_load_unit(const float* pk, int h, float (&wr)[FsPk<D, C>::S]) {
  const float4* w4 = reinterpret_cast<const float4*>(pk + h * FsPk<D, C>::S);
#pragma unroll
  for (int i = 0; i < FsPk<D, C>::S / 4; ++i) {
    const float4 v = w4[i];
    wr[4 * i] = v.x; wr[4 * i + 1] = v.y; wr[4 * i + 2] = v.z; wr[4 * i + 3] = v.w;
  }
}

// one pass of phase 1 over the rows r0 + t + k * 256 (k < RT, r < re): forward, loss, dZ2 -> sm.dz2; returns this
// thread's loss sum.  Per row the arithmetic (and its order) is the same whatever RT is.
template <int D, int C, int ACT, int RT>
__device__ __forceinline__ double fs_phase1_pass(const FsParams& p, const FsSmem& sm, const float (&b2)[C], float sc, int r0,
                                                 int re) {
  constexpr int PKW = D + 1 + C;
  const int act1 = ACT >= 0 ? ACT : p.act1;
  const int t = threadIdx.x, H = p.H;
  float z2[RT][C];
  if (RT == 1 && r0 + (t & ~31) >= re) return 0.0;      // partial last pass: warps without a row skip it (warp-uniform)
  if (RT >= 2) {
    // rows k = 2i, 2i + 1 in the two halves of packed registers; the unit's parameters are broadcast operands
    constexpr int RP = RT / 2 > 0 ? RT / 2 : 1;
    fs_f2 x[RP][D], zp[RP][C];
#pragma unroll
    for (int i = 0; i < RP; ++i) {
      const int ra = r0 + t + 2 * i * FS_THREADS, rb2 = ra + FS_THREADS;
#pragma unroll
      for (int d = 0; d < D; ++d)
        x[i][d] = fs_pack2(ra < re ? sm.xd[fs_xi<D, C>(ra, d)] : 0.f, rb2 < re ? sm.xd[fs_xi<D, C>(rb2, d)] : 0.f);
#pragma unroll
      for (int c = 0; c < C; ++c) zp[i][c] = fs_pack2(b2[c], b2[c]);
    }
    for (int h = 0; h < H; ++h) {
      float wr[FsPk<D, C>::S];
      fs_load_unit<D, C>(sm.pk, h, wr);
      fs_f2 wb[PKW];
#pragma unroll
      for (int i = 0; i < PKW; ++i) wb[i] = fs_pack2(wr[i], wr[i]);
#pragma unroll
      for (int i = 0; i < RP; ++i) {
        fs_f2 z = wb[D];
#pragma unroll
        for (int d = 0; d < D; ++d) z = fs_fma2(x[i][d], wb[d], z);
        float z0, z1;
        fs_unpack2(z, z0, z1);
        const fs_f2 a = fs_pack2(act_apply(z0, act1), act_apply(z1, act1));
#pragma unroll
        for (int c = 0; c < C; ++c) zp[i][c] = fs_fma2(a, wb[D + 1 + c], zp[i][c]);
      }
    }
#pragma unroll
    for (int i = 0; i < RP; ++i)
#pragma unroll
      for (int c = 0; c < C; ++c) fs_unpack2(zp[i][c], z2[(2 * i) % RT][c], z2[(2 * i + 1) % RT][c]);
  } else {
    float x[D];
    const int r = r0 + t;
#pragma unroll
    for (int d = 0; d < D; ++d) x[d] = (r < re) ? sm.xd[fs_xi<D, C>(r, d)] : 0.f;
#pragma unroll
    for (int c = 0; c < C; ++c) z2[0][c] = b2[c];
    for (int h = 0; h < H; ++h) {
      float wr[FsPk<D, C>::S];
      fs_load_unit<D, C>(sm.pk, h, wr);
      float z = wr[D];
#pragma unroll
      for (int d = 0; d < D; ++d) z = fmaf(x[d], wr[d], z);
      const float a = act_apply(z, act1);
#pragma unroll
      for (int c = 0; c < C; ++c) z2[0][c] = fmaf(a, wr[D + 1 + c], z2[0][c]);
    }
  }
  double loss_acc = 0.0;
#pragma unroll
  for (int k = 0; k < RT; ++k) {
    const int r = r0 + t + k * FS_THREADS;
    if (r >= re) break;
    float dz[C];
    if (p.loss_kind == PYB_LOSS_SPARSE_CE) {
      float mx = z2[k][0];
#pragma unroll
      for (int c = 1; c < C; ++c) mx = fmaxf(mx, z2[k][c]);
      float se = 0.f;
#pragma unroll
      for (int c = 0; c < C; ++c) se += expf(z2[k][c] - mx);
      const int yi = __float_as_int(sm.ys[r]);
      float zy = 0.f;
#pragma unroll
      for (int c = 0; c < C; ++c) if (c == yi) zy = z2[k][c];
      loss_acc += (double)(logf(se) - (zy - mx));
      const float inv = 1.0f / se;
#pragma unroll
      for (int c = 0; c < C; ++c) dz[c] = (expf(z2[k][c] - mx) * inv - (c == yi ? 1.f : 0.f)) * sc;
    } else {
      float acc = 0.f;
#pragma unroll
      for (int c = 0; c < C; ++c) {
        float a = act_apply(z2[k][c], p.out_act);
        float df = a - sm.ys[r * C + c];
        acc += df * df;
        dz[c] = (2.0f * sc / (float)C) * df * act_grad_from_output(a, p.out_act);
      }
      loss_acc += (double)(acc / (float)C);
    }
#pragma unroll
    for (int c = 0; c < C; ++c) sm.xd[fs_dzi<D, C>(r, c)] = dz[c];
  }
  return loss_acc;
}

// over the data rows [rb, re): loss SUM (returned to every thread) and gout = scale/N * d(sum loss)/d theta for the
// parameters in sm.qs (N = all rows of the dataset: partial results of disjoint row ranges simply add up)
template <int D, int C, int ACT>
__device__ double fs_eval_rows(const FsParams& p, const FsSmem& sm, float scale, int rb, int re, float* gout) {
  constexpr int PKW = D + 1 + C;
  const int t = threadIdx.x, H = p.H, N = p.N;
  // ACT >= 0: the hidden activation is a compile-time constant (relu: the shipped models) and the per-(row, unit)
  // switches in act_apply / act_grad_from_output fold away; ACT < 0: any activation, selected at run time
  const int act1 = ACT >= 0 ? ACT : p.act1;
  // pack per-unit parameters: {W1[0..D)[h], b1[h], W2[h][0..C)}
  constexpr int PKS = FsPk<D, C>::S;
  for (int i = t; i < H * PKW; i += FS_THREADS) {
    int h = i / PKW, k = i - h * PKW;
    float v;
    if (k < D) v = sm.qs[p.w1_off + (int64_t)k * H + h];
    else if (k == D) v = sm.qs[p.b1_off + h];
    else v = sm.qs[p.w2_off + (int64_t)h * C + (k - D - 1)];
    sm.pk[h * PKS + k] = v;
  }
  __syncthreads();
  float b2[C];
#pragma unroll
  for (int c = 0; c < C; ++c) b2[c] = sm.qs[p.b2_off + c];
  // ---- phase 1: thread == RT data rows (r, r + 256, ...): every per-unit parameter fetched from shared memory feeds
  // RT rows.  Passes of 4 x 256, then 2 x 256, then 1 x 256 rows and a partial last pass: the choice depends only on
  // the rows left, so it is uniform over the block and no pass carries masked-off row slots
  double loss_acc = 0.0;
  const float sc = scale / (float)N;
  int r0 = rb;
  while (re - r0 >= 4 * FS_THREADS) { loss_acc += fs_phase1_pass<D, C, ACT, 4>(p, sm, b2, sc, r0, re); r0 += 4 * FS_THREADS; }
  if (re - r0 >= 2 * FS_THREADS) { loss_acc += fs_phase1_pass<D, C, ACT, 2>(p, sm, b2, sc, r0, re); r0 += 2 * FS_THREADS; }
  while (r0 < re) { loss_acc += fs_phase1_pass<D, C, ACT, 1>(p, sm, b2, sc, r0, re); r0 += FS_THREADS; }
  const double loss_tot = fs_block_sum_all<double>(loss_acc, sm.red);   // contains the __syncthreads dz2 needs
  // ---- phase 2: thread == (hidden unit, row slice)
  const int n_slices = FS_THREADS / H > 0 ? FS_THREADS / H : 1;
  const int h = t % H, slice = t / H;
  const int NG = H * PKW;
  if (slice < n_slices && t < n_slices * H) {
    float w[PKS];
    fs_load_unit<D, C>(sm.pk, h, w);
    // two rows (2j, 2j + 1) per step in the two halves of packed registers; the weights sit in both halves
    fs_f2 w1[D], w2[C], gw1[D], gw2[C], gb1 = 0ull;                  // (0.f, 0.f) is the all-zero bit pattern
    const fs_f2 b1 = fs_pack2(w[D], w[D]);
#pragma unroll
    for (int d = 0; d < D; ++d) { w1[d] = fs_pack2(w[d], w[d]); gw1[d] = 0ull; }
#pragma unroll
    for (int c = 0; c < C; ++c) { w2[c] = fs_pack2(w[D + 1 + c], w[D + 1 + c]); gw2[c] = 0ull; }
    auto step = [&](const fs_f2 (&x)[D], const fs_f2 (&dzr)[C]) {
      fs_f2 z = b1;
#pragma unroll
      for (int d = 0; d < D; ++d) z = fs_fma2(x[d], w1[d], z);
      float z0, z1;
      fs_unpack2(z, z0, z1);
      const float a0 = act_apply(z0, act1), a1 = act_apply(z1, act1);
      fs_f2 da = 0ull;
#pragma unroll
      for (int c = 0; c < C; ++c) da = fs_fma2(dzr[c], w2[c], da);
      const fs_f2 d1 = fs_mul2(da, fs_pack2(act_grad_from_output(a0, act1), act_grad_from_output(a1, act1)));
      const fs_f2 a = fs_pack2(a0, a1);
#pragma unroll
      for (int d = 0; d < D; ++d) gw1[d] = fs_fma2(x[d], d1, gw1[d]);
      gb1 = fs_add2(gb1, d1);
#pragma unroll
      for (int c = 0; c < C; ++c) gw2[c] = fs_fma2(a, dzr[c], gw2[c]);
    };
    // rb is even (fs_eval_cluster rounds the row ranges): pairs [rb / 2, re / 2) are whole, an odd re leaves one half pair
    constexpr int PW2 = 2 * (D + C);
    const int j0 = rb >> 1, j_full = re >> 1;
    uint32_t pa = fs_smem_u32(sm.xd) + (uint32_t)((j0 + slice) * PW2 * 4);
    const uint32_t pstep = (uint32_t)(n_slices * PW2 * 4);
    int j = j0 + slice;
#pragma unroll 2
    for (; j < j_full; j += n_slices, pa += pstep) {
      fs_f2 v[D + C];
      fs_lds_pairs<D + C>(pa, v);
      fs_f2 x[D], dzr[C];
#pragma unroll
      for (int d = 0; d < D; ++d) x[d] = v[d];
#pragma unroll
      for (int c = 0; c < C; ++c) dzr[c] = v[D + c];
      step(x, dzr);
    }
    if ((re & 1) && j == j_full) {                   // the odd tail row gets a zero partner: it adds nothing anywhere
      fs_f2 x[D], dzr[C];
#pragma unroll
      for (int d = 0; d < D; ++d) x[d] = fs_pack2(sm.xd[fs_xi<D, C>(re - 1, d)], 0.f);
#pragma unroll
      for (int c = 0; c < C; ++c) dzr[c] = fs_pack2(sm.xd[fs_dzi<D, C>(re - 1, c)], 0.f);
      step(x, dzr);
    }
    auto hsum = [](fs_f2 v) { float x, y; fs_unpack2(v, x, y); return x + y; };
    float* o = sm.part + slice * NG + h * PKW;
#pragma unroll
    for (int d = 0; d < D; ++d) o[d] = hsum(gw1[d]);
    o[D] = hsum(gb1);
#pragma unroll
    for (int c = 0; c < C; ++c) o[D + 1 + c] = hsum(gw2[c]);
  }
  __syncthreads();
  // combine slices in a fixed order and scatter into the flat gradient layout
  for (int i = t; i < NG; i += FS_THREADS) {
    float s = 0.f;
    for (int sl = 0; sl < n_slices; ++sl) s += sm.part[sl * NG + i];
    int hh = i / PKW, k = i - hh * PKW;
    int64_t dst = (k < D) ? p.w1_off + (int64_t)k * H + hh : (k == D ? p.b1_off + hh : p.w2_off + (int64_t)hh * C + (k - D - 1));
    gout[dst] = s;
  }
  // db2[c] = sum_r dZ2[r][c]: one warp per class
  {
    const int wid = t >> 5, lane = t & 31;
    if (wid < C) {
      float s = 0.f;
      for (int r = rb + lane; r < re; r += 32) s += sm.xd[fs_dzi<D, C>(r, wid)];
      s = warp_sum(s);
      if (lane == 0) gout[p.b2_off + wid] = s;
    }
  }
  __syncthreads();
  return loss_tot;
}
// whole dataset in this CTA: mean loss, gradient in sm.gs
template <int D, int C, int ACT>
__device__ float fs_eval(const FsParams& p, const FsSmem& sm, float scale) {
  return (float)(fs_eval_rows<D, C, ACT>(p, sm, scale, 0, p.N, sm.gs) / (double)p.N);
}
// this CTA's share of the rows, then the cluster-wide sum through distributed shared memory.  `n_eval` alternates the
// exchange buffer: a CTA may already write the next evaluation's partials while a slower one still reads these
template <int D, int C, int ACT>
__device__ float fs_eval_cluster(const FsParams& p, const FsSmem& sm, float scale, int rank, int n_ctas, int& n_eval) {
  namespace cg = cooperative_groups;
  cg::cluster_group cl = cg::this_cluster();
  const int t = threadIdx.x;
  const int64_t P = p.P, GX = ((P + 1) & ~(int64_t)1) + 2;
  float* gx = sm.gx + (n_eval & 1) * GX;
  ++n_eval;
  // even boundaries: a row pair of the interleaved array belongs to one CTA
  const int rb = (int)((int64_t)p.N * rank / n_ctas) & ~1;
  const int re = rank + 1 == n_ctas ? p.N : ((int)((int64_t)p.N * (rank + 1) / n_ctas) & ~1);
  const double lsum = fs_eval_rows<D, C, ACT>(p, sm, scale, rb, re, gx);
  if (t == 0) *reinterpret_cast<double*>(gx + GX - 2) = lsum;
  cl.sync();
  for (int64_t i = t; i < P; i += FS_THREADS) {
    float sacc = 0.f;
    for (int rr = 0; rr < n_ctas; ++rr) sacc += cl.map_shared_rank(gx, rr)[i];     // fixed order: identical in every CTA
    sm.gs[i] = sacc;
  }
  double lt = 0.0;
  for (int rr = 0; rr < n_ctas; ++rr) lt += *reinterpret_cast<const double*>(cl.map_shared_rank(gx, rr) + GX - 2);
  __syncthreads();
  return (float)(lt / (double)p.N);
}

template <int D, int C>
__device__ void fs_setup(const FsParams& p, FsSmem& sm, float* base) {
  const int N = p.N;
  const int64_t P = p.P;
  constexpr int PKW = D + 1 + C;
  const int n_slices = FS_THREADS / p.H > 0 ? FS_THREADS / p.H : 1;
  float* cur = base;
  const int np = (N + 1) & ~1;
  sm.red = (double*)cur; cur += 64;
  sm.kc = cur; cur += 4;
  sm.xd = cur; cur += (int64_t)np * (D + C);
  sm.ys = cur; cur += (int64_t)N * (p.loss_kind == PYB_LOSS_SPARSE_CE ? 1 : C);
  sm.qs = cur; cur += P;
  sm.ps = cur; cur += P;
  sm.gs = cur; cur += P;
  cur = (float*)(((uintptr_t)cur + 15) & ~(uintptr_t)15);
  sm.pk = cur; cur += p.H * FsPk<D, C>::S;
  sm.part = cur; cur += n_slices * p.H * PKW;
  cur = (float*)(((uintptr_t)cur + 7) & ~(uintptr_t)7);
  sm.gx = cur; cur += 2 * (((P + 1) & ~(int64_t)1) + 2);
  for (int i = threadIdx.x; i < N * D; i += FS_THREADS) { const int r = i / D, d = i - r * D; sm.xd[fs_xi<D, C>(r, d)] = p.X[i]; }
  if (np > N && threadIdx.x < D + C)                 // the pad row of an odd N: never read as data, kept finite
    sm.xd[(N >> 1) * (2 * (D + C)) + 2 * threadIdx.x + 1] = 0.f;
  if (p.loss_kind == PYB_LOSS_SPARSE_CE) {
    for (int i = threadIdx.x; i < N; i += FS_THREADS) sm.ys[i] = __int_as_float(p.y_i[i]);
  } else {
    for (int i = threadIdx.x; i < N * C; i += FS_THREADS) sm.ys[i] = p.y_f[i];
  }
}

// eval-only: loss + scale * d(mean loss)/d theta  (parity hook, SVGD gradients)
template <int D, int C, int ACT>
__global__ void __launch_bounds__(FS_THREADS, 4) k_fs_eval(FsParams p) {
  extern __shared__ __align__(16) float fs_smem[];
  FsSmem sm;
  fs_setup<D, C>(p, sm, fs_smem);
  const int64_t s = blockIdx.x;
  for (int64_t i = threadIdx.x; i < p.P; i += FS_THREADS) sm.qs[i] = p.theta[s * p.P + i];
  __syncthreads();
  float loss = fs_eval<D, C, ACT>(p, sm, p.scale);
  if (p.grad_out)
    for (int64_t i = threadIdx.x; i < p.P; i += FS_THREADS) p.grad_out[s * p.P + i] = sm.gs[i];
  if (threadIdx.x == 0 && p.loss_out) p.loss_out[s] = loss;
}

// one full HMC iteration of one chain
template <int D, int C, int ACT>
__global__ void __launch_bounds__(FS_THREADS, 4) k_fs_hmc(FsParams p) {
  extern __shared__ __align__(16) float fs_smem[];
  FsSmem sm;
  fs_setup<D, C>(p, sm, fs_smem);
  const int n_ctas = p.cluster;
  const int rank = n_ctas > 1 ? (int)cooperative_groups::this_cluster().block_rank() : 0;
  const int64_t s = blockIdx.x / n_ctas, P = p.P;
  const int t = threadIdx.x;
  const bool writer = rank == 0;          // every CTA of the cluster holds the same state; one writes it back
  // the chain's leapfrog coefficients and inverse temperature (1 without a ladder; beta g rounds to g exactly), kept in
  // shared memory rather than in registers for the whole kernel; the per-chain step size is read here, before the
  // writer's Metropolis tail may update it (adaptation)
  if (t == 0) {
    const StepCoef c = p.step ? step_coef(p.step[s], p.m) : StepCoef{p.eps, p.half_eps, p.drift};
    sm.kc[0] = c.eps; sm.kc[1] = c.half; sm.kc[2] = c.drift;
    sm.kc[3] = p.beta ? p.beta[s] : 1.f;
  }
  int n_eval = 0;
  auto eval = [&]() -> float {
    return n_ctas > 1 ? fs_eval_cluster<D, C, ACT>(p, sm, p.n_train, rank, n_ctas, n_eval) : fs_eval<D, C, ACT>(p, sm, p.n_train);
  };
  // q, momentum (HMC.py:78), K0 (:79)
  double k0 = 0.0;
  for (int64_t i = t; i < P; i += FS_THREADS) sm.qs[i] = p.q[s * P + i];
  if (p.inj_p) {
    for (int64_t i = t; i < P; i += FS_THREADS) sm.ps[i] = p.inj_p[s * P + i];
  } else {
    for (int64_t blk = t; blk * 4 < P; blk += FS_THREADS) {
      float z[4];
      philox_normal4((uint32_t)blk, (uint32_t)(p.chain_offset + s), p.iter, STREAM_MOMENTUM, p.seed, z);
      for (int j = 0; j < 4; ++j)
        if (blk * 4 + j < P) sm.ps[blk * 4 + j] = z[j] * p.stdv;
    }
  }
  __syncthreads();
  for (int64_t i = t; i < P; i += FS_THREADS) k0 += (double)sm.ps[i] * (double)sm.ps[i];
  const float K0 = (float)(fs_block_sum_all<double>(k0, sm.red) * (double)p.inv2m);
  // U0 and the first half kick share the evaluation at q0 (HMC.py:80-82)
  const float loss0 = eval();
  double e0 = 0.0;
  const float half_eps0 = sm.kc[1], drift0 = sm.kc[2], beta0 = sm.kc[3];
  for (int64_t i = t; i < P; i += FS_THREADS) {
    float q = sm.qs[i], d = q - p.mu[i], iv = p.inv_var[i];
    e0 += 0.5 * (double)(d * d * iv);
    if (writer) p.q0[s * P + i] = q;
    float pp = sm.ps[i] - half_eps0 * (__fmul_rn(beta0, sm.gs[i]) + d * iv);
    sm.ps[i] = pp;
    sm.qs[i] = q + drift0 * pp;
  }
  const float Up0 = (float)fs_block_sum_all<double>(e0, sm.red);
  float loss1 = loss0, Up1 = 0.f, K1 = 0.f;
  for (int step = 1; step <= p.L; ++step) {
    loss1 = eval();
    const float eps = sm.kc[0], half_eps = sm.kc[1], drift = sm.kc[2], beta = sm.kc[3];
    if (step < p.L) {
      for (int64_t i = t; i < P; i += FS_THREADS) {
        float q = sm.qs[i], d = q - p.mu[i];
        float pp = sm.ps[i] - eps * (__fmul_rn(beta, sm.gs[i]) + d * p.inv_var[i]);
        sm.ps[i] = pp;
        sm.qs[i] = q + drift * pp;
      }
      __syncthreads();
    } else {
      double e1 = 0.0, k1 = 0.0;
      for (int64_t i = t; i < P; i += FS_THREADS) {
        float q = sm.qs[i], d = q - p.mu[i], iv = p.inv_var[i];
        float gt = __fmul_rn(beta, sm.gs[i]) + d * iv;
        e1 += 0.5 * (double)(d * d * iv);
        float pp = sm.ps[i];
        if (p.semantics == PYB_HMC_REFERENCE) {   // L-th full kick, then the trailing half kick (HMC.py:85-87)
          pp = pp - eps * gt;
          pp = pp - half_eps * gt;
        } else {
          pp = pp - half_eps * gt;
        }
        sm.ps[i] = pp;
        k1 += (double)pp * (double)pp;
      }
      Up1 = (float)fs_block_sum_all<double>(e1, sm.red);
      K1 = (float)(fs_block_sum_all<double>(k1, sm.red) * (double)p.inv2m);
    }
  }
  if (writer)
    for (int64_t i = t; i < P; i += FS_THREADS) {
      p.q[s * P + i] = sm.qs[i];
      p.p[s * P + i] = sm.ps[i];
    }
  if (n_ctas > 1) cooperative_groups::this_cluster().sync();     // nobody leaves while a peer may still read its shared memory
  if (t == 0 && writer) {
    // Metropolis test (HMC.py:91), same expression order as k_accept
    const float tl0 = __fmul_rn(sm.kc[3], loss0), tl1 = __fmul_rn(sm.kc[3], loss1);
    float U0 = (Up0 + p.prior_const) + tl0 * p.n_train;
    float U1 = (Up1 + p.prior_const) + tl1 * p.n_train;
    float la = ((K0 + U0) - K1) - U1;
    float alpha = expf(la);
    float u = p.inj_u ? p.inj_u[s] : philox_uniform((uint32_t)(p.chain_offset + s), p.iter, STREAM_UNIFORM, p.seed);
    int acc = p.burning ? 1 : ((u < alpha) ? 1 : 0);
    p.U0[s] = U0; p.U1[s] = U1; p.K0[s] = K0; p.K1[s] = K1; p.log_alpha[s] = la; p.accepted[s] = acc;
    if (p.da) dual_average(p.da + 4 * s, p.step + s, la, p.da_target, p.da_t);
    float rl = acc ? loss1 : loss0;
    p.ret_loss[s] = rl;
    if (acc) atomicAdd(&p.counters[0], 1ull);
    atomicAdd(&p.counters[1], 1ull);
    if (la != la) atomicAdd(&p.counters[2], 1ull);
    atomicAdd(p.loss_sum, (double)rl);
  }
}

// ------------------------------------------------------------------------------------------
static size_t fs_smem_bytes(const pyb_handle* h) {
  const Model& m = h->model;
  const int D = m.layer[0].fan_in, H = m.layer[0].fan_out, C = m.layer[1].fan_out;
  const int n_slices = FS_THREADS / H > 0 ? FS_THREADS / H : 1;
  const size_t np = ((size_t)h->N + 1) & ~(size_t)1;
  size_t f = 64 + 4 + np * D + (size_t)h->N * (h->loss_kind == PYB_LOSS_SPARSE_CE ? 1 : C) + np * C +
             3 * (size_t)m.P + (size_t)H * (D + 1 + C) * n_slices + (size_t)H * (((D + 1 + C) + 3) / 4 * 4) + 4 + 2 * (((size_t)m.P + 1) / 2 * 2 + 2) + 2;
  return f * sizeof(float) + 16;
}

template <int D, int C, int ACT>
static void fs_launch(pyb_handle* h, const FsParams& p, int64_t S, bool hmc) {
  size_t smem = fs_smem_bytes(h);
  if (hmc) {
    PYB_CUDA(cudaFuncSetAttribute(k_fs_hmc<D, C, ACT>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    if (p.cluster > 1) {
      cudaLaunchConfig_t cfg = {};
      cfg.gridDim = dim3((unsigned)(S * p.cluster)); cfg.blockDim = dim3(FS_THREADS);
      cfg.dynamicSmemBytes = smem; cfg.stream = h->stream;
      cudaLaunchAttribute at[1];
      at[0].id = cudaLaunchAttributeClusterDimension;
      at[0].val.clusterDim.x = (unsigned)p.cluster; at[0].val.clusterDim.y = 1; at[0].val.clusterDim.z = 1;
      cfg.attrs = at; cfg.numAttrs = 1;
      PYB_CUDA(cudaLaunchKernelEx(&cfg, k_fs_hmc<D, C, ACT>, p));
    } else {
      k_fs_hmc<D, C, ACT><<<(unsigned)S, FS_THREADS, smem, h->stream>>>(p);
    }
  } else {
    PYB_CUDA(cudaFuncSetAttribute(k_fs_eval<D, C, ACT>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    k_fs_eval<D, C, ACT><<<(unsigned)S, FS_THREADS, smem, h->stream>>>(p);
  }
  count_launch(h);
}


// one translation unit per input width D (fused_small_d1.cu .. _d4.cu) instantiates the kernels for C = 1..4 and the
// two activation modes, so that the 64 kernels compile in parallel
#define FS_DEFINE_LAUNCH_D(d)                                                                              \
  void fs_launch_d##d(pyb_handle* h, const FsParams& p, int64_t S, bool hmc) {                              \
    const int C = h->model.layer[1].fan_out;                                                               \
    const bool relu = p.act1 == PYB_ACT_RELU;                                                              \
    switch (C) {                                                                                           \
      case 1: relu ? fs_launch<d, 1, PYB_ACT_RELU>(h, p, S, hmc) : fs_launch<d, 1, -1>(h, p, S, hmc); break; \
      case 2: relu ? fs_launch<d, 2, PYB_ACT_RELU>(h, p, S, hmc) : fs_launch<d, 2, -1>(h, p, S, hmc); break; \
      case 3: relu ? fs_launch<d, 3, PYB_ACT_RELU>(h, p, S, hmc) : fs_launch<d, 3, -1>(h, p, S, hmc); break; \
      case 4: relu ? fs_launch<d, 4, PYB_ACT_RELU>(h, p, S, hmc) : fs_launch<d, 4, -1>(h, p, S, hmc); break; \
      default: throw Error(PYB_ERR_UNSUPPORTED, "fused small path: unsupported output width");            \
    }                                                                                                      \
  }
void fs_launch_d1(pyb_handle* h, const FsParams& p, int64_t S, bool hmc);
void fs_launch_d2(pyb_handle* h, const FsParams& p, int64_t S, bool hmc);
void fs_launch_d3(pyb_handle* h, const FsParams& p, int64_t S, bool hmc);
void fs_launch_d4(pyb_handle* h, const FsParams& p, int64_t S, bool hmc);

}  // namespace pyb
