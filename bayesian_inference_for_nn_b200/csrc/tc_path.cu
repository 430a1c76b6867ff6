// tc_path.cu — tensor-core path for the MNIST-width case (BASELINE config C3/C4/C5 shapes):
// two-layer Dense MLP whose first layer is a real dense contraction (D x H with H <= 256).
//
// What runs where, per chain batch (Bc chains), per log-posterior evaluation:
//   k_split_transpose      theta -> W1^T split into bf16 hi/lo, K-major [Bc*H, D]                (SIMT, tiny)
//   tc_g1_layer2_fused     Z1 = X W1 on tcgen05; epilogue: a1 = relu(z1 + b1) -> A1^T hi/lo, logits, softmax-CE / MSE,
//                          loss, dZ2, db2, dZ1 = (dZ2 W2^T) relu' -> dZ1^T hi/lo          (tc_fused.cuh; relu, H = 128/256)
//     or tc_gemm_pair_bf16x3 + k_layer2 for other hidden activations / widths               (tc_gemm.cuh, tc_layer2.cuh)
//   tc_gemm_bf16x3         dW2 = A1^T dZ2 -> grad[:, w2_off : w2_off + H*C]                  (N = 16, HBM-bound)
//   tc_gemm_pair_dual_bf16x3  [dW1; db1] = dZ1^T [X^T; 1]^T -> grad[:, 0 : D*H + H]         (hidden-major, two tiles per item)
// fp32-grade products on bf16 tensor cores: every operand is split x = hi + lo (bf16 each) and the
// MMA issues hi*hi + lo*hi + hi*lo into one fp32 TMEM accumulator (relative error ~2^-16 per
// product, far inside the 1e-4 parity budget; single-pass BF16/TF32 would not be).
//
// This file is the host side: tensor maps, operand preparation, chain batching, kernel selection and launch.
// The kernels live in tc_ptx.cuh (PTX helpers), tc_gemm.cuh, tc_layer2.cuh and tc_fused.cuh.
#include <cstdlib>
#include <cstring>
#include "tc_fused_mma.cuh"
#include <algorithm>

namespace pyb {

// ------------------------------------------------------------------------------------------
// host side
// ------------------------------------------------------------------------------------------
typedef CUresult (*PFN_encodeTiled)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*,
                                    const cuuint64_t*, const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave,
                                    CUtensorMapSwizzle, CUtensorMapL2promotion, CUtensorMapFloatOOBfill);
static PFN_encodeTiled get_encode() {
  static PFN_encodeTiled fn = nullptr;
  if (!fn) {
    void* f = nullptr;
    cudaDriverEntryPointQueryResult q;
    PYB_CUDA(cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &f, cudaEnableDefault, &q));
    PYB_REQUIRE(f != nullptr && q == cudaDriverEntryPointSuccess, PYB_ERR_CUDA, "cuTensorMapEncodeTiled unavailable");
    fn = (PFN_encodeTiled)f;
  }
  return fn;
}
// 2-D bf16 tensor [rows, k] with row pitch ld_elems, box [TC_BK, box_rows], SWIZZLE_64B, zero OOB fill
// row-tile-blocked bf16 tensor [blocks][rows_per_block][128]: box [TC_BK, box_rows, 1], SWIZZLE_64B
static CUtensorMap make_map_blocked(const void* base, int64_t blocks, int rows_per_block, int box_rows) {
  CUtensorMap m;
  cuuint64_t dims[3] = {128, (cuuint64_t)rows_per_block, (cuuint64_t)blocks};
  cuuint64_t strides[2] = {256, (cuuint64_t)rows_per_block * 256};
  cuuint32_t box[3] = {(cuuint32_t)TC_BK, (cuuint32_t)box_rows, 1};
  cuuint32_t es[3] = {1, 1, 1};
  CUresult r = get_encode()(&m, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 3, const_cast<void*>(base), dims, strides, box, es,
                            CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_64B, CU_TENSOR_MAP_L2_PROMOTION_L2_128B,
                            CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  PYB_REQUIRE(r == CUDA_SUCCESS, PYB_ERR_CUDA, "cuTensorMapEncodeTiled (blocked) failed");
  return m;
}
static CUtensorMap make_map(const void* base, int64_t k, int64_t rows, int64_t ld_elems, int box_rows) {
  CUtensorMap m;
  cuuint64_t dims[2] = {(cuuint64_t)k, (cuuint64_t)rows};
  cuuint64_t strides[1] = {(cuuint64_t)ld_elems * 2};
  cuuint32_t box[2] = {(cuuint32_t)TC_BK, (cuuint32_t)box_rows};
  cuuint32_t es[2] = {1, 1};
  PYB_REQUIRE((ld_elems * 2) % 16 == 0, PYB_ERR_INVALID, "tensor map pitch must be a multiple of 16 bytes");
  CUresult r = get_encode()(&m, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 2, const_cast<void*>(base), dims, strides, box, es,
                            CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_64B, CU_TENSOR_MAP_L2_PROMOTION_L2_128B,
                            CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  PYB_REQUIRE(r == CUDA_SUCCESS, PYB_ERR_CUDA, "cuTensorMapEncodeTiled failed");
  return m;
}

// 8-bit tensors (int8 slices): 2-D [rows][kbytes] with box [64, box_rows]; row-tile-blocked 3-D [blocks][rows_per_block][128]
static CUtensorMap make_map_u8p(const void* base, int64_t kbytes, int64_t rows, int64_t pitch, int box_rows) {
  CUtensorMap m;
  cuuint64_t dims[2] = {(cuuint64_t)kbytes, (cuuint64_t)rows};
  cuuint64_t strides[1] = {(cuuint64_t)pitch};
  cuuint32_t box[2] = {64, (cuuint32_t)box_rows};
  cuuint32_t es[2] = {1, 1};
  PYB_REQUIRE(pitch % 16 == 0, PYB_ERR_INVALID, "tensor map pitch must be a multiple of 16 bytes");
  CUresult r = get_encode()(&m, CU_TENSOR_MAP_DATA_TYPE_UINT8, 2, const_cast<void*>(base), dims, strides, box, es,
                            CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_64B, CU_TENSOR_MAP_L2_PROMOTION_L2_128B,
                            CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  PYB_REQUIRE(r == CUDA_SUCCESS, PYB_ERR_CUDA, "cuTensorMapEncodeTiled (8-bit) failed");
  return m;
}
static CUtensorMap make_map_blocked_u8(const void* base, int64_t blocks, int rows_per_block, int box_rows) {
  CUtensorMap m;
  cuuint64_t dims[3] = {128, (cuuint64_t)rows_per_block, (cuuint64_t)blocks};
  cuuint64_t strides[2] = {128, (cuuint64_t)rows_per_block * 128};
  cuuint32_t box[3] = {64, (cuuint32_t)box_rows, 1};
  cuuint32_t es[3] = {1, 1, 1};
  CUresult r = get_encode()(&m, CU_TENSOR_MAP_DATA_TYPE_UINT8, 3, const_cast<void*>(base), dims, strides, box, es,
                            CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_64B, CU_TENSOR_MAP_L2_PROMOTION_L2_128B,
                            CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  PYB_REQUIRE(r == CUDA_SUCCESS, PYB_ERR_CUDA, "cuTensorMapEncodeTiled (8-bit, blocked) failed");
  return m;
}

struct TcData {   // split bf16 operands derived from one [N, D] fp32 matrix resident in HBM
  bool ready = false;
  int64_t N = 0, Npad = 0;
  int D = 0;
  DevBuf<__nv_bfloat16> x_hi, x_lo, xt_hi, xt_lo;       // [N][D], [D+1][Npad]
  DevBuf<__nv_bfloat16> xtq_hi, xtq_lo;                 // [D+1][Npad] with the fused epilogue's row order (fused_row_pos)
  CUtensorMap mX_hi, mX_lo, mXT_hi, mXT_lo, mXTp_hi, mXTp_lo;   // mXTp: half-tile boxes for the hidden-major pair GEMM
  CUtensorMap mXTq_hi, mXTq_lo, mXTqp_hi, mXTqp_lo;     // the same two views of xtq
  // int8 slices (tc_i8.cuh): centred rows [N][Dk] with per-row scales for the forward GEMM, [X^T;1] [D+1][Npad] in the
  // fused row order with per-feature scales for the dW1 GEMM
  int i8 = 0, Dk = 0;                                    // 0: none, 1: forward operand, 2: + backward operand
  DevBuf<int8_t> xs_hi, xs_lo, xts_hi, xts_lo;
  DevBuf<float> sx, col_mean, col_absmax, sf, stat_max;
  DevBuf<double> stat_sum;
  CUtensorMap mXs_hi, mXs_lo, mXTs_hi, mXTs_lo;
};
struct TcState {
  TcData train, aux;                                    // resident training set / minibatch or test inputs
  TcData track;                                         // inputs of the streamed HMC predictive (prepared once per tracking)
  int D = 0, H = 0, C = 0;
  int64_t cap_chains = 0, cap_blocks = 0;               // capacity: chains, and 128-row blocks over all chains
  DevBuf<__nv_bfloat16> w_hi, w_lo;                     // W1^T  [chains*H][D]
  DevBuf<__nv_bfloat16> z_hi, z_lo;                     // dZ1^T blocked [block][H][128]
  DevBuf<__nv_bfloat16> a_hi, a_lo;                     // A1^T  blocked [block][H][128]
  DevBuf<__nv_bfloat16> z2_hi, z2_lo;                   // dZ2^T blocked [block][16][128]
  DevBuf<float> b2_partial;
  DevBuf<float> kpart, gpart;                           // split-K partial sums (gradient GEMMs / exported GEMM)
  DevBuf<double> loss_partial;
  CUtensorMap mW_hi, mW_lo, mWp_hi, mWp_lo, mZ_hi, mZ_lo, mZa_hi, mZa_lo, mA_hi, mA_lo, mZ2_hi, mZ2_lo;
  // int8 slices: W1^T [chains*H][Dk], dZ1^T blocked [block][H][128], per (chain, unit) factors (k_pack_w1_i8)
  int64_t cap_chains_i8 = 0, cap_blocks_i8 = 0;
  DevBuf<unsigned long long> dbg;                        // option "tc_timeline": per-CTA cycle sums of the fused kernel's phases
  DevBuf<int8_t> ws_hi, ws_lo, zi_hi, zi_lo;
  DevBuf<float> cw, b1c, zq, zd;
  CUtensorMap mWs_hi, mWs_lo, mZi_hi, mZi_lo;
};
static TcState* tc_state(pyb_handle* h) {
  if (!h->tc) h->tc = new TcState();
  return (TcState*)h->tc;
}
void tc_release(pyb_handle* h) {
  if (h->tc) delete (TcState*)h->tc;
  h->tc = nullptr;
}
void tc_read_timeline(pyb_handle* h, unsigned long long* out_8x160) {
  if (!h->tc || !((TcState*)h->tc)->dbg.p) { memset(out_8x160, 0, 8 * 160 * 8); return; }
  PYB_CUDA(cudaMemcpy(out_8x160, ((TcState*)h->tc)->dbg.p, 8 * 160 * 8, cudaMemcpyDeviceToHost));
}
int tc_resident_split(const pyb_handle* h) {   // operand split the resident dataset was prepared for: 0 bf16x3, 1 / 2 int8 slices
  return h->tc ? ((TcState*)h->tc)->train.i8 : 0;
}
void tc_invalidate_dataset(pyb_handle* h) {
  if (h->tc) ((TcState*)h->tc)->train.ready = false;
}
void tc_invalidate_track(pyb_handle* h) {
  if (h->tc) ((TcState*)h->tc)->track.ready = false;
}

// shape conditions of the tensor path for a batch of n_rows data rows
bool tc_supported_rows(pyb_handle* h, int64_t n_rows) {
  const Model& m = h->model;
  if (m.n_layers != 2) return false;
  const LayerDesc& L1 = m.layer[0];
  const LayerDesc& L2 = m.layer[1];
  if (!L1.use_bias || !L2.use_bias) return false;
  if (L1.fan_out % 16 != 0 || L1.fan_out < 16 || L1.fan_out > 256) return false;
  if (L1.fan_in % 8 != 0 || L1.fan_in < 64) return false;
  if (L2.fan_out > L2_CMAX) return false;
  if (L1.act == PYB_ACT_SOFTMAX) return false;
  return n_rows >= 128;
}
bool tc_supported(pyb_handle* h, int64_t S) {
  (void)S;
  return h->have_data && tc_supported_rows(h, h->N);
}

template <int EPI, int ACT>
static void launch_gemm_inst(pyb_handle* h, int grid, const CUtensorMap& a_hi, const CUtensorMap& a_lo,
                             const CUtensorMap& b_hi, const CUtensorMap& b_lo, const TcGemmParams& p) {
  // per device and per instantiation; cheap enough to repeat (a process may drive several GPUs)
  PYB_CUDA(cudaFuncSetAttribute(tc_gemm_bf16x3<EPI, ACT>, cudaFuncAttributeMaxDynamicSharedMemorySize, TC_SMEM_BYTES));
  tc_gemm_bf16x3<EPI, ACT><<<grid, TC_THREADS, TC_SMEM_BYTES, h->stream>>>(a_hi, a_lo, b_hi, b_lo, p);
}
template <int EPI, int ACT>
static void launch_pair_inst(pyb_handle* h, int grid, const CUtensorMap& a_hi, const CUtensorMap& a_lo,
                             const CUtensorMap& b_hi, const CUtensorMap& b_lo, const TcGemmParams& p) {
  PYB_CUDA(cudaFuncSetAttribute(tc_gemm_pair_bf16x3<EPI, ACT>, cudaFuncAttributeMaxDynamicSharedMemorySize, TP_SMEM_BYTES));
  tc_gemm_pair_bf16x3<EPI, ACT><<<grid, TP_THREADS, TP_SMEM_BYTES, h->stream>>>(a_hi, a_lo, b_hi, b_lo, p);
}
// CTA-pair kernel: plain 2-D operands, H a multiple of 32, an even number of M tiles' worth of work per item
static bool pair_ok(const pyb_handle* h, const TcGemmParams& p) {
  if (!h->opt_tc_pair || p.b_blocked || p.H < 32 || p.n_mtiles < 2) return false;
  if (p.n_btiles > 0) return p.a_blocked && p.n_mtiles == 2 && (p.H % 16) == 0;   // hidden-major gradient GEMM
  if ((p.H % 32) != 0) return false;
  return !p.a_blocked && p.a_batch_rows == 0;
}
// bp_hi/bp_lo: the SAME B tensors described with half-height TMA boxes (H/2 rows) for the CTA-pair kernel, or null
static void launch_gemm_tc(pyb_handle* h, const CUtensorMap& a_hi, const CUtensorMap& a_lo,
                           const CUtensorMap& b_hi, const CUtensorMap& b_lo, TcGemmParams p, double flops,
                           const CUtensorMap* bp_hi = nullptr, const CUtensorMap* bp_lo = nullptr) {
  if (p.k_splits <= 1) { p.k_splits = 1; p.chunks_per_split = (p.K + TC_BK - 1) / TC_BK; p.split_stride = 0; }
  p.vec_store = p.epi == EPI_STORE && ((uintptr_t)p.out % 16 == 0) && (p.out_stride % 4 == 0) && (p.out_ld % 4 == 0) &&
                (p.split_stride % 4 == 0);
  int grid = std::min(p.total_items, h->sm_count);
  prof_begin(h);
  if (bp_hi && bp_lo && pair_ok(h, p) && p.n_btiles > 1 && p.epi == EPI_STORE && p.transpose_out && h->opt_tc_dual &&
      p.H <= 256 && (p.H / 2) * TC_BK * 2 <= 8192) {
    // hidden-major gradient GEMM: two feature tiles per item share every A stage
    p.total_items = p.n_batch * p.k_splits * ((p.n_btiles + 1) / 2);
    grid = std::min(2 * p.total_items, (h->sm_count / 2) * 2);
    PYB_CUDA(cudaFuncSetAttribute(tc_gemm_pair_dual_bf16x3, cudaFuncAttributeMaxDynamicSharedMemorySize, TD_SMEM_BYTES));
    tc_gemm_pair_dual_bf16x3<<<grid, TP_THREADS, TD_SMEM_BYTES, h->stream>>>(a_hi, a_lo, *bp_hi, *bp_lo, p);
    prof_end(h, flops);
    count_launch(h);
    return;
  }
  if (bp_hi && bp_lo && pair_ok(h, p)) {
    grid = std::min(2 * p.total_items, (h->sm_count / 2) * 2);
    if (p.epi == EPI_STORE) launch_pair_inst<EPI_STORE, 0>(h, grid, a_hi, a_lo, *bp_hi, *bp_lo, p);
    else if (p.act == PYB_ACT_RELU) launch_pair_inst<EPI_BIAS_ACT_T_SPLIT, PYB_ACT_RELU>(h, grid, a_hi, a_lo, *bp_hi, *bp_lo, p);
    else if (p.act == PYB_ACT_TANH) launch_pair_inst<EPI_BIAS_ACT_T_SPLIT, PYB_ACT_TANH>(h, grid, a_hi, a_lo, *bp_hi, *bp_lo, p);
    else if (p.act == PYB_ACT_SIGMOID) launch_pair_inst<EPI_BIAS_ACT_T_SPLIT, PYB_ACT_SIGMOID>(h, grid, a_hi, a_lo, *bp_hi, *bp_lo, p);
    else launch_pair_inst<EPI_BIAS_ACT_T_SPLIT, PYB_ACT_LINEAR>(h, grid, a_hi, a_lo, *bp_hi, *bp_lo, p);
    prof_end(h, flops);
    count_launch(h);
    return;
  }
  if (p.epi == EPI_STORE) launch_gemm_inst<EPI_STORE, 0>(h, grid, a_hi, a_lo, b_hi, b_lo, p);
  else if (p.act == PYB_ACT_RELU) launch_gemm_inst<EPI_BIAS_ACT_T_SPLIT, PYB_ACT_RELU>(h, grid, a_hi, a_lo, b_hi, b_lo, p);
  else if (p.act == PYB_ACT_TANH) launch_gemm_inst<EPI_BIAS_ACT_T_SPLIT, PYB_ACT_TANH>(h, grid, a_hi, a_lo, b_hi, b_lo, p);
  else if (p.act == PYB_ACT_SIGMOID) launch_gemm_inst<EPI_BIAS_ACT_T_SPLIT, PYB_ACT_SIGMOID>(h, grid, a_hi, a_lo, b_hi, b_lo, p);
  else launch_gemm_inst<EPI_BIAS_ACT_T_SPLIT, PYB_ACT_LINEAR>(h, grid, a_hi, a_lo, b_hi, b_lo, p);
  prof_end(h, flops);
  count_launch(h);
}


template <int CP, bool FWD, int I8>
static void launch_fused_i8(pyb_handle* h, int grid, const CUtensorMap& a_hi, const CUtensorMap& a_lo,
                            const CUtensorMap& b_hi, const CUtensorMap& b_lo, const TcGemmParams& p, const Layer2Params& l2) {
  PYB_CUDA(cudaFuncSetAttribute(tc_g1_layer2_fused<CP, FWD, I8>, cudaFuncAttributeMaxDynamicSharedMemorySize, TfCfg<CP>::SMEM_I8));
  tc_g1_layer2_fused<CP, FWD, I8><<<grid, TF_THREADS, TfCfg<CP>::SMEM_I8, h->stream>>>(a_hi, a_lo, b_hi, b_lo, p, l2);
}
template <int CP>
static void launch_fused_inst(pyb_handle* h, int grid, const CUtensorMap& a_hi, const CUtensorMap& a_lo,
                              const CUtensorMap& b_hi, const CUtensorMap& b_lo, const TcGemmParams& p, const Layer2Params& l2,
                              int i8 = 0) {
  if (i8 && !l2.fwd_out && h->opt_tc_epi_mma) {
    // layer-2 products of the epilogue on mma.sync (tc_fused_mma.cuh)
    if (i8 >= 2) {
      PYB_CUDA(cudaFuncSetAttribute(tc_fused_i8_mma<CP, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, TfmCfg::SMEM));
      tc_fused_i8_mma<CP, true><<<grid, TFM_THREADS, TfmCfg::SMEM, h->stream>>>(a_hi, a_lo, b_hi, b_lo, p, l2);
    } else {
      PYB_CUDA(cudaFuncSetAttribute(tc_fused_i8_mma<CP, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, TfmCfg::SMEM));
      tc_fused_i8_mma<CP, false><<<grid, TFM_THREADS, TfmCfg::SMEM, h->stream>>>(a_hi, a_lo, b_hi, b_lo, p, l2);
    }
    return;
  }
  if (i8) {
    if (l2.fwd_out) launch_fused_i8<CP, true, 1>(h, grid, a_hi, a_lo, b_hi, b_lo, p, l2);
    else if (i8 >= 2) launch_fused_i8<CP, false, 2>(h, grid, a_hi, a_lo, b_hi, b_lo, p, l2);
    else launch_fused_i8<CP, false, 1>(h, grid, a_hi, a_lo, b_hi, b_lo, p, l2);
    return;
  }
  if (l2.fwd_out) {
    PYB_CUDA(cudaFuncSetAttribute(tc_g1_layer2_fused<CP, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, TfCfg<CP>::SMEM));
    tc_g1_layer2_fused<CP, true><<<grid, TF_THREADS, TfCfg<CP>::SMEM, h->stream>>>(a_hi, a_lo, b_hi, b_lo, p, l2);
    return;
  }
  PYB_CUDA(cudaFuncSetAttribute(tc_g1_layer2_fused<CP, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, TfCfg<CP>::SMEM));
  tc_g1_layer2_fused<CP, false><<<grid, TF_THREADS, TfCfg<CP>::SMEM, h->stream>>>(a_hi, a_lo, b_hi, b_lo, p, l2);
}
// fused G1 + layer 2 applies to: relu hidden layer of 128 or 256 units, CTA pairs enabled
static bool fused_ok(const pyb_handle* h, int H, int act1) {
  return h->opt_tc_pair && h->opt_tc_fuse && act1 == PYB_ACT_RELU && (H == 128 || H == 256);
}

// int8-slice mode of an evaluation: 0 bf16x3, 1 forward GEMM on slices, 2 forward and dW1 GEMMs on slices.
// The dW1 operand dZ1 needs an a-priori bound of its magnitude, which exists for the softmax cross-entropy only, and the
// kernel takes one 256-unit chain per CTA pair.
// Option tc_i8 = -1 (default): the slices are used where the 1e-4 parity budget is what the caller is held to — the
// full-data log-posterior gradient of HMC on the RESIDENT dataset (`resident`); minibatch gradients (SVGD / SGLD / SWAG
// feed them to Adam or a Langevin step, whose first steps are sign-like in the gradient) and the predictive stay on
// bf16x3.  0 / 1 / 2 force a mode everywhere it applies.
static int i8_mode(const pyb_handle* h, bool backward, bool resident) {
  const Model& m = h->model;
  int want = h->opt_tc_i8;
  if (want < 0) want = (resident && backward && h->i8_guard_ok) ? 2 : 0;
  if (want <= 0 || !fused_ok(h, m.layer[0].fan_out, m.layer[0].act) || m.layer[1].fan_out > L2_CMAX) return 0;
  if (m.layer[0].fan_in > 32768) return 0;                       // int32 range of the hi*lo + lo*hi accumulator
  if (!backward) return 1;
  const bool ce = h->loss_kind == PYB_LOSS_SPARSE_CE && m.layer[1].act == PYB_ACT_SOFTMAX;
  return (want >= 2 && ce && m.layer[0].fan_out == 256) ? 2 : 1;
}

static void tc_prepare_data_i8(pyb_handle* h, TcData& d, const float* X, int64_t N, int mode) {
  const int D = d.D;
  const int64_t Npad = d.Npad;
  d.Dk = (D + 15) / 16 * 16;
  d.col_mean.alloc(D); d.col_absmax.alloc(D); d.sx.alloc(N); d.sf.alloc(D + 1);
  d.xs_hi.alloc(N * d.Dk); d.xs_lo.alloc(N * d.Dk);
  d.stat_sum.alloc((size_t)I8_STAT_CHUNKS * D); d.stat_max.alloc((size_t)I8_STAT_CHUNKS * D);
  k_col_stats<<<dim3((D + 31) / 32, I8_STAT_CHUNKS), dim3(32, 32), 0, h->stream>>>(X, N, D, d.stat_sum.p, d.stat_max.p);
  k_col_stats_final<<<(D + 255) / 256, 256, 0, h->stream>>>(d.stat_sum.p, d.stat_max.p, I8_STAT_CHUNKS, N, D, d.col_mean.p,
                                                           d.col_absmax.p);
  count_launch(h);
  const int wpb = 8;
  k_slice_x_rows_i8<<<(unsigned)std::min<int64_t>((N + wpb - 1) / wpb, 8 * (int64_t)h->sm_count), wpb * 32, 0, h->stream>>>(
      X, N, D, d.col_mean.p, d.xs_hi.p, d.xs_lo.p, d.sx.p, d.Dk);
  count_launch(h, 2);
  d.mXs_hi = make_map_u8p(d.xs_hi.p, d.Dk, N, d.Dk, 128);
  d.mXs_lo = make_map_u8p(d.xs_lo.p, d.Dk, N, d.Dk, 128);
  if (mode >= 2) {
    d.xts_hi.alloc((int64_t)(D + 1) * Npad); d.xts_lo.alloc((int64_t)(D + 1) * Npad);
    PYB_CUDA(cudaMemsetAsync(d.xts_hi.p, 0, (size_t)(D + 1) * Npad, h->stream));
    PYB_CUDA(cudaMemsetAsync(d.xts_lo.p, 0, (size_t)(D + 1) * Npad, h->stream));
    dim3 g2((D + 31) / 32, (unsigned)((N + 31) / 32), 1), blk(32, 8);
    k_slice_xt_i8<<<g2, blk, 0, h->stream>>>(X, N, D, d.col_absmax.p, d.xts_hi.p, d.xts_lo.p, Npad);
    k_xt_i8_tail<<<(unsigned)((std::max<int64_t>(N, D + 1) + 255) / 256), 256, 0, h->stream>>>(
        d.xts_hi.p + (int64_t)D * Npad, N, d.col_absmax.p, d.sf.p, D);
    count_launch(h, 2);
    const int n_t = (D + 1 + 255) / 256, Ht = (((D + 1 + n_t - 1) / n_t) + 15) / 16 * 16;
    d.mXTs_hi = make_map_u8p(d.xts_hi.p, Npad, D + 1, Npad, Ht / 2);
    d.mXTs_lo = make_map_u8p(d.xts_lo.p, Npad, D + 1, Npad, Ht / 2);
  }
  d.i8 = mode;
}

static void tc_prepare_data(pyb_handle* h, TcData& d, const float* X, int64_t N, bool need_xt, bool resident = false) {
  const Model& m = h->model;
  const int D = m.layer[0].fan_in;
  d.N = N; d.D = D;
  d.Npad = ((N + L2_ROWS - 1) / L2_ROWS) * L2_ROWS;
  const int64_t Npad = d.Npad;
  d.x_hi.alloc(N * D); d.x_lo.alloc(N * D);
  k_split_rows<<<(unsigned)std::min<int64_t>((N * D + 255) / 256, 65535), 256, 0, h->stream>>>(X, N, D, D, d.x_hi.p, d.x_lo.p, D);
  count_launch(h);
  d.mX_hi = make_map(d.x_hi.p, D, N, D, 128);
  d.mX_lo = make_map(d.x_lo.p, D, N, D, 128);
  if (need_xt) {
    d.xt_hi.alloc((int64_t)(D + 1) * Npad); d.xt_lo.alloc((int64_t)(D + 1) * Npad);
    PYB_CUDA(cudaMemsetAsync(d.xt_hi.p, 0, (size_t)(D + 1) * Npad * 2, h->stream));
    PYB_CUDA(cudaMemsetAsync(d.xt_lo.p, 0, (size_t)(D + 1) * Npad * 2, h->stream));
    dim3 g2((D + 31) / 32, (unsigned)((N + 31) / 32), 1), blk(32, 8);
    k_split_transpose<<<g2, blk, 0, h->stream>>>(X, 0, (int)N, D, D, d.xt_hi.p, d.xt_lo.p, 0, Npad);
    k_fill_bf16<<<(unsigned)((N + 255) / 256), 256, 0, h->stream>>>(d.xt_hi.p + (int64_t)D * Npad, N, 1.0f);  // ones row -> db1
    count_launch(h, 2);
    d.mXT_hi = make_map(d.xt_hi.p, Npad, D + 1, Npad, 128);
    d.mXT_lo = make_map(d.xt_lo.p, Npad, D + 1, Npad, 128);
    const int n_t = (D + 1 + 255) / 256, Ht = (((D + 1 + n_t - 1) / n_t) + 15) / 16 * 16;
    d.mXTp_hi = make_map(d.xt_hi.p, Npad, D + 1, Npad, Ht / 2);
    d.mXTp_lo = make_map(d.xt_lo.p, Npad, D + 1, Npad, Ht / 2);
    if (fused_ok(h, m.layer[0].fan_out, m.layer[0].act)) {
      d.xtq_hi.alloc((int64_t)(D + 1) * Npad); d.xtq_lo.alloc((int64_t)(D + 1) * Npad);
      PYB_CUDA(cudaMemsetAsync(d.xtq_hi.p, 0, (size_t)(D + 1) * Npad * 2, h->stream));
      PYB_CUDA(cudaMemsetAsync(d.xtq_lo.p, 0, (size_t)(D + 1) * Npad * 2, h->stream));
      k_split_transpose<<<g2, blk, 0, h->stream>>>(X, 0, (int)N, D, D, d.xtq_hi.p, d.xtq_lo.p, 0, Npad, 1);
      k_fill_ones_perm<<<(unsigned)((N + 255) / 256), 256, 0, h->stream>>>(d.xtq_hi.p + (int64_t)D * Npad, (int)N);
      count_launch(h, 2);
      d.mXTq_hi = make_map(d.xtq_hi.p, Npad, D + 1, Npad, 128);
      d.mXTq_lo = make_map(d.xtq_lo.p, Npad, D + 1, Npad, 128);
      d.mXTqp_hi = make_map(d.xtq_hi.p, Npad, D + 1, Npad, Ht / 2);
      d.mXTqp_lo = make_map(d.xtq_lo.p, Npad, D + 1, Npad, Ht / 2);
    }
  }
  d.i8 = 0;
  const int mode = i8_mode(h, need_xt, resident);
  if (mode) tc_prepare_data_i8(h, d, X, N, mode);
  d.ready = true;
}

// chain batch for S chains over Npad rows; grows the shared buffers (and their tensor maps) on demand
static int64_t tc_prepare_bufs(pyb_handle* h, TcState* st, int64_t S, int64_t Npad, bool backward, int mode) {
  const Model& m = h->model;
  st->D = m.layer[0].fan_in; st->H = m.layer[0].fan_out; st->C = m.layer[1].fan_out;
  const int H = st->H, D = st->D;
  const int64_t k_tiles = Npad / 128;
  // intermediates: A1^T hi/lo (+ dZ1^T hi/lo) = 4 (+4) bytes per (chain, hidden, row)
  int64_t per_chain = (int64_t)H * Npad * (backward ? 8 : 4) + (int64_t)H * D * 4;
  int64_t budget = (int64_t)(std::max(h->opt_workspace_mb, 20000.0) * 1024.0 * 1024.0);
  int64_t bc = std::max<int64_t>(1, budget / per_chain);
  if (h->opt_chain_batch > 0) bc = std::min<int64_t>(bc, h->opt_chain_batch);
  bc = std::min<int64_t>(bc, S);
  if (bc >= h->sm_count) bc = (bc / h->sm_count) * h->sm_count;      // whole waves of per-chain GEMM work
  bc = std::min<int64_t>(bc, 16384);
  const int64_t need_blocks = bc * k_tiles;
  if (bc > st->cap_chains || need_blocks > st->cap_blocks) {
    PYB_CUDA(cudaStreamSynchronize(h->stream));
    st->cap_chains = std::max(st->cap_chains, bc);
    st->cap_blocks = std::max(st->cap_blocks, need_blocks);
    const int64_t cb = st->cap_blocks, cc = st->cap_chains;
    st->w_hi.alloc(cc * H * D); st->w_lo.alloc(cc * H * D);
    st->a_hi.alloc(cb * H * 128); st->a_lo.alloc(cb * H * 128);
    st->z_hi.alloc(cb * H * 128); st->z_lo.alloc(cb * H * 128);
    st->z2_hi.alloc(cb * L2_CMAX * 128); st->z2_lo.alloc(cb * L2_CMAX * 128);
    // every block a kernel reads is fully rewritten by the producer kernels of the same evaluation
    // (G1 zero-fills rows >= N, k_layer2 writes whole 256-row tiles), so no clearing is needed
    st->mW_hi = make_map(st->w_hi.p, D, cc * H, D, H);
    st->mW_lo = make_map(st->w_lo.p, D, cc * H, D, H);
    st->mWp_hi = make_map(st->w_hi.p, D, cc * H, D, std::max(H / 2, 8));
    st->mWp_lo = make_map(st->w_lo.p, D, cc * H, D, std::max(H / 2, 8));
    st->mZ_hi = make_map_blocked(st->z_hi.p, cb, H, H);
    st->mZ_lo = make_map_blocked(st->z_lo.p, cb, H, H);
    st->mZa_hi = make_map_blocked(st->z_hi.p, cb, H, std::min(H, 128));   // dZ1^T as an A operand (128-row boxes)
    st->mZa_lo = make_map_blocked(st->z_lo.p, cb, H, std::min(H, 128));
    st->mA_hi = make_map_blocked(st->a_hi.p, cb, H, std::min(H, 128));
    st->mA_lo = make_map_blocked(st->a_lo.p, cb, H, std::min(H, 128));
    st->mZ2_hi = make_map_blocked(st->z2_hi.p, cb, L2_CMAX, L2_CMAX);
    st->mZ2_lo = make_map_blocked(st->z2_lo.p, cb, L2_CMAX, L2_CMAX);
  }
  if (mode && (bc > st->cap_chains_i8 || (mode >= 2 && need_blocks > st->cap_blocks_i8))) {
    PYB_CUDA(cudaStreamSynchronize(h->stream));
    st->cap_chains_i8 = std::max(st->cap_chains_i8, bc);
    const int64_t cc = st->cap_chains_i8, Dk = (D + 15) / 16 * 16;
    st->ws_hi.alloc(cc * H * Dk); st->ws_lo.alloc(cc * H * Dk);
    st->cw.alloc(cc * H); st->b1c.alloc(cc * H); st->zq.alloc(cc * H); st->zd.alloc(cc * H);
    st->mWs_hi = make_map_u8p(st->ws_hi.p, Dk, cc * H, Dk, H / 2);
    st->mWs_lo = make_map_u8p(st->ws_lo.p, Dk, cc * H, Dk, H / 2);
    if (mode >= 2) {
      st->cap_blocks_i8 = std::max(st->cap_blocks_i8, need_blocks);
      const int64_t cb = st->cap_blocks_i8;
      st->zi_hi.alloc(cb * H * 128); st->zi_lo.alloc(cb * H * 128);
      st->mZi_hi = make_map_blocked_u8(st->zi_hi.p, cb, H, 128);
      st->mZi_lo = make_map_blocked_u8(st->zi_lo.p, cb, H, 128);
    }
  }
  return bc;
}

static void tc_pack_and_g1(pyb_handle* h, TcState* st, TcData& d, const float* th, int nb,
                           const Layer2Params* fused = nullptr, int i8 = 0) {
  const Model& m = h->model;
  const LayerDesc& L1 = m.layer[0];
  const int D = st->D, H = st->H;
  const int64_t N = d.N, Npad = d.Npad, P = m.P;
  if (i8) {
    // W1 [D,H] per chain -> W1^T int8 slices [H, Dk] + the per (chain, unit) factors of the scheme
    const float invN = fused->fwd_out ? 1.0f : fused->scale / (float)fused->N;
    k_pack_w1_i8<<<dim3((H + 31) / 32, nb), dim3(32, 8), 0, h->stream>>>(
        th, P, L1.w_off, L1.b_off, m.layer[1].w_off, D, H, m.layer[1].fan_out, d.col_mean.p, invN, st->ws_hi.p, st->ws_lo.p,
        d.Dk, st->cw.p, st->b1c.p, st->zq.p, st->zd.p);
  } else {
  // W1 [D,H] per chain -> W1^T hi/lo [H, D]
  dim3 g((H + 31) / 32, (D + 31) / 32, nb), blk(32, 8);
  k_split_transpose<<<g, blk, 0, h->stream>>>(th + L1.w_off, P, D, H, H, st->w_hi.p, st->w_lo.p, (int64_t)H * D, D);
  }
  count_launch(h);
  // G1: A1^T = act(X W1 + b1)^T, split bf16 (all Npad/128 row tiles: rows >= N are written as zeros)
  TcGemmParams p = {};
  p.K = D; p.n_mtiles = (int)(Npad / 128); p.n_pairs = (p.n_mtiles + 1) / 2; p.n_batch = nb; p.H = H;
  p.a_batch_rows = 0; p.a_box_rows = 128; p.order = 1; p.sub_batch = 32; p.total_items = p.n_pairs * nb;
  p.epi = EPI_BIAS_ACT_T_SPLIT;
  p.bias = th + L1.b_off; p.bias_stride = P; p.act = L1.act;
  p.out_hi = st->a_hi.p; p.out_lo = st->a_lo.p; p.out_tiles = (int)(Npad / 128);
  p.M_valid = (int)N; p.N_valid = H;
  if (fused) {
    // G1 with layer 2 (+ loss, dZ2, dZ1) in its epilogue
    const int grid = std::min(2 * p.total_items, (h->sm_count / 2) * 2);
    const int C = fused->C;
    Layer2Params f2 = *fused;
    const CUtensorMap &a_hi = i8 ? d.mXs_hi : d.mX_hi, &a_lo = i8 ? d.mXs_lo : d.mX_lo;
    const CUtensorMap &b_hi = i8 ? st->mWs_hi : st->mWp_hi, &b_lo = i8 ? st->mWs_lo : st->mWp_lo;
    if (i8) {
      p.bias = st->b1c.p; p.bias_stride = H;                      // b1 + mu^T W1: the slices hold the centred data
      f2.dbg = nullptr; f2.dbg_flags = h->opt_tc_timeline & ~1;
      if (h->opt_tc_timeline) { st->dbg.alloc(8 * 160); f2.dbg = st->dbg.p; }
      f2.sx = d.sx.p; f2.cw = st->cw.p; f2.zq = st->zq.p; f2.zi_hi = st->zi_hi.p; f2.zi_lo = st->zi_lo.p;
    }
    prof_begin(h);
    if (C <= 4) launch_fused_inst<4>(h, grid, a_hi, a_lo, b_hi, b_lo, p, f2, i8);
    else if (C <= 8) launch_fused_inst<8>(h, grid, a_hi, a_lo, b_hi, b_lo, p, f2, i8);
    else if (C <= 12) launch_fused_inst<12>(h, grid, a_hi, a_lo, b_hi, b_lo, p, f2, i8);
    else launch_fused_inst<16>(h, grid, a_hi, a_lo, b_hi, b_lo, p, f2, i8);
    prof_end(h, 2.0 * N * (D * (double)H + (fused->fwd_out ? 1.0 : 3.0) * H * C) * nb);
    count_launch(h);
    return;
  }
  launch_gemm_tc(h, d.mX_hi, d.mX_lo, st->mW_hi, st->mW_lo, p, 2.0 * N * D * (double)H * nb, &st->mWp_hi, &st->mWp_lo);
}

static void tc_eval_on(pyb_handle* h, TcState* st, TcData& d, const int32_t* y_i, const float* y_f, const float* theta,
                       int64_t S, float scale, float* loss_out, float* grad_out) {
  const Model& m = h->model;
  const int64_t Bc = tc_prepare_bufs(h, st, S, d.Npad, true, d.i8);
  const LayerDesc& L1 = m.layer[0];
  const LayerDesc& L2 = m.layer[1];
  const int D = st->D, H = st->H, C = st->C;
  const int64_t N = d.N, Npad = d.Npad, P = m.P;
  const int n_tiles = (int)(Npad / L2_ROWS);
  const bool fused = fused_ok(h, H, L1.act) && C <= L2_CMAX;
  const int i8 = d.i8;
  // fused: one partial per (128-row tile, lane quadrant); unfused: one per k_layer2 block
  const int n_groups = fused ? (int)(Npad / 128) * 4
                             : std::min(n_tiles, std::max(1, (int)((8 * (int64_t)h->sm_count + Bc - 1) / Bc)));
  st->b2_partial.alloc((size_t)Bc * n_groups * L2_CMAX);
  st->loss_partial.alloc((size_t)Bc * n_groups);
  for (int64_t b0 = 0; b0 < S; b0 += Bc) {
    const int nb = (int)std::min<int64_t>(Bc, S - b0);
    const float* th = theta + b0 * P;
    float* gr = grad_out + b0 * P;
    // layer 2 + loss + dZ1^T, dZ2^T: inside G1's epilogue when the shape allows, else a separate pass over A1^T
    {
      Layer2Params p = {};
      p.a_hi = st->a_hi.p; p.a_lo = st->a_lo.p; p.zt_hi = st->z_hi.p; p.zt_lo = st->z_lo.p;
      p.z2_hi = st->z2_hi.p; p.z2_lo = st->z2_lo.p; p.k_tiles = (int)(Npad / 128);
      p.theta = th; p.P = P; p.w2_off = L2.w_off; p.b2_off = L2.b_off;
      p.H = H; p.C = C; p.N = (int)N; p.act1 = L1.act; p.out_act = L2.act; p.loss_kind = h->loss_kind;
      p.y_i = y_i; p.y_f = y_f; p.scale = scale;
      p.loss_partial = st->loss_partial.p; p.b2_partial = st->b2_partial.p; p.n_groups = n_groups;
      p.n_tiles = n_tiles;
      if (fused) {
        tc_pack_and_g1(h, st, d, th, nb, &p, i8);
      } else {
        tc_pack_and_g1(h, st, d, th, nb);
        dim3 g(n_groups, nb);
        if (C <= 4) k_layer2<4><<<g, 128, 0, h->stream>>>(p);
        else if (C <= 8) k_layer2<8><<<g, 128, 0, h->stream>>>(p);
        else if (C <= 12) k_layer2<12><<<g, 128, 0, h->stream>>>(p);
        else k_layer2<16><<<g, 128, 0, h->stream>>>(p);
      }
      k_layer2_reduce<<<nb, 256, 0, h->stream>>>(st->b2_partial.p, st->loss_partial.p, n_groups, C, gr, P, L2.b_off,
                                                loss_out ? loss_out + b0 : nullptr, (int)N);
      count_launch(h, 2);
    }
    // the two reductions over the data rows are split-K (accumulator truncation, see TcGemmParams)
    const int nk_rows = (int)(Npad / TC_BK);
    const int splits = (nk_rows + TC_SPLIT_CHUNKS - 1) / TC_SPLIT_CHUNKS;
    const int64_t cnt1 = (int64_t)(D + 1) * H, cnt2 = (int64_t)H * C;
    if (splits > 1 || i8 >= 2) st->kpart.alloc((size_t)(splits + 1) * nb * std::max(cnt1, cnt2));
    // G3: dW2[h][c] = sum_r a1[r][h] dZ2[r][c]   (A = A1^T per chain, B = dZ2^T per chain, N = 16)
    {
      TcGemmParams p = {};
      p.K = (int)Npad; p.n_mtiles = (H + 127) / 128; p.n_pairs = (p.n_mtiles + 1) / 2; p.n_batch = nb; p.H = L2_CMAX;
      p.a_blocked = 1; p.b_blocked = 1; p.k_tiles = (int)(Npad / 128); p.a_box_rows = std::min(H, 128);
      p.a_batch_rows = H; p.order = 0; p.sub_batch = nb;
      p.epi = EPI_STORE; p.out_ld = C; p.M_valid = H; p.N_valid = C;
      if (splits > 1) {
        p.k_splits = splits; p.chunks_per_split = TC_SPLIT_CHUNKS; p.split_stride = nb * cnt2;
        p.out = st->kpart.p; p.out_stride = cnt2;
      } else {
        p.out = gr + L2.w_off; p.out_stride = P;
      }
      p.total_items = p.n_pairs * nb * std::max(splits, 1);
      launch_gemm_tc(h, st->mA_hi, st->mA_lo, st->mZ2_hi, st->mZ2_lo, p, 2.0 * N * (double)H * C * nb);
      if (splits > 1) {
        dim3 rg((unsigned)std::min<int64_t>((cnt2 + 255) / 256, 64), nb);
        k_reduce_ksplits<<<rg, 256, 0, h->stream>>>(st->kpart.p, splits, nb * cnt2, cnt2, cnt2, gr + L2.w_off, P);
        count_launch(h);
      }
    }
    // G2: [dW1; db1] = [X^T; 1] dZ1
    // two 128-unit chains per CTA pair: only the dual kernel knows that mode, and it needs at least two feature tiles
    const bool chain_pairs = H == 128 && h->opt_tc_dual && h->opt_tc_h128_pairs && (D + 1 + 255) / 256 > 1;
    int splits_red = splits;                                      // partial sums the reduction below has to add up
    if (i8 >= 2) {
      // hidden-major on int8 slices: one feature tile per item, exact int32 accumulation (tc_i8.cuh)
      const int n_t = (D + 1 + 255) / 256;
      const int Ht = (((D + 1 + n_t - 1) / n_t) + 15) / 16 * 16;
      const int nk64 = (int)(Npad / 64), cps = TC_SPLIT_CHUNKS / 2;   // 128 stages of 64 rows = the same 8192-row segments
      const int sp = (nk64 + cps - 1) / cps;
      splits_red = sp;
      TcGemmParams p = {};
      p.K = (int)Npad; p.n_mtiles = 2; p.n_pairs = 1; p.n_batch = nb; p.H = Ht; p.n_chains = nb;
      p.a_blocked = 1; p.k_tiles = (int)(Npad / 128); p.a_box_rows = 128;
      p.n_btiles = n_t; p.b_row0 = 0; p.transpose_out = 1; p.n_cols_total = D + 1;
      p.epi = EPI_STORE; p.out_ld = H; p.M_valid = H; p.N_valid = Ht;
      p.k_splits = sp; p.chunks_per_split = cps;
      if (sp > 1) {
        p.split_stride = nb * cnt1; p.out = st->kpart.p; p.out_stride = cnt1;
      } else {
        p.split_stride = 0; p.out = gr; p.out_stride = P;
      }
      p.total_items = nb * sp * n_t;
      const int grid = std::min(2 * p.total_items, (h->sm_count / 2) * 2);
      prof_begin(h);
      PYB_CUDA(cudaFuncSetAttribute(tc_gemm_pair_dw1_i8, cudaFuncAttributeMaxDynamicSharedMemorySize, TI_SMEM_BYTES));
      tc_gemm_pair_dw1_i8<<<grid, TP_THREADS, TI_SMEM_BYTES, h->stream>>>(st->mZi_hi, st->mZi_lo, d.mXTs_hi, d.mXTs_lo, p,
                                                                         st->zd.p, d.sf.p);
      prof_end(h, 2.0 * N * (double)(D + 1) * H * nb);
      count_launch(h);
    } else if ((H == 256 || chain_pairs) && h->opt_tc_pair) {
      // hidden-major on the CTA-pair kernel: D[h, f] = sum_r dZ1^T[h, r] [X^T;1][f, r].  M = 256 hidden units is
      // exactly one CTA pair (no M padding), the D+1 feature rows are the N dimension in tiles of 256 plus one
      // narrow remainder tile, the accumulators are double-buffered so the partial-sum stores overlap the MMAs
      // (N = D+1 = 785 -> 4 tiles of 208 columns: 6 % padding instead of the 12.5 % of 7 x 128 M tiles)
      const int n_t = (D + 1 + 255) / 256;
      const int Ht = (((D + 1 + n_t - 1) / n_t) + 15) / 16 * 16;
      TcGemmParams p = {};
      p.K = (int)Npad; p.n_mtiles = 2; p.n_pairs = 1; p.n_batch = chain_pairs ? (nb + 1) / 2 : nb; p.H = Ht;
      p.chain_pairs = chain_pairs ? 1 : 0; p.n_chains = nb;
      p.a_blocked = 1; p.b_blocked = 0; p.k_tiles = (int)(Npad / 128); p.a_box_rows = 128;
      p.n_btiles = n_t; p.b_row0 = 0; p.transpose_out = 1; p.n_cols_total = D + 1;
      p.epi = EPI_STORE; p.out_ld = H; p.M_valid = H; p.N_valid = Ht;
      if (splits > 1) {
        p.k_splits = splits; p.chunks_per_split = TC_SPLIT_CHUNKS; p.split_stride = nb * cnt1;
        p.out = st->kpart.p; p.out_stride = cnt1;
      } else {
        p.out = gr; p.out_stride = P;
      }
      p.total_items = p.n_batch * std::max(splits, 1) * n_t;
      launch_gemm_tc(h, st->mZa_hi, st->mZa_lo, fused ? d.mXTq_hi : d.mXT_hi, fused ? d.mXTq_lo : d.mXT_lo, p,
                     2.0 * N * (double)(D + 1) * H * nb, fused ? &d.mXTqp_hi : &d.mXTp_hi, fused ? &d.mXTqp_lo : &d.mXTp_lo);
    } else {
      TcGemmParams p = {};
      p.K = (int)Npad; p.n_mtiles = (D + 1 + 127) / 128; p.n_pairs = (p.n_mtiles + 1) / 2; p.n_batch = nb; p.H = H;
      p.a_blocked = 0; p.b_blocked = 1; p.k_tiles = (int)(Npad / 128); p.a_box_rows = 128;
      p.a_batch_rows = 0; p.order = 0; p.sub_batch = nb;
      p.epi = EPI_STORE; p.out_ld = H; p.M_valid = D + 1; p.N_valid = H;
      if (splits > 1) {
        p.k_splits = splits; p.chunks_per_split = TC_SPLIT_CHUNKS; p.split_stride = nb * cnt1;
        p.out = st->kpart.p; p.out_stride = cnt1;
      } else {
        p.out = gr; p.out_stride = P;
      }
      p.total_items = p.n_pairs * nb * std::max(splits, 1);
      launch_gemm_tc(h, fused ? d.mXTq_hi : d.mXT_hi, fused ? d.mXTq_lo : d.mXT_lo, st->mZ_hi, st->mZ_lo, p,
                     2.0 * N * (double)(D + 1) * H * nb);
    }
    if (splits_red > 1) {
      dim3 rg((unsigned)std::min<int64_t>((cnt1 + 255) / 256, 256), nb);
      k_reduce_ksplits<<<rg, 256, 0, h->stream>>>(st->kpart.p, splits_red, nb * cnt1, cnt1, cnt1, gr, P);
      count_launch(h);
    }
  }
  PYB_CUDA(cudaGetLastError());
}

void tc_eval(pyb_handle* h, const float* theta, int64_t S, float scale, float* loss_out, float* grad_out) {
  TcState* st = tc_state(h);
  if (!st->train.ready || st->train.i8 != i8_mode(h, true, true)) tc_prepare_data(h, st->train, h->X.p, h->N, true, true);
  tc_eval_on(h, st, st->train, h->y_i.p, h->y_f.p, theta, S, scale, loss_out, grad_out);
}

// loss + gradient on an arbitrary device-resident batch (SVGD minibatches): operands are re-derived per call
void tc_eval_batch(pyb_handle* h, const float* Xb, const int32_t* yb_i, const float* yb_f, int64_t Nb, const float* theta,
                   int64_t S, float scale, float* loss_out, float* grad_out) {
  TcState* st = tc_state(h);
  tc_prepare_data(h, st->aux, Xb, Nb, true);
  tc_eval_on(h, st, st->aux, yb_i, yb_f, theta, S, scale, loss_out, grad_out);
}

static void tc_forward_on(pyb_handle* h, TcState* st, TcData& d, const float* theta, int64_t S, int64_t N, float* out) {
  const Model& m = h->model;
  const int64_t Bc = tc_prepare_bufs(h, st, S, d.Npad, false, d.i8);
  const LayerDesc& L2 = m.layer[1];
  const int64_t P = m.P;
  const bool fused = fused_ok(h, st->H, m.layer[0].act) && st->C <= L2_CMAX;
  for (int64_t b0 = 0; b0 < S; b0 += Bc) {
    const int nb = (int)std::min<int64_t>(Bc, S - b0);
    const float* th = theta + b0 * P;
    if (fused) {
      // layer 2 and the output activation inside the layer-1 GEMM's epilogue: A1 never leaves the SM
      Layer2Params f = {};
      f.theta = th; f.P = P; f.w2_off = L2.w_off; f.b2_off = L2.b_off;
      f.H = st->H; f.C = st->C; f.N = (int)N; f.out_act = L2.act; f.scale = 1.0f;
      f.fwd_out = out + b0 * N * st->C;
      tc_pack_and_g1(h, st, d, th, nb, &f, d.i8);
      continue;
    }
    tc_pack_and_g1(h, st, d, th, nb);
    Layer2FwdParams p = {};
    p.a_hi = st->a_hi.p; p.a_lo = st->a_lo.p; p.k_tiles = (int)(d.Npad / 128);
    p.theta = th; p.P = P; p.w2_off = L2.w_off; p.b2_off = L2.b_off;
    p.H = st->H; p.C = st->C; p.N = (int)N; p.out_act = L2.act; p.n_tiles = (int)(d.Npad / L2_ROWS);
    p.out = out + b0 * N * st->C;
    dim3 g(std::min(p.n_tiles, 64), nb);
    k_layer2_fwd<<<g, 128, 0, h->stream>>>(p);
    count_launch(h);
  }
  PYB_CUDA(cudaGetLastError());
}

// forward only: out [S, N, C] (softmax / output activation applied) for device-resident inputs x [N, D]
void tc_forward(pyb_handle* h, const float* theta, int64_t S, const float* x, int64_t N, float* out) {
  TcState* st = tc_state(h);
  tc_prepare_data(h, st->aux, x, N, false);
  tc_forward_on(h, st, st->aux, theta, S, N, out);
}

// the same forward on the tracked inputs of the streamed HMC predictive: their split operands are derived once per
// tracking (tc_invalidate_track) instead of once per sampling iteration, and the minibatch / test-input set `aux`
// stays untouched
void tc_forward_tracked(pyb_handle* h, const float* theta, int64_t S, const float* x, int64_t N, float* out) {
  TcState* st = tc_state(h);
  if (!st->track.ready || st->track.N != N || st->track.i8 != i8_mode(h, false, false))
    tc_prepare_data(h, st->track, x, N, false);
  tc_forward_on(h, st, st->track, theta, S, N, out);
}

// ---- building blocks exported to svgd.cu (Gram matrix and Stein contraction on the tensor cores) ----
void tc_split_rows(pyb_handle* h, const float* src, int64_t R, int C, int64_t lds, void* hi, void* lo, int64_t ldd) {
  const bool pairs = (C % 2 == 0) && (lds % 2 == 0) && (ldd % 2 == 0) && ((uintptr_t)src % 8 == 0) &&
                     ((uintptr_t)hi % 4 == 0) && ((uintptr_t)lo % 4 == 0);
  if (pairs)
    k_split_rows2<<<(unsigned)std::min<int64_t>((R * (C / 2) + 255) / 256, 16 * (int64_t)h->sm_count), 256, 0, h->stream>>>(
        src, R, C / 2, lds, (__nv_bfloat16*)hi, (__nv_bfloat16*)lo, ldd);
  else
    k_split_rows<<<(unsigned)std::min<int64_t>((R * C + 255) / 256, 65535), 256, 0, h->stream>>>(
        src, R, C, lds, (__nv_bfloat16*)hi, (__nv_bfloat16*)lo, ldd);
  count_launch(h);
}
// src [R, C] fp32 -> hi/lo [C, R] bf16 with row pitch ldd
void tc_split_transpose(pyb_handle* h, const float* src, int R, int C, int64_t lds, void* hi, void* lo, int64_t ldd) {
  dim3 g((C + 31) / 32, (R + 31) / 32, 1), blk(32, 8);
  k_split_transpose<<<g, blk, 0, h->stream>>>(src, 0, R, C, lds, (__nv_bfloat16*)hi, (__nv_bfloat16*)lo, 0, ldd);
  count_launch(h);
}
// out[m][n] = sum_k A[a_row0+m][k] B[n][k] for m < M, n < Nn; split operands, K-major, pitches in elements
// A == B with a_row0 == 0 and M == Nn is a Gram matrix: the CTA-pair kernel then computes only the 256x256 tiles on and
// above the diagonal and the rest is mirrored (exactly symmetric result, ~45 % fewer MMAs)
void tc_gemm_split(pyb_handle* h, const void* a_hi, const void* a_lo, int64_t lda, int64_t a_rows_total, int a_row0, int M,
                   const void* b_hi, const void* b_lo, int64_t ldb, int Nn, int64_t K, float* out, int64_t ldc) {
  PYB_REQUIRE(lda % 8 == 0 && ldb % 8 == 0, PYB_ERR_INVALID, "operand pitches must be multiples of 8 elements");
  CUtensorMap ma_h = make_map(a_hi, K, a_rows_total, lda, 128), ma_l = make_map(a_lo, K, a_rows_total, lda, 128);
  const int Hn = Nn >= 256 ? 256 : ((Nn + 15) / 16) * 16;
  CUtensorMap mb_h = make_map(b_hi, K, Nn, ldb, Hn), mb_l = make_map(b_lo, K, Nn, ldb, Hn);
  TcGemmParams p = {};
  p.K = (int)K; p.n_mtiles = (M + 127) / 128; p.n_pairs = (p.n_mtiles + 1) / 2; p.n_batch = (Nn + Hn - 1) / Hn; p.H = Hn;
  p.a_row0 = a_row0; p.a_batch_rows = 0; p.a_box_rows = 128; p.order = 1; p.sub_batch = 8;
  p.epi = EPI_STORE; p.out = out; p.out_stride = Hn; p.out_ld = (int)ldc; p.M_valid = M; p.N_valid = Hn; p.n_cols_total = Nn;
  const int nk = (int)((K + TC_BK - 1) / TC_BK);
  const int splits = (nk + TC_SPLIT_CHUNKS - 1) / TC_SPLIT_CHUNKS;
  TcState* st = tc_state(h);
  if (splits > 1) {      // long reductions (Gram over P = 1e5 parameters): split-K partials, fixed-order sum
    st->gpart.alloc((size_t)splits * M * ldc);
    p.k_splits = splits; p.chunks_per_split = TC_SPLIT_CHUNKS; p.split_stride = (int64_t)M * ldc; p.out = st->gpart.p;
  }
  p.total_items = p.n_pairs * p.n_batch * std::max(splits, 1);
  CUtensorMap mp_h = make_map(b_hi, K, Nn, ldb, std::max(Hn / 2, 8)), mp_l = make_map(b_lo, K, Nn, ldb, std::max(Hn / 2, 8));
  const bool gram = a_hi == b_hi && a_lo == b_lo && a_row0 == 0 && M == Nn && lda == ldb && Hn == 256 && pair_ok(h, p) &&
                    h->opt_tc_gram_sym;
  p.sym_skip = gram ? 1 : 0;
  launch_gemm_tc(h, ma_h, ma_l, mb_h, mb_l, p, 2.0 * M * (double)Nn * (double)K, &mp_h, &mp_l);
  if (splits > 1) {
    const int64_t cnt = (int64_t)M * ldc;
    dim3 rg((unsigned)std::min<int64_t>((cnt + 255) / 256, 4096), 1);
    k_reduce_ksplits<<<rg, 256, 0, h->stream>>>(st->gpart.p, splits, cnt, 0, cnt, out, 0);
    count_launch(h);
  }
  if (gram) {
    dim3 gm((unsigned)((M + 31) / 32), (unsigned)((M + 31) / 32)), bm(32, 8);
    k_mirror_lower_tiles<<<gm, bm, 0, h->stream>>>(out, M, ldc);
    count_launch(h);
  }
}

// the debug GEMM entry repeats its kernel launch PYB_DEBUG_GEMM_REPS times (default 1) so that a timing tool can read
// per-launch device times from the "profile" option's CUDA events
static int debug_gemm_reps() {
  const char* e = getenv("PYB_DEBUG_GEMM_REPS");
  const int r = e ? atoi(e) : 1;
  return r < 1 ? 1 : (r > 1000 ? 1000 : r);
}
// debug / unit-test entry: D[M,Nn] = A[M,K] B[Nn,K]^T through the tcgen05 kernel (host pointers)
void tc_debug_gemm(pyb_handle* h, const float* A, const float* B, int M, int Nn, int K, float* Dout) {
  PYB_REQUIRE(Nn % 16 == 0 && Nn >= 16 && Nn <= 256 && K % 8 == 0, PYB_ERR_INVALID, "Nn%16, Nn<=256, K%8 required");
  DevBuf<float> dA, dB, dD;
  DevBuf<__nv_bfloat16> ah, al, bh, bl;
  dA.alloc((size_t)M * K); dB.alloc((size_t)Nn * K); dD.alloc((size_t)M * Nn);
  ah.alloc((size_t)M * K); al.alloc((size_t)M * K); bh.alloc((size_t)Nn * K); bl.alloc((size_t)Nn * K);
  PYB_CUDA(cudaMemcpyAsync(dA.p, A, (size_t)M * K * 4, cudaMemcpyHostToDevice, h->stream));
  PYB_CUDA(cudaMemcpyAsync(dB.p, B, (size_t)Nn * K * 4, cudaMemcpyHostToDevice, h->stream));
  PYB_CUDA(cudaMemsetAsync(dD.p, 0xff, (size_t)M * Nn * 4, h->stream));
  k_split_rows<<<1024, 256, 0, h->stream>>>(dA.p, M, K, K, ah.p, al.p, K);
  k_split_rows<<<1024, 256, 0, h->stream>>>(dB.p, Nn, K, K, bh.p, bl.p, K);
  CUtensorMap ma_h = make_map(ah.p, K, M, K, 128), ma_l = make_map(al.p, K, M, K, 128);
  CUtensorMap mb_h = make_map(bh.p, K, Nn, K, Nn), mb_l = make_map(bl.p, K, Nn, K, Nn);
  TcGemmParams p = {};
  p.K = K; p.n_mtiles = (M + 127) / 128; p.n_pairs = (p.n_mtiles + 1) / 2; p.n_batch = 1; p.H = Nn;
  p.order = 0; p.sub_batch = 1; p.total_items = p.n_pairs;
  p.epi = EPI_STORE; p.out = dD.p; p.out_stride = 0; p.out_ld = Nn; p.M_valid = M; p.N_valid = Nn; p.a_batch_rows = 0; p.a_box_rows = 128;
  CUtensorMap mp_h = make_map(bh.p, K, Nn, K, std::max(Nn / 2, 8)), mp_l = make_map(bl.p, K, Nn, K, std::max(Nn / 2, 8));
  for (int r = 0; r < debug_gemm_reps(); ++r)
    launch_gemm_tc(h, ma_h, ma_l, mb_h, mb_l, p, 2.0 * M * Nn * (double)K, &mp_h, &mp_l);
  PYB_CUDA(cudaMemcpyAsync(Dout, dD.p, (size_t)M * Nn * 4, cudaMemcpyDeviceToHost, h->stream));
  PYB_CUDA(cudaStreamSynchronize(h->stream));
  PYB_CUDA(cudaGetLastError());
  prof_resolve(h);
}

// relu'(z1) as the LAST tensor-path evaluation used it, for one chain of its (single) chain batch: read back from the
// A1^T hi/lo blocks the fused kernel left in the workspace (a1 > 0 <=> one of its two bf16 parts is non-zero)
__global__ void k_relu_mask_from_a1(const uint16_t* __restrict__ a_hi, const uint16_t* __restrict__ a_lo, int64_t chain,
                                    int k_tiles, int H, int64_t N, int fused_order, uint8_t* __restrict__ out) {
  const int64_t total = N * H;
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (int64_t)gridDim.x * blockDim.x) {
    const int64_t r = i / H;
    const int hh = (int)(i - r * H);
    const int pos = fused_order ? fused_row_pos((int)(r & 127)) : (int)(r & 127);
    const int64_t o = (((chain * k_tiles + (r >> 7)) * H) + hh) * 128 + pos;
    out[i] = ((a_hi[o] & 0x7fffu) | (a_lo[o] & 0x7fffu)) ? 1 : 0;
  }
}
void tc_debug_relu_mask(pyb_handle* h, int64_t chain, uint8_t* out_host) {
  PYB_REQUIRE(h->tc != nullptr, PYB_ERR_STATE, "no tensor-path evaluation has run on this handle");
  TcState* st = (TcState*)h->tc;
  const Model& m = h->model;
  PYB_REQUIRE(st->train.ready && m.layer[0].act == PYB_ACT_RELU && st->cap_chains > 0, PYB_ERR_STATE,
              "the relu mask is available after a tensor-path evaluation of a relu network on the resident dataset");
  PYB_REQUIRE(chain >= 0 && chain < st->cap_chains, PYB_ERR_INVALID, "chain outside the last chain batch");
  const int H = st->H;
  const int64_t N = st->train.N;
  DevBuf<uint8_t> out;
  out.alloc((size_t)N * H);
  const bool fused = fused_ok(h, H, m.layer[0].act) && st->C <= L2_CMAX;
  k_relu_mask_from_a1<<<(unsigned)std::min<int64_t>((N * H + 255) / 256, 16 * (int64_t)h->sm_count), 256, 0, h->stream>>>(
      (const uint16_t*)st->a_hi.p, (const uint16_t*)st->a_lo.p, chain, (int)(st->train.Npad / 128), H, N, fused ? 1 : 0, out.p);
  PYB_CUDA(cudaMemcpyAsync(out_host, out.p, (size_t)N * H, cudaMemcpyDeviceToHost, h->stream));
  PYB_CUDA(cudaStreamSynchronize(h->stream));
  PYB_CUDA(cudaGetLastError());
}

}  // namespace pyb

extern "C" int pyb_debug_relu_mask(pyb_handle* h, int64_t chain, uint8_t* mask_out) {
  try {
    if (!h || !mask_out) throw pyb::Error(PYB_ERR_INVALID, "NULL argument");
    PYB_CUDA(cudaSetDevice(h->device));
    pyb::tc_debug_relu_mask(h, chain, mask_out);
  } catch (const pyb::Error& e) {
    pyb::set_last_error(e.what());
    return e.code;
  }
  return PYB_OK;
}

extern "C" int pyb_debug_tc_gemm(pyb_handle* h, const float* A, const float* B, int32_t M, int32_t Nn, int32_t K,
                                 float* D) {
  try {
    if (!h || !A || !B || !D) throw pyb::Error(PYB_ERR_INVALID, "NULL argument");
    PYB_CUDA(cudaSetDevice(h->device));
    pyb::tc_debug_gemm(h, A, B, M, Nn, K, D);
  } catch (const pyb::Error& e) {
    pyb::set_last_error(e.what());
    return e.code;
  }
  return PYB_OK;
}
