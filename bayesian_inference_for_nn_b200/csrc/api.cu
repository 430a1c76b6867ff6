// api.cu — the extern "C" boundary of libpyesian_b200.so (declared in include/pyesian_b200.h).
// Exceptions stop here: every entry point returns a pyb_status and records pyb_last_error().
#include "common.cuh"
#include <math.h>
#include <string.h>
#include <new>
#include <algorithm>

namespace pyb {
static thread_local std::string g_last_error;
void set_last_error(const std::string& m) { g_last_error = m; }

// flag[0] |= (a differs from b anywhere), 32-bit words, bit patterns (a NaN equals itself); grid-stride
__global__ void k_differs(const uint32_t* __restrict__ a, const uint32_t* __restrict__ b, size_t n, int32_t* flag) {
  uint32_t d = 0;
  for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (size_t)gridDim.x * blockDim.x) d |= a[i] ^ b[i];
  if (__any_sync(0xffffffffu, d != 0) && (threadIdx.x & 31) == 0) atomicOr(flag, 1);
}
__global__ void k_check_labels(const int32_t* __restrict__ y, int64_t n, int C, int32_t* flag) {
  bool bad = false;
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x)
    bad |= y[i] < 0 || y[i] >= C;
  if (__any_sync(0xffffffffu, bad) && (threadIdx.x & 31) == 0) atomicOr(flag, 1);
}

// fused_small.cu / tc_path.cu
bool fused_small_supported(pyb_handle* h);
void fused_small_eval(pyb_handle* h, const float* theta, int64_t S, float scale, float* loss, float* grad);
bool tc_supported(pyb_handle* h, int64_t S);
void tc_eval(pyb_handle* h, const float* theta, int64_t S, float scale, float* loss, float* grad);
void tc_release(pyb_handle* h);
void tc_invalidate_dataset(pyb_handle* h);
int tc_resident_split(const pyb_handle* h);
void tc_read_timeline(pyb_handle* h, unsigned long long* out_8x160);

int resolve_path(pyb_handle* h, int64_t S, bool with_grad) {
  int path = h->opt_path;
  if (path == PYB_PATH_AUTO) {
    if (with_grad && tc_supported(h, S)) path = PYB_PATH_TENSOR;
    else if (with_grad && fused_small_supported(h)) path = PYB_PATH_FUSED_SMALL;
    else path = PYB_PATH_GENERIC;
  }
  return path;
}

void eval_loss_grad(pyb_handle* h, const float* theta, int64_t S, float scale, float* loss_out, float* grad_out) {
  NvtxRange nv("pyb.eval.fwd_bwd");
  int path = resolve_path(h, S, grad_out != nullptr);
  if (path == PYB_PATH_TENSOR) {
    PYB_REQUIRE(tc_supported(h, S), PYB_ERR_UNSUPPORTED, "tensor path does not support this model/dataset shape");
    PYB_REQUIRE(grad_out != nullptr, PYB_ERR_UNSUPPORTED, "tensor path computes loss and gradient together");
    tc_eval(h, theta, S, scale, loss_out, grad_out);
  } else if (path == PYB_PATH_FUSED_SMALL) {
    PYB_REQUIRE(fused_small_supported(h), PYB_ERR_UNSUPPORTED, "fused small path does not support this model shape");
    PYB_REQUIRE(grad_out != nullptr, PYB_ERR_UNSUPPORTED, "fused small path computes loss and gradient together");
    fused_small_eval(h, theta, S, scale, loss_out, grad_out);
  } else {
    generic_eval(h, theta, S, h->X.p, h->y_i.p, h->y_f.p, h->N, scale, loss_out, grad_out);
  }
  h->path_used = path;
}
void eval_on_batch(pyb_handle* h, const float* theta, int64_t S, const float* Xb, const int32_t* yb_i, const float* yb_f,
                   int64_t Nb, float scale, float* loss_out, float* grad_out) {
  if (Xb == h->X.p && Nb == h->N) { eval_loss_grad(h, theta, S, scale, loss_out, grad_out); return; }
  NvtxRange nv("pyb.eval.fwd_bwd.minibatch");
  const bool tensor_ok = grad_out && tc_supported_rows(h, Nb) && (h->opt_path == PYB_PATH_AUTO || h->opt_path == PYB_PATH_TENSOR);
  const bool small_ok = grad_out && Nb <= h->N && fused_small_supported(h) &&
                        (h->opt_path == PYB_PATH_AUTO || h->opt_path == PYB_PATH_FUSED_SMALL);
  if (tensor_ok) { tc_eval_batch(h, Xb, yb_i, yb_f, Nb, theta, S, scale, loss_out, grad_out); h->path_used = PYB_PATH_TENSOR; }
  else if (small_ok) {   // small-width nets: one launch, parameters and the batch in shared memory
    fused_small_eval_on(h, theta, S, Xb, yb_i, yb_f, Nb, scale, loss_out, grad_out); h->path_used = PYB_PATH_FUSED_SMALL;
  }
  else { generic_eval(h, theta, S, Xb, yb_i, yb_f, Nb, scale, loss_out, grad_out); h->path_used = PYB_PATH_GENERIC; }
}
}  // namespace pyb

using namespace pyb;

#define PYB_TRY try {
#define PYB_CATCH                                      \
  }                                                    \
  catch (const pyb::Error& e) {                        \
    pyb::set_last_error(e.what());                     \
    return e.code;                                     \
  }                                                    \
  catch (const std::bad_alloc&) {                      \
    pyb::set_last_error("host allocation failed");     \
    return PYB_ERR_OOM;                                \
  }                                                    \
  catch (const std::exception& e) {                    \
    pyb::set_last_error(e.what());                     \
    return PYB_ERR_INVALID;                            \
  }                                                    \
  return PYB_OK;

static void use_device(const pyb_handle* h) { PYB_CUDA(cudaSetDevice(h->device)); }

extern "C" {

int pyb_version(void) { return PYB_ABI_VERSION; }
const char* pyb_last_error(void) { return pyb::g_last_error.c_str(); }

int pyb_device_count(int32_t* n_out) {
  PYB_TRY
  PYB_REQUIRE(n_out, PYB_ERR_INVALID, "n_out is NULL");
  int n = 0;
  cudaError_t e = cudaGetDeviceCount(&n);
  if (e != cudaSuccess) { cudaGetLastError(); n = 0; }
  *n_out = n;
  PYB_CATCH
}

int pyb_create(const pyb_model_desc* d, int32_t device_id, uint64_t seed, pyb_handle** out) {
  PYB_TRY
  PYB_REQUIRE(d && out, PYB_ERR_INVALID, "NULL argument");
  PYB_REQUIRE(d->n_layers >= 1 && d->n_layers <= kMaxLayers, PYB_ERR_INVALID, "n_layers must be in [1,16]");
  PYB_REQUIRE(d->in_dim >= 1, PYB_ERR_INVALID, "in_dim must be >= 1");
  PYB_REQUIRE(d->units && d->activation && d->use_bias, PYB_ERR_INVALID, "NULL layer arrays");
  int ndev = 0;
  cudaError_t e = cudaGetDeviceCount(&ndev);
  if (e != cudaSuccess || ndev == 0) {
    cudaGetLastError();
    throw Error(PYB_ERR_CUDA, "no CUDA device: libpyesian_b200 has no CPU fallback");
  }
  PYB_REQUIRE(device_id >= 0 && device_id < ndev, PYB_ERR_INVALID, "device_id out of range");
  cudaDeviceProp prop;
  PYB_CUDA(cudaGetDeviceProperties(&prop, device_id));
  PYB_REQUIRE(prop.major == 10, PYB_ERR_CUDA, "device is not sm_100-class (B200): this library is sm_100a only");
  pyb_handle* h = new pyb_handle();
  h->device = device_id;
  h->sm_count = prop.multiProcessorCount;
  h->seed = seed;
  if (const char* ev = getenv("PYB_TC_I8")) {   // development: default operand split of the tensor path (the tc_i8 option overrides it)
    const int v = atoi(ev);
    if (v >= -1 && v <= 2) h->opt_tc_i8 = v;
  }
  Model& m = h->model;
  m.n_layers = d->n_layers;
  m.in_dim = d->in_dim;
  int fin = d->in_dim;
  int64_t off = 0;
  for (int l = 0; l < d->n_layers; ++l) {
    LayerDesc& L = m.layer[l];
    if (d->units[l] < 1) { delete h; throw Error(PYB_ERR_INVALID, "units must be >= 1"); }
    int act = d->activation[l];
    if (act < 0 || act > PYB_ACT_SIGMOID || (act == PYB_ACT_SOFTMAX && l != d->n_layers - 1)) {
      delete h;
      throw Error(PYB_ERR_UNSUPPORTED, "unsupported activation (softmax is only supported on the output layer)");
    }
    L.fan_in = fin; L.fan_out = d->units[l]; L.act = act; L.use_bias = d->use_bias[l] ? 1 : 0;
    L.w_off = off; off += (int64_t)fin * L.fan_out;
    L.b_off = -1;
    if (L.use_bias) { L.b_off = off; off += L.fan_out; }
    if (L.fan_out > m.max_width) m.max_width = L.fan_out;
    fin = L.fan_out;
  }
  m.P = off;
  m.out_dim = fin;
  try {
    PYB_CUDA(cudaSetDevice(device_id));
    PYB_CUDA(cudaStreamCreateWithFlags(&h->stream, cudaStreamNonBlocking));
    PYB_CUDA(cudaEventCreate(&h->ev0));
    PYB_CUDA(cudaEventCreate(&h->ev1));
  } catch (...) { delete h; throw; }
  *out = h;
  PYB_CATCH
}

int pyb_destroy(pyb_handle* h) {
  PYB_TRY
  if (!h) return PYB_OK;
  cudaSetDevice(h->device);
  if (h->stream) cudaStreamSynchronize(h->stream);
  tc_release(h);
  if (h->svgd.comm_stream) cudaStreamSynchronize(h->svgd.comm_stream);
  if (h->svgd.gram_stream) {
    cudaStreamSynchronize(h->svgd.gram_stream);
    cudaStreamDestroy(h->svgd.gram_stream); h->svgd.gram_stream = nullptr;
    cudaEvent_t* evs[] = {&h->svgd.ev_kernel, &h->svgd.ev_gh[0], &h->svgd.ev_gh[1], &h->svgd.ev_p1, &h->svgd.ev_p2, &h->svgd.ev_back};
    for (cudaEvent_t* e : evs) { if (*e) cudaEventDestroy(*e); *e = nullptr; }
  }
  svgd_p2p_release(h);
  if (h->svgd.nccl_comm3) { nccl_comm_destroy(h->svgd.nccl_comm3); h->svgd.nccl_comm3 = nullptr; }
  if (h->svgd.nccl_comm2) { nccl_comm_destroy(h->svgd.nccl_comm2); h->svgd.nccl_comm2 = nullptr; }
  if (h->svgd.nccl_comm) { nccl_comm_destroy(h->svgd.nccl_comm); h->svgd.nccl_comm = nullptr; }
  if (h->svgd.comm_stream) {
    cudaStreamDestroy(h->svgd.comm_stream); h->svgd.comm_stream = nullptr;
    cudaEventDestroy(h->svgd.ev_fork); cudaEventDestroy(h->svgd.ev_theta); cudaEventDestroy(h->svgd.ev_grad);
    h->svgd.ev_fork = h->svgd.ev_theta = h->svgd.ev_grad = nullptr;
  }
  for (auto* b : h->ws.act) delete b;
  for (cudaEvent_t e : h->prof_events) cudaEventDestroy(e);
  h->ws.act.clear();
  if (h->ev0) cudaEventDestroy(h->ev0);
  if (h->ev1) cudaEventDestroy(h->ev1);
  if (h->stream) cudaStreamDestroy(h->stream);
  delete h;
  PYB_CATCH
}

int pyb_param_count(const pyb_handle* h, int64_t* n) {
  PYB_TRY
  PYB_REQUIRE(h && n, PYB_ERR_INVALID, "NULL argument");
  *n = h->model.P;
  PYB_CATCH
}

int pyb_set_option(pyb_handle* h, const char* key, double v) {
  PYB_TRY
  PYB_REQUIRE(h && key, PYB_ERR_INVALID, "NULL argument");
  if (!strcmp(key, "path")) {
    PYB_REQUIRE(v >= 0 && v <= 3, PYB_ERR_INVALID, "path must be 0..3");
    h->opt_path = (int)v;
  } else if (!strcmp(key, "workspace_mb")) {
    PYB_REQUIRE(v >= 1, PYB_ERR_INVALID, "workspace_mb must be >= 1");
    h->opt_workspace_mb = v;
  } else if (!strcmp(key, "chain_batch")) {
    h->opt_chain_batch = (int64_t)v;
  } else if (!strcmp(key, "tc_pair")) {
    h->opt_tc_pair = v != 0;
  } else if (!strcmp(key, "tc_dual")) {
    h->opt_tc_dual = v != 0;
  } else if (!strcmp(key, "tc_h128_pairs")) {
    h->opt_tc_h128_pairs = v != 0;
  } else if (!strcmp(key, "tc_gram_sym")) {
    h->opt_tc_gram_sym = v != 0;
  } else if (!strcmp(key, "fs_cluster")) {
    h->opt_fs_cluster = v != 0;
  } else if (!strcmp(key, "live_cta")) {
    h->opt_live_cta = v != 0;
  } else if (!strcmp(key, "live_fused")) {
    h->opt_live_fused = v != 0;
  } else if (!strcmp(key, "hmc_carry")) {
    h->opt_hmc_carry = v != 0;
    h->hmc.have_cur = false;
  } else if (!strcmp(key, "hmc_swap")) {
    h->opt_hmc_swap = v != 0;
  } else if (!strcmp(key, "hmc_keep_samples")) {
    PYB_REQUIRE(!h->hmc.sampling_started, PYB_ERR_STATE,
                "hmc_keep_samples cannot change during a sampling phase (set it before, or after pyb_hmc_reset_samples)");
    h->opt_hmc_keep_samples = v != 0;
  } else if (!strcmp(key, "predict_sharded")) {
    h->opt_predict_sharded = v != 0;
  } else if (!strcmp(key, "tc_fuse")) {
    h->opt_tc_fuse = v != 0;
  } else if (!strcmp(key, "tc_timeline")) {
    h->opt_tc_timeline = (int)v;
  } else if (!strcmp(key, "tc_epi_mma")) {
    h->opt_tc_epi_mma = v != 0;
  } else if (!strcmp(key, "svgd_pshard")) {
    h->opt_svgd_pshard = v != 0;
  } else if (!strcmp(key, "svgd_chain_fused")) {
    h->opt_svgd_chain_fused = v != 0;
  } else if (!strcmp(key, "select_compact")) {
    h->opt_select_compact = (int)v;
  } else if (!strcmp(key, "svgd_gram_sync")) {
    h->opt_svgd_gram_sync = v != 0;
  } else if (!strcmp(key, "svgd_halves")) {
    h->opt_svgd_halves = v != 0;
  } else if (!strcmp(key, "svgd_p2p")) {
    h->opt_svgd_p2p = v != 0;
    h->svgd.p2p_tried = false;
    h->svgd.ps_ready = false;
  } else if (!strcmp(key, "tc_i8_min_loss")) {
    PYB_REQUIRE(v >= 0, PYB_ERR_INVALID, "tc_i8_min_loss must be >= 0");
    h->opt_i8_min_loss = v;
  } else if (!strcmp(key, "tc_i8")) {
    PYB_REQUIRE(v == -1 || v == 0 || v == 1 || v == 2, PYB_ERR_INVALID, "tc_i8 must be -1 (auto), 0 (bf16x3), 1 or 2 (int8 slices)");
    h->opt_tc_i8 = (int)v;
  } else if (!strcmp(key, "profile")) {
    h->prof_enabled = v != 0;
    h->prof_ms = h->prof_flops = 0; h->prof_launches = 0; h->prof_used = 0;
  } else {
    throw Error(PYB_ERR_INVALID, std::string("unknown option: ") + key);
  }
  PYB_CATCH
}

int pyb_get_info(const pyb_handle* h, const char* key, double* out) {
  PYB_TRY
  PYB_REQUIRE(h && key && out, PYB_ERR_INVALID, "NULL argument");
  if (!strcmp(key, "path_used")) *out = h->path_used;
  else if (!strcmp(key, "kernel_launches")) *out = (double)h->kernel_launches;
  else if (!strcmp(key, "last_device_ms")) *out = h->last_device_ms;
  else if (!strcmp(key, "sm_count")) *out = h->sm_count;
  else if (!strcmp(key, "fs_cluster_used")) *out = h->fs_cluster_used;
  else if (!strcmp(key, "svgd_stein_used")) *out = h->svgd_stein_used;
  else if (!strcmp(key, "hmc_param_bytes")) *out = (double)hmc_params_bytes(h);
  else if (!strcmp(key, "prof_ms")) *out = h->prof_ms;
  else if (!strcmp(key, "prof_flops")) *out = h->prof_flops;
  else if (!strcmp(key, "prof_launches")) *out = (double)h->prof_launches;
  else if (!strcmp(key, "n_train")) *out = (double)h->n_train;
  else if (!strncmp(key, "tc_timeline_", 12) && key[12] >= '0' && key[12] <= '9' && !key[13]) {
    // mean over the CTAs (of cluster leaders for the issuer's entries) of the last fused launch's phase k, in cycles per item
    std::vector<unsigned long long> t(8 * 160);
    tc_read_timeline(const_cast<pyb_handle*>(h), t.data());
    int k = key[12] - '0';
    double s = 0, n = 0;
    if (k >= 8) {                                        // 8 / 9: the odd CTAs' epilogue entries kept in slots 0 / 1
      for (int c = 1; c < 148; c += 2) {
        const unsigned long long items = t[(c & ~1) * 8 + 3];
        if (items) { s += (double)t[c * 8 + k - 8] / (double)items; n += 1; }
      }
      *out = n ? s / n : 0.0;
      return PYB_OK;
    }
    for (int c = 0; c < 148; ++c) {
      const unsigned long long items = t[(c & ~1) * 8 + 3];
      if (items && (k >= 4 || !(c & 1))) { s += k == 3 ? (double)items : (double)t[c * 8 + k] / (double)items; n += 1; }
    }
    *out = n ? s / n : 0.0;
  }
  else if (!strcmp(key, "hmc_arena_rows")) *out = (double)h->hmc.arena_cap;
  else if (!strcmp(key, "i8_guard_ok")) *out = h->i8_guard_ok ? 1.0 : 0.0;
  else if (!strcmp(key, "i8_guard_trips")) *out = (double)h->i8_guard_trips;
  else if (!strcmp(key, "svgd_h")) *out = h->svgd.last_h;
  else if (!strcmp(key, "svgd_p2p")) *out = h->svgd.p2p_ready ? 1.0 : 0.0;
  else if (!strncmp(key, "svgd_phase_ms_", 14) && key[14] >= '0' && key[14] <= '6' && !key[15]) *out = h->svgd.ps_ms[key[14] - '0'];
  else if (!strcmp(key, "tc_split")) *out = (double)tc_resident_split(h);
  else if (!strcmp(key, "dataset_uploads")) *out = (double)h->dataset_uploads;
  else if (!strcmp(key, "dataset_kept")) *out = (double)h->dataset_kept;
  else throw Error(PYB_ERR_INVALID, std::string("unknown info key: ") + key);
  PYB_CATCH
}

int pyb_set_dataset(pyb_handle* h, const float* X, int64_t N, const void* y, int32_t loss_kind, int32_t mem,
                    int64_t n_train) {
  PYB_TRY
  PYB_REQUIRE(h && X && y, PYB_ERR_INVALID, "NULL argument");
  PYB_REQUIRE(N >= 1 && N < (1ll << 31), PYB_ERR_INVALID, "N must be in [1, 2^31)");
  PYB_REQUIRE(loss_kind == PYB_LOSS_SPARSE_CE || loss_kind == PYB_LOSS_MSE, PYB_ERR_INVALID, "bad loss_kind");
  PYB_REQUIRE(mem == PYB_MEM_HOST || mem == PYB_MEM_DEVICE, PYB_ERR_INVALID, "bad mem");
  const Model& m = h->model;
  int last_act = m.layer[m.n_layers - 1].act;
  if (loss_kind == PYB_LOSS_SPARSE_CE)
    PYB_REQUIRE(last_act == PYB_ACT_SOFTMAX, PYB_ERR_UNSUPPORTED,
                "SparseCategoricalCrossentropy needs a softmax output layer (logits path of Keras 2.15)");
  else
    PYB_REQUIRE(last_act != PYB_ACT_SOFTMAX, PYB_ERR_UNSUPPORTED, "MeanSquaredError on a softmax output is not supported");
  use_device(h);
  if (mem == PYB_MEM_DEVICE) PYB_CUDA(cudaDeviceSynchronize());   // the producer's stream is not ours (header: "device pointers")
  const bool ce = loss_kind == PYB_LOSS_SPARSE_CE;
  // labels are validated BEFORE any handle state changes (the loss kernels index the logits with them)
  if (ce && mem == PYB_MEM_HOST) {
    const int32_t* yi = (const int32_t*)y;
    for (int64_t i = 0; i < N; ++i)
      if (yi[i] < 0 || yi[i] >= m.out_dim) throw Error(PYB_ERR_INVALID, "label out of range [0, out_dim)");
  }
  h->flag.alloc(2);
  PYB_CUDA(cudaMemsetAsync(h->flag.p, 0, 2 * sizeof(int32_t), h->stream));
  if (ce && mem == PYB_MEM_DEVICE) {
    k_check_labels<<<(unsigned)std::min<int64_t>((N + 255) / 256, 1024), 256, 0, h->stream>>>((const int32_t*)y, N, m.out_dim,
                                                                                          h->flag.p + 1);
    int32_t bad = 0;
    PYB_CUDA(cudaMemcpyAsync(&bad, h->flag.p + 1, sizeof(int32_t), cudaMemcpyDeviceToHost, h->stream));
    PYB_CUDA(cudaStreamSynchronize(h->stream));
    if (bad) throw Error(PYB_ERR_INVALID, "label out of range [0, out_dim)");
  }
  const cudaMemcpyKind kind = mem == PYB_MEM_HOST ? cudaMemcpyHostToDevice : cudaMemcpyDeviceToDevice;
  const size_t xb = (size_t)N * m.in_dim * sizeof(float);
  const size_t yb = ce ? (size_t)N * sizeof(int32_t) : (size_t)N * m.out_dim * sizeof(float);
  const int64_t nt = n_train > 0 ? n_train : N;
  // A caller that re-submits the SAME data (a training loop that passes its dataset every step) keeps everything derived
  // from it: the incoming copy is compared bit for bit with the resident one on the device (one pass at HBM rate), and
  // only a different dataset replaces it, invalidating the split / sliced operands and the carried HMC evaluation.
  const bool comparable = h->have_data && h->N == N && h->loss_kind == loss_kind && h->n_train == nt;
  bool same = false;
  if (comparable) {
    const float* Xin = X;
    const void* yin = y;
    if (mem == PYB_MEM_HOST) {
      h->X_stage.alloc((size_t)N * m.in_dim);
      PYB_CUDA(cudaMemcpyAsync(h->X_stage.p, X, xb, kind, h->stream));
      Xin = h->X_stage.p;
      if (ce) { h->yi_stage.alloc(N); PYB_CUDA(cudaMemcpyAsync(h->yi_stage.p, y, yb, kind, h->stream)); yin = h->yi_stage.p; }
      else { h->yf_stage.alloc((size_t)N * m.out_dim); PYB_CUDA(cudaMemcpyAsync(h->yf_stage.p, y, yb, kind, h->stream)); yin = h->yf_stage.p; }
    }
    const void* yres = ce ? (const void*)h->y_i.p : (const void*)h->y_f.p;
    k_differs<<<(unsigned)std::min<size_t>((xb / 4 + 1023) / 1024, 8 * (size_t)h->sm_count), 256, 0, h->stream>>>(
        (const uint32_t*)Xin, (const uint32_t*)h->X.p, xb / 4, h->flag.p);
    k_differs<<<(unsigned)std::min<size_t>((yb / 4 + 1023) / 1024, 8 * (size_t)h->sm_count), 256, 0, h->stream>>>(
        (const uint32_t*)yin, (const uint32_t*)yres, yb / 4, h->flag.p);
    int32_t diff = 1;
    PYB_CUDA(cudaMemcpyAsync(&diff, h->flag.p, sizeof(int32_t), cudaMemcpyDeviceToHost, h->stream));
    PYB_CUDA(cudaStreamSynchronize(h->stream));
    same = diff == 0;
    if (!same) {
      if (mem == PYB_MEM_HOST) {          // the staged copy becomes the resident one
        h->X.swap(h->X_stage);
        if (ce) h->y_i.swap(h->yi_stage); else h->y_f.swap(h->yf_stage);
      } else {
        PYB_CUDA(cudaMemcpyAsync(h->X.p, X, xb, kind, h->stream));
        PYB_CUDA(cudaMemcpyAsync(ce ? (void*)h->y_i.p : (void*)h->y_f.p, y, yb, kind, h->stream));
      }
    }
  } else {
    h->have_data = false;                 // nothing below may leave a stale N against reallocated buffers
    h->X.alloc((size_t)N * m.in_dim);
    PYB_CUDA(cudaMemcpyAsync(h->X.p, X, xb, kind, h->stream));
    if (ce) { h->y_i.alloc(N); PYB_CUDA(cudaMemcpyAsync(h->y_i.p, y, yb, kind, h->stream)); }
    else { h->y_f.alloc((size_t)N * m.out_dim); PYB_CUDA(cudaMemcpyAsync(h->y_f.p, y, yb, kind, h->stream)); }
  }
  PYB_CUDA(cudaStreamSynchronize(h->stream));
  h->N = N;
  h->n_train = nt;
  h->loss_kind = loss_kind;
  h->have_data = true;
  h->dataset_uploads += 1;
  if (same) {
    h->dataset_kept += 1;
  } else {
    h->hmc.have_cur = false;      // a new dataset invalidates the carried loss / gradient
    tc_invalidate_dataset(h);
  }
  PYB_CATCH
}

int pyb_set_prior_gaussian(pyb_handle* h, const float* mean, const float* sigma, int32_t form) {
  PYB_TRY
  PYB_REQUIRE(h && mean && sigma, PYB_ERR_INVALID, "NULL argument");
  const Model& m = h->model;
  std::vector<float> mu(m.P), sg(m.P), iv(m.P);
  if (form == PYB_PRIOR_SCALAR) {
    for (int64_t i = 0; i < m.P; ++i) { mu[i] = mean[0]; sg[i] = sigma[0]; }
  } else if (form == PYB_PRIOR_PER_VARIABLE) {
    int v = 0;
    for (int l = 0; l < m.n_layers; ++l) {
      const LayerDesc& L = m.layer[l];
      for (int64_t i = 0; i < (int64_t)L.fan_in * L.fan_out; ++i) { mu[L.w_off + i] = mean[v]; sg[L.w_off + i] = sigma[v]; }
      ++v;
      if (L.use_bias) {
        for (int i = 0; i < L.fan_out; ++i) { mu[L.b_off + i] = mean[v]; sg[L.b_off + i] = sigma[v]; }
        ++v;
      }
    }
  } else if (form == PYB_PRIOR_PER_ELEMENT) {
    for (int64_t i = 0; i < m.P; ++i) { mu[i] = mean[i]; sg[i] = sigma[i]; }
  } else {
    throw Error(PYB_ERR_INVALID, "bad prior form");
  }
  double c = 0.0;
  for (int64_t i = 0; i < m.P; ++i) {
    PYB_REQUIRE(sg[i] != 0.f, PYB_ERR_INVALID, "sigma must be non-zero");
    iv[i] = 1.0f / (sg[i] * sg[i]);
    c += (double)logf(sg[i]) + 0.9189385332046727;  // log sigma + 1/2 log 2pi; NaN for sigma<0 as tfp (SURVEY B-1)
  }
  use_device(h);
  h->mu.alloc(m.P); h->sigma.alloc(m.P); h->inv_var.alloc(m.P);
  PYB_CUDA(cudaMemcpy(h->mu.p, mu.data(), m.P * sizeof(float), cudaMemcpyHostToDevice));
  PYB_CUDA(cudaMemcpy(h->sigma.p, sg.data(), m.P * sizeof(float), cudaMemcpyHostToDevice));
  PYB_CUDA(cudaMemcpy(h->inv_var.p, iv.data(), m.P * sizeof(float), cudaMemcpyHostToDevice));
  h->prior_const = c;
  h->have_prior = true;
  PYB_CATCH
}

int pyb_hmc_init(pyb_handle* h, int64_t S, int64_t chain_offset, double eps, double m, int32_t L, int32_t sem,
                 const float* q0) {
  PYB_TRY
  PYB_REQUIRE(h, PYB_ERR_INVALID, "NULL handle");
  use_device(h);
  hmc_init(h, S, chain_offset, eps, m, L, sem, q0);
  PYB_CATCH
}

int pyb_hmc_inject(pyb_handle* h, const float* p, const float* u) {
  PYB_TRY
  PYB_REQUIRE(h, PYB_ERR_INVALID, "NULL handle");
  HmcState& st = h->hmc;
  PYB_REQUIRE(st.inited, PYB_ERR_STATE, "pyb_hmc_init must be called first");
  use_device(h);
  const int64_t P = h->model.P;
  if (p) {
    st.inj_p.alloc(st.S * P);
    PYB_CUDA(cudaMemcpy(st.inj_p.p, p, st.S * P * sizeof(float), cudaMemcpyHostToDevice));
    st.have_inj_p = true;
  }
  if (u) {
    st.inj_u.alloc(st.S);
    PYB_CUDA(cudaMemcpy(st.inj_u.p, u, st.S * sizeof(float), cudaMemcpyHostToDevice));
    st.have_inj_u = true;
  }
  PYB_CATCH
}

int pyb_hmc_run(pyb_handle* h, int32_t n_iters, int32_t burning, int32_t sampling, pyb_hmc_diag* out) {
  PYB_TRY
  PYB_REQUIRE(h, PYB_ERR_INVALID, "NULL handle");
  use_device(h);
  hmc_run(h, n_iters, burning != 0, sampling != 0, out);
  PYB_CATCH
}

int pyb_hmc_eval(pyb_handle* h, const float* q, int64_t S, float* U, float* loss, float* grad) {
  PYB_TRY
  PYB_REQUIRE(h && q, PYB_ERR_INVALID, "NULL argument");
  use_device(h);
  hmc_eval(h, q, S, U, loss, grad);
  PYB_CATCH
}

int pyb_hmc_get_state(pyb_handle* h, float* q, float* p) {
  PYB_TRY
  PYB_REQUIRE(h, PYB_ERR_INVALID, "NULL handle");
  HmcState& st = h->hmc;
  PYB_REQUIRE(st.inited, PYB_ERR_STATE, "pyb_hmc_init must be called first");
  use_device(h);
  size_t n = (size_t)st.S * h->model.P * sizeof(float);
  PYB_CUDA(cudaStreamSynchronize(h->stream));
  if (q) PYB_CUDA(cudaMemcpy(q, st.q.p, n, cudaMemcpyDeviceToHost));
  if (p) PYB_CUDA(cudaMemcpy(p, st.p.p, n, cudaMemcpyDeviceToHost));
  PYB_CATCH
}

int pyb_hmc_last(pyb_handle* h, float* U0, float* K0, float* U1, float* K1, float* log_alpha, int32_t* accepted,
                 float* loss) {
  PYB_TRY
  PYB_REQUIRE(h, PYB_ERR_INVALID, "NULL handle");
  HmcState& st = h->hmc;
  PYB_REQUIRE(st.inited && st.iter > 0, PYB_ERR_STATE, "no iteration has run yet");
  use_device(h);
  PYB_CUDA(cudaStreamSynchronize(h->stream));
  size_t n = (size_t)st.S * sizeof(float);
  if (U0) PYB_CUDA(cudaMemcpy(U0, st.U0.p, n, cudaMemcpyDeviceToHost));
  if (K0) PYB_CUDA(cudaMemcpy(K0, st.K0.p, n, cudaMemcpyDeviceToHost));
  if (U1) PYB_CUDA(cudaMemcpy(U1, st.U1.p, n, cudaMemcpyDeviceToHost));
  if (K1) PYB_CUDA(cudaMemcpy(K1, st.K1.p, n, cudaMemcpyDeviceToHost));
  if (log_alpha) PYB_CUDA(cudaMemcpy(log_alpha, st.log_alpha.p, n, cudaMemcpyDeviceToHost));
  if (accepted) PYB_CUDA(cudaMemcpy(accepted, st.accepted.p, n, cudaMemcpyDeviceToHost));
  if (loss) PYB_CUDA(cudaMemcpy(loss, st.ret_loss.p, n, cudaMemcpyDeviceToHost));
  PYB_CATCH
}

int pyb_hmc_reset_samples(pyb_handle* h) {
  PYB_TRY
  PYB_REQUIRE(h, PYB_ERR_INVALID, "NULL handle");
  HmcState& st = h->hmc;
  PYB_REQUIRE(st.inited, PYB_ERR_STATE, "pyb_hmc_init must be called first");
  use_device(h);
  PYB_CUDA(cudaStreamSynchronize(h->stream));
  PYB_CUDA(cudaMemset(st.arena_count.p, 0, sizeof(int32_t)));
  PYB_CUDA(cudaMemset(st.pending_freq.p, 0, st.S * sizeof(int32_t)));
  PYB_CUDA(cudaMemset(st.last_idx.p, 0xff, st.S * sizeof(int32_t)));
  st.arena_used_upper = 0;
  st.host_samples.clear(); st.host_freq.clear(); st.host_chain.clear();
  st.host_last_idx.assign(st.S, -1);
  st.sampling_started = false;
  hmc_track_clear(h);
  hmc_params_clear(h);
  PYB_CATCH
}

int pyb_hmc_sample_count(pyb_handle* h, int64_t* n) {
  PYB_TRY
  PYB_REQUIRE(h && n, PYB_ERR_INVALID, "NULL argument");
  HmcState& st = h->hmc;
  PYB_REQUIRE(st.inited, PYB_ERR_STATE, "pyb_hmc_init must be called first");
  use_device(h);
  hmc_flush_arena(h);
  *n = (int64_t)st.host_freq.size();
  PYB_CATCH
}

int pyb_hmc_samples(pyb_handle* h, float* samples, int32_t* freq, int32_t* chain) {
  PYB_TRY
  PYB_REQUIRE(h, PYB_ERR_INVALID, "NULL handle");
  HmcState& st = h->hmc;
  PYB_REQUIRE(st.inited, PYB_ERR_STATE, "pyb_hmc_init must be called first");
  use_device(h);
  hmc_flush_arena(h);
  // chain-major, acceptance order within a chain (stable counting sort on the chain id)
  const int64_t P = h->model.P, n = (int64_t)st.host_freq.size();
  std::vector<int64_t> start(st.S + 1, 0);
  for (int64_t i = 0; i < n; ++i) start[st.host_chain[i] - st.chain_offset + 1]++;
  for (int64_t s = 0; s < st.S; ++s) start[s + 1] += start[s];
  for (int64_t i = 0; i < n; ++i) {
    int64_t d = start[st.host_chain[i] - st.chain_offset]++;
    if (samples) memcpy(samples + d * P, st.host_samples.data() + i * P, P * sizeof(float));
    if (freq) freq[d] = st.host_freq[i];
    if (chain) chain[d] = st.host_chain[i];
  }
  PYB_CATCH
}

int pyb_hmc_adapt_begin(pyb_handle* h, double target_accept) {
  PYB_TRY
  PYB_REQUIRE(h, PYB_ERR_INVALID, "NULL handle");
  use_device(h);
  hmc_adapt_begin(h, target_accept);
  PYB_CATCH
}

int pyb_hmc_adapt_end(pyb_handle* h) {
  PYB_TRY
  PYB_REQUIRE(h, PYB_ERR_INVALID, "NULL handle");
  use_device(h);
  hmc_adapt_end(h);
  PYB_CATCH
}

int pyb_hmc_step_sizes(pyb_handle* h, double* eps_out) {
  PYB_TRY
  PYB_REQUIRE(h, PYB_ERR_INVALID, "NULL handle");
  use_device(h);
  hmc_step_sizes(h, eps_out);
  PYB_CATCH
}

int pyb_hmc_set_step_sizes(pyb_handle* h, const double* eps) {
  PYB_TRY
  PYB_REQUIRE(h, PYB_ERR_INVALID, "NULL handle");
  use_device(h);
  hmc_set_step_sizes(h, eps);
  PYB_CATCH
}

int pyb_hmc_set_temperatures(pyb_handle* h, const double* beta, int32_t R) {
  PYB_TRY
  PYB_REQUIRE(h, PYB_ERR_INVALID, "NULL handle");
  use_device(h);
  hmc_set_temperatures(h, beta, R);
  PYB_CATCH
}

int pyb_hmc_tempering_stats(pyb_handle* h, int64_t* rung_accepted, int64_t* rung_total, int64_t* swap_attempted,
                            int64_t* swap_accepted) {
  PYB_TRY
  PYB_REQUIRE(h, PYB_ERR_INVALID, "NULL handle");
  use_device(h);
  hmc_tempering_stats(h, rung_accepted, rung_total, swap_attempted, swap_accepted);
  PYB_CATCH
}

int pyb_hmc_last_swaps(pyb_handle* h, float* log_r, int32_t* swapped) {
  PYB_TRY
  PYB_REQUIRE(h, PYB_ERR_INVALID, "NULL handle");
  use_device(h);
  hmc_last_swaps(h, log_r, swapped);
  PYB_CATCH
}

int pyb_hmc_track_predictive(pyb_handle* h, const float* x, int64_t Nt, const int32_t* y) {
  PYB_TRY
  PYB_REQUIRE(h, PYB_ERR_INVALID, "NULL handle");
  use_device(h);
  if (!x) {
    PYB_CUDA(cudaStreamSynchronize(h->stream));
    hmc_track_stop(h);
  } else {
    hmc_track_start(h, x, Nt, y);
  }
  PYB_CATCH
}

int pyb_hmc_predictive_sums(pyb_handle* h, double* sums_out, double* s2_out, int64_t* n_draws_out) {
  PYB_TRY
  PYB_REQUIRE(h && sums_out, PYB_ERR_INVALID, "NULL argument");
  use_device(h);
  hmc_track_sums(h, sums_out, s2_out, n_draws_out);
  PYB_CATCH
}

int pyb_hmc_predictive_finish(pyb_handle* h, const double* sums, const double* s2, int64_t n_chains, int64_t n_draws,
                              int32_t uq_semantics, double divisor, float* mean_out, float* var_out, float* rhat_out,
                              float* total_out, float* aleatoric_out, float* epistemic_out) {
  PYB_TRY
  PYB_REQUIRE(h, PYB_ERR_INVALID, "NULL handle");
  use_device(h);
  const bool want_uq = total_out || aleatoric_out || epistemic_out;
  if (want_uq)
    PYB_REQUIRE(uq_semantics == PYB_UQ_REFERENCE || uq_semantics == PYB_UQ_CANONICAL, PYB_ERR_INVALID, "bad semantics");
  UncertaintyReq uq{nullptr, uq_semantics == PYB_UQ_REFERENCE ? 1 : 0, divisor, total_out, aleatoric_out, epistemic_out};
  hmc_track_finish(h, sums, s2, n_chains, n_draws, want_uq ? &uq : nullptr, mean_out, var_out, rhat_out);
  PYB_CATCH
}

int pyb_hmc_track_params(pyb_handle* h, int64_t n_planned, int32_t batch) {
  PYB_TRY
  PYB_REQUIRE(h, PYB_ERR_INVALID, "NULL handle");
  use_device(h);
  if (n_planned == 0) {
    PYB_CUDA(cudaStreamSynchronize(h->stream));
    hmc_params_stop(h);
  } else {
    hmc_params_start(h, n_planned, batch);
  }
  PYB_CATCH
}

int pyb_hmc_param_sums(pyb_handle* h, double* sums_out, int64_t* n_draws_out) {
  PYB_TRY
  PYB_REQUIRE(h && sums_out, PYB_ERR_INVALID, "NULL argument");
  use_device(h);
  hmc_params_sums(h, sums_out, n_draws_out);
  PYB_CATCH
}

int pyb_hmc_param_finish(pyb_handle* h, const double* sums, int64_t n_chains, int64_t n_draws, int64_t n_planned,
                         int32_t batch, double* mean_out, double* sd_out, double* rhat_out, double* ess_out,
                         double* mcse_out) {
  PYB_TRY
  PYB_REQUIRE(h, PYB_ERR_INVALID, "NULL handle");
  use_device(h);
  hmc_params_finish(h, sums, n_chains, n_draws, n_planned, batch, mean_out, sd_out, rhat_out, ess_out, mcse_out);
  PYB_CATCH
}

int pyb_svgd_init(pyb_handle* h, int64_t S, int64_t offset, double lr, int32_t sem, const double* p0) {
  PYB_TRY
  PYB_REQUIRE(h, PYB_ERR_INVALID, "NULL handle");
  use_device(h);
  svgd_init(h, S, offset, lr, sem, p0);
  PYB_CATCH
}

int pyb_svgd_step(pyb_handle* h, const int32_t* idx, int64_t B, double* loss_out) {
  PYB_TRY
  PYB_REQUIRE(h, PYB_ERR_INVALID, "NULL handle");
  use_device(h);
  if (idx)
    for (int64_t i = 0; i < B; ++i)
      PYB_REQUIRE(idx[i] >= 0 && idx[i] < h->N, PYB_ERR_INVALID, "batch index out of range");
  svgd_step(h, idx, B, loss_out);
  PYB_CATCH
}

int pyb_svgd_phi(pyb_handle* h, const double* X, const float* G, int64_t S, int32_t sem, float* phi, double* h_out) {
  PYB_TRY
  PYB_REQUIRE(h && X && G && phi, PYB_ERR_INVALID, "NULL argument");
  PYB_REQUIRE(sem == PYB_SVGD_REFERENCE_LIVE || sem == PYB_SVGD_CANONICAL_MEDIAN, PYB_ERR_INVALID, "bad semantics");
  use_device(h);
  svgd_phi(h, X, G, S, sem, phi, h_out);
  PYB_CATCH
}

int pyb_svgd_set_validation(pyb_handle* h, const float* X, const void* y, int64_t N) {
  PYB_TRY
  PYB_REQUIRE(h, PYB_ERR_INVALID, "NULL handle");
  use_device(h);
  svgd_set_validation(h, X, y, N);
  PYB_CATCH
}

int pyb_svgd_validation_loss(pyb_handle* h, double* mean_loss_out, float* per_particle_out) {
  PYB_TRY
  PYB_REQUIRE(h, PYB_ERR_INVALID, "NULL handle");
  use_device(h);
  svgd_validation_loss(h, mean_loss_out, per_particle_out);
  PYB_CATCH
}

__global__ void k_f32_to_f64(const float* a, double* b, int64_t n) {
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x)
    b[i] = (double)a[i];
}

int pyb_svgd_get_particles(pyb_handle* h, double* out) {
  PYB_TRY
  PYB_REQUIRE(h && out, PYB_ERR_INVALID, "NULL argument");
  SvgdState& sv = h->svgd;
  PYB_REQUIRE(sv.inited, PYB_ERR_STATE, "pyb_svgd_init must be called first");
  use_device(h);
  int64_t n = sv.S * h->model.P;
  DevBuf<double> tmp;
  tmp.alloc(n);
  k_f32_to_f64<<<(unsigned)((n + 255) / 256 > 4096 ? 4096 : (n + 255) / 256), 256, 0, h->stream>>>(sv.theta.p, tmp.p, n);
  count_launch(h);
  PYB_CUDA(cudaMemcpyAsync(out, tmp.p, n * sizeof(double), cudaMemcpyDeviceToHost, h->stream));
  PYB_CUDA(cudaStreamSynchronize(h->stream));
  PYB_CATCH
}

int pyb_svgd_set_comm(pyb_handle* h, int32_t rank, int32_t world, const void* id) {
  PYB_TRY
  PYB_REQUIRE(h, PYB_ERR_INVALID, "NULL handle");
  PYB_REQUIRE(world >= 1 && rank >= 0 && rank < world, PYB_ERR_INVALID, "bad rank/world");
  use_device(h);
  svgd_p2p_release(h);
  if (h->svgd.nccl_comm3) { nccl_comm_destroy(h->svgd.nccl_comm3); h->svgd.nccl_comm3 = nullptr; }
  if (h->svgd.nccl_comm2) { nccl_comm_destroy(h->svgd.nccl_comm2); h->svgd.nccl_comm2 = nullptr; }
  if (h->svgd.nccl_comm) { nccl_comm_destroy(h->svgd.nccl_comm); h->svgd.nccl_comm = nullptr; }
  if (world > 1) {
    PYB_REQUIRE(id != nullptr, PYB_ERR_INVALID, "nccl unique id is NULL");
    h->svgd.nccl_comm = nccl_comm_init(rank, world, id);
  }
  h->svgd.rank = rank; h->svgd.world = world;
  PYB_CATCH
}

int pyb_set_comm(pyb_handle* h, int32_t rank, int32_t world, const void* id) { return pyb_svgd_set_comm(h, rank, world, id); }

int pyb_nccl_unique_id(void* out_128) {
  PYB_TRY
  PYB_REQUIRE(out_128, PYB_ERR_INVALID, "NULL argument");
  nccl_unique_id(out_128);
  PYB_CATCH
}

int pyb_sg_init(pyb_handle* h, int64_t S, int64_t chain_offset, int32_t kind, int32_t k_dev, int32_t frequency,
                const float* theta0, int32_t theta0_rows) {
  PYB_TRY
  PYB_REQUIRE(h, PYB_ERR_INVALID, "NULL handle");
  use_device(h);
  sg_init(h, S, chain_offset, kind, k_dev, frequency, theta0, theta0_rows);
  PYB_CATCH
}

int pyb_sg_step(pyb_handle* h, const int32_t* idx, int64_t B, double lr, const float* noise, float* loss_out,
                double* mean_loss_out) {
  PYB_TRY
  PYB_REQUIRE(h, PYB_ERR_INVALID, "NULL handle");
  use_device(h);
  if (idx)
    for (int64_t i = 0; i < B; ++i)
      PYB_REQUIRE(idx[i] >= 0 && idx[i] < h->N, PYB_ERR_INVALID, "batch index out of range");
  sg_step(h, idx, B, lr, noise, loss_out, mean_loss_out);
  PYB_CATCH
}

int pyb_sg_get(pyb_handle* h, float* theta, float* mean, float* sq_mean, float* dev, int32_t* n_cols, int64_t* n_steps) {
  PYB_TRY
  PYB_REQUIRE(h, PYB_ERR_INVALID, "NULL handle");
  use_device(h);
  sg_get(h, theta, mean, sq_mean, dev, n_cols, n_steps);
  PYB_CATCH
}

int pyb_predict(pyb_handle* h, const float* W, int64_t n, const float* weight, const float* x, int64_t Nt, float* mean,
                float* var, float* all) {
  PYB_TRY
  PYB_REQUIRE(h, PYB_ERR_INVALID, "NULL handle");
  use_device(h);
  predict(h, W, n, weight, x, Nt, mean, var, all);
  PYB_CATCH
}

int pyb_predict_uncertainty(pyb_handle* h, const float* W, int64_t n, const float* weight, const float* x, int64_t Nt,
                            const int32_t* y, int32_t semantics, double divisor, float* total_out,
                            float* aleatoric_out, float* epistemic_out, float* mean_out) {
  PYB_TRY
  PYB_REQUIRE(h, PYB_ERR_INVALID, "NULL handle");
  use_device(h);
  PYB_REQUIRE(semantics == PYB_UQ_REFERENCE || semantics == PYB_UQ_CANONICAL, PYB_ERR_INVALID, "bad semantics");
  UncertaintyReq uq{y, semantics == PYB_UQ_REFERENCE ? 1 : 0, divisor, total_out, aleatoric_out, epistemic_out};
  predict(h, W, n, weight, x, Nt, mean_out, nullptr, nullptr, &uq);
  PYB_CATCH
}

int pyb_buffer_create(pyb_handle* h, const void* host_or_null, int64_t bytes, void** dev_out) {
  PYB_TRY
  PYB_REQUIRE(h && dev_out && bytes > 0, PYB_ERR_INVALID, "bad arguments");
  use_device(h);
  void* d = nullptr;
  PYB_CUDA(cudaMalloc(&d, (size_t)bytes));
  if (host_or_null) {
    cudaError_t e = cudaMemcpyAsync(d, host_or_null, (size_t)bytes, cudaMemcpyDefault, h->stream);
    if (e == cudaSuccess) e = cudaStreamSynchronize(h->stream);
    if (e != cudaSuccess) { cudaFree(d); PYB_CUDA(e); }
  }
  *dev_out = d;
  PYB_CATCH
}

int pyb_buffer_destroy(pyb_handle* h, void* dev) {
  PYB_TRY
  PYB_REQUIRE(h, PYB_ERR_INVALID, "NULL handle");
  use_device(h);
  if (dev) {
    PYB_CUDA(cudaStreamSynchronize(h->stream));
    PYB_CUDA(cudaFree(dev));
  }
  PYB_CATCH
}

int pyb_gather_rows(pyb_handle* h, const float* src, const int64_t* idx, int64_t n, int64_t row_len, float* dst) {
  PYB_TRY
  PYB_REQUIRE(h && src && idx && dst && n > 0 && row_len > 0, PYB_ERR_INVALID, "bad arguments");
  use_device(h);
  PYB_CUDA(cudaDeviceSynchronize());      // src / dst are caller-owned device buffers (header: "device pointers")
  gather_rows_f32(h, src, idx, n, row_len, dst);
  PYB_CATCH
}

}  // extern "C"
