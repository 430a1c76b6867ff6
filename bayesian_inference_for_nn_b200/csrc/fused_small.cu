// fused_small.cu — host side of the small-width path (kernels: fused_small.cuh, instantiated in fused_small_d*.cu)
#include "fused_small.cuh"

namespace pyb {

bool fused_small_supported(pyb_handle* h) {
  const Model& m = h->model;
  if (m.n_layers != 2 || !h->have_data) return false;
  const LayerDesc& L1 = m.layer[0];
  const LayerDesc& L2 = m.layer[1];
  if (!L1.use_bias || !L2.use_bias) return false;
  if (L1.fan_in < 1 || L1.fan_in > 4 || L2.fan_out < 1 || L2.fan_out > 4) return false;
  if (L1.fan_out > FS_HMAX || L1.act == PYB_ACT_SOFTMAX) return false;
  if (fs_smem_bytes(h) > 200 * 1024) return false;
  return true;
}

static void fs_dispatch(pyb_handle* h, const FsParams& p, int64_t S, bool hmc) {
  const int D = h->model.layer[0].fan_in;
  const double flops = 1.0;  // roofline for this path is reported per grad-eval by bench/tests, not per launch
  prof_begin(h);
  switch (D) {
    case 1: fs_launch_d1(h, p, S, hmc); break;
    case 2: fs_launch_d2(h, p, S, hmc); break;
    case 3: fs_launch_d3(h, p, S, hmc); break;
    case 4: fs_launch_d4(h, p, S, hmc); break;
    default: throw Error(PYB_ERR_UNSUPPORTED, "fused small path: unsupported input width");
  }
  prof_end(h, flops);
}

static FsParams fs_base(pyb_handle* h) {
  const Model& m = h->model;
  FsParams p = {};
  p.N = (int)h->N; p.H = m.layer[0].fan_out; p.act1 = m.layer[0].act; p.out_act = m.layer[1].act;
  p.loss_kind = h->loss_kind; p.P = m.P;
  p.w1_off = m.layer[0].w_off; p.b1_off = m.layer[0].b_off; p.w2_off = m.layer[1].w_off; p.b2_off = m.layer[1].b_off;
  p.X = h->X.p; p.y_i = h->y_i.p; p.y_f = h->y_f.p; p.mu = h->mu.p; p.inv_var = h->inv_var.p;
  p.n_train = (float)h->n_train;
  return p;
}

void fused_small_eval(pyb_handle* h, const float* theta, int64_t S, float scale, float* loss, float* grad) {
  FsParams p = fs_base(h);
  p.theta = theta; p.loss_out = loss; p.grad_out = grad; p.scale = scale;
  fs_dispatch(h, p, S, false);
  PYB_CUDA(cudaGetLastError());
}

// the same on an arbitrary device-resident batch of at most h->N rows (minibatches gathered from the resident dataset:
// SVGD / SGLD / SWAG steps); the shared-memory plan is the one sized for the full dataset
void fused_small_eval_on(pyb_handle* h, const float* theta, int64_t S, const float* Xb, const int32_t* yb_i,
                         const float* yb_f, int64_t Nb, float scale, float* loss, float* grad) {
  PYB_REQUIRE(Nb > 0 && Nb <= h->N, PYB_ERR_INVALID, "fused small path: batch larger than the resident dataset");
  FsParams p = fs_base(h);
  p.X = Xb; p.y_i = yb_i; p.y_f = yb_f; p.N = (int)Nb;
  p.theta = theta; p.loss_out = loss; p.grad_out = grad; p.scale = scale;
  fs_dispatch(h, p, S, false);
  PYB_CUDA(cudaGetLastError());
}

// one HMC iteration for all chains in ONE launch (sampler.cu records samples afterwards)
void fused_small_hmc_iteration(pyb_handle* h, bool burning) {
  HmcState& st = h->hmc;
  FsParams p = fs_base(h);
  p.q = st.q.p; p.p = st.p.p; p.q0 = st.q0.p;
  p.inj_p = st.have_inj_p ? st.inj_p.p : nullptr;
  p.inj_u = st.have_inj_u ? st.inj_u.p : nullptr;
  const StepCoef c = step_coef(st.eps, st.m);
  p.eps = c.eps; p.half_eps = c.half; p.drift = c.drift;
  p.step = st.step.p; p.m = st.m;
  p.da = st.adapting ? st.da.p : nullptr; p.da_target = st.adapt_target; p.da_t = st.adapt_t;
  p.beta = st.R ? st.beta.p : nullptr;
  p.stdv = (st.semantics == PYB_HMC_REFERENCE) ? (float)st.m : (float)sqrt(st.m);
  p.inv2m = (float)(1.0 / (2.0 * st.m));
  p.prior_const = (float)h->prior_const;
  p.L = st.L; p.semantics = st.semantics; p.burning = burning ? 1 : 0;
  p.seed = h->seed; p.iter = (uint32_t)st.iter; p.chain_offset = st.chain_offset;
  // few chains: spread each over a cluster (the row ranges must stay worth a CTA: >= 64 rows each)
  p.cluster = 1;
  if (h->opt_fs_cluster)
    for (int c = 8; c >= 2; c >>= 1)
      if (st.S * c <= h->sm_count && h->N / c >= 64) { p.cluster = c; break; }
  h->fs_cluster_used = p.cluster;
  p.U0 = st.U0.p; p.U1 = st.U1.p; p.K0 = st.K0.p; p.K1 = st.K1.p; p.log_alpha = st.log_alpha.p;
  p.ret_loss = st.ret_loss.p; p.accepted = st.accepted.p; p.counters = st.counters.p; p.loss_sum = st.loss_sum.p;
  fs_dispatch(h, p, st.S, true);
}

}  // namespace pyb
