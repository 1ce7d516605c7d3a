// C-ABI entry points for the forward pass, the loss and the fused training step.
#include <algorithm>

#include "common.cuh"
#include "tile_params.cuh"

namespace {

__global__ void loss_grad_kernel(const float* __restrict__ logits, const float* __restrict__ label,
                                 const float* __restrict__ teacher, float alpha, int64_t B,
                                 float invB, double* __restrict__ loss_accum,
                                 float* __restrict__ dlogit) {
  float ls = 0.f;
  for (int64_t b = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; b < B;
       b += (int64_t)gridDim.x * blockDim.x) {
    float t = 0.f;
    if (teacher != nullptr) t = teacher[b];
    const SampleLoss r = sample_loss(logits[b], label[b], teacher != nullptr, t, alpha, invB);
    ls += r.loss;
    if (dlogit != nullptr) dlogit[b] = r.dlogit;
  }
  __shared__ float part[32];
  ls = warp_sum(ls);
  if ((threadIdx.x & 31) == 0) part[threadIdx.x >> 5] = ls;
  __syncthreads();
  if (threadIdx.x < 32) {
    float v = (threadIdx.x < (blockDim.x >> 5)) ? part[threadIdx.x] : 0.f;
    v = warp_sum(v);
    if (threadIdx.x == 0 && loss_accum != nullptr) atomicAdd(loss_accum, (double)v * (double)invB);
  }
}

int64_t scratch_floats(const NcfModel* m, int64_t B) {
  if (m->model_type == NCF_GMF) return 0;
  ncf::TowerShape ts = ncf::make_tower_shape(m->model_type, m->factor_num, m->num_layers);
  int64_t n = 0;
  for (int k = 1; k < ts.L; ++k) n += B * ts.width[k];   // act[k]
  for (int k = 1; k <= ts.L; ++k) n += B * ts.width[k];  // delta[k]
  return n;
}

}  // namespace

namespace ncf {

// Forward over p.B samples on whichever tile kernel the shape is eligible for.  The tensor-pipe
// path needs mma_split_floats(p) floats of workspace for the pre-split weights.
int forward_dispatch(TileParams& p, const NcfModel* m, void* workspace, int64_t workspace_bytes,
                     cudaStream_t st) {
  if (small_eligible(p)) {
    g_tile_path = 4;
    return launch_small_forward(p, st);
  }
  if (umma_eligible(p)) {
    const int64_t need = umma_forward_workspace_floats(p, p.B) * 4;
    if (!workspace || workspace_bytes < need) {
      set_error("forward: workspace too small (%lld < %lld)", (long long)workspace_bytes, (long long)need);
      return NCF_ERR_WORKSPACE;
    }
    g_tile_path = 3;
    return launch_umma_forward(p, tower_passes(m), (float*)workspace, st);
  }
  if (wide_eligible(p)) {
    const int64_t need = wide_workspace_floats(p, p.B) * 4;
    if (!workspace || workspace_bytes < need) {
      set_error("forward: workspace too small (%lld < %lld)", (long long)workspace_bytes, (long long)need);
      return NCF_ERR_WORKSPACE;
    }
    g_tile_path = 5;
    return launch_wide_forward(p, (float*)workspace, st);
  }
  g_tile_path = mma_tile_rows(p) == 0 ? 1 : 2;
  if (mma_tile_rows(p) == 0) return launch_generic_forward(p, st);
  const int64_t need = mma_split_floats(p) * 4;
  if (!workspace || workspace_bytes < need) {
    set_error("forward: workspace too small (%lld < %lld)", (long long)workspace_bytes, (long long)need);
    return NCF_ERR_WORKSPACE;
  }
  int rc = mma_prepare_weights(p, (float*)workspace, st);
  if (rc != NCF_OK) return rc;
  return launch_mma_forward(p, tower_passes(m), st);
}

// Workspace of forward_dispatch for any batch up to p.B (with p.user_div as the caller will pass it).
int64_t forward_workspace_bytes(const TileParams& p) {
  const int64_t B = p.B;
  int64_t bytes = mma_tile_rows(p) ? align_up(mma_split_floats(p) * 4, 256) : 0;
  if (umma_eligible(p))
    bytes = std::max(bytes, align_up(umma_forward_workspace_floats(p, B) * 4, 256) + 256);
  // any batch up to B may be passed with a workspace of this size: cover the small-batch path as well
  TileParams ps = p;
  ps.B = std::min<int64_t>(B, 2048);
  if (ps.B > 0 && wide_eligible(ps))
    bytes = std::max(bytes, align_up(wide_workspace_floats(ps, ps.B) * 4, 256));
  return bytes;
}

}  // namespace ncf

extern "C" int64_t ncf_forward_workspace_bytes(const NcfModel* m, int64_t B) {
  if (ncf::validate_model(m) != NCF_OK) return -1;
  TileParams p{};
  ncf::fill_model_params(p, m);
  p.B = B;
  return ncf::forward_workspace_bytes(p);
}

extern "C" int ncf_forward(const NcfModel* m, const int64_t* user, const int64_t* item, int64_t B,
                           float* logits, void* workspace, int64_t workspace_bytes, void* stream) {
  int rc = ncf::validate_model(m);
  if (rc != NCF_OK) return rc;
  NCF_REQUIRE(B >= 0, "ncf_forward: negative batch");
  if (B == 0) return NCF_OK;
  NCF_REQUIRE(user && item && logits, "ncf_forward: null pointer");
  TileParams p{};
  ncf::fill_model_params(p, m);
  p.user = user;
  p.item = item;
  p.B = B;
  p.invB = 1.f / (float)B;
  p.logits = logits;
  return ncf::forward_dispatch(p, m, workspace, workspace_bytes, (cudaStream_t)stream);
}

extern "C" int ncf_loss_grad(const float* logits, const float* label, const float* teacher_logits,
                             float alpha, int64_t B, double* loss_accum, float* dlogit,
                             void* stream) {
  NCF_REQUIRE(B > 0, "ncf_loss_grad: empty batch");
  NCF_REQUIRE(logits && label, "ncf_loss_grad: null pointer");
  int64_t blocks = (B + 255) / 256;
  if (blocks > 4 * ncf::num_sms()) blocks = 4 * ncf::num_sms();
  loss_grad_kernel<<<(int)blocks, 256, 0, (cudaStream_t)stream>>>(
      logits, label, teacher_logits, alpha, B, 1.f / (float)B, loss_accum, dlogit);
  NCF_LAUNCH_CHECK("loss_grad_kernel");
  return NCF_OK;
}

extern "C" int64_t ncf_train_workspace_bytes(const NcfModel* m, int64_t B) {
  if (ncf::validate_model(m) != NCF_OK || B < 0) return -1;
  TileParams p{};
  ncf::fill_model_params(p, m);
  p.B = B;
  int64_t floats = ncf::mma_tile_rows(p) ? ncf::mma_split_floats(p) : scratch_floats(m, B);
  if (ncf::umma_eligible(p)) floats = std::max(floats, ncf::umma_train_workspace_floats(p, B));
  return ncf::align_up(floats * 4, 256) + 256;
}

static int train_common(const NcfModel* m, const NcfGrads* g, const int64_t* user,
                        const int64_t* item, const float* label, const float* teacher_logits,
                        const float* dlogit_in, float alpha, int64_t B, double* loss_accum,
                        float* logits_out, void* workspace, int64_t workspace_bytes, void* stream,
                        int64_t B_norm = 0);

extern "C" int ncf_backward(const NcfModel* m, const NcfGrads* g, const int64_t* user,
                            const int64_t* item, const float* dlogit, int64_t B, void* workspace,
                            int64_t workspace_bytes, void* stream) {
  NCF_REQUIRE(dlogit != nullptr, "ncf_backward: dlogit is NULL");
  return train_common(m, g, user, item, nullptr, nullptr, dlogit, 1.f, B, nullptr, nullptr,
                      workspace, workspace_bytes, stream);
}

extern "C" int ncf_train_step_grads(const NcfModel* m, const NcfGrads* g, const int64_t* user,
                                    const int64_t* item, const float* label,
                                    const float* teacher_logits, float alpha, int64_t B,
                                    double* loss_accum, float* logits_out, void* workspace,
                                    int64_t workspace_bytes, void* stream) {
  NCF_REQUIRE(label && loss_accum, "ncf_train_step_grads: null pointer");
  return train_common(m, g, user, item, label, teacher_logits, nullptr, alpha, B, loss_accum,
                      logits_out, workspace, workspace_bytes, stream);
}

extern "C" int ncf_train_step_grads_norm(const NcfModel* m, const NcfGrads* g, const int64_t* user,
                                         const int64_t* item, const float* label,
                                         const float* teacher_logits, float alpha, int64_t B,
                                         int64_t B_norm, double* loss_accum, float* logits_out,
                                         void* workspace, int64_t workspace_bytes, void* stream) {
  NCF_REQUIRE(label && loss_accum, "ncf_train_step_grads_norm: null pointer");
  NCF_REQUIRE(B_norm >= B, "ncf_train_step_grads_norm: B_norm must be >= B");
  return train_common(m, g, user, item, label, teacher_logits, nullptr, alpha, B, loss_accum,
                      logits_out, workspace, workspace_bytes, stream, B_norm);
}

static int train_common(const NcfModel* m, const NcfGrads* g, const int64_t* user,
                        const int64_t* item, const float* label, const float* teacher_logits,
                        const float* dlogit_in, float alpha, int64_t B, double* loss_accum,
                        float* logits_out, void* workspace, int64_t workspace_bytes, void* stream,
                        int64_t B_norm) {
  int rc = ncf::validate_model(m);
  if (rc != NCF_OK) return rc;
  NCF_REQUIRE(B > 0, "ncf_train_step_grads: empty batch");
  NCF_REQUIRE(g && user && item, "ncf_train_step_grads: null pointer");
  NCF_REQUIRE(g->g_tower && g->user_flag && g->item_flag && g->user_list && g->item_list &&
                  g->touched_count,
              "ncf_train_step_grads: incomplete NcfGrads");
  if (m->model_type != NCF_MLP)
    NCF_REQUIRE(g->g_user_gmf && g->g_item_gmf, "ncf_train_step_grads: GMF grad buffers are NULL");
  if (m->model_type != NCF_GMF)
    NCF_REQUIRE(g->g_user_mlp && g->g_item_mlp, "ncf_train_step_grads: MLP grad buffers are NULL");
  const int64_t need = ncf_train_workspace_bytes(m, B);
  if (workspace_bytes < need || (need > 256 && !workspace)) {
    ncf::set_error("ncf_train_step_grads: workspace too small (%lld < %lld)",
                   (long long)workspace_bytes, (long long)need);
    return NCF_ERR_WORKSPACE;
  }
  TileParams p{};
  ncf::fill_model_params(p, m);
  ncf::fill_grad_params(p, g);
  p.user = user;
  p.item = item;
  p.label = label;
  p.teacher = teacher_logits;
  p.dlogit_in = dlogit_in;
  p.alpha = teacher_logits ? alpha : 1.f;
  p.B = B;
  p.invB = 1.f / (float)(B_norm > 0 ? B_norm : B);  // mean over the (global) batch
  p.logits = logits_out;
  p.loss_accum = loss_accum;
  if (ncf::small_eligible(p)) {
    ncf::g_tile_path = 4;
    rc = ncf::launch_small_train(p, (cudaStream_t)stream);
    if (rc != NCF_OK) return rc;
    return ncf::mark_embedding_grads_done((cudaStream_t)stream);
  }
  if (ncf::umma_eligible(p)) {
    ncf::g_tile_path = 3;
    return ncf::launch_umma_train(p, ncf::tower_passes(m), (float*)workspace, (cudaStream_t)stream);
  }
  ncf::g_tile_path = ncf::mma_tile_rows(p) != 0 ? 2 : 1;
  if (ncf::mma_tile_rows(p) != 0) {
    rc = ncf::mma_prepare_weights(p, (float*)workspace, (cudaStream_t)stream);
    if (rc != NCF_OK) return rc;
    rc = ncf::launch_mma_train(p, ncf::tower_passes(m), (cudaStream_t)stream);
    if (rc != NCF_OK) return rc;
    return ncf::mark_embedding_grads_done((cudaStream_t)stream);
  }
  if (m->model_type != NCF_GMF) {
    float* ws = (float*)workspace;
    for (int k = 1; k < p.L; ++k) { p.act[k] = ws; ws += B * p.W[k]; }
    for (int k = 1; k <= p.L; ++k) { p.delta[k] = ws; ws += B * p.W[k]; }
  }
  rc = ncf::launch_generic_train(p, (cudaStream_t)stream);
  if (rc != NCF_OK) return rc;
  return ncf::mark_embedding_grads_done((cudaStream_t)stream);
}
