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

// tile_path below the thread-per-sample kernel.  The training query sizes for this path: the thread-per-sample
// kernel needs no workspace, and the query then does not depend on the weight alignment that kernel checks.
int tensor_path(const TileParams& p, bool train) {
  if (ncf::umma_eligible(p)) return 3;
  if (!train && ncf::wide_eligible(p)) return 5;
  return ncf::mma_tile_rows(p) != 0 ? 2 : 1;
}

int64_t train_workspace_bytes(const TileParams& p) {
  return ncf::align_up(ncf::tile_workspace_floats(tensor_path(p, true), p, p.B, true) * 4, 256) + 256;
}

// The one workspace rule of the forward and training entry points: a call that needs `need` > 0 bytes gets a
// non-NULL workspace of at least that size.
int check_workspace(const char* who, const void* workspace, int64_t workspace_bytes, int64_t need) {
  if (need > 0 && (!workspace || workspace_bytes < need)) {
    ncf::set_error("%s: workspace too small (%lld < %lld)", who, (long long)workspace_bytes, (long long)need);
    return NCF_ERR_WORKSPACE;
  }
  return NCF_OK;
}

}  // namespace

namespace ncf {

int tile_path(const TileParams& p, bool train) { return small_eligible(p) ? 4 : tensor_path(p, train); }

int64_t tile_workspace_floats(int path, const TileParams& p, int64_t B, bool train) {
  switch (path) {
    case 1: return train ? scratch_floats(p, B, true) : 0;  // the generic forward keeps its rows on chip
    case 2: return image_floats(p);
    // + 64: the scratch starts at the next 256-byte boundary after the images
    case 3: return image_floats(p) + scratch_floats(p, train ? B : std::min(B, forward_sub(p)), train) + 64;
    case 5: return wide_workspace_floats(p, B);
    default: return 0;
  }
}

int forward_dispatch(TileParams& p, const NcfModel* m, void* workspace, int64_t workspace_bytes,
                     cudaStream_t st) {
  const int path = tile_path(p, false);
  int rc = check_workspace("forward", workspace, workspace_bytes, tile_workspace_floats(path, p, p.B, false) * 4);
  if (rc != NCF_OK) return rc;
  g_tile_path = path;
  float* ws = (float*)workspace;
  switch (path) {
    case 4: return launch_small_forward(p, st);
    case 3: return launch_umma_forward(p, tower_passes(m), ws, st);
    case 5: return launch_wide_forward(p, ws, st);
    case 2:
      rc = mma_prepare_weights(p, ws, st);
      return rc != NCF_OK ? rc : launch_mma_forward(p, mma_tile_rows(p), tower_passes(m), st);
    default: return launch_generic_forward(p, st);
  }
}

// The most any batch up to p.B can need: each path that consumes workspace, at the largest batch its own rule
// admits (the order of tile_path is not applied, so the value is an upper bound).
int64_t forward_workspace_bytes(const TileParams& p) {
  int64_t bytes = 0;
  if (mma_tile_rows(p)) bytes = align_up(tile_workspace_floats(2, p, p.B, false) * 4, 256);
  if (umma_eligible(p))
    bytes = std::max(bytes, align_up(tile_workspace_floats(3, p, p.B, false) * 4, 256) + 256);
  TileParams ps = p;
  ps.B = std::min(p.B, kWideMaxB);
  if (wide_eligible(ps)) bytes = std::max(bytes, align_up(tile_workspace_floats(5, ps, ps.B, false) * 4, 256));
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
  return train_workspace_bytes(p);
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
  const int path = ncf::tile_path(p, true);
  rc = check_workspace("ncf_train_step_grads", workspace, workspace_bytes, train_workspace_bytes(p));
  if (rc != NCF_OK) return rc;
  ncf::g_tile_path = path;
  float* ws = (float*)workspace;
  const cudaStream_t st = (cudaStream_t)stream;
  switch (path) {
    case 4: rc = ncf::launch_small_train(p, st); break;
    case 3: return ncf::launch_umma_train(p, ncf::tower_passes(m), ws, st);  // marks the embedding grads itself
    case 2:
      rc = ncf::mma_prepare_weights(p, ws, st);
      if (rc == NCF_OK) rc = ncf::launch_mma_train(p, ncf::mma_tile_rows(p), ncf::tower_passes(m), st);
      break;
    default:
      ncf::carve_scratch(p, ws, B, true);
      rc = ncf::launch_generic_train(p, st);
  }
  if (rc != NCF_OK) return rc;
  return ncf::mark_embedding_grads_done(st);
}
