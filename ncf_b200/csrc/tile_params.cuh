// Kernel-argument block shared by the forward / training-step kernels.
#pragma once
#include "common.cuh"

struct TileParams {
  // model (device pointers)
  int type, f, d, L, predict_size;
  int W[NCF_MAX_LAYERS + 1];
  const float *eug, *eig, *eum, *eim;
  const float* w[NCF_MAX_LAYERS];
  const float* b[NCF_MAX_LAYERS];
  const float *pw, *pb;
  int64_t U, I;
  // batch
  const int64_t* user;
  const int64_t* item;
  int user_div;          // >0: sample b uses user[b / user_div] (evaluation: one user, C candidates)
  const float* label;    // NULL => inference
  const float* teacher;  // NULL => plain BCE
  const float* dlogit_in; // non-NULL => use this dloss/dlogit instead of evaluating the loss
  float alpha, invB;
  int64_t B;
  float* logits;         // nullable
  double* loss_accum;
  // gradients
  float *gug, *gig, *gum, *gim, *gt;
  int32_t *uflag, *iflag, *tcount;
  int64_t *ulist, *ilist;
  int64_t w_off[NCF_MAX_LAYERS], b_off[NCF_MAX_LAYERS], pw_off, pb_off;
  // HBM scratch of per-sample activations / deltas (generic training, tcgen05), laid out by carve_scratch
  float* act[NCF_MAX_LAYERS + 1];    // act[k],   k = 1..L-1 : [B, W[k]]
  float* delta[NCF_MAX_LAYERS + 1];  // delta[k], k = 1..L   : [B, W[k]]
  // (hi, lo) weight images of the mma.sync and tcgen05 paths, forward operand and transposed operand, laid out
  // by point_images
  float* wsplit_f[NCF_MAX_LAYERS];
  float* wsplit_b[NCF_MAX_LAYERS];
  // shared-memory layout (float offsets), filled by the launcher
  int smem_off[NCF_MAX_LAYERS + 1];
  int gmf_off, stage_off, misc_off;
};

namespace ncf {

inline void fill_model_params(TileParams& p, const NcfModel* m) {
  TowerShape ts = make_tower_shape(m->model_type, m->factor_num, m->num_layers);
  p.type = m->model_type;
  p.f = m->factor_num;
  p.d = m->mlp_dim;
  p.L = m->num_layers;
  p.predict_size = ts.predict_size;
  for (int k = 0; k <= p.L; ++k) p.W[k] = ts.width[k];
  p.eug = m->embed_user_gmf;
  p.eig = m->embed_item_gmf;
  p.eum = m->embed_user_mlp;
  p.eim = m->embed_item_mlp;
  for (int k = 0; k < p.L; ++k) {
    p.w[k] = m->mlp_w[k];
    p.b[k] = m->mlp_b[k];
    p.w_off[k] = ts.w_off[k];
    p.b_off[k] = ts.b_off[k];
  }
  p.pw = m->predict_w;
  p.pb = m->predict_b;
  p.pw_off = ts.pw_off;
  p.pb_off = ts.pb_off;
  p.U = m->user_num;
  p.I = m->item_num;
}

inline void fill_grad_params(TileParams& p, const NcfGrads* g) {
  p.gug = g->g_user_gmf;
  p.gig = g->g_item_gmf;
  p.gum = g->g_user_mlp;
  p.gim = g->g_item_mlp;
  p.gt = g->g_tower;
  p.uflag = g->user_flag;
  p.iflag = g->item_flag;
  p.ulist = g->user_list;
  p.ilist = g->item_list;
  p.tcount = g->touched_count;
}

// Workspace layouts shared by the tile paths.  Weight images: per layer k, 2 * W[k] * W[k+1] floats of
// forward operand, then as many of transposed operand.
inline int64_t image_floats(const TileParams& p) {
  int64_t n = 0;
  for (int k = 0; k < p.L; ++k) n += 2 * 2 * (int64_t)p.W[k] * p.W[k + 1];
  return n;
}
// points wsplit_f / wsplit_b into ws; returns the end of the images
inline float* point_images(TileParams& p, float* ws) {
  for (int k = 0; k < p.L; ++k) {
    const int64_t n = 2 * (int64_t)p.W[k] * p.W[k + 1];
    p.wsplit_f[k] = ws;
    p.wsplit_b[k] = ws + n;
    ws += 2 * n;
  }
  return ws;
}
// act[1..L-1] and, when training, delta[1..L] for B samples; GMF has no tower and no scratch
inline int64_t scratch_floats(const TileParams& p, int64_t B, bool train) {
  if (p.type == NCF_GMF) return 0;
  int64_t n = 0;
  for (int k = 1; k < p.L; ++k) n += B * p.W[k];
  if (train)
    for (int k = 1; k <= p.L; ++k) n += B * p.W[k];
  return n;
}
inline void carve_scratch(TileParams& p, float* ws, int64_t B, bool train) {
  if (p.type == NCF_GMF) return;
  for (int k = 1; k < p.L; ++k) { p.act[k] = ws; ws += B * p.W[k]; }
  if (train)
    for (int k = 1; k <= p.L; ++k) { p.delta[k] = ws; ws += B * p.W[k]; }
}

// The tile path of a forward (train = false) or training call, as ncf_last_tile_path() reports it: 4 the
// thread-per-sample kernel, 3 tcgen05, 5 the layer-per-launch forward (inference only), 2 mma.sync, 1 generic;
// the first in that order whose eligibility rule below admits p.  step.cu holds this order and nothing else
// restates it: the launchers and the workspace queries go through tile_path / tile_workspace_floats.
int tile_path(const TileParams& p, bool train);
// floats of workspace that `path` consumes for a call over B samples
int64_t tile_workspace_floats(int path, const TileParams& p, int64_t B, bool train);
// forward over p.B samples on tile_path(p, false), with the workspace checked against its need
int forward_dispatch(TileParams& p, const NcfModel* m, void* workspace, int64_t workspace_bytes, cudaStream_t st);
// workspace that serves forward_dispatch for every batch up to p.B (with p.user_div as the caller will pass it)
int64_t forward_workspace_bytes(const TileParams& p);

int launch_generic_forward(TileParams& p, cudaStream_t st);
int launch_generic_train(TileParams& p, cudaStream_t st);

// tensor-pipe path (tile_mma.cu): eligible when mma_tile_rows(p) != 0, the tile height (32 or 64)
int mma_tile_rows(const TileParams& p);
int mma_prepare_weights(TileParams& p, float* ws, cudaStream_t st);
int launch_mma_forward(TileParams& p, int tile_rows, int passes, cudaStream_t st);
int launch_mma_train(TileParams& p, int tile_rows, int passes, cudaStream_t st);
inline int tower_passes(const NcfModel* m) { return m->tower_math == NCF_MATH_TF32 ? 1 : 3; }

// narrow towers, one thread per sample on the FMA pipe (tile_small.cu): factor_num 8, 1..3 layers
bool small_eligible(const TileParams& p);
int launch_small_forward(TileParams& p, cudaStream_t st);
int launch_small_train(TileParams& p, cudaStream_t st);

// wide towers at small batches, forward only: one launch per layer over many CTAs (tile_wide.cu)
constexpr int64_t kWideMaxB = 2048;       // largest batch it takes
bool wide_eligible(const TileParams& p);  // reads p.B
int64_t wide_workspace_floats(const TileParams& p, int64_t B);
int launch_wide_forward(TileParams& p, float* ws, cudaStream_t st);

// tcgen05 path (tile_umma.cu): large batches, tower widths that are power-of-two multiples of 32
bool umma_eligible(const TileParams& p);  // reads p.B
int64_t forward_sub(const TileParams& p);  // rows of one inference sub-batch
int launch_umma_forward(TileParams& p, int passes, float* ws, cudaStream_t st);
int launch_umma_train(TileParams& p, int passes, float* ws, cudaStream_t st);

}  // namespace ncf
