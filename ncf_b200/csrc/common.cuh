// Shared helpers for the ncf_b200 kernels (sm_100a only).
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>
#include <stdio.h>
#include <string>

#include "../../include/ncf_b200.h"

namespace ncf {

void set_error(const char* fmt, ...);
int check_cuda(cudaError_t e, const char* what);
int num_sms();
// records "embedding-row gradients complete" on `st` (see ncf_wait_embedding_grads)
int mark_embedding_grads_done(cudaStream_t st);
// ncf_last_tile_path: 1 generic, 2 mma.sync, 3 tcgen05, 4 thread-per-sample, 5 layer-per-launch forward; chosen
// by ncf::tile_path (step.cu)
extern thread_local int g_tile_path;

#define NCF_REQUIRE(cond, ...)        \
  do {                                \
    if (!(cond)) {                    \
      ncf::set_error(__VA_ARGS__);    \
      return NCF_ERR_ARG;             \
    }                                 \
  } while (0)

#define NCF_CUDA(expr)                                        \
  do {                                                        \
    int _rc = ncf::check_cuda((expr), #expr);                 \
    if (_rc != NCF_OK) return _rc;                            \
  } while (0)

#define NCF_LAUNCH_CHECK(name) NCF_CUDA((cudaGetLastError()))

// Tower shape derived from (f, L): width[0] = f * 2^L (input), width[k+1] = width[k] / 2.
struct TowerShape {
  int L;
  int width[NCF_MAX_LAYERS + 1];
  int64_t w_off[NCF_MAX_LAYERS];  // offsets into the flat tower buffer
  int64_t b_off[NCF_MAX_LAYERS];
  int64_t pw_off, pb_off, total;
  int predict_size;
};

inline TowerShape make_tower_shape(int model_type, int f, int L) {
  TowerShape t{};
  t.L = L;
  t.width[0] = f << L;
  int64_t off = 0;
  for (int k = 0; k < L; ++k) {
    t.width[k + 1] = t.width[k] / 2;
    t.w_off[k] = off;
    off += (int64_t)t.width[k] * t.width[k + 1];
    t.b_off[k] = off;
    off += t.width[k + 1];
  }
  t.predict_size = (model_type == NCF_NEUMF) ? 2 * f : f;
  t.pw_off = off;
  off += t.predict_size;
  t.pb_off = off;
  off += 1;
  t.total = off;
  return t;
}

inline int64_t align_up(int64_t x, int64_t a) { return (x + a - 1) / a * a; }

int validate_model(const NcfModel* m);

}  // namespace ncf

// ---- device helpers ----------------------------------------------------------------------
__device__ __forceinline__ float warp_sum(float v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  return v;
}

__device__ __forceinline__ float4 ldg4(const float* p) {
  return __ldg(reinterpret_cast<const float4*>(p));
}

// Registers `row` in a touched list (the dedup the optimisers walk): the one thread that flips flag[row] from 0
// appends the row to `list`, whose length is *count.  Returns whether this thread won.
__device__ __forceinline__ bool claim_row(int32_t* flag, int64_t* list, int32_t* count, int64_t row) {
  if (atomicExch(&flag[row], 1) != 0) return false;
  list[atomicAdd(count, 1)] = row;
  return true;
}

// The per-sample training objective, defined once for every tile kernel and loss_grad_kernel (the KD
// objective of distill.cu is a different one): BCE-with-logits of logit x against label y, mixed with
// the squared distance to the teacher logit t when there is a teacher (alpha weights the BCE term).
// `loss` is the sample's term of the batch sum; `dlogit` is d(mean loss)/dx, i.e. already scaled by
// invB = 1 / batch size.
struct SampleLoss {
  float loss, dlogit;
};
__device__ __forceinline__ SampleLoss sample_loss(float x, float y, bool has_teacher, float t, float alpha,
                                                  float invB) {
  const float e = expf(-fabsf(x));
  const float bce = fmaxf(x, 0.f) - x * y + log1pf(e);
  const float sig = (x >= 0.f) ? 1.f / (1.f + e) : e / (1.f + e);
  if (!has_teacher) return {bce, (sig - y) * invB};
  const float df = x - t;
  return {alpha * bce + (1.f - alpha) * df * df, (alpha * (sig - y) + (1.f - alpha) * 2.f * df) * invB};
}

// 16-byte vector reduction into global memory (RED.E.ADD.F32x4 on sm_90+).
__device__ __forceinline__ void red_add4(float* p, float4 v) {
  asm volatile("red.global.add.v4.f32 [%0], {%1, %2, %3, %4};" ::"l"(p), "f"(v.x), "f"(v.y),
               "f"(v.z), "f"(v.w)
               : "memory");
}
