// a11 leave-one-out evaluation: warp-level top-k over each user's candidate scores and the
// HR / NDCG of the held-out item (candidate 0).  Replaces torch.topk + torch.take + the numpy
// membership test of reference src/training/metrics.py:12-23 (one warp per user instead of one
// forward + two host syncs per user).
#include <math.h>

#include "common.cuh"
#include "tile_params.cuh"

namespace {

constexpr int kThreads = 256;
constexpr int kWarps = kThreads / 32;
constexpr int kMaxPerLane = 32;  // C <= 1024

// Order: larger score first; equal scores (-0.0 == +0.0): lower candidate index first.  NaN is not a
// candidate: it is marked taken when loaded, so `better` only ever compares numbers (the order of
// ncf_topk_rows).  A NaN in the order would break it: every comparison with NaN is false.
__device__ __forceinline__ bool better(float v, int i, float bv, int bi) {
  return (v > bv) || (v == bv && i < bi);
}

__global__ void __launch_bounds__(kThreads) eval_rank_kernel(const float* __restrict__ scores,
                                                             int64_t n, int C, int k,
                                                             uint8_t* __restrict__ hit,
                                                             int32_t* __restrict__ rank,
                                                             float* __restrict__ ndcg,
                                                             int32_t* __restrict__ topk_idx) {
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const int64_t nw = (int64_t)gridDim.x * kWarps;
  for (int64_t u = (int64_t)blockIdx.x * kWarps + warp; u < n; u += nw) {
    const float* s = scores + u * C;
    const int nq = (C + 31) >> 5;
    float v[kMaxPerLane];
    uint32_t taken = 0;
#pragma unroll
    for (int q = 0; q < kMaxPerLane; ++q) {
      const int c = lane + 32 * q;
      v[q] = (q < nq && c < C) ? s[c] : 0.f;
      if (c >= C || v[q] != v[q]) taken |= (1u << q);
    }
    int my_rank = -1;
    for (int j = 0; j < k; ++j) {
      float bv = 0.f;
      int bi = 0x7fffffff;
#pragma unroll
      for (int q = 0; q < kMaxPerLane; ++q) {
        const int c = lane + 32 * q;
        if (q < nq && !(taken >> q & 1u) && (bi == 0x7fffffff || better(v[q], c, bv, bi))) { bv = v[q]; bi = c; }
      }
#pragma unroll
      for (int o = 16; o > 0; o >>= 1) {
        const float ov = __shfl_xor_sync(0xffffffffu, bv, o);
        const int oi = __shfl_xor_sync(0xffffffffu, bi, o);
        if (oi != 0x7fffffff && (bi == 0x7fffffff || better(ov, oi, bv, bi))) { bv = ov; bi = oi; }
      }
      if (bi == 0x7fffffff) {  // fewer than k candidates in the row (warp-uniform): pad with -1
        if (lane == 0 && topk_idx != nullptr)
          for (int jj = j; jj < k; ++jj) topk_idx[u * k + jj] = -1;
        break;
      }
      if ((bi & 31) == lane) taken |= 1u << (bi >> 5);
      if (bi == 0) my_rank = j;
      if (lane == 0 && topk_idx != nullptr) topk_idx[u * k + j] = bi;
    }
    if (lane == 0) {
      if (hit) hit[u] = my_rank >= 0 ? 1 : 0;
      if (rank) rank[u] = my_rank;
      if (ndcg) ndcg[u] = my_rank >= 0 ? 1.f / log2f((float)(my_rank + 2)) : 0.f;
    }
  }
}

}  // namespace

extern "C" int ncf_eval_rank(const float* scores, int64_t n, int32_t C, int32_t k, uint8_t* hit,
                             int32_t* rank, float* ndcg, int32_t* topk_idx, void* stream) {
  NCF_REQUIRE(n >= 0, "ncf_eval_rank: negative n");
  NCF_REQUIRE(C >= 1 && C <= 32 * kMaxPerLane, "ncf_eval_rank: C=%d outside [1,1024]", C);
  NCF_REQUIRE(k >= 1 && k <= C, "ncf_eval_rank: k=%d outside [1,C=%d]", k, C);
  if (n == 0) return NCF_OK;
  NCF_REQUIRE(scores != nullptr, "ncf_eval_rank: scores is NULL");
  int64_t blocks = (n + kWarps - 1) / kWarps;
  const int64_t cap = (int64_t)ncf::num_sms() * 8;
  if (blocks > cap) blocks = cap;
  eval_rank_kernel<<<(int)blocks, kThreads, 0, (cudaStream_t)stream>>>(scores, n, C, k, hit, rank,
                                                                      ndcg, topk_idx);
  NCF_LAUNCH_CHECK("eval_rank_kernel");
  return NCF_OK;
}

// workspace = [scores n*C floats (used only when scores_out is NULL)] [forward workspace]
extern "C" int64_t ncf_eval_workspace_bytes(const NcfModel* m, int64_t n, int32_t C) {
  if (n < 0 || C < 1) return -1;
  // user_div = 0 bounds the call's user_div = C: for C <= 1024 the tcgen05 sub-batch floor(262144 / C) * C <= 262144
  const int64_t fw = ncf_forward_workspace_bytes(m, n * C);
  if (fw < 0) return -1;
  return ncf::align_up(n * C * 4, 256) + fw + 256;
}

extern "C" int ncf_eval_users(const NcfModel* m, const int64_t* users, const int64_t* cands,
                              int64_t n, int32_t C, int32_t k, uint8_t* hit, int32_t* rank,
                              float* ndcg, int32_t* topk_idx, float* scores_out, void* workspace,
                              int64_t workspace_bytes, void* stream) {
  int rc = ncf::validate_model(m);
  if (rc != NCF_OK) return rc;
  NCF_REQUIRE(n >= 0, "ncf_eval_users: negative n");
  NCF_REQUIRE(C >= 1 && C <= 32 * kMaxPerLane, "ncf_eval_users: C=%d outside [1,1024]", C);
  NCF_REQUIRE(k >= 1 && k <= C, "ncf_eval_users: k=%d outside [1,C=%d]", k, C);
  if (n == 0) return NCF_OK;
  NCF_REQUIRE(users && cands, "ncf_eval_users: null pointer");
  if (!workspace || workspace_bytes < ncf_eval_workspace_bytes(m, n, C)) {
    ncf::set_error("ncf_eval_users: workspace too small");
    return NCF_ERR_WORKSPACE;
  }
  float* scores = scores_out ? scores_out : (float*)workspace;
  char* fw = (char*)workspace + ncf::align_up(n * C * 4, 256);
  const int64_t fw_bytes = workspace_bytes - ncf::align_up(n * C * 4, 256);
  TileParams p{};
  ncf::fill_model_params(p, m);
  p.user = users;
  p.user_div = C;
  p.item = cands;
  p.B = n * C;
  p.invB = 1.f;
  p.logits = scores;
  rc = ncf::forward_dispatch(p, m, fw, fw_bytes, (cudaStream_t)stream);
  if (rc != NCF_OK) return rc;
  return ncf_eval_rank(scores, n, C, k, hit, rank, ndcg, topk_idx, stream);
}
