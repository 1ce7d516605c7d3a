// Full-catalog recommendation: exclusion of each user's seen items, per-row top-k selection over rows of
// up to millions of scores, and the pipeline that scores users against every item of the model
// (ncf::forward_dispatch, the kernels of the forward pass), masks and selects chunk by chunk.
//
// Selection order (the rule of ncf_eval_rank): larger score first, equal scores -> lower column first,
// -0.0 == +0.0, NaN = not a candidate.  Scores map to order-preserving uint32 keys (NaN -> 0, never a
// valid key); the k-th largest key is found by a radix select over 11/11/10-bit digits with shared-memory
// histograms, the keys above it and the lowest-column ties at it are collected in one more read of the
// row, and the <= 1024 survivors are bitonic-sorted in shared memory.  Each score is read four times,
// whatever k is.
#include <math.h>

#include <algorithm>

#include "common.cuh"
#include "tile_params.cuh"

namespace {

constexpr int kSelThreads = 256;
constexpr int kSelWarps = kSelThreads / 32;
constexpr int kMaxK = 1024;
constexpr int kBins = 2048;
constexpr int kMaskThreads = 128;
// one forward of ncf_recommend scores at most this many (user, item) pairs
constexpr int64_t kMaxChunkPairs = int64_t(1) << 28;

__device__ __forceinline__ uint32_t order_key(float v) {
  uint32_t b = __float_as_uint(v);
  if (v != v) return 0u;
  if (b == 0x80000000u) b = 0u;  // -0.0 == +0.0
  return (b & 0x80000000u) ? ~b : (b | 0x80000000u);
}

// Sum of v over the threads of the block with a higher index (a suffix scan, exclusive).  Every thread
// of the block must call it; `tot` is kSelWarps words of shared memory.
__device__ __forceinline__ uint32_t block_sum_above(uint32_t v, uint32_t* tot) {
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  uint32_t x = v;
#pragma unroll
  for (int o = 1; o < 32; o <<= 1) {
    const uint32_t y = __shfl_down_sync(0xffffffffu, x, o);
    if (lane + o < 32) x += y;
  }
  __syncthreads();  // tot of an earlier call has been read
  if (lane == 0) tot[warp] = x;
  __syncthreads();
  uint32_t above = x - v;
  for (int w = warp + 1; w < kSelWarps; ++w) above += tot[w];
  return above;
}

struct SelShared {
  uint32_t hist[kBins];
  unsigned long long cand[kMaxK];  // (key << 32) | (0x7fffffff - column): larger = better
  uint32_t tot[kSelWarps];
  uint32_t ties[2][kSelWarps];
  uint32_t bin, above, n_valid, n_gt;
  int32_t rank_part[kSelWarps];
  uint32_t target_key;
};

// Finds the digit bin that holds the `remaining`-th largest key of the histogram (nb bins, counted from the
// top) and how many keys lie in the bins above it.  Result in s.bin / s.above.
__device__ void pick_bin(SelShared& s, int nb, uint32_t remaining) {
  const int per = nb / kSelThreads;
  const int lo = threadIdx.x * per;
  uint32_t mine = 0;
  for (int b = 0; b < per; ++b) mine += s.hist[lo + b];
  uint32_t above = block_sum_above(mine, s.tot);
  for (int b = per - 1; b >= 0; --b) {
    const uint32_t h = s.hist[lo + b];
    if (above < remaining && above + h >= remaining) {
      s.bin = lo + b;
      s.above = above;
    }
    above += h;
  }
  __syncthreads();
}

__global__ void __launch_bounds__(kSelThreads) topk_rows_kernel(
    const float* __restrict__ scores, int64_t n, int64_t C, int k, const int64_t* __restrict__ target,
    int64_t* __restrict__ topk_item, float* __restrict__ topk_score, int32_t* __restrict__ target_rank) {
  __shared__ SelShared s;
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  for (int64_t r = blockIdx.x; r < n; r += gridDim.x) {
    const float* row = scores + r * C;
    int64_t tcol = -1;
    if (target != nullptr) {
      tcol = target[r];
      if (tcol < 0 || tcol >= C) tcol = -1;
    }
    if (tid == 0) s.target_key = tcol >= 0 ? order_key(row[tcol]) : 0u;

    // ---- radix select of the k-th largest key: digits [31:21], [20:10], [9:0] ----------------------------
    uint32_t prefix = 0, pmask = 0, remaining = 0, k_eff = 0;
#pragma unroll 1
    for (int pass = 0; pass < 3; ++pass) {
      const int shift = pass == 0 ? 21 : (pass == 1 ? 10 : 0);
      const int nb = pass == 2 ? 1024 : 2048;
      for (int b = tid; b < nb; b += kSelThreads) s.hist[b] = 0;
      __syncthreads();
      for (int64_t c = tid; c < C; c += kSelThreads) {
        const uint32_t key = order_key(__ldg(row + c));
        if (key != 0u && (key & pmask) == prefix) atomicAdd(&s.hist[(key >> shift) & (nb - 1)], 1u);
      }
      __syncthreads();
      if (pass == 0) {
        uint32_t mine = 0;
        for (int b = tid; b < nb; b += kSelThreads) mine += s.hist[b];
        const uint32_t total = block_sum_above(mine, s.tot) + mine;  // thread 0 holds the block total
        if (tid == 0) s.n_valid = total;
        __syncthreads();
        k_eff = min((uint32_t)k, s.n_valid);
        remaining = k_eff;
        if (k_eff == 0) break;
      }
      pick_bin(s, nb, remaining);
      remaining -= s.above;
      prefix |= s.bin << shift;
      pmask |= (uint32_t)(nb - 1) << shift;
    }
    const uint32_t thr = prefix;        // the k_eff-th largest key (when k_eff > 0)
    const uint32_t n_gt = k_eff - remaining;  // keys strictly above thr; `remaining` ties at thr are taken
    const uint32_t tkey = s.target_key;

    // ---- collection + target rank: one read of the row in column order ----------------------------------
    if (tid == 0) s.n_gt = 0;
    __syncthreads();
    uint32_t ties_seen = 0;
    int32_t before_target = 0;
    int buf = 0;
    for (int64_t base = 0; base < C; base += kSelThreads) {
      const int64_t c = base + tid;
      const uint32_t key = c < C ? order_key(__ldg(row + c)) : 0u;
      if (key != 0u && (key > tkey || (key == tkey && c < tcol))) ++before_target;
      if (k_eff == 0) continue;
      if (key > thr) {
        const uint32_t slot = atomicAdd(&s.n_gt, 1u);
        s.cand[slot] = ((unsigned long long)key << 32) | (uint32_t)(0x7fffffff - c);
      }
      if (ties_seen < remaining) {  // uniform across the block
        const bool eq = key == thr;
        const uint32_t bal = __ballot_sync(0xffffffffu, eq);
        if (lane == 0) s.ties[buf][warp] = __popc(bal);
        __syncthreads();
        uint32_t off = ties_seen, total = 0;
        for (int w = 0; w < kSelWarps; ++w) {
          const uint32_t t = s.ties[buf][w];
          if (w < warp) off += t;
          total += t;
        }
        if (eq) {
          const uint32_t idx = off + __popc(bal & ((1u << lane) - 1u));
          if (idx < remaining) s.cand[n_gt + idx] = ((unsigned long long)key << 32) | (uint32_t)(0x7fffffff - c);
        }
        ties_seen += total;
        buf ^= 1;
      }
    }
    if (target_rank != nullptr) {
      int32_t v = before_target;
#pragma unroll
      for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
      if (lane == 0) s.rank_part[warp] = v;
    }
    // ---- bitonic sort of the k_eff survivors, best first --------------------------------------------------
    int P = 1;
    while (P < (int)k_eff) P <<= 1;
    for (int j = (int)k_eff + tid; j < P; j += kSelThreads) s.cand[j] = 0ull;
    __syncthreads();
    if (target_rank != nullptr && tid == 0) {
      int32_t v = 0;
      for (int w = 0; w < kSelWarps; ++w) v += s.rank_part[w];
      target_rank[r] = tkey != 0u ? v : -1;
    }
    for (int size = 2; size <= P; size <<= 1) {
      for (int stride = size >> 1; stride > 0; stride >>= 1) {
        for (int i = tid; i < P / 2; i += kSelThreads) {
          const int a = 2 * stride * (i / stride) + (i % stride), b = a + stride;
          const unsigned long long x = s.cand[a], y = s.cand[b];
          if ((x < y) == ((a & size) == 0)) {
            s.cand[a] = y;
            s.cand[b] = x;
          }
        }
        __syncthreads();
      }
    }
    for (int j = tid; j < k; j += kSelThreads) {
      if (j < (int)k_eff) {
        const int64_t c = 0x7fffffff - (int64_t)(uint32_t)(s.cand[j] & 0xffffffffull);
        topk_item[r * k + j] = c;
        topk_score[r * k + j] = row[c];
      } else {
        topk_item[r * k + j] = -1;
        topk_score[r * k + j] = __int_as_float(0x7fc00000);
      }
    }
    __syncthreads();  // shared state is reused by the next row
  }
}

__global__ void __launch_bounds__(kMaskThreads) mask_items_kernel(float* __restrict__ scores, int64_t n, int64_t C,
                                                                  const int64_t* __restrict__ users, int64_t user_num,
                                                                  const int64_t* __restrict__ rowptr,
                                                                  const int32_t* __restrict__ col) {
  const float nan = __int_as_float(0x7fc00000);
  for (int64_t r = blockIdx.x; r < n; r += gridDim.x) {
    float* s = scores + r * C;
    const int64_t u = users[r];
    if (u < 0 || u >= user_num) {
      for (int64_t c = threadIdx.x; c < C; c += kMaskThreads) s[c] = nan;
      continue;
    }
    const int64_t e = rowptr[u + 1];
    for (int64_t j = rowptr[u] + threadIdx.x; j < e; j += kMaskThreads) {
      const int32_t c = col[j];
      if (c >= 0 && c < C) s[c] = nan;
    }
  }
}

__global__ void catalog_ids_kernel(int64_t* __restrict__ ids, int64_t total, int64_t item_num) {
  for (int64_t j = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; j < total; j += (int64_t)gridDim.x * blockDim.x)
    ids[j] = j % item_num;
}

int grid_for(int64_t n, int per_sm) {
  return (int)std::min<int64_t>(n, (int64_t)ncf::num_sms() * per_sm);
}

}  // namespace

extern "C" int ncf_mask_items(float* scores, int64_t n, int64_t C, const int64_t* users, int64_t user_num,
                              const int64_t* rowptr, const int32_t* col, void* stream) {
  NCF_REQUIRE(n >= 0, "ncf_mask_items: negative n");
  NCF_REQUIRE(C >= 1, "ncf_mask_items: C=%lld < 1", (long long)C);
  NCF_REQUIRE(user_num >= 0, "ncf_mask_items: negative user_num");
  if (n == 0) return NCF_OK;
  NCF_REQUIRE(scores && users && rowptr && col, "ncf_mask_items: null pointer");
  mask_items_kernel<<<grid_for(n, 16), kMaskThreads, 0, (cudaStream_t)stream>>>(scores, n, C, users, user_num,
                                                                              rowptr, col);
  NCF_LAUNCH_CHECK("mask_items_kernel");
  return NCF_OK;
}

extern "C" int64_t ncf_topk_rows_workspace_bytes(int64_t n, int64_t C, int32_t k) {
  if (n < 0 || C < 1 || C > INT32_MAX || k < 1 || k > kMaxK || k > C) return -1;
  return 0;  // the selection keeps its state in shared memory
}

extern "C" int ncf_topk_rows(const float* scores, int64_t n, int64_t C, int32_t k, const int64_t* target,
                             int64_t* topk_item, float* topk_score, int32_t* target_rank, void* workspace,
                             int64_t workspace_bytes, void* stream) {
  NCF_REQUIRE(n >= 0, "ncf_topk_rows: negative n");
  NCF_REQUIRE(C >= 1 && C <= INT32_MAX, "ncf_topk_rows: C=%lld outside [1, 2^31)", (long long)C);
  NCF_REQUIRE(k >= 1 && k <= kMaxK, "ncf_topk_rows: k=%d outside [1,1024]", k);
  NCF_REQUIRE(k <= C, "ncf_topk_rows: k=%d > C=%lld", k, (long long)C);
  if (n == 0) return NCF_OK;
  NCF_REQUIRE(scores && topk_item && topk_score, "ncf_topk_rows: null pointer");
  NCF_REQUIRE(!target || target_rank, "ncf_topk_rows: target given without target_rank");
  if (workspace_bytes < ncf_topk_rows_workspace_bytes(n, C, k)) {
    ncf::set_error("ncf_topk_rows: workspace too small");
    return NCF_ERR_WORKSPACE;
  }
  (void)workspace;
  topk_rows_kernel<<<grid_for(n, 8), kSelThreads, 0, (cudaStream_t)stream>>>(
      scores, n, C, k, target, topk_item, topk_score, target_rank);
  NCF_LAUNCH_CHECK("topk_rows_kernel");
  return NCF_OK;
}

// workspace = [scores chunk_users * item_num floats] [item ids chunk_users * item_num int64] [forward workspace]
static int64_t recommend_forward_bytes(const NcfModel* m, int64_t chunk_users) {
  TileParams p{};
  ncf::fill_model_params(p, m);
  p.B = chunk_users * m->item_num;
  p.user_div = (int)m->item_num;
  return ncf::forward_workspace_bytes(p);
}

extern "C" int64_t ncf_recommend_workspace_bytes(const NcfModel* m, int64_t chunk_users, int32_t k) {
  if (ncf::validate_model(m) != NCF_OK) return -1;
  if (m->item_num > INT32_MAX || k < 1 || k > kMaxK || k > m->item_num) return -1;
  if (chunk_users < 1 || chunk_users > kMaxChunkPairs / m->item_num) return -1;
  const int64_t pairs = chunk_users * m->item_num;
  return ncf::align_up(pairs * 4, 256) + ncf::align_up(pairs * 8, 256) + recommend_forward_bytes(m, chunk_users) + 256;
}

extern "C" int ncf_recommend(const NcfModel* m, const int64_t* users, int64_t n, int32_t k, const int64_t* rowptr,
                             const int32_t* col, const int64_t* target, int64_t chunk_users, int64_t* topk_item,
                             float* topk_score, int32_t* target_rank, void* workspace, int64_t workspace_bytes,
                             void* stream) {
  int rc = ncf::validate_model(m);
  if (rc != NCF_OK) return rc;
  const int64_t I = m->item_num;
  NCF_REQUIRE(I <= INT32_MAX, "ncf_recommend: item_num=%lld >= 2^31", (long long)I);
  NCF_REQUIRE(n >= 0, "ncf_recommend: negative n");
  NCF_REQUIRE(k >= 1 && k <= kMaxK, "ncf_recommend: k=%d outside [1,1024]", k);
  NCF_REQUIRE(k <= I, "ncf_recommend: k=%d > item_num=%lld", k, (long long)I);
  NCF_REQUIRE(chunk_users >= 1, "ncf_recommend: chunk_users=%lld < 1", (long long)chunk_users);
  NCF_REQUIRE((rowptr == nullptr) == (col == nullptr), "ncf_recommend: rowptr and col must both be given or both NULL");
  if (n == 0) return NCF_OK;
  const int64_t chunk = std::min(chunk_users, n);
  NCF_REQUIRE(chunk <= kMaxChunkPairs / I, "ncf_recommend: a chunk of %lld users exceeds 2^28 pairs (at most %lld users)",
              (long long)chunk, (long long)(kMaxChunkPairs / I));
  NCF_REQUIRE(users && topk_item && topk_score, "ncf_recommend: null pointer");
  NCF_REQUIRE(!target || target_rank, "ncf_recommend: target given without target_rank");
  if (!workspace || workspace_bytes < ncf_recommend_workspace_bytes(m, chunk, k)) {
    ncf::set_error("ncf_recommend: workspace too small (%lld < %lld)", (long long)workspace_bytes,
                   (long long)ncf_recommend_workspace_bytes(m, chunk, k));
    return NCF_ERR_WORKSPACE;
  }
  cudaStream_t st = (cudaStream_t)stream;
  const int64_t pairs = chunk * I;
  float* scores = (float*)workspace;
  int64_t* ids = (int64_t*)((char*)workspace + ncf::align_up(pairs * 4, 256));
  char* fw = (char*)ids + ncf::align_up(pairs * 8, 256);
  const int64_t fw_bytes = workspace_bytes - (fw - (char*)workspace);
  catalog_ids_kernel<<<grid_for((pairs + 255) / 256, 8), 256, 0, st>>>(ids, pairs, I);
  NCF_LAUNCH_CHECK("catalog_ids_kernel");
  for (int64_t lo = 0; lo < n; lo += chunk) {
    const int64_t cn = std::min(chunk, n - lo);
    TileParams p{};
    ncf::fill_model_params(p, m);
    p.user = users + lo;
    p.user_div = (int)I;
    p.item = ids;
    p.B = cn * I;
    p.invB = 1.f;
    p.logits = scores;
    rc = ncf::forward_dispatch(p, m, fw, fw_bytes, st);
    if (rc != NCF_OK) return rc;
    if (rowptr != nullptr) {
      rc = ncf_mask_items(scores, cn, I, users + lo, m->user_num, rowptr, col, stream);
      if (rc != NCF_OK) return rc;
    }
    rc = ncf_topk_rows(scores, cn, I, k, target ? target + lo : nullptr, topk_item + lo * k, topk_score + lo * k,
                       target ? target_rank + lo : nullptr, nullptr, 0, stream);
    if (rc != NCF_OK) return rc;
  }
  return NCF_OK;
}
