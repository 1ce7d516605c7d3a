// Row-sharded tables (BASELINE config 5): the device-side pieces of the embedding-row exchange.
// Row r of a table lives on rank r % world at local index r / world.  Per step a rank (i) buckets
// its samples by the owner of their item row, (ii) asks the owners for the rows, (iii) runs the
// fused step on its local user rows + the received item rows, (iv) returns the item-row gradients
// to the owners.  The collectives themselves are NCCL all-to-alls issued by the host
// (ncf_b200/dist.py); the kernels here pack, unpack and scatter-add.  HBM-bound byte shuffling.
#include "common.cuh"

namespace {

constexpr int kMaxWorld = 64;

// Owner of an item row.  A negative id (ncf_sample_neg writes -1 for a user without a legal negative) is
// given to rank 0 with local index -1, which ncf_gather_rows zero-fills and ncf_scatter_add_rows skips;
// `it % world` would be negative there and index outside the histogram and the cursor array.
__device__ __forceinline__ int owner_of(int64_t it, int world) { return it < 0 ? 0 : (int)(it % world); }

__global__ void owner_count_kernel(const int64_t* __restrict__ item, int64_t n, int world,
                                   int32_t* __restrict__ counts) {
  __shared__ int32_t h[kMaxWorld];
  for (int i = threadIdx.x; i < world; i += blockDim.x) h[i] = 0;
  __syncthreads();
  for (int64_t b = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; b < n;
       b += (int64_t)gridDim.x * blockDim.x)
    atomicAdd(&h[owner_of(item[b], world)], 1);
  __syncthreads();
  for (int i = threadIdx.x; i < world; i += blockDim.x)
    if (h[i]) atomicAdd(&counts[i], h[i]);
}

// counts[0..world) -> cursor[0..world) = exclusive prefix (single thread; world <= 64)
__global__ void owner_scan_kernel(const int32_t* __restrict__ counts, int world,
                                  int32_t* __restrict__ cursor) {
  if (threadIdx.x == 0 && blockIdx.x == 0) {
    int32_t run = 0;
    for (int i = 0; i < world; ++i) { cursor[i] = run; run += counts[i]; }
  }
}

// perm[pos] = sample index, grouped by owner (order inside a group is arbitrary);
// local_idx[pos] = item / world of that sample (-1 for a negative item).
__global__ void owner_place_kernel(const int64_t* __restrict__ item, int64_t n, int world,
                                   int32_t* __restrict__ cursor, int64_t* __restrict__ perm,
                                   int64_t* __restrict__ local_idx) {
  for (int64_t b = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; b < n;
       b += (int64_t)gridDim.x * blockDim.x) {
    const int64_t it = item[b];
    const int pos = atomicAdd(&cursor[owner_of(it, world)], 1);
    perm[pos] = b;
    local_idx[pos] = it < 0 ? -1 : it / world;
  }
}

// out[i][:] = table[idx[i]][:]   (one warp per row, 16-byte pieces when dim % 4 == 0)
__global__ void gather_rows_kernel(const float* __restrict__ table, const int64_t* __restrict__ idx,
                                   int64_t n, int dim, int64_t rows, float* __restrict__ out) {
  const int lane = threadIdx.x & 31;
  const int64_t w = (blockIdx.x * (int64_t)blockDim.x + threadIdx.x) >> 5;
  const int64_t nw = ((int64_t)gridDim.x * blockDim.x) >> 5;
  for (int64_t i = w; i < n; i += nw) {
    const int64_t r = idx[i];
    const bool ok = r >= 0 && r < rows;
    const float* src = table + (ok ? r : 0) * dim;
    float* dst = out + i * dim;
    if ((dim & 3) == 0) {
      for (int c = lane * 4; c < dim; c += 128)
        *reinterpret_cast<float4*>(dst + c) = ok ? ldg4(src + c) : make_float4(0, 0, 0, 0);
    } else {
      for (int c = lane; c < dim; c += 32) dst[c] = ok ? __ldg(src + c) : 0.f;
    }
  }
}

// table[idx[i]][:] += in[i][:]   (vector REDs; duplicates in idx accumulate)
__global__ void scatter_add_rows_kernel(float* __restrict__ table, const int64_t* __restrict__ idx,
                                        int64_t n, int dim, int64_t rows,
                                        const float* __restrict__ in) {
  const int lane = threadIdx.x & 31;
  const int64_t w = (blockIdx.x * (int64_t)blockDim.x + threadIdx.x) >> 5;
  const int64_t nw = ((int64_t)gridDim.x * blockDim.x) >> 5;
  for (int64_t i = w; i < n; i += nw) {
    const int64_t r = idx[i];
    if (r < 0 || r >= rows) continue;
    float* dst = table + r * dim;
    const float* src = in + i * dim;
    if ((dim & 3) == 0) {
      for (int c = lane * 4; c < dim; c += 128) red_add4(dst + c, ldg4(src + c));
    } else {
      for (int c = lane; c < dim; c += 32) atomicAdd(dst + c, __ldg(src + c));
    }
  }
}

// out[i] = in[perm[i]]  for int64 / float payloads
template <typename T>
__global__ void permute_kernel(const T* __restrict__ in, const int64_t* __restrict__ perm, int64_t n,
                               T* __restrict__ out) {
  for (int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; i < n;
       i += (int64_t)gridDim.x * blockDim.x)
    out[i] = in[perm[i]];
}

inline int blocks_for(int64_t n, int per_block) {
  int64_t b = (n + per_block - 1) / per_block;
  const int64_t cap = (int64_t)ncf::num_sms() * 8;
  if (b > cap) b = cap;
  return (int)(b < 1 ? 1 : b);
}

}  // namespace

extern "C" int ncf_bucket_by_owner(const int64_t* item, int64_t n, int32_t world, int64_t* perm,
                                   int64_t* local_idx, int32_t* counts, int32_t* cursor,
                                   void* stream) {
  NCF_REQUIRE(n >= 0 && world >= 1 && world <= kMaxWorld, "ncf_bucket_by_owner: bad n/world");
  NCF_REQUIRE(counts && cursor, "ncf_bucket_by_owner: null pointer");
  cudaStream_t st = (cudaStream_t)stream;
  NCF_CUDA(cudaMemsetAsync(counts, 0, sizeof(int32_t) * world, st));
  if (n > 0) {
    NCF_REQUIRE(item && perm && local_idx, "ncf_bucket_by_owner: null pointer");
    owner_count_kernel<<<blocks_for(n, 256), 256, 0, st>>>(item, n, world, counts);
    NCF_LAUNCH_CHECK("owner_count_kernel");
  }
  owner_scan_kernel<<<1, 32, 0, st>>>(counts, world, cursor);
  NCF_LAUNCH_CHECK("owner_scan_kernel");
  if (n > 0) {
    owner_place_kernel<<<blocks_for(n, 256), 256, 0, st>>>(item, n, world, cursor, perm, local_idx);
    NCF_LAUNCH_CHECK("owner_place_kernel");
  }
  return NCF_OK;
}

extern "C" int ncf_gather_rows(const float* table, const int64_t* idx, int64_t n, int32_t dim,
                               int64_t rows, float* out, void* stream) {
  NCF_REQUIRE(n >= 0 && dim > 0 && rows > 0, "ncf_gather_rows: bad sizes");
  if (n == 0) return NCF_OK;
  NCF_REQUIRE(table && idx && out, "ncf_gather_rows: null pointer");
  gather_rows_kernel<<<blocks_for(n, 8), 256, 0, (cudaStream_t)stream>>>(table, idx, n, dim, rows, out);
  NCF_LAUNCH_CHECK("gather_rows_kernel");
  return NCF_OK;
}

extern "C" int ncf_scatter_add_rows(float* table, const int64_t* idx, int64_t n, int32_t dim,
                                    int64_t rows, const float* in, void* stream) {
  NCF_REQUIRE(n >= 0 && dim > 0 && rows > 0, "ncf_scatter_add_rows: bad sizes");
  if (n == 0) return NCF_OK;
  NCF_REQUIRE(table && idx && in, "ncf_scatter_add_rows: null pointer");
  scatter_add_rows_kernel<<<blocks_for(n, 8), 256, 0, (cudaStream_t)stream>>>(table, idx, n, dim, rows, in);
  NCF_LAUNCH_CHECK("scatter_add_rows_kernel");
  return NCF_OK;
}

extern "C" int ncf_permute_i64(const int64_t* in, const int64_t* perm, int64_t n, int64_t* out,
                               void* stream) {
  NCF_REQUIRE(n >= 0, "ncf_permute_i64: negative n");
  if (n == 0) return NCF_OK;
  NCF_REQUIRE(in && perm && out, "ncf_permute_i64: null pointer");
  permute_kernel<int64_t><<<blocks_for(n, 256), 256, 0, (cudaStream_t)stream>>>(in, perm, n, out);
  NCF_LAUNCH_CHECK("permute_kernel<i64>");
  return NCF_OK;
}

extern "C" int ncf_permute_f32(const float* in, const int64_t* perm, int64_t n, float* out,
                               void* stream) {
  NCF_REQUIRE(n >= 0, "ncf_permute_f32: negative n");
  if (n == 0) return NCF_OK;
  NCF_REQUIRE(in && perm && out, "ncf_permute_f32: null pointer");
  permute_kernel<float><<<blocks_for(n, 256), 256, 0, (cudaStream_t)stream>>>(in, perm, n, out);
  NCF_LAUNCH_CHECK("permute_kernel<f32>");
  return NCF_OK;
}

// ---- the same exchange over peer memory (one NVLink node) -----------------------------------------------------
// Instead of three NCCL all-to-alls with host-known split sizes, the ranks write into each other's
// buffers directly (CUDA-IPC mappings, ncf_peer_alloc / ncf_ipc_open):
//   requester r:  request (local row index, slot) -> inbox of the owner        [ncf_shard_request]
//   owner o:      registers the requested rows (mark + catch-up by the caller), then PUSHES each row
//                 into the requester's receive buffers at the slot it named    [ncf_shard_push_rows]
//   requester r:  after its fused step, REDs every per-sample item-row gradient straight into the
//                 owner's gradient table over NVLink                           [ncf_shard_push_grads]
// No split sizes ever reach the host; the caller separates the three phases by rank barriers
// (stream-ordered one-element all-reduces).  slot = the sample's position in the requester's batch, so
// the received rows line up with the batch and nothing has to be permuted.
namespace {

constexpr int kMaxPeers = 8;
struct PeerPtrs {
  void* p[kMaxPeers];
};

__device__ __forceinline__ void red_add4_sys(float* p, float4 v) {
  asm volatile("red.relaxed.sys.global.add.v4.f32 [%0], {%1, %2, %3, %4};" ::"l"(p), "f"(v.x), "f"(v.y), "f"(v.z),
               "f"(v.w)
               : "memory");
}

// inbox of owner o: int64 [world][cap], entry = (local_row << 32) | slot; cursor[o] counts this rank's
// requests to owner o (zeroed by the launcher)
__global__ void shard_request_kernel(const int64_t* __restrict__ item, int64_t n, int world, int rank, int64_t cap,
                                     int64_t item_num, PeerPtrs inbox, int32_t* __restrict__ cursor) {
  for (int64_t s = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; s < n; s += (int64_t)gridDim.x * blockDim.x) {
    const int64_t it = item[s];
    if (it < 0 || it >= item_num) continue;   // the fused step reports the bad index (NaN logit)
    const int o = (int)(it % world);
    const int j = atomicAdd(&cursor[o], 1);
    reinterpret_cast<int64_t*>(inbox.p[o])[(int64_t)rank * cap + j] = ((it / world) << 32) | s;
  }
}

__global__ void shard_publish_counts_kernel(const int32_t* __restrict__ cursor, int world, int rank, PeerPtrs inbox_cnt) {
  const int o = threadIdx.x;
  if (o < world) reinterpret_cast<int32_t*>(inbox_cnt.p[o])[rank] = cursor[o];
}

// owner: registers every requested row in the touched list of the item side
__global__ void shard_mark_requests_kernel(const int64_t* __restrict__ inbox, const int32_t* __restrict__ cnt, int world,
                                           int64_t cap, int64_t limit, int32_t* flag, int64_t* list, int32_t* count) {
  const int64_t total = (int64_t)world * cap;
  for (int64_t e = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; e < total; e += (int64_t)gridDim.x * blockDim.x) {
    const int r = (int)(e / cap);
    const int64_t j = e - (int64_t)r * cap;
    if (j >= cnt[r]) continue;
    const int64_t row = inbox[e] >> 32;
    if (row < 0 || row >= limit) continue;
    if (atomicExch(&flag[row], 1) == 0) list[atomicAdd(count, 1)] = row;
  }
}

// owner: one warp per request, 16-byte pieces, stores go to the requester's memory
__global__ void shard_push_rows_kernel(const int64_t* __restrict__ inbox, const int32_t* __restrict__ cnt, int world,
                                       int64_t cap, int64_t limit, const float* __restrict__ tab_gmf,
                                       const float* __restrict__ tab_mlp, int f, int d, PeerPtrs rows_gmf, PeerPtrs rows_mlp) {
  const int lane = threadIdx.x & 31;
  const int64_t w = (blockIdx.x * (int64_t)blockDim.x + threadIdx.x) >> 5;
  const int64_t nw = ((int64_t)gridDim.x * blockDim.x) >> 5;
  const int64_t total = (int64_t)world * cap;
  for (int64_t e = w; e < total; e += nw) {
    const int r = (int)(e / cap);
    const int64_t j = e - (int64_t)r * cap;
    if (j >= cnt[r]) {   // the rest of this source's block is empty: jump to the next source
      const int64_t next = (int64_t)(r + 1) * cap;
      e += (next - e - 1) / nw * nw;   // stays congruent to w modulo nw; the loop increment does the last hop
      continue;
    }
    const int64_t ent = inbox[e];
    const int64_t row = ent >> 32, slot = ent & 0xffffffffll;
    const bool ok = row >= 0 && row < limit;
    if (tab_gmf != nullptr) {
      float* dst = reinterpret_cast<float*>(rows_gmf.p[r]) + slot * f;
      const float* src = tab_gmf + (ok ? row : 0) * f;
      for (int c = lane * 4; c < f; c += 128)
        *reinterpret_cast<float4*>(dst + c) = ok ? ldg4(src + c) : make_float4(0, 0, 0, 0);
    }
    if (tab_mlp != nullptr) {
      float* dst = reinterpret_cast<float*>(rows_mlp.p[r]) + slot * d;
      const float* src = tab_mlp + (ok ? row : 0) * d;
      for (int c = lane * 4; c < d; c += 128)
        *reinterpret_cast<float4*>(dst + c) = ok ? ldg4(src + c) : make_float4(0, 0, 0, 0);
    }
  }
}

// requester: per-sample item-row gradients -> the owners' gradient tables (vector REDs over NVLink)
__global__ void shard_push_grads_kernel(const int64_t* __restrict__ item, int64_t n, int world, int64_t item_num,
                                        const float* __restrict__ g_gmf, const float* __restrict__ g_mlp, int f, int d,
                                        PeerPtrs tab_gmf, PeerPtrs tab_mlp) {
  const int lane = threadIdx.x & 31;
  const int64_t w = (blockIdx.x * (int64_t)blockDim.x + threadIdx.x) >> 5;
  const int64_t nw = ((int64_t)gridDim.x * blockDim.x) >> 5;
  for (int64_t s = w; s < n; s += nw) {
    const int64_t it = item[s];
    if (it < 0 || it >= item_num) continue;
    const int o = (int)(it % world);
    const int64_t row = it / world;
    if (g_gmf != nullptr) {
      float* dst = reinterpret_cast<float*>(tab_gmf.p[o]) + row * f;
      for (int c = lane * 4; c < f; c += 128) red_add4_sys(dst + c, ldg4(g_gmf + s * f + c));
    }
    if (g_mlp != nullptr) {
      float* dst = reinterpret_cast<float*>(tab_mlp.p[o]) + row * d;
      for (int c = lane * 4; c < d; c += 128) red_add4_sys(dst + c, ldg4(g_mlp + s * d + c));
    }
  }
}

int fill_peers(PeerPtrs& pp, void* const* ptrs, int world, bool required, const char* what) {
  for (int r = 0; r < kMaxPeers; ++r) pp.p[r] = nullptr;
  if (ptrs == nullptr) {
    NCF_REQUIRE(!required, "%s: peer pointer array is NULL", what);
    return NCF_OK;
  }
  for (int r = 0; r < world; ++r) {
    NCF_REQUIRE(ptrs[r] != nullptr && ((uintptr_t)ptrs[r] & 15) == 0, "%s: peer buffer %d is NULL or misaligned", what, r);
    pp.p[r] = ptrs[r];
  }
  return NCF_OK;
}

}  // namespace

extern "C" int ncf_shard_request(const int64_t* item, int64_t n, int32_t world, int32_t rank, int64_t cap,
                                 int64_t item_num, void* const* inbox_peers, void* const* inbox_count_peers,
                                 int32_t* cursor, void* stream) {
  NCF_REQUIRE(world >= 1 && world <= kMaxPeers && rank >= 0 && rank < world, "ncf_shard_request: world must be 1..8");
  NCF_REQUIRE(n >= 0 && n <= cap && cap < (1ll << 31) && item_num > 0, "ncf_shard_request: n=%lld exceeds the inbox capacity %lld",
              (long long)n, (long long)cap);
  NCF_REQUIRE(cursor != nullptr, "ncf_shard_request: cursor is NULL");
  PeerPtrs ib, ic;
  int rc;
  if ((rc = fill_peers(ib, inbox_peers, world, true, "ncf_shard_request")) != NCF_OK) return rc;
  if ((rc = fill_peers(ic, inbox_count_peers, world, true, "ncf_shard_request")) != NCF_OK) return rc;
  cudaStream_t st = (cudaStream_t)stream;
  NCF_CUDA(cudaMemsetAsync(cursor, 0, sizeof(int32_t) * world, st));
  if (n > 0) {
    NCF_REQUIRE(item != nullptr, "ncf_shard_request: item is NULL");
    shard_request_kernel<<<blocks_for(n, 256), 256, 0, st>>>(item, n, world, rank, cap, item_num, ib, cursor);
    NCF_LAUNCH_CHECK("shard_request_kernel");
  }
  shard_publish_counts_kernel<<<1, 32, 0, st>>>(cursor, world, rank, ic);
  NCF_LAUNCH_CHECK("shard_publish_counts_kernel");
  return NCF_OK;
}

extern "C" int ncf_shard_mark_requests(const NcfModel* m, const NcfGrads* g, const int64_t* inbox, const int32_t* inbox_count,
                                       int32_t world, int64_t cap, void* stream) {
  int rc = ncf::validate_model(m);
  if (rc != NCF_OK) return rc;
  NCF_REQUIRE(g && g->item_flag && g->item_list && g->touched_count && inbox && inbox_count,
              "ncf_shard_mark_requests: null pointer");
  NCF_REQUIRE(world >= 1 && world <= kMaxPeers && cap > 0, "ncf_shard_mark_requests: bad world / cap");
  shard_mark_requests_kernel<<<blocks_for((int64_t)world * cap, 256), 256, 0, (cudaStream_t)stream>>>(
      inbox, inbox_count, world, cap, m->item_num, g->item_flag, g->item_list, g->touched_count + 1);
  NCF_LAUNCH_CHECK("shard_mark_requests_kernel");
  return NCF_OK;
}

extern "C" int ncf_shard_push_rows(const NcfModel* m, const int64_t* inbox, const int32_t* inbox_count, int32_t world,
                                   int64_t cap, void* const* rows_gmf_peers, void* const* rows_mlp_peers, void* stream) {
  int rc = ncf::validate_model(m);
  if (rc != NCF_OK) return rc;
  NCF_REQUIRE(inbox && inbox_count && world >= 1 && world <= kMaxPeers && cap > 0, "ncf_shard_push_rows: bad argument");
  const bool gmf = m->model_type != NCF_MLP, mlp = m->model_type != NCF_GMF;
  NCF_REQUIRE((!gmf || (m->factor_num & 3) == 0) && (!mlp || (m->mlp_dim & 3) == 0),
              "ncf_shard_push_rows: row widths must be multiples of 4 floats");
  PeerPtrs pg, pm;
  if ((rc = fill_peers(pg, rows_gmf_peers, world, gmf, "ncf_shard_push_rows")) != NCF_OK) return rc;
  if ((rc = fill_peers(pm, rows_mlp_peers, world, mlp, "ncf_shard_push_rows")) != NCF_OK) return rc;
  shard_push_rows_kernel<<<ncf::num_sms() * 8, 256, 0, (cudaStream_t)stream>>>(
      inbox, inbox_count, world, cap, m->item_num, gmf ? m->embed_item_gmf : nullptr, mlp ? m->embed_item_mlp : nullptr,
      m->factor_num, m->mlp_dim, pg, pm);
  NCF_LAUNCH_CHECK("shard_push_rows_kernel");
  return NCF_OK;
}

extern "C" int ncf_shard_push_grads(const int64_t* item, int64_t n, int32_t world, int64_t item_num, const float* g_gmf,
                                    const float* g_mlp, int32_t f, int32_t d, void* const* grad_gmf_peers,
                                    void* const* grad_mlp_peers, void* stream) {
  NCF_REQUIRE(world >= 1 && world <= kMaxPeers && n >= 0 && item_num > 0, "ncf_shard_push_grads: bad argument");
  NCF_REQUIRE((g_gmf == nullptr || (f > 0 && (f & 3) == 0)) && (g_mlp == nullptr || (d > 0 && (d & 3) == 0)),
              "ncf_shard_push_grads: row widths must be multiples of 4 floats");
  if (n == 0) return NCF_OK;
  NCF_REQUIRE(item != nullptr, "ncf_shard_push_grads: item is NULL");
  PeerPtrs pg, pm;
  int rc;
  if ((rc = fill_peers(pg, grad_gmf_peers, world, g_gmf != nullptr, "ncf_shard_push_grads")) != NCF_OK) return rc;
  if ((rc = fill_peers(pm, grad_mlp_peers, world, g_mlp != nullptr, "ncf_shard_push_grads")) != NCF_OK) return rc;
  shard_push_grads_kernel<<<blocks_for(n, 8), 256, 0, (cudaStream_t)stream>>>(item, n, world, item_num, g_gmf, g_mlp, f, d,
                                                                            pg, pm);
  NCF_LAUNCH_CHECK("shard_push_grads_kernel");
  return NCF_OK;
}
