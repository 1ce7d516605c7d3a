// tcgen05 / TMEM version of the tower arithmetic for large batches (sm_100a).
//
// The tower (reference: src/ncf/models.py:86-107, MLP_layers + predict_layer, and autograd's
// backward of it) runs as 128-sample x N GEMMs on the 5th-generation tensor cores:
// `tcgen05.mma.cta_group::1.kind::tf32`, fp32 accumulators in tensor memory.  fp32 parity comes from
// the error-compensated split the mma.sync kernel uses as well (x = hi + lo, hi = x with the low 13
// mantissa bits cleared - which is what the tensor core does to an fp32 operand by itself):
// D += A_hi*B_hi + A_lo*B_hi + A_hi*B_lo.
//
//   umma_weight_images_kernel   W_k -> swizzled (hi, lo) operand images, forward and transposed
//   umma_tower_kernel<TRAIN>    fused: gather -> tower forward -> predict / loss -> backward-data ->
//                               scatter for one 128-sample tile at a time, every A operand in TMEM
//                               (towers whose operand chain fits the 512 TMEM columns: f <= 64 and
//                               W[1] <= 128, e.g. the bench config f = 32, L = 3)
//   umma_gemm_kernel<EPI>       the same GEMMs as separate launches, operands from shared memory
//                               (fallback for wider towers, e.g. f = 64 with L = 3):
//       EPI_RELU_STORE  forward layer:  act[k+1] = relu(D + b)
//       EPI_PREDICT(_TRAIN)  last layer: h_L = relu(D + b); logit (+ loss, dlogit, predict grads,
//                                       GMF-branch scatter, delta_L)
//       EPI_MASK_STORE  backward data:  delta[k] = D * (act[k] > 0)
//       EPI_SCATTER     backward data of layer 0: D -> RED.128 into the embedding-gradient rows
//   umma_wgrad_kernel           dW_k = delta[k+1]^T act[k] summed over the CTA's samples with the
//                               accumulator resident in TMEM; both operands MN-major (128B_BASE32B)
//
// Layouts, issue rates and hand-off costs were measured on this hardware first: tools/umma_probe.cu,
// tools/mma_issue_probe.cu, tools/sync_probe.cu (outputs and the kernel's phase trace in profiles/).
#include <algorithm>
#include <cstdlib>

#include "common.cuh"
#include "tile_params.cuh"

namespace {

constexpr int kTile = 128;  // samples per accumulator tile (UMMA M)
constexpr uint32_t kHiMask = 0xffffe000u;
constexpr int kProducerWarps = 8;   // two groups of four (even / odd panels)
constexpr int kLoaderWarp = 17;     // weight-panel bulk copies
constexpr int kGemmThreads = 576;   // warps 0-7 A producers, 8 MMA, 9-12 / 13-16 epilogue (even / odd tiles), 17 loader
constexpr int kMaxStages = 4;

enum { EPI_RELU_STORE = 0, EPI_PREDICT = 1, EPI_PREDICT_TRAIN = 2, EPI_MASK_STORE = 3, EPI_SCATTER = 4 };

struct GemmArgs {
  int K;        // reduction width (multiple of 8)
  int N;        // output columns of one block (<= 256, multiple of 16)
  int n_total;  // rows of the weight image / leading dimension of the output
  int passes;   // 3 = fp32-parity split, 1 = plain TF32
  int layer;    // tower layer index k
  int gather;   // A rows are [embed_user_MLP[u] | embed_item_MLP[i]] instead of a dense matrix
  int stages;
  const float* a;      // dense A [B][K]
  const float* b_img;  // weight image: [panel][hi|lo][n_total rows][32]
  const float* bias;
  float* out;
  const float* mask_src;
};

struct WgradJob {
  int k, mb, nb, cta0, nctas;
  int S;  // samples per stage: scaled so that every job moves the same bytes per hand-off
};
struct WgradArgs {
  int njobs, passes;
  WgradJob job[12];
};

// ---- PTX wrappers -----------------------------------------------------------------------------------
__device__ __forceinline__ uint32_t smem_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }

__device__ __forceinline__ void mbar_init(uint64_t* b, uint32_t count) {
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(b)), "r"(count));
}
__device__ __forceinline__ void mbar_arrive(uint64_t* b) {
  asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(smem_u32(b)) : "memory");
}
__device__ __forceinline__ void mbar_expect_tx(uint64_t* b, uint32_t bytes) {
  asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(b)), "r"(bytes) : "memory");
}
// Bounded wait: a protocol bug must end in a trap (launch failure), never in a hung GPU.
// NCF_MBAR_POLL: busy-poll with test_wait instead of the suspending try_wait.
__device__ __forceinline__ void mbar_wait(uint64_t* b, uint32_t parity) {
  const uint32_t addr = smem_u32(b);
  for (uint32_t spin = 0; spin < (1u << 26); ++spin) {
    uint32_t done;
#ifdef NCF_MBAR_POLL
    asm volatile(
        "{\n\t.reg .pred p;\n\tmbarrier.test_wait.parity.shared::cta.b64 p, [%1], %2;\n\tselp.u32 %0, 1, 0, p;\n\t}"
        : "=r"(done) : "r"(addr), "r"(parity) : "memory");
#else
    asm volatile(
        "{\n\t.reg .pred p;\n\tmbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\tselp.u32 %0, 1, 0, p;\n\t}"
        : "=r"(done) : "r"(addr), "r"(parity) : "memory");
#endif
    if (done) return;
  }
  __trap();
}
// Non-blocking probe of a phase, warp-uniform result.
__device__ __forceinline__ bool mbar_test_warp(uint64_t* b, uint32_t parity) {
  uint32_t done = 0;
  if ((threadIdx.x & 31) == 0)
    asm volatile(
        "{\n\t.reg .pred p;\n\tmbarrier.test_wait.parity.shared::cta.b64 p, [%1], %2;\n\tselp.u32 %0, 1, 0, p;\n\t}"
        : "=r"(done) : "r"(smem_u32(b)), "r"(parity) : "memory");
  return __shfl_sync(0xffffffffu, done, 0) != 0;
}
// One lane polls / arrives for its warp: 32 arrivals on one mbarrier serialise in shared memory.
__device__ __forceinline__ void mbar_wait_warp(uint64_t* b, uint32_t parity) {
  if ((threadIdx.x & 31) == 0) mbar_wait(b, parity);
  __syncwarp();
}
__device__ __forceinline__ void mbar_arrive_warp(uint64_t* b) {
  __syncwarp();
  if ((threadIdx.x & 31) == 0) mbar_arrive(b);
}
__device__ __forceinline__ void bulk_g2s(void* dst, const void* src, uint32_t bytes, uint64_t* bar) {
  asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];"
               ::"r"(smem_u32(dst)), "l"(src), "r"(bytes), "r"(smem_u32(bar)) : "memory");
}
// 16-byte global -> shared copy through L2 only; !valid writes zeros (src-size 0, nothing is read)
__device__ __forceinline__ void cp_async16_zfill(void* dst, const void* src, bool valid) {
  asm volatile("cp.async.cg.shared.global [%0], [%1], 16, %2;" ::"r"(smem_u32(dst)), "l"(src), "r"(valid ? 16 : 0) : "memory");
}
__device__ __forceinline__ void fence_async_smem() { asm volatile("fence.proxy.async.shared::cta;" ::: "memory"); }
__device__ __forceinline__ void tc_fence_before() { asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void tc_fence_after() { asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void tc_commit(uint64_t* bar) {
  asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(smem_u32(bar)) : "memory");
}
__device__ __forceinline__ void tc_mma(uint32_t d_tmem, uint64_t da, uint64_t db, uint32_t idesc, uint32_t accumulate) {
  asm volatile(
      "{\n\t.reg .pred p;\n\tsetp.ne.b32 p, %4, 0;\n\t"
      "tcgen05.mma.cta_group::1.kind::tf32 [%0], %1, %2, %3, p;\n\t}"
      ::"r"(d_tmem), "l"(da), "l"(db), "r"(idesc), "r"(accumulate) : "memory");
}
// 32 lanes x 32 consecutive columns: thread = TMEM lane (row), r[j] = column j
__device__ __forceinline__ void tc_ld32(uint32_t taddr, float (&v)[32]) {
  uint32_t r[32];
  asm volatile(
      "tcgen05.ld.sync.aligned.32x32b.x32.b32 "
      "{%0,%1,%2,%3,%4,%5,%6,%7,%8,%9,%10,%11,%12,%13,%14,%15,"
      "%16,%17,%18,%19,%20,%21,%22,%23,%24,%25,%26,%27,%28,%29,%30,%31}, [%32];"
      : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]),
        "=r"(r[8]), "=r"(r[9]), "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15]),
        "=r"(r[16]), "=r"(r[17]), "=r"(r[18]), "=r"(r[19]), "=r"(r[20]), "=r"(r[21]), "=r"(r[22]), "=r"(r[23]),
        "=r"(r[24]), "=r"(r[25]), "=r"(r[26]), "=r"(r[27]), "=r"(r[28]), "=r"(r[29]), "=r"(r[30]), "=r"(r[31])
      : "r"(taddr));
  asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory");
#pragma unroll
  for (int j = 0; j < 32; ++j) v[j] = __uint_as_float(r[j]);
}

// shared-memory matrix descriptor (sm_100 version 1): start, leading/stride byte offsets, layout type
__device__ __forceinline__ uint64_t make_desc(uint32_t addr, uint32_t lbo, uint32_t sbo, uint32_t layout) {
  uint64_t d = (uint64_t)(layout & 7) << 61;
  d |= (uint64_t)((addr >> 4) & 0x3fff);
  d |= (uint64_t)((lbo >> 4) & 0x3fff) << 16;
  d |= (uint64_t)((sbo >> 4) & 0x3fff) << 32;
  d |= (uint64_t)1 << 46;
  return d;
}
// instruction descriptor: kind::tf32, fp32 accumulate, M x N, operand majors (0 = K-major, 1 = MN-major)
__device__ __forceinline__ uint32_t make_idesc(int m, int n, int a_mn, int b_mn) {
  uint32_t d = 0;
  d |= 1u << 4;
  d |= 2u << 7;
  d |= 2u << 10;
  d |= (uint32_t)a_mn << 15;
  d |= (uint32_t)b_mn << 16;
  d |= (uint32_t)(n >> 3) << 17;
  d |= (uint32_t)(m >> 4) << 24;
  return d;
}

__device__ __forceinline__ void split4(const float4 x, float4& hi, float4& lo) {
  hi.x = __uint_as_float(__float_as_uint(x.x) & kHiMask);
  hi.y = __uint_as_float(__float_as_uint(x.y) & kHiMask);
  hi.z = __uint_as_float(__float_as_uint(x.z) & kHiMask);
  hi.w = __uint_as_float(__float_as_uint(x.w) & kHiMask);
  lo = make_float4(x.x - hi.x, x.y - hi.y, x.z - hi.z, x.w - hi.w);
}

// Column sums over the warp: v[j] = this lane's value of column j; lane c returns the sum of column c.
__device__ __forceinline__ float warp_colsum32(float (&v)[32], int lane) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) {
    const bool upper = (lane & o) != 0;
#pragma unroll
    for (int i = 0; i < o; ++i) {
      const float send = upper ? v[i] : v[i + o];
      const float keep = upper ? v[i + o] : v[i];
      v[i] = keep + __shfl_xor_sync(0xffffffffu, send, o);
    }
  }
  return v[0];
}

__device__ __forceinline__ void named_bar(int id, int count) {
  asm volatile("bar.sync %0, %1;" ::"r"(id), "r"(count) : "memory");
}

// ---- weight images -----------------------------------------------------------------------------------
// K-major SWIZZLE_128B image of a logical [rows][K] matrix: panel pi = 32 columns,
//   [pi][hi|lo][row][128 B], 16-byte chunk index ^= row % 8.
// dir 0: rows = W[k+1] (n_out), K = W[k]   (forward B operand:  elem(n, c) = w[n][c])
// dir 1: rows = W[k]   (k_in),  K = W[k+1] (backward-data B operand: elem(n, c) = w[c][n])
__global__ void umma_weight_images_kernel(const TileParams p) {
  const int k = blockIdx.y >> 1, dir = blockIdx.y & 1;
  const int kin = p.W[k], nout = p.W[k + 1];
  const int rows = dir ? kin : nout, K = dir ? nout : kin;
  const int panels = (K + 31) / 32;
  const float* w = p.w[k];
  float* img = dir ? p.wsplit_b[k] : p.wsplit_f[k];
  const int64_t total = (int64_t)panels * rows * 32;
  for (int64_t idx = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; idx < total;
       idx += (int64_t)gridDim.x * blockDim.x) {
    const int cc = (int)(idx & 31);
    const int r = (int)((idx >> 5) % rows);
    const int pi = (int)((idx >> 5) / rows);
    const int c = pi * 32 + cc;
    float x = 0.f;
    if (c < K) x = dir ? w[(int64_t)c * kin + r] : w[(int64_t)r * kin + c];
    const float hi = __uint_as_float(__float_as_uint(x) & kHiMask);
    const int64_t off = (int64_t)pi * 2 * rows * 32 + (int64_t)r * 32 + ((((cc >> 2) ^ (r & 7)) << 2) | (cc & 3));
    img[off] = hi;
    img[off + (int64_t)rows * 32] = x - hi;
  }
}

// ---- GEMM kernel ------------------------------------------------------------------------------------
struct GemmBars {
  uint64_t full[kMaxStages], empty[kMaxStages], acc_full[2], acc_empty[2];
  uint32_t tmem_base;
  float pg[2 * 128 + 4];  // predict-weight / predict-bias gradient of this CTA (EPI_PREDICT_TRAIN)
};

template <int EPI>
__global__ void __launch_bounds__(kGemmThreads, 1)
umma_gemm_kernel(const __grid_constant__ TileParams p, const __grid_constant__ GemmArgs g) {
  extern __shared__ __align__(1024) uint8_t smem_raw[];
  __shared__ GemmBars bars;
  // 1024-byte alignment of the swizzle atoms
  uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~(uintptr_t)1023);
  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  const int K = g.K, N = g.N;
  const int panels = (K + 31) >> 5;
  const uint32_t a_bytes = kTile * 128, b_bytes = (uint32_t)N * 128;
  const uint32_t stage_bytes = 2 * a_bytes + 2 * b_bytes;
  const int nb = blockIdx.y;  // output-column block
  const int64_t ntiles = (p.B + kTile - 1) / kTile;
  uint32_t tmem_cols = 32;
  while (tmem_cols < 2u * N) tmem_cols <<= 1;

  if (tid == 0) {
    for (int s = 0; s < g.stages; ++s) { mbar_init(&bars.full[s], kProducerWarps / 2 + 1); mbar_init(&bars.empty[s], 1); }
    for (int a = 0; a < 2; ++a) { mbar_init(&bars.acc_full[a], 1); mbar_init(&bars.acc_empty[a], 4); }
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  }
  if (EPI == EPI_PREDICT_TRAIN)
    for (int i = tid; i < 2 * 128 + 4; i += kGemmThreads) bars.pg[i] = 0.f;
  if (warp == kProducerWarps) {
    asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(&bars.tmem_base)), "r"(tmem_cols));
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;");
  }
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem = bars.tmem_base;

  if (warp < kProducerWarps) {
    // ===== A producers.  Two groups of four warps take alternate panels of the flat (tile, panel)
    // sequence, so two hand-off chains (wait -> copy -> split -> fence -> arrive) run concurrently.
    // A thread copies global -> shared with cp.async (raw fp32 is the "hi" image: the tensor core
    // ignores the low 13 mantissa bits) and later derives the "lo" image from its own pieces.
    const int grp = warp >> 2;        // parity of the panels this group serves
    const int u = tid & 127;          // thread within the group: rows r0 and r0 + 64,
    const int r0 = u >> 1, hq = u & 1;  // 16-byte pieces 2c + hq (a lane pair covers one 32-byte sector)
    const int d = p.d;
    const int64_t my_tiles = (blockIdx.x < ntiles) ? (ntiles - blockIdx.x + gridDim.x - 1) / gridDim.x : 0;
    const int64_t n_iter = my_tiles * panels;
    const int64_t n_own = (n_iter + 1 - grp) / 2;
    const int tile_step = (panels == 1) ? 2 : 1;  // distance to the next tile this group touches
    // issue cursor
    int64_t is_tl = 0, cur_tl = -1;
    int is_pi = grp, is_s = grp, cs = grp;
    uint32_t is_ph = 0;
    while (is_pi >= panels) { is_pi -= panels; ++is_tl; }
    bool ok[2] = {false, false};
    const float *src_u[2] = {nullptr, nullptr}, *src_i[2] = {nullptr, nullptr};
    int64_t pre_u[2] = {-1, -1}, pre_it[2] = {-1, -1};  // indices of the group's next tile, fetched a tile early
    auto prefetch_idx = [&](int64_t tl) {
#pragma unroll
      for (int j = 0; j < 2; ++j) {
        pre_u[j] = -1;
        pre_it[j] = -1;
        const int64_t row = (blockIdx.x + tl * gridDim.x) * kTile + r0 + 64 * j;
        if (tl < my_tiles && row < p.B) {
          pre_u[j] = p.user[p.user_div > 0 ? row / p.user_div : row];
          pre_it[j] = p.item[row];
        }
      }
    };
    auto enter_tile = [&](int64_t tl) {
#pragma unroll
      for (int j = 0; j < 2; ++j) {
        const int64_t row = (blockIdx.x + tl * gridDim.x) * kTile + r0 + 64 * j;
        ok[j] = row < p.B;
        if (g.gather) {
          const int64_t uu = pre_u[j], it = pre_it[j];
          if (uu < 0 || uu >= p.U || it < 0 || it >= p.I) ok[j] = false;
          else { src_u[j] = p.eum + uu * d; src_i[j] = p.eim + it * d; }
        } else if (ok[j]) {
          src_u[j] = g.a + row * (int64_t)K;
        }
      }
      if (g.gather) prefetch_idx(tl + tile_step);
    };
    // blocking == false: copy only if the stage is already free (returns whether it did)
    auto issue = [&](bool blocking) -> bool {
      if (blocking) mbar_wait_warp(&bars.empty[is_s], is_ph ^ 1);
      else if (!mbar_test_warp(&bars.empty[is_s], is_ph ^ 1)) return false;
      if (is_tl != cur_tl) { enter_tile(is_tl); cur_tl = is_tl; }
      uint8_t* st = smem + (size_t)is_s * stage_bytes;
      const int c0 = is_pi * 32;
#pragma unroll
      for (int j = 0; j < 2; ++j) {
        const int r = r0 + 64 * j;
        const float* src = nullptr;
        if (ok[j]) src = g.gather ? (c0 < d ? src_u[j] + c0 : src_i[j] + (c0 - d)) : src_u[j] + c0;
#pragma unroll
        for (int c = 0; c < 4; ++c) {
          const int piece = 2 * c + hq;
          const bool valid = src != nullptr && c0 + piece * 4 < K;
          cp_async16_zfill(st + r * 128 + ((piece ^ (r & 7)) << 4), valid ? src + piece * 4 : g.b_img, valid);
        }
      }
      asm volatile("cp.async.commit_group;" ::: "memory");
      is_pi += 2;
      while (is_pi >= panels) { is_pi -= panels; ++is_tl; }
      is_s += 2;
      if (is_s >= g.stages) { is_s -= g.stages; is_ph ^= 1; }
      return true;
    };
    auto consume = [&](bool more_pending) {
      if (more_pending) asm volatile("cp.async.wait_group 1;" ::: "memory");
      else asm volatile("cp.async.wait_group 0;" ::: "memory");
      uint8_t* st = smem + (size_t)cs * stage_bytes;
      if (g.passes == 3) {
#pragma unroll
        for (int j = 0; j < 2; ++j) {
          const int r = r0 + 64 * j;
#pragma unroll
          for (int c = 0; c < 4; ++c) {
            const int off = r * 128 + (((2 * c + hq) ^ (r & 7)) << 4);
            float4 hi, lo;
            split4(*reinterpret_cast<const float4*>(st + off), hi, lo);
            *reinterpret_cast<float4*>(st + a_bytes + off) = lo;
          }
        }
      }
      fence_async_smem();
      mbar_arrive_warp(&bars.full[cs]);
      cs += 2;
      if (cs >= g.stages) cs -= g.stages;
    };
    if (g.gather) prefetch_idx(is_tl);
    // The next own panel is copied before this one is split only when its stage is already free:
    // a blocking wait there would hold back the hand-off of the panel the MMA warp is waiting for.
    if (n_own > 0) issue(true);
    for (int64_t k = 0; k < n_own; ++k) {
      const bool more = k + 1 < n_own;
      const bool early = more && g.stages >= 3 && issue(false);
      consume(early);
      if (more && !early) issue(true);
    }
  } else if (warp == kLoaderWarp) {
    // ===== weight-panel loader: one thread, bulk copies of the pre-split (hi, lo) images ======================
    if (lane == 0) {
      const int64_t my_tiles = (blockIdx.x < ntiles) ? (ntiles - blockIdx.x + gridDim.x - 1) / gridDim.x : 0;
      const int64_t n_iter = my_tiles * panels;
      int s = 0, pi = 0;
      uint32_t ph = 0;
      for (int64_t i = 0; i < n_iter; ++i) {
        mbar_wait(&bars.empty[s], ph ^ 1);
        uint8_t* st = smem + (size_t)s * stage_bytes;
        const float* bsrc = g.b_img + (int64_t)pi * 2 * g.n_total * 32 + (int64_t)nb * N * 32;
        if (g.passes == 3) {
          mbar_expect_tx(&bars.full[s], 2 * b_bytes);
          bulk_g2s(st + 2 * a_bytes, bsrc, b_bytes, &bars.full[s]);
          bulk_g2s(st + 2 * a_bytes + b_bytes, bsrc + (int64_t)g.n_total * 32, b_bytes, &bars.full[s]);
        } else {
          mbar_expect_tx(&bars.full[s], b_bytes);
          bulk_g2s(st + 2 * a_bytes, bsrc, b_bytes, &bars.full[s]);
        }
        if (++pi == panels) pi = 0;
        if (++s == g.stages) { s = 0; ph ^= 1; }
      }
    }
  } else if (warp == kProducerWarps) {
    // ===== MMA issuer =======================================================================================
    if (lane == 0) {
      const uint32_t idesc = make_idesc(kTile, N, 0, 0);
      uint32_t lt = 0, ph = 0;
      int s = 0;
      for (int64_t tile = blockIdx.x; tile < ntiles; tile += gridDim.x, ++lt) {
        const int a = lt & 1;
        mbar_wait(&bars.acc_empty[a], ((lt >> 1) & 1) ^ 1);
        tc_fence_after();
        const uint32_t d_tmem = tmem + a * N;
        for (int pi = 0; pi < panels; ++pi) {
          mbar_wait(&bars.full[s], ph);
          tc_fence_after();
          const uint32_t base = smem_u32(smem + (size_t)s * stage_bytes);
          const uint32_t ahi = base, alo = base + a_bytes, bhi = base + 2 * a_bytes, blo = bhi + b_bytes;
          const int ksteps = min(4, (K - pi * 32) >> 3);
          for (int ks = 0; ks < ksteps; ++ks) {
            const uint64_t dah = make_desc(ahi + ks * 32, 16, 1024, 2);
            const uint64_t dbh = make_desc(bhi + ks * 32, 16, 1024, 2);
            tc_mma(d_tmem, dah, dbh, idesc, (pi > 0 || ks > 0) ? 1u : 0u);
            if (g.passes == 3) {
              const uint64_t dal = make_desc(alo + ks * 32, 16, 1024, 2);
              const uint64_t dbl = make_desc(blo + ks * 32, 16, 1024, 2);
              tc_mma(d_tmem, dal, dbh, idesc, 1u);
              tc_mma(d_tmem, dah, dbl, idesc, 1u);
            }
          }
          tc_commit(&bars.empty[s]);
          if (++s == g.stages) { s = 0; ph ^= 1; }
        }
        tc_commit(&bars.acc_full[a]);
      }
    }
  } else {
    // ===== epilogue: warp quarter q owns TMEM lanes [32q, 32q+32) ============================================
    const int q = warp & 3;
    const int grp = (warp - kProducerWarps - 1) >> 2;  // epilogue group: even / odd local tiles
    const int f = p.f, dmlp = p.d;
    const int mlp_off = (p.type == NCF_NEUMF) ? f : 0;
    const bool has_gmf = p.type != NCF_MLP;
    uint32_t lt = 0;
    for (int64_t tile = blockIdx.x; tile < ntiles; tile += gridDim.x, ++lt) {
      const int a = lt & 1;
      if (a != grp) continue;
      mbar_wait_warp(&bars.acc_full[a], (lt >> 1) & 1);
      tc_fence_after();
      const int64_t row = tile * kTile + q * 32 + lane;
      const bool valid = row < p.B;
      const uint32_t taddr = tmem + ((uint32_t)(q * 32) << 16) + a * N;
      float v[32];

      if (EPI == EPI_RELU_STORE) {
        float* out = g.out + row * (int64_t)g.n_total + nb * N;
        const float* bias = g.bias + nb * N;
        for (int c0 = 0; c0 < N; c0 += 32) {
          tc_ld32(taddr + c0, v);
          if (valid) {
#pragma unroll
            for (int j = 0; j < 32; j += 4) {
              const float4 bb = ldg4(bias + c0 + j);
              *reinterpret_cast<float4*>(out + c0 + j) =
                  make_float4(fmaxf(v[j] + bb.x, 0.f), fmaxf(v[j + 1] + bb.y, 0.f),
                              fmaxf(v[j + 2] + bb.z, 0.f), fmaxf(v[j + 3] + bb.w, 0.f));
            }
          }
        }
      } else if (EPI == EPI_MASK_STORE) {
        float* out = g.out + row * (int64_t)g.n_total + nb * N;
        const float* h = g.mask_src + row * (int64_t)g.n_total + nb * N;
        for (int c0 = 0; c0 < N; c0 += 32) {
          tc_ld32(taddr + c0, v);
          if (valid) {
#pragma unroll
            for (int j = 0; j < 32; j += 4) {
              const float4 hh = ldg4(h + c0 + j);
              *reinterpret_cast<float4*>(out + c0 + j) =
                  make_float4(hh.x > 0.f ? v[j] : 0.f, hh.y > 0.f ? v[j + 1] : 0.f,
                              hh.z > 0.f ? v[j + 2] : 0.f, hh.w > 0.f ? v[j + 3] : 0.f);
            }
          }
        }
      } else if (EPI == EPI_SCATTER) {
        int64_t u = -1, it = -1;
        if (valid) {
          u = p.user[p.user_div > 0 ? row / p.user_div : row];
          it = p.item[row];
          if (u < 0 || u >= p.U || it < 0 || it >= p.I) u = -1;
        }
        for (int c0 = 0; c0 < N; c0 += 32) {
          tc_ld32(taddr + c0, v);
          if (u >= 0) {
            const int col = nb * N + c0;
            float* dst = (col < dmlp) ? p.gum + u * dmlp + col : p.gim + it * dmlp + (col - dmlp);
#pragma unroll
            for (int j = 0; j < 32; j += 4) red_add4(dst + j, make_float4(v[j], v[j + 1], v[j + 2], v[j + 3]));
          }
        }
      } else {  // EPI_PREDICT / EPI_PREDICT_TRAIN: N == f (the last tower layer), nb == 0
        constexpr bool TRAIN = (EPI == EPI_PREDICT_TRAIN);
        int64_t u = -1, it = -1;
        bool bad = false;
        if (valid) {
          u = p.user[p.user_div > 0 ? row / p.user_div : row];
          it = p.item[row];
          if (u < 0 || u >= p.U || it < 0 || it >= p.I) { u = -1; bad = true; }
        }
        const bool ok = u >= 0;
        float acc = 0.f;
        for (int c0 = 0; c0 < N; c0 += 32) {
          tc_ld32(taddr + c0, v);
#pragma unroll
          for (int j = 0; j < 32; ++j)
            acc = fmaf(__ldg(&p.pw[mlp_off + c0 + j]), fmaxf(v[j] + __ldg(&g.bias[c0 + j]), 0.f), acc);
        }
        if (has_gmf && ok) {
          const float* ru = p.eug + u * f;
          const float* ri = p.eig + it * f;
          for (int c = 0; c < f; c += 4) {
            const float4 gu = ldg4(ru + c), gi = ldg4(ri + c), w = ldg4(p.pw + c);
            acc = fmaf(w.x, gu.x * gi.x, acc);
            acc = fmaf(w.y, gu.y * gi.y, acc);
            acc = fmaf(w.z, gu.z * gi.z, acc);
            acc = fmaf(w.w, gu.w * gi.w, acc);
          }
        }
        float x = acc + __ldg(p.pb);
        if (bad) x = __int_as_float(0x7fc00000);  // out-of-range index: NaN
        if (valid && p.logits != nullptr) p.logits[row] = x;
        if (TRAIN) {
          float dl = 0.f, ls = 0.f;
          if (ok && p.dlogit_in != nullptr) {
            dl = p.dlogit_in[row];
          } else if (ok) {
            const bool kd = p.teacher != nullptr;
            const SampleLoss r = sample_loss(x, p.label[row], kd, kd ? p.teacher[row] : 0.f, p.alpha, p.invB);
            ls = r.loss;
            dl = r.dlogit;
          }
          const float ls_w = warp_sum(ls), dl_w = warp_sum(dl);
          if (lane == 0) {
            if (p.loss_accum != nullptr) atomicAdd(p.loss_accum, (double)ls_w * (double)p.invB);
            atomicAdd(&bars.pg[p.predict_size], dl_w);
          }
          // delta_L and the predict-weight gradient of the tower half
          float* dz = g.out + row * (int64_t)N;
          for (int c0 = 0; c0 < N; c0 += 32) {
            tc_ld32(taddr + c0, v);
            float z[32];
#pragma unroll
            for (int j = 0; j < 32; ++j) {
              const float h = fmaxf(v[j] + __ldg(&g.bias[c0 + j]), 0.f);
              z[j] = (h > 0.f) ? dl * __ldg(&p.pw[mlp_off + c0 + j]) : 0.f;
              v[j] = dl * h;
            }
            if (valid) {
#pragma unroll
              for (int j = 0; j < 32; j += 4)
                *reinterpret_cast<float4*>(dz + c0 + j) = make_float4(z[j], z[j + 1], z[j + 2], z[j + 3]);
            }
            const float s = warp_colsum32(v, lane);
            atomicAdd(&bars.pg[mlp_off + c0 + lane], s);
          }
          // GMF branch: predict-weight gradient and the scatter into the GMF embedding-gradient rows
          if (has_gmf) {
            for (int c0 = 0; c0 < f; c0 += 32) {
#pragma unroll
              for (int j = 0; j < 32; j += 4) {
                float4 gu = make_float4(0.f, 0.f, 0.f, 0.f), gi = gu;
                if (ok) {
                  gu = ldg4(p.eug + u * f + c0 + j);
                  gi = ldg4(p.eig + it * f + c0 + j);
                  const float4 w = ldg4(p.pw + c0 + j);
                  const float4 wd = make_float4(w.x * dl, w.y * dl, w.z * dl, w.w * dl);
                  red_add4(p.gug + u * f + c0 + j, make_float4(wd.x * gi.x, wd.y * gi.y, wd.z * gi.z, wd.w * gi.w));
                  red_add4(p.gig + it * f + c0 + j, make_float4(wd.x * gu.x, wd.y * gu.y, wd.z * gu.z, wd.w * gu.w));
                }
                v[j] = dl * (gu.x * gi.x);
                v[j + 1] = dl * (gu.y * gi.y);
                v[j + 2] = dl * (gu.z * gi.z);
                v[j + 3] = dl * (gu.w * gi.w);
              }
              const float s = warp_colsum32(v, lane);
              atomicAdd(&bars.pg[c0 + lane], s);
            }
          }
        }
      }
      tc_fence_before();
      mbar_arrive_warp(&bars.acc_empty[a]);
    }
  }
  tc_fence_before();
  __syncthreads();
  if (EPI == EPI_PREDICT_TRAIN)
    for (int i = tid; i <= p.predict_size; i += kGemmThreads) atomicAdd(&p.gt[p.pw_off + i], bars.pg[i]);
  if (warp == kProducerWarps) asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem), "r"(tmem_cols));
}

// ---- fused tower kernel ------------------------------------------------------------------------------
// One 128-sample tile runs the whole tower forward and its backward-data pass without leaving the
// SM: the A operand of every GEMM lives in tensor memory (gathered embedding rows for layer 0, the
// previous epilogue's output for every other GEMM), so shared memory only carries the streamed
// weight panels and the activations never go through shared memory at all.
//   TMEM columns (f=32, L=3: widths 256,128,64,32):
//     H[k] / Lo[k], k = 1..L (W[k] columns each): H[k] accumulates Z_k and then holds X_k (hi);
//     Lo[k] holds X_k (lo), later accumulates dX_k and then holds dZ_k (hi) while dZ_k (lo) replaces
//     X_k in H[k].  Layer 0's gathered panels go through a ring of 64-column stages laid over
//     everything but H[1]; dX_0 accumulates in [2 W[1], 2 W[1] + W[0]).
// Roles: warps 0-7 gather producers (two groups, alternate panels), then the MMA issuers (one thread can
// start a tcgen05.mma only every ~105 cycles and a tf32 MMA covers just K = 8, so the three products
// of the split, hi*hi / lo*hi / hi*lo, are issued by three warps into the same accumulator, which the
// preceding epilogue has zeroed; two such sets take alternate panels), eight epilogue warps (lane
// quarter x column half) and the weight-panel loader warp.  Activations and deltas are also written to
// the HBM scratch for the weight-gradient kernel.
constexpr int kMaxGemms = 2 * NCF_MAX_LAYERS;
constexpr int kRingMax = 6;
constexpr int kBStages = 3;

struct TowerGemm {
  int kind;       // 0 forward layer k, 1 backward-data of layer k
  int k, N, K;
  int a_hi, a_lo; // TMEM columns of the A operand (-1: the gather ring)
  int d_col;      // TMEM column of the accumulator
  int n_total, row0;  // the weight image has n_total rows; this GEMM uses rows [row0, row0 + N)
  int new_operand;    // the A operand was written by the epilogue of the previous GEMM (wait for it)
  const float* img;
};
struct TowerArgs {
  int passes, ng;
  int ring_col, ring_stages;
  int hcol[NCF_MAX_LAYERS + 1], lcol[NCF_MAX_LAYERS + 1];
  TowerGemm gemm[kMaxGemms];
};

struct TowerBars {
  uint64_t a_full[kRingMax], a_empty[kRingMax], b_full[kBStages], b_empty[kBStages];
  uint64_t acc_ready[2], opnd_ready, tile_done, dl_ready;
  uint64_t panel_ready[8];  // 32-column panel c of the operand the running epilogue is producing is in TMEM
  uint32_t tmem_base;
  float pg[2 * 64 + 8];  // predict-layer gradient of this CTA (the fused kernel serves f <= 64)
  float xch[kTile];      // hand-off between the two epilogue warps of a lane quarter: GMF logit, then dlogit
};

__device__ __forceinline__ void tc_st32(uint32_t taddr, const float (&v)[32]) {
  asm volatile(
      "tcgen05.st.sync.aligned.32x32b.x32.b32 [%0], {%1,%2,%3,%4,%5,%6,%7,%8,%9,%10,%11,%12,%13,%14,%15,%16,"
      "%17,%18,%19,%20,%21,%22,%23,%24,%25,%26,%27,%28,%29,%30,%31,%32};"
      ::"r"(taddr), "r"(__float_as_uint(v[0])), "r"(__float_as_uint(v[1])), "r"(__float_as_uint(v[2])),
        "r"(__float_as_uint(v[3])), "r"(__float_as_uint(v[4])), "r"(__float_as_uint(v[5])), "r"(__float_as_uint(v[6])),
        "r"(__float_as_uint(v[7])), "r"(__float_as_uint(v[8])), "r"(__float_as_uint(v[9])), "r"(__float_as_uint(v[10])),
        "r"(__float_as_uint(v[11])), "r"(__float_as_uint(v[12])), "r"(__float_as_uint(v[13])), "r"(__float_as_uint(v[14])),
        "r"(__float_as_uint(v[15])), "r"(__float_as_uint(v[16])), "r"(__float_as_uint(v[17])), "r"(__float_as_uint(v[18])),
        "r"(__float_as_uint(v[19])), "r"(__float_as_uint(v[20])), "r"(__float_as_uint(v[21])), "r"(__float_as_uint(v[22])),
        "r"(__float_as_uint(v[23])), "r"(__float_as_uint(v[24])), "r"(__float_as_uint(v[25])), "r"(__float_as_uint(v[26])),
        "r"(__float_as_uint(v[27])), "r"(__float_as_uint(v[28])), "r"(__float_as_uint(v[29])), "r"(__float_as_uint(v[30])),
        "r"(__float_as_uint(v[31])) : "memory");
}
__device__ __forceinline__ void tc_wait_st() { asm volatile("tcgen05.wait::st.sync.aligned;" ::: "memory"); }
__device__ __forceinline__ void tc_mma_ts(uint32_t d_tmem, uint32_t a_tmem, uint64_t db, uint32_t idesc, uint32_t accumulate) {
  asm volatile(
      "{\n\t.reg .pred p;\n\tsetp.ne.b32 p, %4, 0;\n\t"
      "tcgen05.mma.cta_group::1.kind::tf32 [%0], [%1], %2, %3, p;\n\t}"
      ::"r"(d_tmem), "r"(a_tmem), "l"(db), "r"(idesc), "r"(accumulate) : "memory");
}
__device__ __forceinline__ float lo_of(float x) { return x - __uint_as_float(__float_as_uint(x) & kHiMask); }

// Epilogue threads own one sample row each (TMEM lane), so a plain 16-byte store touches 32 cache
// lines per instruction and the LSU serialises them.  Transposing 8x8 blocks of float4 inside groups
// of 8 lanes (48 shuffles per 32 columns) lets 8 lanes write one full 128-byte line of a row instead:
// on return, v[4i..4i+3] of lane l hold columns [4(l%8), 4(l%8)+4) of the row owned by lane (l & ~7) + i.
__device__ __forceinline__ void quad8_transpose(float (&v)[32], int lane) {
#pragma unroll
  for (int o = 4; o > 0; o >>= 1) {
    const bool upper = (lane & o) != 0;
#pragma unroll
    for (int i = 0; i < 8; ++i) {
      if ((i & o) == 0) {
#pragma unroll
        for (int e = 0; e < 4; ++e) {
          const float send = upper ? v[4 * i + e] : v[4 * (i + o) + e];
          const float recv = __shfl_xor_sync(0xffffffffu, send, o);
          if (upper) v[4 * i + e] = recv; else v[4 * (i + o) + e] = recv;
        }
      }
    }
  }
}
// v after quad8_transpose: this lane's float4 of 8 rows -> dst[row][c0 ..], rows of the warp start at wrow0
__device__ __forceinline__ void store_rows_t(const float (&v)[32], float* dst, int64_t ld, int64_t wrow0, int64_t nrows, int c0, int lane) {
  const int64_t r0 = wrow0 + (lane & ~7);
  float* p0 = dst + r0 * ld + c0 + 4 * (lane & 7);
#pragma unroll
  for (int i = 0; i < 8; ++i)
    if (r0 + i < nrows) *reinterpret_cast<float4*>(p0 + i * ld) = make_float4(v[4 * i], v[4 * i + 1], v[4 * i + 2], v[4 * i + 3]);
}

constexpr int kTowerMmaSets = 1;     // sets of three issuing warps taking alternate panels (2 sets: the 80-register cap of
                                     // 736 threads costs the epilogues more than the issue overlap gains: 215 vs 191 us)
constexpr int kTowerThreads = (8 + 3 * kTowerMmaSets + 8 + 1) * 32;
constexpr int kTowerEpiWarps = 8;
constexpr int kTowerMmaWarp = 8;     // .. + 3 * kTowerMmaSets - 1
constexpr int kTowerEpiWarp0 = kTowerMmaWarp + 3 * kTowerMmaSets;
constexpr int kTowerLoaderWarp = kTowerEpiWarp0 + kTowerEpiWarps;

template <bool TRAIN>
__global__ void __launch_bounds__(kTowerThreads, 1)
umma_tower_kernel(const __grid_constant__ TileParams p, const __grid_constant__ TowerArgs g) {
  extern __shared__ __align__(1024) uint8_t smem_raw[];
  __shared__ TowerBars bars;
  uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~(uintptr_t)1023);
  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  const int L = p.L;
  const int64_t ntiles = (p.B + kTile - 1) / kTile;
  const int64_t my_tiles = (blockIdx.x < ntiles) ? (ntiles - blockIdx.x + gridDim.x - 1) / gridDim.x : 0;
  const int P0 = p.W[0] >> 5;               // gathered panels per tile
  const uint32_t b_stage = 128u * 256u;     // largest panel: 128 rows x (hi + lo) x 128 B
  uint8_t* land = smem + kBStages * b_stage;  // landing zone of the gathered rows: [panel][row][128 B], swizzled
  const int NA = g.ring_stages;

  if (tid == 0) {
    const int nm = (g.passes == 3) ? 3 : 1;  // MMA-issuing warps, each commits for its own instructions
    for (int s = 0; s < NA; ++s) { mbar_init(&bars.a_full[s], 4); mbar_init(&bars.a_empty[s], nm); }
    for (int s = 0; s < kBStages; ++s) { mbar_init(&bars.b_full[s], 1); mbar_init(&bars.b_empty[s], nm); }
    mbar_init(&bars.acc_ready[0], nm * kTowerMmaSets);
    mbar_init(&bars.acc_ready[1], nm * kTowerMmaSets);
    mbar_init(&bars.opnd_ready, kTowerEpiWarps);
    for (int c = 0; c < 8; ++c) mbar_init(&bars.panel_ready[c], 4);  // one warp per lane quarter
    mbar_init(&bars.tile_done, kTowerEpiWarps);
    mbar_init(&bars.dl_ready, kTowerEpiWarps / 2);
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  }
  for (int i = tid; i < 2 * 64 + 8; i += kTowerThreads) bars.pg[i] = 0.f;
  if (warp == 8) {
    asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], 512;" ::"r"(smem_u32(&bars.tmem_base)));
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;");
  }
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem = bars.tmem_base;

  if (warp < 8) {
    // ===== gather producers: thread = sample row (TMEM lane), group = parity of the panel ===================
    // The rows of the NEXT tile are copied into the landing zone (cp.async, one commit group per panel)
    // while this tile runs, so the gather latency is off the critical path: moving a panel into the
    // TMEM ring is a shared-memory read of the thread's own row.
    const int grp = warp >> 2, q = warp & 3;
    const int r = q * 32 + lane;
    const int d = p.d;
    const int own = P0 / 2;  // own panels per tile: grp, grp + 2, ...
    const uint32_t lane_addr = tmem + ((uint32_t)(q * 32) << 16);
    int s = grp;            // ring stage of the next own panel (flat over tiles: P0 is even)
    uint32_t ph = 0;
    auto copy_panel = [&](int64_t tl, int pi, int64_t uu, int64_t ii) {
      const bool ok = tl < my_tiles && uu >= 0 && uu < p.U && ii >= 0 && ii < p.I;
      const int c0 = pi * 32;
      const float* src = p.eum;
      if (ok) src = (c0 < d) ? p.eum + uu * d + c0 : p.eim + ii * d + (c0 - d);
      uint8_t* dst = land + pi * (kTile * 128) + r * 128;
#pragma unroll
      for (int c = 0; c < 8; ++c) cp_async16_zfill(dst + ((c ^ (r & 7)) << 4), src + c * 4, ok);
      asm volatile("cp.async.commit_group;" ::: "memory");
    };
    auto row_idx = [&](int64_t tl, int64_t& uu, int64_t& ii) {
      uu = -1;
      ii = -1;
      const int64_t row = (blockIdx.x + tl * gridDim.x) * kTile + r;
      if (tl < my_tiles && row < p.B) {
        uu = p.user[p.user_div > 0 ? row / p.user_div : row];
        ii = p.item[row];
      }
    };
    int64_t nu, nit;
    row_idx(0, nu, nit);
    for (int j = 0; j < own; ++j) copy_panel(0, grp + 2 * j, nu, nit);
    const int f = p.f;
    const bool has_gmf = p.type != NCF_MLP;
    for (int64_t tl = 0; tl < my_tiles; ++tl) {
      const int64_t u = nu, it = nit;  // this tile's row
      const bool ok = u >= 0 && u < p.U && it >= 0 && it < p.I;
      row_idx(tl + 1, nu, nit);
      // the ring overlays columns the previous tile's backward pass was still using
      mbar_wait_warp(&bars.tile_done, (uint32_t)tl & 1);
      for (int pi = grp; pi < P0; pi += 2) {
        // pending groups: the rest of this tile's own panels, then the next tile's first ones
        if (own == 4) asm volatile("cp.async.wait_group 3;" ::: "memory");
        else if (own == 2) asm volatile("cp.async.wait_group 1;" ::: "memory");
        else asm volatile("cp.async.wait_group 0;" ::: "memory");
        float cur[32];
        const uint8_t* src = land + pi * (kTile * 128) + r * 128;
#pragma unroll
        for (int c = 0; c < 8; ++c) {
          const float4 x = *reinterpret_cast<const float4*>(src + ((c ^ (r & 7)) << 4));
          cur[4 * c] = x.x; cur[4 * c + 1] = x.y; cur[4 * c + 2] = x.z; cur[4 * c + 3] = x.w;
        }
        mbar_wait_warp(&bars.a_empty[s], ph ^ 1);
        tc_fence_after();
        const uint32_t col = lane_addr + g.ring_col + s * 64;
        tc_st32(col, cur);
        if (g.passes == 3) {
#pragma unroll
          for (int j = 0; j < 32; ++j) cur[j] = lo_of(cur[j]);
          tc_st32(col + 32, cur);
        }
        tc_wait_st();
        tc_fence_before();
        mbar_arrive_warp(&bars.a_full[s]);
        // refill the slot this thread has just read with the next tile's row - after the hand-off:
        // the copies would otherwise sit in front of it in the warp's memory-instruction queue
        copy_panel(tl + 1, pi, nu, nit);
        s += 2;
        if (s >= NA) { s -= NA; ph ^= 1; }
      }
      // GMF branch backward (group 0, idle until the next tile): wait for this tile's dloss/dlogit
      if (TRAIN && grp == 0) {
        mbar_wait_warp(&bars.dl_ready, (uint32_t)tl & 1);
        const float dl = bars.xch[r];
        float v[32];
              if (has_gmf) {
                for (int c0 = 0; c0 < f; c0 += 32) {
                  float gu_[32], gi_[32];
#pragma unroll
                  for (int j = 0; j < 32; j += 4) {
                    float4 gu = make_float4(0.f, 0.f, 0.f, 0.f), gi4 = gu;
                    if (ok) {
                      gu = ldg4(p.eug + u * f + c0 + j);
                      gi4 = ldg4(p.eig + it * f + c0 + j);
                    }
                    const float4 w = ldg4(p.pw + c0 + j);
                    const float4 wd = make_float4(w.x * dl, w.y * dl, w.z * dl, w.w * dl);
                    v[j] = dl * (gu.x * gi4.x);
                    v[j + 1] = dl * (gu.y * gi4.y);
                    v[j + 2] = dl * (gu.z * gi4.z);
                    v[j + 3] = dl * (gu.w * gi4.w);
                    gu_[j] = wd.x * gi4.x; gu_[j + 1] = wd.y * gi4.y; gu_[j + 2] = wd.z * gi4.z; gu_[j + 3] = wd.w * gi4.w;
                    gi_[j] = wd.x * gu.x; gi_[j + 1] = wd.y * gu.y; gi_[j + 2] = wd.z * gu.z; gi_[j + 3] = wd.w * gu.w;
                  }
                  const float s = warp_colsum32(v, lane);
                  atomicAdd(&bars.pg[c0 + lane], s);
                  // full-line REDs: 8 lanes per embedding-gradient row
                  quad8_transpose(gu_, lane);
                  quad8_transpose(gi_, lane);
                  const int64_t mu = ok ? u : -1, mi = ok ? it : -1;
#pragma unroll
                  for (int i = 0; i < 8; ++i) {
                    const int64_t ru = __shfl_sync(0xffffffffu, mu, (lane & ~7) + i);
                    const int64_t ri = __shfl_sync(0xffffffffu, mi, (lane & ~7) + i);
                    if (ru >= 0) {
                      red_add4(p.gug + ru * f + c0 + 4 * (lane & 7), make_float4(gu_[4 * i], gu_[4 * i + 1], gu_[4 * i + 2], gu_[4 * i + 3]));
                      red_add4(p.gig + ri * f + c0 + 4 * (lane & 7), make_float4(gi_[4 * i], gi_[4 * i + 1], gi_[4 * i + 2], gi_[4 * i + 3]));
                    }
                  }
                }
              }
      }
    }
    asm volatile("cp.async.wait_group 0;" ::: "memory");
  } else if (warp == kTowerLoaderWarp) {
    // ===== weight-panel loader ==================================================================================
    if (lane == 0) {
      int s = 0;
      uint32_t ph = 0;
      for (int64_t tl = 0; tl < my_tiles; ++tl)
        for (int gi = 0; gi < g.ng; ++gi) {
          const TowerGemm& G = g.gemm[gi];
          const int panels = G.K >> 5;
          const uint32_t bytes = (uint32_t)G.N * (g.passes == 3 ? 256u : 128u);
          for (int pi = 0; pi < panels; ++pi) {
            mbar_wait(&bars.b_empty[s], ph ^ 1);
            const float* src = G.img + (int64_t)pi * 2 * G.n_total * 32 + (int64_t)G.row0 * 32;
            uint8_t* dst = smem + (size_t)s * b_stage;
            if (G.N == G.n_total) {  // hi and lo of the panel are contiguous
              mbar_expect_tx(&bars.b_full[s], bytes);
              bulk_g2s(dst, src, bytes, &bars.b_full[s]);
            } else {
              mbar_expect_tx(&bars.b_full[s], bytes);
              bulk_g2s(dst, src, (uint32_t)G.N * 128, &bars.b_full[s]);
              if (g.passes == 3)
                bulk_g2s(dst + G.N * 128, src + (int64_t)G.n_total * 32, (uint32_t)G.N * 128, &bars.b_full[s]);
            }
            if (++s == kBStages) { s = 0; ph ^= 1; }
          }
        }
    }
  } else if (warp >= kTowerMmaWarp && warp < kTowerEpiWarp0) {
    // ===== MMA issuers: per set, one warp each for hi*hi, lo*hi, hi*lo (accumulators are pre-zeroed); the
    // sets take alternate panels, so the ~0.7 k cycles of barrier waits per panel of one set overlap the
    // issue of the other ===========================================================================================
    const int pass = (warp - kTowerMmaWarp) % 3, set = (warp - kTowerMmaWarp) / 3;
    if (lane == 0 && (pass == 0 || g.passes == 3)) {
      int sa = 0, sb = 0;
      uint32_t pha = 0, phb = 0, n_opnd = 0, n_panel = 0, ppar = 0;
      for (int64_t tl = 0; tl < my_tiles; ++tl)
        for (int gi = 0; gi < g.ng; ++gi) {
          const TowerGemm& G = g.gemm[gi];
          const int panels = G.K >> 5;
          const uint32_t idesc = make_idesc(kTile, G.N, 0, 0);
          const uint32_t d_tmem = tmem + G.d_col;
          if (G.new_operand) {  // operand written by the previous epilogue
            mbar_wait(&bars.opnd_ready, n_opnd & 1);
            ++n_opnd;
            tc_fence_after();
          }
          for (int pi = 0; pi < panels; ++pi, ++n_panel) {
            if ((int)(n_panel % kTowerMmaSets) != set) {  // the other set's panel: only keep the ring cursors in step
              if (G.a_hi >= 0 && G.new_operand) ppar ^= 1u << pi;
              if (G.a_hi < 0 && ++sa == NA) { sa = 0; pha ^= 1; }
              if (++sb == kBStages) { sb = 0; phb ^= 1; }
              continue;
            }
            uint32_t a_hi, a_lo;
            if (G.a_hi < 0) {
              mbar_wait(&bars.a_full[sa], pha);
              a_hi = tmem + g.ring_col + sa * 64;
              a_lo = a_hi + 32;
            } else {
              if (G.new_operand) {  // the epilogue hands its output over panel by panel
                mbar_wait(&bars.panel_ready[pi], (ppar >> pi) & 1);
                ppar ^= 1u << pi;
              }
              a_hi = tmem + G.a_hi + pi * 32;
              a_lo = tmem + G.a_lo + pi * 32;
            }
            mbar_wait(&bars.b_full[sb], phb);
            tc_fence_after();
            const uint32_t bhi = smem_u32(smem + (size_t)sb * b_stage);
            // the k-step only moves the start-address field of the descriptor (32 B = 2 units of 16 B)
            const uint64_t dbh0 = make_desc(bhi, 16, 1024, 2);
            const uint64_t dbl0 = make_desc(bhi + (uint32_t)G.N * 128, 16, 1024, 2);
            const uint32_t a_op = (pass == 1) ? a_lo : a_hi;
            const uint64_t b_op = (pass == 2) ? dbl0 : dbh0;
#pragma unroll
            for (int ks = 0; ks < 4; ++ks) tc_mma_ts(d_tmem, a_op + ks * 8, b_op + 2 * ks, idesc, 1u);
            if (G.a_hi < 0) {
              tc_commit(&bars.a_empty[sa]);
              if (++sa == NA) { sa = 0; pha ^= 1; }
            }
            tc_commit(&bars.b_empty[sb]);
            if (++sb == kBStages) { sb = 0; phb ^= 1; }
          }
          tc_commit(&bars.acc_ready[gi & 1]);
        }
    }
  } else {
    // ===== epilogue warps: lane quarter q, column half hf ============================================================
    const int q = warp & 3, hf = (warp - kTowerEpiWarp0) >> 2;
    const int f = p.f, dmlp = p.d;
    const int mlp_off = (p.type == NCF_NEUMF) ? f : 0;
    const bool has_gmf = p.type != NCF_MLP;
    const uint32_t lane_addr = tmem + ((uint32_t)(q * 32) << 16);
    uint32_t n_acc[2] = {0, 0};
    float v[32];
    // every MMA accumulates: the accumulator of a GEMM is cleared by the epilogue that precedes it
    auto zero_cols = [&](int col, int n) {
      const int nchunk = n >> 5;
      const int c_begin = (nchunk >= 2) ? hf * (nchunk / 2) * 32 : 0;
      const int c_end = (nchunk >= 2) ? (hf + 1) * (nchunk / 2) * 32 : (hf == 0 ? n : 0);
      float z[32];
#pragma unroll
      for (int j = 0; j < 32; ++j) z[j] = 0.f;
      for (int c0 = c_begin; c0 < c_end; c0 += 32) tc_st32(lane_addr + col + c0, z);
    };
    zero_cols(g.gemm[0].d_col, g.gemm[0].N);
    tc_wait_st();
    tc_fence_before();
    mbar_arrive_warp(&bars.tile_done);  // phase 0: "the tile before the first one is done"
    for (int64_t tl = 0; tl < my_tiles; ++tl) {
      const int64_t row = (blockIdx.x + tl * gridDim.x) * kTile + q * 32 + lane;
      const bool valid = row < p.B;
      int64_t u = -1, it = -1;
      bool bad = false;
      if (valid) {
        u = p.user[p.user_div > 0 ? row / p.user_div : row];
        it = p.item[row];
        if (u < 0 || u >= p.U || it < 0 || it >= p.I) { u = -1; bad = true; }
      }
      const bool ok = u >= 0;
      float dl = 0.f, pre_label = 0.f, pre_teacher = 0.f;
      for (int gi = 0; gi < g.ng; ++gi) {
        const TowerGemm& G = g.gemm[gi];
        float gd = 0.f;
        if (G.kind == 0 && G.k + 1 == L) {
          // while the last layer is still running: half 1 gathers the GMF rows and reduces the GMF part
          // of the logit, half 0 fetches the label
          if (hf == 1) {
            if (has_gmf && ok) {
              const float* ru = p.eug + u * f;
              const float* ri = p.eig + it * f;
              for (int c = 0; c < f; c += 4) {
                const float4 gu = ldg4(ru + c), gi4 = ldg4(ri + c), w = ldg4(p.pw + c);
                gd = fmaf(w.x, gu.x * gi4.x, gd);
                gd = fmaf(w.y, gu.y * gi4.y, gd);
                gd = fmaf(w.z, gu.z * gi4.z, gd);
                gd = fmaf(w.w, gu.w * gi4.w, gd);
              }
            }
          } else if (TRAIN && ok && p.dlogit_in == nullptr) {
            pre_label = p.label[row];
            if (p.teacher != nullptr) pre_teacher = p.teacher[row];
          }
        }
        mbar_wait_warp(&bars.acc_ready[gi & 1], n_acc[gi & 1] & 1);
        ++n_acc[gi & 1];
        tc_fence_after();
        // published only now: the accumulator of this tile's last layer is ready, so its layer-0 panels
        // have been supplied, so gather group 0 is done reading the previous tile's dlogit from xch[]
        if (G.kind == 0 && G.k + 1 == L && hf == 1) bars.xch[q * 32 + lane] = gd;
        // First clear the accumulators of the GEMMs that consume this epilogue's output (every MMA
        // accumulates) and let them start: they then follow this epilogue panel by panel.
        // (a one-layer tower in inference has a single GEMM: its accumulator is the one this epilogue is
        // about to read, so it is cleared after the read instead)
        const bool zero_late = (gi + 1 == g.ng) && G.d_col == g.gemm[0].d_col;
        if (gi + 1 == g.ng) {
          if (!zero_late) {
            zero_cols(g.gemm[0].d_col, g.gemm[0].N);
            tc_wait_st();
          }
        } else if (g.gemm[gi + 1].new_operand) {
          for (int gj = gi + 1; gj < g.ng && (gj == gi + 1 || !g.gemm[gj].new_operand); ++gj)
            zero_cols(g.gemm[gj].d_col, g.gemm[gj].N);
          tc_wait_st();
          tc_fence_before();
          mbar_arrive_warp(&bars.opnd_ready);
        }
        const int N = G.N, k = G.k;
        // column range of this warp: half of the accumulator, whole 32-column chunks
        const int nchunk = N >> 5;
        const int c_begin = (nchunk >= 2) ? hf * (nchunk / 2) * 32 : 0;
        const int c_end = (nchunk >= 2) ? (hf + 1) * (nchunk / 2) * 32 : (hf == 0 ? N : 0);
        // The branch order steers ptxas' register allocation at the 96-register cap, and was chosen for the
        // training kernel: with the forward layers first it spills 40 more bytes (996 vs 956).  The
        // backward-data branches are compiled into the training kernel only (launch_tower<false> queues
        // forward GEMMs only); in the inference kernel they would cost spills, not just dead code.
        if (G.kind == 0 && k + 1 == L) {
          // ---- last layer + predict layer (+ loss, predict grads, GMF scatter, delta_L) ---------------------
          // The two warps of a lane quarter split the work: half 0 owns the tower side (logit, loss,
          // delta_L), half 1 the GMF branch (its partial logit was computed before the accumulator was
          // ready; the GMF gradients once half 0 has published dloss/dlogit).
          const int trow = q * 32 + lane;
          if (hf == 0) {
            const float* bias = p.b[k];
            float acc = 0.f;
            for (int c0 = 0; c0 < N; c0 += 32) {
              tc_ld32(lane_addr + g.hcol[L] + c0, v);
#pragma unroll
              for (int j = 0; j < 32; ++j)
                acc = fmaf(__ldg(&p.pw[mlp_off + c0 + j]), fmaxf(v[j] + __ldg(&bias[c0 + j]), 0.f), acc);
            }
            named_bar(1 + q, 64);  // half 1 has written the GMF partial logit
            float x = acc + bars.xch[trow] + __ldg(p.pb);
            if (bad) x = __int_as_float(0x7fc00000);  // out-of-range index: NaN
            if (valid && p.logits != nullptr) p.logits[row] = x;
            if (TRAIN) {
              float ls = 0.f;
              if (ok && p.dlogit_in != nullptr) {
                dl = p.dlogit_in[row];
              } else if (ok) {
                const SampleLoss r = sample_loss(x, pre_label, p.teacher != nullptr, pre_teacher, p.alpha, p.invB);
                ls = r.loss;
                dl = r.dlogit;
              }
              bars.xch[trow] = dl;
              mbar_arrive_warp(&bars.dl_ready);  // the GMF-branch gradients are the idle gather warps' job
              const float ls_w = warp_sum(ls), dl_w = warp_sum(dl);
              if (lane == 0) {
                if (p.loss_accum != nullptr) atomicAdd(p.loss_accum, (double)ls_w * (double)p.invB);
                atomicAdd(&bars.pg[p.predict_size], dl_w);
              }
              for (int c0 = 0; c0 < N; c0 += 32) {
                tc_ld32(lane_addr + g.hcol[L] + c0, v);
                float z[32];
#pragma unroll
                for (int j = 0; j < 32; ++j) {
                  const float h = fmaxf(v[j] + __ldg(&bias[c0 + j]), 0.f);
                  z[j] = (h > 0.f) ? dl * __ldg(&p.pw[mlp_off + c0 + j]) : 0.f;
                  v[j] = dl * h;
                }
                tc_st32(lane_addr + g.hcol[L] + c0, z);
                const float s = warp_colsum32(v, lane);
                atomicAdd(&bars.pg[mlp_off + c0 + lane], s);
                if (g.passes == 3) {
#pragma unroll
                  for (int j = 0; j < 32; ++j) v[j] = lo_of(z[j]);
                  tc_st32(lane_addr + g.lcol[L] + c0, v);
                }
                quad8_transpose(z, lane);
                tc_wait_st();
                tc_fence_before();
                mbar_arrive_warp(&bars.panel_ready[c0 >> 5]);
                store_rows_t(z, p.delta[L], N, row - lane, p.B, c0, lane);
              }
            }
          } else {
            named_bar(1 + q, 64);
          }
        } else if (G.kind == 0) {
          // ---- forward layer: X = relu(Z + b) -> scratch, TMEM hi (in place) and lo ------------------------
          const int kk = k + 1;
          const float* bias = p.b[k];
          for (int c0 = c_begin; c0 < c_end; c0 += 32) {
            tc_ld32(lane_addr + g.hcol[kk] + c0, v);
#pragma unroll
            for (int j = 0; j < 32; ++j) v[j] = fmaxf(v[j] + __ldg(&bias[c0 + j]), 0.f);
            tc_st32(lane_addr + g.hcol[kk] + c0, v);
            if (g.passes == 3) {
              float lo[32];
#pragma unroll
              for (int j = 0; j < 32; ++j) lo[j] = lo_of(v[j]);
              tc_st32(lane_addr + g.lcol[kk] + c0, lo);
            }
            if (TRAIN) quad8_transpose(v, lane);  // shuffle work while the TMEM stores drain
            tc_wait_st();
            tc_fence_before();
            mbar_arrive_warp(&bars.panel_ready[c0 >> 5]);
            if (TRAIN) store_rows_t(v, p.act[kk], N, row - lane, p.B, c0, lane);
          }

        } else if (TRAIN && k > 0) {
          // ---- backward data: dZ_k = dX_k * (X_k > 0) -> scratch, TMEM hi (in place) and lo (over X_k) --------
          for (int c0 = c_begin; c0 < c_end; c0 += 32) {
            float x[32];
            tc_ld32(lane_addr + g.lcol[k] + c0, v);
            tc_ld32(lane_addr + g.hcol[k] + c0, x);
#pragma unroll
            for (int j = 0; j < 32; ++j) v[j] = (x[j] > 0.f) ? v[j] : 0.f;
            tc_st32(lane_addr + g.lcol[k] + c0, v);
            if (g.passes == 3) {
#pragma unroll
              for (int j = 0; j < 32; ++j) x[j] = lo_of(v[j]);
              tc_st32(lane_addr + g.hcol[k] + c0, x);
            }
            quad8_transpose(v, lane);
            tc_wait_st();
            tc_fence_before();
            mbar_arrive_warp(&bars.panel_ready[c0 >> 5]);
            store_rows_t(v, p.delta[k], N, row - lane, p.B, c0, lane);
          }
        } else if (TRAIN) {
          // ---- backward data of layer 0: scatter into the embedding-gradient rows -------------------------------
          for (int c0 = c_begin; c0 < c_end; c0 += 32) {
            tc_ld32(lane_addr + G.d_col + c0, v);
            quad8_transpose(v, lane);  // 8 lanes now hold one full 128-byte line of a row
            const int col = G.row0 + c0;
            const bool to_user = col < dmlp;
            const int64_t my_idx = ok ? (to_user ? u : it) : -1;
            float* tab = (to_user ? p.gum + col : p.gim + (col - dmlp)) + 4 * (lane & 7);
#pragma unroll
            for (int i = 0; i < 8; ++i) {
              const int64_t idx = __shfl_sync(0xffffffffu, my_idx, (lane & ~7) + i);
              if (idx >= 0) red_add4(tab + idx * dmlp, make_float4(v[4 * i], v[4 * i + 1], v[4 * i + 2], v[4 * i + 3]));
            }
          }
        }
        if (zero_late) zero_cols(g.gemm[0].d_col, g.gemm[0].N);  // both halves are past the named barrier: the read is over
        tc_wait_st();
        tc_fence_before();
        if (gi + 1 == g.ng) mbar_arrive_warp(&bars.tile_done);
      }
    }
  }
  tc_fence_before();
  __syncthreads();
  if (TRAIN)
    for (int i = tid; i <= p.predict_size; i += kTowerThreads) atomicAdd(&p.gt[p.pw_off + i], bars.pg[i]);
  if (warp == 8) asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, 512;" ::"r"(tmem));
}

// ---- weight-gradient kernel -----------------------------------------------------------------------------
// dW_k[n][c] = sum_s delta[k+1][s][n] * act[k][s][c].  The reduction runs over samples, the slow
// dimension of both operands, so both are MN-major: image rows = samples (128 B = 32 features per
// row and panel), 4-row atoms with the 32-byte chunk index ^= row % 4 (128B_BASE32B, the only
// MN-major layout the tf32 kind accepts).  One CTA owns one [<=128 x <=256] block of one layer's dW
// for its share of the batch; the accumulator stays in TMEM until the CTA's last chunk.
constexpr int kWgProducerWarps = 8;
constexpr int kWgProducers = kWgProducerWarps * 32;
constexpr int kWgradThreads = kWgProducers + 96;  // + three MMA-issuing warps (one per product of the split)

constexpr int kWgStages = 2;  // measured at the bench workload: 2 x 96 KB 79 us, 3 x 72 KB 86 us, 4 x 48 KB 104 us:
                              // the hand-off per chunk costs more than the copies it would hide
struct WgradBars {
  uint64_t full[kWgStages], empty[kWgStages], acc_full;
  uint32_t tmem_base;
  float db[128];
};

// byte offset of feature fo (multiple of 4) of sample row s in an image of S rows per panel
__device__ __forceinline__ uint32_t mn_offset(int s, int fo, int S) {
  const int panel = fo >> 5, cc = fo & 31;
  return (uint32_t)(panel * (S * 128) + s * 128 + (((cc >> 3) ^ (s & 3)) << 5) + ((cc & 7) << 2));
}

__global__ void __launch_bounds__(kWgradThreads, 1)
umma_wgrad_kernel(const __grid_constant__ TileParams p, const __grid_constant__ WgradArgs g) {
  extern __shared__ __align__(1024) uint8_t smem_raw[];
  __shared__ WgradBars bars;
  uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~(uintptr_t)1023);
  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  int ji = 0;
  while (ji + 1 < g.njobs && (int)blockIdx.x >= g.job[ji + 1].cta0) ++ji;
  const WgradJob job = g.job[ji];
  const int k = job.k, kin = p.W[k], nout = p.W[k + 1];
  const int MB = min(128, nout - job.mb * 128), NB = min(256, kin - job.nb * 256);
  const int local = (int)blockIdx.x - job.cta0;
  const int S = job.S;
  const int64_t nchunks = (p.B + S - 1) / S;
  const uint32_t a_img = (uint32_t)MB * S * 4, b_img = (uint32_t)NB * S * 4;
  const uint32_t stage_bytes = 2 * a_img + 2 * b_img;
  const int64_t my_chunks = (local < nchunks) ? (nchunks - local + job.nctas - 1) / job.nctas : 0;

  if (tid == 0) {
    const int nm = (g.passes == 3) ? 3 : 1;
    for (int s = 0; s < kWgStages; ++s) { mbar_init(&bars.full[s], kWgProducerWarps); mbar_init(&bars.empty[s], nm); }
    mbar_init(&bars.acc_full, nm);
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  }
  if (tid < 128) bars.db[tid] = 0.f;
  if (warp == kWgProducerWarps) {
    asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], 256;" ::"r"(smem_u32(&bars.tmem_base)));
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;");
  }
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem = bars.tmem_base;
  // every MMA accumulates (three warps issue into the same block): clear the accumulator first
  if (warp < kWgProducerWarps) {
    float z[32];
#pragma unroll
    for (int j = 0; j < 32; ++j) z[j] = 0.f;
    for (int c0 = (warp >> 2) * 128; c0 < (warp >> 2) * 128 + 128; c0 += 32)
      tc_st32(tmem + ((uint32_t)((warp & 3) * 32) << 16) + c0, z);
    tc_wait_st();
  }
  tc_fence_before();
  __syncthreads();
  tc_fence_after();

  if (warp < kWgProducerWarps) {
    // Producers: every thread copies its 16-byte pieces of the chunk global -> shared with cp.async
    // (raw fp32 = the "hi" image: the tensor core ignores the low 13 mantissa bits), one chunk ahead
    // of the chunk whose "lo" image it is computing from the pieces it copied itself.
    const int t = tid, d = p.d;
    const float* delta = p.delta[k + 1];
    const float* actk = (k > 0) ? p.act[k] : nullptr;
    const int pa = MB >> 2, pb = NB >> 2;       // 16-byte pieces per sample row
    const int na = S * pa / kWgProducers, nbp = S * pb / kWgProducers;  // pieces per thread and chunk (<= 4, <= 8)
    const int ca = t % pa, sa0 = t / pa, sas = kWgProducers / pa;
    const int cb = t % pb, sb0 = t / pb, sbs = kWgProducers / pb;
    float4 dbsum = make_float4(0.f, 0.f, 0.f, 0.f);
    // layer 0: the activation operand is gathered.  A thread always reads the same 4 columns, so it
    // needs one of the two tables only; its sample indices are fetched one chunk ahead so that the
    // row copies never wait on an index load.
    const int fo = job.nb * 256 + cb * 4;
    const bool from_user = fo < d;
    const int64_t* idx_src = from_user ? p.user : p.item;
    const float* tab = from_user ? p.eum + fo : p.eim + (fo - d);
    const int64_t idx_lim = from_user ? p.U : p.I;
    // two chunks ahead (a chunk's copies are often issued right after the previous chunk's)
    int64_t idx_even[8], idx_odd[8];
    auto issue_idx = [&](int64_t ci, int64_t (&idxv)[8]) {
      const int64_t row0 = (local + ci * job.nctas) * S;
#pragma unroll
      for (int i = 0; i < 8; ++i) {
        const int64_t row = row0 + sb0 + i * sbs;
        idxv[i] = (i < nbp && ci < my_chunks && row < p.B) ? idx_src[row] : -1;
      }
    };
    // blocking == false: copy only if the stage is already free (returns whether it did), so that a
    // busy stage never holds back the hand-off of the chunk the MMA warps are waiting for
    auto issue = [&](int64_t ci, bool blocking) -> bool {
      const int s = (int)(ci % kWgStages);
      const uint32_t par = (uint32_t)((ci / kWgStages) & 1) ^ 1;
      if (blocking) mbar_wait_warp(&bars.empty[s], par);
      else if (!mbar_test_warp(&bars.empty[s], par)) return false;
      uint8_t* st = smem + (size_t)s * stage_bytes;
      const int64_t row0 = (local + ci * job.nctas) * S;
#pragma unroll
      for (int i = 0; i < 4; ++i) {
        if (i < na) {
          const int64_t row = row0 + sa0 + i * sas;
          const bool ok = row < p.B;
          cp_async16_zfill(st + mn_offset(sa0 + i * sas, ca * 4, S),
                           ok ? delta + row * nout + job.mb * 128 + ca * 4 : delta, ok);
        }
      }
#pragma unroll
      for (int i = 0; i < 8; ++i) {
        if (i < nbp) {
          const float* src;
          bool ok;
          if (k == 0) {
            const int64_t ix = (ci & 1) ? idx_odd[i] : idx_even[i];
            ok = ix >= 0 && ix < idx_lim;
            src = ok ? tab + ix * d : tab;
          } else {
            const int64_t row = row0 + sb0 + i * sbs;
            ok = row < p.B;
            src = ok ? actk + row * kin + fo : actk;
          }
          cp_async16_zfill(st + 2 * a_img + mn_offset(sb0 + i * sbs, cb * 4, S), src, ok);
        }
      }
      asm volatile("cp.async.commit_group;" ::: "memory");
      if (k == 0) {
        if (ci & 1) issue_idx(ci + 2, idx_odd);
        else issue_idx(ci + 2, idx_even);
      }
      return true;
    };
    auto consume = [&](int64_t ci, int newer) {  // newer: chunks copied after this one, still allowed to be in flight
      const int s = (int)(ci % kWgStages);
      uint8_t* st = smem + (size_t)s * stage_bytes;
      if (newer >= 3) asm volatile("cp.async.wait_group 3;" ::: "memory");
      else if (newer == 2) asm volatile("cp.async.wait_group 2;" ::: "memory");
      else if (newer == 1) asm volatile("cp.async.wait_group 1;" ::: "memory");
      else asm volatile("cp.async.wait_group 0;" ::: "memory");
#pragma unroll
      for (int i = 0; i < 4; ++i) {
        if (i < na) {
          const uint32_t off = mn_offset(sa0 + i * sas, ca * 4, S);
          const float4 x = *reinterpret_cast<const float4*>(st + off);
          float4 hi, lo;
          split4(x, hi, lo);
          dbsum.x += x.x; dbsum.y += x.y; dbsum.z += x.z; dbsum.w += x.w;
          if (g.passes == 3) *reinterpret_cast<float4*>(st + a_img + off) = lo;
        }
      }
#pragma unroll
      for (int i = 0; i < 8; ++i) {
        if (i < nbp && g.passes == 3) {
          const uint32_t off = 2 * a_img + mn_offset(sb0 + i * sbs, cb * 4, S);
          const float4 x = *reinterpret_cast<const float4*>(st + off);
          float4 hi, lo;
          split4(x, hi, lo);
          *reinterpret_cast<float4*>(st + b_img + off) = lo;
        }
      }
      fence_async_smem();
      mbar_arrive_warp(&bars.full[s]);
    };
    if (k == 0) {
      issue_idx(0, idx_even);
      issue_idx(1, idx_odd);
    }
    int64_t issued = 0;
    for (int64_t ci = 0; ci < my_chunks; ++ci) {
      if (issued == ci) issue(issued++, true);  // nothing staged: wait for the stage
      // run ahead while stages are free, but never block in front of a chunk that is ready to hand off
      while (issued < my_chunks && issued - ci < kWgStages && issue(issued, false)) ++issued;
      consume(ci, (int)(issued - ci - 1));
    }
    // bias gradient: column sums of delta (thread t always sees the same 4 columns)
    if (job.nb == 0) {
      atomicAdd(&bars.db[ca * 4 + 0], dbsum.x);
      atomicAdd(&bars.db[ca * 4 + 1], dbsum.y);
      atomicAdd(&bars.db[ca * 4 + 2], dbsum.z);
      atomicAdd(&bars.db[ca * 4 + 3], dbsum.w);
    }
    named_bar(1, kWgProducers);
    if (job.nb == 0 && t < MB && my_chunks > 0) atomicAdd(&p.gt[p.b_off[k] + job.mb * 128 + t], bars.db[t]);
    // flush the accumulator block: warp w reads TMEM lanes 32*(w%4).., column half w/4
    if (my_chunks > 0) {
      mbar_wait_warp(&bars.acc_full, 0);
      tc_fence_after();
      const int q = warp & 3, part = warp >> 2, parts = min(kWgProducerWarps / 4, NB / 32);
      const int m = q * 32 + lane;
      float* dst = p.gt + p.w_off[k] + (int64_t)(job.mb * 128 + m) * kin + job.nb * 256;
      float v[32];
      for (int c0 = part * (NB / parts); c0 < (part + 1) * (NB / parts) && part < parts; c0 += 32) {
        tc_ld32(tmem + ((uint32_t)(q * 32) << 16) + c0, v);
        if (m < MB) {
#pragma unroll
          for (int j = 0; j < 32; j += 4) red_add4(dst + c0 + j, make_float4(v[j], v[j + 1], v[j + 2], v[j + 3]));
        }
      }
    }
  } else if (lane == 0 && (warp == kWgProducerWarps || g.passes == 3)) {
    const int pass = warp - kWgProducerWarps;  // 0 hi*hi, 1 lo*hi, 2 hi*lo
    const uint32_t idesc = make_idesc(128, NB, 1, 1);
    for (int64_t ci = 0; ci < my_chunks; ++ci) {
      const int s = (int)(ci % kWgStages);
      mbar_wait(&bars.full[s], (uint32_t)(ci / kWgStages) & 1);
      tc_fence_after();
      const uint32_t base = smem_u32(smem + (size_t)s * stage_bytes);
      const uint32_t ahi = base, alo = base + a_img, bhi = base + 2 * a_img, blo = bhi + b_img;
      // the k-step (8 sample rows = 1024 B) only moves the start-address field: +64 units of 16 B
      const uint64_t da0 = make_desc(pass == 1 ? alo : ahi, S * 128, 512, 1);
      const uint64_t db0 = make_desc(pass == 2 ? blo : bhi, S * 128, 512, 1);
      for (int ks = 0; ks < S / 8; ++ks) tc_mma(tmem, da0 + 64 * ks, db0 + 64 * ks, idesc, 1u);
      tc_commit(&bars.empty[s]);
    }
    if (my_chunks > 0) tc_commit(&bars.acc_full);
  }
  tc_fence_before();
  __syncthreads();
  if (warp == kWgProducerWarps) asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, 256;" ::"r"(tmem));
}

// ---- launchers ---------------------------------------------------------------------------------------------
constexpr size_t kSmemBudget = 200 * 1024;

template <int EPI>
int launch_gemm(const TileParams& p, GemmArgs g, int nblocks, cudaStream_t st) {
  const size_t stage = 2 * (size_t)kTile * 128 + 2 * (size_t)g.N * 128;
  int stages = (int)(kSmemBudget / stage);
  if (stages > kMaxStages) stages = kMaxStages;
  if (stages < 2) {
    ncf::set_error("umma gemm: stage of %zu bytes does not fit twice", stage);
    return NCF_ERR_ARG;
  }
  g.stages = stages;
  const size_t smem = stages * stage + 1024;
  auto kern = umma_gemm_kernel<EPI>;
  NCF_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
  const int64_t ntiles = (p.B + kTile - 1) / kTile;
  int64_t grid = ncf::num_sms();
  if (grid > ntiles) grid = ntiles;
  kern<<<dim3((unsigned)grid, (unsigned)nblocks), kGemmThreads, smem, st>>>(p, g);
  NCF_LAUNCH_CHECK("umma_gemm_kernel");
  return NCF_OK;
}

int launch_wgrad(const TileParams& p, int passes, cudaStream_t st) {
  WgradArgs g{};
  g.passes = passes;
  // one job per [128 x 256] block of every layer's dW; CTAs shared out by operand bytes per sample
  double weight[12], total = 0;
  for (int k = 0; k < p.L; ++k) {
    const int mbs = (p.W[k + 1] + 127) / 128, nbs = (p.W[k] + 255) / 256;
    for (int mb = 0; mb < mbs; ++mb)
      for (int nb = 0; nb < nbs; ++nb) {
        if (g.njobs >= 12) {
          ncf::set_error("umma wgrad: too many weight blocks");
          return NCF_ERR_ARG;
        }
        const int MB = std::min(128, p.W[k + 1] - mb * 128), NB = std::min(256, p.W[k] - nb * 256);
        // samples per stage: 96 KB of (hi, lo) images, i.e. 4 + 8 sixteen-byte pieces per producer thread
        int S = std::min(4096 / MB, 8192 / NB) / 8 * 8;
        S = std::max(8, std::min(S, 256));
        g.job[g.njobs] = WgradJob{k, mb, nb, 0, 0, S};
        weight[g.njobs] = 1.0 / S;  // hand-offs per sample; every hand-off costs about the same
        total += weight[g.njobs];
        ++g.njobs;
      }
  }
  const int sms = ncf::num_sms();
  int cta = 0;
  size_t smem = 0;
  for (int j = 0; j < g.njobs; ++j) {
    const int64_t nchunks = (p.B + g.job[j].S - 1) / g.job[j].S;
    int n = (int)(weight[j] / total * sms);
    if (n < 1) n = 1;
    if (n > nchunks) n = (int)nchunks;
    g.job[j].cta0 = cta;
    g.job[j].nctas = n;
    cta += n;
    const int k = g.job[j].k;
    const int MB = std::min(128, p.W[k + 1] - g.job[j].mb * 128), NB = std::min(256, p.W[k] - g.job[j].nb * 256);
    smem = std::max(smem, (size_t)kWgStages * 2 * (MB + NB) * g.job[j].S * 4);
  }
  smem += 1024;  // alignment slack (an M=128 descriptor over a narrow A' image reads on into the same stage)
  NCF_CUDA(cudaFuncSetAttribute(umma_wgrad_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
  umma_wgrad_kernel<<<cta, kWgradThreads, smem, st>>>(p, g);
  NCF_LAUNCH_CHECK("umma_wgrad_kernel");
  return NCF_OK;
}

// Per-launch CUDA-event times of one training step on the tcgen05 path.  Enabled by
// ncf_profile_enable(1), read back with ncf_profile_read.  Profiling synchronises the stream after
// every step: measurement aid, not for production.
struct StepProfile {
  int enabled = 0, n = 0;
  float ms[16];
  const char* name[16];
};
thread_local StepProfile g_profile;

struct StepTimer {
  bool on;
  cudaStream_t st;
  cudaEvent_t ev[32];
  const char* name[32];
  int n = 0;
  static thread_local StepTimer* g_timer;
  StepTimer(cudaStream_t s) : on(g_profile.enabled), st(s) {
    g_timer = this;
    mark("start");
  }
  void mark(const char* what) {
    if (!on || n >= 32) return;
    cudaEventCreate(&ev[n]);
    cudaEventRecord(ev[n], st);
    name[n++] = what;
  }
  ~StepTimer() {
    g_timer = nullptr;
    if (!on) return;
    cudaStreamSynchronize(st);
    g_profile.n = 0;
    for (int i = 1; i < n; ++i) {
      float ms = 0;
      cudaEventElapsedTime(&ms, ev[i - 1], ev[i]);
      if (g_profile.n < 16) {
        g_profile.ms[g_profile.n] = ms;
        g_profile.name[g_profile.n++] = name[i];
      }
    }
    for (int i = 0; i < n; ++i) cudaEventDestroy(ev[i]);
  }
};

thread_local StepTimer* StepTimer::g_timer = nullptr;

GemmArgs forward_args(const TileParams& p, int k, int passes) {
  GemmArgs g{};
  g.K = p.W[k];
  g.n_total = p.W[k + 1];
  g.N = std::min(256, g.n_total);
  g.passes = passes;
  g.layer = k;
  g.gather = (k == 0);
  g.a = (k == 0) ? nullptr : p.act[k];
  g.b_img = p.wsplit_f[k];
  g.bias = p.b[k];
  return g;
}

int tower_forward(TileParams& p, int passes, bool train, cudaStream_t st) {
  for (int k = 0; k < p.L; ++k) {
    GemmArgs g = forward_args(p, k, passes);
    int rc;
    if (k + 1 < p.L) {
      g.out = p.act[k + 1];
      rc = launch_gemm<EPI_RELU_STORE>(p, g, g.n_total / g.N, st);
    } else if (train) {
      g.out = p.delta[p.L];
      rc = launch_gemm<EPI_PREDICT_TRAIN>(p, g, 1, st);
    } else {
      rc = launch_gemm<EPI_PREDICT>(p, g, 1, st);
    }
    if (rc != NCF_OK) return rc;
    if (StepTimer::g_timer) StepTimer::g_timer->mark(k == 0 ? "fwd0" : k == 1 ? "fwd1" : "fwd2+");
  }
  return NCF_OK;
}

// The fused kernel needs the whole tile's operand chain in the 512 TMEM columns.  NCF_UMMA_FUSED=0 is a
// test hook that forces the per-layer GEMMs; it is read per call, so a test can switch it between calls.
bool tower_fused_ok(const TileParams& p) {
  const char* off = getenv("NCF_UMMA_FUSED");
  if (off != nullptr && off[0] == '0') return false;
  if (p.W[0] > 256 || p.W[p.L] < 32 || p.f > 64) return false;
  int cols = 0;
  for (int k = 1; k <= p.L; ++k) cols += 2 * p.W[k];
  return cols <= 512 && 2 * p.W[1] + p.W[0] <= 512;
}

template <bool TRAIN>
int launch_tower(const TileParams& p, int passes, cudaStream_t st) {
  TowerArgs g{};
  g.passes = passes;
  int col = 0;
  for (int k = 1; k <= p.L; ++k) {
    g.hcol[k] = col;
    col += p.W[k];
    g.lcol[k] = col;
    col += p.W[k];
  }
  g.ring_col = p.W[1];
  g.ring_stages = std::min(kRingMax, (512 - p.W[1]) / 64);
  for (int k = 0; k < p.L; ++k)
    g.gemm[g.ng++] = TowerGemm{0, k, p.W[k + 1], p.W[k], k == 0 ? -1 : g.hcol[k], k == 0 ? -1 : g.lcol[k],
                               g.hcol[k + 1], p.W[k + 1], 0, k > 0, p.wsplit_f[k]};
  if (TRAIN)
    for (int k = p.L - 1; k >= 0; --k) {
      const bool top = (k + 1 == p.L);
      const int a_hi = top ? g.hcol[p.L] : g.lcol[k + 1], a_lo = top ? g.lcol[p.L] : g.hcol[k + 1];
      // accumulators are at most 128 columns wide (weight panels of <= 32 KB): wider outputs in blocks
      for (int n0 = 0; n0 < p.W[k]; n0 += 128) {
        const int N = std::min(128, p.W[k] - n0);
        g.gemm[g.ng++] = TowerGemm{1, k, N, p.W[k + 1], a_hi, a_lo, (k >= 1 ? g.lcol[k] : 2 * p.W[1]) + n0,
                                   p.W[k], n0, n0 == 0, p.wsplit_b[k]};
      }
    }
  const size_t smem = (size_t)kBStages * 128 * 256 + (size_t)(p.W[0] / 32) * kTile * 128 + 1024;
  auto kern = umma_tower_kernel<TRAIN>;
  NCF_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
  const int64_t ntiles = (p.B + kTile - 1) / kTile;
  int64_t grid = ncf::num_sms();
  if (grid > ntiles) grid = ntiles;
  kern<<<(unsigned)grid, kTowerThreads, smem, st>>>(p, g);
  NCF_LAUNCH_CHECK("umma_tower_kernel");
  return NCF_OK;
}

}  // namespace

namespace ncf {

// Eligible: a tower whose widths are power-of-two multiples of 32 (panels of 32 fp32, accumulator
// chunks of 32 columns) and a batch large enough that ~10 launches beat one fused launch.
// Test hooks, read per call: NCF_UMMA_DISABLE=1 keeps the path off, NCF_UMMA_MIN_B lowers the batch
// threshold so that small test batches run it.
bool umma_eligible(const TileParams& p) {
  const char* off = getenv("NCF_UMMA_DISABLE");
  if (off != nullptr && off[0] == '1') return false;
  const char* mb = getenv("NCF_UMMA_MIN_B");
  const int64_t min_b = mb ? atoll(mb) : 8192;
  if (p.B < min_b) return false;
  if (p.type == NCF_GMF) return false;
  if (p.f < 32 || p.f > 128 || (p.f & (p.f - 1)) != 0) return false;
  // the weight-gradient kernel's job table holds 12 [128 x 256] blocks: towers with a wider input
  // layer (f = 64 with L = 4, f = 128 with L = 3, ...) stay on the mma.sync / generic kernels
  int blocks = 0;
  for (int k = 0; k < p.L; ++k) blocks += ((p.W[k + 1] + 127) / 128) * ((p.W[k] + 255) / 256);
  return blocks <= 12;
}

int64_t umma_image_floats(const TileParams& p) {
  int64_t n = 0;
  for (int k = 0; k < p.L; ++k) n += 2 * 2 * (int64_t)p.W[k] * p.W[k + 1];
  return n;
}

int64_t umma_scratch_floats(const TileParams& p, int64_t B, bool train) {
  int64_t n = 0;
  for (int k = 1; k < p.L; ++k) n += B * p.W[k];
  if (train)
    for (int k = 1; k <= p.L; ++k) n += B * p.W[k];
  return n;
}

constexpr int64_t kForwardSub = 262144;  // inference sub-batch: bounds the activation scratch

// rows of one inference sub-batch: a whole number of users when one user covers user_div rows
static int64_t forward_sub(const TileParams& p) {
  return p.user_div > 0 ? std::max<int64_t>(1, kForwardSub / p.user_div) * p.user_div : kForwardSub;
}

int64_t umma_forward_workspace_floats(const TileParams& p, int64_t B) {
  return umma_image_floats(p) + umma_scratch_floats(p, std::min<int64_t>(B, forward_sub(p)), false) + 64;
}
int64_t umma_train_workspace_floats(const TileParams& p, int64_t B) {
  return umma_image_floats(p) + umma_scratch_floats(p, B, true) + 64;
}

static float* carve(TileParams& p, float* ws, int64_t B, bool train, cudaStream_t st, int* rc) {
  for (int k = 0; k < p.L; ++k) {
    const int64_t n = 2 * (int64_t)p.W[k] * p.W[k + 1];
    p.wsplit_f[k] = ws;
    p.wsplit_b[k] = ws + n;
    ws += 2 * n;
  }
  ws = (float*)(((uintptr_t)ws + 255) & ~(uintptr_t)255);
  for (int k = 1; k < p.L; ++k) { p.act[k] = ws; ws += B * p.W[k]; }
  if (train)
    for (int k = 1; k <= p.L; ++k) { p.delta[k] = ws; ws += B * p.W[k]; }
  umma_weight_images_kernel<<<dim3(64, 2 * p.L), 256, 0, st>>>(p);
  *rc = check_cuda(cudaGetLastError(), "umma_weight_images_kernel");
  return ws;
}

int launch_umma_forward(TileParams& p, int passes, float* ws, cudaStream_t st) {
  int rc;
  const int64_t B = p.B;
  if (tower_fused_ok(p)) {
    carve(p, ws, 0, false, st, &rc);
    if (rc != NCF_OK) return rc;
    return launch_tower<false>(p, passes, st);
  }
  const int64_t sub = forward_sub(p);
  carve(p, ws, std::min(B, sub), false, st, &rc);
  if (rc != NCF_OK) return rc;
  const int64_t* user = p.user;
  const int64_t* item = p.item;
  float* logits = p.logits;
  for (int64_t off = 0; off < B; off += sub) {
    p.B = std::min(sub, B - off);
    p.user = (p.user_div > 0) ? user + off / p.user_div : user + off;
    p.item = item + off;
    p.logits = logits + off;
    rc = tower_forward(p, passes, false, st);
    if (rc != NCF_OK) return rc;
  }
  return NCF_OK;
}

int launch_umma_train(TileParams& p, int passes, float* ws, cudaStream_t st) {
  int rc;
  StepTimer timer(st);
  carve(p, ws, p.B, true, st, &rc);
  if (rc != NCF_OK) return rc;
  timer.mark("images");
  if (tower_fused_ok(p)) {
    rc = launch_tower<true>(p, passes, st);
    if (rc != NCF_OK) return rc;
    if ((rc = mark_embedding_grads_done(st)) != NCF_OK) return rc;
    timer.mark("tower");
    rc = launch_wgrad(p, passes, st);
    timer.mark("wgrad");
    return rc;
  }
  rc = tower_forward(p, passes, true, st);
  if (rc != NCF_OK) return rc;
  for (int k = p.L - 1; k >= 0; --k) {
    GemmArgs g{};
    g.K = p.W[k + 1];
    g.n_total = p.W[k];
    g.N = std::min(256, g.n_total);
    g.passes = passes;
    g.layer = k;
    g.a = p.delta[k + 1];
    g.b_img = p.wsplit_b[k];
    if (k > 0) {
      g.out = p.delta[k];
      g.mask_src = p.act[k];
      rc = launch_gemm<EPI_MASK_STORE>(p, g, g.n_total / g.N, st);
    } else {
      rc = launch_gemm<EPI_SCATTER>(p, g, g.n_total / g.N, st);
    }
    if (rc != NCF_OK) return rc;
    timer.mark(k == 2 ? "dgrad2" : k == 1 ? "dgrad1" : k == 0 ? "dgrad0" : "dgrad");
  }
  if ((rc = mark_embedding_grads_done(st)) != NCF_OK) return rc;
  rc = launch_wgrad(p, passes, st);
  timer.mark("wgrad");
  return rc;
}

}  // namespace ncf

extern "C" int ncf_profile_enable(int32_t on) {
  g_profile.enabled = on;
  g_profile.n = 0;
  return NCF_OK;
}

extern "C" int ncf_profile_read(float* ms, char* names, int32_t cap, int32_t name_len) {
  int n = g_profile.n < cap ? g_profile.n : cap;
  for (int i = 0; i < n; ++i) {
    ms[i] = g_profile.ms[i];
    if (names != nullptr && name_len > 0) snprintf(names + (size_t)i * name_len, name_len, "%s", g_profile.name[i]);
  }
  return n;
}
