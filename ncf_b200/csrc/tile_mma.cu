// Tensor-pipe version of the fused forward / forward+loss+backward tile kernel for towers whose
// widths are multiples of 8 (factor_num % 8 == 0).  Same data flow as tile_generic.cu — one CTA
// owns a tile of TM samples whose activations stay in shared memory for the whole
// forward+backward — but every contraction runs on warp-level mma.sync.m16n8k8 TF32 tiles:
//
//   PASSES == 3 ("fp32"): error-compensated 3xTF32.  Each fp32 operand x is split into
//       hi = tf32(x), lo = tf32(x - hi) and  x*w ~= lo*hi' + hi*lo' + hi*hi'  accumulated in fp32,
//       which keeps logits / gradients within the 1e-5 parity bar of the fp32 reference;
//   PASSES == 1 ("tf32"): plain TF32 (10-bit mantissa), 3x fewer MMAs, stated looser tolerance.
//
// Three GEMM flavours per layer k (tile = TM samples):
//   forward   H_{k+1}[m][n] = relu(sum_c H_k[m][c] W_k[n][c] + b_k[n])       A: smem act, B: W_k
//   backward  d_k[m][c]     = (sum_n d_{k+1}[m][n] W_k[n][c]) * [H_k > 0]     A: smem act, B: W_k^T
//   wgrad     dW_k[n][c]   += sum_m d_{k+1}[m][n] H_k[m][c]                   A, B: smem act
// Weights are pre-split (hi, lo) once per step by split_weights_kernel into the exact fragment
// order the B operand is consumed in, and streamed from L2 through a double-buffered cp.async
// stage; activations are split in registers when their fragments are loaded.  wgrad results and
// embedding-row gradients leave the CTA as vector REDs (dW_k is small and L2-resident).
//
// Replaces reference src/ncf/models.py:97-118 and scripts/train_neumf.py:112-114.
#include "common.cuh"
#include "tile_params.cuh"

namespace {

constexpr int kThreads = 512;          // 16 warps: 4 per scheduler to hide the split / LDS latencies
constexpr int kWarps = 16;
constexpr int kStageRow = 48;          // floats per staged weight row: 2 k-steps x 16 + 16 pad
constexpr int kStageRows = 128;        // output rows per staged block
constexpr int kStageFloats = kStageRows * kStageRow;
constexpr int kStages = 3;             // cp.async ring depth
// Activation row stride = width + 4 floats: stride % 32 == 4 makes the 8 rows of an ldmatrix
// phase hit 8 distinct 16-byte bank groups, and rows 2t apart (wgrad operand loads) 32 bytes apart.
constexpr int kActPad = 4;
static_assert(kThreads == 4 * kStageRows, "staging maps one thread to one 16-byte piece of a row");

__device__ __forceinline__ uint32_t f2tf32(float x) {
  uint32_t r;
  asm("cvt.rna.tf32.f32 %0, %1;" : "=r"(r) : "f"(x));
  return r;
}

// Activation split for 3xTF32.  The tensor core reads only the upper 19 bits of a tf32 operand
// register (sign, 8 exponent, 10 mantissa bits), i.e. it truncates.  So hi is x itself (consumed as
// trunc(x)), and lo = x - trunc(x) is exact in fp32 and in turn consumed truncated to 10 bits:
// x*w = trunc(x)*w + lo*w with a relative defect <= 2^-21 — two full-rate instructions per element.
struct Split {
  uint32_t hi, lo;
};
template <int PASSES>
__device__ __forceinline__ Split split_tf32(float x) {
  Split s;
  s.hi = __float_as_uint(x);
  s.lo = 0;
  if (PASSES == 3) s.lo = __float_as_uint(x - __uint_as_float(s.hi & 0xffffe000u));
  return s;
}

__device__ __forceinline__ void mma_tf32(float (&c)[4], const uint32_t (&a)[4], uint32_t b0,
                                         uint32_t b1) {
  asm volatile(
      "mma.sync.aligned.m16n8k8.row.col.f32.tf32.tf32.f32 {%0,%1,%2,%3}, {%4,%5,%6,%7}, {%8,%9}, "
      "{%0,%1,%2,%3};"
      : "+f"(c[0]), "+f"(c[1]), "+f"(c[2]), "+f"(c[3])
      : "r"(a[0]), "r"(a[1]), "r"(a[2]), "r"(a[3]), "r"(b0), "r"(b1));
}

__device__ __forceinline__ void cp_async16(void* smem, const void* gmem) {
  uint32_t s = (uint32_t)__cvta_generic_to_shared(smem);
  asm volatile("cp.async.cg.shared.global [%0], [%1], 16;" ::"r"(s), "l"(gmem));
}
__device__ __forceinline__ void cp_async_commit() { asm volatile("cp.async.commit_group;"); }
template <int N>
__device__ __forceinline__ void cp_async_wait() {
  asm volatile("cp.async.wait_group %0;" ::"n"(N));
}

__device__ __forceinline__ void ldmatrix_x4(uint32_t (&r)[4], uint32_t addr) {
  asm volatile("ldmatrix.sync.aligned.m8n8.x4.shared.b16 {%0,%1,%2,%3}, [%4];"
               : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3])
               : "r"(addr));
}
__device__ __forceinline__ float4 lds128(uint32_t addr) {
  float4 v;
  asm volatile("ld.shared.v4.f32 {%0,%1,%2,%3}, [%4];" : "=f"(v.x), "=f"(v.y), "=f"(v.z), "=f"(v.w) : "r"(addr));
  return v;
}

__device__ __forceinline__ void red_add2(float* p, float a, float b) {
  asm volatile("red.global.add.v2.f32 [%0], {%1, %2};" ::"l"(p), "f"(a), "f"(b) : "memory");
}

// ---- pre-split weights ---------------------------------------------------------------------------
// For a GEMM with `rows` output rows and contraction length `len` (multiple of 8), element
// (r, c) lands at  [c/8][r][ (c%4)*4 + (c%8)/4 ]  (hi)  and  +2 (lo): one 16-float record per
// (k-step, row); lane t reads its B fragment [hi(k=t), hi(k=t+4), lo(k=t), lo(k=t+4)] as one float4.
__global__ void split_weights_kernel(const TileParams p) {
  const int k = blockIdx.y;
  if (k >= p.L) return;
  const int K = p.W[k], N = p.W[k + 1];
  const float* W = p.w[k];
  float* wf = p.wsplit_f[k];
  float* wb = p.wsplit_b[k];
  for (int idx = blockIdx.x * blockDim.x + threadIdx.x; idx < N * K; idx += gridDim.x * blockDim.x) {
    const int n = idx / K, c = idx % K;
    const float x = W[idx];
    const float hi = __uint_as_float(f2tf32(x));
    const float lo = __uint_as_float(f2tf32(x - hi));
    {  // forward operand: rows = n, contraction = c
      float* d = wf + ((int64_t)(c >> 3) * N + n) * 16 + (c & 3) * 4 + ((c >> 2) & 1);
      d[0] = hi;
      d[2] = lo;
    }
    {  // backward operand: rows = c, contraction = n
      float* d = wb + ((int64_t)(n >> 3) * K + c) * 16 + (n & 3) * 4 + ((n >> 2) & 1);
      d[0] = hi;
      d[2] = lo;
    }
  }
}

// ---- flavour 1: A = activations in smem [TM][len] (stride lda), B = streamed pre-split weights -----
// Output block: TM x nb (nb <= 128, multiple of 8) starting at output row `row0` of the weight
// operand.  Warp (wm, wn) owns rows [wm*16*MT, +16*MT) x cols [wn*8*NT, +8*NT).
// epi(m, col, v0, v1) receives the pairs (col, col+1) of row m.
template <int PASSES, int MT, int NT, typename Epi>
__device__ __forceinline__ void gemm_act_weight(const float* __restrict__ A, int lda, int len,
                                                const float* __restrict__ wsplit, int rows_total,
                                                int row0, int nb, int WN, int tm_rows, float* stage,
                                                Epi epi) {
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const int g = lane >> 2, t = lane & 3;
  const int wm = warp / WN, wn = warp % WN;
  const bool active = wm * 16 * MT < tm_rows;  // surplus warps only help with staging and syncs
  const int nks = len >> 3;                 // k-steps
  const int nchunks = (nks + 1) >> 1;       // 2 k-steps per staged chunk
  float acc[MT][NT][4];
#pragma unroll
  for (int i = 0; i < MT; ++i)
#pragma unroll
    for (int j = 0; j < NT; ++j)
#pragma unroll
      for (int q = 0; q < 4; ++q) acc[i][j][q] = 0.f;

  // Staging: thread (r = tid/4, quad = tid%4) copies the 16-byte piece `quad` of row r of each
  // k-step of the chunk — 512 threads cover the 128 rows exactly, no index arithmetic in the loop.
  const int st_r = tid >> 2, st_q = tid & 3;
  const bool st_on = st_r < nb;
  const float* st_src = wsplit + ((int64_t)row0 + st_r) * 16 + st_q * 4;
  const int64_t st_ks_stride = (int64_t)rows_total * 16;
  const int st_dst = st_r * kStageRow + st_q * 4;
  auto load_chunk = [&](int c, float* buf) {
    if (st_on) {
      const float* src = st_src + (int64_t)(c * 2) * st_ks_stride;
      cp_async16(buf + st_dst, src);
      if (c * 2 + 1 < nks) cp_async16(buf + st_dst + 16, src + st_ks_stride);
    }
    cp_async_commit();
  };

  // Per-thread fragment addresses (32-bit shared-window addresses so that every access in the
  // loop is base register + immediate).  A fragments come from ldmatrix.x4 on the fp32 tile
  // viewed as 8x(16 byte) rows: lane l supplies row (l%8) + 8*((l/8)%2) at column 4*(l/16), and
  // receives a0..a3 = (g,t), (g+8,t), (g,t+4), (g+8,t+4) — exactly the m16n8k8 TF32 A layout.
  const uint32_t a_sh = (uint32_t)__cvta_generic_to_shared(A) +
                        4u * ((wm * 16 * MT + (lane & 7) + 8 * ((lane >> 3) & 1)) * lda + 4 * (lane >> 4));
  const uint32_t a_tile = 64u * lda;  // 16 rows, in bytes
  const uint32_t b_sh0 = (uint32_t)__cvta_generic_to_shared(stage) +
                         4u * ((wn * 8 * NT + g) * kStageRow + t * 4);

  auto k_step = [&](uint32_t a_addr, uint32_t b_addr) {
    uint32_t ahi[MT][4], alo[MT][4];
#pragma unroll
    for (int i = 0; i < MT; ++i) {
      ldmatrix_x4(ahi[i], a_addr + i * a_tile);
      if (PASSES == 3) {
#pragma unroll
        for (int q = 0; q < 4; ++q)
          alo[i][q] = __float_as_uint(__uint_as_float(ahi[i][q]) - __uint_as_float(ahi[i][q] & 0xffffe000u));
      }
    }
    uint32_t bh[NT][2], bl[NT][2];
#pragma unroll
    for (int j = 0; j < NT; ++j) {
      const float4 b = lds128(b_addr + j * (8 * kStageRow * 4));
      bh[j][0] = __float_as_uint(b.x); bh[j][1] = __float_as_uint(b.y);
      bl[j][0] = __float_as_uint(b.z); bl[j][1] = __float_as_uint(b.w);
    }
    // Issue order: MT*NT independent accumulators per pass, so consecutive MMAs never depend on
    // each other (the warp issues in order; a dependent chain would expose the MMA latency).
    if (PASSES == 3) {
#pragma unroll
      for (int j = 0; j < NT; ++j)
#pragma unroll
        for (int i = 0; i < MT; ++i) mma_tf32(acc[i][j], alo[i], bh[j][0], bh[j][1]);
#pragma unroll
      for (int j = 0; j < NT; ++j)
#pragma unroll
        for (int i = 0; i < MT; ++i) mma_tf32(acc[i][j], ahi[i], bl[j][0], bl[j][1]);
    }
#pragma unroll
    for (int j = 0; j < NT; ++j)
#pragma unroll
      for (int i = 0; i < MT; ++i) mma_tf32(acc[i][j], ahi[i], bh[j][0], bh[j][1]);
  };

  // 3-deep ring, one barrier per chunk: the barrier that publishes chunk c also certifies that
  // every warp is done with chunk c-1, whose buffer the load of chunk c+2 then overwrites.
  // (Rotating the chunk order per CTA to de-synchronise the L2 requests of the 148 CTAs was
  // measured and makes no difference — profiles/ablation_r01.md — so the walk is in order.)
  auto logical = [&](int c) { return c; };
  load_chunk(logical(0), stage);
  if (nchunks > 1) load_chunk(logical(1), stage + kStageFloats);
  int slot = 0;
  for (int c = 0; c < nchunks; ++c) {
    const uint32_t b_addr = b_sh0 + slot * (kStageFloats * 4);
    if (c + 1 < nchunks) cp_async_wait<1>(); else cp_async_wait<0>();
    __syncthreads();
    if (c + 2 < nchunks) {
      const int s2 = slot + 2 >= kStages ? slot + 2 - kStages : slot + 2;
      load_chunk(logical(c + 2), stage + s2 * kStageFloats);
    }
    slot = slot + 1 == kStages ? 0 : slot + 1;
    if (active) {
      const int cc = logical(c);
      const uint32_t a_addr = a_sh + cc * 64;  // 2 k-steps x 8 floats
      k_step(a_addr, b_addr);
      if (cc * 2 + 1 < nks) k_step(a_addr + 32, b_addr + 64);
    }
  }
  __syncthreads();  // stage buffers are free again; also orders the epilogue after all A reads
  if (!active) return;
#pragma unroll
  for (int i = 0; i < MT; ++i)
#pragma unroll
    for (int j = 0; j < NT; ++j) {
      const int m = wm * 16 * MT + i * 16 + g;
      const int col = row0 + wn * 8 * NT + j * 8 + 2 * t;
      epi(m, col, acc[i][j][0], acc[i][j][1]);
      epi(m + 8, col, acc[i][j][2], acc[i][j][3]);
    }
}

// Dispatch on the (MT, NT) tiling for a TM x nb output block.
template <int PASSES, int TM, typename Epi>
__device__ __forceinline__ void gemm_act_weight_block(const float* A, int lda, int len,
                                                      const float* wsplit, int rows_total, int row0,
                                                      int nb, float* stage, Epi epi) {
  // warps along n: up to 4 (8 when TM == 32 and nb allows); the rest along m
  constexpr int MTILES = TM / 16;
  // (MT, NT, warps along n): 16 warps = (TM / (16*MT)) x WN when the block is large enough
  if (TM == 64) {
    if (nb == 128) gemm_act_weight<PASSES, 2, 2>(A, lda, len, wsplit, rows_total, row0, nb, 8, TM, stage, epi);
    else if (nb == 64) gemm_act_weight<PASSES, 2, 1>(A, lda, len, wsplit, rows_total, row0, nb, 8, TM, stage, epi);
    else if (nb == 32) gemm_act_weight<PASSES, 1, 1>(A, lda, len, wsplit, rows_total, row0, nb, 4, TM, stage, epi);
    else if (nb == 16) gemm_act_weight<PASSES, 1, 1>(A, lda, len, wsplit, rows_total, row0, nb, 2, TM, stage, epi);
    else gemm_act_weight<PASSES, 1, 1>(A, lda, len, wsplit, rows_total, row0, nb, 1, TM, stage, epi);
  } else {
    static_assert(MTILES == 2 || MTILES == 4, "TM must be 32 or 64");
    if (nb == 128) gemm_act_weight<PASSES, 1, 2>(A, lda, len, wsplit, rows_total, row0, nb, 8, TM, stage, epi);
    else if (nb == 64) gemm_act_weight<PASSES, 1, 1>(A, lda, len, wsplit, rows_total, row0, nb, 8, TM, stage, epi);
    else if (nb == 32) gemm_act_weight<PASSES, 1, 1>(A, lda, len, wsplit, rows_total, row0, nb, 4, TM, stage, epi);
    else if (nb == 16) gemm_act_weight<PASSES, 1, 1>(A, lda, len, wsplit, rows_total, row0, nb, 2, TM, stage, epi);
    else gemm_act_weight<PASSES, 1, 1>(A, lda, len, wsplit, rows_total, row0, nb, 1, TM, stage, epi);
  }
}

// ---- flavour 2: dW[n][c] += sum_m D[m][n] * H[m][c], both operands are smem activations ---------------
// Output tiles of (16*MT) x (8*NT) are dealt round-robin to the warps; NT is even.  Results leave
// as 16-byte REDs: thanks to the column interleave a thread owns 4 consecutive c per (row, tile pair).
template <int PASSES, int TM, int MT, int NT>
__device__ __forceinline__ void gemm_wgrad(const float* __restrict__ D, int ldd, int N,
                                           const float* __restrict__ H, int ldh, int K,
                                           float* __restrict__ gw) {
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const int g = lane >> 2, t = lane & 3;
  const int tiles_n = (N + 16 * MT - 1) / (16 * MT), tiles_c = K / (8 * NT);
  for (int tile = warp; tile < tiles_n * tiles_c; tile += kWarps) {
    const int n0 = (tile / tiles_c) * 16 * MT, c0 = (tile % tiles_c) * 8 * NT;
    float acc[MT][NT][4];
#pragma unroll
    for (int i = 0; i < MT; ++i)
#pragma unroll
      for (int j = 0; j < NT; ++j)
#pragma unroll
        for (int q = 0; q < 4; ++q) acc[i][j][q] = 0.f;
    // k-slot t <-> sample row m0 + 2t, slot t+4 <-> m0 + 2t + 1 (any bijection works as long as A
    // and B agree; this one keeps the four rows of a half-warp 8 banks apart)
    const float* d_base = D + 2 * t * ldd + n0 + 2 * g;   // MMA rows g, g+8 <-> n, n+1
    const float* h_base = H + 2 * t * ldh + c0 + 2 * g;   // tile 2jj col g <-> c, tile 2jj+1 col g <-> c+1
    for (int m0 = 0; m0 < TM; m0 += 8) {
      uint32_t ahi[MT][4], alo[MT][4];
#pragma unroll
      for (int i = 0; i < MT; ++i) {
        float2 x0 = make_float2(0.f, 0.f), x1 = make_float2(0.f, 0.f);
        if (n0 + i * 16 + 2 * g < N) {
          x0 = *reinterpret_cast<const float2*>(d_base + m0 * ldd + i * 16);
          x1 = *reinterpret_cast<const float2*>(d_base + (m0 + 1) * ldd + i * 16);
        }
        const Split s0 = split_tf32<PASSES>(x0.x), s1 = split_tf32<PASSES>(x0.y);
        const Split s2 = split_tf32<PASSES>(x1.x), s3 = split_tf32<PASSES>(x1.y);
        ahi[i][0] = s0.hi; ahi[i][1] = s1.hi; ahi[i][2] = s2.hi; ahi[i][3] = s3.hi;
        alo[i][0] = s0.lo; alo[i][1] = s1.lo; alo[i][2] = s2.lo; alo[i][3] = s3.lo;
      }
      uint32_t bh[NT][2], bl[NT][2];
#pragma unroll
      for (int jj = 0; jj < NT / 2; ++jj) {
        const float2 y0 = *reinterpret_cast<const float2*>(h_base + m0 * ldh + jj * 16);
        const float2 y1 = *reinterpret_cast<const float2*>(h_base + (m0 + 1) * ldh + jj * 16);
        const Split e0 = split_tf32<PASSES>(y0.x), o0 = split_tf32<PASSES>(y0.y);
        const Split e1 = split_tf32<PASSES>(y1.x), o1 = split_tf32<PASSES>(y1.y);
        bh[2 * jj][0] = e0.hi; bh[2 * jj][1] = e1.hi; bl[2 * jj][0] = e0.lo; bl[2 * jj][1] = e1.lo;
        bh[2 * jj + 1][0] = o0.hi; bh[2 * jj + 1][1] = o1.hi; bl[2 * jj + 1][0] = o0.lo; bl[2 * jj + 1][1] = o1.lo;
      }
      if (PASSES == 3) {
#pragma unroll
        for (int j = 0; j < NT; ++j)
#pragma unroll
          for (int i = 0; i < MT; ++i) mma_tf32(acc[i][j], alo[i], bh[j][0], bh[j][1]);
#pragma unroll
        for (int j = 0; j < NT; ++j)
#pragma unroll
          for (int i = 0; i < MT; ++i) mma_tf32(acc[i][j], ahi[i], bl[j][0], bl[j][1]);
      }
#pragma unroll
      for (int j = 0; j < NT; ++j)
#pragma unroll
        for (int i = 0; i < MT; ++i) mma_tf32(acc[i][j], ahi[i], bh[j][0], bh[j][1]);
    }
#pragma unroll
    for (int i = 0; i < MT; ++i) {
      const int n = n0 + i * 16 + 2 * g;
#pragma unroll
      for (int jj = 0; jj < NT / 2; ++jj) {
        const int c = c0 + jj * 16 + 4 * t;
        const float* e = acc[i][2 * jj];
        const float* o = acc[i][2 * jj + 1];
        if (n < N) red_add4(gw + (int64_t)n * K + c, make_float4(e[0], o[0], e[1], o[1]));
        if (n + 1 < N) red_add4(gw + (int64_t)(n + 1) * K + c, make_float4(e[2], o[2], e[3], o[3]));
      }
    }
  }
}

template <int PASSES, int TM>
__device__ __forceinline__ void wgrad_dispatch(const float* D, int ldd, int N, const float* H, int ldh,
                                               int K, float* gw) {
  // 32x32 tiles when there are enough of them to occupy every warp, 16x16 tiles otherwise
  if ((N & 31) == 0 && (K & 31) == 0 && (N >> 5) * (K >> 5) >= kWarps)
    gemm_wgrad<PASSES, TM, 2, 4>(D, ldd, N, H, ldh, K, gw);
  else
    gemm_wgrad<PASSES, TM, 1, 2>(D, ldd, N, H, ldh, K, gw);
}

// ---- the tile kernel --------------------------------------------------------------------------------
template <int PASSES, int TM, bool TRAIN>
__global__ void __launch_bounds__(kThreads, 1) ncf_mma_tile_kernel(const TileParams p) {
  extern __shared__ __align__(16) float smem[];
  constexpr int MI = TM / kWarps;
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const bool has_gmf = p.type != NCF_MLP, has_mlp = p.type != NCF_GMF;
  const int f = p.f, d = p.d, L = p.L;

  float* gu_s = smem + p.gmf_off;
  float* gi_s = gu_s + TM * f;
  float* stage = smem + p.stage_off;
  float* dl_s = smem + p.misc_off;
  float* ls_s = dl_s + TM;
  int64_t* u_s = reinterpret_cast<int64_t*>(ls_s + TM);
  int64_t* i_s = u_s + TM;
  float* pg_s = reinterpret_cast<float*>(i_s + TM);  // [predict_size] predict-weight gradient of the tile
  auto act = [&](int k) { return smem + p.smem_off[k]; };
  auto lda = [&](int k) { return p.W[k] + kActPad; };

  const int64_t ntiles = (p.B + TM - 1) / TM;
  for (int64_t tile = blockIdx.x; tile < ntiles; tile += gridDim.x) {
    const int64_t base = tile * TM;
    __syncthreads();
    if (tid < TM) {
      const int64_t b = base + tid;
      int64_t u = -1, it = -1;
      if (b < p.B) {
        u = p.user[p.user_div > 0 ? b / p.user_div : b];
        it = p.item[b];
        if (u < 0 || u >= p.U || it < 0 || it >= p.I) { u = -2; it = -2; }
      }
      u_s[tid] = u;
      i_s[tid] = it;
    }
    __syncthreads();

    // ---- gather (one warp per sample row; 16-byte coalesced loads) -------------------------------
    // cp.async: every 16-byte piece of the warp's rows is in flight before anything is waited on
#pragma unroll
    for (int i = 0; i < MI; ++i) {
      const int m = warp + kWarps * i;
      const int64_t u = u_s[m], it = i_s[m];
      const bool ok = u >= 0;
      if (has_mlp) {
        float* x = act(0) + m * lda(0);
        const float* ru = p.eum + (ok ? u : 0) * d;
        const float* ri = p.eim + (ok ? it : 0) * d;
        for (int c = lane * 4; c < d; c += 128) {
          if (ok) {
            cp_async16(x + c, ru + c);
            cp_async16(x + d + c, ri + c);
          } else {
            *reinterpret_cast<float4*>(x + c) = make_float4(0, 0, 0, 0);
            *reinterpret_cast<float4*>(x + d + c) = make_float4(0, 0, 0, 0);
          }
        }
      }
      if (has_gmf) {
        const float* ru = p.eug + (ok ? u : 0) * f;
        const float* ri = p.eig + (ok ? it : 0) * f;
        for (int c = lane * 4; c < 2 * f; c += 128) {  // f % 8 == 0: 16-byte pieces never straddle
          float* dst = (c < f) ? gu_s + m * f + c : gi_s + m * f + (c - f);
          const float* src = (c < f) ? ru + c : ri + (c - f);
          if (ok) cp_async16(dst, src);
          else *reinterpret_cast<float4*>(dst) = make_float4(0, 0, 0, 0);
        }
      }
    }
    cp_async_commit();
    cp_async_wait<0>();
    __syncthreads();

    // ---- tower forward ------------------------------------------------------------------------------
    if (has_mlp) {
      for (int k = 0; k < L; ++k) {
        const int K = p.W[k], N = p.W[k + 1];
        float* out = act(k + 1);
        const int ldo = lda(k + 1);
        const float* bias = p.b[k];
        for (int n0 = 0; n0 < N; n0 += kStageRows) {
          const int nb = min(kStageRows, N - n0);
          gemm_act_weight_block<PASSES, TM>(act(k), lda(k), K, p.wsplit_f[k], N, n0, nb, stage,
                                            [&](int m, int col, float v0, float v1) {
                                              const float2 bb = __ldg(reinterpret_cast<const float2*>(bias + col));
                                              *reinterpret_cast<float2*>(out + m * ldo + col) =
                                                  make_float2(fmaxf(v0 + bb.x, 0.f), fmaxf(v1 + bb.y, 0.f));
                                            });
        }
      }
    }
    __syncthreads();

    // ---- predict layer: one warp per sample row computes the logit ------------------------------------------
    const float* hL = act(L);
    const int ldL = lda(L);
    const int fl = p.W[L];
    const int mlp_w_off = (p.type == NCF_NEUMF) ? f : 0;
#pragma unroll
    for (int i = 0; i < MI; ++i) {
      const int m = warp + kWarps * i;
      float s = 0.f;
      if (has_gmf)
        for (int c = lane; c < f; c += 32) s = fmaf(__ldg(&p.pw[c]), gu_s[m * f + c] * gi_s[m * f + c], s);
      if (has_mlp)
        for (int c = lane; c < fl; c += 32) s = fmaf(__ldg(&p.pw[mlp_w_off + c]), hL[m * ldL + c], s);
      s = warp_sum(s);
      if (lane == 0) ls_s[m] = s + __ldg(p.pb);
    }
    __syncthreads();
    // ---- loss and dloss/dlogit: one thread per sample row ---------------------------------------------------------
    if (tid < TM) {
      const int m = tid;
      const int64_t b = base + m;
      float x = ls_s[m];
      const bool ok = (b < p.B) && u_s[m] >= 0;
      if (b < p.B && u_s[m] == -2) x = __int_as_float(0x7fc00000);  // out-of-range index: NaN
      if (b < p.B && p.logits != nullptr) p.logits[b] = x;
      if (TRAIN) {
        float dl = 0.f, ls = 0.f;
        if (ok && p.dlogit_in != nullptr) {
          dl = p.dlogit_in[b];
        } else if (ok) {
          const bool kd = p.teacher != nullptr;
          const SampleLoss r = sample_loss(x, p.label[b], kd, kd ? p.teacher[b] : 0.f, p.alpha, p.invB);
          ls = r.loss;
          dl = r.dlogit;
        }
        dl_s[m] = dl;
        ls_s[m] = ls;
      }
    }
    if (!TRAIN) continue;
    for (int c = tid; c < p.predict_size; c += kThreads) pg_s[c] = 0.f;
    __syncthreads();

    // ---- loss, predict-layer gradients, GMF branch backward: one warp per sample row --------------------------------
    if (warp == 0) {
      float ls = 0.f, dsum = 0.f;
      for (int m = lane; m < TM; m += 32) { ls += ls_s[m]; dsum += dl_s[m]; }
      ls = warp_sum(ls);
      dsum = warp_sum(dsum);
      if (lane == 0) {
        if (p.loss_accum != nullptr) atomicAdd(p.loss_accum, (double)ls * (double)p.invB);
        atomicAdd(&p.gt[p.pb_off], dsum);
      }
    }
    {
      // lane c keeps the partial predict-weight gradient of columns c, c+32, ... over the warp's rows
      float pg[4] = {0.f, 0.f, 0.f, 0.f};
#pragma unroll
      for (int i = 0; i < MI; ++i) {
        const int m = warp + kWarps * i;
        const float dl = dl_s[m];
        const int64_t u = u_s[m], it = i_s[m];
        if (has_gmf) {
#pragma unroll
          for (int q = 0; q < 4; ++q) {
            const int c = lane + 32 * q;
            if (c < f) {
              const float gu = gu_s[m * f + c], gi = gi_s[m * f + c];
              pg[q] = fmaf(dl, gu * gi, pg[q]);
              if (u >= 0) {
                const float w = __ldg(&p.pw[c]) * dl;
                atomicAdd(&p.gug[u * f + c], w * gi);
                atomicAdd(&p.gig[it * f + c], w * gu);
              }
            }
          }
        }
      }
      if (has_gmf) {
#pragma unroll
        for (int q = 0; q < 4; ++q)
          if (lane + 32 * q < f) atomicAdd(&pg_s[lane + 32 * q], pg[q]);
      }
      if (has_mlp) {
        float pm[4] = {0.f, 0.f, 0.f, 0.f};
#pragma unroll
        for (int i = 0; i < MI; ++i) {
          const int m = warp + kWarps * i;
          const float dl = dl_s[m];
#pragma unroll
          for (int q = 0; q < 4; ++q)
            if (lane + 32 * q < fl) pm[q] = fmaf(dl, hL[m * ldL + lane + 32 * q], pm[q]);
        }
#pragma unroll
        for (int q = 0; q < 4; ++q)
          if (lane + 32 * q < fl) atomicAdd(&pg_s[mlp_w_off + lane + 32 * q], pm[q]);
      }
    }
    __syncthreads();
    for (int c = tid; c < p.predict_size; c += kThreads) atomicAdd(&p.gt[p.pw_off + c], pg_s[c]);

    // ---- tower backward ----------------------------------------------------------------------------------------
    if (has_mlp) {
      {  // delta_L = dl * predict_w_mlp * relu'(h_L), in place
        float* dL = act(L);
        for (int idx = tid; idx < TM * fl; idx += kThreads) {
          const int m = idx / fl, c = idx % fl;
          const float h = dL[m * ldL + c];
          dL[m * ldL + c] = (h > 0.f) ? dl_s[m] * __ldg(&p.pw[mlp_w_off + c]) : 0.f;
        }
      }
      __syncthreads();
      for (int k = L - 1; k >= 0; --k) {
        const int K = p.W[k], N = p.W[k + 1];
        const float* dn = act(k + 1);  // delta_{k+1} [TM][N]
        const int ldd = lda(k + 1);
        // bias gradient: column sums of delta_{k+1}
        {
          // thread (n, part) sums TM/parts rows of column n; parts = as many as the CTA can field
          int parts = kThreads / N;
          parts = parts > 16 ? 16 : (parts < 1 ? 1 : parts);
          const int rows = (TM + parts - 1) / parts;
          for (int idx = tid; idx < N * parts; idx += kThreads) {
            const int n = idx % N, m0 = (idx / N) * rows;
            float s = 0.f;
            for (int m = m0; m < min(TM, m0 + rows); ++m) s += dn[m * ldd + n];
            atomicAdd(&p.gt[p.b_off[k] + n], s);
          }
        }
        // weight gradient
        wgrad_dispatch<PASSES, TM>(dn, ldd, N, act(k), lda(k), K, p.gt + p.w_off[k]);
        __syncthreads();  // every read of H_k is done before it is overwritten by delta_k
        float* hk = act(k);
        const int ldh = lda(k);
        for (int c0 = 0; c0 < K; c0 += kStageRows) {
          const int nb = min(kStageRows, K - c0);
          if (k > 0) {
            gemm_act_weight_block<PASSES, TM>(dn, ldd, N, p.wsplit_b[k], K, c0, nb, stage,
                                              [&](int m, int col, float v0, float v1) {
                                                float2* q = reinterpret_cast<float2*>(hk + m * ldh + col);
                                                const float2 h = *q;
                                                *q = make_float2(h.x > 0.f ? v0 : 0.f, h.y > 0.f ? v1 : 0.f);
                                              });
          } else {
            gemm_act_weight_block<PASSES, TM>(dn, ldd, N, p.wsplit_b[k], K, c0, nb, stage,
                                              [&](int m, int col, float v0, float v1) {
                                                const int64_t u = u_s[m];
                                                if (u >= 0) {
                                                  if (col < d) red_add2(p.gum + u * d + col, v0, v1);
                                                  else red_add2(p.gim + i_s[m] * d + (col - d), v0, v1);
                                                }
                                              });
          }
        }
        __syncthreads();
      }
    }
  }
}

template <int TM>
size_t mma_smem_bytes(TileParams& p) {
  int off = 0;
  const bool has_mlp = p.type != NCF_GMF;
  for (int k = 0; k <= p.L; ++k) {
    p.smem_off[k] = off;
    if (has_mlp) off += TM * (p.W[k] + kActPad);
  }
  p.gmf_off = off;
  off += 2 * TM * p.f;
  off = (off + 3) & ~3;
  p.stage_off = off;
  off += kStages * kStageFloats;
  p.misc_off = off;
  off += 2 * TM + 4 * TM + ((p.predict_size + 3) & ~3);
  return (size_t)off * sizeof(float);
}

template <int PASSES, int TM, bool TRAIN>
int launch_mma(TileParams& p, cudaStream_t st) {
  const size_t smem = mma_smem_bytes<TM>(p);
  auto kern = ncf_mma_tile_kernel<PASSES, TM, TRAIN>;
  NCF_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
  const int64_t ntiles = (p.B + TM - 1) / TM;
  int per_sm = (int)(225 * 1024 / (smem + 1024));
  if (per_sm < 1) per_sm = 1;
  if (per_sm > 2) per_sm = 2;
  int64_t grid = (int64_t)ncf::num_sms() * per_sm;
  if (grid > ntiles) grid = ntiles;
  kern<<<(int)grid, kThreads, smem, st>>>(p);
  NCF_LAUNCH_CHECK("ncf_mma_tile_kernel");
  return NCF_OK;
}

constexpr size_t kSmemLimit = 227 * 1024;

}  // namespace

namespace ncf {

// 0 = not eligible, else the tile height (64 or 32).
int mma_tile_rows(const TileParams& p_in) {
  if (p_in.type == NCF_GMF) return 0;          // no tower: the generic kernel is already a pure gather
  if (p_in.f < 8 || (p_in.f & (p_in.f - 1)) != 0) return 0;  // block shapes assume power-of-two widths
  TileParams p = p_in;
  const bool fit64 = mma_smem_bytes<64>(p) <= kSmemLimit, fit32 = mma_smem_bytes<32>(p) <= kSmemLimit;
  // a batch that leaves most SMs idle with 64-row tiles (the reference's 256: 4 CTAs) runs on twice as many CTAs
  if (fit32 && p.B > 0 && (p.B + 63) / 64 * 2 <= ncf::num_sms()) return 32;
  if (fit64) return 64;
  if (fit32) return 32;
  return 0;
}

// ws: image_floats(p) floats.  Points p.wsplit_f / p.wsplit_b into it and launches the split.
int mma_prepare_weights(TileParams& p, float* ws, cudaStream_t st) {
  point_images(p, ws);
  split_weights_kernel<<<dim3(32, p.L), 256, 0, st>>>(p);
  NCF_LAUNCH_CHECK("split_weights_kernel");
  return NCF_OK;
}

int launch_mma_forward(TileParams& p, int tile_rows, int passes, cudaStream_t st) {
  if (tile_rows == 64) return passes == 3 ? launch_mma<3, 64, false>(p, st) : launch_mma<1, 64, false>(p, st);
  return passes == 3 ? launch_mma<3, 32, false>(p, st) : launch_mma<1, 32, false>(p, st);
}

int launch_mma_train(TileParams& p, int tile_rows, int passes, cudaStream_t st) {
  if (tile_rows == 64) return passes == 3 ? launch_mma<3, 64, true>(p, st) : launch_mma<1, 64, true>(p, st);
  return passes == 3 ? launch_mma<3, 32, true>(p, st) : launch_mma<1, 32, true>(p, st);
}

}  // namespace ncf
