// Narrow towers (factor_num = 8: widths 8*2^L -> ... -> 8, the reference's ML-100K / ML-1M configurations,
// BASELINE configs 1-3) on the fp32 FMA pipe, one THREAD per sample.
//
// north_star asks for tensor-core MMAs "only for tower layers wide enough to be a real dense contraction":
// a 64 -> 32 -> 16 -> 8 tower is 2.7 k MACs per sample - one warp of the mma.sync tile kernel spends more
// time staging fragments than multiplying (37 us for a batch of 256 on 4 CTAs).  Here a CTA of four warps owns
// a tile of 32 samples: lane = sample, warp = a quarter of every layer's outputs.  The sample's rows are
// gathered into its own shared-memory row, the tower runs forward and backward over those rows with the layer
// weights (and their transposes) resident in shared memory, and the CTA then forms the weight gradients of
// its 32 samples cooperatively (register tiles over the staged activations / deltas) before adding them to
// the global gradient buffer.  (One warp doing all four quarters measured 29 us for a batch of 256: a single
// dependent instruction stream per sample.)  Exact fp32: no operand split, no tolerance
// caveat.  Same contract as the other tile kernels (TileParams; tile_params.cuh).
//
// Replaces reference src/ncf/models.py:97-118 (forward), scripts/train_neumf.py:112-114 (criterion + backward)
// and src/distillation/base.py:40-50 + response.py:28-32 (KD loss) for these shapes.
#include "common.cuh"
#include "tile_params.cuh"

namespace {

constexpr int kF = 8;          // factor_num served here
constexpr int kPad = 4;        // row stride = width + 4 floats: 16-byte loads of 8 lanes hit 8 distinct bank groups

template <int L>
struct Shape {
  static constexpr int W0 = kF << L;
  __host__ __device__ static constexpr int W(int k) { return kF << (L - k); }
  // floats of shared memory
  static constexpr int weights() {   // W_k [n][c], W_k^T [c][n], b_k for every layer
    int n = 0;
    for (int k = 0; k < L; ++k) n += 2 * W(k) * W(k + 1) + W(k + 1);
    return n;
  }
  static constexpr int acts() {      // per-lane rows of h_0 .. h_L
    int n = 0;
    for (int k = 0; k <= L; ++k) n += 32 * (W(k) + kPad);
    return n;
  }
  static constexpr int delta() { return 32 * (W(1) + kPad); }   // widest delta row block
};

struct Ptrs {
  const float* w[NCF_MAX_LAYERS];    // shared-memory W_k  [W(k+1)][W(k)]
  const float* wt[NCF_MAX_LAYERS];   // shared-memory W_k^T [W(k)][W(k+1)]
  const float* b[NCF_MAX_LAYERS];
  float* h[NCF_MAX_LAYERS + 1];      // activations, row stride W(k) + kPad
};

constexpr int kWarps = 4;       // warps per tile of 32 samples: lane = sample, warp = a quarter of every layer's work
constexpr int kThreads = 32 * kWarps;

// out_row[n0 + j] = relu(bias + sum_c in_row[c] * Wt[c][n0 + j]), j < NW: the warp's NW = N / kWarps outputs
template <int C, int N, int NW>
__device__ __forceinline__ void fwd_part(const float* __restrict__ in_row, const float* __restrict__ wt,
                                         const float* __restrict__ bias, float* __restrict__ out_row, int n0) {
  float acc[NW];
#pragma unroll
  for (int j = 0; j < NW; ++j) acc[j] = bias[n0 + j];
#pragma unroll 2
  for (int c = 0; c < C; c += 4) {
    const float4 x = *reinterpret_cast<const float4*>(in_row + c);
    const float xs[4] = {x.x, x.y, x.z, x.w};
#pragma unroll
    for (int q = 0; q < 4; ++q) {
      const float* wr = wt + (c + q) * N + n0;
      if constexpr (NW % 4 == 0) {
#pragma unroll
        for (int j = 0; j < NW; j += 4) {
          const float4 w4 = *reinterpret_cast<const float4*>(wr + j);
          acc[j] = fmaf(xs[q], w4.x, acc[j]); acc[j + 1] = fmaf(xs[q], w4.y, acc[j + 1]);
          acc[j + 2] = fmaf(xs[q], w4.z, acc[j + 2]); acc[j + 3] = fmaf(xs[q], w4.w, acc[j + 3]);
        }
      } else {
        const float2 w2 = *reinterpret_cast<const float2*>(wr);
        acc[0] = fmaf(xs[q], w2.x, acc[0]); acc[1] = fmaf(xs[q], w2.y, acc[1]);
      }
    }
  }
#pragma unroll
  for (int j = 0; j < NW; ++j) out_row[n0 + j] = fmaxf(acc[j], 0.f);
}

// out_row[c0 + j] = (sum_n delta_row[n] * W[n][c0 + j]) [* (h_row[c0 + j] > 0) if MASK], j < CW = C / kWarps
template <int C, int N, int CW, bool MASK>
__device__ __forceinline__ void bwd_part(const float* __restrict__ delta_row, const float* __restrict__ w,
                                         const float* __restrict__ h_row, float* __restrict__ out_row, int c0) {
  float acc[CW];
#pragma unroll
  for (int j = 0; j < CW; ++j) acc[j] = 0.f;
#pragma unroll 2
  for (int n = 0; n < N; n += 4) {
    const float4 d4 = *reinterpret_cast<const float4*>(delta_row + n);
    const float ds[4] = {d4.x, d4.y, d4.z, d4.w};
#pragma unroll
    for (int q = 0; q < 4; ++q) {
      const float* wr = w + (n + q) * C + c0;
#pragma unroll
      for (int j = 0; j < CW; j += 4) {
        const float4 w4 = *reinterpret_cast<const float4*>(wr + j);
        acc[j] = fmaf(ds[q], w4.x, acc[j]); acc[j + 1] = fmaf(ds[q], w4.y, acc[j + 1]);
        acc[j + 2] = fmaf(ds[q], w4.z, acc[j + 2]); acc[j + 3] = fmaf(ds[q], w4.w, acc[j + 3]);
      }
    }
  }
#pragma unroll
  for (int j = 0; j < CW; ++j) out_row[c0 + j] = (!MASK || h_row[c0 + j] > 0.f) ? acc[j] : 0.f;
}

// dW[n][c] += sum_s delta[s][n] * h[s][c] over the tile's 32 samples for the warp's columns [cw0, cw0 + C / kWarps):
// lane owns an (N/8) x (C/16) register tile
template <int C, int N>
__device__ __forceinline__ void wgrad_part(const float* __restrict__ delta_s, const float* __restrict__ h_s,
                                           float* __restrict__ gw, int lane, int cw0) {
  constexpr int NB = N / 8, CB = C / (4 * kWarps);
  constexpr int SD = N + kPad, SH = C + kPad;
  const int n0 = (lane >> 2) * NB, c0 = cw0 + (lane & 3) * CB;
  float acc[NB][CB];
#pragma unroll
  for (int i = 0; i < NB; ++i)
#pragma unroll
    for (int j = 0; j < CB; ++j) acc[i][j] = 0.f;
#pragma unroll 4
  for (int s = 0; s < 32; ++s) {
    float dv[NB], hv[CB];
#pragma unroll
    for (int i = 0; i < NB; ++i) dv[i] = delta_s[s * SD + n0 + i];
#pragma unroll
    for (int j = 0; j < CB; ++j) hv[j] = h_s[s * SH + c0 + j];
#pragma unroll
    for (int i = 0; i < NB; ++i)
#pragma unroll
      for (int j = 0; j < CB; ++j) acc[i][j] = fmaf(dv[i], hv[j], acc[i][j]);
  }
#pragma unroll
  for (int i = 0; i < NB; ++i)
#pragma unroll
    for (int j = 0; j < CB; ++j) atomicAdd(gw + (n0 + i) * C + c0 + j, acc[i][j]);
}

template <int L, bool TRAIN>
__global__ void __launch_bounds__(kThreads) ncf_small_tile_kernel(const TileParams p) {
  using S = Shape<L>;
  extern __shared__ __align__(16) float smem_small[];
  float* w_sm = smem_small;
  float* h_sm = w_sm + S::weights();
  float* d_sm = h_sm + S::acts();          // TRAIN: two delta blocks, then dl[32]
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const bool has_gmf = p.type != NCF_MLP;
  const int mlp_off = has_gmf ? kF : 0;

  // ---- weights -> shared memory (row-major and transposed), once per CTA ---------------------------------
  Ptrs q;
  {
    float* wp = w_sm;
#pragma unroll
    for (int k = 0; k < L; ++k) {
      const int C = S::W(k), N = S::W(k + 1);
      float* w = wp; float* wt = wp + C * N; float* b = wp + 2 * C * N;
      // W_k: coalesced 16-byte loads straight into the row-major image; W_k^T: a second pass over the same
      // (now L1-resident) words with the OUTPUT index fastest, so that the shared-memory stores of a warp fall
      // into 32 different banks (one pass storing wt[c * N + n] for consecutive c put all 32 lanes on one bank)
      const float4* src4 = reinterpret_cast<const float4*>(p.w[k]);
      for (int i = tid; i < C * N / 4; i += kThreads) reinterpret_cast<float4*>(w)[i] = __ldg(src4 + i);
      for (int j = tid; j < C * N; j += kThreads) wt[j] = __ldg(p.w[k] + (j % N) * C + j / N);
      for (int i = tid; i < N; i += kThreads) b[i] = __ldg(p.b[k] + i);
      q.w[k] = w; q.wt[k] = wt; q.b[k] = b;
      wp += 2 * C * N + N;
    }
    float* hp = h_sm;
#pragma unroll
    for (int k = 0; k <= L; ++k) { q.h[k] = hp; hp += 32 * (S::W(k) + kPad); }
  }
  constexpr int d = S::W0 / 2;
  constexpr int Q0 = S::W0 / kWarps;        // columns of the gathered row per warp (a piece of one table's row)

  const int64_t ntiles = (p.B + 31) / 32;
  for (int64_t tile = blockIdx.x; tile < ntiles; tile += gridDim.x) {
    __syncthreads();   // weights staged (first pass) / the previous tile's rows are no longer read
    const int64_t row = tile * 32 + lane;
    const bool valid = row < p.B;
    int64_t u = -1, it = -1;
    bool bad = false;
    if (valid) {
      u = p.user[p.user_div > 0 ? row / p.user_div : row];
      it = p.item[row];
      if (u < 0 || u >= p.U || it < 0 || it >= p.I) { u = -1; bad = true; }
    }
    const bool ok = u >= 0;
    // ---- gather: the warp's piece of the lane's row ---------------------------------------------------------
    float* h0 = q.h[0] + lane * (S::W0 + kPad);
    {
      const int c0 = warp * Q0;                       // [0, d): user row, [d, 2d): item row
      const float* src = (c0 < d) ? p.eum + (ok ? u : 0) * d + c0 : p.eim + (ok ? it : 0) * d + (c0 - d);
#pragma unroll
      for (int c = 0; c < Q0; c += 4)
        *reinterpret_cast<float4*>(h0 + c0 + c) = ok ? ldg4(src + c) : make_float4(0, 0, 0, 0);
    }
    float gu[kF], gi[kF];
#pragma unroll
    for (int c = 0; c < kF; c += 4) {
      const float4 a = (ok && has_gmf) ? ldg4(p.eug + u * kF + c) : make_float4(0, 0, 0, 0);
      const float4 b4 = (ok && has_gmf) ? ldg4(p.eig + it * kF + c) : make_float4(0, 0, 0, 0);
      gu[c] = a.x; gu[c + 1] = a.y; gu[c + 2] = a.z; gu[c + 3] = a.w;
      gi[c] = b4.x; gi[c + 1] = b4.y; gi[c + 2] = b4.z; gi[c + 3] = b4.w;
    }
    __syncthreads();
    // ---- tower forward: every warp computes a quarter of each layer's outputs for its lane's sample ---------------
    fwd_part<S::W(0), S::W(1), S::W(1) / kWarps>(h0, q.wt[0], q.b[0], q.h[1] + lane * (S::W(1) + kPad), warp * (S::W(1) / kWarps));
    __syncthreads();
    if constexpr (L >= 2) {
      fwd_part<S::W(1), S::W(2), S::W(2) / kWarps>(q.h[1] + lane * (S::W(1) + kPad), q.wt[1], q.b[1],
                                                   q.h[2] + lane * (S::W(2) + kPad), warp * (S::W(2) / kWarps));
      __syncthreads();
    }
    if constexpr (L >= 3) {
      fwd_part<S::W(2), S::W(3), S::W(3) / kWarps>(q.h[2] + lane * (S::W(2) + kPad), q.wt[2], q.b[2],
                                                   q.h[3] + lane * (S::W(3) + kPad), warp * (S::W(3) / kWarps));
      __syncthreads();
    }
    const float* hL = q.h[L] + lane * (kF + kPad);
    // ---- predict layer (every warp computes it for its lane: 16 FMAs, no hand-off needed) -----------------------------
    float x = __ldg(p.pb);
    if (has_gmf) {
#pragma unroll
      for (int c = 0; c < kF; ++c) x = fmaf(__ldg(p.pw + c), gu[c] * gi[c], x);
    }
#pragma unroll
    for (int c = 0; c < kF; ++c) x = fmaf(__ldg(p.pw + mlp_off + c), hL[c], x);
    if (bad) x = __int_as_float(0x7fc00000);   // out-of-range index: NaN
    if (warp == 0 && valid && p.logits != nullptr) p.logits[row] = x;
    if (!TRAIN) continue;

    // ---- loss and dloss/dlogit -------------------------------------------------------------------------------------
    float dl = 0.f, ls = 0.f;
    if (ok && p.dlogit_in != nullptr) {
      dl = p.dlogit_in[row];
    } else if (ok) {
      const bool kd = p.teacher != nullptr;
      const SampleLoss r = sample_loss(x, p.label[row], kd, kd ? p.teacher[row] : 0.f, p.alpha, p.invB);
      ls = r.loss;
      dl = r.dlogit;
    }
    if (warp == 0) {
      const float ls_w = warp_sum(ls), dl_w = warp_sum(dl);
      if (lane == 0) {
        if (p.loss_accum != nullptr && p.dlogit_in == nullptr) atomicAdd(p.loss_accum, (double)ls_w * (double)p.invB);
        atomicAdd(p.gt + p.pb_off, dl_w);
      }
    }
    // predict-weight gradient: sum over the tile's samples of dl * feature (warp 1: GMF half, warp 2: tower half)
    if (warp == 1 && has_gmf) {
#pragma unroll
      for (int c = 0; c < kF; ++c) {
        const float s = warp_sum(dl * gu[c] * gi[c]);
        if (lane == 0) atomicAdd(p.gt + p.pw_off + c, s);
      }
    }
    if (warp == 2) {
#pragma unroll
      for (int c = 0; c < kF; ++c) {
        const float s = warp_sum(dl * hL[c]);
        if (lane == 0) atomicAdd(p.gt + p.pw_off + mlp_off + c, s);
      }
    }
    // GMF branch: embedding-row gradients (warp 3)
    if (warp == 3 && has_gmf && ok) {
#pragma unroll
      for (int c = 0; c < kF; c += 4) {
        const float4 w = ldg4(p.pw + c);
        red_add4(p.gug + u * kF + c, make_float4(dl * w.x * gi[c], dl * w.y * gi[c + 1], dl * w.z * gi[c + 2], dl * w.w * gi[c + 3]));
        red_add4(p.gig + it * kF + c, make_float4(dl * w.x * gu[c], dl * w.y * gu[c + 1], dl * w.z * gu[c + 2], dl * w.w * gu[c + 3]));
      }
    }
    // ---- tower backward: delta rows ping-pong between the two staging blocks -----------------------------------------
    float* dA = d_sm;
    float* dB = d_sm + S::delta();
    {
      float* dr = dA + lane * (kF + kPad);          // delta_L: the warp's two columns
#pragma unroll
      for (int c = warp * (kF / kWarps); c < (warp + 1) * (kF / kWarps); ++c)
        dr[c] = hL[c] > 0.f ? dl * __ldg(p.pw + mlp_off + c) : 0.f;
    }
    __syncthreads();
#define NCF_SMALL_BACK(K)                                                                                          \
    if constexpr (L > K) {                                                                                          \
      constexpr int k = L - 1 - K;                               /* layer index, from the top */                    \
      constexpr int C = S::W(k), N = S::W(k + 1);                                                                   \
      float* din = (K & 1) ? dB : dA;                                                                               \
      float* dout = (K & 1) ? dA : dB;                                                                              \
      wgrad_part<C, N>(din, q.h[k], p.gt + p.w_off[k], lane, warp * (C / kWarps));                                  \
      if (lane < N) {                                            /* bias gradient: column sums of delta, */        \
        float sum = 0.f;                                         /* eight samples per warp                */        \
        for (int s2 = warp * (32 / kWarps); s2 < (warp + 1) * (32 / kWarps); ++s2) sum += din[s2 * (N + kPad) + lane]; \
        atomicAdd(p.gt + p.b_off[k] + lane, sum);                                                                   \
      }                                                                                                             \
      __syncthreads();                                           /* every thread is done reading every row */     \
      if constexpr (k > 0) {                                                                                        \
        bwd_part<C, N, C / kWarps, true>(din + lane * (N + kPad), q.w[k], q.h[k] + lane * (C + kPad),               \
                                         dout + lane * (C + kPad), warp * (C / kWarps));                            \
      } else {                                                   /* dx_0 over the lane's input row */               \
        bwd_part<C, N, C / kWarps, false>(din + lane * (N + kPad), q.w[k], nullptr, h0, warp * (C / kWarps));       \
      }                                                                                                             \
      __syncthreads();                                                                                              \
    }
    NCF_SMALL_BACK(0)
    NCF_SMALL_BACK(1)
    NCF_SMALL_BACK(2)
#undef NCF_SMALL_BACK
    // ---- scatter dx_0 into the MLP embedding-gradient rows: the warp's piece of the lane's row ------------------------------
    if (ok) {
      const int c0 = warp * Q0;
      float* dst = (c0 < d) ? p.gum + u * d + c0 : p.gim + it * d + (c0 - d);
#pragma unroll
      for (int c = 0; c < Q0; c += 4) red_add4(dst + c, *reinterpret_cast<const float4*>(h0 + c0 + c));
    }
  }
}

template <int L, bool TRAIN>
int launch(const TileParams& p, cudaStream_t st) {
  const int64_t ntiles = (p.B + 31) / 32;
  int64_t grid = (int64_t)ncf::num_sms() * 8;
  if (grid > ntiles) grid = ntiles;
  using S = Shape<L>;
  const size_t smem = sizeof(float) * (S::weights() + S::acts() + (TRAIN ? 2 * S::delta() : 0));
  auto kern = ncf_small_tile_kernel<L, TRAIN>;
  if (smem > 48 * 1024) NCF_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
  kern<<<(int)grid, kThreads, smem, st>>>(p);
  NCF_LAUNCH_CHECK("ncf_small_tile_kernel");
  return NCF_OK;
}

}  // namespace

namespace ncf {

// factor_num 8, 1..3 tower layers, MLP / NeuMF (GMF has no tower: the generic kernel is a pure gather)
bool small_eligible(const TileParams& p) {
  if (p.f != kF || p.type == NCF_GMF || p.L < 1 || p.L > 3) return false;
  for (int k = 0; k < p.L; ++k)
    if (reinterpret_cast<uintptr_t>(p.w[k]) & 15) return false;   // weights are staged with 16-byte loads
  return true;
}

int launch_small_forward(TileParams& p, cudaStream_t st) {
  switch (p.L) {
    case 1: return launch<1, false>(p, st);
    case 2: return launch<2, false>(p, st);
    default: return launch<3, false>(p, st);
  }
}

int launch_small_train(TileParams& p, cudaStream_t st) {
  switch (p.L) {
    case 1: return launch<1, true>(p, st);
    case 2: return launch<2, true>(p, st);
    default: return launch<3, true>(p, st);
  }
}

}  // namespace ncf
