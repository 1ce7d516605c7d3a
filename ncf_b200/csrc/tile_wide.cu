// Forward pass of a wide tower over a SMALL batch (the frozen teacher of a distillation step at the
// reference's batch of 256, model scoring of a few hundred pairs): one launch per layer, every launch spread
// over (batch / 32) x (outputs / 32) CTAs.
//
// The fused tile kernels keep a sample's whole tower inside one CTA, which is right when the batch fills the
// machine - at 256 samples it leaves a 512 -> 256 -> 128 -> 64 tower (172 k MACs per sample) on 4-8 CTAs that
// each stream every weight through shared memory: 55 us, plus 13 us to pre-split the weights for the tensor
// pipe.  Here layer k is the plain product H_{k+1} = relu(H_k W_k^T + b_k) on 32 x 32 output tiles (64 CTAs
// for the first layer of that tower), fp32 FMA - exact, no operand split - with the gather of the embedding
// rows folded into the first layer's operand loads; activations go through a [B, W_k] scratch that stays in L2.
//
// Replaces reference src/ncf/models.py:97-118 (forward) for these calls; same contract as the other forward
// kernels (TileParams; tile_params.cuh): out-of-range indices give NaN logits, user_div > 0 = one user per
// user_div candidates.
#include "common.cuh"
#include "tile_params.cuh"

namespace {

constexpr int kT = 32;          // output tile: 32 samples x 32 outputs, K walked in chunks of 32
constexpr int kWideThreads = 256;
constexpr int64_t kWideMaxB = 2048;

struct WideLayer {
  const float* in;       // [B, K] activations (layers > 0)
  const float* w;        // [N, K]
  const float* bias;     // [N]
  float* out;            // [B, N]
  int K, N;
};

// GATHER: the input row of sample b is [embed_user_MLP[user_b] ; embed_item_MLP[item_b]] (K = 2 d)
template <bool GATHER>
__global__ void __launch_bounds__(kWideThreads) wide_layer_kernel(const TileParams p, const WideLayer q) {
  __shared__ float a_sm[kT][kT + 1];
  __shared__ float w_sm[kT][kT + 1];
  __shared__ int64_t u_sm[kT], i_sm[kT];
  const int tid = threadIdx.x, tx = tid & 15, ty = tid >> 4;
  const int64_t b0 = (int64_t)blockIdx.y * kT;
  const int n0 = blockIdx.x * kT;
  if (GATHER && tid < kT) {
    const int64_t row = b0 + tid;
    int64_t u = -1, it = -1;
    if (row < p.B) {
      u = p.user[p.user_div > 0 ? row / p.user_div : row];
      it = p.item[row];
      if (u < 0 || u >= p.U || it < 0 || it >= p.I) u = -1;   // bad pair: zero row here, NaN logit in the predict kernel
    }
    u_sm[tid] = u;
    i_sm[tid] = it;
  }
  if (GATHER) __syncthreads();
  // loader role: thread -> (row r of the tile, 4 consecutive k)
  const int r = tid >> 3, c4 = (tid & 7) * 4;
  const int64_t arow = b0 + r;
  const int wn = n0 + r;
  auto load_a = [&](int k0) -> float4 {
    const int c = k0 + c4;
    if (GATHER) {
      const int64_t u = u_sm[r];
      if (u < 0) return make_float4(0.f, 0.f, 0.f, 0.f);
      return (c < p.d) ? ldg4(p.eum + u * p.d + c) : ldg4(p.eim + i_sm[r] * p.d + (c - p.d));
    }
    return (arow < p.B) ? ldg4(q.in + arow * q.K + c) : make_float4(0.f, 0.f, 0.f, 0.f);
  };
  auto load_w = [&](int k0) -> float4 {
    return (wn < q.N) ? ldg4(q.w + (int64_t)wn * q.K + k0 + c4) : make_float4(0.f, 0.f, 0.f, 0.f);
  };
  float acc[2][2] = {{0.f, 0.f}, {0.f, 0.f}};
  float4 an = load_a(0), wnx = load_w(0);
  for (int k0 = 0; k0 < q.K; k0 += kT) {
    __syncthreads();                       // the previous chunk has been consumed
    a_sm[r][c4] = an.x; a_sm[r][c4 + 1] = an.y; a_sm[r][c4 + 2] = an.z; a_sm[r][c4 + 3] = an.w;
    w_sm[r][c4] = wnx.x; w_sm[r][c4 + 1] = wnx.y; w_sm[r][c4 + 2] = wnx.z; w_sm[r][c4 + 3] = wnx.w;
    __syncthreads();
    if (k0 + kT < q.K) {                   // next chunk's loads fly while this one is multiplied
      an = load_a(k0 + kT);
      wnx = load_w(k0 + kT);
    }
#pragma unroll
    for (int k = 0; k < kT; ++k) {
      const float a0 = a_sm[2 * ty][k], a1 = a_sm[2 * ty + 1][k];
      const float w0 = w_sm[2 * tx][k], w1 = w_sm[2 * tx + 1][k];
      acc[0][0] = fmaf(a0, w0, acc[0][0]); acc[0][1] = fmaf(a0, w1, acc[0][1]);
      acc[1][0] = fmaf(a1, w0, acc[1][0]); acc[1][1] = fmaf(a1, w1, acc[1][1]);
    }
  }
#pragma unroll
  for (int i = 0; i < 2; ++i) {
    const int64_t row = b0 + 2 * ty + i;
    if (row >= p.B) continue;
#pragma unroll
    for (int j = 0; j < 2; ++j) {
      const int n = n0 + 2 * tx + j;
      if (n < q.N) q.out[row * q.N + n] = fmaxf(acc[i][j] + __ldg(q.bias + n), 0.f);
    }
  }
}

// logits[b] = predict_w . [gmf_u * gmf_i ; h_L] + predict_b, one warp per sample
__global__ void __launch_bounds__(256) wide_predict_kernel(const TileParams p, const float* __restrict__ hL) {
  const int lane = threadIdx.x & 31;
  const int64_t wid = (blockIdx.x * (int64_t)blockDim.x + threadIdx.x) >> 5, nw = ((int64_t)gridDim.x * blockDim.x) >> 5;
  const bool has_gmf = p.type != NCF_MLP;
  const int mlp_off = has_gmf ? p.f : 0;
  for (int64_t row = wid; row < p.B; row += nw) {
    const int64_t u = p.user[p.user_div > 0 ? row / p.user_div : row], it = p.item[row];
    const bool bad = u < 0 || u >= p.U || it < 0 || it >= p.I;
    float x = 0.f;
    if (!bad) {
      if (has_gmf)
        for (int c = lane; c < p.f; c += 32) x = fmaf(__ldg(p.pw + c), __ldg(p.eug + u * p.f + c) * __ldg(p.eig + it * p.f + c), x);
      for (int c = lane; c < p.f; c += 32) x = fmaf(__ldg(p.pw + mlp_off + c), hL[row * p.f + c], x);
    }
    x = warp_sum(x);
    if (lane == 0) p.logits[row] = bad ? __int_as_float(0x7fc00000) : x + __ldg(p.pb);
  }
}

}  // namespace

namespace ncf {

// forward only; MLP / NeuMF; every layer input a multiple of 32 wide (factor_num a multiple of 16); small batch
bool wide_eligible(const TileParams& p) {
  if (p.type == NCF_GMF || p.L < 1 || p.B < 1 || p.B > kWideMaxB) return false;
  if (p.f < 16 || (p.f & 15) != 0 || (p.d & 3) != 0) return false;
  for (int k = 0; k < p.L; ++k)
    if ((p.W[k] & 31) != 0 || (reinterpret_cast<uintptr_t>(p.w[k]) & 15) != 0) return false;
  return (reinterpret_cast<uintptr_t>(p.eum) & 15) == 0 && (reinterpret_cast<uintptr_t>(p.eim) & 15) == 0;
}

int64_t wide_workspace_floats(const TileParams& p, int64_t B) {
  int64_t n = 0;
  for (int k = 1; k <= p.L; ++k) n += B * p.W[k];
  return n;
}

int launch_wide_forward(TileParams& p, float* ws, cudaStream_t st) {
  const float* in = nullptr;
  for (int k = 0; k < p.L; ++k) {
    WideLayer q{in, p.w[k], p.b[k], ws, p.W[k], p.W[k + 1]};
    const dim3 grid((unsigned)((q.N + kT - 1) / kT), (unsigned)((p.B + kT - 1) / kT));
    if (k == 0) wide_layer_kernel<true><<<grid, kWideThreads, 0, st>>>(p, q);
    else wide_layer_kernel<false><<<grid, kWideThreads, 0, st>>>(p, q);
    NCF_LAUNCH_CHECK("wide_layer_kernel");
    in = ws;
    ws += p.B * q.N;
  }
  if (p.logits != nullptr) {
    int64_t blocks = (p.B + 7) / 8;
    if (blocks > 4 * num_sms()) blocks = 4 * num_sms();
    wide_predict_kernel<<<(int)blocks, 256, 0, st>>>(p, in);
    NCF_LAUNCH_CHECK("wide_predict_kernel");
  }
  return NCF_OK;
}

}  // namespace ncf
