// Generic (any factor_num / num_layers) fused forward and forward+loss+backward kernels on the
// fp32 FMA pipe.  One CTA owns a tile of TM samples: it gathers the embedding rows into shared
// memory, runs the tower layer by layer out of shared memory (weights staged chunk-wise from
// L2), evaluates the predict layer and the loss, and — when training — walks the tower backwards
// in place, scatter-adding the embedding-row gradients with vector REDs.  The tower weight
// gradients are a split-K GEMM over the batch (tower_wgrad_kernel) fed from an HBM scratch of the
// per-sample activations / deltas.
//
// Replaces reference src/ncf/models.py:97-118 (forward), scripts/train_neumf.py:112-114
// (criterion + backward) and src/distillation/base.py:40-50 + response.py:28-32 (KD loss).
#include "common.cuh"
#include "tile_params.cuh"

namespace {

constexpr int kThreads = 256;
constexpr int kWarps = kThreads / 32;
constexpr int KC = 32;        // contraction rows staged per chunk
constexpr int CB = 256;       // output columns per pass
constexpr int SP = CB + 1;    // padded stage stride (odd => transposing stores are conflict-free)

// out[m][cb..] = sum_c in[m][c] * Wstage[c][.] for the TM samples of the tile.
//   FWD : in = H_k  (width CL = in_w),  W[n][k] contracted over k, NO = out_w = N, + bias, relu
//   !FWD: in = d_{k+1} (width CL = N),  W[n][k] contracted over n, NO = K
template <int TM, bool FWD, typename Epilogue>
__device__ __forceinline__ void tile_gemm(const float* __restrict__ in_s, int CL, int NO,
                                          const float* __restrict__ Wg, float* __restrict__ stage,
                                          Epilogue epi) {
  constexpr int MI = TM / kWarps;
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  for (int cb = 0; cb < NO; cb += CB) {
    const int ncols = min(CB, NO - cb);
    const int nj = (ncols + 31) >> 5;
    float acc[MI][8];
#pragma unroll
    for (int i = 0; i < MI; ++i)
#pragma unroll
      for (int j = 0; j < 8; ++j) acc[i][j] = 0.f;
    for (int c0 = 0; c0 < CL; c0 += KC) {
      const int kc = min(KC, CL - c0);
      __syncthreads();
      if (FWD) {
        for (int idx = tid; idx < nj * 32 * KC; idx += kThreads) {
          const int oc = idx / KC, cc = idx % KC;
          float v = 0.f;
          if (oc < ncols && cc < kc) v = __ldg(&Wg[(int64_t)(cb + oc) * CL + c0 + cc]);
          stage[cc * SP + oc] = v;
        }
      } else {
        for (int idx = tid; idx < KC * nj * 32; idx += kThreads) {
          const int cc = idx / (nj * 32), oc = idx % (nj * 32);
          float v = 0.f;
          if (oc < ncols && cc < kc) v = __ldg(&Wg[(int64_t)(c0 + cc) * NO + cb + oc]);
          stage[cc * SP + oc] = v;
        }
      }
      __syncthreads();
      for (int cc = 0; cc < kc; ++cc) {
        float a[MI];
#pragma unroll
        for (int i = 0; i < MI; ++i) a[i] = in_s[(warp + kWarps * i) * CL + c0 + cc];
#pragma unroll
        for (int j = 0; j < 8; ++j) {
          if (j < nj) {
            const float wv = stage[cc * SP + lane + 32 * j];
#pragma unroll
            for (int i = 0; i < MI; ++i) acc[i][j] = fmaf(a[i], wv, acc[i][j]);
          }
        }
      }
    }
#pragma unroll
    for (int j = 0; j < 8; ++j) {
      const int c = cb + lane + 32 * j;
      if (j < nj && c < NO) {
#pragma unroll
        for (int i = 0; i < MI; ++i) epi(warp + kWarps * i, c, acc[i][j]);
      }
    }
  }
}

template <int TM, bool TRAIN>
__global__ void __launch_bounds__(kThreads) ncf_tile_kernel(const TileParams p) {
  extern __shared__ __align__(16) float smem[];
  constexpr int MI = TM / kWarps;
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const bool has_gmf = p.type != NCF_MLP, has_mlp = p.type != NCF_GMF;
  const int f = p.f, d = p.d, L = p.L;

  float* gu_s = smem + p.gmf_off;            // [TM][f]
  float* gi_s = gu_s + TM * f;               // [TM][f]
  float* stage = smem + p.stage_off;         // [KC][SP]
  float* dl_s = smem + p.misc_off;           // [TM] dloss/dlogit
  float* ls_s = dl_s + TM;                   // [TM] per-sample loss
  int64_t* u_s = reinterpret_cast<int64_t*>(ls_s + TM);  // [TM]
  int64_t* i_s = u_s + TM;                                // [TM]

  const int64_t ntiles = (p.B + TM - 1) / TM;
  for (int64_t tile = blockIdx.x; tile < ntiles; tile += gridDim.x) {
    const int64_t base = tile * TM;
    __syncthreads();  // previous tile fully consumed
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

    // ---- gather: one warp per sample row ------------------------------------------------
#pragma unroll
    for (int i = 0; i < MI; ++i) {
      const int m = warp + kWarps * i;
      const int64_t u = u_s[m], it = i_s[m];
      const bool ok = u >= 0;
      if (has_mlp) {
        float* x = smem + p.smem_off[0] + m * (2 * d);
        const float* ru = p.eum + (ok ? u : 0) * d;
        const float* ri = p.eim + (ok ? it : 0) * d;
        if ((d & 3) == 0) {
          for (int c = lane * 4; c < d; c += 128) {
            float4 a = ok ? ldg4(ru + c) : make_float4(0, 0, 0, 0);
            float4 b4 = ok ? ldg4(ri + c) : make_float4(0, 0, 0, 0);
            *reinterpret_cast<float4*>(x + c) = a;
            *reinterpret_cast<float4*>(x + d + c) = b4;
          }
        } else {
          for (int c = lane; c < d; c += 32) {
            x[c] = ok ? __ldg(ru + c) : 0.f;
            x[d + c] = ok ? __ldg(ri + c) : 0.f;
          }
        }
      }
      if (has_gmf) {
        const float* ru = p.eug + (ok ? u : 0) * f;
        const float* ri = p.eig + (ok ? it : 0) * f;
        for (int c = lane; c < f; c += 32) {
          gu_s[m * f + c] = ok ? __ldg(ru + c) : 0.f;
          gi_s[m * f + c] = ok ? __ldg(ri + c) : 0.f;
        }
      }
    }

    // ---- tower forward -------------------------------------------------------------------
    if (has_mlp) {
      for (int k = 0; k < L; ++k) {
        const float* in_s = smem + p.smem_off[k];
        float* out_s = smem + p.smem_off[k + 1];
        const int K = p.W[k], N = p.W[k + 1];
        const float* bias = p.b[k];
        float* act_g = (TRAIN && k + 1 < L) ? p.act[k + 1] : nullptr;
        tile_gemm<TM, true>(in_s, K, N, p.w[k], stage, [&](int m, int c, float acc) {
          const float h = fmaxf(acc + __ldg(&bias[c]), 0.f);
          out_s[m * N + c] = h;
          if (TRAIN && act_g != nullptr && base + m < p.B) act_g[(base + m) * N + c] = h;
        });
      }
    }
    __syncthreads();

    // ---- predict layer + loss: one warp per sample ----------------------------------------
    const float* hL = smem + p.smem_off[L];
    const int fl = p.W[L];  // == f
    const int mlp_w_off = (p.type == NCF_NEUMF) ? f : 0;
#pragma unroll
    for (int i = 0; i < MI; ++i) {
      const int m = warp + kWarps * i;
      const int64_t b = base + m;
      float s = 0.f;
      if (has_gmf)
        for (int c = lane; c < f; c += 32) s = fmaf(__ldg(&p.pw[c]), gu_s[m * f + c] * gi_s[m * f + c], s);
      if (has_mlp)
        for (int c = lane; c < fl; c += 32) s = fmaf(__ldg(&p.pw[mlp_w_off + c]), hL[m * fl + c], s);
      s = warp_sum(s);
      if (lane == 0) {
        float x = s + __ldg(p.pb);
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
    }
    if (!TRAIN) continue;
    __syncthreads();

    // ---- loss, predict-layer gradients, touched lists ----------------------------------------
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
    for (int c = tid; c < p.predict_size; c += kThreads) {
      float s = 0.f;
      if (has_gmf && c < f) {
        for (int m = 0; m < TM; ++m) s = fmaf(dl_s[m], gu_s[m * f + c] * gi_s[m * f + c], s);
      } else {
        const int j = c - mlp_w_off;
        for (int m = 0; m < TM; ++m) s = fmaf(dl_s[m], hL[m * fl + j], s);
      }
      atomicAdd(&p.gt[p.pw_off + c], s);
    }
    __syncthreads();  // hL reads above complete before delta_L overwrites it

    // ---- GMF branch backward: scatter row gradients --------------------------------------------
    if (has_gmf) {
#pragma unroll
      for (int i = 0; i < MI; ++i) {
        const int m = warp + kWarps * i;
        const int64_t u = u_s[m], it = i_s[m];
        if (u < 0) continue;
        const float dl = dl_s[m];
        for (int c = lane; c < f; c += 32) {
          const float w = __ldg(&p.pw[c]) * dl;
          atomicAdd(&p.gug[u * f + c], w * gi_s[m * f + c]);
          atomicAdd(&p.gig[it * f + c], w * gu_s[m * f + c]);
        }
      }
    }

    // ---- tower backward (in place over the activations) -------------------------------------------
    if (has_mlp) {
      {  // delta_L = dl * predict_w_mlp * relu'(h_L)
        float* dL = smem + p.smem_off[L];
        float* dg = p.delta[L];
        for (int idx = tid; idx < TM * fl; idx += kThreads) {
          const int m = idx / fl, c = idx % fl;
          const float h = dL[idx];
          const float v = (h > 0.f) ? dl_s[m] * __ldg(&p.pw[mlp_w_off + c]) : 0.f;
          dL[idx] = v;
          if (base + m < p.B) dg[(base + m) * fl + c] = v;
        }
      }
      for (int k = L - 1; k >= 0; --k) {
        const float* in_s = smem + p.smem_off[k + 1];  // delta_{k+1}  [TM][N]
        float* out_s = smem + p.smem_off[k];           // H_k -> delta_k [TM][K]
        const int K = p.W[k], N = p.W[k + 1];
        if (k > 0) {
          float* dg = p.delta[k];
          tile_gemm<TM, false>(in_s, N, K, p.w[k], stage, [&](int m, int c, float acc) {
            const float v = (out_s[m * K + c] > 0.f) ? acc : 0.f;
            out_s[m * K + c] = v;
            if (base + m < p.B) dg[(base + m) * K + c] = v;
          });
        } else {
          tile_gemm<TM, false>(in_s, N, K, p.w[k], stage, [&](int m, int c, float acc) {
            const int64_t u = u_s[m];
            if (u >= 0) {
              if (c < d) atomicAdd(&p.gum[u * d + c], acc);
              else atomicAdd(&p.gim[i_s[m] * d + (c - d)], acc);
            }
          });
        }
      }
    }
  }
}

// dW_k[n][c] += sum_b delta_{k+1}[b][n] * H_k[b][c];  db_k[n] += sum_b delta_{k+1}[b][n].
// grid.x = output tiles of all layers, grid.y = batch splits.  64x64 output tile per CTA.
constexpr int WT = 64, WMC = 32;

__global__ void __launch_bounds__(kThreads) tower_wgrad_kernel(const TileParams p, int nsplit) {
  __shared__ __align__(16) float ds[WMC][WT];
  __shared__ __align__(16) float hs[WMC][WT];
  // locate (layer, n-tile, c-tile)
  int t = blockIdx.x, k = 0, tn_cnt = 0, tc_cnt = 0;
  for (k = 0; k < p.L; ++k) {
    tn_cnt = (p.W[k + 1] + WT - 1) / WT;
    tc_cnt = (p.W[k] + WT - 1) / WT;
    if (t < tn_cnt * tc_cnt) break;
    t -= tn_cnt * tc_cnt;
  }
  if (k >= p.L) return;
  const int n0 = (t / tc_cnt) * WT, c0 = (t % tc_cnt) * WT;
  const int K = p.W[k], N = p.W[k + 1], d = p.d;
  const float* delta = p.delta[k + 1];
  const float* act = (k > 0) ? p.act[k] : nullptr;
  const int64_t per = (p.B + nsplit - 1) / nsplit;
  const int64_t b_lo = blockIdx.y * per, b_hi = min(p.B, b_lo + per);
  const int tid = threadIdx.x, tn = tid >> 4, tc = tid & 15;

  float acc[4][4];
  float bsum[4] = {0.f, 0.f, 0.f, 0.f};
#pragma unroll
  for (int i = 0; i < 4; ++i)
#pragma unroll
    for (int j = 0; j < 4; ++j) acc[i][j] = 0.f;

  for (int64_t b0 = b_lo; b0 < b_hi; b0 += WMC) {
    __syncthreads();
    for (int idx = tid; idx < WMC * WT; idx += kThreads) {
      const int mm = idx / WT, cc = idx % WT;
      const int64_t b = b0 + mm;
      float dv = 0.f, hv = 0.f;
      if (b < b_hi) {
        if (n0 + cc < N) dv = delta[b * N + n0 + cc];
        const int c = c0 + cc;
        if (c < K) {
          if (k > 0) {
            hv = act[b * K + c];
          } else {
            const int64_t u = p.user[b], it = p.item[b];
            if (u >= 0 && u < p.U && it >= 0 && it < p.I)
              hv = (c < d) ? __ldg(&p.eum[u * d + c]) : __ldg(&p.eim[it * d + (c - d)]);
          }
        }
      }
      ds[mm][cc] = dv;
      hs[mm][cc] = hv;
    }
    __syncthreads();
#pragma unroll 8
    for (int mm = 0; mm < WMC; ++mm) {
      const float4 dv = *reinterpret_cast<const float4*>(&ds[mm][tn * 4]);
      const float4 hv = *reinterpret_cast<const float4*>(&hs[mm][tc * 4]);
      const float dn[4] = {dv.x, dv.y, dv.z, dv.w};
      const float hc[4] = {hv.x, hv.y, hv.z, hv.w};
#pragma unroll
      for (int i = 0; i < 4; ++i) {
        bsum[i] += dn[i];
#pragma unroll
        for (int j = 0; j < 4; ++j) acc[i][j] = fmaf(dn[i], hc[j], acc[i][j]);
      }
    }
  }
  float* gw = p.gt + p.w_off[k];
#pragma unroll
  for (int i = 0; i < 4; ++i) {
    const int n = n0 + tn * 4 + i;
    if (n >= N) continue;
#pragma unroll
    for (int j = 0; j < 4; ++j) {
      const int c = c0 + tc * 4 + j;
      if (c < K) atomicAdd(&gw[(int64_t)n * K + c], acc[i][j]);
    }
    if (c0 == 0 && tc == 0) atomicAdd(&p.gt[p.b_off[k] + n], bsum[i]);
  }
}

template <int TM>
size_t tile_smem_bytes(TileParams& p) {
  int off = 0;
  const bool has_mlp = p.type != NCF_GMF;
  for (int k = 0; k <= p.L; ++k) {
    p.smem_off[k] = off;
    if (has_mlp) off += TM * p.W[k];
  }
  p.gmf_off = off;
  off += 2 * TM * p.f;
  off = (off + 3) & ~3;
  p.stage_off = off;
  off += KC * SP;
  off = (off + 3) & ~3;
  p.misc_off = off;
  off += 2 * TM;            // dl_s, ls_s
  off += 4 * TM;            // u_s, i_s (int64)
  return (size_t)off * sizeof(float);
}

template <int TM, bool TRAIN>
int launch_tile(TileParams& p, cudaStream_t st) {
  const size_t smem = tile_smem_bytes<TM>(p);
  auto kern = ncf_tile_kernel<TM, TRAIN>;
  NCF_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
  const int64_t ntiles = (p.B + TM - 1) / TM;
  int per_sm = (int)(220 * 1024 / (smem + 1024));
  if (per_sm < 1) per_sm = 1;
  if (per_sm > 4) per_sm = 4;
  int64_t grid = (int64_t)ncf::num_sms() * per_sm;
  if (grid > ntiles) grid = ntiles;
  kern<<<(int)grid, kThreads, smem, st>>>(p);
  NCF_LAUNCH_CHECK("ncf_tile_kernel");
  return NCF_OK;
}

}  // namespace

namespace ncf {

// Picks the largest sample tile whose shared-memory footprint fits one CTA.
int generic_tile_rows(const TileParams& p_in) {
  TileParams p = p_in;
  const size_t limit = 200 * 1024;
  if (tile_smem_bytes<32>(p) <= limit / 2) return 32;  // two CTAs per SM
  if (tile_smem_bytes<32>(p) <= limit) return 32;
  if (tile_smem_bytes<16>(p) <= limit) return 16;
  if (tile_smem_bytes<8>(p) <= limit) return 8;
  return 0;
}

int launch_generic_forward(TileParams& p, cudaStream_t st) {
  switch (generic_tile_rows(p)) {
    case 32: return launch_tile<32, false>(p, st);
    case 16: return launch_tile<16, false>(p, st);
    case 8: return launch_tile<8, false>(p, st);
  }
  set_error("model too wide for the generic tile kernel (f=%d, L=%d)", p.f, p.L);
  return NCF_ERR_ARG;
}

int launch_generic_train(TileParams& p, cudaStream_t st) {
  int rc;
  switch (generic_tile_rows(p)) {
    case 32: rc = launch_tile<32, true>(p, st); break;
    case 16: rc = launch_tile<16, true>(p, st); break;
    case 8: rc = launch_tile<8, true>(p, st); break;
    default:
      set_error("model too wide for the generic tile kernel (f=%d, L=%d)", p.f, p.L);
      return NCF_ERR_ARG;
  }
  if (rc != NCF_OK) return rc;
  if (p.type != NCF_GMF) {
    int tiles = 0;
    for (int k = 0; k < p.L; ++k)
      tiles += ((p.W[k + 1] + WT - 1) / WT) * ((p.W[k] + WT - 1) / WT);
    int nsplit = (4 * num_sms() + tiles - 1) / tiles;
    const int64_t max_split = (p.B + 4 * WMC - 1) / (4 * WMC);
    if (nsplit > max_split) nsplit = (int)max_split;
    if (nsplit < 1) nsplit = 1;
    tower_wgrad_kernel<<<dim3(tiles, nsplit), kThreads, 0, st>>>(p, nsplit);
    NCF_LAUNCH_CHECK("tower_wgrad_kernel");
  }
  return NCF_OK;
}

}  // namespace ncf
