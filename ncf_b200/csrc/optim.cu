// a10 optimisers.  Adam over the touched embedding rows only, numerically equivalent to the
// reference's DENSE optim.Adam (scripts/train_neumf.py:90,115) through lazy replay of the skipped
// zero-gradient steps; dense Adam over the (small) tower; plain SGD (train_neumf.py:88).
// HBM-bound: one warp per touched row streams g, p, m, v once (read) and p, m, v, g (write).
//
// torch.optim.Adam single-tensor math (torch 2.11 optim/adam.py), per step t = 1, 2, ...:
//   m <- m + (1-b1)(g - m);  v <- b2 v + (1-b2) g^2
//   p <- p - (lr / (1-b1^t)) * m / (sqrt(v)/sqrt(1-b2^t) + eps)
// A row whose gradient is zero at step s still moves: m <- b1 m, v <- b2 v, same p update.
#include <math.h>

#include "adam_math.cuh"
#include "common.cuh"

namespace {

constexpr int kThreads = 256;
constexpr int kWarps = kThreads / 32;
// One warp updates one table row of `dim` floats.  g == nullptr => replay only (flush).
template <int V>
__device__ __forceinline__ void adam_row(float* __restrict__ P, float* __restrict__ M,
                                         float* __restrict__ Vv, float* __restrict__ G, int dim,
                                         int gap, const float* c1s, const float* c2s, float c1t,
                                         float c2t, const AdamConst& c, int lane) {
  if (V == 4) {
    for (int e = lane * 4; e < dim; e += 128) {
      float4 p4 = *reinterpret_cast<float4*>(P + e);
      float4 m4 = *reinterpret_cast<float4*>(M + e);
      float4 v4 = *reinterpret_cast<float4*>(Vv + e);
      float4 g4 = make_float4(0, 0, 0, 0);
      if (G) g4 = *reinterpret_cast<float4*>(G + e);
      float pp[4] = {p4.x, p4.y, p4.z, p4.w}, mp[4] = {m4.x, m4.y, m4.z, m4.w}, vp[4] = {v4.x, v4.y, v4.z, v4.w};
      const float* gp = &g4.x;
      replay_zero_steps_n<4>(pp, mp, vp, gap, c1s, c2s, c);
      if (G) {
#pragma unroll
        for (int q = 0; q < 4; ++q) adam_real_step(pp[q], mp[q], vp[q], gp[q], c1t, c2t, c);
      }
      p4 = make_float4(pp[0], pp[1], pp[2], pp[3]);
      m4 = make_float4(mp[0], mp[1], mp[2], mp[3]);
      v4 = make_float4(vp[0], vp[1], vp[2], vp[3]);
      *reinterpret_cast<float4*>(P + e) = p4;
      *reinterpret_cast<float4*>(M + e) = m4;
      *reinterpret_cast<float4*>(Vv + e) = v4;
      if (G) *reinterpret_cast<float4*>(G + e) = make_float4(0, 0, 0, 0);
    }
  } else {
    for (int e = lane; e < dim; e += 32) {
      float p = P[e], m = M[e], v = Vv[e];
      replay_zero_steps(p, m, v, gap, c1s, c2s, c);
      if (G) {
        adam_real_step(p, m, v, G[e], c1t, c2t, c);
        G[e] = 0.f;
      }
      P[e] = p; M[e] = m; Vv[e] = v;
    }
  }
}

struct RowsParams {
  // side 0 = users, side 1 = items
  float *p_gmf[2], *m_gmf[2], *v_gmf[2], *g_gmf[2];
  float *p_mlp[2], *m_mlp[2], *v_mlp[2], *g_mlp[2];
  int32_t* last[2];
  int32_t* flag[2];
  const int64_t* list[2];
  const int32_t* tcount;
  int64_t rows[2];
  int64_t row0[2];  // first row of the all-rows modes (1, 3): rows [row0, row0 + rows) of each side
  const int64_t* step;
  int f, d, has_gmf, has_mlp;
  AdamConst c;
};

struct DenseSeg {
  float* p;
  int64_t off, n;
};
struct DenseParams {
  DenseSeg seg[2 * NCF_MAX_LAYERS + 2];
  int nseg;
  float *g, *m, *v;
  const int64_t* step;
  AdamConst c;
};

// ---- end of an optimiser step, folded into the last kernel that touches the tables -----------------------
// Every CTA updates its slice of the tower (dense Adam), then takes a ticket; the CTA that draws the last one
// knows every other CTA of the grid is done and closes the step: step counter + 1, touched lists emptied.
// (Two launches less per step: at the reference's batch of 256 they were 15 % of the step.)
// touched_count[2] is the ticket word; it is zero between kernels.
struct StepTail {
  DenseParams dq;     // dq.nseg == 0: the tower is not updated by this call
  int64_t* step;
  int32_t* tcount;
};

__device__ __forceinline__ void step_tail(const StepTail& t, int64_t step_now) {
  if (t.dq.nseg > 0) {
    const float tt = (float)(step_now + 1);
    const float c1t = bias_c1(t.dq.c, tt), c2t = bias_c2(t.dq.c, tt);
    const int64_t tid = blockIdx.x * (int64_t)blockDim.x + threadIdx.x, nt = (int64_t)gridDim.x * blockDim.x;
    for (int sg = 0; sg < t.dq.nseg; ++sg) {
      const DenseSeg& s = t.dq.seg[sg];
      for (int64_t i = tid; i < s.n; i += nt) {
        float p = s.p[i], m = t.dq.m[s.off + i], v = t.dq.v[s.off + i];
        adam_real_step(p, m, v, t.dq.g[s.off + i], c1t, c2t, t.dq.c);
        s.p[i] = p;
        t.dq.m[s.off + i] = m;
        t.dq.v[s.off + i] = v;
        t.dq.g[s.off + i] = 0.f;
      }
    }
  }
  __threadfence();
  __syncthreads();
  if (threadIdx.x == 0) {
    unsigned int* ticket = reinterpret_cast<unsigned int*>(t.tcount + 2);
    if (atomicAdd(ticket, 1u) == gridDim.x - 1) {
      *ticket = 0;
      *t.step = step_now + 1;
      t.tcount[0] = 0;
      t.tcount[1] = 0;
    }
  }
}

__global__ void step_tail_kernel(const StepTail tail) { step_tail(tail, *tail.step); }

// mode 0: Adam step on the touched rows; mode 1: flush (all rows, replay only);
// mode 2: catch-up (touched rows, replay only) — run BEFORE the forward of a step so that the rows
// the batch is about to read are at the dense-Adam state of the previous step;
// mode 3: Adam step on ALL rows (the reference's dense optimiser as it is): when a step touches a
// large share of the tables, streaming every row once is cheaper than list + catch-up + row gather.
template <int MODE>
__device__ __forceinline__ void adam_rows_body(const RowsParams& q, int64_t step_now);

// mode 0 ends the step (step_tail); the other modes ignore `tail`
template <int MODE>
__global__ void __launch_bounds__(kThreads) adam_rows_kernel(const RowsParams q, const StepTail tail) {
  const int64_t step_now = *q.step;
  adam_rows_body<MODE>(q, step_now);
  if (MODE == 0) step_tail(tail, step_now);
}

template <int MODE>
__device__ __forceinline__ void adam_rows_body(const RowsParams& q, const int64_t step_now) {
  __shared__ float c1_sm[kWarps][kMaxReplay];
  __shared__ float c2_sm[kWarps][kMaxReplay];
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  float* c1s = c1_sm[warp];
  float* c2s = c2_sm[warp];
  constexpr bool kStep = (MODE == 0 || MODE == 3);   // consumes gradients
  constexpr bool kList = (MODE == 0 || MODE == 2);   // iterates the touched lists
  const int64_t t = kStep ? step_now + 1 : step_now;  // state is brought to "after step t"
  const float c1t = bias_c1(q.c, (float)t), c2t = bias_c2(q.c, (float)t);
  const bool vec = ((q.f & 3) == 0) && ((q.d & 3) == 0);
  int64_t n0, n1;
  if (kList) { n0 = q.tcount[0]; n1 = q.tcount[1]; } else { n0 = q.rows[0]; n1 = q.rows[1]; }
  const int64_t total = n0 + n1;
  const int64_t wid = (int64_t)blockIdx.x * kWarps + warp, nw = (int64_t)gridDim.x * kWarps;
  // Fast path (NeuMF with rows of at most 128 floats, the bench shapes): a lane owns one float4 of the
  // GMF row and one of the MLP row; all eight loads of a row are issued before anything is used, and
  // the next row's list entry and last-step word are fetched while this row is in flight.
  if (vec && q.has_gmf && q.has_mlp && q.f <= 128 && q.d <= 128) {
    const bool lg = lane * 4 < q.f, lm = lane * 4 < q.d;
    auto fetch = [&](int64_t e, int& side, int64_t& r, int32_t& last) {
      side = e < n0 ? 0 : 1;
      r = 0;
      last = 0;
      if (e < total) {
        r = kList ? q.list[side][side ? e - n0 : e] : q.row0[side] + (side ? e - n0 : e);
        last = q.last[side][r];
      }
    };
    int side, nside;
    int64_t r, nr;
    int32_t last, nlast;
    fetch(wid, side, r, last);
    for (int64_t e = wid; e < total; e += nw, side = nside, r = nr, last = nlast) {
      fetch(e + nw, nside, nr, nlast);
      int gap;
      if (kStep) {
        gap = (last > 0) ? (int)(t - 1 - last) : 0;
      } else {
        if (last <= 0 || last >= t) continue;
        gap = (int)(t - last);
      }
      const int64_t og = r * q.f + lane * 4, om = r * q.d + lane * 4;
      float4 pg = make_float4(0, 0, 0, 0), mg = pg, vg = pg, gg = pg, pm = pg, mm = pg, vm = pg, gm = pg;
      if (lg) {
        pg = *reinterpret_cast<const float4*>(q.p_gmf[side] + og);
        mg = *reinterpret_cast<const float4*>(q.m_gmf[side] + og);
        vg = *reinterpret_cast<const float4*>(q.v_gmf[side] + og);
        if (kStep) gg = *reinterpret_cast<const float4*>(q.g_gmf[side] + og);
      }
      if (lm) {
        pm = *reinterpret_cast<const float4*>(q.p_mlp[side] + om);
        mm = *reinterpret_cast<const float4*>(q.m_mlp[side] + om);
        vm = *reinterpret_cast<const float4*>(q.v_mlp[side] + om);
        if (kStep) gm = *reinterpret_cast<const float4*>(q.g_mlp[side] + om);
      }
      __syncwarp();
      const int n = min(gap, kMaxReplay);
      for (int j = lane; j < n; j += 32) {
        const float s = (float)(last + 1 + j);
        c1s[j] = bias_c1(q.c, s);
        c2s[j] = bias_c2(q.c, s);
      }
      __syncwarp();
      // the lane's eight elements (4 of the GMF row, 4 of the MLP row) replay together
      float pe[8] = {pg.x, pg.y, pg.z, pg.w, pm.x, pm.y, pm.z, pm.w};
      float me[8] = {mg.x, mg.y, mg.z, mg.w, mm.x, mm.y, mm.z, mm.w};
      float ve[8] = {vg.x, vg.y, vg.z, vg.w, vm.x, vm.y, vm.z, vm.w};
      replay_zero_steps_n<8>(pe, me, ve, gap, c1s, c2s, q.c);
      if (kStep) {
        const float ge[8] = {gg.x, gg.y, gg.z, gg.w, gm.x, gm.y, gm.z, gm.w};
#pragma unroll
        for (int k = 0; k < 8; ++k) adam_real_step(pe[k], me[k], ve[k], ge[k], c1t, c2t, q.c);
      }
      pg = make_float4(pe[0], pe[1], pe[2], pe[3]); pm = make_float4(pe[4], pe[5], pe[6], pe[7]);
      mg = make_float4(me[0], me[1], me[2], me[3]); mm = make_float4(me[4], me[5], me[6], me[7]);
      vg = make_float4(ve[0], ve[1], ve[2], ve[3]); vm = make_float4(ve[4], ve[5], ve[6], ve[7]);
      if (lg) {
        *reinterpret_cast<float4*>(q.p_gmf[side] + og) = pg;
        *reinterpret_cast<float4*>(q.m_gmf[side] + og) = mg;
        *reinterpret_cast<float4*>(q.v_gmf[side] + og) = vg;
        if (kStep) *reinterpret_cast<float4*>(q.g_gmf[side] + og) = make_float4(0, 0, 0, 0);
      }
      if (lm) {
        *reinterpret_cast<float4*>(q.p_mlp[side] + om) = pm;
        *reinterpret_cast<float4*>(q.m_mlp[side] + om) = mm;
        *reinterpret_cast<float4*>(q.v_mlp[side] + om) = vm;
        if (kStep) *reinterpret_cast<float4*>(q.g_mlp[side] + om) = make_float4(0, 0, 0, 0);
      }
      if (lane == 0) {
        q.last[side][r] = (int32_t)t;
        if (kStep) q.flag[side][r] = 0;
      }
    }
    return;
  }
  for (int64_t e = wid; e < total; e += nw) {
    const int side = e < n0 ? 0 : 1;
    const int64_t r = kList ? q.list[side][side ? e - n0 : e] : q.row0[side] + (side ? e - n0 : e);
    const int32_t last = q.last[side][r];
    int gap;
    if (kStep) {
      gap = (last > 0) ? (int)(t - 1 - last) : 0;
    } else {
      if (last <= 0 || last >= t) continue;
      gap = (int)(t - last);
    }
    __syncwarp();
    const int n = min(gap, kMaxReplay);
    for (int j = lane; j < n; j += 32) {
      const float s = (float)(last + 1 + j);
      c1s[j] = bias_c1(q.c, s);
      c2s[j] = bias_c2(q.c, s);
    }
    __syncwarp();
    if (q.has_gmf) {
      const int64_t o = r * q.f;
      float* G = kStep ? q.g_gmf[side] + o : nullptr;
      if (vec) adam_row<4>(q.p_gmf[side] + o, q.m_gmf[side] + o, q.v_gmf[side] + o, G, q.f, gap, c1s, c2s, c1t, c2t, q.c, lane);
      else adam_row<1>(q.p_gmf[side] + o, q.m_gmf[side] + o, q.v_gmf[side] + o, G, q.f, gap, c1s, c2s, c1t, c2t, q.c, lane);
    }
    if (q.has_mlp) {
      const int64_t o = r * q.d;
      float* G = kStep ? q.g_mlp[side] + o : nullptr;
      if (vec) adam_row<4>(q.p_mlp[side] + o, q.m_mlp[side] + o, q.v_mlp[side] + o, G, q.d, gap, c1s, c2s, c1t, c2t, q.c, lane);
      else adam_row<1>(q.p_mlp[side] + o, q.m_mlp[side] + o, q.v_mlp[side] + o, G, q.d, gap, c1s, c2s, c1t, c2t, q.c, lane);
    }
    if (lane == 0) {
      q.last[side][r] = (int32_t)t;
      if (kStep) q.flag[side][r] = 0;
    }
  }
}

__global__ void sgd_dense_kernel(const DenseParams q, float lr) {
  const DenseSeg s = q.seg[blockIdx.y];
  for (int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; i < s.n;
       i += (int64_t)gridDim.x * blockDim.x) {
    s.p[i] -= lr * q.g[s.off + i];
    q.g[s.off + i] = 0.f;
  }
}

__global__ void __launch_bounds__(kThreads) sgd_rows_kernel(const RowsParams q, float lr) {
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const int64_t n0 = q.tcount[0], total = n0 + q.tcount[1];
  const int64_t wid = (int64_t)blockIdx.x * kWarps + warp, nw = (int64_t)gridDim.x * kWarps;
  for (int64_t e = wid; e < total; e += nw) {
    const int side = e < n0 ? 0 : 1;
    const int64_t r = q.list[side][side ? e - n0 : e];
    if (q.has_gmf) {
      float* P = q.p_gmf[side] + r * q.f;
      float* G = q.g_gmf[side] + r * q.f;
      for (int c = lane; c < q.f; c += 32) { P[c] -= lr * G[c]; G[c] = 0.f; }
    }
    if (q.has_mlp) {
      float* P = q.p_mlp[side] + r * q.d;
      float* G = q.g_mlp[side] + r * q.d;
      for (int c = lane; c < q.d; c += 32) { P[c] -= lr * G[c]; G[c] = 0.f; }
    }
    if (lane == 0) q.flag[side][r] = 0;
  }
}

// Registers the distinct rows of a batch in the touched lists (same protocol as the training
// kernel, which then finds the flags already set).
__global__ void mark_rows_kernel(const int64_t* __restrict__ user, const int64_t* __restrict__ item,
                                 int64_t B, int64_t U, int64_t I, int32_t* uflag, int32_t* iflag,
                                 int64_t* ulist, int64_t* ilist, int32_t* tcount) {
  for (int64_t b = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; b < B;
       b += (int64_t)gridDim.x * blockDim.x) {
    const int64_t u = user[b], it = item[b];
    if (u < 0 || u >= U || it < 0 || it >= I) continue;
    if (atomicExch(&uflag[u], 1) == 0) ulist[atomicAdd(&tcount[0], 1)] = u;
    if (atomicExch(&iflag[it], 1) == 0) ilist[atomicAdd(&tcount[1], 1)] = it;
  }
}

// ncf_adam_prepare as ONE launch: a warp takes one (sample, side) of the batch; lane 0 registers the row in the
// touched list, and the warp that won the registration replays the row's pending zero-gradient Adam steps right
// away (lanes across the row, as in adam_rows_kernel<2>) instead of leaving that to a second kernel that walks
// the list.  At the reference's batch of 256 the second launch was a quarter of the optimiser's time.
__global__ void __launch_bounds__(kThreads) mark_catchup_kernel(const RowsParams q, const int64_t* __restrict__ user,
                                                                const int64_t* __restrict__ item, int64_t B,
                                                                int64_t* ulist, int64_t* ilist, int32_t* tcount) {
  __shared__ float c1_sm[kWarps][kMaxReplay];
  __shared__ float c2_sm[kWarps][kMaxReplay];
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  float* c1s = c1_sm[warp];
  float* c2s = c2_sm[warp];
  const int64_t t = *q.step;   // rows are brought to "after step t"
  const bool vec = ((q.f & 3) == 0) && ((q.d & 3) == 0);
  const int64_t wid = (int64_t)blockIdx.x * kWarps + warp, nw = (int64_t)gridDim.x * kWarps;
  for (int64_t e = wid; e < 2 * B; e += nw) {
    const int64_t b = e >> 1;
    const int side = (int)(e & 1);
    const int64_t u = user[b], it = item[b];
    if (u < 0 || u >= q.rows[0] || it < 0 || it >= q.rows[1]) continue;   // same rule as mark_rows_kernel
    const int64_t r = side ? it : u;
    int32_t last = 0;
    if (lane == 0) {
      if (atomicExch(&q.flag[side][r], 1) == 0) {
        (side ? ilist : ulist)[atomicAdd(&tcount[side], 1)] = r;
        last = q.last[side][r];
        if (last >= t) last = 0;
      }
    }
    last = __shfl_sync(0xffffffffu, last, 0);
    if (last <= 0) continue;   // lost the registration, never stepped, or current already
    const int gap = (int)(t - last);
    __syncwarp();
    const int n = min(gap, kMaxReplay);
    for (int j = lane; j < n; j += 32) {
      const float sj = (float)(last + 1 + j);
      c1s[j] = bias_c1(q.c, sj);
      c2s[j] = bias_c2(q.c, sj);
    }
    __syncwarp();
    if (q.has_gmf) {
      const int64_t o = r * q.f;
      if (vec) adam_row<4>(q.p_gmf[side] + o, q.m_gmf[side] + o, q.v_gmf[side] + o, nullptr, q.f, gap, c1s, c2s, 0.f, 0.f, q.c, lane);
      else adam_row<1>(q.p_gmf[side] + o, q.m_gmf[side] + o, q.v_gmf[side] + o, nullptr, q.f, gap, c1s, c2s, 0.f, 0.f, q.c, lane);
    }
    if (q.has_mlp) {
      const int64_t o = r * q.d;
      if (vec) adam_row<4>(q.p_mlp[side] + o, q.m_mlp[side] + o, q.v_mlp[side] + o, nullptr, q.d, gap, c1s, c2s, 0.f, 0.f, q.c, lane);
      else adam_row<1>(q.p_mlp[side] + o, q.m_mlp[side] + o, q.v_mlp[side] + o, nullptr, q.d, gap, c1s, c2s, 0.f, 0.f, q.c, lane);
    }
    if (lane == 0) q.last[side][r] = (int32_t)t;
  }
}

// One side only (users or items): rows[] need not pair up with anything (row-sharded tables: a
// rank registers its own users and, separately, the item rows other ranks asked it for).
__global__ void mark_side_kernel(const int64_t* __restrict__ rows, int64_t n, int64_t limit,
                                 int32_t* flag, int64_t* list, int32_t* count) {
  for (int64_t b = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; b < n;
       b += (int64_t)gridDim.x * blockDim.x) {
    const int64_t r = rows[b];
    if (r < 0 || r >= limit) continue;
    if (atomicExch(&flag[r], 1) == 0) list[atomicAdd(count, 1)] = r;
  }
}

// ---- the all-rows step as a streaming kernel ------------------------------------------------------------
// A thread owns float4s of the four tables (user GMF, item GMF, user MLP, item MLP) taken as one flat index
// space, so the four streams p, m, v, g are read and written fully coalesced.  `last` is only
// read here (both tables of a row need the same gap); stamp_rows_kernel sets it afterwards.
struct FlatTable {
  float *p, *m, *v, *g;
  const int32_t* last;
  int64_t n4;   // float4s in the table
  int q4;       // float4s per row
};
struct FlatParams {
  FlatTable tab[4];
  const int64_t* step;
  AdamConst c;
};

__global__ void __launch_bounds__(256) adam_flat_kernel(const FlatParams q) {
  // One index space over the four tables, so that every CTA streams the same number of float4s whatever the
  // table sizes are (one grid row per table left the CTAs of the small tables idle for most of the kernel).
  const int64_t e1 = q.tab[0].n4, e2 = e1 + q.tab[1].n4, e3 = e2 + q.tab[2].n4, total = e3 + q.tab[3].n4;
  const int64_t t = *q.step + 1;
  const float c1t = bias_c1(q.c, (float)t), c2t = bias_c2(q.c, (float)t);
  for (int64_t j = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; j < total; j += (int64_t)gridDim.x * blockDim.x) {
    const int ti = j < e1 ? 0 : j < e2 ? 1 : j < e3 ? 2 : 3;
    const FlatTable& T = q.tab[ti];
    const int64_t i = j - (ti == 0 ? 0 : ti == 1 ? e1 : ti == 2 ? e2 : e3);
    float4* P = reinterpret_cast<float4*>(T.p);
    float4* M = reinterpret_cast<float4*>(T.m);
    float4* V = reinterpret_cast<float4*>(T.v);
    float4* G = reinterpret_cast<float4*>(T.g);
    float4 p4 = P[i], m4 = M[i], v4 = V[i];
    const float4 g4 = G[i];
    const int32_t last = __ldg(&T.last[i / T.q4]);
    const int gap = (last > 0) ? (int)(t - 1 - last) : 0;
    float* pp = &p4.x; float* mp = &m4.x; float* vp = &v4.x;
    const float* gp = &g4.x;
#pragma unroll
    for (int k = 0; k < 4; ++k) {
      if (gap > 0) replay_inline(pp[k], mp[k], vp[k], last, gap, q.c);
      adam_real_step(pp[k], mp[k], vp[k], gp[k], c1t, c2t, q.c);
    }
    P[i] = p4; M[i] = m4; V[i] = v4;
    // rows the step did not touch hold zeros already: do not write them again (half of the rows at the bench shape)
    if (g4.x != 0.f || g4.y != 0.f || g4.z != 0.f || g4.w != 0.f) G[i] = make_float4(0.f, 0.f, 0.f, 0.f);
  }
}

// (last_u / flag_u already point at the first user row of the range)
// ... and closes the step (tower update, counter, touched lists: step_tail)
__global__ void stamp_rows_kernel(int32_t* last_u, int32_t* flag_u, int64_t nu, int32_t* last_i, int32_t* flag_i,
                                  int64_t ni, const StepTail tail) {
  const int64_t step_now = *tail.step;
  const int32_t t = (int32_t)(step_now + 1);
  for (int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; i < nu + ni; i += (int64_t)gridDim.x * blockDim.x) {
    if (i < nu) { last_u[i] = t; flag_u[i] = 0; }
    else { last_i[i - nu] = t; flag_i[i - nu] = 0; }
  }
  step_tail(tail, step_now);
}

// Elementwise Adam step over a flat range (data-parallel optimiser sharding: every rank updates its
// own slice of the flat parameter buffer; requires every row to be current, i.e. all-rows mode).
__global__ void __launch_bounds__(256) adam_range_kernel(float4* __restrict__ P, float4* __restrict__ M,
                                                         float4* __restrict__ V, float4* __restrict__ G, int64_t n4,
                                                         const int64_t* __restrict__ step, AdamConst c) {
  const int64_t t = *step + 1;
  const float c1t = bias_c1(c, (float)t), c2t = bias_c2(c, (float)t);
  for (int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; i < n4; i += (int64_t)gridDim.x * blockDim.x) {
    float4 p4 = P[i], m4 = M[i], v4 = V[i];
    const float4 g4 = G[i];
    adam_real_step(p4.x, m4.x, v4.x, g4.x, c1t, c2t, c);
    adam_real_step(p4.y, m4.y, v4.y, g4.y, c1t, c2t, c);
    adam_real_step(p4.z, m4.z, v4.z, g4.z, c1t, c2t, c);
    adam_real_step(p4.w, m4.w, v4.w, g4.w, c1t, c2t, c);
    P[i] = p4; M[i] = m4; V[i] = v4;
    G[i] = make_float4(0.f, 0.f, 0.f, 0.f);
  }
}

// The same step with the gradient exchange inside the kernel (single node, peer memory over NVLink):
// the rank owns elements [lo4, lo4 + n4) of the flat layout, reads that slice of EVERY rank's gradient
// buffer (local + world-1 peer loads, all in flight together), averages in rank order, updates its
// moments and writes the new parameters into EVERY rank's parameter buffer (peer stores).  Replaces
// reduce-scatter -> adam_range_kernel -> all-gather; the caller brackets it with two rank barriers.
struct PeerBufs {
  const float4* g[8];
  float4* p[8];
};
__global__ void __launch_bounds__(256) adam_p2p_kernel(const __grid_constant__ PeerBufs b, const float4* own_p,
                                                       float4* __restrict__ M, float4* __restrict__ V,
                                                       int64_t lo4, int64_t n4, int world, float inv_world,
                                                       const int64_t* __restrict__ step, AdamConst c) {
  const int64_t t = *step + 1;
  const float c1t = bias_c1(c, (float)t), c2t = bias_c2(c, (float)t);
  for (int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; i < n4; i += (int64_t)gridDim.x * blockDim.x) {
    const int64_t e = lo4 + i;
    float4 gr[8];
#pragma unroll
    for (int r = 0; r < 8; ++r)
      gr[r] = (r < world) ? b.g[r][e] : make_float4(0.f, 0.f, 0.f, 0.f);
    float4 p4 = own_p[e], m4 = M[i], v4 = V[i];
    float4 g4 = gr[0];
#pragma unroll
    for (int r = 1; r < 8; ++r) { g4.x += gr[r].x; g4.y += gr[r].y; g4.z += gr[r].z; g4.w += gr[r].w; }
    g4.x *= inv_world; g4.y *= inv_world; g4.z *= inv_world; g4.w *= inv_world;
    adam_real_step(p4.x, m4.x, v4.x, g4.x, c1t, c2t, c);
    adam_real_step(p4.y, m4.y, v4.y, g4.y, c1t, c2t, c);
    adam_real_step(p4.z, m4.z, v4.z, g4.z, c1t, c2t, c);
    adam_real_step(p4.w, m4.w, v4.w, g4.w, c1t, c2t, c);
    M[i] = m4; V[i] = v4;
#pragma unroll
    for (int r = 0; r < 8; ++r)
      if (r < world) b.p[r][e] = p4;
  }
}

__global__ void finalize_step_kernel(int64_t* step, int32_t* tcount) {
  if (step) *step += 1;
  tcount[0] = 0;
  tcount[1] = 0;
}

// Upper bound on the rows registered since the last optimiser step (set by the mark / prepare entries, which
// know the batch size).  Only a launch-size hint: the row kernels walk the touched lists with grid-stride
// loops, so any grid is correct - but 1184 CTAs for the 512 rows of a batch of 256 cost 11 us of launch and
// drain where 64 CTAs cost 4.
thread_local int64_t g_rows_hint = 0;

int rows_grid(int64_t rows) {
  const int64_t cap = (int64_t)ncf::num_sms() * 8;
  if (rows <= 0) return (int)cap;
  int64_t blocks = (rows + kWarps - 1) / kWarps;   // one warp per row
  if (blocks > cap) blocks = cap;
  return (int)(blocks < 1 ? 1 : blocks);
}

AdamConst make_const(NcfAdamHyper h) { return make_adam_const(h.lr, h.beta1, h.beta2, h.eps); }

void fill_rows(RowsParams& q, const NcfModel* m, const NcfGrads* g, const NcfAdamState* s) {
  q.p_gmf[0] = m->embed_user_gmf; q.p_gmf[1] = m->embed_item_gmf;
  q.p_mlp[0] = m->embed_user_mlp; q.p_mlp[1] = m->embed_item_mlp;
  if (g) {
    q.g_gmf[0] = g->g_user_gmf; q.g_gmf[1] = g->g_item_gmf;
    q.g_mlp[0] = g->g_user_mlp; q.g_mlp[1] = g->g_item_mlp;
    q.flag[0] = g->user_flag; q.flag[1] = g->item_flag;
    q.list[0] = g->user_list; q.list[1] = g->item_list;
    q.tcount = g->touched_count;
  }
  if (s) {
    q.m_gmf[0] = s->m_user_gmf; q.m_gmf[1] = s->m_item_gmf;
    q.v_gmf[0] = s->v_user_gmf; q.v_gmf[1] = s->v_item_gmf;
    q.m_mlp[0] = s->m_user_mlp; q.m_mlp[1] = s->m_item_mlp;
    q.v_mlp[0] = s->v_user_mlp; q.v_mlp[1] = s->v_item_mlp;
    q.last[0] = s->user_last_step; q.last[1] = s->item_last_step;
    q.step = s->step;
  }
  q.rows[0] = m->user_num; q.rows[1] = m->item_num;
  q.f = m->factor_num; q.d = m->mlp_dim;
  q.has_gmf = m->model_type != NCF_MLP;
  q.has_mlp = m->model_type != NCF_GMF;
}

void fill_dense(DenseParams& q, const NcfModel* m) {
  ncf::TowerShape ts = ncf::make_tower_shape(m->model_type, m->factor_num, m->num_layers);
  int n = 0;
  if (m->model_type != NCF_GMF) {
    for (int k = 0; k < ts.L; ++k) {
      q.seg[n++] = {m->mlp_w[k], ts.w_off[k], (int64_t)ts.width[k] * ts.width[k + 1]};
      q.seg[n++] = {m->mlp_b[k], ts.b_off[k], (int64_t)ts.width[k + 1]};
    }
  }
  q.seg[n++] = {m->predict_w, ts.pw_off, (int64_t)ts.predict_size};
  q.seg[n++] = {m->predict_b, ts.pb_off, 1};
  q.nseg = n;
}

int check_state(const NcfModel* m, const NcfAdamState* s) {
  NCF_REQUIRE(s && s->step && s->user_last_step && s->item_last_step && s->m_tower && s->v_tower,
              "incomplete NcfAdamState");
  if (m->model_type != NCF_MLP)
    NCF_REQUIRE(s->m_user_gmf && s->v_user_gmf && s->m_item_gmf && s->v_item_gmf,
                "NcfAdamState: GMF moments are NULL");
  if (m->model_type != NCF_GMF)
    NCF_REQUIRE(s->m_user_mlp && s->v_user_mlp && s->m_item_mlp && s->v_item_mlp,
                "NcfAdamState: MLP moments are NULL");
  return NCF_OK;
}

int check_grads(const NcfModel* m, const NcfGrads* g) {
  NCF_REQUIRE(g && g->g_tower && g->user_flag && g->item_flag && g->user_list && g->item_list &&
                  g->touched_count,
              "incomplete NcfGrads");
  if (m->model_type != NCF_MLP) NCF_REQUIRE(g->g_user_gmf && g->g_item_gmf, "GMF grads are NULL");
  if (m->model_type != NCF_GMF) NCF_REQUIRE(g->g_user_mlp && g->g_item_mlp, "MLP grads are NULL");
  return NCF_OK;
}

}  // namespace

constexpr int kPartUsers = 1, kPartItems = 2, kPartTower = 4, kPartAll = 7;
static int adam_step_impl(const NcfModel* m, const NcfGrads* g, const NcfAdamState* s, NcfAdamHyper h,
                          void* stream, bool all_rows, int64_t user_lo, int64_t user_hi, int parts = kPartAll);

extern "C" int ncf_adam_step(const NcfModel* m, const NcfGrads* g, const NcfAdamState* s,
                             NcfAdamHyper h, void* stream) {
  return adam_step_impl(m, g, s, h, stream, false, 0, 0);
}

extern "C" int ncf_adam_step_dense(const NcfModel* m, const NcfGrads* g, const NcfAdamState* s,
                                   NcfAdamHyper h, void* stream) {
  return adam_step_impl(m, g, s, h, stream, true, 0, m ? m->user_num : 0);
}

extern "C" int ncf_adam_step_dense_range(const NcfModel* m, const NcfGrads* g, const NcfAdamState* s,
                                         NcfAdamHyper h, int64_t user_lo, int64_t user_hi, int32_t parts, void* stream) {
  NCF_REQUIRE(m && user_lo >= 0 && user_lo <= user_hi && user_hi <= m->user_num,
              "ncf_adam_step_dense_range: user range [%lld, %lld) outside the table", (long long)user_lo,
              (long long)user_hi);
  NCF_REQUIRE(parts >= 0 && parts <= kPartAll, "ncf_adam_step_dense_range: parts must be a mask of 1 | 2 | 4");
  return adam_step_impl(m, g, s, h, stream, true, user_lo, user_hi, parts);
}

static int adam_step_impl(const NcfModel* m, const NcfGrads* g, const NcfAdamState* s, NcfAdamHyper h,
                          void* stream, bool all_rows, int64_t user_lo, int64_t user_hi, int parts) {
  int rc = ncf::validate_model(m);
  if (rc != NCF_OK) return rc;
  if ((rc = check_grads(m, g)) != NCF_OK) return rc;
  if ((rc = check_state(m, s)) != NCF_OK) return rc;
  NCF_REQUIRE(h.beta1 > 0.f && h.beta1 < 1.f && h.beta2 > 0.f && h.beta2 < 1.f && h.eps > 0.f,
              "ncf_adam_step: bad hyper-parameters");
  cudaStream_t st = (cudaStream_t)stream;
  RowsParams q{};
  fill_rows(q, m, g, s);
  q.c = make_const(h);
  const bool vec = ((q.f & 3) == 0) && ((q.d & 3) == 0);
  if (all_rows) {  // users [user_lo, user_hi) (data-parallel ranks own a range of the user rows), every item
    q.row0[0] = user_lo;
    q.rows[0] = user_hi - user_lo;
  }
  StepTail tail{};
  if (parts & kPartTower) {
    fill_dense(tail.dq, m);
    tail.dq.g = g->g_tower; tail.dq.m = s->m_tower; tail.dq.v = s->v_tower; tail.dq.step = s->step; tail.dq.c = q.c;
  } else {
    tail.dq.nseg = 0;
  }
  tail.step = s->step;
  tail.tcount = g->touched_count;
  if (all_rows && vec) {
    FlatParams fp{};
    fp.step = q.step;
    fp.c = q.c;
    for (int side = 0; side < 2; ++side) {
      if (!(parts & (side ? kPartItems : kPartUsers))) continue;   // that side was updated elsewhere (peer-memory step)
      const int64_t r0 = q.row0[side];
      if (q.has_gmf)
        fp.tab[side] = FlatTable{q.p_gmf[side] + r0 * q.f, q.m_gmf[side] + r0 * q.f, q.v_gmf[side] + r0 * q.f,
                                 q.g_gmf[side] + r0 * q.f, q.last[side] + r0, q.rows[side] * q.f / 4, q.f / 4};
      if (q.has_mlp)
        fp.tab[2 + side] = FlatTable{q.p_mlp[side] + r0 * q.d, q.m_mlp[side] + r0 * q.d, q.v_mlp[side] + r0 * q.d,
                                     q.g_mlp[side] + r0 * q.d, q.last[side] + r0, q.rows[side] * q.d / 4, q.d / 4};
    }
    adam_flat_kernel<<<ncf::num_sms() * 16, 256, 0, st>>>(fp);
    NCF_LAUNCH_CHECK("adam_flat_kernel");
    stamp_rows_kernel<<<ncf::num_sms(), 256, 0, st>>>(q.last[0] + q.row0[0], q.flag[0] + q.row0[0], q.rows[0], q.last[1],
                                                     q.flag[1], q.rows[1], tail);
    NCF_LAUNCH_CHECK("stamp_rows_kernel");
  } else if (all_rows) {
    NCF_REQUIRE(parts == kPartAll, "ncf_adam_step_dense_range: partial steps need row widths that are multiples of 4");
    adam_rows_kernel<3><<<ncf::num_sms() * 8, kThreads, 0, st>>>(q, StepTail{});
    NCF_LAUNCH_CHECK("adam_rows_kernel");
    step_tail_kernel<<<32, 256, 0, st>>>(tail);
    NCF_LAUNCH_CHECK("step_tail_kernel");
  } else {
    adam_rows_kernel<0><<<rows_grid(g_rows_hint), kThreads, 0, st>>>(q, tail);
    NCF_LAUNCH_CHECK("adam_rows_kernel");
  }
  g_rows_hint = 0;
  return NCF_OK;
}

static int launch_mark(const NcfModel* m, const NcfGrads* g, const int64_t* user,
                       const int64_t* item, int64_t B, cudaStream_t st) {
  int64_t blocks = (B + 255) / 256;
  if (blocks > 4 * ncf::num_sms()) blocks = 4 * ncf::num_sms();
  mark_rows_kernel<<<(int)blocks, 256, 0, st>>>(user, item, B, m->user_num, m->item_num,
                                               g->user_flag, g->item_flag, g->user_list,
                                               g->item_list, g->touched_count);
  NCF_LAUNCH_CHECK("mark_rows_kernel");
  g_rows_hint += 2 * B;
  return NCF_OK;
}

extern "C" int ncf_mark_rows(const NcfModel* m, const NcfGrads* g, const int64_t* user,
                             const int64_t* item, int64_t B, void* stream) {
  int rc = ncf::validate_model(m);
  if (rc != NCF_OK) return rc;
  if ((rc = check_grads(m, g)) != NCF_OK) return rc;
  NCF_REQUIRE(B > 0 && user && item, "ncf_mark_rows: empty batch or null pointer");
  return launch_mark(m, g, user, item, B, (cudaStream_t)stream);
}

extern "C" int ncf_mark_rows_side(const NcfModel* m, const NcfGrads* g, const int64_t* rows, int64_t n,
                                  int32_t side, void* stream) {
  int rc = ncf::validate_model(m);
  if (rc != NCF_OK) return rc;
  if ((rc = check_grads(m, g)) != NCF_OK) return rc;
  NCF_REQUIRE(side == 0 || side == 1, "ncf_mark_rows_side: side must be 0 (users) or 1 (items)");
  NCF_REQUIRE(n >= 0, "ncf_mark_rows_side: negative n");
  if (n == 0) return NCF_OK;
  NCF_REQUIRE(rows != nullptr, "ncf_mark_rows_side: rows is NULL");
  int64_t blocks = (n + 255) / 256;
  if (blocks > 4 * ncf::num_sms()) blocks = 4 * ncf::num_sms();
  mark_side_kernel<<<(int)blocks, 256, 0, (cudaStream_t)stream>>>(
      rows, n, side ? m->item_num : m->user_num, side ? g->item_flag : g->user_flag,
      side ? g->item_list : g->user_list, g->touched_count + side);
  NCF_LAUNCH_CHECK("mark_side_kernel");
  g_rows_hint += n;
  return NCF_OK;
}

extern "C" int ncf_adam_catchup(const NcfModel* m, const NcfGrads* g, const NcfAdamState* s,
                                NcfAdamHyper h, void* stream) {
  int rc = ncf::validate_model(m);
  if (rc != NCF_OK) return rc;
  if ((rc = check_grads(m, g)) != NCF_OK) return rc;
  if ((rc = check_state(m, s)) != NCF_OK) return rc;
  RowsParams q{};
  fill_rows(q, m, g, s);
  q.c = make_const(h);
  adam_rows_kernel<2><<<rows_grid(g_rows_hint), kThreads, 0, (cudaStream_t)stream>>>(q, StepTail{});
  NCF_LAUNCH_CHECK("adam_rows_kernel<catchup>");
  return NCF_OK;
}

extern "C" int ncf_adam_prepare(const NcfModel* m, const NcfGrads* g, const NcfAdamState* s,
                                NcfAdamHyper h, const int64_t* user, const int64_t* item, int64_t B,
                                void* stream) {
  int rc = ncf::validate_model(m);
  if (rc != NCF_OK) return rc;
  if ((rc = check_grads(m, g)) != NCF_OK) return rc;
  if ((rc = check_state(m, s)) != NCF_OK) return rc;
  NCF_REQUIRE(B > 0 && user && item, "ncf_adam_prepare: empty batch or null pointer");
  cudaStream_t st = (cudaStream_t)stream;
  RowsParams q{};
  fill_rows(q, m, g, s);
  q.c = make_const(h);
  if (B > 4096) {
    // large batches: a thread per sample registers (one warp per sample-side would serialise 2B dependent
    // chains on a few thousand resident warps), then a warp per DISTINCT row replays
    if ((rc = launch_mark(m, g, user, item, B, st)) != NCF_OK) return rc;
    adam_rows_kernel<2><<<rows_grid(g_rows_hint), kThreads, 0, st>>>(q, StepTail{});
    NCF_LAUNCH_CHECK("adam_rows_kernel<catchup>");
    return NCF_OK;
  }
  mark_catchup_kernel<<<rows_grid(2 * B), kThreads, 0, st>>>(q, user, item, B, g->user_list, g->item_list,
                                                             g->touched_count);
  NCF_LAUNCH_CHECK("mark_catchup_kernel");
  g_rows_hint += 2 * B;
  return NCF_OK;
}

extern "C" int ncf_adam_flush(const NcfModel* m, const NcfAdamState* s, NcfAdamHyper h,
                              void* stream) {
  int rc = ncf::validate_model(m);
  if (rc != NCF_OK) return rc;
  if ((rc = check_state(m, s)) != NCF_OK) return rc;
  RowsParams q{};
  fill_rows(q, m, nullptr, s);
  q.c = make_const(h);
  adam_rows_kernel<1><<<ncf::num_sms() * 8, kThreads, 0, (cudaStream_t)stream>>>(q, StepTail{});
  NCF_LAUNCH_CHECK("adam_rows_kernel<flush>");
  return NCF_OK;
}

extern "C" int ncf_sgd_step(const NcfModel* m, const NcfGrads* g, float lr, void* stream) {
  int rc = ncf::validate_model(m);
  if (rc != NCF_OK) return rc;
  if ((rc = check_grads(m, g)) != NCF_OK) return rc;
  cudaStream_t st = (cudaStream_t)stream;
  RowsParams q{};
  fill_rows(q, m, g, nullptr);
  sgd_rows_kernel<<<rows_grid(g_rows_hint), kThreads, 0, st>>>(q, lr);
  g_rows_hint = 0;
  NCF_LAUNCH_CHECK("sgd_rows_kernel");
  DenseParams dq{};
  fill_dense(dq, m);
  dq.g = g->g_tower;
  sgd_dense_kernel<<<dim3(32, dq.nseg), 256, 0, st>>>(dq, lr);
  NCF_LAUNCH_CHECK("sgd_dense_kernel");
  finalize_step_kernel<<<1, 1, 0, st>>>(nullptr, g->touched_count);
  NCF_LAUNCH_CHECK("finalize_step_kernel");
  return NCF_OK;
}


extern "C" int ncf_adam_range(float* p, float* m, float* v, float* g, int64_t n, const int64_t* step,
                              NcfAdamHyper h, void* stream) {
  NCF_REQUIRE(p && m && v && g && step, "ncf_adam_range: null pointer");
  NCF_REQUIRE(n >= 0 && (n & 3) == 0, "ncf_adam_range: n must be a multiple of 4");
  NCF_REQUIRE((((uintptr_t)p | (uintptr_t)m | (uintptr_t)v | (uintptr_t)g) & 15) == 0,
              "ncf_adam_range: pointers must be 16-byte aligned");
  NCF_REQUIRE(h.beta1 > 0.f && h.beta1 < 1.f && h.beta2 > 0.f && h.beta2 < 1.f && h.eps > 0.f,
              "ncf_adam_range: bad hyper-parameters");
  if (n == 0) return NCF_OK;
  adam_range_kernel<<<ncf::num_sms() * 8, 256, 0, (cudaStream_t)stream>>>(
      reinterpret_cast<float4*>(p), reinterpret_cast<float4*>(m), reinterpret_cast<float4*>(v),
      reinterpret_cast<float4*>(g), n / 4, step, make_const(h));
  NCF_LAUNCH_CHECK("adam_range_kernel");
  return NCF_OK;
}

extern "C" int ncf_adam_p2p(const void* const* grad_bufs, void* const* param_bufs, float* m, float* v, int64_t lo,
                            int64_t n, int32_t world, int32_t rank, float grad_scale, const int64_t* step,
                            NcfAdamHyper h, void* stream) {
  NCF_REQUIRE(grad_bufs && param_bufs && m && v && step, "ncf_adam_p2p: null pointer");
  NCF_REQUIRE(world >= 1 && world <= 8 && rank >= 0 && rank < world, "ncf_adam_p2p: world must be 1..8 (one node)");
  NCF_REQUIRE(lo >= 0 && n >= 0 && (lo & 3) == 0 && (n & 3) == 0, "ncf_adam_p2p: lo and n must be multiples of 4");
  NCF_REQUIRE((((uintptr_t)m | (uintptr_t)v) & 15) == 0, "ncf_adam_p2p: pointers must be 16-byte aligned");
  NCF_REQUIRE(h.beta1 > 0.f && h.beta1 < 1.f && h.beta2 > 0.f && h.beta2 < 1.f && h.eps > 0.f,
              "ncf_adam_p2p: bad hyper-parameters");
  PeerBufs b{};
  for (int r = 0; r < world; ++r) {
    NCF_REQUIRE(grad_bufs[r] && param_bufs[r], "ncf_adam_p2p: null peer buffer");
    NCF_REQUIRE((((uintptr_t)grad_bufs[r] | (uintptr_t)param_bufs[r]) & 15) == 0,
                "ncf_adam_p2p: peer buffers must be 16-byte aligned");
    b.g[r] = reinterpret_cast<const float4*>(grad_bufs[r]);
    b.p[r] = reinterpret_cast<float4*>(param_bufs[r]);
  }
  if (n == 0) return NCF_OK;
  adam_p2p_kernel<<<ncf::num_sms() * 8, 256, 0, (cudaStream_t)stream>>>(
      b, b.p[rank], reinterpret_cast<float4*>(m), reinterpret_cast<float4*>(v), lo / 4, n / 4, world,
      grad_scale, step, make_const(h));
  NCF_LAUNCH_CHECK("adam_p2p_kernel");
  return NCF_OK;
}

extern "C" int ncf_adam_finish_dense(const NcfModel* m, const NcfGrads* g, const NcfAdamState* s, void* stream) {
  int rc = ncf::validate_model(m);
  if (rc != NCF_OK) return rc;
  if ((rc = check_grads(m, g)) != NCF_OK) return rc;
  if ((rc = check_state(m, s)) != NCF_OK) return rc;
  cudaStream_t st = (cudaStream_t)stream;
  StepTail tail{};
  tail.step = s->step;
  tail.tcount = g->touched_count;
  stamp_rows_kernel<<<ncf::num_sms(), 256, 0, st>>>(s->user_last_step, g->user_flag, m->user_num, s->item_last_step,
                                                   g->item_flag, m->item_num, tail);
  NCF_LAUNCH_CHECK("stamp_rows_kernel");
  return NCF_OK;
}
