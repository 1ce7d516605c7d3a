// Adam arithmetic of the optimiser kernels (optim.cu).  torch.optim.Adam single-tensor math (torch 2.11
// optim/adam.py), per step t = 1, 2, ...:
//   m <- m + (1-b1)(g - m);  v <- b2 v + (1-b2) g^2
//   p <- p - (lr / (1-b1^t)) * m / (sqrt(v)/sqrt(1-b2^t) + eps)
// A row whose gradient is zero at step s still moves: m <- b1 m, v <- b2 v, same p update.
#pragma once
#include <cuda_runtime.h>

// Zero-gradient steps replayed exactly per row.  The per-step term decays like
// (b1/sqrt(b2))^j ~ 0.9005^j times the change of the bias corrections, so what is dropped beyond 160 steps
// sums to < 1.4e-6 of the first term (worst for a row last stepped at step 12; DESIGN §3.2).
constexpr int kMaxReplay = 160;

struct AdamConst {
  float lr, b1, b2, eps, ln_b1, ln_b2, sqrt_b2;
};

__device__ __forceinline__ float bias_c1(const AdamConst& c, float s) {  // lr / (1 - b1^s)
  return c.lr / (-expm1f(s * c.ln_b1));
}
__device__ __forceinline__ float bias_c2(const AdamConst& c, float s) {  // 1 / sqrt(1 - b2^s)
  return 1.f / sqrtf(-expm1f(s * c.ln_b2));
}

// Brings N elements of one row from "state after step `last`" to "state after step last+gap" under zero
// gradient.  c1s / c2s hold the bias terms of steps last+1 .. last+min(gap, kMaxReplay).  The N chains are
// independent and advance together, step by step: a row 160 steps behind is the critical path of a small-batch
// step, and eight elements replayed one after the other were eight times that path.  Per element the arithmetic
// is what it always was (an element with m = 0 subtracts exact zeros).
template <int N>
__device__ __forceinline__ void replay_zero_steps_n(float* p, float* m, float* v, int gap, const float* c1s,
                                                    const float* c2s, const AdamConst& c) {
  if (gap <= 0) return;
  const int n = min(gap, kMaxReplay);
  float mm[N], r[N];
#pragma unroll
  for (int i = 0; i < N; ++i) { mm[i] = m[i]; r[i] = sqrtf(v[i]); }
#pragma unroll 2
  for (int j = 0; j < n; ++j) {
    const float c1 = c1s[j], c2 = c2s[j];
#pragma unroll
    for (int i = 0; i < N; ++i) {
      mm[i] *= c.b1;
      r[i] *= c.sqrt_b2;
      p[i] -= c1 * __fdividef(mm[i], fmaf(r[i], c2, c.eps));
    }
  }
  const float dm = expf((float)gap * c.ln_b1), dv = expf((float)gap * c.ln_b2);
#pragma unroll
  for (int i = 0; i < N; ++i) { m[i] *= dm; v[i] *= dv; }
}

__device__ __forceinline__ void replay_zero_steps(float& p, float& m, float& v, int gap,
                                                  const float* c1s, const float* c2s,
                                                  const AdamConst& c) {
  replay_zero_steps_n<1>(&p, &m, &v, gap, c1s, c2s, c);
}

// The same replay with the bias terms evaluated on the fly (rows whose steps are not in a caller's table).
__device__ __forceinline__ void replay_inline(float& p, float& m, float& v, int last, int gap, const AdamConst& c) {
  const int n = min(gap, kMaxReplay);
  const float m0 = m, v0 = v;
  float mm = m0, r = sqrtf(v0);
  if (m0 != 0.f) {
    for (int j = 0; j < n; ++j) {
      const float s = (float)(last + 1 + j);
      mm *= c.b1;
      r *= c.sqrt_b2;
      p -= bias_c1(c, s) * __fdividef(mm, fmaf(r, bias_c2(c, s), c.eps));
    }
  }
  m = m0 * expf((float)gap * c.ln_b1);
  v = v0 * expf((float)gap * c.ln_b2);
}

__device__ __forceinline__ void adam_real_step(float& p, float& m, float& v, float g, float c1t,
                                               float c2t, const AdamConst& c) {
  m = fmaf(1.f - c.b1, g - m, m);
  v = fmaf(c.b2, v, (1.f - c.b2) * g * g);
  p -= c1t * (m / fmaf(sqrtf(v), c2t, c.eps));
}

inline AdamConst make_adam_const(float lr, float beta1, float beta2, float eps) {
  AdamConst c;
  c.lr = lr; c.b1 = beta1; c.b2 = beta2; c.eps = eps;
  c.ln_b1 = (float)log((double)beta1);
  c.ln_b2 = (float)log((double)beta2);
  c.sqrt_b2 = (float)sqrt((double)beta2);
  return c;
}
