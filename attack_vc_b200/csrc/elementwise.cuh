// elementwise.cuh -- HBM-bound kernels of the perturbation loop: layout conversion, InstanceNorm +
// AdaIN + activation (+skip) forward/backward, MSE loss + gradient, the fused perturb/tanh/Adam
// update, the speaker-encoder dense tail and the AdaIN affine layers.  All fp32, float4 accesses,
// deterministic (fixed-order) reductions -- no float atomics anywhere.
#pragma once
#include "common.cuh"

namespace avc {

// ---------------------------------------------------------------------------------------------
// [B, C, T] strided (reference layout, attack.py:49-50)  <->  [B, T, ld] time-major
// ---------------------------------------------------------------------------------------------
__global__ void layout_in_kernel(const float* __restrict__ src, long long sb, long long sc, long long st,
                                 float* __restrict__ dst, long long d_bs, int d_rs, int B, int C, int T) {
  pdl_enter();
  long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  long long n = (long long)B * T * C;
  if (i >= n) return;
  int c = (int)(i % C);
  long long bt = i / C;
  int t = (int)(bt % T), b = (int)(bt / T);
  dst[(long long)b * d_bs + (long long)t * d_rs + c] = src[b * sb + c * sc + t * st];
}

__global__ void layout_out_kernel(const float* __restrict__ src, long long s_bs, int s_rs,
                                  float* __restrict__ dst, long long sb, long long sc, long long st,
                                  int B, int C, int T) {
  pdl_enter();
  long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  long long n = (long long)B * T * C;
  if (i >= n) return;
  int c = (int)(i % C);
  long long bt = i / C;
  int t = (int)(bt % T), b = (int)(bt / T);
  dst[b * sb + c * sc + t * st] = src[(long long)b * s_bs + (long long)t * s_rs + c];
}

// packed time-major [sum_b T_b, C] (utterance b's rows start at row offs[b])  <->  [B, T_max, ld] padded time-major:
// one CTA row per utterance (blockIdx.y), rows past T_b = offs[b+1] - offs[b] are neither read nor written
__global__ void layout_in_varlen_kernel(const float* __restrict__ src, const int* __restrict__ offs,
                                        float* __restrict__ dst, long long d_bs, int d_rs, int C) {
  pdl_enter();
  const int b = blockIdx.y;
  const long long r0 = offs[b], n = (long long)(offs[b + 1] - offs[b]) * C;
  for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (long long)gridDim.x * blockDim.x) {
    const int c = (int)(i % C), t = (int)(i / C);
    dst[(long long)b * d_bs + (long long)t * d_rs + c] = src[r0 * C + i];
  }
}

__global__ void layout_out_varlen_kernel(const float* __restrict__ src, long long s_bs, int s_rs, const int* __restrict__ offs,
                                         float* __restrict__ dst, int C) {
  pdl_enter();
  const int b = blockIdx.y;
  const long long r0 = offs[b], n = (long long)(offs[b + 1] - offs[b]) * C;
  for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (long long)gridDim.x * blockDim.x) {
    const int c = (int)(i % C), t = (int)(i / C);
    dst[r0 * C + i] = src[(long long)b * s_bs + (long long)t * s_rs + c];
  }
}

// ---------------------------------------------------------------------------------------------
// InstanceNorm1d(affine=False) + AdaIN + act (+ skip)            (models.py:66-79, 176, 396, 414-431)
//   out[b,t,c] = act( ((y - mu_bc) * rstd_bc) * std_bc + mean_bc ) + skip
// grid (C/32, B) -- strips of one utterance are neighbours in launch order, so a row's 512-byte line is fetched by
// co-resident CTAs; 256 threads = 8 float4 channel lanes (one full 128-byte line per row) x 32 time
// lanes.  The CTA's [T, 32] slice is staged in shared memory while the first pass sums it, so the
// centred second pass and the normalising third pass never go back to HBM: 8 B/element forward
// (+4 with a skip), 12 B/element backward, each tensor touched exactly once.  Statistics are
// two-pass (mean, then centred sum of squares; biased variance, eps 1e-5) and every reduction has
// a fixed order.  Slices longer than the staging capacity fall back to re-reading (L2).
// ---------------------------------------------------------------------------------------------
constexpr int kNormCh = 32;      // narrowest strip (channels)
constexpr int kNormSmemMax = 216 * 1024;

struct NormArgs {
  const float* y; int T; int C;        // [B,T,C] contiguous conv output (already pixel-shuffled)
  const float* cond; int cond_bs;      // [B, ...] row with mean at [0,C), std at [C,2C); nullptr: mean 0, std 1
  const float* stats_in;               // optional precomputed [B,C,2]
  float* stats_out;                    // optional [B,C,2] (mean, rstd)
  float* out;                          // [B,T,C]
  ResArgs res;
  float slope;
  int stage;                           // 1: the slice fits the dynamic shared memory of this launch
};

// sum over the 256 / CL time lanes for each of the CL float4 channel lanes; result broadcast to all threads
template <int CL>
__device__ __forceinline__ float4 block_reduce_t(float4 v, float4 (*red)[CL], int lane_c) {
#pragma unroll
  for (int o = CL; o <= 16; o <<= 1) {
    v.x += __shfl_xor_sync(0xffffffffu, v.x, o); v.y += __shfl_xor_sync(0xffffffffu, v.y, o);
    v.z += __shfl_xor_sync(0xffffffffu, v.z, o); v.w += __shfl_xor_sync(0xffffffffu, v.w, o);
  }
  const int warp = threadIdx.x >> 5;
  if ((threadIdx.x & 31) < CL) red[warp][lane_c] = v;
  __syncthreads();
  float4 r = red[0][lane_c];
#pragma unroll
  for (int w = 1; w < 8; ++w) r = f4add(r, red[w][lane_c]);
  __syncthreads();
  return r;
}

// CL = float4 channel lanes of a CTA (strip of 4*CL channels: 128 / 256 / 512 bytes of every row); the host takes the widest
// strip whose [T, 4*CL] slice still fits the staging memory with several CTAs per SM and that leaves >= 2 CTAs per SM
template <int CL>
__global__ void __launch_bounds__(256) norm_act_fwd_kernel(const NormArgs p) {
  extern __shared__ __align__(16) float4 ntile[];   // [T][CL] when p.stage
  __shared__ float4 red[8][CL];
  constexpr int kNormTL = 256 / CL;
  pdl_enter();
  const int lane_c = threadIdx.x % CL, lane_t = threadIdx.x / CL;
  const int b = blockIdx.y, c = blockIdx.x * (4 * CL) + lane_c * 4;
  const float* yb = p.y + (long long)b * p.T * p.C + c;
  const bool staged = p.stage && !p.stats_in;
  float4 mu, rstd;
  if (p.stats_in) {
    const float* s = p.stats_in + ((long long)b * p.C + c) * 2;
    float4 s0 = ld4(s), s1 = ld4(s + 4);
    mu = make_float4(s0.x, s0.z, s1.x, s1.z);
    rstd = make_float4(s0.y, s0.w, s1.y, s1.w);
  } else {
    float4 sum = f4zero();
    int t = lane_t;
    for (; t + 7 * kNormTL < p.T; t += 8 * kNormTL) {      // eight independent 16-byte loads in flight per thread
      float4 v[8];
#pragma unroll
      for (int j = 0; j < 8; ++j) v[j] = ld4(yb + (long long)(t + j * kNormTL) * p.C);
#pragma unroll
      for (int j = 0; j < 8; ++j) {
        if (staged) ntile[(t + j * kNormTL) * CL + lane_c] = v[j];
        sum = f4add(sum, v[j]);
      }
    }
    for (; t < p.T; t += kNormTL) {
      const float4 v = ld4(yb + (long long)t * p.C);
      if (staged) ntile[t * CL + lane_c] = v;
      sum = f4add(sum, v);
    }
    sum = block_reduce_t<CL>(sum, red, lane_c);
    const float invT = 1.f / (float)p.T;
    mu = f4scale(sum, invT);
    float4 sq = f4zero();
    for (int t = lane_t; t < p.T; t += kNormTL) {
      const float4 v = staged ? ntile[t * CL + lane_c] : ld4(yb + (long long)t * p.C);
      float dx = v.x - mu.x, dy = v.y - mu.y, dz = v.z - mu.z, dw = v.w - mu.w;
      sq.x = fmaf(dx, dx, sq.x); sq.y = fmaf(dy, dy, sq.y); sq.z = fmaf(dz, dz, sq.z); sq.w = fmaf(dw, dw, sq.w);
    }
    sq = block_reduce_t<CL>(sq, red, lane_c);
    rstd = make_float4(rsqrtf(sq.x * invT + 1e-5f), rsqrtf(sq.y * invT + 1e-5f),
                       rsqrtf(sq.z * invT + 1e-5f), rsqrtf(sq.w * invT + 1e-5f));
  }
  if (p.stats_out && lane_t == 0) {
    float* s = p.stats_out + ((long long)b * p.C + c) * 2;
    st4(s, make_float4(mu.x, rstd.x, mu.y, rstd.y));
    st4(s + 4, make_float4(mu.z, rstd.z, mu.w, rstd.w));
  }
  if (!p.out) return;
  float4 cm = f4zero(), cs = make_float4(1.f, 1.f, 1.f, 1.f);
  if (p.cond) {
    cm = ld4(p.cond + (long long)b * p.cond_bs + c);
    cs = ld4(p.cond + (long long)b * p.cond_bs + p.C + c);
  }
  float* ob = p.out + (long long)b * p.T * p.C + c;
#pragma unroll 4
  for (int t = lane_t; t < p.T; t += kNormTL) {
    const float4 v = staged ? ntile[t * CL + lane_c] : ld4(yb + (long long)t * p.C);
    float4 a;
    a.x = fmaf((v.x - mu.x) * rstd.x, cs.x, cm.x);
    a.y = fmaf((v.y - mu.y) * rstd.y, cs.y, cm.y);
    a.z = fmaf((v.z - mu.z) * rstd.z, cs.z, cm.z);
    a.w = fmaf((v.w - mu.w) * rstd.w, cs.w, cm.w);
    a = act4(a, p.slope);
    if (p.res.mode != RES_NONE) a = f4add(a, res_load4(p.res, b, t, p.T, c));
    st4(ob + (long long)t * p.C, a);
  }
}

struct NormBwdArgs {
  const float* g;       // [B,T,C] upstream gradient w.r.t. the activation output
  const float* y;       // [B,T,C] conv output saved by forward
  const float* stats;   // [B,C,2]
  const float* cond; int cond_bs;
  float* gy;            // [B,T,C] or nullptr (first AdaIN of the decoder: only gcond is needed)
  float* gcond; int gcond_bs;   // row b: d mean at [0,C), d std at [C,2C); nullptr for plain InstanceNorm
  int T; int C;
  float slope;
  int stage;            // 1: y and g slices both fit the dynamic shared memory of this launch
};

template <int CL>
__global__ void __launch_bounds__(256) norm_act_bwd_kernel(const NormBwdArgs p) {
  extern __shared__ __align__(16) float4 ntile[];   // [T][CL][2] (xhat, ga) when p.stage
  __shared__ float4 red[8][CL];
  constexpr int kNormTL = 256 / CL;
  pdl_enter();
  const int lane_c = threadIdx.x % CL, lane_t = threadIdx.x / CL;
  const int b = blockIdx.y, c = blockIdx.x * (4 * CL) + lane_c * 4;
  const float* yb = p.y + (long long)b * p.T * p.C + c;
  const float* gb = p.g + (long long)b * p.T * p.C + c;
  const float* s = p.stats + ((long long)b * p.C + c) * 2;
  const float4 s0 = ld4(s), s1 = ld4(s + 4);
  const float4 mu = make_float4(s0.x, s0.z, s1.x, s1.z), rstd = make_float4(s0.y, s0.w, s1.y, s1.w);
  float4 cm = f4zero(), cs = make_float4(1.f, 1.f, 1.f, 1.f);
  if (p.cond) {
    cm = ld4(p.cond + (long long)b * p.cond_bs + c);
    cs = ld4(p.cond + (long long)b * p.cond_bs + p.C + c);
  }
  const bool staged = p.stage && p.gy;
  // pass 1: S1 = sum_t ga, S2 = sum_t ga * xhat,  ga = g * act'(a)
  float4 S1 = f4zero(), S2 = f4zero();
#pragma unroll 4
  for (int t = lane_t; t < p.T; t += kNormTL) {
    const float4 v = ld4(yb + (long long)t * p.C), g = ld4(gb + (long long)t * p.C);
    const float4 xh = make_float4((v.x - mu.x) * rstd.x, (v.y - mu.y) * rstd.y, (v.z - mu.z) * rstd.z, (v.w - mu.w) * rstd.w);
    const float4 a = make_float4(fmaf(xh.x, cs.x, cm.x), fmaf(xh.y, cs.y, cm.y), fmaf(xh.z, cs.z, cm.z), fmaf(xh.w, cs.w, cm.w));
    const float4 ga = dact4mul(g, a, p.slope);
    if (staged) { ntile[(t * CL + lane_c) * 2] = xh; ntile[(t * CL + lane_c) * 2 + 1] = ga; }
    S1 = f4add(S1, ga);
    S2.x = fmaf(ga.x, xh.x, S2.x); S2.y = fmaf(ga.y, xh.y, S2.y); S2.z = fmaf(ga.z, xh.z, S2.z); S2.w = fmaf(ga.w, xh.w, S2.w);
  }
  S1 = block_reduce_t<CL>(S1, red, lane_c);
  S2 = block_reduce_t<CL>(S2, red, lane_c);
  if (p.gcond && lane_t == 0) {
    st4(p.gcond + (long long)b * p.gcond_bs + c, S1);
    st4(p.gcond + (long long)b * p.gcond_bs + p.C + c, S2);
  }
  if (!p.gy) return;
  // pass 2: gy = rstd * std * (ga - S1/T - xhat * S2/T)
  const float invT = 1.f / (float)p.T;
  const float4 m1 = f4scale(S1, invT), m2 = f4scale(S2, invT);
  const float4 k = make_float4(rstd.x * cs.x, rstd.y * cs.y, rstd.z * cs.z, rstd.w * cs.w);
  float* ob = p.gy + (long long)b * p.T * p.C + c;
#pragma unroll 4
  for (int t = lane_t; t < p.T; t += kNormTL) {
    float4 xh, ga;
    if (staged) {
      xh = ntile[(t * CL + lane_c) * 2]; ga = ntile[(t * CL + lane_c) * 2 + 1];
    } else {
      const float4 v = ld4(yb + (long long)t * p.C), g = ld4(gb + (long long)t * p.C);
      xh = make_float4((v.x - mu.x) * rstd.x, (v.y - mu.y) * rstd.y, (v.z - mu.z) * rstd.z, (v.w - mu.w) * rstd.w);
      const float4 a = make_float4(fmaf(xh.x, cs.x, cm.x), fmaf(xh.y, cs.y, cm.y), fmaf(xh.z, cs.z, cm.z), fmaf(xh.w, cs.w, cm.w));
      ga = dact4mul(g, a, p.slope);
    }
    float4 o;
    o.x = k.x * (ga.x - m1.x - xh.x * m2.x);
    o.y = k.y * (ga.y - m1.y - xh.y * m2.y);
    o.z = k.z * (ga.z - m1.z - xh.z * m2.z);
    o.w = k.w * (ga.w - m1.w - xh.w * m2.w);
    st4(ob + (long long)t * p.C, o);
  }
}

// ---------------------------------------------------------------------------------------------
// e2e loss (attack_utils.py:43):  L = mean((o-tgt)^2) - 0.1*mean((o-org)^2) over ALL elements,
// dL/do = 2*inv_norm*((o-tgt) - 0.1*(o-org)).  One partial per CTA -> loss_parts[step][cta].
// 16 B/element (read o,tgt,org; write g).
// ---------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(256) mse_grad_kernel(const float* __restrict__ o, const float* __restrict__ tgt,
                                                       const float* __restrict__ org, float* __restrict__ g,
                                                       long long n4, float inv_norm, float* __restrict__ loss_parts,
                                                       const int* __restrict__ step, int parts_per_step) {
  pdl_enter();
  __shared__ float wsum[8];
  float acc = 0.f;
  const float k = 2.f * inv_norm;
  for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < n4; i += (long long)gridDim.x * blockDim.x) {
    const float4 a = ld4(o + i * 4), t = ld4(tgt + i * 4), r = ld4(org + i * 4);
    const float4 d = make_float4(a.x - t.x, a.y - t.y, a.z - t.z, a.w - t.w);
    const float4 e = make_float4(a.x - r.x, a.y - r.y, a.z - r.z, a.w - r.w);
    acc += (d.x * d.x + d.y * d.y + d.z * d.z + d.w * d.w) - 0.1f * (e.x * e.x + e.y * e.y + e.z * e.z + e.w * e.w);
    st4(g + i * 4, make_float4(k * (d.x - 0.1f * e.x), k * (d.y - 0.1f * e.y), k * (d.z - 0.1f * e.z), k * (d.w - 0.1f * e.w)));
  }
  acc = warp_sum(acc);
  if ((threadIdx.x & 31) == 0) wsum[threadIdx.x >> 5] = acc;
  __syncthreads();
  if (threadIdx.x == 0) {
    float s = 0.f;
    for (int i = 0; i < 8; ++i) s += wsum[i];
    if (loss_parts) loss_parts[(long long)(*step) * parts_per_step + blockIdx.x] = s * inv_norm;
  }
}

__global__ void loss_sum_kernel(const float* __restrict__ parts, int parts_per_step, int n_iters, float* __restrict__ loss) {
  pdl_enter();
  int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n_iters) return;
  double s = 0.0;
  for (int p = 0; p < parts_per_step; ++p) s += (double)parts[(long long)i * parts_per_step + p];
  loss[i] = (float)s;
}

// ---------------------------------------------------------------------------------------------
// Fused perturbation update (attack_utils.py:40,44-46 + torch/optim/adam.py _single_tensor_adam):
//   y = tanh(w); g_w = (g_adv*eps) * (1 - y*y)
//   m = m + (g_w - m)*(1-b1);  v = v*b2 + (1-b2)*g_w*g_w
//   w = w + (-step_size * m) / (sqrt(v)/bc2_sqrt + 1e-8);   adv = x + eps*tanh(w)
// step_size = lr/(1-b1^t) and bc2_sqrt = sqrt(1-b2^t) come from a host-computed (fp64) table indexed
// by the device step counter, so one captured graph serves every iteration.
// 36 B/element: read g,w,m,v,x ; write w,m,v,adv.
// ---------------------------------------------------------------------------------------------
struct UpdateArgs {
  const float* g_adv; long long g_bs; int g_rs;   // [B,T,C] gradient w.r.t. adv
  const float* g_part[2]; int n_gpart;             // contiguous [B,T,C] partials added to g_adv in order (K-split bank dgrad)
  const float* x;                                  // [B,T,C] contiguous
  float* w; float* m; float* v;                    // contiguous
  float* adv; long long adv_bs; int adv_rs;        // may live inside the bank "cat" buffer
  float* gw_out;                                   // optional contiguous copy of g_w
  int B, T, C;
  float eps;
  const float2* table;                             // [n_iters] (step_size, bc2_sqrt)
  int* step;                                       // device step counter (0-based); incremented by the last CTA
  unsigned int* done;                              // CTA arrival counter
};

__global__ void __launch_bounds__(256) adam_tanh_update_kernel(const UpdateArgs p) {
  pdl_enter();
  const int c4n = p.C >> 2;
  const long long n4 = (long long)p.B * p.T * c4n;
  const int step = *p.step;
  const float2 tab = p.table[step];
  const float step_size = tab.x, bc2s = tab.y;
  const float b1w = (float)(1.0 - 0.9), b2 = 0.999f, b2w = (float)(1.0 - 0.999);
  for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < n4; i += (long long)gridDim.x * blockDim.x) {
    const int c = (int)(i % c4n) << 2;
    const long long bt = i / c4n;
    const int t = (int)(bt % p.T), b = (int)(bt / p.T);
    const long long lin = i * 4;
    float4 g = ld4(p.g_adv + (long long)b * p.g_bs + (long long)t * p.g_rs + c);
    for (int q = 0; q < p.n_gpart; ++q) g = f4add(g, ld4(p.g_part[q] + lin));
    float4 w = ld4(p.w + lin), m = ld4(p.m + lin), v = ld4(p.v + lin);
    const float4 x = ld4(p.x + lin);
    float gw[4], wa[4] = {w.x, w.y, w.z, w.w}, ma[4] = {m.x, m.y, m.z, m.w}, va[4] = {v.x, v.y, v.z, v.w};
    const float ga[4] = {g.x, g.y, g.z, g.w}, xa[4] = {x.x, x.y, x.z, x.w};
    float adv[4];
#pragma unroll
    for (int j = 0; j < 4; ++j) {
      const float y = tanhf(wa[j]);
      gw[j] = (ga[j] * p.eps) * (1.f - y * y);
      ma[j] = ma[j] + (gw[j] - ma[j]) * b1w;
      va[j] = va[j] * b2 + (b2w * gw[j]) * gw[j];
      const float denom = sqrtf(va[j]) / bc2s + 1e-8f;
      wa[j] = wa[j] + (-step_size * ma[j]) / denom;
      adv[j] = xa[j] + p.eps * tanhf(wa[j]);
    }
    st4(p.w + lin, make_float4(wa[0], wa[1], wa[2], wa[3]));
    st4(p.m + lin, make_float4(ma[0], ma[1], ma[2], ma[3]));
    st4(p.v + lin, make_float4(va[0], va[1], va[2], va[3]));
    st4(p.adv + (long long)b * p.adv_bs + (long long)t * p.adv_rs + c, make_float4(adv[0], adv[1], adv[2], adv[3]));
    if (p.gw_out) st4(p.gw_out + lin, make_float4(gw[0], gw[1], gw[2], gw[3]));
  }
  // last CTA to finish advances the step counter (every CTA has read it by then)
  __syncthreads();
  if (threadIdx.x == 0 && p.done) {
    __threadfence();
    const unsigned int prev = atomicAdd(p.done, 1u);
    if (prev == gridDim.x - 1) {
      *p.done = 0u;
      *p.step = step + 1;
      __threadfence();
    }
  }
}

// adv = x + eps*tanh(w) only (initial perturbation and final result, attack_utils.py:40,48)
__global__ void perturb_kernel(const float* __restrict__ x, const float* __restrict__ w, float* __restrict__ adv,
                               long long adv_bs, int adv_rs, int B, int T, int C, float eps) {
  pdl_enter();
  const int c4n = C >> 2;
  const long long n4 = (long long)B * T * c4n;
  for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < n4; i += (long long)gridDim.x * blockDim.x) {
    const int c = (int)(i % c4n) << 2;
    const long long bt = i / c4n;
    const int t = (int)(bt % T), b = (int)(bt / T);
    const float4 xv = ld4(x + i * 4), wv = ld4(w + i * 4);
    st4(adv + (long long)b * adv_bs + (long long)t * adv_rs + c,
        make_float4(xv.x + eps * tanhf(wv.x), xv.y + eps * tanhf(wv.y), xv.z + eps * tanhf(wv.z), xv.w + eps * tanhf(wv.w)));
  }
}

// ---------------------------------------------------------------------------------------------
// Universal perturbation header (reference models/header_model.py:25-68): ONE perturbation h [T, C]
// shared by the whole batch.
//   perturb:  adv[b,t,c] = clamp(x[b,t,c] + h[t,c], -1, 1)                           (:42-45)
//   grad:     g_h[t,c]   = sum_b g_adv[b,t,c] * [-1 <= x + h <= 1]                   (clamp backward; fixed order over b)
//   apply:    Adam(lr) on h with g_h (torch/optim/adam.py), h = clamp(h, -eps, eps)  (:59-65), then the next adv
// grad and apply are separate kernels because a sharded batch all-reduces g_h between them.
// ---------------------------------------------------------------------------------------------
__global__ void header_perturb_kernel(const float* __restrict__ x, const float* __restrict__ h, float* __restrict__ adv,
                                      long long adv_bs, int adv_rs, int B, int T, int C) {
  pdl_enter();
  const int c4n = C >> 2;
  const long long n4 = (long long)B * T * c4n;
  for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < n4; i += (long long)gridDim.x * blockDim.x) {
    const int c = (int)(i % c4n) << 2;
    const long long bt = i / c4n;
    const int t = (int)(bt % T), b = (int)(bt / T);
    const float4 xv = ld4(x + i * 4), hv = ld4(h + ((long long)t * C + c));
    st4(adv + (long long)b * adv_bs + (long long)t * adv_rs + c,
        make_float4(fminf(fmaxf(xv.x + hv.x, -1.f), 1.f), fminf(fmaxf(xv.y + hv.y, -1.f), 1.f),
                    fminf(fmaxf(xv.z + hv.z, -1.f), 1.f), fminf(fmaxf(xv.w + hv.w, -1.f), 1.f)));
  }
}

__global__ void header_grad_kernel(const float* __restrict__ g_adv, long long g_bs, int g_rs, const float* __restrict__ gp0,
                                   const float* __restrict__ gp1, const float* __restrict__ x,
                                   const float* __restrict__ h, float* __restrict__ gh, int B, int T, int C) {
  pdl_enter();
  const int c4n = C >> 2;
  const long long n4 = (long long)T * c4n;
  for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < n4; i += (long long)gridDim.x * blockDim.x) {
    const int c = (int)(i % c4n) << 2;
    const int t = (int)(i / c4n);
    const float4 hv = ld4(h + i * 4);
    float4 s = f4zero();
    for (int b = 0; b < B; ++b) {
      const float4 xv = ld4(x + ((long long)b * T + t) * C + c);
      float4 g = ld4(g_adv + (long long)b * g_bs + (long long)t * g_rs + c);
      if (gp0) g = f4add(g, ld4(gp0 + ((long long)b * T + t) * C + c));     // K-split partials of the bank dgrad, in order
      if (gp1) g = f4add(g, ld4(gp1 + ((long long)b * T + t) * C + c));
      const float p0 = xv.x + hv.x, p1 = xv.y + hv.y, p2 = xv.z + hv.z, p3 = xv.w + hv.w;
      s.x += (p0 >= -1.f && p0 <= 1.f) ? g.x : 0.f;
      s.y += (p1 >= -1.f && p1 <= 1.f) ? g.y : 0.f;
      s.z += (p2 >= -1.f && p2 <= 1.f) ? g.z : 0.f;
      s.w += (p3 >= -1.f && p3 <= 1.f) ? g.w : 0.f;
    }
    st4(gh + i * 4, s);
  }
}

// d loss / d input of the speaker encoder, written in the reference's [B, C, T] layout with caller strides
// (train_predictive.py:113-123 as a gradient service: loss.backward() down to perturbed_mels).  gp0 / gp1: K-split
// partials of the bank dgrad (small-M plans), added in a fixed order.
__global__ void spk_grad_out_kernel(const float* __restrict__ g_in, long long g_bs, int g_rs, const float* __restrict__ gp0,
                                    const float* __restrict__ gp1, float* __restrict__ dst, long long sb, long long sc, long long st,
                                    int B, int T, int C) {
  pdl_enter();
  const long long n = (long long)B * T * C;
  for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (long long)gridDim.x * blockDim.x) {
    const int c = (int)(i % C);
    const long long bt = i / C;
    const int t = (int)(bt % T), b = (int)(bt / T);
    float g = g_in[(long long)b * g_bs + (long long)t * g_rs + c];
    if (gp0) g += gp0[i];
    if (gp1) g += gp1[i];
    dst[b * sb + c * sc + t * st] = g;
  }
}

struct HeaderApplyArgs {
  const float* gh; float* h; float* m; float* v;     // [T, C]
  const float* x; float* adv; long long adv_bs; int adv_rs;
  int B, T, C;
  float eps;
  const float2* table;   // [n_iters] (lr/(1-b1^t), sqrt(1-b2^t))
  int* step; unsigned int* done;
};
__global__ void __launch_bounds__(256) header_apply_kernel(const HeaderApplyArgs p) {
  pdl_enter();
  const int c4n = p.C >> 2;
  const long long n4 = (long long)p.T * c4n;
  const int step = *p.step;
  const float2 tab = p.table[step];
  const float step_size = tab.x, bc2s = tab.y;
  const float b1w = (float)(1.0 - 0.9), b2 = 0.999f, b2w = (float)(1.0 - 0.999);
  for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < n4; i += (long long)gridDim.x * blockDim.x) {
    const int c = (int)(i % c4n) << 2;
    const int t = (int)(i / c4n);
    const float4 g = ld4(p.gh + i * 4);
    float4 h = ld4(p.h + i * 4), m = ld4(p.m + i * 4), v = ld4(p.v + i * 4);
    float ga[4] = {g.x, g.y, g.z, g.w}, ha[4] = {h.x, h.y, h.z, h.w}, ma[4] = {m.x, m.y, m.z, m.w}, va[4] = {v.x, v.y, v.z, v.w};
#pragma unroll
    for (int j = 0; j < 4; ++j) {
      ma[j] = ma[j] + (ga[j] - ma[j]) * b1w;
      va[j] = va[j] * b2 + (b2w * ga[j]) * ga[j];
      const float denom = sqrtf(va[j]) / bc2s + 1e-8f;
      ha[j] = ha[j] + (-step_size * ma[j]) / denom;
      ha[j] = fminf(fmaxf(ha[j], -p.eps), p.eps);
    }
    st4(p.h + i * 4, make_float4(ha[0], ha[1], ha[2], ha[3]));
    st4(p.m + i * 4, make_float4(ma[0], ma[1], ma[2], ma[3]));
    st4(p.v + i * 4, make_float4(va[0], va[1], va[2], va[3]));
    for (int b = 0; b < p.B; ++b) {
      const float4 xv = ld4(p.x + ((long long)b * p.T + t) * p.C + c);
      st4(p.adv + (long long)b * p.adv_bs + (long long)t * p.adv_rs + c,
          make_float4(fminf(fmaxf(xv.x + ha[0], -1.f), 1.f), fminf(fmaxf(xv.y + ha[1], -1.f), 1.f),
                      fminf(fmaxf(xv.z + ha[2], -1.f), 1.f), fminf(fmaxf(xv.w + ha[3], -1.f), 1.f)));
    }
  }
  __syncthreads();
  if (threadIdx.x == 0 && p.done) {
    __threadfence();
    const unsigned int prev = atomicAdd(p.done, 1u);
    if (prev == gridDim.x - 1) {
      *p.done = 0u;
      *p.step = step + 1;
      __threadfence();
    }
  }
}

// ---------------------------------------------------------------------------------------------
// Speaker-encoder tail: AdaptiveAvgPool1d(1) -> 6 residual dense blocks -> output Linear
// (models.py:307-325, 340-342), the emb/fb loss (attack_utils.py:81,125) and the whole backward of
// the tail, one CTA (1024 threads = 8 K-slices x 128 outputs) per utterance.  Requires c_h = c_out = 128.
// ---------------------------------------------------------------------------------------------
constexpr int kTailMaxDense = 8;
enum TailMode : int { TAIL_FWD = 1, TAIL_LOSS = 2, TAIL_BWD = 4 };

struct TailArgs {
  const float* h; long long h_bs; int h_rs; int T_h;   // last conv block output [B,T_h,128]
  int n_dense;
  const float* Wt1[kTailMaxDense]; const float* Wt2[kTailMaxDense];   // transposed [c][n] (forward)
  const float* W1[kTailMaxDense];  const float* W2[kTailMaxDense];    // PyTorch [n][c]  (backward)
  const float* b1[kTailMaxDense];  const float* b2[kTailMaxDense];
  const float* Wto; const float* Wo; const float* bo;
  float slope;
  int mode;
  float* acts;            // [B][2*n_dense+1][128] saved activations: pooled v0, then (y1,y2) per block... see kernel
  float* emb;             // [B,128] output embedding (TAIL_FWD)
  const float* tgt; const float* org;   // [B,128] (TAIL_LOSS)
  float inv_norm;
  float lam;              // weight of the 'away from the original' term: 0.1 in the attacks (attack_utils.py:43,81,125), lambda_param in header_model.py:56
  float* loss_parts; const int* step; int parts_per_step;
  const float* gemb; int gemb_parts;    // TAIL_BWD without TAIL_LOSS: d emb = sum_p gemb[b][p][128]
  float* gpool;           // [B,128]: d h[b,t,:] for every t (already divided by T_h)
  const int* lens_h;      // ragged batches (kernels with VL = true): valid rows of h per utterance, device int32 [B]; T_h is their maximum
};

__device__ __forceinline__ float part_sum(float (*part)[128], int n) {
  float s = 0.f;
#pragma unroll
  for (int g = 0; g < 8; ++g) s += part[g][n];
  return s;
}

// rows of h that utterance b pools over
template <bool VL>
__device__ __forceinline__ int tail_len(const TailArgs& p, int b) {
  if constexpr (VL) return p.lens_h[b];
  else return p.T_h;
}

constexpr int kTailRing = 3;                       // weight matrices in flight (64 KB each)
constexpr int kTailSmem = kTailRing * 128 * 128 * 4;

// The chain is 13 dependent 128x128 mat-vecs forward and 13 backward for ONE utterance per CTA: pure
// latency.  The matrices do not depend on the data, so they stream through a 3-deep ring of bulk copies two
// layers ahead of the arithmetic (the first two and the biases before the dependency wait).
template <bool VL = false>
__global__ void __launch_bounds__(1024) se_tail_kernel(const TailArgs p) {
  extern __shared__ __align__(16) float wring[];    // [kTailRing][128*128]
  __shared__ float part[8][128];
  __shared__ float va[2 * kTailMaxDense + 2][128];   // va[0]=pooled v0; block l: va[1+2l]=y1, va[2+2l]=y2; running v in vcur
  __shared__ float vcur[128];
  __shared__ float gv[128], gt[128];
  __shared__ float lred[4];
  __shared__ __align__(8) uint64_t tbar[kTailRing];   // "matrix i has landed in ring slot i % kTailRing"
  __shared__ float bsm[2 * kTailMaxDense + 1][128];   // biases (loop constants): fetched before the dependency wait, not one L2 round trip per layer
  const int tid = threadIdx.x, b = blockIdx.x, n = tid & 127;
  const int nsave = 2 * p.n_dense + 1;
  const int nd = p.n_dense;
  float* acts_b = p.acts + (long long)b * (nsave + p.n_dense) * 128;   // + per-block inputs v_l

  // matrix sequence of this launch: forward Wt1[0],Wt2[0],...,Wto then backward Wo,W2[nd-1],W1[nd-1],...,W2[0],W1[0]
  const int n_fwd = (p.mode & TAIL_FWD) ? 2 * nd + 1 : 0;
  const int n_all = n_fwd + ((p.mode & TAIL_BWD) ? 2 * nd + 1 : 0);
  auto mat_at = [&](int i) -> const float* {
    if (i < n_fwd) return i == 2 * nd ? p.Wto : ((i & 1) ? p.Wt2[i >> 1] : p.Wt1[i >> 1]);
    const int j = i - n_fwd;
    if (j == 0) return p.Wo;
    const int l = nd - 1 - ((j - 1) >> 1);
    return ((j - 1) & 1) ? p.W1[l] : p.W2[l];
  };
  // one elected thread streams each 64 KB matrix with two bulk copies (TMA engine, mbarrier complete_tx): per-thread
  // cp.async moved a matrix into this one SM in ~3k clk, which was the whole cost of a layer at batch 1
  auto issue = [&](int i) {
    if (i < n_all && tid == 0) {
      const float* M = mat_at(i);
      const uint32_t bar = smem_u32(&tbar[i % kTailRing]);
      const uint32_t dst = smem_u32(wring + (size_t)(i % kTailRing) * 16384);
      mbar_expect_tx(bar, 65536u);
      bulk_g2s(dst, M, 32768u, bar);
      bulk_g2s(dst + 32768u, M + 8192, 32768u, bar);
    }
  };
  int seq = 0;
  // part[g][n] = sum_{c in slice g} M[c*128+n] * vin[c] for the next matrix of the sequence
  auto dense_step = [&](const float* vin) {
    mbar_wait(smem_u32(&tbar[seq % kTailRing]), (uint32_t)(seq / kTailRing) & 1u);
    __syncthreads();                 // matrix `seq` landed for everyone, vin is visible, matrix seq-1 is no longer read
    issue(seq + 2);
    const float* M = wring + (size_t)(seq % kTailRing) * 16384;
    const int g = tid >> 7;
    float a = 0.f;
#pragma unroll
    for (int q = 0; q < 16; ++q) {
      const int c = g * 16 + q;
      a = fmaf(M[c * 128 + n], vin[c], a);
    }
    part[g][n] = a;
    ++seq;
    __syncthreads();
  };
  pdl_launch_dependents();
  if (tid == 0) {
    for (int i = 0; i < kTailRing; ++i) mbar_init(smem_u32(&tbar[i]), 1);
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  }
  __syncthreads();
  issue(0);
  issue(1);
  if ((p.mode & TAIL_FWD) && tid < 128) {
    float bl[2 * kTailMaxDense + 1];
#pragma unroll
    for (int l = 0; l < kTailMaxDense; ++l) {     // all loads in flight before the first store
      bl[2 * l] = l < p.n_dense ? p.b1[l][n] : 0.f;
      bl[2 * l + 1] = l < p.n_dense ? p.b2[l][n] : 0.f;
    }
    bl[2 * kTailMaxDense] = p.bo[n];
#pragma unroll
    for (int i = 0; i < 2 * kTailMaxDense; ++i) bsm[i][n] = bl[i];
    bsm[2 * p.n_dense][n] = bl[2 * kTailMaxDense];
  }
  pdl_wait();   // weights are loop constants; everything below reads the predecessor's output

  if (p.mode & TAIL_FWD) {
    // global average pool over time
    {
      const int g = tid >> 7;
      float a = 0.f;
      const float* hb = p.h + (long long)b * p.h_bs + n;
      for (int t = g; t < tail_len<VL>(p, b); t += 8) a += hb[(long long)t * p.h_rs];
      part[g][n] = a;
      __syncthreads();
      if (tid < 128) { vcur[n] = part_sum(part, n) / (float)tail_len<VL>(p, b); va[0][n] = vcur[n]; }
    }
    for (int l = 0; l < p.n_dense; ++l) {
      dense_step(vcur);
      if (tid < 128) {
        acts_b[(nsave + l) * 128 + n] = vcur[n];     // block input v_l (for nothing but completeness)
        va[1 + 2 * l][n] = actf(part_sum(part, n) + bsm[2 * l][n], p.slope);
      }
      dense_step(va[1 + 2 * l]);
      if (tid < 128) { float y2 = actf(part_sum(part, n) + bsm[2 * l + 1][n], p.slope); va[2 + 2 * l][n] = y2; vcur[n] = y2 + vcur[n]; }
    }
    dense_step(vcur);
    if (tid < 128) {
      gt[n] = part_sum(part, n) + bsm[2 * p.n_dense][n];     // embedding
      if (p.emb) p.emb[(long long)b * 128 + n] = gt[n];
    }
    if (tid < 128) for (int i = 0; i < nsave; ++i) acts_b[i * 128 + n] = va[i][n];
    __syncthreads();
  } else {
    if (tid < 128) for (int i = 0; i < nsave; ++i) va[i][n] = acts_b[i * 128 + n];
    __syncthreads();
  }
  if (!(p.mode & TAIL_BWD)) return;

  // ---- d emb ------------------------------------------------------------------------------
  if (p.mode & TAIL_LOSS) {
    float lp = 0.f;
    if (tid < 128) {
      const float e = gt[n], d = e - p.tgt[(long long)b * 128 + n], o = e - p.org[(long long)b * 128 + n];
      lp = d * d - p.lam * (o * o);
      gv[n] = 2.f * p.inv_norm * (d - p.lam * o);
      lp = warp_sum(lp);
      if ((tid & 31) == 0) lred[tid >> 5] = lp;
    }
    __syncthreads();
    if (tid == 0 && p.loss_parts)
      p.loss_parts[(long long)(*p.step) * p.parts_per_step + b] = (lred[0] + lred[1] + lred[2] + lred[3]) * p.inv_norm;
  } else {
    if (tid < 128) {
      float s = 0.f;
      for (int q = 0; q < p.gemb_parts; ++q) s += p.gemb[((long long)b * p.gemb_parts + q) * 128 + n];
      gv[n] = s;
    }
  }
  // ---- output layer: g_v = Wo^T g_emb  (Wo is [n_out][c]: contraction over n_out) ----------------
  dense_step(gv);
  if (tid < 128) gv[n] = part_sum(part, n);
  for (int l = p.n_dense - 1; l >= 0; --l) {
    // v_{l+1} = y2 + v_l ; y2 = act(W2 y1 + b2) ; y1 = act(W1 v_l + b1)
    __syncthreads();
    if (tid < 128) gt[n] = gv[n] * dactf(va[2 + 2 * l][n], p.slope);     // d pre-act 2
    dense_step(gt);
    if (tid < 128) gt[n] = part_sum(part, n) * dactf(va[1 + 2 * l][n], p.slope);   // d pre-act 1
    dense_step(gt);
    if (tid < 128) gv[n] = gv[n] + part_sum(part, n);
  }
  __syncthreads();
  if (tid < 128) p.gpool[(long long)b * 128 + n] = gv[n] / (float)tail_len<VL>(p, b);
}

// ---------------------------------------------------------------------------------------------
// The same tail for SMALL batches (B * 8 <= SMs): one CLUSTER of 8 CTAs per utterance.  At batch 1 the kernel above is
// one SM pulling 13-26 matrices of 64 KB through its L2 port (~12 us net per launch).  Here CTA r of the cluster owns rows
// [16r, 16r+16) of every matrix (8 KB, contiguous in both the forward [c][n] and the backward [n][c] images: the split
// is over the CONTRACTION index either way), keeps all its slices resident in shared memory (one bulk-copy burst before
// the dependency wait), multiplies its 16 inputs into a 128-wide partial vector, and the partials are reduce-scattered
// through distributed shared memory: thread n stores its partial into CTA n/16, which sums the 8 partials of its 16
// outputs in CTA order -- the same 8 x 16 summation tree as se_tail_kernel, so the results are bit-identical.
// One cluster barrier per layer; the receive buffer is double-buffered.
// ---------------------------------------------------------------------------------------------
constexpr int kTclN = 8, kTclS = 16;                 // CTAs per utterance, vector elements per CTA
constexpr int kTclMatBytes = kTclS * 128 * 4;        // one matrix slice
__device__ __forceinline__ void st_cluster_f32(float* local, uint32_t rank, float v) {
  asm volatile("{\n\t.reg .b32 ra;\n\tmapa.shared::cluster.u32 ra, %0, %1;\n\tst.shared::cluster.f32 [ra], %2;\n\t}"
               ::"r"(smem_u32(local)), "r"(rank), "f"(v) : "memory");
}

template <bool VL = false>
__global__ void __launch_bounds__(128) se_tail_cluster_kernel(const TailArgs p) {
  extern __shared__ __align__(16) float wsl[];          // [n_all][16][128] this CTA's matrix slices
  __shared__ float recv[2][kTclN][kTclS];
  __shared__ float va[2 * kTailMaxDense + 2][kTclS];
  __shared__ float bsm[2 * kTailMaxDense + 1][kTclS];
  __shared__ float vcur[kTclS], gv[kTclS], gt[kTclS];
  __shared__ float red[8][kTclS];
  __shared__ float lossbuf[kTclN];
  __shared__ __align__(8) uint64_t wbar;
  const int tid = threadIdx.x, j = tid & 15;
  const uint32_t r = cluster_ctarank();
  const int b = blockIdx.x / kTclN;
  const int nd = p.n_dense, nsave = 2 * nd + 1;
  const int c0 = (int)r * kTclS;                        // my slice of every 128-vector
  float* acts_b = p.acts + (long long)b * (nsave + nd) * 128;
  const int n_fwd = (p.mode & TAIL_FWD) ? 2 * nd + 1 : 0;
  const int n_all = n_fwd + ((p.mode & TAIL_BWD) ? 2 * nd + 1 : 0);
  auto mat_at = [&](int i) -> const float* {
    if (i < n_fwd) return i == 2 * nd ? p.Wto : ((i & 1) ? p.Wt2[i >> 1] : p.Wt1[i >> 1]);
    const int q = i - n_fwd;
    if (q == 0) return p.Wo;
    const int l = nd - 1 - ((q - 1) >> 1);
    return ((q - 1) & 1) ? p.W1[l] : p.W2[l];
  };
  pdl_launch_dependents();
  if (tid == 0) {
    mbar_init(smem_u32(&wbar), 1);
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    mbar_expect_tx(smem_u32(&wbar), (uint32_t)n_all * kTclMatBytes);
    for (int i = 0; i < n_all; ++i)
      bulk_g2s(smem_u32(wsl + (size_t)i * kTclS * 128), mat_at(i) + (size_t)c0 * 128, kTclMatBytes, smem_u32(&wbar));
  }
  if ((p.mode & TAIL_FWD) && tid < kTclS) {
    float bl[2 * kTailMaxDense + 1];
#pragma unroll
    for (int l = 0; l < kTailMaxDense; ++l) {     // all loads in flight before the first store
      bl[2 * l] = l < nd ? p.b1[l][c0 + j] : 0.f;
      bl[2 * l + 1] = l < nd ? p.b2[l][c0 + j] : 0.f;
    }
    bl[2 * kTailMaxDense] = p.bo[c0 + j];
#pragma unroll
    for (int i = 0; i < 2 * kTailMaxDense; ++i) bsm[i][j] = bl[i];
    bsm[2 * nd][j] = bl[2 * kTailMaxDense];
  }
  cluster_sync_all();      // every CTA of the cluster is running (its shared memory may be written) and the barrier is initialised
  pdl_wait();              // weights and biases are loop constants; everything below reads the predecessor's output
  mbar_wait(smem_u32(&wbar), 0);
  int seq = 0, buf = 0;
  // out[n] (n in my slice, returned to threads tid < 16) = sum_c M[c][n] vin[c]: my 16 rows times my 16 inputs -> a
  // 128-wide partial, element n stored into CTA n/16; after the cluster barrier the 8 partials are summed in CTA order
  auto dense_step = [&](const float* vin) -> float {
    const float* M = wsl + (size_t)seq * kTclS * 128;
    float a = 0.f;
#pragma unroll
    for (int q = 0; q < kTclS; ++q) a = fmaf(M[q * 128 + tid], vin[q], a);
    st_cluster_f32(&recv[buf][r][tid & 15], (uint32_t)(tid >> 4), a);
    cluster_sync_all();
    float y = 0.f;
    if (tid < kTclS) {
#pragma unroll
      for (int g = 0; g < kTclN; ++g) y += recv[buf][g][j];
    }
    ++seq; buf ^= 1;
    return y;
  };

  if (p.mode & TAIL_FWD) {
    {   // global average pool over time of my 16 channels (8 time lanes, summed in lane order)
      const int g = tid >> 4;
      float a = 0.f;
      const float* hb = p.h + (long long)b * p.h_bs + c0 + j;
      for (int t = g; t < tail_len<VL>(p, b); t += 8) a += hb[(long long)t * p.h_rs];
      red[g][j] = a;
      __syncthreads();
      if (tid < kTclS) {
        float s2 = 0.f;
#pragma unroll
        for (int g2 = 0; g2 < 8; ++g2) s2 += red[g2][j];
        vcur[j] = s2 / (float)tail_len<VL>(p, b); va[0][j] = vcur[j];
      }
      __syncthreads();
    }
    for (int l = 0; l < nd; ++l) {
      float y = dense_step(vcur);
      if (tid < kTclS) {
        acts_b[(nsave + l) * 128 + c0 + j] = vcur[j];
        va[1 + 2 * l][j] = actf(y + bsm[2 * l][j], p.slope);
      }
      __syncthreads();
      y = dense_step(va[1 + 2 * l]);
      if (tid < kTclS) { const float y2 = actf(y + bsm[2 * l + 1][j], p.slope); va[2 + 2 * l][j] = y2; vcur[j] = y2 + vcur[j]; }
      __syncthreads();
    }
    const float y = dense_step(vcur);
    if (tid < kTclS) {
      gt[j] = y + bsm[2 * nd][j];     // embedding
      if (p.emb) p.emb[(long long)b * 128 + c0 + j] = gt[j];
      for (int i = 0; i < nsave; ++i) acts_b[i * 128 + c0 + j] = va[i][j];
    }
    __syncthreads();
  } else {
    if (tid < kTclS) for (int i = 0; i < nsave; ++i) va[i][j] = acts_b[i * 128 + c0 + j];
    __syncthreads();
  }
  if (p.mode & TAIL_BWD) {
    // ---- d emb ----
    if (p.mode & TAIL_LOSS) {
      float lp = 0.f;
      if (tid < kTclS) {
        const float e = gt[j], d = e - p.tgt[(long long)b * 128 + c0 + j], o = e - p.org[(long long)b * 128 + c0 + j];
        lp = d * d - p.lam * (o * o);
        gv[j] = 2.f * p.inv_norm * (d - p.lam * o);
      }
      if (tid < 32) {
        lp = warp_sum(lp);
        if (tid == 0) st_cluster_f32(&lossbuf[r], 0u, lp);     // summed by CTA 0 after the next cluster barrier
      }
    } else if (tid < kTclS) {
      float s2 = 0.f;
      for (int q = 0; q < p.gemb_parts; ++q) s2 += p.gemb[((long long)b * p.gemb_parts + q) * 128 + c0 + j];
      gv[j] = s2;
    }
    __syncthreads();
    // ---- output layer: g_v = Wo^T g_emb (contraction over the rows of Wo: my slice of g_emb times my rows) ----
    float y = dense_step(gv);
    if ((p.mode & TAIL_LOSS) && r == 0 && tid == 0 && p.loss_parts) {
      float s2 = 0.f;
      for (int g = 0; g < kTclN; ++g) s2 += lossbuf[g];
      p.loss_parts[(long long)(*p.step) * p.parts_per_step + b] = s2 * p.inv_norm;
    }
    if (tid < kTclS) gv[j] = y;
    for (int l = nd - 1; l >= 0; --l) {
      __syncthreads();
      if (tid < kTclS) gt[j] = gv[j] * dactf(va[2 + 2 * l][j], p.slope);     // d pre-act 2
      __syncthreads();
      y = dense_step(gt);
      if (tid < kTclS) gt[j] = y * dactf(va[1 + 2 * l][j], p.slope);          // d pre-act 1
      __syncthreads();
      y = dense_step(gt);
      if (tid < kTclS) gv[j] = gv[j] + y;
    }
    __syncthreads();
    if (tid < kTclS) p.gpool[(long long)b * 128 + c0 + j] = gv[j] / (float)tail_len<VL>(p, b);
  }
  cluster_sync_all();      // nobody leaves while a peer may still store into its shared memory
}

// ---------------------------------------------------------------------------------------------
// AdaIN affine layers: cond_l = Linear_l(emb), l < 2*n_blocks  (models.py:397-399, 420, 427)
// forward grid (B, L): 256 outputs per CTA.  backward grid (B, L): partial d emb per layer, summed
// (fixed order) by the tail kernel.
// ---------------------------------------------------------------------------------------------
constexpr int kMaxAffine = 2 * 8;
struct AffineArgs {
  const float* Wt[kMaxAffine];   // [c][2C] transposed
  const float* W[kMaxAffine];    // [2C][c]
  const float* bias[kMaxAffine];
  const float* emb;              // [B,128]
  float* cond;                   // [B][L][256]
  const float* gcond;            // [B][L][256]
  float* gemb_parts;             // [B][L][128]
  int L;
};

__global__ void __launch_bounds__(1024) affine_fwd_kernel(const AffineArgs p) {
  __shared__ float e[128];
  __shared__ float part[4][256];
  const int b = blockIdx.x, l = blockIdx.y, tid = threadIdx.x, n = tid & 255, g = tid >> 8;
  pdl_launch_dependents();
  const float* M = p.Wt[l];
  float wv[32];
#pragma unroll
  for (int q = 0; q < 32; ++q) wv[q] = M[(g * 32 + q) * 256 + n];   // loop constants: fetched before the dependency wait
  pdl_wait();
  if (tid < 128) e[tid] = p.emb[(long long)b * 128 + tid];
  __syncthreads();
  float a = 0.f;
#pragma unroll
  for (int q = 0; q < 32; ++q) a = fmaf(wv[q], e[g * 32 + q], a);
  part[g][n] = a;
  __syncthreads();
  if (tid < 256) p.cond[((long long)b * p.L + l) * 256 + n] = part[0][n] + part[1][n] + part[2][n] + part[3][n] + p.bias[l][n];
}

__global__ void __launch_bounds__(1024) affine_bwd_kernel(const AffineArgs p) {
  __shared__ float gc[256];
  __shared__ float part[8][128];
  const int b = blockIdx.x, l = blockIdx.y, tid = threadIdx.x, c = tid & 127, g = tid >> 7;
  pdl_launch_dependents();
  const float* M = p.W[l];   // [n][c]
  float wv[32];
#pragma unroll
  for (int q = 0; q < 32; ++q) wv[q] = M[(g * 32 + q) * 128 + c];   // loop constants: fetched before the dependency wait
  pdl_wait();
  if (tid < 256) gc[tid] = p.gcond[((long long)b * p.L + l) * 256 + tid];
  __syncthreads();
  float a = 0.f;
#pragma unroll
  for (int q = 0; q < 32; ++q) a = fmaf(wv[q], gc[g * 32 + q], a);
  part[g][c] = a;
  __syncthreads();
  if (tid < 128) {
    float s = 0.f;
#pragma unroll
    for (int q = 0; q < 8; ++q) s += part[q][c];
    p.gemb_parts[((long long)b * p.L + l) * 128 + c] = s;
  }
}

}  // namespace avc
