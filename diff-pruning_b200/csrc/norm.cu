// norm.cu — GroupNorm (+SiLU, +dropout) forward/backward over NHWC views.  HBM-bound: every kernel reads rows
// of C contiguous floats (coalesced), each thread owns fixed channel(s) so per-channel scale/shift live in
// registers, and all cross-block reductions go through fixed-order partial buffers (no atomics).
#include <cuda_bf16.h>
#include "common.cuh"

namespace {
constexpr int NT = 256;
constexpr int MAXCPT = 4;  // channels per thread when C > 256 (C <= 1024)

struct Map {  // thread -> (channel slot, pixel lane)
  int CT, PL, PPC, nchunks;
};
static inline Map make_map(int HW, int C) {
  Map m;
  if (C >= NT) { m.CT = NT; m.PL = 1; }
  else { int ct = 32; while (ct < C) ct <<= 1; m.CT = ct; m.PL = NT / ct; }
  int ppc = 8192 / C; if (ppc < m.PL) ppc = m.PL; if (ppc > HW) ppc = HW; if (ppc < 1) ppc = 1;
  m.PPC = ppc; m.nchunks = (HW + ppc - 1) / ppc;
  return m;
}

// Dropout keep-mask: a counter-based hash (splitmix64) of (seed, element index / 4) yields 64 bits = one 16-bit uniform for each of
// 4 consecutive elements (the float4 kernels hash once per load); keep if u16 >= thr = round(p * 65536), survivors scaled by
// 65536 / (65536 - thr) (the exact inverse keep rate).  Forward and backward regenerate the same mask from the element index alone.
struct Drop {
  uint64_t seed; uint32_t thr; float inv; bool on;
};
__device__ __forceinline__ Drop make_drop(const dp_gn_args& a) {
  Drop d;
  d.on = a.dropout_p > 0.f;
  d.seed = a.dropout_seed + ((d.on && a.dropout_seed_dev) ? *a.dropout_seed_dev : 0ull);
  d.thr = d.on ? __float2uint_rn(a.dropout_p * 65536.f) : 0u;
  d.inv = 65536.f / (float)(65536u - d.thr);
  return d;
}
__device__ __forceinline__ uint64_t drop_bits(uint64_t seed, uint64_t group) {
  uint64_t z = seed + 0x9E3779B97F4A7C15ull * (group + 1);
  z = (z ^ (z >> 30)) * 0xBF58476D1CE4E5B9ull;
  z = (z ^ (z >> 27)) * 0x94D049BB133111EBull;
  return z ^ (z >> 31);
}
__device__ __forceinline__ float keep_scale(const Drop& d, uint64_t idx) {
  const uint32_t u = (uint32_t)(drop_bits(d.seed, idx >> 2) >> (16 * (int)(idx & 3))) & 0xFFFFu;
  return u >= d.thr ? d.inv : 0.f;
}
__device__ __forceinline__ void keep_scale4(const Drop& d, uint64_t idx0 /* % 4 == 0 */, float (&k)[4]) {
  const uint64_t z = drop_bits(d.seed, idx0 >> 2);
#pragma unroll
  for (int e = 0; e < 4; ++e) k[e] = ((uint32_t)(z >> (16 * e)) & 0xFFFFu) >= d.thr ? d.inv : 0.f;
}
// SiLU through the special-function unit: ex2.approx + rcp.approx (~3e-7 relative on the sigmoid, an order below the 22-bit operand
// split of the convolutions that consume it).  The accurate expf + correctly rounded reciprocal cost ~16 instructions per element and made
// every GroupNorm kernel with a SiLU issue-bound at ~40 % of the HBM rate (profiles/r02_experiments.md, section 17).
__device__ __forceinline__ float sigmoidf_fast(float x) {
  float e, r;
  asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(e) : "f"(-1.4426950408889634f * x));
  asm("rcp.approx.ftz.f32 %0, %1;" : "=f"(r) : "f"(1.0f + e));
  return r;
}

__global__ void __launch_bounds__(NT) gn_stats_kernel(const dp_gn_args a, const Map mp, double* __restrict__ ws) {
  extern __shared__ double sh[];  // [2][PL*CT or C]
  const int n = blockIdx.y, chunk = blockIdx.x, tid = threadIdx.x;
  const int ct = tid % mp.CT, pl = tid / mp.CT;
  const int p0 = chunk * mp.PPC, p1 = min(a.HW, p0 + mp.PPC);
  double s[MAXCPT] = {0, 0, 0, 0}, q[MAXCPT] = {0, 0, 0, 0};
  const float* xb = a.x + (long long)n * a.HW * a.ldx;
  for (int pix = p0 + pl; pix < p1; pix += mp.PL) {
    const float* row = xb + (long long)pix * a.ldx;
#pragma unroll
    for (int u = 0; u < MAXCPT; ++u) {
      int c = ct + u * NT;
      if (c < a.C) { float v = __ldg(row + c); s[u] += v; q[u] += (double)v * v; }
    }
  }
  const int slots = (a.C > NT) ? a.C : mp.PL * mp.CT;
  double* shs = sh; double* shq = sh + slots;
  if (a.C > NT) {
#pragma unroll
    for (int u = 0; u < MAXCPT; ++u) { int c = ct + u * NT; if (c < a.C) { shs[c] = s[u]; shq[c] = q[u]; } }
  } else { shs[pl * mp.CT + ct] = s[0]; shq[pl * mp.CT + ct] = q[0]; }
  __syncthreads();
  const int cpg = a.C / a.G;
  for (int g = tid; g < a.G; g += NT) {
    double ts = 0, tq = 0;
    for (int c = g * cpg; c < (g + 1) * cpg; ++c) {
      if (a.C > NT) { ts += shs[c]; tq += shq[c]; }
      else for (int l = 0; l < mp.PL; ++l) { ts += shs[l * mp.CT + c]; tq += shq[l * mp.CT + c]; }
    }
    double* o = ws + (((long long)n * mp.nchunks + chunk) * a.G + g) * 2;
    o[0] = ts; o[1] = tq;
  }
}

// mean / rstd of a group from its fp64 sum / sum of squares
__device__ __forceinline__ void gn_stats_final(const dp_gn_args& a, double ts, double tq, float& mean_f, float& rstd_f) {
  double m = (double)a.HW * (a.C / a.G);
  double mean = ts / m, var = tq / m - mean * mean;
  if (var < 0) var = 0;
  mean_f = (float)mean;
  rstd_f = (float)(1.0 / sqrt(var + (double)a.eps));
}
// mean / rstd of (n, g) from the stats partials: fixed-order fp64 sums over the chunks
__device__ __forceinline__ void gn_finalize_one(const dp_gn_args& a, const Map& mp, const double* __restrict__ ws, int n, int g,
                                                float& mean_f, float& rstd_f) {
  double ts = 0, tq = 0;
#pragma unroll 4
  for (int ch = 0; ch < mp.nchunks; ++ch) {
    const double* o = ws + (((long long)n * mp.nchunks + ch) * a.G + g) * 2;
    ts += o[0]; tq += o[1];
  }
  gn_stats_final(a, ts, tq, mean_f, rstd_f);
}

// Images of many chunks (LSUN 256x256: 512-1024 per image): one WARP per (n, g) — lane l sums chunks l, l + 32, ... in order, then a fixed
// butterfly.  (One thread per (n, g) walked all chunks serially: N * G = 128 threads in one block, ~100 us per 256x256 layer, more than
// the stats and apply passes over the 134 MB tensor take together.)
__global__ void __launch_bounds__(256) gn_finalize_kernel(const dp_gn_args a, const Map mp, const double* __restrict__ ws) {
  const int i = blockIdx.x * 8 + (threadIdx.x >> 5), lane = threadIdx.x & 31;  // (n, g), whole warps
  if (i >= a.N * a.G) return;
  const int n = i / a.G, g = i - n * a.G;
  double ts = 0, tq = 0;
  for (int ch = lane; ch < mp.nchunks; ch += 32) {
    const double* o = ws + (((long long)n * mp.nchunks + ch) * a.G + g) * 2;
    ts += o[0]; tq += o[1];
  }
  ts = warp_sum_d(ts); tq = warp_sum_d(tq);
  if (lane == 0) gn_stats_final(a, ts, tq, a.mean[i], a.rstd[i]);
}

// Folded finalize (images of at most GN_FOLD_FWD chunks): there is no finalize launch; every block of the apply pass re-derives the
// statistics of its image from the partials (G x nchunks fp64 pairs out of L2: the same sums in the same order, so every block gets
// the same bits) into shared memory, and the chunk-0 block stores them for the backward.  One tiny dependent launch less per layer on
// a chain that is launch-latency bound (51 GroupNorms per C1 pass).
constexpr int GN_FOLD_FWD = 32;
__device__ __forceinline__ void gn_fold_stats(const dp_gn_args& a, const Map& mp, const double* __restrict__ ws, int n, bool store,
                                              float* smean, float* srstd) {
  for (int g = threadIdx.x; g < a.G; g += NT) {
    float mu, rs;
    gn_finalize_one(a, mp, ws, n, g, mu, rs);
    smean[g] = mu; srstd[g] = rs;
    if (store) { a.mean[n * a.G + g] = mu; a.rstd[n * a.G + g] = rs; }
  }
  __syncthreads();
}

__global__ void __launch_bounds__(NT) gn_apply_kernel(const dp_gn_args a, const Map mp, const double* __restrict__ fold_ws) {
  extern __shared__ float shst[];   // folded finalize: [2][G]
  const int n = blockIdx.y, chunk = blockIdx.x, tid = threadIdx.x;
  const int ct = tid % mp.CT, pl = tid / mp.CT;
  const int p0 = chunk * mp.PPC, p1 = min(a.HW, p0 + mp.PPC);
  const int cpg = a.C / a.G;
  const float* gmean = a.mean + n * a.G;
  const float* grstd = a.rstd + n * a.G;
  if (fold_ws) { gn_fold_stats(a, mp, fold_ws, n, chunk == 0, shst, shst + a.G); gmean = shst; grstd = shst + a.G; }
  float sc[MAXCPT], shf[MAXCPT];
#pragma unroll
  for (int u = 0; u < MAXCPT; ++u) {
    int c = ct + u * NT;
    if (c < a.C) {
      int g = c / cpg;
      float mu = gmean[g], rs = grstd[g];
      float ga = __ldg(a.gamma + c), be = __ldg(a.beta + c);
      sc[u] = rs * ga; shf[u] = be - mu * rs * ga;
    } else { sc[u] = 0.f; shf[u] = 0.f; }
  }
  const float* xb = a.x + (long long)n * a.HW * a.ldx;
  float* yb = a.y + (long long)n * a.HW * a.ldy;
  const Drop drop = make_drop(a);
  float amax = 0.f;
  for (int pix = p0 + pl; pix < p1; pix += mp.PL) {
    const float* row = xb + (long long)pix * a.ldx;
    float* orow = yb + (long long)pix * a.ldy;
#pragma unroll
    for (int u = 0; u < MAXCPT; ++u) {
      int c = ct + u * NT;
      if (c < a.C) {
        float y = fmaf(__ldg(row + c), sc[u], shf[u]);
        if (a.silu) y = y * sigmoidf_fast(y);
        if (drop.on) y *= keep_scale(drop, ((uint64_t)n * a.HW + pix) * a.C + c);
        if (a.y) orow[c] = y;
        if (a.y_bf16) reinterpret_cast<__nv_bfloat16*>(a.y_bf16)[((long long)n * a.HW + pix) * a.ldyb + c] = __float2bfloat16_rn(y);
        amax = fmaxf(amax, fabsf(y));
      }
    }
  }
  if (a.amax_y) amax_commit(a.amax_y, amax);
}

// ---- backward ----
__device__ __forceinline__ float gn_dy(const dp_gn_args& a, float g, float y) {   // g: dy with the dropout keep-scale already applied
  if (a.silu) { float s = sigmoidf_fast(y); g *= s * (1.f + y * (1.f - s)); }
  return g;
}

__global__ void __launch_bounds__(NT) gn_bwd_partial_kernel(const dp_gn_args a, const Map mp, float* __restrict__ part) {
  extern __shared__ float shf32[];  // [2][PL*CT]   (only used when C <= NT)
  const int n = blockIdx.y, chunk = blockIdx.x, tid = threadIdx.x;
  const int ct = tid % mp.CT, pl = tid / mp.CT;
  const int p0 = chunk * mp.PPC, p1 = min(a.HW, p0 + mp.PPC);
  const int cpg = a.C / a.G;
  float mu[MAXCPT], rs[MAXCPT], ga[MAXCPT], be[MAXCPT], s1[MAXCPT], s2[MAXCPT];
#pragma unroll
  for (int u = 0; u < MAXCPT; ++u) {
    int c = ct + u * NT; s1[u] = 0.f; s2[u] = 0.f;
    if (c < a.C) { int g = c / cpg; mu[u] = a.mean[n * a.G + g]; rs[u] = a.rstd[n * a.G + g]; ga[u] = __ldg(a.gamma + c); be[u] = __ldg(a.beta + c); }
    else { mu[u] = rs[u] = ga[u] = be[u] = 0.f; }
  }
  const float* xb = a.x + (long long)n * a.HW * a.ldx;
  const float* db = a.dy + (long long)n * a.HW * a.lddy;
  const Drop drop = make_drop(a);
  for (int pix = p0 + pl; pix < p1; pix += mp.PL) {
#pragma unroll
    for (int u = 0; u < MAXCPT; ++u) {
      int c = ct + u * NT;
      if (c < a.C) {
        float xh = (__ldg(xb + (long long)pix * a.ldx + c) - mu[u]) * rs[u];
        float y = fmaf(xh, ga[u], be[u]);
        float g = __ldg(db + (long long)pix * a.lddy + c);
        if (drop.on) g *= keep_scale(drop, ((uint64_t)n * a.HW + pix) * a.C + c);
        g = gn_dy(a, g, y);
        s1[u] += g; s2[u] += g * xh;
      }
    }
  }
  float* o = part + ((long long)n * mp.nchunks + chunk) * 2 * a.C;
  if (a.C > NT) {
#pragma unroll
    for (int u = 0; u < MAXCPT; ++u) { int c = ct + u * NT; if (c < a.C) { o[c] = s1[u]; o[a.C + c] = s2[u]; } }
  } else {
    float* sa = shf32; float* sb = shf32 + mp.PL * mp.CT;
    sa[pl * mp.CT + ct] = s1[0]; sb[pl * mp.CT + ct] = s2[0];
    __syncthreads();
    if (pl == 0 && ct < a.C) {
      float t1 = 0.f, t2 = 0.f;
      for (int l = 0; l < mp.PL; ++l) { t1 += sa[l * mp.CT + ct]; t2 += sb[l * mp.CT + ct]; }
      o[ct] = t1; o[a.C + ct] = t2;
    }
  }
}

// Per image: channel sums over the `nrows` partial rows (fixed order, fp64) -> fin[n][2][C] for the dgamma / dbeta kernel (written when
// `store`), then the two gamma-weighted group means -> coef[g][2].  shc: [2][C] floats of shared memory; coef: shared memory.
__device__ __forceinline__ void gn_bwd_coef(const dp_gn_args& a, int nrows, const float* part, float* fin,   // part == fin when nrows == 1
                                            int n, bool store, float* shc, float* coef) {
  const int tid = threadIdx.x;
  for (int c = tid; c < a.C; c += NT) {
    double t1 = 0, t2 = 0;
#pragma unroll 4
    for (int ch = 0; ch < nrows; ++ch) {
      const float* o = part + ((long long)n * nrows + ch) * 2 * a.C;
      t1 += o[c]; t2 += o[a.C + c];
    }
    if (store) {
      fin[((long long)n * 2) * a.C + c] = (float)t1;
      fin[((long long)n * 2 + 1) * a.C + c] = (float)t2;
    }
    float ga = __ldg(a.gamma + c);
    shc[c] = (float)t1 * ga; shc[a.C + c] = (float)t2 * ga;
  }
  __syncthreads();
  const int cpg = a.C / a.G;
  const double inv_m = 1.0 / ((double)a.HW * cpg);
  for (int g = tid; g < a.G; g += NT) {
    double u1 = 0, u2 = 0;
    for (int c = g * cpg; c < (g + 1) * cpg; ++c) { u1 += shc[c]; u2 += shc[a.C + c]; }
    coef[g * 2] = (float)(u1 * inv_m);
    coef[g * 2 + 1] = (float)(u2 * inv_m);
  }
  __syncthreads();
}
// There is no finalize launch in the backward: every block of the apply pass derives the coefficients of its image itself, from the
// chunk partials when an image has at most GN_FOLD_BWD of them (2 C nchunks floats out of L2; the chunk-0 block also stores fin), else
// from fin, which gn_bwd_reduce_kernel fills first: block = 32 channels x 32 chunk lanes, lane l sums chunks l, l + 32, ... in order, then
// a fixed-order sum over the lanes (deterministic).  (The former per-image finalize block walked all chunks serially per channel: N = 4
// blocks and ~100 us per 256x256 LSUN layer.)
constexpr int GN_FOLD_BWD = 8;
__global__ void __launch_bounds__(1024) gn_bwd_reduce_kernel(const dp_gn_args a, const Map mp, const float* __restrict__ part,
                                                             float* __restrict__ fin) {
  __shared__ double s1[32][33], s2[32][33];
  const int cx = threadIdx.x & 31, ly = threadIdx.x >> 5;
  const int c = blockIdx.x * 32 + cx, n = blockIdx.y;
  double t1 = 0, t2 = 0;
  if (c < a.C)
    for (int ch = ly; ch < mp.nchunks; ch += 32) {
      const float* o = part + ((long long)n * mp.nchunks + ch) * 2 * a.C;
      t1 += o[c]; t2 += o[a.C + c];
    }
  s1[ly][cx] = t1; s2[ly][cx] = t2;
  __syncthreads();
  if (ly == 0 && c < a.C) {
    for (int l = 1; l < 32; ++l) { t1 += s1[l][cx]; t2 += s2[l][cx]; }
    fin[((long long)n * 2) * a.C + c] = (float)t1;
    fin[((long long)n * 2 + 1) * a.C + c] = (float)t2;
  }
}

__global__ void __launch_bounds__(1024) gn_bwd_param_kernel(const dp_gn_args a, const float* __restrict__ fin) {
  // block = 32 channels x 32 image lanes; fixed-order tree over the lanes (deterministic), coalesced 128-byte rows.  The grid is
  // only C/32 blocks, so the per-lane serial walk over images is the critical path: 32 lanes keep it at N/32 dependent loads.
  __shared__ double sb[32][33], sg[32][33];
  const int cx = threadIdx.x & 31, ly = threadIdx.x >> 5;
  const int c = blockIdx.x * 32 + cx;
  double tb = 0, tg = 0;
  if (c < a.C)
    for (int n = ly; n < a.N; n += 32) { tb += fin[((long long)n * 2) * a.C + c]; tg += fin[((long long)n * 2 + 1) * a.C + c]; }
  sb[ly][cx] = tb; sg[ly][cx] = tg;
  __syncthreads();
  if (ly == 0 && c < a.C) {
    for (int l = 1; l < 32; ++l) { tb += sb[l][cx]; tg += sg[l][cx]; }
    if (a.dbeta) a.dbeta[c] += (float)tb;
    if (a.dgamma) a.dgamma[c] += (float)tg;
  }
}

__global__ void __launch_bounds__(NT) gn_bwd_apply_kernel(const dp_gn_args a, const Map mp, const float* part, int nrows, float* fin) {
  extern __shared__ float shfold[];   // folded finalize: [2][C] weighted sums + [G][2] coefficients
  const int n = blockIdx.y, chunk = blockIdx.x, tid = threadIdx.x;
  const int ct = tid % mp.CT, pl = tid / mp.CT;
  const int p0 = chunk * mp.PPC, p1 = min(a.HW, p0 + mp.PPC);
  const int cpg = a.C / a.G;
  const float* coef = shfold + 2 * a.C;
  gn_bwd_coef(a, nrows, part, fin, n, chunk == 0 && part != fin, shfold, shfold + 2 * a.C);
  float mu[MAXCPT], rs[MAXCPT], ga[MAXCPT], be[MAXCPT], c1[MAXCPT], c2[MAXCPT];
#pragma unroll
  for (int u = 0; u < MAXCPT; ++u) {
    int c = ct + u * NT;
    if (c < a.C) {
      int g = c / cpg; mu[u] = a.mean[n * a.G + g]; rs[u] = a.rstd[n * a.G + g]; ga[u] = __ldg(a.gamma + c); be[u] = __ldg(a.beta + c);
      c1[u] = coef[g * 2]; c2[u] = coef[g * 2 + 1];
    } else { mu[u] = rs[u] = ga[u] = be[u] = c1[u] = c2[u] = 0.f; }
  }
  const float* xb = a.x + (long long)n * a.HW * a.ldx;
  const float* db = a.dy + (long long)n * a.HW * a.lddy;
  const Drop drop = make_drop(a);
  float* ob = a.dx + (long long)n * a.HW * a.lddx;
  const float* ab = a.dx_add ? a.dx_add + (long long)n * a.HW * a.ldadd : nullptr;
  const float* ab2 = a.dx_add2 ? a.dx_add2 + (long long)n * a.HW * a.ldadd2 : nullptr;
  float amax = 0.f;
  for (int pix = p0 + pl; pix < p1; pix += mp.PL) {
#pragma unroll
    for (int u = 0; u < MAXCPT; ++u) {
      int c = ct + u * NT;
      if (c < a.C) {
        float xh = (__ldg(xb + (long long)pix * a.ldx + c) - mu[u]) * rs[u];
        float y = fmaf(xh, ga[u], be[u]);
        float g = __ldg(db + (long long)pix * a.lddy + c);
        if (drop.on) g *= keep_scale(drop, ((uint64_t)n * a.HW + pix) * a.C + c);
        g = gn_dy(a, g, y);
        float d = rs[u] * (ga[u] * g - c1[u] - xh * c2[u]);
        if (ab) d += ab[(long long)pix * a.ldadd + c];
        if (ab2) d += ab2[(long long)pix * a.ldadd2 + c];
        ob[(long long)pix * a.lddx + c] = d;
        amax = fmaxf(amax, fabsf(d));
      }
    }
  }
  if (a.amax_dx) amax_commit(a.amax_dx, amax);
}


// ------------------------------------------------------------------------------------------------------------
// float4 variants (C % 4 == 0, 16-byte aligned views): each thread owns 4 consecutive channels, 8 pixel lanes for
// C = 128.  Same partial-buffer layouts as the scalar kernels, so finalize/param kernels are shared.
static inline Map make_map4(int HW, int C) {
  Map m;
  int c4 = C / 4, ct = 8;
  while (ct < c4) ct <<= 1;
  m.CT = ct; m.PL = NT / ct;
  int ppc = 16384 / C; if (ppc < m.PL) ppc = m.PL; if (ppc > HW) ppc = HW; if (ppc < 1) ppc = 1;
  m.PPC = ppc; m.nchunks = (HW + ppc - 1) / ppc;
  return m;
}
__device__ __forceinline__ float4 ld4(const float* p) { return __ldg(reinterpret_cast<const float4*>(p)); }
constexpr int GU = 4;      // pixels per software-pipeline group of the float4 kernels

__global__ void __launch_bounds__(NT) gn_stats4_kernel(const dp_gn_args a, const Map mp, double* __restrict__ ws) {
  extern __shared__ double sh[];  // [2][PL][CT*4]
  const int n = blockIdx.y, chunk = blockIdx.x, tid = threadIdx.x;
  const int ct = tid % mp.CT, pl = tid / mp.CT, c0 = ct * 4;
  const int p0 = chunk * mp.PPC, p1 = min(a.HW, p0 + mp.PPC);
  double s[4] = {0, 0, 0, 0}, q[4] = {0, 0, 0, 0};
  const float* xb = a.x + (long long)n * a.HW * a.ldx + c0;
  if (c0 < a.C) {
    // groups of GU pixels, the next group's loads in flight while this one is summed: these kernels are bound by the serial chain of
    // memory round trips inside a block (ncu: 14-26 % DRAM utilisation), not by bandwidth.  Same summation order as a plain loop.
    float4 cur[GU], nxt[GU];
    const int gstep = GU * mp.PL;
    auto load = [&](int base, float4 (&buf)[GU]) {
#pragma unroll
      for (int u = 0; u < GU; ++u) { const int px = base + u * mp.PL; buf[u] = px < p1 ? ld4(xb + (long long)px * a.ldx) : make_float4(0, 0, 0, 0); }
    };
    int base = p0 + pl;
    if (base < p1) load(base, cur);
    for (; base < p1; base += gstep) {
      const bool more = base + gstep < p1;
      if (more) load(base + gstep, nxt);
#pragma unroll
      for (int u = 0; u < GU; ++u)
        if (base + u * mp.PL < p1) {
          const float4 v = cur[u];
          s[0] += v.x; q[0] += (double)v.x * v.x; s[1] += v.y; q[1] += (double)v.y * v.y;
          s[2] += v.z; q[2] += (double)v.z * v.z; s[3] += v.w; q[3] += (double)v.w * v.w;
        }
      if (more) {
#pragma unroll
        for (int u = 0; u < GU; ++u) cur[u] = nxt[u];
      }
    }
  }
  const int W4 = mp.CT * 4;
  double* shs = sh; double* shq = sh + mp.PL * W4;
#pragma unroll
  for (int e = 0; e < 4; ++e) { shs[pl * W4 + c0 + e] = s[e]; shq[pl * W4 + c0 + e] = q[e]; }
  __syncthreads();
  const int cpg = a.C / a.G;
  for (int g = tid; g < a.G; g += NT) {
    double ts = 0, tq = 0;
    for (int c = g * cpg; c < (g + 1) * cpg; ++c)
      for (int l = 0; l < mp.PL; ++l) { ts += shs[l * W4 + c]; tq += shq[l * W4 + c]; }
    double* o = ws + (((long long)n * mp.nchunks + chunk) * a.G + g) * 2;
    o[0] = ts; o[1] = tq;
  }
}

// Bound of |y| known before y exists, from gamma / beta alone (every block derives the same bits, on every launch: safe under graph
// replay and after a weight update).  Over a group of n values |x - mean| <= sqrt(n - 1) * std (Samuelson) and rstd <= 1 / std, so
// |x_hat| <= sqrt(n - 1) and |gn(x)| <= B = max|gamma| sqrt(n - 1) + max|beta|; |silu(v)| <= max(|v|, 0.2785); dropout scales by its
// exact inverse keep rate.  Rounded up, plus 2^-10 for the fp32 rounding of the statistics and of the SiLU.  Block (0, 0) stores B as
// the output's amax slot; the return value is the convolutions' operand scale for that slot.  Called by all threads of the block.
__device__ float gn_split_scale(const dp_gn_args& a, const Drop& drop, int cpg) {
  __shared__ float red[2][NT / 32];
  float gm = 0.f, bm = 0.f;
  for (int c = threadIdx.x; c < a.C; c += NT) { gm = fmaxf(gm, fabsf(__ldg(a.gamma + c))); bm = fmaxf(bm, fabsf(__ldg(a.beta + c))); }
  gm = warp_max(gm); bm = warp_max(bm);
  if ((threadIdx.x & 31) == 0) { red[0][threadIdx.x >> 5] = gm; red[1][threadIdx.x >> 5] = bm; }
  __syncthreads();
  gm = 0.f; bm = 0.f;
#pragma unroll
  for (int w = 0; w < NT / 32; ++w) { gm = fmaxf(gm, red[0][w]); bm = fmaxf(bm, red[1][w]); }
  const long long n = (long long)cpg * a.HW;
  float B = __fmaf_ru(gm, __fsqrt_ru((float)(n - 1)), bm);
  if (a.silu) B = fmaxf(B, 0.2785f);
  if (drop.on) B = __fmul_ru(B, drop.inv);
  B = __fmul_ru(B, 1.0f + 0x1p-10f);
  const uint32_t bits = __float_as_uint(B);
  if (blockIdx.x == 0 && blockIdx.y == 0 && threadIdx.x == 0) *a.amax_y = bits;
  return scale_up(amax_exponent_bits(bits));
}

// SPLIT: also write the split output (dp_groupnorm_fwd_split).  Its own instantiation, with room for the extra live registers (at 4 blocks per SM it spilled)
template <bool SPLIT>
__global__ void __launch_bounds__(NT, SPLIT ? 3 : 4) gn_apply4_kernel(const dp_gn_args a, const Map mp, const double* __restrict__ fold_ws, __half* __restrict__ ysplit,
                                                             const long long ldys) {
  extern __shared__ float shst[];   // folded finalize: [2][G]
  const int n = blockIdx.y, chunk = blockIdx.x, tid = threadIdx.x;
  const int ct = tid % mp.CT, pl = tid / mp.CT, c0 = ct * 4;
  const float* gmean = a.mean + n * a.G;
  const float* grstd = a.rstd + n * a.G;
  if (fold_ws) { gn_fold_stats(a, mp, fold_ws, n, chunk == 0, shst, shst + a.G); gmean = shst; grstd = shst + a.G; }
  const Drop drop = make_drop(a);
  const int cpg = a.C / a.G;
  float ssplit = 0.f;       // split output: scale of the bound B, the same in every block
  if constexpr (SPLIT) ssplit = gn_split_scale(a, drop, cpg);
  if (c0 >= a.C) return;
  const int p0 = chunk * mp.PPC, p1 = min(a.HW, p0 + mp.PPC);
  float sc[4], shf[4];
#pragma unroll
  for (int e = 0; e < 4; ++e) {
    int c = c0 + e, g = c / cpg;
    float mu = gmean[g], rs = grstd[g], ga = __ldg(a.gamma + c), be = __ldg(a.beta + c);
    sc[e] = rs * ga; shf[e] = be - mu * rs * ga;
  }
  const float* xb = a.x + (long long)n * a.HW * a.ldx + c0;
  float* yb = a.y + (long long)n * a.HW * a.ldy + c0;
  __half* ysb = ysplit + (long long)n * a.HW * 2 * ldys + c0;
  float amax = 0.f;
  float4 cur[GU], nxt[GU];       // software pipeline: see gn_stats4_kernel
  const int gstep = GU * mp.PL;
  auto load = [&](int base, float4 (&buf)[GU]) {
#pragma unroll
    for (int u = 0; u < GU; ++u) { const int px = base + u * mp.PL; if (px < p1) buf[u] = ld4(xb + (long long)px * a.ldx); }
  };
  if (p0 + pl < p1) load(p0 + pl, cur);
  for (int base = p0 + pl; base < p1; base += gstep) {
   const bool more = base + gstep < p1;
   if (more) load(base + gstep, nxt);
#pragma unroll
   for (int u = 0; u < GU; ++u) {
    const int pix = base + u * mp.PL;
    if (pix >= p1) break;
    const float4 v = cur[u];
    float y[4] = {fmaf(v.x, sc[0], shf[0]), fmaf(v.y, sc[1], shf[1]), fmaf(v.z, sc[2], shf[2]), fmaf(v.w, sc[3], shf[3])};
#pragma unroll
    for (int e = 0; e < 4; ++e) {
      if (a.silu) y[e] = y[e] * sigmoidf_fast(y[e]);
    }
    if (drop.on) {
      float k[4];
      keep_scale4(drop, ((uint64_t)n * a.HW + pix) * a.C + c0, k);
#pragma unroll
      for (int e = 0; e < 4; ++e) y[e] *= k[e];
    }
    if (a.y) *reinterpret_cast<float4*>(yb + (long long)pix * a.ldy) = make_float4(y[0], y[1], y[2], y[3]);
    if (a.y_bf16) {   // the next convolution's bf16 operand (c0 % 4 == 0 and ldyb % 8 == 0: 8-byte aligned)
      __nv_bfloat162 lo = __floats2bfloat162_rn(y[0], y[1]), hi = __floats2bfloat162_rn(y[2], y[3]);
      uint2 pk = make_uint2(*reinterpret_cast<uint32_t*>(&lo), *reinterpret_cast<uint32_t*>(&hi));
      *reinterpret_cast<uint2*>(reinterpret_cast<__nv_bfloat16*>(a.y_bf16) + ((long long)n * a.HW + pix) * a.ldyb + c0) = pk;
    }
    if constexpr (SPLIT) {  // the convolutions' hi / lo' operand pair, exactly what their splitter makes of y with the same scale (8-byte aligned)
      uint2 h, l;
      split2(y[0] * ssplit, y[1] * ssplit, h.x, l.x);
      split2(y[2] * ssplit, y[3] * ssplit, h.y, l.y);
      __half* dst = ysb + (long long)pix * 2 * ldys;
      *reinterpret_cast<uint2*>(dst) = h;
      *reinterpret_cast<uint2*>(dst + ldys) = l;
    }
    amax = fmaxf(fmaxf(amax, fmaxf(fabsf(y[0]), fabsf(y[1]))), fmaxf(fabsf(y[2]), fabsf(y[3])));
   }
   if (more) {
#pragma unroll
    for (int u = 0; u < GU; ++u) cur[u] = nxt[u];
   }
  }
  if (a.amax_y && !SPLIT) amax_commit(a.amax_y, amax);
}

__global__ void __launch_bounds__(NT, 4) gn_bwd_partial4_kernel(const dp_gn_args a, const Map mp, float* __restrict__ part) {
  extern __shared__ float shf32[];  // [2][PL][CT*4]
  const int n = blockIdx.y, chunk = blockIdx.x, tid = threadIdx.x;
  const int ct = tid % mp.CT, pl = tid / mp.CT, c0 = ct * 4;
  const int p0 = chunk * mp.PPC, p1 = min(a.HW, p0 + mp.PPC);
  const int cpg = a.C / a.G;
  float mu[4], rs[4], ga[4], be[4], s1[4] = {0, 0, 0, 0}, s2[4] = {0, 0, 0, 0};
  const bool act = c0 < a.C;
#pragma unroll
  for (int e = 0; e < 4; ++e) {
    int c = act ? c0 + e : 0, g = c / cpg;
    mu[e] = a.mean[n * a.G + g]; rs[e] = a.rstd[n * a.G + g]; ga[e] = __ldg(a.gamma + c); be[e] = __ldg(a.beta + c);
  }
  if (act) {
    const float* xb = a.x + (long long)n * a.HW * a.ldx + c0;
    const float* db = a.dy + (long long)n * a.HW * a.lddy + c0;
    const Drop drop = make_drop(a);
    // groups of PU pixels with ALL their loads issued before the first use: the SiLU / dropout branches inside the body are basic-block
    // boundaries the compiler does not move loads across, so a plain (even unrolled) loop keeps one pixel = two 16-byte loads in flight
    // per thread — 24 KB per SM, a quarter of what HBM needs (profiles/r02_experiments.md, section 18).  Same summation order.
    constexpr int PU = 2;
    const int gstep = PU * mp.PL;
    for (int base = p0 + pl; base < p1; base += gstep) {
      float4 xg[PU], dg[PU];
#pragma unroll
      for (int u = 0; u < PU; ++u) {
        const int px = base + u * mp.PL;
        xg[u] = dg[u] = make_float4(0.f, 0.f, 0.f, 0.f);
        if (px < p1) { xg[u] = ld4(xb + (long long)px * a.ldx); dg[u] = ld4(db + (long long)px * a.lddy); }
      }
#pragma unroll
      for (int u = 0; u < PU; ++u) {
        const int pix = base + u * mp.PL;
        if (pix < p1) {
          float xs[4] = {xg[u].x, xg[u].y, xg[u].z, xg[u].w}, ds[4] = {dg[u].x, dg[u].y, dg[u].z, dg[u].w};
          if (drop.on) {
            float k[4];
            keep_scale4(drop, ((uint64_t)n * a.HW + pix) * a.C + c0, k);
#pragma unroll
            for (int e = 0; e < 4; ++e) ds[e] *= k[e];
          }
#pragma unroll
          for (int e = 0; e < 4; ++e) {
            float xh = (xs[e] - mu[e]) * rs[e];
            float g = gn_dy(a, ds[e], fmaf(xh, ga[e], be[e]));
            s1[e] += g; s2[e] += g * xh;
          }
        }
      }
    }
  }
  const int W4 = mp.CT * 4;
  float* sa = shf32; float* sb = shf32 + mp.PL * W4;
#pragma unroll
  for (int e = 0; e < 4; ++e) { sa[pl * W4 + c0 + e] = s1[e]; sb[pl * W4 + c0 + e] = s2[e]; }
  __syncthreads();
  float* o = part + ((long long)n * mp.nchunks + chunk) * 2 * a.C;
  for (int c = tid; c < a.C; c += NT) {
    float t1 = 0.f, t2 = 0.f;
    for (int l = 0; l < mp.PL; ++l) { t1 += sa[l * W4 + c]; t2 += sb[l * W4 + c]; }
    o[c] = t1; o[a.C + c] = t2;
  }
}

__global__ void __launch_bounds__(NT, 4) gn_bwd_apply4_kernel(const dp_gn_args a, const Map mp, const float* part, int nrows, float* fin) {
  extern __shared__ float shfold[];   // folded finalize: [2][C] weighted sums + [G][2] coefficients
  const int n = blockIdx.y, chunk = blockIdx.x, tid = threadIdx.x;
  const int ct = tid % mp.CT, pl = tid / mp.CT, c0 = ct * 4;
  const float* coef = shfold + 2 * a.C;
  gn_bwd_coef(a, nrows, part, fin, n, chunk == 0 && part != fin, shfold, shfold + 2 * a.C);
  if (c0 >= a.C) return;
  const int p0 = chunk * mp.PPC, p1 = min(a.HW, p0 + mp.PPC);
  const int cpg = a.C / a.G;
  float mu[4], rs[4], ga[4], be[4], k1[4], k2[4];
#pragma unroll
  for (int e = 0; e < 4; ++e) {
    int c = c0 + e, g = c / cpg;
    mu[e] = a.mean[n * a.G + g]; rs[e] = a.rstd[n * a.G + g]; ga[e] = __ldg(a.gamma + c); be[e] = __ldg(a.beta + c);
    k1[e] = coef[g * 2]; k2[e] = coef[g * 2 + 1];
  }
  const float* xb = a.x + (long long)n * a.HW * a.ldx + c0;
  const float* db = a.dy + (long long)n * a.HW * a.lddy + c0;
  const Drop drop = make_drop(a);
  float* ob = a.dx + (long long)n * a.HW * a.lddx + c0;
  const float* ab = a.dx_add ? a.dx_add + (long long)n * a.HW * a.ldadd + c0 : nullptr;
  const float* ab2 = a.dx_add2 ? a.dx_add2 + (long long)n * a.HW * a.ldadd2 + c0 : nullptr;
  float amax = 0.f;
  // pairs of pixels with all eight loads (x, dy and the two optional addends) issued before the first use — see gn_bwd_partial4_kernel.
  // dx_add may alias dx: every element is read by the thread that later writes it, and a pair's reads precede the pair's stores
  constexpr int BU = 2;
  const int gstep = BU * mp.PL;
  for (int base = p0 + pl; base < p1; base += gstep) {
    float4 xg[BU], dg[BU], ag[BU], bg[BU];
#pragma unroll
    for (int u = 0; u < BU; ++u) {
      const int px = base + u * mp.PL;
      xg[u] = dg[u] = ag[u] = bg[u] = make_float4(0.f, 0.f, 0.f, 0.f);
      if (px < p1) {
        xg[u] = ld4(xb + (long long)px * a.ldx); dg[u] = ld4(db + (long long)px * a.lddy);
        if (ab) ag[u] = *reinterpret_cast<const float4*>(ab + (long long)px * a.ldadd);
        if (ab2) bg[u] = ld4(ab2 + (long long)px * a.ldadd2);
      }
    }
#pragma unroll
    for (int u = 0; u < BU; ++u) {
      const int pix = base + u * mp.PL;
      if (pix < p1) {
        float xs[4] = {xg[u].x, xg[u].y, xg[u].z, xg[u].w}, ds[4] = {dg[u].x, dg[u].y, dg[u].z, dg[u].w}, d[4];
        if (drop.on) {
          float k[4];
          keep_scale4(drop, ((uint64_t)n * a.HW + pix) * a.C + c0, k);
#pragma unroll
          for (int e = 0; e < 4; ++e) ds[e] *= k[e];
        }
#pragma unroll
        for (int e = 0; e < 4; ++e) {
          float xh = (xs[e] - mu[e]) * rs[e];
          float g = gn_dy(a, ds[e], fmaf(xh, ga[e], be[e]));
          d[e] = rs[e] * (ga[e] * g - k1[e] - xh * k2[e]);
        }
        if (ab) { d[0] += ag[u].x; d[1] += ag[u].y; d[2] += ag[u].z; d[3] += ag[u].w; }
        if (ab2) { d[0] += bg[u].x; d[1] += bg[u].y; d[2] += bg[u].z; d[3] += bg[u].w; }
        *reinterpret_cast<float4*>(ob + (long long)pix * a.lddx) = make_float4(d[0], d[1], d[2], d[3]);
        amax = fmaxf(fmaxf(amax, fmaxf(fabsf(d[0]), fabsf(d[1]))), fmaxf(fabsf(d[2]), fabsf(d[3])));
      }
    }
  }
  if (a.amax_dx) amax_commit(a.amax_dx, amax);
}


static inline bool al16(const void* p, long long ld) { return p == nullptr || ((((uintptr_t)p) & 15) == 0 && (ld % 4) == 0); }

// ------------------------------------------------------------------------------------------------------------
// LayerNorm = GroupNorm with ONE group over the channels of a ONE-pixel "image" (the LDM transformer blocks call it on every token:
// N = tokens).  The chunked kernels above would spend a whole 256-thread block on one token; here a warp owns a row: float4 loads,
// two passes over registers (mean, then centred sum of squares), warp-shuffle reductions.  Rows of up to 4 * 32 * LN_V = 1280 channels.
constexpr int LN_V = 10;
__device__ __forceinline__ float warp_sum_all(float v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  return v;
}
__global__ void __launch_bounds__(256) ln_fwd_kernel(const dp_gn_args a) {
  const int lane = threadIdx.x & 31;
  const long long row = (long long)blockIdx.x * 8 + (threadIdx.x >> 5);
  if (row >= a.N) return;
  const int nv = a.C >> 2;
  const float* xr = a.x + row * a.ldx;
  float4 v[LN_V];
  float s = 0.f;
#pragma unroll
  for (int j = 0; j < LN_V; ++j) {
    const int i = lane + 32 * j;
    v[j] = i < nv ? ld4(xr + 4 * i) : make_float4(0, 0, 0, 0);
    s += (v[j].x + v[j].y) + (v[j].z + v[j].w);
  }
  const float mean = warp_sum_all(s) / (float)a.C;
  float q = 0.f;
#pragma unroll
  for (int j = 0; j < LN_V; ++j)
    if (lane + 32 * j < nv) {
      const float dx = v[j].x - mean, dy = v[j].y - mean, dz = v[j].z - mean, dw = v[j].w - mean;
      q += (dx * dx + dy * dy) + (dz * dz + dw * dw);
    }
  const float rstd = 1.0f / sqrtf(warp_sum_all(q) / (float)a.C + a.eps);
  if (lane == 0) { a.mean[row] = mean; a.rstd[row] = rstd; }
  float* yr = a.y + row * a.ldy;
  float amax = 0.f;
#pragma unroll
  for (int j = 0; j < LN_V; ++j) {
    const int i = lane + 32 * j;
    if (i < nv) {
      const float4 g = ld4(a.gamma + 4 * i), b = ld4(a.beta + 4 * i);
      float4 y;
      y.x = fmaf((v[j].x - mean) * rstd, g.x, b.x); y.y = fmaf((v[j].y - mean) * rstd, g.y, b.y);
      y.z = fmaf((v[j].z - mean) * rstd, g.z, b.z); y.w = fmaf((v[j].w - mean) * rstd, g.w, b.w);
      *reinterpret_cast<float4*>(yr + 4 * i) = y;
      amax = fmaxf(fmaxf(amax, fmaxf(fabsf(y.x), fabsf(y.y))), fmaxf(fabsf(y.z), fabsf(y.w)));
    }
  }
  if (a.amax_y) amax_commit(a.amax_y, amax);
}
// dx = rstd * (g - mean(g) - xhat * mean(g * xhat)) (+ addends), g = dy * gamma
__global__ void __launch_bounds__(256) ln_bwd_dx_kernel(const dp_gn_args a) {
  const int lane = threadIdx.x & 31;
  const long long row = (long long)blockIdx.x * 8 + (threadIdx.x >> 5);
  if (row >= a.N) return;
  const int nv = a.C >> 2;
  const float mean = a.mean[row], rstd = a.rstd[row];
  const float* xr = a.x + row * a.ldx;
  const float* dr = a.dy + row * a.lddy;
  float4 xh[LN_V], g[LN_V];
  float s1 = 0.f, s2 = 0.f;
#pragma unroll
  for (int j = 0; j < LN_V; ++j) {
    const int i = lane + 32 * j;
    if (i < nv) {
      const float4 x = ld4(xr + 4 * i), d = ld4(dr + 4 * i), ga = ld4(a.gamma + 4 * i);
      xh[j] = make_float4((x.x - mean) * rstd, (x.y - mean) * rstd, (x.z - mean) * rstd, (x.w - mean) * rstd);
      g[j] = make_float4(d.x * ga.x, d.y * ga.y, d.z * ga.z, d.w * ga.w);
      s1 += (g[j].x + g[j].y) + (g[j].z + g[j].w);
      s2 += (g[j].x * xh[j].x + g[j].y * xh[j].y) + (g[j].z * xh[j].z + g[j].w * xh[j].w);
    } else { xh[j] = make_float4(0, 0, 0, 0); g[j] = xh[j]; }
  }
  const float m1 = warp_sum_all(s1) / (float)a.C, m2 = warp_sum_all(s2) / (float)a.C;
  float* out = a.dx + row * a.lddx;
  const float* ab = a.dx_add ? a.dx_add + row * a.ldadd : nullptr;
  const float* ab2 = a.dx_add2 ? a.dx_add2 + row * a.ldadd2 : nullptr;
  float amax = 0.f;
#pragma unroll
  for (int j = 0; j < LN_V; ++j) {
    const int i = lane + 32 * j;
    if (i < nv) {
      float4 d = make_float4(rstd * (g[j].x - m1 - xh[j].x * m2), rstd * (g[j].y - m1 - xh[j].y * m2),
                             rstd * (g[j].z - m1 - xh[j].z * m2), rstd * (g[j].w - m1 - xh[j].w * m2));
      if (ab) { const float4 t = *reinterpret_cast<const float4*>(ab + 4 * i); d.x += t.x; d.y += t.y; d.z += t.z; d.w += t.w; }
      if (ab2) { const float4 t = ld4(ab2 + 4 * i); d.x += t.x; d.y += t.y; d.z += t.z; d.w += t.w; }
      *reinterpret_cast<float4*>(out + 4 * i) = d;
      amax = fmaxf(fmaxf(amax, fmaxf(fabsf(d.x), fabsf(d.y))), fmaxf(fabsf(d.z), fabsf(d.w)));
    }
  }
  if (a.amax_dx) amax_commit(a.amax_dx, amax);
}
// dgamma / dbeta partials: block = 32 float4 column groups x 8 row lanes over a chunk of LN_ROWS rows; part[chunk][2][C]
constexpr int LN_ROWS = 256;
__global__ void __launch_bounds__(256) ln_bwd_param_partial_kernel(const dp_gn_args a, float* __restrict__ part) {
  __shared__ float4 sg[8][33], sb[8][33];
  const int cx = threadIdx.x & 31, ly = threadIdx.x >> 5;
  const int i = blockIdx.x * 32 + cx;                 // float4 column group
  const int nv = a.C >> 2;
  const long long r0 = (long long)blockIdx.y * LN_ROWS, r1 = min((long long)a.N, r0 + LN_ROWS);
  float4 tg = make_float4(0, 0, 0, 0), tb = tg;
  if (i < nv)
    for (long long r = r0 + ly; r < r1; r += 8) {
      const float mean = a.mean[r], rstd = a.rstd[r];
      const float4 x = ld4(a.x + r * a.ldx + 4 * i), d = ld4(a.dy + r * a.lddy + 4 * i);
      tg.x += d.x * ((x.x - mean) * rstd); tg.y += d.y * ((x.y - mean) * rstd);
      tg.z += d.z * ((x.z - mean) * rstd); tg.w += d.w * ((x.w - mean) * rstd);
      tb.x += d.x; tb.y += d.y; tb.z += d.z; tb.w += d.w;
    }
  sg[ly][cx] = tg; sb[ly][cx] = tb;
  __syncthreads();
  if (ly == 0 && i < nv) {
    for (int l = 1; l < 8; ++l) {
      tg.x += sg[l][cx].x; tg.y += sg[l][cx].y; tg.z += sg[l][cx].z; tg.w += sg[l][cx].w;
      tb.x += sb[l][cx].x; tb.y += sb[l][cx].y; tb.z += sb[l][cx].z; tb.w += sb[l][cx].w;
    }
    float* o = part + (long long)blockIdx.y * 2 * a.C;
    *reinterpret_cast<float4*>(o + 4 * i) = tg;
    *reinterpret_cast<float4*>(o + a.C + 4 * i) = tb;
  }
}
__global__ void ln_bwd_param_final_kernel(const dp_gn_args a, const float* __restrict__ part, int chunks) {
  const int c = blockIdx.x * blockDim.x + threadIdx.x;
  if (c >= a.C) return;
  double tg = 0, tb = 0;
  for (int ch = 0; ch < chunks; ++ch) { tg += part[(long long)ch * 2 * a.C + c]; tb += part[(long long)ch * 2 * a.C + a.C + c]; }
  if (a.dgamma) a.dgamma[c] += (float)tg;
  if (a.dbeta) a.dbeta[c] += (float)tb;
}
static inline bool ln_fast(const dp_gn_args* a) {     // the row kernels take what the LDM transformer blocks ask for
  return a->HW == 1 && a->G == 1 && a->C % 4 == 0 && a->C <= 4 * 32 * LN_V && !a->silu && a->dropout_p == 0.f && !a->y_bf16;
}


static size_t align256(size_t v) { return (v + 255) & ~(size_t)255; }

}  // namespace

extern "C" size_t dp_groupnorm_workspace_bytes(int32_t N, int32_t HW, int32_t C, int32_t G) {
  if (N <= 0 || HW <= 0 || C <= 0 || G <= 0) return 0;
  Map mp = make_map(HW, C);
  if (C % 4 == 0) { Map m4 = make_map4(HW, C); if (m4.nchunks > mp.nchunks) mp.nchunks = m4.nchunks; }
  size_t fwd = (size_t)N * mp.nchunks * G * 2 * sizeof(double);
  size_t bwd = align256((size_t)N * mp.nchunks * 2 * C * sizeof(float)) + align256((size_t)N * 2 * C * sizeof(float)) +
               align256((size_t)N * G * 2 * sizeof(float));
  return align256(fwd > bwd ? fwd : bwd);
}

static int gn_validate(const dp_gn_args* a) {
  DP_REQUIRE(a && a->x && a->gamma && a->beta && a->mean && a->rstd && a->workspace, DP_ERR_NULL);
  DP_REQUIRE(a->N > 0 && a->HW > 0 && a->C > 0 && a->G > 0 && a->C % a->G == 0, DP_ERR_SHAPE);
  DP_REQUIRE((a->C <= NT * MAXCPT || ln_fast(a)) && a->G <= 1024, DP_ERR_UNSUPPORTED);
  DP_REQUIRE(a->N <= 65535, DP_ERR_SHAPE);
  DP_REQUIRE(a->ldx >= a->C, DP_ERR_SHAPE);
  DP_REQUIRE(a->dropout_p >= 0.f && a->dropout_p < 1.f, DP_ERR_SHAPE);
  return DP_OK;
}

static int gn_fwd(const dp_gn_args* a, void* ysplit, int64_t ldys, dp_stream_t stream) {
  int rc = gn_validate(a);
  if (rc) return rc;
  DP_REQUIRE(a->y || a->y_bf16 || ysplit, DP_ERR_NULL);
  DP_REQUIRE(!a->y || a->ldy >= a->C, DP_ERR_SHAPE);
  DP_REQUIRE(!a->y_bf16 || (a->ldyb >= a->C && a->ldyb % 8 == 0 && (((uintptr_t)a->y_bf16) & 15) == 0), DP_ERR_ALIGN);
  DP_REQUIRE(!ysplit || a->amax_y, DP_ERR_NULL);
  DP_REQUIRE(!ysplit || (ldys >= a->C && ldys % 8 == 0 && (((uintptr_t)ysplit) & 15) == 0), DP_ERR_ALIGN);
  cudaStream_t st = (cudaStream_t)stream;
  const bool v4 = (a->C % 4 == 0) && al16(a->x, a->ldx) && al16(a->y, a->ldy);
  DP_REQUIRE(!ysplit || (v4 && !ln_fast(a)), DP_ERR_UNSUPPORTED);    // the split output is written by the float4 apply kernel only
  if (v4 && a->y && ln_fast(a) && al16(a->gamma, 0) && al16(a->beta, 0)) {     // LayerNorm over tokens: one warp per row
    ln_fwd_kernel<<<(unsigned)((a->N + 7) / 8), 256, 0, st>>>(*a);
    return dp_check_launch();
  }
  Map mp = v4 ? make_map4(a->HW, a->C) : make_map(a->HW, a->C);
  dim3 grid(mp.nchunks, a->N);
  if (v4) {
    gn_stats4_kernel<<<grid, NT, 2 * mp.PL * mp.CT * 4 * sizeof(double), st>>>(*a, mp, (double*)a->workspace);
  } else {
    int slots = (a->C > NT) ? a->C : mp.PL * mp.CT;
    gn_stats_kernel<<<grid, NT, 2 * slots * sizeof(double), st>>>(*a, mp, (double*)a->workspace);
  }
  if ((rc = dp_check_launch())) return rc;
  const bool fold = mp.nchunks <= GN_FOLD_FWD;
  if (!fold) {
    gn_finalize_kernel<<<(a->N * a->G + 7) / 8, 256, 0, st>>>(*a, mp, (const double*)a->workspace);
    if ((rc = dp_check_launch())) return rc;
  }
  const double* fws = fold ? (const double*)a->workspace : nullptr;
  const size_t fsm = fold ? 2 * (size_t)a->G * sizeof(float) : 0;
  if (v4 && ysplit) gn_apply4_kernel<true><<<grid, NT, fsm, st>>>(*a, mp, fws, (__half*)ysplit, ldys);
  else if (v4) gn_apply4_kernel<false><<<grid, NT, fsm, st>>>(*a, mp, fws, nullptr, 0);
  else gn_apply_kernel<<<grid, NT, fsm, st>>>(*a, mp, fws);
  return dp_check_launch();
}

extern "C" int dp_groupnorm_fwd(const dp_gn_args* a, dp_stream_t stream) { return gn_fwd(a, nullptr, 0, stream); }
extern "C" int dp_groupnorm_fwd_split(const dp_gn_args* a, void* y_split, int64_t ldys, dp_stream_t stream) {
  DP_REQUIRE(y_split, DP_ERR_NULL);
  return gn_fwd(a, y_split, ldys, stream);
}

extern "C" int dp_groupnorm_bwd(const dp_gn_args* a, dp_stream_t stream) {
  int rc = gn_validate(a);
  if (rc) return rc;
  DP_REQUIRE(a->dy && a->dx, DP_ERR_NULL);
  DP_REQUIRE(a->lddy >= a->C && a->lddx >= a->C, DP_ERR_SHAPE);
  cudaStream_t st = (cudaStream_t)stream;
  const bool v4 = (a->C % 4 == 0) && al16(a->x, a->ldx) && al16(a->dy, a->lddy) && al16(a->dx, a->lddx) &&
                  al16(a->dx_add, a->ldadd) && al16(a->dx_add2, a->ldadd2);
  DP_REQUIRE(!(a->fin && ln_fast(a)), DP_ERR_UNSUPPORTED);     // the row kernels take dgamma / dbeta from x and dy, not from fin
  if (v4 && ln_fast(a) && al16(a->gamma, 0)) {      // LayerNorm over tokens: row kernel for dx, chunked column sums for dgamma / dbeta
    ln_bwd_dx_kernel<<<(unsigned)((a->N + 7) / 8), 256, 0, st>>>(*a);
    if ((rc = dp_check_launch())) return rc;
    if (a->dgamma || a->dbeta) {
      const int chunks = (a->N + LN_ROWS - 1) / LN_ROWS;       // partials [chunks][2][C] fit the GroupNorm workspace (N * 2 * C floats and more)
      ln_bwd_param_partial_kernel<<<dim3((a->C / 4 + 31) / 32, chunks), 256, 0, st>>>(*a, (float*)a->workspace);
      if ((rc = dp_check_launch())) return rc;
      ln_bwd_param_final_kernel<<<(a->C + 127) / 128, 128, 0, st>>>(*a, (const float*)a->workspace, chunks);
      rc = dp_check_launch();
    }
    return rc;
  }
  Map mp = v4 ? make_map4(a->HW, a->C) : make_map(a->HW, a->C);
  char* ws = (char*)a->workspace;
  float* part = (float*)ws;
  float* fin = (float*)(ws + align256((size_t)a->N * mp.nchunks * 2 * a->C * sizeof(float)));
  if (a->fin) fin = a->fin;      // caller-owned: outlives the shared workspace, dgamma / dbeta are taken later (dp_groupnorm_bwd_param)
  dim3 grid(mp.nchunks, a->N);
  if (v4) gn_bwd_partial4_kernel<<<grid, NT, 2 * mp.PL * mp.CT * 4 * sizeof(float), st>>>(*a, mp, part);
  else gn_bwd_partial_kernel<<<grid, NT, 2 * mp.PL * mp.CT * sizeof(float), st>>>(*a, mp, part);
  if ((rc = dp_check_launch())) return rc;
  const bool fold = mp.nchunks <= GN_FOLD_BWD;
  if (!fold) {
    gn_bwd_reduce_kernel<<<dim3((a->C + 31) / 32, a->N), 1024, 0, st>>>(*a, mp, part, fin);
    if ((rc = dp_check_launch())) return rc;
  }
  const float* src = fold ? part : fin;
  const int nrows = fold ? mp.nchunks : 1;
  const size_t fsm = (2 * (size_t)a->C + 2 * (size_t)a->G) * sizeof(float);
  if (v4) gn_bwd_apply4_kernel<<<grid, NT, fsm, st>>>(*a, mp, src, nrows, fin);
  else gn_bwd_apply_kernel<<<grid, NT, fsm, st>>>(*a, mp, src, nrows, fin);
  if ((rc = dp_check_launch())) return rc;
  if (!a->fin && (a->dgamma || a->dbeta)) {      // after the apply pass: its chunk-0 blocks write fin in the folded form
    gn_bwd_param_kernel<<<(a->C + 31) / 32, 1024, 0, st>>>(*a, fin);
    rc = dp_check_launch();
  }
  return rc;
}

extern "C" int dp_groupnorm_bwd_param(const dp_gn_args* a, dp_stream_t stream) {
  DP_REQUIRE(a && a->fin, DP_ERR_NULL);
  DP_REQUIRE(a->N > 0 && a->C > 0, DP_ERR_SHAPE);
  DP_REQUIRE(!ln_fast(a), DP_ERR_UNSUPPORTED);
  if (!a->dgamma && !a->dbeta) return DP_OK;
  gn_bwd_param_kernel<<<(a->C + 31) / 32, 1024, 0, (cudaStream_t)stream>>>(*a, a->fin);
  return dp_check_launch();
}
