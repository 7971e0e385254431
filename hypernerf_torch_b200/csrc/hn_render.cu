// HBM-bound per-ray stages of the HyperNeRF hot path: stratified sampling, inverse-CDF resampling and
// alpha compositing (forward + reverse).  One warp owns one ray; every lane owns C consecutive samples so
// global loads are contiguous across the warp and scans are lane-local + one shuffle scan.
//
// Reference semantics (cited per kernel): hypernerf/model_utils.py of songrise/HyperNeRF-torch.
#include <stdint.h>
#include "hn_api_internal.h"

namespace hn {

static constexpr int kWarpsPerBlock = 8;
static constexpr unsigned kFull = 0xffffffffu;

// ------------------------------------------------------------------------------------------------
// hn_sample_coarse — model_utils.py:6-41.  z = lower + (upper-lower)*u, each op separately rounded like the
// reference's three torch elementwise kernels; points = o + z*d likewise (no FMA contraction).
// ------------------------------------------------------------------------------------------------
__global__ void sample_coarse_kernel(const float* __restrict__ o, const float* __restrict__ d,
                                     const float* __restrict__ u, const float* __restrict__ lower,
                                     const float* __restrict__ upper, int64_t n, int Nc, float* __restrict__ z,
                                     float* __restrict__ pts) {
  int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  int64_t b = i / Nc;
  int s = (int)(i - b * Nc);
  float lo = lower[s];
  float zz = lo;
  if (u != nullptr) zz = __fadd_rn(lo, __fmul_rn(__fsub_rn(upper[s], lo), u[i]));
  z[i] = zz;
  if (pts != nullptr) {
#pragma unroll
    for (int c = 0; c < 3; ++c) pts[i * 3 + c] = __fadd_rn(o[b * 3 + c], __fmul_rn(zz, d[b * 3 + c]));
  }
}

// Nc % 4 == 0 and 16-byte aligned rows: a thread owns 4 consecutive depths of one ray (same arithmetic; one 16-byte load of
// the draws, one 16-byte store of the depths and three of the 48 contiguous bytes of points instead of 16 scalar accesses)
__global__ void __launch_bounds__(256) sample_coarse_v4_kernel(const float* __restrict__ o, const float* __restrict__ d,
                                                               const float4* __restrict__ u, const float4* __restrict__ lower,
                                                               const float4* __restrict__ upper, int64_t n4, int Nc4,
                                                               float4* __restrict__ z, float4* __restrict__ pts) {
  const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n4) return;
  const int64_t b = i / Nc4;
  const int s = (int)(i - b * Nc4);
  const float4 lo = __ldg(lower + s);
  float zz[4] = {lo.x, lo.y, lo.z, lo.w};
  if (u != nullptr) {
    const float4 up = __ldg(upper + s), uu = __ldg(u + i);
    zz[0] = __fadd_rn(lo.x, __fmul_rn(__fsub_rn(up.x, lo.x), uu.x));
    zz[1] = __fadd_rn(lo.y, __fmul_rn(__fsub_rn(up.y, lo.y), uu.y));
    zz[2] = __fadd_rn(lo.z, __fmul_rn(__fsub_rn(up.z, lo.z), uu.z));
    zz[3] = __fadd_rn(lo.w, __fmul_rn(__fsub_rn(up.w, lo.w), uu.w));
  }
  z[i] = make_float4(zz[0], zz[1], zz[2], zz[3]);
  if (pts != nullptr) {
    const float ox = __ldg(o + b * 3), oy = __ldg(o + b * 3 + 1), oz = __ldg(o + b * 3 + 2);
    const float dx = __ldg(d + b * 3), dy = __ldg(d + b * 3 + 1), dz = __ldg(d + b * 3 + 2);
    float pv[12];
#pragma unroll
    for (int j = 0; j < 4; ++j) {
      pv[3 * j] = __fadd_rn(ox, __fmul_rn(zz[j], dx));
      pv[3 * j + 1] = __fadd_rn(oy, __fmul_rn(zz[j], dy));
      pv[3 * j + 2] = __fadd_rn(oz, __fmul_rn(zz[j], dz));
    }
    pts[i * 3] = make_float4(pv[0], pv[1], pv[2], pv[3]);
    pts[i * 3 + 1] = make_float4(pv[4], pv[5], pv[6], pv[7]);
    pts[i * 3 + 2] = make_float4(pv[8], pv[9], pv[10], pv[11]);
  }
}

// ------------------------------------------------------------------------------------------------
// warp scans
// ------------------------------------------------------------------------------------------------
__device__ __forceinline__ float warp_excl_scan_mul(float v, int lane) {
  // returns product of v over lanes < lane
  float inc = v;
#pragma unroll
  for (int o = 1; o < 32; o <<= 1) {
    float t = __shfl_up_sync(kFull, inc, o);
    if (lane >= o) inc *= t;
  }
  float ex = __shfl_up_sync(kFull, inc, 1);
  return lane == 0 ? 1.f : ex;
}
__device__ __forceinline__ float warp_excl_scan_add(float v, int lane) {
  float inc = v;
#pragma unroll
  for (int o = 1; o < 32; o <<= 1) {
    float t = __shfl_up_sync(kFull, inc, o);
    if (lane >= o) inc += t;
  }
  float ex = __shfl_up_sync(kFull, inc, 1);
  return lane == 0 ? 0.f : ex;
}
__device__ __forceinline__ float warp_excl_rscan_add(float v, int lane) {
  // sum of v over lanes > lane
  float inc = v;
#pragma unroll
  for (int o = 1; o < 32; o <<= 1) {
    float t = __shfl_down_sync(kFull, inc, o);
    if (lane + o < 32) inc += t;
  }
  float ex = __shfl_down_sync(kFull, inc, 1);
  return lane == 31 ? 0.f : ex;
}
__device__ __forceinline__ float warp_sum(float v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(kFull, v, o);
  return v;
}
__device__ __forceinline__ double warp_sum_d(double v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(kFull, v, o);
  return v;
}

// contiguous per-lane loads of CNT floats with the widest aligned vector
template <int CNT>
__device__ __forceinline__ void load_run(const float* __restrict__ p, float* out) {
  if constexpr (CNT % 4 == 0) {
#pragma unroll
    for (int i = 0; i < CNT / 4; ++i) {
      float4 v = __ldg(reinterpret_cast<const float4*>(p) + i);
      out[4 * i] = v.x; out[4 * i + 1] = v.y; out[4 * i + 2] = v.z; out[4 * i + 3] = v.w;
    }
  } else if constexpr (CNT % 2 == 0) {
#pragma unroll
    for (int i = 0; i < CNT / 2; ++i) {
      float2 v = __ldg(reinterpret_cast<const float2*>(p) + i);
      out[2 * i] = v.x; out[2 * i + 1] = v.y;
    }
  } else {
#pragma unroll
    for (int i = 0; i < CNT; ++i) out[i] = __ldg(p + i);
  }
}
template <int CNT>
__device__ __forceinline__ void store_run(float* __restrict__ p, const float* v) {
  if constexpr (CNT % 4 == 0) {
#pragma unroll
    for (int i = 0; i < CNT / 4; ++i)
      reinterpret_cast<float4*>(p)[i] = make_float4(v[4 * i], v[4 * i + 1], v[4 * i + 2], v[4 * i + 3]);
  } else if constexpr (CNT % 2 == 0) {
#pragma unroll
    for (int i = 0; i < CNT / 2; ++i) reinterpret_cast<float2*>(p)[i] = make_float2(v[2 * i], v[2 * i + 1]);
  } else {
#pragma unroll
    for (int i = 0; i < CNT; ++i) p[i] = v[i];
  }
}

// Per-lane view of one ray's samples.  EXACT: S == 32*C (vector loads); otherwise guarded scalar loads.
template <int C, bool EXACT>
struct RayLane {
  float sigma[C], z[C], alpha[C], T[C], w[C], dist[C];
  int base;  // first sample index of this lane

  __device__ __forceinline__ void load(const float* __restrict__ sg, const float* __restrict__ zz, int64_t ray,
                                       int S, int lane) {
    base = lane * C;
    const float* ps = sg + ray * S + base;
    const float* pz = zz + ray * S + base;
    if constexpr (EXACT) {
      load_run<C>(ps, sigma);
      load_run<C>(pz, z);
    } else {
#pragma unroll
      for (int j = 0; j < C; ++j) {
        bool ok = base + j < S;
        sigma[j] = ok ? __ldg(ps + j) : 0.f;
        z[j] = ok ? __ldg(pz + j) : 0.f;
      }
    }
  }
  // alpha, transmittance, weights (model_utils.py:70-87)
  __device__ __forceinline__ void composite(int S, int lane, float dnorm, float eps, float last_delta) {
    float znext = __shfl_down_sync(kFull, z[0], 1);
    float p[C];
    float run = 1.f;
#pragma unroll
    for (int j = 0; j < C; ++j) {
      int s = base + j;
      float zn = (j + 1 < C) ? z[j + 1] : znext;
      float dl = (s == S - 1) ? last_delta : (zn - z[j]);
      dist[j] = dl * dnorm;
      float a = 1.f - expf(-sigma[j] * dist[j]);
      if (s >= S) a = 0.f;
      alpha[j] = a;
      p[j] = (s < S) ? (1.f - a + eps) : 1.f;
      T[j] = run;  // lane-local exclusive product
      run *= p[j];
    }
    float pre = warp_excl_scan_mul(run, lane);
#pragma unroll
    for (int j = 0; j < C; ++j) {
      T[j] *= pre;
      w[j] = alpha[j] * T[j];
    }
  }
};

// ------------------------------------------------------------------------------------------------
// hn_composite_fwd — model_utils.py:43-107 + compute_depth_index/compute_depth_map (:319-362)
// ------------------------------------------------------------------------------------------------
template <int C, bool EXACT>
__global__ void __launch_bounds__(kWarpsPerBlock * 32)
composite_fwd_kernel(const float* __restrict__ sigma, const float* __restrict__ rgb, const float* __restrict__ z,
                     const float* __restrict__ dirs, int64_t B, int S, int flags, float eps, float last_delta,
                     float* __restrict__ out_rgb, float* __restrict__ depth, float* __restrict__ med_depth,
                     float* __restrict__ acc, float* __restrict__ weights, int64_t* __restrict__ med_idx) {
  const int lane = threadIdx.x & 31;
  const int64_t ray = (int64_t)blockIdx.x * kWarpsPerBlock + (threadIdx.x >> 5);
  if (ray >= B) return;
  RayLane<C, EXACT> r;
  r.load(sigma, z, ray, S, lane);
  float dx = __ldg(dirs + ray * 3), dy = __ldg(dirs + ray * 3 + 1), dz = __ldg(dirs + ray * 3 + 2);
  float dnorm = sqrtf(dx * dx + dy * dy + dz * dz);
  r.composite(S, lane, dnorm, eps, last_delta);

  float col[3 * C];
  const float* pc = rgb + (ray * S + r.base) * 3;
  if constexpr (EXACT) {
    load_run<3 * C>(pc, col);
  } else {
#pragma unroll
    for (int j = 0; j < 3 * C; ++j) col[j] = (r.base + j / 3 < S) ? __ldg(pc + j) : 0.f;
  }
  float sr = 0.f, sg = 0.f, sb = 0.f, sd = 0.f, sa = 0.f, sall = 0.f, cs = 0.f;
#pragma unroll
  for (int j = 0; j < C; ++j) {
    float w = r.w[j];
    sr += w * col[3 * j];
    sg += w * col[3 * j + 1];
    sb += w * col[3 * j + 2];
    sd += w * r.z[j];
    sall += w;
    if ((flags & HN_COMP_ACC_ALL) || (r.base + j < S - 1)) sa += w;
    cs += w;
  }
  // median depth: first sample whose inclusive cumsum(w) >= 0.5
  float pre = warp_excl_scan_add(cs, lane);
  int first = -1;
  float run = pre;
#pragma unroll
  for (int j = 0; j < C; ++j) {
    run += r.w[j];
    if (first < 0 && r.base + j < S && run >= 0.5f) first = j;
  }
  unsigned hit = __ballot_sync(kFull, first >= 0);
  int src = hit ? (__ffs(hit) - 1) : 0;
  float zsel = 0.f;
#pragma unroll
  for (int j = 0; j < C; ++j)
    if (j == first) zsel = r.z[j];
  float mz = __shfl_sync(kFull, zsel, src);
  int mj = __shfl_sync(kFull, first, src);
  sr = warp_sum(sr); sg = warp_sum(sg); sb = warp_sum(sb);
  sd = warp_sum(sd); sa = warp_sum(sa); sall = warp_sum(sall);

  if (weights != nullptr) {
    float* pw = weights + ray * S + r.base;
    if constexpr (EXACT) {
      store_run<C>(pw, r.w);
    } else {
#pragma unroll
      for (int j = 0; j < C; ++j)
        if (r.base + j < S) pw[j] = r.w[j];
    }
  }
  if (lane == 0) {
    if (flags & HN_COMP_WHITE_BKGD) {
      float bg = 1.f - sall;
      sr += bg; sg += bg; sb += bg;
    }
    out_rgb[ray * 3] = sr; out_rgb[ray * 3 + 1] = sg; out_rgb[ray * 3 + 2] = sb;
    depth[ray] = sd;
    acc[ray] = sa;
    if (med_depth != nullptr) med_depth[ray] = hit ? mz : 0.f;
    if (med_idx != nullptr) med_idx[ray] = hit ? (int64_t)(src * C + mj) : 0;
  }
}

// S == 64 (the coarse level): two rays per warp, 16 lanes x 4 consecutive samples each.  The scans, reductions and the
// median search are a fixed per-WARP cost; with one ray per warp they, not the 1.6 KB of loads, bound the S = 64 case
// (issue-active 76 %, 0.68 of the HBM peak against 0.98 at S = 128).  Same formulas as RayLane::composite above.
__global__ void __launch_bounds__(kWarpsPerBlock * 32)
composite_fwd_s64_kernel(const float* __restrict__ sigma, const float* __restrict__ rgb, const float* __restrict__ z,
                         const float* __restrict__ dirs, int64_t B, int flags, float eps, float last_delta,
                         float* __restrict__ out_rgb, float* __restrict__ depth, float* __restrict__ med_depth,
                         float* __restrict__ acc, float* __restrict__ weights, int64_t* __restrict__ med_idx) {
  constexpr int C = 4, S = 64, W = 16;
  const int lane = threadIdx.x & 31, sub = lane & (W - 1), half = lane >> 4;
  const int64_t ray_w = ((int64_t)blockIdx.x * kWarpsPerBlock + (threadIdx.x >> 5)) * 2;
  if (ray_w >= B) return;
  const bool live = ray_w + half < B;           // odd B: the upper half of the last warp idles along (shuffles need it)
  const int64_t ray = live ? ray_w + half : ray_w;
  const int base = sub * C;
  float sg[C], zz[C], w[C];
  load_run<C>(sigma + ray * S + base, sg);
  load_run<C>(z + ray * S + base, zz);
  const float dx = __ldg(dirs + ray * 3), dy = __ldg(dirs + ray * 3 + 1), dz = __ldg(dirs + ray * 3 + 2);
  const float dnorm = sqrtf(dx * dx + dy * dy + dz * dz);
  const float znext = __shfl_down_sync(kFull, zz[0], 1, W);
  float alpha[C], T[C];
  float run = 1.f;
#pragma unroll
  for (int j = 0; j < C; ++j) {
    const int s = base + j;
    const float zn = (j + 1 < C) ? zz[j + 1] : znext;
    const float dl = (s == S - 1) ? last_delta : (zn - zz[j]);
    const float a = 1.f - expf(-sg[j] * (dl * dnorm));
    alpha[j] = a;
    T[j] = run;
    run *= 1.f - a + eps;
  }
  float inc = run;                               // exclusive product over the lanes of this half
#pragma unroll
  for (int o = 1; o < W; o <<= 1) {
    const float t = __shfl_up_sync(kFull, inc, o, W);
    if (sub >= o) inc *= t;
  }
  float pre = __shfl_up_sync(kFull, inc, 1, W);
  if (sub == 0) pre = 1.f;
  float col[3 * C];
  load_run<3 * C>(rgb + (ray * S + base) * 3, col);
  float sr = 0.f, sgn = 0.f, sb = 0.f, sd = 0.f, sa = 0.f, sall = 0.f, cs = 0.f;
#pragma unroll
  for (int j = 0; j < C; ++j) {
    w[j] = alpha[j] * (T[j] * pre);
    sr += w[j] * col[3 * j];
    sgn += w[j] * col[3 * j + 1];
    sb += w[j] * col[3 * j + 2];
    sd += w[j] * zz[j];
    sall += w[j];
    if ((flags & HN_COMP_ACC_ALL) || (base + j < S - 1)) sa += w[j];
    cs += w[j];
  }
  // median depth: first sample whose inclusive cumsum(w) >= 0.5
  float cinc = cs;
#pragma unroll
  for (int o = 1; o < W; o <<= 1) {
    const float t = __shfl_up_sync(kFull, cinc, o, W);
    if (sub >= o) cinc += t;
  }
  float runw = cinc - cs;
  int first = -1;
#pragma unroll
  for (int j = 0; j < C; ++j) {
    runw += w[j];
    if (first < 0 && runw >= 0.5f) first = j;
  }
  const unsigned hit = (__ballot_sync(kFull, first >= 0) >> (W * half)) & 0xffffu;
  const int src = hit ? (__ffs(hit) - 1) : 0;
  float zsel = 0.f;
#pragma unroll
  for (int j = 0; j < C; ++j)
    if (j == first) zsel = zz[j];
  const float mz = __shfl_sync(kFull, zsel, src, W);
  const int mj = __shfl_sync(kFull, first, src, W);
#pragma unroll
  for (int o = W / 2; o > 0; o >>= 1) {
    sr += __shfl_xor_sync(kFull, sr, o); sgn += __shfl_xor_sync(kFull, sgn, o); sb += __shfl_xor_sync(kFull, sb, o);
    sd += __shfl_xor_sync(kFull, sd, o); sa += __shfl_xor_sync(kFull, sa, o); sall += __shfl_xor_sync(kFull, sall, o);
  }
  if (!live) return;
  if (weights != nullptr) store_run<C>(weights + ray * S + base, w);
  if (sub == 0) {
    if (flags & HN_COMP_WHITE_BKGD) {
      const float bg = 1.f - sall;
      sr += bg; sgn += bg; sb += bg;
    }
    out_rgb[ray * 3] = sr; out_rgb[ray * 3 + 1] = sgn; out_rgb[ray * 3 + 2] = sb;
    depth[ray] = sd;
    acc[ray] = sa;
    if (med_depth != nullptr) med_depth[ray] = hit ? mz : 0.f;
    if (med_idx != nullptr) med_idx[ray] = hit ? (int64_t)(src * C + mj) : 0;
  }
}

// ------------------------------------------------------------------------------------------------
// hn_composite_bwd — reverse of the above.
//   G_i = g_rgb . c_i + g_depth z_i + g_acc [i counted] + g_w_i (+ white bkgd: -sum(g_rgb))
//   dL/dalpha_i = G_i T_i - (sum_{k>i} G_k w_k) / (1 - alpha_i + eps)
//   dL/dsigma_i = dL/dalpha_i * dist_i * (1 - alpha_i) ;  dL/dc_i = w_i g_rgb
// ------------------------------------------------------------------------------------------------
template <int C, bool EXACT>
__global__ void __launch_bounds__(kWarpsPerBlock * 32, C <= 4 ? 6 : 1)
composite_bwd_kernel(const float* __restrict__ sigma, const float* __restrict__ rgb, const float* __restrict__ z,
                     const float* __restrict__ dirs, int64_t B, int S, int flags, float eps, float last_delta,
                     const float* __restrict__ g_out_rgb, const float* __restrict__ g_depth,
                     const float* __restrict__ g_acc, const float* __restrict__ g_weights,
                     float* __restrict__ g_sigma, float* __restrict__ g_rgb) {
  const int lane = threadIdx.x & 31;
  const int64_t ray = (int64_t)blockIdx.x * kWarpsPerBlock + (threadIdx.x >> 5);
  if (ray >= B) return;
  RayLane<C, EXACT> r;
  r.load(sigma, z, ray, S, lane);
  float dx = __ldg(dirs + ray * 3), dy = __ldg(dirs + ray * 3 + 1), dz = __ldg(dirs + ray * 3 + 2);
  float dnorm = sqrtf(dx * dx + dy * dy + dz * dz);
  r.composite(S, lane, dnorm, eps, last_delta);

  float col[3 * C];
  const float* pc = rgb + (ray * S + r.base) * 3;
  if constexpr (EXACT) {
    load_run<3 * C>(pc, col);
  } else {
#pragma unroll
    for (int j = 0; j < 3 * C; ++j) col[j] = (r.base + j / 3 < S) ? __ldg(pc + j) : 0.f;
  }
  float gr = 0.f, gg = 0.f, gb = 0.f;
  if (g_out_rgb != nullptr) {
    gr = __ldg(g_out_rgb + ray * 3); gg = __ldg(g_out_rgb + ray * 3 + 1); gb = __ldg(g_out_rgb + ray * 3 + 2);
  }
  float gd = g_depth ? __ldg(g_depth + ray) : 0.f;
  float ga = g_acc ? __ldg(g_acc + ray) : 0.f;
  float gbg = (flags & HN_COMP_WHITE_BKGD) ? -(gr + gg + gb) : 0.f;
  float gw[C];
  if (g_weights != nullptr) {
    const float* pg = g_weights + ray * S + r.base;
    if constexpr (EXACT) {
      load_run<C>(pg, gw);
    } else {
#pragma unroll
      for (int j = 0; j < C; ++j) gw[j] = (r.base + j < S) ? __ldg(pg + j) : 0.f;
    }
  } else {
#pragma unroll
    for (int j = 0; j < C; ++j) gw[j] = 0.f;
  }
  float G[C], Gw[C];
  float tot = 0.f;
#pragma unroll
  for (int j = 0; j < C; ++j) {
    int s = r.base + j;
    float g = gr * col[3 * j] + gg * col[3 * j + 1] + gb * col[3 * j + 2] + gd * r.z[j] + gw[j] + gbg;
    if ((flags & HN_COMP_ACC_ALL) || s < S - 1) g += ga;
    if (s >= S) g = 0.f;
    G[j] = g;
    Gw[j] = g * r.w[j];
    tot += Gw[j];
  }
  float suf = warp_excl_rscan_add(tot, lane);  // sum over later lanes
  float gs[C], gc[3 * C];
#pragma unroll
  for (int j = C - 1; j >= 0; --j) {
    float p = 1.f - r.alpha[j] + eps;
    float dalpha = G[j] * r.T[j] - suf / p;
    gs[j] = dalpha * r.dist[j] * (1.f - r.alpha[j]);
    suf += Gw[j];
    gc[3 * j] = r.w[j] * gr; gc[3 * j + 1] = r.w[j] * gg; gc[3 * j + 2] = r.w[j] * gb;
  }
  float* ps = g_sigma + ray * S + r.base;
  float* pr = g_rgb + (ray * S + r.base) * 3;
  if constexpr (EXACT) {
    store_run<C>(ps, gs);
    store_run<3 * C>(pr, gc);
  } else {
#pragma unroll
    for (int j = 0; j < C; ++j)
      if (r.base + j < S) {
        ps[j] = gs[j];
        pr[3 * j] = gc[3 * j]; pr[3 * j + 1] = gc[3 * j + 1]; pr[3 * j + 2] = gc[3 * j + 2];
      }
  }
}

// S == 64: two rays per warp (16 lanes x 4 consecutive samples), like composite_fwd_s64_kernel; 16-byte loads / stores.
__global__ void __launch_bounds__(kWarpsPerBlock * 32)
composite_bwd_s64_kernel(const float* __restrict__ sigma, const float* __restrict__ rgb, const float* __restrict__ z,
                         const float* __restrict__ dirs, int64_t B, int flags, float eps, float last_delta,
                         const float* __restrict__ g_out_rgb, const float* __restrict__ g_depth,
                         const float* __restrict__ g_acc, const float* __restrict__ g_weights,
                         float* __restrict__ g_sigma, float* __restrict__ g_rgb) {
  constexpr int C = 4, S = 64, W = 16;
  const int lane = threadIdx.x & 31, sub = lane & (W - 1), half = lane >> 4;
  const int64_t ray_w = ((int64_t)blockIdx.x * kWarpsPerBlock + (threadIdx.x >> 5)) * 2;
  if (ray_w >= B) return;
  const bool live = ray_w + half < B;
  const int64_t ray = live ? ray_w + half : ray_w;
  const int base = sub * C;
  float sg[C], zz[C];
  load_run<C>(sigma + ray * S + base, sg);
  load_run<C>(z + ray * S + base, zz);
  const float dx = __ldg(dirs + ray * 3), dy = __ldg(dirs + ray * 3 + 1), dz = __ldg(dirs + ray * 3 + 2);
  const float dnorm = sqrtf(dx * dx + dy * dy + dz * dz);
  const float znext = __shfl_down_sync(kFull, zz[0], 1, W);
  float alpha[C], T[C], dist[C];
  float run = 1.f;
#pragma unroll
  for (int j = 0; j < C; ++j) {
    const int s = base + j;
    const float zn = (j + 1 < C) ? zz[j + 1] : znext;
    const float dl = (s == S - 1) ? last_delta : (zn - zz[j]);
    dist[j] = dl * dnorm;
    const float a = 1.f - expf(-sg[j] * dist[j]);
    alpha[j] = a;
    T[j] = run;
    run *= 1.f - a + eps;
  }
  float inc = run;                               // exclusive product over the lanes of this half
#pragma unroll
  for (int o = 1; o < W; o <<= 1) {
    const float t = __shfl_up_sync(kFull, inc, o, W);
    if (sub >= o) inc *= t;
  }
  float pre = __shfl_up_sync(kFull, inc, 1, W);
  if (sub == 0) pre = 1.f;
  float col[3 * C];
  load_run<3 * C>(rgb + (ray * S + base) * 3, col);
  float gr = 0.f, gg = 0.f, gb = 0.f;
  if (g_out_rgb != nullptr) {
    gr = __ldg(g_out_rgb + ray * 3); gg = __ldg(g_out_rgb + ray * 3 + 1); gb = __ldg(g_out_rgb + ray * 3 + 2);
  }
  const float gd = g_depth ? __ldg(g_depth + ray) : 0.f;
  const float ga = g_acc ? __ldg(g_acc + ray) : 0.f;
  const float gbg = (flags & HN_COMP_WHITE_BKGD) ? -(gr + gg + gb) : 0.f;
  float gw[C];
  if (g_weights != nullptr) {
    load_run<C>(g_weights + ray * S + base, gw);
  } else {
#pragma unroll
    for (int j = 0; j < C; ++j) gw[j] = 0.f;
  }
  float w[C], G[C], Gw[C];
  float tot = 0.f;
#pragma unroll
  for (int j = 0; j < C; ++j) {
    T[j] *= pre;
    w[j] = alpha[j] * T[j];
    float g = gr * col[3 * j] + gg * col[3 * j + 1] + gb * col[3 * j + 2] + gd * zz[j] + gw[j] + gbg;
    if ((flags & HN_COMP_ACC_ALL) || base + j < S - 1) g += ga;
    G[j] = g;
    Gw[j] = g * w[j];
    tot += Gw[j];
  }
  float rinc = tot;                              // sum over the later lanes of this half
#pragma unroll
  for (int o = 1; o < W; o <<= 1) {
    const float t = __shfl_down_sync(kFull, rinc, o, W);
    if (sub + o < W) rinc += t;
  }
  float suf = __shfl_down_sync(kFull, rinc, 1, W);
  if (sub == W - 1) suf = 0.f;
  float gs[C], gc[3 * C];
#pragma unroll
  for (int j = C - 1; j >= 0; --j) {
    const float p = 1.f - alpha[j] + eps;
    const float dalpha = G[j] * T[j] - suf / p;
    gs[j] = dalpha * dist[j] * (1.f - alpha[j]);
    suf += Gw[j];
    gc[3 * j] = w[j] * gr; gc[3 * j + 1] = w[j] * gg; gc[3 * j + 2] = w[j] * gb;
  }
  if (!live) return;
  store_run<C>(g_sigma + ray * S + base, gs);
  store_run<3 * C>(g_rgb + (ray * S + base) * 3, gc);
}

// ------------------------------------------------------------------------------------------------
// hn_sample_pdf — model_utils.py:160-232 (+ the slicing at models.py:752-755).
// Arithmetic contract (DESIGN.md "resampling"): w' = fl32(w + 1e-5); S = fl32(sum w') and
// cdf_j = fl32(sum_{k<=j} pdf_k) with the sums carried in fp64 — exact for these magnitudes, hence
// independent of summation order, and identical to torch.cumsum on CPU; every other op is a single
// round-to-nearest fp32 operation (no FMA contraction), like the reference's separate torch kernels.
// ------------------------------------------------------------------------------------------------
static constexpr int kPdfMaxN = 512;  // Nc + Nf padded to a power of two must fit

__device__ __forceinline__ void bitonic_sort_warp(float* a, int n2, int lane) {
  for (int k = 2; k <= n2; k <<= 1) {
    for (int j = k >> 1; j > 0; j >>= 1) {
      for (int i = lane; i < n2; i += 32) {
        int ixj = i ^ j;
        if (ixj > i) {
          float x = a[i], y = a[ixj];
          bool up = (i & k) == 0;
          if ((x > y) == up) { a[i] = y; a[ixj] = x; }
        }
      }
      __syncwarp();
    }
  }
}

// The same network on registers: element e = r * 32 + lane lives in v[r] of its lane; partners closer than 32 are reached
// with a shuffle, the others are another register of the same lane.  n = 32 R elements, ascending.
template <int R>
__device__ __forceinline__ void bitonic_sort_regs(float* a, int lane) {
  float v[R];
#pragma unroll
  for (int r = 0; r < R; ++r) v[r] = a[r * 32 + lane];
#pragma unroll
  for (int k = 2; k <= 32 * R; k <<= 1) {
#pragma unroll
    for (int j = k >> 1; j > 0; j >>= 1) {
      if (j >= 32) {
#pragma unroll
        for (int r = 0; r < R; ++r) {
          const int q = r ^ (j >> 5);
          if (q > r) {
            const bool up = (((r * 32) & k) == 0);   // lane bits do not reach k when k > 32
            const float lo = fminf(v[r], v[q]), hi = fmaxf(v[r], v[q]);
            v[r] = up ? lo : hi; v[q] = up ? hi : lo;
          }
        }
      } else {
#pragma unroll
        for (int r = 0; r < R; ++r) {
          const int e = r * 32 + lane;
          const float other = __shfl_xor_sync(kFull, v[r], j);
          const bool up = (e & k) == 0;
          const bool lower = (lane & j) == 0;        // this lane holds the smaller index of the pair
          v[r] = (lower == up) ? fminf(v[r], other) : fmaxf(v[r], other);
        }
      }
    }
  }
#pragma unroll
  for (int r = 0; r < R; ++r) a[r * 32 + lane] = v[r];
  __syncwarp();
}
// n2 a power of two; below 32 or above 512 the shared-memory network
__device__ __forceinline__ void sort_warp(float* a, int n2, int lane) {
  switch (n2) {
    case 32: bitonic_sort_regs<1>(a, lane); break;
    case 64: bitonic_sort_regs<2>(a, lane); break;
    case 128: bitonic_sort_regs<4>(a, lane); break;
    case 256: bitonic_sort_regs<8>(a, lane); break;
    default: bitonic_sort_warp(a, n2, lane); break;
  }
}

__global__ void __launch_bounds__(4 * 32)
sample_pdf_kernel(const float* __restrict__ zc, const float* __restrict__ bins_in, const float* __restrict__ wc,
                  int64_t w_stride, const float* __restrict__ u, const float* __restrict__ o,
                  const float* __restrict__ d, int64_t B, int Nc, int nb, int Nf, int n2c, int n2, float* __restrict__ zf,
                  float* __restrict__ pts, int32_t* __restrict__ bin_idx, int32_t* __restrict__ pos_c,
                  int32_t* __restrict__ pos_n) {
  extern __shared__ float sm[];
  const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
  const int64_t ray = (int64_t)blockIdx.x * 4 + wid;
  if (ray >= B) return;
  // per warp: bins[nb+1] | cdf[nb+1] | srt[n2c] coarse depths | smp[n2] new samples (both padded to powers of two)
  //           | merged[Nc + Nf]
  float* bins = sm + (size_t)wid * (2 * (nb + 1) + n2c + n2 + Nc + Nf);
  float* cdf = bins + nb + 1;
  float* srt = cdf + nb + 1;
  float* smp = srt + n2c;
  float* merged = smp + n2;
  const float* zr = zc + ray * Nc;
  const float* wr = wc + ray * w_stride - 1;  // wr[1 + i] = weight of bin i
  const float eps = 1e-5f;

  for (int i = lane; i < Nc; i += 32) srt[i] = __ldg(zr + i);
  __syncwarp();
  if (bins_in != nullptr) {
    for (int i = lane; i < nb + 1; i += 32) bins[i] = __ldg(bins_in + ray * (nb + 1) + i);
  } else {
    for (int i = lane; i < nb + 1; i += 32) bins[i] = __fmul_rn(0.5f, __fadd_rn(srt[i + 1], srt[i]));
  }
  // sum of w' in fp64 (exact)
  double part = 0.0;
  for (int i = lane; i < nb; i += 32) part += (double)__fadd_rn(__ldg(wr + 1 + i), eps);
  float Ssum = (float)warp_sum_d(part);
  // inclusive prefix of pdf in fp64: lane owns a contiguous run of bins
  const int per = (nb + 31) / 32;
  const int b0 = lane * per;
  double loc = 0.0;
  for (int j = 0; j < per; ++j) {
    int i = b0 + j;
    if (i < nb) loc += (double)__fdiv_rn(__fadd_rn(__ldg(wr + 1 + i), eps), Ssum);
  }
  double inc = loc;
#pragma unroll
  for (int off = 1; off < 32; off <<= 1) {
    double t = __shfl_up_sync(kFull, inc, off);
    if (lane >= off) inc += t;
  }
  double run = inc - loc;  // exclusive prefix of this lane
  if (lane == 0) cdf[0] = 0.f;
  for (int j = 0; j < per; ++j) {
    int i = b0 + j;
    if (i < nb) {
      run += (double)__fdiv_rn(__fadd_rn(__ldg(wr + 1 + i), eps), Ssum);
      cdf[i + 1] = (float)run;
    }
  }
  __syncwarp();
  const int ncdf = nb + 1;
  for (int i = lane; i < Nf; i += 32) {
    float uu = __ldg(u + ray * Nf + i);
    // searchsorted(cdf, u, right=True): number of entries <= u
    int lo = 0, hi = ncdf;
    while (lo < hi) {
      int mid = (lo + hi) >> 1;
      if (cdf[mid] <= uu) lo = mid + 1; else hi = mid;
    }
    int inds = lo;
    int below = max(inds - 1, 0), above = min(inds, nb);
    float c0 = cdf[below], c1 = cdf[above];
    float g0 = bins[below], g1 = bins[above];
    float denom = __fsub_rn(c1, c0);
    if (denom < eps) denom = 1.f;
    float t = __fdiv_rn(__fsub_rn(uu, c0), denom);
    smp[i] = __fadd_rn(g0, __fmul_rn(t, __fsub_rn(g1, g0)));
    if (bin_idx != nullptr) bin_idx[ray * Nf + i] = inds;
  }
  __syncwarp();
  // torch.sort(cat([z_vals, z_samples])) (model_utils.py:227) as sort(new samples) + merge with the sorted coarse depths:
  // same multiset in ascending order, hence the same values.  The inverse CDF is monotone in u, so deterministic
  // (linspace) draws arrive sorted and skip the sort.
  bool ordered = true;
  for (int i = lane; i < Nf; i += 32) ordered &= (i == 0) || (smp[i - 1] <= smp[i]);
  if (!__all_sync(kFull, ordered)) {
    for (int i = Nf + lane; i < n2; i += 32) smp[i] = __int_as_float(0x7f800000);
    __syncwarp();
    sort_warp(smp, n2, lane);
  }
  // the coarse depths of sample_along_rays are ascending; any other caller's are sorted here (the bins above were
  // formed from the original order, as the reference does)
  ordered = true;
  for (int i = lane; i < Nc; i += 32) ordered &= (i == 0) || (srt[i - 1] <= srt[i]);
  if (!__all_sync(kFull, ordered)) {
    for (int i = Nc + lane; i < n2c; i += 32) srt[i] = __int_as_float(0x7f800000);
    __syncwarp();
    sort_warp(srt, n2c, lane);
  }
  // ranks: a coarse depth goes after the new samples strictly below it, a new sample after the coarse depths <= it
  for (int i = lane; i < Nc; i += 32) {
    const float v = srt[i];
    int lo = 0, hi = Nf;
    while (lo < hi) { int mid = (lo + hi) >> 1; if (smp[mid] < v) lo = mid + 1; else hi = mid; }
    merged[i + lo] = v;
    if (pos_c != nullptr) pos_c[ray * Nc + i] = i + lo;
  }
  for (int i = lane; i < Nf; i += 32) {
    const float v = smp[i];
    int lo = 0, hi = Nc;
    while (lo < hi) { int mid = (lo + hi) >> 1; if (srt[mid] <= v) lo = mid + 1; else hi = mid; }
    merged[i + lo] = v;
    if (pos_n != nullptr) pos_n[ray * Nf + i] = i + lo;
  }
  __syncwarp();
  srt = merged;
  const int S = Nc + Nf;
  float ox = 0.f, oy = 0.f, oz = 0.f, dx = 0.f, dy = 0.f, dz = 0.f;
  if (pts != nullptr) {
    ox = __ldg(o + ray * 3); oy = __ldg(o + ray * 3 + 1); oz = __ldg(o + ray * 3 + 2);
    dx = __ldg(d + ray * 3); dy = __ldg(d + ray * 3 + 1); dz = __ldg(d + ray * 3 + 2);
  }
  for (int i = lane; i < S; i += 32) {
    float zz = srt[i];
    zf[ray * S + i] = zz;
    if (pts != nullptr) {
      float* p = pts + (ray * S + i) * 3;
      p[0] = __fadd_rn(ox, __fmul_rn(zz, dx));
      p[1] = __fadd_rn(oy, __fmul_rn(zz, dy));
      p[2] = __fadd_rn(oz, __fmul_rn(zz, dz));
    }
  }
}

// ------------------------------------------------------------------------------------------------
// Fast path of hn_sample_pdf for the shapes the model uses: in-kernel mid-point bins, Nc = 32 CP coarse depths,
// Nf = 32 FP new samples (CP, FP in {2, 4}).  Same arithmetic contract, different organisation:
//   * the draws u are sorted FIRST (plain keys on registers); the inverse CDF is monotone, so the samples come out
//     ascending and every sample still knows its CDF bin k.  (If rounding ever breaks the order by an ulp — checked —
//     the generic merge below takes over; the multiset of samples is the same either way.)
//   * the bins are the mid-points of the ascending coarse depths, so a sample of bin k lies between mid(z_k, z_k+1) and
//     mid(z_k+1, z_k+2): its rank among the coarse depths is k + 1 + [z_k+1 <= s], corrected by a (normally empty)
//     linear fix-up loop instead of a binary search;
//   * the coarse depths take the slots the samples left free: a bit mask of the taken slots + popcounts, no second search;
//   * depths and points leave as 16-byte vectors (a lane owns 4 consecutive samples = 48 contiguous bytes of points).
// ------------------------------------------------------------------------------------------------
template <int CP, int FP>
__global__ void __launch_bounds__(4 * 32)
sample_pdf_fast_kernel(const float* __restrict__ zc_g, const float* __restrict__ wc, int64_t w_stride,
                       const float* __restrict__ u_g, const float* __restrict__ o, const float* __restrict__ d, int64_t B,
                       float* __restrict__ zf, float* __restrict__ pts, int32_t* __restrict__ bin_idx,
                       int32_t* __restrict__ pos_c, int32_t* __restrict__ pos_n) {
  constexpr int Nc = 32 * CP, Nf = 32 * FP, nb = Nc - 2, ncdf = nb + 1, S = Nc + Nf, NW = S / 32;
  __shared__ float sm_all[4][3 * Nc + Nf + S];
  __shared__ int sm_cnt[4][Nf];     // bucket counts / bucket starts of the draw sort
  const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
  const int64_t ray = (int64_t)blockIdx.x * 4 + wid;
  if (ray >= B) return;
  float* zc = sm_all[wid];          // [Nc] coarse depths (ascending, or sorted below)
  float* bins = zc + Nc;            // [Nc - 1]
  float* cdf = bins + Nc;           // [Nc - 1]
  float* smp = cdf + Nc;            // [Nf]
  float* merged = smp + Nf;         // [S]
  const float eps = 1e-5f;

  // coarse depths, mid-point bins
  bool c_sorted = true;
#pragma unroll
  for (int r = 0; r < CP; ++r) zc[r * 32 + lane] = __ldg(zc_g + ray * Nc + r * 32 + lane);
  __syncwarp();
#pragma unroll
  for (int r = 0; r < CP; ++r) {
    const int i = r * 32 + lane;
    if (i < ncdf) {
      bins[i] = __fmul_rn(0.5f, __fadd_rn(zc[i + 1], zc[i]));
      c_sorted &= zc[i] <= zc[i + 1];
    }
  }
  c_sorted = __all_sync(kFull, c_sorted);

  // pdf and its inclusive prefix: lane owns bins [lane CP, lane CP + CP); sums carried in fp64 (exact)
  float wl[CP];
  double part = 0.0;
#pragma unroll
  for (int j = 0; j < CP; ++j) {
    const int i = lane * CP + j;
    wl[j] = i < nb ? __fadd_rn(__ldg(wc + ray * w_stride + i), eps) : 0.f;
    part += (double)wl[j];
  }
  const float Ssum = (float)warp_sum_d(part);
  double loc[CP];
  double run = 0.0;
#pragma unroll
  for (int j = 0; j < CP; ++j) {
    const int i = lane * CP + j;
    if (i < nb) run += (double)__fdiv_rn(wl[j], Ssum);
    loc[j] = run;
  }
  double inc = run;
#pragma unroll
  for (int off = 1; off < 32; off <<= 1) {
    const double t = __shfl_up_sync(kFull, inc, off);
    if (lane >= off) inc += t;
  }
  const double excl = inc - run;
  if (lane == 0) cdf[0] = 0.f;
#pragma unroll
  for (int j = 0; j < CP; ++j) {
    const int i = lane * CP + j;
    if (i < nb) cdf[i + 1] = (float)(excl + loc[j]);
  }

  // draws: sorted unless they arrive ascending (deterministic linspace draws)
  float uu[FP];
  bool ordered = true;
#pragma unroll
  for (int r = 0; r < FP; ++r) {
    uu[r] = __ldg(u_g + ray * Nf + r * 32 + lane);
    smp[r * 32 + lane] = uu[r];
  }
  __syncwarp();
  if (bin_idx != nullptr) {   // (parity tests) bin of every draw in its original order
#pragma unroll
    for (int r = 0; r < FP; ++r) {
      int pos = 0;
#pragma unroll
      for (int st = Nc / 2; st > 0; st >>= 1)
        if (cdf[pos + st - 1] <= uu[r]) pos += st;
      bin_idx[ray * Nf + r * 32 + lane] = pos;
    }
  }
#pragma unroll
  for (int r = 0; r < FP; ++r) {
    const int e = r * 32 + lane;
    if (e > 0) ordered &= smp[e - 1] <= uu[r];
  }
  if (!__all_sync(kFull, ordered)) {
    // Bucket sort: torch.rand draws are uniform on [0, 1) whatever the weights look like, so bucket floor(u Nf) holds one
    // draw on average (Poisson): count per bucket (shared-memory atomics hand out arrival numbers), exclusive prefix,
    // then every draw ranks itself among the few members of its own bucket.  floor(u Nf) is monotone in u, so the
    // result is the ascending order of the draws (equal draws are interchangeable).  A crowded bucket (> 8 members:
    // draws that are not uniform) sends the ray through the bitonic network instead.
    int* cnt = sm_cnt[wid];
#pragma unroll
    for (int r = 0; r < FP; ++r) cnt[r * 32 + lane] = 0;
    __syncwarp();
    int bk[FP], arr[FP];
#pragma unroll
    for (int r = 0; r < FP; ++r) {
      bk[r] = min(max((int)(uu[r] * (float)Nf), 0), Nf - 1);
      arr[r] = atomicAdd(&cnt[bk[r]], 1);
    }
    __syncwarp();
    int c[FP], tot = 0, cmax = 0;
#pragma unroll
    for (int j = 0; j < FP; ++j) {
      c[j] = cnt[lane * FP + j];
      tot += c[j];
      cmax = max(cmax, c[j]);
    }
    int inc = tot;
#pragma unroll
    for (int off = 1; off < 32; off <<= 1) {
      const int t = __shfl_up_sync(kFull, inc, off);
      if (lane >= off) inc += t;
    }
    const int m = __reduce_max_sync(kFull, cmax);   // fullest bucket of the ray (warp-uniform)
    if (m > 8) {
      bitonic_sort_regs<FP>(smp, lane);
    } else {
      int ex = inc - tot;
#pragma unroll
      for (int j = 0; j < FP; ++j) { cnt[lane * FP + j] = ex; ex += c[j]; }   // counts -> bucket starts
      float* tmp = merged;   // free until the merge; [Nf] draws grouped by bucket + 8 x +inf
      if (lane < 8) tmp[Nf + lane] = __int_as_float(0x7f800000);
#pragma unroll
      for (int r = 0; r < FP; ++r) smp[r * 32 + lane] = __int_as_float(0x7fc00000);   // NaN: "slot not written yet"
      __syncwarp();
      int s0[FP];
#pragma unroll
      for (int r = 0; r < FP; ++r) {
        s0[r] = cnt[bk[r]];
        tmp[s0[r] + arr[r]] = uu[r];
      }
      __syncwarp();
      // rank = bucket start + members below the draw.  The m entries from the bucket's start cover the bucket; what
      // follows it belongs to later buckets (strictly larger) or is the padding.  Equal draws inside one bucket (1e-4 of
      // the rays with torch.rand's 24-bit draws) get the same rank and leave a slot unwritten: detected below.
      int rank[FP];
#pragma unroll
      for (int r = 0; r < FP; ++r) rank[r] = s0[r];
#pragma unroll
      for (int j = 0; j < 8; ++j) {
        if (j >= m) break;
#pragma unroll
        for (int r = 0; r < FP; ++r) rank[r] += (tmp[s0[r] + j] < uu[r]) ? 1 : 0;
      }
#pragma unroll
      for (int r = 0; r < FP; ++r) smp[rank[r]] = uu[r];
      __syncwarp();
      bool hole = false;
#pragma unroll
      for (int r = 0; r < FP; ++r) { const float v = smp[r * 32 + lane]; hole |= v != v; }
      if (__any_sync(kFull, hole)) {
        __syncwarp();
#pragma unroll
        for (int r = 0; r < FP; ++r) smp[r * 32 + lane] = uu[r];
        __syncwarp();
        bitonic_sort_regs<FP>(smp, lane);
      }
    }
#pragma unroll
    for (int r = 0; r < FP; ++r) uu[r] = smp[r * 32 + lane];
  }
  __syncwarp();

  // inverse CDF of the sorted draws; sample e = r 32 + lane keeps its bin
  float sv[FP];
  int kb[FP];
#pragma unroll
  for (int r = 0; r < FP; ++r) {
    int pos = 0;   // searchsorted(cdf, u, right=True): entries <= u among the Nc - 1
#pragma unroll
    for (int st = Nc / 2; st > 0; st >>= 1)
      if (cdf[pos + st - 1] <= uu[r]) pos += st;
    const int below = max(pos - 1, 0), above = min(pos, nb);
    const float c0 = cdf[below], c1 = cdf[above];
    const float g0 = bins[below], g1 = bins[above];
    float denom = __fsub_rn(c1, c0);
    if (denom < eps) denom = 1.f;
    const float t = __fdiv_rn(__fsub_rn(uu[r], c0), denom);
    sv[r] = __fadd_rn(g0, __fmul_rn(t, __fsub_rn(g1, g0)));
    kb[r] = below;
  }
  __syncwarp();
#pragma unroll
  for (int r = 0; r < FP; ++r) smp[r * 32 + lane] = sv[r];
  __syncwarp();
  ordered = true;
#pragma unroll
  for (int r = 0; r < FP; ++r) {
    const int e = r * 32 + lane;
    if (e > 0) ordered &= smp[e - 1] <= sv[r];
  }
  ordered = __all_sync(kFull, ordered);

  if (ordered && c_sorted) {
    // ranks from the bins: a new sample goes after the coarse depths <= it; mask[t] = slots [32 t, 32 t + 32) taken by
    // new samples (warp-wide OR reductions, every lane ends up with all words)
    uint32_t mask[NW];
#pragma unroll
    for (int t = 0; t < NW; ++t) mask[t] = 0u;
#pragma unroll
    for (int r = 0; r < FP; ++r) {
      const int e = r * 32 + lane;
      const float v = sv[r];
      int c = kb[r] + 1;                       // 1 .. Nc - 1
      if (zc[c] <= v) ++c;
      if ((c < Nc && zc[min(c, Nc - 1)] <= v) || zc[c - 1] > v) {   // (normally not taken)
        while (c < Nc && zc[c] <= v) ++c;
        while (c > 0 && zc[c - 1] > v) --c;
      }
      const int p = e + c;
      merged[p] = v;
      if (pos_n != nullptr) pos_n[ray * Nf + e] = p;
      // sample e = 32 r + lane lands in [32 r, 32 r + Nc + 32): only those words can receive its bit
#pragma unroll
      for (int t = r; t < NW && t <= r + CP; ++t)
        mask[t] |= __reduce_or_sync(kFull, (p >> 5) == t ? (1u << (p & 31)) : 0u);
    }
    // the coarse depths fill the free slots in order
    int before = 0;
#pragma unroll
    for (int t = 0; t < NW; ++t) {
      const uint32_t word = mask[t];
      if (!((word >> lane) & 1u)) {
        const int q = t * 32 + lane;
        const int i = q - (before + __popc(word & ((1u << lane) - 1u)));
        merged[q] = zc[i];
        if (pos_c != nullptr) pos_c[ray * Nc + i] = q;
      }
      before += __popc(word);
    }
  } else {
    // generic merge (sample_pdf_kernel): sort what is not ascending, ranks by binary search
    if (!ordered) bitonic_sort_regs<FP>(smp, lane);
    if (!c_sorted) bitonic_sort_regs<CP>(zc, lane);
    __syncwarp();
#pragma unroll
    for (int r = 0; r < CP; ++r) {
      const int i = r * 32 + lane;
      const float v = zc[i];
      int lo = 0, hi = Nf;
      while (lo < hi) { const int mid = (lo + hi) >> 1; if (smp[mid] < v) lo = mid + 1; else hi = mid; }
      merged[i + lo] = v;
      if (pos_c != nullptr) pos_c[ray * Nc + i] = i + lo;
    }
#pragma unroll
    for (int r = 0; r < FP; ++r) {
      const int i = r * 32 + lane;
      const float v = smp[i];
      int lo = 0, hi = Nc;
      while (lo < hi) { const int mid = (lo + hi) >> 1; if (zc[mid] <= v) lo = mid + 1; else hi = mid; }
      merged[i + lo] = v;
      if (pos_n != nullptr) pos_n[ray * Nf + i] = i + lo;
    }
  }
  __syncwarp();

  // depths and points: a lane owns 4 consecutive samples
  float ox = 0.f, oy = 0.f, oz = 0.f, dx = 0.f, dy = 0.f, dz = 0.f;
  if (pts != nullptr) {
    ox = __ldg(o + ray * 3); oy = __ldg(o + ray * 3 + 1); oz = __ldg(o + ray * 3 + 2);
    dx = __ldg(d + ray * 3); dy = __ldg(d + ray * 3 + 1); dz = __ldg(d + ray * 3 + 2);
  }
  for (int g = lane; g < S / 4; g += 32) {
    const float4 z4 = *reinterpret_cast<const float4*>(merged + 4 * g);
    reinterpret_cast<float4*>(zf + ray * S)[g] = z4;
    if (pts != nullptr) {
      const float zz[4] = {z4.x, z4.y, z4.z, z4.w};
      float pv[12];
#pragma unroll
      for (int j = 0; j < 4; ++j) {
        pv[3 * j] = __fadd_rn(ox, __fmul_rn(zz[j], dx));
        pv[3 * j + 1] = __fadd_rn(oy, __fmul_rn(zz[j], dy));
        pv[3 * j + 2] = __fadd_rn(oz, __fmul_rn(zz[j], dz));
      }
      float4* dst = reinterpret_cast<float4*>(pts + (ray * S + 4 * g) * 3);
      dst[0] = make_float4(pv[0], pv[1], pv[2], pv[3]);
      dst[1] = make_float4(pv[4], pv[5], pv[6], pv[7]);
      dst[2] = make_float4(pv[8], pv[9], pv[10], pv[11]);
    }
  }
}

template <int C>
static int launch_comp_fwd(bool exact, dim3 g, cudaStream_t st, const float* sigma, const float* rgb, const float* z,
                           const float* dirs, int64_t B, int S, int flags, float eps, float ld, float* o_rgb,
                           float* depth, float* med, float* acc, float* w, int64_t* mi) {
  if (exact)
    composite_fwd_kernel<C, true><<<g, kWarpsPerBlock * 32, 0, st>>>(sigma, rgb, z, dirs, B, S, flags, eps, ld, o_rgb,
                                                                   depth, med, acc, w, mi);
  else
    composite_fwd_kernel<C, false><<<g, kWarpsPerBlock * 32, 0, st>>>(sigma, rgb, z, dirs, B, S, flags, eps, ld,
                                                                    o_rgb, depth, med, acc, w, mi);
  return 0;
}
template <int C>
static int launch_comp_bwd(bool exact, dim3 g, cudaStream_t st, const float* sigma, const float* rgb, const float* z,
                           const float* dirs, int64_t B, int S, int flags, float eps, float ld, const float* g1,
                           const float* g2, const float* g3, const float* g4, float* gs, float* gc) {
  if (exact)
    composite_bwd_kernel<C, true><<<g, kWarpsPerBlock * 32, 0, st>>>(sigma, rgb, z, dirs, B, S, flags, eps, ld, g1, g2,
                                                                   g3, g4, gs, gc);
  else
    composite_bwd_kernel<C, false><<<g, kWarpsPerBlock * 32, 0, st>>>(sigma, rgb, z, dirs, B, S, flags, eps, ld, g1,
                                                                    g2, g3, g4, gs, gc);
  return 0;
}

}  // namespace hn

using namespace hn;

extern "C" int hn_sample_coarse(const float* origins, const float* dirs, const float* u, const float* lower,
                                const float* upper, int64_t B, int Nc, float* z, float* points, void* stream) {
  if (B < 0 || Nc <= 0) return set_error(-1, "hn_sample_coarse: bad B/Nc");
  if (!origins || !dirs || !lower || !upper || !z) return set_error(-2, "hn_sample_coarse: null pointer");
  if (B == 0) return 0;
  int64_t n = B * Nc;
  int threads = 256;
  auto aligned16 = [](const void* p) { return p == nullptr || (reinterpret_cast<uintptr_t>(p) & 15) == 0; };
  if (Nc % 4 == 0 && aligned16(u) && aligned16(lower) && aligned16(upper) && aligned16(z) && aligned16(points)) {
    const int64_t n4 = n / 4;
    sample_coarse_v4_kernel<<<(unsigned)((n4 + threads - 1) / threads), threads, 0, (cudaStream_t)stream>>>(
        origins, dirs, reinterpret_cast<const float4*>(u), reinterpret_cast<const float4*>(lower),
        reinterpret_cast<const float4*>(upper), n4, Nc / 4, reinterpret_cast<float4*>(z), reinterpret_cast<float4*>(points));
    return set_cuda_error(cudaGetLastError(), "hn_sample_coarse");
  }
  int64_t blocks = (n + threads - 1) / threads;
  sample_coarse_kernel<<<(unsigned)blocks, threads, 0, (cudaStream_t)stream>>>(origins, dirs, u, lower, upper, n, Nc,
                                                                              z, points);
  return set_cuda_error(cudaGetLastError(), "hn_sample_coarse");
}

static int sample_pdf_impl(const float* z_coarse, const float* bins, const float* weights, int64_t w_stride,
                           const float* u, const float* origins, const float* dirs, int64_t B, int Nc, int nb, int Nf,
                           float* z_fine, float* points, int32_t* bin_idx, int32_t* pos_coarse, int32_t* pos_new,
                           void* stream) {
  if (B < 0 || Nc < 1 || nb < 1 || Nf <= 0) return set_error(-1, "hn_sample_pdf: need Nc >= 1, nb >= 1, Nf >= 1");
  if (bins == nullptr && nb != Nc - 2) return set_error(-1, "hn_sample_pdf: in-kernel bins need nb == Nc - 2");
  if (Nc + Nf > kPdfMaxN || nb + 1 > kPdfMaxN) return set_error(-1, "hn_sample_pdf: Nc + Nf > 512 unsupported");
  if (!z_coarse || !weights || !u || !z_fine) return set_error(-2, "hn_sample_pdf: null pointer");
  if (points && (!origins || !dirs)) return set_error(-2, "hn_sample_pdf: points need origins and dirs");
  if (B == 0) return 0;
  // the model's shapes (in-kernel bins, 64 / 128 coarse depths, 64 / 128 new samples) take the fast kernel
  const bool aligned = (reinterpret_cast<uintptr_t>(z_fine) & 15) == 0 && (!points || (reinterpret_cast<uintptr_t>(points) & 15) == 0);
  if (bins == nullptr && aligned && (Nc == 64 || Nc == 128) && (Nf == 64 || Nf == 128)) {
    const unsigned blocks4 = (unsigned)((B + 3) / 4);
#define HN_PDF_FAST(CP, FP)                                                                                                 \
    sample_pdf_fast_kernel<CP, FP><<<blocks4, 128, 0, (cudaStream_t)stream>>>(z_coarse, weights, w_stride, u, origins, dirs, B, \
                                                                              z_fine, points, bin_idx, pos_coarse, pos_new)
    if (Nc == 64 && Nf == 64) HN_PDF_FAST(2, 2);
    else if (Nc == 64) HN_PDF_FAST(2, 4);
    else if (Nf == 64) HN_PDF_FAST(4, 2);
    else HN_PDF_FAST(4, 4);
#undef HN_PDF_FAST
    return set_cuda_error(cudaGetLastError(), "hn_sample_pdf");
  }
  int n2 = 1, n2c = 1;   // new samples and coarse depths are sorted on their own (padded to powers of two), then merged
  while (n2 < Nf) n2 <<= 1;
  while (n2c < Nc) n2c <<= 1;
  size_t smem = (size_t)4 * (2 * (nb + 1) + n2c + n2 + Nc + Nf) * sizeof(float);
  int64_t blocks = (B + 3) / 4;
  sample_pdf_kernel<<<(unsigned)blocks, 128, smem, (cudaStream_t)stream>>>(z_coarse, bins, weights, w_stride, u, origins,
                                                                          dirs, B, Nc, nb, Nf, n2c, n2, z_fine, points, bin_idx, pos_coarse,
                                                                          pos_new);
  return set_cuda_error(cudaGetLastError(), "hn_sample_pdf");
}

extern "C" int hn_sample_pdf(const float* z_coarse, const float* bins, const float* weights, int64_t w_stride,
                             const float* u, const float* origins, const float* dirs, int64_t B, int Nc, int nb, int Nf,
                             float* z_fine, float* points, int32_t* bin_idx, void* stream) {
  return sample_pdf_impl(z_coarse, bins, weights, w_stride, u, origins, dirs, B, Nc, nb, Nf, z_fine, points, bin_idx, nullptr,
                         nullptr, stream);
}

extern "C" int hn_sample_pdf_ranks(const float* z_coarse, const float* bins, const float* weights, int64_t w_stride,
                                   const float* u, const float* origins, const float* dirs, int64_t B, int Nc, int nb, int Nf,
                                   float* z_fine, float* points, int32_t* bin_idx, int32_t* pos_coarse, int32_t* pos_new,
                                   void* stream) {
  if (!pos_coarse || !pos_new) return set_error(-2, "hn_sample_pdf_ranks: null pointer");
  return sample_pdf_impl(z_coarse, bins, weights, w_stride, u, origins, dirs, B, Nc, nb, Nf, z_fine, points, bin_idx,
                         pos_coarse, pos_new, stream);
}

#define HN_DISPATCH_C(FN, ...)                                              \
  switch (C) {                                                              \
    case 1: FN<1>(__VA_ARGS__); break;                                      \
    case 2: FN<2>(__VA_ARGS__); break;                                      \
    case 3: FN<3>(__VA_ARGS__); break;                                      \
    case 4: FN<4>(__VA_ARGS__); break;                                      \
    case 5: FN<5>(__VA_ARGS__); break;                                      \
    case 6: FN<6>(__VA_ARGS__); break;                                      \
    case 7: FN<7>(__VA_ARGS__); break;                                      \
    case 8: FN<8>(__VA_ARGS__); break;                                      \
    case 12: FN<12>(__VA_ARGS__); break;                                    \
    default: FN<16>(__VA_ARGS__); break;                                    \
  }

static int comp_c(int S) {
  int C = (S + 31) / 32;
  if (C > 8 && C <= 12) C = 12;
  else if (C > 12) C = 16;
  return C;
}

extern "C" int hn_composite_fwd(const float* sigma, const float* rgb, const float* z, const float* dirs, int64_t B,
                                int S, int flags, float eps, float last_delta, float* out_rgb, float* depth,
                                float* med_depth, float* acc, float* weights, int64_t* med_idx, void* stream) {
  if (B < 0 || S <= 0 || S > 512) return set_error(-1, "hn_composite_fwd: need 1 <= S <= 512");
  if (!sigma || !rgb || !z || !dirs || !out_rgb || !depth || !acc) return set_error(-2, "hn_composite_fwd: null pointer");
  if (B == 0) return 0;
  int C = comp_c(S);
  bool exact = (S == 32 * C);
  const bool aligned = ((reinterpret_cast<uintptr_t>(sigma) | reinterpret_cast<uintptr_t>(z) | reinterpret_cast<uintptr_t>(rgb) |
                         reinterpret_cast<uintptr_t>(weights)) & 15) == 0;
  if (S == 64 && aligned) {   // two rays per warp
    dim3 g2((unsigned)((B + 2 * kWarpsPerBlock - 1) / (2 * kWarpsPerBlock)));
    composite_fwd_s64_kernel<<<g2, kWarpsPerBlock * 32, 0, (cudaStream_t)stream>>>(sigma, rgb, z, dirs, B, flags, eps, last_delta,
                                                                                  out_rgb, depth, med_depth, acc, weights, med_idx);
    return set_cuda_error(cudaGetLastError(), "hn_composite_fwd");
  }
  dim3 g((unsigned)((B + kWarpsPerBlock - 1) / kWarpsPerBlock));
  HN_DISPATCH_C(launch_comp_fwd, exact, g, (cudaStream_t)stream, sigma, rgb, z, dirs, B, S, flags, eps, last_delta,
                out_rgb, depth, med_depth, acc, weights, med_idx);
  return set_cuda_error(cudaGetLastError(), "hn_composite_fwd");
}

extern "C" int hn_composite_bwd(const float* sigma, const float* rgb, const float* z, const float* dirs, int64_t B,
                                int S, int flags, float eps, float last_delta, const float* g_out_rgb,
                                const float* g_depth, const float* g_acc, const float* g_weights, float* g_sigma,
                                float* g_rgb, void* stream) {
  if (B < 0 || S <= 0 || S > 512) return set_error(-1, "hn_composite_bwd: need 1 <= S <= 512");
  if (!sigma || !rgb || !z || !dirs || !g_sigma || !g_rgb) return set_error(-2, "hn_composite_bwd: null pointer");
  if (B == 0) return 0;
  int C = comp_c(S);
  bool exact = (S == 32 * C);
  if (S == 64) {
    dim3 g2((unsigned)((B + 2 * kWarpsPerBlock - 1) / (2 * kWarpsPerBlock)));
    composite_bwd_s64_kernel<<<g2, kWarpsPerBlock * 32, 0, (cudaStream_t)stream>>>(sigma, rgb, z, dirs, B, flags, eps, last_delta,
                                                                                   g_out_rgb, g_depth, g_acc, g_weights, g_sigma, g_rgb);
    return set_cuda_error(cudaGetLastError(), "hn_composite_bwd");
  }
  dim3 g((unsigned)((B + kWarpsPerBlock - 1) / kWarpsPerBlock));
  HN_DISPATCH_C(launch_comp_bwd, exact, g, (cudaStream_t)stream, sigma, rgb, z, dirs, B, S, flags, eps, last_delta,
                g_out_rgb, g_depth, g_acc, g_weights, g_sigma, g_rgb);
  return set_cuda_error(cudaGetLastError(), "hn_composite_bwd");
}


// ------------------------------------------------------------------------------------------------------
// hn_mse_loss — losses.py:9-14 (MSE(coarse.rgb) + MSE(fine.rgb), mean reduction) fused with its gradient seed
// and the fine-level MSE that metrics.py:4-13 turns into PSNR.  One pass over (B,3) predictions: sums[0] +=
// sum (c - t)^2, sums[1] += sum (f - t)^2 (fp32 block partials, one atomic per block and level) and
// g_level = 2 (pred - t) * grad_scale (grad_scale = upstream_grad / (3 B_global)).
// ------------------------------------------------------------------------------------------------------
namespace hn {
__global__ void __launch_bounds__(256) mse_loss_kernel(const float* __restrict__ pc, const float* __restrict__ pf,
                                                       const float* __restrict__ tg, int64_t n, float grad_scale,
                                                       float* __restrict__ sums, float* __restrict__ gc, float* __restrict__ gf) {
  float sc = 0.f, sf = 0.f;
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x) {
    const float t = __ldg(tg + i);
    const float dc = __ldg(pc + i) - t;
    sc += dc * dc;
    if (gc != nullptr) gc[i] = 2.f * dc * grad_scale;
    if (pf != nullptr) {
      const float df = __ldg(pf + i) - t;
      sf += df * df;
      if (gf != nullptr) gf[i] = 2.f * df * grad_scale;
    }
  }
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) { sc += __shfl_xor_sync(kFull, sc, o); sf += __shfl_xor_sync(kFull, sf, o); }
  __shared__ float red[2][8];
  const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
  if (lane == 0) { red[0][wid] = sc; red[1][wid] = sf; }
  __syncthreads();
  if (wid == 0) {
    sc = lane < 8 ? red[0][lane] : 0.f;
    sf = lane < 8 ? red[1][lane] : 0.f;
#pragma unroll
    for (int o = 4; o > 0; o >>= 1) { sc += __shfl_xor_sync(kFull, sc, o); sf += __shfl_xor_sync(kFull, sf, o); }
    if (lane == 0) { atomicAdd(sums, sc); if (pf != nullptr) atomicAdd(sums + 1, sf); }
  }
}
}  // namespace hn

extern "C" int hn_mse_loss(const float* rgb_coarse, const float* rgb_fine, const float* targets, int64_t B, float grad_scale,
                           float* sums, float* g_coarse, float* g_fine, void* stream) {
  if (!rgb_coarse || !targets || !sums) return hn::set_error(-2, "hn_mse_loss: null pointer");
  if (B < 0) return hn::set_error(-1, "hn_mse_loss: negative B");
  if (B == 0) return 0;
  const int64_t n = B * 3;
  const int blocks = (int)std::min<int64_t>((n + 255) / 256, 4 * (int64_t)hn::num_sms());
  hn::mse_loss_kernel<<<blocks, 256, 0, (cudaStream_t)stream>>>(rgb_coarse, rgb_fine, targets, n, grad_scale, sums, g_coarse, g_fine);
  return hn::set_cuda_error(cudaGetLastError(), "hn_mse_loss");
}


// ------------------------------------------------------------------------------------------------------
// hn_filter_sigma — filter_sigma (models.py:35-63): out = mask * values with mask = (sigma >= dust_threshold) and
// (point inside the bounding box), either test optional.  Forward: values = sigma; backward: values = upstream gradient
// (the reference multiplies by the boolean masks, so the gradient passes where the mask is set).
// ------------------------------------------------------------------------------------------------------
namespace hn {
struct BBox { float v[6]; };
__global__ void __launch_bounds__(256) filter_sigma_kernel(const float* __restrict__ points, const float* __restrict__ sigma,
                                                           const float* __restrict__ values, int64_t n, float dust, int use_dust,
                                                           BBox b, int use_bbox, float* __restrict__ out) {
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x) {
    bool keep = true;
    // the two tests compose as in the reference: the bounding-box product sees the dust-filtered value, which changes
    // nothing for the mask itself
    if (use_dust) keep = __ldg(sigma + i) >= dust;
    if (use_bbox) {
      const float x = __ldg(points + 3 * i), y = __ldg(points + 3 * i + 1), z = __ldg(points + 3 * i + 2);
      keep = keep && x >= b.v[0] && x <= b.v[1] && y >= b.v[2] && y <= b.v[3] && z >= b.v[4] && z <= b.v[5];
    }
    out[i] = keep ? __ldg(values + i) : 0.f;
  }
}
}  // namespace hn

extern "C" int hn_filter_sigma(const float* points, const float* sigma, const float* values, int64_t n, float dust_threshold,
                               int use_dust, const float* bbox_host, float* out, void* stream) {
  if (!sigma || !values || !out || (bbox_host && !points)) return hn::set_error(-2, "hn_filter_sigma: null pointer");
  if (n < 0) return hn::set_error(-1, "hn_filter_sigma: negative n");
  if (n == 0) return 0;
  hn::BBox b{};
  if (bbox_host) for (int k = 0; k < 6; ++k) b.v[k] = bbox_host[k];
  const int blocks = (int)std::min<int64_t>((n + 255) / 256, 8 * (int64_t)hn::num_sms());
  hn::filter_sigma_kernel<<<blocks, 256, 0, (cudaStream_t)stream>>>(points, sigma, values, n, dust_threshold, use_dust, b,
                                                                    bbox_host != nullptr, out);
  return hn::set_cuda_error(cudaGetLastError(), "hn_filter_sigma");
}


// ------------------------------------------------------------------------------------------------------
// hn_make_ndc_rays — datasets/ray_utils.py:5-93 (get_ray_directions -> get_rays -> get_ndc_rays) + the ray-row layout
// of datasets/llff.py:261-264 / 316-332 for one full frame, on the device: pixel (i = column, j = row) ->
// camera direction ((i - W/2)/f, -(j - H/2)/f, -1) -> world (rotate by c2w[:, :3], normalise) -> NDC origin /
// direction -> row [o(3), d(3), near = 0, far = 1, image id].  c2w: 12 floats, row-major (3,4), passed by value.
// ------------------------------------------------------------------------------------------------------
namespace hn {
struct C2W { float m[12]; };
__global__ void __launch_bounds__(256) make_ndc_rays_kernel(int H, int W, float focal, C2W c, float near_plane, float image_id,
                                                            int cols, float* __restrict__ rays) {
  const int64_t n = (int64_t)H * W;
  for (int64_t p = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; p < n; p += (int64_t)gridDim.x * blockDim.x) {
    const float i = (float)(p % W), j = (float)(p / W);
    const float cx = (i - W / 2.f) / focal, cy = -(j - H / 2.f) / focal, cz = -1.f;
    float dx = cx * c.m[0] + cy * c.m[1] + cz * c.m[2];
    float dy = cx * c.m[4] + cy * c.m[5] + cz * c.m[6];
    float dz = cx * c.m[8] + cy * c.m[9] + cz * c.m[10];
    const float inv = 1.f / sqrtf(dx * dx + dy * dy + dz * dz);
    dx *= inv; dy *= inv; dz *= inv;
    float ox = c.m[3], oy = c.m[7], oz = c.m[11];
    const float t = -(near_plane + oz) / dz;                 // shift the origin to the near plane
    ox += t * dx; oy += t * dy; oz += t * dz;
    const float ox_oz = ox / oz, oy_oz = oy / oz;
    const float sx = -1.f / (W / (2.f * focal)), sy = -1.f / (H / (2.f * focal));
    const float o2 = 1.f + 2.f * near_plane / oz;
    float* r = rays + p * cols;
    r[0] = sx * ox_oz; r[1] = sy * oy_oz; r[2] = o2;
    r[3] = sx * (dx / dz - ox_oz); r[4] = sy * (dy / dz - oy_oz); r[5] = 1.f - o2;
    r[6] = 0.f; r[7] = 1.f;
    if (cols > 8) r[8] = image_id;
  }
}
}  // namespace hn

extern "C" int hn_make_ndc_rays(int H, int W, float focal, const float* c2w_host, float near_plane, float image_id, int cols,
                                float* rays, void* stream) {
  if (!c2w_host || !rays) return hn::set_error(-2, "hn_make_ndc_rays: null pointer");
  if (H <= 0 || W <= 0 || focal <= 0.f || (cols != 8 && cols != 9)) return hn::set_error(-1, "hn_make_ndc_rays: bad H/W/focal/cols");
  hn::C2W c;
  for (int k = 0; k < 12; ++k) c.m[k] = c2w_host[k];
  const int64_t n = (int64_t)H * W;
  const int blocks = (int)std::min<int64_t>((n + 255) / 256, 8 * (int64_t)hn::num_sms());
  hn::make_ndc_rays_kernel<<<blocks, 256, 0, (cudaStream_t)stream>>>(H, W, focal, c, near_plane, image_id, cols, rays);
  return hn::set_cuda_error(cudaGetLastError(), "hn_make_ndc_rays");
}

// ======================================================================================================
// optimizer: torch.optim.Adam.step over the flat parameter / gradient buffers in one launch
// ======================================================================================================
namespace hn {
struct AdamArgs { float beta1, beta2, eps, weight_decay, step_size, inv_bc2_sqrt, grad_scale; };

__device__ __forceinline__ void adam_one(float& p, float g, float& m, float& v, const AdamArgs& a) {
  g *= a.grad_scale;
  if (a.weight_decay != 0.f) g = fmaf(a.weight_decay, p, g);     // L2 form: grad + wd * param
  m = m + (g - m) * (1.f - a.beta1);                              // lerp, as torch's exp_avg.lerp_(grad, 1 - beta1)
  v = a.beta2 * v + (1.f - a.beta2) * g * g;
  const float denom = sqrtf(v) * a.inv_bc2_sqrt + a.eps;
  p = p - a.step_size * (m / denom);
}

__global__ void __launch_bounds__(256) adam_kernel(float* __restrict__ params, const float* __restrict__ grads,
                                                   float* __restrict__ exp_avg, float* __restrict__ exp_avg_sq, int64_t n,
                                                   AdamArgs a) {
  const int64_t n4 = n >> 2;
  const int64_t stride = (int64_t)gridDim.x * blockDim.x;
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n4; i += stride) {
    float4 p = reinterpret_cast<float4*>(params)[i];
    const float4 g = reinterpret_cast<const float4*>(grads)[i];
    float4 m = reinterpret_cast<float4*>(exp_avg)[i];
    float4 v = reinterpret_cast<float4*>(exp_avg_sq)[i];
    adam_one(p.x, g.x, m.x, v.x, a); adam_one(p.y, g.y, m.y, v.y, a);
    adam_one(p.z, g.z, m.z, v.z, a); adam_one(p.w, g.w, m.w, v.w, a);
    reinterpret_cast<float4*>(params)[i] = p;
    reinterpret_cast<float4*>(exp_avg)[i] = m;
    reinterpret_cast<float4*>(exp_avg_sq)[i] = v;
  }
  for (int64_t i = (n4 << 2) + (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += stride)
    adam_one(params[i], grads[i], exp_avg[i], exp_avg_sq[i], a);
}
}  // namespace hn

extern "C" int hn_adam_step(float* params, const float* grads, float* exp_avg, float* exp_avg_sq, int64_t n, float lr,
                            float beta1, float beta2, float eps, float weight_decay, int64_t step, float grad_scale,
                            void* stream) {
  if (!params || !grads || !exp_avg || !exp_avg_sq) return hn::set_error(-2, "hn_adam_step: null pointer");
  if (n < 0 || step < 1) return hn::set_error(-1, "hn_adam_step: n < 0 or step < 1");
  if ((reinterpret_cast<uintptr_t>(params) | reinterpret_cast<uintptr_t>(grads) | reinterpret_cast<uintptr_t>(exp_avg) |
       reinterpret_cast<uintptr_t>(exp_avg_sq)) & 15)
    return hn::set_error(-3, "hn_adam_step: buffers must be 16-byte aligned");
  if (n == 0) return 0;
  // bias corrections in double, as torch's Python scalars
  const double bc1 = 1.0 - pow((double)beta1, (double)step), bc2 = 1.0 - pow((double)beta2, (double)step);
  hn::AdamArgs a{beta1, beta2, eps, weight_decay, (float)((double)lr / bc1), (float)(1.0 / sqrt(bc2)), grad_scale};
  const int blocks = (int)std::min<int64_t>(((n >> 2) + 255) / 256 + 1, 8 * (int64_t)hn::num_sms());
  hn::adam_kernel<<<blocks, 256, 0, (cudaStream_t)stream>>>(params, grads, exp_avg, exp_avg_sq, n, a);
  return hn::set_cuda_error(cudaGetLastError(), "hn_adam_step");
}
