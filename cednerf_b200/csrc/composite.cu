// K4 — segmented transmittance / alpha compositing and its backward (HBM-bound).
//
// Replaces, behind the same semantics, the nerfacc calls the reference makes at
//   cednerf/render.py:52-54, :81-87   render_transmittance/weight_from_density
//   cednerf/render.py:158-174         accumulate_along_rays x3 + depth normalise + background
//   cednerf/utils.py:274-299          prefix_trans variant + in-place accumulation
// Samples are packed by ray (ray_indices sorted, as the marcher emits them); a group of G lanes
// (G = 4..32, picked from the mean samples/ray) owns one ray and walks its samples in chunks of G with
// shuffle scans: one forward exclusive scan of sigma*dt, one reverse exclusive scan in the backward.
#include <type_traits>

#include "common.cuh"

namespace {

template <int G>
__device__ __forceinline__ unsigned group_mask() {
  if constexpr (G == 32) {
    return 0xffffffffu;
  } else {
    const int lane = threadIdx.x & 31;
    return ((1u << G) - 1u) << (lane / G * G);
  }
}

template <int G>
__device__ __forceinline__ float group_incl_scan(float v, int gl, unsigned gm) {
#pragma unroll
  for (int o = 1; o < G; o <<= 1) {
    float n = __shfl_up_sync(gm, v, o, G);
    if (gl >= o) v += n;
  }
  return v;
}

template <int G>
__device__ __forceinline__ float group_incl_scan_rev(float v, int gl, unsigned gm) {
#pragma unroll
  for (int o = 1; o < G; o <<= 1) {
    float n = __shfl_down_sync(gm, v, o, G);
    if (gl + o < G) v += n;
  }
  return v;
}

template <int G>
__device__ __forceinline__ float group_sum(float v, unsigned gm) {
#pragma unroll
  for (int o = G / 2; o > 0; o >>= 1) v += __shfl_xor_sync(gm, v, o, G);
  return v;
}

// G from the mean samples per ray S / n_rays: <= 6 -> 4, <= 12 -> 8, <= 24 -> 16, else 32 (compared in integers)
__host__ __device__ __forceinline__ int pick_group(int64_t S, int64_t n_rays) {
  if (S <= 6 * n_rays) return 4;
  if (S <= 12 * n_rays) return 8;
  if (S <= 24 * n_rays) return 16;
  return 32;
}

// The group width changes the order of the per-ray scans and sums, so it is part of the result.  The per-ray kernels take
// it from the LIVE sample count offsets[n_rays] on the device (g_fixed = 0): a capacity-sized sample set (buffers larger
// than the live prefix, ops.counts_of) then gives the same bits as the exact-size set, whatever its capacity.  The launch
// is sized from the host's estimate and every group walks its rays in a grid-stride loop, so any G is covered.
// f(std::integral_constant<int, G>{}, ray, gl, gm) runs once per ray on its G lanes; `return` in f moves to the next ray.
template <int G, class F>
__device__ __forceinline__ void ray_groups_g(int64_t n_rays, F& f) {
  const int gl = threadIdx.x % G;
  const unsigned gm = group_mask<G>();
  const int64_t stride = (int64_t)gridDim.x * blockDim.x / G;
  for (int64_t ray = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) / G; ray < n_rays; ray += stride)
    f(std::integral_constant<int, G>{}, ray, gl, gm);
}

template <class F>
__device__ __forceinline__ void for_each_ray_group(const int64_t* offsets, int64_t n_rays, int g_fixed, F f) {
  switch (g_fixed > 0 ? g_fixed : pick_group(offsets[n_rays], n_rays)) {
    case 4: ray_groups_g<4>(n_rays, f); break;
    case 8: ray_groups_g<8>(n_rays, f); break;
    case 16: ray_groups_g<16>(n_rays, f); break;
    default: ray_groups_g<32>(n_rays, f); break;
  }
}

// offsets[r] = index of the first sample whose ray index is >= r; offsets[n_rays] = S.
__global__ void ray_offsets_kernel(const int64_t* __restrict__ ridx, int64_t S, int64_t n_rays,
                                   int64_t* __restrict__ offsets) {
  int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i > S) return;
  int64_t prev = (i == 0) ? -1 : ridx[i - 1];
  int64_t cur = (i == S) ? n_rays : ridx[i];
  if (cur > n_rays) cur = n_rays;
  for (int64_t r = prev + 1; r <= cur; ++r) offsets[r] = i;
}

struct CompositeFwdArgs {
  const float* t0;
  const float* t1;
  const float* sigma;
  const float* rgb;      // [S,3] or null
  const float* prefix;   // [S] or null
  const int64_t* offsets;  // [n_rays+1]
  const float* bkgd;     // null, [3] (stride 0) or [n_rays,3] (stride 3)
  int bkgd_stride;
  int64_t n_rays;
  float* w;      // [S] or null
  float* trans;  // [S] or null
  float* alpha;  // [S] or null
  float* colors;   // [n_rays,3] or null
  float* opacity;  // [n_rays] or null
  float* depth;    // [n_rays] or null
  float* depth_raw;  // [n_rays] or null (un-normalised, saved for backward)
  int accumulate_inplace;  // 1: += into colors/opacity/depth, no normalise / background; 2: same, prefix = 1 - opacity[ray]
  float depth_eps;
  // device-resident marching rounds (cednerf_render_round_composite): `offsets` is indexed by SLOT of the alive list,
  // the ray of a slot is slot_ray[slot], only the first round_state[0] slots are live, and a ray that stays alive
  // (opacity <= 1 - alive_eps and it marched its full k = round_state[1] samples) gets next_flags[slot] = 1
  const int32_t* slot_ray;
  const int32_t* round_state;
  const int32_t* slot_counts;
  float alive_eps;
  int32_t* next_flags;
};

__global__ void __launch_bounds__(256, 8) composite_fwd_kernel(CompositeFwdArgs a, int g_fixed) {
  for_each_ray_group(a.offsets, a.n_rays, g_fixed, [&](auto g_, int64_t slot, int gl, unsigned gm) {
    constexpr int G = decltype(g_)::value;
    bool live = true;
    if (a.round_state && slot >= (int64_t)a.round_state[0]) live = false;
    if (!a.next_flags && !live) return;  // whole groups exit together
    const int64_t ray = live ? (a.slot_ray ? (int64_t)a.slot_ray[slot] : slot) : 0;
    const int64_t s0 = live ? a.offsets[slot] : 0, s1 = live ? a.offsets[slot + 1] : 0;
    float carry = 0.f, cr = 0.f, cg = 0.f, cb = 0.f, co = 0.f, cd = 0.f;
    // mode 2: continue a ray across marching rounds - the transmittance so far is 1 - opacity[ray] (utils.py:274-281)
    const float ray_prefix = (a.accumulate_inplace == 2 && s0 < s1) ? 1.f - a.opacity[ray] : 1.f;
    for (int64_t base = s0; base < s1; base += G) {
      const int64_t i = base + gl;
      const bool ok = i < s1;
      float ta = 0.f, tb = 0.f, sg = 0.f, pf = ray_prefix;
      if (ok) {
        ta = a.t0[i];
        tb = a.t1[i];
        sg = a.sigma[i];
        if (a.prefix) pf = a.prefix[i];
      }
      const float sd = sg * (tb - ta);
      const float incl = group_incl_scan<G>(sd, gl, gm);
      const float T = expf(-(carry + (incl - sd))) * pf;
      const float al = 1.f - expf(-sd);
      const float w = T * al;
      carry += __shfl_sync(gm, incl, G - 1, G);
      if (ok) {
        if (a.w) a.w[i] = w;
        if (a.trans) a.trans[i] = T;
        if (a.alpha) a.alpha[i] = al;
        co += w;
        cd += w * ((ta + tb) * 0.5f);
        if (a.rgb) {
          cr += w * a.rgb[3 * i];
          cg += w * a.rgb[3 * i + 1];
          cb += w * a.rgb[3 * i + 2];
        }
      }
    }
    if (!a.opacity && !a.colors && !a.depth) return;
    cr = group_sum<G>(cr, gm);
    cg = group_sum<G>(cg, gm);
    cb = group_sum<G>(cb, gm);
    co = group_sum<G>(co, gm);
    cd = group_sum<G>(cd, gm);
    bool keep = false;  // round mode: this lane speaks for a ray that stays alive
    if (gl == 0 && live) {
      if (a.accumulate_inplace) {
        if (a.colors) {
          a.colors[3 * ray] += cr;
          a.colors[3 * ray + 1] += cg;
          a.colors[3 * ray + 2] += cb;
        }
        float op = co;
        if (a.opacity) {
          op += a.opacity[ray];
          a.opacity[ray] = op;
        }
        if (a.depth) a.depth[ray] += cd;
        // alive = (opacity <= 1 - early_stop_eps) & (n_samples == k)   (cednerf/utils.py:300-304)
        if (a.next_flags) keep = op <= 1.f - a.alive_eps && a.slot_counts[slot] == a.round_state[1];
      } else {
        if (a.depth_raw) a.depth_raw[ray] = cd;
        if (a.opacity) a.opacity[ray] = co;
        if (a.depth) a.depth[ray] = cd / fmaxf(co, a.depth_eps);
        if (a.colors) {
          float br = 0.f, bg = 0.f, bb = 0.f;
          if (a.bkgd) {
            const float* b = a.bkgd + (int64_t)a.bkgd_stride * ray;
            br = b[0] * (1.f - co);
            bg = b[1] * (1.f - co);
            bb = b[2] * (1.f - co);
          }
          a.colors[3 * ray] = cr + br;
          a.colors[3 * ray + 1] = cg + bg;
          a.colors[3 * ray + 2] = cb + bb;
        }
      }
    }
    // round mode: a flag per slot (0 beyond the live part of the list); the next round's list is the ORDERED compaction
    // of the flagged rays (scan + cednerf_render_round_compact), so the list stays in pixel order and the lanes of a warp
    // keep marching neighbouring rays.  (Measured: an unordered per-ray atomic append cost 45 % in the marcher and 30 % in
    // the field kernel; CTA-sized ordered chunks in arbitrary order still 12 % and 6 %.)
    if (a.next_flags && gl == 0) a.next_flags[slot] = keep ? 1 : 0;
  });
}

struct CompositeBwdArgs {
  const float* t0;
  const float* t1;
  const float* rgb;     // [S,3] or null
  const float* trans;   // [S] saved
  const float* alpha;   // [S] saved
  const int64_t* offsets;
  const float* bkgd;
  int bkgd_stride;
  int64_t n_rays;
  const float* opacity;    // [n_rays] saved (for depth normalisation), may be null
  const float* depth_raw;  // [n_rays] saved, may be null
  const float* g_colors;   // [n_rays,3] or null
  const float* g_opacity;  // [n_rays] or null
  const float* g_depth;    // [n_rays] or null (gradient of the NORMALISED depth)
  const float* g_w;        // [S] or null
  const float* g_trans;    // [S] or null
  const float* g_alpha;    // [S] or null
  float* g_sigma;          // [S]
  float* g_rgb;            // [S,3] or null
  float depth_eps;
};

__global__ void __launch_bounds__(256) composite_bwd_kernel(CompositeBwdArgs a) {
  for_each_ray_group(a.offsets, a.n_rays, 0, [&](auto g_, int64_t ray, int gl, unsigned gm) {
    constexpr int G = decltype(g_)::value;
    const int64_t s0 = a.offsets[ray], s1 = a.offsets[ray + 1];
    if (s0 >= s1) return;
    // per-ray upstream gradients, folded back through depth normalisation and background blend
    float gcr = 0.f, gcg = 0.f, gcb = 0.f, gO = 0.f, gD = 0.f;
    if (a.g_colors) {
      gcr = a.g_colors[3 * ray];
      gcg = a.g_colors[3 * ray + 1];
      gcb = a.g_colors[3 * ray + 2];
      if (a.bkgd) {
        const float* b = a.bkgd + (int64_t)a.bkgd_stride * ray;
        gO -= gcr * b[0] + gcg * b[1] + gcb * b[2];
      }
    }
    if (a.g_opacity) gO += a.g_opacity[ray];
    if (a.g_depth && a.opacity && a.depth_raw) {
      const float o = a.opacity[ray], gd = a.g_depth[ray];
      const float den = fmaxf(o, a.depth_eps);
      gD = gd / den;
      if (o > a.depth_eps) gO -= gd * a.depth_raw[ray] / (den * den);
    }
    float carry = 0.f;  // sum over later samples of GT_s * T_s
    const int64_t n = s1 - s0;
    const int64_t n_chunks = (n + G - 1) / G;
    for (int64_t c = n_chunks - 1; c >= 0; --c) {
      const int64_t i = s0 + c * G + gl;
      const bool ok = i < s1;
      float T = 0.f, al = 0.f, ta = 0.f, tb = 0.f, r = 0.f, g = 0.f, b = 0.f;
      float gw = 0.f, gT = 0.f, ga = 0.f;
      if (ok) {
        T = a.trans[i];
        al = a.alpha[i];
        ta = a.t0[i];
        tb = a.t1[i];
        if (a.rgb) {
          r = a.rgb[3 * i];
          g = a.rgb[3 * i + 1];
          b = a.rgb[3 * i + 2];
        }
        if (a.g_w) gw = a.g_w[i];
        if (a.g_trans) gT = a.g_trans[i];
        if (a.g_alpha) ga = a.g_alpha[i];
      }
      gw += gcr * r + gcg * g + gcb * b + gO + gD * ((ta + tb) * 0.5f);
      const float GT = gT + gw * al;
      const float GA = ga + gw * T;
      const float v = ok ? GT * T : 0.f;
      const float incl = group_incl_scan_rev<G>(v, gl, gm);
      const float later = carry + (incl - v);
      carry += __shfl_sync(gm, incl, 0, G);
      if (ok) {
        a.g_sigma[i] = (tb - ta) * (GA * (1.f - al) - later);
        if (a.g_rgb) {
          const float w = T * al;
          a.g_rgb[3 * i] = w * gcr;
          a.g_rgb[3 * i + 1] = w * gcg;
          a.g_rgb[3 * i + 2] = w * gcb;
        }
      }
    }
  });
}

// visibility mask of nerfacc's render_visibility_from_density, fused with the scan
__global__ void __launch_bounds__(256)
visibility_kernel(const float* __restrict__ t0, const float* __restrict__ t1, const float* __restrict__ sigma,
                  const int64_t* __restrict__ offsets, int64_t n_rays, float early_stop_eps, float alpha_thre,
                  uint8_t* __restrict__ keep, int32_t* __restrict__ kept_counts) {
  for_each_ray_group(offsets, n_rays, 0, [&](auto g_, int64_t ray, int gl, unsigned gm) {
    constexpr int G = decltype(g_)::value;
    const int64_t s0 = offsets[ray], s1 = offsets[ray + 1];
    float carry = 0.f;
    int kept = 0;
    for (int64_t base = s0; base < s1; base += G) {
      const int64_t i = base + gl;
      const bool ok = i < s1;
      const float sd = ok ? sigma[i] * (t1[i] - t0[i]) : 0.f;
      const float incl = group_incl_scan<G>(sd, gl, gm);
      const float T = expf(-(carry + (incl - sd)));
      const float al = 1.f - expf(-sd);
      carry += __shfl_sync(gm, incl, G - 1, G);
      const bool k = ok && (T >= early_stop_eps) && (alpha_thre <= 0.f || al >= alpha_thre);
      if (ok) keep[i] = k;
      if (kept_counts) kept += __popc(__ballot_sync(gm, k) & gm);
    }
    if (kept_counts && gl == 0) kept_counts[ray] = kept;
  });
}

// Compaction of the visible samples (what OccGridEstimator.sampling returns): every ray's kept samples move, in order,
// to out_starts[ray] + rank.  One group of G lanes per ray; the rank inside a chunk is a popcount of the group's ballot.
template <int G>
__global__ void __launch_bounds__(256)
compact_samples_kernel(const uint8_t* __restrict__ keep, const int64_t* __restrict__ offsets,
                       const int64_t* __restrict__ out_starts, const float* __restrict__ t0, const float* __restrict__ t1,
                       int64_t n_rays, int64_t* __restrict__ ridx_out, float* __restrict__ t0_out,
                       float* __restrict__ t1_out, int capped) {
  const int gl = threadIdx.x % G;
  const unsigned gm = group_mask<G>();
  const int shift = (threadIdx.x & 31) / G * G;
  const int64_t ray = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) / G;
  if (ray >= n_rays) return;
  const int64_t s0 = offsets[ray], s1 = offsets[ray + 1];
  int64_t dst = out_starts[ray];
  // capped: out_starts = offsets [n_rays + 1] clamped to the capacity of the outputs; nothing lands at or beyond the
  // clamped end of the ray's range
  const int64_t dst_end = capped ? out_starts[ray + 1] : INT64_MAX;
  for (int64_t base = s0; base < s1; base += G) {
    const int64_t i = base + gl;
    const bool k = i < s1 && keep[i] != 0;
    const unsigned bits = (__ballot_sync(gm, k) & gm) >> shift;
    if (k && dst + __popc(bits & ((1u << gl) - 1u)) < dst_end) {
      const int64_t o = dst + __popc(bits & ((1u << gl) - 1u));
      ridx_out[o] = ray;
      t0_out[o] = t0[i];
      t1_out[o] = t1[i];
    }
    dst += __popc(bits);
  }
}

// generic per-ray weighted sum of C channels: out[r,c] (+)= sum_s w_s * v[s,c]   (v null -> 1)
__global__ void __launch_bounds__(256, 8)
accumulate_fwd_kernel(const float* __restrict__ w, const float* __restrict__ v, int C,
                      const int64_t* __restrict__ offsets, int64_t n_rays, float* __restrict__ out, int inplace) {
  for_each_ray_group(offsets, n_rays, 0, [&](auto g_, int64_t ray, int gl, unsigned gm) {
    constexpr int G = decltype(g_)::value;
    const int64_t s0 = offsets[ray], s1 = offsets[ray + 1];
    for (int c = 0; c < C; ++c) {
      float acc = 0.f;
      for (int64_t i = s0 + gl; i < s1; i += G) acc += w[i] * (v ? v[i * C + c] : 1.f);
      acc = group_sum<G>(acc, gm);
      if (gl == 0) {
        if (inplace) out[ray * C + c] += acc;
        else out[ray * C + c] = acc;
      }
    }
  });
}

__global__ void accumulate_bwd_kernel(const float* __restrict__ w, const float* __restrict__ v, int C,
                                      const int64_t* __restrict__ ridx, int64_t S, const float* __restrict__ g_out,
                                      float* __restrict__ g_w, float* __restrict__ g_v, const int64_t* __restrict__ S_dev) {
  int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= S || (S_dev && i >= *S_dev)) return;
  const int64_t r = ridx[i];
  const float wi = w[i];
  float acc = 0.f;
  for (int c = 0; c < C; ++c) {
    const float go = g_out[r * C + c];
    acc += go * (v ? v[i * C + c] : 1.f);
    if (g_v) g_v[i * C + c] = wi * go;
  }
  if (g_w) g_w[i] = acc;
}

// wide-channel variants (C in 8..32): one warp per ray / per sample, lane = channel, rows read as coalesced lines
__global__ void __launch_bounds__(256)
accumulate_wide_fwd_kernel(const float* __restrict__ w, const float* __restrict__ v, int C,
                           const int64_t* __restrict__ offsets, int64_t n_rays, float* __restrict__ out, int inplace) {
  const int lane = threadIdx.x & 31;
  const int64_t ray = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
  if (ray >= n_rays || lane >= C) return;
  const int64_t s0 = offsets[ray], s1 = offsets[ray + 1];
  float acc = 0.f;
  for (int64_t i = s0; i < s1; ++i) acc += w[i] * v[i * C + lane];
  if (inplace) out[ray * C + lane] += acc;
  else out[ray * C + lane] = acc;
}

__global__ void __launch_bounds__(256)
accumulate_wide_bwd_kernel(const float* __restrict__ w, const float* __restrict__ v, int C,
                           const int64_t* __restrict__ ridx, int64_t S, const float* __restrict__ g_out,
                           float* __restrict__ g_w, float* __restrict__ g_v, const int64_t* __restrict__ S_dev) {
  const int lane = threadIdx.x & 31;
  const int64_t i = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
  if (i >= S || (S_dev && i >= *S_dev)) return;
  const int64_t r = ridx[i];
  const float go = lane < C ? g_out[r * C + lane] : 0.f;
  if (g_v && lane < C) g_v[i * C + lane] = w[i] * go;
  if (g_w) {
    float acc = lane < C ? go * v[i * C + lane] : 0.f;
    acc = warp_sum(acc);
    if (lane == 0) g_w[i] = acc;
  }
}

// C == 32 (the latent-loss reduction): eight lanes per row with 16-byte accesses, four rays / samples per warp - a
// quarter of the warp instructions of the lane-per-channel kernels above for the same bytes
__global__ void __launch_bounds__(256)
accumulate_c32_fwd_kernel(const float* __restrict__ w, const float4* __restrict__ v, const int64_t* __restrict__ offsets,
                          int64_t n_rays, float4* __restrict__ out, int inplace) {
  const int64_t t = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  const int64_t ray = t >> 3;
  const int c = (int)(t & 7);
  if (ray >= n_rays) return;
  const int64_t s0 = offsets[ray], s1 = offsets[ray + 1];
  float4 acc = make_float4(0.f, 0.f, 0.f, 0.f);
  for (int64_t i = s0; i < s1; ++i) {
    const float wi = w[i];
    const float4 x = v[i * 8 + c];
    acc.x += wi * x.x, acc.y += wi * x.y, acc.z += wi * x.z, acc.w += wi * x.w;
  }
  if (inplace) {
    const float4 o = out[ray * 8 + c];
    acc.x += o.x, acc.y += o.y, acc.z += o.z, acc.w += o.w;
  }
  out[ray * 8 + c] = acc;
}

__global__ void __launch_bounds__(256)
accumulate_c32_bwd_kernel(const float* __restrict__ w, const float4* __restrict__ v, const int64_t* __restrict__ ridx,
                          int64_t S, const float4* __restrict__ g_out, float* __restrict__ g_w, float4* __restrict__ g_v,
                          const int64_t* __restrict__ S_dev) {
  const int64_t t = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  const int64_t i = t >> 3;
  const int c = (int)(t & 7);
  const bool ok = i < S && (!S_dev || i < *S_dev);
  float part = 0.f;
  if (ok) {
    const float4 go = g_out[ridx[i] * 8 + c];
    if (g_v) {
      const float wi = w[i];
      g_v[i * 8 + c] = make_float4(wi * go.x, wi * go.y, wi * go.z, wi * go.w);
    }
    if (g_w) {
      const float4 x = v[i * 8 + c];
      part = go.x * x.x + go.y * x.y + go.z * x.z + go.w * x.w;
    }
  }
  if (g_w) {  // sum over the eight lanes of the row
    part += __shfl_xor_sync(0xffffffffu, part, 4);
    part += __shfl_xor_sync(0xffffffffu, part, 2);
    part += __shfl_xor_sync(0xffffffffu, part, 1);
    if (ok && c == 0) g_w[i] = part;
  }
}

}  // namespace

// kernels that choose their group width on the device: the grid has G lanes per ray for the host's estimate of G
#define LAUNCH_PER_RAY(KERNEL, S_, ...)                                                                      \
  KERNEL<<<cednerf_blocks(n_rays * pick_group(S_, n_rays), 256), 256, 0, st>>>(__VA_ARGS__)

#define DISPATCH_G(G_, KERNEL, ...)                                                          \
  do {                                                                                       \
    const int threads = 256;                                                                 \
    switch (G_) {                                                                            \
      case 4: KERNEL<4><<<cednerf_blocks(n_rays * 4, threads), threads, 0, st>>>(__VA_ARGS__); break;   \
      case 8: KERNEL<8><<<cednerf_blocks(n_rays * 8, threads), threads, 0, st>>>(__VA_ARGS__); break;   \
      case 16: KERNEL<16><<<cednerf_blocks(n_rays * 16, threads), threads, 0, st>>>(__VA_ARGS__); break; \
      default: KERNEL<32><<<cednerf_blocks(n_rays * 32, threads), threads, 0, st>>>(__VA_ARGS__); break; \
    }                                                                                        \
  } while (0)

CEDNERF_EXPORT int cednerf_ray_offsets(const int64_t* ray_indices, int64_t n_samples, int64_t n_rays,
                                       int64_t* offsets, void* stream) {
  CEDNERF_REQUIRE(n_samples >= 0 && n_rays >= 0 && offsets, "bad sizes");
  cudaStream_t st = (cudaStream_t)stream;
  ray_offsets_kernel<<<cednerf_blocks(n_samples + 1, 256), 256, 0, st>>>(ray_indices, n_samples, n_rays, offsets);
  return cednerf_check_launch("cednerf_ray_offsets");
}

CEDNERF_EXPORT int cednerf_composite_fwd(const float* t_starts, const float* t_ends, const float* sigmas,
                                         const float* rgbs, const float* prefix_trans, const int64_t* offsets,
                                         const float* bkgd, int bkgd_stride, int64_t n_samples, int64_t n_rays,
                                         float* weights, float* trans, float* alphas, float* colors, float* opacity,
                                         float* depth, float* depth_raw, int accumulate_inplace, float depth_eps,
                                         void* stream) {
  CEDNERF_REQUIRE(n_rays >= 0 && n_samples >= 0, "bad sizes");
  if (n_rays == 0) return 0;
  cudaStream_t st = (cudaStream_t)stream;
  CompositeFwdArgs a{t_starts, t_ends, sigmas, rgbs, prefix_trans, offsets, bkgd, bkgd_stride, n_rays, weights,
                     trans, alphas, colors, opacity, depth, depth_raw, accumulate_inplace, depth_eps};
  LAUNCH_PER_RAY(composite_fwd_kernel, n_samples, a, 0);
  return cednerf_check_launch("cednerf_composite_fwd");
}

// One marching round of render_image_test with the alive list on the device (cednerf/utils.py:274-304): for every live
// slot, weights with prefix transmittance 1 - opacity[ray], rgb / opacity / depth accumulated in place, and
// alive_flags[slot] = 1 when the ray stays alive (0 for the slots beyond the live part of the list, up to n_bound).
// offsets / slot_counts are indexed by slot (cednerf_exclusive_scan_capped / cednerf_march_round); k_hint sizes the lane
// group per ray.  cednerf_exclusive_scan_capped(alive_flags) + cednerf_render_round_compact then build the next list.
CEDNERF_EXPORT int cednerf_render_round_composite(const float* t_starts, const float* t_ends, const float* sigmas,
                                                  const float* rgbs, const int64_t* offsets, const int32_t* alive,
                                                  int32_t* round_state, const int32_t* slot_counts, int64_t n_bound,
                                                  int k_hint, float early_stop_eps, float* colors, float* opacity,
                                                  float* depth, int32_t* alive_flags, void* stream) {
  CEDNERF_REQUIRE(n_bound >= 0 && offsets && alive && round_state && slot_counts && colors && opacity && depth && alive_flags,
                  "bad arguments");
  if (n_bound == 0) return 0;
  cudaStream_t st = (cudaStream_t)stream;
  CompositeFwdArgs a{t_starts, t_ends, sigmas, rgbs, nullptr, offsets, nullptr, 0, n_bound, nullptr, nullptr, nullptr,
                     colors, opacity, depth, nullptr, 2, 0.f, alive, round_state, slot_counts, early_stop_eps, alive_flags};
  const int64_t n_rays = n_bound;
  // the group width of a round follows k_hint, not the live count: the rounds' launches are fixed in advance
  const int g = pick_group((int64_t)k_hint * n_bound, n_bound);
  composite_fwd_kernel<<<cednerf_blocks(n_rays * g, 256), 256, 0, st>>>(a, g);
  return cednerf_check_launch("cednerf_render_round_composite");
}

namespace {
__global__ void render_round_compact_kernel(const int32_t* __restrict__ flags, const int64_t* __restrict__ pos,
                                            const int32_t* __restrict__ cur, int64_t n_bound, int32_t* __restrict__ state,
                                            int32_t* __restrict__ next, int64_t n_rays, int max_samples, int min_samples,
                                            const int64_t* __restrict__ round_totals, int64_t* __restrict__ total) {
  const int64_t slot = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (slot < n_bound && flags[slot]) next[pos[slot]] = cur[slot];
  if (slot == 0) {   // nobody else in this launch reads the state: start the NEXT round here (saves a launch per round)
    state[3] = (int32_t)pos[n_bound];   // rays alive in the next round
    if (max_samples > 0) cednerf_round_begin(state, n_rays, max_samples, min_samples, round_totals, total);
  }
}
}  // namespace

// next[pos[slot]] = alive[slot] for the flagged slots (pos = exclusive scan of alive_flags, [n_bound + 1]); state[3] <- count
// max_samples > 0: the same launch also performs cednerf_render_round_begin for the next round (with this round's scan
// totals added to *total)
CEDNERF_EXPORT int cednerf_render_round_compact(const int32_t* alive_flags, const int64_t* positions, const int32_t* alive,
                                                int64_t n_bound, int32_t* round_state, int32_t* next_alive, int64_t n_rays,
                                                int max_samples, int min_samples, const int64_t* round_totals,
                                                int64_t* total, void* stream) {
  CEDNERF_REQUIRE(n_bound >= 0 && alive_flags && positions && alive && round_state && next_alive, "bad arguments");
  if (n_bound == 0) return 0;
  render_round_compact_kernel<<<cednerf_blocks(n_bound, 256), 256, 0, (cudaStream_t)stream>>>(
      alive_flags, positions, alive, n_bound, round_state, next_alive, n_rays, max_samples, min_samples, round_totals, total);
  return cednerf_check_launch("cednerf_render_round_compact");
}

CEDNERF_EXPORT int cednerf_composite_bwd(const float* t_starts, const float* t_ends, const float* rgbs,
                                         const float* trans, const float* alphas, const int64_t* offsets,
                                         const float* bkgd, int bkgd_stride, int64_t n_samples, int64_t n_rays,
                                         const float* opacity, const float* depth_raw, const float* g_colors,
                                         const float* g_opacity, const float* g_depth, const float* g_weights,
                                         const float* g_trans, const float* g_alphas, float* g_sigmas, float* g_rgbs,
                                         float depth_eps, void* stream) {
  CEDNERF_REQUIRE(n_rays >= 0 && n_samples >= 0 && (n_samples == 0 || g_sigmas), "bad sizes");
  if (n_rays == 0 || n_samples == 0) return 0;
  cudaStream_t st = (cudaStream_t)stream;
  CompositeBwdArgs a{t_starts, t_ends, rgbs, trans, alphas, offsets, bkgd, bkgd_stride, n_rays, opacity, depth_raw,
                     g_colors, g_opacity, g_depth, g_weights, g_trans, g_alphas, g_sigmas, g_rgbs, depth_eps};
  LAUNCH_PER_RAY(composite_bwd_kernel, n_samples, a);
  return cednerf_check_launch("cednerf_composite_bwd");
}

CEDNERF_EXPORT int cednerf_visibility_mask(const float* t_starts, const float* t_ends, const float* sigmas,
                                           const int64_t* offsets, int64_t n_samples, int64_t n_rays,
                                           float early_stop_eps, float alpha_thre, uint8_t* keep,
                                           int32_t* kept_counts, void* stream) {
  CEDNERF_REQUIRE(n_rays >= 0 && n_samples >= 0, "bad sizes");
  if (n_rays == 0) return 0;
  cudaStream_t st = (cudaStream_t)stream;
  LAUNCH_PER_RAY(visibility_kernel, n_samples, t_starts, t_ends, sigmas, offsets, n_rays,
             early_stop_eps, alpha_thre, keep, kept_counts);
  return cednerf_check_launch("cednerf_visibility_mask");
}

// keep [S] + offsets [n_rays+1] of the marched samples, out_starts [n_rays] = exclusive scan of the per-ray kept counts
// (cednerf_visibility_mask's kept_counts through cednerf_exclusive_scan) -> the kept (ray_indices, t_starts, t_ends).
CEDNERF_EXPORT int cednerf_compact_samples(const uint8_t* keep, const int64_t* offsets, const int64_t* out_starts,
                                           const float* t_starts, const float* t_ends, int64_t n_samples, int64_t n_rays,
                                           int64_t* ray_indices_out, float* t_starts_out, float* t_ends_out,
                                           void* stream) {
  CEDNERF_REQUIRE(n_rays >= 0 && n_samples >= 0 && keep && offsets && out_starts, "bad arguments");
  if (n_rays == 0 || n_samples == 0) return 0;
  cudaStream_t st = (cudaStream_t)stream;
  DISPATCH_G(pick_group(n_samples, n_rays), compact_samples_kernel, keep, offsets, out_starts, t_starts, t_ends, n_rays,
             ray_indices_out, t_starts_out, t_ends_out, 0);
  return cednerf_check_launch("cednerf_compact_samples");
}

// The same compaction into outputs of a fixed capacity: out_offsets [n_rays + 1] from cednerf_exclusive_scan_capped over
// the kept counts (kept samples at or beyond the capacity are dropped); n_samples is only an estimate for the launch shape.
CEDNERF_EXPORT int cednerf_compact_samples_capped(const uint8_t* keep, const int64_t* offsets, const int64_t* out_offsets,
                                                  const float* t_starts, const float* t_ends, int64_t n_samples,
                                                  int64_t n_rays, int64_t* ray_indices_out, float* t_starts_out,
                                                  float* t_ends_out, void* stream) {
  CEDNERF_REQUIRE(n_rays >= 0 && n_samples >= 0 && keep && offsets && out_offsets, "bad arguments");
  if (n_rays == 0) return 0;
  cudaStream_t st = (cudaStream_t)stream;
  DISPATCH_G(pick_group(n_samples, n_rays), compact_samples_kernel, keep, offsets, out_offsets, t_starts, t_ends, n_rays,
             ray_indices_out, t_starts_out, t_ends_out, 1);
  return cednerf_check_launch("cednerf_compact_samples_capped");
}

CEDNERF_EXPORT int cednerf_accumulate_fwd(const float* weights, const float* values, int n_channels,
                                          const int64_t* offsets, int64_t n_samples, int64_t n_rays, float* outputs,
                                          int inplace, void* stream) {
  CEDNERF_REQUIRE(n_rays >= 0 && n_samples >= 0 && n_channels >= 1, "bad sizes");
  if (n_rays == 0) return 0;
  cudaStream_t st = (cudaStream_t)stream;
  if (values && n_channels == 32 && (((uintptr_t)values | (uintptr_t)outputs) & 15) == 0) {
    accumulate_c32_fwd_kernel<<<cednerf_blocks(n_rays * 8, 256), 256, 0, st>>>(
        weights, reinterpret_cast<const float4*>(values), offsets, n_rays, reinterpret_cast<float4*>(outputs), inplace);
    return cednerf_check_launch("cednerf_accumulate_fwd");
  }
  if (values && n_channels >= 8 && n_channels <= 32) {
    accumulate_wide_fwd_kernel<<<cednerf_blocks(n_rays * 32, 256), 256, 0, st>>>(weights, values, n_channels, offsets,
                                                                                 n_rays, outputs, inplace);
    return cednerf_check_launch("cednerf_accumulate_fwd");
  }
  LAUNCH_PER_RAY(accumulate_fwd_kernel, n_samples, weights, values, n_channels, offsets, n_rays,
             outputs, inplace);
  return cednerf_check_launch("cednerf_accumulate_fwd");
}

CEDNERF_EXPORT int cednerf_accumulate_bwd(const float* weights, const float* values, int n_channels,
                                          const int64_t* ray_indices, int64_t n_samples, const float* g_outputs,
                                          float* g_weights, float* g_values, const int64_t* n_device, void* stream) {
  CEDNERF_REQUIRE(n_samples >= 0 && n_channels >= 1, "bad sizes");
  if (n_samples == 0) return 0;
  cudaStream_t st = (cudaStream_t)stream;
  if (values && n_channels == 32 &&
      (((uintptr_t)values | (uintptr_t)g_outputs | (uintptr_t)g_values) & 15) == 0) {
    accumulate_c32_bwd_kernel<<<cednerf_blocks(n_samples * 8, 256), 256, 0, st>>>(
        weights, reinterpret_cast<const float4*>(values), ray_indices, n_samples,
        reinterpret_cast<const float4*>(g_outputs), g_weights, reinterpret_cast<float4*>(g_values), n_device);
    return cednerf_check_launch("cednerf_accumulate_bwd");
  }
  if (values && n_channels >= 8 && n_channels <= 32) {
    accumulate_wide_bwd_kernel<<<cednerf_blocks(n_samples * 32, 256), 256, 0, st>>>(
        weights, values, n_channels, ray_indices, n_samples, g_outputs, g_weights, g_values, n_device);
    return cednerf_check_launch("cednerf_accumulate_bwd");
  }
  accumulate_bwd_kernel<<<cednerf_blocks(n_samples, 256), 256, 0, st>>>(weights, values, n_channels, ray_indices,
                                                                       n_samples, g_outputs, g_weights, g_values, n_device);
  return cednerf_check_launch("cednerf_accumulate_bwd");
}
