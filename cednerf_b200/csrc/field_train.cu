// Fused radiance-field TRAINING step on packed ray samples: one forward kernel (all four networks, hash encode,
// time / SH / Frequency encodings, trunc_exp, sigmoid, huber latent loss) that keeps what the backward needs, and a
// backward made of one tensor-core kernel per network whose prologue / epilogue do the element-wise glue in registers.
//
// Replaces, for the gradient-carrying pass of render_image (cednerf/utils.py:90-104 -> DNGPradianceField.forward,
// cednerf/model.py:468-488 with return_interal=True), the ~120 PyTorch / tcnn launches per step that sit between the
// sampler and rendering(): torch.cat / slicing / casts, tcnn Frequency / SH / HashGrid / 4 x FullyFusedMLP forward and
// backward, huber_loss, tanh, exp, sigmoid and their autograd nodes.
//
// Backward order: colour net -> density net (its epilogue also subtracts the feature predictor's output gradient from
// the hash-feature gradient: the features are that net's huber target) -> hash-table gradient -> feature predictor ->
// dL/dx of the encoding -> deformation net.  Everything after the table gradient can run under its all-reduce.  Gradient dtype flow is tcnn's (DESIGN.md §2): gradients that cross a
// module boundary are fp16, hidden gradients are fp16, weight / table gradients and dL/dx are fp32.
#include <stdlib.h>

#include "field_common.cuh"

namespace {

struct SavedLayout {
  int64_t h1, o1, in2, h2, o2, h3, h4, o4, xn, total, tiles;
};

__host__ __device__ inline SavedLayout saved_layout(const CednerfFieldDesc& d, int64_t n) {
  SavedLayout s;
  int64_t off = 0;
  // hidden activations: tile-blocked, every 128-sample tile as its 16 KB swizzled shared-memory image (one TMA bulk
  // copy out in the forward, one in in the backward), [layer][tile]; everything else row-major per sample
  const int64_t tiles = (n + MLP_TILE - 1) / MLP_TILE;
  s.tiles = tiles;
  s.h1 = off, off += (int64_t)(d.f1.n_layers - 1) * tiles * MLP_TILE_BYTES;
  s.o1 = off, off += n * 32;
  s.in2 = off, off += n * d.f2.dim_in[0] * 2;
  s.h2 = off, off += (int64_t)(d.f2.n_layers - 1) * tiles * MLP_TILE_BYTES;
  s.o2 = off, off += n * 32;
  s.h3 = off, off += (int64_t)(d.f3.n_layers - 1) * tiles * MLP_TILE_BYTES;
  s.h4 = off, off += d.f4.n_layers > 0 ? (int64_t)(d.f4.n_layers - 1) * tiles * MLP_TILE_BYTES : 0;
  s.o4 = off, off += d.f4.n_layers > 0 ? n * 64 : 0;
  s.xn = off, off += (n * 12 + 15) / 16 * 16;
  s.total = off;
  return s;
}

struct BwdWorkLayout {
  int64_t d_o2, d_in2, d_in4, g_xn, dy_lm, total;
};

__host__ __device__ inline BwdWorkLayout bwd_layout(const CednerfFieldDesc& d, int64_t n) {
  BwdWorkLayout w;
  int64_t off = 0;
  w.d_o2 = off, off += n * 32;
  w.d_in2 = off, off += n * d.f2.dim_in[0] * 2;
  w.d_in4 = off, off += n * 64;
  w.g_xn = off, off += (n * 12 + 15) / 16 * 16;
  w.dy_lm = off, off += (int64_t)d.levels.n_levels * n * 4;  // hash-feature gradient, [level][sample] half2
  w.total = off;
  return w;
}

struct TrainArgs {
  const int64_t* ridx;
  const float* t0;
  const float* t1;
  const float* rays_o;
  const float* rays_d;
  const float* t;
  int t_stride;
  int64_t n;             // capacity of the sample arrays: layouts and strides
  const int64_t* n_dev;  // nullable: live sample count on the device (min(n, *n_dev) samples are processed)
  const uint8_t* img[4];
  const __half* table;
  // forward outputs (also read by the backward)
  float* sigma;       // [n]
  float* rgb;         // [n,3]
  float* latent;      // [n,32] or null
  uint8_t* selector;  // [n]
  float* move;        // [n,3]
  uint8_t* saved;
  // backward inputs / outputs
  const float* d_sigma;   // [n]
  const float* d_rgb;     // [n,3]
  const float* d_latent;  // [n,32] or null
  uint8_t* work;
  float* d_params[4];
  uint32_t tmem_cols;
  int flush_tiles;  // > 0: flush the TMEM weight-gradient accumulators every this many tiles of a group
  CednerfFieldDesc d;
};

__device__ __forceinline__ int64_t live_count(const TrainArgs& a) {
  if (!a.n_dev) return a.n;
  const int64_t v = *a.n_dev;
  return v < a.n ? v : a.n;
}

__device__ __forceinline__ float huber(float x) {
  const float ax = fabsf(x);
  return ax < 1.f ? 0.5f * x * x : ax - 0.5f;
}

__device__ __forceinline__ void load_off(const TrainArgs& a, const SavedLayout& sl, int64_t s, float* off6) {
  const uint4 w = *reinterpret_cast<const uint4*>(a.saved + sl.o1 + s * 32);
  const uint32_t ww[4] = {w.x, w.y, w.z, w.w};
#pragma unroll
  for (int j = 0; j < 3; ++j) {
    const float2 f = __half22float2(*reinterpret_cast<const __half2*>(&ww[j]));
    off6[2 * j] = f.x;
    off6[2 * j + 1] = f.y;
  }
}

// -DFIELD_PHASE_CLOCKS (make debug; profiles/tools/exp_field_train.py): cycles per phase of a tile, summed over the first
// thread of every warp-group; slot 11 counts tiles
#ifdef FIELD_PHASE_CLOCKS
__device__ unsigned long long g_train_phase_clocks[12];
#define TPHASE_MARK(i)                                                           \
  do {                                                                           \
    if (gtid == 0) {                                                             \
      const long long now_ = clock64();                                          \
      atomicAdd(&g_train_phase_clocks[i], (unsigned long long)(now_ - phase_t)); \
      phase_t = now_;                                                            \
    }                                                                            \
  } while (0)
#else
#define TPHASE_MARK(i) do {} while (0)
#endif

// =============================================================================================== forward
#ifndef TRAIN_FWD_GROUPS
#define TRAIN_FWD_GROUPS 5   // 128-sample tiles in flight per SM (one warp-group each); measured 4 / 5 / 6 / 7: 0.60 / 0.57 /
                             // 0.63 / 0.64 ms on the 1.01 M visible samples of the DyNeRF-shaped step (96 registers per thread at 5)
#endif
#ifndef TRAIN_FWD_LG
#define TRAIN_FWD_LG 4       // hash levels (8 gathers each) in flight per thread
#endif
__global__ void __launch_bounds__(TRAIN_FWD_GROUPS * 128, 1) field_train_fwd_kernel(TrainArgs a) {
  extern __shared__ __align__(1024) uint8_t smem_raw[];
  uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~(uintptr_t)1023);
  const CednerfFieldDesc& d = a.d;
  const bool has4 = d.f4.n_layers > 0;
  const int n_groups = blockDim.x / MLP_TILE;
  const int tid = threadIdx.x, warp = tid >> 5, group = tid / MLP_TILE, gtid = tid % MLP_TILE;
  uint8_t* w1 = smem;
  uint8_t* w2 = w1 + d.f1.image_bytes;
  uint8_t* w3 = w2 + d.f2.image_bytes;
  uint8_t* w4 = w3 + d.f3.image_bytes;
  uint8_t* abuf = reinterpret_cast<uint8_t*>(
                      (reinterpret_cast<uintptr_t>(w4 + (has4 ? d.f4.image_bytes : 0)) + 1023) & ~(uintptr_t)1023) +
                  (size_t)group * MLP_TILE_BYTES;
  __shared__ uint64_t bars[8];
  __shared__ uint32_t tmem_base_s;
  uint64_t* bar = &bars[group];
  {
    const uint8_t* src[4] = {a.img[0], a.img[1], a.img[2], a.img[3]};
    uint8_t* dst[4] = {w1, w2, w3, w4};
    const int bytes[4] = {d.f1.image_bytes, d.f2.image_bytes, d.f3.image_bytes, has4 ? d.f4.image_bytes : 0};
    for (int k = 0; k < 4; ++k)
      for (int q = tid; q < bytes[k] / 16; q += blockDim.x)
        reinterpret_cast<uint4*>(dst[k])[q] = __ldg(reinterpret_cast<const uint4*>(src[k]) + q);
  }
  const uint32_t tmem_cols = n_groups <= 1 ? 64 : (n_groups == 2 ? 128 : (n_groups <= 4 ? 256 : 512));
  if (warp == 0) tmem_alloc(&tmem_base_s, tmem_cols);
  if (gtid == 0) mbar_init(bar, 1);
  if (tid == 0) fence_barrier_init();
  fence_proxy_async();
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = tmem_base_s + 64u * (uint32_t)group;
  const uint32_t tmem_warp = tmem_base + ((uint32_t)((warp & 3) * 32) << 16);
  uint32_t phase = 0;
  const int64_t n = a.n, nl = live_count(a);
  const int64_t n_tiles = (nl + MLP_TILE - 1) / MLP_TILE;
  const int L = d.levels.n_levels;
  const uint32_t one2 = 0x3C003C00u;
  const SavedLayout sl = saved_layout(d, n);
  const int k2 = d.f2.dim_in[0];

  for (int64_t tile = blockIdx.x + (int64_t)gridDim.x * group; tile < n_tiles; tile += (int64_t)gridDim.x * n_groups) {
    const int64_t s = tile * MLP_TILE + gtid;
    const bool ok = s < nl;
    const int rows_valid = (int)((nl - tile * MLP_TILE) < MLP_TILE ? (nl - tile * MLP_TILE) : MLP_TILE);
    float x[3] = {0.f, 0.f, 0.f}, tv = 0.f;
    int64_t ray = 0;
#ifdef FIELD_PHASE_CLOCKS
    long long phase_t = clock64();
    if (gtid == 0) atomicAdd(&g_train_phase_clocks[11], 1ull);
#endif
    if (ok) packed_sample(a.ridx, a.t0, a.t1, a.rays_o, a.rays_d, a.t, a.t_stride, s, x, tv, ray);
    // ---- deformation net ---------------------------------------------------------------------------------------
    frequency_row<true>(abuf, gtid, x[0], x[1], x[2], tv);
    fence_proxy_async();
    tc_fence_before();
    group_sync(group);
    TPHASE_MARK(0);
    run_chain(d.f1, w1, abuf, tmem_base, tmem_warp, bar, phase, gtid, group, a.saved + sl.h1,
              sl.tiles, tile * MLP_TILE, rows_valid);
    TPHASE_MARK(1);
    float xn[3], mv[3], mvnorm;
    bool selector;
    {
      uint32_t r[16];
      tmem_ld16(tmem_warp, r);
      tmem_ld_wait();
      uint32_t p[8];
#pragma unroll
      for (int j = 0; j < 8; ++j) p[j] = pack_h2(__uint_as_float(r[2 * j]), __uint_as_float(r[2 * j + 1]));
      if (ok) {
        uint4* dst = reinterpret_cast<uint4*>(a.saved + sl.o1 + s * 32);
        dst[0] = make_uint4(p[0], p[1], p[2], p[3]);
        dst[1] = make_uint4(p[4], p[5], p[6], p[7]);
      }
      float off6[6];
#pragma unroll
      for (int k = 0; k < 6; ++k) off6[k] = rnd16(r[k]);
      apply_move(d, x, off6, mv, xn, selector);
      mvnorm = sqrtf(mv[0] * mv[0] + mv[1] * mv[1] + mv[2] * mv[2]);
    }
    if (ok) {
      float* xs = reinterpret_cast<float*>(a.saved + sl.xn) + 3 * s;
      xs[0] = xn[0], xs[1] = xn[1], xs[2] = xn[2];
      a.move[3 * s] = mv[0], a.move[3 * s + 1] = mv[1], a.move[3 * s + 2] = mv[2];
      a.selector[s] = (uint8_t)selector;
    }
    TPHASE_MARK(2);
    // ---- density net input: [hash 2L | time 9 | 1.0 ...] ---------------------------------------------------------
    float temb[9];
    {
      auto put_word = [&](int w, uint32_t v) {
        *reinterpret_cast<uint32_t*>(abuf + swz(gtid, w >> 2) + ((w & 3) << 2)) = v;
      };
      if ((L % TRAIN_FWD_LG) == 0 && (L & 3) == 0) {
#pragma unroll 1
        for (int l0 = 0; l0 < L; l0 += TRAIN_FWD_LG) {
          uint32_t fw[TRAIN_FWD_LG];
          hash_levels<TRAIN_FWD_LG>(xn, a.table, d.levels, 0, fw, l0);
          if constexpr (TRAIN_FWD_LG >= 4) {
#pragma unroll
            for (int q = 0; q < TRAIN_FWD_LG / 4; ++q)
              *reinterpret_cast<uint4*>(abuf + swz(gtid, (l0 >> 2) + q)) = make_uint4(fw[4 * q], fw[4 * q + 1], fw[4 * q + 2], fw[4 * q + 3]);
          } else {
            *reinterpret_cast<uint2*>(abuf + swz(gtid, l0 >> 2) + ((l0 & 2) << 2)) = make_uint2(fw[0], fw[1]);
          }
        }
      } else {
#pragma unroll 1
        for (int l0 = 0; l0 < L; ++l0) {
          uint32_t f1w[1];
          hash_levels<1>(xn, a.table, d.levels, 0, f1w, l0);
          put_word(l0, f1w[0]);
        }
      }
      TPHASE_MARK(3);
      if (d.time_mode) time_embedding<true>(tv, mvnorm, d.time_mode, temb);
      int w = L;
      if (d.time_mode && d.time_before_sigma) {
#pragma unroll
        for (int j = 0; j < 4; ++j) put_word(L + j, pack_h2(temb[2 * j], temb[2 * j + 1]));
        put_word(L + 4, pack_h2(temb[8], 1.f));
        w = L + 5;
      }
      for (; 2 * w < k2; ++w) put_word(w, one2);
    }
    fence_proxy_async();
    tc_fence_before();
    group_sync(group);
    TPHASE_MARK(4);
    // (the density net's input rows are kept too: weight gradient of its first layer, huber target of the predictor)
    run_chain(d.f2, w2, abuf, tmem_base, tmem_warp, bar, phase, gtid, group, a.saved + sl.h2,
              sl.tiles, tile * MLP_TILE, rows_valid, a.saved + sl.in2);
    TPHASE_MARK(5);
    {
      uint32_t o2[16];
      tmem_ld16(tmem_warp, o2);
      tmem_ld_wait();
      uint32_t p[8];
#pragma unroll
      for (int j = 0; j < 8; ++j) p[j] = pack_h2(__uint_as_float(o2[2 * j]), __uint_as_float(o2[2 * j + 1]));
      if (ok) {
        uint4* dst = reinterpret_cast<uint4*>(a.saved + sl.o2 + s * 32);
        dst[0] = make_uint4(p[0], p[1], p[2], p[3]);
        dst[1] = make_uint4(p[4], p[5], p[6], p[7]);
        a.sigma[s] = selector ? expf(rnd16(o2[0]) - 1.f) : 0.f;
      }
      // ---- colour net ------------------------------------------------------------------------------------------
      float dir[3] = {0.f, 0.f, 1.f}, feat15[15];
      if (ok) dir[0] = a.rays_d[3 * ray], dir[1] = a.rays_d[3 * ray + 1], dir[2] = a.rays_d[3 * ray + 2];
#pragma unroll
      for (int j = 0; j < 15; ++j) feat15[j] = rnd16(o2[1 + j]);
      colour_input_row(d, abuf, gtid, dir, feat15, temb);
    }
    fence_proxy_async();
    tc_fence_before();
    group_sync(group);
    TPHASE_MARK(6);
    run_chain(d.f3, w3, abuf, tmem_base, tmem_warp, bar, phase, gtid, group, a.saved + sl.h3,
              sl.tiles, tile * MLP_TILE, rows_valid);
    TPHASE_MARK(7);
    {
      uint32_t r[16];
      tmem_ld16(tmem_warp, r);
      tmem_ld_wait();
      if (ok) {
#pragma unroll
        for (int k = 0; k < 3; ++k) a.rgb[3 * s + k] = 1.f / (1.f + expf(-rnd16(r[k])));
      }
    }
    if (has4) {
      // ---- hash-feature predictor on Frequency(x_norm, t) and its huber loss against the hash features ------------
      frequency_row<true>(abuf, gtid, xn[0], xn[1], xn[2], tv);
      fence_proxy_async();
      tc_fence_before();
      group_sync(group);
      TPHASE_MARK(8);
      run_chain(d.f4, w4, abuf, tmem_base, tmem_warp, bar, phase, gtid, group, a.saved + sl.h4,
                sl.tiles, tile * MLP_TILE, rows_valid);
      TPHASE_MARK(9);
#pragma unroll
      for (int cb = 0; cb < 2; ++cb) {
        uint32_t r[16];
        tmem_ld16(tmem_warp + cb * 16, r);
        tmem_ld_wait();
        if (ok) {
          uint32_t p[8];
#pragma unroll
          for (int j = 0; j < 8; ++j) p[j] = pack_h2(__uint_as_float(r[2 * j]), __uint_as_float(r[2 * j + 1]));
          uint4* dst = reinterpret_cast<uint4*>(a.saved + sl.o4 + s * 64) + 2 * cb;
          dst[0] = make_uint4(p[0], p[1], p[2], p[3]);
          dst[1] = make_uint4(p[4], p[5], p[6], p[7]);
          if (a.latent) {
            const uint4* fsrc = reinterpret_cast<const uint4*>(a.saved + sl.in2 + s * k2 * 2) + 2 * cb;
            const uint4 f0 = fsrc[0], f1 = fsrc[1];
            const uint32_t fw[8] = {f0.x, f0.y, f0.z, f0.w, f1.x, f1.y, f1.z, f1.w};
            float4* lo = reinterpret_cast<float4*>(a.latent + s * 32 + cb * 16);
            float lv[16];
#pragma unroll
            for (int j = 0; j < 8; ++j) {
              const float2 f = __half22float2(*reinterpret_cast<const __half2*>(&fw[j]));
              lv[2 * j] = selector ? huber(rnd16(r[2 * j]) - f.x) : 0.f;
              lv[2 * j + 1] = selector ? huber(rnd16(r[2 * j + 1]) - f.y) : 0.f;
            }
#pragma unroll
            for (int j = 0; j < 4; ++j) lo[j] = make_float4(lv[4 * j], lv[4 * j + 1], lv[4 * j + 2], lv[4 * j + 3]);
          }
        }
      }
    }
    tc_fence_before();
    group_sync(group);
    TPHASE_MARK(10);
  }
  tc_fence_before();
  __syncthreads();
  if (warp == 0) tmem_dealloc(tmem_base_s, tmem_cols);
}

// =============================================================================================== backward
// One network per launch.  NET: 1 deformation, 2 density, 3 colour, 4 feature predictor.  Structure of mlp_bwd_kernel
// (mlp.cu): per 128-sample tile, for each layer from the last: wgrad (M = 64, both operands MN-major, K = 128 samples,
// accumulated in TMEM across the CTA's tiles) and dgrad (B = the forward weight image read MN-major), ReLU mask from the
// saved activations.  What differs per network is how a thread forms its row of the output-gradient tile, its row of the
// network-input tile, and what it does with its row of the input gradient.
template <int NET>
__device__ __forceinline__ const CednerfMlpDesc& net_desc(const CednerfFieldDesc& d) {
  if constexpr (NET == 1) return d.f1;
  else if constexpr (NET == 2) return d.f2;
  else if constexpr (NET == 3) return d.f3;
  else return d.f4;
}

// Output gradient of the feature predictor for 16 of its 32 columns (chunk pair cb of sample s), as 8 packed half2 words:
// dL/dpred = d_latent * huber'(pred - hash_feat) * selector, huber'(x) = clamp(x, -1, 1)  (model.py:435-438).  The hash
// features are the huber target too, so the same words are subtracted from the density net's input gradient.
__device__ __forceinline__ void predictor_dout(const TrainArgs& a, const SavedLayout& sl, int64_t s, int cb, uint32_t* dw) {
  const int k2 = a.d.f2.dim_in[0];
  const uint4* ps = reinterpret_cast<const uint4*>(a.saved + sl.o4 + s * 64) + 2 * cb;
  const uint4* fs = reinterpret_cast<const uint4*>(a.saved + sl.in2 + s * k2 * 2) + 2 * cb;
  const bool sel = a.selector[s] != 0;
#pragma unroll
  for (int c = 0; c < 2; ++c) {
    const uint4 p = ps[c], f = fs[c];
    const uint32_t pw[4] = {p.x, p.y, p.z, p.w}, fw[4] = {f.x, f.y, f.z, f.w};
    const float4 l0 = *reinterpret_cast<const float4*>(a.d_latent + s * 32 + (2 * cb + c) * 8);
    const float4 l1 = *reinterpret_cast<const float4*>(a.d_latent + s * 32 + (2 * cb + c) * 8 + 4);
    const float lg[8] = {l0.x, l0.y, l0.z, l0.w, l1.x, l1.y, l1.z, l1.w};
#pragma unroll
    for (int j = 0; j < 4; ++j) {
      const float2 pv = __half22float2(*reinterpret_cast<const __half2*>(&pw[j]));
      const float2 fv = __half22float2(*reinterpret_cast<const __half2*>(&fw[j]));
      const float d0 = sel ? lg[2 * j] * fminf(fmaxf(pv.x - fv.x, -1.f), 1.f) : 0.f;
      const float d1 = sel ? lg[2 * j + 1] * fminf(fmaxf(pv.y - fv.y, -1.f), 1.f) : 0.f;
      dw[4 * c + j] = pack_h2(d0, d1);
    }
  }
}

template <int NET>
__device__ __forceinline__ void make_dout(const TrainArgs& a, const SavedLayout& sl, const BwdWorkLayout& wl, uint8_t* tile,
                                          int row, int64_t s, bool ok) {
  const CednerfFieldDesc& d = a.d;
  uint32_t w[16];  // up to 32 halves
#pragma unroll
  for (int j = 0; j < 16; ++j) w[j] = 0u;
  // rows past the end are zero-filled over the WHOLE width of this network's output gradient (a stale NaN pattern in
  // shared memory would otherwise meet a zero activation in the weight-gradient MMA: 0 x NaN)
  const int n_chunks = NET == 4 ? 4 : 2;
  if (ok) {
    if constexpr (NET == 3) {
      float g[3];
#pragma unroll
      for (int k = 0; k < 3; ++k) {
        const float c = a.rgb[3 * s + k];
        g[k] = a.d_rgb[3 * s + k] * c * (1.f - c);  // sigmoid backward (model.py:464-465)
      }
      w[0] = pack_h2(g[0], g[1]);
      w[1] = pack_h2(g[2], 0.f);
    } else if constexpr (NET == 2) {
      const uint4* src = reinterpret_cast<const uint4*>(a.work + wl.d_o2 + s * 32);
      const uint4 g0 = src[0], g1 = src[1];
      w[0] = g0.x, w[1] = g0.y, w[2] = g0.z, w[3] = g0.w, w[4] = g1.x, w[5] = g1.y, w[6] = g1.z, w[7] = g1.w;
      const __half raw = *reinterpret_cast<const __half*>(a.saved + sl.o2 + s * 32);
      // trunc_exp backward: g * exp(clamp(raw - 1, max = 15)), times the selector (utils.py:27-43, model.py:414-417)
      const float gs = a.selector[s] ? a.d_sigma[s] * expf(fminf(__half2float(raw) - 1.f, 15.f)) : 0.f;
      const float hi = __half2float(__ushort_as_half((unsigned short)(w[0] >> 16)));
      w[0] = pack_h2(gs, hi);
    } else if constexpr (NET == 4) {
      predictor_dout(a, sl, s, 0, w);
      predictor_dout(a, sl, s, 1, w + 8);
    } else {  // NET == 1: through aabb normalisation, x + move, move = o[:3]*MS + tanh(o[3:])*MS
      const float* gx = reinterpret_cast<const float*>(a.work + wl.g_xn) + 3 * s;
      float g[3] = {gx[0], gx[1], gx[2]};
      if (d.f4.n_layers > 0 && a.d_latent) {  // Frequency backward of the predictor's input (x_norm part)
        const float* xs = reinterpret_cast<const float*>(a.saved + sl.xn) + 3 * s;
        const uint4* src = reinterpret_cast<const uint4*>(a.work + wl.d_in4 + s * 64);
#pragma unroll
        for (int dim = 0; dim < 3; ++dim) {
          const uint4 q = src[dim];
          const uint32_t qw[4] = {q.x, q.y, q.z, q.w};
          float acc = 0.f;
#pragma unroll
          for (int k = 0; k < 4; ++k) {
            const float2 gv = __half22float2(*reinterpret_cast<const __half2*>(&qw[k]));
            const float sc = (float)(1 << k);
            float sn, cs;  // d/dx sin(pi ph) = pi 2^k cos(pi ph); d/dx sin(pi (ph + 1/2)) = -pi 2^k sin(pi ph)
            sincospi_fast(xs[dim] * sc, sn, cs);
            acc += (gv.x * cs - gv.y * sn) * sc * 3.14159265358979323846f;
          }
          g[dim] += acc;
        }
      }
      float off6[6];
      load_off(a, sl, s, off6);
      float o[6] = {0.f, 0.f, 0.f, 0.f, 0.f, 0.f};
#pragma unroll
      for (int k = 0; k < 3; ++k) {
        const float gm = g[k] / (d.aabb[3 + k] - d.aabb[k]);
        o[k] = gm * d.moving_step;
        if (d.use_div_offsets) {
          const float th = tanhf(off6[3 + k]);
          o[3 + k] = gm * d.moving_step * (1.f - th * th);
        }
      }
      w[0] = pack_h2(o[0], o[1]);
      w[1] = pack_h2(o[2], o[3]);
      w[2] = pack_h2(o[4], o[5]);
    }
  }
#pragma unroll
  for (int c = 0; c < 4; ++c)
    if (c < n_chunks) *reinterpret_cast<uint4*>(tile + swz(row, c)) = make_uint4(w[4 * c], w[4 * c + 1], w[4 * c + 2], w[4 * c + 3]);
}

template <int NET>
__device__ __forceinline__ void make_input(const TrainArgs& a, const SavedLayout& sl, uint8_t* tile, int row, int64_t s,
                                           bool ok) {
  const CednerfFieldDesc& d = a.d;
  if (!ok) {  // rows past the end contribute nothing to the weight gradients
    const int chunks = net_desc<NET>(d).dim_in[0] / 8;
    for (int c = 0; c < chunks; ++c) *reinterpret_cast<uint4*>(tile + swz(row, c)) = make_uint4(0u, 0u, 0u, 0u);
    return;
  }
  if constexpr (NET == 2) {
    const int k2 = d.f2.dim_in[0];
    const uint4* src = reinterpret_cast<const uint4*>(a.saved + sl.in2 + s * k2 * 2);
    for (int c = 0; c < k2 / 8; ++c) *reinterpret_cast<uint4*>(tile + swz(row, c)) = src[c];
    return;
  }
  float x[3], tv;
  int64_t ray;
  packed_sample(a.ridx, a.t0, a.t1, a.rays_o, a.rays_d, a.t, a.t_stride, s, x, tv, ray);
  if constexpr (NET == 1) {
    frequency_row<true>(tile, row, x[0], x[1], x[2], tv);
  } else if constexpr (NET == 4) {
    const float* xs = reinterpret_cast<const float*>(a.saved + sl.xn) + 3 * s;
    frequency_row<true>(tile, row, xs[0], xs[1], xs[2], tv);
  } else {  // NET == 3
    float temb[9];
    if (d.time_mode && !d.time_before_sigma) {
      float off6[6], mv[3], xn[3];
      bool sel;
      load_off(a, sl, s, off6);
      apply_move(d, x, off6, mv, xn, sel);
      time_embedding<true>(tv, sqrtf(mv[0] * mv[0] + mv[1] * mv[1] + mv[2] * mv[2]), d.time_mode, temb);
    }
    const uint4* src = reinterpret_cast<const uint4*>(a.saved + sl.o2 + s * 32);
    const uint4 q0 = src[0], q1 = src[1];
    const uint32_t qw[8] = {q0.x, q0.y, q0.z, q0.w, q1.x, q1.y, q1.z, q1.w};
    float o2[16];
#pragma unroll
    for (int j = 0; j < 8; ++j) {
      const float2 f = __half22float2(*reinterpret_cast<const __half2*>(&qw[j]));
      o2[2 * j] = f.x, o2[2 * j + 1] = f.y;
    }
    const float dir[3] = {a.rays_d[3 * ray], a.rays_d[3 * ray + 1], a.rays_d[3 * ray + 2]};
    colour_input_row(d, tile, row, dir, o2 + 1, temb);
  }
}

// Four 128-sample tiles in flight per SM (one warp-group each, one CTA per SM).  Every group owns its tile buffers and
// its input-gradient accumulator; the weight-gradient accumulators are SHARED by the groups: tcgen05.mma instructions
// of a CTA execute in issue order, whichever thread issued them, so D += A*B from different groups onto the same TMEM
// tile is the same read-modify-write chain as the k-loop of one thread.  They are zeroed once (tcgen05.st) and flushed
// once per CTA with fp32 atomics.
#define BWD_GROUPS 4
#define BWD_GROUP_SMEM (3 * MLP_TILE_BYTES)

template <int NET>
__global__ void __launch_bounds__(BWD_GROUPS * MLP_TILE, 1) field_bwd_kernel(TrainArgs a) {
  extern __shared__ __align__(1024) uint8_t smem_raw[];
  uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~(uintptr_t)1023);
  const CednerfMlpDesc& d = net_desc<NET>(a.d);
  const int n_groups = blockDim.x / MLP_TILE;
  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31, group = tid / MLP_TILE, gtid = tid % MLP_TILE;
  uint8_t* wsm = smem;
  uint8_t* gsm = smem + ((d.image_bytes + 1023) & ~1023) + (size_t)group * BWD_GROUP_SMEM;
  uint8_t* gbuf = gsm;  // output-gradient tile of the current layer; the next layer's is written over it in place
  uint8_t* ibuf[2] = {gsm + MLP_TILE_BYTES, gsm + 2 * MLP_TILE_BYTES};
  __shared__ uint64_t bars[BWD_GROUPS];
  __shared__ uint32_t tmem_base_s;
  uint64_t* bar = &bars[group];
  const int64_t n = a.n, nl = live_count(a);
  const SavedLayout sl = saved_layout(a.d, n);
  const BwdWorkLayout wl = bwd_layout(a.d, n);
  const uint8_t* image = a.img[NET - 1];
  const uint8_t* hidden = a.saved + (NET == 1 ? sl.h1 : (NET == 2 ? sl.h2 : (NET == 3 ? sl.h3 : sl.h4)));
  __shared__ uint64_t lbars[BWD_GROUPS];  // completion of the TMA loads of this group's activation tiles
  uint64_t* lbar = &lbars[group];
  uint32_t lphase = 0;
  // one elected thread fetches the saved 16 KB tile image (layer, tile) into an operand buffer with one bulk copy
  auto fetch_tile = [&](uint8_t* dst, int layer, int64_t tile_idx) {
    if (gtid == 0) {
      asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(lbar)), "r"((uint32_t)MLP_TILE_BYTES)
                   : "memory");
      asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(smem_u32(dst)),
                   "l"(hidden + ((int64_t)layer * sl.tiles + tile_idx) * MLP_TILE_BYTES), "r"((uint32_t)MLP_TILE_BYTES),
                   "r"(smem_u32(lbar))
                   : "memory");
    }
  };
  auto await_tile = [&]() {  // every thread of the group: the fetched tile is in shared memory
    mbar_wait(lbar, lphase);
    lphase ^= 1;
  };
  float* d_params = a.d_params[NET - 1];
  const int L = d.n_layers;
  for (int q = tid; q < d.image_bytes / 16; q += blockDim.x)
    reinterpret_cast<uint4*>(wsm)[q] = __ldg(reinterpret_cast<const uint4*>(image) + q);
  if (warp == 0) tmem_alloc(&tmem_base_s, a.tmem_cols);
  if (gtid == 0) {
    mbar_init(bar, 1);
    mbar_init(lbar, 1);
  }
  if (tid == 0) fence_barrier_init();
  fence_proxy_async();
  tc_fence_before();
  __syncthreads();
  if (gtid == 0) fence_barrier_init();
  tc_fence_after();
  const uint32_t tmem_base = tmem_base_s;
  const uint32_t tmem_grp = tmem_base + 64u * (uint32_t)group;                    // dgrad accumulator of this group
  const uint32_t tmem_warp = tmem_grp + ((uint32_t)((warp & 3) * 32) << 16);
  const uint32_t wg_base = tmem_base + 64u * (uint32_t)n_groups;                  // shared wgrad accumulators
  const uint32_t wg_warp = wg_base + ((uint32_t)((warp & 3) * 32) << 16);
  if (group == 0) {
    for (int cb = 0; cb < 4 * ((L + 1) / 2); ++cb) tmem_st16_fill(wg_warp + cb * 16, 0u);
    tmem_st_wait();
  }
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  uint32_t phase = 0;
  const int64_t n_tiles = (nl + MLP_TILE - 1) / MLP_TILE;
  const bool want_dx = NET != 1;  // the deformation net's input (x, t) carries no gradient

  // flush: TMEM weight-gradient accumulators -> d_params (fp32 atomics); with rezero the accumulation starts over
  auto flush_wgrad = [&](bool rezero) {
    if (group == 0) {
      for (int l = 0; l < L; ++l) {
        const int K_in = d.dim_in[l], N_out = d.dim_out[l];
        const int half = l & 1;                       // which 16-lane half of the sub-partition holds this layer
        const int m = warp * 16 + (lane & 15);
        for (int cb = 0; cb < K_in / 16; ++cb) {
          uint32_t r[16];
          tmem_ld16(wg_warp + 64u * (uint32_t)(l >> 1) + cb * 16, r);
          tmem_ld_wait();
          if ((lane >> 4) == half && m < N_out) {
            float* dst = d_params + d.param_off[l] + m * K_in + cb * 16;
#pragma unroll
            for (int j = 0; j < 16; ++j) atomicAdd(dst + j, __uint_as_float(r[j]));
          }
        }
      }
      if (rezero) {
        for (int cb = 0; cb < 4 * ((L + 1) / 2); ++cb) tmem_st16_fill(wg_warp + cb * 16, 0u);
        tmem_st_wait();
      }
      tc_fence_before();
    }
  };
  const int64_t stride = (int64_t)gridDim.x * n_groups;
  const int64_t first = blockIdx.x + (int64_t)gridDim.x * group;
  // the same trip count for every group of the CTA (the periodic flush below synchronises the whole CTA)
  const int64_t n_iter = (n_tiles - blockIdx.x + stride - 1) / stride;
  for (int64_t it = 0; it < n_iter; ++it) {
    const int64_t tile = first + it * stride;
    if (a.flush_tiles > 0 && it > 0 && (it % a.flush_tiles) == 0) {
      tc_fence_before();
      __syncthreads();
      tc_fence_after();
      flush_wgrad(true);
      __syncthreads();
      tc_fence_after();
    }
    if (tile >= n_tiles) continue;
    const int64_t row0 = tile * MLP_TILE;
    const int rows_valid = (int)((nl - row0) < MLP_TILE ? (nl - row0) : MLP_TILE);
    const int64_t s = row0 + gtid;
    const bool ok = gtid < rows_valid;
    if (L > 1) fetch_tile(ibuf[0], L - 2, tile);
    else make_input<NET>(a, sl, ibuf[0], gtid, s, ok);
    make_dout<NET>(a, sl, wl, gbuf, gtid, s, ok);
    if (L > 1) await_tile();
    fence_proxy_async();
    tc_fence_before();
    group_sync(group);
    int cur = 0;
    for (int l = L - 1; l >= 0; --l) {
      const int K_in = d.dim_in[l], N_out = d.dim_out[l];
      const bool need_dgrad = (l > 0) || want_dx;
      if (gtid == 0) {
        tc_fence_after();
        {
          const uint64_t ad = make_desc(smem_u32(gbuf), 64, 64);
          const uint64_t bd = make_desc(smem_u32(ibuf[cur]), 64, 64);
          const uint32_t id = make_idesc(64, K_in, 1, 1);
          // M = 64 accumulators occupy 16 of the 32 lanes of each TMEM sub-partition: two layers share a column block
          const uint32_t acc = wg_base + 64u * (uint32_t)(l >> 1) + ((uint32_t)((l & 1) * 16) << 16);
          for (int k = 0; k < MLP_TILE / 16; ++k) umma(acc, ad + 128 * k, bd + 128 * k, id, 1u);
        }
        if (need_dgrad) {
          const uint64_t ad = make_desc(smem_u32(gbuf), 1, 64);
          const uint64_t bd = make_desc(smem_u32(wsm + d.image_off[l]), 64, 64);
          const uint32_t id = make_idesc(128, K_in, 0, 1);
          for (int k = 0; k < N_out / 16; ++k) umma(tmem_grp, ad + 2 * k, bd + 128 * k, id, k > 0);
        }
        umma_commit(bar);
      }
      if (l > 0) {
        if (l > 1) fetch_tile(ibuf[cur ^ 1], l - 2, tile);
        else make_input<NET>(a, sl, ibuf[cur ^ 1], gtid, s, ok);
      }
      if ((gtid >> 5) == 0) {  // one polling warp per group, the others block on the named barrier
        mbar_wait(bar, phase);
        tc_fence_after();
        tc_fence_before();
      }
      group_sync(group);
      phase ^= 1;
      tc_fence_after();
      if (l > 0) {
        const uint8_t* act = ibuf[cur];
#pragma unroll
        for (int cb = 0; cb < 4; ++cb) {
          uint32_t r[16];
          tmem_ld16(tmem_warp + cb * 16, r);
          tmem_ld_wait();
          const uint4 m0 = *reinterpret_cast<const uint4*>(act + swz(gtid, 2 * cb));
          const uint4 m1 = *reinterpret_cast<const uint4*>(act + swz(gtid, 2 * cb + 1));
          const uint32_t mw[8] = {m0.x, m0.y, m0.z, m0.w, m1.x, m1.y, m1.z, m1.w};
          uint32_t p[8];
#pragma unroll
          for (int j = 0; j < 8; ++j) {
            // ReLU mask from the saved post-ReLU activations: one packed compare (0xffff per half that is > 0) and
            // one AND on the packed gradient - exact zeroing, three instructions per pair of elements
            const unsigned keep = __hgt2_mask(*reinterpret_cast<const __half2*>(&mw[j]), __float2half2_rn(0.f));
            p[j] = pack_h2(__uint_as_float(r[2 * j]), __uint_as_float(r[2 * j + 1])) & keep;
          }
          // in place: every MMA that read this tile has completed, and a thread only touches its own row
          *reinterpret_cast<uint4*>(gbuf + swz(gtid, 2 * cb)) = make_uint4(p[0], p[1], p[2], p[3]);
          *reinterpret_cast<uint4*>(gbuf + swz(gtid, 2 * cb + 1)) = make_uint4(p[4], p[5], p[6], p[7]);
        }
      } else if (want_dx) {
        if constexpr (NET == 3) {
          // keep only the gradient of the 15 geometry features (columns 4..18 of the colour-net input): it becomes
          // columns 1..15 of the density net's output gradient; column 0 (sigma) is filled by that net's prologue
          uint32_t r0[16], r1[16];
          tmem_ld16(tmem_warp, r0);
          tmem_ld16(tmem_warp + 16, r1);
          tmem_ld_wait();
          if (ok) {
            float v[16];
            v[0] = 0.f;
#pragma unroll
            for (int j = 1; j <= 12; ++j) v[j] = __uint_as_float(r0[3 + j]);
#pragma unroll
            for (int j = 13; j <= 15; ++j) v[j] = __uint_as_float(r1[j - 13]);
            uint4* dst = reinterpret_cast<uint4*>(a.work + wl.d_o2 + s * 32);
            dst[0] = make_uint4(pack_h2(v[0], v[1]), pack_h2(v[2], v[3]), pack_h2(v[4], v[5]), pack_h2(v[6], v[7]));
            dst[1] = make_uint4(pack_h2(v[8], v[9]), pack_h2(v[10], v[11]), pack_h2(v[12], v[13]), pack_h2(v[14], v[15]));
          }
        } else {
          uint8_t* out = a.work + (NET == 2 ? wl.d_in2 + s * K_in * 2 : wl.d_in4 + s * 64);
          for (int cb = 0; cb < K_in / 16; ++cb) {
            uint32_t r[16];
            tmem_ld16(tmem_warp + cb * 16, r);
            tmem_ld_wait();
            if (ok) {
              uint32_t p[8];
#pragma unroll
              for (int j = 0; j < 8; ++j) p[j] = pack_h2(__uint_as_float(r[2 * j]), __uint_as_float(r[2 * j + 1]));
              if constexpr (NET == 2) {
                // the hash features are also the huber target of the feature predictor: its output gradient is
                // subtracted here, so the table gradient does not have to wait for the predictor's backward kernel
                if (a.d.f4.n_layers > 0 && a.d_latent && cb < 2) {
                  uint32_t dw[8];
                  predictor_dout(a, sl, s, cb, dw);
#pragma unroll
                  for (int j = 0; j < 8; ++j) {
                    const __half2 q = __hsub2(*reinterpret_cast<const __half2*>(&p[j]), *reinterpret_cast<const __half2*>(&dw[j]));
                    p[j] = *reinterpret_cast<const uint32_t*>(&q);
                  }
                }
                // level-major hash-feature gradient for the table-gradient and dL/dx kernels (nothing else reads the
                // density net's input gradient)
                uint32_t* lm = reinterpret_cast<uint32_t*>(a.work + wl.dy_lm);
#pragma unroll
                for (int j = 0; j < 8; ++j)
                  if (8 * cb + j < a.d.levels.n_levels) lm[(int64_t)(8 * cb + j) * n + s] = p[j];
              } else {
                reinterpret_cast<uint4*>(out)[2 * cb] = make_uint4(p[0], p[1], p[2], p[3]);
                reinterpret_cast<uint4*>(out)[2 * cb + 1] = make_uint4(p[4], p[5], p[6], p[7]);
              }
            }
          }
        }
      }
      if (l > 1) await_tile();  // the prefetched next-layer tile has landed
      fence_proxy_async();
      tc_fence_before();
      group_sync(group);
      cur ^= 1;
    }
  }
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  flush_wgrad(false);  // every CTA added into zero-initialised accumulators: flush them all (zeros where it had no tile)
  __syncthreads();
  if (warp == 0) tmem_dealloc(tmem_base, a.tmem_cols);
}

// dL/dx_norm of the hash encoding from the level-major feature gradient (tcnn's kernel_grid_backward_input form,
// SURVEY.md E2q): one thread per sample walks all levels with the gather arithmetic of the forward (two levels = 16
// gathers in flight), reads its 4 bytes of dy per level coalesced, keeps the three sums in registers and writes them
// once.  Replaces the (sample, level)-per-thread kernel of hashgrid.cu on this path (0.38 ms -> see profiles/).
__global__ void __launch_bounds__(256) hashgrid_bwd_input_lm_kernel(const float* __restrict__ xn, int64_t n,
                                                                    const __half* __restrict__ table, CednerfGridLevels lv,
                                                                    const __half2* __restrict__ dy_lm, float* __restrict__ g_x,
                                                                    const int64_t* __restrict__ n_dev) {
  const int64_t s = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (s >= n || (n_dev && s >= *n_dev)) return;
  const float x[3] = {xn[3 * s], xn[3 * s + 1], xn[3 * s + 2]};
  float gx[3] = {0.f, 0.f, 0.f};
  const int L = lv.n_levels;
  auto level_terms = [&](const float* f, const __half2* v, int l) {
    const float2 d = __half22float2(dy_lm[(int64_t)l * n + s]);
    float dot[8];
#pragma unroll
    for (int k = 0; k < 8; ++k) {
      const float2 t = __half22float2(v[k]);
      dot[k] = t.x * d.x + t.y * d.y;
    }
    const float wx[2] = {1.f - f[0], f[0]}, wy[2] = {1.f - f[1], f[1]}, wz[2] = {1.f - f[2], f[2]};
    float a[3] = {0.f, 0.f, 0.f};
#pragma unroll
    for (int q = 0; q < 2; ++q)
#pragma unroll
      for (int p = 0; p < 2; ++p) {
        a[0] += wy[p] * wz[q] * (dot[1 + 2 * p + 4 * q] - dot[0 + 2 * p + 4 * q]);
        a[1] += wx[p] * wz[q] * (dot[p + 2 + 4 * q] - dot[p + 0 + 4 * q]);
        a[2] += wx[p] * wy[q] * (dot[p + 2 * q + 4] - dot[p + 2 * q]);
      }
    const float sc = lv.scale[l];
    gx[0] += a[0] * sc, gx[1] += a[1] * sc, gx[2] += a[2] * sc;
  };
  int l0 = 0;
#pragma unroll 1
  for (; l0 + 2 <= L; l0 += 2) {
    float frac[2][3];
    __half2 v[2][8];
    hash_issue<2>(x, table, lv, l0, frac, v);
    level_terms(frac[0], v[0], l0);
    level_terms(frac[1], v[1], l0 + 1);
  }
  if (l0 < L) {
    float frac[1][3];
    __half2 v[1][8];
    hash_issue<1>(x, table, lv, l0, frac, v);
    level_terms(frac[0], v[0], l0);
  }
  g_x[3 * s] = gx[0], g_x[3 * s + 1] = gx[1], g_x[3 * s + 2] = gx[2];
}

constexpr int BWD_SMEM_MAX = 226 * 1024;  // 227 KB opt-in limit minus the kernel's 1 KB of static shared memory

int check_train_desc(const CednerfFieldDesc* d) {
  if (!d) return 0;
  const int L = d->levels.n_levels;
  if (L < 1 || L > 16 || d->time_mode < 0 || d->time_mode > 2) return 0;
  const CednerfMlpDesc* nets[4] = {&d->f1, &d->f2, &d->f3, &d->f4};
  for (int k = 0; k < 4; ++k) {
    const int nl = nets[k]->n_layers;
    if (k == 3 && nl == 0) continue;
    if (nl < 1 || nl > MLP_MAX_LAYERS) return 0;
  }
  if (d->f1.dim_in[0] != 32 || d->f1.dim_out[d->f1.n_layers - 1] != 16) return 0;
  const int in2 = 2 * L + ((d->time_mode && d->time_before_sigma) ? 9 : 0);
  if (d->f2.dim_in[0] != (in2 + 15) / 16 * 16 || d->f2.dim_out[d->f2.n_layers - 1] != 16) return 0;
  const int in3 = 19 + ((d->time_mode && !d->time_before_sigma) ? 9 : 0);
  if (d->f3.dim_in[0] != (in3 + 15) / 16 * 16 || d->f3.dim_out[d->f3.n_layers - 1] != 16) return 0;
  if (d->f4.n_layers > 0 && (L != 16 || d->f4.dim_in[0] != 32 || d->f4.dim_out[d->f4.n_layers - 1] != 32)) return 0;
  return 1;
}

template <int NET>
int launch_bwd(TrainArgs a, cudaStream_t st) {
  static CednerfOncePerDevice configured;
  if (int e = cednerf_opt_in_smem(field_bwd_kernel<NET>, BWD_SMEM_MAX, configured, "cednerf_field_train_bwd")) return e;
  const CednerfMlpDesc& d = NET == 1 ? a.d.f1 : (NET == 2 ? a.d.f2 : (NET == 3 ? a.d.f3 : a.d.f4));
  int groups = BWD_GROUPS;  // as many tiles in flight as shared memory (weights + 48 KB per group) and TMEM allow
  if (const char* env = getenv("CEDNERF_BWD_GROUPS")) {  // diagnostic: 1 = no weight-gradient accumulator is shared
    const int g = atoi(env);
    if (g >= 1 && g < groups) groups = g;
  }
  const int fixed = ((d.image_bytes + 1023) & ~1023) + 2048;
  while (groups > 1 && (fixed + groups * BWD_GROUP_SMEM > BWD_SMEM_MAX || 64 * (groups + (d.n_layers + 1) / 2) > 512)) --groups;
  uint32_t cols = 64u * (uint32_t)(groups + (d.n_layers + 1) / 2), alloc = 64;
  while (alloc < cols) alloc <<= 1;
  a.tmem_cols = alloc;
  a.flush_tiles = 0;
  if (const char* env = getenv("CEDNERF_BWD_FLUSH_TILES")) a.flush_tiles = atoi(env);
  const int64_t tiles = (a.n + MLP_TILE - 1) / MLP_TILE;
  const int64_t max_ctas = (int64_t)cednerf_num_sms();
  field_bwd_kernel<NET><<<(unsigned)(tiles < max_ctas ? tiles : max_ctas), groups * MLP_TILE, fixed + groups * BWD_GROUP_SMEM, st>>>(a);
  return 0;
}

}  // namespace

// hash-grid backward of hashgrid.cu (table gradient with run aggregation, dL/dx)
extern "C" int cednerf_hashgrid_bwd_table_lm_dev(const float* x, int x_stride, int64_t n, const int64_t* n_device,
                                                 const CednerfGridLevels* levels, const void* dy_lm_f16, float* g_table,
                                                 void* stream);
extern "C" int cednerf_hashgrid_bwd(const float* x, int x_stride, int64_t n, const void* table_f16,
                                    const CednerfGridLevels* levels, const void* dy, int dy_stride, int dy_is_f16,
                                    float* g_table, float* g_x, void* stream);

CEDNERF_EXPORT int64_t cednerf_field_saved_bytes(const CednerfFieldDesc* desc, int64_t n) {
  return desc ? saved_layout(*desc, n).total : -1;
}
CEDNERF_EXPORT int64_t cednerf_field_bwd_workspace_bytes(const CednerfFieldDesc* desc, int64_t n) {
  return desc ? bwd_layout(*desc, n).total : -1;
}

// DNGPradianceField.forward (training, return_interal=True) on packed ray samples, keeping activations in `saved`
// (cednerf_field_saved_bytes).  latent == NULL or desc->f4.n_layers == 0: no feature predictor.
CEDNERF_EXPORT int cednerf_field_train_fwd(const int64_t* ray_indices, const float* t_starts, const float* t_ends,
                                           const float* rays_o, const float* rays_d, const float* timestamps,
                                           int t_stride, int64_t n, const void* image_deform, const void* image_density,
                                           const void* image_colour, const void* image_predict, const void* table_f16,
                                           const CednerfFieldDesc* desc, float* sigma, float* rgb, float* latent,
                                           uint8_t* selector, float* move, void* saved, const int64_t* n_device,
                                           void* stream) {
  CEDNERF_REQUIRE(check_train_desc(desc), "bad field descriptor");
  CEDNERF_REQUIRE(n >= 0 && ray_indices && t_starts && t_ends && rays_o && rays_d && timestamps && sigma && rgb &&
                      selector && move && saved,
                  "bad arguments");
  CEDNERF_REQUIRE(desc->f4.n_layers == 0 || image_predict, "feature predictor image missing");
  if (n == 0) return 0;
  const int n_groups = TRAIN_FWD_GROUPS;  // one CTA per SM: the tiles in flight (one warp-group each) share one copy of the weight images
  const int smem = desc->f1.image_bytes + desc->f2.image_bytes + desc->f3.image_bytes +
                   (desc->f4.n_layers > 0 ? desc->f4.image_bytes : 0) + n_groups * MLP_TILE_BYTES + 2048;
  CEDNERF_REQUIRE(smem <= 224 * 1024, "networks too large for the fused kernel");
  static CednerfOncePerDevice configured;
  if (int e = cednerf_opt_in_smem(field_train_fwd_kernel, 224 * 1024, configured, "cednerf_field_train_fwd")) return e;
  TrainArgs a{};
  a.ridx = ray_indices, a.t0 = t_starts, a.t1 = t_ends, a.rays_o = rays_o, a.rays_d = rays_d, a.t = timestamps;
  a.t_stride = t_stride, a.n = n, a.n_dev = n_device;
  a.img[0] = (const uint8_t*)image_deform, a.img[1] = (const uint8_t*)image_density;
  a.img[2] = (const uint8_t*)image_colour, a.img[3] = (const uint8_t*)image_predict;
  a.table = (const __half*)table_f16;
  a.sigma = sigma, a.rgb = rgb, a.latent = desc->f4.n_layers > 0 ? latent : nullptr, a.selector = selector, a.move = move;
  a.saved = (uint8_t*)saved;
  a.d = *desc;
  const int64_t tiles = (n + MLP_TILE - 1) / MLP_TILE;
  const int64_t ctas = tiles;  // tiles go round-robin over CTAs first, then over the groups of a CTA
  const int64_t max_ctas = (int64_t)cednerf_num_sms();
  field_train_fwd_kernel<<<(unsigned)(ctas < max_ctas ? ctas : max_ctas), n_groups * MLP_TILE, smem, (cudaStream_t)stream>>>(a);
  return cednerf_check_launch("cednerf_field_train_fwd");
}

// Backward of cednerf_field_train_fwd.  d_params_* and g_table are ACCUMULATED into (caller zeroes); work from
// cednerf_field_bwd_workspace_bytes.  d_latent == NULL: no gradient through the latent loss.
CEDNERF_EXPORT int cednerf_field_train_bwd(const int64_t* ray_indices, const float* t_starts, const float* t_ends,
                                           const float* rays_o, const float* rays_d, const float* timestamps,
                                           int t_stride, int64_t n, const void* image_deform, const void* image_density,
                                           const void* image_colour, const void* image_predict, const void* table_f16,
                                           const CednerfFieldDesc* desc, const float* sigma, const float* rgb,
                                           const uint8_t* selector, const void* saved, const float* d_sigma,
                                           const float* d_rgb, const float* d_latent, void* work, float* d_params_deform,
                                           float* d_params_density, float* d_params_colour, float* d_params_predict,
                                           float* g_table, int phase, const int64_t* n_device, void* stream) {
  CEDNERF_REQUIRE(check_train_desc(desc), "bad field descriptor");
  CEDNERF_REQUIRE(phase >= 0 && phase <= 2, "phase: 0 all, 1 up to the table gradient, 2 the rest");
  CEDNERF_REQUIRE(n >= 0 && ray_indices && t_starts && t_ends && rays_o && rays_d && timestamps && rgb && selector &&
                      saved && d_sigma && d_rgb && work && d_params_deform && d_params_density && d_params_colour &&
                      g_table,
                  "bad arguments");
  const bool has4 = desc->f4.n_layers > 0 && d_latent != nullptr;
  CEDNERF_REQUIRE(!has4 || (image_predict && d_params_predict), "feature predictor buffers missing");
  if (n == 0) return 0;
  cudaStream_t st = (cudaStream_t)stream;
  TrainArgs a{};
  a.ridx = ray_indices, a.t0 = t_starts, a.t1 = t_ends, a.rays_o = rays_o, a.rays_d = rays_d, a.t = timestamps;
  a.t_stride = t_stride, a.n = n, a.n_dev = n_device;
  a.img[0] = (const uint8_t*)image_deform, a.img[1] = (const uint8_t*)image_density;
  a.img[2] = (const uint8_t*)image_colour, a.img[3] = (const uint8_t*)image_predict;
  a.table = (const __half*)table_f16;
  a.sigma = const_cast<float*>(sigma), a.rgb = const_cast<float*>(rgb), a.selector = const_cast<uint8_t*>(selector);
  a.saved = (uint8_t*)saved;
  a.d_sigma = d_sigma, a.d_rgb = d_rgb, a.d_latent = d_latent, a.work = (uint8_t*)work;
  a.d_params[0] = d_params_deform, a.d_params[1] = d_params_density, a.d_params[2] = d_params_colour;
  a.d_params[3] = d_params_predict;
  a.d = *desc;
  const SavedLayout sl = saved_layout(*desc, n);  // offsets follow the FORWARD's descriptor
  const BwdWorkLayout wl = bwd_layout(*desc, n);
  int rc, launches = 0;
  const float* xn = reinterpret_cast<const float*>((const uint8_t*)saved + sl.xn);
  float* g_xn = reinterpret_cast<float*>((uint8_t*)work + wl.g_xn);
  if (phase != 2) {
    if ((rc = launch_bwd<3>(a, st))) return rc;
    if ((rc = launch_bwd<2>(a, st))) return rc;
    launches += 2;
    rc = cednerf_hashgrid_bwd_table_lm_dev(xn, 3, n, n_device, &desc->levels, (const uint8_t*)work + wl.dy_lm, g_table, stream);
    if (rc) return rc;
    // g_table is complete here: with phase == 1 the caller can start its all-reduce while phase 2 runs
    if (phase == 1) return cednerf_check_launch("cednerf_field_train_bwd", launches);
  }
  if (has4) {  // the predictor's own backward (its weight gradients and dL/dx_norm through its Frequency input)
    if ((rc = launch_bwd<4>(a, st))) return rc;
    ++launches;
  }
  hashgrid_bwd_input_lm_kernel<<<cednerf_blocks(n, 256), 256, 0, st>>>(
      xn, n, (const __half*)table_f16, desc->levels, reinterpret_cast<const __half2*>((const uint8_t*)work + wl.dy_lm), g_xn,
      n_device);
  if ((rc = launch_bwd<1>(a, st))) return rc;
  return cednerf_check_launch("cednerf_field_train_bwd", launches + 2);
}

#ifdef FIELD_PHASE_CLOCKS
// debug build only: the accumulated phase clocks of the training forward (12 x uint64 on the host), cleared on read
CEDNERF_EXPORT int cednerf_debug_train_phase_clocks(unsigned long long* out) {
  unsigned long long zero[12] = {0};
  if (cudaMemcpyFromSymbol(out, g_train_phase_clocks, sizeof(zero)) != cudaSuccess) return 1;
  return cudaMemcpyToSymbol(g_train_phase_clocks, zero, sizeof(zero)) != cudaSuccess;
}
#endif
