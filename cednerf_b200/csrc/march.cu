// K1 — occupancy-grid ray marching (count -> device scan -> fill), ray/aabb slab test and boundary sort.
//
// Same per-ray algorithm as the nerfacc calls the reference makes:
//   ray_aabb_intersect   cednerf/utils.py:215
//   sort of boundaries   cednerf/utils.py:219-225
//   traverse_grids       cednerf/utils.py:241-264 (eval: steps limit + over-allocate + ray mask),
//                        and inside OccGridEstimator.sampling, cednerf/utils.py:115-125 (train: two pass)
// restated in SURVEY.md Appendix A.4-A.6.  This translation unit is compiled with -fmad=false: every
// fp32 operation is individually rounded in the order oracle/march_oracle.c fixes, which is what makes
// per-ray sample counts, ray_indices and the packed t values bit-comparable with the oracle.
// Occupancy is read from a bit-packed copy of `binaries` (1 bit/cell, same x*R*R+y*R+z order): 1 MB for
// 4x128^3, L1/L2 resident.  One thread per ray; per-ray counts are turned into packed offsets by a
// three-kernel device scan so that no host round trip sits between count and fill.
#include "common.cuh"

#define MARCH_MAX_LEVELS 8

namespace {

struct MarchArgs {
  const float* rays_o;
  const float* rays_d;
  int64_t n_rays;
  const uint32_t* occ_bits;
  const float* aabbs;  // [L,6]
  int n_levels;
  int res;
  const float* near;  // [n] or null -> near_const
  const float* far;   // [n] or null -> far_const
  float near_const, far_const;
  float step_size, cone_angle;
  int limit;
  const uint8_t* mask;       // [n] or null
  const float* t_sorted;     // [n,2L] or null (computed in-kernel)
  const int64_t* t_indices;  // [n,2L] or null
  const uint8_t* hits;       // [n,L] or null
  // fill-pass inputs
  const int64_t* iv_starts;
  const int64_t* sm_starts;
  // nerfacc-shaped outputs (nullable)
  float* iv_vals;
  uint8_t* iv_left;
  uint8_t* iv_right;
  int64_t* iv_ray;
  float* sm_vals;
  int64_t* sm_ray;
  uint8_t* sm_valid;
  // packed outputs (nullable)
  float* t_starts;
  float* t_ends;
  int64_t* ray_indices;
  // per-ray outputs (nullable)
  int32_t* n_intervals;
  int32_t* n_samples;
  float* termination;
  // run recording (count pass, nullable): a run = maximal stretch of back-to-back samples; (t of its first left edge,
  // number of samples) is all the fill pass needs to regenerate it with the same recurrence
  float* run_t;      // [n, run_cap]
  int32_t* run_n;    // [n, run_cap]
  int32_t* n_runs;   // [n]  (may exceed run_cap: the ray then takes the full-march fill)
  int run_cap;
  const int32_t* order;  // nullable: thread i marches ray order[i] (rays sorted for coherence); outputs stay indexed by ray
  // marching rounds of render_image_test kept on the device (cednerf_march_round): `order` is the list of alive rays,
  // only its first *n_active_dev entries are live, the per-round sample limit is read from *limit_dev, and every
  // per-ray array except near / termination (mask, counts, runs, fill offsets) is indexed by SLOT in that list
  const int32_t* n_active_dev;
  const int32_t* limit_dev;
  int by_slot;
  // nullable: one bit per 4x4x4 block of cells (cednerf_occ_coarsen), set when any cell of the block is occupied.  Inside
  // an empty block the DDA is stepped without looking the cells up (same fp32 additions, same results, a third of the
  // instructions): most of a ray's path is empty space.
  const uint32_t* coarse;
};

__device__ __forceinline__ float clampf(float v, float lo, float hi) { return fminf(fmaxf(v, lo), hi); }
__device__ __forceinline__ int clampi(int v, int lo, int hi) { return v < lo ? lo : (v > hi ? hi : v); }
__device__ __forceinline__ float step_dt(float t, float cone, float step) { return clampf(t * cone, step, 1e10f); }

// The catch-up recurrence of traverse_grids (SURVEY.md A.6): t <- t + clamp(t cone, step, 1e10) until t + dt / 2 >= target.
// A ray walks it over every stretch of empty space - about a thousand iterations per ray on the DyNeRF-shaped scene (t
// grows by 0.4 % per step from 0.25 to the far side of the outermost grid) - and it is one serial chain.  Where the clamp
// cannot bind its two FMNMX leave the chain (same values, bit for bit: clamp returns its argument unchanged inside the
// bounds): t cone >= step holds for the rest of the walk once it holds (t only grows, the rounded product is monotone)
// and t cone < 1e10 holds while t < target; with cone == 0 the increment is the constant step.
__device__ __forceinline__ void advance_to(float& t_last, float t_target, float cone, float step_size) {
  if (step_size <= 0.0f) {
    t_last = t_target;
    return;
  }
  if (cone == 0.0f && step_size <= 1e10f && t_last == t_last && t_last - t_last == 0.0f) {  // finite t: t * 0 = 0 -> dt = step
    const float half = step_size * 0.5f;
    while (t_last + half < t_target) t_last += step_size;
    return;
  }
  while (!(t_last * cone >= step_size && t_target * cone < 1e10f)) {  // the general form, until the clamp stops binding
    const float dt = step_dt(t_last, cone, step_size);
    if (t_last + dt * 0.5f >= t_target) return;
    t_last += dt;
  }
  // four steps per trip: the step chain (one add and one multiply per step) runs ahead of the four stop tests, which hang
  // off it side by side instead of sitting on it; the first test that holds names the value to keep (same operations,
  // same roundings - the steps past the stop are computed and dropped)
  float t = t_last;
  for (;;) {
    const float d0 = t * cone;
    const float t1 = t + d0, d1 = t1 * cone;
    const float t2 = t1 + d1, d2 = t2 * cone;
    const float t3 = t2 + d2, d3 = t3 * cone;
    const bool e0 = t + d0 * 0.5f >= t_target, e1 = t1 + d1 * 0.5f >= t_target;
    const bool e2 = t2 + d2 * 0.5f >= t_target, e3 = t3 + d3 * 0.5f >= t_target;
    if (e0 | e1 | e2 | e3) {
      t_last = e0 ? t : (e1 ? t1 : (e2 ? t2 : t3));
      return;
    }
    t = t3 + d3;
  }
}

__device__ __forceinline__ void slab(const float* o, const float* inv, const float* bx, float near, float far,
                                     float miss, float& t_min, float& t_max, bool& hit) {
  float tmin = -INFINITY, tmax = INFINITY;
#pragma unroll
  for (int a = 0; a < 3; ++a) {
    const float t1 = (bx[a] - o[a]) * inv[a];
    const float t2 = (bx[3 + a] - o[a]) * inv[a];
    tmin = fmaxf(tmin, fminf(t1, t2));
    tmax = fminf(tmax, fmaxf(t1, t2));
  }
  hit = (tmax > tmin) && (tmax > 0.0f);
  t_min = hit ? clampf(tmin, near, far) : miss;
  t_max = hit ? clampf(tmax, near, far) : miss;
}

__global__ void ray_aabb_kernel(const float* __restrict__ rays_o, const float* __restrict__ rays_d, int64_t n,
                                const float* __restrict__ aabbs, int L, float near, float far, float miss,
                                float* __restrict__ t_mins, float* __restrict__ t_maxs, uint8_t* __restrict__ hits) {
  const int64_t r = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (r >= n) return;
  const float o[3] = {rays_o[3 * r], rays_o[3 * r + 1], rays_o[3 * r + 2]};
  const float inv[3] = {1.0f / rays_d[3 * r], 1.0f / rays_d[3 * r + 1], 1.0f / rays_d[3 * r + 2]};
  for (int l = 0; l < L; ++l) {
    float a, b;
    bool h;
    slab(o, inv, aabbs + 6 * l, near, far, miss, a, b, h);
    t_mins[r * L + l] = a;
    t_maxs[r * L + l] = b;
    hits[r * L + l] = (uint8_t)h;
  }
}

// stable insertion sort of the 2L boundary values (ties keep the lower original slot)
__device__ __forceinline__ void sort_bounds(float* v, int* id, int m) {
  for (int i = 1; i < m; ++i) {
    const float kv = v[i];
    const int ki = id[i];
    int j = i - 1;
    while (j >= 0 && v[j] > kv) {
      v[j + 1] = v[j];
      id[j + 1] = id[j];
      --j;
    }
    v[j + 1] = kv;
    id[j + 1] = ki;
  }
}

__global__ void sort_boundaries_kernel(const float* __restrict__ t_mins, const float* __restrict__ t_maxs, int64_t n,
                                       int L, float* __restrict__ t_sorted, int64_t* __restrict__ t_indices) {
  const int64_t r = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (r >= n) return;
  float v[2 * MARCH_MAX_LEVELS];
  int id[2 * MARCH_MAX_LEVELS];
  const int m = 2 * L;
  for (int l = 0; l < L; ++l) {
    v[l] = t_mins[r * L + l];
    v[L + l] = t_maxs[r * L + l];
  }
  for (int i = 0; i < m; ++i) id[i] = i;
  sort_bounds(v, id, m);
  for (int i = 0; i < m; ++i) {
    t_sorted[r * m + i] = v[i];
    t_indices[r * m + i] = id[i];
  }
}

#ifndef MARCH_MIN_BLOCKS
#define MARCH_MIN_BLOCKS 6   // resident CTAs of 128 rays per SM -> 78 registers; measured 5 / 6 / 7 / 8: 0.592 / 0.566 / 0.570 /
#endif                       // 0.598 ms on the count pass of the DyNeRF-shaped batch (rounds of a frame: 7.09 / 7.20 / 7.23 / 7.37)
// COARSE: the 4^3-block bits are given (a.coarse != null).  A template parameter, not a run-time test: the block
// coordinates and their three compares sat in the per-cell path of every launch, also of those without the bits.
template <bool FILL, bool COARSE = false>
__global__ void __launch_bounds__(128, MARCH_MIN_BLOCKS) march_kernel(MarchArgs a) {
  const int64_t slot = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (slot >= a.n_rays) return;
  if (a.n_active_dev && slot >= (int64_t)*a.n_active_dev) {  // beyond the live part of the alive list
    if (!FILL && a.n_samples) a.n_samples[slot] = 0;
    if (!FILL && a.n_runs) a.n_runs[slot] = 0;
    return;
  }
  const int64_t r = a.order ? (int64_t)a.order[slot] : slot;
  const int64_t oi = a.by_slot ? slot : r;  // index of this ray's entries in the count / run / offset arrays
  const float near = a.near ? a.near[r] : a.near_const;
  const float far = a.far ? a.far[r] : a.far_const;
  if (a.mask && !a.mask[oi]) {
    if (a.n_intervals) a.n_intervals[oi] = 0;
    if (a.n_samples) a.n_samples[oi] = 0;
    // (by slot, near and termination are one array, and the fill pass leaves the planes of the rays it skips as they are)
    if (a.termination && !(FILL && a.by_slot)) a.termination[r] = near;
    if (!FILL && a.n_runs) a.n_runs[oi] = 0;
    return;
  }
  const int L = a.n_levels, m = 2 * L, res = a.res;
  const float eps = 1e-6f;
  const float o[3] = {a.rays_o[3 * r], a.rays_o[3 * r + 1], a.rays_o[3 * r + 2]};
  const float d[3] = {a.rays_d[3 * r], a.rays_d[3 * r + 1], a.rays_d[3 * r + 2]};
  const float inv[3] = {1.0f / d[0], 1.0f / d[1], 1.0f / d[2]};
  const float fres = (float)res;
  const int64_t cells_per_level = (int64_t)res * res * res;

  float ts[2 * MARCH_MAX_LEVELS];
  int ti[2 * MARCH_MAX_LEVELS];
  bool hit[MARCH_MAX_LEVELS];
  if (a.t_sorted) {
    for (int i = 0; i < m; ++i) {
      ts[i] = a.t_sorted[r * m + i];
      ti[i] = (int)a.t_indices[r * m + i];
    }
    for (int l = 0; l < L; ++l) hit[l] = a.hits[r * L + l] != 0;
  } else {
    for (int l = 0; l < L; ++l) slab(o, inv, a.aabbs + 6 * l, -INFINITY, INFINITY, INFINITY, ts[l], ts[L + l], hit[l]);
    for (int i = 0; i < m; ++i) ti[i] = i;
    sort_bounds(ts, ti, m);
  }

  const int64_t iv_base = FILL && a.iv_starts ? a.iv_starts[oi] : 0;
  const int64_t sm_base = FILL && a.sm_starts ? a.sm_starts[oi] : 0;
  int n_iv = 0, n_sm = 0;
  float t_last = near;
  int continuous = 0;  // (int, not bool: the compiler packs bools into byte lanes and shuffles them with PRMT in the cell loop)
  int runs = 0, run_len = 0;  // run bookkeeping (count pass with run recording)
  const int limit = a.limit_dev ? *a.limit_dev : a.limit;
  const float step_size = a.step_size, cone = a.cone_angle;

  for (int i = 0; i < m - 1; ++i) {
    const int bi = ti[i];
    const bool entering = bi < L;
    int level = bi % L;
    if (!hit[level]) continue;
    if (!entering) {
      const int bn = ti[i + 1];
      if (bn < L) continue;  // gap between boxes
      level = bn % L;
      if (!hit[level]) continue;
    }
    const float this_tmin = fmaxf(ts[i], near);
    const float this_tmax = fminf(ts[i + 1], far);
    if (this_tmin >= this_tmax) continue;

    if (!continuous) advance_to(t_last, this_tmin, cone, step_size);

    const float* bx = a.aabbs + 6 * level;
    float tdist[3], delta[3];
    int cur[3], overflow[3], stepi[3];
    const float tstart = this_tmin + eps, tend = this_tmax - eps;
#pragma unroll
    for (int ax = 0; ax < 3; ++ax) {
      const float extent = bx[3 + ax] - bx[ax];
      const float voxel = extent / fres;
      const float start = o[ax] + d[ax] * tstart;
      const float end = o[ax] + d[ax] * tend;
      int c = (int)(((start - bx[ax]) / extent) * fres);
      int f = (int)(((end - bx[ax]) / extent) * fres);
      c = clampi(c, 0, res - 1);
      f = clampi(f, 0, res - 1);
      const int start_idx = c + (d[ax] > 0.0f ? 1 : 0);
      const float tmax_a = ((bx[ax] + (((float)start_idx * voxel) - start)) * inv[ax]) + this_tmin;
      const float stepf = (d[ax] == 0.0f) ? 0.0f : (d[ax] > 0.0f ? 1.0f : -1.0f);
      tdist[ax] = (d[ax] == 0.0f) ? this_tmax : tmax_a;
      delta[ax] = (d[ax] == 0.0f) ? this_tmax : (voxel * inv[ax]) * stepf;
      stepi[ax] = (int)stepf;
      cur[ax] = c;
      overflow[ax] = f + stepi[ax];
    }

    // Empty cells only move a catch-up target: t_last is caught up to the exit plane of the LAST empty cell when the next
    // occupied cell (or the end of the segment) needs it.  The cell-by-cell catch-up stops at the first t_last with
    // t_last + dt/2 >= plane, and the planes increase along the ray, so catching up once to the last plane walks the same
    // recurrence to the same stop.  With the coarse bits, cells of a block known to be empty are not even looked up.
    float t_pend = 0.0f;
    int pend = 0;
    int eb0 = -1, eb1 = -1, eb2 = -1;  // the 4^3 block known to be empty (-1: none)
    auto catch_up = [&](float t_target) { advance_to(t_last, t_target, cone, step_size); };
    // the cell's bit index, kept incrementally (one add per DDA step; 32 bits: the entry point checks L res^3 < 2^31)
    uint32_t cell = ((uint32_t)cur[0] * (uint32_t)res + (uint32_t)cur[1]) * (uint32_t)res + (uint32_t)cur[2] +
                    (uint32_t)level * (uint32_t)cells_per_level;
    int dcell[3] = {stepi[0] * res * res, stepi[1] * res, stepi[2]};
    asm volatile("" : "+r"(dcell[0]), "+r"(dcell[1]));  // keep the products in registers (ptxas re-formed them per step)
    while (limit <= 0 || n_sm < limit) {
      const float t_trav = fminf(fminf(tdist[0], fminf(tdist[1], tdist[2])), this_tmax);
      bool occupied = false;
      if (!(COARSE && (cur[0] >> 2) == eb0 && (cur[1] >> 2) == eb1 && (cur[2] >> 2) == eb2)) {
        occupied = (__ldg(a.occ_bits + (cell >> 5)) >> (cell & 31u)) & 1u;
        if (COARSE && !occupied) {
          const int cres = res >> 2;
          const int64_t cb = ((int64_t)(cur[0] >> 2) * cres + (cur[1] >> 2)) * cres + (cur[2] >> 2) +
                             (int64_t)level * cres * cres * cres;
          const bool block_occupied = (__ldg(a.coarse + (cb >> 5)) >> (cb & 31)) & 1u;
          eb0 = block_occupied ? -1 : (cur[0] >> 2);
          eb1 = cur[1] >> 2;
          eb2 = cur[2] >> 2;
        }
      }
      if (!occupied) {
        t_pend = t_trav;
        pend = 1;
        continuous = 0;
      } else {
        if (pend) {
          catch_up(t_pend);
          pend = 0;
        }
        while (limit <= 0 || n_sm < limit) {
          float t_next;
          if (step_size <= 0.0f) {
            t_next = t_trav;
          } else {
            const float dt = step_dt(t_last, cone, step_size);
            if (t_last + dt * 0.5f >= t_trav) break;
            t_next = t_last + dt;
          }
          if (FILL) {
            if (a.iv_vals) {
              const int64_t k = iv_base + n_iv;
              if (!continuous) {
                a.iv_vals[k] = t_last;
                a.iv_ray[k] = r;
                a.iv_left[k] = 1;
                a.iv_vals[k + 1] = t_next;
                a.iv_ray[k + 1] = r;
                a.iv_right[k + 1] = 1;
              } else {
                a.iv_vals[k] = t_next;
                a.iv_ray[k] = r;
                a.iv_left[k - 1] = 1;
                a.iv_right[k] = 1;
              }
            }
            const int64_t k = sm_base + n_sm;
            if (a.sm_vals) {
              a.sm_vals[k] = (t_next + t_last) * 0.5f;
              a.sm_ray[k] = r;
              a.sm_valid[k] = 1;
            }
            if (a.t_starts) {
              a.t_starts[k] = t_last;
              a.t_ends[k] = t_next;
              a.ray_indices[k] = r;
            }
          }
          if (!FILL && a.run_t) {
            if (!continuous) {  // a new run starts at t_last
              if (runs > 0 && runs <= a.run_cap) a.run_n[oi * a.run_cap + runs - 1] = run_len;
              if (runs < a.run_cap) a.run_t[oi * a.run_cap + runs] = t_last;
              ++runs;
              run_len = 0;
            }
            ++run_len;
          }
          n_iv += continuous ? 1 : 2;
          n_sm += 1;
          continuous = 1;
          t_last = t_next;
          if (t_next >= t_trav) break;
        }
      }
      // advance along the axis whose plane comes first - written with selects, not a three-way branch: the lanes of a
      // warp pick different axes at every step, and a branch runs the three arms one after the other.  (The add for the
      // two other axes is computed and dropped: same values for the chosen one.)
      const bool s0 = tdist[0] < tdist[1] && tdist[0] < tdist[2];
      const bool s1 = !s0 && tdist[1] < tdist[2];
      const bool s2 = !s0 && !s1;
      const float n0 = tdist[0] + delta[0], n1 = tdist[1] + delta[1], n2 = tdist[2] + delta[2];
      tdist[0] = s0 ? n0 : tdist[0];
      tdist[1] = s1 ? n1 : tdist[1];
      tdist[2] = s2 ? n2 : tdist[2];
      cur[0] += s0 ? stepi[0] : 0;
      cur[1] += s1 ? stepi[1] : 0;
      cur[2] += s2 ? stepi[2] : 0;
      cell += (uint32_t)(s0 ? dcell[0] : (s1 ? dcell[1] : dcell[2]));
      const bool done = (s0 & (cur[0] == overflow[0])) | (s1 & (cur[1] == overflow[1])) | (s2 & (cur[2] == overflow[2]));
      if (done) break;
    }
    if (pend) catch_up(t_pend);
  }
  if (!FILL && a.run_t) {
    if (runs > 0 && runs <= a.run_cap) a.run_n[oi * a.run_cap + runs - 1] = run_len;
    a.n_runs[oi] = runs;
  }
  if (a.n_intervals) a.n_intervals[oi] = n_iv;
  if (a.n_samples) a.n_samples[oi] = n_sm;
  // By slot (cednerf_march_round) near and termination are one array.  A ray over the run limit is marched a second time
  // by the full-march fill, which must start from the same plane: the count pass leaves that plane in place, and the fill
  // pass writes the termination plane instead (the same fp32 operations from the same start, so the same value).
  const bool refilled = a.by_slot && !FILL && runs > a.run_cap;
  if (a.termination && !refilled) a.termination[r] = t_last;
}

// Fill pass from recorded runs: no grid traversal, just the step recurrence t <- t + clamp(t*cone, step, 1e10) replayed
// from each run's first left edge (identical fp32 operations, so identical bits).  Rays whose run list overflowed are
// flagged in `overflow` and filled by the full-march kernel with that flag array as its ray mask.
__global__ void __launch_bounds__(128)
march_fill_runs_kernel(int64_t n_rays, const int64_t* __restrict__ sm_starts, const float* __restrict__ run_t,
                       const int32_t* __restrict__ run_n, const int32_t* __restrict__ n_runs, int run_cap,
                       float step_size, float cone, float* __restrict__ t_starts, float* __restrict__ t_ends,
                       int64_t* __restrict__ ray_indices, uint8_t* __restrict__ overflow,
                       const int32_t* __restrict__ capped_counts, const int32_t* __restrict__ slot_ray = nullptr,
                       const int32_t* __restrict__ n_active_dev = nullptr) {
  const int64_t r = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;  // ray, or slot in the alive list (slot_ray)
  if (r >= n_rays) return;
  if (n_active_dev && r >= (int64_t)*n_active_dev) {
    overflow[r] = 0;
    return;
  }
  const int64_t ray_id = slot_ray ? (int64_t)slot_ray[r] : r;
  const int runs = n_runs[r];
  bool over = runs > run_cap;
  int64_t k = sm_starts[r];
  // capped mode (sm_starts = offsets [n_rays + 1] clamped to the capacity of the packed buffers, capped_counts = the
  // unclamped per-ray counts): nothing is written at or beyond the clamped end of the ray's range
  const int64_t k_end = capped_counts ? sm_starts[r + 1] : INT64_MAX;
  if (capped_counts && over && k_end - k != (int64_t)capped_counts[r]) {
    // a truncated ray cannot take the full-march fallback (it writes its whole range): leave harmless samples
    for (; k < k_end; ++k) t_starts[k] = 0.0f, t_ends[k] = 0.0f, ray_indices[k] = ray_id;
    over = false;
    overflow[r] = 0;
    return;
  }
  overflow[r] = (uint8_t)over;
  if (over) return;
  auto next = [&](float t) { return (step_size <= 0.0f) ? t : t + step_dt(t, cone, step_size); };
  for (int j = 0; j < runs; ++j) {
    float t = run_t[r * run_cap + j];
    int cnt = run_n[r * run_cap + j];
    if ((int64_t)cnt > k_end - k) cnt = (int)(k_end - k);
    int i = 0;
    // A ray's samples are consecutive in the packed arrays but neighbouring lanes write ~one ray length apart: scalar
    // stores put 4 useful bytes into every 32-byte sector they touch.  Four samples at a time as 16-byte stores (once k
    // is a multiple of 4) quarter the number of store transactions.
    for (; i < cnt && (k & 3); ++i, ++k) {
      const float t_next = next(t);
      t_starts[k] = t, t_ends[k] = t_next, ray_indices[k] = ray_id;
      t = t_next;
    }
    for (; i + 4 <= cnt; i += 4, k += 4) {
      const float a1 = next(t), a2 = next(a1), a3 = next(a2), a4 = next(a3);
      *reinterpret_cast<float4*>(t_starts + k) = make_float4(t, a1, a2, a3);
      *reinterpret_cast<float4*>(t_ends + k) = make_float4(a1, a2, a3, a4);
      const longlong2 rr = make_longlong2((long long)ray_id, (long long)ray_id);
      *reinterpret_cast<longlong2*>(ray_indices + k) = rr;
      *reinterpret_cast<longlong2*>(ray_indices + k + 2) = rr;
      t = a4;
    }
    for (; i < cnt; ++i, ++k) {
      const float t_next = next(t);
      t_starts[k] = t, t_ends[k] = t_next, ray_indices[k] = ray_id;
      t = t_next;
    }
  }
}

// ---- bit packing of the occupancy grid ------------------------------------------------------------
__global__ void pack_bits_kernel(const uint8_t* __restrict__ bin, int64_t n_cells, uint32_t* __restrict__ bits) {
  const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;  // one cell per thread, one word per warp
  const bool b = i < n_cells && bin[i] != 0;
  const unsigned w = __ballot_sync(0xffffffffu, b);
  if ((threadIdx.x & 31) == 0 && i < n_cells) bits[i >> 5] = w;
}

// occs -> binaries (bool bytes) + bit field:  binaries = occs > thre   (SURVEY A.2 last line)
__global__ void occ_threshold_kernel(const float* __restrict__ occs, int64_t n_cells, const float* __restrict__ thre,
                                     uint8_t* __restrict__ bin, uint32_t* __restrict__ bits) {
  const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  const bool b = i < n_cells && occs[i] > *thre;
  const unsigned w = __ballot_sync(0xffffffffu, b);
  if (i < n_cells) {
    bin[i] = (uint8_t)b;
    if ((threadIdx.x & 31) == 0) bits[i >> 5] = w;
  }
}

// ---- int32 counts -> int64 exclusive offsets (+ total) -----------------------------------------------
constexpr int SCAN_THREADS = 256;
constexpr int SCAN_ITEMS = 16;
constexpr int SCAN_TILE = SCAN_THREADS * SCAN_ITEMS;

__device__ __forceinline__ int64_t block_excl_scan(int64_t v, int64_t* total, int64_t* smem) {
  const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
  int64_t x = v;
#pragma unroll
  for (int o = 1; o < 32; o <<= 1) {
    const int64_t y = __shfl_up_sync(0xffffffffu, x, o);
    if (lane >= o) x += y;
  }
  if (lane == 31) smem[wid] = x;
  __syncthreads();
  if (wid == 0) {
    int64_t w = lane < SCAN_THREADS / 32 ? smem[lane] : 0;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
      const int64_t y = __shfl_up_sync(0xffffffffu, w, o);
      if (lane >= o) w += y;
    }
    if (lane < SCAN_THREADS / 32) smem[lane] = w;
  }
  __syncthreads();
  const int64_t warp_off = wid ? smem[wid - 1] : 0;
  *total = smem[SCAN_THREADS / 32 - 1];
  __syncthreads();
  return warp_off + x - v;
}

__global__ void __launch_bounds__(SCAN_THREADS)
scan_tile_sums_kernel(const int32_t* __restrict__ counts, int64_t n, int64_t* __restrict__ tile_sums) {
  __shared__ int64_t smem[SCAN_THREADS / 32];
  const int64_t base = (int64_t)blockIdx.x * SCAN_TILE + (int64_t)threadIdx.x * SCAN_ITEMS;
  int64_t s = 0;
  for (int k = 0; k < SCAN_ITEMS; ++k)
    if (base + k < n) s += counts[base + k];
  int64_t total;
  block_excl_scan(s, &total, smem);
  if (threadIdx.x == 0) tile_sums[blockIdx.x] = total;
}

__global__ void __launch_bounds__(SCAN_THREADS)
scan_tile_offsets_kernel(int64_t* __restrict__ tile_sums, int64_t n_tiles, int64_t* __restrict__ total_out) {
  __shared__ int64_t smem[SCAN_THREADS / 32];
  int64_t carry = 0;
  for (int64_t base = 0; base < n_tiles; base += SCAN_THREADS) {
    const int64_t i = base + threadIdx.x;
    const int64_t v = i < n_tiles ? tile_sums[i] : 0;
    int64_t total;
    const int64_t ex = block_excl_scan(v, &total, smem);
    if (i < n_tiles) tile_sums[i] = carry + ex;
    carry += total;
  }
  if (threadIdx.x == 0 && total_out) *total_out = carry;
}

__global__ void __launch_bounds__(SCAN_THREADS)
scan_apply_kernel(const int32_t* __restrict__ counts, int64_t n, const int64_t* __restrict__ tile_offsets,
                  int64_t* __restrict__ starts, int64_t* __restrict__ packed_info) {
  __shared__ int64_t smem[SCAN_THREADS / 32];
  const int64_t base = (int64_t)blockIdx.x * SCAN_TILE + (int64_t)threadIdx.x * SCAN_ITEMS;
  int32_t c[SCAN_ITEMS];
  int64_t s = 0;
#pragma unroll
  for (int k = 0; k < SCAN_ITEMS; ++k) {
    c[k] = base + k < n ? counts[base + k] : 0;
    s += c[k];
  }
  int64_t total;
  int64_t off = tile_offsets[blockIdx.x] + block_excl_scan(s, &total, smem);
#pragma unroll
  for (int k = 0; k < SCAN_ITEMS; ++k) {
    if (base + k < n) {
      if (starts) starts[base + k] = off;
      if (packed_info) {
        packed_info[2 * (base + k)] = off;
        packed_info[2 * (base + k) + 1] = c[k];
      }
    }
    off += c[k];
  }
}

// The capped scan in ONE pass (decoupled look-back): tiles take tickets in launch order, publish their aggregate, then
// add up the published values of their predecessors (aggregate -> keep looking back, inclusive prefix -> stop).
// state[0] = ticket counter, state[1 + t] = (flag << 62) | value with flag 1 = aggregate, 2 = inclusive prefix; zeroed by
// the launcher.  One launch instead of three: the marching rounds of a frame scan twice per round.
__global__ void __launch_bounds__(SCAN_THREADS)
scan_capped_onepass_kernel(const int32_t* __restrict__ counts, int64_t n, int64_t capacity, int64_t* __restrict__ offsets,
                           int64_t* __restrict__ totals, unsigned long long* __restrict__ state) {
  __shared__ int64_t smem[SCAN_THREADS / 32];
  __shared__ int64_t tile_s, excl_s;
  if (threadIdx.x == 0) tile_s = (int64_t)atomicAdd(state, 1ull);
  __syncthreads();
  const int64_t tile = tile_s;
  const int64_t base = tile * SCAN_TILE + (int64_t)threadIdx.x * SCAN_ITEMS;
  int32_t c[SCAN_ITEMS];
  int64_t s = 0;
#pragma unroll
  for (int k = 0; k < SCAN_ITEMS; ++k) {
    c[k] = base + k < n ? counts[base + k] : 0;
    s += c[k];
  }
  int64_t total;
  const int64_t local = block_excl_scan(s, &total, smem);
  if (threadIdx.x == 0) {
    volatile unsigned long long* st = state + 1;
    const unsigned long long FLAG_AGG = 1ull << 62, FLAG_INC = 2ull << 62, MASK = (1ull << 62) - 1ull;
    if (tile > 0) {
      st[tile] = FLAG_AGG | (unsigned long long)total;
      __threadfence();
    }
    int64_t excl = 0;
    for (int64_t j = tile - 1; j >= 0; --j) {
      unsigned long long v;
      do {
        v = st[j];
      } while ((v >> 62) == 0ull);
      excl += (int64_t)(v & MASK);
      if ((v >> 62) == 2ull) break;
    }
    st[tile] = FLAG_INC | (unsigned long long)(excl + total);
    __threadfence();
    excl_s = excl;
    if ((tile + 1) * SCAN_TILE >= n) {  // the last tile knows the grand total
      const int64_t t = excl + total;
      offsets[n] = t < capacity ? t : capacity;
      totals[0] = t < capacity ? t : capacity;
      totals[1] = t;
    }
  }
  __syncthreads();
  int64_t off = excl_s + local;
#pragma unroll
  for (int k = 0; k < SCAN_ITEMS; ++k) {
    if (base + k < n) offsets[base + k] = off < capacity ? off : capacity;
    off += c[k];
  }
}

}  // namespace

CEDNERF_EXPORT int cednerf_ray_aabb_intersect(const float* rays_o, const float* rays_d, int64_t n_rays,
                                              const float* aabbs, int n_levels, float near_plane, float far_plane,
                                              float miss_value, float* t_mins, float* t_maxs, uint8_t* hits,
                                              void* stream) {
  CEDNERF_REQUIRE(n_rays >= 0 && n_levels >= 1, "bad sizes");
  if (n_rays == 0) return 0;
  ray_aabb_kernel<<<cednerf_blocks(n_rays, 256), 256, 0, (cudaStream_t)stream>>>(
      rays_o, rays_d, n_rays, aabbs, n_levels, near_plane, far_plane, miss_value, t_mins, t_maxs, hits);
  return cednerf_check_launch("cednerf_ray_aabb_intersect");
}

CEDNERF_EXPORT int cednerf_sort_boundaries(const float* t_mins, const float* t_maxs, int64_t n_rays, int n_levels,
                                           float* t_sorted, int64_t* t_indices, void* stream) {
  CEDNERF_REQUIRE(n_rays >= 0 && n_levels >= 1 && n_levels <= MARCH_MAX_LEVELS, "bad sizes (levels <= 8)");
  if (n_rays == 0) return 0;
  sort_boundaries_kernel<<<cednerf_blocks(n_rays, 256), 256, 0, (cudaStream_t)stream>>>(t_mins, t_maxs, n_rays,
                                                                                       n_levels, t_sorted, t_indices);
  return cednerf_check_launch("cednerf_sort_boundaries");
}

// bits holds ceil(n_cells / 32) words; the unused high bits of the last one are zero
CEDNERF_EXPORT int cednerf_occ_pack_bits(const uint8_t* binaries, int64_t n_cells, uint32_t* bits, void* stream) {
  CEDNERF_REQUIRE(n_cells > 0, "empty grid");
  pack_bits_kernel<<<cednerf_blocks(n_cells, 256), 256, 0, (cudaStream_t)stream>>>(binaries, n_cells, bits);
  return cednerf_check_launch("cednerf_occ_pack_bits");
}

CEDNERF_EXPORT int cednerf_occ_threshold_pack(const float* occs, int64_t n_cells, const float* threshold_dev,
                                              uint8_t* binaries, uint32_t* bits, void* stream) {
  CEDNERF_REQUIRE(n_cells > 0 && (n_cells % 32) == 0, "cell count must be a multiple of 32");
  occ_threshold_kernel<<<cednerf_blocks(n_cells, 256), 256, 0, (cudaStream_t)stream>>>(occs, n_cells, threshold_dev,
                                                                                      binaries, bits);
  return cednerf_check_launch("cednerf_occ_threshold_pack");
}

namespace {

// OccGridEstimator.mark_invisible_cells (nerfacc; called at train_real.py:205-211): a cell (its lower corner mapped with
// coord / (res - 1), as nerfacc does) stays valid (occs = 0) when at least one camera sees it at depth >= near_plane
// and no camera sees it closer than near_plane; every other cell gets occs = -1 and is never sampled or updated again.
// One thread per cell, cameras staged through shared memory; every product and sum is individually rounded in the
// order oracle/nerfacc_ref.py fixes, so the result is bit-comparable.
__global__ void __launch_bounds__(256) occ_mark_invisible_kernel(const float* __restrict__ K, int n_K,
                                                                 const float* __restrict__ c2w, int n_cams, int c2w_rows,
                                                                 const float* __restrict__ aabbs, int res,
                                                                 int64_t cells_per_level, int64_t n_cells, float width,
                                                                 float height, float near, float* __restrict__ occs) {
  __shared__ float cam[64][21];  // w2c_R (9), w2c_T (3), K (9)
  const int64_t cell = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  const bool active = cell < n_cells;
  float xw[3] = {0.f, 0.f, 0.f};
  if (active) {
    const int level = (int)(cell / cells_per_level);
    const int64_t c = cell - (int64_t)level * cells_per_level;
    const int coord[3] = {(int)(c / ((int64_t)res * res)), (int)((c / res) % res), (int)(c % res)};
    const float* bx = aabbs + 6 * level;
#pragma unroll
    for (int k = 0; k < 3; ++k) {
      const float x01 = __fdiv_rn((float)coord[k], (float)(res - 1));
      xw[k] = __fadd_rn(bx[k], __fmul_rn(x01, __fsub_rn(bx[3 + k], bx[k])));
    }
  }
  bool covered = false, too_near = false;
  for (int c0 = 0; c0 < n_cams; c0 += 64) {
    const int nc = n_cams - c0 < 64 ? n_cams - c0 : 64;
    __syncthreads();
    for (int q = threadIdx.x; q < nc; q += blockDim.x) {
      const float* m = c2w + (int64_t)(c0 + q) * c2w_rows * 4;
      const float* k = K + (n_K == 1 ? 0 : (int64_t)(c0 + q) * 9);
      float* d = cam[q];
#pragma unroll
      for (int i = 0; i < 3; ++i) {
#pragma unroll
        for (int j = 0; j < 3; ++j) d[3 * i + j] = m[4 * j + i];  // w2c_R = R^T
        d[9 + i] = -__fadd_rn(__fadd_rn(__fmul_rn(m[i], m[3]), __fmul_rn(m[4 + i], m[7])), __fmul_rn(m[8 + i], m[11]));
      }
#pragma unroll
      for (int j = 0; j < 9; ++j) d[12 + j] = k[j];
    }
    __syncthreads();
    if (active) {
      for (int q = 0; q < nc; ++q) {
        const float* d = cam[q];
        float xc[3], uvd[3];
#pragma unroll
        for (int i = 0; i < 3; ++i)
          xc[i] = __fadd_rn(__fadd_rn(__fadd_rn(__fmul_rn(d[3 * i], xw[0]), __fmul_rn(d[3 * i + 1], xw[1])),
                                      __fmul_rn(d[3 * i + 2], xw[2])),
                            d[9 + i]);
#pragma unroll
        for (int i = 0; i < 3; ++i)
          uvd[i] = __fadd_rn(__fadd_rn(__fmul_rn(d[12 + 3 * i], xc[0]), __fmul_rn(d[12 + 3 * i + 1], xc[1])),
                             __fmul_rn(d[12 + 3 * i + 2], xc[2]));
        const float u = __fdiv_rn(uvd[0], uvd[2]), v = __fdiv_rn(uvd[1], uvd[2]);
        const bool in_image = uvd[2] >= 0.f && u >= 0.f && u < width && v >= 0.f && v < height;
        covered = covered || (uvd[2] >= near && in_image);
        too_near = too_near || (uvd[2] < near && in_image);
      }
    }
  }
  if (active) occs[cell] = (covered && !too_near) ? 0.f : -1.f;
}

}  // namespace

// K: [n_K, 3, 3] with n_K == 1 (shared intrinsics) or n_cams; c2w: [n_cams, c2w_rows (3 or 4), 4]; occs: [L * res^3].
CEDNERF_EXPORT int cednerf_occ_mark_invisible(const float* K, int n_K, const float* c2w, int n_cams, int c2w_rows,
                                              const float* aabbs, int n_levels, int resolution, int width, int height,
                                              float near_plane, float* occs, void* stream) {
  CEDNERF_REQUIRE(K && c2w && aabbs && occs, "null argument");
  CEDNERF_REQUIRE(n_cams >= 1 && (n_K == 1 || n_K == n_cams) && (c2w_rows == 3 || c2w_rows == 4), "bad camera arrays");
  CEDNERF_REQUIRE(n_levels >= 1 && resolution >= 2, "bad grid");
  const int64_t cpl = (int64_t)resolution * resolution * resolution, n_cells = cpl * n_levels;
  occ_mark_invisible_kernel<<<cednerf_blocks(n_cells, 256), 256, 0, (cudaStream_t)stream>>>(
      K, n_K, c2w, n_cams, c2w_rows, aabbs, resolution, cpl, n_cells, (float)width, (float)height, near_plane, occs);
  return cednerf_check_launch("cednerf_occ_mark_invisible");
}

namespace {

// 20-bit Morton code of the ray direction (octahedral map, 10 bits per axis): rays with neighbouring codes cross the
// nested grids along neighbouring paths.  Sorting a batch of random training rays by it before the count pass raises the
// marcher's SIMT efficiency (it is an instruction-bound kernel whose lanes otherwise sit in unrelated cells).
__global__ void ray_coherence_keys_kernel(const float* __restrict__ rays_d, int64_t n, int32_t* __restrict__ keys) {
  const int64_t r = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (r >= n) return;
  const float x = rays_d[3 * r], y = rays_d[3 * r + 1], z = rays_d[3 * r + 2];
  const float inv = 1.0f / fmaxf(fabsf(x) + fabsf(y) + fabsf(z), 1e-20f);
  float u = x * inv, v = y * inv;
  if (z < 0.0f) {
    const float fu = (1.0f - fabsf(v)) * (u >= 0.0f ? 1.0f : -1.0f), fv = (1.0f - fabsf(u)) * (v >= 0.0f ? 1.0f : -1.0f);
    u = fu, v = fv;
  }
  uint32_t qu = (uint32_t)fminf(fmaxf((u * 0.5f + 0.5f) * 1023.0f, 0.0f), 1023.0f);
  uint32_t qv = (uint32_t)fminf(fmaxf((v * 0.5f + 0.5f) * 1023.0f, 0.0f), 1023.0f);
  auto spread = [](uint32_t b) {  // 10 bits -> every other bit of 20
    b = (b | (b << 8)) & 0x00ff00ffu;
    b = (b | (b << 4)) & 0x0f0f0f0fu;
    b = (b | (b << 2)) & 0x33333333u;
    b = (b | (b << 1)) & 0x55555555u;
    return b;
  };
  keys[r] = (int32_t)(spread(qu) | (spread(qv) << 1));
}

// one bit per 4x4x4 block of cells: set when any cell of the block is occupied
__global__ void occ_coarsen_kernel(const uint32_t* __restrict__ bits, int n_levels, int res, uint32_t* __restrict__ coarse) {
  const int cres = res >> 2;
  const int64_t per_level = (int64_t)cres * cres * cres, total = per_level * n_levels;
  const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;  // one coarse WORD (32 blocks) per thread
  if (i * 32 >= total) return;
  uint32_t w = 0u;
  for (int j = 0; j < 32; ++j) {
    const int64_t cb = i * 32 + j;
    if (cb >= total) break;
    const int level = (int)(cb / per_level);
    const int64_t r = cb - level * per_level;
    const int bz = (int)(r % cres), by = (int)((r / cres) % cres), bx = (int)(r / ((int64_t)cres * cres));
    bool any = false;
    for (int dx = 0; dx < 4 && !any; ++dx)
      for (int dy = 0; dy < 4 && !any; ++dy) {
        const int64_t c0 = ((int64_t)(4 * bx + dx) * res + (4 * by + dy)) * res + 4 * bz + (int64_t)level * res * res * res;
        for (int dz = 0; dz < 4; ++dz) {
          const int64_t c = c0 + dz;
          any = any || ((bits[c >> 5] >> (c & 31)) & 1u);
        }
      }
    if (any) w |= 1u << j;
  }
  coarse[i] = w;
}

// ---- bucket order by coherence key: histogram -> scan -> scatter (order inside a bucket is irrelevant: the permutation
// only decides which rays share a warp, every output stays indexed by ray) -------------------------------------------
#define ORDER_BINS 16384   // the top 14 bits of the 20-bit key: 128 x 128 direction cells
__global__ void order_hist_kernel(const int32_t* __restrict__ keys, int64_t n, uint32_t* __restrict__ hist) {
  const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i < n) atomicAdd(hist + (((uint32_t)keys[i]) >> 6), 1u);
}
__global__ void __launch_bounds__(1024) order_scan_kernel(uint32_t* __restrict__ hist) {  // exclusive scan of 16384 bins
  __shared__ uint32_t warp_tot[32];
  uint32_t v[16], s = 0;
#pragma unroll
  for (int k = 0; k < 16; ++k) v[k] = hist[threadIdx.x * 16 + k], s += v[k];
  uint32_t incl = s;
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
#pragma unroll
  for (int o = 1; o < 32; o <<= 1) {
    const uint32_t t = __shfl_up_sync(0xffffffffu, incl, o);
    if (lane >= o) incl += t;
  }
  if (lane == 31) warp_tot[warp] = incl;
  __syncthreads();
  if (warp == 0) {
    uint32_t w = warp_tot[lane], wi = w;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
      const uint32_t t = __shfl_up_sync(0xffffffffu, wi, o);
      if (lane >= o) wi += t;
    }
    warp_tot[lane] = wi - w;
  }
  __syncthreads();
  uint32_t off = warp_tot[warp] + incl - s;
#pragma unroll
  for (int k = 0; k < 16; ++k) hist[threadIdx.x * 16 + k] = off, off += v[k];
}
__global__ void order_scatter_kernel(const int32_t* __restrict__ keys, int64_t n, uint32_t* __restrict__ cursor,
                                     int32_t* __restrict__ order) {
  const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i < n) order[atomicAdd(cursor + (((uint32_t)keys[i]) >> 6), 1u)] = (int32_t)i;
}

}  // namespace

// order [n] = a permutation of the rays that groups equal leading key bits (cednerf_ray_coherence_keys): the ray_order
// argument of cednerf_march.  workspace: 64 KB.  Replaces a general radix sort (4 launches, ~0.1 ms on 2^18 keys).
CEDNERF_EXPORT int cednerf_ray_coherence_order(const int32_t* keys, int64_t n_rays, int32_t* order, void* workspace,
                                               void* stream) {
  CEDNERF_REQUIRE(n_rays >= 0 && n_rays < (1ll << 31) && keys && order && workspace, "bad arguments");
  if (n_rays == 0) return 0;
  cudaStream_t st = (cudaStream_t)stream;
  uint32_t* hist = (uint32_t*)workspace;
  cudaMemsetAsync(hist, 0, ORDER_BINS * sizeof(uint32_t), st);
  order_hist_kernel<<<cednerf_blocks(n_rays, 256), 256, 0, st>>>(keys, n_rays, hist);
  order_scan_kernel<<<1, 1024, 0, st>>>(hist);
  order_scatter_kernel<<<cednerf_blocks(n_rays, 256), 256, 0, st>>>(keys, n_rays, hist, order);
  return cednerf_check_launch("cednerf_ray_coherence_order", 3);
}

// coarse occupancy for the marcher's empty-space skip: one bit per 4x4x4 block of cells of every level (resolution a
// multiple of 4); coarse holds ceil(n_levels (resolution / 4)^3 / 32) words
CEDNERF_EXPORT int cednerf_occ_coarsen(const uint32_t* occ_bits, int n_levels, int resolution, uint32_t* coarse, void* stream) {
  CEDNERF_REQUIRE(occ_bits && coarse && n_levels >= 1 && resolution >= 4 && resolution % 4 == 0, "bad arguments");
  const int cres = resolution / 4;
  const int64_t words = ((int64_t)cres * cres * cres * n_levels + 31) / 32;
  occ_coarsen_kernel<<<cednerf_blocks(words, 128), 128, 0, (cudaStream_t)stream>>>(occ_bits, n_levels, resolution, coarse);
  return cednerf_check_launch("cednerf_occ_coarsen");
}

// keys[r] = coherence key of ray r (sort by it, pass the permutation to cednerf_march as ray_order)
CEDNERF_EXPORT int cednerf_ray_coherence_keys(const float* rays_d, int64_t n_rays, int32_t* keys, void* stream) {
  CEDNERF_REQUIRE(n_rays >= 0 && rays_d && keys, "bad arguments");
  if (n_rays == 0) return 0;
  ray_coherence_keys_kernel<<<cednerf_blocks(n_rays, 256), 256, 0, (cudaStream_t)stream>>>(rays_d, n_rays, keys);
  return cednerf_check_launch("cednerf_ray_coherence_keys");
}

// March one pass.  fill == 0: count only (n_intervals / n_samples / termination).  fill == 1: write the
// outputs at the offsets given by iv_starts / sm_starts.  near/far: per-ray arrays or null (constants).
CEDNERF_EXPORT int cednerf_march(int fill, const float* rays_o, const float* rays_d, int64_t n_rays,
                                 const uint32_t* occ_bits, const float* aabbs, int n_levels, int resolution,
                                 const float* near_planes, const float* far_planes, float near_const, float far_const,
                                 float step_size, float cone_angle, int steps_limit, const uint8_t* rays_mask,
                                 const float* t_sorted, const int64_t* t_indices, const uint8_t* hits,
                                 const int64_t* iv_starts, const int64_t* sm_starts, float* iv_vals, uint8_t* iv_left,
                                 uint8_t* iv_right, int64_t* iv_ray, float* sm_vals, int64_t* sm_ray,
                                 uint8_t* sm_valid, float* t_starts, float* t_ends, int64_t* ray_indices,
                                 int32_t* n_intervals, int32_t* n_samples, float* termination, float* run_t,
                                 int32_t* run_n, int32_t* n_runs, int run_cap, const int32_t* ray_order,
                                 const uint32_t* occ_coarse, void* stream) {
  CEDNERF_REQUIRE(!run_t || (!fill && run_n && n_runs && run_cap > 0 && step_size > 0.0f),
                  "run recording: count pass, positive step size");
  CEDNERF_REQUIRE((int64_t)n_levels * resolution * resolution * resolution < (1ll << 31), "occupancy grid too large");
  CEDNERF_REQUIRE(n_rays >= 0 && n_levels >= 1 && n_levels <= MARCH_MAX_LEVELS && resolution >= 1,
                  "bad sizes (levels <= 8)");
  CEDNERF_REQUIRE((t_sorted == nullptr) == (t_indices == nullptr) && (t_sorted == nullptr) == (hits == nullptr),
                  "t_sorted, t_indices and hits go together");
  CEDNERF_REQUIRE(!fill || ((!t_starts && !sm_vals) || sm_starts) , "fill pass needs sm_starts");
  CEDNERF_REQUIRE(!fill || !iv_vals || iv_starts, "fill pass needs iv_starts");
  CEDNERF_REQUIRE(!t_starts || (t_ends && ray_indices), "packed outputs go together");
  if (n_rays == 0) return 0;
  MarchArgs a{rays_o, rays_d, n_rays, occ_bits, aabbs, n_levels, resolution, near_planes, far_planes, near_const,
              far_const, step_size, cone_angle, steps_limit, rays_mask, t_sorted, t_indices, hits, iv_starts,
              sm_starts, iv_vals, iv_left, iv_right, iv_ray, sm_vals, sm_ray, sm_valid, t_starts, t_ends, ray_indices,
              n_intervals, n_samples, termination, run_t, run_n, n_runs, run_cap, ray_order, nullptr, nullptr, 0,
              (resolution % 4 == 0) ? occ_coarse : nullptr};
  const unsigned grid = cednerf_blocks(n_rays, 128);
  if (a.coarse) {
    if (fill) march_kernel<true, true><<<grid, 128, 0, (cudaStream_t)stream>>>(a);
    else march_kernel<false, true><<<grid, 128, 0, (cudaStream_t)stream>>>(a);
  } else {
    if (fill) march_kernel<true><<<grid, 128, 0, (cudaStream_t)stream>>>(a);
    else march_kernel<false><<<grid, 128, 0, (cudaStream_t)stream>>>(a);
  }
  return cednerf_check_launch("cednerf_march");
}

// Packed fill from the runs a count pass recorded (see march_fill_runs_kernel); `overflow` [n] receives 1 for rays
// whose run list did not fit - fill those with cednerf_march(fill = 1, rays_mask = overflow, ...).
CEDNERF_EXPORT int cednerf_march_fill_runs(int64_t n_rays, const int64_t* sm_starts, const float* run_t,
                                           const int32_t* run_n, const int32_t* n_runs, int run_cap, float step_size,
                                           float cone_angle, float* t_starts, float* t_ends, int64_t* ray_indices,
                                           uint8_t* overflow, void* stream) {
  CEDNERF_REQUIRE(n_rays >= 0 && run_cap > 0 && step_size > 0.0f, "bad arguments");
  CEDNERF_REQUIRE((((uintptr_t)t_starts | (uintptr_t)t_ends | (uintptr_t)ray_indices) & 15) == 0,
                  "packed outputs must be 16-byte aligned");
  if (n_rays == 0) return 0;
  march_fill_runs_kernel<<<cednerf_blocks(n_rays, 128), 128, 0, (cudaStream_t)stream>>>(
      n_rays, sm_starts, run_t, run_n, n_runs, run_cap, step_size, cone_angle, t_starts, t_ends, ray_indices, overflow,
      nullptr);
  return cednerf_check_launch("cednerf_march_fill_runs");
}

// The same fill for buffers of a fixed capacity (no host read of the sample total): `offsets` [n_rays + 1] comes from
// cednerf_exclusive_scan_capped and `n_samples` holds the unclamped per-ray counts; samples at or beyond the capacity are
// dropped (totals[1] > totals[0] of the scan tells the caller).  Rays flagged in `overflow` go through
// cednerf_march(fill = 1, rays_mask = overflow, sm_starts = offsets) as before; a ray that is both truncated and over
// the run limit gets zero-length samples instead.
CEDNERF_EXPORT int cednerf_march_fill_runs_capped(int64_t n_rays, const int64_t* offsets, const int32_t* n_samples,
                                                  const float* run_t, const int32_t* run_n, const int32_t* n_runs,
                                                  int run_cap, float step_size, float cone_angle, float* t_starts,
                                                  float* t_ends, int64_t* ray_indices, uint8_t* overflow, void* stream) {
  CEDNERF_REQUIRE(n_rays >= 0 && run_cap > 0 && step_size > 0.0f && offsets && n_samples, "bad arguments");
  CEDNERF_REQUIRE((((uintptr_t)t_starts | (uintptr_t)t_ends | (uintptr_t)ray_indices) & 15) == 0,
                  "packed outputs must be 16-byte aligned");
  if (n_rays == 0) return 0;
  march_fill_runs_kernel<<<cednerf_blocks(n_rays, 128), 128, 0, (cudaStream_t)stream>>>(
      n_rays, offsets, run_t, run_n, n_runs, run_cap, step_size, cone_angle, t_starts, t_ends, ray_indices, overflow,
      n_samples);
  return cednerf_check_launch("cednerf_march_fill_runs_capped");
}

CEDNERF_EXPORT int64_t cednerf_scan_workspace_bytes(int64_t n) {
  const int64_t tiles = (n + SCAN_TILE - 1) / SCAN_TILE;
  return 8 * (tiles + 1);
}

// counts int32[n] -> starts int64[n] (exclusive), optional packed_info int64[n,2] = (start, count),
// optional total int64[1]; workspace from cednerf_scan_workspace_bytes.
CEDNERF_EXPORT int cednerf_exclusive_scan(const int32_t* counts, int64_t n, int64_t* starts, int64_t* packed_info,
                                          int64_t* total, void* workspace, void* stream) {
  CEDNERF_REQUIRE(n >= 0 && workspace, "bad arguments");
  cudaStream_t st = (cudaStream_t)stream;
  if (n == 0) {
    if (total) cudaMemsetAsync(total, 0, 8, st);
    return 0;
  }
  const int64_t tiles = (n + SCAN_TILE - 1) / SCAN_TILE;
  int64_t* tile_sums = (int64_t*)workspace;
  scan_tile_sums_kernel<<<(unsigned)tiles, SCAN_THREADS, 0, st>>>(counts, n, tile_sums);
  scan_tile_offsets_kernel<<<1, SCAN_THREADS, 0, st>>>(tile_sums, tiles, total);
  scan_apply_kernel<<<(unsigned)tiles, SCAN_THREADS, 0, st>>>(counts, n, tile_sums, starts, packed_info);
  return cednerf_check_launch("cednerf_exclusive_scan", 3);
}

// The scan for fixed-capacity buffers: offsets int64[n + 1] = min(exclusive prefix sums, capacity) (offsets[n] = the
// clamped total), totals int64[2] = {min(total, capacity), total}.  Nothing has to be read back by the host: kernels
// downstream take their live count from totals[0] and per-ray ranges from `offsets`.
CEDNERF_EXPORT int cednerf_exclusive_scan_capped(const int32_t* counts, int64_t n, int64_t capacity, int64_t* offsets,
                                                 int64_t* totals, void* workspace, void* stream) {
  CEDNERF_REQUIRE(n >= 0 && capacity >= 0 && offsets && totals && workspace, "bad arguments");
  cudaStream_t st = (cudaStream_t)stream;
  if (n == 0) {
    cudaMemsetAsync(offsets, 0, 8, st);
    cudaMemsetAsync(totals, 0, 16, st);
    return 0;
  }
  const int64_t tiles = (n + SCAN_TILE - 1) / SCAN_TILE;
  // one pass: ticket counter + one state word per tile (workspace holds 8 (tiles + 1) bytes), zeroed by a memset node
  cudaMemsetAsync(workspace, 0, 8 * (size_t)(tiles + 1), st);
  scan_capped_onepass_kernel<<<(unsigned)tiles, SCAN_THREADS, 0, st>>>(counts, n, capacity, offsets, totals,
                                                                       (unsigned long long*)workspace);
  return cednerf_check_launch("cednerf_exclusive_scan_capped", 1);
}

// ---- marching rounds of render_image_test kept on the device (cednerf/utils.py:224-318) ---------------------------
// state (int32 [8], device): [0] alive rays of this round, [1] k = samples per ray this round, [2] samples per ray marched
// so far ("done"), [3] rays appended to the NEXT round's list by the compositing kernel, [4] round index, [5] 1 once the
// loop is over.  total (int64 [1]) accumulates the rounds' sample totals.
namespace {
__global__ void render_round_begin_kernel(int32_t* __restrict__ state, int64_t n_rays, int max_samples, int min_samples,
                                          const int64_t* __restrict__ prev_totals, int64_t* __restrict__ total) {
  cednerf_round_begin(state, n_rays, max_samples, min_samples, prev_totals, total);
}
}  // namespace

// start of a round: state[0] <- state[3] (rays the previous round kept alive; the caller seeds state[3] = n_rays),
// k and done are advanced as the reference's host loop does; prev_totals (nullable): the previous round's scan totals
CEDNERF_EXPORT int cednerf_render_round_begin(int32_t* state, int64_t n_rays, int max_samples, int min_samples,
                                              const int64_t* prev_totals, int64_t* total, void* stream) {
  CEDNERF_REQUIRE(state && n_rays >= 0 && max_samples > 0 && min_samples > 0, "bad arguments");
  render_round_begin_kernel<<<1, 1, 0, (cudaStream_t)stream>>>(state, n_rays, max_samples, min_samples, prev_totals, total);
  return cednerf_check_launch("cednerf_render_round_begin");
}

// One marching pass of a round over the alive list (first state[0] entries of `alive`; n_bound >= state[0] sizes the
// launch).  near_term [n_rays]: the rays' start planes on entry, their termination planes once both passes have run: the
// count pass (fill == 0) writes them for the rays within the run limit, the fill pass for the rays over it (it marches
// those again from their start planes).  Per-slot outputs: n_samples, runs.  fill == 1: the full-march fill for the slots
// flagged in slot_mask (rays over the run limit), at offsets[slot].  It writes a ray's whole count, so the packed
// buffers must hold every sample of the round: the rounds of render_image_test allocate n_rays * max(1, min_samples) >=
// n_alive * k (utils._render_rounds_gen) and never truncate.  The sample limit k is read from state[1].
CEDNERF_EXPORT int cednerf_march_round(int fill, const float* rays_o, const float* rays_d, int64_t n_bound,
                                       const uint32_t* occ_bits, const float* aabbs, int n_levels, int resolution,
                                       float* near_term, float far_const, float step_size, float cone_angle,
                                       const float* t_sorted, const int64_t* t_indices, const uint8_t* hits,
                                       const int32_t* alive, const int32_t* state, const uint8_t* slot_mask,
                                       const int64_t* offsets, float* t_starts, float* t_ends, int64_t* ray_indices,
                                       int32_t* n_samples, float* run_t, int32_t* run_n, int32_t* n_runs, int run_cap,
                                       const uint32_t* occ_coarse, void* stream) {
  CEDNERF_REQUIRE((int64_t)n_levels * resolution * resolution * resolution < (1ll << 31), "occupancy grid too large");
  CEDNERF_REQUIRE(n_bound >= 0 && n_levels >= 1 && n_levels <= MARCH_MAX_LEVELS && resolution >= 1 && alive && state &&
                      near_term && t_sorted && t_indices && hits,
                  "bad arguments");
  CEDNERF_REQUIRE(fill ? (slot_mask && offsets && t_starts && t_ends && ray_indices)
                       : (n_samples && run_t && run_n && n_runs && run_cap > 0 && step_size > 0.0f),
                  "count pass: counts and runs; fill pass: mask, offsets and packed outputs");
  if (n_bound == 0) return 0;
  MarchArgs a{};
  a.rays_o = rays_o, a.rays_d = rays_d, a.n_rays = n_bound, a.occ_bits = occ_bits, a.aabbs = aabbs;
  a.n_levels = n_levels, a.res = resolution, a.near = near_term, a.far = nullptr, a.near_const = 0.0f, a.far_const = far_const;
  a.step_size = step_size, a.cone_angle = cone_angle, a.limit = 0, a.mask = fill ? slot_mask : nullptr;
  a.t_sorted = t_sorted, a.t_indices = t_indices, a.hits = hits;
  a.sm_starts = offsets, a.t_starts = t_starts, a.t_ends = t_ends, a.ray_indices = ray_indices;
  a.n_samples = fill ? nullptr : n_samples, a.termination = near_term;
  a.run_t = fill ? nullptr : run_t, a.run_n = fill ? nullptr : run_n, a.n_runs = fill ? nullptr : n_runs, a.run_cap = run_cap;
  a.order = alive, a.n_active_dev = state, a.limit_dev = state + 1, a.by_slot = 1;
  a.coarse = (resolution % 4 == 0) ? occ_coarse : nullptr;
  const unsigned grid = cednerf_blocks(n_bound, 128);
  if (a.coarse) {
    if (fill) march_kernel<true, true><<<grid, 128, 0, (cudaStream_t)stream>>>(a);
    else march_kernel<false, true><<<grid, 128, 0, (cudaStream_t)stream>>>(a);
  } else {
    if (fill) march_kernel<true><<<grid, 128, 0, (cudaStream_t)stream>>>(a);
    else march_kernel<false><<<grid, 128, 0, (cudaStream_t)stream>>>(a);
  }
  return cednerf_check_launch("cednerf_march_round");
}

// packed fill of a round from the recorded runs: slot-indexed offsets (cednerf_exclusive_scan_capped over n_samples),
// ray ids taken from the alive list; overflow[slot] = 1 where the run list did not fit (-> cednerf_march_round(fill = 1))
CEDNERF_EXPORT int cednerf_march_fill_runs_round(int64_t n_bound, const int64_t* offsets, const int32_t* n_samples,
                                                 const float* run_t, const int32_t* run_n, const int32_t* n_runs,
                                                 int run_cap, float step_size, float cone_angle, const int32_t* alive,
                                                 const int32_t* state, float* t_starts, float* t_ends,
                                                 int64_t* ray_indices, uint8_t* overflow, void* stream) {
  CEDNERF_REQUIRE(n_bound >= 0 && run_cap > 0 && step_size > 0.0f && offsets && n_samples && alive && state, "bad arguments");
  CEDNERF_REQUIRE((((uintptr_t)t_starts | (uintptr_t)t_ends | (uintptr_t)ray_indices) & 15) == 0,
                  "packed outputs must be 16-byte aligned");
  if (n_bound == 0) return 0;
  march_fill_runs_kernel<<<cednerf_blocks(n_bound, 128), 128, 0, (cudaStream_t)stream>>>(
      n_bound, offsets, run_t, run_n, n_runs, run_cap, step_size, cone_angle, t_starts, t_ends, ray_indices, overflow,
      n_samples, alive, state);
  return cednerf_check_launch("cednerf_march_fill_runs_round");
}
