/*
 * cednerf_b200 — C ABI of libcednerf_b200.so (sm_100a).
 *
 * The reference (Linyou/Ced-NeRF) has no FFI of its own: its per-ray rendering hot path calls three
 * third-party CUDA/JIT packages from Python (nerfacc, tiny-cuda-nn, Taichi).  The entry points below are
 * what a Python binding for that path binds instead; each one names the reference call it stands behind.
 * INTEGRATION.md shows the ctypes stubs.
 *
 * Conventions
 *   - every pointer is a DEVICE pointer unless its name ends in _host or its type is a descriptor struct
 *     (descriptors are small host structs passed by pointer and copied at launch);
 *   - the caller owns all memory, including workspaces; the library never allocates or frees device memory
 *     and keeps no pointer after returning;
 *   - functions only enqueue work on `stream` (a cudaStream_t) and return; no device synchronisation;
 *   - return value 0 = ok, > 0 = cudaError_t, < 0 = library error (CEDNERF_ERR_*);
 *     cednerf_last_error() returns a thread-local message;
 *   - nullable arguments are marked (nullable).
 */
#ifndef CEDNERF_B200_H
#define CEDNERF_B200_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define CEDNERF_ERR_BAD_ARG (-1)
#define CEDNERF_ERR_UNSUPPORTED (-2)

#define CEDNERF_MAX_LEVELS 32
#define CEDNERF_MLP_MAX_LAYERS 5

/* ---- library ------------------------------------------------------------------------------------ */
const char* cednerf_last_error(void);
int cednerf_abi_version(void);
int cednerf_check_device(void); /* 0 iff the current device is compute capability 10.x */
int64_t cednerf_launch_count(void); /* kernels launched by this library so far in this process */

/* ---- K1: marching --------------------------------------------------------------------------------
 * nerfacc.ray_aabb_intersect — reference call site cednerf/utils.py:215 */
int cednerf_ray_aabb_intersect(const float* rays_o, const float* rays_d, int64_t n_rays, const float* aabbs,
                               int n_levels, float near_plane, float far_plane, float miss_value, float* t_mins,
                               float* t_maxs, uint8_t* hits, void* stream);
/* torch.sort of cat([t_mins, t_maxs]) — cednerf/utils.py:219-225 (stable; ties keep the lower slot) */
int cednerf_sort_boundaries(const float* t_mins, const float* t_maxs, int64_t n_rays, int n_levels, float* t_sorted,
                            int64_t* t_indices, void* stream);
/* OccGridEstimator.binaries (bool bytes [L,R,R,R]) -> 1 bit per cell, same cell order */
int cednerf_occ_pack_bits(const uint8_t* binaries, int64_t n_cells, uint32_t* bits /*ceil(n_cells / 32) words*/, void* stream);
/* binaries = occs > *threshold_dev, plus the bit field (last line of OccGridEstimator._update; train_real.py:332-336) */
int cednerf_occ_threshold_pack(const float* occs, int64_t n_cells, const float* threshold_dev, uint8_t* binaries,
                               uint32_t* bits, void* stream);
/* OccGridEstimator.mark_invisible_cells(K, c2w, width, height, near_plane) — train_real.py:205-211 (nerfacc): occs = -1
 * for cells no camera sees at depth >= near_plane or some camera sees closer than that, else 0.
 * K [n_K,3,3] (n_K == 1 or n_cams), c2w [n_cams, c2w_rows (3|4), 4], occs [n_levels * resolution^3]. */
int cednerf_occ_mark_invisible(const float* K, int n_K, const float* c2w, int n_cams, int c2w_rows, const float* aabbs,
                               int n_levels, int resolution, int width, int height, float near_plane, float* occs,
                               void* stream);
/* nerfacc.traverse_grids — cednerf/utils.py:245-264 (eval) and inside OccGridEstimator.sampling,
 * cednerf/utils.py:115-125 (train).  fill == 0 counts (n_intervals / n_samples / termination);
 * fill == 1 writes at iv_starts / sm_starts.  near/far: per-ray arrays or (nullable) -> the constants.
 * t_sorted / t_indices / hits (nullable, all or none): computed in-kernel when absent.
 * Output groups (each nullable): nerfacc intervals (iv_*), nerfacc samples (sm_*), packed
 * (t_starts, t_ends, ray_indices). */
/* coarse occupancy for the marcher's empty-space skip: one bit per 4x4x4 block of cells (resolution % 4 == 0),
 * ceil(n_levels (resolution / 4)^3 / 32) words.  Passing it changes no result: inside an empty block the DDA is stepped
 * with the same fp32 additions, only the per-cell look-ups are skipped. */
int cednerf_occ_coarsen(const uint32_t* occ_bits, int n_levels, int resolution, uint32_t* coarse, void* stream);
int cednerf_ray_coherence_keys(const float* rays_d, int64_t n_rays, int32_t* keys, void* stream);
/* order [n] = permutation grouping the rays by the leading 14 bits of that key (bucket order: histogram, scan, scatter;
 * workspace 64 KB) - the ray_order argument of cednerf_march */
int cednerf_ray_coherence_order(const int32_t* keys, int64_t n_rays, int32_t* order, void* workspace, void* stream);
int cednerf_march(int fill, const float* rays_o, const float* rays_d, int64_t n_rays, const uint32_t* occ_bits,
                  const float* aabbs, int n_levels, int resolution, const float* near_planes, const float* far_planes,
                  float near_const, float far_const, float step_size, float cone_angle, int steps_limit,
                  const uint8_t* rays_mask, const float* t_sorted, const int64_t* t_indices, const uint8_t* hits,
                  const int64_t* iv_starts, const int64_t* sm_starts, float* iv_vals, uint8_t* iv_left,
                  uint8_t* iv_right, int64_t* iv_ray, float* sm_vals, int64_t* sm_ray, uint8_t* sm_valid,
                  float* t_starts, float* t_ends, int64_t* ray_indices, int32_t* n_intervals, int32_t* n_samples,
                  float* termination, float* run_t /*nullable: [n,run_cap], count pass only*/,
                  int32_t* run_n /*[n,run_cap]*/, int32_t* n_runs /*[n]*/, int run_cap,
                  const int32_t* ray_order /*nullable: thread i marches ray ray_order[i], outputs stay indexed by ray*/,
                  const uint32_t* occ_coarse /*nullable: cednerf_occ_coarsen*/, void* stream);
/* Packed fill that replays the runs a count pass recorded (first left edge + length of every stretch of back-to-back
 * samples): no second grid traversal.  overflow[r] = 1 where a ray had more than run_cap runs; fill those rays with
 * cednerf_march(fill = 1, rays_mask = overflow). */
int cednerf_march_fill_runs(int64_t n_rays, const int64_t* sm_starts, const float* run_t, const int32_t* run_n,
                            const int32_t* n_runs, int run_cap, float step_size, float cone_angle, float* t_starts,
                            float* t_ends, int64_t* ray_indices, uint8_t* overflow, void* stream);
/* The same fill into buffers of a FIXED CAPACITY (no host read of the sample total - SURVEY.md 7 "hard parts"): offsets
 * [n_rays + 1] and the drop rule come from cednerf_exclusive_scan_capped, n_samples = the unclamped per-ray counts. */
int cednerf_march_fill_runs_capped(int64_t n_rays, const int64_t* offsets, const int32_t* n_samples, const float* run_t,
                                   const int32_t* run_n, const int32_t* n_runs, int run_cap, float step_size,
                                   float cone_angle, float* t_starts, float* t_ends, int64_t* ray_indices,
                                   uint8_t* overflow, void* stream);
/* cumsum between the two traversal passes (nerfacc: torch.cumsum + .item()); stays on the device */
int64_t cednerf_scan_workspace_bytes(int64_t n);
int cednerf_exclusive_scan(const int32_t* counts, int64_t n, int64_t* starts /*nullable*/,
                           int64_t* packed_info /*nullable, [n,2]*/, int64_t* total /*nullable*/, void* workspace,
                           void* stream);
/* the scan for fixed-capacity buffers: offsets [n + 1] = min(exclusive prefix sums, capacity); totals [2] =
 * {min(total, capacity), total}.  Kernels downstream read their live count from totals[0] (their `n_device`). */
int cednerf_exclusive_scan_capped(const int32_t* counts, int64_t n, int64_t capacity, int64_t* offsets, int64_t* totals,
                                  void* workspace, void* stream);

/* ---- K2: hash-grid encoders ------------------------------------------------------------------------ */
typedef struct CednerfGridLevels {
  int n_levels;
  float scale[CEDNERF_MAX_LEVELS];     /* base * exp(l * log_b) - 1   (hash_encoder_half.py:96-103) */
  uint32_t res[CEDNERF_MAX_LEVELS];    /* ceil(scale) + 1 */
  uint32_t size[CEDNERF_MAX_LEVELS];   /* min(max_params, align8(res^3)) */
  uint32_t offset[CEDNERF_MAX_LEVELS]; /* prefix sum of size */
  uint32_t hashed[CEDNERF_MAX_LEVELS]; /* res^3 > size */
} CednerfGridLevels;
/* tcnn.Encoding(HashGrid) forward — cednerf/model.py:384; Taichi twin hash_encoder_half.py:112-161.
 * table: fp16 [sum size, 2]; out: fp16, row stride out_stride (>= 2*n_levels) */
int cednerf_hashgrid_fwd(const float* x, int x_stride, int64_t n, const void* table_f16,
                         const CednerfGridLevels* levels, void* out_f16, int out_stride, void* stream);
/* backward: g_table fp32 [sum size, 2] is accumulated into (caller zeroes); g_x fp32 [n,3] (nullable) */
int cednerf_hashgrid_bwd(const float* x, int x_stride, int64_t n, const void* table_f16,
                         const CednerfGridLevels* levels, const void* dy, int dy_stride, int dy_is_f16,
                         float* g_table /*nullable*/, float* g_x /*nullable*/, void* stream);
/* table gradient from a level-major fp16 gradient dy_lm[level][sample][2] (written by the fused density-net backward) */
int cednerf_hashgrid_bwd_table_lm(const float* x, int x_stride, int64_t n, const CednerfGridLevels* levels,
                                  const void* dy_lm_f16, float* g_table, void* stream);
/* 4-D (xyz+t, 4 key-frames x 2 features per entry) — hash_encoder_inter.py:121-199 / :202-275 */
int cednerf_hashgrid4d_fwd(const float* xyzt, int x_stride, int64_t n, const void* table_f16,
                           const CednerfGridLevels* levels, void* out_f16, int out_stride, int taichi_compat,
                           void* stream);
int cednerf_hashgrid4d_bwd(const float* xyzt, int x_stride, int64_t n, const CednerfGridLevels* levels, const void* dy,
                           int dy_stride, int dy_is_f16, float* g_table, int taichi_compat, void* stream);
/* fp32 master -> fp16 working copy (hash_encoder_half.py:381-385 does this on every call) */
int cednerf_cast_f32_to_f16(const float* src, void* dst_f16, int64_t n, void* stream);

/* ---- parameter-free encodings ----------------------------------------------------------------------- */
/* tcnn Frequency(n): out[j] = sin(2^k pi x_dim + phase), dim = j/(2n), k = (j/2)%n, phase = (j%2) pi/2 —
 * cednerf/model.py:205-213, :316-319, :333-336.  Columns [width, pad_to) are filled with pad_value
 * (tcnn pads MLP inputs to a multiple of 16 with 1.0). */
int cednerf_frequency_fwd(const float* x, int n_dims, int64_t n, int n_frequencies, void* out_f16, int out_stride,
                          int pad_to, float pad_value, void* stream);
int cednerf_frequency_bwd(const float* x, int n_dims, int64_t n, int n_frequencies, const void* dy, int dy_stride,
                          int dy_is_f16, float* dx, void* stream);
/* tcnn SphericalHarmonics(degree 2), input in [0,1]^3 — cednerf/model.py:226-239, :450-455 */
int cednerf_sh2_fwd(const float* d01, int64_t n, void* out_f16, int out_stride, void* stream);
/* SinusoidalEncoder(1,0,4,True) (move_norm == NULL) / SinusoidalEncoderWithExp(1,0,4,True) —
 * cednerf/encoder.py:28-44, :69-90; out fp32 [n,9] */
int cednerf_time_embed(const float* t, const float* move_norm /*nullable*/, int64_t n, float* out, void* stream);

/* ---- K3: fully fused 64-wide MLPs (tcgen05) -------------------------------------------------------- */
typedef struct CednerfMlpDesc {
  int n_layers;                          /* hidden layers + 1 */
  int dim_in[CEDNERF_MLP_MAX_LAYERS];    /* padded to 16; 64 for every layer but the first */
  int dim_out[CEDNERF_MLP_MAX_LAYERS];   /* 64 for hidden layers; padded n_out for the last */
  int param_off[CEDNERF_MLP_MAX_LAYERS]; /* element offset of W_l [dim_out, dim_in] in the flat fp32 params */
  int image_off[CEDNERF_MLP_MAX_LAYERS]; /* byte offset of W_l's image: dim_out rows x 128 B, 128-byte swizzle */
  int image_bytes;
} CednerfMlpDesc;
/* tcnn.Network — cednerf/model.py:200-222, :280-290, :292-309, :312-344 */
int cednerf_mlp_pack_weights(const float* params, const CednerfMlpDesc* desc, void* image, void* stream);
int cednerf_mlp_fwd(const void* x_f16, const void* weight_image, const CednerfMlpDesc* desc, int64_t n, void* out_f16,
                    void* hidden_f16 /*nullable: [n_layers-1][n][64]*/, void* stream);
int cednerf_mlp_bwd(const void* x_f16, const void* hidden_f16, const void* d_out_f16, const void* weight_image,
                    const CednerfMlpDesc* desc, int64_t n, void* d_x /*nullable*/, int dx_is_f32,
                    float* d_params /*nullable, accumulated into*/,
                    void* d_hidden_f16 /*nullable: [n_layers-1][n][64] masked hidden gradients, for inspection*/,
                    void* stream);

/* ---- fused field query (K2 + K3 in one kernel) -------------------------------------------------------- */
typedef struct CednerfFieldDesc {
  float aabb[6];
  float moving_step;
  int use_div_offsets;   /* deformation net emits 6 values: move = o[:3]*MS + tanh(o[3:])*MS (model.py:358-363) */
  int time_mode;         /* 0 none, 1 SinusoidalEncoder, 2 SinusoidalEncoderWithExp */
  int time_before_sigma; /* 1: density input = [hash | time9]; 0: colour input = [sh4 | feat15 | time9] */
  CednerfMlpDesc f1, f2, f3; /* deformation (xyz_wrap), density (mlp_base), colour (mlp_head) */
  CednerfMlpDesc f4;         /* hash-feature predictor (mlp_feat_prediction, -f); n_layers == 0 when absent */
  CednerfGridLevels levels;
} CednerfFieldDesc;
/* DNGPradianceField.query_density / .forward without autograd (cednerf/model.py:367-488) fused with the position
 * closure of cednerf/utils.py:74-104.  Samples: packed ray samples (ray_indices, t_starts, t_ends, rays_o, rays_d;
 * timestamps indexed by ray) or explicit points (x, dirs; timestamps indexed by point); t_stride 0 = one timestamp
 * for all.  rgb == NULL: density only. */
int cednerf_field_fwd(const int64_t* ray_indices, const float* t_starts, const float* t_ends, const float* rays_o,
                      const float* rays_d, const float* x, const float* dirs, const float* timestamps, int t_stride,
                      int64_t n, const void* image_deform, const void* image_density, const void* image_colour,
                      const void* table_f16, const CednerfFieldDesc* desc, float* sigma, float* rgb,
                      const int64_t* n_device /*nullable: live sample count on the device, n = capacity*/, void* stream);

/* Occupancy-grid update of one level, fused (SURVEY.md 8f N1; nerfacc OccGridEstimator._update as the reference calls
 * it, train_real.py:324-336, occ_eval_fn(x) = query_density(x, t)["density"] * render_step_size): one jittered point per
 * entry of `cells` (NULL: every cell of the level once - the warm-up case) goes through deformation net, hash grid and
 * density net, and occs_level[cell] = max(occs_level[cell] * ema_decay, sigma * step_scale) is written by the same
 * kernel.  level_aabb: HOST array of 6 floats.  Cells with duplicates: pass zero-initialised cand [R^3] and touched [R^3]
 * (the largest candidate wins, as scatter-amax; both come back cleared). */
int cednerf_occ_update_level(const int64_t* cells /*nullable*/, int64_t n, const float* jitter /*[n,3]*/,
                             const float* timestamps /*[n]*/, const float* level_aabb /*host, [6]*/, int resolution,
                             float step_scale, float ema_decay, const void* image_deform, const void* image_density,
                             const void* table_f16, const CednerfFieldDesc* desc, float* occs_level,
                             float* cand /*nullable*/, uint8_t* touched /*nullable*/, void* stream);

/* DNGPradianceField.forward in training (cednerf/model.py:468-488, return_interal=True) on packed ray samples, and its
 * backward.  `saved` (cednerf_field_saved_bytes) carries the activations; the backward accumulates into the fp32
 * parameter gradients (tcnn flat layout) and the fp32 hash-table gradient (caller zeroes), using `work`
 * (cednerf_field_bwd_workspace_bytes).  latent / d_latent: huber loss of the feature predictor against the hash
 * features, [n,32] (nullable: no predictor). */
int64_t cednerf_field_saved_bytes(const CednerfFieldDesc* desc, int64_t n);
int64_t cednerf_field_bwd_workspace_bytes(const CednerfFieldDesc* desc, int64_t n);
int cednerf_field_train_fwd(const int64_t* ray_indices, const float* t_starts, const float* t_ends, const float* rays_o,
                            const float* rays_d, const float* timestamps, int t_stride, int64_t n,
                            const void* image_deform, const void* image_density, const void* image_colour,
                            const void* image_predict, const void* table_f16, const CednerfFieldDesc* desc, float* sigma,
                            float* rgb, float* latent, uint8_t* selector, float* move, void* saved,
                            const int32_t* sample_order /*nullable: cednerf_sample_order*/,
                            const int64_t* n_device /*nullable: live sample count on the device, n = capacity*/,
                            void* stream);
int cednerf_field_train_bwd(const int64_t* ray_indices, const float* t_starts, const float* t_ends, const float* rays_o,
                            const float* rays_d, const float* timestamps, int t_stride, int64_t n,
                            const void* image_deform, const void* image_density, const void* image_colour,
                            const void* image_predict, const void* table_f16, const CednerfFieldDesc* desc,
                            const float* sigma, const float* rgb, const uint8_t* selector, const void* saved,
                            const float* d_sigma, const float* d_rgb, const float* d_latent, void* work,
                            float* d_params_deform, float* d_params_density, float* d_params_colour,
                            float* d_params_predict, float* g_table, int phase,
                            const int32_t* sample_order /*nullable, the forward's*/,
                            const int64_t* n_device /*nullable, as in the forward*/, void* stream);
/* phase: 0 = the whole backward; 1 = colour and density nets + table gradient (g_table is complete on return: a
 * data-parallel caller starts its all-reduce here); 2 = the rest (predictor net, dL/dx of the encoding, deformation net). */

/* Spatial bucket order of packed samples for the two calls above (csrc/sample_order.cu): `order` [n] int32 walks the live
 * samples bucket by bucket of a 128^3 Morton grid over the box [lo, hi] (position = o + d (t0 + t1) / 2), so that the
 * lanes of a warp are neighbours in space and the hash-grid gathers of the coarse and middle levels coalesce.  With an
 * order, kernel-internal sample s reads / writes entry order[s] of every per-sample array named in the signatures above;
 * `saved` and `work` are laid out by s.  workspace: cednerf_sample_order_workspace_bytes(n).  n_device nullable. */
int64_t cednerf_sample_order_workspace_bytes(int64_t n);
int cednerf_sample_order(const int64_t* ray_indices, const float* t_starts, const float* t_ends, const float* rays_o,
                         const float* rays_d, int64_t n, const int64_t* n_device, float lo0, float lo1, float lo2,
                         float hi0, float hi1, float hi2, void* workspace, int32_t* order, void* stream);

/* ---- K4: compositing ------------------------------------------------------------------------------- */
/* offsets[r] = first sample of ray r (ray_indices sorted); offsets[n_rays] = n_samples */
int cednerf_ray_offsets(const int64_t* ray_indices, int64_t n_samples, int64_t n_rays, int64_t* offsets, void* stream);
/* accumulate_inplace: 0 = write colours/opacity/depth (normalised depth, background blend); 1 = add the raw sums into
 * them (accumulate_along_rays_); 2 = as 1 with prefix transmittance 1 - opacity[ray] read before the update (one marching
 * round of render_image_test, cednerf/utils.py:274-299).
 * nerfacc.render_weight_from_density (+ accumulate_along_rays x3, depth normalise, background) —
 * cednerf/render.py:81-87, :158-174; prefix_trans / in-place form cednerf/utils.py:274-299 */
int cednerf_composite_fwd(const float* t_starts, const float* t_ends, const float* sigmas, const float* rgbs,
                          const float* prefix_trans, const int64_t* offsets, const float* bkgd, int bkgd_stride,
                          int64_t n_samples, int64_t n_rays, float* weights, float* trans, float* alphas,
                          float* colors, float* opacity, float* depth, float* depth_raw, int accumulate_inplace,
                          float depth_eps, void* stream);
int cednerf_composite_bwd(const float* t_starts, const float* t_ends, const float* rgbs, const float* trans,
                          const float* alphas, const int64_t* offsets, const float* bkgd, int bkgd_stride,
                          int64_t n_samples, int64_t n_rays, const float* opacity, const float* depth_raw,
                          const float* g_colors, const float* g_opacity, const float* g_depth, const float* g_weights,
                          const float* g_trans, const float* g_alphas, float* g_sigmas, float* g_rgbs, float depth_eps,
                          void* stream);
/* nerfacc.render_visibility_from_density — inside OccGridEstimator.sampling (cednerf/utils.py:115-125) */
int cednerf_visibility_mask(const float* t_starts, const float* t_ends, const float* sigmas, const int64_t* offsets,
                            int64_t n_samples, int64_t n_rays, float early_stop_eps, float alpha_thre, uint8_t* keep,
                            int32_t* kept_counts /*nullable: per-ray number of kept samples*/, void* stream);
/* the compaction that follows it in .sampling: kept samples of every ray, in order, to out_starts[ray] + rank
 * (out_starts = exclusive scan of kept_counts) */
int cednerf_compact_samples(const uint8_t* keep, const int64_t* offsets, const int64_t* out_starts, const float* t_starts,
                            const float* t_ends, int64_t n_samples, int64_t n_rays, int64_t* ray_indices_out,
                            float* t_starts_out, float* t_ends_out, void* stream);
/* ... into outputs of a fixed capacity: out_offsets [n_rays + 1] from cednerf_exclusive_scan_capped over kept_counts */
int cednerf_compact_samples_capped(const uint8_t* keep, const int64_t* offsets, const int64_t* out_offsets,
                                   const float* t_starts, const float* t_ends, int64_t n_samples, int64_t n_rays,
                                   int64_t* ray_indices_out, float* t_starts_out, float* t_ends_out, void* stream);
/* ---- marching rounds of render_image_test kept on the device (cednerf/utils.py:224-318): the alive-ray list, the
 * per-round sample limit k and the termination test never leave the GPU; the host only enqueues rounds and looks at a
 * lagged copy of `state` to know when to stop.  state int32[8]: [0] alive rays of this round, [1] k, [2] samples per ray
 * marched so far, [3] rays kept alive for the next round (seed with n_rays), [4] round index, [5] 1 when the loop is
 * over. */
int cednerf_render_round_begin(int32_t* state, int64_t n_rays, int max_samples, int min_samples,
                               const int64_t* prev_totals /*nullable*/, int64_t* total /*nullable, += prev_totals[0]*/,
                               void* stream);
int cednerf_march_round(int fill, const float* rays_o, const float* rays_d, int64_t n_bound, const uint32_t* occ_bits,
                        const float* aabbs, int n_levels, int resolution, float* near_term /*[n_rays] in: start planes. out (count pass, then fill pass for the rays over the run limit): termination planes*/, float far_const, float step_size, float cone_angle,
                        const float* t_sorted, const int64_t* t_indices, const uint8_t* hits, const int32_t* alive,
                        const int32_t* state, const uint8_t* slot_mask /*fill*/, const int64_t* offsets /*fill*/,
                        float* t_starts, float* t_ends, int64_t* ray_indices, int32_t* n_samples /*count, per slot*/,
                        float* run_t, int32_t* run_n, int32_t* n_runs, int run_cap,
                        const uint32_t* occ_coarse /*nullable*/, void* stream);
int cednerf_march_fill_runs_round(int64_t n_bound, const int64_t* offsets, const int32_t* n_samples, const float* run_t,
                                  const int32_t* run_n, const int32_t* n_runs, int run_cap, float step_size,
                                  float cone_angle, const int32_t* alive, const int32_t* state, float* t_starts,
                                  float* t_ends, int64_t* ray_indices, uint8_t* overflow, void* stream);
int cednerf_render_round_composite(const float* t_starts, const float* t_ends, const float* sigmas, const float* rgbs,
                                   const int64_t* offsets, const int32_t* alive, int32_t* round_state,
                                   const int32_t* slot_counts, int64_t n_bound, int k_hint, float early_stop_eps,
                                   float* colors, float* opacity, float* depth, int32_t* alive_flags /*[n_bound]*/,
                                   void* stream);
/* ordered compaction of the flagged slots into the next round's list (positions = cednerf_exclusive_scan_capped of the
 * flags): neighbouring lanes keep marching neighbouring pixels.  state[3] <- number of rays kept. */
int cednerf_render_round_compact(const int32_t* alive_flags, const int64_t* positions, const int32_t* alive,
                                 int64_t n_bound, int32_t* round_state, int32_t* next_alive, int64_t n_rays,
                                 int max_samples /*> 0: also begin the next round, as cednerf_render_round_begin*/,
                                 int min_samples, const int64_t* round_totals, int64_t* total, void* stream);
/* One marching round behind one call (the eight launches above, in the order render_image_test needs them): a frame is
 * 40-220 rounds, and eight calls with ~25 arguments each per round made the host the bound of the interleaved rounds.
 * Everything that stays the same over the rounds of a frame lives in the struct; `alive` / `next_alive` swap every
 * round and n_bound (an upper bound of the live part of `alive`) only shrinks. */
typedef struct CednerfRenderRound {
  const float* rays_o;
  const float* rays_d;
  int64_t n_rays;
  const uint32_t* occ_bits;
  const float* aabbs;
  int n_levels, resolution;
  float* near_term;
  float far_const, step_size, cone_angle, early_stop_eps;
  const float* t_sorted;
  const int64_t* t_indices;
  const uint8_t* hits;
  int32_t* state;
  int64_t* total;
  int32_t* n_samples;
  float* run_t;
  int32_t* run_n;
  int32_t* n_runs;
  const uint32_t* occ_coarse;
  int64_t capacity;
  int64_t* offsets;
  int64_t* totals;
  void* scan_workspace;
  float* t_starts;
  float* t_ends;
  int64_t* ray_indices;
  uint8_t* overflow;
  const float* timestamps;
  const void* image_deform;
  const void* image_density;
  const void* image_colour;
  const void* table_f16;
  const CednerfFieldDesc* desc;
  float* sigma;
  float* rgbs;
  float* colors;
  float* opacity;
  float* depth;
  int32_t* alive_flags;
  int64_t* positions;
  int64_t* position_totals;
  int run_cap, k_hint, max_samples, min_samples;
} CednerfRenderRound;
int64_t cednerf_render_round_bytes(void);
int cednerf_render_round(const CednerfRenderRound* round, int64_t n_bound, const int32_t* alive, int32_t* next_alive,
                         void* stream);
/* nerfacc.accumulate_along_rays / accumulate_along_rays_ — cednerf/render.py:158-169, cednerf/utils.py:282-299 */
int cednerf_accumulate_fwd(const float* weights, const float* values /*nullable*/, int n_channels,
                           const int64_t* offsets, int64_t n_samples, int64_t n_rays, float* outputs, int inplace,
                           void* stream);
int cednerf_accumulate_bwd(const float* weights, const float* values /*nullable*/, int n_channels,
                           const int64_t* ray_indices, int64_t n_samples, const float* g_outputs,
                           float* g_weights /*nullable*/, float* g_values /*nullable*/,
                           const int64_t* n_device /*nullable: live sample count, n_samples = capacity*/, void* stream);


/* ------------------------------------------------------------------------------------------------------------------
 * Optimiser step of the training loop (SURVEY.md 8f N2): grad_scaler.step(optimizer) with apex.optimizers.FusedAdam /
 * torch.optim.Adam(lr, eps=1e-15) — train_real.py:252, 267-274, 412-420.  Up to 8 parameter tensors per call. */
#define CEDNERF_OPT_MAX_TENSORS 8
typedef struct CednerfAdamTensors {
  int n_tensors;
  float* p[CEDNERF_OPT_MAX_TENSORS];        /* fp32 master parameters (updated in place) */
  const float* g[CEDNERF_OPT_MAX_TENSORS];  /* gradients (scaled by the loss scale) */
  float* m[CEDNERF_OPT_MAX_TENSORS];        /* exp_avg */
  float* v[CEDNERF_OPT_MAX_TENSORS];        /* exp_avg_sq */
  void* p16[CEDNERF_OPT_MAX_TENSORS];       /* nullable: fp16 working copy written with p (hash table) */
  int64_t n[CEDNERF_OPT_MAX_TENSORS];
  float lr[CEDNERF_OPT_MAX_TENSORS];
  float weight_decay[CEDNERF_OPT_MAX_TENSORS];
  int64_t chunk_begin[CEDNERF_OPT_MAX_TENSORS + 1]; /* scratch, filled by the library */
} CednerfAdamTensors;
/* GradScaler's inf/nan check (torch._amp_foreach_non_finite_check_and_unscale_ without the write-back):
 * *found_inf (device, caller-zeroed) = 1 when any gradient element is not finite. */
int cednerf_nonfinite_check(const CednerfAdamTensors* tensors, float* found_inf, void* stream);
/* unscale (g / *grad_scale) + Adam + fp16 copy in one pass; skipped when *found_inf != 0; *step (device float) advances
 * first (advance_step != 0) unless skipped and feeds the bias corrections.  adam_w_mode: apex's decoupled weight decay,
 * else torch Adam's L2 term (identical for weight_decay == 0, the reference's setting). */
int cednerf_adam_step(const CednerfAdamTensors* tensors, float* step, int advance_step, const float* grad_scale /*nullable*/,
                      const float* found_inf /*nullable*/, float beta1, float beta2, float eps, int adam_w_mode,
                      void* stream);


/* ------------------------------------------------------------------------------------------------------------------
 * Data-parallel optimiser step over NVLink peer memory (SURVEY.md 2.3 / 8e; no reference counterpart - the reference
 * trains on cuda:0 only, train_real.py:81).  One process per GPU.  Gradient, fp32 master and fp16 working copy of the
 * hash table live in cednerf_peer_alloc memory that the other ranks map with cednerf_ipc_open (the caller exchanges
 * the 64-byte handles).  cednerf_dp_barrier -> cednerf_dp_found_inf -> cednerf_dp_adam -> cednerf_dp_barrier, all
 * stream-ordered, replace gradient all-reduce + replicated Adam: every rank sums ITS range of all ranks' gradients
 * over NVLink (reduce-scatter), applies unscale + Adam to that range and stores the new fp32 / fp16 values into all
 * replicas (all-gather).  Up to 8 ranks. */
#define CEDNERF_DP_MAX_RANKS 8
typedef struct CednerfDpCtrl {   /* one per rank, in peer-visible memory, zero-initialised */
  uint32_t arrive[CEDNERF_DP_MAX_RANKS];
  float found_inf;               /* this rank's local non-finite flag (cednerf_nonfinite_check target) */
  uint32_t timed_out;            /* != 0: a barrier gave up waiting for a peer */
} CednerfDpCtrl;
typedef struct CednerfDpPeers {
  int world, rank;
  CednerfDpCtrl* ctrl[CEDNERF_DP_MAX_RANKS];  /* every rank's control block as mapped in this process */
} CednerfDpPeers;
typedef struct CednerfDpAdam {
  int world, rank;
  const float* grad[CEDNERF_DP_MAX_RANKS];    /* every rank's gradient buffer (same layout), as mapped here */
  int n_out;                                  /* replicas to update: world (broadcast) or 1 (local only) */
  float* p32_out[CEDNERF_DP_MAX_RANKS];       /* fp32 replicas; entry 0 = the local master (also the input), others nullable */
  void* p16_out[CEDNERF_DP_MAX_RANKS];        /* fp16 working copies (nullable entries) */
  float* m;                                   /* Adam moments of the owned range, indexed from lo */
  float* v;
  int64_t lo, hi;                             /* owned element range, lo % 4 == 0 */
  float lr, weight_decay, grad_div;           /* summed gradient / grad_div (world: average) */
  const float* grad_mc;                       /* nullable: multicast address of the gradient buffers (NVLS ld_reduce) */
  void* p16_mc;                               /* nullable: multicast address of the fp16 copies (NVLS multimem.st) */
} CednerfDpAdam;
#define CEDNERF_DP_SMALL_MAX 8
typedef struct CednerfDpSmall {   /* the small (MLP) tensors of a step: summed from all ranks in rank order, updated locally */
  int world, n_tensors;
  const float* grad[CEDNERF_DP_MAX_RANKS];   /* every rank's staging region of the small gradients, as mapped here */
  float* p[CEDNERF_DP_SMALL_MAX];
  float* m[CEDNERF_DP_SMALL_MAX];
  float* v[CEDNERF_DP_SMALL_MAX];
  int64_t off[CEDNERF_DP_SMALL_MAX];         /* element offset of the tensor's gradient inside the staging region */
  int64_t n[CEDNERF_DP_SMALL_MAX];
  float lr[CEDNERF_DP_SMALL_MAX];
  float weight_decay[CEDNERF_DP_SMALL_MAX];
  float grad_div;
  int64_t chunk_begin[CEDNERF_DP_SMALL_MAX + 1]; /* scratch */
} CednerfDpSmall;
int cednerf_peer_alloc(int64_t bytes, void** ptr);            /* cudaMalloc + zero fill */
int cednerf_peer_free(void* ptr);
int cednerf_ipc_export(void* ptr, void* handle64);            /* cudaIpcGetMemHandle of a cednerf_peer_alloc pointer */
int cednerf_ipc_open(const void* handle64, void** ptr);       /* map a peer's allocation on the current device */
int cednerf_ipc_close(void* ptr);
int64_t cednerf_dp_ctrl_bytes(void);
/* epoch increases by one per barrier, identically on all ranks; after timeout_ms the wait gives up and sets timed_out */
int cednerf_dp_barrier(const CednerfDpPeers* peers, uint32_t epoch, int timeout_ms, void* stream);
/* *found_out (nullable) = OR of all ranks' found_inf; *step (nullable) += 1 unless set */
int cednerf_dp_found_inf(const CednerfDpPeers* peers, float* found_out, float* step, void* stream);
int cednerf_dp_adam_small(const CednerfDpSmall* args, const float* step, const float* grad_scale /*nullable*/,
                          const float* found_inf /*nullable*/, float beta1, float beta2, float eps, int adam_w_mode,
                          void* stream);
int cednerf_dp_adam(const CednerfDpAdam* args, const float* step, const float* grad_scale /*nullable*/,
                    const float* found_inf /*nullable*/, float beta1, float beta2, float eps, int adam_w_mode, void* stream);

/* ------------------------------------------------------------------------------------------------------------------
 * Training loss of the reference loop for the canonical flags (train_real.py:369-409): F.mse_loss(rgb, pixels)
 * + w_entropy * acc-entropy (-ae, 1e-3) + w_rgbper * weighted per-sample colour loss (-wr, 1e-3) + latent_losses.mean()
 * (-f).  acc / rgbs / latent nullable (term absent).  sums: 4 doubles of workspace; loss: 1 float. */
int cednerf_training_loss_fwd(const float* rgb, const float* acc, const float* pixels, int64_t n_rays, const float* rgbs,
                              const float* weights, const int64_t* ray_indices, int64_t n_samples, const float* latent,
                              int n_latent, float w_entropy, float w_rgbper, double* sums, float* loss,
                              const int64_t* n_device /*nullable: live sample count, n_samples = capacity*/, void* stream);
/* its gradients times g_loss[0] (device scalar); any of d_rgb [R,3], d_acc [R], d_rgbs [S,3], d_latent [R,n_latent] null */
int cednerf_training_loss_bwd(const float* g_loss, const float* rgb, const float* acc, const float* pixels, int64_t n_rays,
                              const float* rgbs, const float* weights, const int64_t* ray_indices, int64_t n_samples,
                              int n_latent, float w_entropy, float w_rgbper, float* d_rgb, float* d_acc, float* d_rgbs,
                              float* d_latent, const int64_t* n_device /*nullable*/, void* stream);

/* ------------------------------------------------------------------------------------------------------------------
 * The steps either side of the hot path (SURVEY.md 8f N4).
 * Pixel -> ray generation (datasets/dnerf_3d_video_IS.py:330-358, datasets/dnerf_synthetic.py:196-224): camera_dirs =
 * [(x - cx + 0.5) / fx, (y - cy + 0.5) / fy * s, s], s = -1 for OpenGL cameras; directions = R camera_dirs; viewdirs =
 * directions / |directions|; origins = translation.  px / py nullable (ray i = pixel (i % width, i / width)); cam nullable
 * (pose index per ray into c2w [n_cams, c2w_rows, 4]); directions nullable. */
int cednerf_generate_rays(const int64_t* px, const int64_t* py, const int64_t* cam, const float* c2w, int c2w_rows,
                          float fx, float fy, float cx, float cy, int width, int opengl, int64_t n, float* origins,
                          float* viewdirs, float* directions, void* stream);
/* Distortion loss (cednerf/losses.py:4-11 = torch_efficient_distloss.flatten_eff_distloss on weights, interval
 * mid-points and lengths) of packed samples: sum_rays sum_i [d_i w_i^2 / 3 + 2 w_i (m_i W_i - M_i)] / (max ray + 1).
 * work: cednerf_distortion_workspace_bytes() (per-block fp64 partials: no atomics, deterministic); loss, inv_rays: one float
 * each (inv_rays feeds the backward).  Gradient w.r.t. the weights only. */
int64_t cednerf_distortion_workspace_bytes(void);
int cednerf_distortion_fwd(const float* weights, const float* t_starts, const float* t_ends, const int64_t* offsets,
                           int64_t n_rays, void* work, float* loss, float* inv_rays, void* stream);
int cednerf_distortion_bwd(const float* weights, const float* t_starts, const float* t_ends, const int64_t* offsets,
                           int64_t n_rays, const float* g_loss, const float* inv_rays, float* g_weights, void* stream);

/* ------------------------------------------------------------------------------------------------------------------
 * Importance-sampled training batches (SURVEY.md 8f N4): the training branch of SubjectLoader.fetch_data,
 * datasets/dnerf_3d_video_IS.py:401-445 (torch.multinomial over the ISG / IST weights of a uniform random subset) and
 * :447-497 (s x s pixel expansion, colour gather, ray generation).  torch.multinomial without replacement is a top-k of
 * weights / Exp(1) noise; the three calls below are that top-k and the batch assembly, with no host read.
 * keys[i] = bits of weights[subset ? subset[i] : i] / exp_noise[i] (0 for non-positive weights). */
int cednerf_importance_keys(const float* weights, const int64_t* subset /*nullable*/, const float* exp_noise, int64_t n,
                            uint32_t* keys, void* stream);
int64_t cednerf_topk_workspace_bytes(int64_t n);
/* out [k]: the positions (mapped through `subset` when given) of the k largest keys, in ascending position order; ties at
 * the threshold go to the lowest positions.  The int32 at byte 16 of the workspace is set to 1 when the k-th largest key
 * is zero (fewer than k positive weights: torch.multinomial raises there). */
int cednerf_topk_select(const uint32_t* keys, int64_t n, int64_t k, const int64_t* subset /*nullable*/, int64_t* out,
                        void* workspace, void* stream);
/* Ray j = sub * k + i (sub = ah * s + aw) is pixel (xsub * s + aw, ysub * s + ah) of image cells[i] / (hsub * wsub) with
 * hsub = height / s, wsub = width / s: rgb = images[image, y, x] / 255, the ray of cednerf_generate_rays, the image's
 * timestamp.  images uint8 [n_images, height, width, 3]; c2w [n_images, c2w_rows, 4]; timestamps [n_images];
 * image_id_out / pixel_index_out nullable. */
int cednerf_importance_batch(const int64_t* cells, int64_t k, int subsample, int width, int height, const uint8_t* images,
                             const float* c2w, int c2w_rows, float fx, float fy, float cx, float cy, int opengl,
                             const float* timestamps, float* origins, float* viewdirs, float* rgb, float* timestamps_out,
                             int64_t* image_id_out, int64_t* pixel_index_out, void* stream);

#ifdef __cplusplus
}
#endif
#endif /* CEDNERF_B200_H */
