// MS-SSIM of the evaluation after training (train_real.py:497-499 -> pytorch_msssim.ms_ssim v1.0, 4-D inputs, default
// window and weights), restated in oracle/metrics_ref.py:
//   per scale: mu = gf(X), gf = valid 11-tap Gaussian cross-correlation along H, then along W; sigma1_sq = gf(X*X) - mu1^2,
//   sigma2_sq = gf(Y*Y) - mu2^2, sigma12 = gf(X*Y) - mu1 mu2; cs_map = (2 sigma12 + C2) / (sigma1_sq + sigma2_sq + C2),
//   ssim_map = ((2 mu1 mu2 + C1) / (mu1^2 + mu2^2 + C1)) * cs_map; then X, Y = avg_pool2d(., 2, padding=[H % 2, W % 2])
//   (count_include_pad: a window over padding is still divided by 4).
//   value[n, c] = prod_{i<4} relu(mean cs_i)^w_i * relu(mean ssim_4)^w_4.
// One launch per scale over (tile, image x channel): the CTA stages its tile of X and Y with the halo in shared memory,
// runs the vertical then the horizontal pass for the five maps, writes one fp64 (ssim, cs) partial (no atomics: the
// result is the same from run to run) and the next scale's pooled planes.  One finishing launch reduces the partials in
// a fixed order.  The file is built with -fmad=false: a contraction of mu1_sq + mu2_sq into fma(mu1, mu1, mu2_sq) would
// break ms_ssim(x, x) == 1.
#include "common.cuh"

namespace {

#define SSIM_SCALES 5
#define SSIM_WIN 11
#define SSIM_TH 16                      // output rows of a tile
#define SSIM_TW 32                      // output columns of a tile
#define SSIM_SH (SSIM_TH + SSIM_WIN)    // staged rows: one above the tile (odd-side pooling), the tile, the 10-row halo
#define SSIM_SW (SSIM_TW + SSIM_WIN)
#define SSIM_VW (SSIM_TW + SSIM_WIN - 1)  // columns of the vertical pass
#define FINISH_THREADS 1024

struct SsimTaps {
  float g[SSIM_WIN];
};

struct SsimScale {
  const float* x;
  const float* y;
  int64_t xs[4], ys[4];  // element strides (n, c, h, w)
  int c, h, w;           // channels and this scale's sides
  float* px;             // next scale's planes [n * c, hn, wn] (null at the last scale)
  float* py;
  int hn, wn, pad_h, pad_w;
  double* partial;  // [n * c][tiles][2]: (sum ssim_map, sum cs_map) of each tile
  float c1, c2;
};

__global__ void __launch_bounds__(256) ms_ssim_scale_kernel(SsimScale a, SsimTaps t) {
  __shared__ float sx[SSIM_SH][SSIM_SW], sy[SSIM_SH][SSIM_SW];
  __shared__ float v[5][SSIM_TH][SSIM_VW];
  __shared__ double red[2][8];
  const int nc = blockIdx.y, n = nc / a.c, ch = nc % a.c;
  const int tiles_x = (a.w + SSIM_TW - 1) / SSIM_TW;
  const int r0 = (blockIdx.x / tiles_x) * SSIM_TH, c0 = (blockIdx.x % tiles_x) * SSIM_TW;
  const float* X = a.x + n * a.xs[0] + ch * a.xs[1];
  const float* Y = a.y + n * a.ys[0] + ch * a.ys[1];
  // stage rows r0-1 .. r0+TH+9 and columns c0-1 .. c0+TW+9; outside the image: 0 (only read by outputs that are skipped)
  for (int i = threadIdx.x; i < SSIM_SH * SSIM_SW; i += blockDim.x) {
    const int rr = i / SSIM_SW, cc = i % SSIM_SW;
    const int r = r0 - 1 + rr, col = c0 - 1 + cc;
    const bool in = r >= 0 && r < a.h && col >= 0 && col < a.w;
    sx[rr][cc] = in ? X[r * a.xs[2] + col * a.xs[3]] : 0.f;
    sy[rr][cc] = in ? Y[r * a.ys[2] + col * a.ys[3]] : 0.f;
  }
  __syncthreads();

  // next scale: the pooled pixel (i, j) belongs to the tile holding input pixel (2i, 2j).  Like torch's avg_pool2d the
  // window's pixels inside the image are summed row-major from 0 and the sum is divided by 4.
  if (a.px && threadIdx.x < (SSIM_TH / 2) * (SSIM_TW / 2)) {
    const int i = r0 / 2 + threadIdx.x / (SSIM_TW / 2), j = c0 / 2 + threadIdx.x % (SSIM_TW / 2);
    if (i < a.hn && j < a.wn) {
      float qx = 0.f, qy = 0.f;
#pragma unroll
      for (int dr = 0; dr < 2; ++dr) {
        const int r = 2 * i - a.pad_h + dr;
        if (r < 0 || r >= a.h) continue;
#pragma unroll
        for (int dc = 0; dc < 2; ++dc) {
          const int col = 2 * j - a.pad_w + dc;
          if (col < 0 || col >= a.w) continue;
          qx = __fadd_rn(qx, sx[r - r0 + 1][col - c0 + 1]);
          qy = __fadd_rn(qy, sy[r - r0 + 1][col - c0 + 1]);
        }
      }
      const int64_t o = ((int64_t)nc * a.hn + i) * a.wn + j;
      a.px[o] = __fdiv_rn(qx, 4.f);
      a.py[o] = __fdiv_rn(qy, 4.f);
    }
  }

  // vertical pass of the five maps x, y, x*x, y*y, x*y (products rounded to fp32 before filtering, as gf(X*X))
  for (int i = threadIdx.x; i < SSIM_TH * SSIM_VW; i += blockDim.x) {
    const int r = i / SSIM_VW, cc = i % SSIM_VW;
    float m0 = 0.f, m1 = 0.f, m2 = 0.f, m3 = 0.f, m4 = 0.f;
#pragma unroll
    for (int k = 0; k < SSIM_WIN; ++k) {
      const float xv = sx[r + 1 + k][cc + 1], yv = sy[r + 1 + k][cc + 1], g = t.g[k];
      m0 += g * xv;
      m1 += g * yv;
      m2 += g * (xv * xv);
      m3 += g * (yv * yv);
      m4 += g * (xv * yv);
    }
    v[0][r][cc] = m0, v[1][r][cc] = m1, v[2][r][cc] = m2, v[3][r][cc] = m3, v[4][r][cc] = m4;
  }
  __syncthreads();

  // horizontal pass and the two maps, in the order of the restatement
  double s_acc = 0.0, c_acc = 0.0;
  for (int i = threadIdx.x; i < SSIM_TH * SSIM_TW; i += blockDim.x) {
    const int r = i / SSIM_TW, cc = i % SSIM_TW;
    if (r0 + r >= a.h - (SSIM_WIN - 1) || c0 + cc >= a.w - (SSIM_WIN - 1)) continue;
    float h[5] = {0.f, 0.f, 0.f, 0.f, 0.f};
#pragma unroll
    for (int k = 0; k < SSIM_WIN; ++k) {
#pragma unroll
      for (int m = 0; m < 5; ++m) h[m] += t.g[k] * v[m][r][cc + k];
    }
    const float mu1 = h[0], mu2 = h[1];
    const float mu1_sq = mu1 * mu1, mu2_sq = mu2 * mu2, mu1_mu2 = mu1 * mu2;
    const float sigma1_sq = h[2] - mu1_sq, sigma2_sq = h[3] - mu2_sq, sigma12 = h[4] - mu1_mu2;
    const float cs = __fdiv_rn(2.f * sigma12 + a.c2, sigma1_sq + sigma2_sq + a.c2);
    const float ssim = __fdiv_rn(2.f * mu1_mu2 + a.c1, mu1_sq + mu2_sq + a.c1) * cs;
    s_acc += (double)ssim;
    c_acc += (double)cs;
  }
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) {
    s_acc += __shfl_xor_sync(0xffffffffu, s_acc, o);
    c_acc += __shfl_xor_sync(0xffffffffu, c_acc, o);
  }
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  if (lane == 0) red[0][warp] = s_acc, red[1][warp] = c_acc;
  __syncthreads();
  if (threadIdx.x == 0) {
    double ts = 0.0, tc = 0.0;
    for (int q = 0; q < 8; ++q) ts += red[0][q], tc += red[1][q];
    double* p = a.partial + ((int64_t)nc * gridDim.x + blockIdx.x) * 2;
    p[0] = ts;
    p[1] = tc;
  }
}

struct SsimFinish {
  const double* partial[SSIM_SCALES];
  int tiles[SSIM_SCALES];
  double pixels[SSIM_SCALES];  // output pixels of each scale's maps
  int n, c;
  double* means;  // [scale][n * c][2]: mean ssim_map, mean cs_map
  float* out;     // [n + 1]: per-image value (mean over channels), then the mean over all images and channels
};

// pytorch_msssim's weights, as the fp32 tensor it builds from them
__constant__ float c_ms_ssim_weights[SSIM_SCALES] = {0.0448f, 0.2856f, 0.3001f, 0.2363f, 0.1333f};

__device__ __forceinline__ double ms_ssim_value(const double* means, int nc, int n_nc) {
  double v = 1.0;
  for (int s = 0; s < SSIM_SCALES; ++s) {
    const double m = means[((int64_t)s * n_nc + nc) * 2 + (s == SSIM_SCALES - 1 ? 0 : 1)];  // cs below the last scale
    v *= pow(m < 0.0 ? 0.0 : m, (double)c_ms_ssim_weights[s]);  // relu
  }
  return v;
}

__global__ void __launch_bounds__(FINISH_THREADS) ms_ssim_finish_kernel(SsimFinish a) {
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5, n_warps = FINISH_THREADS / 32;
  const int n_nc = a.n * a.c;
  // one warp per (scale, image x channel): lanes stride over the tiles, then a fixed xor fold
  for (int q = warp; q < SSIM_SCALES * n_nc; q += n_warps) {
    const int s = q / n_nc, nc = q % n_nc;
    const double* p = a.partial[s] + (int64_t)nc * a.tiles[s] * 2;
    double ss = 0.0, cs = 0.0;
    for (int t = lane; t < a.tiles[s]; t += 32) ss += p[2 * t], cs += p[2 * t + 1];
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
      ss += __shfl_xor_sync(0xffffffffu, ss, o);
      cs += __shfl_xor_sync(0xffffffffu, cs, o);
    }
    if (lane == 0) {
      a.means[(int64_t)q * 2] = ss / a.pixels[s];
      a.means[(int64_t)q * 2 + 1] = cs / a.pixels[s];
    }
  }
  __syncthreads();
  for (int n = threadIdx.x; n <= a.n; n += blockDim.x) {
    double sum = 0.0;
    const int lo = n < a.n ? n * a.c : 0, hi = n < a.n ? lo + a.c : n_nc;  // n == a.n: every image
    for (int nc = lo; nc < hi; ++nc) sum += ms_ssim_value(a.means, nc, n_nc);
    a.out[n] = (float)(sum / (double)(hi - lo));
  }
}

// sides of every scale, and where the pooled planes, the means and the partials sit in the workspace
struct SsimLayout {
  int h[SSIM_SCALES], w[SSIM_SCALES], tiles[SSIM_SCALES];
  int64_t plane_x[SSIM_SCALES], plane_y[SSIM_SCALES];  // byte offsets (scales 1..4)
  int64_t means, partial[SSIM_SCALES], bytes;
};

bool ms_ssim_layout(int64_t n, int64_t c, int64_t h, int64_t w, SsimLayout& L) {
  if (n < 1 || c < 1 || h <= (SSIM_WIN - 1) * 16 || w <= (SSIM_WIN - 1) * 16 || h > (1 << 16) || w > (1 << 16)) return false;
  const int64_t nc = n * c;
  int64_t off = 0;
  for (int s = 0; s < SSIM_SCALES; ++s) {
    L.h[s] = (int)(s == 0 ? h : (L.h[s - 1] + 1) / 2);
    L.w[s] = (int)(s == 0 ? w : (L.w[s - 1] + 1) / 2);
    L.tiles[s] = ((L.h[s] + SSIM_TH - 1) / SSIM_TH) * ((L.w[s] + SSIM_TW - 1) / SSIM_TW);
    L.plane_x[s] = L.plane_y[s] = -1;
    if (s > 0) {
      const int64_t bytes = nc * L.h[s] * L.w[s] * 4;
      L.plane_x[s] = off;
      L.plane_y[s] = off + bytes;
      off += 2 * bytes;
    }
  }
  off = (off + 15) / 16 * 16;
  L.means = off;
  off += (int64_t)SSIM_SCALES * nc * 16;
  for (int s = 0; s < SSIM_SCALES; ++s) {
    L.partial[s] = off;
    off += nc * L.tiles[s] * 16;
  }
  L.bytes = off;
  return true;
}

}  // namespace

CEDNERF_EXPORT int64_t cednerf_ms_ssim_workspace_bytes(int64_t n, int64_t c, int64_t h, int64_t w) {
  SsimLayout L;
  return ms_ssim_layout(n, c, h, w, L) ? L.bytes : -1;
}

CEDNERF_EXPORT int cednerf_ms_ssim(const float* x, const int64_t* x_strides_host, const float* y,
                                   const int64_t* y_strides_host, int64_t n, int64_t c, int64_t h, int64_t w,
                                   const float* taps_host, float c1, float c2,
                                   void* work, float* out, void* stream) {
  SsimLayout L;
  CEDNERF_REQUIRE(x && y && x_strides_host && y_strides_host && taps_host && work && out, "bad arguments");
  CEDNERF_REQUIRE(ms_ssim_layout(n, c, h, w, L), "need n, c >= 1 and sides in (160, 65536]");
  CEDNERF_REQUIRE(n * c <= 65535, "more than 65535 image channels in one call");
  cudaStream_t st = (cudaStream_t)stream;
  char* base = (char*)work;
  SsimTaps t;
  for (int k = 0; k < SSIM_WIN; ++k) t.g[k] = taps_host[k];
  SsimFinish f;
  for (int s = 0; s < SSIM_SCALES; ++s) {
    SsimScale a;
    if (s == 0) {
      a.x = x, a.y = y;
      for (int k = 0; k < 4; ++k) a.xs[k] = x_strides_host[k], a.ys[k] = y_strides_host[k];
    } else {
      a.x = (const float*)(base + L.plane_x[s]), a.y = (const float*)(base + L.plane_y[s]);
      const int64_t plane = (int64_t)L.h[s] * L.w[s];
      a.xs[0] = a.ys[0] = c * plane, a.xs[1] = a.ys[1] = plane, a.xs[2] = a.ys[2] = L.w[s], a.xs[3] = a.ys[3] = 1;
    }
    a.c = (int)c, a.h = L.h[s], a.w = L.w[s];
    const bool last = s == SSIM_SCALES - 1;
    a.px = last ? nullptr : (float*)(base + L.plane_x[s + 1]);
    a.py = last ? nullptr : (float*)(base + L.plane_y[s + 1]);
    a.hn = last ? 0 : L.h[s + 1], a.wn = last ? 0 : L.w[s + 1];
    a.pad_h = L.h[s] % 2, a.pad_w = L.w[s] % 2;
    a.partial = (double*)(base + L.partial[s]);
    a.c1 = c1, a.c2 = c2;
    ms_ssim_scale_kernel<<<dim3(L.tiles[s], (unsigned)(n * c)), 256, 0, st>>>(a, t);
    f.partial[s] = a.partial;
    f.tiles[s] = L.tiles[s];
    f.pixels[s] = (double)(L.h[s] - (SSIM_WIN - 1)) * (double)(L.w[s] - (SSIM_WIN - 1));
  }
  f.n = (int)n, f.c = (int)c;
  f.means = (double*)(base + L.means);
  f.out = out;
  ms_ssim_finish_kernel<<<1, FINISH_THREADS, 0, st>>>(f);
  return cednerf_check_launch("cednerf_ms_ssim", SSIM_SCALES + 1);
}
