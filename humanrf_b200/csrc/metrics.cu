// Image-quality metrics for validation on the device: the bounding box of a foreground mask (cv2.boundingRect) and
// PSNR / SSIM of an image pair (actorshq/evaluation/evaluate.py:76-85, humanrf/trainer.py:373-419 without LPIPS).
// SSIM follows skimage.metrics.structural_similarity as the reference calls it: 7x7 uniform window, sample covariance
// (49/48), K1 = 0.01, K2 = 0.03, per-channel map cropped by 3 pixels on every side, mean over the channels.
#include "common.cuh"

namespace hrf {

// ---------------------------------------------------------------------------------------
// bounding box of mask > 0.  box[4] starts at -1 (memset 0xff) and collects, by atomicMax, (W-1-min x, H-1-min y,
// max x, max y); box_finish_kernel turns that into (x, y, w, h) in place.
// ---------------------------------------------------------------------------------------
__global__ void __launch_bounds__(256) mask_box_kernel(const uint8_t* __restrict__ mask, int height, int width,
                                                       int32_t* __restrict__ box) {
  int nx = -1, ny = -1, mx = -1, my = -1;     // -1: nothing seen
  for (int y = blockIdx.x; y < height; y += gridDim.x) {
    const uint8_t* row = mask + (int64_t)y * width;
    for (int x = threadIdx.x; x < width; x += blockDim.x) {
      if (row[x] != 0) {
        nx = max(nx, width - 1 - x), mx = max(mx, x);
        ny = max(ny, height - 1 - y), my = max(my, y);
      }
    }
  }
  nx = __reduce_max_sync(0xffffffffu, nx), ny = __reduce_max_sync(0xffffffffu, ny);
  mx = __reduce_max_sync(0xffffffffu, mx), my = __reduce_max_sync(0xffffffffu, my);
  if ((threadIdx.x & 31) == 0 && mx >= 0) {
    atomicMax(box + 0, nx), atomicMax(box + 1, ny), atomicMax(box + 2, mx), atomicMax(box + 3, my);
  }
}

__global__ void box_finish_kernel(int height, int width, int32_t* __restrict__ box) {
  if (box[2] < 0) {   // empty mask: cv2.boundingRect gives (0, 0, 0, 0)
    box[0] = box[1] = box[2] = box[3] = 0;
    return;
  }
  const int x0 = width - 1 - box[0], y0 = height - 1 - box[1];
  box[2] = box[2] - x0 + 1, box[3] = box[3] - y0 + 1;
  box[0] = x0, box[1] = y0;
}

// ---------------------------------------------------------------------------------------
// PSNR + SSIM.  One CTA per 32x16 tile.  For SSIM the tiles are anchored at the ROI's cropped map (ROI-relative
// x >= 3, y >= 3), so a tile reads its 7x7 windows from ROI pixels only: skimage's reflected padding reaches just the
// 3-pixel border it crops away, and that border is never computed.  Tiles past the cropped map exit at once.  For PSNR
// the same grid covers the whole image with absolute tiles.
// ---------------------------------------------------------------------------------------
constexpr int kTW = 32, kTH = 16, kThreads = 256;
constexpr int kHW = kTW + 6, kHH = kTH + 6;    // tile + 3-pixel halo

struct MetricsArgs {
  const void* a;
  const void* b;
  const int32_t* roi;          // device (x, y, w, h) or NULL
  const uint8_t* mask;         // [H, W] or NULL
  double* partials;            // [3][tiles]: SSIM sum, squared error sum, masked pixel count
  double* out;                 // [4]
  int64_t row_stride;          // elements between image rows
  int height, width, tiles_x, tiles_y;
  float data_range;
  int want_ssim, want_psnr;
};

template <typename T>
__device__ __forceinline__ float ld(const T* p, int64_t i) { return (float)p[i]; }

__device__ __forceinline__ double block_sum(double v, double* red) {
#pragma unroll
  for (int d = 16; d > 0; d >>= 1) v += __shfl_xor_sync(0xffffffffu, v, d);
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  __syncthreads();                             // red[] may still be read by a previous call
  if (lane == 0) red[warp] = v;
  __syncthreads();
  v = 0.0;
  if (warp == 0) {
    v = lane < (int)(blockDim.x >> 5) ? red[lane] : 0.0;
#pragma unroll
    for (int d = 16; d > 0; d >>= 1) v += __shfl_xor_sync(0xffffffffu, v, d);
  }
  return v;                                    // valid in thread 0
}

// ROI intersected with the image, as [x0, x1) x [y0, y1)
__device__ __forceinline__ void roi_bounds(const MetricsArgs& a, int& x0, int& y0, int& w, int& h) {
  x0 = 0, y0 = 0, w = a.width, h = a.height;
  if (a.roi != nullptr) {
    const int rx = a.roi[0], ry = a.roi[1], rw = a.roi[2], rh = a.roi[3];
    x0 = min(max(rx, 0), a.width), y0 = min(max(ry, 0), a.height);
    w = max(min(rx + rw, a.width) - x0, 0), h = max(min(ry + rh, a.height) - y0, 0);
  }
}

template <typename T>
__global__ void __launch_bounds__(kThreads) image_metrics_kernel(const __grid_constant__ MetricsArgs a) {
  __shared__ float sx[3][kHH][kHW], sy[3][kHH][kHW];
  __shared__ float hs[5][kHH][kTW];
  __shared__ double red[kThreads / 32];
  const int tid = threadIdx.x;
  const int tile = blockIdx.y * a.tiles_x + blockIdx.x, tiles = a.tiles_x * a.tiles_y;
  const T* A = static_cast<const T*>(a.a);
  const T* B = static_cast<const T*>(a.b);

  if (a.want_psnr) {
    double se = 0.0, cnt = 0.0;
    for (int i = tid; i < kTW * kTH; i += kThreads) {
      const int x = blockIdx.x * kTW + (i % kTW), y = blockIdx.y * kTH + i / kTW;
      if (x < a.width && y < a.height && (a.mask == nullptr || a.mask[(int64_t)y * a.width + x] != 0)) {
        const int64_t p = (int64_t)y * a.row_stride + 3 * x;
        double e = 0.0;
#pragma unroll
        for (int c = 0; c < 3; ++c) {
          const double d = (double)ld(A, p + c) - (double)ld(B, p + c);
          e += d * d;
        }
        se += e / 3.0, cnt += 1.0;
      }
    }
    se = block_sum(se, red);
    cnt = block_sum(cnt, red);
    if (tid == 0) a.partials[tiles + tile] = se, a.partials[2 * tiles + tile] = cnt;
  }
  if (!a.want_ssim) return;

  int x0, y0, w, h;
  roi_bounds(a, x0, y0, w, h);
  // ROI-relative origin of this tile's halo; its outputs start 3 pixels further in
  const int hx = blockIdx.x * kTW, hy = blockIdx.y * kTH;
  if (w < 7 || h < 7 || hx + 3 >= w - 3 || hy + 3 >= h - 3) return;

  // Moments about a per-tile, per-channel shift s (the tile's first pixel of im1): variances and the covariance do not
  // change under it, and the fp32 box sums of a flat background stay near zero instead of cancelling large terms.
  const float R = a.data_range;
  const int64_t p0 = (int64_t)(y0 + hy) * a.row_stride + 3 * (x0 + hx);
  const float s0 = ld(A, p0) / R, s1 = ld(A, p0 + 1) / R, s2 = ld(A, p0 + 2) / R;
  auto shift = [&](int c) { return c == 0 ? s0 : (c == 1 ? s1 : s2); };
  for (int k = tid; k < kHH * kHW * 3; k += kThreads) {
    const int r = k / (kHW * 3), rem = k - r * (kHW * 3), col = rem / 3, c = rem - col * 3;
    // halo cells past the ROI only feed outputs of the cropped border; clamp them to stay inside the ROI
    const int gy = y0 + min(hy + r, h - 1), gx = x0 + min(hx + col, w - 1);
    const int64_t p = (int64_t)gy * a.row_stride + 3 * gx + c;
    const float sc = shift(c);
    sx[c][r][col] = ld(A, p) / R - sc;
    sy[c][r][col] = ld(B, p) / R - sc;
  }
  const float C1 = 1e-4f, C2 = 9e-4f, inv49 = 1.f / 49.f, cov_norm = 49.f / 48.f;
  double acc = 0.0;
  for (int c = 0; c < 3; ++c) {
    const float sc = shift(c);
    __syncthreads();                           // tile loaded / hs of the previous channel consumed
    for (int i = tid; i < kHH * kTW; i += kThreads) {
      const int r = i / kTW, col = i % kTW;
      float x1 = 0.f, y1 = 0.f, xx = 0.f, yy = 0.f, xy = 0.f;
#pragma unroll
      for (int j = 0; j < 7; ++j) {
        const float u = sx[c][r][col + j], v = sy[c][r][col + j];
        x1 += u, y1 += v, xx = fmaf(u, u, xx), yy = fmaf(v, v, yy), xy = fmaf(u, v, xy);
      }
      hs[0][r][col] = x1, hs[1][r][col] = y1, hs[2][r][col] = xx, hs[3][r][col] = yy, hs[4][r][col] = xy;
    }
    __syncthreads();
    for (int i = tid; i < kTH * kTW; i += kThreads) {
      const int r = i / kTW, col = i % kTW;
      if (hx + col + 3 >= w - 3 || hy + r + 3 >= h - 3) continue;   // cropped border / past the ROI
      float q[5] = {0.f, 0.f, 0.f, 0.f, 0.f};
#pragma unroll
      for (int j = 0; j < 7; ++j) {
#pragma unroll
        for (int m = 0; m < 5; ++m) q[m] += hs[m][r + j][col];
      }
      const float mx = q[0] * inv49, my = q[1] * inv49;
      const float vx = cov_norm * (q[2] * inv49 - mx * mx), vy = cov_norm * (q[3] * inv49 - my * my);
      const float vxy = cov_norm * (q[4] * inv49 - mx * my);
      const float ux = mx + sc, uy = my + sc;
      const float S = ((2.f * ux * uy + C1) * (2.f * vxy + C2)) / ((ux * ux + uy * uy + C1) * (vx + vy + C2));
      acc += (double)S;
    }
  }
  acc = block_sum(acc, red);
  if (tid == 0) a.partials[tile] = acc;
}

// Fixed-order reduction of the per-tile partials (one CTA, so two calls give identical bits).
__global__ void __launch_bounds__(1024) image_metrics_finish_kernel(const __grid_constant__ MetricsArgs a) {
  __shared__ double red[32];
  const int tiles = a.tiles_x * a.tiles_y;
  double ssim = 0.0, se = 0.0, cnt = 0.0;
  int x0, y0, w, h;
  roi_bounds(a, x0, y0, w, h);
  // tiles that ran the SSIM part: the first ceil((w-6)/kTW) x ceil((h-6)/kTH) of the grid
  const int ax = w >= 7 ? (w - 6 + kTW - 1) / kTW : 0, ay = h >= 7 ? (h - 6 + kTH - 1) / kTH : 0;
  if (a.want_ssim)
    for (int k = threadIdx.x; k < ax * ay; k += blockDim.x) ssim += a.partials[(k / ax) * a.tiles_x + k % ax];
  if (a.want_psnr)
    for (int k = threadIdx.x; k < tiles; k += blockDim.x) se += a.partials[tiles + k], cnt += a.partials[2 * tiles + k];
  ssim = block_sum(ssim, red);
  se = block_sum(se, red);
  cnt = block_sum(cnt, red);
  if (threadIdx.x == 0) {
    const double nan = __longlong_as_double(0x7ff8000000000000ll);
    const double R = a.data_range;
    const double mse = se / cnt / (R * R);
    a.out[0] = (a.want_ssim && ax > 0 && ay > 0) ? ssim / (3.0 * (double)(w - 6) * (double)(h - 6)) : nan;
    a.out[1] = a.want_psnr ? -10.0 * log10(mse) : nan;
    a.out[2] = a.want_psnr ? se / (R * R) : nan;
    a.out[3] = a.want_psnr ? cnt : nan;
  }
}

static inline int tiles_x(int width) { return (width + kTW - 1) / kTW; }
static inline int tiles_y(int height) { return (height + kTH - 1) / kTH; }

}  // namespace hrf

using namespace hrf;

extern "C" int hrf_mask_bbox(const uint8_t* mask, int height, int width, int32_t* box, void* stream) {
  HRF_REQUIRE(mask != nullptr && box != nullptr, "null pointer");
  HRF_REQUIRE(height >= 0 && width >= 0, "negative image size");
  cudaStream_t st = reinterpret_cast<cudaStream_t>(stream);
  HRF_CUDA(cudaMemsetAsync(box, 0xff, 4 * sizeof(int32_t), st));
  if (height > 0 && width > 0) {
    const int grid = std::min(height, sm_count() * 8);
    mask_box_kernel<<<grid, 256, 0, st>>>(mask, height, width, box);
    HRF_CHECK_LAUNCH();
  }
  box_finish_kernel<<<1, 1, 0, st>>>(height, width, box);
  HRF_CHECK_LAUNCH();
  return 0;
}

extern "C" int64_t hrf_image_metrics_workspace_bytes(int height, int width) {
  return 3 * (int64_t)tiles_x(width) * tiles_y(height) * (int64_t)sizeof(double);
}

extern "C" int hrf_image_metrics(const void* im1, const void* im2, int is_uint8, int height, int width,
                                 int64_t row_stride, const int32_t* roi, float data_range, const uint8_t* psnr_mask,
                                 int what, double* out, void* workspace, void* stream) {
  HRF_REQUIRE(im1 != nullptr && im2 != nullptr && out != nullptr && workspace != nullptr, "null pointer");
  HRF_REQUIRE(height > 0 && width > 0 && row_stride >= 3 * (int64_t)width, "bad image size or row stride");
  HRF_REQUIRE(data_range > 0.f, "data_range must be positive");
  HRF_REQUIRE((what & ~3) == 0 && what != 0, "what: bit 0 = SSIM, bit 1 = PSNR");
  HRF_REQUIRE(psnr_mask == nullptr || row_stride == 3 * (int64_t)width, "a PSNR mask needs a contiguous image");
  HRF_REQUIRE(tiles_y(height) <= 65535, "image too tall");
  MetricsArgs a{im1, im2, roi, psnr_mask, static_cast<double*>(workspace), out, row_stride, height, width,
                tiles_x(width), tiles_y(height), data_range, what & 1, (what >> 1) & 1};
  cudaStream_t st = reinterpret_cast<cudaStream_t>(stream);
  const dim3 grid(a.tiles_x, a.tiles_y);
  if (is_uint8) image_metrics_kernel<uint8_t><<<grid, kThreads, 0, st>>>(a);
  else image_metrics_kernel<float><<<grid, kThreads, 0, st>>>(a);
  HRF_CHECK_LAUNCH();
  image_metrics_finish_kernel<<<1, 1024, 0, st>>>(a);
  HRF_CHECK_LAUNCH();
  return 0;
}
