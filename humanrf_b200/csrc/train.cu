// Training-step kernels that are not the field itself: the per-ray loss (forward + backward in one launch) and the
// multi-tensor fused Adam with device-side step counters and active flags.  Together with the device-side sample counts
// (hrf_samples.num_samples_dev) they make FusedTrainer.step free of host synchronisation.
// Reference semantics: humanrf/trainer.py:205-215,229-255, humanrf/utils/loss.py:4-10, humanrf/run.py:101-104.
#include <algorithm>

#include "common.cuh"

namespace hrf {

// element i of a `vectors` tensor [4, VR, 32] inside its transposed copy [4, 16, VR, 2]
__device__ __forceinline__ int64_t vectors_t_index(int64_t i, int vr) {
  const int c = (int)(i & 31);
  const int64_t row = (i >> 5) % vr, axis = (i >> 5) / vr;
  return ((axis * 16 + (c >> 1)) * vr + row) * 2 + (c & 1);
}

__global__ void transpose_vectors_kernel(const float* __restrict__ v, float* __restrict__ vt, int vr) {
  const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i < (int64_t)4 * vr * 32) vt[vectors_t_index(i, vr)] = v[i];
}

__device__ __forceinline__ float block_sum_256(float v) {
  __shared__ float part[8];
#pragma unroll
  for (int d = 16; d > 0; d >>= 1) v += __shfl_xor_sync(0xffffffffu, v, d);
  if ((threadIdx.x & 31) == 0) part[threadIdx.x >> 5] = v;
  __syncthreads();
  v = threadIdx.x < 8 ? part[threadIdx.x] : 0.f;
  if (threadIdx.x < 32) {
#pragma unroll
    for (int d = 4; d > 0; d >>= 1) v += __shfl_xor_sync(0xffffffffu, v, d);
  }
  return v;  // valid in thread 0
}

// trainer.py:237-238 gt = rgb*mask + bg*(1-mask); :209 HuberLoss(delta, mean); :213-215 bce_weight * mean(bce_loss)
__global__ void __launch_bounds__(256) train_loss_kernel(const float* __restrict__ color, const float* __restrict__ wsum,
                                                         const float* __restrict__ rgba, const float* __restrict__ bg,
                                                         int64_t num_rays, float delta, float bce_w,
                                                         const float* __restrict__ scale_dev, float* __restrict__ d_color,
                                                         float* __restrict__ d_wsum, float* __restrict__ loss_out) {
  const int64_t r = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  const float scale = scale_dev != nullptr ? __ldg(scale_dev) : 1.f;
  const float inv3r = 1.f / (3.f * (float)num_rays), invr = 1.f / (float)num_rays;
  float loss = 0.f;
  if (r < num_rays) {
    const float m = rgba[4 * r + 3];
#pragma unroll
    for (int c = 0; c < 3; ++c) {
      const float gt = rgba[4 * r + c] * m + bg[3 * r + c] * (1.f - m);
      const float x = color[3 * r + c] - gt, ax = fabsf(x);
      const bool quad = ax < delta;
      loss += (quad ? 0.5f * x * x : delta * (ax - 0.5f * delta)) * inv3r;
      d_color[3 * r + c] = (quad ? x : copysignf(delta, x)) * inv3r * scale;
    }
    // utils/loss.py:4-10 : clamp to [0,1], eps 1e-10 inside both logs
    const float w = wsum[r];
    const float pc = fminf(fmaxf(w, 0.f), 1.f);
    loss += -(m * logf(pc + 1e-10f) + (1.f - m) * logf(1.f - pc + 1e-10f)) * invr * bce_w;
    const float dpc = -(m / (pc + 1e-10f) - (1.f - m) / (1.f - pc + 1e-10f));
    d_wsum[r] = (w >= 0.f && w <= 1.f) ? dpc * invr * bce_w * scale : 0.f;   // torch.clamp passes the gradient on [min, max]
  }
  loss = block_sum_256(loss);
  if (threadIdx.x == 0 && loss_out != nullptr) atomicAdd(loss_out, loss);
}

// ---- multi-tensor Adam ---------------------------------------------------------------------------------------
__global__ void adam_steps_kernel(const hrf_adam_tensor* __restrict__ T, int num) {
  const int t = blockIdx.x * blockDim.x + threadIdx.x;
  if (t >= num) return;
  if (T[t].active != nullptr && *T[t].active == 0) return;
  *T[t].step += 1;
}

__global__ void __launch_bounds__(256) adam_multi_kernel(const hrf_adam_tensor* __restrict__ T, int num, float lr, float b1,
                                                         float b2, float eps, float gscale, int zero_grad) {
  // block -> tensor: last t with first_block <= blockIdx.x
  int lo = 0, hi = num - 1;
  const int64_t b = blockIdx.x;
  while (lo < hi) {
    const int mid = (lo + hi + 1) >> 1;
    if (T[mid].first_block <= b) lo = mid;
    else hi = mid - 1;
  }
  const hrf_adam_tensor t = T[lo];
  if (t.active != nullptr && *t.active == 0) return;
  const int step = *t.step;   // already advanced by adam_steps_kernel
  const float bc1 = 1.f - powf(b1, (float)step);
  const float bc2s = sqrtf(1.f - powf(b2, (float)step));
  const float lr1 = lr / bc1;
  const int64_t start = (b - t.first_block) * HRF_ADAM_BLOCK_ELEMS;
  const int64_t end = start + HRF_ADAM_BLOCK_ELEMS < t.n ? start + HRF_ADAM_BLOCK_ELEMS : t.n;
  __nv_bfloat16* sh = reinterpret_cast<__nv_bfloat16*>(t.shadow_bf16);
  auto upd = [&](float& p, float& m, float& v, float g) {
    g *= gscale;
    m = b1 * m + (1.f - b1) * g;
    v = b2 * v + (1.f - b2) * g * g;
    // torch: denom = sqrt(v)/sqrt(bias_correction2) + eps ; p -= lr/bias_correction1 * m/denom
    p = p - lr1 * (m / (sqrtf(v) / bc2s + eps));
  };
  const bool vec = t.blob_perm == nullptr &&
                   ((reinterpret_cast<uintptr_t>(t.param) | reinterpret_cast<uintptr_t>(t.exp_avg) |
                     reinterpret_cast<uintptr_t>(t.exp_avg_sq) | reinterpret_cast<uintptr_t>(t.grad)) & 15u) == 0 &&
                   (reinterpret_cast<uintptr_t>(t.shadow_bf16) & 7u) == 0 && ((end - start) & 3) == 0;
  if (vec) {
    for (int64_t i = start + 4 * (int64_t)threadIdx.x; i < end; i += 4 * 256) {
      float4 p = *reinterpret_cast<float4*>(t.param + i), m = *reinterpret_cast<float4*>(t.exp_avg + i),
             v = *reinterpret_cast<float4*>(t.exp_avg_sq + i);
      const float4 g = *reinterpret_cast<const float4*>(t.grad + i);
      upd(p.x, m.x, v.x, g.x), upd(p.y, m.y, v.y, g.y), upd(p.z, m.z, v.z, g.z), upd(p.w, m.w, v.w, g.w);
      *reinterpret_cast<float4*>(t.param + i) = p;
      *reinterpret_cast<float4*>(t.exp_avg + i) = m;
      *reinterpret_cast<float4*>(t.exp_avg_sq + i) = v;
      if (zero_grad) *reinterpret_cast<float4*>(t.grad + i) = make_float4(0.f, 0.f, 0.f, 0.f);
      if (sh != nullptr) *reinterpret_cast<uint2*>(sh + i) = make_uint2(pack_bf16x2(p.x, p.y), pack_bf16x2(p.z, p.w));
      if (t.vectors_t != nullptr) {   // (i is a multiple of 4: two feature pairs = two levels of one row)
        *reinterpret_cast<float2*>(t.vectors_t + vectors_t_index(i, t.vec_res)) = make_float2(p.x, p.y);
        *reinterpret_cast<float2*>(t.vectors_t + vectors_t_index(i + 2, t.vec_res)) = make_float2(p.z, p.w);
      }
    }
  } else {
    for (int64_t i = start + threadIdx.x; i < end; i += 256) {
      float p = t.param[i], m = t.exp_avg[i], v = t.exp_avg_sq[i];
      upd(p, m, v, t.grad[i]);
      t.param[i] = p, t.exp_avg[i] = m, t.exp_avg_sq[i] = v;
      if (zero_grad) t.grad[i] = 0.f;
      if (sh != nullptr) sh[t.blob_perm != nullptr ? (int64_t)t.blob_perm[i] : i] = __float2bfloat16_rn(p);
      if (t.vectors_t != nullptr) t.vectors_t[vectors_t_index(i, t.vec_res)] = p;
    }
  }
}

}  // namespace hrf

using namespace hrf;

extern "C" int hrf_train_loss(const float* color, const float* weights_sum, const float* rgba, const float* background,
                              int64_t num_rays, float huber_delta, float bce_weight, const float* loss_scale_dev,
                              float* d_color, float* d_weights_sum, float* loss_out, void* stream) {
  HRF_REQUIRE(color && weights_sum && rgba && background && d_color && d_weights_sum, "null argument");
  if (num_rays == 0) return 0;
  train_loss_kernel<<<(unsigned)((num_rays + 255) / 256), 256, 0, reinterpret_cast<cudaStream_t>(stream)>>>(
      color, weights_sum, rgba, background, num_rays, huber_delta, bce_weight, loss_scale_dev, d_color, d_weights_sum, loss_out);
  HRF_CHECK_LAUNCH();
  return 0;
}

extern "C" int hrf_transpose_vectors(const float* vectors, float* vectors_t, int vec_res, void* stream) {
  HRF_REQUIRE(vectors != nullptr && vectors_t != nullptr && vec_res >= 1, "bad argument");
  const int64_t n = (int64_t)4 * vec_res * 32;
  transpose_vectors_kernel<<<(unsigned)((n + 255) / 256), 256, 0, reinterpret_cast<cudaStream_t>(stream)>>>(vectors, vectors_t, vec_res);
  HRF_CHECK_LAUNCH();
  return 0;
}

extern "C" int hrf_adam_multi(const hrf_adam_tensor* tensors, int num_tensors, int64_t total_blocks, float lr, float beta1,
                              float beta2, float eps, float grad_scale, int zero_grad, void* stream) {
  HRF_REQUIRE(tensors != nullptr && num_tensors >= 1, "no tensors");
  if (total_blocks == 0) return 0;
  HRF_REQUIRE(total_blocks < (1ll << 31), "too many blocks");
  cudaStream_t st = reinterpret_cast<cudaStream_t>(stream);
  adam_steps_kernel<<<(num_tensors + 127) / 128, 128, 0, st>>>(tensors, num_tensors);
  HRF_CHECK_LAUNCH();
  adam_multi_kernel<<<(unsigned)total_blocks, 256, 0, st>>>(tensors, num_tensors, lr, beta1, beta2, eps, grad_scale, zero_grad);
  HRF_CHECK_LAUNCH();
  return 0;
}
