// Error plumbing, device info, fused Adam, bf16 cast and the tcgen05 descriptor self-test.
#include <mutex>

#include "field_common.cuh"

namespace hrf {

static thread_local std::string g_last_error;
void set_error(const std::string& msg) { g_last_error = msg; }
int cuda_fail(cudaError_t e, const char* what, const char* file, int line) {
  g_last_error = std::string("CUDA error ") + cudaGetErrorName(e) + " (" + cudaGetErrorString(e) + ") in " + what +
                 " at " + file + ":" + std::to_string(line);
  return (int)e ? (int)e : -2;
}
int sm_count() {
  static int cached = 0;
  if (cached == 0) {
    int dev = 0, n = 0;
    if (cudaGetDevice(&dev) == cudaSuccess &&
        cudaDeviceGetAttribute(&n, cudaDevAttrMultiProcessorCount, dev) == cudaSuccess && n > 0)
      cached = n;
    else
      return 148;
  }
  return cached;
}

// ---------------------------------------------------------------------------------------
// Adam (torch.optim.Adam semantics, run.py:101: betas=(0.9,0.99), eps=1e-15, no weight decay)
// ---------------------------------------------------------------------------------------
__global__ void adam_kernel(float* __restrict__ p, float* __restrict__ m, float* __restrict__ v,
                            const float* __restrict__ g, __nv_bfloat16* __restrict__ shadow, int64_t n, float lr,
                            float b1, float b2, float eps, float bc1, float bc2_sqrt, float gscale) {
  const int64_t stride = (int64_t)gridDim.x * blockDim.x;
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += stride) {
    const float gi = g[i] * gscale;
    const float mi = b1 * m[i] + (1.f - b1) * gi;
    const float vi = b2 * v[i] + (1.f - b2) * gi * gi;
    m[i] = mi;
    v[i] = vi;
    // torch: denom = sqrt(v)/sqrt(bias_correction2) + eps ; p -= lr/bias_correction1 * m/denom
    const float denom = sqrtf(vi) / bc2_sqrt + eps;
    const float pi = p[i] - (lr / bc1) * (mi / denom);
    p[i] = pi;
    if (shadow != nullptr) shadow[i] = __float2bfloat16_rn(pi);
  }
}

__global__ void cast_bf16_kernel(const float* __restrict__ s, __nv_bfloat16* __restrict__ d, int64_t n) {
  const int64_t stride = (int64_t)gridDim.x * blockDim.x;
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += stride) d[i] = __float2bfloat16_rn(s[i]);
}

// ---------------------------------------------------------------------------------------
// tcgen05 descriptor self-test: D[M,N] = A[M,K] * B[N,K]^T with caller-chosen placement
// strides and descriptor fields.
// ---------------------------------------------------------------------------------------
struct SelfTestArgs {
  const __nv_bfloat16* a;
  const __nv_bfloat16* b;
  float* d;
  int m, n, k;
  uint32_t a_kstride, a_mstride, b_kstride, b_nstride;  // physical placement (bytes)
  uint32_t a_lbo, a_sbo, b_lbo, b_sbo;                  // descriptor fields (bytes)
  int mn_major;
};

__global__ void __launch_bounds__(128, 1) selftest_umma_kernel(const SelfTestArgs t) {
  extern __shared__ unsigned char smem_raw[];
  unsigned char* base = reinterpret_cast<unsigned char*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~uintptr_t(1023));
  unsigned char* sa = base;            // up to 64 KB
  unsigned char* sb = base + 65536;    // up to 64 KB
  __shared__ uint64_t bar;
  __shared__ uint32_t tmem_base;
  const int tid = threadIdx.x;
  if (tid == 0) {
    mbar_init(&bar, 1);
    fence_mbar_init();
  }
  if (tid < 32) {
    tmem_alloc(&tmem_base, 256);
    tmem_relinquish();
  }
  // operand placement
  for (int e = tid; e < t.m * t.k; e += blockDim.x) {
    const int r = e / t.k, k = e % t.k;
    uint32_t off;
    if (!(t.mn_major & 1))
      off = (uint32_t)(k >> 3) * t.a_kstride + (uint32_t)(r >> 3) * t.a_mstride + (uint32_t)(r & 7) * 16u + (uint32_t)(k & 7) * 2u;
    else
      off = (uint32_t)(r >> 3) * t.a_mstride + (uint32_t)(k >> 3) * t.a_kstride + (uint32_t)(k & 7) * 16u + (uint32_t)(r & 7) * 2u;
    *reinterpret_cast<__nv_bfloat16*>(sa + off) = t.a[e];
  }
  for (int e = tid; e < t.n * t.k; e += blockDim.x) {
    const int r = e / t.k, k = e % t.k;
    uint32_t off;
    if (!(t.mn_major & 2))
      off = (uint32_t)(k >> 3) * t.b_kstride + (uint32_t)(r >> 3) * t.b_nstride + (uint32_t)(r & 7) * 16u + (uint32_t)(k & 7) * 2u;
    else
      off = (uint32_t)(r >> 3) * t.b_nstride + (uint32_t)(k >> 3) * t.b_kstride + (uint32_t)(k & 7) * 16u + (uint32_t)(r & 7) * 2u;
    *reinterpret_cast<__nv_bfloat16*>(sb + off) = t.b[e];
  }
  tc_fence_before();
  fence_proxy_async_smem();
  __syncthreads();
  tc_fence_after();
  if (tid == 0) {
    const uint32_t idesc = make_idesc_bf16(t.m, t.n, t.mn_major & 1, (t.mn_major >> 1) & 1);
    for (int k = 0; k < t.k / 16; ++k) {
      const uint64_t ad = make_smem_desc(smem_u32(sa) + (uint32_t)k * 2u * t.a_kstride, t.a_lbo, t.a_sbo);
      const uint64_t bd = make_smem_desc(smem_u32(sb) + (uint32_t)k * 2u * t.b_kstride, t.b_lbo, t.b_sbo);
      umma_bf16(tmem_base, ad, bd, idesc, k > 0);
    }
    umma_commit(&bar);
  }
  mbar_wait(&bar, 0);
  tc_fence_after();
  // read back: lane L of warp w holds row: M=128 -> row = 32w+L ; M=64 -> rows live in lanes 0..15 of each warp
  const int lane = tid & 31, warp = tid >> 5;
  int row = -1;
  if (t.m == 128) row = tid;
  else if (lane < 16) row = warp * 16 + lane;
  for (int c0 = 0; c0 < t.n; c0 += 16) {
    float v[16];
    tmem_ld16(tmem_base + ((uint32_t)(warp * 32) << 16) + (uint32_t)c0, v);
    if (row >= 0)
      for (int j = 0; j < 16; ++j) t.d[(int64_t)row * t.n + c0 + j] = v[j];
  }
  tc_fence_before();
  __syncthreads();
  if (tid < 32) tmem_dealloc(tmem_base, 256);
}

}  // namespace hrf

using namespace hrf;

extern "C" const char* hrf_last_error(void) { return g_last_error.c_str(); }
extern "C" int hrf_version(void) { return 2; }
extern "C" int hrf_device_info(int* out3) {
  int dev = 0;
  HRF_CUDA(cudaGetDevice(&dev));
  HRF_CUDA(cudaDeviceGetAttribute(&out3[0], cudaDevAttrMultiProcessorCount, dev));
  HRF_CUDA(cudaDeviceGetAttribute(&out3[1], cudaDevAttrComputeCapabilityMajor, dev));
  HRF_CUDA(cudaDeviceGetAttribute(&out3[2], cudaDevAttrComputeCapabilityMinor, dev));
  return 0;
}

extern "C" int hrf_adam_step(float* param, float* exp_avg, float* exp_avg_sq, const float* grad, void* shadow_bf16,
                             int64_t n, float lr, float beta1, float beta2, float eps, int step, float grad_scale,
                             void* stream) {
  HRF_REQUIRE(step >= 1, "Adam step counter starts at 1");
  if (n == 0) return 0;
  const float bc1 = 1.f - powf(beta1, (float)step);
  const float bc2 = 1.f - powf(beta2, (float)step);
  const int grid = (int)std::min<int64_t>((n + 255) / 256, (int64_t)sm_count() * 8);
  adam_kernel<<<grid, 256, 0, reinterpret_cast<cudaStream_t>(stream)>>>(
      param, exp_avg, exp_avg_sq, grad, reinterpret_cast<__nv_bfloat16*>(shadow_bf16), n, lr, beta1, beta2, eps, bc1,
      sqrtf(bc2), grad_scale);
  HRF_CHECK_LAUNCH();
  return 0;
}

extern "C" int hrf_cast_bf16(const float* src, void* dst, int64_t n, void* stream) {
  if (n == 0) return 0;
  const int grid = (int)std::min<int64_t>((n + 255) / 256, (int64_t)sm_count() * 8);
  cast_bf16_kernel<<<grid, 256, 0, reinterpret_cast<cudaStream_t>(stream)>>>(src, reinterpret_cast<__nv_bfloat16*>(dst), n);
  HRF_CHECK_LAUNCH();
  return 0;
}

extern "C" int hrf_selftest_umma(const void* a_bf16, const void* b_bf16, float* d, int m, int n, int k,
                                 uint32_t a_kstride, uint32_t a_mstride, uint32_t b_kstride, uint32_t b_nstride,
                                 uint32_t a_lbo, uint32_t a_sbo, uint32_t b_lbo, uint32_t b_sbo, int mn_major,
                                 void* stream) {
  HRF_REQUIRE(m == 64 || m == 128, "M must be 64 or 128");
  HRF_REQUIRE(n % 16 == 0 && n >= 16 && n <= 256 && k % 16 == 0 && k >= 16 && k <= 128, "bad N/K");
  SelfTestArgs t{(const __nv_bfloat16*)a_bf16, (const __nv_bfloat16*)b_bf16, d, m, n, k, a_kstride, a_mstride,
                 b_kstride, b_nstride, a_lbo, a_sbo, b_lbo, b_sbo, mn_major};
  const int smem = 2 * 65536 + 1024;
  HRF_CUDA(cudaFuncSetAttribute(selftest_umma_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, smem));
  selftest_umma_kernel<<<1, 128, smem, reinterpret_cast<cudaStream_t>(stream)>>>(t);
  HRF_CHECK_LAUNCH();
  return 0;
}
