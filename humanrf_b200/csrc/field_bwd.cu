// Fused backward of the HumanRF radiance field for sm_100a (autograd of humanrf.py:158-208).
// Per 128-sample tile (thread r = sample r = operand row r = TMEM lane r):
//   1. forward recompute of both MLPs from the saved composed features (or a re-encode),
//      keeping every activation tile in shared memory (bf16, UMMA K-major core-matrix layout);
//   2. MLP backward on the tensor cores.  The SAME shared-memory tiles serve three roles by
//      switching descriptors only:  K-major A operand of the forward / dgrad GEMMs, and
//      MN-major A / B operands of the wgrad GEMMs (contraction over the 128 samples).  The
//      packed forward weight blob is re-used as the MN-major B operand of the dgrad GEMMs.
//      Weight-gradient accumulators live in TMEM for the whole persistent CTA (M=64 tiles)
//      and are flushed once with fp32 atomics;
//   3. d(composed features) goes to a level-major [16][N] workspace, with each sample's position and segment; the
//      table / vector gradient scatter (grid_scatter_v3_kernel, scatter_v3.cu) reads them in a second, high-occupancy
//      kernel.  (One fused kernel was latency-bound at 12.5 % occupancy: profiles/r1_ncu_full_bwd.)
#include <cstdlib>

#include "field_common.cuh"

namespace hrf {

struct __align__(1024) BwdSmem {
  unsigned char w[kWBlobBytesMax];
  unsigned char feat[kTile * 32 * 2];  // composed features            (A32)
  unsigned char cin[kTile * 48 * 2];   // colour-net input              (A32 / A48)
  unsigned char hs[kTile * 64 * 2];    // sigma hidden, then d(hidden)  (A64)
  unsigned char h1[kTile * 64 * 2];    // colour hidden 1, then its gradient, then dFeat staging
  unsigned char h2[kTile * 64 * 2];    // colour hidden 2, then its gradient
  unsigned char g3[kTile * 16 * 2];    // d(colour pre-activation)  [128,16]
  unsigned char gs[kTile * 16 * 2];    // d(sigma-net output)       [128,16]
  uint64_t bar_w, bar_mma;
  uint32_t tmem_base;
};

// TMEM column map (256 columns allocated): work area + persistent weight-gradient accumulators
constexpr uint32_t kColWork = 0;     // 64 cols: layer outputs / dgrad results
constexpr uint32_t kColW1s = 64;     // dW1s   [64 out, 32 in]
constexpr uint32_t kColW2s = 96;     // dW2s^T [64 in, 16 out]
constexpr uint32_t kColW1c = 112;    // dW1c   [64 out, 32|48 in]
constexpr uint32_t kColW2c = 160;    // dW2c   [64 out, 64 in]
constexpr uint32_t kColW3c = 224;    // dW3c^T [64 in, 16 out]
constexpr uint32_t kTmemCols = 256;

struct BwdArgs {
  hrf_field f;
  hrf_samples s;
  const hrf_segment_grads* seg_grads;
  const float* d_sigma;
  const float* d_rgb;
  const float* d_geo;    // [N,15] gradient of the geometry features, or NULL
  const uint4* feat_in;  // bf16 [M,32] saved by a forward pass, or NULL (re-encode)
  const int32_t* feat_index;  // row of feat_in per sample, or NULL (identity)
  float* d_mlp;
  float* d_emb;   // camera-embedding gradient [num_cameras, E] or NULL
  float2* dfeat;  // [16][N] float2 workspace: d(composed features)
  float4* pos4;   // [N] normalised (x,y,z,t) of every sample, for the scatter (scatter_v3.cu)
  uint8_t* seg8;  // [N] segment index (255 = no segment)
};

// D[128,Nin] = G[128,Kout] * W[Kout,Nin]  : A = gradient tile (K-major), B = forward blob read MN-major
__device__ __forceinline__ void issue_dgrad(uint32_t tmem_d, uint32_t g_addr, uint32_t w_addr, int Nin, int Kout) {
  const uint32_t idesc = make_idesc_bf16(kTile, Nin, 0, 1);
  const uint32_t b_sbo = (uint32_t)(Kout >> 3) * 128u;
  for (int k = 0; k < Kout / 16; ++k) {
    const uint64_t ad = make_smem_desc(g_addr + (uint32_t)k * 2u * kAChunk, kAChunk, 128u);
    const uint64_t bd = make_smem_desc(w_addr + (uint32_t)k * 256u, 128u, b_sbo);
    umma_bf16(tmem_d, ad, bd, idesc, k > 0 ? 1u : 0u);
  }
}
// D[64,N] (+)= X^T[64,128] * Y[128,N] : both tiles read MN-major, contraction over the 128 samples
__device__ __forceinline__ void issue_wgrad(uint32_t tmem_d, uint32_t x_addr, uint32_t y_addr, int N, bool acc) {
  const uint32_t idesc = make_idesc_bf16(64, N, 1, 1);
  for (int k = 0; k < kTile / 16; ++k) {
    const uint64_t ad = make_smem_desc(x_addr + (uint32_t)k * 256u, 128u, kAChunk);
    const uint64_t bd = make_smem_desc(y_addr + (uint32_t)k * 256u, 128u, kAChunk);
    umma_bf16(tmem_d, ad, bd, idesc, (acc || k > 0) ? 1u : 0u);
  }
}

template <class F>
__device__ __forceinline__ void mma_round(BwdSmem& sm, uint32_t& phase, F&& issue) {
  tc_fence_before();
  fence_proxy_async_smem();
  __syncthreads();
  if (threadIdx.x == 0) {
    tc_fence_after();
    issue();
    umma_commit(&sm.bar_mma);
  }
  mbar_wait(&sm.bar_mma, phase);
  phase ^= 1u;
  tc_fence_after();
}

// store relu(v) as a K=64 bf16 tile row
__device__ __forceinline__ void store_relu64(unsigned char* buf, uint32_t roff, const float* v) {
#pragma unroll
  for (int kg = 0; kg < 8; ++kg) {
    uint4 q;
    q.x = pack_bf16x2(fmaxf(v[kg * 8 + 0], 0.f), fmaxf(v[kg * 8 + 1], 0.f));
    q.y = pack_bf16x2(fmaxf(v[kg * 8 + 2], 0.f), fmaxf(v[kg * 8 + 3], 0.f));
    q.z = pack_bf16x2(fmaxf(v[kg * 8 + 4], 0.f), fmaxf(v[kg * 8 + 5], 0.f));
    q.w = pack_bf16x2(fmaxf(v[kg * 8 + 6], 0.f), fmaxf(v[kg * 8 + 7], 0.f));
    *reinterpret_cast<uint4*>(buf + kg * kAChunk + roff) = q;
  }
}
// in place: tile row holds relu(h) (bf16); replace by g * (h > 0) (bf16)
__device__ __forceinline__ void relu_backward_inplace64(unsigned char* buf, uint32_t roff, const float* g) {
#pragma unroll
  for (int kg = 0; kg < 8; ++kg) {
    uint4* p = reinterpret_cast<uint4*>(buf + kg * kAChunk + roff);
    const uint4 a = *p;
    const uint32_t av[4] = {a.x, a.y, a.z, a.w};
    uint32_t o[4];
#pragma unroll
    for (int j = 0; j < 4; ++j) {
      const float lo = (av[j] & 0x7fffu) != 0u && !(av[j] & 0x8000u) ? g[kg * 8 + 2 * j] : 0.f;
      const float hi = (av[j] & 0x7fff0000u) != 0u && !(av[j] & 0x80000000u) ? g[kg * 8 + 2 * j + 1] : 0.f;
      o[j] = pack_bf16x2(lo, hi);
    }
    *p = make_uint4(o[0], o[1], o[2], o[3]);
  }
}

__device__ __forceinline__ void red_add_v4(float* addr, float a, float b, float c, float d) {   // addr 16-byte aligned
  asm volatile("red.global.add.v4.f32 [%0], {%1, %2, %3, %4};" ::"l"(addr), "f"(a), "f"(b), "f"(c), "f"(d) : "memory");
}

// kLevelUnroll: levels unrolled in the re-encode loop (only taken when the forward's features were not saved)
template <int kLevelUnroll = 4>
__global__ void __launch_bounds__(kTile, 2) field_backward_kernel(const __grid_constant__ BwdArgs args) {
  extern __shared__ unsigned char smem_raw[];
  BwdSmem& sm = *reinterpret_cast<BwdSmem*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~uintptr_t(1023));
  const int tid = threadIdx.x;
  const hrf_field& f = args.f;
  const uint32_t roff = a_row_off(tid);

  if (tid == 0) {
    mbar_init(&sm.bar_w, 1);
    mbar_init(&sm.bar_mma, 1);
    fence_mbar_init();
  }
  if (tid < 32) {
    tmem_alloc(&sm.tmem_base, kTmemCols);
    tmem_relinquish();
  }
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  if (tid == 0) {
    mbar_arrive_expect_tx(&sm.bar_w, w_blob_bytes(f.color_in_width));
    tma_load_1d(sm.w, f.mlp_blob, w_blob_bytes(f.color_in_width), &sm.bar_w);
  }
  const uint32_t tm = sm.tmem_base;
  const uint32_t trow = tm + ((uint32_t)(tid & ~31) << 16);  // this warp's TMEM lanes
  const uint32_t wbase = smem_u32(sm.w);
  const uint32_t a_feat = smem_u32(sm.feat), a_cin = smem_u32(sm.cin), a_hs = smem_u32(sm.hs),
                 a_h1 = smem_u32(sm.h1), a_h2 = smem_u32(sm.h2), a_g3 = smem_u32(sm.g3), a_gs = smem_u32(sm.gs);
  bool weights_ready = false, have_acc = false;
  uint32_t phase = 0;

  const int64_t n = live_samples(args.s);
  const int64_t ns = args.s.num_samples;   // row length of the level-major workspace
  const int64_t num_tiles = (n + kTile - 1) / kTile;
  for (int64_t tile = blockIdx.x; tile < num_tiles; tile += gridDim.x) {
    const int64_t i = tile * kTile + tid;
    const bool valid = i < n;
    const Sample s = load_sample(f, args.s, i, n);
    if (valid) {
      args.pos4[i] = make_float4(s.x, s.y, s.z, s.t);
      args.seg8[i] = s.seg != nullptr ? (uint8_t)(s.seg - f.segments) : (uint8_t)255;
    }
    if (args.feat_in != nullptr) {
      const int64_t row = !(valid && s.seg != nullptr) ? -1 : (args.feat_index != nullptr ? (int64_t)__ldg(args.feat_index + i) : i);
#pragma unroll
      for (int kg = 0; kg < 4; ++kg)
        *reinterpret_cast<uint4*>(sm.feat + kg * kAChunk + roff) =
            row >= 0 ? __ldg(args.feat_in + row * 4 + kg) : make_uint4(0, 0, 0, 0);
    } else {
      encode_to_smem<false, kLevelUnroll>(f, s, sm.feat, tid);
    }
    // Everything else this tile will read from global memory is requested here, before the ten MMA rounds: each round
    // ends in asm statements that clobber memory, so the compiler cannot move a later load above them, and at 8 warps
    // per SM a load issued where its value is needed is a fully exposed round trip.
    const View vw = load_view(f, args.s, i, n);
    float up_sigma = 0.f, up_rgb[3] = {0.f, 0.f, 0.f};
    if (valid) {
      if (args.d_sigma != nullptr) up_sigma = __ldg(args.d_sigma + i);
      if (args.d_rgb != nullptr) up_rgb[0] = __ldg(args.d_rgb + 3 * i), up_rgb[1] = __ldg(args.d_rgb + 3 * i + 1), up_rgb[2] = __ldg(args.d_rgb + 3 * i + 2);
    }
    if (!weights_ready) {
      mbar_wait(&sm.bar_w, 0);
      weights_ready = true;
    }
    float v[64], o[16];
    // ---------------- forward recompute ----------------
    mma_round(sm, phase, [&] { issue_layer(tm + kColWork, a_feat, wbase + kWSig1, 64, 32); });
    tmem_ld64(trow + kColWork, v);
    store_relu64(sm.hs, roff, v);
    mma_round(sm, phase, [&] { issue_layer(tm + kColWork, a_hs, wbase + kWSig2, 16, 64); });
    tmem_ld16(trow + kColWork, o);
    const float h0 = o[0];
    write_color_input(f, sm.cin, roff, vw, o);
    const int K1 = f.color_in_width;
    mma_round(sm, phase, [&] { issue_layer(tm + kColWork, a_cin, wbase + kWCol1, 64, K1); });
    tmem_ld64(trow + kColWork, v);
    store_relu64(sm.h1, roff, v);
    mma_round(sm, phase, [&] { issue_layer(tm + kColWork, a_h1, wbase + w_col2(f.color_in_width), 64, 64); });
    tmem_ld64(trow + kColWork, v);
    store_relu64(sm.h2, roff, v);
    mma_round(sm, phase, [&] { issue_layer(tm + kColWork, a_h2, wbase + w_col3(f.color_in_width), 16, 64); });
    tmem_ld16(trow + kColWork, o);

    // ---------------- backward ----------------
    {  // d(colour pre-activation) = d_rgb * rgb * (1 - rgb), cols 3..15 = 0
      float d3[3] = {0.f, 0.f, 0.f};
      if (valid && args.d_rgb != nullptr) {
#pragma unroll
        for (int c = 0; c < 3; ++c) {
          const float r = 1.f / (1.f + __expf(-o[c]));
          d3[c] = up_rgb[c] * r * (1.f - r);
        }
      }
      *reinterpret_cast<uint4*>(sm.g3 + 0 * kAChunk + roff) =
          make_uint4(pack_bf16x2(d3[0], d3[1]), pack_bf16x2(d3[2], 0.f), 0u, 0u);
      *reinterpret_cast<uint4*>(sm.g3 + 1 * kAChunk + roff) = make_uint4(0u, 0u, 0u, 0u);
    }
    mma_round(sm, phase, [&] {
      issue_wgrad(tm + kColW3c, a_h2, a_g3, 16, have_acc);                   // dW3c^T += H2^T dO3
      issue_dgrad(tm + kColWork, a_g3, wbase + w_col3(f.color_in_width), 64, 16);              // dH2 = dO3 W3c
    });
    tmem_ld64(trow + kColWork, v);
    relu_backward_inplace64(sm.h2, roff, v);
    mma_round(sm, phase, [&] {
      issue_wgrad(tm + kColW2c, a_h2, a_h1, 64, have_acc);                   // dW2c += dH2^T H1
      issue_dgrad(tm + kColWork, a_h2, wbase + w_col2(f.color_in_width), 64, 64);              // dH1 = dH2 W2c
    });
    tmem_ld64(trow + kColWork, v);
    relu_backward_inplace64(sm.h1, roff, v);
    mma_round(sm, phase, [&] {
      issue_wgrad(tm + kColW1c, a_h1, a_cin, K1, have_acc);                  // dW1c += dH1^T Cin
      issue_dgrad(tm + kColWork, a_h1, wbase + kWCol1, K1, 64);              // dCin = dH1 W1c
    });
    {
      float dc[48];
      tmem_ld32(trow + kColWork, dc);
      if (K1 == 48) tmem_ld16(trow + kColWork + 32, dc + 32);
      if (args.d_emb != nullptr && vw.cam >= 0) {  // d(camera embedding): colour-input features 31..30+E
        const int E = f.camera_embedding_dim;
#pragma unroll
        for (int e = 0; e < HRF_MAX_CAMERA_EMBEDDING_DIM; ++e)
          if (e < E) atomicAdd(args.d_emb + (size_t)vw.cam * E + e, dc[31 + e]);
      }
      // d(sigma-net output): col 0 from the density (truncated_exp backward, activation.py:21), 1..15 = d geo: what the
      // colour net sends back plus the caller's own gradient of QueryOutput.geometry_features (humanrf.py:185-186)
      if (args.d_geo != nullptr && valid) {
#pragma unroll
        for (int j = 0; j < HRF_GEO_DIM; ++j) dc[16 + j] += __ldg(args.d_geo + i * HRF_GEO_DIM + j);
      }
      float dh0 = 0.f;
      if (valid && args.d_sigma != nullptr)
        dh0 = up_sigma * f.density_scale * __expf(fminf(fmaxf(h0, -15.f), 15.f));
      *reinterpret_cast<uint4*>(sm.gs + 0 * kAChunk + roff) = make_uint4(
          pack_bf16x2(dh0, dc[16]), pack_bf16x2(dc[17], dc[18]), pack_bf16x2(dc[19], dc[20]), pack_bf16x2(dc[21], dc[22]));
      *reinterpret_cast<uint4*>(sm.gs + 1 * kAChunk + roff) = make_uint4(
          pack_bf16x2(dc[23], dc[24]), pack_bf16x2(dc[25], dc[26]), pack_bf16x2(dc[27], dc[28]), pack_bf16x2(dc[29], dc[30]));
    }
    mma_round(sm, phase, [&] {
      issue_wgrad(tm + kColW2s, a_hs, a_gs, 16, have_acc);                   // dW2s^T += Hs^T dOs
      issue_dgrad(tm + kColWork, a_gs, wbase + kWSig2, 64, 16);              // dHs = dOs W2s
    });
    tmem_ld64(trow + kColWork, v);
    relu_backward_inplace64(sm.hs, roff, v);
    mma_round(sm, phase, [&] {
      issue_wgrad(tm + kColW1s, a_hs, a_feat, 32, have_acc);                 // dW1s += dHs^T feat
      issue_dgrad(tm + kColWork, a_hs, wbase + kWSig1, 32, 64);              // dFeat = dHs W1s
    });
    have_acc = true;
    {
      // d(composed features) -> global, level-major [16][N] float2 (coalesced here and in the scatter)
      float df[32];
      tmem_ld32(trow + kColWork, df);
      if (valid) {
#pragma unroll
        for (int l = 0; l < 16; ++l) args.dfeat[(size_t)l * ns + i] = make_float2(df[2 * l], df[2 * l + 1]);
      }
    }
  }

  if (!weights_ready) mbar_wait(&sm.bar_w, 0);
  // ---------------- flush the weight-gradient accumulators ----------------
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  if (have_acc && args.d_mlp != nullptr) {
    const int lane = tid & 31, warp = tid >> 5;
    const int m = warp * 16 + lane;  // M=64 accumulators: row m lives in lane m%16 of sub-partition m/16
    // Every CTA adds its 11 264 partial sums into the same 44 KB at the same moment (persistent CTAs finish together):
    // rows that are contiguous per lane go out as 16-byte REDs, a quarter of the operations on those hot lines.
    const bool v4ok = (reinterpret_cast<uintptr_t>(args.d_mlp) & 15u) == 0;
    auto add_row = [&](float* dst, const float* a, int n) {   // n multiple of 4, dst 16-byte aligned when v4ok
      if (v4ok) {
#pragma unroll
        for (int c = 0; c < 64; c += 4)
          if (c < n) red_add_v4(dst + c, a[c], a[c + 1], a[c + 2], a[c + 3]);
      } else {
#pragma unroll
        for (int c = 0; c < 64; ++c)
          if (c < n) atomicAdd(dst + c, a[c]);
      }
    };
    float acc[64];
    tmem_ld32(trow + kColW1s, acc);
    if (lane < 16) add_row(args.d_mlp + kGSig1 + m * 32, acc, 32);
    tmem_ld16(trow + kColW2s, acc);
    if (lane < 16)
      for (int c = 0; c < 16; ++c) atomicAdd(args.d_mlp + kGSig2 + c * 64 + m, acc[c]);
    const int K1 = f.color_in_width;
    const int gcol2 = kGCol1 + 64 * K1, gcol3 = gcol2 + 4096;
    tmem_ld32(trow + kColW1c, acc);
    if (K1 == 48) tmem_ld16(trow + kColW1c + 32, acc + 32);
    if (lane < 16) add_row(args.d_mlp + kGCol1 + m * K1, acc, K1);
    tmem_ld64(trow + kColW2c, acc);
    if (lane < 16) add_row(args.d_mlp + gcol2 + m * 64, acc, 64);
    tmem_ld16(trow + kColW3c, acc);
    if (lane < 16)
      for (int c = 0; c < 16; ++c) atomicAdd(args.d_mlp + gcol3 + c * 64 + m, acc[c]);
  }
  tc_fence_before();
  __syncthreads();
  if (tid < 32) tmem_dealloc(sm.tmem_base, kTmemCols);
}

}  // namespace hrf

using namespace hrf;

extern "C" int hrf_field_backward_mlp(const hrf_field* f, const hrf_samples* s, const float* d_sigma, const float* d_rgb,
                                      const float* d_geo, const void* feat_bf16, const int32_t* feat_index, float* d_mlp,
                                      float* d_camera_embeddings, void* workspace, void* stream) {
  HRF_REQUIRE(f != nullptr && s != nullptr, "null argument");
  HRF_REQUIRE(f->num_segments < 255, "at most 254 temporal segments");
  if (s->num_samples == 0) return 0;
  HRF_REQUIRE(workspace != nullptr, "hrf_field_backward needs a workspace of 160 bytes per sample");
  HRF_REQUIRE(d_sigma != nullptr || d_rgb != nullptr || d_geo != nullptr, "no upstream gradient given");
  if (s->ray_origins == nullptr) {
    HRF_REQUIRE(s->positions && s->frame_numbers, "query form needs positions and frame numbers");
    HRF_REQUIRE(d_rgb == nullptr || s->directions, "radiance gradients need directions");
  }
  BwdArgs a;
  a.f = *f;
  a.s = *s;
  a.seg_grads = nullptr;
  a.d_sigma = d_sigma;
  a.d_rgb = d_rgb;
  a.d_geo = d_geo;
  a.feat_in = reinterpret_cast<const uint4*>(feat_bf16);
  a.feat_index = feat_bf16 != nullptr ? feat_index : nullptr;
  a.d_mlp = d_mlp;
  a.d_emb = d_camera_embeddings;
  a.dfeat = reinterpret_cast<float2*>(workspace);
  a.pos4 = reinterpret_cast<float4*>(reinterpret_cast<char*>(workspace) + 128 * (size_t)s->num_samples);
  a.seg8 = reinterpret_cast<uint8_t*>(reinterpret_cast<char*>(workspace) + 144 * (size_t)s->num_samples);
  const int64_t tiles = (s->num_samples + kTile - 1) / kTile;
  const int smem = (int)sizeof(BwdSmem) + 1024;
  const int64_t max_ctas = (int64_t)sm_count() * 2;
  const int grid = (int)(tiles < max_ctas ? tiles : max_ctas);
  // HRF_BWD_UNROLL=1: experiment for round 2 (the forward gained 19 % from the smaller loop; this kernel is 155 KB of SASS)
  static const bool compact = [] { const char* e = getenv("HRF_BWD_UNROLL"); return e && e[0] == '1'; }();
  if (compact) {
    HRF_CUDA(cudaFuncSetAttribute(field_backward_kernel<1>, cudaFuncAttributeMaxDynamicSharedMemorySize, smem));
    field_backward_kernel<1><<<grid, kTile, smem, reinterpret_cast<cudaStream_t>(stream)>>>(a);
  } else {
    HRF_CUDA(cudaFuncSetAttribute(field_backward_kernel<4>, cudaFuncAttributeMaxDynamicSharedMemorySize, smem));
    field_backward_kernel<4><<<grid, kTile, smem, reinterpret_cast<cudaStream_t>(stream)>>>(a);
  }
  HRF_CHECK_LAUNCH();
  return 0;
}

extern "C" int hrf_field_backward(const hrf_field* f, const hrf_samples* s, const hrf_segment_grads* seg_grads,
                                  const float* d_sigma, const float* d_rgb, const float* d_geo, const void* feat_bf16,
                                  const void* grid_feat_bf16, const int32_t* feat_index, int64_t grid_feat_stride,
                                  float* d_mlp, float* d_camera_embeddings, void* workspace, void* stream) {
  HRF_REQUIRE(seg_grads != nullptr, "null argument");
  if (int rc = hrf_field_backward_mlp(f, s, d_sigma, d_rgb, d_geo, feat_bf16, feat_index, d_mlp, d_camera_embeddings, workspace,
                                      stream))
    return rc;
  return hrf_field_backward_tables(f, s, seg_grads, grid_feat_bf16, feat_index, grid_feat_stride, workspace, 0, 4, stream);
}
