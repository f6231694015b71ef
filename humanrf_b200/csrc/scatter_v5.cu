// Table / vector gradient scatter, fifth generation (replaces tcnn kernel_grid_backward + compose_tensors_backward,
// tensor_composition.cu:57-118).  Same arithmetic as scatter_v3.cu (and the former v4); the change is what ONE RED
// INSTRUCTION carries to the L2.
//
// ncu on v3 and v4 (profiles/r2g_*, r2i_*): two kernels with very different SM-side pictures (39 % / 49 % of the issue
// slots, 20 / 32 warps per SM) take the same 1.47 ms, and both send 145 M RED requests of ONE sector each to the L2
// (lts__t_tag_requests: 44 % on average, 69 % on the busiest slice, half of the requests crossing the die fabric).  A
// thread owns all vertices of its sample, so the 32 lanes of a RED instruction address 32 unrelated cells: one request
// per lane.  But the two vertices of a cell that differ in the FIRST axis are neighbours in the table (tcnn's hash
// multiplies the first axis by 1; a dense level is x-major): 15 times out of 16 they lie in the same 128-byte line.
// Here the 8 parity slots of a sample chunk are split over the two lanes of a LANE PAIR by the parity of the first-axis
// vertex, and the pair flushes a slot TOGETHER (when either lane's entry changed): both entries leave in the same RED
// instruction and share one L2 request.  A lane that flushes early only splits its sum in two adds.
// The vector-row gradient is split the same way: the even lane owns tap row i0, the odd lane row i1.
#include <cstddef>
#include <cstdlib>

#include "field_common.cuh"

namespace hrf {

constexpr int kV5Threads = 256, kV5Chunk = 8, kV5Chunks = kV5Threads / 2, kV5Samples = kV5Chunks * kV5Chunk, kV5Levels = 8,
              kV5Row = kV5Chunk + 1, kV5WarpSamples = 16 * kV5Chunk, kV5Stage = kV5WarpSamples / 32;

struct ScatterV5Args {
  hrf_field f;
  hrf_samples s;
  const hrf_segment_grads* seg_grads;
  const float2* dfeat;        // [16 levels][stride] float2, written by field_backward_kernel
  const float4* pos4;         // [N] (x,y,z,t)
  const uint8_t* seg8;        // [N]
  const uint32_t* egrid;      // bf16x2 [16*4][egrid_stride] per-grid features of a forward pass, or NULL (re-gather)
  const int32_t* feat_index;  // column of sample i inside egrid, or NULL
  int64_t egrid_stride;
  int grid_first, grid_count;
};

struct __align__(16) V5Smem {
  float4 pos[kV5Chunks * kV5Row];
  float2 df[kV5Chunks * kV5Row];
  uint32_t eg[kV5Chunks * kV5Row];
  uint8_t seg[kV5Samples];
};

__device__ __forceinline__ void red2v5(float* addr, float a, float b) {
  asm volatile("red.global.add.v2.f32 [%0], {%1, %2};" ::"l"(addr), "f"(a), "f"(b));
}

struct RowTap5 {
  uint32_t i0, i1;
  float frac;
};
__device__ __forceinline__ RowTap5 make_row_tap5(float coord, int vec_res) {
  const float c = __fmaf_rn(coord, (float)vec_res, -0.5f);
  const float fl = floorf(c);
  RowTap5 t;
  t.frac = c - fl;
  t.i0 = (uint32_t)min(max((int)fmaxf(fl, 0.f), 0), vec_res - 1);
  t.i1 = (uint32_t)min(max((int)fminf(fl + 1.f, (float)(vec_res - 1)), 0), vec_res - 1);
  return t;
}

// Table entries of the 4 vertices of a cell whose FIRST-axis vertex has parity p, in parity-slot order (slot bit 0 = parity
// of the second-axis vertex, bit 1 = of the third-axis vertex).  hashed: tcnn's coherent prime hash; dense: one
// conditional subtraction (cell inside the grid, see corner_indices).
__device__ __forceinline__ void slot_indices5(uint32_t p, Cell A, Cell B, Cell C, bool hashed, uint32_t mulY, uint32_t mulZ,
                                              uint32_t hmask, uint32_t lsize, uint32_t (&v)[4]) {
  const uint32_t nx = p ? (A.g | 1u) : ((A.g + 1u) & ~1u);
  const uint32_t ny0 = ((B.g + 1u) & ~1u) * mulY, ny1 = (B.g | 1u) * mulY;
  const uint32_t nz0 = ((C.g + 1u) & ~1u) * mulZ, nz1 = (C.g | 1u) * mulZ;
  if (hashed) {
#pragma unroll
    for (int q = 0; q < 4; ++q) v[q] = (nx ^ ((q & 1) ? ny1 : ny0) ^ ((q & 2) ? nz1 : nz0)) & hmask;
  } else {
#pragma unroll
    for (int q = 0; q < 4; ++q) {
      const uint32_t t = nx + ((q & 1) ? ny1 : ny0) + ((q & 2) ? nz1 : nz0);   // < 2 * lsize (see corner_indices)
      v[q] = t >= lsize ? t - lsize : t;
    }
  }
}

// cold path: a sample outside a dense level's grid (all 8 corners, the forward's general index wrap); even lane only
template <bool kGather>
__device__ __noinline__ void scatter_sample_slow5(const uint32_t* tab, float* gtab, float* gvec, const float* vecs, bool hashed,
                                                  uint32_t res, uint32_t lsize, Cell A, Cell B, Cell C, VecTap tp, int l, float2 dO,
                                                  uint32_t ev) {
  uint32_t idx[8];
  float w[8];
  corner_indices(hashed, res, lsize, A, B, C, idx);
  corner_weights(A, B, C, w);
  const float2 v0 = __ldg(reinterpret_cast<const float2*>(vecs + tp.o0 + 2 * l)), v1 = __ldg(reinterpret_cast<const float2*>(vecs + tp.o1 + 2 * l));
  const float gx = (v0.x + tp.frac * (v1.x - v0.x)) * dO.x, gy = (v0.y + tp.frac * (v1.y - v0.y)) * dO.y;
  float ex = bf16_lo(ev), ey = bf16_hi(ev);
  if (kGather) {
    ex = ey = 0.f;
    for (int q = 0; q < 8; ++q) {
      const uint32_t r = __ldg(tab + idx[q]);
      ex = __fmaf_rn(w[q], bf16_lo(r), ex), ey = __fmaf_rn(w[q], bf16_hi(r), ey);
    }
  }
  for (int q = 0; q < 8; ++q) red2v5(gtab + 2 * (size_t)idx[q], w[q] * gx, w[q] * gy);
  const float dx = ex * dO.x, dy = ey * dO.y;
  red2v5(gvec + tp.o0 + 2 * l, dx * (1.f - tp.frac), dy * (1.f - tp.frac));
  red2v5(gvec + tp.o1 + 2 * l, dx * tp.frac, dy * tp.frac);
}

// kGrid: 0 xyz, 1 xyt, 2 yzt, 3 xzt (decomposition4d.py:126-129); its vector axis is t, z, x, y (tensor_composition.cu:49-52)
template <int kGrid, bool kGather>
__device__ __forceinline__ void scatter_levels5(const ScatterV5Args& a, V5Smem& sm, int l0, int64_t base, int valid) {
  const hrf_field& f = a.f;
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const uint32_t p = (uint32_t)lane & 1u;          // parity of the first-axis vertex this lane owns; tap row it owns
  const int ch = warp * 16 + (lane >> 1);          // the chunk of 8 consecutive samples the lane pair walks
  const int64_t ns = a.s.num_samples;
  constexpr int kAxis = (kGrid == 0) ? 3 : (kGrid == 1) ? 2 : (kGrid == 2) ? 0 : 1;
  const int row = ch * kV5Row;
  const int w0 = warp * kV5WarpSamples;            // the warp stages the 128 samples its own lanes walk
  int32_t col4[kV5Stage];                          // columns of this lane's staging slots inside egrid (same for every level)
  if (!kGather) {
#pragma unroll
    for (int r = 0; r < kV5Stage; ++r) {
      const int s = w0 + lane + 32 * r;
      col4[r] = s < valid ? (a.feat_index == nullptr ? (int32_t)(base + s) : __ldg(a.feat_index + base + s)) : -1;
    }
  }
#pragma unroll 1
  for (int li = 0; li < kV5Levels; ++li) {
    const int l = l0 + li;
    __syncwarp();  // this warp's lanes are done with the previous level's df / eg
    {
      const float2* __restrict__ dfl = a.dfeat + (size_t)l * ns + base;
      float2 d4[kV5Stage];
#pragma unroll
      for (int r = 0; r < kV5Stage; ++r) {
        const int s = w0 + lane + 32 * r;
        d4[r] = s < valid ? __ldg(dfl + s) : make_float2(0.f, 0.f);
      }
      uint32_t e4[kV5Stage];
      if (!kGather) {
        const uint32_t* __restrict__ eg = a.egrid + (size_t)(4 * l + kGrid) * a.egrid_stride;
#pragma unroll
        for (int r = 0; r < kV5Stage; ++r) e4[r] = col4[r] >= 0 ? __ldg(eg + col4[r]) : 0u;
      }
#pragma unroll
      for (int r = 0; r < kV5Stage; ++r) {
        const int s = w0 + lane + 32 * r;
        sm.df[(s >> 3) * kV5Row + (s & 7)] = d4[r];
        if (!kGather) sm.eg[(s >> 3) * kV5Row + (s & 7)] = e4[r];
      }
    }
    __syncwarp();
    const float scale = f.level_scale[l];
    const uint32_t res = f.level_res[l];

    uint32_t cur_sgi = 255u;
    uint32_t idx[4], raw[4];      // table entry of the vertex each of this lane's parity slots holds, its bf16x2 value
    float accx[4], accy[4];
#pragma unroll
    for (int q = 0; q < 4; ++q) accx[q] = accy[q] = 0.f, idx[q] = 0u, raw[q] = 0u;
    float* gtab = nullptr;
    float* gvec = nullptr;
    const uint32_t* tab = nullptr;
    const float* vecs = nullptr;
    uint32_t lsize = 1u, mulY = 0u, mulZ = 0u, hmask = 0u, vstride = 2u;
    bool hashed = false;
    uint32_t to = 0u;             // the tap row of the vector axis this lane accumulates for (i0 on even lanes, i1 on odd)
    float va0 = 0.f, va1 = 0.f;
    uint32_t slow_mask = 0u;

    // Uniform trip count: every lane of the warp reaches the pair shuffle of every step (slots past `valid` carry segment
    // id 255 and do nothing).  `ok` and all branches below are the same in both lanes of a pair.
#pragma unroll 1
    for (int j = 0; j < kV5Chunk; ++j) {
      const uint32_t sgi = sm.seg[ch * kV5Chunk + j];
      bool ok = sgi != 255u;                           // 255: no temporal segment / past the end: no gradient
      uint32_t changed = 0u;
      uint32_t nidx[4] = {0u, 0u, 0u, 0u};
      Cell A{0u, 0.f}, B{0u, 0.f}, C{0u, 0.f};
      RowTap5 tp{0u, 0u, 0.f};
      float2 dO = make_float2(0.f, 0.f);
      if (ok) {
        const float4 p4 = sm.pos[row + j];
        dO = sm.df[row + j];
        const float c0 = (kGrid == 2) ? p4.y : p4.x;
        const float c1 = (kGrid == 0 || kGrid == 1) ? p4.y : p4.z;
        const float c2 = (kGrid == 0) ? p4.z : p4.w;
        const float cv = (kAxis == 0) ? p4.x : (kAxis == 1) ? p4.y : (kAxis == 2) ? p4.z : p4.w;
        tp = make_row_tap5(cv, f.vec_res);
        A = to_cell(scale, c0), B = to_cell(scale, c1), C = to_cell(scale, c2);
        if (sgi != cur_sgi) {                           // (rare) new temporal segment: flush everything, new constants
          if (gtab != nullptr) {
#pragma unroll
            for (int q = 0; q < 4; ++q) {
              red2v5(gtab + 2 * (size_t)idx[q], accx[q], accy[q]);
              accx[q] = accy[q] = 0.f;
            }
            red2v5(gvec + to * HRF_N_FEATURES, va0, va1);
            va0 = va1 = 0.f;
          }
          const hrf_segment* sg = f.segments + sgi;
          const uint32_t off = sg->level_offset[l];
          lsize = sg->level_size[l];
          hashed = ((sg->hashed_mask >> l) & 1u) != 0u;
          mulY = hashed ? kPrimeY : res;
          mulZ = hashed ? kPrimeZ : res * res;
          hmask = hashed ? lsize - 1u : 0xffffffffu;
          tab = sg->grid[kGrid] + off;
          vstride = sg->vectors_t != nullptr ? 2u : (uint32_t)HRF_N_FEATURES;
          vecs = sg->vectors_t != nullptr ? sg->vectors_t + (size_t)(kAxis * HRF_N_LEVELS + l) * f.vec_res * 2
                                          : sg->vectors + (size_t)kAxis * f.vec_res * HRF_N_FEATURES + 2 * l;
          gvec = a.seg_grads[sgi].vectors + (size_t)kAxis * f.vec_res * HRF_N_FEATURES + 2 * l;
          gtab = a.seg_grads[sgi].grid[kGrid] + 2 * (size_t)off;
          // start the runs AT this sample (nothing to flush below, no "slot is empty" test on the hot path)
          to = p ? tp.i1 : tp.i0;
          if (hashed || (A.g < res && B.g < res && C.g < res)) {
            slot_indices5(p, A, B, C, hashed, mulY, mulZ, hmask, lsize, idx);
          } else {
#pragma unroll
            for (int q = 0; q < 4; ++q) idx[q] = 0u;     // (out-of-grid sample: any valid entry; it only ever receives +0)
          }
          if (kGather) {
#pragma unroll
            for (int q = 0; q < 4; ++q) raw[q] = __ldg(tab + idx[q]);
          }
          cur_sgi = sgi;
        }
        if (!hashed && (A.g >= res || B.g >= res || C.g >= res)) {   // outside a dense grid (never for samples inside the AABB)
          slow_mask |= 1u << j;
          ok = false;
        } else {
          slot_indices5(p, A, B, C, hashed, mulY, mulZ, hmask, lsize, nidx);
#pragma unroll
          for (int q = 0; q < 4; ++q) changed |= (nidx[q] != idx[q]) ? (1u << q) : 0u;
        }
      }
      // a slot is flushed by BOTH lanes of the pair when either lane's entry changed: the two entries (first-axis
      // neighbours, same 128-byte line 15 times out of 16) travel in one RED instruction
      const uint32_t flush = changed | __shfl_xor_sync(0xffffffffu, changed, 1);
      float ex = 0.f, ey = 0.f;
      float w[4] = {0.f, 0.f, 0.f, 0.f};
      if (ok) {
        // vector rows of this sample (tensor_composition.cu:37-45): both lanes need the lerped value v
        const float2 tv0 = __ldg(reinterpret_cast<const float2*>(vecs + tp.i0 * vstride));
        const float2 tv1 = __ldg(reinterpret_cast<const float2*>(vecs + tp.i1 * vstride));
        const uint32_t trow = p ? tp.i1 : tp.i0;
        if (trow != to) {                               // a new tap row flushes this lane's vector-gradient run
          red2v5(gvec + to * HRF_N_FEATURES, va0, va1);
          va0 = va1 = 0.f;
          to = trow;
        }
#pragma unroll
        for (int q = 0; q < 4; ++q) {
          if ((flush >> q) & 1u) {
            red2v5(gtab + 2 * (size_t)idx[q], accx[q], accy[q]);
            accx[q] = accy[q] = 0.f;
            if (kGather) {
              if (nidx[q] != idx[q]) raw[q] = __ldg(tab + nidx[q]);
            }
            idx[q] = nidx[q];
          }
        }
        // corner weights in slot order: even vertex = the LOWER corner iff the cell coordinate is even
        const float wx = ((A.g & 1u) != 0u) == (p == 0u) ? A.f : 1.f - A.f;   // even vertex (p 0): upper corner iff the cell is odd
        const float ay = (B.g & 1u) ? B.f : 1.f - B.f, by = (B.g & 1u) ? 1.f - B.f : B.f;
        const float az = (C.g & 1u) ? C.f : 1.f - C.f, bz = (C.g & 1u) ? 1.f - C.f : C.f;
#pragma unroll
        for (int q = 0; q < 4; ++q) w[q] = (wx * ((q & 1) ? by : ay)) * ((q & 2) ? bz : az);   // same product order as corner_weights
        const float2 v = make_float2(tv0.x + tp.frac * (tv1.x - tv0.x), tv0.y + tp.frac * (tv1.y - tv0.y));
        const float gx = v.x * dO.x, gy = v.y * dO.y;
#pragma unroll
        for (int q = 0; q < 4; ++q) {
          accx[q] = __fmaf_rn(w[q], gx, accx[q]);
          accy[q] = __fmaf_rn(w[q], gy, accy[q]);
        }
        if (!kGather) {
          const uint32_t ev = sm.eg[row + j];
          ex = bf16_lo(ev), ey = bf16_hi(ev);
        } else {   // this lane's share of the blend
#pragma unroll
          for (int q = 0; q < 4; ++q) {
            ex = __fmaf_rn(w[q], bf16_lo(raw[q]), ex);
            ey = __fmaf_rn(w[q], bf16_hi(raw[q]), ey);
          }
        }
      }
      if (kGather) {   // the other lane's share (uniform: every lane shuffles)
        ex += __shfl_xor_sync(0xffffffffu, ex, 1);
        ey += __shfl_xor_sync(0xffffffffu, ey, 1);
      }
      if (ok) {
        // d vectors[axis][i0 | i1][2l..2l+1] = e_k * dOut * (1-frac | frac)   (tensor_composition.cu:109-111)
        const float tw = p ? tp.frac : 1.f - tp.frac;
        va0 = __fmaf_rn(ex * dO.x, tw, va0), va1 = __fmaf_rn(ey * dO.y, tw, va1);
      }
    }
    if (gtab != nullptr) {
#pragma unroll
      for (int q = 0; q < 4; ++q) red2v5(gtab + 2 * (size_t)idx[q], accx[q], accy[q]);
      if (kAxis != 3) red2v5(gvec + to * HRF_N_FEATURES, va0, va1);
    }
    if (kAxis == 3)   // grid xyz: the vector axis is time, a few hot rows: summed across the warp first (field_common.cuh)
      warp_combine_red2(gtab != nullptr ? ((cur_sgi << 24) | to) : 0xffffffffu, gvec + to * HRF_N_FEATURES, va0, va1);
    if (p == 0u && slow_mask != 0u) {   // cold: samples outside a dense level's grid, all 8 corners, even lane only
      for (int j = 0; j < kV5Chunk; ++j) {
        if (!((slow_mask >> j) & 1u)) continue;
        const uint32_t sgi = sm.seg[ch * kV5Chunk + j];
        const float4 p4 = sm.pos[row + j];
        const float c0 = (kGrid == 2) ? p4.y : p4.x, c1 = (kGrid == 0 || kGrid == 1) ? p4.y : p4.z, c2 = (kGrid == 0) ? p4.z : p4.w;
        const float cv = (kAxis == 0) ? p4.x : (kAxis == 1) ? p4.y : (kAxis == 2) ? p4.z : p4.w;
        const hrf_segment* sg = f.segments + sgi;
        const uint32_t off = sg->level_offset[l];
        scatter_sample_slow5<kGather>(sg->grid[kGrid] + off, a.seg_grads[sgi].grid[kGrid] + 2 * (size_t)off, a.seg_grads[sgi].vectors,
                                      sg->vectors, ((sg->hashed_mask >> l) & 1u) != 0u, res, sg->level_size[l], to_cell(scale, c0),
                                      to_cell(scale, c1), to_cell(scale, c2), make_tap(cv, f.vec_res, kAxis), l, sm.df[row + j],
                                      kGather ? 0u : sm.eg[row + j]);
      }
    }
  }
}

template <bool kGather>
__global__ void __launch_bounds__(kV5Threads, 4) grid_scatter_v5_kernel(const __grid_constant__ ScatterV5Args a) {
  extern __shared__ __align__(16) unsigned char v5_raw[];
  V5Smem& sm = *reinterpret_cast<V5Smem*>(v5_raw);
  const int64_t n = live_samples(a.s);
  const int64_t base = (int64_t)blockIdx.x * kV5Samples;
  if (base >= n) return;
  const int k = a.grid_first + (int)blockIdx.y % a.grid_count;
  const int l0 = ((int)blockIdx.y / a.grid_count) * kV5Levels;
  const int valid = (int)((n - base) < kV5Samples ? (n - base) : kV5Samples);
  {   // positions / segment ids of the 128 samples this warp's lanes walk (warp-private: no block barrier anywhere)
    const int lane = threadIdx.x & 31, w0 = (threadIdx.x >> 5) * kV5WarpSamples;
#pragma unroll
    for (int r = 0; r < kV5Stage; ++r) {
      const int s = w0 + lane + 32 * r;
      const bool ok = s < valid;
      sm.pos[(s >> 3) * kV5Row + (s & 7)] = ok ? __ldg(a.pos4 + base + s) : make_float4(0.f, 0.f, 0.f, 0.f);
      sm.seg[s] = ok ? a.seg8[base + s] : (uint8_t)255;
    }
  }
  if (k == 0) scatter_levels5<0, kGather>(a, sm, l0, base, valid);       // (k is uniform over the CTA)
  else if (k == 1) scatter_levels5<1, kGather>(a, sm, l0, base, valid);
  else if (k == 2) scatter_levels5<2, kGather>(a, sm, l0, base, valid);
  else scatter_levels5<3, kGather>(a, sm, l0, base, valid);
}

}  // namespace hrf

using namespace hrf;

// called from hrf_field_backward_tables (scatter_v3.cu); HRF_SCATTER=5
int hrf_launch_scatter_v5(const hrf_field* f, const hrf_samples* s, const hrf_segment_grads* seg_grads, const void* grid_feat_bf16,
                          const int32_t* feat_index, int64_t grid_feat_stride, const void* workspace, int grid_first, int grid_count,
                          cudaStream_t st) {
  HRF_REQUIRE(f->vec_res < (1 << 24), "scatter v5 keys vector rows in 24 bits");
  ScatterV5Args a;
  a.f = *f;
  a.s = *s;
  a.seg_grads = seg_grads;
  a.dfeat = reinterpret_cast<const float2*>(workspace);
  a.pos4 = reinterpret_cast<const float4*>(reinterpret_cast<const char*>(workspace) + 128 * (size_t)s->num_samples);
  a.seg8 = reinterpret_cast<const uint8_t*>(reinterpret_cast<const char*>(workspace) + 144 * (size_t)s->num_samples);
  a.egrid = reinterpret_cast<const uint32_t*>(grid_feat_bf16);
  a.feat_index = grid_feat_bf16 != nullptr ? feat_index : nullptr;
  a.egrid_stride = grid_feat_stride > 0 ? grid_feat_stride : s->num_samples;
  a.grid_first = grid_first;
  a.grid_count = grid_count;
  const int64_t blocks = (s->num_samples + kV5Samples - 1) / kV5Samples;
  const dim3 grid((unsigned)blocks, (HRF_N_LEVELS / kV5Levels) * grid_count);
  const int smem = (int)sizeof(V5Smem);
  if (grid_feat_bf16 != nullptr) grid_scatter_v5_kernel<false><<<grid, kV5Threads, smem, st>>>(a);
  else grid_scatter_v5_kernel<true><<<grid, kV5Threads, smem, st>>>(a);
  HRF_CHECK_LAUNCH();
  return 0;
}
