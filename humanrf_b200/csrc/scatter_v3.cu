// Table / vector gradient scatter, third generation (replaces tcnn kernel_grid_backward + compose_tensors_backward,
// tensor_composition.cu:57-118).  Same algorithm as the second generation, v2 (DESIGN.md section 3.2: parity-slot
// accumulators, the shared-corner carry of the run-length scheme as straight-line code), restructured around what ncu
// showed on v2 (profiles/r2c_*): 28 % issue-slot
// utilisation, 54 % of the stall samples on long-scoreboard waits spread over (a) the shared-memory staging of every
// level behind block-wide barriers, (b) the two vector-row loads of every step, which miss the 28 KB of L1 left beside
// 200 KB of shared memory because `vectors` is [axis][row][32 features]: the 8 bytes one (level, row) needs sit in a
// 128-byte line of their own.
//   * staging is WARP-private: a warp stages the 256 samples its own lanes walk (coalesced loads, __syncwarp), so the
//     warps of a CTA no longer stop together at every level and one warp's staging latency hides behind the others' steps;
//   * a CTA covers 8 levels (not 4) of its samples: positions / segment ids are staged half as often;
//   * the vector rows are read from a TRANSPOSED fp32 copy, vectors_t[axis][level][row][2] (hrf_segment.vectors_t, kept
//     current by the Adam kernels): the rows a warp touches at one level are contiguous, 16 to a line, and stay in L1.
#include <cstdlib>

#include "field_common.cuh"

namespace hrf {

constexpr int kV3Threads = 128, kV3Chunk = 8, kV3Samples = kV3Threads * kV3Chunk, kV3Levels = 8, kV3Row = kV3Chunk + 1;

struct ScatterV3Args {
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

struct __align__(16) V3Smem {
  float4 pos[kV3Threads * kV3Row];
  float2 df[kV3Threads * kV3Row];
  uint32_t eg[kV3Threads * kV3Row];
  uint8_t seg[kV3Samples];
};

__device__ __forceinline__ void red2(float* addr, float a, float b) {
  // (no "memory" clobber: the gradient buffers are never read in this kernel, and the clobber would pin every load of
  //  the next step behind the REDs of this one)
  asm volatile("red.global.add.v2.f32 [%0], {%1, %2};" ::"l"(addr), "f"(a), "f"(b));
}
// Table entries of the 8 vertices of a cell in parity-slot order (slot bit a = parity of the vertex coordinate on axis a).
// hashed: tcnn's coherent prime hash; dense: x + y res + z res^2, one conditional subtraction (cell inside the grid).
__device__ __forceinline__ void slot_indices(Cell A, Cell B, Cell C, bool hashed, uint32_t mulY, uint32_t mulZ, uint32_t hmask,
                                             uint32_t lsize, uint32_t (&v)[8]) {
  const uint32_t nx0 = (A.g + 1u) & ~1u, nx1 = A.g | 1u;                   // even / odd vertex on each axis
  const uint32_t ny0 = ((B.g + 1u) & ~1u) * mulY, ny1 = (B.g | 1u) * mulY;
  const uint32_t nz0 = ((C.g + 1u) & ~1u) * mulZ, nz1 = (C.g | 1u) * mulZ;
  if (hashed) {   // (uniform over the warp unless the 32 x 8 samples straddle temporal segments of different sizes)
#pragma unroll
    for (int q = 0; q < 8; ++q) v[q] = (((q & 1) ? nx1 : nx0) ^ ((q & 2) ? ny1 : ny0) ^ ((q & 4) ? nz1 : nz0)) & hmask;
  } else {
#pragma unroll
    for (int q = 0; q < 8; ++q) {
      const uint32_t t = ((q & 1) ? nx1 : nx0) + ((q & 2) ? ny1 : ny0) + ((q & 4) ? nz1 : nz0);   // < 2 * lsize (see corner_indices)
      v[q] = t >= lsize ? t - lsize : t;
    }
  }
}

// A sample whose cell lies outside a DENSE level's grid (a position outside the unit cube: only reachable through the
// QueryInput API, never through ray batches inside the AABB): the forward wraps its indices with the general modulo
// (corner_indices); the straight-line step below assumes one conditional subtraction.  Such samples take this cold,
// out-of-line path: 8 direct REDs with exactly the forward's indices, and the two vector-row REDs.
template <bool kGather>
__device__ __noinline__ void scatter_sample_slow(const uint32_t* tab, float* gtab, float* gvec, const float* vecs, bool hashed,
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
  for (int q = 0; q < 8; ++q) red2(gtab + 2 * (size_t)idx[q], w[q] * gx, w[q] * gy);
  const float dx = ex * dO.x, dy = ey * dO.y;
  red2(gvec + tp.o0 + 2 * l, dx * (1.f - tp.frac), dy * (1.f - tp.frac));
  red2(gvec + tp.o1 + 2 * l, dx * tp.frac, dy * tp.frac);
}

// kGrid: 0 xyz, 1 xyt, 2 yzt, 3 xzt (decomposition4d.py:126-129); its vector axis is t, z, x, y (tensor_composition.cu:49-52)
template <int kGrid, bool kGather>
__device__ __forceinline__ void scatter_levels(const ScatterV3Args& a, V3Smem& sm, int l0, int64_t base, int valid) {
  const hrf_field& f = a.f;
  const int tid = threadIdx.x;
  const int64_t ns = a.s.num_samples;
  constexpr int kAxis = (kGrid == 0) ? 3 : (kGrid == 1) ? 2 : (kGrid == 2) ? 0 : 1;
  const int row = tid * kV3Row;
  const int cnt = min(max(valid - tid * kV3Chunk, 0), kV3Chunk);
  // columns of this lane's 8 staging slots inside egrid: the same for every level, fetched once (per level they would
  // be a second, dependent global load in front of every staged value: 19 % of the stall samples of the first v3 cut)
  int32_t col8[kV3Chunk];        // (a launch covers < 2^31 samples)
  if (!kGather) {
    const int w0 = (tid & ~31) * kV3Chunk, lane = tid & 31;
#pragma unroll
    for (int r = 0; r < kV3Chunk; ++r) {
      const int s = w0 + lane + 32 * r;
      col8[r] = s < valid ? (a.feat_index == nullptr ? (int32_t)(base + s) : __ldg(a.feat_index + base + s)) : -1;
    }
  }
#pragma unroll 1
  for (int li = 0; li < kV3Levels; ++li) {
    const int l = l0 + li;
    __syncwarp();  // this warp's lanes are done with the previous level's df / eg
    {
      // the warp stages the 256 samples its own lanes walk (rows of threads 32w .. 32w+31): 8 coalesced loads per lane
      const int w0 = (tid & ~31) * kV3Chunk, lane = tid & 31;
      const float2* __restrict__ dfl = a.dfeat + (size_t)l * ns + base;
      float2 d8[kV3Chunk];
#pragma unroll
      for (int r = 0; r < kV3Chunk; ++r) {
        const int s = w0 + lane + 32 * r;
        d8[r] = s < valid ? __ldg(dfl + s) : make_float2(0.f, 0.f);
      }
      uint32_t e8[kV3Chunk];
      if (!kGather) {
        const uint32_t* __restrict__ eg = a.egrid + (size_t)(4 * l + kGrid) * a.egrid_stride;
#pragma unroll
        for (int r = 0; r < kV3Chunk; ++r) e8[r] = col8[r] >= 0 ? __ldg(eg + col8[r]) : 0u;
      }
#pragma unroll
      for (int r = 0; r < kV3Chunk; ++r) {
        const int s = w0 + lane + 32 * r;
        sm.df[(s >> 3) * kV3Row + (s & 7)] = d8[r];
        if (!kGather) sm.eg[(s >> 3) * kV3Row + (s & 7)] = e8[r];
      }
    }
    __syncwarp();
    const float scale = f.level_scale[l];
    const uint32_t res = f.level_res[l];

    uint32_t cur_sgi = 255u;
    uint32_t idx[8], raw[8];      // table entry of the vertex each parity slot holds, its bf16x2 value
    float accx[8], accy[8];
#pragma unroll
    for (int q = 0; q < 8; ++q) accx[q] = accy[q] = 0.f, idx[q] = 0xffffffffu, raw[q] = 0u;
    float* gtab = nullptr;
    float* gvec = nullptr;
    const uint32_t* tab = nullptr;
    const float* vecs = nullptr;
    uint32_t lsize = 1u, mulY = 0u, mulZ = 0u, hmask = 0u, vstride = 2u;
    bool hashed = false;
    uint32_t to0 = 0u, to1 = 0u;          // current tap rows of the vector axis (valid once gtab != nullptr)
    float va0 = 0.f, va1 = 0.f, vb0 = 0.f, vb1 = 0.f;
    uint32_t slow_mask = 0u;
    // the vector rows of sample j+1 are requested during step j (software pipelining: a whole step of independent work
    // between the load and its use; the dependent `tv1 - tv0` was the most-stalled instruction of the first cut)
    RowTap2 ntp{0u, 0u, 0.f};
    float2 ntv0 = make_float2(0.f, 0.f), ntv1 = make_float2(0.f, 0.f);
    bool pf = false;

#pragma unroll 1
    for (int j = 0; j < cnt; ++j) {
      const uint32_t sgi = sm.seg[tid * kV3Chunk + j];
      if (sgi == 255u) {                               // sample without a temporal segment: no gradient
        pf = false;
        continue;
      }
      const float4 p4 = sm.pos[row + j];
      const float2 dO = sm.df[row + j];
      const float c0 = (kGrid == 2) ? p4.y : p4.x;
      const float c1 = (kGrid == 0 || kGrid == 1) ? p4.y : p4.z;
      const float c2 = (kGrid == 0) ? p4.z : p4.w;
      const float cv = (kAxis == 0) ? p4.x : (kAxis == 1) ? p4.y : (kAxis == 2) ? p4.z : p4.w;
      const bool use_pf = pf && sgi == cur_sgi;
      const RowTap2 tp = use_pf ? ntp : make_row_tap2(cv, f.vec_res);
      const Cell A = to_cell(scale, c0), B = to_cell(scale, c1), C = to_cell(scale, c2);
      if (sgi != cur_sgi) {                             // (rare) new temporal segment: flush everything, new constants
        if (gtab != nullptr) {
#pragma unroll
          for (int q = 0; q < 8; ++q) {
            red2(gtab + 2 * (size_t)idx[q], accx[q], accy[q]);
            accx[q] = accy[q] = 0.f;
          }
          red2(gvec + to0 * HRF_N_FEATURES, va0, va1);
          red2(gvec + to1 * HRF_N_FEATURES, vb0, vb1);
          va0 = va1 = vb0 = vb1 = 0.f;
        }
        const hrf_segment* sg = f.segments + sgi;
        const uint32_t off = sg->level_offset[l];
        lsize = sg->level_size[l];
        hashed = ((sg->hashed_mask >> l) & 1u) != 0u;
        mulY = hashed ? kPrimeY : res;
        mulZ = hashed ? kPrimeZ : res * res;
        hmask = hashed ? lsize - 1u : 0xffffffffu;
        tab = sg->grid[kGrid] + off;
        // this level's feature pair of every row of the grid's vector axis: from the transposed copy (row stride 2) when
        // the segment has one, else from `vectors` itself (row stride 32)
        vstride = sg->vectors_t != nullptr ? 2u : (uint32_t)HRF_N_FEATURES;
        vecs = sg->vectors_t != nullptr ? sg->vectors_t + (size_t)(kAxis * HRF_N_LEVELS + l) * f.vec_res * 2
                                        : sg->vectors + (size_t)kAxis * f.vec_res * HRF_N_FEATURES + 2 * l;
        gvec = a.seg_grads[sgi].vectors + (size_t)kAxis * f.vec_res * HRF_N_FEATURES + 2 * l;   // (row stride 32)
        gtab = a.seg_grads[sgi].grid[kGrid] + 2 * (size_t)off;
        // start the runs AT this sample: its own vertices / taps are the current ones, so the step below finds nothing to
        // flush (the accumulators are zero) and the hot path needs no "slot is empty" test
        to0 = tp.i0, to1 = tp.i1;
        if (hashed || (A.g < res && B.g < res && C.g < res)) {
          slot_indices(A, B, C, hashed, mulY, mulZ, hmask, lsize, idx);
        } else {
#pragma unroll
          for (int q = 0; q < 8; ++q) idx[q] = 0u;       // (out-of-grid sample: any valid entry; it only ever receives +0)
        }
        if (kGather) {
#pragma unroll
          for (int q = 0; q < 8; ++q) raw[q] = __ldg(tab + idx[q]);
        }
        cur_sgi = sgi;
      }
      uint32_t ev = 0u;
      if (!kGather) ev = sm.eg[row + j];
      if (!hashed && (A.g >= res || B.g >= res || C.g >= res)) {   // outside a dense grid (never for samples inside the AABB):
        slow_mask |= 1u << j;                                       // handled after the loop, out of line (keeps the call, and
        pf = false;                                                 // what it does to register allocation, out of the hot loop)
        continue;
      }
      // ---- vector tap of this sample (tensor_composition.cu:37-45); a new tap pair flushes the gradient run.  The two
      // rows are fetched every step (L1 hits, issued here, consumed after the index work below): no stall on them.
      if (tp.i0 != to0 || tp.i1 != to1) {
        red2(gvec + to0 * HRF_N_FEATURES, va0, va1);
        red2(gvec + to1 * HRF_N_FEATURES, vb0, vb1);
        va0 = va1 = vb0 = vb1 = 0.f;
        to0 = tp.i0, to1 = tp.i1;
      }
      float2 tv0 = ntv0, tv1 = ntv1;
      if (!use_pf) {                                     // first sample of the thread / after a skipped sample / new segment
        tv0 = __ldg(reinterpret_cast<const float2*>(vecs + tp.i0 * vstride));
        tv1 = __ldg(reinterpret_cast<const float2*>(vecs + tp.i1 * vstride));
      }
      pf = j + 1 < cnt;
      if (pf) {
        const float4 pn = sm.pos[row + j + 1];
        ntp = make_row_tap2((kAxis == 0) ? pn.x : (kAxis == 1) ? pn.y : (kAxis == 2) ? pn.z : pn.w, f.vec_res);
        ntv0 = __ldg(reinterpret_cast<const float2*>(vecs + ntp.i0 * vstride));
        ntv1 = __ldg(reinterpret_cast<const float2*>(vecs + ntp.i1 * vstride));
      }
      // ---- cell -> the 8 vertex indices in parity-slot order; a slot whose index changed is flushed and re-keyed
      // (two different vertices that hash to the same entry keep accumulating into one slot: same table entry anyway)
      uint32_t nidx[8];
      slot_indices(A, B, C, hashed, mulY, mulZ, hmask, lsize, nidx);
#pragma unroll
      for (int q = 0; q < 8; ++q) {
        if (nidx[q] != idx[q]) {
          red2(gtab + 2 * (size_t)idx[q], accx[q], accy[q]);
          accx[q] = accy[q] = 0.f;
          idx[q] = nidx[q];
          if (kGather) raw[q] = __ldg(tab + nidx[q]);
        }
      }
      // ---- corner weights in slot order: slot bit 0 <-> even vertex = the LOWER corner iff the cell coordinate is even
      const float ax = (A.g & 1u) ? A.f : 1.f - A.f, bx = (A.g & 1u) ? 1.f - A.f : A.f;   // even-vertex / odd-vertex weight, x
      const float ay = (B.g & 1u) ? B.f : 1.f - B.f, by = (B.g & 1u) ? 1.f - B.f : B.f;
      const float az = (C.g & 1u) ? C.f : 1.f - C.f, bz = (C.g & 1u) ? 1.f - C.f : C.f;
      float w[8];
#pragma unroll
      for (int q = 0; q < 8; ++q) w[q] = (((q & 1) ? bx : ax) * ((q & 2) ? by : ay)) * ((q & 4) ? bz : az);   // same product order as corner_weights
      const float2 v = make_float2(tv0.x + tp.frac * (tv1.x - tv0.x), tv0.y + tp.frac * (tv1.y - tv0.y));
      const float gx = v.x * dO.x, gy = v.y * dO.y;
#pragma unroll
      for (int q = 0; q < 8; ++q) {
        accx[q] = __fmaf_rn(w[q], gx, accx[q]);
        accy[q] = __fmaf_rn(w[q], gy, accy[q]);
      }
      float ex = 0.f, ey = 0.f;
      if (!kGather) {
        ex = bf16_lo(ev), ey = bf16_hi(ev);
      } else {
#pragma unroll
        for (int q = 0; q < 8; ++q) {
          ex = __fmaf_rn(w[q], bf16_lo(raw[q]), ex);
          ey = __fmaf_rn(w[q], bf16_hi(raw[q]), ey);
        }
      }
      // d vectors[axis][i0/i1][2l..2l+1] = e_k * dOut * (1-frac | frac)   (tensor_composition.cu:109-111)
      const float dx = ex * dO.x, dy = ey * dO.y;
      va0 = __fmaf_rn(dx, 1.f - tp.frac, va0), va1 = __fmaf_rn(dy, 1.f - tp.frac, va1);
      vb0 = __fmaf_rn(dx, tp.frac, vb0), vb1 = __fmaf_rn(dy, tp.frac, vb1);
    }
    if (gtab != nullptr) {
#pragma unroll
      for (int q = 0; q < 8; ++q) red2(gtab + 2 * (size_t)idx[q], accx[q], accy[q]);
      if (kAxis != 3) {
        red2(gvec + to0 * HRF_N_FEATURES, va0, va1);
        red2(gvec + to1 * HRF_N_FEATURES, vb0, vb1);
      }
    }
    if (kAxis == 3) {   // grid xyz: the vector axis is time, a few hot rows: summed across the warp first (field_common.cuh)
      warp_combine_red2(gtab != nullptr ? ((cur_sgi << 24) | to0) : 0xffffffffu, gvec + to0 * HRF_N_FEATURES, va0, va1);
      warp_combine_red2(gtab != nullptr ? ((cur_sgi << 24) | to1) : 0xffffffffu, gvec + to1 * HRF_N_FEATURES, vb0, vb1);
    }
    if (slow_mask != 0u) {   // cold: samples outside a dense level's grid, one by one with the forward's general index wrap
      for (int j = 0; j < cnt; ++j) {
        if (!((slow_mask >> j) & 1u)) continue;
        const uint32_t sgi = sm.seg[tid * kV3Chunk + j];
        const float4 p4 = sm.pos[row + j];
        const float c0 = (kGrid == 2) ? p4.y : p4.x, c1 = (kGrid == 0 || kGrid == 1) ? p4.y : p4.z, c2 = (kGrid == 0) ? p4.z : p4.w;
        const float cv = (kAxis == 0) ? p4.x : (kAxis == 1) ? p4.y : (kAxis == 2) ? p4.z : p4.w;
        const hrf_segment* sg = f.segments + sgi;
        const uint32_t off = sg->level_offset[l];
        scatter_sample_slow<kGather>(sg->grid[kGrid] + off, a.seg_grads[sgi].grid[kGrid] + 2 * (size_t)off, a.seg_grads[sgi].vectors,
                                     sg->vectors, ((sg->hashed_mask >> l) & 1u) != 0u, res, sg->level_size[l], to_cell(scale, c0),
                                     to_cell(scale, c1), to_cell(scale, c2), make_tap(cv, f.vec_res, kAxis), l, sm.df[row + j],
                                     kGather ? 0u : sm.eg[row + j]);
      }
    }
  }
}

// 5 CTAs per SM: 96 registers, so the prefetch registers and the 8 staging columns fit
template <bool kGather>
__global__ void __launch_bounds__(kV3Threads, 5) grid_scatter_v3_kernel(const __grid_constant__ ScatterV3Args a) {
  extern __shared__ __align__(16) unsigned char v3_raw[];
  V3Smem& sm = *reinterpret_cast<V3Smem*>(v3_raw);
  const int64_t n = live_samples(a.s);
  const int64_t base = (int64_t)blockIdx.x * kV3Samples;
  if (base >= n) return;
  const int tid = threadIdx.x;
  const int k = a.grid_first + (int)blockIdx.y % a.grid_count;
  const int l0 = ((int)blockIdx.y / a.grid_count) * kV3Levels;
  const int valid = (int)((n - base) < kV3Samples ? (n - base) : kV3Samples);
  {   // positions / segment ids of the 256 samples this warp's lanes walk (warp-private: no block barrier anywhere)
    const int w0 = (tid & ~31) * kV3Chunk, lane = tid & 31;
#pragma unroll
    for (int r = 0; r < kV3Chunk; ++r) {
      const int s = w0 + lane + 32 * r;
      const bool ok = s < valid;
      sm.pos[(s >> 3) * kV3Row + (s & 7)] = ok ? __ldg(a.pos4 + base + s) : make_float4(0.f, 0.f, 0.f, 0.f);
      sm.seg[s] = ok ? a.seg8[base + s] : (uint8_t)255;
    }
  }
  if (k == 0) scatter_levels<0, kGather>(a, sm, l0, base, valid);       // (k is uniform over the CTA)
  else if (k == 1) scatter_levels<1, kGather>(a, sm, l0, base, valid);
  else if (k == 2) scatter_levels<2, kGather>(a, sm, l0, base, valid);
  else scatter_levels<3, kGather>(a, sm, l0, base, valid);
}

}  // namespace hrf

using namespace hrf;

int hrf_launch_scatter_v5(const hrf_field* f, const hrf_samples* s, const hrf_segment_grads* seg_grads, const void* grid_feat_bf16,
                          const int32_t* feat_index, int64_t grid_feat_stride, const void* workspace, int grid_first, int grid_count,
                          cudaStream_t st);   // scatter_v5.cu

extern "C" int hrf_field_backward_tables(const hrf_field* f, const hrf_samples* s, const hrf_segment_grads* seg_grads,
                                         const void* grid_feat_bf16, const int32_t* feat_index, int64_t grid_feat_stride,
                                         const void* workspace, int grid_first, int grid_count, void* stream) {
  HRF_REQUIRE(f != nullptr && s != nullptr && seg_grads != nullptr, "null argument");
  HRF_REQUIRE(grid_first >= 0 && grid_count >= 1 && grid_first + grid_count <= 4, "grids are 0..3 (xyz, xyt, yzt, xzt)");
  if (s->num_samples == 0) return 0;
  HRF_REQUIRE(workspace != nullptr, "needs the workspace hrf_field_backward_mlp filled");
  // HRF_SCATTER=5 (read per call: the tests switch it) runs scatter_v5.cu, which once measured faster than this kernel on
  // one workload (saved features, segment_sizes=(100,100,50)); kept for a follow-up comparison, DESIGN.md section 3.2
  if (const char* e = getenv("HRF_SCATTER"); e != nullptr && e[0] == '5' && e[1] == '\0')
    return hrf_launch_scatter_v5(f, s, seg_grads, grid_feat_bf16, feat_index, grid_feat_stride, workspace, grid_first, grid_count,
                                 reinterpret_cast<cudaStream_t>(stream));
  HRF_REQUIRE(f->vec_res < (1 << 24), "the scatter keys vector rows in 24 bits");
  ScatterV3Args a;
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
  const int64_t blocks = (s->num_samples + kV3Samples - 1) / kV3Samples;
  const dim3 grid((unsigned)blocks, (HRF_N_LEVELS / kV3Levels) * grid_count);
  const int smem = (int)sizeof(V3Smem);
  cudaStream_t st = reinterpret_cast<cudaStream_t>(stream);
  if (grid_feat_bf16 != nullptr) grid_scatter_v3_kernel<false><<<grid, kV3Threads, smem, st>>>(a);
  else grid_scatter_v3_kernel<true><<<grid, kV3Threads, smem, st>>>(a);
  HRF_CHECK_LAUNCH();
  return 0;
}
