// msda_fast.cuh -- the sm_100a MSDeformAttn kernels for head dims 16/32/64/128 (float or bf16 value).
//
// Work decomposition (forward and backward): a "row" is one (image b, query q, head h); its D
// channels are covered by LANES = D/4 adjacent lanes holding 4 channels each, so every bilinear
// corner is ONE vectorised load per lane (16 B for float, 8 B for bf16) and a warp instruction
// covers 32/LANES rows at once (D=32: four rows per warp, 128 contiguous bytes per corner per row).
// The reference instead runs one scalar thread per channel (cuh:237-299) and, in backward, one
// D-thread block per row with two barriers and a serial reduction per point (cuh:301-403).
//
// Per row the L*P sampling locations and attention weights are turned ONCE into compact records
// in shared memory (cell offset + corner validity + weights) by the row's own lanes -- the
// coordinate arithmetic of msda_coords.cuh is done once per point, not once per channel -- and
// then broadcast-read by all lanes of the row in the gather loop.  Corner loads, their FMAs (forward)
// and dot products (backward) are predicated on the record's validity bits: a padded, gated or masked
// corner is never loaded (see PointRec).
//
// Row order (which rows a CTA works on; results never depend on it):
//   LINEAR  rows in memory order (b, q, h): a CTA = THREADS/LANES consecutive rows.
//   STRIP   a CTA = THREADS/LANES consecutive queries of ONE head (any Q).
//   TILE2D  encoder self-attention only (Q == S, query i IS pixel i of the level pyramid): a CTA = a
//           TW x TH block of pixels of ONE level and ONE head.  The tile table is derived in-kernel from the
//           DEVICE spatial_shapes, so no host copy of the shapes (and no sync) is needed.
// (Round 1 also carried a persistent 1024-thread TILED order, a head-major STRIP variant and a shared-memory
// accumulation of the coarse levels; all three were measured slower -- profiles/r01*_experiments.txt, DESIGN.md
// section 6 -- and were removed from the library in round 2.)
//
// Backward: per point each lane forms 4 partial dot products <grad_out, corner_k> over its 4
// channels; partials of 4 points are transposed-and-reduced across the row's lanes with a
// butterfly of shuffles (no shared memory, no barriers), after which one lane per point finishes
// grad_attn_weight / grad_sampling_loc; the row writes them out in full lines at its end.  grad_value is scattered with 128-bit
// vector reductions (red.global.add.v4.f32, SASS REDG.E.ADD.F32x4) -- 4x fewer atomic
// instructions than the reference's scalar atomicAdd (cuh:125-152).
#pragma once
#include <cuda_bf16.h>
#include <cuda_fp16.h>
#include <cuda_runtime.h>
#include <stdint.h>

#include <type_traits>

#include "msda_coords.cuh"

// -DMSDA_DEBUG_BOUNDS (variant builds only, tools/build_variant.sh): every corner offset that is about to be
// dereferenced -- gather, scatter, padding-mask byte -- is checked against the image; a violation prints and traps.
// The records hold UNCLAMPED offsets whose validity bits alone keep the loops inside the map, and compute-sanitizer
// is not available on the GPU pool, so this is the memcheck of the parity suite (tools/gpu_calls/gpu_r02n.sh).
#ifdef MSDA_DEBUG_BOUNDS
#include <cstdio>
#define MSDA_CHECK_OFFSET(off, limit, what)                                                                  \
  do {                                                                                                       \
    if ((unsigned)(off) >= (unsigned)(limit)) {                                                              \
      printf("msda bounds: %s offset %d outside [0, %d) (block %d thread %d)\n", what, (int)(off), (int)(limit), \
             (int)blockIdx.x, (int)threadIdx.x);                                                             \
      __trap();                                                                                              \
    }                                                                                                        \
  } while (0)
#else
#define MSDA_CHECK_OFFSET(off, limit, what) ((void)0)
#endif

namespace msda {

constexpr int kFastMaxLevels = 16;
constexpr int kFastMaxPoints = 64;  // L*P per row

// ---- 4-channel vector access --------------------------------------------------------------
__device__ __forceinline__ float4 ld4(const float* p) { return __ldg(reinterpret_cast<const float4*>(p)); }
__device__ __forceinline__ float4 ld4(const __nv_bfloat16* p) {
  const uint2 u = __ldg(reinterpret_cast<const uint2*>(p));
  float4 r;
  r.x = __uint_as_float(u.x << 16);
  r.y = __uint_as_float(u.x & 0xffff0000u);
  r.z = __uint_as_float(u.y << 16);
  r.w = __uint_as_float(u.y & 0xffff0000u);
  return r;
}
// float16 -> float32: __half22float2 is ONE HADD2.F32 (FMA pipe, not the F2F conversion unit) per two channels, and
// it is exact: every half (subnormals, Inf, NaN included) widens to the float32 with the same value
__device__ __forceinline__ float2 half2_bits_to_float2(unsigned u) {
  return __half22float2(*reinterpret_cast<const __half2*>(&u));
}
__device__ __forceinline__ unsigned pack_f16x2(float lo, float hi) {
  const __half2 t = __floats2half2_rn(lo, hi);
  return *reinterpret_cast<const unsigned*>(&t);
}
__device__ __forceinline__ float4 ld4(const __half* p) {
  const uint2 u = __ldg(reinterpret_cast<const uint2*>(p));
  const float2 a = half2_bits_to_float2(u.x), b = half2_bits_to_float2(u.y);
  return make_float4(a.x, a.y, b.x, b.y);
}
__device__ __forceinline__ void st4(float* p, const float4 v) { *reinterpret_cast<float4*>(p) = v; }
__device__ __forceinline__ void st4(__nv_bfloat16* p, const float4 v) {
  const __nv_bfloat162 lo = __floats2bfloat162_rn(v.x, v.y), hi = __floats2bfloat162_rn(v.z, v.w);
  uint2 u;
  u.x = *reinterpret_cast<const unsigned*>(&lo);
  u.y = *reinterpret_cast<const unsigned*>(&hi);
  *reinterpret_cast<uint2*>(p) = u;
}
__device__ __forceinline__ void st4(__half* p, const float4 v) {
  *reinterpret_cast<uint2*>(p) = make_uint2(pack_f16x2(v.x, v.y), pack_f16x2(v.z, v.w));
}
__device__ __forceinline__ void fma4(float4& acc, const float s, const float4 v) {
  acc.x = fmaf(s, v.x, acc.x); acc.y = fmaf(s, v.y, acc.y); acc.z = fmaf(s, v.z, acc.z); acc.w = fmaf(s, v.w, acc.w);
}
__device__ __forceinline__ float dot4(const float4 a, const float4 b) {
  return fmaf(a.w, b.w, fmaf(a.z, b.z, fmaf(a.y, b.y, a.x * b.x)));
}

// ---- CPL-channel lane vectors: 4 channels per lane (one 16-byte float load, or 8 bytes of bf16), or 8 bf16
// channels per lane (one 16-byte load).  The L1 data path is limited per 16-byte lane access, not per byte
// (profiles/r01m_microbench_ceilings.txt, item 5), so bf16 rows are gathered with 8 channels per lane.
template <int N>
struct Vec {
  float v[N];
};
template <int N>
__device__ __forceinline__ Vec<N> vzero() {
  Vec<N> r;
#pragma unroll
  for (int i = 0; i < N; ++i) r.v[i] = 0.0f;
  return r;
}
template <int N>
__device__ __forceinline__ Vec<N> ldv(const float* p) {
  static_assert(N == 4, "float rows use 4 channels per lane");
  const float4 t = __ldg(reinterpret_cast<const float4*>(p));
  Vec<4> r;
  r.v[0] = t.x; r.v[1] = t.y; r.v[2] = t.z; r.v[3] = t.w;
  return r;
}
template <int N>
__device__ __forceinline__ Vec<N> ldv(const __nv_bfloat16* p) {
  Vec<N> r;
  if constexpr (N == 4) {
    const uint2 u = __ldg(reinterpret_cast<const uint2*>(p));
    r.v[0] = __uint_as_float(u.x << 16); r.v[1] = __uint_as_float(u.x & 0xffff0000u);
    r.v[2] = __uint_as_float(u.y << 16); r.v[3] = __uint_as_float(u.y & 0xffff0000u);
  } else {
    const uint4 u = __ldg(reinterpret_cast<const uint4*>(p));
    r.v[0] = __uint_as_float(u.x << 16); r.v[1] = __uint_as_float(u.x & 0xffff0000u);
    r.v[2] = __uint_as_float(u.y << 16); r.v[3] = __uint_as_float(u.y & 0xffff0000u);
    r.v[4] = __uint_as_float(u.z << 16); r.v[5] = __uint_as_float(u.z & 0xffff0000u);
    r.v[6] = __uint_as_float(u.w << 16); r.v[7] = __uint_as_float(u.w & 0xffff0000u);
  }
  return r;
}
// float16: the same vector loads, widened pairwise (half2_bits_to_float2)
__device__ __forceinline__ void widen_f16x2(float* dst, unsigned u) {
  const float2 f = half2_bits_to_float2(u);
  dst[0] = f.x;
  dst[1] = f.y;
}
template <int N>
__device__ __forceinline__ Vec<N> ldv(const __half* p) {
  Vec<N> r;
  if constexpr (N == 4) {
    const uint2 u = __ldg(reinterpret_cast<const uint2*>(p));
    widen_f16x2(r.v, u.x); widen_f16x2(r.v + 2, u.y);
  } else {
    const uint4 u = __ldg(reinterpret_cast<const uint4*>(p));
    widen_f16x2(r.v, u.x); widen_f16x2(r.v + 2, u.y); widen_f16x2(r.v + 4, u.z); widen_f16x2(r.v + 6, u.w);
  }
  return r;
}
// The bits of one lane load, converted to floats only where they are consumed (the forward keeps several
// predicated loads in flight; holding them as packed bf16 keeps the kernel inside its register budget).
template <int N, typename VT>
struct Raw;
template <>
struct Raw<4, float> {
  float4 r;
};
template <>
struct Raw<4, __nv_bfloat16> {
  uint2 r = {0u, 0u};
};
template <>
struct Raw<8, __nv_bfloat16> {
  uint4 r = {0u, 0u, 0u, 0u};
};
template <>
struct Raw<4, __half> {
  uint2 r = {0u, 0u};
};
template <>
struct Raw<8, __half> {
  uint4 r = {0u, 0u, 0u, 0u};
};
template <int N>
__device__ __forceinline__ Raw<N, float> ldraw(const float* p) {
  static_assert(N == 4, "float rows use 4 channels per lane");
  Raw<4, float> x;
  x.r = __ldg(reinterpret_cast<const float4*>(p));
  return x;
}
template <int N>
__device__ __forceinline__ Raw<N, __nv_bfloat16> ldraw(const __nv_bfloat16* p) {
  Raw<N, __nv_bfloat16> x;
  if constexpr (N == 4) x.r = __ldg(reinterpret_cast<const uint2*>(p));
  else x.r = __ldg(reinterpret_cast<const uint4*>(p));
  return x;
}
template <int N>
__device__ __forceinline__ Raw<N, __half> ldraw(const __half* p) {
  Raw<N, __half> x;
  if constexpr (N == 4) x.r = __ldg(reinterpret_cast<const uint2*>(p));
  else x.r = __ldg(reinterpret_cast<const uint4*>(p));
  return x;
}
__device__ __forceinline__ Vec<4> unpack(const Raw<4, float>& x) {
  Vec<4> r;
  r.v[0] = x.r.x; r.v[1] = x.r.y; r.v[2] = x.r.z; r.v[3] = x.r.w;
  return r;
}
__device__ __forceinline__ Vec<4> unpack(const Raw<4, __nv_bfloat16>& x) {
  Vec<4> r;
  r.v[0] = __uint_as_float(x.r.x << 16); r.v[1] = __uint_as_float(x.r.x & 0xffff0000u);
  r.v[2] = __uint_as_float(x.r.y << 16); r.v[3] = __uint_as_float(x.r.y & 0xffff0000u);
  return r;
}
__device__ __forceinline__ Vec<8> unpack(const Raw<8, __nv_bfloat16>& x) {
  Vec<8> r;
  r.v[0] = __uint_as_float(x.r.x << 16); r.v[1] = __uint_as_float(x.r.x & 0xffff0000u);
  r.v[2] = __uint_as_float(x.r.y << 16); r.v[3] = __uint_as_float(x.r.y & 0xffff0000u);
  r.v[4] = __uint_as_float(x.r.z << 16); r.v[5] = __uint_as_float(x.r.z & 0xffff0000u);
  r.v[6] = __uint_as_float(x.r.w << 16); r.v[7] = __uint_as_float(x.r.w & 0xffff0000u);
  return r;
}
__device__ __forceinline__ Vec<4> unpack(const Raw<4, __half>& x) {
  Vec<4> r;
  widen_f16x2(r.v, x.r.x); widen_f16x2(r.v + 2, x.r.y);
  return r;
}
__device__ __forceinline__ Vec<8> unpack(const Raw<8, __half>& x) {
  Vec<8> r;
  widen_f16x2(r.v, x.r.x); widen_f16x2(r.v + 2, x.r.y); widen_f16x2(r.v + 4, x.r.z); widen_f16x2(r.v + 6, x.r.w);
  return r;
}
template <int N>
__device__ __forceinline__ void stv(float* p, const Vec<N>& a) {
  static_assert(N == 4, "float rows use 4 channels per lane");
  *reinterpret_cast<float4*>(p) = make_float4(a.v[0], a.v[1], a.v[2], a.v[3]);
}
__device__ __forceinline__ unsigned pack_bf16x2(float lo, float hi) {
  const __nv_bfloat162 t = __floats2bfloat162_rn(lo, hi);
  return *reinterpret_cast<const unsigned*>(&t);
}
template <int N>
__device__ __forceinline__ void stv(__nv_bfloat16* p, const Vec<N>& a) {
  if constexpr (N == 4) {
    *reinterpret_cast<uint2*>(p) = make_uint2(pack_bf16x2(a.v[0], a.v[1]), pack_bf16x2(a.v[2], a.v[3]));
  } else {
    *reinterpret_cast<uint4*>(p) = make_uint4(pack_bf16x2(a.v[0], a.v[1]), pack_bf16x2(a.v[2], a.v[3]),
                                              pack_bf16x2(a.v[4], a.v[5]), pack_bf16x2(a.v[6], a.v[7]));
  }
}
template <int N>
__device__ __forceinline__ void stv(__half* p, const Vec<N>& a) {
  if constexpr (N == 4) {
    *reinterpret_cast<uint2*>(p) = make_uint2(pack_f16x2(a.v[0], a.v[1]), pack_f16x2(a.v[2], a.v[3]));
  } else {
    *reinterpret_cast<uint4*>(p) = make_uint4(pack_f16x2(a.v[0], a.v[1]), pack_f16x2(a.v[2], a.v[3]),
                                              pack_f16x2(a.v[4], a.v[5]), pack_f16x2(a.v[6], a.v[7]));
  }
}
template <int N>
__device__ __forceinline__ void fmav(Vec<N>& acc, const float s, const Vec<N>& x) {
#pragma unroll
  for (int i = 0; i < N; ++i) acc.v[i] = fmaf(s, x.v[i], acc.v[i]);
}
template <int N>
__device__ __forceinline__ float dotv(const Vec<N>& a, const Vec<N>& b) {
  float r = a.v[0] * b.v[0];
#pragma unroll
  for (int i = 1; i < N; ++i) r = fmaf(a.v[i], b.v[i], r);
  return r;
}

// ---- level / tile table in shared memory -----------------------------------------------------
// Packed batches (kPrePacked) keep H / W = the padded level (location scaling and gating), start = the level's first
// token inside the image, and the image's valid rectangle h_v x w_v in the tile fields, which they do not use.
struct LevelTab {
  int H[kFastMaxLevels];
  int W[kFastMaxLevels];
  int start[kFastMaxLevels];
  union {
    int tiles_x[kFastMaxLevels];   // tile orders only
    int Wv[kFastMaxLevels];        // packed only: valid width = row pitch of the level inside the image
  };
  union {
    int tile_begin[kFastMaxLevels];  // tile orders only: first tile index of the level
    int Hv[kFastMaxLevels];          // packed only: valid height
  };
  int total_tiles;                 // tile orders only
  int cells_per_bh;                // EMIT only (deterministic sorted path): bins per (image, head), see msda_det.cuh
  int cell_begin[kFastMaxLevels];  // EMIT only: first bin of the level inside one (image, head) block
  int pad[2];
};

template <int TW, int TH>
__device__ __forceinline__ void load_levels(LevelTab* tab, const int64_t* shapes, const int64_t* lsi, int L) {
  if (threadIdx.x < L) {
    tab->H[threadIdx.x] = (int)shapes[2 * threadIdx.x];
    tab->W[threadIdx.x] = (int)shapes[2 * threadIdx.x + 1];
    tab->start[threadIdx.x] = (int)lsi[threadIdx.x];
  }
  __syncthreads();
  if (threadIdx.x == 0) {
    int acc = 0;
    for (int l = 0; l < L; ++l) {
      const int tx = (tab->W[l] + TW - 1) / TW, ty = (tab->H[l] + TH - 1) / TH;
      tab->tiles_x[l] = tx;
      tab->tile_begin[l] = acc;
      acc += tx * ty;
    }
    tab->total_tiles = acc;
  }
  __syncthreads();
}

// Bins one level owns on the deterministic sorted path: the cells of its extended (H+1) x (W+1) grid.  An empty level
// (H or W <= 0) holds no valid point, so it owns none -- (H+1)(W+1) would add W+1 or H+1 bins without adding to S and
// break det_cells_bound (msda_det.cuh).  Every table of that path (load_cell_tab, load_levels_plain<true>,
// set_single_level<..., true>) sums this.
__host__ __device__ __forceinline__ int level_cells(int H, int W) { return (H > 0 && W > 0) ? (H + 1) * (W + 1) : 0; }

// LINEAR / STRIP orders need no tile table: one barrier, no serial section.  CELLS: also the bin table of the
// deterministic sorted path (cells of the extended (H+1) x (W+1) grids, msda_det.cuh) -- thread l sums its own prefix.
template <bool CELLS = false>
__device__ __forceinline__ void load_levels_plain(LevelTab* tab, const int64_t* shapes, const int64_t* lsi, int L) {
  if (threadIdx.x < L) {
    tab->H[threadIdx.x] = (int)shapes[2 * threadIdx.x];
    tab->W[threadIdx.x] = (int)shapes[2 * threadIdx.x + 1];
    tab->start[threadIdx.x] = (int)lsi[threadIdx.x];
    if constexpr (CELLS) {
      int acc = 0;
      for (int k = 0; k < (int)threadIdx.x; ++k) acc += level_cells((int)shapes[2 * k], (int)shapes[2 * k + 1]);
      tab->cell_begin[threadIdx.x] = acc;
      if ((int)threadIdx.x == L - 1)
        tab->cells_per_bh = acc + level_cells((int)shapes[2 * threadIdx.x], (int)shapes[2 * threadIdx.x + 1]);
    }
  }
  __syncthreads();
}

// ---- packed batches (kPrePacked) -----------------------------------------------------------------
// Image b's metadata row, kPackedMetaFixed + 3*L int64: {value_start, value_count, query_start, query_count} and, per
// level, {h_v, w_v, start of the level inside the image}.  A CTA works on rows of ONE image, so the row is loaded once.
constexpr int kPackedMetaFixed = 4;
__host__ __device__ constexpr int packed_meta_stride(int L) { return kPackedMetaFixed + 3 * L; }

__device__ __forceinline__ void load_levels_packed(LevelTab* tab, const int64_t* shapes, const int64_t* img, int L) {
  if (threadIdx.x < L) {
    const int64_t* lv = img + kPackedMetaFixed + 3 * threadIdx.x;
    tab->H[threadIdx.x] = (int)shapes[2 * threadIdx.x];
    tab->W[threadIdx.x] = (int)shapes[2 * threadIdx.x + 1];
    tab->Hv[threadIdx.x] = (int)lv[0];
    tab->Wv[threadIdx.x] = (int)lv[1];
    tab->start[threadIdx.x] = (int)lv[2];
  }
  __syncthreads();
}

// DCNv3: a single level whose shape comes with the call, not from device tensors.  CELLS: also the bin table of the
// deterministic sorted path (one extended (H+1) x (W+1) grid).
template <int TW, int TH, bool CELLS = false>
__device__ __forceinline__ void set_single_level(LevelTab* tab, int H, int W) {
  if (threadIdx.x == 0) {
    tab->H[0] = H;
    tab->W[0] = W;
    tab->start[0] = 0;
    tab->tiles_x[0] = (W + TW - 1) / TW;
    tab->tile_begin[0] = 0;
    tab->total_tiles = tab->tiles_x[0] * ((H + TH - 1) / TH);
    if constexpr (CELLS) {
      tab->cell_begin[0] = 0;
      tab->cells_per_bh = level_cells(H, W);
    }
  }
  __syncthreads();
}

template <int PT>
__device__ __forceinline__ int level_of(int pt, int P) {
  if constexpr (PT > 0) {
    return pt / PT;
  } else {
    return pt / P;
  }
}

template <int D, int THREADS>
struct Geom {
  static constexpr int LANES = D / 4;
  static constexpr int RPC = THREADS / LANES;                 // rows per CTA pass
  static constexpr int TW = (RPC >= 128) ? 16 : ((RPC >= 32) ? 8 : ((RPC >= 4) ? 4 : RPC));   // tile orders only
  static constexpr int TH = RPC / TW;
  static_assert(TW * TH == RPC, "tile must cover the CTA's rows");
};

struct RowRef {
  int64_t row;   // (b*Q + q)*H + h; 0 when !live
  int b, h;
  bool live;
};

// shared-memory words per row (host and device must agree)
__host__ __device__ constexpr int fwd_row_words(int NP) {
  // float4 cw[NP] | int oc[NP] | pad
  return ((((5 * NP + 1) & ~1) + 3) & ~3) + 4;
}
__host__ __device__ constexpr int bwd_row_words(int NP) {
  // float4 cw[NP] | int4 fin[NP] | pad
  return 8 * NP + 4;
}

// Row iterator: yields this thread's row for every work item of the CTA.
// ORDER: 0 = LINEAR, 2 = STRIP (one CTA = RPC consecutive queries of ONE head; x-adjacent queries of a head share
// bilinear corners, so the CTA re-uses lines in L1 -- needs no knowledge of the level shapes and works for any Q),
// 3 = TILE2D (encoder form, Q == S: one CTA = a TW x TH pixel tile of one level and ONE head, tile index
// slowest; the grid is an upper bound computed from S alone -- surplus CTAs exit, a grid-stride step covers
// pathological pyramids -- so the level shapes never have to be known on the host).  (1 was round 1's TILED.)
template <int D, int THREADS, int ORDER>
struct RowWalk {
  static_assert(ORDER == 0 || ORDER == 2 || ORDER == 3, "row orders: LINEAR, STRIP, TILE2D");
  using G = Geom<D, THREADS>;
  int64_t item, n_items, rows;
  int rin, BH;
  __device__ __forceinline__ RowWalk() {}
  // LINEAR / STRIP do not read `tab`, so they may start before the level table is loaded
  __device__ __forceinline__ RowWalk(const LevelTab* tab, int B, int H, int64_t rows_) : rows(rows_) {
    rin = threadIdx.x / G::LANES;
    item = blockIdx.x;
    BH = B * H;
    if (ORDER == 3) n_items = (int64_t)B * H * tab->total_tiles;
    else if (ORDER == 2) n_items = (int64_t)B * H * ((rows / ((int64_t)B * H) + G::RPC - 1) / G::RPC);
    else n_items = (rows + G::RPC - 1) / G::RPC;
  }
  __device__ __forceinline__ bool done() const { return item >= n_items; }
  // LINEAR / STRIP kernels are launched with one CTA per item: a single pass, no loop-carried state.
  __device__ __forceinline__ void next() { item = (ORDER == 3) ? item + gridDim.x : n_items; }
  __device__ __forceinline__ RowRef get(const LevelTab* tab, int L, int H, int Q) const {
    RowRef r;
    if (ORDER == 2) {
      const int chunks = (Q + G::RPC - 1) / G::RPC;
      // item = blockIdx.x fits 32 bits: unsigned arithmetic instead of three 64-bit divisions per thread
      const unsigned it = (unsigned)item, bc = it / (unsigned)H, bb = bc / (unsigned)chunks;
      const int h = (int)(it - bc * (unsigned)H);
      const int q = (int)(bc - bb * (unsigned)chunks) * G::RPC + rin;
      const int b = (int)bb;
      r.live = q < Q;
      r.b = b;
      r.h = h;
      r.row = r.live ? ((int64_t)b * Q + q) * H + h : 0;
    } else if (ORDER == 3) {
      // image slowest, then tile, then head: the CTAs in flight work on one or two images, whose value / grad_value
      // (2 x 22.7 MB each at DINO-R50 shapes) stay in L2.  (Tile slowest -- round 1's order -- spreads the resident CTAs
      // over every image of the batch and doubles the DRAM traffic.)
      const unsigned it = (unsigned)item, per_img = (unsigned)H * (unsigned)tab->total_tiles;
      const unsigned bb = it / per_img, rem = it - bb * per_img;
      const unsigned t = rem / (unsigned)H;
      const int b = (int)bb, h = (int)(rem - t * (unsigned)H);
      int l = 0;
#pragma unroll 1
      for (int k = 1; k < L; ++k)
        if ((int)t >= tab->tile_begin[k]) l = k;
      const int tt = (int)t - tab->tile_begin[l];
      const int ty = tt / tab->tiles_x[l], tx = tt - ty * tab->tiles_x[l];
      const int y = ty * G::TH + rin / G::TW, x = tx * G::TW + rin % G::TW;
      const int q = tab->start[l] + y * tab->W[l] + x;
      r.live = (y < tab->H[l]) && (x < tab->W[l]) && (q < Q);
      r.b = b;
      r.h = h;
      r.row = r.live ? ((int64_t)b * Q + q) * H + h : 0;
    } else {
      const int64_t row = item * G::RPC + rin;
      r.live = row < rows;
      r.row = r.live ? row : 0;
      r.h = (int)(r.row % H);
      r.b = (int)(r.row / H / Q);
    }
    return r;
  }
};

// The CTA's image and this thread's row.  LINEAR (forward): blockIdx.x = image * chunks + chunk, a chunk = RPC
// consecutive (query, head) rows of the image, chunks = ceil(max_q * H / RPC).  STRIP (backward): blockIdx.x =
// (image * chunks + chunk) * H + head, a chunk = RPC consecutive queries, chunks = ceil(max_q / RPC).  Every image
// gets the grid of the largest one; a CTA past its image's rows is surplus (uniform over the CTA) and exits.
struct PackedRow {
  RowRef r;
  const int64_t* img;   // the image's metadata row
  bool surplus;
};
template <int RPC, int ORDER>
__device__ __forceinline__ PackedRow packed_row(const int64_t* meta, int L, int H, int max_q, int rin) {
  static_assert(ORDER == 0 || ORDER == 2, "packed batches: LINEAR forward, STRIP backward");
  PackedRow p;
  const unsigned it = blockIdx.x;
  unsigned b, chunk;
  int h = 0;
  if (ORDER == 2) {
    const unsigned chunks = (unsigned)((max_q + RPC - 1) / RPC), bc = it / (unsigned)H;
    h = (int)(it - bc * (unsigned)H);
    b = bc / chunks;
    chunk = bc - b * chunks;
  } else {
    const unsigned chunks = (unsigned)((max_q * H + RPC - 1) / RPC);
    b = it / chunks;
    chunk = it - b * chunks;
  }
  p.img = meta + (int64_t)b * packed_meta_stride(L);
  const int64_t q0 = __ldg(p.img + 2);
  const int nq = (int)__ldg(p.img + 3);
  p.r.b = (int)b;
  if (ORDER == 2) {
    const int q = (int)chunk * RPC + rin;
    p.surplus = (int)chunk * RPC >= nq;
    p.r.live = q < nq;
    p.r.h = h;
    p.r.row = p.r.live ? (q0 + q) * H + h : 0;
  } else {
    const int local = (int)chunk * RPC + rin;
    p.surplus = (int)chunk * RPC >= nq * H;
    p.r.live = local < nq * H;
    p.r.h = local % H;
    p.r.row = p.r.live ? q0 * H + local : 0;
  }
  return p;
}

// The validity bits of a cell restricted to the image's valid rectangle [0, w_v) x [0, h_v) -- what a
// key_padding_mask that is exactly that rectangle does to the bits (apply_value_mask) -- for a level stored with
// row pitch w_v.
__device__ __forceinline__ Cell<float> clip_to_rect(Cell<float> c, int hv, int wv) {
  const bool x0 = c.x0 < wv, x1 = c.x0 + 1 < wv, y0 = c.y0 < hv, y1 = c.y0 + 1 < hv;
  c.valid &= (unsigned)(y0 && x0) | ((unsigned)(y0 && x1) << 1) | ((unsigned)(y1 && x0) << 2) |
             ((unsigned)(y1 && x1) << 3);
  return c;
}

// ---- per-point record --------------------------------------------------------------------------
// oc = element offset, inside the image, of the bilinear cell's (x0, y0) corner -- NOT clamped: it lies outside the
// map when that corner is padded, and is then never dereferenced -- with four corner-validity bits in its low bits
// (the offset is a multiple of D >= 16):
//   bit k  corner k = (x0 + (k & 1), y0 + (k >> 1)) is inside the map (and, in the fused module path, not under the
//          padding mask); k: 0=(y0,x0) 1=(y0,x0+1) 2=(y0+1,x0) 3=(y0+1,x0+1)   (v1..v4 of cuh:56-80)
// The corner offsets are oc, oc + H*D, oc + W_l*H*D, oc + (W_l+1)*H*D: no selects in the loops.  A corner whose bit
// is clear is NOT LOADED (the loads are predicated on the bits), exactly as the reference's per-corner bounds checks
// skip it (cuh:56-80): it costs no L1 data-pipe wavefront -- on model-like inputs ~14 % of all corners are padded --
// and a non-finite value in a pixel that is padded or masked for this point cannot leak into the result.  All bits
// clear = the point is gated out (cuh:288) and contributes nothing.
struct PointRec {
  float4 cw;     // corner weights (v1..v4 of cuh:56-80) x attention weight, exactly 0 where the bit is clear
  int oc;
  int pix;       // pixel index (inside the image) of the (x0, y0) corner, not clamped: oc == ((pix*H + h)*D) | bits
  float lw, lh;  // fractional parts
};

// DCNv3 gives pixel coordinates directly (cuh:262-263 gate, :48-58 cell), no exact-product trick needed.  DCNv2
// (msda_dcnv2.cu) has the same gate and cell, in float or -- its generic kernels -- double.
template <typename T>
__device__ __forceinline__ Cell<T> locate_pixel(T px, T py, int H, int W) {
  Cell<T> c;
  const bool ok = (py > (T)-1) && (px > (T)-1) && (py < (T)H) && (px < (T)W);
  const T fy = floor(py), fx = floor(px);
  c.y0 = ok ? (int)fy : 0;
  c.x0 = ok ? (int)fx : 0;
  c.lh = ok ? py - fy : (T)0;
  c.lw = ok ? px - fx : (T)0;
  unsigned v = 0;
  if (ok) {
    const bool y0ok = c.y0 >= 0, y1ok = c.y0 + 1 <= H - 1, x0ok = c.x0 >= 0, x1ok = c.x0 + 1 <= W - 1;
    v = (unsigned)(y0ok && x0ok) | ((unsigned)(y0ok && x1ok) << 1) | ((unsigned)(y1ok && x0ok) << 2) |
        ((unsigned)(y1ok && x1ok) << 3);
  }
  c.valid = v;
  return c;
}

__device__ __forceinline__ PointRec record_from_cell(const Cell<float> c, float aw, int Wl, int start, int H, int h,
                                                     int D) {
  PointRec r;
  const float hh = 1.0f - c.lh, hw = 1.0f - c.lw;
  r.cw.x = (c.valid & 1u) ? hh * hw * aw : 0.0f;
  r.cw.y = (c.valid & 2u) ? hh * c.lw * aw : 0.0f;
  r.cw.z = (c.valid & 4u) ? c.lh * hw * aw : 0.0f;
  r.cw.w = (c.valid & 8u) ? c.lh * c.lw * aw : 0.0f;
  r.pix = (c.valid == 0u) ? 0 : start + c.y0 * Wl + c.x0;
  r.oc = ((r.pix * H + h) * D) | (int)c.valid;
  r.lw = c.lw;
  r.lh = c.lh;
  return r;
}

__device__ __forceinline__ PointRec make_record(float x, float y, float aw, int Hl, int Wl, int start, int H, int h,
                                                int D) {
  return record_from_cell(locate<float>(x, y, Hl, Wl), aw, Wl, start, H, h, D);
}

// ---- fused pre-op chain (SURVEY section 8f-1) -----------------------------------------------------
// FUSED kernels take what the module's two Linear layers produce -- raw sampling offsets
// [B,Q,H,L,P,2] and attention logits [B,Q,H,L*P] -- plus the reference points [B,Q,L,2|4], and do the
// softmax over L*P and the sampling-location affine (multi_scale_deform_attn.py:300-332) while they
// build the records, so sampling_locations / attention_weights never exist in HBM.  The arithmetic
// keeps torch's operation order (separate div / mul / add roundings, no fma), so the locations are
// bit-identical to the unfused module's.
struct FusedArgs {
  const float* ref;   // reference_points [B, Q, L, ref_dim]
  // key_padding_mask [B, S] (one byte per pixel, non-zero = padded), or null: the module's
  // value.masked_fill(key_padding_mask[..., None], 0) (multi_scale_deform_attn.py:291-292) folded into the
  // kernels -- a masked pixel's row reads as zeros, see apply_value_mask
  const unsigned char* value_mask;
  int ref_dim;        // 2: loc = ref + off / (W_l, H_l);  4: loc = ref_xy + off / P * ref_wh * 0.5
  float inv_P;        // 1 / P (backward chain rule)
  float num_P;        // P as a float: the forward divides (torch computes off / P, not off * (1/P))
  // PRE == 2 (DCNv3, SURVEY section 8f-4): the same gather/scatter core driven by a convolution-style
  // sampling grid (detrex/layers/csrc/DCNv3/dcnv3_im2col_cuda.cuh:217-275): rows are (n, output pixel,
  // group), the K = kernel_w*kernel_h points of a row sit at
  //   loc_w = p0_w - (dil_w*(kw-1)/2)*scale + (i*dil_w + offset_w)*scale   (pixel units, i outer, j inner)
  // `loc` holds the offsets [N, Ho, Wo, G*K*2], `w` the mask [N, Ho, Wo, G*K]; one level = the input map.
  // PRE == 3 (fused DCNv3 module path): the same grid, `w` the mask LOGITS -- the DCNv3 module's softmax over the K
  // points of a (pixel, group) row runs inside the kernels, as the fused MSDA chain's softmax over L*P does.
  int kernel_h, kernel_w, stride_h, stride_w, pad_h, pad_w, dil_h, dil_w;
  int height_in, width_in, width_out;
  float offset_scale;
};
// PRE: 0 = sampling_locations / attention_weights given (the reference operator), 1 = fused module chain,
//      2 = DCNv3 sampling grid, 3 = DCNv3 sampling grid + softmax over the row's mask logits,
//      4 = fused module chain over a packed batch (valid pixels only, see packed_row; `lsi` is then the per-image
//          metadata and `S` unused)
constexpr int kPrePlain = 0, kPreFused = 1, kPreDcn = 2, kPreDcnSoftmax = 3, kPrePacked = 4;
// the record modes whose `w` holds logits: the row softmax in forward, its chain rule in backward
__host__ __device__ constexpr bool pre_softmax(int pre) {
  return pre == kPreFused || pre == kPreDcnSoftmax || pre == kPrePacked;
}
// the record modes of the MSDA module chain: location affine from raw offsets and reference points
__host__ __device__ constexpr bool pre_fused(int pre) { return pre == kPreFused || pre == kPrePacked; }
// the record modes on the DCNv3 convolution grid
__host__ __device__ constexpr bool pre_dcn(int pre) { return pre == kPreDcn || pre == kPreDcnSoftmax; }

__device__ __forceinline__ float2 fused_location(const float2 off, const float* r, int ref_dim, int Hl, int Wl,
                                                 float num_P) {
  float2 loc;
  if (ref_dim == 2) {
    loc.x = __fadd_rn(__ldg(r + 0), __fdiv_rn(off.x, (float)Wl));
    loc.y = __fadd_rn(__ldg(r + 1), __fdiv_rn(off.y, (float)Hl));
  } else {
    loc.x = __fadd_rn(__ldg(r + 0), __fmul_rn(__fmul_rn(__fdiv_rn(off.x, num_P), __ldg(r + 2)), 0.5f));
    loc.y = __fadd_rn(__ldg(r + 1), __fmul_rn(__fmul_rn(__fdiv_rn(off.y, num_P), __ldg(r + 3)), 0.5f));
  }
  return loc;
}

// Padding mask folded into the records.  A masked pixel's value row counts as zeros: the corner's validity bit is
// cleared and its weight set to 0, so the forward neither loads it nor adds anything for it, the backward scatters
// nothing into it (grad_value of a masked pixel stays 0, which is masked_fill's own backward) and drops its value
// from grad_sampling_loc / grad_attn_weight -- whereas a corner whose weight merely happens to be 0 (lw == 0, say)
// keeps its bit and still enters the location gradient.  Only the mask bytes of in-map corners are read.
__device__ __forceinline__ void apply_value_mask(PointRec& r, const unsigned char* mask_img, int Wl, int S) {
  const int v = r.oc & 15;
#ifdef MSDA_DEBUG_BOUNDS
  if (v & 1) MSDA_CHECK_OFFSET(r.pix, S, "mask k0");
  if (v & 2) MSDA_CHECK_OFFSET(r.pix + 1, S, "mask k1");
  if (v & 4) MSDA_CHECK_OFFSET(r.pix + Wl, S, "mask k2");
  if (v & 8) MSDA_CHECK_OFFSET(r.pix + Wl + 1, S, "mask k3");
#else
  (void)S;
#endif
  const bool k0 = (v & 1) && __ldg(mask_img + r.pix) == 0, k1 = (v & 2) && __ldg(mask_img + r.pix + 1) == 0;
  const bool k2 = (v & 4) && __ldg(mask_img + r.pix + Wl) == 0, k3 = (v & 8) && __ldg(mask_img + r.pix + Wl + 1) == 0;
  r.cw.x = k0 ? r.cw.x : 0.0f;
  r.cw.y = k1 ? r.cw.y : 0.0f;
  r.cw.z = k2 ? r.cw.z : 0.0f;
  r.cw.w = k3 ? r.cw.w : 0.0f;
  r.oc = (r.oc & ~15) | (int)k0 | ((int)k1 << 1) | ((int)k2 << 2) | ((int)k3 << 3);
}

// DCNv3 sampling position of kernel point `pt` (= i*kernel_h + j, i over kernel_w) for output pixel q,
// in input-pixel units (dcnv3_im2col_cuda.cuh:232-260).
__device__ __forceinline__ float2 dcn_location(const float2 off, int pt, int q, const FusedArgs& a) {
  const int wo = q % a.width_out, ho = q / a.width_out;
  const int i = pt / a.kernel_h, j = pt - i * a.kernel_h;
  const int cw = (a.dil_w * (a.kernel_w - 1)) >> 1, ch = (a.dil_h * (a.kernel_h - 1)) >> 1;
  const float p0w = (float)(cw - a.pad_w + wo * a.stride_w) - (float)cw * a.offset_scale;
  const float p0h = (float)(ch - a.pad_h + ho * a.stride_h) - (float)ch * a.offset_scale;
  float2 loc;
  loc.x = fmaf((float)(i * a.dil_w) + off.x, a.offset_scale, p0w);
  loc.y = fmaf((float)(j * a.dil_h) + off.y, a.offset_scale, p0h);
  return loc;
}

// ---- element type of loc / w and their gradients (AT) ----------------------------------------------------------
// float, or -- in the record modes whose `w` holds logits (fused MSDA chain, fused DCNv3) -- the value's own 16-bit
// type, which is what the module's Linear layers produce under autocast.  Widening f16 / bf16 to float is exact, so the
// kernels compute on the same floats either way; gradients are rounded once, to nearest even, as a cast would.
__device__ __forceinline__ float2 ld_xy(const float* base, int pt) {   // the (x, y) pair of point pt
  return __ldg(reinterpret_cast<const float2*>(base) + pt);
}
__device__ __forceinline__ float2 ld_xy(const __half* base, int pt) {
  const unsigned u = __ldg(reinterpret_cast<const unsigned*>(base) + pt);
  return __half22float2(*reinterpret_cast<const __half2*>(&u));
}
__device__ __forceinline__ float2 ld_xy(const __nv_bfloat16* base, int pt) {
  const unsigned u = __ldg(reinterpret_cast<const unsigned*>(base) + pt);
  return __bfloat1622float2(*reinterpret_cast<const __nv_bfloat162*>(&u));
}
__device__ __forceinline__ float ld_aux(const float* p) { return __ldg(p); }
__device__ __forceinline__ float ld_aux(const __half* p) { return __half2float(__ldg(p)); }
__device__ __forceinline__ float ld_aux(const __nv_bfloat16* p) { return __bfloat162float(__ldg(p)); }
// two gradients as one store: 8 bytes of float, 4 of f16 / bf16
__device__ __forceinline__ void st_aux2(float* p, float a, float b) { *reinterpret_cast<float2*>(p) = make_float2(a, b); }
__device__ __forceinline__ void st_aux2(__half* p, float a, float b) { *reinterpret_cast<unsigned*>(p) = pack_f16x2(a, b); }
__device__ __forceinline__ void st_aux2(__nv_bfloat16* p, float a, float b) {
  const __nv_bfloat162 t = __floats2bfloat162_rn(a, b);
  *reinterpret_cast<unsigned*>(p) = *reinterpret_cast<const unsigned*>(&t);
}
// four gradients as one store: 16 bytes of float, 8 of f16 / bf16
__device__ __forceinline__ void st_aux4(float* p, float4 v) { *reinterpret_cast<float4*>(p) = v; }
__device__ __forceinline__ void st_aux4(__half* p, float4 v) { st4(p, v); }
__device__ __forceinline__ void st_aux4(__nv_bfloat16* p, float4 v) { st4(p, v); }
__device__ __forceinline__ void st_aux1(float* p, float a) { *p = a; }
__device__ __forceinline__ void st_aux1(__half* p, float a) { *p = __float2half_rn(a); }
__device__ __forceinline__ void st_aux1(__nv_bfloat16* p, float a) { *p = __float2bfloat16_rn(a); }
// the (value type, aux type) pairs the kernels are built for: AT == float, or AT == VT (16-bit) in a logits mode
// (kPreFused, kPreDcnSoftmax) and the one row order per pass the product library carries for it (ORDER_16)
template <typename VT, typename AT, int PRE, int ORDER, int ORDER_16>
__host__ __device__ constexpr bool aux_ok() {
  return std::is_same_v<AT, float> ||
         (std::is_same_v<AT, VT> && sizeof(VT) == 2 && (PRE == 1 || PRE == 3 || PRE == 4) && ORDER == ORDER_16);
}

// softmax over the row's NP logits by the row's LANES lanes; e_i = exp(x_i - max) is left in
// scratch[pt] (one float per point, any 4-byte stride) and the sum is returned: w_i = e_i / sum.
// VLANES = 2 * LANES (rows of 8 channels per lane) forms the sum in the order of VLANES lanes: lane `sub` adds up the
// points of virtual lanes sub and sub + LANES separately and then the two -- the first butterfly step of the wider
// order -- so the weights are bit for bit those of the 4-channel-per-lane rows (f16 forward == f32 forward).
template <int LANES, int STRIDE, int VLANES = LANES, typename AT>
__device__ __forceinline__ float row_softmax(const AT* logits_row, float* scratch, int NP, int sub) {
  static_assert(VLANES == LANES || VLANES == 2 * LANES, "one or two virtual lanes per lane");
  float m = -3.402823466e38f;
  for (int pt = sub; pt < NP; pt += LANES) {
    const float x = ld_aux(logits_row + pt);
    scratch[pt * STRIDE] = x;
    m = fmaxf(m, x);
  }
#pragma unroll
  for (int k = LANES / 2; k > 0; k >>= 1) m = fmaxf(m, __shfl_xor_sync(0xffffffffu, m, k));
  auto partial = [&](int first) {
    float s = 0.0f;
    for (int pt = first; pt < NP; pt += VLANES) {
      const float e = expf(scratch[pt * STRIDE] - m);
      scratch[pt * STRIDE] = e;
      s += e;
    }
    return s;
  };
  float sum = partial(sub);
  if constexpr (VLANES != LANES) sum += partial(sub + LANES);
#pragma unroll
  for (int k = LANES / 2; k > 0; k >>= 1) sum += __shfl_xor_sync(0xffffffffu, sum, k);
  return sum;
}

// =============================================================================================
// Forward
// =============================================================================================
// One pass per CTA (TILE2D: a grid-stride step for pathological pyramids); phase 1 reads loc/w straight from
// global memory.
template <int D, typename VT, int PT, int THREADS, int ORDER, int PRE, int CPL, typename AT = float>
#ifndef MSDA_FWD_MINB
#define MSDA_FWD_MINB 6
#endif
__global__ void __launch_bounds__(THREADS, MSDA_FWD_MINB * (256 / THREADS))
msda_fwd_fast_kernel(const VT* __restrict__ value, const int64_t* __restrict__ shapes,
                     const int64_t* __restrict__ lsi, const AT* __restrict__ loc,
                     const AT* __restrict__ w, VT* __restrict__ out, const FusedArgs fused, int B, int S, int H,
                     int L, int Q, int P, int64_t rows) {
  // FUSED: `loc` holds raw sampling offsets and `w` attention logits (see FusedArgs)
  static_assert(THREADS <= 256, "single-pass CTAs");
  static_assert(aux_ok<VT, AT, PRE, ORDER, 0>(), "16-bit offsets / logits: fused modes, value's dtype, LINEAR forward");
  constexpr int DL = D * 4 / CPL;               // lane geometry: LANES = D / CPL lanes per row
  using G = Geom<DL, THREADS>;
  constexpr int LANES = G::LANES;
  // f16 rows sum the fused softmax in the f32 rows' lane order (row_softmax), so the f16 forward is the f32 forward
  // on the widened value; bf16 keeps its own order
  constexpr int SM_LANES = std::is_same_v<VT, __half> ? D / 4 : LANES;
  constexpr bool SOFTMAX = pre_softmax(PRE);    // `w` holds logits: row softmax (fused MSDA chain, fused DCNv3)
  constexpr bool FUSED = pre_fused(PRE);        // MSDA chain only: location affine, reference points, padding mask
  constexpr bool PACKED = (PRE == kPrePacked);  // packed batch: `lsi` = per-image metadata, one image per CTA
  static_assert(!PACKED || ORDER == 0, "the packed forward is LINEAR");
  constexpr bool DCN = pre_dcn(PRE);
  extern __shared__ __align__(16) unsigned char smem_raw[];
  LevelTab* tab = reinterpret_cast<LevelTab*>(smem_raw);
  float* recs = reinterpret_cast<float*>(smem_raw + sizeof(LevelTab));
  const int NP = L * P;
  const int row_words = fwd_row_words(NP);

  const int sub = (threadIdx.x & 31) % LANES;            // lane inside the row
  const int rin = threadIdx.x / LANES;                   // row inside the CTA
  const int HD = H * D;
  float* my = recs + (size_t)rin * row_words;
  float4* s_cw = reinterpret_cast<float4*>(my);
  int* s_oc = reinterpret_cast<int*>(my + 4 * NP);
  // -DMSDA_FWD_REC16=1 (experiment, VERDICT r01 task 4): a 16-byte record {oc | validity bits, lw, (1-lh)*aw, lh*aw}
  // whose four corner weights the gather loop forms itself (1 FADD + 4 FMUL): ONE LDS.128 per point = 2 L1 data-pipe
  // wavefronts per point and warp instead of 3 (LDS.128 + LDS.32).  Measured with the clamped-address loop of round 1:
  // cfg2 model 0.609 -> 0.589 ms, cfg2 test 0.566 -> 0.579 ms; with the predicated loads below it buys nothing
  // (0.551 either way) and still costs the inputs without locality (0.583 -> 0.615 ms): off (profiles/r02j_*).
#ifndef MSDA_FWD_REC16
#define MSDA_FWD_REC16 0
#endif
  constexpr bool REC16 = MSDA_FWD_REC16 != 0;
  int4* s_rec = reinterpret_cast<int4*>(my);             // REC16 only (s_oc stays the fused softmax's scratch)

  // Single-pass orders (LINEAR, STRIP) know their row without the level table, so the first locations / weights
  // of the row are requested BEFORE the table's load + barrier: the two global-memory latencies of a CTA's
  // start-up overlap instead of adding up.
  // (FUSED: the raw offsets are requested and the row's softmax is done before the barrier.)
  constexpr bool EARLY = (ORDER == 0 || ORDER == 2) && !DCN;
  constexpr int kEarly = 2;                              // row-loop iterations whose loads are issued early
  float2 early_xy[kEarly];
  float early_w[kEarly];
  float early_sum = 1.0f;                                // SOFTMAX: softmax denominator of the row
  RowWalk<DL, THREADS, ORDER> walk;
  RowRef cur;
  const int64_t* pimg = nullptr;                         // PACKED: the CTA's image metadata row
  if constexpr (EARLY) {
    if constexpr (PACKED) {
      const PackedRow p = packed_row<G::RPC, ORDER>(lsi, L, H, Q, rin);
      if (p.surplus) return;                             // uniform over the CTA
      cur = p.r;
      pimg = p.img;
    } else {
      walk = RowWalk<DL, THREADS, ORDER>(tab, B, H, rows);
      if (walk.done()) return;                             // uniform over the CTA
      cur = walk.get(tab, L, H, Q);
    }
#pragma unroll
    for (int i = 0; i < kEarly; ++i) {
      const int pt = sub + i * LANES;
      const bool on = cur.live && pt < NP;
      early_xy[i] = on ? ld_xy(loc + cur.row * (int64_t)NP * 2, pt) : make_float2(0.f, 0.f);
      early_w[i] = (on && !SOFTMAX) ? ld_aux(w + cur.row * (int64_t)NP + pt) : 0.0f;
    }
    // the softmax shuffles need the whole warp; dead rows read row 0 and simply produce nothing
    if constexpr (SOFTMAX) early_sum = row_softmax<LANES, 1, SM_LANES>(w + cur.row * (int64_t)NP, reinterpret_cast<float*>(s_oc), NP, sub);
    if constexpr (PACKED) load_levels_packed(tab, shapes, pimg, L);
    else load_levels_plain(tab, shapes, lsi, L);
  } else {
    if constexpr (DCN) set_single_level<G::TW, G::TH>(tab, fused.height_in, fused.width_in);
    else if constexpr (ORDER == 0 || ORDER == 2) load_levels_plain(tab, shapes, lsi, L);
    else load_levels<G::TW, G::TH>(tab, shapes, lsi, L);
    walk = RowWalk<DL, THREADS, ORDER>(tab, B, H, rows);
    if (walk.done()) return;
    cur = walk.get(tab, L, H, Q);
  }
  while (true) {
    // ---- phase 1: records ----
    {
      const AT* lp = loc + cur.row * (int64_t)NP * 2;
      const AT* wp = w + cur.row * (int64_t)NP;
      float sm_sum = early_sum;
      if constexpr (SOFTMAX && !EARLY) sm_sum = row_softmax<LANES, 1, SM_LANES>(wp, reinterpret_cast<float*>(s_oc), NP, sub);
      if (cur.live) {
        const float* rp = FUSED ? fused.ref + (cur.row / H) * (int64_t)L * fused.ref_dim : nullptr;
        // one record from a point's raw location / weight (FUSED: raw offset; SOFTMAX: the weight comes from the
        // softmax)
        auto build = [&](int pt, float2 xy, float aw) {
          const int l = level_of<PT>(pt, P);
          if constexpr (SOFTMAX) aw = __fdiv_rn(__int_as_float(s_oc[pt]), sm_sum);
          if constexpr (FUSED)
            xy = fused_location(xy, rp + l * fused.ref_dim, fused.ref_dim, tab->H[l], tab->W[l], fused.num_P);
          PointRec r;
          if constexpr (DCN) {
            const float2 px = dcn_location(xy, pt, (int)((cur.row / H) % Q), fused);
            r = record_from_cell(locate_pixel(px.x, px.y, tab->H[0], tab->W[0]), aw, tab->W[0], 0, H, cur.h, D);
          } else if constexpr (PACKED) {
            r = record_from_cell(clip_to_rect(locate<float>(xy.x, xy.y, tab->H[l], tab->W[l]), tab->Hv[l], tab->Wv[l]),
                                 aw, tab->Wv[l], tab->start[l], H, cur.h, D);
          } else {
            r = make_record(xy.x, xy.y, aw, tab->H[l], tab->W[l], tab->start[l], H, cur.h, D);
          }
          if constexpr (FUSED && !PACKED) {
            if (fused.value_mask) apply_value_mask(r, fused.value_mask + (int64_t)cur.b * S, tab->W[l], S);
          }
          if constexpr (REC16) {
            s_rec[pt] = make_int4(r.oc, __float_as_int(r.lw), __float_as_int((1.0f - r.lh) * aw), __float_as_int(r.lh * aw));
          } else {
            s_cw[pt] = r.cw;
            s_oc[pt] = r.oc;
          }
        };
        int pt = sub;
        if constexpr (EARLY) {   // the loads of these iterations were issued before the level table's barrier
#pragma unroll
          for (int i = 0; i < kEarly; ++i, pt += LANES)
            if (pt < NP) build(pt, early_xy[i], early_w[i]);
        }
        for (; pt < NP; pt += LANES) build(pt, ld_xy(lp, pt), SOFTMAX ? 0.0f : ld_aux(wp + pt));
      }
    }
    __syncwarp();

    // ---- phase 2: gather ----
    if (cur.live) {
      const VT* vimg = value + (PACKED ? __ldg(pimg) * HD : (int64_t)cur.b * S * HD) + sub * CPL;
      asm volatile("" : "+l"(vimg));   // keep the row base as ONE 64-bit register: corner address = base + off*4 (IMAD.WIDE)
#ifdef MSDA_DEBUG_BOUNDS
      const int lim = PACKED ? (int)__ldg(pimg + 1) * HD : S * HD;   // the image's elements
#endif
      Vec<CPL> acc = vzero<CPL>();
      int pt = 0;
      for (int l = 0; l < L; ++l) {
        const int dyl = (PACKED ? tab->Wv[l] : tab->W[l]) * HD;   // row pitch of the level inside the image
        const int np = (PT > 0) ? PT : P;
#pragma unroll
        for (int p = 0; p < np; ++p, ++pt) {
          int oc;
          float4 cw;
          if constexpr (REC16) {
            const int4 r = s_rec[pt];
            oc = r.x;
            const float lw = __int_as_float(r.y), wy0 = __int_as_float(r.z), wy1 = __int_as_float(r.w);
            const float hw = 1.0f - lw;
            cw = make_float4(wy0 * hw, wy0 * lw, wy1 * hw, wy1 * lw);
          } else {
            oc = s_oc[pt];
            cw = s_cw[pt];
          }
          // A corner whose validity bit is clear is neither loaded nor added (its offset may lie outside the map).
          // Loads first, then the FMAs: both compile to predicated instructions (R2P + @P LDG.E.128 / @P FFMA), no
          // branches, and the loads of the next point are scheduled under the FMAs of this one.
          const int o00 = oc & ~15;
#ifdef MSDA_DEBUG_BOUNDS
          if (oc & 1) MSDA_CHECK_OFFSET(o00, lim, "fwd k0");
          if (oc & 2) MSDA_CHECK_OFFSET(o00 + HD, lim, "fwd k1");
          if (oc & 4) MSDA_CHECK_OFFSET(o00 + dyl, lim, "fwd k2");
          if (oc & 8) MSDA_CHECK_OFFSET(o00 + dyl + HD, lim, "fwd k3");
#endif
          if constexpr (sizeof(VT) == 4) {
            Raw<CPL, VT> v0, v1, v2, v3;
            if (oc & 1) v0 = ldraw<CPL>(vimg + o00);
            if (oc & 2) v1 = ldraw<CPL>(vimg + (o00 + HD));
            if (oc & 4) v2 = ldraw<CPL>(vimg + (o00 + dyl));
            if (oc & 8) v3 = ldraw<CPL>(vimg + (o00 + dyl + HD));
            if (oc & 1) fmav(acc, cw.x, unpack(v0));
            if (oc & 2) fmav(acc, cw.y, unpack(v1));
            if (oc & 4) fmav(acc, cw.z, unpack(v2));
            if (oc & 8) fmav(acc, cw.w, unpack(v3));
          } else {
            // bf16: unpack + FMA of 8 channels is too long a body for the compiler to predicate (it branches, and the
            // rows of a warp diverge), so the packed bits start as zeros and only the load is predicated
            Raw<CPL, VT> v0 = Raw<CPL, VT>(), v1 = Raw<CPL, VT>(), v2 = Raw<CPL, VT>(), v3 = Raw<CPL, VT>();
            if (oc & 1) v0 = ldraw<CPL>(vimg + o00);
            if (oc & 2) v1 = ldraw<CPL>(vimg + (o00 + HD));
            if (oc & 4) v2 = ldraw<CPL>(vimg + (o00 + dyl));
            if (oc & 8) v3 = ldraw<CPL>(vimg + (o00 + dyl + HD));
            fmav(acc, cw.x, unpack(v0));
            fmav(acc, cw.y, unpack(v1));
            fmav(acc, cw.z, unpack(v2));
            fmav(acc, cw.w, unpack(v3));
          }
        }
      }
      stv<CPL>(out + cur.row * D + sub * CPL, acc);
    }
    if constexpr (PACKED) break;   // single pass
    walk.next();    // single-pass orders end here; TILE2D only continues for a pathological pyramid
    if (walk.done()) break;
    __syncwarp();
    cur = walk.get(tab, L, H, Q);
  }
}

// =============================================================================================
// Backward
// =============================================================================================
// records per row: float4 cw[NP] (as forward) | int4 fin[NP] = { oc, lw, lh, aw } (floats bit-cast)
//
// grad_value accumulation: float (vector red, fast, order-dependent rounding) or, for
// MSDA_FLAG_DETERMINISTIC, 64-bit fixed point (integer red: the sum is order independent).
// ACC = NoScatter compiles the grad_value scatter out (the sorted deterministic path computes grad_value
// elsewhere, msda_det.cuh, and only needs this kernel's grad_sampling_loc / grad_attn_weight).
struct NoScatter {
  char unused;
};
// ACC = EmitEntries: no scatter either, but every in-range point files a 16-byte entry {row, lw, lh, attention weight}
// under its bilinear cell for the sorted deterministic path (msda_det.cuh) -- this replaces that path's separate fill
// pass (which re-read every location / weight and redid the coordinate arithmetic) with one cursor atomic and one
// 16-byte store per point issued from the lane that has just built the point's record.
struct EmitEntries {
  char unused[3];
};
struct EmitArgs {
  int* cursor;            // [bins] zero-initialised fill counters
  const int* bin_start;   // [bins + 1] exclusive scan of the per-bin counts
  int4* entries;          // [points in range]
  // [2][warps of the grid], or null: every warp leaves max |grad_out| and max |attention weight| of its rows here (float
  // bit patterns, +Inf = "not finite", msda_amax_kernel's rule); the host reduces the two short arrays instead of
  // sweeping grad_out and the weights a second time for the fixed-point scale.  (One atomicMax per warp on two shared
  // words was measured first: the two hot L2 lines cost +0.3 / +0.5 ms at cfg 2 / cfg 5.)
  float* warp_amax;
};

// running max |x| with msda_amax_kernel's rule: NaN, Inf or beyond float range turns the maximum into +Inf
__device__ __forceinline__ float amax_step(float m, float x) {
  const float a = fabsf(x);
  return (a <= 3.0e38f) ? fmaxf(m, a) : __int_as_float(0x7f800000);
}

__device__ __forceinline__ void scatter4(float* g, const float c, const float4 go, float /*scale*/) {
  // red (no return value) on purpose: atomicAdd(float4*) may compile to ATOM.E.ADD.F32x4 with a dead
  // destination, which pays the return trip; inline PTX pins SASS REDG.E.ADD.F32x4.
  asm volatile("red.global.add.v4.f32 [%0], {%1, %2, %3, %4};" ::"l"(g), "f"(c * go.x), "f"(c * go.y), "f"(c * go.z),
               "f"(c * go.w)
               : "memory");
}
// `go` is in SCATTER layout: component block i (4 floats) belongs to channels i*HALF + 4*sub .. +3, and `g`
// already points at channel 4*sub, so the LANES lanes of a row write 16*LANES CONTIGUOUS bytes per instruction
// (with 8 channels per lane the gather layout would put two separate 16-byte reds into every 32-byte
// sector and double the L2 reduction work: measured 1.75 -> 2.9 ms).
template <int N, int HALF>
__device__ __forceinline__ void scatterv(float* g, const float c, const Vec<N>& go) {
#pragma unroll
  for (int i = 0; i < N; i += 4)
    asm volatile("red.global.add.v4.f32 [%0], {%1, %2, %3, %4};" ::"l"(g + (i / 4) * HALF), "f"(c * go.v[i]),
                 "f"(c * go.v[i + 1]), "f"(c * go.v[i + 2]), "f"(c * go.v[i + 3])
                 : "memory");
}

// grad_out row in scatter layout (see scatterv): for 4 channels per lane it is the gather layout itself
template <int N, int D, typename VT>
__device__ __forceinline__ Vec<N> load_scatter_layout(const VT* row, int sub, const Vec<N>& gather_layout) {
  if constexpr (N == 4) {
    return gather_layout;
  } else {
    const Vec<4> a = ldv<4>(row + sub * 4), b = ldv<4>(row + D / 2 + sub * 4);
    Vec<8> r;
#pragma unroll
    for (int i = 0; i < 4; ++i) {
      r.v[i] = a.v[i];
      r.v[4 + i] = b.v[i];
    }
    return r;
  }
}

// Deterministic flavour: `go` holds the TRANSPOSED channels (component i = channel i*LANES + sub, see
// transpose_channels), and g already points at channel `sub`, so the LANES lanes of a row write 8*LANES
// contiguous bytes per instruction: every 32-byte sector receives one full-width 64-bit red per lane
// instead of four partial ones (there is no vector form of the 64-bit integer red).
template <int LANES>
__device__ __forceinline__ void scatter4_det(unsigned long long* g, const float c, const float4 go, float scale) {
  // the weight is scaled by the power of two first (exact), then its product with grad_out is rounded to an integer:
  // det_weight / det_contrib (msda_coords.cuh) are shared with msda_det.cuh so that all three paths give the same bits
  const det_factor cs = (det_factor)det_weight(c, scale);
  atomicAdd(g + 0 * LANES, (unsigned long long)det_contrib(cs, (det_factor)go.x));
  atomicAdd(g + 1 * LANES, (unsigned long long)det_contrib(cs, (det_factor)go.y));
  atomicAdd(g + 2 * LANES, (unsigned long long)det_contrib(cs, (det_factor)go.z));
  atomicAdd(g + 3 * LANES, (unsigned long long)det_contrib(cs, (det_factor)go.w));
}

// lane `sub` owns channels 4*sub..4*sub+3 in v; returns channels {sub, LANES+sub, 2*LANES+sub, 3*LANES+sub}
template <int LANES>
__device__ __forceinline__ float4 transpose_channels(const float4 v, int sub) {
  const int comp = sub & 3;
  // channel i*LANES + sub lives in lane (i*LANES + sub)/4, component sub%4; every lane must publish the
  // component its READERS want, which is the reader's sub%4 -- so do it in 4 rounds, one per component
  float4 r;
  float got[4];
#pragma unroll
  for (int i = 0; i < 4; ++i) {
    const int src = (i * LANES + sub) >> 2;
    const float c0 = __shfl_sync(0xffffffffu, v.x, src, LANES);
    const float c1 = __shfl_sync(0xffffffffu, v.y, src, LANES);
    const float c2 = __shfl_sync(0xffffffffu, v.z, src, LANES);
    const float c3 = __shfl_sync(0xffffffffu, v.w, src, LANES);
    got[i] = comp == 0 ? c0 : (comp == 1 ? c1 : (comp == 2 ? c2 : c3));
  }
  r.x = got[0]; r.y = got[1]; r.z = got[2]; r.w = got[3];
  return r;
}

template <int LANES>
__device__ __forceinline__ void transpose_reduce_4x4(float (&d)[16], int sub) {
  // d[j*4+k]: partial dot k of point j.  After this, lane `sub` holds in d[0..3] the four dots of
  // point sub / (LANES/4), summed over all LANES lanes of the row.
  {
    const bool up = (sub & (LANES / 2)) != 0;
#pragma unroll
    for (int i = 0; i < 8; ++i) {
      const float send = up ? d[i] : d[i + 8];
      const float keep = up ? d[i + 8] : d[i];
      d[i] = keep + __shfl_xor_sync(0xffffffffu, send, LANES / 2);
    }
  }
  {
    const bool up = (sub & (LANES / 4)) != 0;
#pragma unroll
    for (int i = 0; i < 4; ++i) {
      const float send = up ? d[i] : d[i + 4];
      const float keep = up ? d[i + 4] : d[i];
      d[i] = keep + __shfl_xor_sync(0xffffffffu, send, LANES / 4);
    }
  }
#pragma unroll
  for (int m = LANES / 8; m > 0; m >>= 1) {
#pragma unroll
    for (int i = 0; i < 4; ++i) d[i] += __shfl_xor_sync(0xffffffffu, d[i], m);
  }
}

#ifndef MSDA_BWD_MINB
#define MSDA_BWD_MINB 4
#endif
template <int D, typename VT, int PT, int THREADS, int ORDER, typename ACC, int PRE, int CPL, typename AT = float>
__global__ void __launch_bounds__(THREADS, MSDA_BWD_MINB * (256 / THREADS))
msda_bwd_fast_kernel(const VT* __restrict__ grad_out, const VT* __restrict__ value,
                     const int64_t* __restrict__ shapes, const int64_t* __restrict__ lsi,
                     const AT* __restrict__ loc, const AT* __restrict__ w,
                     ACC* __restrict__ grad_value, AT* __restrict__ grad_loc,
                     AT* __restrict__ grad_w, const DetScale* __restrict__ det, const FusedArgs fused,
                     const EmitArgs emit, int B, int S, int H, int L, int Q, int P, int64_t rows) {
  // FUSED: loc = raw offsets, w = logits in; grad_loc = grad of the offsets, grad_w = grad of the logits out
  static_assert(THREADS <= 256, "single-pass CTAs");
  constexpr bool EMIT = sizeof(ACC) == sizeof(EmitEntries);
  // LINEAR only: EmitArgs::warp_amax has one slot pair per warp of the LINEAR grid (bwd_fast_emit / bwd_dcn_emit)
  static_assert(!EMIT || (ORDER == 0 && (PRE == kPrePlain || PRE == kPreDcn)),
                "entries are emitted by the plain and DCNv3 LINEAR backward");
  // the fused DCNv3 module path has no deterministic or no-scatter form (its deterministic backward is composed
  // around the kPreDcn kernels, ir_ads_b200/dcnv3.py)
  static_assert(PRE != kPreDcnSoftmax || std::is_same_v<ACC, float>, "the fused DCNv3 backward uses float reds");
  static_assert(aux_ok<VT, AT, PRE, ORDER, 2>() && (std::is_same_v<AT, float> || std::is_same_v<ACC, float>),
                "16-bit offsets / logits: fused modes, value's dtype, float reds, STRIP backward");
  constexpr int DL = D * 4 / CPL;
  using G = Geom<DL, THREADS>;
  constexpr int LANES = G::LANES;
  constexpr bool SOFTMAX = pre_softmax(PRE);    // `w` holds logits: softmax and its chain rule (grad_w = logits' grad)
  constexpr bool FUSED = pre_fused(PRE);        // MSDA chain only: location affine, reference points, padding mask
  constexpr bool PACKED = (PRE == kPrePacked);  // packed batch: `lsi` = per-image metadata, one image per CTA
  static_assert(!PACKED || (ORDER == 2 && std::is_same_v<ACC, float>), "the packed backward is STRIP with float reds");
  constexpr bool DCN = pre_dcn(PRE);
  extern __shared__ __align__(16) unsigned char smem_raw[];
  LevelTab* tab = reinterpret_cast<LevelTab*>(smem_raw);
  float* recs = reinterpret_cast<float*>(smem_raw + sizeof(LevelTab));
  const int NP = L * P;
  const int row_words = bwd_row_words(NP);

  const int sub = (threadIdx.x & 31) % LANES;
  const int rin = threadIdx.x / LANES;
  const int HD = H * D;
  float* my = recs + (size_t)rin * row_words;
  float4* s_cw = reinterpret_cast<float4*>(my);
  int4* s_fin = reinterpret_cast<int4*>(my + 4 * NP);
  const float4 zero = make_float4(0.f, 0.f, 0.f, 0.f);
  const float gscale = det ? det->scale : 1.0f;

  // Single-pass orders know their row without the level table: the row's grad_out and its first locations /
  // weights are requested before the table's load + barrier (see the forward kernel).
  constexpr bool EARLY = (ORDER == 0 || ORDER == 2) && !DCN;
  constexpr int kEarly = 2;
  float2 early_xy[kEarly];
  float early_w[kEarly];
  float early_sum = 1.0f;                                // SOFTMAX: softmax denominator of the row
  // A warp stays converged for the full-mask shuffles below: rows that do not exist (edge tiles,
  // the tail of the last CTA) get all-zero weights, so they scatter nothing and never write.
  RowWalk<DL, THREADS, ORDER> walk;
  RowRef cur;
  Vec<CPL> go = vzero<CPL>();
  const int64_t* pimg = nullptr;                         // PACKED: the CTA's image metadata row
  if constexpr (EARLY) {
    if constexpr (PACKED) {
      const PackedRow p = packed_row<G::RPC, ORDER>(lsi, L, H, Q, rin);
      if (p.surplus) return;                             // uniform over the CTA
      cur = p.r;
      pimg = p.img;
    } else {
      walk = RowWalk<DL, THREADS, ORDER>(tab, B, H, rows);
      if (walk.done()) return;                             // uniform over the CTA
      cur = walk.get(tab, L, H, Q);
    }
    if (cur.live) go = ldv<CPL>(grad_out + cur.row * D + sub * CPL);
#pragma unroll
    for (int i = 0; i < kEarly; ++i) {
      const int pt = sub + i * LANES;
      const bool on = cur.live && pt < NP;
      early_xy[i] = on ? ld_xy(loc + cur.row * (int64_t)NP * 2, pt) : make_float2(0.f, 0.f);
      early_w[i] = (on && !SOFTMAX) ? ld_aux(w + cur.row * (int64_t)NP + pt) : 0.0f;
    }
    if constexpr (SOFTMAX)
      early_sum = row_softmax<LANES, 4>(w + cur.row * (int64_t)NP, reinterpret_cast<float*>(s_fin) + 3, NP, sub);
    if constexpr (PACKED) load_levels_packed(tab, shapes, pimg, L);
    else load_levels_plain<EMIT>(tab, shapes, lsi, L);
  } else {
    if constexpr (DCN) set_single_level<G::TW, G::TH, EMIT>(tab, fused.height_in, fused.width_in);
    else if constexpr (ORDER == 0 || ORDER == 2) load_levels_plain(tab, shapes, lsi, L);
    else load_levels<G::TW, G::TH>(tab, shapes, lsi, L);
    walk = RowWalk<DL, THREADS, ORDER>(tab, B, H, rows);
    if (walk.done()) return;
    cur = walk.get(tab, L, H, Q);
  }
  // file a point's entry under the bin of its cell (cells of the extended grid, det_bin_kernel's index exactly)
  auto emit_entry = [&](const Cell<float> c, int l, float aw) {
    const int bin = (cur.b * H + cur.h) * tab->cells_per_bh + tab->cell_begin[l] + (c.y0 + 1) * (tab->W[l] + 1) +
                    (c.x0 + 1);
    const int pos = __ldg(emit.bin_start + bin) + atomicAdd(emit.cursor + bin, 1);
#ifdef MSDA_DEBUG_BOUNDS   // the count pass must have counted this point in this very bin
    MSDA_CHECK_OFFSET(pos - __ldg(emit.bin_start + bin), __ldg(emit.bin_start + bin + 1) - __ldg(emit.bin_start + bin),
                      "emit entry");
#endif
    emit.entries[pos] = make_int4((int)cur.row, __float_as_int(c.lw), __float_as_int(c.lh), __float_as_int(aw));
  };
  while (true) {
    if constexpr (!EARLY) go = cur.live ? ldv<CPL>(grad_out + cur.row * D + sub * CPL) : vzero<CPL>();
    const float* rp = FUSED ? fused.ref + (cur.row / H) * (int64_t)L * fused.ref_dim : nullptr;
    {
      const AT* lp = loc + cur.row * (int64_t)NP * 2;
      const AT* wp = w + cur.row * (int64_t)NP;
      float sm_sum = early_sum;
      if constexpr (SOFTMAX && !EARLY) sm_sum = row_softmax<LANES, 4>(wp, reinterpret_cast<float*>(s_fin) + 3, NP, sub);
      // one record from a point's raw location / weight (FUSED: raw offset; SOFTMAX: the weight comes from the
      // softmax); rows that do not exist get all-zero records
      auto build = [&](int pt, float2 xy, float aw) {
        float4 cw = zero;
        int4 fin = make_int4(0, 0, 0, 0);      // no validity bits: nothing is loaded, scattered or written
        if (cur.live) {
          const int l = level_of<PT>(pt, P);
          if constexpr (SOFTMAX) aw = __fdiv_rn(__int_as_float(s_fin[pt].w), sm_sum);
          if constexpr (FUSED)
            xy = fused_location(xy, rp + l * fused.ref_dim, fused.ref_dim, tab->H[l], tab->W[l], fused.num_P);
          PointRec r;
          if constexpr (DCN) {
            const float2 px = dcn_location(xy, pt, (int)((cur.row / H) % Q), fused);
            const Cell<float> c = locate_pixel(px.x, px.y, tab->H[0], tab->W[0]);
            r = record_from_cell(c, aw, tab->W[0], 0, H, cur.h, D);
            if constexpr (EMIT) {
              if (c.valid != 0u) emit_entry(c, 0, aw);
            }
          } else if constexpr (EMIT) {
            const Cell<float> c = locate<float>(xy.x, xy.y, tab->H[l], tab->W[l]);
            r = record_from_cell(c, aw, tab->W[l], tab->start[l], H, cur.h, D);
            if (c.valid != 0u) emit_entry(c, l, aw);
          } else if constexpr (PACKED) {
            r = record_from_cell(clip_to_rect(locate<float>(xy.x, xy.y, tab->H[l], tab->W[l]), tab->Hv[l], tab->Wv[l]),
                                 aw, tab->Wv[l], tab->start[l], H, cur.h, D);
          } else {
            r = make_record(xy.x, xy.y, aw, tab->H[l], tab->W[l], tab->start[l], H, cur.h, D);
          }
          if constexpr (FUSED && !PACKED) {
            if (fused.value_mask) apply_value_mask(r, fused.value_mask + (int64_t)cur.b * S, tab->W[l], S);
          }
          cw = r.cw;
          fin = make_int4(r.oc, __float_as_int(r.lw), __float_as_int(r.lh), __float_as_int(aw));
        }
        s_cw[pt] = cw;
        s_fin[pt] = fin;
      };
      int pt = sub;
      if constexpr (EARLY) {   // the loads of these iterations were issued before the level table's barrier
#pragma unroll
        for (int i = 0; i < kEarly; ++i, pt += LANES)
          if (pt < NP) build(pt, early_xy[i], early_w[i]);
      }
      for (; pt < NP; pt += LANES) {
        float2 xy = make_float2(0.f, 0.f);
        float aw = 0.0f;
        if (cur.live) {
          xy = ld_xy(lp, pt);
          if constexpr (!SOFTMAX) aw = ld_aux(wp + pt);
        }
        build(pt, xy, aw);
      }
    }
    __syncwarp();

    constexpr bool DET = sizeof(ACC) == 8;
    constexpr bool SCATTER = sizeof(ACC) != sizeof(NoScatter) && !EMIT;
    static_assert(!(sizeof(ACC) == 8 && CPL != 4), "the fixed-point red path transposes 4 channels per lane");

    const int64_t img = (PACKED ? __ldg(pimg) * HD : (int64_t)cur.b * S * HD) + sub * CPL;
#ifdef MSDA_DEBUG_BOUNDS
    const int lim = PACKED ? (int)__ldg(pimg + 1) * HD : S * HD;   // the image's elements
#endif
    const VT* vimg = value + img;
    ACC* gimg = grad_value + (DET ? img - sub * 3 : img);   // DET: lane offset is `sub`, not 4*sub
    asm volatile("" : "+l"(vimg), "+l"(gimg));
    float4 go_s = make_float4(0.f, 0.f, 0.f, 0.f);           // DET only: channels transposed across the lanes
    if constexpr (DET) go_s = transpose_channels<LANES>(make_float4(go.v[0], go.v[1], go.v[2], go.v[3]), sub);
    // float scatter: grad_out in scatter layout, base pointer at channel 4*sub (== the gather base for CPL 4)
    Vec<CPL> go_sc = go;
    float* gsc = nullptr;
    if constexpr (SCATTER && !DET) {
      go_sc = load_scatter_layout<CPL, D>(grad_out + cur.row * D, sub, go);
      gsc = reinterpret_cast<float*>(grad_value) + (PACKED ? __ldg(pimg) * HD : (int64_t)cur.b * S * HD) + sub * 4;
      asm volatile("" : "+l"(gsc));
    }   // one 64-bit register each: address = base + off*size (IMAD.WIDE)
    AT* glp = grad_loc + cur.row * (int64_t)NP * 2;
    AT* gwp = grad_w + cur.row * (int64_t)NP;

    float sm_dot = 0.0f;   // SOFTMAX: sum_j grad_aw_j * aw_j of the row (softmax backward)
    for (int c0 = 0; c0 < NP; c0 += 4) {
      float d[16];
#pragma unroll
      for (int j = 0; j < 4; ++j) {
        const int pt = c0 + j;
        if (pt < NP) {
          const int oc = s_fin[pt].x;
          const float4 cw = s_cw[pt];
          const int l = level_of<PT>(pt, P);
          const int o00 = oc & ~15;
          const int o01 = o00 + HD;
          const int o10 = o00 + (PACKED ? tab->Wv[l] : tab->W[l]) * HD, o11 = o10 + HD;
          // a corner whose validity bit is clear is not loaded (its offset may lie outside the map); its dot stays 0
          float d0 = 0.0f, d1 = 0.0f, d2 = 0.0f, d3 = 0.0f;
#ifdef MSDA_DEBUG_BOUNDS
          if ((oc & 1) || cw.x != 0.0f) MSDA_CHECK_OFFSET(o00, lim, "bwd k0");
          if ((oc & 2) || cw.y != 0.0f) MSDA_CHECK_OFFSET(o01, lim, "bwd k1");
          if ((oc & 4) || cw.z != 0.0f) MSDA_CHECK_OFFSET(o10, lim, "bwd k2");
          if ((oc & 8) || cw.w != 0.0f) MSDA_CHECK_OFFSET(o11, lim, "bwd k3");
#endif
#ifdef MSDA_EXP_NO_GATHER   // experiment builds only (tools/ablate.sh): what does the scatter cost alone?
          d0 = d1 = d2 = d3 = dotv(go, go);
#else
          if (oc & 1) d0 = dotv(go, ldv<CPL>(vimg + o00));
          if (oc & 2) d1 = dotv(go, ldv<CPL>(vimg + o01));
          if (oc & 4) d2 = dotv(go, ldv<CPL>(vimg + o10));
          if (oc & 8) d3 = dotv(go, ldv<CPL>(vimg + o11));
#endif
          d[4 * j + 0] = d0;
          d[4 * j + 1] = d1;
          d[4 * j + 2] = d2;
          d[4 * j + 3] = d3;
#ifdef MSDA_EXP_NO_RED      // experiment builds only: what does the gather cost alone?
          if (cw.x == 12345.678f) scatterv<CPL, D / 2>(reinterpret_cast<float*>(gimg) + o00, cw.x, go);
#else
          if constexpr (!SCATTER) {
            (void)gscale;
          } else if constexpr (DET) {
            if (cw.x != 0.0f) scatter4_det<LANES>(gimg + o00, cw.x, go_s, gscale);
            if (cw.y != 0.0f) scatter4_det<LANES>(gimg + o01, cw.y, go_s, gscale);
            if (cw.z != 0.0f) scatter4_det<LANES>(gimg + o10, cw.z, go_s, gscale);
            if (cw.w != 0.0f) scatter4_det<LANES>(gimg + o11, cw.w, go_s, gscale);
          } else {
            if (cw.x != 0.0f) scatterv<CPL, D / 2>(gsc + o00, cw.x, go_sc);
            if (cw.y != 0.0f) scatterv<CPL, D / 2>(gsc + o01, cw.y, go_sc);
            if (cw.z != 0.0f) scatterv<CPL, D / 2>(gsc + o10, cw.z, go_sc);
            if (cw.w != 0.0f) scatterv<CPL, D / 2>(gsc + o11, cw.w, go_sc);
          }
#endif
        } else {
          d[4 * j + 0] = 0.f; d[4 * j + 1] = 0.f; d[4 * j + 2] = 0.f; d[4 * j + 3] = 0.f;
        }
      }
      transpose_reduce_4x4<LANES>(d, sub);
      const int mine = c0 + sub / (LANES / 4);
      if (cur.live && (sub % (LANES / 4)) == 0 && mine < NP) {
        const int4 r = s_fin[mine];
        const float lw = __int_as_float(r.y), lh = __int_as_float(r.z), aw = __int_as_float(r.w);
        float g_aw = 0.0f, g_x = 0.0f, g_y = 0.0f;      // a gated point's grads stay 0 (cuh:369)
        if (r.x & 15) {
          // d[k] = <grad_out, v_k>; padded (and masked) corners were not loaded and contribute 0 (cuh:119-158)
          const float d0 = d[0], d1 = d[1], d2 = d[2], d3 = d[3];
          const float hh = 1.0f - lh, hw = 1.0f - lw;
          const int l = level_of<PT>(mine, P);
          g_aw = hh * hw * d0 + hh * lw * d1 + lh * hw * d2 + lh * lw * d3;
          g_x = (hh * (d1 - d0) + lh * (d3 - d2)) * aw;    // d / d(pixel coordinate)
          g_y = (hw * (d2 - d0) + lw * (d3 - d1)) * aw;
          if constexpr (DCN) {                                // offsets are in pixels x offset_scale (dcnv3 cuh:150-157)
            g_x *= fused.offset_scale;
            g_y *= fused.offset_scale;
          } else {                                            // locations are normalised by the level size
            g_x *= (float)tab->W[l];
            g_y *= (float)tab->H[l];
          }
        }
        if constexpr (FUSED) {
          // chain rule through loc = ref + off / (W,H)   or   ref_xy + off / P * ref_wh * 0.5
          const int l = level_of<PT>(mine, P);
          float2 g_off;
          if (fused.ref_dim == 2) {
            g_off = make_float2(__fdiv_rn(g_x, (float)tab->W[l]), __fdiv_rn(g_y, (float)tab->H[l]));
          } else {
            const float* r4 = rp + l * 4;
            g_off = make_float2(g_x * 0.5f * __ldg(r4 + 2) * fused.inv_P, g_y * 0.5f * __ldg(r4 + 3) * fused.inv_P);
          }
          // this point's record is finished: park the three gradients in it ({g_x, g_aw, g_y, aw}); the row writes
          // them out in full lines below
          s_fin[mine] = make_int4(__float_as_int(g_off.x), __float_as_int(g_aw), __float_as_int(g_off.y), r.w);
          sm_dot = fmaf(g_aw, aw, sm_dot);
        } else {
          s_fin[mine] = make_int4(__float_as_int(g_x), __float_as_int(g_aw), __float_as_int(g_y), r.w);
          if constexpr (SOFTMAX) sm_dot = fmaf(g_aw, aw, sm_dot);
        }
      }
    }
    if constexpr (SOFTMAX) {
      // softmax backward: grad_logit_i = aw_i * (grad_aw_i - sum_j grad_aw_j aw_j)
#pragma unroll
      for (int k = LANES / 2; k > 0; k >>= 1) sm_dot += __shfl_xor_sync(0xffffffffu, sm_dot, k);
    }
    __syncwarp();
    // Write-out.  One lane per point storing 4 + 8 bytes as it finishes would send every 16-byte piece of grad_attn_weight
    // and every 32-byte piece of grad_sampling_loc through the SM's crossbar port as a request of its own (header + one
    // sector each: 16 port cycles per row at L*P = 16); the port is what binds this kernel.  Parked in the records and
    // written by the row's lanes two points at a time, a row leaves as one 128-byte and one 64-byte request (16-bit AT:
    // the same full lines at half the bytes).
    if (cur.live) {
      auto gw_of = [&](const int4 r) {
        const float g_aw = __int_as_float(r.y);
        return SOFTMAX ? __int_as_float(r.w) * (g_aw - sm_dot) : g_aw;
      };
      if ((NP & 1) == 0) {      // both row bases are then 16- / 8-byte aligned
        for (int pt = 2 * sub; pt < NP; pt += 2 * LANES) {
          const int4 a = s_fin[pt], b = s_fin[pt + 1];
          st_aux4(glp + 2 * pt,
                  make_float4(__int_as_float(a.x), __int_as_float(a.z), __int_as_float(b.x), __int_as_float(b.z)));
          st_aux2(gwp + pt, gw_of(a), gw_of(b));
        }
      } else {
        for (int pt = sub; pt < NP; pt += LANES) {
          const int4 a = s_fin[pt];
          st_aux2(glp + 2 * pt, __int_as_float(a.x), __int_as_float(a.z));
          st_aux1(gwp + pt, gw_of(a));
        }
      }
    }
    if constexpr (EMIT) {
      if (emit.warp_amax) {   // uniform over the grid; EMIT is a single-pass order: one slot pair per warp
        float m_go = 0.0f, m_w = 0.0f;
        if (cur.live) {
#pragma unroll
          for (int i = 0; i < CPL; ++i) m_go = amax_step(m_go, go.v[i]);
          for (int pt = sub; pt < NP; pt += LANES) m_w = amax_step(m_w, __int_as_float(s_fin[pt].w));   // .w is still aw
        }
#pragma unroll
        for (int k = 16; k > 0; k >>= 1) {
          m_go = fmaxf(m_go, __shfl_xor_sync(0xffffffffu, m_go, k));
          m_w = fmaxf(m_w, __shfl_xor_sync(0xffffffffu, m_w, k));
        }
        if ((threadIdx.x & 31) == 0) {
          const int64_t n_warps = (int64_t)gridDim.x * (THREADS / 32);
          const int64_t wid = (int64_t)blockIdx.x * (THREADS / 32) + (threadIdx.x >> 5);
          emit.warp_amax[wid] = m_go;
          emit.warp_amax[n_warps + wid] = m_w;
        }
      }
    }
    if constexpr (PACKED) break;   // single pass
    walk.next();
    if (walk.done()) break;
    __syncwarp();
    cur = walk.get(tab, L, H, Q);
  }
}

}  // namespace msda
