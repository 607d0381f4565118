// msda_det.cuh -- deterministic grad_value by sorted segment reduction (MSDA_FLAG_DETERMINISTIC, fast shapes).
//
// The atomic backward scatters 4 corner rows per sampling point into grad_value; float reds make the
// rounding depend on arrival order.  This path removes the scatter altogether:
//   1. det_bin_kernel<false>  every point finds its bilinear cell (same coordinate code as the other
//                             kernels) and counts itself in that cell's bin
//   2. scan (3 small kernels) bin counts -> bin start offsets
//   3. det_bin_kernel<true>   every point writes a 16-byte entry {row, lw, lh, attention weight} into its bin
//   4a. det_gather_kernel     (sparse problems: fewer than kDetDenseRatio points per pixel and head, e.g. decoder
//                             cross-attention) one lane group per (image, pixel, head): walks the (up to) four
//                             bins whose cells have this pixel as a corner, gathers grad_out rows and accumulates
//                             in 64-bit fixed point IN REGISTERS, writes the pixel's D channels once.
//   4b. det_cell_reduce_kernel (dense problems, e.g. encoder self-attention) one lane group per slice of 64
//                             consecutive entries: every entry is read once, the four corner sums of a cell are
//                             kept in registers and handed to a fixed-point accumulation buffer with 64-bit
//                             integer reds when the cell changes; msda_det_finalize_kernel converts.
// Bins are filled in arbitrary order (an atomic cursor), but integer accumulation is order independent,
// so the result is bit-reproducible -- and bit-identical to the fixed-point reds of the generic
// deterministic path (same products, same scale).  No atomics touch grad_value, no zero-fill is needed.
// grad_sampling_loc / grad_attn_weight come from the regular backward kernel with the scatter compiled
// out (ACC = NoScatter).
//
// Cells live on the extended grid (H_l+1) x (W_l+1) of every level (the low corner of a cell can be -1),
// bins are indexed [image][head][level cells].
#pragma once
#include <cuda_bf16.h>
#include <cuda_runtime.h>
#include <stdint.h>

#include "msda_coords.cuh"
#include "msda_fast.cuh"

namespace msda {

struct CellTab {
  int H[kFastMaxLevels];
  int W[kFastMaxLevels];
  int start[kFastMaxLevels];
  int cell_begin[kFastMaxLevels];   // first bin of the level inside one (image, head) block
  int cells_per_bh;
  int pad[3];
};

__device__ __forceinline__ void load_cell_tab(CellTab* t, const int64_t* shapes, const int64_t* lsi, int L) {
  if (threadIdx.x == 0) {
    int acc = 0;
    for (int l = 0; l < L; ++l) {
      t->H[l] = (int)shapes[2 * l];
      t->W[l] = (int)shapes[2 * l + 1];
      t->start[l] = (int)lsi[l];
      t->cell_begin[l] = acc;
      acc += level_cells(t->H[l], t->W[l]);
    }
    t->cells_per_bh = acc;
  }
  __syncthreads();
}

// dense problems (points per pixel and head >= this) take the cell reduce, sparse ones the per-pixel gather:
// cfg 3 (1.4 points per pixel-head) 0.60 vs 0.81 ms, cfg 2 (16) 3.31 vs 3.02 ms, cfg 5 (39) 8.26 vs 5.65 ms
constexpr int kDetDenseRatio = 4;

// upper bound of bins per (image, head) that needs only S and L: (H+1)(W+1) <= 2HW + 2 for H, W >= 1, and an empty
// level owns no bins (level_cells)
__host__ __device__ constexpr int64_t det_cells_bound(int64_t S, int64_t L) { return 2 * S + 2 * L; }

// Division of a 31-bit unsigned by a run-time constant as multiply-high + shift (Granlund-Montgomery, the round-up
// form: m = ceil(2^(31+s) / d), s = ceil(log2 d), exact for n < 2^31).  The count pass below decomposes every
// point index with four divisions; as `n / d` each costs an I2F + MUFU.RCP + F2I sequence on the quarter-rate
// conversion pipe, and the pass is bound by its instruction issue.
struct FastDiv {
  unsigned m, s;   // d == 1: m == 0 (the quotient is n itself)
};
// host + device (msda_debug_fastdiv in include/msda.h lets the CPU tests check the constants against `/`)
__host__ __device__ __forceinline__ FastDiv fastdiv_make(unsigned d) {
  FastDiv f;
  if (d <= 1u) {
    f.m = 0u;
    f.s = 0u;
  } else {
#ifdef __CUDA_ARCH__
    const unsigned lg = 32u - (unsigned)__clz((int)(d - 1u));          // ceil(log2 d), d >= 2
#else
    const unsigned lg = 32u - (unsigned)__builtin_clz(d - 1u);
#endif
    f.m = (unsigned)(((1ull << (31u + lg)) + d - 1u) / d);
    f.s = lg - 1u;
  }
  return f;
}
__host__ __device__ __forceinline__ unsigned fastdiv(unsigned n, const FastDiv f) {
#ifdef __CUDA_ARCH__
  return f.m ? (__umulhi(n, f.m) >> f.s) : n;
#else
  return f.m ? ((unsigned)(((unsigned long long)n * f.m) >> 32) >> f.s) : n;
#endif
}

// FILL == false: count points per bin.  FILL == true: write entries (bins already scanned into `bin_start`).
// PRE == kPreDcn: DCNv3 (L == 1, P == K, H == groups, Q == H_out * W_out): `loc` holds the offsets [N, Ho, Wo, G*K*2]
// and `w` the mask; point pt = ((b*Q + q)*G + g)*K + k lands at dcn_location + locate_pixel -- the device functions
// the DCN records of the backward kernel use, so this pass and the entry-filing backward agree on every cell.
template <bool FILL, int PRE = kPrePlain>
__global__ void __launch_bounds__(256)
det_bin_kernel(const float* __restrict__ loc, const float* __restrict__ w, const int64_t* __restrict__ shapes,
               const int64_t* __restrict__ lsi, int H, int L, int Q, int P, int64_t n_points, int* __restrict__ counter,
               const int* __restrict__ bin_start, int4* __restrict__ entries, const FusedArgs dcn) {
  static_assert(PRE == kPrePlain || PRE == kPreDcn, "plain or DCNv3 points");
  __shared__ CellTab tab;
  __shared__ FastDiv div[4];   // by NP, P, H, Q
  const int NP = L * P;
  if (threadIdx.x < 4) div[threadIdx.x] = fastdiv_make((unsigned)(threadIdx.x == 0 ? NP : (threadIdx.x == 1 ? P : (threadIdx.x == 2 ? H : Q))));
  load_cell_tab(&tab, shapes, lsi, L);   // ends with a barrier
  const FastDiv dNP = div[0], dP = div[1], dH = div[2], dQ = div[3];
  for (int64_t pt = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; pt < n_points;
       pt += (int64_t)gridDim.x * blockDim.x) {
    // 32-bit index arithmetic: the sorted path is only taken when n_points < 2^31 (det_sorted_ok), and this kernel
    // was bound by its divisions (64-bit: issue slots 79 % busy at cfg 5; 32-bit `/`: 76 %)
    const unsigned p32 = (unsigned)pt;
    const unsigned row = fastdiv(p32, dNP);
    const int l = (int)fastdiv(p32 - row * (unsigned)NP, dP);
    const unsigned bq = fastdiv(row, dH);
    const int h = (int)(row - bq * (unsigned)H);
    const int64_t b = fastdiv(bq, dQ);
    const float2 xy = __ldg(reinterpret_cast<const float2*>(loc) + pt);
    Cell<float> c;
    if constexpr (PRE == kPreDcn) {   // NP == P == K: l == 0, k = p32 - row * K
      const float2 px = dcn_location(xy, (int)(p32 - row * (unsigned)NP), (int)(bq - (unsigned)b * (unsigned)Q), dcn);
      c = locate_pixel(px.x, px.y, tab.H[0], tab.W[0]);
    } else {
      c = locate<float>(xy.x, xy.y, tab.H[l], tab.W[l]);
    }
    if (c.valid == 0u) continue;
    const int64_t bin = (b * H + h) * (int64_t)tab.cells_per_bh + tab.cell_begin[l] + (c.y0 + 1) * (tab.W[l] + 1) + (c.x0 + 1);
    if (!FILL) {
      atomicAdd(counter + bin, 1);
    } else {
      const int pos = bin_start[bin] + atomicAdd(counter + bin, 1);
      entries[pos] = make_int4((int)row, __float_as_int(c.lw), __float_as_int(c.lh), __float_as_int(__ldg(w + pt)));
    }
  }
}

// DCNv3 has no spatial_shapes / level_start_index tensors, only H_in and W_in: one thread writes the one-level table
// {H_in, W_in}, {0} into a slot of the caller's workspace, and the count / gather / cell-reduce kernels read it like the
// plain operator's.  No host copy and no sync, so the call stays capturable in a CUDA graph.
__global__ void det_one_level_kernel(int64_t* __restrict__ table, int H, int W) {
  table[0] = H;
  table[1] = W;
  table[2] = 0;
}

// ---- exclusive scan of n ints, 2048 per block --------------------------------------------------------
constexpr int kScanPerBlock = 2048;

__global__ void __launch_bounds__(256) det_scan_block_kernel(const int* __restrict__ in, int* __restrict__ out,
                                                           int* __restrict__ block_sums, int64_t n) {
  __shared__ int warp_tot[8];
  const int64_t base = (int64_t)blockIdx.x * kScanPerBlock + threadIdx.x * 8;
  int v[8], sum = 0;
#pragma unroll
  for (int k = 0; k < 8; ++k) {
    v[k] = (base + k < n) ? in[base + k] : 0;
    sum += v[k];
  }
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  int inc = sum;
#pragma unroll
  for (int o = 1; o < 32; o <<= 1) {
    const int t = __shfl_up_sync(0xffffffffu, inc, o);
    if (lane >= o) inc += t;
  }
  if (lane == 31) warp_tot[warp] = inc;
  __syncthreads();
  int off = 0;
  for (int k = 0; k < warp; ++k) off += warp_tot[k];
  int run = off + inc - sum;   // exclusive prefix of this thread's first element inside the block
#pragma unroll
  for (int k = 0; k < 8; ++k) {
    if (base + k < n) out[base + k] = run;
    run += v[k];
  }
  if (threadIdx.x == 255) block_sums[blockIdx.x] = run;
}

__global__ void __launch_bounds__(1024) det_scan_sums_kernel(int* __restrict__ block_sums, int n_blocks) {
  __shared__ int part[1024];
  const int per = (n_blocks + 1023) / 1024;
  const int b0 = threadIdx.x * per;
  int sum = 0;
  for (int k = 0; k < per; ++k)
    if (b0 + k < n_blocks) sum += block_sums[b0 + k];
  part[threadIdx.x] = sum;
  __syncthreads();
  if (threadIdx.x == 0) {
    int run = 0;
    for (int k = 0; k < 1024; ++k) {
      const int t = part[k];
      part[k] = run;
      run += t;
    }
  }
  __syncthreads();
  int run = part[threadIdx.x];
  for (int k = 0; k < per; ++k)
    if (b0 + k < n_blocks) {
      const int t = block_sums[b0 + k];
      block_sums[b0 + k] = run;
      run += t;
    }
}

__global__ void __launch_bounds__(256) det_scan_add_kernel(int* __restrict__ out, const int* __restrict__ block_sums,
                                                         int64_t n) {
  const int64_t base = (int64_t)blockIdx.x * kScanPerBlock + threadIdx.x * 8;
  const int off = block_sums[blockIdx.x];
#pragma unroll
  for (int k = 0; k < 8; ++k)
    if (base + k < n) out[base + k] += off;
}

// ---- gather: one LANES-wide lane group per (image, pixel, head) -----------------------------------------
// Walks the pixel's four bins (it is corner k of cell (y-dy, x-dx)), gathers the grad_out row of every entry
// and accumulates in 64-bit fixed point in registers.  Pixels are taken from the coarsest level down: a
// coarse pixel owns hundreds of entries, a fine one a handful, and the long items must not start last.
// (Measured alternatives, all slower at cfg 2: one warp per pixel with interleaved entries, a flattened
// 4-deep software pipeline over the four bins, and a magic-number replacement of the 64-bit F2I -- the
// kernel is bound by its instruction count, ~45 per entry, not by the conversion or by load latency.)
template <int D, typename VT>
__global__ void __launch_bounds__(256)
det_gather_kernel(const VT* __restrict__ grad_out, const int4* __restrict__ entries, const int* __restrict__ bin_start,
                  const int64_t* __restrict__ shapes, const int64_t* __restrict__ lsi,
                  const DetScale* __restrict__ det, VT* __restrict__ grad_value, int B, int S, int H, int L) {
  constexpr int LANES = D / 4;
  constexpr int RPC = 256 / LANES;
  __shared__ CellTab tab;
  load_cell_tab(&tab, shapes, lsi, L);
  const int sub = (threadIdx.x & 31) % LANES;
  const int64_t item = (int64_t)blockIdx.x * RPC + threadIdx.x / LANES;   // (b, reversed s, h), h fastest
  if (item >= (int64_t)B * S * H) return;
  const int h = (int)(item % H);
  const int64_t bs = item / H;
  const int s = S - 1 - (int)(bs % S);
  const int64_t b = bs / S;
  int l = 0;
  for (int k = 1; k < L; ++k)
    if (s >= tab.start[k]) l = k;
  const int Wl = tab.W[l];
  const int local = s - tab.start[l];
  const int y = local / Wl, x = local - y * Wl;
  const float scale = det->scale;
  const int64_t bin0 = (b * H + h) * (int64_t)tab.cells_per_bh + tab.cell_begin[l];
  long long a0 = 0, a1 = 0, a2 = 0, a3 = 0;
  if (y < tab.H[l]) {   // guards a malformed pyramid (sum of level sizes < S)
#pragma unroll
    for (int k = 0; k < 4; ++k) {
      const int dy = k >> 1, dx = k & 1;   // this pixel is corner k (v1..v4 of cuh:56-80) of cell (y-dy, x-dx)
      const int64_t bin = bin0 + (y - dy + 1) * (Wl + 1) + (x - dx + 1);
      const int e0 = __ldg(bin_start + bin), e1 = __ldg(bin_start + bin + 1);
      for (int e = e0; e < e1; ++e) {
        const int4 ent = __ldg(entries + e);
        const float lw = __int_as_float(ent.y), lh = __int_as_float(ent.z), aw = __int_as_float(ent.w);
        const float hh = 1.0f - lh, hw = 1.0f - lw;
        const det_factor c =
            (det_factor)det_weight((k == 0 ? hh * hw : (k == 1 ? hh * lw : (k == 2 ? lh * hw : lh * lw))) * aw, scale);
        const float4 go = ld4(grad_out + (int64_t)ent.x * D + sub * 4);
        a0 += det_contrib(c, (det_factor)go.x);
        a1 += det_contrib(c, (det_factor)go.y);
        a2 += det_contrib(c, (det_factor)go.z);
        a3 += det_contrib(c, (det_factor)go.w);
      }
    }
  }
  const double inv = (double)det->inv_scale;
  const float4 r = make_float4((float)((double)a0 * inv), (float)((double)a1 * inv), (float)((double)a2 * inv),
                               (float)((double)a3 * inv));
  st4(grad_value + ((b * S + s) * H + h) * (int64_t)D + sub * 4, r);
}

// ---- cell reduce: one pass over the sorted entries ---------------------------------------------------------
// The per-pixel gather above visits every entry four times (once per corner pixel) and gives a coarse pixel's
// hundreds of entries to ONE lane group.  Here the entry array is cut into slices of kDetSlice consecutive
// entries; one LANES-wide lane group walks a slice, keeps the four corner sums of the current cell in 64-bit
// fixed point in registers (16 accumulators per lane) and, whenever the cell changes, adds them to the fixed-point
// accumulation buffer [B, S, H, D] with 64-bit integer reds.  Work per group is bounded whatever the
// entries-per-cell distribution is, every entry (and its grad_out row) is read once, and the number of reds is
// ~(cells + slices) x 4 instead of points x 4.  Integer addition commutes, so the result is bit-identical to the
// gather's and to the fixed-point red path's (same products, same scale); msda_det_finalize_kernel converts.
// Lane `sub` owns channels {sub, LANES+sub, 2*LANES+sub, 3*LANES+sub}: the lanes of a group then write
// 8*LANES contiguous bytes per red instruction (full 32-byte sectors; there is no vector form of the 64-bit red).
constexpr int kDetSlice = 64;   // measured at cfg 2 / cfg 5: 32 -> 3.44 / 6.36 ms, 64 -> 3.02 / 5.65 ms, 128 -> 3.33 / 6.05 ms

__device__ __forceinline__ float det_ld(const float* p) { return __ldg(p); }
__device__ __forceinline__ float det_ld(const __nv_bfloat16* p) {
  return __uint_as_float((unsigned)__ldg(reinterpret_cast<const unsigned short*>(p)) << 16);
}
__device__ __forceinline__ float det_ld(const __half* p) {
  return __half2float(__ushort_as_half(__ldg(reinterpret_cast<const unsigned short*>(p))));
}

// No minimum-blocks bound on purpose: ptxas settles at 80 registers (3 CTAs per SM) and 2.09 ms at cfg 5; asking for
// 4 CTAs (64 registers, 40 bytes of spills) gave 2.49 ms, and even a bound of 1 -- same register count, another
// schedule -- 2.66 ms (profiles/r02af_det_variants.txt).  MSDA_DET_REDUCE_MINB > 0 is for variant builds.
#ifndef MSDA_DET_REDUCE_MINB
#define MSDA_DET_REDUCE_MINB 0
#endif
template <int D, typename VT>
#if MSDA_DET_REDUCE_MINB > 0
__global__ void __launch_bounds__(256, MSDA_DET_REDUCE_MINB)
#else
__global__ void __launch_bounds__(256)
#endif
det_cell_reduce_kernel(const VT* __restrict__ grad_out, const int4* __restrict__ entries,
                       const int* __restrict__ bin_start, int n_bins, const int64_t* __restrict__ shapes,
                       const int64_t* __restrict__ lsi, const DetScale* __restrict__ det,
                       unsigned long long* __restrict__ acc, int S, int H, int L) {
  constexpr int LANES = D / 4;
  constexpr int GPC = 256 / LANES;   // lane groups per CTA
  __shared__ CellTab tab;
  load_cell_tab(&tab, shapes, lsi, L);
  const int sub = (threadIdx.x & 31) % LANES;
  const int total = __ldg(bin_start + n_bins);                       // entries actually written (gated-out points have none)
  const int64_t slice = (int64_t)blockIdx.x * GPC + threadIdx.x / LANES;
  if (slice * kDetSlice >= total) return;
  const int e_begin = (int)(slice * kDetSlice);
  const int e_end = min(e_begin + kDetSlice, total);
  const float scale = det->scale;

  // the (non-empty) bin that holds entry e: the last bin whose start is <= e
  auto find_bin = [&](int e, int lo) {
    int hi = n_bins;                                                 // bin_start[n_bins] == total > e
    while (hi - lo > 1) {
      const int mid = lo + ((hi - lo) >> 1);
      if (__ldg(bin_start + mid) <= e) lo = mid;
      else hi = mid;
    }
    return lo;
  };
  long long a[4][4];
  auto clear = [&] {
#pragma unroll
    for (int k = 0; k < 4; ++k)
#pragma unroll
      for (int i = 0; i < 4; ++i) a[k][i] = 0;
  };
  // add the four corner sums of cell `bin` to the accumulation buffer (corners outside the map are dropped)
  auto flush = [&](int bin) {
    const int bh = bin / tab.cells_per_bh, rem = bin - bh * tab.cells_per_bh;
    int l = 0;
    for (int k = 1; k < L; ++k)
      if (rem >= tab.cell_begin[k]) l = k;
    const int Wl = tab.W[l], Hl = tab.H[l], W1 = Wl + 1;
    const int local = rem - tab.cell_begin[l];
    const int cy = local / W1, y0 = cy - 1, x0 = local - cy * W1 - 1;
    const int b = bh / H, h = bh - b * H;
    unsigned long long* base = acc + ((int64_t)b * S * H + h) * D + sub;
#pragma unroll
    for (int k = 0; k < 4; ++k) {
      const int yy = y0 + (k >> 1), xx = x0 + (k & 1);
      if (yy >= 0 && yy < Hl && xx >= 0 && xx < Wl) {
        unsigned long long* p = base + (int64_t)(tab.start[l] + yy * Wl + xx) * H * D;
#pragma unroll
        for (int i = 0; i < 4; ++i)
          if (a[k][i] != 0) atomicAdd(p + i * LANES, (unsigned long long)a[k][i]);
      }
    }
  };
  auto load_go = [&](int row, float (&g)[4]) {
    const VT* r = grad_out + (int64_t)row * D + sub;
#pragma unroll
    for (int i = 0; i < 4; ++i) g[i] = det_ld(r + i * LANES);
  };

  int bin = find_bin(e_begin, 0);
  int bin_end = __ldg(bin_start + bin + 1);
  clear();
  // software pipeline: entry e+2 and the grad_out row of entry e+1 are in flight while entry e is accumulated
  int4 ent = __ldg(entries + e_begin);
  int4 ent1 = (e_begin + 1 < e_end) ? __ldg(entries + e_begin + 1) : ent;
  float g[4], g1[4];
  load_go(ent.x, g);
  for (int e = e_begin; e < e_end; ++e) {
    const int4 ent2 = (e + 2 < e_end) ? __ldg(entries + e + 2) : ent1;
    if (e + 1 < e_end) load_go(ent1.x, g1);
    if (e >= bin_end) {                                              // the cell changes: hand its sums over
      flush(bin);
      clear();
      ++bin;
      bin_end = __ldg(bin_start + bin + 1);
      if (e >= bin_end) {                                            // a run of empty cells: search instead of walking
        bin = find_bin(e, bin);
        bin_end = __ldg(bin_start + bin + 1);
      }
    }
    const float lw = __int_as_float(ent.y), lh = __int_as_float(ent.z), aw = __int_as_float(ent.w);
    const float hh = 1.0f - lh, hw = 1.0f - lw;
    const det_factor c[4] = {(det_factor)det_weight(hh * hw * aw, scale), (det_factor)det_weight(hh * lw * aw, scale),
                             (det_factor)det_weight(lh * hw * aw, scale), (det_factor)det_weight(lh * lw * aw, scale)};
    const det_factor gd[4] = {(det_factor)g[0], (det_factor)g[1], (det_factor)g[2], (det_factor)g[3]};
#pragma unroll
    for (int k = 0; k < 4; ++k)
#pragma unroll
      for (int i = 0; i < 4; ++i) a[k][i] += det_contrib(c[k], gd[i]);
    ent = ent1;
    ent1 = ent2;
#pragma unroll
    for (int i = 0; i < 4; ++i) g[i] = g1[i];
  }
  flush(bin);
}

}  // namespace msda
