// msda_generic.cuh -- shape-agnostic MSDeformAttn kernels (any D, L, P; float / double / bf16 / f16 value).
//
// These cover what the fast kernels (msda_fast.cuh) do not: head dims outside {16,32,64,128},
// float64 (the reference's gradcheck path, tests/test_ms_deform_attn.py:131-133 walks
// D in {30,32,64,71,1025}), more than 16 levels, images too large for 32-bit offsets.
// They play the role of the reference's forward kernel (cuh:237-299) and of its six backward
// kernels (cuh:301-920) at once: one forward kernel, one backward kernel, any channel count.
//
//   forward   one thread per output element (b,q,h,c), grid-stride; channel is the fastest index
//             so a warp reads consecutive channels of one pixel.
//   backward  one CTA per (b,q,h) row, threads stride over channels; per point the three
//             reductions over channels (grad_attn_weight, grad_loc.x, grad_loc.y) are done with
//             warp shuffles + one shared-memory hop; grad_value goes out as scalar atomics.
#pragma once
#include <cuda_bf16.h>
#include <cuda_fp16.h>
#include <cuda_runtime.h>
#include <stdint.h>

#include "msda_coords.cuh"
#include "msda_scalar.cuh"

namespace msda {

// value/out: VT; loc/w: CT (= float for float, bf16 and f16 values, double for double).
template <typename VT, typename CT>
__global__ void __launch_bounds__(256)
msda_fwd_generic_kernel(const VT* __restrict__ value, const int64_t* __restrict__ shapes,
                        const int64_t* __restrict__ lsi, const CT* __restrict__ loc,
                        const CT* __restrict__ w, VT* __restrict__ out, int S, int H, int D, int L,
                        int Q, int P, int64_t total) {
  for (int64_t idx = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; idx < total;
       idx += (int64_t)gridDim.x * blockDim.x) {
    const int c = (int)(idx % D);
    const int64_t row = idx / D;             // (b*Q + q)*H + h
    const int h = (int)(row % H);
    const int64_t b = row / H / Q;
    const VT* vimg = value + b * (int64_t)S * H * D + (int64_t)h * D + c;
    const CT* lp = loc + row * (int64_t)L * P * 2;
    const CT* wp = w + row * (int64_t)L * P;
    CT acc = 0;
    for (int l = 0; l < L; ++l) {
      const int Hl = (int)shapes[2 * l], Wl = (int)shapes[2 * l + 1];
      const VT* vlev = vimg + lsi[l] * (int64_t)H * D;
      for (int p = 0; p < P; ++p) {
        const CT lx = lp[0], ly = lp[1], aw = wp[0];
        lp += 2;
        wp += 1;
        const Cell<CT> cell = locate<CT>(lx, ly, Hl, Wl);
        if (cell.valid == 0) continue;
        const CT hh = (CT)1 - cell.lh, hw = (CT)1 - cell.lw;
        const int64_t o00 = ((int64_t)cell.y0 * Wl + cell.x0) * H * D;
        const int64_t dx = (int64_t)H * D, dy = (int64_t)Wl * H * D;
        CT val = 0;
        if (cell.valid & 1u) val += hh * hw * load_as<CT>(vlev + o00);
        if (cell.valid & 2u) val += hh * cell.lw * load_as<CT>(vlev + o00 + dx);
        if (cell.valid & 4u) val += cell.lh * hw * load_as<CT>(vlev + o00 + dy);
        if (cell.valid & 8u) val += cell.lh * cell.lw * load_as<CT>(vlev + o00 + dx + dy);
        acc += val * aw;
      }
    }
    store_as<VT, CT>(out + idx, acc);
  }
}

template <typename CT>
__device__ __forceinline__ CT warp_sum(CT v) {
#pragma unroll
  for (int m = 16; m > 0; m >>= 1) v += __shfl_xor_sync(0xffffffffu, v, m);
  return v;
}

template <typename CT>
__device__ __forceinline__ void accumulate(CT* g, CT v, float) { atomicAdd(g, v); }
__device__ __forceinline__ void accumulate(unsigned long long* g, float v, float scale) {
  atomicAdd(g, (unsigned long long)__float2ll_rn(v * scale));
}
__device__ __forceinline__ void accumulate(unsigned long long* g, double v, float scale) {
  atomicAdd(g, (unsigned long long)__double2ll_rn(v * (double)scale));
}

// grad_value accumulates in ACC: CT (float scratch for bf16 values; the caller converts afterwards)
// or 64-bit fixed point for MSDA_FLAG_DETERMINISTIC.
template <typename VT, typename CT, typename ACC>
__global__ void __launch_bounds__(256)
msda_bwd_generic_kernel(const VT* __restrict__ grad_out, const VT* __restrict__ value,
                        const int64_t* __restrict__ shapes, const int64_t* __restrict__ lsi,
                        const CT* __restrict__ loc, const CT* __restrict__ w, ACC* __restrict__ grad_value,
                        CT* __restrict__ grad_loc, CT* __restrict__ grad_w, const DetScale* __restrict__ det,
                        int S, int H, int D, int L, int Q, int P, int64_t rows) {
  const float gscale = det ? det->scale : 1.0f;
  __shared__ CT red[3][8];
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5, nwarp = blockDim.x >> 5;
  for (int64_t row = blockIdx.x; row < rows; row += gridDim.x) {
    const int h = (int)(row % H);
    const int64_t b = row / H / Q;
    const int64_t img = b * (int64_t)S * H * D + (int64_t)h * D;
    const VT* go = grad_out + row * D;
    const CT* lp = loc + row * (int64_t)L * P * 2;
    const CT* wp = w + row * (int64_t)L * P;
    CT* glp = grad_loc + row * (int64_t)L * P * 2;
    CT* gwp = grad_w + row * (int64_t)L * P;
    for (int l = 0; l < L; ++l) {
      const int Hl = (int)shapes[2 * l], Wl = (int)shapes[2 * l + 1];
      const int64_t lev = img + lsi[l] * (int64_t)H * D;
      for (int p = 0; p < P; ++p, lp += 2, wp += 1, glp += 2, gwp += 1) {
        const CT lx = lp[0], ly = lp[1], aw = wp[0];
        const Cell<CT> cell = locate<CT>(lx, ly, Hl, Wl);   // block-uniform
        if (cell.valid == 0) {
          if (threadIdx.x == 0) { glp[0] = 0; glp[1] = 0; gwp[0] = 0; }
          continue;
        }
        const CT lh = cell.lh, lw = cell.lw, hh = (CT)1 - lh, hw = (CT)1 - lw;
        const int64_t o00 = lev + ((int64_t)cell.y0 * Wl + cell.x0) * H * D;
        const int64_t dx = (int64_t)H * D, dy = (int64_t)Wl * H * D;
        CT s_w = 0, s_x = 0, s_y = 0;
        for (int c = threadIdx.x; c < D; c += blockDim.x) {
          const CT top = load_as<CT>(go + c);
          const CT tgv = top * aw;
          CT v1 = 0, v2 = 0, v3 = 0, v4 = 0;
          if (cell.valid & 1u) { v1 = load_as<CT>(value + o00 + c); accumulate(grad_value + o00 + c, hh * hw * tgv, gscale); }
          if (cell.valid & 2u) { v2 = load_as<CT>(value + o00 + dx + c); accumulate(grad_value + o00 + dx + c, hh * lw * tgv, gscale); }
          if (cell.valid & 4u) { v3 = load_as<CT>(value + o00 + dy + c); accumulate(grad_value + o00 + dy + c, lh * hw * tgv, gscale); }
          if (cell.valid & 8u) { v4 = load_as<CT>(value + o00 + dx + dy + c); accumulate(grad_value + o00 + dx + dy + c, lh * lw * tgv, gscale); }
          const CT val = hh * hw * v1 + hh * lw * v2 + lh * hw * v3 + lh * lw * v4;
          s_w += top * val;
          s_x += (hh * (v2 - v1) + lh * (v4 - v3)) * tgv;   // cuh:119-153 grad_w_weight
          s_y += (hw * (v3 - v1) + lw * (v4 - v2)) * tgv;   // grad_h_weight
        }
        s_w = warp_sum(s_w); s_x = warp_sum(s_x); s_y = warp_sum(s_y);
        if (nwarp > 1) {
          if (lane == 0) { red[0][warp] = s_w; red[1][warp] = s_x; red[2][warp] = s_y; }
          __syncthreads();
          if (threadIdx.x == 0) {
            s_w = red[0][0]; s_x = red[1][0]; s_y = red[2][0];
            for (int k = 1; k < nwarp; ++k) { s_w += red[0][k]; s_x += red[1][k]; s_y += red[2][k]; }
          }
          __syncthreads();
        }
        if (threadIdx.x == 0) {
          gwp[0] = s_w;
          glp[0] = (CT)Wl * s_x;   // cuh:157
          glp[1] = (CT)Hl * s_y;   // cuh:158
        }
      }
    }
  }
}

// scratch (float) -> bf16 / f16 grad_value
template <typename VT>
__global__ void msda_cast_f32_kernel(const float* __restrict__ src, VT* __restrict__ dst, int64_t n) {
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x)
    store_as<VT, float>(dst + i, src[i]);
}

// ---- deterministic mode helpers ------------------------------------------------------------
// max |x| over a tensor, as the bit pattern of a non-negative float (atomicMax on unsigned is
// order independent, so the scale -- and with it every bit of the result -- is reproducible).
template <typename T>
__global__ void msda_amax_kernel(const T* __restrict__ x, int64_t n, unsigned* __restrict__ out_bits) {
  float m = 0.0f;
  bool bad = false;
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x) {
    const double v = fabs((double)load_as<typename Compute<T>::type, T>(x + i));
    if (!(v <= 3.0e38)) bad = true;              // NaN, Inf or beyond float range
    m = fmaxf(m, __double2float_ru(v));
  }
  if (bad) m = __int_as_float(0x7f800000);       // +Inf marks "not finite"
#pragma unroll
  for (int k = 16; k > 0; k >>= 1) m = fmaxf(m, __shfl_xor_sync(0xffffffffu, m, k));
  if ((threadIdx.x & 31) == 0) atomicMax(out_bits, __float_as_uint(m));
}

// scale = 2^k with max|go| * max|w| * 2^k <= 2^38 (double: 2^44); one thread.
__global__ void msda_det_scale_kernel(const unsigned* __restrict__ amax_bits, DetScale* __restrict__ out, int target_log2) {
  const float a = __uint_as_float(amax_bits[0]), b = __uint_as_float(amax_bits[1]);
  const float bound = a * b;
  DetScale r;
  if (!(bound < 3.0e38f)) {
    r.scale = 0.0f;
    r.inv_scale = __int_as_float(0x7fc00000);    // NaN in, NaN out
  } else if (bound == 0.0f) {
    r.scale = 1.0f;
    r.inv_scale = 1.0f;
  } else {
    int e;
    frexpf(bound, &e);                           // bound = m * 2^e, m in [0.5, 1)  =>  bound < 2^e
    int k = target_log2 - e;
    k = k > 120 ? 120 : (k < -120 ? -120 : k);
    r.scale = ldexpf(1.0f, k);
    r.inv_scale = ldexpf(1.0f, -k);
  }
  *out = r;
}

// fixed point -> grad_value
template <typename VT>
__global__ void msda_det_finalize_kernel(const long long* __restrict__ acc, VT* __restrict__ dst, int64_t n,
                                         const DetScale* __restrict__ det) {
  const double inv = (double)det->inv_scale;
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x)
    store_as<VT, typename Compute<VT>::type>(dst + i, (typename Compute<VT>::type)((double)acc[i] * inv));
}

// Test hook, see include/msda.h::msda_debug_bookkeeping: generic-kernel flavour (locate<float> + the reference's
// per-corner bounds tests).  The fast kernels' own records are dumped by msda_fast_records_kernel (msda_capi.cu).
__global__ void msda_bookkeeping_kernel(const float* __restrict__ loc, const int64_t* __restrict__ shapes,
                                        const int64_t* __restrict__ lsi, int S, int H, int D, int L, int Q, int P,
                                        int64_t npts, int64_t* __restrict__ offs, float* __restrict__ frac) {
  for (int64_t pt = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; pt < npts; pt += (int64_t)gridDim.x * blockDim.x) {
    const int l = (int)((pt / P) % L);
    const int64_t row = pt / P / L;
    const int h = (int)(row % H);
    const int64_t b = row / H / Q;
    const int Hl = (int)shapes[2 * l], Wl = (int)shapes[2 * l + 1];
    const Cell<float> cell = locate<float>(loc[2 * pt], loc[2 * pt + 1], Hl, Wl);
    const int ys[4] = {cell.y0, cell.y0, cell.y0 + 1, cell.y0 + 1};
    const int xs[4] = {cell.x0, cell.x0 + 1, cell.x0, cell.x0 + 1};
#pragma unroll
    for (int k = 0; k < 4; ++k) {
      int64_t o = -1;
      if (cell.valid & (1u << k)) o = (b * S + lsi[l] + (int64_t)ys[k] * Wl + xs[k]) * H * D + (int64_t)h * D;
      offs[4 * pt + k] = o;
    }
    frac[2 * pt] = cell.valid ? cell.lw : 0.0f;
    frac[2 * pt + 1] = cell.valid ? cell.lh : 0.0f;
  }
}

}  // namespace msda
