// msda_dcnv2.cu -- deformable convolution v1 / v2 (detectron2's DeformConv / ModulatedDeformConv) as im2col + GEMM:
// these kernels build the column matrix and scatter its gradient back; the products with the weight are dense GEMMs
// on the caller's side (cuBLAS through torch).  They replace detectron2/layers/csrc/deformable/
// deform_conv_cuda_kernel.cu: deformable_im2col (DCNv1), modulated_deformable_im2col_cuda (DCNv2) and
// modulated_deformable_col2im_cuda + modulated_deformable_col2im_coord_cuda (backward).
//
// A point is (image, output pixel, deformable group d, kernel tap k = i*kw + j).  It samples the C/dg channels of group
// d at y = (ho*stride_h - pad_h + i*dil_h) + dy, x likewise (torchvision's arithmetic: the integer base converted,
// then ONE rounded add of the offset), with DCNv3's gate and cell (locate_pixel) and, in the fast kernels, the record
// of the MSDeformAttn kernels (record_from_cell: unclamped corner offset + validity bits + corner weights x mask).  A
// corner outside the map is not loaded.  Layouts are in include/msda.h; the column order [pixel][conv group][k][c]
// makes every conv group's weight a plain reshape of weight.permute(0, 2, 3, 1).
//
// Fast kernels (C/dg and C/groups multiples of 16, float / bf16 / f16 input): LANES = D/CPL adjacent lanes own one
// point and walk its row in chunks of D channels, CPL channels per lane (one 16-byte load per corner).  Backward: the
// four <grad_row, corner> dot products are summed over the chunks inside each lane in chunk order, then across the
// LANES lanes by a fixed xor butterfly -- no float atomics, so grad_offset / grad_mask are bit-reproducible; grad_input
// gets 128-bit float reds.
// Generic kernels (any channel count, float64 too): im2col one thread per (point, channel), col2im one thread per
// point that walks its channels in order (grad_offset / grad_mask bit-reproducible there too).
#include "msda_host.h"

#include <type_traits>

#include "msda_scalar.cuh"

namespace msda {

using msda_host::Dcn2Dims;

namespace {

// Point p (inside one image): output pixel, deformable group, tap and the integer part of its sampling position.
struct Dcn2Tap {
  int pix, d, k;
  int base_y, base_x;
};
__device__ __forceinline__ Dcn2Tap dcn2_tap(const Dcn2Dims& g, int p) {
  Dcn2Tap t;
  const int K = g.K();
  t.k = p % K;
  const int r = p / K;
  t.d = r % g.dg;
  t.pix = r / g.dg;
  const int ho = t.pix / g.Wo, wo = t.pix - ho * g.Wo;
  const int i = t.k / g.kw, j = t.k - i * g.kw;
  t.base_y = ho * g.sh - g.ph + i * g.dh;
  t.base_x = wo * g.sw - g.pw + j * g.dw;
  return t;
}

// Element offset, inside one image's columns, of input channel c of point (pix, k): [pix][c / Cg][k][c % Cg].
__device__ __forceinline__ int64_t dcn2_col(const Dcn2Dims& g, int pix, int k, int c) {
  const int Cg = g.Cg(), grp = c / Cg;
  return ((int64_t)pix * g.groups + grp) * g.K() * Cg + (int64_t)k * Cg + (c - grp * Cg);
}

// Mask and (dy, dx) gradients of one point from d_k = <grad_row, corner_k> (0 for a corner outside the map):
// grad_mask = <grad_row, v(p)>, grad_offset = m * <grad_row, dv/dp>.  A gated point gets 0.
template <typename T>
struct Dcn2Grads {
  T gm, gy, gx;
};
template <typename T>
__device__ __forceinline__ Dcn2Grads<T> dcn2_point_grads(bool live, T lh, T lw, T m, T d0, T d1, T d2, T d3) {
  Dcn2Grads<T> r{(T)0, (T)0, (T)0};
  if (live) {
    const T hh = (T)1 - lh, hw = (T)1 - lw;
    r.gm = hh * hw * d0 + hh * lw * d1 + lh * hw * d2 + lh * lw * d3;
    r.gy = (hw * (d2 - d0) + lw * (d3 - d1)) * m;
    r.gx = (hh * (d1 - d0) + lh * (d3 - d2)) * m;
  }
  return r;
}

// The fast kernels' record of point p of image b: corner offset (channel 0 of corner (y0, x0) inside the image, | the
// validity bits; C is a multiple of 16) and corner weights x mask m.  `off` points at the image's offset rows.
template <typename AT>
__device__ __forceinline__ PointRec dcn2_record(const Dcn2Dims& g, const Dcn2Tap& t, const AT* off, int p, float m) {
  const float2 dyx = ld_xy(off, p);   // the pair is stored (dy, dx)
  const Cell<float> c =
      locate_pixel(__fadd_rn((float)t.base_x, dyx.y), __fadd_rn((float)t.base_y, dyx.x), g.H, g.W);
  return record_from_cell(c, m, g.W, 0, 1, 0, g.C);
}

}  // namespace

// Grid (ceil(points_per_image*LANES / 256), B); four CTAs an SM (64 registers).
template <int D, int CPL, typename VT, typename AT>
__global__ void __launch_bounds__(256, 4)
msda_dcnv2_im2col_kernel(const VT* __restrict__ input, const AT* __restrict__ offset, const AT* __restrict__ mask,
                         VT* __restrict__ columns, Dcn2Dims g) {
  constexpr int LANES = D / CPL;
  const int ppi = g.points_per_image();
  const int t = blockIdx.x * blockDim.x + threadIdx.x;
  const int p = t / LANES, sub = t % LANES;
  if (p >= ppi) return;
  const int b = blockIdx.y;
  const Dcn2Tap tap = dcn2_tap(g, p);
  const float m = mask ? ld_aux(mask + (int64_t)b * ppi + p) : 1.0f;
  const PointRec r = dcn2_record(g, tap, offset + (int64_t)b * ppi * 2, p, m);
  const VT* img = input + (int64_t)b * g.H * g.W * g.C + sub * CPL;
  VT* col = columns + (int64_t)b * g.Ho * g.Wo * g.K() * g.C + sub * CPL;
  const int o00 = r.oc & ~15, o01 = o00 + g.C, o10 = o00 + g.W * g.C, o11 = o10 + g.C;
  const int c_end = (tap.d + 1) * g.Cdg();
  for (int c = tap.d * g.Cdg(); c < c_end; c += D) {
    Vec<CPL> acc = vzero<CPL>();
    if (r.oc & 1) fmav(acc, r.cw.x, ldv<CPL>(img + o00 + c));
    if (r.oc & 2) fmav(acc, r.cw.y, ldv<CPL>(img + o01 + c));
    if (r.oc & 4) fmav(acc, r.cw.z, ldv<CPL>(img + o10 + c));
    if (r.oc & 8) fmav(acc, r.cw.w, ldv<CPL>(img + o11 + c));
    stv(col + dcn2_col(g, tap.pix, tap.k, c), acc);
  }
}

// Same grid.  grad_input: float [B,H,W,C], accumulated with reds.
template <int D, int CPL, typename VT, typename AT>
__global__ void __launch_bounds__(256, 4)
msda_dcnv2_col2im_kernel(const VT* __restrict__ grad_columns, const VT* __restrict__ input,
                         const AT* __restrict__ offset, const AT* __restrict__ mask, float* __restrict__ grad_input,
                         AT* __restrict__ grad_offset, AT* __restrict__ grad_mask, Dcn2Dims g) {
  constexpr int LANES = D / CPL;
  const int ppi = g.points_per_image();
  const int t = blockIdx.x * blockDim.x + threadIdx.x;
  const int p = t / LANES, sub = t % LANES;
  const bool live = p < ppi;   // no early return: every lane of the warp takes part in the butterfly
  const int b = blockIdx.y;
  const AT* off = offset + (int64_t)b * ppi * 2;
  const AT* msk = mask ? mask + (int64_t)b * ppi : nullptr;
  float d0 = 0.0f, d1 = 0.0f, d2 = 0.0f, d3 = 0.0f, m = 1.0f;
  PointRec r{};
  if (live) {
    const Dcn2Tap tap = dcn2_tap(g, p);
    if (msk) m = ld_aux(msk + p);
    r = dcn2_record(g, tap, off, p, m);
    const int64_t img_base = (int64_t)b * g.H * g.W * g.C + sub * CPL;
    const VT* img = input + img_base;
    float* gimg = grad_input + img_base;
    const VT* gcol = grad_columns + (int64_t)b * g.Ho * g.Wo * g.K() * g.C + sub * CPL;
    const int o00 = r.oc & ~15, o01 = o00 + g.C, o10 = o00 + g.W * g.C, o11 = o10 + g.C;
    const int c_end = (tap.d + 1) * g.Cdg();
    for (int c = tap.d * g.Cdg(); c < c_end; c += D) {
      const Vec<CPL> go = ldv<CPL>(gcol + dcn2_col(g, tap.pix, tap.k, c));
      if (r.oc & 1) d0 += dotv(go, ldv<CPL>(img + o00 + c));
      if (r.oc & 2) d1 += dotv(go, ldv<CPL>(img + o01 + c));
      if (r.oc & 4) d2 += dotv(go, ldv<CPL>(img + o10 + c));
      if (r.oc & 8) d3 += dotv(go, ldv<CPL>(img + o11 + c));
      // CPL contiguous channels per lane: 16-byte reds at g and g + 4
      if (r.cw.x != 0.0f) scatterv<CPL, 4>(gimg + o00 + c, r.cw.x, go);
      if (r.cw.y != 0.0f) scatterv<CPL, 4>(gimg + o01 + c, r.cw.y, go);
      if (r.cw.z != 0.0f) scatterv<CPL, 4>(gimg + o10 + c, r.cw.z, go);
      if (r.cw.w != 0.0f) scatterv<CPL, 4>(gimg + o11 + c, r.cw.w, go);
    }
  }
#pragma unroll
  for (int s = LANES / 2; s > 0; s >>= 1) {
    d0 += __shfl_xor_sync(0xffffffffu, d0, s);
    d1 += __shfl_xor_sync(0xffffffffu, d1, s);
    d2 += __shfl_xor_sync(0xffffffffu, d2, s);
    d3 += __shfl_xor_sync(0xffffffffu, d3, s);
  }
  if (live && sub == 0) {
    const Dcn2Grads<float> gr = dcn2_point_grads<float>((r.oc & 15) != 0, r.lh, r.lw, m, d0, d1, d2, d3);
    st_aux2(grad_offset + (int64_t)b * ppi * 2 + (int64_t)p * 2, gr.gy, gr.gx);
    if (msk) st_aux1(grad_mask + (int64_t)b * ppi + p, gr.gm);
  }
}

// Any channel count and dtype: one thread per (point, channel of its deformable group), grid-stride.
template <typename VT, typename AT, typename CT>
__global__ void __launch_bounds__(256)
msda_dcnv2_im2col_generic_kernel(const VT* __restrict__ input, const AT* __restrict__ offset,
                                 const AT* __restrict__ mask, VT* __restrict__ columns, Dcn2Dims g, int64_t total) {
  const int Cdg = g.Cdg(), ppi = g.points_per_image();
  for (int64_t idx = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; idx < total;
       idx += (int64_t)gridDim.x * blockDim.x) {
    const int64_t pg = idx / Cdg;
    const int b = (int)(pg / ppi), p = (int)(pg - (int64_t)b * ppi);
    const Dcn2Tap t = dcn2_tap(g, p);
    const int c = t.d * Cdg + (int)(idx - pg * Cdg);
    const CT y = (CT)t.base_y + load_as<CT>(offset + 2 * pg), x = (CT)t.base_x + load_as<CT>(offset + 2 * pg + 1);
    const CT m = mask ? load_as<CT>(mask + pg) : (CT)1;
    const Cell<CT> cell = locate_pixel<CT>(x, y, g.H, g.W);
    CT val = 0;
    if (cell.valid) {
      const VT* v = input + (int64_t)b * g.H * g.W * g.C + ((int64_t)cell.y0 * g.W + cell.x0) * g.C + c;
      const int64_t dx = g.C, dy = (int64_t)g.W * g.C;
      const CT hh = (CT)1 - cell.lh, hw = (CT)1 - cell.lw;
      if (cell.valid & 1u) val += hh * hw * load_as<CT>(v);
      if (cell.valid & 2u) val += hh * cell.lw * load_as<CT>(v + dx);
      if (cell.valid & 4u) val += cell.lh * hw * load_as<CT>(v + dy);
      if (cell.valid & 8u) val += cell.lh * cell.lw * load_as<CT>(v + dy + dx);
    }
    store_as<VT, CT>(columns + (int64_t)b * g.Ho * g.Wo * g.K() * g.C + dcn2_col(g, t.pix, t.k, c), m * val);
  }
}

// One thread per point; grad_input (CT: float, or double for float64) accumulated with atomics.
template <typename VT, typename AT, typename CT>
__global__ void __launch_bounds__(256)
msda_dcnv2_col2im_generic_kernel(const VT* __restrict__ grad_columns, const VT* __restrict__ input,
                                 const AT* __restrict__ offset, const AT* __restrict__ mask, CT* __restrict__ grad_input,
                                 AT* __restrict__ grad_offset, AT* __restrict__ grad_mask, Dcn2Dims g, int64_t total) {
  const int Cdg = g.Cdg(), ppi = g.points_per_image();
  for (int64_t pg = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; pg < total;
       pg += (int64_t)gridDim.x * blockDim.x) {
    const int b = (int)(pg / ppi), p = (int)(pg - (int64_t)b * ppi);
    const Dcn2Tap t = dcn2_tap(g, p);
    const CT y = (CT)t.base_y + load_as<CT>(offset + 2 * pg), x = (CT)t.base_x + load_as<CT>(offset + 2 * pg + 1);
    const CT m = mask ? load_as<CT>(mask + pg) : (CT)1;
    const Cell<CT> cell = locate_pixel<CT>(x, y, g.H, g.W);
    CT d0 = 0, d1 = 0, d2 = 0, d3 = 0;
    if (cell.valid) {
      const int64_t o = (int64_t)b * g.H * g.W * g.C + ((int64_t)cell.y0 * g.W + cell.x0) * g.C;
      const VT* v = input + o;
      CT* gv = grad_input + o;
      const int64_t dx = g.C, dy = (int64_t)g.W * g.C;
      const CT hh = (CT)1 - cell.lh, hw = (CT)1 - cell.lw;
      const CT w0 = m * hh * hw, w1 = m * hh * cell.lw, w2 = m * cell.lh * hw, w3 = m * cell.lh * cell.lw;
      const VT* gcol = grad_columns + (int64_t)b * g.Ho * g.Wo * g.K() * g.C;
      for (int c = t.d * Cdg; c < (t.d + 1) * Cdg; ++c) {
        const CT go = load_as<CT>(gcol + dcn2_col(g, t.pix, t.k, c));
        if (cell.valid & 1u) { d0 += go * load_as<CT>(v + c); atomicAdd(gv + c, w0 * go); }
        if (cell.valid & 2u) { d1 += go * load_as<CT>(v + dx + c); atomicAdd(gv + dx + c, w1 * go); }
        if (cell.valid & 4u) { d2 += go * load_as<CT>(v + dy + c); atomicAdd(gv + dy + c, w2 * go); }
        if (cell.valid & 8u) { d3 += go * load_as<CT>(v + dy + dx + c); atomicAdd(gv + dy + dx + c, w3 * go); }
      }
    }
    const Dcn2Grads<CT> gr = dcn2_point_grads<CT>(cell.valid != 0, cell.lh, cell.lw, m, d0, d1, d2, d3);
    store_as<AT, CT>(grad_offset + 2 * pg, gr.gy);
    store_as<AT, CT>(grad_offset + 2 * pg + 1, gr.gx);
    if (mask) store_as<AT, CT>(grad_mask + pg, gr.gm);
  }
}

}  // namespace msda

namespace msda_host {

namespace {

// channels per lane of the fast kernels: one 16-byte load per corner
template <typename VT>
constexpr int dcn2_cpl() { return std::is_same_v<VT, float> ? 4 : 8; }

// D of the fast kernels for this problem, 0 = the generic kernels: the largest of 128 / 64 / 32 / 16 dividing both
// C/dg and C/groups (a chunk never straddles a deformable or a conv group), float / bf16 / f16, 32-bit element
// offsets inside one image (one spare row of slack) and inside one image's thread range, B within grid.y.
template <typename VT>   // float / bf16 / f16
int fast_chunk(const Dcn2Dims& g, unsigned flags) {
  if (flags & MSDA_FLAG_FORCE_GENERIC) return 0;
  if (((int64_t)g.H * g.W + g.W + 1) * g.C >= ((int64_t)1 << 31) || g.B > 65535) return 0;
  for (int D = 128; D >= 16; D /= 2) {
    if (g.Cdg() % D != 0 || g.Cg() % D != 0) continue;
    const int64_t lanes = D / dcn2_cpl<VT>();
    return ((int64_t)g.points_per_image() * lanes + 256 < ((int64_t)1 << 31)) ? D : 0;
  }
  return 0;
}

}  // namespace

#ifdef MSDA_EXP_SLIM
int dcnv2_im2col(cudaStream_t, const Dcn2Dims&, int, unsigned, const void*, const void*, const void*, void*) {
  return fail(MSDA_ERR_UNSUPPORTED, "slim build: no DCNv2 kernels");
}
int dcnv2_col2im(cudaStream_t, const Dcn2Dims&, int, unsigned, const void*, const void*, const void*, const void*,
                 void*, void*, void*) {
  return fail(MSDA_ERR_UNSUPPORTED, "slim build: no DCNv2 kernels");
}
#else
int dcnv2_im2col(cudaStream_t st, const Dcn2Dims& g, int dtype, unsigned flags, const void* input, const void* offset,
                 const void* mask, void* columns) {
  return with_types<AllTags>(dtype, [&](auto t) {
    using VT = typename decltype(t)::VT;
    using AT = typename decltype(t)::AT;
    if constexpr (!std::is_same_v<VT, double>) {
      if (const int D = fast_chunk<VT>(g, flags)) {
        return with_chunk(D, [&](auto DC) {
          constexpr int CPL = dcn2_cpl<VT>();
          const dim3 grid((unsigned)(((int64_t)g.points_per_image() * (DC / CPL) + 255) / 256), (unsigned)g.B);
          msda::msda_dcnv2_im2col_kernel<DC, CPL, VT, AT><<<grid, 256, 0, st>>>(
              (const VT*)input, (const AT*)offset, (const AT*)mask, (VT*)columns, g);
          return launched();
        });
      }
    }
    using CT = typename msda::Compute<VT>::type;
    const int64_t total = g.n_points() * g.Cdg();
    msda::msda_dcnv2_im2col_generic_kernel<VT, AT, CT><<<grid_for(total, 256, 148 * 32), 256, 0, st>>>(
        (const VT*)input, (const AT*)offset, (const AT*)mask, (VT*)columns, g, total);
    return launched();
  });
}

int dcnv2_col2im(cudaStream_t st, const Dcn2Dims& g, int dtype, unsigned flags, const void* grad_columns,
                 const void* input, const void* offset, const void* mask, void* grad_input_acc, void* grad_offset,
                 void* grad_mask) {
  return with_types<AllTags>(dtype, [&](auto t) {
    using VT = typename decltype(t)::VT;
    using AT = typename decltype(t)::AT;
    if constexpr (!std::is_same_v<VT, double>) {
      if (const int D = fast_chunk<VT>(g, flags)) {
        return with_chunk(D, [&](auto DC) {
          constexpr int CPL = dcn2_cpl<VT>();
          const dim3 grid((unsigned)(((int64_t)g.points_per_image() * (DC / CPL) + 255) / 256), (unsigned)g.B);
          msda::msda_dcnv2_col2im_kernel<DC, CPL, VT, AT><<<grid, 256, 0, st>>>(
              (const VT*)grad_columns, (const VT*)input, (const AT*)offset, (const AT*)mask, (float*)grad_input_acc,
              (AT*)grad_offset, (AT*)grad_mask, g);
          return launched();
        });
      }
    }
    using CT = typename msda::Compute<VT>::type;
    const int64_t total = g.n_points();
    msda::msda_dcnv2_col2im_generic_kernel<VT, AT, CT><<<grid_for(total, 256, 148 * 32), 256, 0, st>>>(
        (const VT*)grad_columns, (const VT*)input, (const AT*)offset, (const AT*)mask, (CT*)grad_input_acc,
        (AT*)grad_offset, (AT*)grad_mask, g, total);
    return launched();
  });
}
#endif

}  // namespace msda_host
