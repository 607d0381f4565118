// msda_capi.cu -- host side of libmsda_b200.so: argument checks, kernel selection, launches.
// The C ABI is declared and documented in include/msda.h.
//
// Plays the role of ms_deform_attn_cuda_forward / _backward
// (/root/reference/detrex/layers/csrc/MsDeformAttn/ms_deform_attn_cuda.cu:21-154) and of the
// kernel selector ms_deformable_col2im_cuda (ms_deform_im2col_cuda.cuh:956-1327), minus ATen:
// no allocation, no im2col_step chunk loop (one launch covers the batch), errors returned.
#include "msda_host.h"

#include <atomic>
#include <cstdarg>
#include <cstdio>
#include <cstdlib>
#include <cstring>

#include "msda_generic.cuh"
#include "msda_det.cuh"

namespace {
std::atomic<uint64_t> g_launches{0};
thread_local char g_err[512] = "";
}  // namespace

namespace msda_host {

int fail(int status, const char* fmt, ...) {
  va_list ap;
  va_start(ap, fmt);
  vsnprintf(g_err, sizeof(g_err), fmt, ap);
  va_end(ap);
  return status;
}

int cuda_fail(cudaError_t e, const char* what) {
  cudaGetLastError();   // clear the runtime's sticky last-error so it cannot be blamed on a later, healthy launch
  return fail(MSDA_ERR_CUDA, "%s: %s (%s)", what, cudaGetErrorString(e), cudaGetErrorName(e));
}

void count_launch() { g_launches.fetch_add(1, std::memory_order_relaxed); }

int check_alignment(std::initializer_list<NamedPtr> ptrs) {
  for (const NamedPtr& p : ptrs)
    if (p.ptr && (reinterpret_cast<uintptr_t>(p.ptr) & 15u) != 0)
      return fail(MSDA_ERR_INVALID_ARGUMENT, "%s (%p) is not 16-byte aligned: the kernels use 128-bit accesses", p.name,
                  p.ptr);
  return MSDA_OK;
}

int check_workspace(const void* workspace, size_t workspace_bytes, size_t need) {
  if (need && (!workspace || workspace_bytes < need))
    return fail(MSDA_ERR_WORKSPACE, "workspace of %zu bytes required, %zu given", need, workspace_bytes);
  return MSDA_OK;
}

bool fast_ok(const Dims& d, int dtype, unsigned flags) {
  if (flags & MSDA_FLAG_FORCE_GENERIC) return false;
  if (dtype != MSDA_F32 && dtype != MSDA_BF16 && dtype != MSDA_F16) return false;
  if (!(d.D == 16 || d.D == 32 || d.D == 64 || d.D == 128)) return false;
  if (d.L < 1 || d.L > msda::kFastMaxLevels) return false;
  if (d.L * d.P < 1 || d.L * d.P > msda::kFastMaxPoints) return false;
  // element offsets inside one image are 32-bit in the fast kernels (one spare row/pixel of slack)
  if (((int64_t)d.S + 65536) * d.H * d.D >= ((int64_t)1 << 31)) return false;
  return true;
}

}  // namespace msda_host

namespace {
using namespace msda_host;

// Runs the call on the device that owns `ptr`, restoring the caller's device afterwards
// (the reference has no guard at all: ms_deform_attn_cuda.cu:66 just takes the current stream).
struct DeviceGuard {
  int prev = -1;
  bool switched = false;
  cudaError_t enter(const void* ptr) {
    cudaPointerAttributes attr;
    cudaError_t e = cudaPointerGetAttributes(&attr, ptr);
    if (e != cudaSuccess) return e;
    if (attr.type != cudaMemoryTypeDevice && attr.type != cudaMemoryTypeManaged) return cudaErrorInvalidDevicePointer;
    e = cudaGetDevice(&prev);
    if (e != cudaSuccess) return e;
    if (attr.device != prev) {
      e = cudaSetDevice(attr.device);
      switched = (e == cudaSuccess);
    }
    return e;
  }
  ~DeviceGuard() {
    if (switched) cudaSetDevice(prev);
  }
};

int check_dims(const Dims& d, int dtype) {
  if (d.B < 0 || d.S < 0 || d.H < 0 || d.D < 0 || d.L < 0 || d.Q < 0 || d.P < 0)
    return fail(MSDA_ERR_INVALID_ARGUMENT, "negative dimension (B=%d S=%d H=%d D=%d L=%d Q=%d P=%d)", d.B, d.S, d.H,
                d.D, d.L, d.Q, d.P);
  if (dtype != MSDA_F32 && dtype != MSDA_F64 && dtype != MSDA_BF16 && dtype != MSDA_F16)
    return fail(MSDA_ERR_INVALID_ARGUMENT, "unknown dtype tag %d", dtype);
  return MSDA_OK;
}

// Test hook (msda_debug_bookkeeping with MSDA_DEBUG_FAST_RECORDS): builds the SAME PointRec the fast kernels build
// (msda::make_record: locate + unclamped offset + corner-validity bits) and decodes it the way their gather / scatter
// loops do -- o00 = oc & ~15, +H*D for x+1, +W_l*H*D for y+1, corner k used iff bit k -- so the integers the fast
// kernels actually gather from / scatter to are what the test compares bit for bit.
__global__ void msda_fast_records_kernel(const float* __restrict__ loc, const int64_t* __restrict__ shapes,
                                         const int64_t* __restrict__ lsi, int S, int H, int D, int L, int Q, int P,
                                         int64_t npts, int64_t* __restrict__ offs, float* __restrict__ frac) {
  const int HD = H * D;
  for (int64_t pt = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; pt < npts; pt += (int64_t)gridDim.x * blockDim.x) {
    const int l = (int)((pt / P) % L);
    const int64_t row = pt / P / L;
    const int h = (int)(row % H);
    const int64_t b = row / H / Q;
    const int Hl = (int)shapes[2 * l], Wl = (int)shapes[2 * l + 1];
    const msda::PointRec r = msda::make_record(loc[2 * pt], loc[2 * pt + 1], 1.0f, Hl, Wl, (int)lsi[l], H, h, D);
    const int oc = r.oc;
    const bool gated = (oc & 15) == 0;
    const int o00 = oc & ~15;
    const int o01 = o00 + HD, o10 = o00 + Wl * HD, o11 = o10 + HD;
    const int64_t img = b * (int64_t)S * HD;
    offs[4 * pt + 0] = (oc & 1) ? img + o00 : -1;
    offs[4 * pt + 1] = (oc & 2) ? img + o01 : -1;
    offs[4 * pt + 2] = (oc & 4) ? img + o10 : -1;
    offs[4 * pt + 3] = (oc & 8) ? img + o11 : -1;
    frac[2 * pt] = gated ? 0.0f : r.lw;
    frac[2 * pt + 1] = gated ? 0.0f : r.lh;
  }
}

template <typename VT>
int det_gather(cudaStream_t st, const Dims& d, const void* go, const int4* entries, const int* bin_start,
               const int64_t* shapes, const int64_t* lsi, const msda::DetScale* scale, void* gv) {
  const int64_t items = (int64_t)d.B * d.S * d.H;
  return with_chunk(d.D, [&](auto D) {
    constexpr int RPC = 256 / (D / 4);
    msda::det_gather_kernel<D, VT><<<(unsigned)((items + RPC - 1) / RPC), 256, 0, st>>>(
        (const VT*)go, entries, bin_start, shapes, lsi, scale, (VT*)gv, d.B, d.S, d.H, d.L);
    return launched();
  });
}

// dense problems reduce per cell (one pass over the entries), sparse ones gather per pixel (msda_det.cuh)
bool det_dense(const Dims& d) { return d.n_points() >= (int64_t)msda::kDetDenseRatio * d.B * d.S * d.H; }

template <typename VT>
int det_cell_reduce(cudaStream_t st, const Dims& d, const void* go, const int4* entries, const int* bin_start,
                    int64_t n_bins, const int64_t* shapes, const int64_t* lsi, const msda::DetScale* scale,
                    unsigned long long* acc) {
  const int64_t slices = (d.n_points() + msda::kDetSlice - 1) / msda::kDetSlice;   // upper bound: gated points have no entry
  return with_chunk(d.D, [&](auto D) {
    constexpr int GPC = 256 / (D / 4);
    msda::det_cell_reduce_kernel<D, VT><<<(unsigned)((slices + GPC - 1) / GPC), 256, 0, st>>>(
        (const VT*)go, entries, bin_start, (int)n_bins, shapes, lsi, scale, acc, d.S, d.H, d.L);
    return launched();
  });
}

// 64-bit fixed-point accumulators -> grad_value
template <typename VT>
int det_finalize(cudaStream_t st, const unsigned long long* acc, void* gv, int64_t nv, const msda::DetScale* scale) {
  msda::msda_det_finalize_kernel<VT><<<grid_for(nv, 256, 148 * 16), 256, 0, st>>>(
      reinterpret_cast<const long long*>(acc), (VT*)gv, nv, scale);
  return launched();
}

// Workspace of the sorted deterministic path (all 16-byte aligned):
//   [bins+1 ints: counts -> starts][bins ints: cursors][scan block sums][entries: n_points x 16 B][amax x2, DetScale]
//   [fixed-point accumulators: n_value x 8 B]
struct DetLayout {
  int64_t bins;        // upper bound, B*H*(2S+2L)
  int64_t n_scan;      // bins + 1
  int64_t scan_blocks;
  size_t off_cursor, off_sums, off_entries, off_misc, off_wamax, off_acc, total;
};
DetLayout det_layout(const Dims& d) {
  DetLayout l;
  l.bins = (int64_t)d.B * d.H * msda::det_cells_bound(d.S, d.L);
  l.n_scan = l.bins + 1;
  l.scan_blocks = (l.n_scan + msda::kScanPerBlock - 1) / msda::kScanPerBlock;
  auto up = [](size_t x) { return (x + 255) & ~(size_t)255; };
  l.off_cursor = up((size_t)l.n_scan * 4);
  l.off_sums = l.off_cursor + up((size_t)l.bins * 4);
  l.off_entries = l.off_sums + up((size_t)l.scan_blocks * 4);
  l.off_misc = l.off_entries + up((size_t)d.n_points() * 16);
  l.off_acc = l.off_misc + 256;
  l.off_wamax = l.off_acc + (det_dense(d) ? up((size_t)d.n_value() * 8) : 0);   // accumulators: cell reduce only
  // two floats per warp of the entry-filing backward (<= 256 threads per CTA)
  l.total = l.off_wamax + up((size_t)(d.rows() * d.D / 128 + 8) * 8);
  return l;
}
// the sorted path needs 32-bit bin / entry / row indices
bool det_sorted_ok(const Dims& d, int dtype, unsigned flags) {
  if (flags & MSDA_FLAG_DET_ATOMIC) return false;
  if (!fast_ok(d, dtype, flags)) return false;
  const int64_t lim = ((int64_t)1 << 31) - 4096;
  return (int64_t)d.B * d.H * msda::det_cells_bound(d.S, d.L) < lim && d.n_points() < lim && d.rows() < lim;
}

// ------------------------------------------------------------------------------------------
// generic launches
// ------------------------------------------------------------------------------------------
template <typename VT, typename CT>
int fwd_generic(cudaStream_t st, const Dims& d, const void* value, const int64_t* shapes, const int64_t* lsi,
                const void* loc, const void* w, void* out) {
  const int64_t total = d.rows() * d.D;
  const int grid = grid_for(total, 256, 148 * 32);
  msda::msda_fwd_generic_kernel<VT, CT><<<grid, 256, 0, st>>>((const VT*)value, shapes, lsi, (const CT*)loc,
                                                              (const CT*)w, (VT*)out, d.S, d.H, d.D, d.L, d.Q, d.P,
                                                              total);
  return launched();
}

template <typename VT, typename CT, typename ACC>
int bwd_generic(cudaStream_t st, const Dims& d, const void* go, const void* value, const int64_t* shapes,
                const int64_t* lsi, const void* loc, const void* w, ACC* gv, void* gl, void* gw,
                const msda::DetScale* det = nullptr) {
  int threads = 32;
  while (threads < d.D && threads < 256) threads <<= 1;
  const int64_t rows = d.rows();
  const int grid = (int)(rows < 148 * 64 ? rows : 148 * 64);
  msda::msda_bwd_generic_kernel<VT, CT, ACC><<<grid, threads, 0, st>>>(
      (const VT*)go, (const VT*)value, shapes, lsi, (const CT*)loc, (const CT*)w, gv, (CT*)gl, (CT*)gw, det, d.S, d.H,
      d.D, d.L, d.Q, d.P, rows);
  return launched();
}

// bf16 / f16 values: 2-byte elements, grad_value accumulated in a float workspace and converted at the end
bool two_byte(int dtype) { return dtype == MSDA_BF16 || dtype == MSDA_F16; }

size_t elem_size(int dtype) { return dtype == MSDA_F64 ? 8 : (two_byte(dtype) ? 2 : 4); }

// The autocast tags of the fused entry points (include/msda.h): the value dtype they stand for, and whether the
// offsets / logits and their gradients are 16-bit too.  Every other tag maps to itself.
int fused_value_dtype(int dtype) {
  return dtype == MSDA_BF16_AUX16 ? MSDA_BF16 : (dtype == MSDA_F16_AUX16 ? MSDA_F16 : dtype);
}
size_t aux_size(int dtype) { return (dtype == MSDA_BF16_AUX16 || dtype == MSDA_F16_AUX16) ? 2 : 4; }

// float workspace -> bf16 / f16 grad_value
int cast_from_f32(cudaStream_t st, const float* src, void* dst, int64_t n, int dtype) {
  const int grid = grid_for(n, 256, 148 * 16);
  if (dtype == MSDA_BF16) msda::msda_cast_f32_kernel<__nv_bfloat16><<<grid, 256, 0, st>>>(src, (__nv_bfloat16*)dst, n);
  else msda::msda_cast_f32_kernel<__half><<<grid, 256, 0, st>>>(src, (__half*)dst, n);
  return launched();
}

// The FusedArgs of the MSDeformAttn module path: reference points, the 1/P offset normalisation, the value padding mask
msda::FusedArgs module_args(const float* reference_points, int ref_dim, int num_point, const uint8_t* value_mask) {
  msda::FusedArgs fa{};
  fa.ref = reference_points;
  fa.ref_dim = ref_dim;
  fa.inv_P = 1.0f / (float)num_point;
  fa.num_P = (float)num_point;
  fa.value_mask = value_mask;
  return fa;
}

// Where the points of the deterministic backward come from: the plain operator's sampling_loc / attn_weight, or the
// DCNv3 sampling grid (offset / mask + geometry; `Dims` is then the equivalent one-level problem).  The count, gather
// and cell-reduce kernels read the level table from device memory in both cases (DCNv3: the one-level slot
// det_one_level_kernel writes into the workspace).
struct DetSource {
  const void* loc;               // plain: sampling_loc [B,Q,H,L,P,2]; DCNv3: offset [N,Ho,Wo,G*K*2]
  const void* w;                 // plain: attn_weight;                 DCNv3: mask   [N,Ho,Wo,G*K]
  const int64_t* shapes;
  const int64_t* lsi;
  const msda::FusedArgs* dcn;    // null: plain operator
};

// Bit-reproducible grad_value (MSDA_FLAG_DETERMINISTIC): 64-bit fixed-point accumulation (see include/msda.h), by the
// sorted segment reduction where det_sorted_ok admits the problem, else by fixed-point reds.  `workspace` holds `need`
// bytes laid out as msda_backward_workspace_bytes describes.  Writes every element of grad_value.
int det_backward(cudaStream_t st, const Dims& d, int dtype, unsigned flags, const void* grad_output, const void* value,
                 const DetSource& src, void* grad_value, void* grad_sampling_loc, void* grad_attn_weight,
                 void* workspace, size_t need) {
  const void* sampling_loc = src.loc;
  const void* attn_weight = src.w;
  const int64_t* spatial_shapes = src.shapes;
  const int64_t* level_start_index = src.lsi;
  const msda::FusedArgs dcn = src.dcn ? *src.dcn : msda::FusedArgs{};
  const int64_t nv = d.n_value(), n_out = d.rows() * d.D, n_pts = d.n_points();
  const bool sorted = det_sorted_ok(d, dtype, flags);
  const DetLayout lay = sorted ? det_layout(d) : DetLayout{};
  char* ws = static_cast<char*>(workspace);
  auto* acc = reinterpret_cast<unsigned long long*>(ws + (sorted ? lay.off_acc : 0));
  auto* amax = reinterpret_cast<unsigned*>(ws + (sorted ? lay.off_misc : (size_t)nv * 8));
  auto* scale = reinterpret_cast<msda::DetScale*>(reinterpret_cast<char*>(amax) + 16);
  if (sorted) {   // zero the bins, cursors, {amax, scale} and the accumulators; entries are fully overwritten
    MSDA_CUDA(cudaMemsetAsync(ws, 0, lay.off_sums, st));
    MSDA_CUDA(cudaMemsetAsync(ws + lay.off_misc, 0, lay.total - lay.off_misc, st));
  } else {
    MSDA_CUDA(cudaMemsetAsync(workspace, 0, need, st));
  }
  // The fixed-point scale comes from max |grad_out| x max |weight|.  On the sorted route the backward kernel that
  // files the entries reads both tensors anyway and takes the two maxima itself (EmitArgs::amax); the scale is only
  // needed by the reduction that follows it.  Every other route scatters with the scale and takes them up front.
#ifndef MSDA_DET_AMAX_IN_EMIT
#define MSDA_DET_AMAX_IN_EMIT 1
#endif
  const bool amax_in_emit = MSDA_DET_AMAX_IN_EMIT && sorted && !(flags & MSDA_FLAG_DET_SEPARATE_FILL);
  const int g_out = grid_for(n_out, 256, 148 * 8), g_pts = grid_for(n_pts, 256, 148 * 8);
  if (!amax_in_emit) {
    if (int s = with_types<ValueTags>(dtype, [&](auto t) {
          using VT = typename decltype(t)::VT;
          using AT = typename decltype(t)::AT;
          msda::msda_amax_kernel<VT><<<g_out, 256, 0, st>>>((const VT*)grad_output, n_out, amax);
          count_launch();
          msda::msda_amax_kernel<AT><<<g_pts, 256, 0, st>>>((const AT*)attn_weight, n_pts, amax + 1);
          count_launch();
          msda::msda_det_scale_kernel<<<1, 1, 0, st>>>(amax, scale, std::is_same_v<VT, double> ? 44 : 38);
          return launched();
        }))
      return s;
  }
  if (sorted) {
    // sorted segment reduction (msda_det.cuh): count -> scan -> fill -> gather; no atomics on grad_value
    int* bins = reinterpret_cast<int*>(ws);
    int* cursor = reinterpret_cast<int*>(ws + lay.off_cursor);
    int* sums = reinterpret_cast<int*>(ws + lay.off_sums);
    int4* entries = reinterpret_cast<int4*>(ws + lay.off_entries);
    const float* loc = static_cast<const float*>(sampling_loc);
    const float* w = static_cast<const float*>(attn_weight);
    const int g_bin = grid_for(n_pts, 256, 148 * 32);
    if (src.dcn)
      msda::det_bin_kernel<false, msda::kPreDcn><<<g_bin, 256, 0, st>>>(loc, w, spatial_shapes, level_start_index, d.H,
                                                                       d.L, d.Q, d.P, n_pts, bins, nullptr, nullptr, dcn);
    else
      msda::det_bin_kernel<false><<<g_bin, 256, 0, st>>>(loc, w, spatial_shapes, level_start_index, d.H, d.L, d.Q, d.P,
                                                         n_pts, bins, nullptr, nullptr, dcn);
    count_launch();
    msda::det_scan_block_kernel<<<(unsigned)lay.scan_blocks, 256, 0, st>>>(bins, bins, sums, lay.n_scan);
    count_launch();
    msda::det_scan_sums_kernel<<<1, 1024, 0, st>>>(sums, (int)lay.scan_blocks);
    count_launch();
    msda::det_scan_add_kernel<<<(unsigned)lay.scan_blocks, 256, 0, st>>>(bins, sums, lay.n_scan);
    if (int s = launched()) return s;
    // entries are filed by the backward kernel itself (ACC = EmitEntries): the lane that has just built a point's
    // record takes the cursor atomic and writes the 16-byte entry, so the separate fill pass (det_bin_kernel<true>:
    // re-read of every location / weight + the coordinate arithmetic a second time) is gone
    auto emit = [&](float* wamax, int64_t* n_warps) {
      if (src.dcn)
        return bwd_dcn_emit(st, d, dtype, grad_output, value, sampling_loc, attn_weight, grad_sampling_loc,
                            grad_attn_weight, cursor, bins, entries, wamax, n_warps, dcn);
      return bwd_fast_emit(st, d, dtype, grad_output, value, spatial_shapes, level_start_index, sampling_loc,
                           attn_weight, grad_sampling_loc, grad_attn_weight, cursor, bins, entries, wamax, n_warps);
    };
    if (flags & MSDA_FLAG_DET_SEPARATE_FILL) {
      if (src.dcn)
        msda::det_bin_kernel<true, msda::kPreDcn><<<g_bin, 256, 0, st>>>(loc, w, spatial_shapes, level_start_index, d.H,
                                                                        d.L, d.Q, d.P, n_pts, cursor, bins, entries, dcn);
      else
        msda::det_bin_kernel<true><<<g_bin, 256, 0, st>>>(loc, w, spatial_shapes, level_start_index, d.H, d.L, d.Q, d.P,
                                                          n_pts, cursor, bins, entries, dcn);
      if (int s = launched()) return s;
      if (int s2 = src.dcn ? bwd_dcn_noscatter(st, d, dtype, grad_output, value, sampling_loc, attn_weight,
                                               grad_sampling_loc, grad_attn_weight, dcn)
                           : bwd_fast_noscatter(st, d, dtype, grad_output, value, spatial_shapes, level_start_index,
                                                sampling_loc, attn_weight, grad_sampling_loc, grad_attn_weight))
        return s2;
    } else if (amax_in_emit) {
      // the kernel leaves two maxima per warp; reducing those short arrays replaces the sweeps over grad_out / weights
      float* wamax = reinterpret_cast<float*>(ws + lay.off_wamax);
      int64_t n_warps = 0;
      if (int s2 = emit(wamax, &n_warps)) return s2;
      const int g_w = grid_for(n_warps, 256, 148 * 8);
      msda::msda_amax_kernel<float><<<g_w, 256, 0, st>>>(wamax, n_warps, amax);
      count_launch();
      msda::msda_amax_kernel<float><<<g_w, 256, 0, st>>>(wamax + n_warps, n_warps, amax + 1);
      count_launch();
      msda::msda_det_scale_kernel<<<1, 1, 0, st>>>(amax, scale, 38);   // sorted route: float / bf16 / f16 only
      if (int s = launched()) return s;
    } else if (int s2 = emit(nullptr, nullptr)) {
      return s2;
    }
    return with_types<FastTags>(dtype, [&](auto t) {
      using VT = typename decltype(t)::VT;
      if (!det_dense(d))
        return det_gather<VT>(st, d, grad_output, entries, bins, spatial_shapes, level_start_index, scale, grad_value);
      if (int s = det_cell_reduce<VT>(st, d, grad_output, entries, bins, lay.bins, spatial_shapes, level_start_index,
                                      scale, acc))
        return s;
      return det_finalize<VT>(st, acc, grad_value, nv, scale);
    });
  }
  return with_types<ValueTags>(dtype, [&](auto t) {
    using VT = typename decltype(t)::VT;
    using AT = typename decltype(t)::AT;
    int s;
    if (src.dcn)
      s = bwd_dcn_det(st, d, dtype, grad_output, value, sampling_loc, attn_weight, acc, grad_sampling_loc,
                      grad_attn_weight, scale, dcn);
    else if (fast_ok(d, dtype, flags))
      s = bwd_fast_det(st, d, dtype, grad_output, value, spatial_shapes, level_start_index, sampling_loc, attn_weight,
                       acc, grad_sampling_loc, grad_attn_weight, scale);
    else
      s = bwd_generic<VT, AT, unsigned long long>(st, d, grad_output, value, spatial_shapes, level_start_index,
                                                  sampling_loc, attn_weight, acc, grad_sampling_loc, grad_attn_weight,
                                                  scale);
    if (s != MSDA_OK) return s;
    return det_finalize<VT>(st, acc, grad_value, nv, scale);
  });
}

}  // namespace

// ============================================================================================
extern "C" {

int msda_abi_version(void) { return MSDA_ABI_VERSION; }

unsigned msda_build_config(void) {
  unsigned c = 0;
#ifdef MSDA_EXPERIMENTS
  c |= MSDA_BUILD_EXPERIMENTS;
#endif
#ifdef MSDA_EXP_SLIM
  c |= MSDA_BUILD_SLIM;
#endif
  return c;
}

uint64_t msda_kernel_launch_count(void) { return g_launches.load(std::memory_order_relaxed); }

unsigned msda_debug_fastdiv(unsigned n, unsigned d) { return msda::fastdiv(n, msda::fastdiv_make(d)); }

const char* msda_last_error_message(void) { return g_err; }

const char* msda_status_string(int status) {
  switch (status) {
    case MSDA_OK: return "MSDA_OK";
    case MSDA_ERR_INVALID_ARGUMENT: return "MSDA_ERR_INVALID_ARGUMENT";
    case MSDA_ERR_UNSUPPORTED: return "MSDA_ERR_UNSUPPORTED";
    case MSDA_ERR_WORKSPACE: return "MSDA_ERR_WORKSPACE";
    case MSDA_ERR_CUDA: return "MSDA_ERR_CUDA";
    default: return "MSDA_ERR_UNKNOWN";
  }
}

const char* msda_dispatch_name(int channels, int num_levels, int num_point, int spatial_size, int num_heads,
                               int dtype, unsigned flags, int backward) {
  Dims d{1, spatial_size, num_heads, channels, num_levels, 1, num_point};
  static thread_local char name[64];
  const char* dt = dtype == MSDA_F64 ? "f64" : (dtype == MSDA_BF16 ? "bf16" : (dtype == MSDA_F16 ? "f16" : "f32"));
  if (fast_ok(d, dtype, flags))
    snprintf(name, sizeof(name), "%s_fast_d%d_%s", backward ? "bwd" : "fwd", channels, dt);
  else
    snprintf(name, sizeof(name), "%s_generic_%s", backward ? "bwd" : "fwd", dt);
  return name;
}

int msda_forward(void* stream, const void* value, const int64_t* spatial_shapes, const int64_t* level_start_index,
                 const void* sampling_loc, const void* attn_weight, int batch, int spatial_size, int num_heads,
                 int channels, int num_levels, int num_query, int num_point, void* output, int dtype,
                 unsigned flags) {
  g_err[0] = 0;
  const Dims d{batch, spatial_size, num_heads, channels, num_levels, num_query, num_point};
  if (int s = check_dims(d, dtype)) return s;
  if (d.rows() * d.D == 0) return MSDA_OK;  // nothing to write (the reference would launch a 0-block grid, cuh:942)
  if (!output) return fail(MSDA_ERR_INVALID_ARGUMENT, "output is null");
  if (int s = check_alignment({{"value", value}, {"sampling_loc", sampling_loc}, {"attn_weight", attn_weight},
                               {"output", output}}))
    return s;
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  if (d.n_points() == 0 || d.S == 0) {  // no samples: the sum over an empty set
    DeviceGuard g;
    MSDA_CUDA(g.enter(output));
    MSDA_CUDA(cudaMemsetAsync(output, 0, (size_t)(d.rows() * d.D) * elem_size(dtype), st));
    return MSDA_OK;
  }
  if (!value || !spatial_shapes || !level_start_index || !sampling_loc || !attn_weight)
    return fail(MSDA_ERR_INVALID_ARGUMENT, "null tensor pointer");
  DeviceGuard guard;
  MSDA_CUDA(guard.enter(value));
  if (fast_ok(d, dtype, flags))
    return fwd_fast(st, d, dtype, flags, value, spatial_shapes, level_start_index, sampling_loc, attn_weight, output);
  return with_types<ValueTags>(dtype, [&](auto t) {
    using VT = typename decltype(t)::VT;
    using AT = typename decltype(t)::AT;
    return fwd_generic<VT, AT>(st, d, value, spatial_shapes, level_start_index, sampling_loc, attn_weight, output);
  });
}

size_t msda_backward_workspace_bytes(int batch, int spatial_size, int num_heads, int channels, int num_levels,
                                     int num_query, int num_point, int dtype, unsigned flags) {
  (void)num_levels; (void)num_query; (void)num_point;
  dtype = fused_value_dtype(dtype);   // the autocast tags need what their value dtype needs
  if (batch <= 0 || spatial_size <= 0 || num_heads <= 0 || channels <= 0) return 0;
  const size_t n_value = (size_t)batch * spatial_size * num_heads * channels;
  if (flags & MSDA_FLAG_DETERMINISTIC) {
    const Dims d{batch, spatial_size, num_heads, channels, num_levels, num_query, num_point};
    if (det_sorted_ok(d, dtype, flags)) return det_layout(d).total;   // bins, cursors, scan sums, entries
    return n_value * sizeof(long long) + 64;   // 64-bit fixed-point accumulators + {amax bits x2, DetScale}
  }
  // bf16 / f16 grad_value is accumulated in float and converted at the end
  if (two_byte(dtype)) return n_value * sizeof(float);
  return 0;
}

int msda_backward(void* stream, const void* grad_output, const void* value, const int64_t* spatial_shapes,
                  const int64_t* level_start_index, const void* sampling_loc, const void* attn_weight, int batch,
                  int spatial_size, int num_heads, int channels, int num_levels, int num_query, int num_point,
                  void* grad_value, void* grad_sampling_loc, void* grad_attn_weight, void* workspace,
                  size_t workspace_bytes, int dtype, unsigned flags) {
  g_err[0] = 0;
  const Dims d{batch, spatial_size, num_heads, channels, num_levels, num_query, num_point};
  if (int s = check_dims(d, dtype)) return s;
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  const size_t es = elem_size(dtype);
  const size_t ls = dtype == MSDA_F64 ? 8 : 4;
  if (d.n_value() == 0 && d.n_points() == 0) return MSDA_OK;
  if (int s = check_alignment({{"grad_output", grad_output}, {"value", value}, {"sampling_loc", sampling_loc},
                               {"attn_weight", attn_weight}, {"grad_value", grad_value},
                               {"grad_sampling_loc", grad_sampling_loc}, {"grad_attn_weight", grad_attn_weight},
                               {"workspace", workspace}}))
    return s;
  if ((flags & MSDA_FLAG_NO_GRAD_VALUE) && d.n_value() != 0 && d.n_points() != 0 && fast_ok(d, dtype, flags)) {
    // grad_value not wanted: the regular kernel with the scatter compiled out (no zero-fill, no workspace)
    if (!grad_output || !value || !spatial_shapes || !level_start_index || !sampling_loc || !attn_weight ||
        !grad_sampling_loc || !grad_attn_weight)
      return fail(MSDA_ERR_INVALID_ARGUMENT, "null tensor pointer");
    DeviceGuard guard_ns;
    MSDA_CUDA(guard_ns.enter(value));
    return bwd_fast_noscatter(st, d, dtype, grad_output, value, spatial_shapes, level_start_index, sampling_loc,
                              attn_weight, grad_sampling_loc, grad_attn_weight);
  }
  const void* anchor = d.n_value() ? grad_value : grad_attn_weight;
  if (!anchor) return fail(MSDA_ERR_INVALID_ARGUMENT, "gradient output pointer is null");
  DeviceGuard guard;
  MSDA_CUDA(guard.enter(anchor));
  const bool det = (flags & MSDA_FLAG_DETERMINISTIC) != 0;
  const bool have_samples = d.n_points() != 0 && d.n_value() != 0;
  // zero-fill grad_value -- unless a later pass writes every element anyway: the deterministic finalize / gather,
  // or the float -> bf16 / f16 conversion of the workspace accumulators
  const bool overwritten = have_samples && d.D != 0 && (det || two_byte(dtype));
  if (d.n_value() && !overwritten) {
    if (!grad_value) return fail(MSDA_ERR_INVALID_ARGUMENT, "grad_value is null");
    MSDA_CUDA(cudaMemsetAsync(grad_value, 0, (size_t)d.n_value() * es, st));
  }
  if (d.n_points() == 0) return MSDA_OK;
  if (!grad_sampling_loc || !grad_attn_weight) return fail(MSDA_ERR_INVALID_ARGUMENT, "grad_loc / grad_w is null");
  if (d.n_value() == 0 || d.D == 0) {  // nothing to sample from: all gradients are zero
    MSDA_CUDA(cudaMemsetAsync(grad_sampling_loc, 0, (size_t)d.n_points() * 2 * ls, st));
    MSDA_CUDA(cudaMemsetAsync(grad_attn_weight, 0, (size_t)d.n_points() * ls, st));
    return MSDA_OK;
  }
  if (!grad_output || !value || !spatial_shapes || !level_start_index || !sampling_loc || !attn_weight || !grad_value)
    return fail(MSDA_ERR_INVALID_ARGUMENT, "null tensor pointer");
  const size_t need = msda_backward_workspace_bytes(batch, spatial_size, num_heads, channels, num_levels, num_query,
                                                    num_point, dtype, flags);
  if (int s = check_workspace(workspace, workspace_bytes, need)) return s;
  if (det) {
    const DetSource src{sampling_loc, attn_weight, spatial_shapes, level_start_index, nullptr};
    return det_backward(st, d, dtype, flags, grad_output, value, src, grad_value, grad_sampling_loc, grad_attn_weight,
                        workspace, need);
  }

  float* gv32 = static_cast<float*>(grad_value);
  if (two_byte(dtype)) {
    gv32 = static_cast<float*>(workspace);
    MSDA_CUDA(cudaMemsetAsync(gv32, 0, need, st));
  }

  int s;
  if (fast_ok(d, dtype, flags)) {
    if (fold_applies(d, dtype, flags))
      s = bwd_fold(st, d, dtype, grad_output, value, spatial_shapes, level_start_index, sampling_loc, attn_weight, gv32,
                   grad_sampling_loc, grad_attn_weight, nullptr);
    else
      s = bwd_fast(st, d, dtype, flags, grad_output, value, spatial_shapes, level_start_index, sampling_loc,
                   attn_weight, gv32, grad_sampling_loc, grad_attn_weight);
  } else {
    // grad_value accumulates in AT: float (the workspace for bf16 / f16 values), double for float64
    s = with_types<ValueTags>(dtype, [&](auto t) {
      using VT = typename decltype(t)::VT;
      using AT = typename decltype(t)::AT;
      return bwd_generic<VT, AT, AT>(st, d, grad_output, value, spatial_shapes, level_start_index, sampling_loc,
                                     attn_weight, reinterpret_cast<AT*>(gv32), grad_sampling_loc, grad_attn_weight);
    });
  }
  if (s != MSDA_OK) return s;
  if (two_byte(dtype)) return cast_from_f32(st, gv32, grad_value, d.n_value(), dtype);
  return MSDA_OK;
}

int msda_fused_supported(int channels, int num_levels, int num_point, int spatial_size, int num_heads, int dtype,
                         unsigned flags) {
  const Dims d{1, spatial_size, num_heads, channels, num_levels, 1, num_point};
  return fast_ok(d, fused_value_dtype(dtype), flags) && !(flags & MSDA_FLAG_DETERMINISTIC) ? 1 : 0;
}

int msda_fused_forward(void* stream, const void* value, const int64_t* spatial_shapes,
                       const int64_t* level_start_index, const void* sampling_offsets, const void* attn_logits,
                       const float* reference_points, int ref_dim, const uint8_t* value_padding_mask, int batch,
                       int spatial_size, int num_heads, int channels, int num_levels, int num_query, int num_point,
                       void* output, int dtype, unsigned flags) {
  g_err[0] = 0;
  const Dims d{batch, spatial_size, num_heads, channels, num_levels, num_query, num_point};
  if (int s = check_dims(d, fused_value_dtype(dtype))) return s;
  if (ref_dim != 2 && ref_dim != 4) return fail(MSDA_ERR_INVALID_ARGUMENT, "ref_dim must be 2 or 4, got %d", ref_dim);
  if (d.rows() * d.D == 0) return MSDA_OK;
  if (!msda_fused_supported(channels, num_levels, num_point, spatial_size, num_heads, dtype, flags) || d.S == 0)
    return fail(MSDA_ERR_UNSUPPORTED, "fused path needs D in {16,32,64,128}, float/bf16/f16 value, L<=16, 1<=L*P<=64");
  if (!value || !spatial_shapes || !level_start_index || !sampling_offsets || !attn_logits || !reference_points ||
      !output)
    return fail(MSDA_ERR_INVALID_ARGUMENT, "null tensor pointer");
  if (int s = check_alignment({{"value", value}, {"sampling_offsets", sampling_offsets}, {"attn_logits", attn_logits},
                               {"reference_points", reference_points}, {"output", output}}))
    return s;
  DeviceGuard guard;
  MSDA_CUDA(guard.enter(value));
  const msda::FusedArgs fa = module_args(reference_points, ref_dim, num_point, value_padding_mask);
  return fwd_fused(static_cast<cudaStream_t>(stream), d, dtype, value, spatial_shapes, level_start_index,
                   sampling_offsets, attn_logits, output, fa);
}

int msda_fused_backward(void* stream, const void* grad_output, const void* value, const int64_t* spatial_shapes,
                        const int64_t* level_start_index, const void* sampling_offsets, const void* attn_logits,
                        const float* reference_points, int ref_dim, const uint8_t* value_padding_mask, int batch,
                        int spatial_size, int num_heads, int channels, int num_levels, int num_query, int num_point,
                        void* grad_value, void* grad_offsets, void* grad_logits, void* workspace,
                        size_t workspace_bytes, int dtype, unsigned flags) {
  g_err[0] = 0;
  const Dims d{batch, spatial_size, num_heads, channels, num_levels, num_query, num_point};
  const int vdt = fused_value_dtype(dtype);   // dtype itself selects the kernels (16-bit offsets / logits or not)
  if (int s = check_dims(d, vdt)) return s;
  if (ref_dim != 2 && ref_dim != 4) return fail(MSDA_ERR_INVALID_ARGUMENT, "ref_dim must be 2 or 4, got %d", ref_dim);
  if (!msda_fused_supported(channels, num_levels, num_point, spatial_size, num_heads, dtype, flags) ||
      d.n_value() == 0 || d.n_points() == 0)
    return fail(MSDA_ERR_UNSUPPORTED, "fused path needs a non-empty problem, D in {16,32,64,128}, float/bf16/f16 value");
  if (!grad_output || !value || !spatial_shapes || !level_start_index || !sampling_offsets || !attn_logits ||
      !reference_points || !grad_value || !grad_offsets || !grad_logits)
    return fail(MSDA_ERR_INVALID_ARGUMENT, "null tensor pointer");
  if (int s = check_alignment({{"grad_output", grad_output}, {"value", value}, {"sampling_offsets", sampling_offsets},
                               {"attn_logits", attn_logits}, {"reference_points", reference_points},
                               {"grad_value", grad_value}, {"grad_offsets", grad_offsets}, {"grad_logits", grad_logits},
                               {"workspace", workspace}}))
    return s;
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  DeviceGuard guard;
  MSDA_CUDA(guard.enter(value));
  const size_t need = msda_backward_workspace_bytes(batch, spatial_size, num_heads, channels, num_levels, num_query,
                                                    num_point, dtype, flags);
  if (int s = check_workspace(workspace, workspace_bytes, need)) return s;
  float* gv32 = static_cast<float*>(grad_value);
  if (two_byte(vdt)) gv32 = static_cast<float*>(workspace);
  MSDA_CUDA(cudaMemsetAsync(gv32, 0, (size_t)d.n_value() * sizeof(float), st));
  const msda::FusedArgs fa = module_args(reference_points, ref_dim, num_point, value_padding_mask);
  int s;
  if (fold_applies(d, dtype, flags))
    s = bwd_fold(st, d, dtype, grad_output, value, spatial_shapes, level_start_index, sampling_offsets, attn_logits,
                 gv32, grad_offsets, grad_logits, &fa);
  else
    s = bwd_fused(st, d, dtype, grad_output, value, spatial_shapes, level_start_index, sampling_offsets, attn_logits,
                  gv32, grad_offsets, grad_logits, fa);
  if (s != MSDA_OK) return s;
  if (two_byte(vdt)) return cast_from_f32(st, gv32, grad_value, d.n_value(), vdt);
  return MSDA_OK;
}

namespace {
// Checks shared by msda_packed_forward / _backward.  *d becomes the problem the kernels are launched for: B images,
// S / Q = the largest image's value / query count (grid and 32-bit in-image offsets).  Returns MSDA_OK, an error, or
// -1 for an empty problem (nothing to do).
int packed_setup(int batch, int total_value, int num_heads, int channels, int num_levels, int total_query,
                 int num_point, int max_image_value, int max_image_query, int ref_dim, int dtype, unsigned flags,
                 Dims* d) {
  *d = Dims{batch, max_image_value, num_heads, channels, num_levels, max_image_query, num_point};
  if (int s = check_dims(*d, fused_value_dtype(dtype))) return s;
  if (total_value < 0 || total_query < 0)
    return fail(MSDA_ERR_INVALID_ARGUMENT, "negative token count (T_v=%d T_q=%d)", total_value, total_query);
  if (ref_dim != 2 && ref_dim != 4) return fail(MSDA_ERR_INVALID_ARGUMENT, "ref_dim must be 2 or 4, got %d", ref_dim);
  if (batch == 0 || total_query == 0 || (int64_t)num_heads * channels == 0) return -1;
  if (max_image_query > total_query || max_image_value > total_value ||
      (int64_t)max_image_query * batch < total_query || (int64_t)max_image_value * batch < total_value)
    return fail(MSDA_ERR_INVALID_ARGUMENT, "largest image (%d queries, %d values) does not fit the totals (%d, %d)",
                max_image_query, max_image_value, total_query, total_value);
  if (!fast_ok(*d, fused_value_dtype(dtype), flags & ~MSDA_FLAG_DETERMINISTIC) ||
      (int64_t)max_image_query * num_heads >= ((int64_t)1 << 31))
    return fail(MSDA_ERR_UNSUPPORTED, "packed path needs D in {16,32,64,128}, float/bf16/f16 value, L<=16, 1<=L*P<=64");
  return MSDA_OK;
}
}  // namespace

size_t msda_packed_backward_workspace_bytes(int total_value, int num_heads, int channels, int dtype, unsigned flags) {
  (void)flags;
  if (total_value <= 0 || num_heads <= 0 || channels <= 0) return 0;
  // bf16 / f16 grad_value is accumulated in float and converted at the end
  return two_byte(fused_value_dtype(dtype)) ? (size_t)total_value * num_heads * channels * sizeof(float) : 0;
}

int msda_packed_forward(void* stream, const void* value, const int64_t* spatial_shapes, const int64_t* image_meta,
                        const void* sampling_offsets, const void* attn_logits, const float* reference_points,
                        int ref_dim, int batch, int total_value, int num_heads, int channels, int num_levels,
                        int total_query, int num_point, int max_image_value, int max_image_query, void* output,
                        int dtype, unsigned flags) {
  g_err[0] = 0;
  Dims d;
  const int s0 = packed_setup(batch, total_value, num_heads, channels, num_levels, total_query, num_point,
                              max_image_value, max_image_query, ref_dim, dtype, flags, &d);
  if (s0 == -1) return MSDA_OK;
  if (s0 != MSDA_OK) return s0;
  if (!output) return fail(MSDA_ERR_INVALID_ARGUMENT, "output is null");
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  if (total_value == 0) {   // no valid pixel anywhere: every sample reads zeros
    DeviceGuard g;
    MSDA_CUDA(g.enter(output));
    MSDA_CUDA(cudaMemsetAsync(output, 0, (size_t)total_query * num_heads * channels * elem_size(fused_value_dtype(dtype)),
                              st));
    return MSDA_OK;
  }
  if (!value || !spatial_shapes || !image_meta || !sampling_offsets || !attn_logits || !reference_points)
    return fail(MSDA_ERR_INVALID_ARGUMENT, "null tensor pointer");
  if (int s = check_alignment({{"value", value}, {"image_meta", image_meta}, {"sampling_offsets", sampling_offsets},
                               {"attn_logits", attn_logits}, {"reference_points", reference_points},
                               {"output", output}}))
    return s;
  DeviceGuard guard;
  MSDA_CUDA(guard.enter(value));
  const msda::FusedArgs fa = module_args(reference_points, ref_dim, num_point, nullptr);
  return fwd_packed(st, d, dtype, value, spatial_shapes, image_meta, sampling_offsets, attn_logits, output, fa);
}

int msda_packed_backward(void* stream, const void* grad_output, const void* value, const int64_t* spatial_shapes,
                         const int64_t* image_meta, const void* sampling_offsets, const void* attn_logits,
                         const float* reference_points, int ref_dim, int batch, int total_value, int num_heads,
                         int channels, int num_levels, int total_query, int num_point, int max_image_value,
                         int max_image_query, void* grad_value, void* grad_offsets, void* grad_logits,
                         void* workspace, size_t workspace_bytes, int dtype, unsigned flags) {
  g_err[0] = 0;
  if (flags & MSDA_FLAG_DETERMINISTIC)
    return fail(MSDA_ERR_UNSUPPORTED, "the packed backward has no deterministic form (float reds)");
  Dims d;
  const int s0 = packed_setup(batch, total_value, num_heads, channels, num_levels, total_query, num_point,
                              max_image_value, max_image_query, ref_dim, dtype, flags, &d);
  if (s0 == -1) return MSDA_OK;
  if (s0 != MSDA_OK) return s0;
  if (!grad_offsets || !grad_logits) return fail(MSDA_ERR_INVALID_ARGUMENT, "gradient output pointer is null");
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  const int64_t n_points = (int64_t)total_query * num_heads * num_levels * num_point;
  if (total_value == 0) {   // nothing was sampled: every gradient is zero
    DeviceGuard g;
    MSDA_CUDA(g.enter(grad_offsets));
    MSDA_CUDA(cudaMemsetAsync(grad_offsets, 0, (size_t)n_points * 2 * aux_size(dtype), st));
    MSDA_CUDA(cudaMemsetAsync(grad_logits, 0, (size_t)n_points * aux_size(dtype), st));
    return MSDA_OK;
  }
  if (!grad_output || !value || !spatial_shapes || !image_meta || !sampling_offsets || !attn_logits ||
      !reference_points || !grad_value)
    return fail(MSDA_ERR_INVALID_ARGUMENT, "null tensor pointer");
  if (int s = check_alignment({{"grad_output", grad_output}, {"value", value}, {"image_meta", image_meta},
                               {"sampling_offsets", sampling_offsets}, {"attn_logits", attn_logits},
                               {"reference_points", reference_points}, {"grad_value", grad_value},
                               {"grad_offsets", grad_offsets}, {"grad_logits", grad_logits},
                               {"workspace", workspace}}))
    return s;
  const int vdt = fused_value_dtype(dtype);
  const size_t need = msda_packed_backward_workspace_bytes(total_value, num_heads, channels, dtype, flags);
  if (int s = check_workspace(workspace, workspace_bytes, need)) return s;
  DeviceGuard guard;
  MSDA_CUDA(guard.enter(value));
  const int64_t n_value = (int64_t)total_value * num_heads * channels;
  float* gv32 = two_byte(vdt) ? static_cast<float*>(workspace) : static_cast<float*>(grad_value);
  MSDA_CUDA(cudaMemsetAsync(gv32, 0, (size_t)n_value * sizeof(float), st));
  const msda::FusedArgs fa = module_args(reference_points, ref_dim, num_point, nullptr);
  const int s = bwd_packed(st, d, dtype, grad_output, value, spatial_shapes, image_meta, sampling_offsets, attn_logits,
                           gv32, grad_offsets, grad_logits, fa);
  if (s != MSDA_OK) return s;
  if (two_byte(vdt)) return cast_from_f32(st, gv32, grad_value, n_value, vdt);
  return MSDA_OK;
}

namespace {
// DCNv3 as an MSDeformAttn problem: value = input [N, H_in*W_in, G, C], one level, Q = H_out*W_out, P = K.
int dcn_setup(int kernel_h, int kernel_w, int stride_h, int stride_w, int pad_h, int pad_w, int dilation_h,
              int dilation_w, int group, int group_channels, float offset_scale, int batch, int height_in,
              int width_in, int height_out, int width_out, int dtype, Dims* d, msda::FusedArgs* fa) {
  if (kernel_h < 1 || kernel_w < 1 || stride_h < 1 || stride_w < 1 || dilation_h < 1 || dilation_w < 1 || pad_h < 0 ||
      pad_w < 0 || batch < 0 || height_in < 0 || width_in < 0 || height_out < 0 || width_out < 0 || group < 1 ||
      group_channels < 1)
    return fail(MSDA_ERR_INVALID_ARGUMENT, "dcnv3: bad geometry");
  *d = Dims{batch, height_in * width_in, group, group_channels, 1, height_out * width_out, kernel_h * kernel_w};
  if (dtype != MSDA_F32 && dtype != MSDA_BF16 && dtype != MSDA_F16)
    return fail(MSDA_ERR_UNSUPPORTED, "dcnv3: float32 / bfloat16 / float16 only");
  if (d->rows() * d->D != 0 && !fast_ok(*d, dtype, 0))
    return fail(MSDA_ERR_UNSUPPORTED,
                "dcnv3: needs group_channels in {16,32,64,128} and kernel_h*kernel_w <= 64 (got %d, %d)",
                group_channels, kernel_h * kernel_w);
  msda::FusedArgs a{};
  a.kernel_h = kernel_h; a.kernel_w = kernel_w; a.stride_h = stride_h; a.stride_w = stride_w;
  a.pad_h = pad_h; a.pad_w = pad_w; a.dil_h = dilation_h; a.dil_w = dilation_w;
  a.height_in = height_in; a.width_in = width_in; a.width_out = width_out > 0 ? width_out : 1;
  a.offset_scale = offset_scale;
  *fa = a;
  return MSDA_OK;
}

// the flags msda_dcnv3_backward honours; every other bit is ignored
constexpr unsigned kDcnDetFlags = MSDA_FLAG_DETERMINISTIC | MSDA_FLAG_DET_ATOMIC | MSDA_FLAG_DET_SEPARATE_FILL;
// deterministic workspace: the one-level table {H_in, W_in}, {0} (det_one_level_kernel) first, then the layout of the
// equivalent one-level msda_backward problem
constexpr size_t kDcnLevelSlot = 256;
}  // namespace

size_t msda_dcnv3_backward_workspace_bytes(int kernel_h, int kernel_w, int group, int group_channels, int batch,
                                           int height_in, int width_in, int height_out, int width_out, int dtype,
                                           unsigned flags) {
  dtype = fused_value_dtype(dtype);   // the autocast tags need what their value dtype needs
  if (batch <= 0 || height_in <= 0 || width_in <= 0 || group <= 0 || group_channels <= 0) return 0;
  const size_t n_value = (size_t)batch * height_in * width_in * group * group_channels;
  // empty problems (no output pixel, no kernel point) need what they need without the flag
  if ((flags & MSDA_FLAG_DETERMINISTIC) && height_out > 0 && width_out > 0 && kernel_h > 0 && kernel_w > 0)
    return kDcnLevelSlot + msda_backward_workspace_bytes(batch, height_in * width_in, group, group_channels, 1,
                                                         height_out * width_out, kernel_h * kernel_w, dtype,
                                                         flags & kDcnDetFlags);
  // bf16 / f16 grad_input is accumulated in float and converted at the end
  return two_byte(dtype) ? n_value * sizeof(float) : 0;
}

namespace {
// The body of msda_dcnv3_forward (softmax false: `w` = mask) and msda_dcnv3_fused_forward (softmax true: `w` = mask
// logits; dtype may be an autocast tag), after dcn_setup.
int dcn_forward(void* stream, const Dims& d, const msda::FusedArgs& fa, const void* input, const void* offset,
                const void* w, void* output, int dtype, bool softmax) {
  if (d.rows() * d.D == 0) return MSDA_OK;
  if (!output) return fail(MSDA_ERR_INVALID_ARGUMENT, "output is null");
  if (int s = check_alignment({{"input", input}, {"offset", offset}, {softmax ? "mask_logits" : "mask", w},
                               {"output", output}}))
    return s;
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  DeviceGuard guard;
  MSDA_CUDA(guard.enter(output));
  if (d.S == 0) {
    MSDA_CUDA(cudaMemsetAsync(output, 0, (size_t)(d.rows() * d.D) * elem_size(fused_value_dtype(dtype)), st));
    return MSDA_OK;
  }
  if (!input || !offset || !w) return fail(MSDA_ERR_INVALID_ARGUMENT, "null tensor pointer");
  return softmax ? fwd_dcn_softmax(st, d, dtype, input, offset, w, output, fa)
                 : fwd_dcn(st, d, dtype, input, offset, w, output, fa);
}

// The body of msda_dcnv3_backward (softmax false: `w` = mask, grad_w = its gradient) and msda_dcnv3_fused_backward
// (softmax true: `w` = mask logits, grad_w = their gradient; never with MSDA_FLAG_DETERMINISTIC; dtype may be an
// autocast tag), after dcn_setup.  `need` = msda_dcnv3_backward_workspace_bytes of the problem and flags.
int dcn_backward(void* stream, const Dims& d, const msda::FusedArgs& fa, const void* grad_output, const void* input,
                 const void* offset, const void* w, void* grad_input, void* grad_offset, void* grad_w,
                 void* workspace, size_t workspace_bytes, size_t need, int tag, unsigned flags, bool softmax) {
  const int dtype = fused_value_dtype(tag);   // the value dtype; `tag` selects the kernels
  const char* w_name = softmax ? "mask_logits" : "mask";
  const char* gw_name = softmax ? "grad_mask_logits" : "grad_mask";
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  if (d.n_value() == 0 && d.n_points() == 0) return MSDA_OK;
  const void* anchor = d.n_value() ? grad_input : (const void*)grad_w;
  if (!anchor) return fail(MSDA_ERR_INVALID_ARGUMENT, "gradient output pointer is null");
  if (int s = check_alignment({{"grad_output", grad_output}, {"input", input}, {"offset", offset}, {w_name, w},
                               {"grad_input", grad_input}, {"grad_offset", grad_offset}, {gw_name, grad_w},
                               {"workspace", workspace}}))
    return s;
  DeviceGuard guard;
  MSDA_CUDA(guard.enter(anchor));
  if (int s = check_workspace(workspace, workspace_bytes, need)) return s;
  if ((flags & MSDA_FLAG_DETERMINISTIC) && d.n_value() != 0 && d.n_points() != 0) {
    // bit-reproducible grad_input: the deterministic backward of the equivalent one-level problem, which writes every
    // element of grad_input in its own dtype (no float workspace, no zero-fill, no cast)
    if (!grad_input || !grad_offset || !grad_w || !grad_output || !input || !offset || !w)
      return fail(MSDA_ERR_INVALID_ARGUMENT, "null tensor pointer");
    char* ws = static_cast<char*>(workspace);
    int64_t* table = reinterpret_cast<int64_t*>(ws);
    if (det_sorted_ok(d, dtype, flags)) {   // the count / gather / cell-reduce kernels read the level table
      msda::det_one_level_kernel<<<1, 1, 0, st>>>(table, fa.height_in, fa.width_in);
      if (int s = launched()) return s;
    }
    const DetSource src{offset, w, table, table + 2, &fa};
    return det_backward(st, d, dtype, flags, grad_output, input, src, grad_input, grad_offset, grad_w,
                        ws + kDcnLevelSlot, need - kDcnLevelSlot);
  }
  float* gi32 = two_byte(dtype) ? static_cast<float*>(workspace) : static_cast<float*>(grad_input);
  if (d.n_value()) {
    if (!grad_input) return fail(MSDA_ERR_INVALID_ARGUMENT, "grad_input is null");
    MSDA_CUDA(cudaMemsetAsync(gi32, 0, (size_t)d.n_value() * sizeof(float), st));
    if (two_byte(dtype) && d.n_points() == 0)
      MSDA_CUDA(cudaMemsetAsync(grad_input, 0, (size_t)d.n_value() * 2, st));
  }
  if (d.n_points() == 0) return MSDA_OK;
  if (!grad_offset || !grad_w) return fail(MSDA_ERR_INVALID_ARGUMENT, "grad_offset / %s is null", gw_name);
  if (d.n_value() == 0) {   // nothing to sample: the output does not depend on the offsets or the mask (or its logits)
    MSDA_CUDA(cudaMemsetAsync(grad_offset, 0, (size_t)d.n_points() * 2 * aux_size(tag), st));
    MSDA_CUDA(cudaMemsetAsync(grad_w, 0, (size_t)d.n_points() * aux_size(tag), st));
    return MSDA_OK;
  }
  if (!grad_output || !input || !offset || !w) return fail(MSDA_ERR_INVALID_ARGUMENT, "null tensor pointer");
  if (int s = softmax ? bwd_dcn_softmax(st, d, tag, grad_output, input, offset, w, gi32, grad_offset, grad_w, fa)
                      : bwd_dcn(st, d, dtype, grad_output, input, offset, w, gi32, grad_offset, grad_w, fa))
    return s;
  if (two_byte(dtype)) return cast_from_f32(st, gi32, grad_input, d.n_value(), dtype);
  return MSDA_OK;
}
}  // namespace

int msda_dcnv3_forward(void* stream, const void* input, const float* offset, const float* mask, int kernel_h,
                       int kernel_w, int stride_h, int stride_w, int pad_h, int pad_w, int dilation_h, int dilation_w,
                       int group, int group_channels, float offset_scale, int batch, int height_in, int width_in,
                       int height_out, int width_out, void* output, int dtype, unsigned flags) {
  (void)flags;
  g_err[0] = 0;
  Dims d;
  msda::FusedArgs fa;
  if (int s = dcn_setup(kernel_h, kernel_w, stride_h, stride_w, pad_h, pad_w, dilation_h, dilation_w, group,
                        group_channels, offset_scale, batch, height_in, width_in, height_out, width_out, dtype, &d, &fa))
    return s;
  return dcn_forward(stream, d, fa, input, offset, mask, output, dtype, false);
}

int msda_dcnv3_backward(void* stream, const void* grad_output, const void* input, const float* offset,
                        const float* mask, int kernel_h, int kernel_w, int stride_h, int stride_w, int pad_h, int pad_w,
                        int dilation_h, int dilation_w, int group, int group_channels, float offset_scale, int batch,
                        int height_in, int width_in, int height_out, int width_out, void* grad_input,
                        float* grad_offset, float* grad_mask, void* workspace, size_t workspace_bytes, int dtype,
                        unsigned flags) {
  g_err[0] = 0;
  Dims d;
  msda::FusedArgs fa;
  if (int s = dcn_setup(kernel_h, kernel_w, stride_h, stride_w, pad_h, pad_w, dilation_h, dilation_w, group,
                        group_channels, offset_scale, batch, height_in, width_in, height_out, width_out, dtype, &d, &fa))
    return s;
  flags &= kDcnDetFlags;
  const size_t need = msda_dcnv3_backward_workspace_bytes(kernel_h, kernel_w, group, group_channels, batch, height_in,
                                                          width_in, height_out, width_out, dtype, flags);
  return dcn_backward(stream, d, fa, grad_output, input, offset, mask, grad_input, grad_offset, grad_mask, workspace,
                      workspace_bytes, need, dtype, flags, false);
}

int msda_dcnv3_fused_forward(void* stream, const void* input, const void* offset, const void* mask_logits,
                             int kernel_h, int kernel_w, int stride_h, int stride_w, int pad_h, int pad_w,
                             int dilation_h, int dilation_w, int group, int group_channels, float offset_scale,
                             int batch, int height_in, int width_in, int height_out, int width_out, void* output,
                             int dtype, unsigned flags) {
  (void)flags;
  g_err[0] = 0;
  Dims d;
  msda::FusedArgs fa;
  if (int s = dcn_setup(kernel_h, kernel_w, stride_h, stride_w, pad_h, pad_w, dilation_h, dilation_w, group,
                        group_channels, offset_scale, batch, height_in, width_in, height_out, width_out,
                        fused_value_dtype(dtype), &d, &fa))
    return s;
  return dcn_forward(stream, d, fa, input, offset, mask_logits, output, dtype, true);
}

int msda_dcnv3_fused_backward(void* stream, const void* grad_output, const void* input, const void* offset,
                              const void* mask_logits, int kernel_h, int kernel_w, int stride_h, int stride_w,
                              int pad_h, int pad_w, int dilation_h, int dilation_w, int group, int group_channels,
                              float offset_scale, int batch, int height_in, int width_in, int height_out,
                              int width_out, void* grad_input, void* grad_offset, void* grad_mask_logits,
                              void* workspace, size_t workspace_bytes, int dtype, unsigned flags) {
  g_err[0] = 0;
  Dims d;
  msda::FusedArgs fa;
  if (int s = dcn_setup(kernel_h, kernel_w, stride_h, stride_w, pad_h, pad_w, dilation_h, dilation_w, group,
                        group_channels, offset_scale, batch, height_in, width_in, height_out, width_out,
                        fused_value_dtype(dtype), &d, &fa))
    return s;
  // the float-red kernel is the only fused form: a caller that needs bit-reproducible gradients composes the softmax
  // around msda_dcnv3_backward (refused before any device work, empty problems included)
  if (flags & MSDA_FLAG_DETERMINISTIC)
    return fail(MSDA_ERR_UNSUPPORTED, "dcnv3 fused backward: no deterministic form (use msda_dcnv3_backward)");
  const size_t need = msda_dcnv3_backward_workspace_bytes(kernel_h, kernel_w, group, group_channels, batch, height_in,
                                                          width_in, height_out, width_out, dtype, 0u);
  return dcn_backward(stream, d, fa, grad_output, input, offset, mask_logits, grad_input, grad_offset,
                      grad_mask_logits, workspace, workspace_bytes, need, dtype, 0u, true);
}

namespace {
// Checks the deformable-convolution geometry and dtype tag (no device work) and fills `g`.
int dcnv2_setup(int batch, int channels, int height_in, int width_in, int height_out, int width_out, int kernel_h,
                int kernel_w, int stride_h, int stride_w, int pad_h, int pad_w, int dilation_h, int dilation_w,
                int groups, int deformable_groups, int dtype, Dcn2Dims* g) {
  if (batch < 0 || channels < 0 || height_in < 1 || width_in < 1 || kernel_h < 1 || kernel_w < 1 || stride_h < 1 ||
      stride_w < 1 || pad_h < 0 || pad_w < 0 || dilation_h < 1 || dilation_w < 1 || groups < 1 ||
      deformable_groups < 1)
    return fail(MSDA_ERR_INVALID_ARGUMENT, "dcnv2: bad geometry");
  if (channels % groups != 0 || channels % deformable_groups != 0)
    return fail(MSDA_ERR_INVALID_ARGUMENT, "dcnv2: channels (%d) must be divisible by groups (%d) and deformable_groups (%d)",
                channels, groups, deformable_groups);
  const int64_t ho = ((int64_t)height_in + 2 * pad_h - ((int64_t)dilation_h * (kernel_h - 1) + 1)) / stride_h + 1;
  const int64_t wo = ((int64_t)width_in + 2 * pad_w - ((int64_t)dilation_w * (kernel_w - 1) + 1)) / stride_w + 1;
  if (ho < 1 || wo < 1 || height_out != ho || width_out != wo)
    return fail(MSDA_ERR_INVALID_ARGUMENT, "dcnv2: output %dx%d, the geometry gives %lldx%lld", height_out, width_out,
                (long long)ho, (long long)wo);
  if (dtype != MSDA_F32 && dtype != MSDA_F64 && dtype != MSDA_BF16 && dtype != MSDA_F16 && dtype != MSDA_BF16_AUX16 &&
      dtype != MSDA_F16_AUX16)
    return fail(MSDA_ERR_INVALID_ARGUMENT, "unknown dtype tag %d", dtype);
  if (ho * wo * deformable_groups * kernel_h * kernel_w >= ((int64_t)1 << 31) ||
      (int64_t)height_in * width_in * channels >= ((int64_t)1 << 40))
    return fail(MSDA_ERR_UNSUPPORTED, "dcnv2: image too large");
  *g = Dcn2Dims{batch, channels, height_in, width_in, height_out, width_out, kernel_h, kernel_w, stride_h, stride_w,
                pad_h, pad_w, dilation_h, dilation_w, groups, deformable_groups};
  return MSDA_OK;
}
}  // namespace

size_t msda_dcnv2_col2im_workspace_bytes(int batch, int channels, int height_in, int width_in, int height_out,
                                         int width_out, int kernel_h, int kernel_w, int stride_h, int stride_w,
                                         int pad_h, int pad_w, int dilation_h, int dilation_w, int groups,
                                         int deformable_groups, int dtype, unsigned flags) {
  (void)flags;
  Dcn2Dims g;
  if (dcnv2_setup(batch, channels, height_in, width_in, height_out, width_out, kernel_h, kernel_w, stride_h, stride_w,
                  pad_h, pad_w, dilation_h, dilation_w, groups, deformable_groups, dtype, &g) != MSDA_OK)
    return 0;
  // bf16 / f16 grad_input is accumulated in float and converted at the end
  return two_byte(fused_value_dtype(dtype)) ? (size_t)g.n_input() * sizeof(float) : 0;
}

int msda_dcnv2_im2col(void* stream, const void* input, const void* offset, const void* mask, int batch, int channels,
                      int height_in, int width_in, int height_out, int width_out, int kernel_h, int kernel_w,
                      int stride_h, int stride_w, int pad_h, int pad_w, int dilation_h, int dilation_w, int groups,
                      int deformable_groups, void* columns, int dtype, unsigned flags) {
  g_err[0] = 0;
  Dcn2Dims g;
  if (int s = dcnv2_setup(batch, channels, height_in, width_in, height_out, width_out, kernel_h, kernel_w, stride_h,
                          stride_w, pad_h, pad_w, dilation_h, dilation_w, groups, deformable_groups, dtype, &g))
    return s;
  if (g.n_columns() == 0) return MSDA_OK;
  if (!input || !offset || !columns) return fail(MSDA_ERR_INVALID_ARGUMENT, "null tensor pointer");
  if (int s = check_alignment({{"input", input}, {"offset", offset}, {"mask", mask}, {"columns", columns}})) return s;
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  DeviceGuard guard;
  MSDA_CUDA(guard.enter(columns));
  return dcnv2_im2col(st, g, dtype, flags, input, offset, mask, columns);
}

int msda_dcnv2_col2im(void* stream, const void* grad_columns, const void* input, const void* offset, const void* mask,
                      int batch, int channels, int height_in, int width_in, int height_out, int width_out, int kernel_h,
                      int kernel_w, int stride_h, int stride_w, int pad_h, int pad_w, int dilation_h, int dilation_w,
                      int groups, int deformable_groups, void* grad_input, void* grad_offset, void* grad_mask,
                      void* workspace, size_t workspace_bytes, int dtype, unsigned flags) {
  g_err[0] = 0;
  Dcn2Dims g;
  if (int s = dcnv2_setup(batch, channels, height_in, width_in, height_out, width_out, kernel_h, kernel_w, stride_h,
                          stride_w, pad_h, pad_w, dilation_h, dilation_w, groups, deformable_groups, dtype, &g))
    return s;
  if (flags & MSDA_FLAG_DETERMINISTIC)
    return fail(MSDA_ERR_UNSUPPORTED, "dcnv2 col2im: no deterministic form (grad_input uses float reds)");
  if (g.n_points() == 0) return MSDA_OK;   // batch 0
  const int vdt = fused_value_dtype(dtype);
  const size_t aux = dtype == MSDA_F64 ? 8 : aux_size(dtype);
  if (!grad_offset || (mask && !grad_mask)) return fail(MSDA_ERR_INVALID_ARGUMENT, "grad_offset / grad_mask is null");
  if (g.n_input() != 0 && (!grad_columns || !input || !offset || !grad_input))
    return fail(MSDA_ERR_INVALID_ARGUMENT, "null tensor pointer");
  if (int s = check_alignment({{"grad_columns", grad_columns}, {"input", input}, {"offset", offset}, {"mask", mask},
                               {"grad_input", grad_input}, {"grad_offset", grad_offset},
                               {"grad_mask", mask ? grad_mask : nullptr}, {"workspace", workspace}}))
    return s;
  const size_t need = two_byte(vdt) ? (size_t)g.n_input() * sizeof(float) : 0;
  if (int s = check_workspace(workspace, workspace_bytes, need)) return s;
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  DeviceGuard guard;
  MSDA_CUDA(guard.enter(grad_offset));
  if (g.n_input() == 0) {   // no channels: the output does not depend on the offsets or the mask
    MSDA_CUDA(cudaMemsetAsync(grad_offset, 0, (size_t)g.n_points() * 2 * aux, st));
    if (mask) MSDA_CUDA(cudaMemsetAsync(grad_mask, 0, (size_t)g.n_points() * aux, st));
    return MSDA_OK;
  }
  void* acc = two_byte(vdt) ? workspace : grad_input;
  MSDA_CUDA(cudaMemsetAsync(acc, 0, (size_t)g.n_input() * (vdt == MSDA_F64 ? 8 : 4), st));
  if (int s = dcnv2_col2im(st, g, dtype, flags, grad_columns, input, offset, mask, acc, grad_offset, grad_mask))
    return s;
  if (two_byte(vdt)) return cast_from_f32(st, static_cast<const float*>(acc), grad_input, g.n_input(), vdt);
  return MSDA_OK;
}

int msda_debug_bookkeeping(void* stream, const float* sampling_loc, const int64_t* spatial_shapes,
                           const int64_t* level_start_index, int batch, int spatial_size, int num_heads, int channels,
                           int num_levels, int num_query, int num_point, int64_t* corner_offsets, float* frac) {
  g_err[0] = 0;
  const Dims d{batch, spatial_size, num_heads, channels, num_levels, num_query, num_point};
  if (int s = check_dims(d, MSDA_F32)) return s;
  if (d.n_points() == 0) return MSDA_OK;
  if (!sampling_loc || !spatial_shapes || !level_start_index || !corner_offsets || !frac)
    return fail(MSDA_ERR_INVALID_ARGUMENT, "null tensor pointer");
  DeviceGuard guard;
  MSDA_CUDA(guard.enter(sampling_loc));
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  if (fast_ok(d, MSDA_F32, 0))   // what the fast kernels index with (their own records, decoded)
    msda_fast_records_kernel<<<grid_for(d.n_points(), 256, 148 * 16), 256, 0, st>>>(
        sampling_loc, spatial_shapes, level_start_index, d.S, d.H, d.D, d.L, d.Q, d.P, d.n_points(), corner_offsets,
        frac);
  else
    msda::msda_bookkeeping_kernel<<<grid_for(d.n_points(), 256, 148 * 16), 256, 0, st>>>(
        sampling_loc, spatial_shapes, level_start_index, d.S, d.H, d.D, d.L, d.Q, d.P, d.n_points(), corner_offsets,
        frac);
  return launched();
}

}  // extern "C"
