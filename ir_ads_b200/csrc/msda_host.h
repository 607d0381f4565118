// msda_host.h -- internal host-side interface between the translation units of libmsda_b200.so.
// (The public C ABI is include/msda.h; nothing here is exported.)
//
// The library is split so that the kernel families compile in parallel:
//   msda_capi.cu     the extern "C" entry points, argument checks, generic + deterministic kernels
//   msda_fwd.cu      fast forward kernels (plain / fused module chain / DCNv3)
//   msda_bwd.cu      fast backward kernels, float reds (plain operator, all row orders)
//   msda_bwd_aux.cu  fast backward kernels: fixed-point reds, no-scatter, fused module chain, DCNv3
//   msda_fold.cu     encoder-form backward with on-SM folding of grad_value (msda_fold.cuh)
//   msda_dcnv2.cu    deformable convolution im2col / col2im (fast + generic)
//   msda_epilogue.cu fused residual add + LayerNorm
// Every launch site maps its runtime dtype tag and channel count onto template arguments with the dispatch templates
// below (with_types, with_chunk); the fast units add the point-count and row-order dispatch of msda_fast_launch.cuh.
#pragma once
#include "../../include/msda.h"

#include <cuda_bf16.h>
#include <cuda_fp16.h>
#include <cuda_runtime.h>
#include <stdint.h>

#include <initializer_list>
#include <type_traits>

#include "msda_fast.cuh"

namespace msda_host {

struct Dims {
  int B, S, H, D, L, Q, P;
  int64_t rows() const { return (int64_t)B * Q * H; }
  int64_t n_value() const { return (int64_t)B * S * H * D; }
  int64_t n_points() const { return rows() * L * P; }
};

// sets the calling thread's last-error message and returns `status`
int fail(int status, const char* fmt, ...) __attribute__((format(printf, 2, 3)));
int cuda_fail(cudaError_t e, const char* what);
void count_launch();

#define MSDA_CUDA(call)                                               \
  do {                                                                \
    cudaError_t e__ = (call);                                         \
    if (e__ != cudaSuccess) return ::msda_host::cuda_fail(e__, #call); \
  } while (0)

// The kernels read and write rows with 128-bit accesses (LDG.E.128, REDG...F32x4, STG.E.128): every non-null tensor
// pointer of a compute call must be 16-byte aligned (any torch allocation is; an odd storage offset is not).
// Returns MSDA_OK or MSDA_ERR_INVALID_ARGUMENT naming the first offender.
struct NamedPtr {
  const char* name;
  const void* ptr;
};
int check_alignment(std::initializer_list<NamedPtr> ptrs);

// MSDA_OK, or MSDA_ERR_WORKSPACE when `need` bytes are required and fewer are given
int check_workspace(const void* workspace, size_t workspace_bytes, size_t need);

// The tail of every kernel launch: counts it (msda_kernel_launch_count) and returns MSDA_OK or the launch error.
inline int launched() {
  count_launch();
  MSDA_CUDA(cudaGetLastError());
  return MSDA_OK;
}

// D in {16,32,64,128}, float / bf16 / f16 value, L <= 16, 1 <= L*P <= 64, 32-bit offsets inside one image
bool fast_ok(const Dims& d, int dtype, unsigned flags);

// ---- dispatch templates ----
// Each one calls a generic lambda with the template arguments a runtime value stands for, and instantiates it only
// for the values it lists, so a launch site compiles exactly the kernels it can launch.
template <int N>
using Int = std::integral_constant<int, N>;

// The types a dtype tag stands for: VT of the value (input, output, grad_output), AT of the offsets / weights and
// their gradients (float; double for float64; the value's own type for the autocast tags *_AUX16).
template <int Tag>
struct TagTypes;
template <> struct TagTypes<MSDA_F32> { using VT = float; using AT = float; };
template <> struct TagTypes<MSDA_F64> { using VT = double; using AT = double; };
template <> struct TagTypes<MSDA_BF16> { using VT = __nv_bfloat16; using AT = float; };
template <> struct TagTypes<MSDA_F16> { using VT = __half; using AT = float; };
template <> struct TagTypes<MSDA_BF16_AUX16> { using VT = __nv_bfloat16; using AT = __nv_bfloat16; };
template <> struct TagTypes<MSDA_F16_AUX16> { using VT = __half; using AT = __half; };

// The tag sets a kernel family is instantiated for
template <int... Tags>
struct TagList {};
using FastTags = TagList<MSDA_F32, MSDA_BF16, MSDA_F16>;                                     // fast kernels (fast_ok)
using FusedTags = TagList<MSDA_F32, MSDA_BF16, MSDA_F16, MSDA_BF16_AUX16, MSDA_F16_AUX16>;   // + 16-bit offsets / logits
using ValueTags = TagList<MSDA_F32, MSDA_F64, MSDA_BF16, MSDA_F16>;                          // generic kernels
using AllTags = TagList<MSDA_F32, MSDA_F64, MSDA_BF16, MSDA_F16, MSDA_BF16_AUX16, MSDA_F16_AUX16>;

template <int... Tags, typename F>
int with_types_in(TagList<Tags...>, int tag, F& f) {
  int r = MSDA_OK;
  if (((tag == Tags && (r = f(TagTypes<Tags>{}), true)) || ...)) return r;
  return fail(MSDA_ERR_UNSUPPORTED, "no kernel for dtype tag %d", tag);
}
// Calls f(TagTypes<tag>{}) for a tag of the set List.
template <typename List, typename F>
int with_types(int tag, F&& f) {
  return with_types_in(List{}, tag, f);
}

// Calls f(Int<D>{}) for the channel chunk D of the fast kernels, 16, 32, 64 or 128.
template <typename F>
int with_chunk(int D, F&& f) {
  switch (D) {
    case 16: return f(Int<16>{});
    case 32: return f(Int<32>{});
    case 64: return f(Int<64>{});
    case 128: return f(Int<128>{});
    default: return fail(MSDA_ERR_UNSUPPORTED, "no fast kernel for D=%d", D);
  }
}

inline int grid_for(int64_t work_items, int threads, int cap_blocks) {
  int64_t g = (work_items + threads - 1) / threads;
  if (g > cap_blocks) g = cap_blocks;
  if (g < 1) g = 1;
  return (int)g;
}

template <typename K>
cudaError_t ensure_smem(K kernel, size_t bytes) {
  if (bytes <= 48 * 1024) return cudaSuccess;
  return cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)bytes);
}

// ---- msda_fwd.cu ----
int fwd_fast(cudaStream_t st, const Dims& d, int dtype, unsigned flags, const void* value, const int64_t* shapes,
             const int64_t* lsi, const void* loc, const void* w, void* out);
int fwd_fused(cudaStream_t st, const Dims& d, int dtype, const void* value, const int64_t* shapes, const int64_t* lsi,
              const void* off, const void* logits, void* out, msda::FusedArgs fa);
int fwd_dcn(cudaStream_t st, const Dims& d, int dtype, const void* input, const void* off, const void* mask, void* out,
            msda::FusedArgs fa);
// fused DCNv3 module path (kPreDcnSoftmax): mask logits in, the row softmax runs in the kernel
int fwd_dcn_softmax(cudaStream_t st, const Dims& d, int dtype, const void* input, const void* off,
                    const void* mask_logits, void* out, msda::FusedArgs fa);

// packed batch (kPrePacked): d.B images, d.S / d.Q the largest image's value / query count, `meta` the per-image
// metadata rows (msda::packed_meta_stride), fa.value_mask unused.  LINEAR forward, STRIP backward with float reds.
int fwd_packed(cudaStream_t st, const Dims& d, int dtype, const void* value, const int64_t* shapes,
               const int64_t* meta, const void* off, const void* logits, void* out, msda::FusedArgs fa);

// ---- msda_bwd.cu ----
int bwd_fast(cudaStream_t st, const Dims& d, int dtype, unsigned flags, const void* go, const void* value,
             const int64_t* shapes, const int64_t* lsi, const void* loc, const void* w, float* gv, void* gl, void* gw);

// ---- msda_bwd_aux.cu ----
int bwd_fast_det(cudaStream_t st, const Dims& d, int dtype, const void* go, const void* value, const int64_t* shapes,
                 const int64_t* lsi, const void* loc, const void* w, unsigned long long* acc, void* gl, void* gw,
                 const msda::DetScale* det);
int bwd_fast_noscatter(cudaStream_t st, const Dims& d, int dtype, const void* go, const void* value,
                       const int64_t* shapes, const int64_t* lsi, const void* loc, const void* w, void* gl, void* gw);
int bwd_fast_emit(cudaStream_t st, const Dims& d, int dtype, const void* go, const void* value, const int64_t* shapes,
                  const int64_t* lsi, const void* loc, const void* w, void* gl, void* gw, int* cursor,
                  const int* bin_start, void* entries, float* warp_amax, int64_t* n_warps);
int bwd_fused(cudaStream_t st, const Dims& d, int dtype, const void* go, const void* value, const int64_t* shapes,
              const int64_t* lsi, const void* off, const void* logits, float* gv, void* goff, void* glog,
              msda::FusedArgs fa);
int bwd_fused_noscatter(cudaStream_t st, const Dims& d, int dtype, const void* go, const void* value,
                        const int64_t* shapes, const int64_t* lsi, const void* off, const void* logits, void* goff,
                        void* glog, msda::FusedArgs fa);
int bwd_dcn(cudaStream_t st, const Dims& d, int dtype, const void* go, const void* input, const void* off,
            const void* mask, float* gi, void* goff, void* gmask, msda::FusedArgs fa);
// fused DCNv3 module path: mask logits in, their gradient out (float reds only)
int bwd_dcn_softmax(cudaStream_t st, const Dims& d, int dtype, const void* go, const void* input, const void* off,
                    const void* mask_logits, float* gi, void* goff, void* glogits, msda::FusedArgs fa);
// DCNv3 twins of bwd_fast_det / bwd_fast_noscatter / bwd_fast_emit (deterministic grad_input)
int bwd_dcn_det(cudaStream_t st, const Dims& d, int dtype, const void* go, const void* input, const void* off,
                const void* mask, unsigned long long* acc, void* goff, void* gmask, const msda::DetScale* det,
                msda::FusedArgs fa);
int bwd_dcn_noscatter(cudaStream_t st, const Dims& d, int dtype, const void* go, const void* input, const void* off,
                      const void* mask, void* goff, void* gmask, msda::FusedArgs fa);
int bwd_dcn_emit(cudaStream_t st, const Dims& d, int dtype, const void* go, const void* input, const void* off,
                 const void* mask, void* goff, void* gmask, int* cursor, const int* bin_start, void* entries,
                 float* warp_amax, int64_t* n_warps, msda::FusedArgs fa);

int bwd_packed(cudaStream_t st, const Dims& d, int dtype, const void* go, const void* value, const int64_t* shapes,
               const int64_t* meta, const void* off, const void* logits, float* gv, void* goff, void* glog,
               msda::FusedArgs fa);

// ---- msda_dcnv2.cu ----
// Deformable convolution geometry (msda_dcnv2_im2col / _col2im): input [B,H,W,C], output [B,Ho,Wo,*].  A point is
// (image, output pixel, deformable group, kernel tap); p = ((pixel*dg + d)*K + k) inside one image.
struct Dcn2Dims {
  int B, C, H, W, Ho, Wo, kh, kw, sh, sw, ph, pw, dh, dw, groups, dg;
  __host__ __device__ int K() const { return kh * kw; }
  __host__ __device__ int Cg() const { return C / groups; }
  __host__ __device__ int Cdg() const { return C / dg; }
  __host__ __device__ int points_per_image() const { return Ho * Wo * dg * kh * kw; }
  int64_t n_points() const { return (int64_t)B * points_per_image(); }
  int64_t n_input() const { return (int64_t)B * H * W * C; }
  int64_t n_columns() const { return (int64_t)B * Ho * Wo * K() * C; }
};
// dtype: any tag; MSDA_*_AUX16: offset / mask and their gradients in the value's 16-bit type.
// grad_input_acc: float [B,H,W,C] (double for MSDA_F64), zeroed by the caller; the kernels add into it.
int dcnv2_im2col(cudaStream_t st, const Dcn2Dims& g, int dtype, unsigned flags, const void* input, const void* offset,
                 const void* mask, void* columns);
int dcnv2_col2im(cudaStream_t st, const Dcn2Dims& g, int dtype, unsigned flags, const void* grad_columns,
                 const void* input, const void* offset, const void* mask, void* grad_input_acc, void* grad_offset,
                 void* grad_mask);

// ---- msda_fold.cu ----
// does the folding backward cover this problem (encoder form Q == S, shapes it is instantiated for, flags)?
bool fold_applies(const Dims& d, int dtype, unsigned flags);
// fa == nullptr: the plain operator (loc / w given); else the fused module chain
int bwd_fold(cudaStream_t st, const Dims& d, int dtype, const void* go, const void* value, const int64_t* shapes,
             const int64_t* lsi, const void* loc, const void* w, float* gv, void* gl, void* gw,
             const msda::FusedArgs* fa);

}  // namespace msda_host
