// msda_bwd_aux.cu -- the other fast backward kernels (msda_fast.cuh): 64-bit fixed-point reds (deterministic),
// scatter compiled out (grad_value not wanted / computed by msda_det.cuh), fused module chain, DCNv3.
#include "msda_fast_launch.cuh"

namespace msda_host {

namespace {
// The per-warp slots of EmitArgs::warp_amax of the entry-filing backward (LINEAR order: one CTA per kBwdThreads /
// (D / 4) rows, kBwdThreads / 32 warps each) go to *n_warps.
msda::EmitArgs emit_args(const Dims& d, int* cursor, const int* bin_start, void* entries, float* warp_amax,
                         int64_t* n_warps) {
  const int64_t rpc = kBwdThreads / (d.D / 4);
  if (n_warps) *n_warps = ((d.rows() + rpc - 1) / rpc) * (kBwdThreads / 32);
  return msda::EmitArgs{cursor, bin_start, static_cast<int4*>(entries), warp_amax};
}

// The plain operator's backward without float reds, LINEAR order.  ACC: unsigned long long (64-bit fixed-point reds
// into acc), NoScatter (scatter compiled out: grad_loc / grad_w only) or EmitEntries (no scatter; files every in-range
// point under its bilinear cell for the deterministic sorted path, replacing det_bin_kernel<true> + the no-scatter
// backward).
template <typename ACC>
int bwd_fast_acc(cudaStream_t st, const Dims& d, int dtype, const void* go, const void* value, const int64_t* shapes,
                 const int64_t* lsi, const void* loc, const void* w, ACC* acc, void* gl, void* gw,
                 const msda::DetScale* det, msda::EmitArgs ea = msda::EmitArgs{}) {
  return dispatch_fast<FastTags, OrderList<kLinear>>(d, dtype, 0, [&](auto t, auto D, auto PT, auto order) {
    using VT = typename decltype(t)::VT;
    return launch_bwd_fast<D, VT, PT, kBwdThreads, order, ACC>(st, d, go, value, shapes, lsi, loc, w, acc, gl, gw, det,
                                                               msda::FusedArgs{}, ea);
  });
}
}  // namespace

int bwd_fast_det(cudaStream_t st, const Dims& d, int dtype, const void* go, const void* value, const int64_t* shapes,
                 const int64_t* lsi, const void* loc, const void* w, unsigned long long* acc, void* gl, void* gw,
                 const msda::DetScale* det) {
  return bwd_fast_acc(st, d, dtype, go, value, shapes, lsi, loc, w, acc, gl, gw, det);
}

int bwd_fast_noscatter(cudaStream_t st, const Dims& d, int dtype, const void* go, const void* value,
                       const int64_t* shapes, const int64_t* lsi, const void* loc, const void* w, void* gl, void* gw) {
  return bwd_fast_acc<msda::NoScatter>(st, d, dtype, go, value, shapes, lsi, loc, w, nullptr, gl, gw, nullptr);
}

int bwd_fast_emit(cudaStream_t st, const Dims& d, int dtype, const void* go, const void* value, const int64_t* shapes,
                  const int64_t* lsi, const void* loc, const void* w, void* gl, void* gw, int* cursor,
                  const int* bin_start, void* entries, float* warp_amax, int64_t* n_warps) {
  const msda::EmitArgs ea = emit_args(d, cursor, bin_start, entries, warp_amax, n_warps);
  return bwd_fast_acc<msda::EmitEntries>(st, d, dtype, go, value, shapes, lsi, loc, w, nullptr, gl, gw, nullptr, ea);
}

#ifdef MSDA_EXP_SLIM
int bwd_fused(cudaStream_t, const Dims&, int, const void*, const void*, const int64_t*, const int64_t*, const void*,
              const void*, float*, void*, void*, msda::FusedArgs) {
  return fail(MSDA_ERR_UNSUPPORTED, "slim build: no fused kernels");
}
int bwd_fused_noscatter(cudaStream_t, const Dims&, int, const void*, const void*, const int64_t*, const int64_t*,
                        const void*, const void*, void*, void*, msda::FusedArgs) {
  return fail(MSDA_ERR_UNSUPPORTED, "slim build: no fused kernels");
}
int bwd_packed(cudaStream_t, const Dims&, int, const void*, const void*, const int64_t*, const int64_t*, const void*,
               const void*, float*, void*, void*, msda::FusedArgs) {
  return fail(MSDA_ERR_UNSUPPORTED, "slim build: no packed kernels");
}
int bwd_dcn(cudaStream_t, const Dims&, int, const void*, const void*, const void*, const void*, float*, void*, void*,
            msda::FusedArgs) {
  return fail(MSDA_ERR_UNSUPPORTED, "slim build: no DCNv3 kernels");
}
int bwd_dcn_softmax(cudaStream_t, const Dims&, int, const void*, const void*, const void*, const void*, float*, void*,
                    void*, msda::FusedArgs) {
  return fail(MSDA_ERR_UNSUPPORTED, "slim build: no DCNv3 kernels");
}
int bwd_dcn_det(cudaStream_t, const Dims&, int, const void*, const void*, const void*, const void*,
                unsigned long long*, void*, void*, const msda::DetScale*, msda::FusedArgs) {
  return fail(MSDA_ERR_UNSUPPORTED, "slim build: no DCNv3 kernels");
}
int bwd_dcn_noscatter(cudaStream_t, const Dims&, int, const void*, const void*, const void*, const void*, void*, void*,
                      msda::FusedArgs) {
  return fail(MSDA_ERR_UNSUPPORTED, "slim build: no DCNv3 kernels");
}
int bwd_dcn_emit(cudaStream_t, const Dims&, int, const void*, const void*, const void*, const void*, void*, void*, int*,
                 const int*, void*, float*, int64_t*, msda::FusedArgs) {
  return fail(MSDA_ERR_UNSUPPORTED, "slim build: no DCNv3 kernels");
}
#else
// fused pre-op chain, STRIP order.  PRE kPreFused (lsi: level start index) or kPrePacked (lsi: the per-image metadata
// rows).  ACC float (float reds into gv) or NoScatter (gradients of the raw offsets / logits only).  dtype
// MSDA_*_AUX16 (Tags = FusedTags): offsets / logits and their gradients in the value's 16-bit type
template <int PRE, typename Tags, typename ACC>
int bwd_fused_pre(cudaStream_t st, const Dims& d, int dtype, const void* go, const void* value, const int64_t* shapes,
                  const int64_t* lsi, const void* off, const void* logits, ACC* gv, void* goff, void* glog,
                  msda::FusedArgs fa) {
  return dispatch_fast<Tags, OrderList<kStrip>>(d, dtype, 0, [&](auto t, auto D, auto PT, auto order) {
    using VT = typename decltype(t)::VT;
    using AT = typename decltype(t)::AT;
    return launch_bwd_fast<D, VT, PT, kBwdThreads, order, ACC, PRE, AT>(st, d, go, value, shapes, lsi, off, logits, gv,
                                                                        goff, glog, nullptr, fa);
  });
}

int bwd_fused(cudaStream_t st, const Dims& d, int dtype, const void* go, const void* value, const int64_t* shapes,
              const int64_t* lsi, const void* off, const void* logits, float* gv, void* goff, void* glog,
              msda::FusedArgs fa) {
  return bwd_fused_pre<msda::kPreFused, FusedTags>(st, d, dtype, go, value, shapes, lsi, off, logits, gv, goff, glog,
                                                   fa);
}

int bwd_packed(cudaStream_t st, const Dims& d, int dtype, const void* go, const void* value, const int64_t* shapes,
               const int64_t* meta, const void* off, const void* logits, float* gv, void* goff, void* glog,
               msda::FusedArgs fa) {
  return bwd_fused_pre<msda::kPrePacked, FusedTags>(st, d, dtype, go, value, shapes, meta, off, logits, gv, goff, glog,
                                                    fa);
}

int bwd_fused_noscatter(cudaStream_t st, const Dims& d, int dtype, const void* go, const void* value,
                        const int64_t* shapes, const int64_t* lsi, const void* off, const void* logits, void* goff,
                        void* glog, msda::FusedArgs fa) {
  return bwd_fused_pre<msda::kPreFused, FastTags, msda::NoScatter>(st, d, dtype, go, value, shapes, lsi, off, logits,
                                                                   nullptr, goff, glog, fa);
}

// DCNv3: runtime point count.  PRE kPreDcn (w = mask, gw = its gradient) or kPreDcnSoftmax (w = mask logits, gw = the
// logits' gradient; dtype MSDA_*_AUX16: offset / logits and their gradients in the input's 16-bit type).  ACC: float
// reds, or the deterministic kinds of bwd_fast_acc (kPreDcn only).  STRIP order, except EmitEntries: LINEAR, so that
// the per-warp maxima have exactly the slots emit_args counts for the equivalent one-level problem.
template <int PRE, typename ACC>
int bwd_dcn_pre(cudaStream_t st, const Dims& d, int dtype, const void* go, const void* input, const void* off,
                const void* w, ACC* gi, void* goff, void* gw, const msda::DetScale* det, msda::FusedArgs fa,
                msda::EmitArgs ea = msda::EmitArgs{}) {
  using Tags = std::conditional_t<PRE == msda::kPreDcnSoftmax, FusedTags, FastTags>;
  constexpr int ORDER = std::is_same_v<ACC, msda::EmitEntries> ? kLinear : kStrip;
  return with_types<Tags>(dtype, [&](auto t) {
    using VT = typename decltype(t)::VT;
    using AT = typename decltype(t)::AT;
    return with_chunk(d.D, [&](auto D) {
      return launch_bwd_fast<D, VT, 0, kBwdThreads, ORDER, ACC, PRE, AT>(st, d, go, input, nullptr, nullptr, off, w, gi,
                                                                         goff, gw, det, fa, ea);
    });
  });
}

int bwd_dcn(cudaStream_t st, const Dims& d, int dtype, const void* go, const void* input, const void* off,
            const void* mask, float* gi, void* goff, void* gmask, msda::FusedArgs fa) {
  return bwd_dcn_pre<msda::kPreDcn>(st, d, dtype, go, input, off, mask, gi, goff, gmask, nullptr, fa);
}

// fused DCNv3 module path: the softmax's chain rule runs in the kernel, which writes the mask logits' gradient
int bwd_dcn_softmax(cudaStream_t st, const Dims& d, int dtype, const void* go, const void* input, const void* off,
                    const void* mask_logits, float* gi, void* goff, void* glogits, msda::FusedArgs fa) {
  return bwd_dcn_pre<msda::kPreDcnSoftmax>(st, d, dtype, go, input, off, mask_logits, gi, goff, glogits, nullptr, fa);
}

// 64-bit fixed-point reds: MSDA_FLAG_DET_ATOMIC, or problems beyond the sorted path's 32-bit indices
int bwd_dcn_det(cudaStream_t st, const Dims& d, int dtype, const void* go, const void* input, const void* off,
                const void* mask, unsigned long long* acc, void* goff, void* gmask, const msda::DetScale* det,
                msda::FusedArgs fa) {
  return bwd_dcn_pre<msda::kPreDcn>(st, d, dtype, go, input, off, mask, acc, goff, gmask, det, fa);
}

// without the scatter (grad_offset / grad_mask only): the sorted path with MSDA_FLAG_DET_SEPARATE_FILL
int bwd_dcn_noscatter(cudaStream_t st, const Dims& d, int dtype, const void* go, const void* input, const void* off,
                      const void* mask, void* goff, void* gmask, msda::FusedArgs fa) {
  return bwd_dcn_pre<msda::kPreDcn, msda::NoScatter>(st, d, dtype, go, input, off, mask, nullptr, goff, gmask, nullptr,
                                                     fa);
}

// files every in-range point under its bilinear cell (sorted path)
int bwd_dcn_emit(cudaStream_t st, const Dims& d, int dtype, const void* go, const void* input, const void* off,
                 const void* mask, void* goff, void* gmask, int* cursor, const int* bin_start, void* entries,
                 float* warp_amax, int64_t* n_warps, msda::FusedArgs fa) {
  const msda::EmitArgs ea = emit_args(d, cursor, bin_start, entries, warp_amax, n_warps);
  return bwd_dcn_pre<msda::kPreDcn, msda::EmitEntries>(st, d, dtype, go, input, off, mask, nullptr, goff, gmask,
                                                       nullptr, fa, ea);
}
#endif

}  // namespace msda_host
