// msda_bwd_aux.cu -- the other fast backward kernels (msda_fast.cuh): 64-bit fixed-point reds (deterministic),
// scatter compiled out (grad_value not wanted / computed by msda_det.cuh), fused module chain, DCNv3.
#include "msda_fast_launch.cuh"

namespace msda_host {

// deterministic accumulate: LINEAR order
int bwd_fast_det(cudaStream_t st, const Dims& d, int dtype, const void* go, const void* value, const int64_t* shapes,
                 const int64_t* lsi, const void* loc, const void* w, unsigned long long* acc, void* gl, void* gw,
                 const msda::DetScale* det) {
#define MSDA_DISPATCH_ORDER MSDA_ORDER_LINEAR
#define CALL_BWD(D_, VT_, PT_, ORD_) \
  launch_bwd_fast<D_, VT_, PT_, kBwdThreads, ORD_, unsigned long long>(st, d, go, value, shapes, lsi, loc, w, acc, gl, gw, det)
  MSDA_DISPATCH_VT(CALL_BWD);
#undef CALL_BWD
#undef MSDA_DISPATCH_ORDER
}

// backward without the scatter (grad_loc / grad_w only), LINEAR order
int bwd_fast_noscatter(cudaStream_t st, const Dims& d, int dtype, const void* go, const void* value,
                       const int64_t* shapes, const int64_t* lsi, const void* loc, const void* w, void* gl, void* gw) {
#define MSDA_DISPATCH_ORDER MSDA_ORDER_LINEAR
#define CALL_BWD(D_, VT_, PT_, ORD_)                                                                          \
  launch_bwd_fast<D_, VT_, PT_, kBwdThreads, ORD_, msda::NoScatter>(st, d, go, value, shapes, lsi, loc, w,   \
                                                                    (msda::NoScatter*)nullptr, gl, gw, nullptr)
  MSDA_DISPATCH_VT(CALL_BWD);
#undef CALL_BWD
#undef MSDA_DISPATCH_ORDER
}

// backward without the scatter that also files every in-range point under its bilinear cell (deterministic sorted
// path: replaces det_bin_kernel<true> + the plain no-scatter backward), LINEAR order
int bwd_fast_emit(cudaStream_t st, const Dims& d, int dtype, const void* go, const void* value, const int64_t* shapes,
                  const int64_t* lsi, const void* loc, const void* w, void* gl, void* gw, int* cursor,
                  const int* bin_start, void* entries, float* warp_amax, int64_t* n_warps) {
  // one CTA per kBwdThreads / (D / 4) rows (LINEAR order), kBwdThreads / 32 warps each: the slots of EmitArgs::warp_amax
  const int64_t rpc = kBwdThreads / (d.D / 4);
  if (n_warps) *n_warps = ((d.rows() + rpc - 1) / rpc) * (kBwdThreads / 32);
  msda::EmitArgs ea{cursor, bin_start, static_cast<int4*>(entries), warp_amax};
#define MSDA_DISPATCH_ORDER MSDA_ORDER_LINEAR
#define CALL_BWD(D_, VT_, PT_, ORD_)                                                                            \
  launch_bwd_fast<D_, VT_, PT_, kBwdThreads, ORD_, msda::EmitEntries>(st, d, go, value, shapes, lsi, loc, w,   \
                                                                      (msda::EmitEntries*)nullptr, gl, gw, nullptr, \
                                                                      msda::FusedArgs{}, ea)
  MSDA_DISPATCH_VT(CALL_BWD);
#undef CALL_BWD
#undef MSDA_DISPATCH_ORDER
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
// fused pre-op chain: STRIP order.  dtype MSDA_*_AUX16: offsets / logits and their gradients in the value's 16-bit
// type
int bwd_fused(cudaStream_t st, const Dims& d, int dtype, const void* go, const void* value, const int64_t* shapes,
              const int64_t* lsi, const void* off, const void* logits, float* gv, void* goff, void* glog,
              msda::FusedArgs fa) {
#define MSDA_DISPATCH_ORDER MSDA_ORDER_STRIP
#define CALL_FB(D_, VT_, PT_, ORD_)                                                                               \
  launch_bwd_fast<D_, VT_, PT_, kBwdThreads, ORD_, float, msda::kPreFused>(st, d, go, value, shapes, lsi, off, logits, gv, \
                                                                           goff, glog, nullptr, fa)
#define CALL_FB16(D_, VT_, PT_, ORD_)                                                                          \
  launch_bwd_fast<D_, VT_, PT_, kBwdThreads, ORD_, float, msda::kPreFused, VT_>(st, d, go, value, shapes, lsi, off, \
                                                                                logits, gv, goff, glog, nullptr, fa)
  MSDA_DISPATCH_VT_AUX16(CALL_FB16);
  MSDA_DISPATCH_VT(CALL_FB);
#undef CALL_FB16
#undef CALL_FB
#undef MSDA_DISPATCH_ORDER
}

// fused chain over a packed batch: STRIP order, float reds, the same value / aux types as bwd_fused
int bwd_packed(cudaStream_t st, const Dims& d, int dtype, const void* go, const void* value, const int64_t* shapes,
               const int64_t* meta, const void* off, const void* logits, float* gv, void* goff, void* glog,
               msda::FusedArgs fa) {
#define MSDA_DISPATCH_ORDER MSDA_ORDER_STRIP
#define CALL_PB(D_, VT_, PT_, ORD_)                                                                                  \
  launch_bwd_fast<D_, VT_, PT_, kBwdThreads, ORD_, float, msda::kPrePacked>(st, d, go, value, shapes, meta, off,      \
                                                                            logits, gv, goff, glog, nullptr, fa)
#define CALL_PB16(D_, VT_, PT_, ORD_)                                                                             \
  launch_bwd_fast<D_, VT_, PT_, kBwdThreads, ORD_, float, msda::kPrePacked, VT_>(st, d, go, value, shapes, meta, off, \
                                                                                 logits, gv, goff, glog, nullptr, fa)
  MSDA_DISPATCH_VT_AUX16(CALL_PB16);
  MSDA_DISPATCH_VT(CALL_PB);
#undef CALL_PB16
#undef CALL_PB
#undef MSDA_DISPATCH_ORDER
}

// fused chain, scatter compiled out: gradients of the raw offsets / logits only (deterministic fused backward)
int bwd_fused_noscatter(cudaStream_t st, const Dims& d, int dtype, const void* go, const void* value,
                        const int64_t* shapes, const int64_t* lsi, const void* off, const void* logits, void* goff,
                        void* glog, msda::FusedArgs fa) {
#define MSDA_DISPATCH_ORDER MSDA_ORDER_STRIP
#define CALL_FB(D_, VT_, PT_, ORD_)                                                                              \
  launch_bwd_fast<D_, VT_, PT_, kBwdThreads, ORD_, msda::NoScatter, msda::kPreFused>(                            \
      st, d, go, value, shapes, lsi, off, logits, (msda::NoScatter*)nullptr, goff, glog, nullptr, fa)
  MSDA_DISPATCH_VT(CALL_FB);
#undef CALL_FB
#undef MSDA_DISPATCH_ORDER
}

// DCNv3: runtime point count, STRIP order.  PRE: kPreDcn (w = mask, gw = its gradient) or kPreDcnSoftmax (w = mask
// logits, gw = the logits' gradient; dtype MSDA_*_AUX16: offset / logits and their gradients in the input's 16-bit
// type)
template <int PRE>
int bwd_dcn_pre(cudaStream_t st, const Dims& d, int dtype, const void* go, const void* input, const void* off,
                const void* w, float* gi, void* goff, void* gw, msda::FusedArgs fa) {
#define CALL_DB(D_, VT_, AT_)                                                                                          \
  launch_bwd_fast<D_, VT_, 0, kBwdThreads, 2, float, PRE, AT_>(st, d, go, input, nullptr, nullptr, off, w, gi, goff, gw, \
                                                               nullptr, fa)
#define DCN_D(VT_, AT_)                                                                    \
  switch (d.D) {                                                                           \
    case 16: return CALL_DB(16, VT_, AT_);                                                 \
    case 32: return CALL_DB(32, VT_, AT_);                                                 \
    case 64: return CALL_DB(64, VT_, AT_);                                                 \
    case 128: return CALL_DB(128, VT_, AT_);                                               \
    default: return fail(MSDA_ERR_UNSUPPORTED, "dcnv3: group_channels=%d", d.D);           \
  }
  if constexpr (PRE == msda::kPreDcnSoftmax) {
    if (dtype == MSDA_BF16_AUX16) DCN_D(__nv_bfloat16, __nv_bfloat16)
    if (dtype == MSDA_F16_AUX16) DCN_D(__half, __half)
  }
  if (dtype == MSDA_F32) DCN_D(float, float)
  if (dtype == MSDA_BF16) DCN_D(__nv_bfloat16, float)
  if (dtype == MSDA_F16) DCN_D(__half, float)
  return fail(MSDA_ERR_UNSUPPORTED, "dcnv3: dtype %d", dtype);
#undef DCN_D
#undef CALL_DB
}

int bwd_dcn(cudaStream_t st, const Dims& d, int dtype, const void* go, const void* input, const void* off,
            const void* mask, float* gi, void* goff, void* gmask, msda::FusedArgs fa) {
  return bwd_dcn_pre<msda::kPreDcn>(st, d, dtype, go, input, off, mask, gi, goff, gmask, fa);
}

// fused DCNv3 module path: the softmax's chain rule runs in the kernel, which writes the mask logits' gradient
int bwd_dcn_softmax(cudaStream_t st, const Dims& d, int dtype, const void* go, const void* input, const void* off,
                    const void* mask_logits, float* gi, void* goff, void* glogits, msda::FusedArgs fa) {
  return bwd_dcn_pre<msda::kPreDcnSoftmax>(st, d, dtype, go, input, off, mask_logits, gi, goff, glogits, fa);
}

// the DCNv3 twins of the deterministic backward kernels above, dispatched over group_channels and dtype
#define MSDA_DCN_DISPATCH(CALL)                                                              \
  do {                                                                                       \
    if (dtype != MSDA_F32 && dtype != MSDA_BF16 && dtype != MSDA_F16)                        \
      return fail(MSDA_ERR_UNSUPPORTED, "dcnv3: dtype %d", dtype);                           \
    switch (d.D) {                                                                           \
      case 16: return dtype == MSDA_F32 ? CALL(16, float) : dtype == MSDA_BF16 ? CALL(16, __nv_bfloat16) : CALL(16, __half); \
      case 32: return dtype == MSDA_F32 ? CALL(32, float) : dtype == MSDA_BF16 ? CALL(32, __nv_bfloat16) : CALL(32, __half); \
      case 64: return dtype == MSDA_F32 ? CALL(64, float) : dtype == MSDA_BF16 ? CALL(64, __nv_bfloat16) : CALL(64, __half); \
      case 128: return dtype == MSDA_F32 ? CALL(128, float) : dtype == MSDA_BF16 ? CALL(128, __nv_bfloat16) : CALL(128, __half); \
      default: return fail(MSDA_ERR_UNSUPPORTED, "dcnv3: group_channels=%d", d.D);         \
    }                                                                                        \
  } while (0)

// DCNv3, 64-bit fixed-point reds (MSDA_FLAG_DET_ATOMIC, or problems beyond the sorted path's 32-bit indices): STRIP
// order, as the float-red twin
int bwd_dcn_det(cudaStream_t st, const Dims& d, int dtype, const void* go, const void* input, const void* off,
                const void* mask, unsigned long long* acc, void* goff, void* gmask, const msda::DetScale* det,
                msda::FusedArgs fa) {
#define CALL_DB(D_, VT_)                                                                                         \
  launch_bwd_fast<D_, VT_, 0, kBwdThreads, 2, unsigned long long, msda::kPreDcn>(st, d, go, input, nullptr, nullptr, \
                                                                                 off, mask, acc, goff, gmask, det, fa)
  MSDA_DCN_DISPATCH(CALL_DB);
#undef CALL_DB
}

// DCNv3 without the scatter (grad_offset / grad_mask only): the sorted path with MSDA_FLAG_DET_SEPARATE_FILL
int bwd_dcn_noscatter(cudaStream_t st, const Dims& d, int dtype, const void* go, const void* input, const void* off,
                      const void* mask, void* goff, void* gmask, msda::FusedArgs fa) {
#define CALL_DB(D_, VT_)                                                                                           \
  launch_bwd_fast<D_, VT_, 0, kBwdThreads, 2, msda::NoScatter, msda::kPreDcn>(                                     \
      st, d, go, input, nullptr, nullptr, off, mask, (msda::NoScatter*)nullptr, goff, gmask, nullptr, fa)
  MSDA_DCN_DISPATCH(CALL_DB);
#undef CALL_DB
}

// DCNv3 backward that files every in-range point under its bilinear cell (sorted path).  LINEAR order, so that the
// per-warp maxima have exactly the slots bwd_fast_emit counts for the equivalent one-level problem.
int bwd_dcn_emit(cudaStream_t st, const Dims& d, int dtype, const void* go, const void* input, const void* off,
                 const void* mask, void* goff, void* gmask, int* cursor, const int* bin_start, void* entries,
                 float* warp_amax, int64_t* n_warps, msda::FusedArgs fa) {
  const int64_t rpc = kBwdThreads / (d.D / 4);
  if (n_warps) *n_warps = ((d.rows() + rpc - 1) / rpc) * (kBwdThreads / 32);
  msda::EmitArgs ea{cursor, bin_start, static_cast<int4*>(entries), warp_amax};
#define CALL_DB(D_, VT_)                                                                                           \
  launch_bwd_fast<D_, VT_, 0, kBwdThreads, 0, msda::EmitEntries, msda::kPreDcn>(                                   \
      st, d, go, input, nullptr, nullptr, off, mask, (msda::EmitEntries*)nullptr, goff, gmask, nullptr, fa, ea)
  MSDA_DCN_DISPATCH(CALL_DB);
#undef CALL_DB
}
#undef MSDA_DCN_DISPATCH
#endif

}  // namespace msda_host
