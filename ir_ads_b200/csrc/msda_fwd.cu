// msda_fwd.cu -- instantiations and dispatch of the fast forward kernels (msda_fast.cuh).
#include "msda_fast_launch.cuh"

namespace msda_host {

int fwd_fast(cudaStream_t st, const Dims& d, int dtype, unsigned flags, const void* value, const int64_t* shapes,
             const int64_t* lsi, const void* loc, const void* w, void* out) {
#ifdef MSDA_ALL_ORDERS
#define MSDA_DISPATCH_ORDER MSDA_ORDER_ANY
#else
#define MSDA_DISPATCH_ORDER MSDA_ORDER_LINEAR
  (void)flags;
#endif
#define CALL_FWD(D_, VT_, PT_, ORD_) launch_fwd_fast<D_, VT_, PT_, kFwdThreads, ORD_>(st, d, value, shapes, lsi, loc, w, out)
  MSDA_DISPATCH_VT(CALL_FWD);
#undef CALL_FWD
#undef MSDA_DISPATCH_ORDER
}

#ifdef MSDA_EXP_SLIM
int fwd_fused(cudaStream_t, const Dims&, int, const void*, const int64_t*, const int64_t*, const void*, const void*,
              void*, msda::FusedArgs) {
  return fail(MSDA_ERR_UNSUPPORTED, "slim build: no fused kernels");
}
int fwd_dcn(cudaStream_t, const Dims&, int, const void*, const void*, const void*, void*, msda::FusedArgs) {
  return fail(MSDA_ERR_UNSUPPORTED, "slim build: no DCNv3 kernels");
}
int fwd_dcn_softmax(cudaStream_t, const Dims&, int, const void*, const void*, const void*, void*, msda::FusedArgs) {
  return fail(MSDA_ERR_UNSUPPORTED, "slim build: no DCNv3 kernels");
}
int fwd_packed(cudaStream_t, const Dims&, int, const void*, const int64_t*, const int64_t*, const void*, const void*,
               void*, msda::FusedArgs) {
  return fail(MSDA_ERR_UNSUPPORTED, "slim build: no packed kernels");
}
#else
// fused pre-op chain: LINEAR order.  dtype MSDA_*_AUX16: offsets / logits in the value's 16-bit type
int fwd_fused(cudaStream_t st, const Dims& d, int dtype, const void* value, const int64_t* shapes, const int64_t* lsi,
              const void* off, const void* logits, void* out, msda::FusedArgs fa) {
#define MSDA_DISPATCH_ORDER MSDA_ORDER_LINEAR
#define CALL_FF(D_, VT_, PT_, ORD_) \
  launch_fwd_fast<D_, VT_, PT_, kFwdThreads, ORD_, msda::kPreFused>(st, d, value, shapes, lsi, off, logits, out, fa)
#define CALL_FF16(D_, VT_, PT_, ORD_)                                                                             \
  launch_fwd_fast<D_, VT_, PT_, kFwdThreads, ORD_, msda::kPreFused, VT_>(st, d, value, shapes, lsi, off, logits, out, \
                                                                         fa)
  MSDA_DISPATCH_VT_AUX16(CALL_FF16);
  MSDA_DISPATCH_VT(CALL_FF);
#undef CALL_FF16
#undef CALL_FF
#undef MSDA_DISPATCH_ORDER
}

// fused chain over a packed batch: LINEAR order, the same value / aux types as fwd_fused
int fwd_packed(cudaStream_t st, const Dims& d, int dtype, const void* value, const int64_t* shapes,
               const int64_t* meta, const void* off, const void* logits, void* out, msda::FusedArgs fa) {
#define MSDA_DISPATCH_ORDER MSDA_ORDER_LINEAR
#define CALL_FP(D_, VT_, PT_, ORD_) \
  launch_fwd_fast<D_, VT_, PT_, kFwdThreads, ORD_, msda::kPrePacked>(st, d, value, shapes, meta, off, logits, out, fa)
#define CALL_FP16(D_, VT_, PT_, ORD_)                                                                           \
  launch_fwd_fast<D_, VT_, PT_, kFwdThreads, ORD_, msda::kPrePacked, VT_>(st, d, value, shapes, meta, off, logits, \
                                                                          out, fa)
  MSDA_DISPATCH_VT_AUX16(CALL_FP16);
  MSDA_DISPATCH_VT(CALL_FP);
#undef CALL_FP16
#undef CALL_FP
#undef MSDA_DISPATCH_ORDER
}

// DCNv3: runtime point count (K = kernel_h * kernel_w), LINEAR order.  PRE: kPreDcn (w = mask) or kPreDcnSoftmax
// (w = mask logits; dtype MSDA_*_AUX16: offset / logits in the input's 16-bit type)
template <int PRE>
int fwd_dcn_pre(cudaStream_t st, const Dims& d, int dtype, const void* input, const void* off, const void* w,
                void* out, msda::FusedArgs fa) {
#define CALL_DF(D_, VT_, AT_) \
  launch_fwd_fast<D_, VT_, 0, kFwdThreads, 0, PRE, AT_>(st, d, input, nullptr, nullptr, off, w, out, fa)
#define DCN_D(VT_, AT_)                                                                    \
  switch (d.D) {                                                                           \
    case 16: return CALL_DF(16, VT_, AT_);                                                 \
    case 32: return CALL_DF(32, VT_, AT_);                                                 \
    case 64: return CALL_DF(64, VT_, AT_);                                                 \
    case 128: return CALL_DF(128, VT_, AT_);                                               \
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
#undef CALL_DF
}

int fwd_dcn(cudaStream_t st, const Dims& d, int dtype, const void* input, const void* off, const void* mask, void* out,
            msda::FusedArgs fa) {
  return fwd_dcn_pre<msda::kPreDcn>(st, d, dtype, input, off, mask, out, fa);
}

// fused DCNv3 module path: the softmax over each (pixel, group) row's K mask logits runs in the kernel
int fwd_dcn_softmax(cudaStream_t st, const Dims& d, int dtype, const void* input, const void* off,
                    const void* mask_logits, void* out, msda::FusedArgs fa) {
  return fwd_dcn_pre<msda::kPreDcnSoftmax>(st, d, dtype, input, off, mask_logits, out, fa);
}
#endif

}  // namespace msda_host
