// msda_fwd.cu -- instantiations and dispatch of the fast forward kernels (msda_fast.cuh).
#include "msda_fast_launch.cuh"

namespace msda_host {

int fwd_fast(cudaStream_t st, const Dims& d, int dtype, unsigned flags, const void* value, const int64_t* shapes,
             const int64_t* lsi, const void* loc, const void* w, void* out) {
  return dispatch_fast<FastTags, PlainOrders<kLinear>>(d, dtype, flags, [&](auto t, auto D, auto PT, auto order) {
    using VT = typename decltype(t)::VT;
    return launch_fwd_fast<D, VT, PT, kFwdThreads, order>(st, d, value, shapes, lsi, loc, w, out);
  });
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
// fused pre-op chain, PRE kPreFused (lsi: level start index) or kPrePacked (lsi: the per-image metadata rows): LINEAR
// order.  dtype MSDA_*_AUX16: offsets / logits in the value's 16-bit type
template <int PRE>
int fwd_fused_pre(cudaStream_t st, const Dims& d, int dtype, const void* value, const int64_t* shapes,
                  const int64_t* lsi, const void* off, const void* logits, void* out, msda::FusedArgs fa) {
  return dispatch_fast<FusedTags, OrderList<kLinear>>(d, dtype, 0, [&](auto t, auto D, auto PT, auto order) {
    using VT = typename decltype(t)::VT;
    using AT = typename decltype(t)::AT;
    return launch_fwd_fast<D, VT, PT, kFwdThreads, order, PRE, AT>(st, d, value, shapes, lsi, off, logits, out, fa);
  });
}

int fwd_fused(cudaStream_t st, const Dims& d, int dtype, const void* value, const int64_t* shapes, const int64_t* lsi,
              const void* off, const void* logits, void* out, msda::FusedArgs fa) {
  return fwd_fused_pre<msda::kPreFused>(st, d, dtype, value, shapes, lsi, off, logits, out, fa);
}

int fwd_packed(cudaStream_t st, const Dims& d, int dtype, const void* value, const int64_t* shapes,
               const int64_t* meta, const void* off, const void* logits, void* out, msda::FusedArgs fa) {
  return fwd_fused_pre<msda::kPrePacked>(st, d, dtype, value, shapes, meta, off, logits, out, fa);
}

// DCNv3: runtime point count (K = kernel_h * kernel_w), LINEAR order.  PRE: kPreDcn (w = mask) or kPreDcnSoftmax
// (w = mask logits; dtype MSDA_*_AUX16: offset / logits in the input's 16-bit type)
template <int PRE>
int fwd_dcn_pre(cudaStream_t st, const Dims& d, int dtype, const void* input, const void* off, const void* w,
                void* out, msda::FusedArgs fa) {
  using Tags = std::conditional_t<PRE == msda::kPreDcnSoftmax, FusedTags, FastTags>;
  return with_types<Tags>(dtype, [&](auto t) {
    using VT = typename decltype(t)::VT;
    using AT = typename decltype(t)::AT;
    return with_chunk(d.D, [&](auto D) {
      return launch_fwd_fast<D, VT, 0, kFwdThreads, kLinear, PRE, AT>(st, d, input, nullptr, nullptr, off, w, out, fa);
    });
  });
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
