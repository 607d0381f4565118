// msda_bwd.cu -- instantiations and dispatch of the fast backward kernels with float vector reds (msda_fast.cuh).
#include "msda_fast_launch.cuh"

namespace msda_host {

int bwd_fast(cudaStream_t st, const Dims& d, int dtype, unsigned flags, const void* go, const void* value,
             const int64_t* shapes, const int64_t* lsi, const void* loc, const void* w, float* gv, void* gl, void* gw) {
  // default row order of the backward: STRIP (measured 3 % faster than LINEAR at cfg 2: fewer L1 misses
  // on the crossbar-bound kernel); the forward keeps LINEAR
  if (!(flags & (MSDA_FLAG_ORDER_LINEAR | MSDA_FLAG_ORDER_TILE2D))) flags |= MSDA_FLAG_ORDER_STRIP;
#ifdef MSDA_ALL_ORDERS
#define MSDA_DISPATCH_ORDER MSDA_ORDER_ANY
#else
#define MSDA_DISPATCH_ORDER MSDA_ORDER_STRIP
#endif
#define CALL_BWD(D_, VT_, PT_, ORD_) \
  launch_bwd_fast<D_, VT_, PT_, kBwdThreads, ORD_, float>(st, d, go, value, shapes, lsi, loc, w, gv, gl, gw, nullptr)
  MSDA_DISPATCH_VT(CALL_BWD);
#undef CALL_BWD
#undef MSDA_DISPATCH_ORDER
}

}  // namespace msda_host
