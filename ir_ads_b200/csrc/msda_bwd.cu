// msda_bwd.cu -- instantiations and dispatch of the fast backward kernels with float vector reds (msda_fast.cuh).
#include "msda_fast_launch.cuh"

namespace msda_host {

int bwd_fast(cudaStream_t st, const Dims& d, int dtype, unsigned flags, const void* go, const void* value,
             const int64_t* shapes, const int64_t* lsi, const void* loc, const void* w, float* gv, void* gl, void* gw) {
  // default row order of the backward: STRIP (measured 3 % faster than LINEAR at cfg 2: fewer L1 misses
  // on the crossbar-bound kernel); the forward keeps LINEAR
  if (!(flags & (MSDA_FLAG_ORDER_LINEAR | MSDA_FLAG_ORDER_TILE2D))) flags |= MSDA_FLAG_ORDER_STRIP;
  return dispatch_fast<FastTags, PlainOrders<kStrip>>(d, dtype, flags, [&](auto t, auto D, auto PT, auto order) {
    using VT = typename decltype(t)::VT;
    return launch_bwd_fast<D, VT, PT, kBwdThreads, order, float>(st, d, go, value, shapes, lsi, loc, w, gv, gl, gw,
                                                                  nullptr);
  });
}

}  // namespace msda_host
