// msda_fast_launch.cuh -- launch templates and the shape / row-order dispatch shared by the fast-kernel translation
// units: dispatch_fast(d, dtype, flags, f) calls f(types, D, PT, ORDER) for the one fast kernel a problem runs on.
#pragma once
#include "msda_host.h"

namespace msda_host {

// Row order: TILE2D needs query i == pixel i of the pyramid (encoder self-attention, Q == S).
inline bool use_strip(unsigned flags) {
  return (flags & MSDA_FLAG_ORDER_STRIP) && !(flags & (MSDA_FLAG_ORDER_LINEAR | MSDA_FLAG_ORDER_TILE2D));
}
inline bool use_tile2d(const Dims& d, unsigned flags) {
  return d.Q == d.S && (flags & MSDA_FLAG_ORDER_TILE2D) && !(flags & MSDA_FLAG_ORDER_LINEAR);
}
// TILE2D launches an upper bound on the tile count that needs only S and L (the level shapes stay on the
// device): sum_l ceil(H_l/TH)*ceil(W_l/TW) is ~1.03 * S/RPC for image pyramids; 25 % + 32 tiles per level of
// slack covers them, the kernel's grid-stride step covers anything else.
inline int64_t tile2d_bound(const Dims& d, int rpc) { return ((int64_t)d.S + rpc - 1) / rpc * 5 / 4 + 32 * (int64_t)d.L; }

// CTA sizes.  An SM re-uses a CTA's slot only when the CTA's slowest warp is done, so small CTAs keep more warps
// busy: cfg 2 forward 0.665 / 0.635 / 0.620 ms at 256 / 128 / 64 threads, backward 1.687 / 1.672 / 1.695 ms
// (profiles/r01s_experiments.txt).
#ifndef MSDA_FWD_THREADS
#define MSDA_FWD_THREADS 64
#endif
#ifndef MSDA_BWD_THREADS
#define MSDA_BWD_THREADS 128
#endif
constexpr int kFwdThreads = MSDA_FWD_THREADS, kBwdThreads = MSDA_BWD_THREADS;

// channels per lane: 8 for bf16 / f16 rows of 32+ channels (16-byte lane loads), else 4
template <int D, typename VT>
constexpr int cpl_of() { return (sizeof(VT) == 2 && D >= 32) ? 8 : 4; }

// AT: element type of loc / w (float, or the value's 16-bit type in the logits modes, msda::aux_ok)
template <int D, typename VT, int PT, int THREADS, int ORDER, int PRE = 0, typename AT = float>
int launch_fwd_fast(cudaStream_t st, const Dims& d, const void* value, const int64_t* shapes, const int64_t* lsi,
                    const void* loc, const void* w, void* out, msda::FusedArgs fa = msda::FusedArgs{}) {
  constexpr int CPL = cpl_of<D, VT>();
  using G = msda::Geom<D * 4 / CPL, THREADS>;
  const int NP = d.L * d.P;
  const size_t smem = sizeof(msda::LevelTab) + (size_t)G::RPC * msda::fwd_row_words(NP) * 4;
  auto k = msda::msda_fwd_fast_kernel<D, VT, PT, THREADS, ORDER, PRE, CPL, AT>;
  MSDA_CUDA(ensure_smem(k, smem));
  const int64_t rows = d.rows();
  unsigned grid = (unsigned)((rows + G::RPC - 1) / G::RPC);
  if (ORDER == 2) grid = (unsigned)((int64_t)d.B * d.H * ((d.Q + G::RPC - 1) / G::RPC));
  if (ORDER == 3) grid = (unsigned)((int64_t)d.B * d.H * tile2d_bound(d, G::RPC));
  // packed batch (d.Q = the largest image's query count): every image gets the LINEAR grid of that image
  if (PRE == msda::kPrePacked) grid = (unsigned)((int64_t)d.B * (((int64_t)d.Q * d.H + G::RPC - 1) / G::RPC));
  k<<<grid, THREADS, smem, st>>>((const VT*)value, shapes, lsi, (const AT*)loc, (const AT*)w, (VT*)out, fa,
                                 d.B, d.S, d.H, d.L, d.Q, d.P, rows);
  return launched();
}

template <int D, typename VT, int PT, int THREADS, int ORDER, typename ACC, int PRE = 0, typename AT = float>
int launch_bwd_fast(cudaStream_t st, const Dims& d, const void* go, const void* value, const int64_t* shapes,
                    const int64_t* lsi, const void* loc, const void* w, ACC* gv, void* gl, void* gw,
                    const msda::DetScale* det, msda::FusedArgs fa = msda::FusedArgs{},
                    msda::EmitArgs emit = msda::EmitArgs{}) {
  // The backward keeps 4 channels per lane for every type: it is bound by the grad_value reds, and those run
  // fastest as one full 128-byte line per row and instruction (8 channels per lane -> two 64-byte halves per
  // row: 1.75 -> 2.09 ms at cfg2 with bf16 value), so the faster 16-byte gather buys nothing there.
  constexpr int CPL = 4;
  using G = msda::Geom<D * 4 / CPL, THREADS>;
  const int NP = d.L * d.P;
  const size_t smem = sizeof(msda::LevelTab) + (size_t)G::RPC * msda::bwd_row_words(NP) * 4;
  auto k = msda::msda_bwd_fast_kernel<D, VT, PT, THREADS, ORDER, ACC, PRE, CPL, AT>;
  MSDA_CUDA(ensure_smem(k, smem));
  const int64_t rows = d.rows();
  unsigned grid = (unsigned)((rows + G::RPC - 1) / G::RPC);
  // (packed batches: d.Q = the largest image's query count, the STRIP grid of that image for every image)
  if (ORDER == 2) grid = (unsigned)((int64_t)d.B * d.H * ((d.Q + G::RPC - 1) / G::RPC));
  if (ORDER == 3) grid = (unsigned)((int64_t)d.B * d.H * tile2d_bound(d, G::RPC));
  k<<<grid, THREADS, smem, st>>>((const VT*)go, (const VT*)value, shapes, lsi, (const AT*)loc, (const AT*)w,
                                 gv, (AT*)gl, (AT*)gw, det, fa, emit, d.B, d.S, d.H, d.L, d.Q, d.P, rows);
  return launched();
}

// Calls f(Int<PT>{}) for the point count of the fast kernels: 4 or 8 compiled in, 0 = any (runtime d.P).
template <typename F>
int with_points(int P, F&& f) {
  if (P == 4) return f(Int<4>{});
  if (P == 8) return f(Int<8>{});
  return f(Int<0>{});
}

// Calls f(Int<D>{}, Int<PT>{}) for the channel and point count of the fast kernels.
template <typename F>
int with_shape(const Dims& d, F&& f) {
#ifdef MSDA_EXP_SLIM
  // Kernel-variant experiment builds (tools/build_variant.sh): only D = 32, P in {4, 8} are instantiated, so a variant
  // compiles in well under a minute.  Never defined for the product library.
  if (d.D != 32) return fail(MSDA_ERR_UNSUPPORTED, "slim build: D=%d", d.D);
  if (d.P == 4) return f(Int<32>{}, Int<4>{});
  if (d.P == 8) return f(Int<32>{}, Int<8>{});
  return fail(MSDA_ERR_UNSUPPORTED, "slim build: P=%d", d.P);
#else
  return with_chunk(d.D, [&](auto D) { return with_points(d.P, [&](auto PT) { return f(D, PT); }); });
#endif
}

// Row orders (the kernels' ORDER argument) and the sets a family is instantiated for
constexpr int kLinear = 0, kStrip = 2, kTile2d = 3;
template <int... Orders>
struct OrderList {};
using AllOrders = OrderList<kLinear, kStrip, kTile2d>;

// The product library instantiates ONE row order per pass of the plain operator -- LINEAR forward, STRIP backward, the
// pair that is fastest on every measured config (profiles/r02t_sweep_row_orders.txt) -- and treats MSDA_FLAG_ORDER_*
// as hints it may ignore (results never depend on the order).  Experiment builds (-DMSDA_EXPERIMENTS) and the slim
// variant builds of tools/build_variant.sh carry all three orders for both passes.
#if defined(MSDA_EXPERIMENTS) || defined(MSDA_EXP_SLIM)
template <int Default>
using PlainOrders = AllOrders;
#else
template <int Default>
using PlainOrders = OrderList<Default>;
#endif

// Calls f(Int<ORDER>{}): a family with one order always runs it, one with all three picks it from the flags.
template <int Order, typename F>
int with_order(OrderList<Order>, const Dims&, unsigned, F&& f) {
  return f(Int<Order>{});
}
template <typename F>
int with_order(AllOrders, const Dims& d, unsigned flags, F&& f) {
  if (use_tile2d(d, flags)) return f(Int<kTile2d>{});
  if (use_strip(flags)) return f(Int<kStrip>{});
  return f(Int<kLinear>{});
}

// Calls f(TagTypes<dtype>{}, Int<D>{}, Int<PT>{}, Int<ORDER>{}) for a family instantiated for the dtype tags Tags
// and the row orders Orders.
template <typename Tags, typename Orders, typename F>
int dispatch_fast(const Dims& d, int dtype, unsigned flags, F&& f) {
  return with_types<Tags>(dtype, [&](auto t) {
    return with_shape(d, [&](auto D, auto PT) {
      return with_order(Orders{}, d, flags, [&](auto order) { return f(t, D, PT, order); });
    });
  });
}

}  // namespace msda_host
