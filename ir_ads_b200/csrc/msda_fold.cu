// msda_fold.cu -- instantiations and dispatch of the folding encoder backward (msda_fold.cuh).
//
// EXPERIMENT, compiled only with -DMSDA_EXPERIMENTS (tools/build_variant.sh); the product library carries stubs.
// Measured on B200 at cfg 2 (profiles/r02b_fold_experiment.txt): the fold removes 82 % of the reds (57 M red sectors
// instead of 312 M, crossbar port 9 % busy instead of 93 %) but its bookkeeping costs 2.0 G warp instructions
// against 0.9 G, and the backward takes 3.1 - 4.2 ms instead of 1.67 ms.
#include "msda_fast_launch.cuh"

#ifndef MSDA_EXPERIMENTS
namespace msda_host {
bool fold_applies(const Dims&, int, unsigned) { return false; }
int bwd_fold(cudaStream_t, const Dims&, int, const void*, const void*, const int64_t*, const int64_t*, const void*,
             const void*, float*, void*, void*, const msda::FusedArgs*) {
  return fail(MSDA_ERR_UNSUPPORTED, "the folding backward is compiled into experiment builds only");
}
}  // namespace msda_host
#else
#include "msda_fold.cuh"

namespace msda_host {

namespace {
constexpr size_t kFoldSmemCap = 113 * 1024;   // two CTAs per SM

// query tile: 8 x 8 when its tables fit twice into an SM's shared memory, else 8 x 4 (D = 32 only), else no fold
int fold_tile(const Dims& d) {
  const int NP = d.L * d.P;
  if (msda::fold_smem_bytes(d.D, 64, NP) <= kFoldSmemCap) return 64;
  if (d.D == 32 && msda::fold_smem_bytes(d.D, 32, NP) <= kFoldSmemCap) return 32;
  return 0;
}

template <int D, typename VT, int PT, int NQ, int PRE>
int launch_fold(cudaStream_t st, const Dims& d, const void* go, const void* value, const int64_t* shapes,
                const int64_t* lsi, const void* loc, const void* w, float* gv, void* gl, void* gw, msda::FusedArgs fa) {
  const size_t smem = msda::fold_smem_bytes(D, NQ, d.L * d.P);
  auto k = msda::msda_bwd_fold_kernel<D, VT, PT, NQ, PRE>;
  MSDA_CUDA(ensure_smem(k, smem));
  const unsigned grid = (unsigned)((int64_t)d.B * d.H * tile2d_bound(d, NQ));
  k<<<grid, msda::kFoldThreads, smem, st>>>((const VT*)go, (const VT*)value, shapes, lsi, (const float*)loc,
                                             (const float*)w, gv, (float*)gl, (float*)gw, fa, d.B, d.S, d.H, d.L, d.Q,
                                             d.P);
  return launched();
}

template <int D, typename VT, int PRE>
int fold_pt(cudaStream_t st, const Dims& d, int nq, const void* go, const void* value, const int64_t* shapes,
            const int64_t* lsi, const void* loc, const void* w, float* gv, void* gl, void* gw, msda::FusedArgs fa) {
  auto call = [&](auto PT, auto NQ) {
    return launch_fold<D, VT, PT, NQ, PRE>(st, d, go, value, shapes, lsi, loc, w, gv, gl, gw, fa);
  };
#ifdef MSDA_EXP_SLIM
  // experiment builds: D = 32, P in {4, 8}, the plain operator only
  if constexpr (D == 32 && PRE == msda::kPrePlain) {
    if (d.P == 4 && nq == 64) return call(Int<4>{}, Int<64>{});
    if (d.P == 8 && nq == 32) return call(Int<8>{}, Int<32>{});
  }
  return fail(MSDA_ERR_UNSUPPORTED, "slim build: fold D=%d P=%d", d.D, d.P);
#else
  if constexpr (D == 32) {
    if (nq == 32) return d.P == 8 ? call(Int<8>{}, Int<32>{}) : call(Int<0>{}, Int<32>{});
  }
  return with_points(d.P, [&](auto PT) { return call(PT, Int<64>{}); });
#endif
}
}  // namespace

bool fold_applies(const Dims& d, int dtype, unsigned flags) {
  if (flags & (MSDA_FLAG_FOLD_OFF | MSDA_FLAG_DETERMINISTIC | MSDA_FLAG_FORCE_GENERIC | MSDA_FLAG_ORDER_LINEAR |
               MSDA_FLAG_ORDER_STRIP | MSDA_FLAG_ORDER_TILE2D))
    return false;
  if (dtype != MSDA_F32 && dtype != MSDA_BF16) return false;   // instantiated for float / bf16 values only
  if (!fast_ok(d, dtype, flags)) return false;
  if (d.Q != d.S) return false;                       // query i must be pixel i of the pyramid
  if (!(d.D == 32 || d.D == 64)) return false;
  if (fold_tile(d) == 0) return false;
  return (flags & MSDA_FLAG_FOLD_ON) != 0;
}

int bwd_fold(cudaStream_t st, const Dims& d, int dtype, const void* go, const void* value, const int64_t* shapes,
             const int64_t* lsi, const void* loc, const void* w, float* gv, void* gl, void* gw,
             const msda::FusedArgs* fa) {
  const int nq = fold_tile(d);
  const msda::FusedArgs a = fa ? *fa : msda::FusedArgs{};
  // fold_applies admits float / bf16 values and D in {32, 64}
  return with_types<TagList<MSDA_F32, MSDA_BF16>>(dtype, [&](auto t) {
    using VT = typename decltype(t)::VT;
    auto run = [&](auto PRE) {
      if (d.D == 32) return fold_pt<32, VT, PRE>(st, d, nq, go, value, shapes, lsi, loc, w, gv, gl, gw, a);
      return fold_pt<64, VT, PRE>(st, d, nq, go, value, shapes, lsi, loc, w, gv, gl, gw, a);
    };
    return fa ? run(Int<msda::kPreFused>{}) : run(Int<msda::kPrePlain>{});
  });
}

}  // namespace msda_host
#endif  // MSDA_EXPERIMENTS
