// msda_epilogue.cu -- fused residual add + LayerNorm, the epilogue of the op's callers (SURVEY section 8f-2).
//
// In the reference's encoder / decoder layers every MSDeformAttn call and every FFN is followed by
//   x = x + identity ; x = LayerNorm(x)
// (detrex/layers/transformer.py:152-192 runs "self_attn", "norm", "ffn", "norm"; the attention module adds its own
// residual, multi_scale_deform_attn.py:363; the FFN adds its identity, detrex/layers/mlp.py:127-132), i.e. an
// elementwise add kernel that writes the sum and a LayerNorm kernel that reads it back.  Here both are one pass:
//   forward   y = LN(a + b) * gamma + beta          reads a, b           writes y, mean[row], rstd[row]
//   backward  dx = dLN/d(a+b) (the gradient of BOTH inputs), dgamma, dbeta
//             reads dy, a, b (the sum is recomputed, never stored)       writes dx, per-CTA partials of dgamma / dbeta
// One warp per row, 16-byte lane accesses, two-pass mean / variance in registers (the row stays in registers), fp32
// arithmetic for float, bfloat16 and float16 tensors.  The mixed form (TA = 16-bit `a`, TB = float `b` / y / dy / dx)
// is the one autocast produces -- a 16-bit attention / FFN output plus a float32 residual -- and the backward then
// writes dx twice: as float for `b` and rounded for `a`.  dgamma / dbeta are reduced in a fixed order (per-CTA partial sums, then
// one small kernel), so the whole backward is bit-reproducible.  HBM-bound: 3 tensor passes forward, 4 backward.
#include "msda_host.h"

namespace {
using namespace msda_host;

constexpr int kLnThreads = 256;
constexpr int kLnMaxVec = 8;   // float4 chunks per lane: C <= 32 * 4 * 8 = 1024

__device__ __forceinline__ float4 ld_f4(const float* p) { return *reinterpret_cast<const float4*>(p); }
__device__ __forceinline__ float4 ld_f4(const __nv_bfloat16* p) {
  const uint2 u = *reinterpret_cast<const uint2*>(p);
  return make_float4(__uint_as_float(u.x << 16), __uint_as_float(u.x & 0xffff0000u), __uint_as_float(u.y << 16),
                     __uint_as_float(u.y & 0xffff0000u));
}
__device__ __forceinline__ float4 ld_f4(const __half* p) {
  const uint2 u = *reinterpret_cast<const uint2*>(p);
  const float2 lo = __half22float2(*reinterpret_cast<const __half2*>(&u.x));
  const float2 hi = __half22float2(*reinterpret_cast<const __half2*>(&u.y));
  return make_float4(lo.x, lo.y, hi.x, hi.y);
}
__device__ __forceinline__ void st_f4(float* p, float4 v) { *reinterpret_cast<float4*>(p) = v; }
__device__ __forceinline__ void st_f4(__half* p, float4 v) {
  const __half2 lo = __floats2half2_rn(v.x, v.y), hi = __floats2half2_rn(v.z, v.w);
  uint2 u;
  u.x = *reinterpret_cast<const unsigned*>(&lo);
  u.y = *reinterpret_cast<const unsigned*>(&hi);
  *reinterpret_cast<uint2*>(p) = u;
}
__device__ __forceinline__ void st_f4(__nv_bfloat16* p, float4 v) {
  const __nv_bfloat162 lo = __floats2bfloat162_rn(v.x, v.y), hi = __floats2bfloat162_rn(v.z, v.w);
  uint2 u;
  u.x = *reinterpret_cast<const unsigned*>(&lo);
  u.y = *reinterpret_cast<const unsigned*>(&hi);
  *reinterpret_cast<uint2*>(p) = u;
}
__device__ __forceinline__ float warp_sum(float v) {
#pragma unroll
  for (int k = 16; k > 0; k >>= 1) v += __shfl_xor_sync(0xffffffffu, v, k);
  return v;
}

// NV = float4 chunks per lane (C == 128 * NV exactly when EXACT, else C <= 128 * NV and chunks are predicated).
// T = the type of b and y; TA = the type of a (T, or a 16-bit type when T is float: the mixed form)
template <typename T, int NV, typename TA = T>
__global__ void __launch_bounds__(kLnThreads)
add_layernorm_fwd_kernel(const TA* __restrict__ a, const T* __restrict__ b, const float* __restrict__ gamma,
                         const float* __restrict__ beta, T* __restrict__ y, float* __restrict__ mean,
                         float* __restrict__ rstd, int64_t rows, int C, float eps) {
  const int lane = threadIdx.x & 31;
  const int64_t warp0 = (int64_t)blockIdx.x * (kLnThreads / 32) + (threadIdx.x >> 5);
  const int64_t stride = (int64_t)gridDim.x * (kLnThreads / 32);
  const float inv_c = 1.0f / (float)C;
  for (int64_t row = warp0; row < rows; row += stride) {
    const TA* pa = a + row * C;
    const T* pb = b + row * C;
    float4 s[NV];
    float sum = 0.0f;
#pragma unroll
    for (int v = 0; v < NV; ++v) {
      const int c = (v * 32 + lane) * 4;
      s[v] = make_float4(0.f, 0.f, 0.f, 0.f);
      if (c < C) {
        const float4 x = ld_f4(pa + c), r = ld_f4(pb + c);
        s[v] = make_float4(x.x + r.x, x.y + r.y, x.z + r.z, x.w + r.w);
        sum += (s[v].x + s[v].y) + (s[v].z + s[v].w);
      }
    }
    const float mu = warp_sum(sum) * inv_c;
    float var = 0.0f;
#pragma unroll
    for (int v = 0; v < NV; ++v) {
      const int c = (v * 32 + lane) * 4;
      if (c < C) {
        const float dx = s[v].x - mu, dy = s[v].y - mu, dz = s[v].z - mu, dw = s[v].w - mu;
        var += (dx * dx + dy * dy) + (dz * dz + dw * dw);
      }
    }
    const float rs = rsqrtf(warp_sum(var) * inv_c + eps);
#pragma unroll
    for (int v = 0; v < NV; ++v) {
      const int c = (v * 32 + lane) * 4;
      if (c < C) {
        const float4 g = __ldg(reinterpret_cast<const float4*>(gamma + c)), bt = __ldg(reinterpret_cast<const float4*>(beta + c));
        st_f4(y + row * C + c, make_float4((s[v].x - mu) * rs * g.x + bt.x, (s[v].y - mu) * rs * g.y + bt.y,
                                           (s[v].z - mu) * rs * g.z + bt.z, (s[v].w - mu) * rs * g.w + bt.w));
      }
    }
    if (lane == 0) {
      mean[row] = mu;
      rstd[row] = rs;
    }
  }
}

// dx = rstd * (g - mean(g) - xhat * mean(g * xhat)),  g = dy * gamma,  xhat = (a + b - mean) * rstd
// partial[blockIdx.x][0][c] = sum over the CTA's rows of dy * xhat (dgamma), [1][c] = sum of dy (dbeta)
// Mixed form (TA != T): dx_a = dx rounded to TA, stored in the same pass
template <typename T, int NV, typename TA = T>
__global__ void __launch_bounds__(kLnThreads)
add_layernorm_bwd_kernel(const T* __restrict__ dy, const TA* __restrict__ a, const T* __restrict__ b,
                         const float* __restrict__ gamma, const float* __restrict__ mean,
                         const float* __restrict__ rstd, T* __restrict__ dx, TA* __restrict__ dx_a,
                         float* __restrict__ partial, int64_t rows, int C) {
  static_assert(std::is_same_v<TA, T> || (std::is_same_v<T, float> && sizeof(TA) == 2), "mixed form: 16-bit a, float b");
  extern __shared__ __align__(16) float red[];          // [warps][2][C]
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const int64_t warp0 = (int64_t)blockIdx.x * (kLnThreads / 32) + warp;
  const int64_t stride = (int64_t)gridDim.x * (kLnThreads / 32);
  const float inv_c = 1.0f / (float)C;
  float4 dg[NV], db[NV], gm[NV];
#pragma unroll
  for (int v = 0; v < NV; ++v) {
    const int c = (v * 32 + lane) * 4;
    dg[v] = db[v] = make_float4(0.f, 0.f, 0.f, 0.f);
    gm[v] = (c < C) ? __ldg(reinterpret_cast<const float4*>(gamma + c)) : make_float4(0.f, 0.f, 0.f, 0.f);
  }
  for (int64_t row = warp0; row < rows; row += stride) {
    const float mu = mean[row], rs = rstd[row];
    float4 xh[NV], g[NV];
    float s1 = 0.0f, s2 = 0.0f;
#pragma unroll
    for (int v = 0; v < NV; ++v) {
      const int c = (v * 32 + lane) * 4;
      xh[v] = g[v] = make_float4(0.f, 0.f, 0.f, 0.f);
      if (c < C) {
        const float4 x = ld_f4(a + row * C + c), r = ld_f4(b + row * C + c), d = ld_f4(dy + row * C + c);
        xh[v] = make_float4((x.x + r.x - mu) * rs, (x.y + r.y - mu) * rs, (x.z + r.z - mu) * rs, (x.w + r.w - mu) * rs);
        g[v] = make_float4(d.x * gm[v].x, d.y * gm[v].y, d.z * gm[v].z, d.w * gm[v].w);
        s1 += (g[v].x + g[v].y) + (g[v].z + g[v].w);
        s2 += (g[v].x * xh[v].x + g[v].y * xh[v].y) + (g[v].z * xh[v].z + g[v].w * xh[v].w);
        dg[v].x += d.x * xh[v].x; dg[v].y += d.y * xh[v].y; dg[v].z += d.z * xh[v].z; dg[v].w += d.w * xh[v].w;
        db[v].x += d.x; db[v].y += d.y; db[v].z += d.z; db[v].w += d.w;
      }
    }
    const float m1 = warp_sum(s1) * inv_c, m2 = warp_sum(s2) * inv_c;
#pragma unroll
    for (int v = 0; v < NV; ++v) {
      const int c = (v * 32 + lane) * 4;
      if (c < C) {
        const float4 r = make_float4(rs * (g[v].x - m1 - xh[v].x * m2), rs * (g[v].y - m1 - xh[v].y * m2),
                                     rs * (g[v].z - m1 - xh[v].z * m2), rs * (g[v].w - m1 - xh[v].w * m2));
        st_f4(dx + row * C + c, r);
        if constexpr (!std::is_same_v<TA, T>) st_f4(dx_a + row * C + c, r);
      }
    }
  }
  // CTA-level reduction of dgamma / dbeta in a fixed order (warp 0..7), then one partial row per CTA
  float* mine = red + (size_t)warp * 2 * C;
#pragma unroll
  for (int v = 0; v < NV; ++v) {
    const int c = (v * 32 + lane) * 4;
    if (c < C) {
      *reinterpret_cast<float4*>(mine + c) = dg[v];
      *reinterpret_cast<float4*>(mine + C + c) = db[v];
    }
  }
  __syncthreads();
  for (int i = threadIdx.x; i < 2 * C; i += kLnThreads) {
    float acc = 0.0f;
#pragma unroll
    for (int w = 0; w < kLnThreads / 32; ++w) acc += red[(size_t)w * 2 * C + i];
    partial[(size_t)blockIdx.x * 2 * C + i] = acc;
  }
}

__global__ void add_layernorm_param_grad_kernel(const float* __restrict__ partial, int n_partial, int C,
                                                float* __restrict__ dgamma, float* __restrict__ dbeta) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= 2 * C) return;
  float acc = 0.0f;
  for (int p = 0; p < n_partial; ++p) acc += partial[(size_t)p * 2 * C + i];
  if (i < C) dgamma[i] = acc;
  else dbeta[i - C] = acc;
}

int ln_grid(int64_t rows) {
  int dev = 0, sms = 148;
  if (cudaGetDevice(&dev) == cudaSuccess) cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev);
  const int64_t need = (rows + kLnThreads / 32 - 1) / (kLnThreads / 32);
  const int64_t cap = (int64_t)sms * 8;                  // 8 CTAs of 256 threads per SM
  return (int)(need < cap ? (need < 1 ? 1 : need) : cap);
}

// Calls f(Int<NV>{}) with the float4 chunks per lane the kernels are instantiated for: the least of 1, 2, 4, 8
// covering C channels
template <typename F>
int with_nv(int C, F&& f) {
  switch ((C + 127) / 128) {
    case 1: return f(Int<1>{});
    case 2: return f(Int<2>{});
    case 3: case 4: return f(Int<4>{});
    default: return f(Int<8>{});
  }
}

int check_ln(int64_t rows, int C, int dtype) {
  if (rows < 0 || C < 0) return fail(MSDA_ERR_INVALID_ARGUMENT, "negative size (rows=%lld C=%d)", (long long)rows, C);
  if (dtype != MSDA_F32 && dtype != MSDA_BF16 && dtype != MSDA_F16)
    return fail(MSDA_ERR_UNSUPPORTED, "add_layernorm: float32 / bfloat16 / float16 only");
  if (C % 4 != 0 || C > 128 * kLnMaxVec)
    return fail(MSDA_ERR_UNSUPPORTED, "add_layernorm: channels must be a multiple of 4 and <= %d (got %d)", 128 * kLnMaxVec, C);
  return MSDA_OK;
}

}  // namespace

extern "C" size_t msda_add_layernorm_workspace_bytes(int64_t rows, int channels) {
  if (rows <= 0 || channels <= 0) return 0;
  return (size_t)ln_grid(rows) * 2 * (size_t)channels * sizeof(float);
}

namespace {
// The bodies of the same-dtype entry points (MIXED false: a, b, y, grad_* all `dtype`) and of the mixed ones (MIXED
// true: `a` / grad_a in the 16-bit `dtype`, b, y, grad_y, grad_b float), after check_ln.
template <bool MIXED>
int ln_forward(void* stream, const void* a, const void* b, const float* gamma, const float* beta, int64_t rows,
               int channels, float eps, void* y, float* mean, float* rstd, int dtype) {
  if (rows == 0 || channels == 0) return MSDA_OK;
  if (!a || !b || !gamma || !beta || !y || !mean || !rstd) return fail(MSDA_ERR_INVALID_ARGUMENT, "null tensor pointer");
  if (int s = check_alignment({{"a", a}, {"b", b}, {"gamma", gamma}, {"beta", beta}, {"y", y}})) return s;
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  const int grid = ln_grid(rows);
  return with_types<FastTags>(dtype, [&](auto t) {
    using TA = typename decltype(t)::VT;
    using T = std::conditional_t<MIXED, float, TA>;
    return with_nv(channels, [&](auto NV) {
      add_layernorm_fwd_kernel<T, NV, TA><<<grid, kLnThreads, 0, st>>>((const TA*)a, (const T*)b, gamma, beta, (T*)y,
                                                                       mean, rstd, rows, channels, eps);
      return launched();
    });
  });
}

template <bool MIXED>
int ln_backward(void* stream, const void* grad_y, const void* a, const void* b, const float* gamma, const float* mean,
                const float* rstd, int64_t rows, int channels, void* grad_x, void* grad_a, float* grad_gamma,
                float* grad_beta, void* workspace, size_t workspace_bytes, int dtype) {
  if (channels == 0) return MSDA_OK;
  if (!grad_gamma || !grad_beta) return fail(MSDA_ERR_INVALID_ARGUMENT, "grad_gamma / grad_beta is null");
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  if (rows == 0) {
    MSDA_CUDA(cudaMemsetAsync(grad_gamma, 0, (size_t)channels * sizeof(float), st));
    MSDA_CUDA(cudaMemsetAsync(grad_beta, 0, (size_t)channels * sizeof(float), st));
    return MSDA_OK;
  }
  if (!grad_y || !a || !b || !gamma || !mean || !rstd || !grad_x || (MIXED && !grad_a))
    return fail(MSDA_ERR_INVALID_ARGUMENT, "null tensor pointer");
  if (int s = check_alignment({{"grad_y", grad_y}, {"a", a}, {"b", b}, {"gamma", gamma},
                               {MIXED ? "grad_b" : "grad_x", grad_x}, {"grad_a", MIXED ? grad_a : nullptr},
                               {"workspace", workspace}}))
    return s;
  if (int s = check_workspace(workspace, workspace_bytes, msda_add_layernorm_workspace_bytes(rows, channels))) return s;
  const int grid = ln_grid(rows);
  const size_t smem = (size_t)(kLnThreads / 32) * 2 * channels * sizeof(float);
  float* partial = static_cast<float*>(workspace);
  if (int s = with_types<FastTags>(dtype, [&](auto t) {
        using TA = typename decltype(t)::VT;
        using T = std::conditional_t<MIXED, float, TA>;
        return with_nv(channels, [&](auto NV) {
          auto k = add_layernorm_bwd_kernel<T, NV, TA>;
          MSDA_CUDA(ensure_smem(k, smem));
          k<<<grid, kLnThreads, smem, st>>>((const T*)grad_y, (const TA*)a, (const T*)b, gamma, mean, rstd, (T*)grad_x,
                                            (TA*)grad_a, partial, rows, channels);
          return launched();
        });
      }))
    return s;
  add_layernorm_param_grad_kernel<<<(2 * channels + 255) / 256, 256, 0, st>>>(partial, grid, channels, grad_gamma, grad_beta);
  return launched();
}

// the mixed form: `a` bfloat16 or float16, everything else float
int check_ln_mixed(int64_t rows, int C, int a_dtype) {
  if (a_dtype != MSDA_BF16 && a_dtype != MSDA_F16)
    return fail(MSDA_ERR_UNSUPPORTED, "add_layernorm mixed: `a` must be bfloat16 or float16 (b float32)");
  return check_ln(rows, C, a_dtype);
}
}  // namespace

extern "C" {

int msda_add_layernorm_forward(void* stream, const void* a, const void* b, const float* gamma, const float* beta,
                               int64_t rows, int channels, float eps, void* y, float* mean, float* rstd, int dtype) {
  if (int s = check_ln(rows, channels, dtype)) return s;
  return ln_forward<false>(stream, a, b, gamma, beta, rows, channels, eps, y, mean, rstd, dtype);
}

int msda_add_layernorm_backward(void* stream, const void* grad_y, const void* a, const void* b, const float* gamma,
                                const float* mean, const float* rstd, int64_t rows, int channels, void* grad_x,
                                float* grad_gamma, float* grad_beta, void* workspace, size_t workspace_bytes,
                                int dtype) {
  if (int s = check_ln(rows, channels, dtype)) return s;
  return ln_backward<false>(stream, grad_y, a, b, gamma, mean, rstd, rows, channels, grad_x, nullptr, grad_gamma,
                            grad_beta, workspace, workspace_bytes, dtype);
}

int msda_add_layernorm_mixed_forward(void* stream, const void* a, const float* b, const float* gamma,
                                     const float* beta, int64_t rows, int channels, float eps, float* y, float* mean,
                                     float* rstd, int a_dtype) {
  if (int s = check_ln_mixed(rows, channels, a_dtype)) return s;
  return ln_forward<true>(stream, a, b, gamma, beta, rows, channels, eps, y, mean, rstd, a_dtype);
}

int msda_add_layernorm_mixed_backward(void* stream, const float* grad_y, const void* a, const float* b,
                                      const float* gamma, const float* mean, const float* rstd, int64_t rows,
                                      int channels, void* grad_a, float* grad_b, float* grad_gamma, float* grad_beta,
                                      void* workspace, size_t workspace_bytes, int a_dtype) {
  if (int s = check_ln_mixed(rows, channels, a_dtype)) return s;
  return ln_backward<true>(stream, grad_y, a, b, gamma, mean, rstd, rows, channels, grad_b, grad_a, grad_gamma,
                           grad_beta, workspace, workspace_bytes, a_dtype);
}

}  // extern "C"
