/*
 * msda.h -- C ABI of the B200-native multi-scale deformable attention library (libmsda_b200.so).
 *
 * This is the drop-in boundary for the reference's native MSDeformAttn pair.  A maintainer of
 * the reference binds these entry points where detrex binds its own kernels today
 * (INTEGRATION.md shows the ctypes / pybind stub):
 *
 *   msda_forward   replaces  ms_deformable_im2col_cuda<T>
 *                  (/root/reference/detrex/layers/csrc/MsDeformAttn/ms_deform_im2col_cuda.cuh:923-954),
 *                  i.e. the body of ms_deform_attn_cuda_forward (ms_deform_attn_cuda.cu:21-81),
 *                  exported to Python as detrex._C.ms_deform_attn_forward (csrc/vision.cpp:55).
 *   msda_backward  replaces  ms_deformable_col2im_cuda<T> (ms_deform_im2col_cuda.cuh:956-1327),
 *                  i.e. the body of ms_deform_attn_cuda_backward (ms_deform_attn_cuda.cu:84-154),
 *                  exported as detrex._C.ms_deform_attn_backward (csrc/vision.cpp:56).
 *
 * Argument order and meaning follow those two launchers: stream first, then the tensors, then
 * (batch, spatial_size, num_heads, channels, num_levels, num_query, num_point), then outputs.
 * Differences, all deliberate:
 *   - plain C: no ATen / torch types, `void*` for the stream (a cudaStream_t);
 *   - a dtype tag instead of a C++ template: float, double, bfloat16 or float16 value with float
 *     locations / weights (the reference has float and double only);
 *   - errors are RETURNED (the reference only printf's launch failures, cuh:948-952);
 *   - no im2col_step: the whole batch is one launch (ms_deform_attn_cuda.cu:51-76 chunked it);
 *   - backward takes a caller-owned workspace (size from msda_backward_workspace_bytes) because
 *     the library never allocates device memory.
 *
 * Tensor layouts (all contiguous, all device pointers, as the reference asserts
 * ms_deform_attn_cuda.cu:29-39):
 *   value              [B, S, H, D]        dtype
 *   spatial_shapes     [L, 2]  int64  (H_l, W_l)
 *   level_start_index  [L]     int64
 *   sampling_loc       [B, Q, H, L, P, 2]  (x, y) normalised to [0,1] over the level; float
 *                                          (double when dtype == MSDA_F64)
 *   attn_weight        [B, Q, H, L, P]     same type as sampling_loc
 *   output / grad_output        [B, Q, H*D]   dtype
 *   grad_value         [B, S, H, D]        dtype        (zero-filled by the library)
 *   grad_sampling_loc, grad_attn_weight    shaped/typed like sampling_loc / attn_weight
 *                                          (fully written by the library, no pre-zeroing needed)
 * Every tensor pointer (workspaces included) must be 16-byte aligned: rows are read and written with 128-bit
 * accesses.  A torch / cudaMalloc allocation is; a view with an odd storage offset may not be -- such a call returns
 * MSDA_ERR_INVALID_ARGUMENT (the Python wrappers re-align by copying).  The reference's scalar kernels had no such
 * requirement.
 *
 * Thread safety: re-entrant, no global mutable state except a launch counter and a
 * thread-local last-error string; no library-owned streams, events or locks.  Work is enqueued on `stream` of the device that owns `value`
 * (the library switches to that device for the call and restores the previous one).
 */
#ifndef MSDA_B200_H_
#define MSDA_B200_H_

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define MSDA_ABI_VERSION 3

/* dtype tags */
#define MSDA_F32 0  /* value/out/grads float,  loc/w float  */
#define MSDA_F64 1  /* everything double (gradcheck path; generic kernels only) */
#define MSDA_BF16 2 /* value/out/grad_out/grad_value bfloat16, loc/w and their grads float, fp32 accumulate */
/* value/out/grad_out/grad_value float16, loc/w and their grads float, fp32 accumulate.  Every kernel widens the
 * float16 operands exactly, so out / grad_value equal the MSDA_F32 results on the widened tensors rounded once to
 * float16, and the float gradients equal them bit for bit (grad_value with float reds: up to the run-to-run
 * difference of the red order).  Added in ABI 3 without a version bump: an older library answers
 * MSDA_ERR_INVALID_ARGUMENT ("unknown dtype tag"). */
#define MSDA_F16 3
/* The autocast forms of the fused module paths (msda_fused_*, msda_dcnv3_fused_*): value / output / grad_output /
 * grad_value (input / grad_input for DCNv3) AND the projection tensors -- sampling_offsets / attn_logits (DCNv3:
 * offset / mask_logits) and their gradients -- in that 16-bit type, as the module's Linear layers produce them under
 * autocast; reference_points stay float.  The kernels widen the 16-bit offsets / logits exactly, so output and
 * grad_value are those of MSDA_BF16 / MSDA_F16 called with the widened tensors, and the offset / logit gradients are
 * the float gradients of that call rounded once, to nearest even (what a cast of them gives), except that a NaN
 * gradient's payload may differ from the cast's: only NaN-ness is promised.  Accepted by msda_fused_supported,
 * msda_fused_forward / _backward, msda_dcnv3_fused_forward / _backward and the two backward workspace queries (which
 * answer exactly what they answer for MSDA_BF16 / MSDA_F16); every other entry point refuses them as an unknown tag,
 * before any device work.  Added in ABI 3 without a version bump: an older library refuses them the same way. */
#define MSDA_BF16_AUX16 4
#define MSDA_F16_AUX16 5

/* status codes */
#define MSDA_OK 0
#define MSDA_ERR_INVALID_ARGUMENT 1 /* null pointer, negative size, unknown dtype ...            */
#define MSDA_ERR_UNSUPPORTED 2      /* shape outside what any kernel handles                     */
#define MSDA_ERR_WORKSPACE 3        /* workspace missing or smaller than msda_backward_workspace_bytes */
#define MSDA_ERR_CUDA 4             /* a CUDA runtime call or kernel launch failed; see msda_last_error_message */

/* flags (bit set) */
/* Backward: bit-reproducible grad_value.  Contributions are accumulated as 64-bit fixed point
 * (integer atomics commute, float atomics do not) with a power-of-two scale derived from
 * max|grad_output| * max|attn_weight|, then converted once: run-to-run identical, absolute error
 * <= 2^-38 of that bound per contribution, headroom for 2^25 maximal contributions per element.
 * On the fast shapes the accumulation is a sorted segment reduction (points binned by bilinear cell, one
 * lane group per output pixel gathers its bins and sums in registers: no atomics on grad_value, no
 * zero-fill); elsewhere 64-bit integer reds.  Both produce identical bits.
 * grad_sampling_loc / grad_attn_weight are reproducible in every mode (fixed reduction order). */
#define MSDA_FLAG_DETERMINISTIC (1u << 0)
/* With MSDA_FLAG_DETERMINISTIC: use the fixed-point RED path even where the sorted segment reduction
 * (msda_det.cuh) is available (A/B testing; both give the same bits). */
#define MSDA_FLAG_DET_ATOMIC (1u << 6)
/* With MSDA_FLAG_DETERMINISTIC (sorted path): fill the bins with a separate pass over the locations instead of from
 * the backward kernel itself (A/B testing; both give the same bits, the separate pass is slower). */
#define MSDA_FLAG_DET_SEPARATE_FILL (1u << 14)
#define MSDA_FLAG_FORCE_GENERIC (1u << 1) /* bypass the D in {16,32,64,128} fast kernels             */
/* Row order = which rows a CTA works on.  A scheduling choice only: results never depend on it.  The PRODUCT library
 * carries one order per pass -- forward LINEAR, backward STRIP, the fastest pair on every measured configuration -- and
 * treats the three flags below as hints it ignores; experiment builds (msda_build_config() & MSDA_BUILD_EXPERIMENTS) and
 * the variant builds of tools/build_variant.sh instantiate all three orders for both passes and honour them. */
#define MSDA_FLAG_ORDER_LINEAR (1u << 2)  /* rows in memory order (b, q, h)                              */
/* One CTA = a strip of consecutive queries of ONE head (any Q): x-adjacent queries re-use corner lines in L1. */
#define MSDA_FLAG_ORDER_STRIP (1u << 4)
/* Encoder form only (Q == S): one CTA = a pixel tile (8x4 at D=32) of one level and ONE head. */
#define MSDA_FLAG_ORDER_TILE2D (1u << 5)
/* Bits 3 and 7-10 selected round-1 experiments (persistent TILED order, shared-memory accumulation of the coarse
 * levels on a side stream, head-major strips) that were measured slower and removed; they are reserved and
 * ignored. */

/* EXPERIMENT BUILDS ONLY (msda_build_config() & MSDA_BUILD_EXPERIMENTS; the product library ignores both bits).
 * Backward, encoder form (Q == S, query i is pixel i of the pyramid), D in {32, 64}, float accumulation:
 * grad_value contributions of an 8x8 query tile of one head are pre-added ON THE SM (pixel-keyed lists in
 * shared memory, csrc/msda_fold.cuh) and leave it as ONE vector red per distinct destination row instead of one
 * per (point, corner): 5.5x fewer reds on model-like inputs (profiles/r02a_fold_rate_cfg2.json) -- and 2-2.5x
 * SLOWER, because the bookkeeping more than doubles the instruction count (profiles/r02b_fold_experiment.txt).
 * grad_sampling_loc / grad_attn_weight are bit-identical to the other kernels'; grad_value differs by float
 * summation order only.  FOLD_OFF wins over FOLD_ON; an explicit ORDER_* flag, MSDA_FLAG_DETERMINISTIC and
 * MSDA_FLAG_FORCE_GENERIC also select the non-folding kernels. */
#define MSDA_FLAG_FOLD_ON (1u << 12)
#define MSDA_FLAG_FOLD_OFF (1u << 13)

/* Backward: the caller does not need grad_value (autograd: value.requires_grad is False, e.g. a frozen memory
 * branch).  On the shapes the fast kernels cover (msda_dispatch_name(..., backward=1) is "bwd_fast_...") the
 * grad_value scatter -- the dominant cost of the backward -- is compiled out: grad_value may be NULL and is left
 * untouched, no workspace is needed, grad_sampling_loc / grad_attn_weight are as always.  Elsewhere the flag is
 * ignored and grad_value must be a valid buffer. */
#define MSDA_FLAG_NO_GRAD_VALUE (1u << 11)

int msda_abi_version(void);
/* How this library was built: 0 for the product library. */
#define MSDA_BUILD_EXPERIMENTS 1u /* -DMSDA_EXPERIMENTS: the measured-slower experiments are compiled in   */
#define MSDA_BUILD_SLIM 2u        /* -DMSDA_EXP_SLIM: only D = 32, P in {4, 8} of the plain operator       */
unsigned msda_build_config(void);

/* Forward.  Returns MSDA_OK or an error code.  B*Q*H*D == 0 is a no-op. */
int msda_forward(void* stream, const void* value, const int64_t* spatial_shapes,
                 const int64_t* level_start_index, const void* sampling_loc, const void* attn_weight,
                 int batch, int spatial_size, int num_heads, int channels, int num_levels,
                 int num_query, int num_point, void* output, int dtype, unsigned flags);

/* Bytes of device scratch msda_backward needs for this problem (0 is possible). */
size_t msda_backward_workspace_bytes(int batch, int spatial_size, int num_heads, int channels,
                                     int num_levels, int num_query, int num_point, int dtype,
                                     unsigned flags);

/* Backward: the three gradients of the forward above w.r.t. value, sampling_loc, attn_weight. */
int msda_backward(void* stream, const void* grad_output, const void* value,
                  const int64_t* spatial_shapes, const int64_t* level_start_index,
                  const void* sampling_loc, const void* attn_weight, int batch, int spatial_size,
                  int num_heads, int channels, int num_levels, int num_query, int num_point,
                  void* grad_value, void* grad_sampling_loc, void* grad_attn_weight,
                  void* workspace, size_t workspace_bytes, int dtype, unsigned flags);

/*
 * Fused module path (SURVEY.md section 8f-1; an extension, the reference has no counterpart): the
 * softmax over L*P and the sampling-location arithmetic of MultiScaleDeformableAttention.forward
 * (/root/reference/detrex/layers/multi_scale_deform_attn.py:300-332) run inside the kernels, so
 * sampling_locations / attention_weights and their gradients never exist in HBM.
 *   sampling_offsets  [B, Q, H, L, P, 2] float  raw output of the module's sampling_offsets Linear
 *   attn_logits       [B, Q, H, L*P]     float  raw output of its attention_weights Linear (pre-softmax)
 *   reference_points  [B, Q, L, ref_dim] float  ref_dim 2: loc = ref + off / (W_l, H_l)   (py:320-324)
 *                                               ref_dim 4: loc = ref_xy + off / P * ref_wh * 0.5 (py:326-332)
 *   value_padding_mask [B, S] uint8, or NULL    the module's key_padding_mask (non-zero = padded pixel): its
 *                                               value.masked_fill(key_padding_mask[..., None], 0) (py:291-292)
 *                                               is folded into the kernels -- a masked pixel's value row reads
 *                                               as zeros in the output and in every gradient, and its
 *                                               grad_value is 0 -- so `value` is passed UNMASKED and the
 *                                               masked copy (one read + one write of value per layer, and the
 *                                               same again in backward) never exists
 * Backward returns grad_value plus the gradients w.r.t. the two RAW tensors (what the Linear layers'
 * backward consumes); it uses the same workspace rule as msda_backward.  With MSDA_BF16_AUX16 / MSDA_F16_AUX16
 * sampling_offsets, attn_logits, grad_offsets and grad_logits are in the value's 16-bit type (hence `void*`).
 * Only the fast kernels have a fused form: otherwise MSDA_ERR_UNSUPPORTED is returned (query with
 * msda_fused_supported) and the caller composes softmax / affine itself around msda_forward / msda_backward.
 */
int msda_fused_supported(int channels, int num_levels, int num_point, int spatial_size, int num_heads,
                         int dtype, unsigned flags);
int msda_fused_forward(void* stream, const void* value, const int64_t* spatial_shapes,
                       const int64_t* level_start_index, const void* sampling_offsets,
                       const void* attn_logits, const float* reference_points, int ref_dim,
                       const uint8_t* value_padding_mask, int batch, int spatial_size, int num_heads,
                       int channels, int num_levels, int num_query, int num_point, void* output, int dtype,
                       unsigned flags);
int msda_fused_backward(void* stream, const void* grad_output, const void* value,
                        const int64_t* spatial_shapes, const int64_t* level_start_index,
                        const void* sampling_offsets, const void* attn_logits,
                        const float* reference_points, int ref_dim, const uint8_t* value_padding_mask,
                        int batch, int spatial_size, int num_heads, int channels, int num_levels,
                        int num_query, int num_point, void* grad_value, void* grad_offsets,
                        void* grad_logits, void* workspace, size_t workspace_bytes, int dtype,
                        unsigned flags);

/*
 * Packed (padding-free) form of the fused module path: a batch of differently sized images without padding, the
 * equivalent of FlashAttention's "varlen" interface.  Image b's pixels of level l are its valid top-left rectangle
 * h_v[b,l] x w_v[b,l] of the padded level (H_l, W_l), stored row-major with row pitch w_v; the levels of an image follow
 * each other and the images are concatenated, so
 *   value              [T_v, H, D]             dtype (T_v = total_value, the valid pixels of all images)
 *   sampling_offsets   [T_q, H, L, P, 2]       float or (MSDA_*_AUX16) the value's 16-bit type
 *   attn_logits        [T_q, H, L*P]           as sampling_offsets
 *   reference_points   [T_q, L, ref_dim]       float
 *   output / grad_output  [T_q, H*D]           dtype (T_q = total_query)
 *   grad_value         [T_v, H, D]             dtype; grad_offsets / grad_logits shaped and typed like their inputs
 *   spatial_shapes     [L, 2] int64            the PADDED level shapes (H_l, W_l)
 *   image_meta         [batch, 4 + 3*L] int64  per image {value_start, value_count, query_start, query_count} and per
 *                                              level {h_v, w_v, start of the level inside the image}; query rows
 *                                              query_start .. +query_count belong to image b
 * Queries of image b sample image b only.  Locations stay normalised over the padded level (the location affine and
 * the gate use (H_l, W_l)); a bilinear corner counts iff it lies inside image b's valid rectangle.  So every query's
 * output, grad_offsets and grad_logits are the same bits msda_fused_forward / _backward give for the padded batch with
 * the rectangle as value_padding_mask, and grad_value equals theirs at the valid pixels up to the order of the float
 * reds.  Encoder self-attention: the queries are the value tokens (query_start == value_start); decoder
 * cross-attention: query_start = b*Q over packed memory.
 * max_image_value / max_image_query: the largest value_count / query_count (host integers; the grid is sized for
 * them and every image's value_count * H * D must stay below 2^31).  The metadata is read on the device only -- no
 * host copy, sync or allocation, so both calls are CUDA-graph capturable -- and is TRUSTED: the product library does
 * not check it against the totals; a -DMSDA_DEBUG_BOUNDS build traps on any corner outside its image.
 * Empty problems (batch, total_query or H*D zero) are no-ops; total_value == 0 zero-fills the output (backward: the
 * offset / logit gradients) without a kernel.  The backward uses float reds; with MSDA_FLAG_DETERMINISTIC it returns
 * MSDA_ERR_UNSUPPORTED before any device work (unpack, use msda_fused_* / msda_backward, pack).  Its workspace is
 * msda_packed_backward_workspace_bytes (T_v*H*D floats for 16-bit values, else 0).  Every other flag bit is ignored.
 * Added in ABI 3 without a version bump: an older library lacks the three symbols.
 */
size_t msda_packed_backward_workspace_bytes(int total_value, int num_heads, int channels, int dtype, unsigned flags);
int msda_packed_forward(void* stream, const void* value, const int64_t* spatial_shapes, const int64_t* image_meta,
                        const void* sampling_offsets, const void* attn_logits, const float* reference_points,
                        int ref_dim, int batch, int total_value, int num_heads, int channels, int num_levels,
                        int total_query, int num_point, int max_image_value, int max_image_query, void* output,
                        int dtype, unsigned flags);
int msda_packed_backward(void* stream, const void* grad_output, const void* value, const int64_t* spatial_shapes,
                         const int64_t* image_meta, const void* sampling_offsets, const void* attn_logits,
                         const float* reference_points, int ref_dim, int batch, int total_value, int num_heads,
                         int channels, int num_levels, int total_query, int num_point, int max_image_value,
                         int max_image_query, void* grad_value, void* grad_offsets, void* grad_logits,
                         void* workspace, size_t workspace_bytes, int dtype, unsigned flags);

/*
 * DCNv3 core op (SURVEY.md section 8f-4): the other native op of detrex._C, same gather/scatter core.
 *   msda_dcnv3_forward   replaces dcnv3_im2col_cuda<T>
 *       (/root/reference/detrex/layers/csrc/DCNv3/dcnv3_im2col_cuda.cuh:840-868), i.e. _C.dcnv3_forward
 *       (csrc/vision.cpp:57); msda_dcnv3_backward replaces dcnv3_col2im_cuda<T> (:870-), _C.dcnv3_backward.
 * Argument order follows those launchers.  Layouts (contiguous, channels last, as dcn_v3.py:464-489):
 *   input  [N, H_in, W_in, group*group_channels]   dtype (MSDA_F32, MSDA_BF16 or MSDA_F16)
 *   offset [N, H_out, W_out, group*K*2] float, K = kernel_h*kernel_w, point index = i*kernel_h + j
 *          with i over kernel_w (the reference kernel's loop order), (x, y) per point, in pixels
 *   mask   [N, H_out, W_out, group*K]   float
 *   output / grad_output [N, H_out, W_out, group*group_channels] dtype
 * The input is NOT padded by the caller: pad_h / pad_w only shift the sampling grid and samples outside
 * the map read zeros, exactly like the reference kernel.  Supported: group_channels in {16,32,64,128},
 * K <= 64, float32 / bfloat16 / float16 input (MSDA_ERR_UNSUPPORTED otherwise).
 * The backward's workspace comes from msda_dcnv3_backward_workspace_bytes; less gives MSDA_ERR_WORKSPACE.  Without
 * MSDA_FLAG_DETERMINISTIC that is 0 for float32 and N*H_in*W_in*C floats for bfloat16 / float16 (grad_input is
 * accumulated in float with float reds, whose rounding depends on arrival order).
 * msda_dcnv3_backward honours MSDA_FLAG_DETERMINISTIC, MSDA_FLAG_DET_ATOMIC and MSDA_FLAG_DET_SEPARATE_FILL and ignores
 * every other bit.  With MSDA_FLAG_DETERMINISTIC grad_input is bit-reproducible: it is the deterministic backward of
 * the equivalent one-level msda_backward problem (value = input [N, H_in*W_in, group, group_channels],
 * Q = H_out*W_out, P = K), 64-bit fixed point summed by the sorted segment reduction or, with MSDA_FLAG_DET_ATOMIC or
 * beyond its 32-bit index limits, by integer reds -- all routes give the same bits -- and converted once into the
 * input's dtype.  grad_offset / grad_mask are the same bits as without the flag.  The workspace is then
 *   256 + msda_backward_workspace_bytes(N, H_in*W_in, group, group_channels, 1, H_out*W_out, K, dtype,
 *                                       flags & (DETERMINISTIC | DET_ATOMIC | DET_SEPARATE_FILL))
 * bytes (the first 256 hold the one-level table the kernels read), except for empty problems (N, H_in*W_in or
 * H_out*W_out zero), which need and do exactly what they do without the flag.
 */
size_t msda_dcnv3_backward_workspace_bytes(int kernel_h, int kernel_w, int group, int group_channels, int batch,
                                           int height_in, int width_in, int height_out, int width_out, int dtype,
                                           unsigned flags);
int msda_dcnv3_forward(void* stream, const void* input, const float* offset, const float* mask,
                       int kernel_h, int kernel_w, int stride_h, int stride_w, int pad_h, int pad_w,
                       int dilation_h, int dilation_w, int group, int group_channels, float offset_scale,
                       int batch, int height_in, int width_in, int height_out, int width_out,
                       void* output, int dtype, unsigned flags);
int msda_dcnv3_backward(void* stream, const void* grad_output, const void* input, const float* offset,
                        const float* mask, int kernel_h, int kernel_w, int stride_h, int stride_w,
                        int pad_h, int pad_w, int dilation_h, int dilation_w, int group,
                        int group_channels, float offset_scale, int batch, int height_in, int width_in,
                        int height_out, int width_out, void* grad_input, float* grad_offset,
                        float* grad_mask, void* workspace, size_t workspace_bytes, int dtype,
                        unsigned flags);

/*
 * Fused DCNv3 module path (an extension; the reference has no counterpart): the DCNv3 module's mask softmax
 * (dcn_v3.py:476, softmax over the K points of every (output pixel, group)) runs inside the kernels, so the mask and
 * its gradient never exist in HBM.  Arguments, layouts, geometry, supported shapes and dtypes are those of
 * msda_dcnv3_forward / msda_dcnv3_backward, with
 *   mask_logits       [N, H_out, W_out, group*K] float  the raw output of the module's mask Linear (pre-softmax)
 *   grad_mask_logits  [N, H_out, W_out, group*K] float  its gradient (fully written by the library)
 * in place of mask / grad_mask (with MSDA_BF16_AUX16 / MSDA_F16_AUX16: offset, mask_logits and their gradients in
 * the input's 16-bit type, hence `void*`; before those tags the prototypes read `const float* mask_logits` /
 * `float* grad_mask_logits`, and since a float pointer converts to `void*` implicitly, such callers compile and link
 * unchanged -- the same holds for the four pointers of msda_fused_forward / _backward).  The result equals
 * msda_dcnv3_forward / _backward called with mask = softmax(mask_logits) over each row of K, followed by the softmax's
 * chain rule grad_logit_i = w_i * (grad_mask_i - sum_j grad_mask_j * w_j), up to float rounding of the softmax.
 * Non-finite logits behave as in torch.softmax: a -inf logit gets weight 0 (and gradient 0) while the rest of its row is
 * normalised as usual; a row whose logits are all -inf, or that holds +inf or NaN, has NaN weights: its logits'
 * gradient is NaN, and so are its output pixel and its grad_offset / grad_input contributions wherever one of its
 * points samples inside the map (exactly what msda_dcnv3_* make of torch.softmax's NaN row).
 * Backward uses the workspace rule of msda_dcnv3_backward_workspace_bytes with flags 0 (float reds).  It has no
 * deterministic form: with MSDA_FLAG_DETERMINISTIC it returns MSDA_ERR_UNSUPPORTED before any device work (compose
 * the softmax around msda_dcnv3_backward instead, whose grad_input is bit-reproducible).  Every other flag bit is
 * ignored by both entry points.  Added in ABI 3 without a version bump: an older library lacks the two symbols.
 */
int msda_dcnv3_fused_forward(void* stream, const void* input, const void* offset, const void* mask_logits,
                             int kernel_h, int kernel_w, int stride_h, int stride_w, int pad_h, int pad_w,
                             int dilation_h, int dilation_w, int group, int group_channels, float offset_scale,
                             int batch, int height_in, int width_in, int height_out, int width_out,
                             void* output, int dtype, unsigned flags);
int msda_dcnv3_fused_backward(void* stream, const void* grad_output, const void* input, const void* offset,
                              const void* mask_logits, int kernel_h, int kernel_w, int stride_h, int stride_w,
                              int pad_h, int pad_w, int dilation_h, int dilation_w, int group,
                              int group_channels, float offset_scale, int batch, int height_in, int width_in,
                              int height_out, int width_out, void* grad_input, void* grad_offset,
                              void* grad_mask_logits, void* workspace, size_t workspace_bytes, int dtype,
                              unsigned flags);

/*
 * Deformable convolution v1 / v2 (detectron2's DeformConv / ModulatedDeformConv, SURVEY.md section 2.1 row 12) as
 * im2col + GEMM: these two entry points build the column matrix and scatter its gradient back; the products with the
 * weight are dense GEMMs the caller runs (cuBLAS).  They replace detectron2/layers/csrc/deformable/
 * deform_conv_cuda_kernel.cu:
 *   msda_dcnv2_im2col   deformable_im2col (mask = NULL, DCNv1) and modulated_deformable_im2col_cuda (DCNv2)
 *   msda_dcnv2_col2im   modulated_deformable_col2im_cuda (grad_input) + modulated_deformable_col2im_coord_cuda
 *                       (grad_offset, grad_mask) in one pass; with mask = NULL the DCNv1 deformable_col2im +
 *                       deformable_col2im_coord
 * Layouts (contiguous; K = kernel_h*kernel_w, tap k = i*kernel_w + j; P = H_out*W_out):
 *   input / grad_input       [N, H_in, W_in, C]                   dtype (channels last)
 *   offset / grad_offset     [N, H_out, W_out, dg, K, 2]          (dy, dx) per tap, in pixels (detectron2's channel
 *                                                                 order dg*K*2, channels last)
 *   mask / grad_mask         [N, H_out, W_out, dg, K]             NULL for DCNv1 (grad_mask then unused)
 *   columns / grad_columns   [N*P, groups, K, C/groups]           dtype; the (k, c) order of a row is that of
 *                                                                 weight.permute(0, 2, 3, 1) [C_out, kh, kw, C/groups]
 * dg = deformable_groups; channel c samples with the offsets of group c / (C/dg).  Sampling position of tap (i, j) at
 * output (ho, wo): y = (ho*stride_h - pad_h + i*dilation_h) + dy, x likewise -- the integer base plus the offset, one
 * rounding, as torchvision.ops.deform_conv2d -- bilinear, zero outside the map, a tap contributes only where
 * y > -1 && y < H_in && x > -1 && x < W_in.  columns = mask * sample.  H_out / W_out must be what the geometry gives
 * ((H_in + 2*pad_h - (dilation_h*(kernel_h-1) + 1)) / stride_h + 1), else MSDA_ERR_INVALID_ARGUMENT; C must be
 * divisible by groups and by deformable_groups.
 * dtype: MSDA_F32, MSDA_F64, MSDA_BF16, MSDA_F16 (offset / mask and their gradients float32, float64 for MSDA_F64) or
 * MSDA_BF16_AUX16 / MSDA_F16_AUX16 (offset / mask and their gradients in the input's 16-bit type).  Fast kernels cover
 * C/dg and C/groups multiples of 16 with float32 / bfloat16 / float16 input; every other shape, and float64, runs the
 * generic kernels.  MSDA_FLAG_FORCE_GENERIC selects the generic kernels; every other flag bit is ignored, except that
 * msda_dcnv2_col2im returns MSDA_ERR_UNSUPPORTED for MSDA_FLAG_DETERMINISTIC (grad_input is accumulated with float
 * reds, whose rounding depends on arrival order; grad_offset / grad_mask are bit-reproducible in every case).
 * col2im writes every element of grad_input, grad_offset and grad_mask.  Its workspace is
 * msda_dcnv2_col2im_workspace_bytes: N*H_in*W_in*C floats for bfloat16 / float16 input (the float accumulator of
 * grad_input), 0 otherwise (and 0 for an invalid geometry); less gives MSDA_ERR_WORKSPACE.  N = 0 or C = 0 are empty
 * problems (col2im zero-fills grad_offset / grad_mask when C = 0).  Added in ABI 3 without a version bump: an older
 * library lacks the three symbols.
 */
size_t msda_dcnv2_col2im_workspace_bytes(int batch, int channels, int height_in, int width_in, int height_out,
                                         int width_out, int kernel_h, int kernel_w, int stride_h, int stride_w,
                                         int pad_h, int pad_w, int dilation_h, int dilation_w, int groups,
                                         int deformable_groups, int dtype, unsigned flags);
int msda_dcnv2_im2col(void* stream, const void* input, const void* offset, const void* mask, int batch, int channels,
                      int height_in, int width_in, int height_out, int width_out, int kernel_h, int kernel_w,
                      int stride_h, int stride_w, int pad_h, int pad_w, int dilation_h, int dilation_w, int groups,
                      int deformable_groups, void* columns, int dtype, unsigned flags);
int msda_dcnv2_col2im(void* stream, const void* grad_columns, const void* input, const void* offset, const void* mask,
                      int batch, int channels, int height_in, int width_in, int height_out, int width_out, int kernel_h,
                      int kernel_w, int stride_h, int stride_w, int pad_h, int pad_w, int dilation_h, int dilation_w,
                      int groups, int deformable_groups, void* grad_input, void* grad_offset, void* grad_mask,
                      void* workspace, size_t workspace_bytes, int dtype, unsigned flags);

/*
 * Fused residual add + LayerNorm (SURVEY.md section 8f-2): the epilogue that follows every MSDeformAttn call and every
 * FFN in the reference's transformer layers -- x = x + identity; x = norm(x)
 * (/root/reference/detrex/layers/transformer.py:152-192; the residuals are added at multi_scale_deform_attn.py:363 and
 * detrex/layers/mlp.py:127-132) -- as one pass instead of an add kernel plus a LayerNorm kernel.
 *   a, b, y, grad_y, grad_x   [rows, channels]  dtype (MSDA_F32, MSDA_BF16 or MSDA_F16), contiguous
 *   gamma, beta, grad_gamma, grad_beta  [channels] float;   mean, rstd  [rows] float (saved by forward for backward)
 * forward:  y = (a + b - mean) * rstd * gamma + beta, statistics over the channels, fp32 arithmetic.
 * backward: grad_x = d loss / d (a + b) -- the gradient of BOTH addends -- plus grad_gamma / grad_beta, reduced in a
 *           fixed order (bit-reproducible); a + b is recomputed, never stored.  Needs a workspace of
 *           msda_add_layernorm_workspace_bytes(rows, channels).
 * channels must be a multiple of 4 and at most 1024 (MSDA_ERR_UNSUPPORTED otherwise, also for any other dtype tag).
 *
 * Mixed form, the one autocast produces (a 16-bit attention / FFN output added to a float32 residual): `a` is in
 * a_dtype (MSDA_BF16 or MSDA_F16; anything else is MSDA_ERR_UNSUPPORTED), b / y / grad_y / grad_b are float32.
 *   forward:  y = LayerNorm(float(a) + b) in float32 -- what norm(a + b) gives with torch's type promotion.
 *   backward: grad_b = d loss / d (a + b) (float32) and grad_a = grad_b rounded once to a_dtype, to nearest even (the
 *             cast autograd applies to a's gradient; a NaN's payload may differ, only NaN-ness is promised), written in
 *             one pass; grad_gamma / grad_beta as above, in the same fixed order.  Same workspace query.
 * Added in ABI 3 without a version bump: an older library lacks the two symbols.
 */
size_t msda_add_layernorm_workspace_bytes(int64_t rows, int channels);
int msda_add_layernorm_forward(void* stream, const void* a, const void* b, const float* gamma, const float* beta,
                               int64_t rows, int channels, float eps, void* y, float* mean, float* rstd, int dtype);
int msda_add_layernorm_backward(void* stream, const void* grad_y, const void* a, const void* b, const float* gamma,
                                const float* mean, const float* rstd, int64_t rows, int channels, void* grad_x,
                                float* grad_gamma, float* grad_beta, void* workspace, size_t workspace_bytes,
                                int dtype);
int msda_add_layernorm_mixed_forward(void* stream, const void* a, const float* b, const float* gamma,
                                     const float* beta, int64_t rows, int channels, float eps, float* y, float* mean,
                                     float* rstd, int a_dtype);
int msda_add_layernorm_mixed_backward(void* stream, const float* grad_y, const void* a, const float* b,
                                      const float* gamma, const float* mean, const float* rstd, int64_t rows,
                                      int channels, void* grad_a, float* grad_b, float* grad_gamma, float* grad_beta,
                                      void* workspace, size_t workspace_bytes, int a_dtype);

/*
 * Test hook: the integer bookkeeping the float kernels derive from every sampling point.
 *   corner_offsets [B*Q*H*L*P, 4] int64  flat element offset (channel 0) of the four bilinear
 *                  corners inside `value`, -1 for a zero-padded corner or a gated-out point;
 *   frac           [B*Q*H*L*P, 2] float  (lw, lh) fractional weights.
 * Same definition as msda_oracle_bookkeeping in oracle/msda_oracle.c; compared bit for bit.
 * On the shapes the fast kernels cover (float dispatch name "*_fast_*") the numbers are decoded from the very
 * record the fast kernels build per point (unclamped low-corner offset + four corner-validity bits), i.e. they are
 * the addresses those kernels gather from and scatter to; elsewhere they come from the generic kernels'
 * coordinate code.
 */
int msda_debug_bookkeeping(void* stream, const float* sampling_loc, const int64_t* spatial_shapes,
                           const int64_t* level_start_index, int batch, int spatial_size,
                           int num_heads, int channels, int num_levels, int num_query,
                           int num_point, int64_t* corner_offsets, float* frac);

/* Test hook (host arithmetic only, no GPU): n / d as the deterministic path's count pass computes it -- multiply-high
 * by a constant derived from d (csrc/msda_det.cuh, FastDiv).  Exact for n < 2^31 and 1 <= d < 2^31. */
unsigned msda_debug_fastdiv(unsigned n, unsigned d);

/* Human-readable name of a status code. */
const char* msda_status_string(int status);
/* Detail of the last failure on the calling thread ("" if none). */
const char* msda_last_error_message(void);
/* Number of kernels this library has launched in this process (monotonic). */
uint64_t msda_kernel_launch_count(void);
/* Name of the kernel family the given problem dispatches to ("fast_d32_f32", "generic_f64", ...). */
const char* msda_dispatch_name(int channels, int num_levels, int num_point, int spatial_size,
                               int num_heads, int dtype, unsigned flags, int backward);

#ifdef __cplusplus
}
#endif
#endif /* MSDA_B200_H_ */
