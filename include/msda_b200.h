/*
 * msda_b200.h -- C ABI of the B200-native (sm_100a) multi-scale deformable
 * attention library, libmsda_b200.so.
 *
 * This is the drop-in boundary for the one hot path of
 * HI-ComputerVision/uni-encoder-code that this repository replaces: the two
 * functions its pybind11 module `MultiScaleDeformableAttention` exports
 * (reference: model/modeling/pixel_decoder/ops/src/vision.cpp:18-21, dispatch in
 * ops/src/ms_deform_attn.h:25-66, host wrappers in
 * ops/src/cuda/ms_deform_attn_cuda.cu:25-85 and :88-158).
 *
 * Conventions
 *   - plain pointers and sizes only; every data pointer is a DEVICE pointer
 *     (the reference requires CUDA tensors: ms_deform_attn_cuda.cu:39-43);
 *   - all tensors contiguous, row-major (ms_deform_attn_cuda.cu:33-37):
 *       value          [batch, spatial_size, num_heads, channels]
 *       spatial_shapes [num_levels, 2]  int64 (H_l, W_l), on the device
 *       level_start    [num_levels]     int64,            on the device
 *       sampling_loc   [batch, num_query, num_heads, num_levels, num_point, 2]
 *                      normalised (x, y), x first (ms_deform_im2col_cuda.cuh:286-287)
 *       attn_weight    [batch, num_query, num_heads, num_levels, num_point]
 *       output / grad_output [batch, num_query, num_heads * channels]
 *   - `stream` is a cudaStream_t passed as void* (the reference launches on the
 *     caller's current stream, ms_deform_attn_cuda.cu:70,140); the library never
 *     synchronises the device, allocates or frees, and keeps no mutable state
 *     that affects results: calls are re-entrant and CUDA-graph capturable;
 *   - one launch covers the whole batch with 64-bit base offsets; the
 *     reference's im2col_step chunk loop (ms_deform_attn_cuda.cu:55-80) is a
 *     host-side concern handled (validated, then ignored) by the Python shim;
 *   - return value: 0 on success, a negative MSDA_ERR_* for argument errors, a
 *     positive cudaError_t if the launch failed (the reference only printf()s
 *     launch errors, ms_deform_im2col_cuda.cuh:953-957; we report them).
 */
#ifndef MSDA_B200_H_
#define MSDA_B200_H_

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define MSDA_B200_ABI_VERSION 2

enum {
    MSDA_OK = 0,
    MSDA_ERR_NULL_POINTER = -1,   /* a required pointer is NULL                      */
    MSDA_ERR_BAD_SHAPE = -2,      /* a size is <= 0 or exceeds a supported bound     */
    MSDA_ERR_UNSUPPORTED = -3,    /* e.g. num_levels > MSDA_MAX_LEVELS               */
    MSDA_ERR_BAD_OPTION = -4      /* msda_b200_set_option: unknown name / bad value  */
};

#define MSDA_MAX_LEVELS 16        /* level table kept in shared memory               */

/* Library / ABI identification. */
int msda_b200_abi_version(void);
/* Human-readable text for a code returned by any function here. */
const char *msda_b200_error_string(int code);
/* Number of kernel launches issued through this library since load (all
 * streams); bench.py reports the delta over its timed region as gpu_launches. */
long long msda_b200_launch_count(void);

/*
 * Forward.  Replaces ms_deform_attn_cuda_forward (ms_deform_attn_cuda.cu:25-85)
 * + ms_deformable_im2col_cuda (ms_deform_im2col_cuda.cuh:928-959) + the kernel
 * ms_deformable_im2col_gpu_kernel (cuh:242-304).
 * `output` is fully overwritten (no zero-fill needed; cf. at::zeros at cu:59).
 */
int msda_b200_forward_f32(const float *value, const int64_t *spatial_shapes,
                          const int64_t *level_start, const float *sampling_loc,
                          const float *attn_weight, int batch, int spatial_size,
                          int num_heads, int channels, int num_levels, int num_query,
                          int num_point, float *output, void *stream);
int msda_b200_forward_f64(const double *value, const int64_t *spatial_shapes,
                          const int64_t *level_start, const double *sampling_loc,
                          const double *attn_weight, int batch, int spatial_size,
                          int num_heads, int channels, int num_levels, int num_query,
                          int num_point, double *output, void *stream);

/*
 * Backward.  Replaces ms_deform_attn_cuda_backward (ms_deform_attn_cuda.cu:88-158)
 * + ms_deformable_col2im_cuda (cuh:961-1331) + the seven col2im kernels
 * (cuh:306-925).
 * `grad_value` MUST be zero on entry (it is accumulated with reductions, like
 * the reference's at::zeros_like at cu:126); `grad_sampling_loc` and
 * `grad_attn_weight` are fully overwritten (no zero-fill needed, cf. cu:127-128).
 */
int msda_b200_backward_f32(const float *grad_output, const float *value,
                           const int64_t *spatial_shapes, const int64_t *level_start,
                           const float *sampling_loc, const float *attn_weight,
                           int batch, int spatial_size, int num_heads, int channels,
                           int num_levels, int num_query, int num_point,
                           float *grad_value, float *grad_sampling_loc,
                           float *grad_attn_weight, void *stream);
int msda_b200_backward_f64(const double *grad_output, const double *value,
                           const int64_t *spatial_shapes, const int64_t *level_start,
                           const double *sampling_loc, const double *attn_weight,
                           int batch, int spatial_size, int num_heads, int channels,
                           int num_levels, int num_query, int num_point,
                           double *grad_value, double *grad_sampling_loc,
                           double *grad_attn_weight, void *stream);

/*
 * Deterministic backwards: the same gradients with no order-dependent floating-point sums, so bit-identical
 * inputs give bit-identical outputs on the same device (what torch.use_deterministic_algorithms asks for).
 * Same arguments as the entries above plus `workspace`, device scratch of
 * msda_b200_backward_deterministic_workspace_bytes(...) bytes (value_bytes = 4 for the f32 entries, 8 for f64,
 * 2 for the bf16 / f16 ones below;
 * 16-byte aligned; contents meaningless before and after; 0 = shape not covered: more than 2^31 - 1 corner
 * records, i.e. batch * num_query * num_heads * num_levels * num_point * 4, or batch * spatial_size * num_heads
 * >= 2^31 -- split the batch).  grad_value is fully overwritten (no zero-fill needed).  The backward kernel of
 * the path writes one {grad_value row, weight} record per (sampling point, corner) into a fixed slot, a stable
 * radix sort (CUB) orders the records by row, and one warp per row adds its records up in slot order -- the
 * order of a sequential loop over query, head, level, point, corner.  grad_sampling_loc / grad_attn_weight are
 * computed exactly as by the default entries.  No host read-back or allocation: CUDA-graph capturable.
 * msda_b200_launch_count counts four launches per call: the records kernel, the sort (as one launch, however many
 * kernels CUB runs for it), the bucket bounds and the gather.
 */
long long msda_b200_backward_deterministic_workspace_bytes(int batch, int spatial_size, int num_heads,
                                                          int channels, int num_levels, int num_query,
                                                          int num_point, int value_bytes);
int msda_b200_backward_deterministic_f32(const float *grad_output, const float *value,
                                         const int64_t *spatial_shapes, const int64_t *level_start,
                                         const float *sampling_loc, const float *attn_weight,
                                         int batch, int spatial_size, int num_heads, int channels,
                                         int num_levels, int num_query, int num_point,
                                         float *grad_value, float *grad_sampling_loc,
                                         float *grad_attn_weight, void *workspace, void *stream);
int msda_b200_backward_deterministic_f64(const double *grad_output, const double *value,
                                         const int64_t *spatial_shapes, const int64_t *level_start,
                                         const double *sampling_loc, const double *attn_weight,
                                         int batch, int spatial_size, int num_heads, int channels,
                                         int num_levels, int num_query, int num_point,
                                         double *grad_value, double *grad_sampling_loc,
                                         double *grad_attn_weight, void *workspace, void *stream);

/*
 * Mixed precision (torch.autocast): value, output, grad_output and grad_value are bfloat16 (_bf16) or IEEE
 * half (_f16), passed as uint16_t bit patterns, one type per call; sampling_loc, attn_weight and their
 * gradients stay float.  Every sum is fp32 with the geometry of the f32 entries; the only 16-bit rounding is
 * the final store of output / grad_value (round to nearest even; fp16 overflow gives +-inf).  The results
 * therefore equal the f32 entries applied to the widened 16-bit inputs, up to that one rounding.  Same
 * kernel choice and "bwd_variant" meanings as the f32 entries (each kernel in its default shape); any
 * channels, levels and points (shapes outside the 32-channel kernels take the generic ones).
 *
 * msda_b200_backward_{bf16,f16}: `grad_value_accum` is caller-provided device scratch of
 * batch * spatial_size * num_heads * channels floats, ZERO-FILLED before the call (16-byte aligned for the
 * fastest path); the kernels reduce into it in fp32 and one more launch rounds it into grad_value.  Its
 * contents afterwards are the fp32 grad_value.
 * msda_b200_backward_deterministic_{bf16,f16}: as the f32 twin, workspace of
 * msda_b200_backward_deterministic_workspace_bytes(..., value_bytes = 2) bytes (the records carry fp32
 * weights); the gather sums in fp32 and writes the 16-bit grad_value directly (no accumulation buffer).
 */
int msda_b200_forward_bf16(const uint16_t *value, const int64_t *spatial_shapes, const int64_t *level_start,
                           const float *sampling_loc, const float *attn_weight, int batch, int spatial_size,
                           int num_heads, int channels, int num_levels, int num_query, int num_point,
                           uint16_t *output, void *stream);
int msda_b200_forward_f16(const uint16_t *value, const int64_t *spatial_shapes, const int64_t *level_start,
                          const float *sampling_loc, const float *attn_weight, int batch, int spatial_size,
                          int num_heads, int channels, int num_levels, int num_query, int num_point,
                          uint16_t *output, void *stream);
int msda_b200_backward_bf16(const uint16_t *grad_output, const uint16_t *value, const int64_t *spatial_shapes,
                            const int64_t *level_start, const float *sampling_loc, const float *attn_weight,
                            int batch, int spatial_size, int num_heads, int channels, int num_levels,
                            int num_query, int num_point, float *grad_value_accum, uint16_t *grad_value,
                            float *grad_sampling_loc, float *grad_attn_weight, void *stream);
int msda_b200_backward_f16(const uint16_t *grad_output, const uint16_t *value, const int64_t *spatial_shapes,
                           const int64_t *level_start, const float *sampling_loc, const float *attn_weight,
                           int batch, int spatial_size, int num_heads, int channels, int num_levels,
                           int num_query, int num_point, float *grad_value_accum, uint16_t *grad_value,
                           float *grad_sampling_loc, float *grad_attn_weight, void *stream);
int msda_b200_backward_deterministic_bf16(const uint16_t *grad_output, const uint16_t *value,
                                          const int64_t *spatial_shapes, const int64_t *level_start,
                                          const float *sampling_loc, const float *attn_weight, int batch,
                                          int spatial_size, int num_heads, int channels, int num_levels,
                                          int num_query, int num_point, uint16_t *grad_value,
                                          float *grad_sampling_loc, float *grad_attn_weight, void *workspace,
                                          void *stream);
int msda_b200_backward_deterministic_f16(const uint16_t *grad_output, const uint16_t *value,
                                         const int64_t *spatial_shapes, const int64_t *level_start,
                                         const float *sampling_loc, const float *attn_weight, int batch,
                                         int spatial_size, int num_heads, int channels, int num_levels,
                                         int num_query, int num_point, uint16_t *grad_value,
                                         float *grad_sampling_loc, float *grad_attn_weight, void *workspace,
                                         void *stream);

/*
 * Fused producers (SURVEY.md 8f.1): the same op with the three elementwise steps of its caller
 * folded into the kernels -- ops/modules/ms_deform_attn.py:105-112:
 *     attention_weights = softmax(attn_logits over num_levels*num_point)
 *     sampling_loc      = reference_points[:, :, None, :, None, :] + sampling_offsets / (W_l, H_l)
 *   reference_points  [batch or 1, num_query, num_levels, 2]; ref_batch_stride = elements between
 *                     images (num_query*num_levels*2), or 0 when one set is shared by the batch
 *   sampling_offsets  [batch, num_query, num_heads, num_levels, num_point, 2]  (raw Linear output)
 *   attn_logits       [batch, num_query, num_heads, num_levels*num_point]      (raw Linear output)
 * The backward returns the gradients with respect to sampling_offsets and attn_logits (softmax
 * backward and the 1/(W,H) scaling folded in); reference_points get no gradient here.
 * Only the 32-channel fast path exists (channels == 32, num_levels*num_point in {4,8,12,16}), in fp32
 * and in mixed precision (the _bf16 / _f16 entries below); MSDA_ERR_UNSUPPORTED otherwise, and for views
 * whose alignment the kernels cannot take -- the caller then composes the unfused entry points.
 */
int msda_b200_fused_forward_f32(const float *value, const int64_t *spatial_shapes,
                                const int64_t *level_start, const float *reference_points,
                                long long ref_batch_stride, const float *sampling_offsets,
                                const float *attn_logits, int batch, int spatial_size,
                                int num_heads, int channels, int num_levels, int num_query,
                                int num_point, float *output, void *stream);
/* The fused forward with the raw projections read in place from wider rows: query r's offsets start at
 * sampling_offsets + r * offsets_row_stride and its logits at attn_logits + r * logits_row_stride (floats;
 * offsets_row_stride even).  One [rows, 3*M*L*P] GEMM (sampling_offsets and attention_weights weights
 * stacked, ops/modules/ms_deform_attn.py:105-106) then feeds the kernel without a split copy:
 * sampling_offsets = y, attn_logits = y + 2*M*L*P, both strides 3*M*L*P.
 * offsets_table / logits_table (both or neither; NULL = none): per-QUERY tables with num_query rows laid
 * out with the same row strides, shared by the batch and added to the raw values of query q of every image
 * before the softmax / location arithmetic.  The encoder layer projects `src + pos` (with_pos_embed,
 * msdeformattn.py:123-124, :133); `pos` is the same for every image and every call, so
 * (src + pos) W^T + b = src W^T + (pos W^T + b): the host computes the second term once per layer
 * (num_query x 3*M*L*P), the GEMM runs on `src`, and the `src + pos` pass over the activations disappears. */
int msda_b200_fused_forward_strided_f32(const float *value, const int64_t *spatial_shapes,
                                        const int64_t *level_start, const float *reference_points,
                                        long long ref_batch_stride, const float *sampling_offsets,
                                        int offsets_row_stride, const float *attn_logits,
                                        int logits_row_stride, const float *offsets_table,
                                        const float *logits_table, int batch, int spatial_size,
                                        int num_heads, int channels, int num_levels, int num_query,
                                        int num_point, float *output, void *stream);
int msda_b200_fused_backward_f32(const float *grad_output, const float *value,
                                 const int64_t *spatial_shapes, const int64_t *level_start,
                                 const float *reference_points, long long ref_batch_stride,
                                 const float *sampling_offsets, const float *attn_logits,
                                 int batch, int spatial_size, int num_heads, int channels,
                                 int num_levels, int num_query, int num_point, float *grad_value,
                                 float *grad_sampling_offsets, float *grad_attn_logits,
                                 void *stream);
/* Deterministic twin of the fused backward: the records carry the in-kernel softmax and locations, exactly as
 * the fused forward used them.  Workspace and guarantees as for msda_b200_backward_deterministic_f32
 * (value_bytes = 4). */
int msda_b200_fused_backward_deterministic_f32(const float *grad_output, const float *value,
                                               const int64_t *spatial_shapes, const int64_t *level_start,
                                               const float *reference_points, long long ref_batch_stride,
                                               const float *sampling_offsets, const float *attn_logits,
                                               int batch, int spatial_size, int num_heads, int channels,
                                               int num_levels, int num_query, int num_point, float *grad_value,
                                               float *grad_sampling_offsets, float *grad_attn_logits,
                                               void *workspace, void *stream);

/*
 * Mixed-precision fused producers (what torch.autocast hands the module: every Linear output is 16-bit):
 * value, sampling_offsets, attn_logits, output, grad_output, grad_value, grad_sampling_offsets and
 * grad_attn_logits all bf16 (_bf16) or all fp16 (_f16), as uint16_t bit patterns; reference_points stay
 * fp32.  Everything in between is fp32 -- the widened offsets and logits, ref + offset / (W, H), the
 * softmax and its backward, the 1/(W, H) scaling and every sum -- with the integer geometry of the fp32 op,
 * and each output is rounded once (round-to-nearest-even; fp16 overflow gives +-inf).  For the same widened
 * inputs output, grad_sampling_offsets, grad_attn_logits and the deterministic grad_value are therefore the
 * fp32 fused entries' results rounded to 16 bits, bit for bit.
 * msda_b200_fused_backward_{bf16,f16}: grad_value_accum is a zero-filled fp32 [batch, spatial_size,
 * num_heads, channels] buffer that the kernels reduce into and that is then rounded into grad_value, as for
 * msda_b200_backward_bf16.  The deterministic twins take a workspace of
 * msda_b200_backward_deterministic_workspace_bytes(..., value_bytes = 2) bytes.
 * Alignment: sampling_offsets 4 bytes, reference_points 8, value / output / grad_output 16 (and value 64
 * for the merging backward kernel, otherwise the per-row one runs); MSDA_ERR_UNSUPPORTED otherwise.
 */
int msda_b200_fused_forward_bf16(const uint16_t *value, const int64_t *spatial_shapes, const int64_t *level_start,
                                 const float *reference_points, long long ref_batch_stride,
                                 const uint16_t *sampling_offsets, const uint16_t *attn_logits, int batch,
                                 int spatial_size, int num_heads, int channels, int num_levels, int num_query,
                                 int num_point, uint16_t *output, void *stream);
int msda_b200_fused_forward_f16(const uint16_t *value, const int64_t *spatial_shapes, const int64_t *level_start,
                                const float *reference_points, long long ref_batch_stride,
                                const uint16_t *sampling_offsets, const uint16_t *attn_logits, int batch,
                                int spatial_size, int num_heads, int channels, int num_levels, int num_query,
                                int num_point, uint16_t *output, void *stream);
/* The 16-bit fused forward with row strides and per-query tables, as msda_b200_fused_forward_strided_f32: the raw
 * offsets / logits are 16-bit rows (strides in elements, offsets_row_stride even), e.g. of one [rows, 3*M*L*P]
 * projection output; offsets_table / logits_table (both or neither) stay fp32.  Each raw value is widened first
 * and then gets its table entry added in fp32, so output is bit-identical to msda_b200_fused_forward_strided_f32 run
 * on the widened rows, the widened value and the same tables, rounded once to 16 bits.  Error codes and
 * alignment as for that entry, with sampling_offsets 4-byte aligned. */
int msda_b200_fused_forward_strided_bf16(const uint16_t *value, const int64_t *spatial_shapes,
                                         const int64_t *level_start, const float *reference_points,
                                         long long ref_batch_stride, const uint16_t *sampling_offsets,
                                         int offsets_row_stride, const uint16_t *attn_logits, int logits_row_stride,
                                         const float *offsets_table, const float *logits_table, int batch,
                                         int spatial_size, int num_heads, int channels, int num_levels, int num_query,
                                         int num_point, uint16_t *output, void *stream);
int msda_b200_fused_forward_strided_f16(const uint16_t *value, const int64_t *spatial_shapes,
                                        const int64_t *level_start, const float *reference_points,
                                        long long ref_batch_stride, const uint16_t *sampling_offsets,
                                        int offsets_row_stride, const uint16_t *attn_logits, int logits_row_stride,
                                        const float *offsets_table, const float *logits_table, int batch,
                                        int spatial_size, int num_heads, int channels, int num_levels, int num_query,
                                        int num_point, uint16_t *output, void *stream);
int msda_b200_fused_backward_bf16(const uint16_t *grad_output, const uint16_t *value, const int64_t *spatial_shapes,
                                  const int64_t *level_start, const float *reference_points,
                                  long long ref_batch_stride, const uint16_t *sampling_offsets,
                                  const uint16_t *attn_logits, int batch, int spatial_size, int num_heads,
                                  int channels, int num_levels, int num_query, int num_point,
                                  float *grad_value_accum, uint16_t *grad_value, uint16_t *grad_sampling_offsets,
                                  uint16_t *grad_attn_logits, void *stream);
int msda_b200_fused_backward_f16(const uint16_t *grad_output, const uint16_t *value, const int64_t *spatial_shapes,
                                 const int64_t *level_start, const float *reference_points,
                                 long long ref_batch_stride, const uint16_t *sampling_offsets,
                                 const uint16_t *attn_logits, int batch, int spatial_size, int num_heads,
                                 int channels, int num_levels, int num_query, int num_point,
                                 float *grad_value_accum, uint16_t *grad_value, uint16_t *grad_sampling_offsets,
                                 uint16_t *grad_attn_logits, void *stream);
int msda_b200_fused_backward_deterministic_bf16(const uint16_t *grad_output, const uint16_t *value,
                                                const int64_t *spatial_shapes, const int64_t *level_start,
                                                const float *reference_points, long long ref_batch_stride,
                                                const uint16_t *sampling_offsets, const uint16_t *attn_logits,
                                                int batch, int spatial_size, int num_heads, int channels,
                                                int num_levels, int num_query, int num_point, uint16_t *grad_value,
                                                uint16_t *grad_sampling_offsets, uint16_t *grad_attn_logits,
                                                void *workspace, void *stream);
int msda_b200_fused_backward_deterministic_f16(const uint16_t *grad_output, const uint16_t *value,
                                               const int64_t *spatial_shapes, const int64_t *level_start,
                                               const float *reference_points, long long ref_batch_stride,
                                               const uint16_t *sampling_offsets, const uint16_t *attn_logits,
                                               int batch, int spatial_size, int num_heads, int channels,
                                               int num_levels, int num_query, int num_point, uint16_t *grad_value,
                                               uint16_t *grad_sampling_offsets, uint16_t *grad_attn_logits,
                                               void *workspace, void *stream);

/*
 * Next component on the path's caller side (SURVEY.md section 8f.3): the fp32 nn.Linear layers around
 * the op (ops/modules/ms_deform_attn.py:62-65,97-121 and msdeformattn.py:126-142), which the reference
 * runs as fp32 GEMMs (torch F.linear; autocast disabled, msdeformattn.py:338).
 *     y[rows, out_features] = x[rows, in_features] * weight[out_features, in_features]^T + bias
 * (torch.nn.functional.linear semantics, row-major contiguous fp32; bias may be NULL; relu != 0
 * applies max(., 0) to the result).  Computed on the sm_100a tensor cores with the error-compensated
 * 3 x TF32 split (fp32-class accuracy, fp32 accumulation).  `workspace`: device scratch of
 * 2 * out_features * in_features floats (the split weight; the library never allocates), or NULL: the
 * weight is then split inside the kernel (for a one-shot "weight", e.g. the transposed activations of a
 * weight-gradient GEMM).  When the output has few tiles and in_features is very large the reduction is
 * spread over several CTAs per tile (split-K: y is zero-filled and accumulated with reductions).  Requires
 * in_features % 32 == 0, out_features % 4 == 0 and 16-byte aligned x / weight / workspace / y;
 * MSDA_ERR_UNSUPPORTED otherwise.
 */
int msda_b200_linear_f32(const float *x, const float *weight, const float *bias, float *y,
                         int rows, int out_features, int in_features, int relu, float *workspace,
                         void *stream);
/* Deterministic twin (same arguments): never spreads a tile's reduction over CTAs, so the result does not
 * depend on scheduling.  Where msda_b200_linear_f32 uses split-K, one CTA per output tile computes the same
 * chunks of the reduction in order and adds them in chunk order (same accuracy); elsewhere the result is
 * bit-identical to msda_b200_linear_f32. */
int msda_b200_linear_deterministic_f32(const float *x, const float *weight, const float *bias, float *y,
                                       int rows, int out_features, int in_features, int relu,
                                       float *workspace, void *stream);

/*
 * The same GEMM for a weight that does not change between calls (inference): msda_b200_split_weight_f32 writes
 * the split weight (tf32(W) followed by tf32(W - tf32(W)), 2 * out_features * in_features floats) once,
 * msda_b200_linear_presplit_f32 then runs the GEMM alone -- one launch per Linear instead of two, bit-identical
 * results.  Same shape / alignment requirements; MSDA_ERR_UNSUPPORTED otherwise.
 */
int msda_b200_split_weight_f32(const float *weight, float *split_weight, int out_features, int in_features,
                               void *stream);
int msda_b200_linear_presplit_f32(const float *x, const float *split_weight, const float *bias, float *y,
                                  int rows, int out_features, int in_features, int relu, void *stream);
int msda_b200_linear_presplit_deterministic_f32(const float *x, const float *split_weight, const float *bias,
                                                float *y, int rows, int out_features, int in_features, int relu,
                                                void *stream);

/*
 * y[rows, cols] = LayerNorm(x + residual) * gamma + beta over the last dimension (eps inside the square
 * root, biased variance: torch.nn.functional.layer_norm semantics) -- the `norm(src + sublayer(src))`
 * steps of the encoder layer (msdeformattn.py:134-141) in one pass.  residual may be NULL.
 * cols in {128, 256, 384, 512}, 16-byte aligned pointers; MSDA_ERR_UNSUPPORTED otherwise.
 */
int msda_b200_add_layernorm_f32(const float *x, const float *residual, const float *gamma,
                                const float *beta, float *y, long long rows, int cols, float eps,
                                void *stream);

/*
 * Backward of the above: grad_v[rows, cols] (= gradient of both x and residual), grad_gamma[cols], grad_beta[cols]
 * from grad_y, x, residual (may be NULL) and gamma; mean / rstd are recomputed.  grad_gamma / grad_beta are
 * overwritten.  cols in {128, 256}; MSDA_ERR_UNSUPPORTED otherwise.
 */
int msda_b200_add_layernorm_backward_f32(const float *grad_y, const float *x, const float *residual,
                                         const float *gamma, float *grad_v, float *grad_gamma,
                                         float *grad_beta, long long rows, int cols, float eps, void *stream);
/* Deterministic twin: every CTA stores its grad_gamma / grad_beta partials in `workspace`
 * (msda_b200_add_layernorm_backward_deterministic_workspace_bytes(rows, cols) bytes, computed for the current
 * device) and a second launch adds them in CTA order.  grad_v is bit-identical to the entry above. */
int msda_b200_add_layernorm_backward_deterministic_f32(const float *grad_y, const float *x, const float *residual,
                                                       const float *gamma, float *grad_v, float *grad_gamma,
                                                       float *grad_beta, long long rows, int cols, float eps,
                                                       void *workspace, void *stream);
long long msda_b200_add_layernorm_backward_deterministic_workspace_bytes(long long rows, int cols);

/*
 * Mixed precision (torch.autocast: the sublayer's Linear output is 16-bit, the residual stream fp32):
 * y = LayerNorm(x + widen(residual)) * gamma + beta with x, gamma, beta, y fp32 and residual bf16 (_bf16) or fp16
 * (_f16), as uint16_t bit patterns.  y is bit-identical to msda_b200_add_layernorm_f32(x, widen(residual)): the
 * fp32 arithmetic is that kernel's, residual is widened once on load.  y16 (may be NULL) receives the same rows
 * rounded to the 16-bit type (round-to-nearest-even, == y.to(dtype); fp16 overflow gives +-inf) -- the copy the
 * next GEMMs read.  residual is required.  cols in {128, 256, 384, 512}; x, gamma, beta, y 16-byte aligned,
 * residual and y16 8-byte aligned; MSDA_ERR_UNSUPPORTED otherwise.
 */
int msda_b200_add_layernorm_mixed_bf16(const float *x, const uint16_t *residual, const float *gamma,
                                       const float *beta, float *y, uint16_t *y16, long long rows, int cols,
                                       float eps, void *stream);
int msda_b200_add_layernorm_mixed_f16(const float *x, const uint16_t *residual, const float *gamma,
                                      const float *beta, float *y, uint16_t *y16, long long rows, int cols,
                                      float eps, void *stream);
/* Backward of the entries above with respect to y (grad_y, fp32) and y16 (grad_y16, 16-bit), either of which may
 * be NULL (not both): g = grad_y + widen(grad_y16), one fp32 add per element.  grad_x (fp32) is bit-identical to
 * msda_b200_add_layernorm_backward_f32(g, x, widen(residual)); grad_residual (16-bit) is grad_x rounded once;
 * grad_gamma / grad_beta (fp32, overwritten) are reduced as in that entry.  cols in {128, 256}; alignment as in the
 * forward (grad_y and grad_x 16 bytes, grad_y16 and grad_residual 8); MSDA_ERR_UNSUPPORTED otherwise.  The
 * deterministic twins take the workspace of msda_b200_add_layernorm_backward_deterministic_workspace_bytes(rows,
 * cols) and are bit-identical to msda_b200_add_layernorm_backward_deterministic_f32 fed g. */
int msda_b200_add_layernorm_mixed_backward_bf16(const float *grad_y, const uint16_t *grad_y16, const float *x,
                                                const uint16_t *residual, const float *gamma, float *grad_x,
                                                uint16_t *grad_residual, float *grad_gamma, float *grad_beta,
                                                long long rows, int cols, float eps, void *stream);
int msda_b200_add_layernorm_mixed_backward_f16(const float *grad_y, const uint16_t *grad_y16, const float *x,
                                               const uint16_t *residual, const float *gamma, float *grad_x,
                                               uint16_t *grad_residual, float *grad_gamma, float *grad_beta,
                                               long long rows, int cols, float eps, void *stream);
int msda_b200_add_layernorm_mixed_backward_deterministic_bf16(const float *grad_y, const uint16_t *grad_y16,
                                                              const float *x, const uint16_t *residual,
                                                              const float *gamma, float *grad_x,
                                                              uint16_t *grad_residual, float *grad_gamma,
                                                              float *grad_beta, long long rows, int cols, float eps,
                                                              void *workspace, void *stream);
int msda_b200_add_layernorm_mixed_backward_deterministic_f16(const float *grad_y, const uint16_t *grad_y16,
                                                             const float *x, const uint16_t *residual,
                                                             const float *gamma, float *grad_x,
                                                             uint16_t *grad_residual, float *grad_gamma,
                                                             float *grad_beta, long long rows, int cols, float eps,
                                                             void *workspace, void *stream);

/*
 * GroupNorm over an NCHW fp32 map with the pixel decoder's epilogues fused in (SURVEY 8f.4;
 * msdeformattn.py:233-248, :286-300, :369-379):
 *     y = group_norm(x + channel_bias[c], groups, gamma, beta, eps)    torch.nn.functional.group_norm semantics;
 *                     channel_bias (may be NULL) is the bias of the convolution that produced x, when that
 *                     convolution ran without it (torch adds a convolution's bias in a separate pass)
 *     if relu:        y = max(y, 0)
 *     if up != NULL:  y += bilinear up-sampling of up[N, C, up_h, up_w] to H x W, align_corners=False
 * `workspace` must hold msda_b200_group_norm_workspace_bytes(N, groups) bytes (per-group partial sums;
 * its contents are meaningless before and after the call).  Needs H*W (and, with `up`, W) to be a multiple of 4 and
 * 16-byte aligned x / y; MSDA_ERR_UNSUPPORTED otherwise.  Training: the _train_f32 forwards and the backward
 * entry points below.
 */
int msda_b200_group_norm_nchw_f32(const float *x, const float *channel_bias, const float *gamma,
                                  const float *beta, float *y, int batch, int channels, int height,
                                  int width, int groups, float eps, int relu, const float *up, int up_h,
                                  int up_w, void *workspace, void *stream);
long long msda_b200_group_norm_workspace_bytes(int batch, int groups);
/* The same GroupNorm (+ channel_bias, + ReLU) of x[N, C, plane] written as ROWS,
 *     y_rows[n * image_stride + pixel * row_stride + c],
 * the `[N, pixels, C]` layout the deformable encoder consumes (`src.flatten(2).transpose(1, 2)` followed by the
 * concatenation of the levels, msdeformattn.py:72-79, :87): with y_rows = the level's first row of the
 * concatenated [N, S, C] tensor, row_stride = C and image_stride = S * C every input projection lands in place
 * and torch's transposing `cat` disappears.  channels % 32 == 0, plane % 4 == 0, strides % 4 == 0,
 * 16-byte aligned x / y_rows; MSDA_ERR_UNSUPPORTED otherwise.  Same workspace as above. */
int msda_b200_group_norm_nchw_to_rows_f32(const float *x, const float *channel_bias, const float *gamma,
                                          const float *beta, float *y_rows, long long row_stride,
                                          long long image_stride, int batch, int channels, long long plane,
                                          int groups, float eps, int relu, void *workspace, void *stream);
/*
 * Training forwards: the two GroupNorms above with the same arguments, plus mean_rstd [batch, groups, 2], which
 * receives (mean, rstd) of x + channel_bias per (image, group) as the backward needs them.  y / y_rows are
 * bit-identical to those of the entry points above.
 */
int msda_b200_group_norm_nchw_train_f32(const float *x, const float *channel_bias, const float *gamma,
                                        const float *beta, float *y, float *mean_rstd, int batch, int channels,
                                        int height, int width, int groups, float eps, int relu, const float *up,
                                        int up_h, int up_w, void *workspace, void *stream);
int msda_b200_group_norm_nchw_to_rows_train_f32(const float *x, const float *channel_bias, const float *gamma,
                                                const float *beta, float *y_rows, float *mean_rstd,
                                                long long row_stride, long long image_stride, int batch,
                                                int channels, long long plane, int groups, float eps, int relu,
                                                void *workspace, void *stream);
/*
 * Backward of msda_b200_group_norm_nchw_train_f32 (torch autograd semantics) from grad_y, the forward's inputs and
 * its mean_rstd.  Overwritten: grad_x [N, C, H, W]; grad_gamma [C] and grad_beta [C], summed over the batch;
 * grad_channel_bias [C] (may be NULL: not computed); grad_up [N, C, up_h, up_w] (may be NULL: not computed), the
 * adjoint of the forward's bilinear up-sampling applied to grad_y (the add comes after the ReLU, so grad_y is not
 * masked there).  With relu, the mask is rebuilt from x with the forward's own float expression.  Deterministic (no
 * floating-point atomics).  Three launches (reduce, per-group finalize, apply), a fourth for grad_up.
 * `workspace` must hold msda_b200_group_norm_backward_workspace_bytes(N, C) bytes.  Shape and alignment
 * requirements are the forward's (16-byte aligned grad_y / x / grad_x); MSDA_ERR_UNSUPPORTED otherwise.
 */
int msda_b200_group_norm_backward_nchw_f32(const float *grad_y, const float *x, const float *channel_bias,
                                           const float *gamma, const float *beta, const float *mean_rstd,
                                           float *grad_x, float *grad_gamma, float *grad_beta,
                                           float *grad_channel_bias, float *grad_up, int batch, int channels,
                                           int height, int width, int groups, int relu, int up_h, int up_w,
                                           void *workspace, void *stream);
long long msda_b200_group_norm_backward_workspace_bytes(int batch, int channels);
/* Backward of msda_b200_group_norm_nchw_to_rows_train_f32: the same, with grad_y read from the rows layout
 * (grad_y_rows[n * image_stride + pixel * row_stride + c]) and grad_x written NCHW.  Three launches; same workspace
 * and the forward's requirements. */
int msda_b200_group_norm_rows_backward_f32(const float *grad_y_rows, long long row_stride, long long image_stride,
                                           const float *x, const float *channel_bias, const float *gamma,
                                           const float *beta, const float *mean_rstd, float *grad_x,
                                           float *grad_gamma, float *grad_beta, float *grad_channel_bias, int batch,
                                           int channels, long long plane, int groups, int relu, void *workspace,
                                           void *stream);
/* x[n, c, :] += bias[c] in place over an NCHW fp32 map (plane = H*W, a multiple of 4; 16-byte aligned x):
 * the bias of the decoder's last 1x1 convolution (mask_features, msdeformattn.py:268-275, :381) at the
 * memory roofline instead of torch's broadcasting add. */
int msda_b200_add_channel_bias_nchw_f32(float *x, const float *bias, int batch, int channels,
                                        long long plane, void *stream);

/*
 * Mixed precision (torch.autocast: the convolution in front of each GroupNorm writes bf16 / fp16): the GroupNorms
 * above on a bf16 (_bf16) or fp16 (_f16) map x, passed as uint16_t bit patterns.  channel_bias, gamma, beta, up,
 * mean_rstd and every `float *` output stay fp32; the workspaces are those of the fp32 entries.  Contract: bit
 * identity with the fp32 entry of the same name fed the widened map (the fp32 arithmetic and its grouping are that
 * entry's; x is widened on load):
 *   y, y_rows, mean_rstd, grad_gamma, grad_beta, grad_channel_bias, grad_up == the fp32 entry's on widen(x) and the
 *                      widened incoming gradient;
 *   y16                == y rounded to the 16-bit type (round-to-nearest-even, == y.to(dtype); fp16 overflow gives
 *                      +-inf): the copy the next convolution reads;
 *   grad_x (16-bit)    == the fp32 entry's grad_x rounded once.
 * The NCHW forwards write y and / or y16 (either may be NULL, not both: MSDA_ERR_NULL_POINTER).  The NCHW backward
 * takes the gradient of whichever output the forward wrote: exactly one of grad_y (fp32) and grad_y16 (16-bit);
 * neither gives MSDA_ERR_NULL_POINTER, both MSDA_ERR_UNSUPPORTED.  Requirements are the fp32 twins', with x, y16,
 * grad_y16 and grad_x 8-byte aligned (the fp32 maps 16-byte aligned); MSDA_ERR_UNSUPPORTED otherwise.  Launches as
 * in fp32: two forward, three backward (four with grad_up).
 */
int msda_b200_group_norm_nchw_mixed_bf16(const uint16_t *x, const float *channel_bias, const float *gamma,
                                         const float *beta, float *y, uint16_t *y16, int batch, int channels,
                                         int height, int width, int groups, float eps, int relu, const float *up,
                                         int up_h, int up_w, void *workspace, void *stream);
int msda_b200_group_norm_nchw_mixed_f16(const uint16_t *x, const float *channel_bias, const float *gamma,
                                        const float *beta, float *y, uint16_t *y16, int batch, int channels,
                                        int height, int width, int groups, float eps, int relu, const float *up,
                                        int up_h, int up_w, void *workspace, void *stream);
int msda_b200_group_norm_nchw_mixed_train_bf16(const uint16_t *x, const float *channel_bias, const float *gamma,
                                               const float *beta, float *y, uint16_t *y16, float *mean_rstd,
                                               int batch, int channels, int height, int width, int groups, float eps,
                                               int relu, const float *up, int up_h, int up_w, void *workspace,
                                               void *stream);
int msda_b200_group_norm_nchw_mixed_train_f16(const uint16_t *x, const float *channel_bias, const float *gamma,
                                              const float *beta, float *y, uint16_t *y16, float *mean_rstd,
                                              int batch, int channels, int height, int width, int groups, float eps,
                                              int relu, const float *up, int up_h, int up_w, void *workspace,
                                              void *stream);
/* fp32 rows (the encoder's [N, S, C] input) from a 16-bit NCHW map; strides and requirements of
 * msda_b200_group_norm_nchw_to_rows_f32, x 8-byte aligned. */
int msda_b200_group_norm_nchw_to_rows_mixed_bf16(const uint16_t *x, const float *channel_bias, const float *gamma,
                                                 const float *beta, float *y_rows, long long row_stride,
                                                 long long image_stride, int batch, int channels, long long plane,
                                                 int groups, float eps, int relu, void *workspace, void *stream);
int msda_b200_group_norm_nchw_to_rows_mixed_f16(const uint16_t *x, const float *channel_bias, const float *gamma,
                                                const float *beta, float *y_rows, long long row_stride,
                                                long long image_stride, int batch, int channels, long long plane,
                                                int groups, float eps, int relu, void *workspace, void *stream);
int msda_b200_group_norm_nchw_to_rows_mixed_train_bf16(const uint16_t *x, const float *channel_bias,
                                                       const float *gamma, const float *beta, float *y_rows,
                                                       float *mean_rstd, long long row_stride, long long image_stride,
                                                       int batch, int channels, long long plane, int groups, float eps,
                                                       int relu, void *workspace, void *stream);
int msda_b200_group_norm_nchw_to_rows_mixed_train_f16(const uint16_t *x, const float *channel_bias,
                                                      const float *gamma, const float *beta, float *y_rows,
                                                      float *mean_rstd, long long row_stride, long long image_stride,
                                                      int batch, int channels, long long plane, int groups, float eps,
                                                      int relu, void *workspace, void *stream);
int msda_b200_group_norm_backward_nchw_mixed_bf16(const float *grad_y, const uint16_t *grad_y16, const uint16_t *x,
                                                  const float *channel_bias, const float *gamma, const float *beta,
                                                  const float *mean_rstd, uint16_t *grad_x, float *grad_gamma,
                                                  float *grad_beta, float *grad_channel_bias, float *grad_up,
                                                  int batch, int channels, int height, int width, int groups,
                                                  int relu, int up_h, int up_w, void *workspace, void *stream);
int msda_b200_group_norm_backward_nchw_mixed_f16(const float *grad_y, const uint16_t *grad_y16, const uint16_t *x,
                                                 const float *channel_bias, const float *gamma, const float *beta,
                                                 const float *mean_rstd, uint16_t *grad_x, float *grad_gamma,
                                                 float *grad_beta, float *grad_channel_bias, float *grad_up,
                                                 int batch, int channels, int height, int width, int groups,
                                                 int relu, int up_h, int up_w, void *workspace, void *stream);
/* Backward of the rows forwards: fp32 gradient rows, 16-bit x and grad_x (NCHW). */
int msda_b200_group_norm_rows_backward_mixed_bf16(const float *grad_y_rows, long long row_stride,
                                                  long long image_stride, const uint16_t *x,
                                                  const float *channel_bias, const float *gamma, const float *beta,
                                                  const float *mean_rstd, uint16_t *grad_x, float *grad_gamma,
                                                  float *grad_beta, float *grad_channel_bias, int batch, int channels,
                                                  long long plane, int groups, int relu, void *workspace,
                                                  void *stream);
int msda_b200_group_norm_rows_backward_mixed_f16(const float *grad_y_rows, long long row_stride,
                                                 long long image_stride, const uint16_t *x,
                                                 const float *channel_bias, const float *gamma, const float *beta,
                                                 const float *mean_rstd, uint16_t *grad_x, float *grad_gamma,
                                                 float *grad_beta, float *grad_channel_bias, int batch, int channels,
                                                 long long plane, int groups, int relu, void *workspace,
                                                 void *stream);
/* x[n, c, :] = round16(widen(x[n, c, :]) + bias[c]) in place over a 16-bit NCHW map with an fp32 bias
 * (== (x.float() + bias).to(dtype)); plane % 4 == 0, x 8-byte aligned; MSDA_ERR_UNSUPPORTED otherwise. */
int msda_b200_add_channel_bias_nchw_bf16(uint16_t *x, const float *bias, int batch, int channels, long long plane,
                                         void *stream);
int msda_b200_add_channel_bias_nchw_f16(uint16_t *x, const float *bias, int batch, int channels, long long plane,
                                        void *stream);

/*
 * Weight and bias gradient of the same Linear (torch autograd semantics), 3 x TF32 on the tensor cores
 * without transposing the operands in memory:
 *     grad_weight[out_features, in_features] = grad_y[rows, out_features]^T * x[rows, in_features]
 *     grad_bias[out_features] = column sums of grad_y                      (grad_bias may be NULL)
 * Both outputs are overwritten (zero-filled, then accumulated with reductions: the row range is split over
 * the SMs).  out_features % 4 == 0, in_features % 4 == 0, 16-byte aligned operands; else MSDA_ERR_UNSUPPORTED.
 */
int msda_b200_linear_wgrad_f32(const float *grad_y, const float *x, float *grad_weight, float *grad_bias,
                               long long rows, int out_features, int in_features, void *stream);
/* Deterministic twin: each work item (a chunk of rows of one output tile) stores its partial tile and bias in
 * `workspace` (msda_b200_linear_wgrad_deterministic_workspace_bytes(rows, out_features, in_features) bytes, one
 * grad_weight + grad_bias per row chunk) and a second launch adds the chunks in order. */
int msda_b200_linear_wgrad_deterministic_f32(const float *grad_y, const float *x, float *grad_weight,
                                             float *grad_bias, long long rows, int out_features, int in_features,
                                             void *workspace, void *stream);
long long msda_b200_linear_wgrad_deterministic_workspace_bytes(long long rows, int out_features, int in_features);

/*
 * The same Linear under torch.autocast, on bf16 (_bf16) or fp16 (_f16) operands passed as uint16_t bit patterns:
 *     y[rows, out_features] = round16(x[rows, in_features] * weight16[out_features, in_features]^T + bias)
 * (then ReLU if relu != 0).  bias is fp32 (may be NULL) and is added to the fp32 accumulator; the result is rounded
 * once to nearest-even (fp16 overflow gives +-inf).  The input gradient is the same call with grad_y as x and the
 * transposed weight [in_features, out_features].  in_features % 8 == 0, out_features % 8 == 0 and 16-byte aligned
 * x, weight16 and y; MSDA_ERR_UNSUPPORTED otherwise.  One launch.
 */
int msda_b200_linear_mixed_bf16(const uint16_t *x, const uint16_t *weight16, const float *bias, uint16_t *y, int rows,
                                int out_features, int in_features, int relu, void *stream);
int msda_b200_linear_mixed_f16(const uint16_t *x, const uint16_t *weight16, const float *bias, uint16_t *y, int rows,
                               int out_features, int in_features, int relu, void *stream);
/* Weight and bias gradient of that Linear, in fp32 from 16-bit operands:
 *     grad_weight[out_features, in_features] = grad_y[rows, out_features]^T * x[rows, in_features]
 *     grad_bias[out_features] = column sums of grad_y                      (grad_bias may be NULL)
 * Deterministic by construction: each work item (a chunk of rows of one output tile) stores its partial tile and
 * bias sums in `workspace` (msda_b200_linear_mixed_wgrad_workspace_bytes(rows, out_features, in_features) bytes) and a
 * second launch adds the chunks in chunk order; the chunking depends on the shapes only.  out_features % 8 == 0,
 * in_features % 8 == 0, 16-byte aligned grad_y, x, grad_weight and workspace; MSDA_ERR_UNSUPPORTED otherwise. */
int msda_b200_linear_mixed_wgrad_bf16(const uint16_t *grad_y, const uint16_t *x, float *grad_weight, float *grad_bias,
                                      long long rows, int out_features, int in_features, void *workspace,
                                      void *stream);
int msda_b200_linear_mixed_wgrad_f16(const uint16_t *grad_y, const uint16_t *x, float *grad_weight, float *grad_bias,
                                     long long rows, int out_features, int in_features, void *workspace, void *stream);
long long msda_b200_linear_mixed_wgrad_workspace_bytes(long long rows, int out_features, int in_features);

/* y[cols, rows] = x[rows, cols]^T, fp32 (operand preparation for weight-gradient GEMMs). */
int msda_b200_transpose_f32(const float *x, float *y, long long rows, int cols, void *stream);

/*
 * Integer known-answer hook (no counterpart in the reference; it exposes the
 * integer work of cuh:43-58, 279-293 so tests can pin it bit-exactly).
 * For every (n, q, m, l, p), in sampling_loc order:
 *   idx[4*s+0] = point valid (cuh:293)   idx[4*s+1] = h_low   idx[4*s+2] = w_low
 *   idx[4*s+3] = corner mask, bit k set <=> corner k contributes
 *                (k = 0:(h_low,w_low) 1:(h_low,w_high) 2:(h_high,w_low) 3:(h_high,w_high))
 *   off[4*s+k] = flat element offset (channel 0) of corner k in the whole value
 *                tensor, or -1 if the corner does not contribute.
 * Uses the same device function as the forward/backward fp32 kernels.
 */
int msda_b200_debug_indices_f32(const int64_t *spatial_shapes, const int64_t *level_start,
                                const float *sampling_loc, int batch, int spatial_size,
                                int num_heads, int channels, int num_levels, int num_query,
                                int num_point, int32_t *idx, int64_t *off, void *stream);

/*
 * Tuning knobs for tools/sweep.py and the profiles; they select between
 * kernel variants that all produce the same results (forward: bit-identical;
 * backward: identical up to the order of the grad_value reductions).  Defaults
 * are what the shipped path uses.  Not thread-safe against concurrent launches.
 *   "fwd_variant"  0 = auto, other values select a specific forward kernel
 *   "bwd_variant"  0 = auto: where the queries are the value pixels (Lq == S, D = 32) the in-SM merging
 *                  kernel and the per-row reduction kernel are both launched, every CTA of both probes the
 *                  sampling locations and the kernel the verdict goes against returns at once; 1..8 = CTA
 *                  shapes of the per-row reduction kernel, 20..39 = the merging kernel and its tuning
 *                  variants, 63 = generic kernel
 *   "tile_order"   0 = auto (2-D tiles when the queries are laid out like the value pixels),
 *                  1 = groups of consecutive queries
 *   "ctas_per_sm"  0 = occupancy limit, k > 0 caps the persistent grid at k CTAs per SM
 *   "linear_variant"  msda_b200_linear_f32: 0 = auto (128/96-column tiles, A operand in tensor memory,
 *                  reductions longer than 256 accumulated in chunks of 256 that are added in registers),
 *                  2 = both operands in shared memory with four accumulators in one set, 3 = the same with
 *                  two {main, small} sets, 4 = same as 0
 *   "wgrad_chunk"  msda_b200_linear_wgrad_f32: 32-row blocks per work item (0 = 16, i.e. 512 rows)
 * Only in the profiling build (`make -C uni-encoder-code_b200/csrc profile`, -DMSDA_PROFILE_KNOBS; the
 * shipped library rejects the names): "whatif_drop_reds" and "whatif_linear" make kernels SKIP work on
 * purpose (wrong results) to time what-if experiments for profiles/; see tools/whatif*.py.
 */
int msda_b200_set_option(const char *name, int value);
int msda_b200_get_option(const char *name, int *value);

#ifdef __cplusplus
}
#endif
#endif /* MSDA_B200_H_ */
