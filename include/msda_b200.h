/*
 * msda_b200.h — C ABI of the B200-native multi-scale deformable attention core.
 *
 * This header is the drop-in boundary for the hot path of ViT-Adapter's MSDeformAttn.
 * It replaces the pybind11 surface of the reference extension
 *   detection/ops/src/vision.cpp:13-16            (ms_deform_attn_forward / ms_deform_attn_backward)
 *   detection/ops/src/ms_deform_attn.h:20-61      (device dispatch)
 *   detection/ops/src/cuda/ms_deform_attn_cuda.cu:20-80, :83-153   (host wrappers)
 * with plain pointers + sizes: no torch / ATen types cross this boundary.
 *
 * Conventions
 *   - All tensor pointers are DEVICE pointers to contiguous row-major storage.
 *   - msda_forward / msda_backward accept any pointer aligned to its element size (else MSDA_E_ALIGN); better
 *     aligned tensors may take faster kernels, with results within the same rounding bounds. The fused entry points
 *     need 16-byte aligned value / out / grad_out and 8-byte aligned offsets, but only the element size of a 16-bit
 *     grad_value.
 *   - The library never allocates or frees tensor memory (the reference allocates with
 *     at::zeros inside C++, ms_deform_attn_cuda.cu:54,121-123). The caller owns every buffer.
 *   - `stream` is a cudaStream_t passed as void*; every call is asynchronous w.r.t. the host,
 *     performs no host<->device synchronisation and no allocation, so it is CUDA-graph capturable.
 *   - Return value: 0 on success, a negative MSDA_E_* code for argument errors, or a positive
 *     cudaError_t for CUDA runtime/launch errors (the reference only printf()s launch errors,
 *     ms_deform_im2col_cuda.cuh:948-952,1321-1325; here they are surfaced).
 *     msda_last_error() returns a thread-local human-readable message for the last failure.
 *   - Thread-safe and re-entrant. The only process-wide mutable state is (a) the benchmark knobs of msda_set_tuning()
 *     (atomics; 0 = heuristic, never needed for correctness), (b) the launch counter of msda_launch_count() and (c) a
 *     per-device cache of the SM count. Results never depend on any of them beyond the summation order of atomics.
 *
 * Tensor layouts (identical to the reference, ms_deform_attn_func.py:20-33):
 *   value              [N, S, M, D]        dtype T   (T = f32 | bf16 | f16 | f64)
 *   spatial_shapes     [L, 2]  int64       (H_l, W_l)      -- on device, as in the reference
 *   level_start_index  [L]     int64                         -- on device
 *   sampling_loc       [N, Lq, M, L, P, 2] dtype F   (x, y) normalised to [0,1]
 *   attn_weight        [N, Lq, M, L, P]    dtype F
 *   out / grad_out     [N, Lq, M*D]        dtype T
 *   grad_value         [N, S, M, D]        dtype T
 *   grad_sampling_loc  like sampling_loc, grad_attn_weight like attn_weight (dtype F)
 * where F = f32 for T in {f32, bf16, f16} and F = f64 for T = f64.
 */
#ifndef MSDA_B200_H_
#define MSDA_B200_H_

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define MSDA_ABI_VERSION 1

/* dtype of value / out / grad_out / grad_value */
enum msda_dtype {
  MSDA_F32 = 0,  /* loc/aw f32; the reference's production dtype (custom_fwd casts to fp32)   */
  MSDA_BF16 = 1, /* loc/aw f32, fp32 accumulation; new capability (reference has no bf16 path) */
  MSDA_F64 = 2,  /* loc/aw f64; exists so the reference's fp64 gradcheck (ops/test.py:78-101) runs */
  MSDA_F16 = 3   /* fp16 I/O, loc/aw f32, fp32 accumulation (like MSDA_BF16; for the reference's `fp16 = dict(loss_scale=...)` AMP
                    configs). The Python layer keeps the reference's behaviour - fp32 up-cast under fp16 AMP - unless asked
                    (set_amp_value_dtype(torch.float16)); not available in the shared-memory forward */
};

/* negative error codes */
enum msda_error {
  MSDA_OK = 0,
  MSDA_E_NULL = -1,      /* a required pointer is NULL                                  */
  MSDA_E_DIMS = -2,      /* a dimension is <= 0 or a product overflows int32            */
  MSDA_E_DTYPE = -3,     /* unknown dtype                                               */
  MSDA_E_ALIGN = -4,     /* pointer not aligned to the element size                     */
  MSDA_E_LEVELS = -5,    /* more levels than MSDA_MAX_LEVELS                            */
  MSDA_E_WORKSPACE = -6, /* workspace missing or too small (see msda_backward_workspace_bytes) */
  MSDA_E_STEP = -7,      /* batch not divisible by min(batch, im2col_step)              */
  MSDA_E_UNSUPPORTED = -8 /* no kernel for this configuration (fused entry points only; use the plain ones) */
};

#define MSDA_MAX_LEVELS 16

/* Problem dimensions — the 7 ints the reference host code extracts from the tensors
 * (ms_deform_attn_cuda.cu:40-48). */
typedef struct msda_dims {
  int32_t batch;        /* N  */
  int32_t spatial_size; /* S  = sum_l H_l*W_l */
  int32_t num_heads;    /* M  */
  int32_t channels;     /* D  (per head) */
  int32_t num_levels;   /* L  */
  int32_t num_query;    /* Lq */
  int32_t num_point;    /* P  */
} msda_dims;

/* ABI version of the loaded library (== MSDA_ABI_VERSION it was built with). */
int msda_abi_version(void);

/* Thread-local message describing the last non-zero return on this thread ("" if none). */
const char* msda_last_error(void);

/* Same precondition the reference asserts (ms_deform_attn_cuda.cu:50-52): batch % min(batch, step) == 0.
 * The step is otherwise ignored: one launch covers the whole batch. Returns 0 or MSDA_E_STEP. */
int msda_check_im2col_step(int32_t batch, int32_t im2col_step);

/* Forward: replaces ms_deform_attn_cuda_forward (ms_deform_attn_cuda.cu:20-80) and kernel
 * ms_deformable_im2col_gpu_kernel (ms_deform_im2col_cuda.cuh:237-299).
 * `out` is fully overwritten (no pre-zeroing needed). */
int msda_forward(const msda_dims* dims, int dtype,
                 const void* value,
                 const int64_t* spatial_shapes,
                 const int64_t* level_start_index,
                 const void* sampling_loc,
                 const void* attn_weight,
                 void* out,
                 void* stream);

/* Forward with the level shapes ALSO available on the host (`spatial_shapes_host`: [L,2] int64 in host
 * memory, same values as the device tensor; may be NULL, which makes this identical to msda_forward).
 * Host-known shapes let the library choose kernels that need the level geometry before launch (today: the
 * opt-in shared-memory forward that stages whole level maps with cp.async). The reference reads the shapes only on the device (ms_deform_im2col_cuda.cuh:274-277); a caller
 * that built the shapes tensor from Python ints (adapter_modules.py:30-33) has them on the host for free. */
int msda_forward_ex(const msda_dims* dims, int dtype,
                    const void* value,
                    const int64_t* spatial_shapes,
                    const int64_t* level_start_index,
                    const void* sampling_loc,
                    const void* attn_weight,
                    void* out,
                    const int64_t* spatial_shapes_host,
                    void* stream);

/* Bytes of scratch the backward needs for (dims, dtype); 0 when none is needed.
 * (bf16 / f16 accumulate grad_value in an fp32 scratch of N*S*M*D floats; calls that take the slab-sorted backward -
 * single-level calls with many samples per value token, see msda_set_tuning "bwd_sorted" - add the sort buffers: one
 * 4-byte index per sample plus the histograms. Ask again after changing a tuning key.) */
size_t msda_backward_workspace_bytes(const msda_dims* dims, int dtype);

/* Backward: replaces ms_deform_attn_cuda_backward (ms_deform_attn_cuda.cu:83-153) and the col2im
 * kernels (ms_deform_im2col_cuda.cuh:301-920).
 * grad_value, grad_sampling_loc and grad_attn_weight are fully written by the call (grad_value is
 * zero-filled on `stream` before the scatter; the caller does not pre-zero anything).
 * `workspace` may be NULL when msda_backward_workspace_bytes() == 0. */
int msda_backward(const msda_dims* dims, int dtype,
                  const void* value,
                  const int64_t* spatial_shapes,
                  const int64_t* level_start_index,
                  const void* sampling_loc,
                  const void* attn_weight,
                  const void* grad_out,
                  void* grad_value,
                  void* grad_sampling_loc,
                  void* grad_attn_weight,
                  void* workspace, size_t workspace_bytes,
                  void* stream);

/* Fused entry points: the module arithmetic around the sampling core (reference:
 * detection/ops/modules/ms_deform_attn.py:108-119) is done inside the kernels, in registers:
 *     attention_weights = softmax(attn_logits over the L*P points of each (b, q, m))      [warp shuffles]
 *     sampling_location = reference_point + sampling_offset / (W_l, H_l)
 * so neither tensor is ever materialised in HBM.
 *   reference_points  [ref_batch, Lq, ref_levels, 2] f32, ref_batch in {1, N}, ref_levels in {1, L}
 *                     (the adapter passes [1, Lq, 1, 2]; both broadcasts of the reference's indexing
 *                     `reference_points[:, :, None, :, None, :]` are supported)
 *   sampling_offsets  [N, Lq, M, L, P, 2] f32 — raw output of the `sampling_offsets` linear
 *   attn_logits       [N, Lq, M, L*P]     f32 — raw output of the `attention_weights` linear (pre-softmax)
 *   offsets_row_stride / logits_row_stride: floats between consecutive (b, q) rows of the two tensors; 0 = dense
 *                     (M*L*P*2 and M*L*P). Non-dense strides let both be column blocks of ONE merged GEMM output
 *                     [N*Lq, M*L*P*3] (`sampling_offsets` and `attention_weights` share the same input); the
 *                     gradients are written with the same strides, so they form the merged GEMM's output gradient.
 * The backward returns gradients w.r.t. the raw offsets and logits (softmax backward folded in).
 * Supported: dtype f32 / bf16 / f16, (L, P) in {(3,4), (1,4), (4,4)}, D = 32 or 64 (D*sizeof(T) a multiple of 16 with
 * 2..32 lanes in the forward, D / 4 in {8, 16} in the backward); anything else returns MSDA_E_UNSUPPORTED and the
 * caller uses msda_forward / msda_backward.
 * msda_forward_fused / msda_backward_fused are msda_forward_fused_ref / msda_backward_fused_ref with ref_dim = 2 and
 * grad_reference_points = NULL. */
int msda_forward_fused(const msda_dims* dims, int dtype,
                       const void* value,
                       const int64_t* spatial_shapes,
                       const int64_t* level_start_index,
                       const float* reference_points, int32_t ref_batch, int32_t ref_levels,
                       const float* sampling_offsets,
                       const float* attn_logits,
                       int64_t offsets_row_stride, int64_t logits_row_stride,
                       void* out,
                       void* stream);

int msda_backward_fused(const msda_dims* dims, int dtype,
                        const void* value,
                        const int64_t* spatial_shapes,
                        const int64_t* level_start_index,
                        const float* reference_points, int32_t ref_batch, int32_t ref_levels,
                        const float* sampling_offsets,
                        const float* attn_logits,
                        int64_t offsets_row_stride, int64_t logits_row_stride,
                        const void* grad_out,
                        void* grad_value,
                        float* grad_sampling_offsets,
                        float* grad_attn_logits,
                        void* workspace, size_t workspace_bytes,
                        void* stream);

/* Fused entry points for every reference-point form the reference module accepts (ms_deform_attn.py:115-122):
 *   ref_dim 2: reference_points [ref_batch, Lq, ref_levels, 2]  points (x, y):
 *              sampling_location = reference_point + sampling_offset / (W_l, H_l)
 *   ref_dim 4: reference_points [ref_batch, Lq, ref_levels, 4]  boxes (x, y, w, h), 16-byte aligned:
 *              sampling_location = (x, y) + sampling_offset / P * (w, h) * 0.5
 *              (torch's fp32 operations in torch's order: the locations are bit-identical to the unfused path)
 * anything else returns MSDA_E_DIMS; a misaligned box returns MSDA_E_ALIGN.
 * grad_reference_points: NULL = not wanted (the backward then launches exactly what msda_backward_fused launches), or
 *   f32 [ref_batch, Lq, ref_levels, ref_dim], fully written by the call. The sum over heads, points (and levels /
 *   batch where the reference points broadcast) uses no atomics: the result is bitwise reproducible. It needs the
 *   larger workspace of msda_backward_fused_workspace_bytes(..., with_ref_grad = 1) and one more kernel launch. */
int msda_forward_fused_ref(const msda_dims* dims, int dtype,
                           const void* value,
                           const int64_t* spatial_shapes,
                           const int64_t* level_start_index,
                           const float* reference_points, int32_t ref_batch, int32_t ref_levels, int32_t ref_dim,
                           const float* sampling_offsets,
                           const float* attn_logits,
                           int64_t offsets_row_stride, int64_t logits_row_stride,
                           void* out,
                           void* stream);

int msda_backward_fused_ref(const msda_dims* dims, int dtype,
                            const void* value,
                            const int64_t* spatial_shapes,
                            const int64_t* level_start_index,
                            const float* reference_points, int32_t ref_batch, int32_t ref_levels, int32_t ref_dim,
                            const float* sampling_offsets,
                            const float* attn_logits,
                            int64_t offsets_row_stride, int64_t logits_row_stride,
                            const void* grad_out,
                            void* grad_value,
                            float* grad_sampling_offsets,
                            float* grad_attn_logits,
                            float* grad_reference_points,
                            void* workspace, size_t workspace_bytes,
                            void* stream);

/* Bytes of scratch the fused backward needs (16-byte aligned): the fp32 grad_value accumulator of the 16-bit dtypes
 * (N*S*M*D floats; 0 for f32), then, when with_ref_grad != 0, the reference-point gradient partials at the next
 * 16-byte boundary: N*Lq*M*ref_levels*ref_dim floats. 0 when dims is NULL, ref_dim is not 2 or 4, or the reference
 * points do not broadcast (ref_batch not in {1, N}, ref_levels not in {1, L}). */
size_t msda_backward_fused_workspace_bytes(const msda_dims* dims, int dtype, int32_t ref_batch, int32_t ref_levels,
                                           int32_t ref_dim, int32_t with_ref_grad);

/* ------------------------------------------------------------------------------------------------
 * Adapter ConvFFN depth-wise 3x3 convolution on the token layout (SURVEY.md §8(f) N3).
 * Replaces DWConv.forward of the reference (adapter_modules.py:73-87: slice the [B, 21n, C] sequence into the
 * three maps 2Hx2W / HxW / (H/2)x(W/2), transpose each to NCHW, nn.Conv2d(C, C, 3, 1, 1, groups=C), transpose
 * back, concatenate) with one kernel that reads and writes the tokens in place (channels-last).
 *   x, y, grad_y, grad_x   [B, n_tokens, C]  dtype T (f32 | bf16 | f16 | f64), n_tokens = 21 * H * W / 4, H and W even
 *   weight                 [C, 1, 3, 3]      dtype T ;  bias [C] dtype T or NULL
 *   grad_weight [C*9], grad_bias [C]: fp32 accumulators for T in {f32, bf16, f16}, fp64 for T = f64 (fully written here)
 *   workspace: adapter_dwconv_backward_weight_workspace_bytes(...) bytes of device scratch (per-CTA partial sums of the
 *   deterministic two-stage reduction); 0 = none needed (generic path: f64 or C % 4 != 0, reduced with atomics).
 * ------------------------------------------------------------------------------------------------ */
int adapter_dwconv_forward(int dtype, const void* x, const void* weight, const void* bias, void* y,
                           int32_t batch, int32_t n_tokens, int32_t channels, int32_t H, int32_t W, void* stream);
int adapter_dwconv_backward_input(int dtype, const void* grad_y, const void* weight, void* grad_x,
                                  int32_t batch, int32_t n_tokens, int32_t channels, int32_t H, int32_t W, void* stream);
size_t adapter_dwconv_backward_weight_workspace_bytes(int dtype, int32_t batch, int32_t n_tokens, int32_t channels,
                                                      int32_t H, int32_t W);
int adapter_dwconv_backward_weight(int dtype, const void* x, const void* grad_y, void* grad_weight, void* grad_bias,
                                   int32_t batch, int32_t n_tokens, int32_t channels, int32_t H, int32_t W,
                                   void* workspace, size_t workspace_bytes, void* stream);

/* ------------------------------------------------------------------------------------------------
 * Adapter LayerNorm prologues (SURVEY.md §8(f) N2).
 * Replaces the nn.LayerNorm(dim, eps=1e-6) calls in front of every Linear of the Injector / Extractor
 * (adapter_modules.py:101-103,110-116,133-134,142-145: query_norm, feat_norm, ffn_norm):
 *   y = (x - mean(x)) / sqrt(var(x) + eps) * gamma + beta   per row of C channels, biased variance,
 * with y written directly in the consumer's dtype (bf16 under AMP: torch writes fp32 and the Linear casts it
 * with another full pass) and mean / rstd saved for the backward.
 *   x, grad_x [rows, C] in_dtype ; y, grad_y [rows, C] out_dtype ; (in, out) in {(f32,f32), (f32,bf16), (bf16,bf16), (f32,f16), (f16,f16)}
 *   gamma, beta [C] fp32 (beta may be NULL) ; mean, rstd [rows] fp32 ; grad_gamma, grad_beta [C] fp32 (fully written)
 *   C % 4 == 0 and C <= 1024, else MSDA_E_UNSUPPORTED (the caller keeps torch's LayerNorm)
 *   workspace: adapter_layernorm_backward_workspace_bytes(rows, C) bytes, 16-byte aligned (per-CTA partial sums of the
 *   deterministic two-stage grad_gamma / grad_beta reduction).
 * ------------------------------------------------------------------------------------------------ */
int adapter_layernorm_forward(int in_dtype, int out_dtype, const void* x, const void* gamma, const void* beta, void* y,
                              float* mean, float* rstd, int64_t rows, int32_t channels, float eps, void* stream);
size_t adapter_layernorm_backward_workspace_bytes(int64_t rows, int32_t channels);
/* grad_residual (optional, [rows, C] in_dtype, may be NULL): when x also feeds a residual connection
 * (query + f(LN(query)), adapter_modules.py:113-116), the gradient arriving over that connection; it is added into
 * grad_x here, which removes autograd's separate full-tensor add. */
int adapter_layernorm_backward(int in_dtype, int out_dtype, const void* grad_y, const void* x, const void* gamma,
                               const float* mean, const float* rstd, const void* grad_residual, void* grad_x,
                               float* grad_gamma, float* grad_beta, int64_t rows, int32_t channels, void* workspace,
                               size_t workspace_bytes, void* stream);

/* Residual epilogue of the Extractor (SURVEY.md §8(f) N2; adapter_modules.py:113-116 `query = query + attn`,
 * `query = query + drop_path(ffn(...))`): out[i] = residual[i] + (float)branch[i] with an fp32 stream and an f32 | bf16 | f16
 * branch (the mixed-dtype case torch's add does not vectorise). n % 8 == 0, 16-byte aligned pointers; out may alias
 * residual. Anything else: MSDA_E_UNSUPPORTED / MSDA_E_ALIGN and the caller keeps torch's add. */
int adapter_residual_add(int branch_dtype, const float* residual, const void* branch, float* out, int64_t n, void* stream);

/* ------------------------------------------------------------------------------------------------
 * Bias gradient of the adapter's Linears (SURVEY.md §8(f) N1): out[c] = sum over rows of x[row, c], fp32.
 * Replaces the row reduction inside the backward of every nn.Linear with a bias in MSDeformAttn
 * (ms_deform_attn.py:57-60) and ConvFFN (adapter_modules.py:56,60).
 *   x [rows, C] f32 (C % 4 == 0, C <= 1024) or bf16 / f16 (C % 8 == 0, C <= 2048), 16-byte aligned; out [C] fp32
 *   workspace: adapter_colsum_workspace_bytes(dtype, rows, C) bytes (per-CTA partial rows; deterministic sum)
 *   anything else returns MSDA_E_UNSUPPORTED (the caller keeps torch's sum).
 * ------------------------------------------------------------------------------------------------ */
size_t adapter_colsum_workspace_bytes(int dtype, int64_t rows, int32_t channels);
int adapter_colsum(int dtype, const void* x, int64_t rows, int32_t channels, float* out, void* workspace,
                   size_t workspace_bytes, void* stream);

/* Test hook: for every sampling point (N*Lq*M*L*P of them, same order as attn_weight) write
 *   idx[4*i+0] = h_low, idx[4*i+1] = w_low,
 *   idx[4*i+2] = corner-validity mask (bit k = corner k+1 is read; 0 = sample skipped),
 *   idx[4*i+3] = element offset of corner (h_low, w_low) inside value[b] (token*M*D + m*D)
 * computed by the SAME device routine the kernels use. f32 locations only.
 * Pins the index / level-offset arithmetic of ms_deform_im2col_cuda.cuh:33-53,274-288. */
int msda_debug_point_index(const msda_dims* dims,
                           const int64_t* spatial_shapes,
                           const int64_t* level_start_index,
                           const float* sampling_loc,
                           int32_t* idx,
                           void* stream);

/* Number of kernel launches (ours) issued through this library by the calling process so far. */
uint64_t msda_launch_count(void);

/* Tuning overrides for benchmarking; value 0 restores the built-in heuristic. Process-wide. Keys:
 *   "fwd_chunk", "bwd_chunk"        queries per CTA chunk of the L1-path kernels
 *   "fwd_min_ctas", "bwd_min_ctas"  min-resident-CTAs-per-SM variant (forward 3|4|6, backward 2|3|4)
 *   "fwd_smem"                      2 = use the shared-memory forward whenever a plan exists (default: never;
 *                                   measured no faster than the L1 path, see msda_abi.cu plan_forward_smem)
 *   "fwd_wide"                      fp32 forward with 32-byte lanes (LDG.256): 1 = off, 2 = on
 *   "fwd_smem_threads"              512 | 1024 threads per CTA of the shared-memory forward
 *   "fwd_smem_chunks"               query chunks per (batch, head) of the shared-memory forward
 *   "bwd_cell"                      2 = the cell-bucketed backward (msda_bwd_cell.cu; D in {32, 64}); default: the query-order kernel
 *   "bwd_cell_chunk"                queries per chunk of the cell-bucketed backward
 *   "bwd_packed16"                  2 = bf16 / f16 backward with packed 16-bit reductions straight into grad_value (no fp32
 *                                   scratch, no convert kernel; every contribution rounded to 16 bits - looser numerics)
 *   "bwd_sorted"                    slab-sorted backward (msda_bwd_sorted.cu; D in {32, 64}): 0 = where it measured faster (one
 *                                   level, >= 16 samples per value token and head, and >= 1 M samples at D = 32 / >= 0.25 M at D = 64), 1 = never,
 *                                   2 = wherever it applies. Changes msda_backward_workspace_bytes().
 * Returns 0, or MSDA_E_NULL for an unknown key. */
int msda_set_tuning(const char* key, int32_t value);

#ifdef __cplusplus
}
#endif
#endif /* MSDA_B200_H_ */
