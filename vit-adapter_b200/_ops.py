"""The package's kernels as `torch.library` custom ops (namespace `msda_b200`), for torch.compile and torch.export.

Eager code never goes through these: it calls `_cabi` directly, as it always has. Code that Dynamo or torch.export traces
(`torch.compiler.is_compiling()`) reaches the same `_cabi` functions through the ops below, which the compiler sees as
opaque calls with known output shapes (`register_fake`, symbolic sizes included) and, where a gradient flows, a backward
(`register_autograd`) that calls the matching backward op.

Each op's implementation does, at run time on real tensors, the work Dynamo cannot trace: `.contiguous()` on every tensor
operand (the C ABI needs dense rows, and a caller's `.contiguous()` need not survive Inductor's layout choices), the
8/16-byte alignment copy of fused reference points, the residual kernel's 16-byte alignment, MSDeformAttn's shape check,
and everything `_cabi` does itself (device guard, stream handle, workspaces, `host_shapes`). The AMP value policy, dtype
casts and the `*_supported` predicates stay in the callers, where Dynamo traces them.

Differences from the eager autograd Functions:
  * `layernorm` returns `(y, stats)` only. The eager `_LayerNormRows` can also hand out `x.view_as(x)` and fold the
    residual connection's gradient into its backward kernel; a custom op cannot return an alias of its input, so compiled
    code uses `x` itself for the residual and Inductor adds the two gradients.
  * Custom ops cannot return None in a tensor slot. Backward ops whose gradients are optional return an EMPTY tensor
    (`numel() == 0`) in the slot they were not asked for: `ms_deform_attn_fused_backward` / `ms_deform_attn_merged_backward`
    for the reference-point gradient when `ref_grad` is False, `dwconv_backward` for the input gradient when
    `need_input` is False and for the weight and bias gradients when `need_weight` is False. They launch exactly the
    kernels the eager backward launches for the same flags.
  * `layernorm_backward` returns grad_weight and grad_bias stacked as one fp32 [2, C] tensor (the kernel writes them into
    one buffer, and op outputs may not alias each other).
  * MSDeformAttn checks `(H * W).sum() == Len_in` in its Python forward; compiled code cannot read device data there, so
    the three forward ops run the same check in their implementation, memoised per `spatial_shapes` tensor in a
    `TensorMemo` as the module does, and skipped while a CUDA graph is being captured.
"""
from typing import Optional

import torch

from . import _cabi
from .functions.ms_deform_attn_func import _fused_ref

Tensor = torch.Tensor

_LEN_IN_CHECKED = _cabi.TensorMemo(limit=64)


def _check_len_in(spatial_shapes, len_in):
    """MSDeformAttn's `(H * W).sum() == Len_in`: one device->host read per spatial_shapes tensor (and version, and Len_in),
    none in steady state and none during CUDA-graph capture."""
    if _LEN_IN_CHECKED.get(spatial_shapes, len_in) or torch.cuda.is_current_stream_capturing():
        return
    assert (spatial_shapes[:, 0] * spatial_shapes[:, 1]).sum() == len_in
    _LEN_IN_CHECKED.put(spatial_shapes, True, len_in)


def _dense(*tensors):
    return [t.contiguous() for t in tensors]


# --- plain multi-scale deformable attention (MSDeformAttnFunction) ----------------------------------------------------------
@torch.library.custom_op('msda_b200::ms_deform_attn', mutates_args=())
def ms_deform_attn(value: Tensor, spatial_shapes: Tensor, level_start_index: Tensor, sampling_locations: Tensor,
                   attention_weights: Tensor, im2col_step: int) -> Tensor:
    """out [N, Lq, M*D] in value's dtype (f32 / bf16 / f16 / f64); locations and weights f32 (f64 with f64 values)."""
    value, spatial_shapes, level_start_index, sampling_locations, attention_weights = _dense(
        value, spatial_shapes, level_start_index, sampling_locations, attention_weights)
    _check_len_in(spatial_shapes, value.shape[1])
    return _cabi.forward(value, spatial_shapes, level_start_index, sampling_locations, attention_weights, im2col_step)


@ms_deform_attn.register_fake
def _(value, spatial_shapes, level_start_index, sampling_locations, attention_weights, im2col_step):
    N, _, M, D = value.shape
    return value.new_empty((N, sampling_locations.shape[1], M * D))


@torch.library.custom_op('msda_b200::ms_deform_attn_backward', mutates_args=())
def ms_deform_attn_backward(value: Tensor, spatial_shapes: Tensor, level_start_index: Tensor, sampling_locations: Tensor,
                            attention_weights: Tensor, grad_output: Tensor, im2col_step: int) -> tuple[Tensor, Tensor, Tensor]:
    """(grad_value, grad_sampling_locations, grad_attention_weights); grad_output in value's dtype."""
    return _cabi.backward(*_dense(value, spatial_shapes, level_start_index, sampling_locations, attention_weights, grad_output),
                          im2col_step)


@ms_deform_attn_backward.register_fake
def _(value, spatial_shapes, level_start_index, sampling_locations, attention_weights, grad_output, im2col_step):
    return (value.new_empty(value.shape), sampling_locations.new_empty(sampling_locations.shape),
            attention_weights.new_empty(attention_weights.shape))


def _plain_setup(ctx, inputs, output):
    value, spatial_shapes, level_start_index, loc, attn, im2col_step = inputs
    ctx.save_for_backward(value, spatial_shapes, level_start_index, loc, attn)
    ctx.im2col_step = im2col_step


def _plain_backward(ctx, grad_output):
    value, spatial_shapes, level_start_index, loc, attn = ctx.saved_tensors
    gv, gl, ga = torch.ops.msda_b200.ms_deform_attn_backward(value, spatial_shapes, level_start_index, loc, attn,
                                                             grad_output.to(value.dtype), ctx.im2col_step)
    return gv, None, None, gl, ga, None


ms_deform_attn.register_autograd(_plain_backward, setup_context=_plain_setup)


# --- fused entry: raw offsets and logits (MSDeformAttnFusedFunction) --------------------------------------------------------
@torch.library.custom_op('msda_b200::ms_deform_attn_fused', mutates_args=())
def ms_deform_attn_fused(value: Tensor, spatial_shapes: Tensor, level_start_index: Tensor, reference_points: Tensor,
                         sampling_offsets: Tensor, attn_logits: Tensor) -> Tensor:
    """out [N, Lq, M*D] from raw sampling_offsets [N,Lq,M,L,P,2] and pre-softmax attn_logits [N,Lq,M,L*P] (f32);
    reference_points f32 [1|N, Lq, 1|L, 2 (points) | 4 (boxes)]."""
    value, spatial_shapes, level_start_index, sampling_offsets, attn_logits = _dense(
        value, spatial_shapes, level_start_index, sampling_offsets, attn_logits)
    _check_len_in(spatial_shapes, value.shape[1])
    return _cabi.forward_fused(value, spatial_shapes, level_start_index, _fused_ref(reference_points), sampling_offsets,
                               attn_logits)


@ms_deform_attn_fused.register_fake
def _(value, spatial_shapes, level_start_index, reference_points, sampling_offsets, attn_logits):
    N, _, M, D = value.shape
    return value.new_empty((N, sampling_offsets.shape[1], M * D))


@torch.library.custom_op('msda_b200::ms_deform_attn_fused_backward', mutates_args=())
def ms_deform_attn_fused_backward(value: Tensor, spatial_shapes: Tensor, level_start_index: Tensor, reference_points: Tensor,
                                  sampling_offsets: Tensor, attn_logits: Tensor, grad_output: Tensor,
                                  ref_grad: bool) -> tuple[Tensor, Tensor, Tensor, Tensor]:
    """(grad_value, grad_sampling_offsets, grad_attn_logits, grad_reference_points). grad_reference_points is f32 in the
    shape of reference_points when `ref_grad`, else an EMPTY tensor, and then no kernel is launched for it."""
    value, spatial_shapes, level_start_index, sampling_offsets, attn_logits, grad_output = _dense(
        value, spatial_shapes, level_start_index, sampling_offsets, attn_logits, grad_output)
    ref = _fused_ref(reference_points)
    grads = _cabi.backward_fused(value, spatial_shapes, level_start_index, ref, sampling_offsets, attn_logits, grad_output,
                                 ref_grad=ref_grad)
    return grads if ref_grad else grads + (ref.new_empty((0,)),)


@ms_deform_attn_fused_backward.register_fake
def _(value, spatial_shapes, level_start_index, reference_points, sampling_offsets, attn_logits, grad_output, ref_grad):
    grad_ref = reference_points.new_empty(reference_points.shape if ref_grad else (0,), dtype=torch.float32)
    return (value.new_empty(value.shape), sampling_offsets.new_empty(sampling_offsets.shape),
            attn_logits.new_empty(attn_logits.shape), grad_ref)


def _fused_setup(ctx, inputs, output):
    ctx.save_for_backward(*inputs)


def _fused_backward(ctx, grad_output):
    value, spatial_shapes, level_start_index, ref, offsets, logits = ctx.saved_tensors
    want_ref = ctx.needs_input_grad[3]
    gv, go, gl, gr = torch.ops.msda_b200.ms_deform_attn_fused_backward(
        value, spatial_shapes, level_start_index, ref, offsets, logits, grad_output.to(value.dtype), want_ref)
    return gv, None, None, gr if want_ref else None, go, gl


ms_deform_attn_fused.register_autograd(_fused_backward, setup_context=_fused_setup)


# --- fused entry fed by one GEMM (MSDeformAttnMergedFunction) ---------------------------------------------------------------
@torch.library.custom_op('msda_b200::ms_deform_attn_merged', mutates_args=())
def ms_deform_attn_merged(value: Tensor, spatial_shapes: Tensor, level_start_index: Tensor, reference_points: Tensor,
                          merged: Tensor, n_levels: int, n_points: int) -> Tensor:
    """out [N, Lq, M*D] from merged f32 [N, Lq, M*L*P*3]: raw offsets in the first M*L*P*2 columns, raw logits after."""
    value, spatial_shapes, level_start_index, merged = _dense(value, spatial_shapes, level_start_index, merged)
    _check_len_in(spatial_shapes, value.shape[1])
    return _cabi.forward_fused_merged(value, spatial_shapes, level_start_index, _fused_ref(reference_points), merged,
                                      n_levels, n_points)


@ms_deform_attn_merged.register_fake
def _(value, spatial_shapes, level_start_index, reference_points, merged, n_levels, n_points):
    N, _, M, D = value.shape
    return value.new_empty((N, merged.shape[1], M * D))


@torch.library.custom_op('msda_b200::ms_deform_attn_merged_backward', mutates_args=())
def ms_deform_attn_merged_backward(value: Tensor, spatial_shapes: Tensor, level_start_index: Tensor, reference_points: Tensor,
                                   merged: Tensor, n_levels: int, n_points: int, grad_output: Tensor,
                                   ref_grad: bool) -> tuple[Tensor, Tensor, Tensor]:
    """(grad_value, grad_merged in merged's layout, grad_reference_points): the last is EMPTY unless `ref_grad`."""
    value, spatial_shapes, level_start_index, merged, grad_output = _dense(
        value, spatial_shapes, level_start_index, merged, grad_output)
    ref = _fused_ref(reference_points)
    grads = _cabi.backward_fused_merged(value, spatial_shapes, level_start_index, ref, merged, n_levels, n_points,
                                        grad_output, ref_grad=ref_grad)
    return grads if ref_grad else grads + (ref.new_empty((0,)),)


@ms_deform_attn_merged_backward.register_fake
def _(value, spatial_shapes, level_start_index, reference_points, merged, n_levels, n_points, grad_output, ref_grad):
    grad_ref = reference_points.new_empty(reference_points.shape if ref_grad else (0,), dtype=torch.float32)
    return value.new_empty(value.shape), merged.new_empty(merged.shape), grad_ref


def _merged_setup(ctx, inputs, output):
    value, spatial_shapes, level_start_index, ref, merged, n_levels, n_points = inputs
    ctx.save_for_backward(value, spatial_shapes, level_start_index, ref, merged)
    ctx.lp = (n_levels, n_points)


def _merged_backward(ctx, grad_output):
    value, spatial_shapes, level_start_index, ref, merged = ctx.saved_tensors
    want_ref = ctx.needs_input_grad[3]
    gv, gm, gr = torch.ops.msda_b200.ms_deform_attn_merged_backward(
        value, spatial_shapes, level_start_index, ref, merged, *ctx.lp, grad_output.to(value.dtype), want_ref)
    return gv, None, None, gr if want_ref else None, gm, None, None


ms_deform_attn_merged.register_autograd(_merged_backward, setup_context=_merged_setup)


# --- adapter LayerNorm ------------------------------------------------------------------------------------------------------
@torch.library.custom_op('msda_b200::layernorm', mutates_args=())
def layernorm(x: Tensor, weight: Tensor, bias: Optional[Tensor], eps: float, out_dtype: torch.dtype) -> tuple[Tensor, Tensor]:
    """(y in out_dtype, stats f32 [2, rows] = mean, rstd) of a LayerNorm over x's last dimension (f32 weight / bias)."""
    return _cabi.layernorm_forward(x.contiguous(), weight.contiguous(), bias.contiguous() if bias is not None else None, eps,
                                   out_dtype)


@layernorm.register_fake
def _(x, weight, bias, eps, out_dtype):
    return x.new_empty(x.shape, dtype=out_dtype), x.new_empty((2, x.numel() // x.shape[-1]), dtype=torch.float32)


@torch.library.custom_op('msda_b200::layernorm_backward', mutates_args=())
def layernorm_backward(grad_y: Tensor, x: Tensor, weight: Tensor, stats: Tensor) -> tuple[Tensor, Tensor]:
    """(grad_x in x's dtype, f32 [2, C] = (grad_weight, grad_bias))."""
    return _cabi.layernorm_backward_stacked(*_dense(grad_y, x, weight, stats))


@layernorm_backward.register_fake
def _(grad_y, x, weight, stats):
    return x.new_empty(x.shape), x.new_empty((2, x.shape[-1]), dtype=torch.float32)


def _layernorm_setup(ctx, inputs, output):
    x, weight, bias, eps, out_dtype = inputs
    ctx.save_for_backward(x, weight, output[1])
    ctx.has_bias = bias is not None


def _layernorm_backward(ctx, grad_y, grad_stats):
    x, weight, stats = ctx.saved_tensors
    gx, gwb = torch.ops.msda_b200.layernorm_backward(grad_y, x, weight, stats)
    return gx, gwb[0], (gwb[1] if ctx.has_bias else None), None, None


layernorm.register_autograd(_layernorm_backward, setup_context=_layernorm_setup)


# --- depth-wise 3x3 on the adapter's token layout ------------------------------------------------------------------------
@torch.library.custom_op('msda_b200::dwconv', mutates_args=())
def dwconv(x: Tensor, weight: Tensor, bias: Optional[Tensor], H: int, W: int) -> Tensor:
    """Depth-wise 3x3 over the [B, 21n, C] token sequence of the H/8, H/16, H/32 maps (H, W: the H/16 grid)."""
    return _cabi.dwconv_forward(x.contiguous(), weight.contiguous(), bias.contiguous() if bias is not None else None, H, W)


@dwconv.register_fake
def _(x, weight, bias, H, W):
    return x.new_empty(x.shape)


@torch.library.custom_op('msda_b200::dwconv_backward', mutates_args=())
def dwconv_backward(x: Tensor, weight: Tensor, grad_y: Tensor, H: int, W: int, need_input: bool,
                    need_weight: bool) -> tuple[Tensor, Tensor, Tensor]:
    """(grad_x, grad_weight [C,1,3,3], grad_bias [C]) in x's / weight's dtype; grad_x is EMPTY unless `need_input`,
    grad_weight and grad_bias are EMPTY unless `need_weight` (the kernels for them are then not launched)."""
    gx, gw, gb = _cabi.dwconv_backward(*_dense(x, weight, grad_y), H, W, need_input=need_input, need_weight=need_weight)
    return (gx if need_input else x.new_empty((0,)), gw if need_weight else weight.new_empty((0,)),
            gb if need_weight else weight.new_empty((0,)))


@dwconv_backward.register_fake
def _(x, weight, grad_y, H, W, need_input, need_weight):
    C = x.shape[-1]
    return (x.new_empty(x.shape if need_input else (0,)), weight.new_empty((C, 1, 3, 3) if need_weight else (0,)),
            weight.new_empty((C,) if need_weight else (0,)))


def _dwconv_setup(ctx, inputs, output):
    x, weight, bias, H, W = inputs
    ctx.save_for_backward(x, weight)
    ctx.hw = (H, W)
    ctx.has_bias = bias is not None


def _dwconv_backward(ctx, grad_y):
    x, weight = ctx.saved_tensors
    need_input = ctx.needs_input_grad[0]
    need_weight = ctx.needs_input_grad[1] or ctx.needs_input_grad[2]
    gx, gw, gb = torch.ops.msda_b200.dwconv_backward(x, weight, grad_y, *ctx.hw, need_input, need_weight)
    return (gx if need_input else None, gw if need_weight else None, gb if need_weight and ctx.has_bias else None,
            None, None)


dwconv.register_autograd(_dwconv_backward, setup_context=_dwconv_setup)


# --- residual epilogue ------------------------------------------------------------------------------------------------------
@torch.library.custom_op('msda_b200::residual_add', mutates_args=())
def residual_add(res: Tensor, branch: Tensor) -> Tensor:
    """f32 res + (f32 | bf16 | f16) branch -> f32 in one pass (16-byte accesses: a misaligned operand is copied first)."""
    res, branch = _dense(res, branch)
    res, branch = [t if t.data_ptr() % 16 == 0 else t.clone() for t in (res, branch)]
    return _cabi.residual_add(res, branch)


@residual_add.register_fake
def _(res, branch):
    return res.new_empty(res.shape)


def _residual_setup(ctx, inputs, output):
    ctx.branch_dtype = inputs[1].dtype


def _residual_backward(ctx, grad):
    return grad, (grad.to(ctx.branch_dtype) if ctx.needs_input_grad[1] else None)


residual_add.register_autograd(_residual_backward, setup_context=_residual_setup)


# --- bias gradient of the adapter's Linears ---------------------------------------------------------------------------------
@torch.library.custom_op('msda_b200::colsum', mutates_args=())
def colsum(x: Tensor) -> Tensor:
    """f32 [C] = sum of x [..., C] over all leading dimensions (deterministic two-stage reduction)."""
    return _cabi.colsum(x.contiguous())


@colsum.register_fake
def _(x):
    return x.new_empty((x.shape[-1],), dtype=torch.float32)
