"""MSDeformAttnFunction — autograd entry of the B200-native multi-scale deformable attention.

Drop-in for the reference's `ops.functions.ms_deform_attn_func.MSDeformAttnFunction`
(detection/ops/functions/ms_deform_attn_func.py:19-46): same 6-argument `apply`, gradients for
arguments 0, 3 and 4 only, `once_differentiable` backward. The native side is the C-ABI library
declared in include/msda_b200.h (called through `_cabi`); there is no PyTorch / CPU fallback here.

AMP: the reference decorates forward with `custom_fwd(cast_inputs=torch.float32)` (:21), i.e. under
autocast everything is up-cast to fp32. That stays the default. `set_amp_value_dtype(torch.bfloat16)`
opts in to the bf16 I/O kernels under autocast (value / out in bf16, locations and weights fp32,
fp32 accumulation) — a capability the reference does not have; `torch.float16` does the same for fp16 autocast.

Under torch.compile / torch.export (`torch.compiler.is_compiling()`) the three Functions call the `torch.ops.msda_b200`
custom ops of `_ops.py` instead of `_cabi`: same kernels, but opaque to the compiler, so `apply` traces without a graph
break. Eager calls take the `_cabi` path exactly as before.
"""
import torch
from torch.autograd import Function
from torch.autograd.function import once_differentiable

from .. import _cabi

_AMP_VALUE_DTYPE = torch.float32


def set_amp_value_dtype(dtype):
    """dtype `value` is cast to when the op runs under torch.autocast (float32 = reference behaviour)."""
    global _AMP_VALUE_DTYPE
    if dtype not in (torch.float32, torch.bfloat16, torch.float16):
        raise ValueError('amp value dtype must be torch.float32, torch.bfloat16 or torch.float16')
    _AMP_VALUE_DTYPE = dtype


def _amp_value(value):
    """`value` in the dtype the kernels run on: the AMP value dtype under CUDA autocast, and fp16 up-cast to fp32 unless fp16
    was asked for (the reference's behaviour for fp16 AMP: the core runs in fp32)."""
    if torch.is_autocast_enabled('cuda') and value.is_cuda:
        value = value.to(_AMP_VALUE_DTYPE)
    if value.dtype == torch.float16 and _AMP_VALUE_DTYPE != torch.float16:
        value = value.float()
    return value


def _grad_output(grad_output, value):
    """grad_output contiguous and in value's dtype, as the backward kernels read it."""
    return grad_output.to(value.dtype).contiguous()


def _fused_ref(reference_points):
    """reference_points as the fused kernels read them: fp32, contiguous, and aligned to one point (8 bytes) or box (16
    bytes) - a view with an odd storage offset is copied."""
    ref = reference_points.float().contiguous()
    if ref.data_ptr() % (4 * ref.shape[-1]) != 0:
        ref = ref.clone()
    return ref


def _compiled_ops():
    """torch.ops.msda_b200, registered by importing `_ops` on the first compiled call (eager processes never load it)."""
    from .. import _ops  # noqa: F401
    return torch.ops.msda_b200


def _coord_dtype(value_dtype):
    return torch.float64 if value_dtype == torch.float64 else torch.float32


class MSDeformAttnFunction(Function):

    @staticmethod
    def forward(ctx, value, value_spatial_shapes, value_level_start_index,
                sampling_locations, attention_weights, im2col_step):
        value = _amp_value(value)
        cdt = _coord_dtype(value.dtype)
        # .to() is a no-op (same tensor) when the dtype already matches
        sampling_locations = sampling_locations.to(cdt)
        attention_weights = attention_weights.to(cdt)
        ctx.im2col_step = im2col_step
        if torch.compiler.is_compiling():
            output = _compiled_ops().ms_deform_attn(value, value_spatial_shapes, value_level_start_index,
                                                    sampling_locations, attention_weights, im2col_step)
        else:
            output = _cabi.forward(value, value_spatial_shapes, value_level_start_index,
                                   sampling_locations, attention_weights, im2col_step)
        ctx.save_for_backward(value, value_spatial_shapes, value_level_start_index,
                              sampling_locations, attention_weights)
        return output

    @staticmethod
    @once_differentiable
    def backward(ctx, grad_output):
        value, shapes, level_start, loc, attn = ctx.saved_tensors
        if torch.compiler.is_compiling():
            grad_value, grad_loc, grad_attn = _compiled_ops().ms_deform_attn_backward(
                value, shapes, level_start, loc, attn, _grad_output(grad_output, value), ctx.im2col_step)
            return grad_value, None, None, grad_loc, grad_attn, None
        grad_value, grad_loc, grad_attn = _cabi.backward(
            value, shapes, level_start, loc, attn, _grad_output(grad_output, value), ctx.im2col_step)
        return grad_value, None, None, grad_loc, grad_attn, None


class MSDeformAttnFusedFunction(Function):
    """Sampling core + the module arithmetic around it in one kernel (no reference counterpart as a
    separate Function: it fuses detection/ops/modules/ms_deform_attn.py:108-119 into the op):

        apply(value, spatial_shapes, level_start_index, reference_points, sampling_offsets, attn_logits)

    with RAW `sampling_offsets` [N,Lq,M,L,P,2] and RAW pre-softmax `attn_logits` [N,Lq,M,L*P]; the kernel forms
    softmax(attn_logits) and the sampling locations in registers, so neither tensor is written to HBM, and the
    backward returns gradients w.r.t. the raw offsets / logits. `reference_points` is [1|N, Lq, 1|L, 2] (points:
    reference_point + offset / (W_l, H_l)) or [1|N, Lq, 1|L, 4] (boxes: xy + offset / P * wh * 0.5). Its gradient is
    computed exactly when it requires one (Deformable-DETR style decoders); otherwise, as for the adapter's constant
    grid, the backward launches no extra kernel.
    Same AMP policy as MSDeformAttnFunction. Use `_cabi.fused_supported` to check for a kernel."""

    @staticmethod
    def forward(ctx, value, value_spatial_shapes, value_level_start_index, reference_points, sampling_offsets,
                attn_logits):
        value = _amp_value(value)
        compiling = torch.compiler.is_compiling()
        # (compiled: the op makes its own alignment copy of the reference points, at run time)
        reference_points = reference_points.float().contiguous() if compiling else _fused_ref(reference_points)
        sampling_offsets = sampling_offsets.float().contiguous()
        attn_logits = attn_logits.float().contiguous()
        if compiling:
            output = _compiled_ops().ms_deform_attn_fused(value, value_spatial_shapes, value_level_start_index,
                                                          reference_points, sampling_offsets, attn_logits)
        else:
            output = _cabi.forward_fused(value, value_spatial_shapes, value_level_start_index, reference_points,
                                         sampling_offsets, attn_logits)
        ctx.save_for_backward(value, value_spatial_shapes, value_level_start_index, reference_points,
                              sampling_offsets, attn_logits)
        return output

    @staticmethod
    @once_differentiable
    def backward(ctx, grad_output):
        value, shapes, level_start, ref, offsets, logits = ctx.saved_tensors
        want_ref = ctx.needs_input_grad[3]
        if torch.compiler.is_compiling():
            grads = _compiled_ops().ms_deform_attn_fused_backward(value, shapes, level_start, ref, offsets, logits,
                                                                  _grad_output(grad_output, value), want_ref)
        else:
            grads = _cabi.backward_fused(value, shapes, level_start, ref, offsets, logits, _grad_output(grad_output, value),
                                         ref_grad=want_ref)
        grad_value, grad_off, grad_logits = grads[:3]
        return grad_value, None, None, grads[3] if want_ref else None, grad_off, grad_logits


class MSDeformAttnMergedFunction(Function):
    """Fused entry fed by ONE GEMM: `merged` [N, Lq, M*L*P*3] = query @ cat(W_offsets, W_logits)^T + cat(b_offsets, b_logits)
    (both linears of the reference module read the same `query`, ms_deform_attn.py:108-111). The kernels read the two
    column blocks in place and write their gradient in the same layout, so the backward is also one GEMM.

        apply(value, spatial_shapes, level_start_index, reference_points, merged, n_levels, n_points)

    `reference_points` as in MSDeformAttnFusedFunction: points or boxes, with a gradient exactly when it requires one."""

    @staticmethod
    def forward(ctx, value, value_spatial_shapes, value_level_start_index, reference_points, merged, n_levels, n_points):
        value = _amp_value(value)
        compiling = torch.compiler.is_compiling()
        reference_points = reference_points.float().contiguous() if compiling else _fused_ref(reference_points)
        merged = merged.float().contiguous()
        ctx.lp = (int(n_levels), int(n_points))
        if compiling:
            output = _compiled_ops().ms_deform_attn_merged(value, value_spatial_shapes, value_level_start_index,
                                                           reference_points, merged, *ctx.lp)
        else:
            output = _cabi.forward_fused_merged(value, value_spatial_shapes, value_level_start_index, reference_points,
                                                merged, *ctx.lp)
        ctx.save_for_backward(value, value_spatial_shapes, value_level_start_index, reference_points, merged)
        return output

    @staticmethod
    @once_differentiable
    def backward(ctx, grad_output):
        value, shapes, level_start, ref, merged = ctx.saved_tensors
        want_ref = ctx.needs_input_grad[3]
        if torch.compiler.is_compiling():
            grads = _compiled_ops().ms_deform_attn_merged_backward(value, shapes, level_start, ref, merged, *ctx.lp,
                                                                   _grad_output(grad_output, value), want_ref)
        else:
            grads = _cabi.backward_fused_merged(value, shapes, level_start, ref, merged, *ctx.lp,
                                                _grad_output(grad_output, value), ref_grad=want_ref)
        return grads[0], None, None, grads[2] if want_ref else None, grads[1], None, None
