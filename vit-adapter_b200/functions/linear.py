"""F.linear for the adapter's Linears with the bias gradient done by csrc/adapter_colsum.cu (SURVEY.md §8(f) N1).

Same arithmetic as nn.Linear / autocast(F.linear): inputs are cast to the autocast dtype when autocast is on, the forward
is one cuBLAS GEMM with the bias epilogue, the backward is the same two GEMMs torch runs. Only the third piece of the
backward differs: grad_bias = column sums of grad_output goes through the two-stage column-sum kernel instead of torch's
generic reduction (which at [86 016, 768] bf16 runs ~10x off the HBM roofline on B200). State-dict keys, parameter
dtypes and results (to rounding of the fp32 sum order) are unchanged; anything the kernel does not take calls F.linear.
Compiled code (torch.compile / torch.export) reaches the same kernel through the `msda_b200::colsum` custom op.
"""
import torch
import torch.nn.functional as F

from .. import _cabi
from .ms_deform_attn_func import _compiled_ops


class _LinearColsumBias(torch.autograd.Function):

    @staticmethod
    def forward(ctx, x, weight, bias):
        dt = torch.get_autocast_dtype('cuda') if torch.is_autocast_enabled('cuda') else x.dtype
        xc = x if x.dtype == dt else x.to(dt)
        wc = weight if weight.dtype == dt else weight.to(dt)
        bc = bias if bias.dtype == dt else bias.to(dt)
        y = F.linear(xc, wc, bc)   # operands already share the compute dtype: autocast, if on, has nothing left to cast
        ctx.save_for_backward(xc, wc)
        return y

    @staticmethod
    @torch.autograd.function.once_differentiable
    def backward(ctx, gy):
        xc, wc = ctx.saved_tensors
        gy2 = gy.reshape(-1, gy.shape[-1])
        if not gy2.is_contiguous():
            gy2 = gy2.contiguous()
        gx = gw = gb = None
        if gy2.dtype != wc.dtype:
            gy2 = gy2.to(wc.dtype)
        if ctx.needs_input_grad[0]:
            gx = (gy2 @ wc).view(xc.shape)
        if ctx.needs_input_grad[1]:
            gw = gy2.t() @ xc.reshape(-1, xc.shape[-1])
        if ctx.needs_input_grad[2]:
            if not _cabi.colsum_supported(gy2):
                gb = gy2.sum(0)
            elif torch.compiler.is_compiling():
                gb = _compiled_ops().colsum(gy2)
            else:
                gb = _cabi.colsum(gy2)
        return gx, gw, gb


_OK = (torch.float32, torch.bfloat16, torch.float16)


def linear(x, weight, bias, enabled=True):
    """F.linear(x, weight, bias); on CUDA with a trainable bias the backward's bias gradient uses the column-sum kernel."""
    if enabled and bias is not None and x.is_cuda and torch.is_grad_enabled() and bias.requires_grad:
        if torch.is_autocast_enabled('cuda'):
            ok = torch.get_autocast_dtype('cuda') in (torch.bfloat16, torch.float16) and x.dtype in _OK and weight.dtype in _OK and bias.dtype in _OK
        else:
            ok = x.dtype in _OK and weight.dtype == x.dtype and bias.dtype == x.dtype
        if ok:
            return _LinearColsumBias.apply(x, weight, bias)
    return F.linear(x, weight, bias)
