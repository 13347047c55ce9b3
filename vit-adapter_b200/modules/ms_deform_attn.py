"""MSDeformAttn — the nn.Module around the B200-native sampling core.

Drop-in for the reference's `ops.modules.MSDeformAttn` (detection/ops/modules/ms_deform_attn.py:28-130):
same constructor, same sub-module names (`sampling_offsets`, `attention_weights`, `value_proj`,
`output_proj` — so reference checkpoints load unchanged), same initialisation (:64-81), same forward
arithmetic (:102-129). The four linears stay cuBLAS GEMMs (tensor-core work is not this path); the
sampling core goes through MSDeformAttnFunction -> include/msda_b200.h.

One deliberate difference: the reference evaluates `assert (H*W).sum() == Len_in` on CUDA tensors on
every call (:99-100), which is a device->host synchronisation per forward. Here the same check runs
once per distinct (spatial_shapes tensor object, version, Len_in) and is cached, so steady-state forwards
never synchronise and the module can be captured in a CUDA graph.

Under torch.compile / torch.export the forward traces without a graph break: the Functions call the msda_b200 custom ops,
the shape check runs inside those ops (same memo policy), and the merged query weight is a plain torch.cat.
"""
import math
import warnings

import torch
import torch.nn.functional as F
from torch import nn

from .. import _cabi
from ..functions import MSDeformAttnFunction, MSDeformAttnFusedFunction, MSDeformAttnMergedFunction, linear


class _MergedQueryParams(torch.autograd.Function):
    """cat(sampling_offsets.weight, attention_weights.weight) and cat(their biases) in two PERSISTENT buffers owned by the
    module. The buffers are rewritten only when one of the four parameters changed (version counters / storage), so an
    inference loop or a checkpointed re-forward issues no cat kernel at all, and the backward hands the two halves of the
    merged gradient back as views (no split kernels). State-dict keys are untouched: the buffers are plain attributes."""

    @staticmethod
    def forward(ctx, w_off, w_attn, b_off, b_attn, owner):
        key = tuple((t._version, t.data_ptr(), t.dtype, t.device) for t in (w_off, w_attn, b_off, b_attn))
        cache = owner.__dict__.get('_merged_cache')
        if cache is None or cache[0] != key:
            n = w_off.shape[0] + w_attn.shape[0]
            if cache is not None and cache[1].shape == (n, w_off.shape[1]) and cache[1].dtype == w_off.dtype and cache[1].device == w_off.device:
                w, b = cache[1], cache[2]
            else:
                w = torch.empty((n, w_off.shape[1]), dtype=w_off.dtype, device=w_off.device)
                b = torch.empty((n,), dtype=b_off.dtype, device=b_off.device)
            torch.cat([w_off.detach(), w_attn.detach()], 0, out=w)
            torch.cat([b_off.detach(), b_attn.detach()], 0, out=b)
            owner.__dict__['_merged_cache'] = (key, w, b)
        else:
            w, b = cache[1], cache[2]
        ctx.n_off = w_off.shape[0]
        # views of the buffers, so that autograd sees fresh outputs of this node every call
        return w.view_as(w), b.view_as(b)

    @staticmethod
    def backward(ctx, gw, gb):
        n = ctx.n_off
        return (gw[:n] if gw is not None else None, gw[n:] if gw is not None else None,
                gb[:n] if gb is not None else None, gb[n:] if gb is not None else None, None)


def _is_power_of_2(n):
    if not isinstance(n, int) or n < 0:
        raise ValueError('invalid input for _is_power_of_2: {} (type: {})'.format(n, type(n)))
    return n != 0 and (n & (n - 1)) == 0


class MSDeformAttn(nn.Module):
    """Multi-scale deformable attention (d_model, n_levels, n_heads, n_points, ratio)."""

    def __init__(self, d_model=256, n_levels=4, n_heads=8, n_points=4, ratio=1.0):
        super().__init__()
        if d_model % n_heads != 0:
            raise ValueError('d_model must be divisible by n_heads, but got {} and {}'.format(d_model, n_heads))
        if not _is_power_of_2(d_model // n_heads):
            warnings.warn("You'd better set d_model in MSDeformAttn to make the dimension of each attention "
                          'head a power of 2 which is more efficient in our CUDA implementation.')
        self.im2col_step = 64
        self.d_model = d_model
        self.n_levels = n_levels
        self.n_heads = n_heads
        self.n_points = n_points
        self.ratio = ratio
        d_value = int(d_model * ratio)
        self.sampling_offsets = nn.Linear(d_model, n_heads * n_levels * n_points * 2)
        self.attention_weights = nn.Linear(d_model, n_heads * n_levels * n_points)
        self.value_proj = nn.Linear(d_model, d_value)
        self.output_proj = nn.Linear(d_value, d_model)
        self._checked_shapes = _cabi.TensorMemo(limit=64)
        self._merged_cache = None   # (key, weight, bias) of _MergedQueryParams
        # fuse softmax + location arithmetic into the sampling kernel when a fused kernel exists (CUDA, fp32 / bf16 /
        # fp16, D in {32, 64}, (L,P) in {(3,4),(1,4),(4,4)}; 2-d or 4-d reference points, with or without gradient);
        # results differ from the unfused path only by the rounding of the softmax normalisation and the order of the
        # reference-point gradient's sum. Set to False to force the reference's op sequence.
        self.fused = True
        self.merge_query_linears = True
        # bias gradients of value_proj / output_proj / the merged query linear through the column-sum kernel
        # (functions/linear.py); False = nn.Linear's own backward
        self.colsum_bias_grad = True
        self._reset_parameters()

    def _reset_parameters(self):
        # reference :64-81 — zero offset weights; bias = one ray per head (unit step in the max-norm),
        # point k sits k+1 steps out; uniform attention (zero logits); xavier value/output projections.
        M, L, P = self.n_heads, self.n_levels, self.n_points
        with torch.no_grad():
            self.sampling_offsets.weight.zero_()
            theta = torch.arange(M, dtype=torch.float32) * (2.0 * math.pi / M)
            ray = torch.stack([theta.cos(), theta.sin()], -1)
            ray = ray / ray.abs().max(-1, keepdim=True)[0]
            steps = torch.arange(1, P + 1, dtype=torch.float32).view(1, 1, P, 1)
            bias = ray.view(M, 1, 1, 2).repeat(1, L, P, 1) * steps
            self.sampling_offsets.bias = nn.Parameter(bias.reshape(-1))
            self.attention_weights.weight.zero_()
            self.attention_weights.bias.zero_()
            nn.init.xavier_uniform_(self.value_proj.weight)
            self.value_proj.bias.zero_()
            nn.init.xavier_uniform_(self.output_proj.weight)
            self.output_proj.bias.zero_()

    def __getstate__(self):
        state = self.__dict__.copy()
        state['_merged_cache'] = None   # derived from the four parameters; rebuilt on the next forward
        return state

    def _check_len_in(self, spatial_shapes, len_in):
        # compiled code cannot read device data here: the msda_b200 forward ops run the same memoised check at run time
        if torch.compiler.is_compiling():
            return
        # memo keyed by tensor identity + version (NOT data_ptr: freed addresses are reused by the allocator)
        if self._checked_shapes.get(spatial_shapes, int(len_in)):
            return
        assert (spatial_shapes[:, 0] * spatial_shapes[:, 1]).sum() == len_in
        self._checked_shapes.put(spatial_shapes, True, int(len_in))

    def forward(self, query, reference_points, input_flatten, input_spatial_shapes,
                input_level_start_index, input_padding_mask=None):
        """query (N, Lq, C); reference_points (N|1, Lq, n_levels|1, 2 or 4) in [0,1];
        input_flatten (N, sum H_l*W_l, C); input_spatial_shapes (n_levels, 2) int64 (H, W);
        input_level_start_index (n_levels,) int64; input_padding_mask (N, sum H_l*W_l) bool or None.
        Returns (N, Lq, C)."""
        N, Lq, _ = query.shape
        _, len_in, _ = input_flatten.shape
        self._check_len_in(input_spatial_shapes, len_in)
        M, L, P = self.n_heads, self.n_levels, self.n_points

        cs = self.colsum_bias_grad
        value = linear(input_flatten, self.value_proj.weight, self.value_proj.bias, cs)
        if input_padding_mask is not None:
            value = value.masked_fill(input_padding_mask[..., None], float(0))
        value = value.view(N, len_in, M, int(self.ratio * self.d_model) // M)

        # The fused kernels take points [.., 2] and boxes [.., 4] and return a reference-point gradient exactly when
        # autograd asks for one (Deformable-DETR style decoders learn their reference points, ms_deform_attn.py:115-119);
        # the adapter's constant grid gets none and launches nothing extra for it.
        if self.fused and reference_points.dim() == 4 and reference_points.shape[-1] in (2, 4) \
                and _cabi.fused_supported(value, L, P):
            if self.merge_query_linears:
                # sampling_offsets and attention_weights read the same query: ONE GEMM over the concatenated weights
                # (state-dict keys untouched, cached until a parameter changes); the kernels consume its output in place
                if torch.compiler.is_compiling():
                    # the persistent buffers live in the module's __dict__, which compiled code must not write:
                    # a plain cat, which Inductor schedules (and keeps out of the steady state of a CUDA graph)
                    w = torch.cat([self.sampling_offsets.weight, self.attention_weights.weight], 0)
                    b = torch.cat([self.sampling_offsets.bias, self.attention_weights.bias], 0)
                else:
                    w, b = _MergedQueryParams.apply(self.sampling_offsets.weight, self.attention_weights.weight,
                                                    self.sampling_offsets.bias, self.attention_weights.bias, self)
                merged = linear(query, w, b, cs)
                output = MSDeformAttnMergedFunction.apply(value, input_spatial_shapes, input_level_start_index,
                                                          reference_points, merged, L, P)
            else:
                offsets = self.sampling_offsets(query).view(N, Lq, M, L, P, 2)
                logits = self.attention_weights(query).view(N, Lq, M, L * P)
                output = MSDeformAttnFusedFunction.apply(value, input_spatial_shapes, input_level_start_index,
                                                         reference_points, offsets, logits)
            return linear(output, self.output_proj.weight, self.output_proj.bias, cs)

        offsets = self.sampling_offsets(query).view(N, Lq, M, L, P, 2)
        weights = F.softmax(self.attention_weights(query).view(N, Lq, M, L * P), -1).view(N, Lq, M, L, P)

        if reference_points.shape[-1] == 2:
            # (W_l, H_l) per level: offsets are in pixels of their own level
            wh = torch.stack([input_spatial_shapes[..., 1], input_spatial_shapes[..., 0]], -1)
            locations = reference_points[:, :, None, :, None, :] + offsets / wh[None, None, None, :, None, :]
        elif reference_points.shape[-1] == 4:
            locations = reference_points[:, :, None, :, None, :2] \
                + offsets / P * reference_points[:, :, None, :, None, 2:] * 0.5
        else:
            raise ValueError('Last dim of reference_points must be 2 or 4, but get {} instead.'.format(
                reference_points.shape[-1]))
        output = MSDeformAttnFunction.apply(value, input_spatial_shapes, input_level_start_index,
                                            locations, weights, self.im2col_step)
        return linear(output, self.output_proj.weight, self.output_proj.bias, cs)
