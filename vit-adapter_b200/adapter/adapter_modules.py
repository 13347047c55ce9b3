"""Adapter-side callers of MSDeformAttn: deform_inputs, Injector, Extractor, InteractionBlock[WithCls].

Drop-in for the reference's `adapter_modules.py` (three near-identical copies:
detection/mmdet_custom/models/backbones/adapter_modules.py, segmentation/mmseg_custom/... (adds
InteractionBlockWithCls, :194-234, and `with_cp` on SpatialPriorModule), wsdm2023/...). Same class
names, constructor arguments, sub-module names (state_dict keys) and forward signatures, so the
adapter backbones (vit_adapter.py:109-113) can import these instead.

Differences from the reference, all host-side:
  * `deform_inputs` memoises the (reference_points, spatial_shapes, level_start_index) triples per
    (H, W, device): the reference rebuilds them from Python on every forward (adapter_modules.py:28-47),
    which costs ~20 tiny kernel launches and makes the tensors' storage change every step (defeating
    MSDeformAttn's cached shape check and CUDA-graph capture).
  * DropPath is implemented here (timm is not a dependency).

Under torch.compile / torch.export the LayerNorm, residual-add and depth-wise conv kernels are reached through the
msda_b200 custom ops (`_ops.py`). The one compiled-mode difference: the LayerNorm op returns only y, so the pre-norm
residual uses x itself and its gradient is added by the compiled graph instead of inside the LayerNorm backward kernel.
"""
from functools import partial

import torch
import torch.nn as nn
import torch.utils.checkpoint as cp

from .. import _cabi
from ..functions import linear
from ..functions.ms_deform_attn_func import _compiled_ops
from ..modules import MSDeformAttn


class DropPath(nn.Module):
    """Stochastic depth per sample (what timm.models.layers.DropPath does)."""

    def __init__(self, drop_prob=0.):
        super().__init__()
        self.drop_prob = float(drop_prob)

    def forward(self, x):
        if self.drop_prob == 0. or not self.training:
            return x
        keep = 1.0 - self.drop_prob
        mask = x.new_empty((x.shape[0],) + (1,) * (x.dim() - 1)).bernoulli_(keep)
        return x * mask / keep

    def extra_repr(self):
        return 'drop_prob={:.3f}'.format(self.drop_prob)


def get_reference_points(spatial_shapes, device):
    """Cell centres (x, y) in [0,1] of each (H, W) grid, concatenated: [1, sum H*W, 1, 2]
    (reference adapter_modules.py:13-25: linspace(0.5, H-0.5, H) / H)."""
    pts = []
    for (H, W) in spatial_shapes:
        ys = torch.linspace(0.5, H - 0.5, H, dtype=torch.float32, device=device) / H
        xs = torch.linspace(0.5, W - 0.5, W, dtype=torch.float32, device=device) / W
        yy, xx = torch.meshgrid(ys, xs, indexing='ij')
        pts.append(torch.stack((xx.reshape(-1), yy.reshape(-1)), -1)[None])
    return torch.cat(pts, 1)[:, :, None]


def _level_meta(shapes, device):
    spatial_shapes = torch.as_tensor(shapes, dtype=torch.long, device=device)
    level_start_index = torch.cat((spatial_shapes.new_zeros((1,)), spatial_shapes.prod(1).cumsum(0)[:-1]))
    return spatial_shapes, level_start_index


_DEFORM_CACHE = {}


def deform_inputs(x):
    """x: image batch [N, 3, H, W] (only its shape / device are used). Returns
    deform_inputs1 = [ref points of the H/16 grid, shapes of the H/8, H/16, H/32 levels, level starts]  (Injector)
    deform_inputs2 = [ref points of the three levels, shape of the H/16 grid, [0]]                     (Extractor)
    exactly as reference adapter_modules.py:28-47, memoised per (H, W, device). The memoised tensors are built outside
    inference mode (an inference tensor could not be saved for a later training backward) and are READ-ONLY by contract;
    every call returns fresh list containers around them, so a caller that edits its lists cannot disturb another."""
    _, _, h, w = x.shape
    key = (int(h), int(w), str(x.device))
    hit = _DEFORM_CACHE.get(key)
    if hit is not None:
        return list(hit[0]), list(hit[1])
    with torch.inference_mode(False), torch.no_grad():
        return _build_deform_inputs(x, key, h, w)


def _build_deform_inputs(x, key, h, w):
    pyramid = [(h // 8, w // 8), (h // 16, w // 16), (h // 32, w // 32)]
    vit_grid = [(h // 16, w // 16)]
    shapes1, lsi1 = _level_meta(pyramid, x.device)
    ref1 = get_reference_points(vit_grid, x.device)
    shapes2, lsi2 = _level_meta(vit_grid, x.device)
    ref2 = get_reference_points(pyramid, x.device)
    out = ([ref1, shapes1, lsi1], [ref2, shapes2, lsi2])
    if len(_DEFORM_CACHE) > 32:
        _DEFORM_CACHE.clear()
    _DEFORM_CACHE[key] = out
    return list(out[0]), list(out[1])


class _LayerNormRows(torch.autograd.Function):
    """nn.LayerNorm over the last dimension as one row kernel (csrc/adapter_layernorm.cu): x is read once, y is written
    in the consumer's dtype, mean / rstd are kept for a backward that also reads x once."""

    @staticmethod
    def forward(ctx, x, weight, bias, eps, out_dtype, with_residual):
        x = x.contiguous()
        y, stats = _cabi.layernorm_forward(x, weight, bias, eps, out_dtype)
        ctx.save_for_backward(x, weight, stats)
        ctx.has_bias = bias is not None
        ctx.set_materialize_grads(False)
        if with_residual:
            # second output: x itself, for the residual connection around the normalised branch. Its gradient comes
            # back into THIS node, where the backward kernel adds it to dx (one pass instead of LN backward + add).
            return y, x.view_as(x)
        return y

    @staticmethod
    @torch.autograd.function.once_differentiable
    def backward(ctx, grad_y, grad_res=None):
        x, weight, stats = ctx.saved_tensors
        if grad_y is None:   # only the residual output was used
            return grad_res, None, None, None, None, None
        if grad_res is not None and (grad_res.dtype != x.dtype or not grad_res.is_contiguous()):
            grad_res = grad_res.to(x.dtype).contiguous()
        gx, gw, gb = _cabi.layernorm_backward(grad_y.contiguous(), x, weight, stats, grad_res)
        return gx, gw, (gb if ctx.has_bias else None), None, None, None


def _norm_kernel_dtype(norm, x, fused):
    """Output dtype when the row kernel takes this LayerNorm call, else None."""
    if fused and type(norm) is nn.LayerNorm and norm.elementwise_affine and len(norm.normalized_shape) == 1 and x.is_cuda:
        out_dtype = torch.get_autocast_dtype('cuda') if torch.is_autocast_enabled('cuda') else x.dtype
        if _cabi.layernorm_supported(x, norm.weight, norm.bias, out_dtype):
            return out_dtype
    return None


def apply_norm(norm, x, fused=True):
    """`norm(x)` for the LayerNorms in front of the adapter's Linears (reference adapter_modules.py:110-116,142-145).
    A plain affine nn.LayerNorm on CUDA goes through the row kernel and, under bf16 autocast, hands the Linear a bf16
    tensor directly (torch would write fp32 and cast it again); anything else calls the module as the reference does."""
    out_dtype = _norm_kernel_dtype(norm, x, fused)
    if out_dtype is not None:
        if torch.compiler.is_compiling():
            return _compiled_ops().layernorm(x, norm.weight, norm.bias, norm.eps, out_dtype)[0]
        return _LayerNormRows.apply(x, norm.weight, norm.bias, norm.eps, out_dtype, False)
    return norm(x)


def apply_norm_residual(norm, x, fused=True):
    """(norm(x), x') for the pre-norm residual pattern `x + f(norm(x))` (reference adapter_modules.py:113-116, :145):
    use x' (same values as x) for the residual connection. With the row kernel, the gradient of x' is folded into the
    LayerNorm backward kernel instead of a separate full-tensor add by autograd (not in compiled code: see the module
    docstring)."""
    if torch.compiler.is_compiling():
        return apply_norm(norm, x, fused), x
    out_dtype = _norm_kernel_dtype(norm, x, fused)
    if out_dtype is not None and torch.is_grad_enabled() and x.requires_grad:
        return _LayerNormRows.apply(x, norm.weight, norm.bias, norm.eps, out_dtype, True)
    return apply_norm(norm, x, fused), x


class _ResidualAdd(torch.autograd.Function):
    """fp32 stream + bf16 branch in one vectorised pass (csrc/adapter_residual.cu)."""

    @staticmethod
    def forward(ctx, res, branch):
        ctx.branch_dtype = branch.dtype
        return _cabi.residual_add(res, branch)

    @staticmethod
    @torch.autograd.function.once_differentiable
    def backward(ctx, grad):
        return grad, (grad.to(ctx.branch_dtype) if ctx.needs_input_grad[1] else None)


def residual_add(res, branch, fused=True):
    """`res + branch` (reference adapter_modules.py:113-116); the mixed fp32 + bf16 case goes through the kernel."""
    if torch.compiler.is_compiling():
        # the 16-byte alignment of the operands is known only at run time: the op copies a misaligned one
        if fused and res.dtype != branch.dtype and _cabi.residual_add_layout_supported(res, branch):
            return _compiled_ops().residual_add(res, branch)
        return res + branch
    if fused and res.dtype != branch.dtype and _cabi.residual_add_supported(res, branch):
        return _ResidualAdd.apply(res, branch)
    return res + branch


class _DWConvTokens(torch.autograd.Function):
    """Depth-wise 3x3 on the [B, 21n, C] token layout in one kernel (csrc/adapter_dwconv.cu) instead of the
    reference's slice / transpose / conv2d / transpose / cat sequence."""

    @staticmethod
    def forward(ctx, x, weight, bias, H, W):
        x = x.contiguous()
        ctx.save_for_backward(x, weight)
        ctx.hw = (int(H), int(W))
        ctx.has_bias = bias is not None
        return _cabi.dwconv_forward(x, weight.contiguous(), bias.contiguous() if bias is not None else None, int(H), int(W))

    @staticmethod
    @torch.autograd.function.once_differentiable
    def backward(ctx, grad_y):
        x, weight = ctx.saved_tensors
        gx, gw, gb = _cabi.dwconv_backward(x, weight.contiguous(), grad_y.contiguous(), *ctx.hw,
                                           need_input=ctx.needs_input_grad[0],
                                           need_weight=ctx.needs_input_grad[1] or ctx.needs_input_grad[2])
        return gx, gw, (gb if ctx.has_bias else None), None, None


class DWConv(nn.Module):
    """Depth-wise 3x3 over the three token maps packed in one sequence of 21n tokens
    (16n at H/8, 4n at H/16, n at H/32); reference adapter_modules.py:73-87. Same parameter (`dwconv.weight`,
    `dwconv.bias`); on CUDA the token-layout kernel is used, otherwise the reference's op sequence."""

    def __init__(self, dim=768):
        super().__init__()
        self.dwconv = nn.Conv2d(dim, dim, 3, 1, 1, bias=True, groups=dim)
        self.token_kernel = True

    def forward(self, x, H, W):
        w, b = self.dwconv.weight, self.dwconv.bias
        if self.token_kernel and _cabi.dwconv_supported(x, w.to(x.dtype) if w.dtype != x.dtype else w, H, W):
            if w.dtype != x.dtype:  # autocast: activations bf16, parameters fp32
                w, b = w.to(x.dtype), (b.to(x.dtype) if b is not None else None)
            if torch.compiler.is_compiling():
                return _compiled_ops().dwconv(x, w, b, H, W)
            return _DWConvTokens.apply(x, w, b, H, W)
        B, N, C = x.shape
        n = N // 21
        outs = []
        for (lo, hi, h, w) in ((0, 16 * n, H * 2, W * 2), (16 * n, 20 * n, H, W), (20 * n, N, H // 2, W // 2)):
            fmap = x[:, lo:hi, :].transpose(1, 2).reshape(B, C, h, w)
            outs.append(self.dwconv(fmap).flatten(2).transpose(1, 2))
        return torch.cat(outs, dim=1)


class ConvFFN(nn.Module):
    def __init__(self, in_features, hidden_features=None, out_features=None, act_layer=nn.GELU, drop=0.):
        super().__init__()
        out_features = out_features or in_features
        hidden_features = hidden_features or in_features
        self.fc1 = nn.Linear(in_features, hidden_features)
        self.dwconv = DWConv(hidden_features)
        self.act = act_layer()
        self.fc2 = nn.Linear(hidden_features, out_features)
        self.drop = nn.Dropout(drop)
        self.colsum_bias_grad = True   # bias gradients of fc1 / fc2 through the column-sum kernel (functions/linear.py)

    def forward(self, x, H, W):
        cs = self.colsum_bias_grad
        x = self.drop(self.act(self.dwconv(linear(x, self.fc1.weight, self.fc1.bias, cs), H, W)))
        return self.drop(linear(x, self.fc2.weight, self.fc2.bias, cs))


class Extractor(nn.Module):
    """c <- c + MSDeformAttn(LN(c), ref, LN(x)) ; c <- c + DropPath(ConvFFN(LN(c)))   (reference :90-124)."""

    def __init__(self, dim, num_heads=6, n_points=4, n_levels=1, deform_ratio=1.0, with_cffn=True, cffn_ratio=0.25,
                 drop=0., drop_path=0., norm_layer=partial(nn.LayerNorm, eps=1e-6), with_cp=False):
        super().__init__()
        self.query_norm = norm_layer(dim)
        self.feat_norm = norm_layer(dim)
        self.attn = MSDeformAttn(d_model=dim, n_levels=n_levels, n_heads=num_heads, n_points=n_points,
                                 ratio=deform_ratio)
        self.with_cffn = with_cffn
        self.with_cp = with_cp
        self.fused_norm = True   # LayerNorms through the row kernel (apply_norm); False = torch's, as the reference
        if with_cffn:
            self.ffn = ConvFFN(in_features=dim, hidden_features=int(dim * cffn_ratio), drop=drop)
            self.ffn_norm = norm_layer(dim)
            self.drop_path = DropPath(drop_path) if drop_path > 0. else nn.Identity()

    def forward(self, query, reference_points, feat, spatial_shapes, level_start_index, H, W):
        def inner(query, feat):
            fn = self.fused_norm
            normed, query = apply_norm_residual(self.query_norm, query, fn)
            query = residual_add(query, self.attn(normed, reference_points, apply_norm(self.feat_norm, feat, fn),
                                                  spatial_shapes, level_start_index, None), fn)
            if self.with_cffn:
                normed, query = apply_norm_residual(self.ffn_norm, query, fn)
                query = residual_add(query, self.drop_path(self.ffn(normed, H, W)), fn)
            return query

        if self.with_cp and query.requires_grad:
            return cp.checkpoint(inner, query, feat, use_reentrant=True)
        return inner(query, feat)


class Injector(nn.Module):
    """x <- x + gamma * MSDeformAttn(LN(x), ref, LN(c))   (reference :127-152; gamma starts at init_values)."""

    def __init__(self, dim, num_heads=6, n_points=4, n_levels=1, deform_ratio=1.0,
                 norm_layer=partial(nn.LayerNorm, eps=1e-6), init_values=0., with_cp=False):
        super().__init__()
        self.with_cp = with_cp
        self.query_norm = norm_layer(dim)
        self.feat_norm = norm_layer(dim)
        self.attn = MSDeformAttn(d_model=dim, n_levels=n_levels, n_heads=num_heads, n_points=n_points,
                                 ratio=deform_ratio)
        self.gamma = nn.Parameter(init_values * torch.ones((dim)), requires_grad=True)
        self.fused_norm = True

    def forward(self, query, reference_points, feat, spatial_shapes, level_start_index, return_feat=False):
        """Same as the reference; with return_feat=True also returns `feat` as handed out by its LayerNorm node
        (same values): a caller that goes on using feat (InteractionBlock feeds c to the Extractor next) should use
        that one, so the gradient of the later use is added inside the LayerNorm backward kernel."""
        def inner(query, feat):
            fn = self.fused_norm
            normed, query = apply_norm_residual(self.query_norm, query, fn)
            if return_feat:
                normed_feat, feat = apply_norm_residual(self.feat_norm, feat, fn)
            else:
                normed_feat = apply_norm(self.feat_norm, feat, fn)
            attn = self.attn(normed, reference_points, normed_feat, spatial_shapes, level_start_index, None)
            out = query + self.gamma * attn
            return (out, feat) if return_feat else out

        if self.with_cp and query.requires_grad:
            return cp.checkpoint(inner, query, feat, use_reentrant=True)
        return inner(query, feat)


class _InteractionBase(nn.Module):
    def __init__(self, dim, num_heads=6, n_points=4, norm_layer=partial(nn.LayerNorm, eps=1e-6), drop=0., drop_path=0.,
                 with_cffn=True, cffn_ratio=0.25, init_values=0., deform_ratio=1.0, extra_extractor=False,
                 with_cp=False):
        super().__init__()
        self.injector = Injector(dim=dim, n_levels=3, num_heads=num_heads, init_values=init_values, n_points=n_points,
                                 norm_layer=norm_layer, deform_ratio=deform_ratio, with_cp=with_cp)
        ext = dict(dim=dim, num_heads=num_heads, n_points=n_points, norm_layer=norm_layer, deform_ratio=deform_ratio,
                   with_cffn=with_cffn, cffn_ratio=cffn_ratio, drop=drop, drop_path=drop_path, with_cp=with_cp)
        self.extractor = Extractor(n_levels=1, **ext)
        self.extra_extractors = nn.Sequential(*[Extractor(**ext) for _ in range(2)]) if extra_extractor else None

    def _inject(self, x, c, deform_inputs1):
        """(x after injection, c to keep using): c comes back through the injector's feat_norm node (see Injector.forward)."""
        return self.injector(query=x, reference_points=deform_inputs1[0], feat=c, spatial_shapes=deform_inputs1[1],
                             level_start_index=deform_inputs1[2], return_feat=True)

    def _extract(self, x, c, deform_inputs2, H, W):
        extractors = [self.extractor] + (list(self.extra_extractors) if self.extra_extractors is not None else [])
        for e in extractors:
            c = e(query=c, reference_points=deform_inputs2[0], feat=x, spatial_shapes=deform_inputs2[1],
                  level_start_index=deform_inputs2[2], H=H, W=W)
        return c


class InteractionBlock(_InteractionBase):
    """Injector -> the slice of ViT blocks -> Extractor (+2 extra extractors on the last block);
    reference adapter_modules.py:155-191."""

    def forward(self, x, c, blocks, deform_inputs1, deform_inputs2, H, W):
        x, c = self._inject(x, c, deform_inputs1)
        for blk in blocks:
            x = blk(x, H, W)
        return x, self._extract(x, c, deform_inputs2, H, W)


class InteractionBlockWithCls(_InteractionBase):
    """Same, with BEiT's class token re-attached around the ViT blocks (segmentation copy :194-234)."""

    def forward(self, x, c, cls, blocks, deform_inputs1, deform_inputs2, H, W):
        x, c = self._inject(x, c, deform_inputs1)
        x = torch.cat((cls, x), dim=1)
        for blk in blocks:
            x = blk(x, H, W)
        cls, x = x[:, :1, ], x[:, 1:, ]
        return x, self._extract(x, c, deform_inputs2, H, W), cls


class InteractionBlockWithText(_InteractionBase):
    """The wsdm2023 grounding variant: the ViT blocks also carry text tokens `q` (with their mask) next to the image tokens
    (wsdm2023/mmdet_custom/models/backbones/adapter_modules.py:161-198, where the class is again called InteractionBlock).
    Same sub-modules and state-dict keys; returns (x, c, q)."""

    def forward(self, x, c, q, q_mask, blocks, deform_inputs1, deform_inputs2, H, W):
        x, c = self._inject(x, c, deform_inputs1)
        for blk in blocks:
            x, q = blk(x, q, q_mask, H, W)
        return x, self._extract(x, c, deform_inputs2, H, W), q


class SpatialPriorModule(nn.Module):
    """Convolutional stem producing the 1/4 map and the 1/8, 1/16, 1/32 token sequences the Injector
    reads (reference :194-246). `norm_layer` defaults to nn.SyncBatchNorm as in the reference."""

    def __init__(self, inplanes=64, embed_dim=384, with_cp=False, norm_layer=nn.SyncBatchNorm):
        super().__init__()
        self.with_cp = with_cp

        def conv_bn_relu(cin, cout, stride):
            return [nn.Conv2d(cin, cout, kernel_size=3, stride=stride, padding=1, bias=False), norm_layer(cout),
                    nn.ReLU(inplace=True)]

        self.stem = nn.Sequential(*(conv_bn_relu(3, inplanes, 2) + conv_bn_relu(inplanes, inplanes, 1)
                                    + conv_bn_relu(inplanes, inplanes, 1)
                                    + [nn.MaxPool2d(kernel_size=3, stride=2, padding=1)]))
        self.conv2 = nn.Sequential(*conv_bn_relu(inplanes, 2 * inplanes, 2))
        self.conv3 = nn.Sequential(*conv_bn_relu(2 * inplanes, 4 * inplanes, 2))
        self.conv4 = nn.Sequential(*conv_bn_relu(4 * inplanes, 4 * inplanes, 2))
        self.fc1 = nn.Conv2d(inplanes, embed_dim, kernel_size=1, stride=1, padding=0, bias=True)
        self.fc2 = nn.Conv2d(2 * inplanes, embed_dim, kernel_size=1, stride=1, padding=0, bias=True)
        self.fc3 = nn.Conv2d(4 * inplanes, embed_dim, kernel_size=1, stride=1, padding=0, bias=True)
        self.fc4 = nn.Conv2d(4 * inplanes, embed_dim, kernel_size=1, stride=1, padding=0, bias=True)

    def forward(self, x):
        def inner(x):
            c1 = self.stem(x)
            c2 = self.conv2(c1)
            c3 = self.conv3(c2)
            c4 = self.conv4(c3)
            c1, c2, c3, c4 = self.fc1(c1), self.fc2(c2), self.fc3(c3), self.fc4(c4)
            bs, dim = c1.shape[:2]
            tokens = [c.view(bs, dim, -1).transpose(1, 2) for c in (c2, c3, c4)]  # 8s, 16s, 32s
            return (c1, *tokens)

        if self.with_cp and x.requires_grad:
            return cp.checkpoint(inner, x, use_reentrant=True)
        return inner(x)
