"""torch.compile / torch.export on the B200: the msda_b200 custom ops (opcheck), compiled modules against eager, a
reduce-overhead training step, an exported module, and the eager path left exactly as it was.

Bars: fp32 1e-5 forward / 1e-4 gradients, bf16 1e-2, fp16 2e-3 (relative to the largest magnitude of the eager result).
The sampling kernels' forward outputs and the fused reference-point gradient are deterministic, so compiled and eager must
agree bitwise there; grad_value is accumulated with atomics and gets the tolerance.

This module imports `vit_adapter_b200._ops` only inside tests: `_eager_launches` also runs in a fresh interpreter in which
the ops are never registered."""
import os
import subprocess
import sys

import pytest
import torch
from torch import nn

import vit_adapter_b200 as vab
from vit_adapter_b200 import _cabi
from vit_adapter_b200.adapter import Extractor, Injector, InteractionBlock, InteractionBlockWithCls, deform_inputs
from vit_adapter_b200.functions import MSDeformAttnFunction, MSDeformAttnFusedFunction, MSDeformAttnMergedFunction
from vit_adapter_b200.mmcv_compat import MultiScaleDeformableAttention
from vit_adapter_b200.modules import MSDeformAttn

F32, BF16, F16, F64 = torch.float32, torch.bfloat16, torch.float16, torch.float64
TOL = {F32: (1e-5, 1e-4), F64: (1e-5, 1e-4), BF16: (1e-2, 1e-2), F16: (2e-3, 2e-3)}   # (forward, gradients)
SHAPES = [(16, 16), (8, 8), (4, 4)]
N, M, D, Lq, P = 2, 4, 32, 96, 4
L = len(SHAPES)


def _ops():
    from vit_adapter_b200 import _ops as ops  # noqa: F401
    return torch.ops.msda_b200


def _close(got, want, tol, what=''):
    got, want = got.detach().float(), want.detach().float()
    scale = max(float(want.abs().max()), 1e-6)
    torch.testing.assert_close(got, want, rtol=tol, atol=tol * scale, msg=lambda m: '%s: %s' % (what, m))


def _close_norm(got, want, tol, what=''):
    """Relative L2 error. Gradients of whole bf16-autocast blocks: a last-bit difference upstream (Inductor fuses f32
    arithmetic that eager rounds op by op) can move a sample across a texel edge, where the bilinear location gradient
    jumps; elementwise bars would flag those few elements, the norm bounds the gradient as a whole."""
    got, want = got.detach().double(), want.detach().double()
    err = float((got - want).norm() / want.norm().clamp_min(1e-12))
    assert err <= tol, '%s: relative L2 error %.3g > %g' % (what, err, tol)


def _levels(dev='cuda'):
    shapes = torch.as_tensor(SHAPES, dtype=torch.long, device=dev)
    lsi = torch.cat((shapes.new_zeros((1,)), shapes.prod(1).cumsum(0)[:-1]))
    return shapes, lsi, sum(h * w for h, w in SHAPES)


def _ref(ref_dim, ref_grad, g, dev='cuda'):
    if ref_dim == 2:
        ref = torch.rand(N if ref_grad else 1, Lq, 1, 2, generator=g) * 0.9 + 0.05
    else:
        xy = torch.rand(N, Lq, L, 2, generator=g) * 0.8 + 0.1
        ref = torch.cat([xy, torch.rand(N, Lq, L, 2, generator=g) * 0.3 + 0.05], -1)
    return ref.to(dev).requires_grad_(ref_grad)


# --- opcheck on every op ------------------------------------------------------------------------------------------------
def _op_cases():
    cases = []
    for dt in (F32, BF16, F16, F64):
        cases.append(('plain', dt, 2, False))
    for dt in (F32, BF16, F16):
        for ref_dim in (2, 4):
            for ref_grad in (False, True):
                cases.append(('fused', dt, ref_dim, ref_grad))
                cases.append(('merged', dt, ref_dim, ref_grad))
    return cases


@pytest.mark.gpu
@pytest.mark.parametrize('kind,dtype,ref_dim,ref_grad', _op_cases(),
                         ids=['%s-%s-%s-%s' % (k, str(d)[6:], 'points' if r == 2 else 'boxes', 'ref_grad' if g else 'const')
                              for k, d, r, g in _op_cases()])
def test_opcheck_msda(kind, dtype, ref_dim, ref_grad):
    ops = _ops()
    g = torch.Generator().manual_seed(3)
    shapes, lsi, S = _levels()
    cdt = F64 if dtype == F64 else F32
    tol = TOL[dtype][1]
    value = torch.randn(N, S, M, D, generator=g).to('cuda', dtype).requires_grad_()
    go = torch.randn(N, Lq, M * D, generator=g).to('cuda', dtype)
    if kind == 'plain':
        loc = (torch.rand(N, Lq, M, L, P, 2, generator=g) * 1.1 - 0.05).to('cuda', cdt).requires_grad_()
        aw = torch.softmax(torch.randn(N, Lq, M, L * P, generator=g), -1).view(N, Lq, M, L, P).to('cuda', cdt).requires_grad_()
        torch.library.opcheck(ops.ms_deform_attn, (value, shapes, lsi, loc, aw, 64), atol=tol, rtol=tol)
        torch.library.opcheck(ops.ms_deform_attn_backward, (value.detach(), shapes, lsi, loc.detach(), aw.detach(), go, 64),
                              atol=tol, rtol=tol)
        return
    ref = _ref(ref_dim, ref_grad, g)
    if kind == 'fused':
        off = (torch.randn(N, Lq, M, L, P, 2, generator=g) * 2).cuda().requires_grad_()
        logits = torch.randn(N, Lq, M, L * P, generator=g).cuda().requires_grad_()
        torch.library.opcheck(ops.ms_deform_attn_fused, (value, shapes, lsi, ref, off, logits), atol=tol, rtol=tol)
        torch.library.opcheck(ops.ms_deform_attn_fused_backward,
                              (value.detach(), shapes, lsi, ref.detach(), off.detach(), logits.detach(), go, ref_grad),
                              atol=tol, rtol=tol)
    else:
        merged = torch.randn(N, Lq, M * L * P * 3, generator=g).cuda().requires_grad_()
        torch.library.opcheck(ops.ms_deform_attn_merged, (value, shapes, lsi, ref, merged, L, P), atol=tol, rtol=tol)
        torch.library.opcheck(ops.ms_deform_attn_merged_backward,
                              (value.detach(), shapes, lsi, ref.detach(), merged.detach(), L, P, go, ref_grad),
                              atol=tol, rtol=tol)


@pytest.mark.gpu
@pytest.mark.parametrize('xdt,ydt', [(F32, F32), (F32, BF16), (BF16, BF16), (F32, F16), (F16, F16)],
                         ids=lambda d: str(d)[6:])
def test_opcheck_layernorm(xdt, ydt):
    ops = _ops()
    g = torch.Generator().manual_seed(4)
    C = 96
    x = torch.randn(N, 50, C, generator=g).to('cuda', xdt).requires_grad_()
    w = (1 + 0.1 * torch.randn(C, generator=g)).cuda().requires_grad_()
    b = (0.1 * torch.randn(C, generator=g)).cuda().requires_grad_()
    tol = TOL[ydt][1]
    torch.library.opcheck(ops.layernorm, (x, w, b, 1e-6, ydt), atol=tol, rtol=tol)
    torch.library.opcheck(ops.layernorm, (x, w, None, 1e-6, ydt), atol=tol, rtol=tol)
    y, stats = ops.layernorm(x.detach(), w.detach(), b.detach(), 1e-6, ydt)
    gy = torch.randn(y.shape, generator=g).to('cuda', ydt)
    torch.library.opcheck(ops.layernorm_backward, (gy, x.detach(), w.detach(), stats), atol=tol, rtol=tol)


@pytest.mark.gpu
@pytest.mark.parametrize('dtype', [F32, BF16, F16], ids=lambda d: str(d)[6:])
def test_opcheck_dwconv_residual_colsum(dtype):
    ops = _ops()
    g = torch.Generator().manual_seed(5)
    H = W = 8
    C = 48
    n = 21 * (H // 2) * (W // 2)
    tol = TOL[dtype][1]
    x = torch.randn(N, n, C, generator=g).to('cuda', dtype).requires_grad_()
    w = (0.3 * torch.randn(C, 1, 3, 3, generator=g)).to('cuda', dtype).requires_grad_()
    b = (0.1 * torch.randn(C, generator=g)).to('cuda', dtype).requires_grad_()
    torch.library.opcheck(ops.dwconv, (x, w, b, H, W), atol=tol, rtol=tol)
    gy = torch.randn(N, n, C, generator=g).to('cuda', dtype)
    for need_input, need_weight in ((True, True), (True, False), (False, True)):
        torch.library.opcheck(ops.dwconv_backward, (x.detach(), w.detach(), gy, H, W, need_input, need_weight),
                              atol=tol, rtol=tol)
    res = torch.randn(N, n, C, generator=g).cuda().requires_grad_()
    torch.library.opcheck(ops.residual_add, (res, x), atol=tol, rtol=tol)
    torch.library.opcheck(ops.colsum, (gy,), atol=tol, rtol=tol)


# --- compiled Functions: bitwise forward and reference-point gradient ----------------------------------------------------
def _function_inputs(kind, dtype, ref_dim, ref_grad, seed=7):
    g = torch.Generator().manual_seed(seed)
    shapes, lsi, S = _levels()
    value = torch.randn(N, S, M, D, generator=g).to('cuda', dtype).requires_grad_()
    go = torch.randn(N, Lq, M * D, generator=g).to('cuda', dtype)
    if kind == 'plain':
        cdt = F64 if dtype == F64 else F32
        loc = (torch.rand(N, Lq, M, L, P, 2, generator=g) * 1.1 - 0.05).to('cuda', cdt).requires_grad_()
        aw = torch.softmax(torch.randn(N, Lq, M, L * P, generator=g), -1).view(N, Lq, M, L, P).to('cuda', cdt).requires_grad_()
        return (lambda v, l, a: MSDeformAttnFunction.apply(v, shapes, lsi, l, a, 64)), [value, loc, aw], go
    ref = _ref(ref_dim, ref_grad, g)
    if kind == 'fused':
        off = (torch.randn(N, Lq, M, L, P, 2, generator=g) * 2).cuda().requires_grad_()
        logits = torch.randn(N, Lq, M, L * P, generator=g).cuda().requires_grad_()
        return ((lambda v, r, o, lg: MSDeformAttnFusedFunction.apply(v, shapes, lsi, r, o, lg)),
                [value, ref, off, logits], go)
    merged = torch.randn(N, Lq, M * L * P * 3, generator=g).cuda().requires_grad_()
    return (lambda v, r, m: MSDeformAttnMergedFunction.apply(v, shapes, lsi, r, m, L, P)), [value, ref, merged], go


def _run(fn, leaves, go):
    for t in leaves:
        t.grad = None
    out = fn(*leaves)
    out.backward(go)
    return out.detach(), [t.grad for t in leaves]


_FN_CASES = ([('plain', dt, 2, False) for dt in (F32, BF16, F64)]
             + [(k, dt, r, gr) for k in ('fused', 'merged') for dt in (F32, BF16, F16) for r, gr in ((2, False), (4, True))]
             + [(k, F32, r, gr) for k in ('fused', 'merged') for r, gr in ((2, True), (4, False))])


@pytest.mark.gpu
@pytest.mark.parametrize('kind,dtype,ref_dim,ref_grad', _FN_CASES,
                         ids=['%s-%s-%s-%s' % (k, str(d)[6:], 'points' if r == 2 else 'boxes', 'ref_grad' if g else 'const')
                              for k, d, r, g in _FN_CASES])
def test_compiled_function_matches_eager(kind, dtype, ref_dim, ref_grad):
    torch._dynamo.reset()
    if dtype == F16:
        vab.set_amp_value_dtype(F16)   # otherwise fp16 values run on the fp32 kernels (the reference's policy)
    try:
        fn, leaves, go = _function_inputs(kind, dtype, ref_dim, ref_grad)
        out_e, grads_e = _run(fn, leaves, go)
        out_c, grads_c = _run(torch.compile(fn, fullgraph=True), leaves, go)
    finally:
        vab.set_amp_value_dtype(F32)
    assert out_c.dtype == out_e.dtype and torch.equal(out_c, out_e)
    tol = TOL[dtype][1]
    _close(grads_c[0], grads_e[0], tol, 'grad_value')
    for i, (gc, ge) in enumerate(zip(grads_c[1:], grads_e[1:]), 1):
        if ge is None:
            assert gc is None
        elif kind != 'plain' and i == 1:
            assert torch.equal(gc, ge), 'reference-point gradient'
        else:
            _close(gc, ge, tol, 'grad %d' % i)


# --- compiled modules against eager ---------------------------------------------------------------------------------------
def _clone_module(make):
    torch.manual_seed(11)
    a = make().cuda()
    torch.manual_seed(11)
    b = make().cuda()
    b.load_state_dict(a.state_dict())
    return a, b


def _compare_module(make, inputs, call, dtype=F32, autocast=False):
    """compiled (fullgraph) vs eager: outputs, input gradients and parameter gradients."""
    torch._dynamo.reset()
    mod_e, mod_c = _clone_module(make)
    tol_f, tol_b = TOL[dtype]
    compiled = torch.compile(lambda *a: call(mod_c, *a), fullgraph=True)
    results = []
    for mod, fn in ((mod_e, lambda *a: call(mod_e, *a)), (mod_c, compiled)):
        leaves = [t.detach().clone().requires_grad_(t.requires_grad) for t in inputs]
        with torch.autocast('cuda', dtype=BF16, enabled=autocast):
            outs = fn(*leaves)
        outs = outs if isinstance(outs, tuple) else (outs,)
        loss = sum((o.float() * torch.linspace(-1, 1, o.numel(), device='cuda').view(o.shape)).sum() for o in outs)
        loss.backward()
        results.append(([o.detach() for o in outs], [t.grad for t in leaves if t.requires_grad],
                        {k: p.grad for k, p in mod.named_parameters() if p.grad is not None}))
    assert torch._dynamo.utils.counters['stats']['unique_graphs'] >= 1   # compiled, not an eager fallback
    (outs_e, gin_e, gp_e), (outs_c, gin_c, gp_c) = results
    for i, (oc, oe) in enumerate(zip(outs_c, outs_e)):
        assert oc.dtype == oe.dtype
        _close(oc, oe, tol_f, 'output %d' % i)
    assert gp_c.keys() == gp_e.keys()
    if autocast:
        # bf16: a bias / LayerNorm-affine gradient is a column sum of thousands of bf16-rounded rows whose rounding does not
        # cancel, so the parameter gradients are compared as one vector
        for i, (gc, ge) in enumerate(zip(gin_c, gin_e)):
            _close_norm(gc, ge, tol_b, 'input grad %d' % i)
        _close_norm(torch.cat([gp_c[k].flatten().float() for k in gp_e]), torch.cat([gp_e[k].flatten().float() for k in gp_e]),
                    tol_b, 'parameter gradients')
        return
    for i, (gc, ge) in enumerate(zip(gin_c, gin_e)):
        _close(gc, ge, tol_b, 'input grad %d' % i)
    for k in gp_e:
        _close(gp_c[k], gp_e[k], tol_b, k)


@pytest.mark.gpu
@pytest.mark.parametrize('ref_dim,ref_grad', [(2, False), (4, False), (2, True), (4, True)],
                         ids=['points-const', 'boxes-const', 'points-ref_grad', 'boxes-ref_grad'])
@pytest.mark.parametrize('path', ['merged', 'fused', 'unfused'])
def test_compiled_msdeformattn_matches_eager(path, ref_dim, ref_grad):
    shapes, lsi, S = _levels()
    g = torch.Generator().manual_seed(8)
    q = torch.randn(N, Lq, 128, generator=g).cuda().requires_grad_()
    feat = torch.randn(N, S, 128, generator=g).cuda().requires_grad_()
    ref = _ref(ref_dim, ref_grad, g)

    def make():
        m = MSDeformAttn(128, L, M, P)
        m.fused, m.merge_query_linears = path != 'unfused', path == 'merged'
        with torch.no_grad():
            for p in m.parameters():
                p.add_(0.05 * torch.randn_like(p))
        return m
    _compare_module(make, [q, ref, feat], lambda m, q, r, f: m(q, r, f, shapes, lsi))


@pytest.mark.gpu
def test_compiled_mmcv_shim_matches_eager():
    shapes, lsi, S = _levels()
    g = torch.Generator().manual_seed(9)
    q = torch.randn(Lq, N, 128, generator=g).cuda().requires_grad_()
    v = torch.randn(S, N, 128, generator=g).cuda().requires_grad_()
    ref = _ref(4, False, g)
    _compare_module(lambda: MultiScaleDeformableAttention(128, M, L, P, dropout=0.0), [q, v],
                    lambda m, q, v: m(q, value=v, reference_points=ref, spatial_shapes=shapes, level_start_index=lsi))


class _TinyViTBlock(nn.Module):
    def __init__(self, dim):
        super().__init__()
        self.norm = nn.LayerNorm(dim, eps=1e-6)
        self.fc = nn.Linear(dim, dim)

    def forward(self, x, H, W):
        return x + self.fc(self.norm(x))


def _block_data(side, dim=128, seed=10):
    h = side // 16
    g = torch.Generator().manual_seed(seed)
    di1, di2 = deform_inputs(torch.zeros(N, 3, side, side, device='cuda'))
    x = torch.randn(N, h * h, dim, generator=g).cuda().requires_grad_()
    c = torch.randn(N, 21 * (h // 2) ** 2, dim, generator=g).cuda().requires_grad_()
    return x, c, di1, di2, h


def _make_block(cls=InteractionBlock, dim=128):
    def make():
        blk = cls(dim, 2, 4, deform_ratio=0.5, init_values=0.3, extra_extractor=True)
        blk.vit = nn.ModuleList([_TinyViTBlock(dim)])
        with torch.no_grad():
            for p in blk.parameters():
                p.add_(0.02 * torch.randn_like(p))
        return blk
    return make


@pytest.mark.gpu
@pytest.mark.parametrize('which', ['injector', 'extractor', 'interaction', 'interaction_cls'])
def test_compiled_adapter_modules_match_eager(which):
    x, c, di1, di2, h = _block_data(128)
    if which == 'injector':
        _compare_module(lambda: Injector(128, 2, 4, n_levels=3, deform_ratio=0.5, init_values=0.3), [x, c],
                        lambda m, x, c: m(x, di1[0], c, di1[1], di1[2]))
    elif which == 'extractor':
        _compare_module(lambda: Extractor(128, 2, 4, n_levels=1, deform_ratio=0.5), [x, c],
                        lambda m, x, c: m(c, di2[0], x, di2[1], di2[2], h, h))
    elif which == 'interaction':
        _compare_module(_make_block(), [x, c], lambda m, x, c: m(x, c, m.vit, di1, di2, h, h))
    else:
        cls = torch.randn(N, 1, 128, device='cuda', requires_grad=True)
        _compare_module(_make_block(InteractionBlockWithCls), [x, c, cls],
                        lambda m, x, c, cls: m(x, c, cls, m.vit, di1, di2, h, h))


@pytest.mark.gpu
@pytest.mark.parametrize('value_dtype', [F32, BF16], ids=['amp_value_f32', 'amp_value_bf16'])
def test_compiled_interaction_block_bf16_autocast(value_dtype):
    x, c, di1, di2, h = _block_data(128)
    vab.set_amp_value_dtype(value_dtype)
    try:
        # the AMP value policy is traced: the compiled op runs on values of the chosen dtype
        torch._dynamo.reset()
        fn, leaves, _ = _function_inputs('merged', F32, 2, False)
        with torch.autocast('cuda', dtype=BF16):
            assert torch.compile(fn, fullgraph=True)(*leaves).dtype == value_dtype
        _compare_module(_make_block(), [x, c], lambda m, x, c: m(x, c, m.vit, di1, di2, h, h), dtype=BF16, autocast=True)
    finally:
        vab.set_amp_value_dtype(F32)


@pytest.mark.gpu
def test_compiled_with_checkpointing_matches_eager():
    """with_cp=True: reentrant checkpointing keeps its graph break (no fullgraph), and still computes the eager result."""
    torch._dynamo.reset()
    x, c, di1, di2, h = _block_data(128)

    def make():
        blk = InteractionBlock(128, 2, 4, deform_ratio=0.5, init_values=0.3, extra_extractor=True, with_cp=True)
        with torch.no_grad():
            for p in blk.parameters():
                p.add_(0.02 * torch.randn_like(p))
        return blk
    mod_e, mod_c = _clone_module(make)
    compiled = torch.compile(lambda x, c: mod_c(x, c, [], di1, di2, h, h))
    grads = []
    for fn, mod in ((lambda x, c: mod_e(x, c, [], di1, di2, h, h), mod_e), (compiled, mod_c)):
        xl, cl = x.detach().clone().requires_grad_(), c.detach().clone().requires_grad_()
        xo, co = fn(xl, cl)
        (xo.square().mean() + co.square().mean()).backward()
        grads.append([xo.detach(), co.detach(), xl.grad, cl.grad] + [p.grad for p in mod.parameters()])
    for i, (gc, ge) in enumerate(zip(*grads)):
        _close(gc, ge, TOL[F32][1], 'tensor %d' % i)


@pytest.mark.gpu
def test_compiled_two_resolutions():
    """A second input resolution may recompile; both results must match eager."""
    torch._dynamo.reset()
    mod_e, mod_c = _clone_module(_make_block())
    compiled = torch.compile(lambda x, c, di1, di2, h: mod_c(x, c, mod_c.vit, di1, di2, h, h), fullgraph=True)
    for side in (128, 192):
        x, c, di1, di2, h = _block_data(side, seed=side)
        with torch.no_grad():
            xe, ce = mod_e(x, c, mod_e.vit, di1, di2, h, h)
            xc, cc = compiled(x, c, di1, di2, h)
        _close(xc, xe, TOL[F32][0], 'x at %d' % side)
        _close(cc, ce, TOL[F32][0], 'c at %d' % side)


# --- reduce-overhead training step ----------------------------------------------------------------------------------------
@pytest.mark.gpu
def test_reduce_overhead_training_step():
    torch._dynamo.reset()
    x, c, di1, di2, h = _block_data(128)
    x, c = x.detach(), c.detach()
    mod_e, mod_c = _clone_module(_make_block())

    def make_step(mod, fwd):
        opt = torch.optim.AdamW(mod.parameters(), lr=1e-3, capturable=True, foreach=True)

        def step():
            torch.compiler.cudagraph_mark_step_begin()
            xo, co = fwd(x, c)
            loss = xo.square().mean() + co.square().mean()
            opt.zero_grad(set_to_none=False)
            loss.backward()
            opt.step()
            return loss.detach().clone()
        return step

    eager = make_step(mod_e, lambda x, c: mod_e(x, c, mod_e.vit, di1, di2, h, h))
    compiled = make_step(mod_c, torch.compile(lambda x, c: mod_c(x, c, mod_c.vit, di1, di2, h, h), mode='reduce-overhead',
                                              fullgraph=True))
    for p in list(mod_e.parameters()) + list(mod_c.parameters()):
        p.grad = torch.zeros_like(p)
    losses_e = [float(eager()) for _ in range(4)]
    losses_c = [float(compiled()) for _ in range(3)]    # warm-up, record, replay
    for le, lc in zip(losses_e, losses_c):
        assert abs(lc - le) <= 2e-4 * abs(le), (losses_c, losses_e)
    torch.cuda.synchronize()
    torch.cuda.set_sync_debug_mode('error')
    try:
        loss = compiled()
    finally:
        torch.cuda.set_sync_debug_mode(0)
    assert abs(float(loss) - losses_e[3]) <= 2e-4 * abs(losses_e[3])
    assert losses_c[2] < losses_c[0]


# --- torch.export ---------------------------------------------------------------------------------------------------------
@pytest.mark.gpu
def test_export_module_matches_eager_bitwise():
    x, c, di1, di2, h = _block_data(128)
    torch.manual_seed(12)
    blk = _make_block()().cuda().eval()
    with torch.no_grad():
        want = blk(x, c, [], di1, di2, h, h)
    ep = torch.export.export(blk, (x.detach(), c.detach(), [], di1, di2, h, h))
    targets = {str(n.target) for n in ep.graph.nodes if n.op == 'call_function'}
    assert {'msda_b200.ms_deform_attn_merged.default', 'msda_b200.layernorm.default', 'msda_b200.dwconv.default'} <= targets
    with torch.no_grad():
        got = ep.module()(x, c, [], di1, di2, h, h)
    for gt, wt in zip(got, want):
        assert torch.equal(gt, wt)
    attn = MSDeformAttn(128, L, M, P).cuda()
    shapes, lsi, S = _levels()
    q, feat = torch.randn(N, Lq, 128, device='cuda'), torch.randn(N, S, 128, device='cuda')
    ref = torch.rand(1, Lq, 1, 2, device='cuda')
    with torch.no_grad():
        want = attn(q, ref, feat, shapes, lsi)
        got = torch.export.export(attn, (q, ref, feat, shapes, lsi)).module()(q, ref, feat, shapes, lsi)
    assert torch.equal(got, want)


# --- the eager path is untouched ------------------------------------------------------------------------------------------
def _eager_launches():
    """Library launches of one eager InteractionBlock forward + backward (also run in a fresh interpreter)."""
    x, c, di1, di2, h = _block_data(128)
    torch.manual_seed(13)
    blk = _make_block()().cuda()
    n0 = _cabi.launch_count()
    xo, co = blk(x, c, blk.vit, di1, di2, h, h)
    (xo.square().mean() + co.square().mean()).backward()
    torch.cuda.synchronize()
    return _cabi.launch_count() - n0


@pytest.mark.gpu
def test_eager_dispatches_no_custom_op():
    """An eager forward + backward dispatches nothing through torch.ops.msda_b200, and launches as many library kernels with
    the ops registered as in an interpreter that never imported them."""
    from torch.utils._python_dispatch import TorchDispatchMode
    _ops()   # registered, so that a dispatch through torch.ops.msda_b200 would be seen

    class Record(TorchDispatchMode):
        def __init__(self):
            super().__init__()
            self.names = set()

        def __torch_dispatch__(self, func, types, args=(), kwargs=None):
            self.names.add(func.namespace)
            return func(*args, **(kwargs or {}))

    _eager_launches()   # warm (deform_inputs and shape-check memos)
    rec = Record()
    with rec:
        launches = _eager_launches()
    assert 'aten' in rec.names and 'msda_b200' not in rec.names, rec.names
    here = os.path.dirname(os.path.abspath(__file__))
    code = ('import sys; sys.path[:0] = [%r, %r]; import test_compile_gpu as t; t._eager_launches(); n = t._eager_launches(); '
            'assert "vit_adapter_b200._ops" not in sys.modules; print(n)' % (os.path.dirname(here), here))
    fresh = subprocess.run([sys.executable, '-c', code], capture_output=True, text=True, timeout=600)
    assert fresh.returncode == 0, fresh.stderr[-2000:]
    assert int(fresh.stdout.split()[-1]) == launches == _eager_launches()
