"""torch.compile / torch.export of the package's modules, traced on fake CUDA tensors (no GPU needed).

Checks the msda_b200 custom ops' fake implementations (shapes and dtypes, concrete and symbolic), that Dynamo traces every
caller without a graph break, and that torch.export records the op of the path the eager module takes."""
import pytest
import torch
from torch._subclasses.fake_tensor import FakeTensorMode

import vit_adapter_b200 as vab
from vit_adapter_b200 import _ops  # noqa: F401  (registers torch.ops.msda_b200)
from vit_adapter_b200.adapter import Extractor, Injector, InteractionBlock, InteractionBlockWithCls
from vit_adapter_b200.mmcv_compat import MultiScaleDeformableAttention
from vit_adapter_b200.modules import MSDeformAttn

ops = torch.ops.msda_b200
F32, BF16, F16, F64 = torch.float32, torch.bfloat16, torch.float16, torch.float64
N, S, M, D, L, Lq, P = 2, 336, 4, 32, 3, 64, 4


def _m(*shape, dtype=F32):
    return torch.empty(shape, dtype=dtype, device='meta')


def _meta(dtype=F32):
    return _m(L, 2, dtype=torch.long), _m(L, dtype=torch.long)


def _fake_table():
    """(name, op, args, [(shape, dtype) of each output])."""
    rows = []
    for dt in (F32, BF16, F16, F64):
        cdt = F64 if dt == F64 else F32
        sh, lsi = _meta()
        v, loc, aw = _m(N, S, M, D, dtype=dt), _m(N, Lq, M, L, P, 2, dtype=cdt), _m(N, Lq, M, L, P, dtype=cdt)
        rows.append(('plain-%s' % dt, ops.ms_deform_attn, (v, sh, lsi, loc, aw, 64), [((N, Lq, M * D), dt)]))
        rows.append(('plain_bwd-%s' % dt, ops.ms_deform_attn_backward, (v, sh, lsi, loc, aw, _m(N, Lq, M * D, dtype=dt), 64),
                     [((N, S, M, D), dt), ((N, Lq, M, L, P, 2), cdt), ((N, Lq, M, L, P), cdt)]))
    for dt in (F32, BF16, F16):
        for ref_shape in ((1, Lq, 1, 2), (N, Lq, L, 4)):
            sh, lsi = _meta()
            v, ref = _m(N, S, M, D, dtype=dt), _m(*ref_shape)
            off, logit, merged = _m(N, Lq, M, L, P, 2), _m(N, Lq, M, L * P), _m(N, Lq, M * L * P * 3)
            go = _m(N, Lq, M * D, dtype=dt)
            tag = '%s-%s' % (dt, 'points' if ref_shape[-1] == 2 else 'boxes')
            rows.append(('fused-' + tag, ops.ms_deform_attn_fused, (v, sh, lsi, ref, off, logit), [((N, Lq, M * D), dt)]))
            rows.append(('merged-' + tag, ops.ms_deform_attn_merged, (v, sh, lsi, ref, merged, L, P), [((N, Lq, M * D), dt)]))
            for ref_grad in (False, True):
                gref = (ref_shape if ref_grad else (0,), F32)
                rows.append(('fused_bwd-%s-ref_grad=%s' % (tag, ref_grad), ops.ms_deform_attn_fused_backward,
                             (v, sh, lsi, ref, off, logit, go, ref_grad),
                             [((N, S, M, D), dt), ((N, Lq, M, L, P, 2), F32), ((N, Lq, M, L * P), F32), gref]))
                rows.append(('merged_bwd-%s-ref_grad=%s' % (tag, ref_grad), ops.ms_deform_attn_merged_backward,
                             (v, sh, lsi, ref, merged, L, P, go, ref_grad),
                             [((N, S, M, D), dt), ((N, Lq, M * L * P * 3), F32), gref]))
    C = 96
    for xdt, ydt in ((F32, F32), (F32, BF16), (BF16, BF16), (F16, F16)):
        x, w, b = _m(N, 21, C, dtype=xdt), _m(C), _m(C)
        rows.append(('layernorm-%s-%s' % (xdt, ydt), ops.layernorm, (x, w, b, 1e-6, ydt), [((N, 21, C), ydt), ((2, N * 21), F32)]))
        rows.append(('layernorm-nobias-%s-%s' % (xdt, ydt), ops.layernorm, (x, w, None, 1e-6, ydt),
                     [((N, 21, C), ydt), ((2, N * 21), F32)]))
        rows.append(('layernorm_bwd-%s-%s' % (xdt, ydt), ops.layernorm_backward, (_m(N, 21, C, dtype=ydt), x, w, _m(2, N * 21)),
                     [((N, 21, C), xdt), ((2, C), F32)]))
    H = W = 4
    n = 21 * (H // 2) * (W // 2)
    for dt in (F32, BF16):
        x, w, b = _m(N, n, C, dtype=dt), _m(C, 1, 3, 3, dtype=dt), _m(C, dtype=dt)
        rows.append(('dwconv-%s' % dt, ops.dwconv, (x, w, b, H, W), [((N, n, C), dt)]))
        for need_input, need_weight in ((True, True), (True, False), (False, True)):
            rows.append(('dwconv_bwd-%s-%d%d' % (dt, need_input, need_weight), ops.dwconv_backward,
                         (x, w, _m(N, n, C, dtype=dt), H, W, need_input, need_weight),
                         [((N, n, C) if need_input else (0,), dt), ((C, 1, 3, 3) if need_weight else (0,), dt),
                          ((C,) if need_weight else (0,), dt)]))
        rows.append(('residual_add-%s' % dt, ops.residual_add, (_m(N, n, C), _m(N, n, C, dtype=dt)), [((N, n, C), F32)]))
        rows.append(('colsum-%s' % dt, ops.colsum, (_m(N, n, C, dtype=dt),), [((C,), F32)]))
    return rows


_TABLE = _fake_table()


@pytest.mark.parametrize('row', _TABLE, ids=[r[0] for r in _TABLE])
def test_fake_impl_shapes_and_dtypes(row):
    _, op, args, want = row
    out = op(*args)
    outs = out if isinstance(out, (tuple, list)) else (out,)
    assert [(tuple(o.shape), o.dtype) for o in outs] == [(tuple(s), dt) for s, dt in want]
    assert all(o.device.type == 'meta' and o.is_contiguous() for o in outs)


@pytest.mark.parametrize('row', _TABLE, ids=[r[0] for r in _TABLE])
def test_fake_impl_symbolic_sizes(row):
    """The same table traced with symbolic sizes: every output dimension is an expression of the input sizes."""
    from torch.fx.experimental.proxy_tensor import make_fx
    _, op, args, want = row
    pos = [i for i, a in enumerate(args) if isinstance(a, torch.Tensor)]

    def call(*tensors):
        full = list(args)
        for i, t in zip(pos, tensors):
            full[i] = t
        return op(*full)

    gm = make_fx(call, tracing_mode='symbolic')(*[args[i] for i in pos])
    outs = [n for n in gm.graph.nodes if n.op == 'output'][0].args[0]
    vals = [o.meta['val'] for o in (outs if isinstance(outs, (tuple, list)) else (outs,))]
    hint = lambda d: d.node.hint if isinstance(d, torch.SymInt) else d  # noqa: E731
    assert [(tuple(hint(d) for d in v.shape), v.dtype) for v in vals] == [(tuple(s), dt) for s, dt in want]
    assert any(isinstance(d, torch.SymInt) for v in vals for d in v.shape)


def test_every_op_in_the_table():
    want = {'ms_deform_attn', 'ms_deform_attn_backward', 'ms_deform_attn_fused', 'ms_deform_attn_fused_backward',
            'ms_deform_attn_merged', 'ms_deform_attn_merged_backward', 'layernorm', 'layernorm_backward', 'dwconv',
            'dwconv_backward', 'residual_add', 'colsum'}
    assert {r[1]._qualified_op_name.split('::')[1] for r in _TABLE} == want


# --- Dynamo / export on fake CUDA tensors --------------------------------------------------------------------------------
def _msda_targets(gm):
    """msda_b200 ops called anywhere in a traced graph module (autograd.Function bodies included)."""
    found = set()
    for mod in gm.modules():
        if isinstance(mod, torch.fx.GraphModule):
            for node in mod.graph.nodes:
                if node.op == 'call_function' and str(node.target).startswith('msda_b200.'):
                    found.add(str(node.target).split('.')[1])
    return found


def _explain(fn, *args):
    torch._dynamo.reset()
    ex = torch._dynamo.explain(fn)(*args)
    assert ex.graph_break_count == 0, [str(r.reason) for r in ex.break_reasons]
    assert ex.graph_count == 1
    return set().union(*[_msda_targets(g) for g in ex.graphs])


def _levels(shapes):
    """(spatial_shapes, level_start_index, total tokens); the tensors are fake, their values never read."""
    sizes = [h * w for h, w in shapes]
    return (torch.empty(len(shapes), 2, dtype=torch.long), torch.empty(len(shapes), dtype=torch.long), sum(sizes))


@pytest.fixture
def fake_cuda():
    with FakeTensorMode(), torch.device('cuda'):
        yield


def _attn_case(path, ref_dim, ref_grad, d_model=128, heads=4):
    attn = MSDeformAttn(d_model, L, heads, P)
    attn.fused = path != 'unfused'
    attn.merge_query_linears = path == 'merged'
    shapes, lsi, s = _levels([(16, 16), (8, 8), (4, 4)])
    q = torch.randn(N, Lq, d_model, requires_grad=True)
    feat = torch.randn(N, s, d_model, requires_grad=True)
    ref = torch.rand(N if ref_grad else 1, Lq, L if ref_dim == 4 else 1, ref_dim, requires_grad=ref_grad)
    return attn, (q, ref, feat, shapes, lsi)


_WANT_OP = {'merged': 'ms_deform_attn_merged', 'fused': 'ms_deform_attn_fused', 'unfused': 'ms_deform_attn'}


def _with_backward(*names):
    """Forward ops and the backward ops Dynamo records with them (the Functions' backward bodies are traced too)."""
    return set(names) | {n + '_backward' for n in names}


@pytest.mark.parametrize('ref_grad', [False, True], ids=['const_ref', 'ref_grad'])
@pytest.mark.parametrize('ref_dim', [2, 4], ids=['points', 'boxes'])
@pytest.mark.parametrize('path', ['merged', 'fused', 'unfused'])
def test_msdeformattn_no_graph_break(fake_cuda, path, ref_dim, ref_grad):
    attn, args = _attn_case(path, ref_dim, ref_grad)
    assert _explain(attn, *args) == _with_backward(_WANT_OP[path]) | {'colsum'}


def _block_inputs(dim=128, h=8):
    ds = [(2 * h, 2 * h), (h, h), (h // 2, h // 2)]
    s1, l1, _ = _levels(ds)
    s2, l2, _ = _levels([(h, h)])
    n_c = 21 * (h // 2) ** 2
    di1 = [torch.rand(1, h * h, 1, 2), s1, l1]
    di2 = [torch.rand(1, n_c, 1, 2), s2, l2]
    x = torch.randn(N, h * h, dim, requires_grad=True)
    c = torch.randn(N, n_c, dim, requires_grad=True)
    return x, c, di1, di2, h


def _stand_in_block(x, H, W):
    return x * 1.5


_BLOCK_OPS = {'ms_deform_attn_merged', 'layernorm', 'dwconv'}
# (the LayerNorm and depth-wise conv backward ops come from the ops' registered autograd: AOTAutograd traces them later)
_BLOCK_TRAINING_OPS = _with_backward('ms_deform_attn_merged') | {'layernorm', 'dwconv', 'colsum'}


def test_injector_no_graph_break(fake_cuda):
    inj = Injector(dim=128, num_heads=2, n_points=4, n_levels=3, deform_ratio=0.5, init_values=0.1)
    x, c, di1, _, _ = _block_inputs()
    assert _explain(lambda x, c: inj(x, di1[0], c, di1[1], di1[2]), x, c) == \
        _with_backward('ms_deform_attn_merged') | {'layernorm', 'colsum'}


def test_extractor_no_graph_break(fake_cuda):
    ext = Extractor(dim=128, num_heads=2, n_points=4, n_levels=1, deform_ratio=0.5)
    x, c, _, di2, h = _block_inputs()
    assert _explain(lambda x, c: ext(c, di2[0], x, di2[1], di2[2], h, h), x, c) == _BLOCK_TRAINING_OPS


@pytest.mark.parametrize('extra_extractor', [False, True])
def test_interaction_block_no_graph_break(fake_cuda, extra_extractor):
    blk = InteractionBlock(128, 2, 4, deform_ratio=0.5, init_values=0.1, extra_extractor=extra_extractor)
    x, c, di1, di2, h = _block_inputs()
    assert _explain(lambda x, c: blk(x, c, [_stand_in_block], di1, di2, h, h), x, c) == _BLOCK_TRAINING_OPS


def test_interaction_block_with_cls_no_graph_break(fake_cuda):
    blk = InteractionBlockWithCls(128, 2, 4, deform_ratio=0.5, init_values=0.1)
    x, c, di1, di2, h = _block_inputs()
    cls = torch.randn(N, 1, 128, requires_grad=True)
    assert _explain(lambda x, c, cls: blk(x, c, cls, [_stand_in_block], di1, di2, h, h), x, c, cls) == _BLOCK_TRAINING_OPS


@pytest.mark.parametrize('ref_dim', [2, 4], ids=['points', 'boxes'])
def test_mmcv_shim_no_graph_break(fake_cuda, ref_dim):
    attn = MultiScaleDeformableAttention(embed_dims=128, num_heads=4, num_levels=L, num_points=P)
    shapes, lsi, s = _levels([(16, 16), (8, 8), (4, 4)])
    query = torch.randn(Lq, N, 128, requires_grad=True)     # (num_query, bs, embed_dims): batch_first=False
    value = torch.randn(s, N, 128, requires_grad=True)
    ref = torch.rand(N, Lq, L, ref_dim)
    assert _explain(lambda q, v: attn(q, value=v, reference_points=ref, spatial_shapes=shapes, level_start_index=lsi),
                    query, value) == _with_backward('ms_deform_attn_merged') | {'colsum'}


@pytest.mark.parametrize('dtype', [F32, F64])
def test_bare_function_apply_no_graph_break(fake_cuda, dtype):
    shapes, lsi, s = _levels([(16, 16), (8, 8), (4, 4)])
    value = torch.randn(N, s, M, D, dtype=dtype, requires_grad=True)
    loc = torch.rand(N, Lq, M, L, P, 2, dtype=dtype, requires_grad=True)
    aw = torch.rand(N, Lq, M, L, P, dtype=dtype, requires_grad=True)
    assert _explain(lambda v, l, a: vab.MSDeformAttnFunction.apply(v, shapes, lsi, l, a, 64), value, loc, aw) == \
        _with_backward('ms_deform_attn')


@pytest.mark.parametrize('path', ['merged', 'fused', 'unfused'])
def test_msdeformattn_fullgraph_dynamic_inference(fake_cuda, path):
    """fullgraph + dynamic shapes through AOTAutograd (inference graph: the joint graph needs a real CUDA device for the
    autograd engine and is compiled in test_compile_gpu.py)."""
    torch._dynamo.reset()
    attn, (q, ref, feat, shapes, lsi) = _attn_case(path, 4, False)
    with torch.no_grad():
        out = torch.compile(attn, backend='aot_eager', fullgraph=True, dynamic=True)(q, ref, feat, shapes, lsi)
    assert out.shape == q.shape and out.device.type == 'cuda'


def test_interaction_block_fullgraph_dynamic_inference(fake_cuda):
    torch._dynamo.reset()
    blk = InteractionBlock(128, 2, 4, deform_ratio=0.5, init_values=0.1, extra_extractor=True)
    x, c, di1, di2, h = _block_inputs()
    with torch.no_grad():
        xo, co = torch.compile(lambda x, c: blk(x, c, [_stand_in_block], di1, di2, h, h), backend='aot_eager',
                               fullgraph=True, dynamic=True)(x, c)
    assert xo.shape == x.shape and co.shape == c.shape


def _export_targets(mod, args):
    ep = torch.export.export(mod, args)
    return _msda_targets(ep.graph_module)


@pytest.mark.parametrize('path', ['merged', 'fused', 'unfused'])
def test_export_msdeformattn(fake_cuda, path):
    attn, args = _attn_case(path, 2, False)
    assert _export_targets(attn, tuple(a.detach() for a in args)) == {_WANT_OP[path]}


def test_export_interaction_block(fake_cuda):
    blk = InteractionBlock(128, 2, 4, deform_ratio=0.5, init_values=0.1, extra_extractor=True)
    x, c, di1, di2, h = _block_inputs()
    assert _export_targets(blk, (x.detach(), c.detach(), [], di1, di2, h, h)) == _BLOCK_OPS
