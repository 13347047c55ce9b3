"""Fused entry points with box reference points (x, y, w, h), reference-point gradients and four levels, against the
reference module's op sequence (detection/ops/modules/ms_deform_attn.py:108-128) run through the plain Function."""
import ctypes

import pytest
import torch
import torch.nn.functional as F

from oracle.core_pytorch import ms_deform_attn_core

import vit_adapter_b200 as vab
from vit_adapter_b200 import _cabi

pytestmark = pytest.mark.gpu
DEV = 'cuda:0'
SHAPES = {1: [(12, 10)], 3: [(12, 10), (6, 5), (3, 3)], 4: [(12, 10), (6, 5), (3, 3), (2, 2)]}
TOL = {torch.float32: (1e-5, 1e-4), torch.bfloat16: (1e-2, 1e-2), torch.float16: (2e-3, 2e-3)}   # test_fused_matches_unfused's


def _scale(t):
    return float(t.abs().max()) + 1e-30


def _inputs(N, M, D, Lq, shapes, rb, rl, ref_dim, dtype, seed):
    g = torch.Generator().manual_seed(seed)
    shapes_t = torch.as_tensor(shapes, dtype=torch.long)
    L = shapes_t.shape[0]
    S = int(shapes_t.prod(1).sum())
    lsi = torch.cat((shapes_t.new_zeros((1,)), shapes_t.prod(1).cumsum(0)[:-1]))
    value = torch.randn(N, S, M, D, generator=g).to(dtype)
    ref = torch.rand(rb, Lq, rl, ref_dim, generator=g)
    ref[..., :2] = ref[..., :2] * 1.1 - 0.05                                     # some reference points off-image
    offsets = torch.randn(N, Lq, M, L, 4, 2, generator=g) * 2.5
    if ref_dim == 4:
        ref[..., 2:] = ref[..., 2:] * 0.6
        ref[:, ::7, :, 2] = 0.0                                                  # degenerate boxes: w = 0
        ref[:, 3::11, :, 3] = 0.0                                                # and h = 0
        offsets = offsets * 0.8                                                  # offsets are in box units here
    logits = torch.randn(N, Lq, M, L * 4, generator=g) * 2.0
    grad_out = torch.randn(N, Lq, M * D, generator=g).to(dtype)
    return [t.to(DEV) for t in (value, shapes_t, lsi, ref, offsets, logits, grad_out)]


def _locations(ref, offsets, shapes):
    """The reference module's location arithmetic (ms_deform_attn.py:115-122)."""
    P = offsets.shape[4]
    if ref.shape[-1] == 2:
        wh = torch.stack([shapes[..., 1], shapes[..., 0]], -1)
        return ref[:, :, None, :, None, :] + offsets / wh[None, None, None, :, None, :]
    return ref[:, :, None, :, None, :2] + offsets / P * ref[:, :, None, :, None, 2:] * 0.5


def _unfused(value, shapes, lsi, ref, offsets, logits):
    N, Lq, M, L, P, _ = offsets.shape
    weights = F.softmax(logits, -1).view(N, Lq, M, L, P)
    loc = _locations(ref, offsets, shapes)
    return vab.MSDeformAttnFunction.apply(value, shapes, lsi, loc.contiguous(), weights.contiguous(), 64)


def _leaves(*ts):
    return [t.clone().requires_grad_() for t in ts]


@pytest.mark.parametrize('L, hot', [(1, 2), (4, 2), (4, 5), (4, 11), (4, 12)])
def test_box_locations_are_bit_identical(L, hot):
    """One-hot logits make the softmax exactly {0, 1}: any output difference could only come from the box location
    arithmetic, and there must be none - also for boxes partly off the image and with zero width or height. The hot point
    `hot` lies in level hot // 4, so every level's reference lookup and box arithmetic is checked bit for bit."""
    N, M, D, Lq = 2, 2, 32, 300
    shapes = [(40, 40), (20, 20), (10, 10), (5, 5)][:L]
    value, shapes_t, lsi, ref, offsets, logits, _ = _inputs(N, M, D, Lq, shapes, N, L, 4, torch.float32, 41)
    logits = torch.full_like(logits, -1e4)
    logits[..., hot] = 0.0
    out1 = vab.MSDeformAttnFusedFunction.apply(value, shapes_t, lsi, ref, offsets, logits)
    out2 = _unfused(value, shapes_t, lsi, ref, offsets, logits)
    assert torch.equal(out1, out2)


@pytest.mark.parametrize('dtype', [torch.float32, torch.bfloat16, torch.float16], ids=['f32', 'bf16', 'f16'])
@pytest.mark.parametrize('D', [32, 64])
@pytest.mark.parametrize('L', [1, 3, 4])
@pytest.mark.parametrize('rl', ['1', 'L'])
@pytest.mark.parametrize('rb', ['1', 'N'])
@pytest.mark.parametrize('ref_dim', [2, 4])
def test_fused_with_reference_gradient_matches_unfused(ref_dim, rb, rl, L, D, dtype):
    """Separate tensors and the merged layout against the unfused sequence, with autograd through reference_points; the
    merged layout is bit-identical to the separate tensors, grad_reference_points included."""
    N, M, Lq = 2, 4, 50
    rb_, rl_ = (1 if rb == '1' else N), (1 if rl == '1' else L)
    value, shapes_t, lsi, ref, offsets, logits, go = _inputs(N, M, D, Lq, SHAPES[L], rb_, rl_, ref_dim, dtype, 7 * L + D)
    assert _cabi.fused_supported(value, L, 4)
    if dtype == torch.float16:
        vab.set_amp_value_dtype(torch.float16)
    try:
        v1, r1, o1, l1 = _leaves(value, ref, offsets, logits)
        out1 = vab.MSDeformAttnFusedFunction.apply(v1, shapes_t, lsi, r1, o1, l1)
        out1.backward(go)
        v2, r2, o2, l2 = _leaves(value, ref, offsets, logits)
        out2 = _unfused(v2, shapes_t, lsi, r2, o2, l2)
        out2.backward(go)
        merged = torch.cat([offsets.reshape(N, Lq, -1), logits.reshape(N, Lq, -1)], -1)
        v3, r3, m3 = _leaves(value, ref, merged)
        out3 = vab.MSDeformAttnMergedFunction.apply(v3, shapes_t, lsi, r3, m3, L, 4)
        out3.backward(go)
        torch.cuda.synchronize()
    finally:
        vab.set_amp_value_dtype(torch.float32)
    ft, gt = TOL[dtype]
    torch.testing.assert_close(out1.float(), out2.float(), rtol=ft, atol=ft * max(1.0, _scale(out2.float())))
    torch.testing.assert_close(v1.grad.float(), v2.grad.float(), rtol=gt, atol=gt * _scale(v2.grad.float()))
    torch.testing.assert_close(o1.grad, o2.grad, rtol=gt, atol=gt * _scale(o2.grad))
    torch.testing.assert_close(l1.grad, l2.grad, rtol=gt, atol=gt * _scale(l2.grad))
    assert r1.grad.shape == ref.shape and float(r1.grad.abs().max()) > 0
    torch.testing.assert_close(r1.grad, r2.grad, rtol=gt, atol=gt * _scale(r2.grad))
    assert torch.equal(out1, out3)
    assert torch.equal(r1.grad, r3.grad)
    assert torch.equal(m3.grad, torch.cat([o1.grad.reshape(N, Lq, -1), l1.grad.reshape(N, Lq, -1)], -1))


@pytest.mark.parametrize('ref_dim', [2, 4])
def test_reference_gradient_matches_fp64_oracle(ref_dim):
    """grad_reference_points of the fp32 kernels against fp64 autograd through the reference's pure-PyTorch core."""
    N, M, D, Lq, L = 2, 3, 32, 20, 4
    value, shapes_t, lsi, ref, offsets, logits, go = _inputs(N, M, D, Lq, SHAPES[L], N, L, ref_dim, torch.float32, 5)
    ref[..., :2] = ref[..., :2] * 0.6 + 0.2            # keep every sample inside the image: no boundary kinks
    offsets = offsets * 0.2
    r1 = ref.clone().requires_grad_()
    out = vab.MSDeformAttnFusedFunction.apply(value, shapes_t, lsi, r1, offsets, logits)
    out.backward(go)
    r64 = ref.double().requires_grad_()
    w = F.softmax(logits.double(), -1).view(N, Lq, M, L, 4)
    want = ms_deform_attn_core(value.double(), shapes_t.cpu(), _locations(r64, offsets.double(), shapes_t), w)
    want.backward(go.double())
    torch.testing.assert_close(out.double(), want.detach(), rtol=1e-5, atol=1e-5 * _scale(want))
    torch.testing.assert_close(r1.grad.double(), r64.grad, rtol=1e-4, atol=1e-4 * _scale(r64.grad))


@pytest.mark.parametrize('rl', [1, 4])
def test_reference_gradient_is_bitwise_reproducible(rl):
    N, M, D, Lq, L = 2, 8, 32, 900, 4
    value, shapes_t, lsi, ref, offsets, logits, go = _inputs(N, M, D, Lq, SHAPES[L], 1, rl, 4, torch.float32, 9)
    lib = _cabi.load()
    dims, rb, rl_ = _cabi._fused_dims(value, ref, offsets, logits)
    ws_bytes = lib.msda_backward_fused_workspace_bytes(ctypes.byref(dims), _cabi.MSDA_F32, rb, rl_, 4, 1)
    runs = []
    for _ in range(3):
        # NaN-filled workspace and outputs: a partial or an output element the kernels failed to write shows up as NaN
        ws = torch.full((ws_bytes // 4,), float('nan'), device=DEV)
        outs = [torch.full_like(t, float('nan')) for t in (value, offsets, logits, ref)]
        rc = lib.msda_backward_fused_ref(ctypes.byref(dims), _cabi.MSDA_F32, value.data_ptr(), shapes_t.data_ptr(),
                                         lsi.data_ptr(), ref.data_ptr(), rb, rl_, 4, offsets.data_ptr(), logits.data_ptr(),
                                         0, 0, go.data_ptr(), *[t.data_ptr() for t in outs], ws.data_ptr(), ws_bytes,
                                         torch.cuda.current_stream().cuda_stream)
        assert rc == 0, lib.msda_last_error()
        torch.cuda.synchronize()
        assert not any(t.isnan().any() for t in outs)
        runs.append(outs)
    for r in runs[1:]:
        assert torch.equal(r[3], runs[0][3])
        assert torch.equal(r[1], runs[0][1]) and torch.equal(r[2], runs[0][2])


@pytest.mark.parametrize('dtype', [torch.float32, torch.bfloat16], ids=['f32', 'bf16'])
@pytest.mark.parametrize('ref_dim', [2, 4])
def test_reference_gradient_costs_one_launch_only_when_asked(ref_dim, dtype):
    """Without requires_grad on reference_points the backward issues exactly the launches it always has (the fused
    scatter, plus the fp32 -> 16-bit convert for bf16); with it, one more (the fixed-order sum of the partials)."""
    N, M, D, Lq, L = 2, 4, 32, 64, 3
    value, shapes_t, lsi, ref, offsets, logits, go = _inputs(N, M, D, Lq, SHAPES[L], 1, 1, ref_dim, dtype, 3)
    base = 1 if dtype == torch.float32 else 2
    for want_ref, extra in ((False, 0), (True, 1)):
        v, o, l = _leaves(value, offsets, logits)
        r = ref.clone().requires_grad_(want_ref)
        out = vab.MSDeformAttnFusedFunction.apply(v, shapes_t, lsi, r, o, l)
        n0 = _cabi.launch_count()
        out.backward(go)
        torch.cuda.synchronize()
        assert _cabi.launch_count() - n0 == base + extra
        assert (r.grad is not None) == want_ref


def _decoder_module(mmcv):
    torch.manual_seed(0)
    if mmcv:
        from vit_adapter_b200.mmcv_compat import MultiScaleDeformableAttention
        m = MultiScaleDeformableAttention(embed_dims=256, num_heads=8, num_levels=4, num_points=4, dropout=0.0,
                                          batch_first=True)
    else:
        m = vab.MSDeformAttn(d_model=256, n_levels=4, n_heads=8, n_points=4)
    m = m.to(DEV)
    with torch.no_grad():
        for p in m.parameters():
            p.add_(torch.randn_like(p) * 0.02)
    return m


def _run_module(m, mmcv, query, ref, feat, shapes, lsi):
    if mmcv:
        return m(query, value=feat, reference_points=ref, spatial_shapes=shapes, level_start_index=lsi)
    return m(query, ref, feat, shapes, lsi)


def _ran_fused(out):
    """True when the autograd graph of `out` holds one of the fused Functions."""
    seen, stack = set(), [out.grad_fn]
    while stack:
        f = stack.pop()
        if f is None or f in seen:
            continue
        seen.add(f)
        if type(f).__name__.startswith(('MSDeformAttnMergedFunction', 'MSDeformAttnFusedFunction')):
            return True
        stack.extend(n for n, _ in f.next_functions)
    return False


@pytest.mark.parametrize('mmcv', [False, True], ids=['MSDeformAttn', 'mmcv-shim'])
@pytest.mark.parametrize('ref_kind', ['box', 'box-nograd', 'learned-2d'])
def test_four_level_decoder_takes_the_fused_path_and_matches_unfused(ref_kind, mmcv):
    m = _decoder_module(mmcv)
    shapes = torch.as_tensor([(16, 20), (8, 10), (4, 5), (2, 3)], dtype=torch.long, device=DEV)
    lsi = torch.cat((shapes.new_zeros((1,)), shapes.prod(1).cumsum(0)[:-1]))
    N, Lq = 2, 30
    query = torch.randn(N, Lq, 256, device=DEV)
    feat = torch.randn(N, int(shapes.prod(1).sum()), 256, device=DEV)
    ref0 = torch.rand(N, Lq, 4, 4 if ref_kind.startswith('box') else 2, device=DEV)
    if ref_kind.startswith('box'):
        ref0[..., 2:] *= 0.3
    needs_grad = ref_kind != 'box-nograd'
    res = {}
    for fused in (True, False):
        m.fused = fused
        m.zero_grad(set_to_none=True)
        q = query.clone().requires_grad_()
        r = ref0.clone().requires_grad_(needs_grad)
        out = _run_module(m, mmcv, q, r, feat, shapes, lsi)
        assert _ran_fused(out) == fused
        n0 = _cabi.launch_count()
        out.square().mean().backward()
        torch.cuda.synchronize()
        res[fused] = (out.detach(), q.grad, r.grad, {k: p.grad.clone() for k, p in m.named_parameters()},
                      _cabi.launch_count() - n0)
    m.fused = True
    tol = 1e-4
    for i in (0, 1):
        torch.testing.assert_close(res[True][i], res[False][i], rtol=tol, atol=tol * _scale(res[False][i]))
    if needs_grad:
        torch.testing.assert_close(res[True][2], res[False][2], rtol=tol, atol=tol * _scale(res[False][2]))
    else:
        assert res[True][2] is None
    for k in res[True][3]:
        torch.testing.assert_close(res[True][3][k], res[False][3][k], rtol=tol, atol=tol * _scale(res[False][3][k]), msg=k)
    # the fused path: the same backward without the reference gradient launches exactly one kernel fewer
    m.zero_grad(set_to_none=True)
    out = _run_module(m, mmcv, query, ref0, feat, shapes, lsi)
    n0 = _cabi.launch_count()
    out.square().mean().backward()
    assert res[True][4] - (_cabi.launch_count() - n0) == (1 if needs_grad else 0)


@pytest.mark.parametrize('ref_dim', [2, 4])
def test_reference_points_at_an_odd_storage_offset_are_copied_not_rejected(ref_dim):
    """A contiguous fp32 view that starts 4 bytes into its storage misses the kernels' 8- / 16-byte load alignment: the
    Function copies it (as the unfused sequence would simply read it) and returns the gradient for the view."""
    N, M, D, Lq, L = 2, 4, 32, 40, 4
    value, shapes_t, lsi, ref, offsets, logits, go = _inputs(N, M, D, Lq, SHAPES[L], N, L, ref_dim, torch.float32, 17)
    store = torch.empty(ref.numel() + 1, device=DEV)
    odd = store[1:].view(ref.shape)
    odd.copy_(ref)
    assert odd.is_contiguous() and odd.data_ptr() % 8 == 4
    r1, r2 = odd.detach().requires_grad_(), ref.clone().requires_grad_()
    out1 = vab.MSDeformAttnFusedFunction.apply(value, shapes_t, lsi, r1, offsets, logits)
    out1.backward(go)
    out2 = vab.MSDeformAttnFusedFunction.apply(value, shapes_t, lsi, r2, offsets, logits)
    out2.backward(go)
    assert torch.equal(out1, out2) and torch.equal(r1.grad, r2.grad)


def test_reference_gradient_replays_in_a_cuda_graph():
    N, M, D, Lq, L = 2, 8, 32, 300, 4
    value, shapes_t, lsi, ref, offsets, logits, go = _inputs(N, M, D, Lq, SHAPES[L], N, L, 4, torch.float32, 11)
    leaves = _leaves(value, ref, offsets, logits)

    def step():
        for t in leaves:
            t.grad = None
        out = vab.MSDeformAttnFusedFunction.apply(leaves[0], shapes_t, lsi, leaves[1], leaves[2], leaves[3])
        out.backward(go)
        return out

    s = torch.cuda.Stream()
    s.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(s):
        for _ in range(2):
            step()
    torch.cuda.current_stream().wait_stream(s)
    g = torch.cuda.CUDAGraph()
    for t in leaves:
        t.grad = None
    with torch.cuda.graph(g):
        static_out = step()
    static_grads = [t.grad for t in leaves]
    # new inputs, then replay, against an eager run on the same inputs
    _, _, _, ref2, off2, log2, _ = _inputs(N, M, D, Lq, SHAPES[L], N, L, 4, torch.float32, 12)
    with torch.no_grad():
        leaves[1].copy_(ref2), leaves[2].copy_(off2), leaves[3].copy_(log2)
    g.replay()
    torch.cuda.synchronize()
    eager = _leaves(value, ref2, off2, log2)
    out = vab.MSDeformAttnFusedFunction.apply(eager[0], shapes_t, lsi, eager[1], eager[2], eager[3])
    out.backward(go)
    torch.cuda.synchronize()
    assert torch.equal(static_out, out)
    for i in (1, 2, 3):                                 # no atomics in these: bit-identical
        assert torch.equal(static_grads[i], eager[i].grad)
    torch.testing.assert_close(static_grads[0], eager[0].grad, rtol=1e-5, atol=1e-6 * _scale(eager[0].grad))


@pytest.mark.parametrize('L', [1, 3, 4])
@pytest.mark.parametrize('ref_dim', [2, 4])
def test_packed16_backward_with_reference_gradient(ref_dim, L):
    """bwd_packed16 = 2 runs the same fused kernel template with packed 16-bit grad_value reductions (for (L, P) in
    {(3,4),(1,4)}; (4,4) keeps the fp32 accumulator). The reference-point, offset and logit gradients do not depend on the
    grad_value scatter, so they equal the default path's bit for bit."""
    N, M, D, Lq = 2, 4, 32, 64
    value, shapes_t, lsi, ref, offsets, logits, go = _inputs(N, M, D, Lq, SHAPES[L], N, L, ref_dim, torch.bfloat16, 13)
    res = []
    try:
        for packed in (0, 2):
            _cabi.set_tuning(bwd_packed16=packed)
            n0 = _cabi.launch_count()
            res.append(_cabi.backward_fused(value, shapes_t, lsi, ref, offsets, logits, go, ref_grad=True)
                       + (_cabi.launch_count() - n0,))
            torch.cuda.synchronize()
    finally:
        _cabi.set_tuning(bwd_packed16=0)
    for i in (1, 2, 3):
        assert torch.equal(res[0][i], res[1][i])
    torch.testing.assert_close(res[1][0].float(), res[0][0].float(), rtol=2e-2, atol=2e-2 * _scale(res[0][0].float()))
    assert res[0][4] == 3                               # scatter + convert + reference-gradient sum
    assert res[1][4] == (2 if L in (1, 3) else 3)       # packed scatter (no convert) + reference-gradient sum
