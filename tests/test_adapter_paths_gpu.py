"""Every launch path of the adapter's depth-wise 3x3 convolution (csrc/adapter_dwconv.cu) and LayerNorm row kernels
(csrc/adapter_layernorm.cu) against fp64.

The convolution picks its kernel family from the dtype, C, the map sizes, a shared-memory formula and the alignment of
its pointers, so each case below names the kernels it must launch and checks that they ran (`kernels_launched`).
Inputs are placed at byte offsets inside larger buffers (`at_offset`) to reach the misaligned paths.

Results are compared with the fp64 oracles (oracle/dwconv_ref.py, oracle/layernorm_ref.py) evaluated on the rounded
inputs, within bounds derived from the rounding the kernels do:

    |out - ref| <= u_out * |ref| + (1 + u_out) * acc + floor

u_out is the unit roundoff of the output dtype (2^-8 bf16, 2^-11 f16, 0 when the output is the fp32 / fp64 accumulator),
acc bounds the accumulation error (c * u_acc * sum of |terms| for a sum), floor is half the subnormal spacing of the
output dtype. Each `acc` says where its constant comes from.
"""
import pytest
import torch
import torch.nn.functional as F
from torch import nn

from kernel_paths import assert_within, at_offset, kernel, kernels_launched
from oracle import dwconv_ref, layernorm_ref

pytestmark = pytest.mark.gpu

U32 = 2.0 ** -24
U64 = 2.0 ** -53
B = 3
T_NAME = {torch.float32: 'float', torch.bfloat16: '__nv_bfloat16', torch.float16: '__half', torch.float64: 'double'}
SHORT = {torch.float32: 'f32', torch.bfloat16: 'bf16', torch.float16: 'f16', torch.float64: 'f64'}


# --- helpers -------------------------------------------------------------------------------------------------------------
def assert_kernels(names, expected, what):
    """Every expected pattern matched by exactly one launched kernel of this project, and no other such kernel."""
    ours = [n for n in names if 'adapter_' in n]
    for pat in expected:
        hits = [n for n in ours if pat.search(n)]
        assert len(hits) == 1, '%s: expected one launch of /%s/, got %s' % (what, pat.pattern, ours)
    assert len(ours) == len(expected), '%s: launched %s, expected %s' % (what, ours, [p.pattern for p in expected])


def _sms():
    return torch.cuda.get_device_properties(torch.cuda.current_device()).multi_processor_count


# --- A. depth-wise convolution --------------------------------------------------------------------------------------------
def tile(T, flip, cbq):
    return kernel('adapter_dwconv_tile_kernel', T_NAME[T], 'true' if flip else 'false', cbq)


def run(T, flip):
    return kernel('adapter_dwconv_run_kernel', T_NAME[T], 'true' if flip else 'false')


def generic(T, flip):
    return kernel('adapter_dwconv_kernel', T_NAME[T], 1, 'true' if flip else 'false')


def wgrad_run(T):
    return [kernel('adapter_dwconv_wgrad_run_kernel', T_NAME[T]), kernel('adapter_dwconv_wgrad_sum_kernel')]


def wgrad_atomic(T):
    return [kernel('adapter_dwconv_wgrad_kernel', T_NAME[T])]


def _family(T, fam, flip):
    if fam == 'tile64':
        return tile(T, flip, 16)
    if fam == 'tile32':
        return tile(T, flip, 8)
    return run(T, flip) if fam == 'run' else generic(T, flip)


# (id, dtype, C, H, W, byte offset of x and grad_y, forward / grad_x family, weight-gradient family)
DW_CASES = [
    ('f32-aligned-run', torch.float32, 64, 4, 8, 0, 'run', 'run'),
    ('f32-off4-generic', torch.float32, 64, 4, 8, 4, 'generic', 'atomic'),
    ('f32-C6-generic', torch.float32, 6, 4, 8, 0, 'generic', 'atomic'),
    ('f32-1x1-run', torch.float32, 64, 2, 2, 0, 'run', 'run'),
    ('f64-generic', torch.float64, 64, 4, 8, 0, 'generic', 'atomic'),
    ('f64-1x1-generic', torch.float64, 16, 2, 2, 0, 'generic', 'atomic'),
]
for _T in (torch.bfloat16, torch.float16):
    _s = SHORT[_T]
    DW_CASES += [
        (_s + '-C64-tile64', _T, 64, 4, 8, 0, 'tile64', 'run'),
        (_s + '-C128-tile64', _T, 128, 6, 16, 0, 'tile64', 'run'),
        (_s + '-C96-tile32', _T, 96, 4, 8, 0, 'tile32', 'run'),
        # the 64-channel tile needs 4 rows x 402 tokens x 128 B = 206 992 B (> 200 KB): 32-channel blocks
        (_s + '-W200-tile32', _T, 64, 2, 200, 0, 'tile32', 'run'),
        # the 32-channel tile needs 4 x 802 x 64 B + taps = 205 904 B: no tile
        (_s + '-W400-run', _T, 64, 2, 400, 0, 'run', 'run'),
        (_s + '-W12-run', _T, 64, 4, 12, 0, 'run', 'run'),     # quarter map 6 wide: not a multiple of 4
        (_s + '-W6-run', _T, 64, 4, 6, 0, 'run', 'run'),       # quarter map 3 wide: narrower than 4
        (_s + '-C48-run', _T, 48, 4, 8, 0, 'run', 'run'),      # C % 32 != 0
        (_s + '-off8-run', _T, 64, 4, 8, 8, 'run', 'run'),     # 8-byte aligned: no 16-byte tile loads
        (_s + '-off2-generic', _T, 64, 4, 8, 2, 'generic', 'atomic'),
        (_s + '-1x1-run', _T, 64, 2, 2, 0, 'run', 'run'),
        (_s + '-1x1-generic', _T, 64, 2, 2, 2, 'generic', 'atomic'),
        (_s + '-2x8-tile64', _T, 64, 2, 8, 0, 'tile64', 'run'),  # smallest maps the tile takes: 4x16, 2x8, 1x4
    ]


def _dw_inputs(dtype, C, H, W, seed):
    g = torch.Generator().manual_seed(seed)
    n = 21 * (H // 2) * (W // 2)
    x = torch.randn(B, n, C, generator=g).to(dtype).cuda()
    gy = torch.randn(B, n, C, generator=g).to(dtype).cuda()
    w = (torch.randn(C, 1, 3, 3, generator=g) / 3).to(dtype).cuda()
    b = torch.randn(C, generator=g).to(dtype).cuda()
    return x, gy, w, b


def _dw_reference(x, gy, w, b, H, W):
    """fp64 (y, y without bias, grad_x, grad_w, grad_b) and the matching sums of |terms|."""
    xd, gd, wd, bd = x.double(), gy.double(), w.double(), b.double()
    zero = torch.zeros_like(bd)
    y = dwconv_ref.dwconv_tokens(xd, wd, bd, H, W)
    y0 = dwconv_ref.dwconv_tokens(xd, wd, None, H, W)
    gx, gw, gb = dwconv_ref.dwconv_tokens_backward(xd, wd, bd, H, W, gd)
    s_y = dwconv_ref.dwconv_tokens(xd.abs(), wd.abs(), bd.abs(), H, W)
    s_y0 = dwconv_ref.dwconv_tokens(xd.abs(), wd.abs(), None, H, W)
    s_gx = dwconv_ref.dwconv_tokens_backward(xd, wd.abs(), zero, H, W, gd.abs())[0]
    _, s_gw, s_gb = dwconv_ref.dwconv_tokens_backward(xd.abs(), wd, zero, H, W, gd.abs())
    return (y, y0, gx, gw, gb), (s_y, s_y0, s_gx, s_gw, s_gb)


def _wgrad_depth(C, H, W, run_path):
    """Longest chain of dependent fp32 additions any grad_w / grad_b element goes through (a summation tree of depth d
    is within gamma_d = d * u of the sum of |terms|). Run path: a thread's items x 8 tokens, the CTA's item slots, the
    partial-row sum (<= ceil(rows / 32) + 2 + 32). Atomic path: a thread's tokens, the CTA's 8 rows, one atomic per CTA."""
    maps = ((2 * H, 2 * W), (H, W), (H // 2, W // 2))
    if run_path:
        cvec = C // 4
        ty = 256 // cvec
        items = B * sum(mh * -(-mw // 8) for mh, mw in maps)
        grid = min(-(-items // ty), 148 * 2)
        return -(-items // (grid * ty)) * 8 + ty + -(-grid // 32) + 34
    bt = B * 21 * (H // 2) * (W // 2)
    tpc = max(-(-bt // (2 * _sms())), 64)
    return -(-tpc // 8) + 8 + -(-bt // tpc)


def _dw_check(outs, refs, sums, dtype, C, H, W, wgrad_path, what):
    """Forward and grad_x: nine fused multiply-adds from the bias (or zero), one rounding each -> c = 10 leaves room for
    gamma_9 > 9u. grad_w / grad_b: c = the chain depth of the reduction."""
    ua = U64 if dtype == torch.float64 else U32
    names = ('y', 'y (bias=None)', 'grad_x', 'grad_w', 'grad_b')
    depth = _wgrad_depth(C, H, W, wgrad_path == 'run')
    for k, (o, r, s, nm) in enumerate(zip(outs, refs, sums, names)):
        c = 10 if k < 3 else depth
        assert_within(o, r, c * ua * s, '%s %s' % (what, nm))


@pytest.mark.parametrize('case', DW_CASES, ids=[c[0] for c in DW_CASES])
def test_dwconv_path_table(case):
    from vit_adapter_b200 import _cabi
    cid, dtype, C, H, W, off, fam, wfam = case
    x, gy, w, b = _dw_inputs(dtype, C, H, W, seed=C * 1000 + H * 10 + W)
    xo, gyo = at_offset(x, off), at_offset(gy, off)
    y, names = kernels_launched(lambda: _cabi.dwconv_forward(xo, w, b, H, W))
    assert_kernels(names, [_family(dtype, fam, False)], cid + ' forward')
    y0, names = kernels_launched(lambda: _cabi.dwconv_forward(xo, w, None, H, W))
    assert_kernels(names, [_family(dtype, fam, False)], cid + ' forward, bias=None')
    (gx, _, _), names = kernels_launched(lambda: _cabi.dwconv_backward(xo, w, gyo, H, W, need_weight=False))
    assert_kernels(names, [_family(dtype, fam, True)], cid + ' grad_x')
    (_, gw, gb), names = kernels_launched(lambda: _cabi.dwconv_backward(xo, w, gyo, H, W, need_input=False))
    assert_kernels(names, wgrad_run(dtype) if wfam == 'run' else wgrad_atomic(dtype), cid + ' grad_w')
    refs, sums = _dw_reference(x, gy, w, b, H, W)
    _dw_check((y, y0, gx, gw, gb), refs, sums, dtype, C, H, W, wfam, cid)


@pytest.mark.parametrize('dtype', [torch.float32, torch.bfloat16, torch.float16], ids=['f32', 'bf16', 'f16'])
def test_dwconv_wgrad_run_vs_atomic(dtype):
    """Aligned x and grad_y take the deterministic two-kernel reduction, a misaligned grad_y the one atomic kernel; both
    within the bound, the former bitwise repeatable."""
    from vit_adapter_b200 import _cabi
    C, H, W = 64, 8, 16
    x, gy, w, b = _dw_inputs(dtype, C, H, W, seed=11)
    gy_mis = at_offset(gy, 4 if dtype == torch.float32 else 2)
    refs, sums = _dw_reference(x, gy, w, b, H, W)
    results = {}
    for path, g, expect, launches in (('run', gy, wgrad_run(dtype), 2), ('atomic', gy_mis, wgrad_atomic(dtype), 1)):
        n0 = _cabi.launch_count()
        (_, gw, gb), names = kernels_launched(lambda: _cabi.dwconv_backward(x, w, g, H, W, need_input=False))
        assert _cabi.launch_count() - n0 == launches
        assert_kernels(names, expect, '%s grad_w' % path)
        depth = _wgrad_depth(C, H, W, path == 'run')
        assert_within(gw, refs[3], depth * U32 * sums[3], '%s grad_w' % path)
        assert_within(gb, refs[4], depth * U32 * sums[4], '%s grad_b' % path)
        results[path] = (gw, gb)
    _, gw2, gb2 = _cabi.dwconv_backward(x, w, gy, H, W, need_input=False)
    assert torch.equal(results['run'][0], gw2) and torch.equal(results['run'][1], gb2)


CROSS_SHAPES = [(64, 4, 8), (128, 20, 24)]


@pytest.mark.parametrize('shape', CROSS_SHAPES, ids=['C%d-%dx%d' % s for s in CROSS_SHAPES])
@pytest.mark.parametrize('dtype', [torch.float32, torch.bfloat16, torch.float16], ids=['f32', 'bf16', 'f16'])
def test_dwconv_families_are_bitwise_identical(dtype, shape):
    """Every family starts from the bias (or zero) and applies the nine taps in the same row-major order with one IEEE
    fp32 FMA each (FFMA in the generic kernel, FFMA2 lanes in the run and tile kernels): for finite inputs, forward and
    grad_x agree bit for bit. A difference is an indexing bug in one family."""
    from vit_adapter_b200 import _cabi
    C, H, W = shape
    x, gy, w, b = _dw_inputs(dtype, C, H, W, seed=5)
    fams = (('tile64', 0), ('run', 8), ('generic', 2)) if dtype != torch.float32 else (('run', 0), ('generic', 4))
    ys, gxs = [], []
    for fam, off in fams:
        xo, gyo = at_offset(x, off), at_offset(gy, off)
        y, names = kernels_launched(lambda: _cabi.dwconv_forward(xo, w, b, H, W))
        assert_kernels(names, [_family(dtype, fam, False)], fam + ' forward')
        (gx, _, _), names = kernels_launched(lambda: _cabi.dwconv_backward(xo, w, gyo, H, W, need_weight=False))
        assert_kernels(names, [_family(dtype, fam, True)], fam + ' grad_x')
        ys.append(y)
        gxs.append(gx)
    for (fam, _), y, gx in zip(fams[1:], ys[1:], gxs[1:]):
        assert torch.equal(y, ys[0]), '%s forward differs from %s' % (fam, fams[0][0])
        assert torch.equal(gx, gxs[0]), '%s grad_x differs from %s' % (fam, fams[0][0])


def test_dwconv_module_misaligned_bf16_under_autocast():
    """The autograd path with a bf16 activation at a 2-byte offset: generic forward, atomic grad_w, and grad_x on the
    tile (autograd's grad_y is a fresh allocation)."""
    from vit_adapter_b200.adapter import DWConv
    C, H, W = 64, 4, 8
    x, gy, w, b = _dw_inputs(torch.bfloat16, C, H, W, seed=3)
    m = DWConv(C).cuda()
    with torch.no_grad():
        m.dwconv.weight.copy_(w.float())
        m.dwconv.bias.copy_(b.float())
    xo = at_offset(x, 2).requires_grad_()

    def step():
        with torch.autocast('cuda', dtype=torch.bfloat16):
            y = m(xo, H, W)
        y.backward(gy)
        return y

    y, names = kernels_launched(step)
    assert y.dtype == torch.bfloat16
    assert_kernels(names, [generic(torch.bfloat16, False), tile(torch.bfloat16, True, 16)] + wgrad_atomic(torch.bfloat16),
                   'DWConv module')
    refs, sums = _dw_reference(x, gy, w, b, H, W)
    depth = _wgrad_depth(C, H, W, False)
    assert_within(y.detach(), refs[0], 10 * U32 * sums[0], 'module y')
    assert_within(xo.grad, refs[2], 10 * U32 * sums[2], 'module grad_x')
    # the fp32 parameters receive the bf16 gradients of their bf16 casts: round to bf16, compare in bf16
    assert_within(m.dwconv.weight.grad.to(torch.bfloat16), refs[3], depth * U32 * sums[3], 'module grad_w')
    assert_within(m.dwconv.bias.grad.to(torch.bfloat16), refs[4], depth * U32 * sums[4], 'module grad_b')


# --- B. LayerNorm row kernels ---------------------------------------------------------------------------------------------
LN_COMBOS = [(torch.float32, torch.float32), (torch.float32, torch.bfloat16), (torch.bfloat16, torch.bfloat16),
             (torch.float32, torch.float16), (torch.float16, torch.float16)]
LN_CS = [124, 132, 260, 508, 516, 700, 772, 1024]   # quads per lane (VPL) 1 ... 8, all but 1024 with a ragged last quad
EPS = 1e-6


def _ln_kernels(ti, to, vpl):
    return ([kernel('adapter_ln_fwd_kernel', T_NAME[ti], T_NAME[to], vpl)],
            [kernel('adapter_ln_bwd_kernel', T_NAME[ti], T_NAME[to], vpl), kernel('adapter_ln_param_grad_kernel')])


def _ln_inputs(ti, to, rows, C, seed, residual):
    g = torch.Generator().manual_seed(seed)
    x = (3.0 * torch.randn(rows, C, generator=g) + 1.5).to(ti).cuda()
    gamma = (1 + 0.3 * torch.randn(C, generator=g)).cuda()
    beta = (0.2 * torch.randn(C, generator=g)).cuda()
    gy = torch.randn(rows, C, generator=g).to(to).cuda()
    gres = torch.randn(rows, C, generator=g).to(ti).cuda() if residual else None
    return x, gamma, beta, gy, gres


def _ln_check(ti, to, C, x, gamma, beta, gy, gres, y, stats, gx, gg, gb, what):
    """First-order rounding bounds of the row kernels, doubled to cover the second-order terms. With VPL = ceil(C / 128):
    the mean is m0 + mean(x - m0); the correction's differences, its tree of depth VPL + 7 and * (1/C) give
    (VPL + 10) units of the spread mean|x - mean|, the final add one unit of |mean|; the centred square sum is 4 VPL + 7
    deep, and eps, sqrt and the division add three roundings: rstd is within k_r = 2 VPL + 8 units relative. The
    backward's two row sums are 4 VPL + 7 deep (+ 1/C); dgamma / dbeta are sums over rows of depth
    ceil(rows / (8 CTAs)) + 64 (CTA tree, partial-row sum)."""
    rows = x.shape[0]
    vpl = -(-C // 128)
    u = U32
    xd, gd, bd, dyd = x.double(), gamma.double(), beta.double(), gy.double()
    mean = xd.mean(-1, keepdim=True)
    var = ((xd - mean) ** 2).mean(-1, keepdim=True)
    r = 1.0 / torch.sqrt(var + EPS)
    xh = (xd - mean) * r
    y_ref = layernorm_ref.layernorm(xd, gd, bd, EPS)
    gx_ref, gg_ref, gb_ref = layernorm_ref.layernorm_backward(xd, gd, EPS, dyd)
    if gres is not None:
        gx_ref = gx_ref + gres.double()

    e_mu = (vpl + 10) * u * (xd - mean).abs().mean(-1, keepdim=True) + u * mean.abs()   # absolute, per row
    e_r = (2 * vpl + 8) * u                                     # relative
    assert_within(stats[0], mean.squeeze(-1), 2 * e_mu.squeeze(-1), what + ' mean')
    assert_within(stats[1], r.squeeze(-1), 2 * e_r * r.squeeze(-1), what + ' rstd')
    acc_y = 2 * (gd.abs() * (r * e_mu + xh.abs() * (e_r + 3 * u)) + u * bd.abs())
    assert_within(y, y_ref, acc_y, what + ' y')

    e_xh = r * e_mu + xh.abs() * (e_r + 2 * u)                  # error of the recomputed xhat
    t = dyd * gd
    s1 = t.mean(-1, keepdim=True)
    s2 = (t * xh).mean(-1, keepdim=True)
    k_s = (4 * vpl + 9) * u
    e_s1 = k_s * t.abs().mean(-1, keepdim=True)
    e_s2 = k_s * (t * xh).abs().mean(-1, keepdim=True) + (t.abs() * e_xh).mean(-1, keepdim=True)
    core = t - s1 - xh * s2
    e_core = u * t.abs() + e_s1 + xh.abs() * e_s2 + s2.abs() * e_xh + 3 * u * (t.abs() + s1.abs() + (xh * s2).abs())
    acc_gx = r * e_core + r * core.abs() * (e_r + u)
    if gres is not None:
        acc_gx = acc_gx + u * (r * core.abs() + gres.double().abs())
    assert_within(gx, gx_ref, 2 * acc_gx, what + ' grad_x')
    grid = min(-(-rows // 8), 2 * _sms())
    depth = -(-rows // (8 * grid)) + 64
    acc_gg = (dyd.abs() * e_xh).sum(0) + depth * u * (dyd * xh).abs().sum(0)
    assert_within(gg, gg_ref, 2 * acc_gg, what + ' grad_gamma')
    assert_within(gb, gb_ref, depth * u * dyd.abs().sum(0), what + ' grad_beta')


@pytest.mark.parametrize('residual', [False, True], ids=['plain', 'grad_res'])
@pytest.mark.parametrize('C', LN_CS)
@pytest.mark.parametrize('combo', LN_COMBOS, ids=['%s-%s' % (SHORT[a], SHORT[b]) for a, b in LN_COMBOS])
def test_layernorm_grid(combo, C, residual):
    from vit_adapter_b200 import _cabi
    ti, to = combo
    vpl = -(-C // 128)
    fwd_k, bwd_k = _ln_kernels(ti, to, vpl)
    for rows in (1, 7, 2 * _sms() * 8 + 5):
        what = '%s->%s C=%d rows=%d%s' % (SHORT[ti], SHORT[to], C, rows, ' +grad_res' if residual else '')
        x, gamma, beta, gy, gres = _ln_inputs(ti, to, rows, C, seed=C * 10 + rows, residual=residual)
        (y, stats), names = kernels_launched(lambda: _cabi.layernorm_forward(x, gamma, beta, EPS, to))
        assert_kernels(names, fwd_k, what + ' forward')
        (gx, gg, gb), names = kernels_launched(lambda: _cabi.layernorm_backward(gy, x, gamma, stats, gres))
        assert_kernels(names, bwd_k, what + ' backward')
        assert y.dtype == to and gx.dtype == ti
        _ln_check(ti, to, C, x, gamma, beta, gy, gres, y, stats, gx, gg, gb, what)
        if residual and rows > 8:
            _, gg2, gb2 = _cabi.layernorm_backward(gy, x, gamma, stats, gres)
            assert torch.equal(gg, gg2) and torch.equal(gb, gb2), what + ': parameter gradients not bitwise repeatable'


def test_layernorm_module_bf16_residual_fold():
    """apply_norm_residual on a bf16 activation under bf16 autocast (C = 768): the (bf16, bf16) kernels with the residual
    branch's bf16 gradient staged through shared memory, as a model reaches them."""
    from vit_adapter_b200.adapter.adapter_modules import apply_norm_residual
    C, rows = 768, 2 * 197 + 3
    x, gamma, beta, gy, gres = _ln_inputs(torch.bfloat16, torch.bfloat16, rows, C, seed=768, residual=True)
    m = nn.LayerNorm(C, eps=EPS).cuda()
    with torch.no_grad():
        m.weight.copy_(gamma)
        m.bias.copy_(beta)
    xl = x.clone().requires_grad_()

    def step():
        with torch.autocast('cuda', dtype=torch.bfloat16):
            y, xr = apply_norm_residual(m, xl)
        ((y.float() * gy.float()).sum() + (xr.float() * gres.float()).sum()).backward()
        return y

    y, names = kernels_launched(step)
    fwd_k, bwd_k = _ln_kernels(torch.bfloat16, torch.bfloat16, 6)
    assert y.dtype == torch.bfloat16
    assert_kernels(names, fwd_k + bwd_k, 'module')
    from vit_adapter_b200 import _cabi
    _, stats = _cabi.layernorm_forward(x, gamma, beta, EPS, torch.bfloat16)
    _ln_check(torch.bfloat16, torch.bfloat16, C, x, gamma, beta, gy, gres, y.detach(), stats, xl.grad, m.weight.grad,
              m.bias.grad, 'module')


def _conditioning_rows(kind, rows, C, g):
    if kind == 'offset':   # |mean| / std from 1e3 to 1e4
        std = torch.logspace(-1, 0, rows).unsqueeze(1)
        return 1e3 + std * torch.randn(rows, C, generator=g)
    if kind == 'constant':
        return (10 * torch.randn(rows, 1, generator=g)).expand(rows, C).contiguous()
    x = torch.randn(rows, C, generator=g)   # one large outlier per row
    x[torch.arange(rows), torch.randint(0, C, (rows,), generator=g)] = 1e4 * (1 + torch.rand(rows, generator=g))
    return x


@pytest.mark.parametrize('kind', ['offset', 'constant', 'outlier'])
def test_layernorm_conditioning_no_worse_than_torch(kind):
    """Badly conditioned rows: the row kernel's largest error against fp64 is at most 4x that of torch's own fp32
    LayerNorm (Welford statistics), plus a floor of 2^-20 of the largest reference value."""
    from vit_adapter_b200 import _cabi
    C, rows = 768, 64
    g = torch.Generator().manual_seed(17)
    x = _conditioning_rows(kind, rows, C, g).cuda()
    gamma = (1 + 0.3 * torch.randn(C, generator=g)).cuda()
    beta = (0.2 * torch.randn(C, generator=g)).cuda()
    gy = torch.randn(rows, C, generator=g).cuda()
    y_ref = layernorm_ref.layernorm(x.double(), gamma.double(), beta.double(), EPS)
    gx_ref = layernorm_ref.layernorm_backward(x.double(), gamma.double(), EPS, gy.double())[0]
    y, stats = _cabi.layernorm_forward(x, gamma, beta, EPS, torch.float32)
    gx, _, _ = _cabi.layernorm_backward(gy, x, gamma, stats)
    xt = x.clone().requires_grad_()
    yt = F.layer_norm(xt, (C,), gamma, beta, EPS)
    yt.backward(gy)
    for name, mine, theirs, ref in (('y', y, yt.detach(), y_ref), ('grad_x', gx, xt.grad, gx_ref)):
        e_k = float((mine.double() - ref).abs().max())
        e_t = float((theirs.double() - ref).abs().max())
        floor = 2.0 ** -20 * float(ref.abs().max())
        assert e_k <= 4 * e_t + floor, '%s rows, %s: kernel error %.3e, torch %.3e, floor %.3e' % (kind, name, e_k, e_t, floor)


# --- C. 64-bit offsets ----------------------------------------------------------------------------------------------------
def test_more_than_2pow31_elements():
    """A bf16 convolution and a bf16 LayerNorm over more than 2^31 elements: the last image / rows are bitwise what the
    same kernels compute for them alone."""
    from vit_adapter_b200 import _cabi
    Bn, C, H, W = 98, 1024, 64, 64
    n = 21 * (H // 2) * (W // 2)
    conv_elems = Bn * n * C
    rows, LC = (1 << 21) + 8, 1024
    assert conv_elems > 2 ** 31 and rows * LC > 2 ** 31
    need = max(4 * conv_elems, 5 * rows * LC) * 2
    free, _ = torch.cuda.mem_get_info()
    if free < 3 * need:
        pytest.skip('needs %.1f GB of free device memory, %.1f GB free' % (3 * need / 1e9, free / 1e9))
    gen = torch.Generator(device='cuda').manual_seed(0)
    dev = torch.device('cuda')
    try:
        x = torch.randn(Bn, n, C, generator=gen, device=dev, dtype=torch.bfloat16)
        gy = torch.randn(Bn, n, C, generator=gen, device=dev, dtype=torch.bfloat16)
        w = (torch.randn(C, 1, 3, 3, generator=gen, device=dev) / 3).to(torch.bfloat16)
        b = torch.randn(C, generator=gen, device=dev).to(torch.bfloat16)
        y, names = kernels_launched(lambda: _cabi.dwconv_forward(x, w, b, H, W))
        assert_kernels(names, [tile(torch.bfloat16, False, 16)], 'large forward')
        y_last = y[-1].clone()
        del y
        (gx, _, _), names = kernels_launched(lambda: _cabi.dwconv_backward(x, w, gy, H, W, need_weight=False))
        assert_kernels(names, [tile(torch.bfloat16, True, 16)], 'large grad_x')
        gx_last = gx[-1].clone()
        del gx
        x1, gy1 = x[-1:].clone(), gy[-1:].clone()
        del x, gy
        assert torch.equal(_cabi.dwconv_forward(x1, w, b, H, W)[0], y_last)
        assert torch.equal(_cabi.dwconv_backward(x1, w, gy1, H, W, need_weight=False)[0][0], gx_last)
        del x1, gy1, y_last, gx_last

        tail = 64
        x = torch.randn(rows, LC, generator=gen, device=dev, dtype=torch.bfloat16)
        gamma = 1 + 0.3 * torch.randn(LC, generator=gen, device=dev)
        beta = 0.2 * torch.randn(LC, generator=gen, device=dev)
        y, stats = _cabi.layernorm_forward(x, gamma, beta, EPS, torch.bfloat16)
        y_last, stats_last = y[-tail:].clone(), stats[:, -tail:].clone()
        del y
        gy = torch.randn(rows, LC, generator=gen, device=dev, dtype=torch.bfloat16)
        gres = torch.randn(rows, LC, generator=gen, device=dev, dtype=torch.bfloat16)
        gx, _, _ = _cabi.layernorm_backward(gy, x, gamma, stats, gres)
        gx_last = gx[-tail:].clone()
        xs, gys, gress = x[-tail:].clone(), gy[-tail:].clone(), gres[-tail:].clone()
        del gx, x, gy, gres, stats
        y1, st1 = _cabi.layernorm_forward(xs, gamma, beta, EPS, torch.bfloat16)
        assert torch.equal(y1, y_last) and torch.equal(st1, stats_last)
        assert torch.equal(_cabi.layernorm_backward(gys, xs, gamma, st1, gress)[0], gx_last)
    finally:
        torch.cuda.synchronize()
        torch.cuda.empty_cache()
