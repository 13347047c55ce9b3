"""Every launch path of the plain deformable-attention sampling op (msda_forward / msda_backward: csrc/msda_fwd.cu and
csrc/msda_bwd.cu) against the fp64 C oracle (oracle/msda_oracle.c).

The launchers pick a kernel from the dtype, D, (L, P), the min-CTA tuning keys, the 32-byte-lane switch and the
alignment of seven pointers. Each case names the kernels it must launch, and `kernels_launched` checks that exactly those
ran. tests/test_msda_paths_cpu.py checks that the cases name every plain-path kernel the library compiles.

Reference: the oracle in fp64 on the inputs as the kernels see them (value and grad_out rounded to the I/O dtype, then
widened). Locations are dyadic: multiples of 2^-12 with |loc| * 2^12 * max(H, W) < 2^23. Then fmaf(loc, H, -0.5) is
exact in fp32, the kernels and the oracle pick the same corners and fractions, and the bilinear weights (products of two
12-bit fractions) are exact too. So the location gradient, which jumps at texel edges, is comparable everywhere.

Bounds, elementwise (kernel_paths.assert_within): |out - ref| <= u_out |ref| + (1 + u_out) gamma_n S + floor, where S is
the sum of |terms| of the exact result, gamma_n = n u / (1 - n u) and u = 2^-24 (fp32 arithmetic; 2^-53 for f64). A sum of
m terms in any order is within gamma_{m-1} S, and k roundings in each term's products add gamma_k, so n = m - 1 + k:
    out         m = 4 L P (corners x points)     k = 2 (w * a, then * v)                                 n = 4 L P + 1
    grad_value  m = samples that reach the row    k = 2 (w * a, then * grad_out)                          n = m + 1
    grad_aw     m = 4 D (corners x channels)      k = 2 (grad_out * v, then * w)                          n = 4 D + 1
    grad_loc    m = 4 D                           k = 4 (grad_out * v, * fraction, * W or H, * a)          n = 4 D + 3
Differences of corner values count as additions. S of out, grad_value and grad_aw is the oracle on |value|, |aw| and
|grad_out|: the bilinear weights are non-negative. grad_loc's S is W |a| sum_c |grad_out_c| sum_corners |v_c| (H for y),
an upper bound because the fractions are <= 1.
"""
import re

import pytest
import torch

from kernel_paths import assert_within, at_offset, kernel, kernels_launched
from oracle import c_oracle

pytestmark = pytest.mark.gpu

F32, BF16, F16, F64 = torch.float32, torch.bfloat16, torch.float16, torch.float64
T_NAME = {F32: 'float', BF16: '__nv_bfloat16', F16: '__half', F64: 'double'}
SHORT = {F32: 'f32', BF16: 'bf16', F16: 'f16', F64: 'f64'}
FRAC_BITS = 12
N, M, LQ = 2, 2, 37   # 37 queries: the last chunk of every CTA split is partial


# --- the kernels a call must launch ----------------------------------------------------------------------------------------
def _acc(T):
    return 'double' if T == F64 else 'float'


def fwd_vec(T, G, LT, PT, minb, lane_bytes=16):
    return ('msda_fwd_vec_kernel', (T_NAME[T], G, LT, PT, minb, lane_bytes, 'false', 2))


def bwd_vec(T, G, LT, PT, minb, packed=False):
    return ('msda_bwd_vec_kernel', (T_NAME[T], G, LT, PT, minb, 'false', 'true' if packed else 'false', 2, 'false'))


def fwd_generic(T):
    return ('msda_fwd_generic_kernel', (T_NAME[T], _acc(T)))


def bwd_generic(T):
    return ('msda_bwd_generic_kernel', (T_NAME[T], _acc(T), _acc(T)))


def cvt(T, vector=True):
    return ('msda_cvt_f32_bf16_kernel' if vector else 'msda_cvt_f32_bf16_scalar_kernel', (T_NAME[T],))


SORTED = [re.compile(r'\bmsda_sort_part_kernel\s*<'), re.compile(r'\bmsda_sort_prefix_kernel\b'),
          re.compile(r'\bmsda_sort_part_kernel\s*<'), re.compile(r'\bmsda_bwd_sorted_kernel\s*<')]


def _static(L, P):
    return (L, P) if (L, P) in ((3, 4), (1, 4)) else (0, 0)


def forward_kernel(T, D, L, P, minb=0, wide=False):
    """What msda_forward launches with 32-byte aligned tensors (msda_abi.cu, msda_fwd.cu launch_vec / launch_wide_g)."""
    LT, PT = _static(L, P)
    cpl = 4 if T == F32 else 8
    G = D // cpl
    if T == F64 or D % cpl or G not in (2, 4, 8, 16, 32):
        return fwd_generic(T)
    if wide and T == F32 and D // 8 in (2, 4, 8):
        return fwd_vec(T, D // 8, LT, PT, 3 if minb == 3 and LT else 4, 32)
    if G in (4, 8, 16) and minb in (3, 6):
        return fwd_vec(T, G, LT, PT, minb)
    return fwd_vec(T, G, LT, PT, 3 if T != F32 and G in (4, 8, 16) else 4)


def backward_kernels(T, D, L, P, minb=0):
    """What msda_backward launches with 16-byte aligned tensors: the scatter, then the convert of a 16-bit grad_value."""
    LT, PT = _static(L, P)
    G = D // 4
    if T == F64 or D % 4 or G not in (2, 4, 8, 16, 32):
        k = bwd_generic(T)
    else:
        k = bwd_vec(T, G, LT, PT, minb if G in (4, 8, 16) and minb in (2, 4) else 3)
    return [k] + ([cvt(T)] if T in (BF16, F16) else [])


def assert_msda_kernels(names, expected, what):
    """The sampling op's kernels that ran are exactly `expected`, in order ((name, args) or a regex)."""
    ours = [n for n in names if 'msda_' in n]
    pats = [e if isinstance(e, re.Pattern) else kernel(e[0], *e[1]) for e in expected]
    assert len(ours) == len(pats) and all(p.search(n) for p, n in zip(pats, ours)), \
        '%s: launched %s, expected %s' % (what, ours, [p.pattern for p in pats])


# --- inputs, reference, bounds ---------------------------------------------------------------------------------------------
def dyadic_locations(g, n, Lq, m, shapes, P):
    """[n, Lq, m, L, P, 2] float64 multiples of 2^-12 in [-0.25, 1.25], with these on every level and axis of side s:
    0 and 1 (h_im = -0.5 and s - 0.5) and, when s is a power of two, the texel edges h_im = -1, 0, 1, s/2, s - 1 and s."""
    L = len(shapes)
    one = 1 << FRAC_BITS
    loc = torch.randint(-one // 4, 5 * one // 4 + 1, (n, Lq, m, L, P, 2), generator=g).double() / one
    for l, (H, W) in enumerate(shapes):
        for axis, s in ((0, W), (1, H)):
            special = [0.0, 1.0]
            if s & (s - 1) == 0:
                special += [(e + 0.5) / s for e in (-1, 0, 1, s // 2, s - 1, s)]
            v = loc[:, :, :, l, :, axis].flatten()
            i = torch.arange(v.numel())
            pick = (i % 4 == 0) | (i % 4 == 1 + axis)      # both coordinates special on every fourth point
            v[pick] = torch.tensor(special, dtype=torch.float64)[(i[pick] // 4 + l) % len(special)]
            loc[:, :, :, l, :, axis] = v.view(loc.shape[:3] + (P,))
    side = max(max(s) for s in shapes)
    assert bool(((loc * one).frac() == 0).all()) and bool((loc.abs() * one * side < 2 ** 23).all())
    return loc


def problem(T, D, shapes, P, seed, n=N, m=M, Lq=LQ):
    """CPU inputs: value / grad_out in T, dyadic locations and signed attention weights in f32 (f64 for T = f64)."""
    g = torch.Generator().manual_seed(seed)
    shapes_t = torch.as_tensor(shapes, dtype=torch.long)
    lsi = torch.cat((shapes_t.new_zeros((1,)), shapes_t.prod(1).cumsum(0)[:-1]))
    S = int(shapes_t.prod(1).sum())
    F = F64 if T == F64 else F32
    value = torch.randn(n, S, m, D, generator=g).to(T)
    go = torch.randn(n, Lq, m * D, generator=g).to(T)
    aw = torch.randn(n, Lq, m, len(shapes), P, generator=g).to(F)
    loc = dyadic_locations(g, n, Lq, m, shapes, P).to(F)
    return dict(value=value, shapes=shapes_t, lsi=lsi, loc=loc, aw=aw, grad_out=go)


def _corners(pb):
    """Per sample and corner (h_low / h_high x w_low / w_high): token index and whether the oracle reads it."""
    shapes, lsi, loc = pb['shapes'], pb['lsi'], pb['loc'].double()
    L = shapes.shape[0]
    H = shapes[:, 0].view(1, 1, 1, L, 1)
    W = shapes[:, 1].view(1, 1, 1, L, 1)
    h = loc[..., 1] * H - 0.5
    w = loc[..., 0] * W - 0.5
    inside = (h > -1) & (w > -1) & (h < H) & (w < W)
    h0, w0 = h.floor().long(), w.floor().long()
    out = []
    for dh, dw in ((0, 0), (0, 1), (1, 0), (1, 1)):
        hh, ww = h0 + dh, w0 + dw
        ok = inside & (hh >= 0) & (hh < H) & (ww >= 0) & (ww < W)
        out.append(((lsi.view(1, 1, 1, L, 1) + hh * W + ww).clamp(0, int(shapes.prod(1).sum()) - 1), ok))
    return out


def reference(pb, extra=0, packed=False):
    """fp64 (out, grad_value, grad_loc, grad_aw) and the gamma_n * S of each (see the module docstring). `extra`: more
    roundings in every term. `packed`: grad_value is summed in its 16-bit dtype (bwd_packed16), each contribution rounded
    to it, so its m + 1 roundings are of that dtype's unit."""
    T = pb['value'].dtype
    u = 2.0 ** -53 if T == F64 else 2.0 ** -24
    v, go, loc, aw = pb['value'].double(), pb['grad_out'].double(), pb['loc'].double(), pb['aw'].double()
    sh, lsi = pb['shapes'], pb['lsi']
    n_, S, m, D = v.shape
    Lq, L, P = loc.shape[1], loc.shape[3], loc.shape[4]
    out = c_oracle.forward(v, sh, lsi, loc, aw)
    gv, gl, ga = c_oracle.backward(v, sh, lsi, loc, aw, go)
    s_out = c_oracle.forward(v.abs(), sh, lsi, loc, aw.abs())
    s_gv, _, s_ga = c_oracle.backward(v.abs(), sh, lsi, loc, aw.abs(), go.abs())

    count = torch.zeros(n_ * S * m, dtype=torch.float64)
    vgo = torch.zeros(loc.shape[:-1], dtype=torch.float64)
    b = torch.arange(n_).view(n_, 1, 1, 1, 1).expand(loc.shape[:-1])
    hd = torch.arange(m).view(1, 1, m, 1, 1).expand(loc.shape[:-1])
    ago = go.abs().view(n_, Lq, m, 1, 1, D)
    for tok, ok in _corners(pb):
        count.index_add_(0, ((b * S + tok) * m + hd)[ok], torch.ones(int(ok.sum()), dtype=torch.float64))
        vgo += ok * (v.abs()[b, tok, hd] * ago).sum(-1)
    wh = torch.stack((sh[:, 1], sh[:, 0]), -1).double().view(1, 1, 1, L, 1, 2)
    s_gl = wh * (aw.abs() * vgo).unsqueeze(-1)

    def gamma(n, u=u):
        return n * u / (1 - n * u)
    n_gv = count.view(n_, S, m, 1) + 1 + extra
    acc = (gamma(4 * L * P + 1 + extra) * s_out,
           (gamma(n_gv) + (gamma(n_gv, 2.0 ** -8 if T == BF16 else 2.0 ** -11) if packed else 0)) * s_gv,
           gamma(4 * D + 3 + extra) * s_gl,
           gamma(4 * D + 1 + extra) * s_ga)
    return (out, gv, gl, ga), acc


def check(pb, results, what, packed=False):
    refs = reference(pb, packed=packed)
    for name, got, ref, acc in zip(('out', 'grad_value', 'grad_loc', 'grad_aw'), results, *refs):
        assert got.dtype == (pb['value'].dtype if name in ('out', 'grad_value') else pb['loc'].dtype)
        assert_within(got.cpu(), ref, acc, '%s %s' % (what, name))


def _device(pb):
    return {k: v.cuda() for k, v in pb.items()}


def run_python(pb):
    """out, grad_value, grad_loc, grad_aw through _cabi.forward / backward (fresh, allocator-aligned buffers)."""
    from vit_adapter_b200 import _cabi
    d = _device(pb)
    out = _cabi.forward(d['value'], d['shapes'], d['lsi'], d['loc'], d['aw'], 64)
    return (out,) + _cabi.backward(d['value'], d['shapes'], d['lsi'], d['loc'], d['aw'], d['grad_out'], 64)


def run_cabi(pb, off):
    """The same through the C ABI, each tensor `off.get(name, 0)` bytes past an allocator (256-byte) boundary; outputs
    start NaN-filled."""
    import ctypes
    from vit_adapter_b200 import _cabi
    lib = _cabi.load()
    d = _device(pb)
    T = d['value'].dtype
    put = {k: at_offset(d[k], off.get(k, 0)) for k in ('value', 'loc', 'aw', 'grad_out')}
    nan = float('nan')
    out = at_offset(torch.full(d['grad_out'].shape, nan, dtype=T, device='cuda'), off.get('out', 0))
    gv = at_offset(torch.full(d['value'].shape, nan, dtype=T, device='cuda'), off.get('grad_value', 0))
    gl = at_offset(torch.full_like(d['loc'], nan), off.get('grad_loc', 0))
    ga = at_offset(torch.full_like(d['aw'], nan), off.get('grad_aw', 0))
    dims = _cabi._dims(d['value'], d['shapes'], d['loc'])
    code = _cabi._DTYPES[T]
    ws_bytes = lib.msda_backward_workspace_bytes(ctypes.byref(dims), code)
    ws = at_offset(torch.zeros(ws_bytes, dtype=torch.uint8, device='cuda'), off.get('workspace', 0)) if ws_bytes else None
    stream = torch.cuda.current_stream().cuda_stream
    rc = lib.msda_forward(ctypes.byref(dims), code, put['value'].data_ptr(), d['shapes'].data_ptr(), d['lsi'].data_ptr(),
                          put['loc'].data_ptr(), put['aw'].data_ptr(), out.data_ptr(), stream)
    assert rc == 0, lib.msda_last_error()
    rc = lib.msda_backward(ctypes.byref(dims), code, put['value'].data_ptr(), d['shapes'].data_ptr(), d['lsi'].data_ptr(),
                           put['loc'].data_ptr(), put['aw'].data_ptr(), put['grad_out'].data_ptr(), gv.data_ptr(), gl.data_ptr(),
                           ga.data_ptr(), ws.data_ptr() if ws is not None else None, ws_bytes, stream)
    assert rc == 0, lib.msda_last_error()
    return out, gv, gl, ga


class tuned:
    """msda_set_tuning keys for the duration of a block, restored to 0 (the heuristic) afterwards."""

    def __init__(self, **kv):
        self.kv = kv

    def __enter__(self):
        from vit_adapter_b200 import _cabi
        try:
            _cabi.set_tuning(**self.kv)
        except BaseException:
            self.__exit__()
            raise

    def __exit__(self, *exc):
        from vit_adapter_b200 import _cabi
        _cabi.set_tuning(**{k: 0 for k in self.kv})
        return False


# --- A. launch matrix ------------------------------------------------------------------------------------------------------
LEVELS = {
    'L3P4': ([(8, 8), (4, 6), (3, 2)], 4),          # static (3, 4)
    'L1P4': ([(16, 8)], 4),                         # static (1, 4)
    'L2P3': ([(8, 8), (5, 3)], 3),                  # runtime (L, P)
    'L16P2': ([(1, 1), (2, 3), (4, 4), (3, 5), (8, 2), (1, 7), (6, 6), (2, 2), (5, 1), (4, 8), (7, 3), (1, 2), (3, 3),
               (2, 6), (8, 8), (1, 1)], 2),          # MSDA_MAX_LEVELS ragged levels
    'L1P32': ([(8, 8)], 32),                        # more points than lanes in a group
}
MINB = (('minb-default', 0, 0), ('minb-lo', 3, 2), ('minb-hi', 6, 4))   # (fwd_min_ctas, bwd_min_ctas)

# (id, dtype, D, levels, fwd_min_ctas, bwd_min_ctas, fwd_chunk = bwd_chunk (0 = heuristic), fwd_wide)
CASES = []
for _T, _Ds in ((F32, (8, 16, 32, 64, 128)), (BF16, (8, 16, 32, 64, 128, 256)), (F16, (8, 16, 32, 64, 128, 256))):
    for _D in _Ds:
        for _lv in ('L3P4', 'L1P4', 'L2P3'):
            for _mk, _fm, _bm in MINB:
                CASES.append(('%s-D%d-%s-%s' % (SHORT[_T], _D, _lv, _mk), _T, _D, _lv, _fm, _bm, 0, False))
for _D in (16, 32, 64):
    for _lv in ('L3P4', 'L1P4', 'L2P3'):
        for _mk, _fm in (('minb-default', 0), ('minb-lo', 3)):
            CASES.append(('f32-wide-D%d-%s-%s' % (_D, _lv, _mk), F32, _D, _lv, _fm, 0, 0, True))
for _T in (F32, BF16, F16, F64):
    for _D in (24, 30):
        CASES.append(('%s-D%d-generic' % (SHORT[_T], _D), _T, _D, 'L3P4', 0, 0, 0, False))
    CASES.append(('%s-D32-L16P2' % SHORT[_T], _T, 32, 'L16P2', 0, 0, 0, False))
CASES += [
    ('f64-D32-L3P4', F64, 32, 'L3P4', 0, 0, 0, False),
    ('f32-D32-L1P32', F32, 32, 'L1P32', 0, 0, 0, False),
    ('bf16-D64-L1P32', BF16, 64, 'L1P32', 0, 0, 0, False),
    # short chunks: several CTAs per (b, m), the last one partial
    ('f32-D128-L2P3-chunk8', F32, 128, 'L2P3', 0, 0, 8, False),
    ('f16-D64-L1P4-chunk16', F16, 64, 'L1P4', 0, 0, 16, False),
    ('bf16-D24-L3P4-chunk8', BF16, 24, 'L3P4', 0, 0, 8, False),
]


def case_kernels(case):
    _, T, D, lv, fm, bm, _, wide = case
    shapes, P = LEVELS[lv]
    return [forward_kernel(T, D, len(shapes), P, fm, wide)] + backward_kernels(T, D, len(shapes), P, bm)


@pytest.mark.parametrize('case', CASES, ids=[c[0] for c in CASES])
def test_launch_matrix(case):
    cid, T, D, lv, fm, bm, chunk, wide = case
    shapes, P = LEVELS[lv]
    pb = problem(T, D, shapes, P, seed=D * 100 + len(shapes) * 10 + P)
    with tuned(fwd_min_ctas=fm, bwd_min_ctas=bm, fwd_chunk=chunk, bwd_chunk=chunk, fwd_wide=2 if wide else 0):
        res, names = kernels_launched(lambda: run_python(pb))
    assert_msda_kernels(names, case_kernels(case), cid)
    check(pb, res, cid)


# --- B. pointer alignment through the C ABI --------------------------------------------------------------------------------
def _align_cases():
    """(id, dtype, D, {pointer: byte offset}, tuning, expected kernels): D = 32, (L, P) = (3, 4)."""
    cases = []
    f_vec, b_vec = forward_kernel(F32, 32, 3, 4), backward_kernels(F32, 32, 3, 4)
    f_gen, b_gen = fwd_generic(F32), [bwd_generic(F32)]
    for p, f, b in (('value', f_gen, b_gen), ('out', f_gen, b_vec), ('grad_out', f_vec, b_gen), ('loc', f_gen, b_gen),
                    ('grad_loc', f_vec, b_gen), ('aw', f_vec, b_vec), ('grad_aw', f_vec, b_vec), ('grad_value', f_vec, b_gen)):
        cases.append(('f32-%s+4' % p, F32, 32, {p: 4}, {}, [f] + b))
    # 32-byte lanes need 32-byte aligned value and out: 16 bytes past a boundary takes the 16-byte-lane forward
    for p in ('value', 'out'):
        cases.append(('f32-wide-%s+16' % p, F32, 32, {p: 16}, {'fwd_wide': 2}, [f_vec] + b_vec))
    cases.append(('f32-wide-aligned', F32, 32, {}, {'fwd_wide': 2}, [forward_kernel(F32, 32, 3, 4, wide=True)] + b_vec))
    for T in (BF16, F16):
        s = SHORT[T]
        f_vec, b_vec = forward_kernel(T, 32, 3, 4), [bwd_vec(T, 8, 3, 4, 3)]
        f_gen, b_gen = fwd_generic(T), [bwd_generic(T)]
        for p, offs, f, b in (('value', (2, 8), f_gen, b_gen), ('out', (2, 8), f_gen, b_vec),
                              ('grad_out', (2, 8), f_vec, b_gen), ('loc', (4,), f_gen, b_gen), ('grad_loc', (4,), f_vec, b_gen),
                              ('aw', (4,), f_vec, b_vec), ('grad_aw', (4,), f_vec, b_vec), ('workspace', (16,), f_vec, b_vec)):
            for o in offs:
                cases.append(('%s-%s+%d' % (s, p, o), T, 32, {p: o}, {}, [f] + b + [cvt(T)]))
        # grad_value is written only by the convert (fp32 scratch -> T): any element offset, scalar stores
        for o in (2, 4, 8):
            cases.append(('%s-grad_value+%d' % (s, o), T, 32, {'grad_value': o}, {}, [f_vec] + b_vec + [cvt(T, False)]))
        # packed 16-bit reductions straight into grad_value need 8-byte alignment; otherwise the fp32 scratch + convert
        cases.append(('%s-grad_value+8-packed16' % s, T, 32, {'grad_value': 8}, {'bwd_packed16': 2},
                      [f_vec, bwd_vec(T, 8, 3, 4, 3, packed=True)]))
        for o in (2, 4):
            cases.append(('%s-grad_value+%d-packed16' % (s, o), T, 32, {'grad_value': o}, {'bwd_packed16': 2},
                          [f_vec] + b_vec + [cvt(T, False)]))
        for D in (32, 64):
            cases.append(('%s-D%d-grad_value+2-sorted' % (s, D), T, D, {'grad_value': 2}, {'bwd_sorted': 2},
                          [forward_kernel(T, D, 3, 4)] + SORTED + [cvt(T, False)]))
    return cases


ALIGN_CASES = _align_cases()


@pytest.mark.parametrize('case', ALIGN_CASES, ids=[c[0] for c in ALIGN_CASES])
def test_pointer_alignment(case):
    cid, T, D, off, tuning, expected = case
    shapes, P = LEVELS['L3P4']
    pb = problem(T, D, shapes, P, seed=7)
    with tuned(**tuning):
        res, names = kernels_launched(lambda: run_cabi(pb, off))
    assert_msda_kernels(names, expected, cid)
    check(pb, res, cid, packed=tuning.get('bwd_packed16') == 2 and 'grad_value' in off and off['grad_value'] % 8 == 0)


@pytest.mark.parametrize('offset', [2, 8])
@pytest.mark.parametrize('T', [BF16, F16], ids=['bf16', 'f16'])
def test_fused_backward_16bit_grad_value_at_an_element_offset(T, offset):
    """msda_backward_fused converts its fp32 scratch into a grad_value that is only element-aligned. Locations
    ref + offset / (W, H) are dyadic on power-of-two levels. The reference takes the exact softmax; the kernel's fp32
    softmax of logits within 8 of their maximum (the difference, expf, a sum of L P terms, the division) is within
    L P + 32 roundings of it, which every grad_value term inherits."""
    import ctypes
    from vit_adapter_b200 import _cabi
    lib = _cabi.load()
    shapes, P, D, Lq = [(8, 8), (4, 4), (2, 2)], 4, 32, LQ
    L = len(shapes)
    g = torch.Generator().manual_seed(offset)
    pb = problem(T, D, shapes, P, seed=11)
    ref_pts = torch.randint(0, 4097, (1, Lq, 1, 2), generator=g).float() / 4096
    offs = torch.randint(-16, 17, (N, Lq, M, L, P, 2), generator=g).float() / 8
    logits = torch.randn(N, Lq, M, L * P, generator=g).clamp(-4, 4)
    wh = torch.tensor([[w, h] for h, w in shapes], dtype=torch.float32).view(1, 1, 1, L, 1, 2)
    pb['loc'] = ref_pts.view(1, Lq, 1, 1, 1, 2) + offs / wh
    assert bool(((pb['loc'].double() * 4096).frac() == 0).all())
    pb['aw'] = torch.softmax(logits.double(), -1).view(N, Lq, M, L, P).float()
    d = _device(pb)
    dr, do, dl = ref_pts.cuda(), offs.cuda(), logits.cuda()
    gv = at_offset(torch.full(d['value'].shape, float('nan'), dtype=T, device='cuda'), offset)
    g_off, g_log = torch.empty_like(do), torch.empty_like(dl)
    dims = _cabi._dims(d['value'], d['shapes'], d['loc'])
    ws_bytes = lib.msda_backward_fused_workspace_bytes(ctypes.byref(dims), _cabi._DTYPES[T], 1, 1, 2, 0)
    ws = torch.empty(ws_bytes, dtype=torch.uint8, device='cuda')

    def call():
        rc = lib.msda_backward_fused(ctypes.byref(dims), _cabi._DTYPES[T], d['value'].data_ptr(), d['shapes'].data_ptr(),
                                     d['lsi'].data_ptr(), dr.data_ptr(), 1, 1, do.data_ptr(), dl.data_ptr(), 0, 0,
                                     d['grad_out'].data_ptr(), gv.data_ptr(), g_off.data_ptr(), g_log.data_ptr(), ws.data_ptr(),
                                     ws_bytes, torch.cuda.current_stream().cuda_stream)
        assert rc == 0, lib.msda_last_error()

    _, names = kernels_launched(call)
    fused = ('msda_bwd_vec_kernel', (T_NAME[T], 8, 3, 4, 3, 'true', 'false', 2, 'false'))
    assert_msda_kernels(names, [fused, cvt(T, False)], 'fused grad_value+%d' % offset)
    (_, ref_gv, _, _), (_, acc_gv, _, _) = reference(pb, extra=L * P + 32)
    assert_within(gv.cpu(), ref_gv, acc_gv, 'fused grad_value+%d' % offset)


# --- C. the largest image check_dims accepts -------------------------------------------------------------------------------
# (id, M, D, level 0): S * M * D just below the 2^29 of check_dims, a small 8 x 8 level 1 at the end of every image. The
# kernels address inside an image with 32-bit byte offsets: in f32 the level-1 rows of the first shape sit just below
# 2^31 bytes into their image; with N = 2 the second image lies beyond 2^31 bytes from the start of the tensor in f32
# (beyond 2^32 in f64, which takes the generic kernels); bf16 accumulates in an fp32 scratch with the f32 offsets.
LARGEST = [('M1-D32-4095x4096', 1, 32, (4095, 4096)), ('M16-D64-720x720', 16, 64, (720, 720))]


@pytest.mark.parametrize('T', [F32, BF16, F64], ids=['f32', 'bf16', 'f64'])
@pytest.mark.parametrize('shape', LARGEST, ids=[s[0] for s in LARGEST])
def test_largest_image(shape, T):
    """Level 0 is NaN and every sample on it is out of range; level-1 samples are dyadic and in range. The reference is the
    oracle on the same problem with level 0 shrunk to 1 x 1; level 0 of grad_value must be exactly zero."""
    from vit_adapter_b200 import _cabi
    _, m, D, (H0, W0) = shape
    P, big = 4, H0 * W0
    S = big + 64
    assert 0.98 * 2 ** 29 < S * m * D < 2 ** 29
    es = torch.tensor([], dtype=T).element_size()
    need = 2 * N * S * m * D * es + (N * S * m * D * 4 if T == BF16 else 0)   # value + grad_value (+ fp32 scratch)
    free, _ = torch.cuda.mem_get_info()
    if free < need + (2 << 30):
        pytest.skip('needs %.1f GB of free device memory, %.1f GB free' % (need / 1e9, free / 1e9))
    pb = problem(T, D, [(1, 1), (8, 8)], P, seed=D, m=m)
    loc = pb['loc'].view(N, LQ, m, 2, P, 2)
    loc[:, :, :, 0, :, 0] = torch.where(torch.arange(P) % 2 == 0, -1.5, 2.5).to(loc.dtype)  # outside both level 0s
    refs = reference(pb)
    d = _device(pb)
    dev = torch.device('cuda')
    torch.cuda.synchronize()
    torch.cuda.reset_peak_memory_stats()
    try:
        value = torch.full((N, S, m, D), float('nan'), dtype=T, device=dev)
        value[:, big:] = d['value'][:, 1:]
        shapes = torch.tensor([[H0, W0], [8, 8]], dtype=torch.long, device=dev)
        lsi = torch.tensor([0, big], dtype=torch.long, device=dev)

        def call():
            out = _cabi.forward(value, shapes, lsi, d['loc'], d['aw'], 64)
            return (out,) + _cabi.backward(value, shapes, lsi, d['loc'], d['aw'], d['grad_out'], 64)

        (out, gv, gl, ga), names = kernels_launched(call)
        assert_msda_kernels(names, [forward_kernel(T, D, 2, P)] + backward_kernels(T, D, 2, P), shape[0])
        del value
        assert int(torch.count_nonzero(gv[:, :big])) == 0, 'level 0 of grad_value is not exactly zero'
        gv_small = torch.cat((gv[:, :1], gv[:, big:]), 1)
        del gv
        print('\n%s %s: peak device memory %.2f GB' % (shape[0], SHORT[T], torch.cuda.max_memory_allocated() / 1e9))
        for name, got, ref, acc in zip(('out', 'grad_value', 'grad_loc', 'grad_aw'), (out, gv_small, gl, ga), *refs):
            assert_within(got.cpu(), ref, acc, '%s %s %s' % (shape[0], SHORT[T], name))
    finally:
        torch.cuda.synchronize()
        torch.cuda.empty_cache()
