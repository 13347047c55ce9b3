"""CPU-side checks of the fused entry points for box references and reference-point gradients
(msda_forward_fused_ref / msda_backward_fused_ref / msda_backward_fused_workspace_bytes): every argument is
validated before any CUDA call, so none of these needs a device. The fake device pointers are never dereferenced."""
import ctypes

import pytest

from vit_adapter_b200 import _cabi

F32, BF16, F16 = _cabi.MSDA_F32, _cabi.MSDA_BF16, _cabi.MSDA_F16
E_NULL, E_DIMS, E_ALIGN, E_WORKSPACE, E_UNSUPPORTED = -1, -2, -4, -6, -8
NEW = ('msda_forward_fused_ref', 'msda_backward_fused_ref', 'msda_backward_fused_workspace_bytes')
P = 0x10000  # a 16-byte aligned fake device address


def _dims(N=2, S=340, M=8, D=32, L=4, Lq=300, Pt=4):
    return _cabi.MsdaDims(N, S, M, D, L, Lq, Pt)


def _fwd(lib, d, dtype=F32, ref=P, rb=2, rl=4, ref_dim=4):
    return lib.msda_forward_fused_ref(ctypes.byref(d), dtype, P, P, P, ref, rb, rl, ref_dim, P, P, 0, 0, P, None)


def _bwd(lib, d, dtype=F32, ref=P, rb=2, rl=4, ref_dim=4, grad_ref=P, ws=None, ws_bytes=0):
    return lib.msda_backward_fused_ref(ctypes.byref(d), dtype, P, P, P, ref, rb, rl, ref_dim, P, P, 0, 0, P, P, P, P, grad_ref,
                                       ws, ws_bytes, None)


def _ws(lib, d, dtype, rb, rl, ref_dim, with_grad):
    return lib.msda_backward_fused_workspace_bytes(ctypes.byref(d), dtype, rb, rl, ref_dim, with_grad)


def test_new_fused_symbols_are_exported():
    lib = _cabi.load()
    for name in NEW:
        assert name in _cabi.EXPORTS
        assert getattr(lib, name) is not None


@pytest.mark.parametrize('entry', ['forward', 'backward'])
def test_reference_width_other_than_2_or_4_is_a_dims_error(entry):
    lib = _cabi.load()
    d = _dims()
    for bad in (0, 1, 3, 5, -4):
        rc = _fwd(lib, d, ref_dim=bad) if entry == 'forward' else _bwd(lib, d, ref_dim=bad, ws=P, ws_bytes=1 << 30)
        assert rc == E_DIMS, (bad, rc)
        assert b'ref_dim' in lib.msda_last_error()


@pytest.mark.parametrize('entry', ['forward', 'backward'])
def test_box_references_must_be_16_byte_aligned(entry):
    lib = _cabi.load()
    d = _dims()
    call = (lambda **kw: _fwd(lib, d, **kw)) if entry == 'forward' else (lambda **kw: _bwd(lib, d, ws=P, ws_bytes=1 << 30, **kw))
    assert call(ref=P + 8) == E_ALIGN
    assert b'16-byte' in lib.msda_last_error()
    # points keep their 8-byte requirement
    assert call(ref=P + 4, ref_dim=2) == E_ALIGN
    assert b'8-byte' in lib.msda_last_error()


def test_reference_broadcast_and_null_are_checked():
    lib = _cabi.load()
    d = _dims()
    assert _fwd(lib, d, rb=3) == E_DIMS          # neither 1 nor N
    assert _fwd(lib, d, rl=2) == E_DIMS          # neither 1 nor L
    assert _fwd(lib, d, ref=None) == E_NULL


def test_reference_broadcast_is_checked_before_the_workspace_is_sized():
    """The partials' size depends on ref_levels: a bogus value is a dims error, not a (huge) workspace request."""
    lib = _cabi.load()
    d = _dims()
    for rb, rl in ((2, -1), (2, 2), (3, 4), (-2, 4)):
        assert _bwd(lib, d, rb=rb, rl=rl) == E_DIMS, (rb, rl)
        assert b'broadcast' in lib.msda_last_error()
        assert _ws(lib, d, F32, rb, rl, 4, 1) == 0


def test_short_workspace_for_the_reference_gradient_is_rejected():
    lib = _cabi.load()
    d = _dims()
    need = _ws(lib, d, F32, 2, 4, 4, 1)
    assert need > 0
    assert _bwd(lib, d) == E_WORKSPACE                                 # f32 needs no accumulator, but the partials
    assert _bwd(lib, d, ws=P, ws_bytes=need - 4) == E_WORKSPACE
    assert _bwd(lib, d, ws=P + 8, ws_bytes=need) == E_WORKSPACE          # not 16-byte aligned
    assert b'workspace' in lib.msda_last_error()


def test_reference_gradient_output_must_be_float_aligned():
    lib = _cabi.load()
    d = _dims()
    assert _bwd(lib, d, ws=P, ws_bytes=1 << 30, grad_ref=P + 2) == E_ALIGN


def test_workspace_bytes_are_the_accumulator_then_the_aligned_partials():
    lib = _cabi.load()
    N, S, M, D, L, Lq = 2, 340, 8, 32, 4, 300
    d = _dims(N, S, M, D, L, Lq)
    accum = N * S * M * D * 4
    for rb in (1, N):
        for rl in (1, L):
            for ref_dim in (2, 4):
                partial = N * Lq * M * rl * ref_dim * 4        # per batch element even when the references broadcast
                assert _ws(lib, d, F32, rb, rl, ref_dim, 0) == 0
                assert _ws(lib, d, F32, rb, rl, ref_dim, 1) == partial
                for lowp in (BF16, F16):
                    assert _ws(lib, d, lowp, rb, rl, ref_dim, 0) == accum
                    assert _ws(lib, d, lowp, rb, rl, ref_dim, 1) == (accum + 15) // 16 * 16 + partial
    assert _ws(lib, d, F32, 1, 1, 3, 1) == 0
    assert lib.msda_backward_fused_workspace_bytes(None, F32, 1, 1, 2, 1) == 0
    # without the gradient the size is exactly what msda_backward_fused has always required
    assert _ws(lib, d, BF16, 1, 1, 2, 0) == accum


def test_four_levels_have_a_fused_kernel_and_two_do_not():
    lib = _cabi.load()
    # (L, P) = (4, 4) passes the kernel check and fails later on the misaligned reference, before any CUDA call
    assert _fwd(lib, _dims(L=4), ref=P + 8) == E_ALIGN
    assert _bwd(lib, _dims(L=4), ref=P + 8, ws=P, ws_bytes=1 << 30) == E_ALIGN
    assert _fwd(lib, _dims(L=2), rl=2) == E_UNSUPPORTED
    assert _bwd(lib, _dims(L=2), rl=2, ws=P, ws_bytes=1 << 30) == E_UNSUPPORTED
    assert _fwd(lib, _dims(D=48)) == E_UNSUPPORTED
