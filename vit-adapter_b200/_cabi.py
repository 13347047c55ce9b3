"""ctypes binding of include/msda_b200.h (lib/libmsda_b200.so).

This is the only place Python touches the native library. It passes raw device pointers, the 7
dimensions and the current CUDA stream; it never computes anything itself and there is NO fallback:
if the shared library is missing or a tensor is not on a CUDA device the call raises.

Replaces the pybind11 module of the reference (detection/ops/src/vision.cpp:13-16).
"""
import ctypes
import os
import threading

import torch

_HERE = os.path.dirname(os.path.abspath(__file__))
# (MSDA_B200_LIB names another build of the same library: A/B timing of kernel variants, tools/walker_variants.sh)
LIB_PATH = os.environ.get('MSDA_B200_LIB') or os.path.join(_HERE, 'lib', 'libmsda_b200.so')

MSDA_F32, MSDA_BF16, MSDA_F64 = 0, 1, 2
MSDA_F16 = 3
_DTYPES = {torch.float32: MSDA_F32, torch.bfloat16: MSDA_BF16, torch.float64: MSDA_F64, torch.float16: MSDA_F16}
_ADAPTER_DTYPES = _DTYPES

# every symbol include/msda_b200.h declares
EXPORTS = (
    'msda_abi_version', 'msda_last_error', 'msda_check_im2col_step', 'msda_forward', 'msda_forward_ex',
    'msda_backward_workspace_bytes', 'msda_backward', 'msda_debug_point_index', 'msda_launch_count',
    'msda_set_tuning', 'msda_forward_fused', 'msda_backward_fused',
    'msda_forward_fused_ref', 'msda_backward_fused_ref', 'msda_backward_fused_workspace_bytes',
    'adapter_dwconv_forward', 'adapter_dwconv_backward_input', 'adapter_dwconv_backward_weight',
    'adapter_dwconv_backward_weight_workspace_bytes',
    'adapter_layernorm_forward', 'adapter_layernorm_backward', 'adapter_layernorm_backward_workspace_bytes',
    'adapter_colsum', 'adapter_colsum_workspace_bytes', 'adapter_residual_add',
)


class MsdaDims(ctypes.Structure):
    _fields_ = [(n, ctypes.c_int32) for n in
                ('batch', 'spatial_size', 'num_heads', 'channels', 'num_levels', 'num_query', 'num_point')]


_lib = None
_lock = threading.Lock()


def load():
    """dlopen the C-ABI library (once). Raises if it has not been built — there is no CPU path."""
    global _lib
    if _lib is not None:
        return _lib
    with _lock:
        if _lib is not None:
            return _lib
        if not os.path.exists(LIB_PATH):
            raise RuntimeError(
                'native library %s is missing: build it with `python vit-adapter_b200/build.py` '
                '(or __graft_entry__.build()). There is no CPU / PyTorch fallback for this op.' % LIB_PATH)
        lib = ctypes.CDLL(LIB_PATH)
        vp, i64p = ctypes.c_void_p, ctypes.c_void_p
        dp = ctypes.POINTER(MsdaDims)
        lib.msda_abi_version.restype = ctypes.c_int
        lib.msda_abi_version.argtypes = []
        lib.msda_last_error.restype = ctypes.c_char_p
        lib.msda_last_error.argtypes = []
        lib.msda_check_im2col_step.restype = ctypes.c_int
        lib.msda_check_im2col_step.argtypes = [ctypes.c_int32, ctypes.c_int32]
        lib.msda_forward.restype = ctypes.c_int
        lib.msda_forward.argtypes = [dp, ctypes.c_int, vp, i64p, i64p, vp, vp, vp, vp]
        lib.msda_forward_ex.restype = ctypes.c_int
        lib.msda_forward_ex.argtypes = [dp, ctypes.c_int, vp, i64p, i64p, vp, vp, vp, vp, vp]
        lib.msda_backward_workspace_bytes.restype = ctypes.c_size_t
        lib.msda_backward_workspace_bytes.argtypes = [dp, ctypes.c_int]
        lib.msda_backward.restype = ctypes.c_int
        lib.msda_backward.argtypes = [dp, ctypes.c_int, vp, i64p, i64p, vp, vp, vp, vp, vp, vp, vp,
                                      ctypes.c_size_t, vp]
        lib.msda_forward_fused.restype = ctypes.c_int
        lib.msda_forward_fused.argtypes = [dp, ctypes.c_int, vp, i64p, i64p, vp, ctypes.c_int32, ctypes.c_int32, vp, vp,
                                           ctypes.c_int64, ctypes.c_int64, vp, vp]
        lib.msda_backward_fused.restype = ctypes.c_int
        lib.msda_backward_fused.argtypes = [dp, ctypes.c_int, vp, i64p, i64p, vp, ctypes.c_int32, ctypes.c_int32, vp, vp,
                                            ctypes.c_int64, ctypes.c_int64, vp, vp, vp, vp, vp, ctypes.c_size_t, vp]
        lib.msda_forward_fused_ref.restype = ctypes.c_int
        lib.msda_forward_fused_ref.argtypes = [dp, ctypes.c_int, vp, i64p, i64p, vp, ctypes.c_int32, ctypes.c_int32,
                                               ctypes.c_int32, vp, vp, ctypes.c_int64, ctypes.c_int64, vp, vp]
        lib.msda_backward_fused_ref.restype = ctypes.c_int
        lib.msda_backward_fused_ref.argtypes = [dp, ctypes.c_int, vp, i64p, i64p, vp, ctypes.c_int32, ctypes.c_int32,
                                                ctypes.c_int32, vp, vp, ctypes.c_int64, ctypes.c_int64, vp, vp, vp, vp, vp, vp,
                                                ctypes.c_size_t, vp]
        lib.msda_backward_fused_workspace_bytes.restype = ctypes.c_size_t
        lib.msda_backward_fused_workspace_bytes.argtypes = [dp, ctypes.c_int, ctypes.c_int32, ctypes.c_int32, ctypes.c_int32,
                                                            ctypes.c_int32]
        i32 = ctypes.c_int32
        lib.adapter_dwconv_forward.restype = ctypes.c_int
        lib.adapter_dwconv_forward.argtypes = [ctypes.c_int, vp, vp, vp, vp, i32, i32, i32, i32, i32, vp]
        lib.adapter_dwconv_backward_input.restype = ctypes.c_int
        lib.adapter_dwconv_backward_input.argtypes = [ctypes.c_int, vp, vp, vp, i32, i32, i32, i32, i32, vp]
        lib.adapter_dwconv_backward_weight.restype = ctypes.c_int
        lib.adapter_dwconv_backward_weight.argtypes = [ctypes.c_int, vp, vp, vp, vp, i32, i32, i32, i32, i32, vp, ctypes.c_size_t, vp]
        lib.adapter_dwconv_backward_weight_workspace_bytes.restype = ctypes.c_size_t
        lib.adapter_dwconv_backward_weight_workspace_bytes.argtypes = [ctypes.c_int, i32, i32, i32, i32, i32]
        i64 = ctypes.c_int64
        lib.adapter_layernorm_forward.restype = ctypes.c_int
        lib.adapter_layernorm_forward.argtypes = [ctypes.c_int, ctypes.c_int, vp, vp, vp, vp, vp, vp, i64, i32, ctypes.c_float, vp]
        lib.adapter_layernorm_backward_workspace_bytes.restype = ctypes.c_size_t
        lib.adapter_layernorm_backward_workspace_bytes.argtypes = [i64, i32]
        lib.adapter_colsum_workspace_bytes.restype = ctypes.c_size_t
        lib.adapter_colsum_workspace_bytes.argtypes = [ctypes.c_int, i64, i32]
        lib.adapter_colsum.restype = ctypes.c_int
        lib.adapter_colsum.argtypes = [ctypes.c_int, vp, i64, i32, vp, vp, ctypes.c_size_t, vp]
        lib.adapter_layernorm_backward.restype = ctypes.c_int
        lib.adapter_layernorm_backward.argtypes = [ctypes.c_int, ctypes.c_int, vp, vp, vp, vp, vp, vp, vp, vp, vp, i64, i32, vp,
                                                   ctypes.c_size_t, vp]
        lib.adapter_residual_add.restype = ctypes.c_int
        lib.adapter_residual_add.argtypes = [ctypes.c_int, vp, vp, vp, i64, vp]
        lib.msda_debug_point_index.restype = ctypes.c_int
        lib.msda_debug_point_index.argtypes = [dp, i64p, i64p, vp, vp, vp]
        lib.msda_launch_count.restype = ctypes.c_uint64
        lib.msda_launch_count.argtypes = []
        lib.msda_set_tuning.restype = ctypes.c_int
        lib.msda_set_tuning.argtypes = [ctypes.c_char_p, ctypes.c_int32]
        if lib.msda_abi_version() != 1:
            raise RuntimeError('libmsda_b200.so ABI version %d, expected 1' % lib.msda_abi_version())
        _lib = lib
    return _lib


def _raise(code, what):
    msg = load().msda_last_error().decode('utf-8', 'replace')
    raise RuntimeError('%s failed (code %d): %s' % (what, code, msg))


def _check_cuda(**tensors):
    # Same contract as the reference host code (ms_deform_attn_cuda.cu:28-38): contiguous CUDA
    # tensors are REQUIRED, never silently fixed up; CPU tensors are an error (ms_deform_attn.h:38).
    dev = None
    for name, t in tensors.items():
        if not t.is_cuda:
            raise RuntimeError('%s must be a CUDA tensor (Not implemented on the CPU)' % name)
        if not t.is_contiguous():
            raise RuntimeError('%s tensor has to be contiguous' % name)
        if dev is None:
            dev = t.device
        elif t.device != dev:
            raise RuntimeError('%s is on %s, expected %s' % (name, t.device, dev))
    return dev


def _dims(value, spatial_shapes, sampling_loc):
    if value.dim() != 4 or sampling_loc.dim() != 6 or spatial_shapes.dim() != 2:
        raise RuntimeError('expected value [N,S,M,D], spatial_shapes [L,2], sampling_loc [N,Lq,M,L,P,2]')
    N, S, M, D = value.shape
    L = spatial_shapes.shape[0]
    Lq, P = sampling_loc.shape[1], sampling_loc.shape[4]
    return MsdaDims(N, S, M, D, L, Lq, P)


def _dtype_code(value, sampling_loc, attn_weight):
    code = _DTYPES.get(value.dtype)
    if code is None:
        raise RuntimeError('unsupported value dtype %s (float32, bfloat16, float16, float64)' % value.dtype)
    want = torch.float64 if code == MSDA_F64 else torch.float32
    if sampling_loc.dtype != want or attn_weight.dtype != want:
        raise RuntimeError('sampling_loc / attn_weight must be %s for value dtype %s' % (want, value.dtype))
    return code


def _check_meta(spatial_shapes, level_start_index):
    if spatial_shapes.dtype != torch.int64 or level_start_index.dtype != torch.int64:
        raise RuntimeError('spatial_shapes / level_start_index must be int64 (as in the reference)')


class _NoSwitch:
    def __enter__(self):
        return None

    def __exit__(self, *exc):
        return False


_NO_SWITCH = _NoSwitch()


def _on(dev):
    """Device guard for allocation + launch; free when `dev` is already current (torch.cuda.device() costs ~10 us a call)."""
    return _NO_SWITCH if dev.index == torch.cuda.current_device() else torch.cuda.device(dev)


def _stream():
    # the raw handle of torch's current stream on the current device; torch.cuda.current_stream() builds a Stream
    # object and costs ~18 us a call, which at 2 images per GPU was 15% of an adapter interaction's host time
    return ctypes.c_void_p(torch._C._cuda_getCurrentRawStream(torch.cuda.current_device()))


def _workspace(nbytes, dev):
    """(buffer, pointer) of `nbytes` bytes of device scratch for one call, or (None, None) when none is needed. Keep the
    buffer referenced until the call has been issued."""
    if not nbytes:
        return None, None
    ws = torch.empty((nbytes,), dtype=torch.uint8, device=dev)
    return ws, ws.data_ptr()


class TensorMemo:
    """Memo keyed by tensor IDENTITY (weak reference) + version counter. Keying by data_ptr would be wrong: the
    caching allocator hands a freed address to the next tensor of the same size, with different contents."""

    def __init__(self, limit=256):
        self._d = {}
        self._limit = limit

    def get(self, t, extra=None):
        ent = self._d.get(id(t))
        if ent is not None and ent[0]() is t and ent[1] == (t._version, extra):
            return ent[2]
        return None

    # A memo is derived state: it pickles (torch.save(model), copy.deepcopy, mp.spawn) as an empty memo. The weak
    # references and their callbacks it holds are not picklable and would mean nothing in another process anyway.
    def __getstate__(self):
        return {'_limit': self._limit}

    def __setstate__(self, state):
        self._d = {}
        self._limit = state.get('_limit', 256)

    def __deepcopy__(self, memo):
        return TensorMemo(self._limit)

    def put(self, t, value, extra=None):
        import weakref
        if len(self._d) > self._limit:
            self._d = {k: v for k, v in self._d.items() if v[0]() is not None}
            if len(self._d) > self._limit:
                self._d.clear()
        key = id(t)
        self._d[key] = (weakref.ref(t, lambda _r, k=key, d=self._d: d.pop(k, None)), (t._version, extra), value)
        return value


# Host copies of spatial_shapes tensors (needed only by kernels planned on the host: the opt-in shared-memory
# forward). ONE device->host read the first time a given tensor object is seen, none afterwards: the adapter's
# deform_inputs() memoises its tensors, so steady-state forwards never synchronise.
_HOST_SHAPES = TensorMemo()
_WANT_HOST_SHAPES = False  # switched on by set_tuning(fwd_smem=2)


def host_shapes(spatial_shapes):
    hit = _HOST_SHAPES.get(spatial_shapes)
    if hit is None:
        if torch.cuda.is_current_stream_capturing():
            return None  # never synchronise inside a graph capture; the default kernels need no host shapes
        vals = [int(v) for v in spatial_shapes.detach().reshape(-1).tolist()]
        hit = _HOST_SHAPES.put(spatial_shapes, (ctypes.c_int64 * len(vals))(*vals))
    return hit


def forward(value, spatial_shapes, level_start_index, sampling_loc, attn_weight, im2col_step):
    """ms_deform_attn_forward of the reference pybind module: returns out [N, Lq, M*D]."""
    lib = load()
    dev = _check_cuda(value=value, spatial_shapes=spatial_shapes, level_start_index=level_start_index,
                      sampling_loc=sampling_loc, attn_weight=attn_weight)
    _check_meta(spatial_shapes, level_start_index)
    dims = _dims(value, spatial_shapes, sampling_loc)
    code = _dtype_code(value, sampling_loc, attn_weight)
    rc = lib.msda_check_im2col_step(dims.batch, int(im2col_step))
    if rc != 0:
        _raise(rc, 'ms_deform_attn_forward')
    with _on(dev):
        out = torch.empty((dims.batch, dims.num_query, dims.num_heads * dims.channels),
                          dtype=value.dtype, device=dev)
        hs = host_shapes(spatial_shapes) if _WANT_HOST_SHAPES else None
        rc = lib.msda_forward_ex(ctypes.byref(dims), code, value.data_ptr(), spatial_shapes.data_ptr(),
                                 level_start_index.data_ptr(), sampling_loc.data_ptr(), attn_weight.data_ptr(),
                                 out.data_ptr(), ctypes.cast(hs, ctypes.c_void_p) if hs is not None else None,
                                 _stream())
    if rc != 0:
        _raise(rc, 'ms_deform_attn_forward')
    return out


def backward(value, spatial_shapes, level_start_index, sampling_loc, attn_weight, grad_output, im2col_step):
    """ms_deform_attn_backward of the reference pybind module: (grad_value, grad_loc, grad_attn)."""
    lib = load()
    dev = _check_cuda(value=value, spatial_shapes=spatial_shapes, level_start_index=level_start_index,
                      sampling_loc=sampling_loc, attn_weight=attn_weight, grad_output=grad_output)
    _check_meta(spatial_shapes, level_start_index)
    dims = _dims(value, spatial_shapes, sampling_loc)
    code = _dtype_code(value, sampling_loc, attn_weight)
    if grad_output.dtype != value.dtype:
        raise RuntimeError('grad_output dtype %s != value dtype %s' % (grad_output.dtype, value.dtype))
    rc = lib.msda_check_im2col_step(dims.batch, int(im2col_step))
    if rc != 0:
        _raise(rc, 'ms_deform_attn_backward')
    with _on(dev):
        grad_value = torch.empty_like(value)
        grad_loc = torch.empty_like(sampling_loc)
        grad_aw = torch.empty_like(attn_weight)
        ws_bytes = lib.msda_backward_workspace_bytes(ctypes.byref(dims), code)
        ws, ws_ptr = _workspace(ws_bytes, dev)
        rc = lib.msda_backward(ctypes.byref(dims), code, value.data_ptr(), spatial_shapes.data_ptr(),
                               level_start_index.data_ptr(), sampling_loc.data_ptr(), attn_weight.data_ptr(),
                               grad_output.data_ptr(), grad_value.data_ptr(), grad_loc.data_ptr(),
                               grad_aw.data_ptr(), ws_ptr, ws_bytes, _stream())
    if rc != 0:
        _raise(rc, 'ms_deform_attn_backward')
    return grad_value, grad_loc, grad_aw


MSDA_E_UNSUPPORTED = -8


def fused_supported(value, n_levels, n_points):
    """True when the fused entry points have a kernel for this configuration (else use forward/backward)."""
    if not value.is_cuda or value.dtype not in (torch.float32, torch.bfloat16, torch.float16):
        return False
    D = value.shape[-1]
    if not ((n_levels, n_points) in ((3, 4), (1, 4), (4, 4))) or D % 4 != 0 or (D // 4) not in (8, 16):
        return False
    cpl = 4 if value.dtype == torch.float32 else 8
    return D % cpl == 0 and (D // cpl) in (4, 8, 16)


def _check_fused_meta(spatial_shapes, level_start_index, reference_points, L):
    """The fused kernels index spatial_shapes / level_start_index with the MODULE's level count: a metadata tensor with
    fewer rows would be read out of bounds on the device (the reference fails with a broadcasting error instead)."""
    _check_meta(spatial_shapes, level_start_index)
    if tuple(spatial_shapes.shape) != (L, 2) or level_start_index.numel() != L:
        raise RuntimeError('fused MSDeformAttn: spatial_shapes must be [%d, 2] and level_start_index [%d], got %s and %s'
                           % (L, L, tuple(spatial_shapes.shape), tuple(level_start_index.shape)))
    if reference_points.dim() != 4 or reference_points.shape[-1] not in (2, 4):
        raise RuntimeError('fused MSDeformAttn: reference_points must be [Nr, Lq, Lr, 2|4], got %s' % (tuple(reference_points.shape),))


def _fused_dims(value, reference_points, sampling_offsets, attn_logits):
    if value.dim() != 4 or sampling_offsets.dim() != 6 or reference_points.dim() != 4 or reference_points.shape[-1] not in (2, 4):
        raise RuntimeError('expected value [N,S,M,D], reference_points [Nr,Lq,Lr,2|4], sampling_offsets [N,Lq,M,L,P,2]')
    N, S, M, D = value.shape
    _, Lq, M2, L, P, _ = sampling_offsets.shape
    if M2 != M or attn_logits.numel() != N * Lq * M * L * P or reference_points.shape[1] != Lq:
        raise RuntimeError('fused MSDeformAttn: inconsistent shapes')
    if sampling_offsets.dtype != torch.float32 or attn_logits.dtype != torch.float32 or reference_points.dtype != torch.float32:
        raise RuntimeError('fused MSDeformAttn: reference_points / sampling_offsets / attn_logits must be float32')
    return MsdaDims(N, S, M, D, L, Lq, P), int(reference_points.shape[0]), int(reference_points.shape[2])


def _forward_fused(dims, rb, rl, ref_dim, value, spatial_shapes, level_start_index, reference_points, offsets, logits,
                   row_stride):
    """out [N, Lq, M*D] of the fused entry. `ref_dim`: 2 (points) or 4 (boxes). `row_stride`: floats between consecutive
    (b, q) rows of `offsets` and `logits`, 0 = dense. Runs under the caller's device guard."""
    _check_fused_meta(spatial_shapes, level_start_index, reference_points, dims.num_levels)
    out = torch.empty((dims.batch, dims.num_query, dims.num_heads * dims.channels), dtype=value.dtype, device=value.device)
    rc = load().msda_forward_fused_ref(ctypes.byref(dims), _DTYPES.get(value.dtype), value.data_ptr(), spatial_shapes.data_ptr(),
                                       level_start_index.data_ptr(), reference_points.data_ptr(), rb, rl, ref_dim,
                                       offsets.data_ptr(), logits.data_ptr(), row_stride, row_stride, out.data_ptr(), _stream())
    if rc != 0:
        _raise(rc, 'msda_forward_fused_ref')
    return out


def _backward_fused(dims, rb, rl, ref_dim, value, spatial_shapes, level_start_index, reference_points, offsets, logits,
                    row_stride, grad_output, grad_offsets, grad_logits, grad_ref=None):
    """grad_value of the fused entry; writes the offset and logit gradients into `grad_offsets` / `grad_logits`, which have
    the row stride of `offsets` / `logits`, and, when `grad_ref` (f32, the shape of `reference_points`) is given, the
    reference-point gradient into it. Runs under the caller's device guard."""
    _check_fused_meta(spatial_shapes, level_start_index, reference_points, dims.num_levels)
    if grad_output.dtype != value.dtype:
        raise RuntimeError('grad_output dtype %s != value dtype %s' % (grad_output.dtype, value.dtype))
    lib = load()
    code = _DTYPES.get(value.dtype)
    grad_value = torch.empty_like(value)
    ws_bytes = lib.msda_backward_fused_workspace_bytes(ctypes.byref(dims), code, rb, rl, ref_dim, grad_ref is not None)
    ws, ws_ptr = _workspace(ws_bytes, value.device)
    rc = lib.msda_backward_fused_ref(ctypes.byref(dims), code, value.data_ptr(), spatial_shapes.data_ptr(),
                                     level_start_index.data_ptr(), reference_points.data_ptr(), rb, rl, ref_dim,
                                     offsets.data_ptr(), logits.data_ptr(), row_stride, row_stride, grad_output.data_ptr(),
                                     grad_value.data_ptr(), grad_offsets.data_ptr(), grad_logits.data_ptr(),
                                     grad_ref.data_ptr() if grad_ref is not None else None, ws_ptr, ws_bytes, _stream())
    if rc != 0:
        _raise(rc, 'msda_backward_fused_ref')
    return grad_value


def forward_fused(value, spatial_shapes, level_start_index, reference_points, sampling_offsets, attn_logits):
    """out [N, Lq, M*D] from RAW offsets / logits: softmax and location arithmetic happen inside the kernel."""
    dev = _check_cuda(value=value, spatial_shapes=spatial_shapes, level_start_index=level_start_index,
                      reference_points=reference_points, sampling_offsets=sampling_offsets, attn_logits=attn_logits)
    dims, rb, rl = _fused_dims(value, reference_points, sampling_offsets, attn_logits)
    with _on(dev):
        return _forward_fused(dims, rb, rl, reference_points.shape[-1], value, spatial_shapes, level_start_index,
                              reference_points, sampling_offsets, attn_logits, 0)


def backward_fused(value, spatial_shapes, level_start_index, reference_points, sampling_offsets, attn_logits, grad_output,
                   ref_grad=False):
    """(grad_value, grad_sampling_offsets, grad_attn_logits) of the fused entry, and grad_reference_points (f32, the shape of
    `reference_points`) as a fourth element when `ref_grad`."""
    dev = _check_cuda(value=value, spatial_shapes=spatial_shapes, level_start_index=level_start_index,
                      reference_points=reference_points, sampling_offsets=sampling_offsets, attn_logits=attn_logits,
                      grad_output=grad_output)
    dims, rb, rl = _fused_dims(value, reference_points, sampling_offsets, attn_logits)
    with _on(dev):
        grad_off, grad_logits = torch.empty_like(sampling_offsets), torch.empty_like(attn_logits)
        grad_ref = torch.empty_like(reference_points) if ref_grad else None
        grad_value = _backward_fused(dims, rb, rl, reference_points.shape[-1], value, spatial_shapes, level_start_index,
                                     reference_points, sampling_offsets, attn_logits, 0, grad_output, grad_off, grad_logits,
                                     grad_ref)
    return (grad_value, grad_off, grad_logits) + ((grad_ref,) if ref_grad else ())


def _merged_dims(value, reference_points, merged, n_levels, n_points):
    if value.dim() != 4 or reference_points.dim() != 4 or reference_points.shape[-1] not in (2, 4):
        raise RuntimeError('fused MSDeformAttn (merged): expected value [N,S,M,D] and reference_points [Nr,Lq,Lr,2|4], got %s and %s'
                           % (tuple(value.shape), tuple(reference_points.shape)))
    N, S, M, D = value.shape
    Lq = reference_points.shape[1]
    width = M * n_levels * n_points * 3
    if merged.dim() != 3 or merged.shape != (N, Lq, width) or merged.dtype != torch.float32 or reference_points.dtype != torch.float32:
        raise RuntimeError('fused MSDeformAttn (merged): expected float32 [N, Lq, M*L*P*3] offsets|logits, got %s' % (tuple(merged.shape),))
    return MsdaDims(N, S, M, D, n_levels, Lq, n_points), int(reference_points.shape[0]), int(reference_points.shape[2]), width


def forward_fused_merged(value, spatial_shapes, level_start_index, reference_points, merged, n_levels, n_points):
    """Fused forward reading offsets and logits from ONE buffer [N, Lq, M*L*P*3] — the output of a single GEMM whose
    weight is cat(sampling_offsets.weight, attention_weights.weight): columns [0, M*L*P*2) are the raw offsets,
    columns [M*L*P*2, M*L*P*3) the raw logits."""
    dev = _check_cuda(value=value, spatial_shapes=spatial_shapes, level_start_index=level_start_index,
                      reference_points=reference_points, merged=merged)
    dims, rb, rl, width = _merged_dims(value, reference_points, merged, n_levels, n_points)
    split = width // 3 * 2
    with _on(dev):
        return _forward_fused(dims, rb, rl, reference_points.shape[-1], value, spatial_shapes, level_start_index,
                              reference_points, merged[..., :split], merged[..., split:], width)


def backward_fused_merged(value, spatial_shapes, level_start_index, reference_points, merged, n_levels, n_points, grad_output,
                          ref_grad=False):
    """(grad_value, grad_merged): grad_merged has the layout of `merged`, i.e. it is the merged GEMM's output gradient;
    grad_reference_points (f32, the shape of `reference_points`) follows as a third element when `ref_grad`."""
    dev = _check_cuda(value=value, spatial_shapes=spatial_shapes, level_start_index=level_start_index,
                      reference_points=reference_points, merged=merged, grad_output=grad_output)
    dims, rb, rl, width = _merged_dims(value, reference_points, merged, n_levels, n_points)
    split = width // 3 * 2
    with _on(dev):
        grad_merged = torch.empty_like(merged)
        grad_ref = torch.empty_like(reference_points) if ref_grad else None
        grad_value = _backward_fused(dims, rb, rl, reference_points.shape[-1], value, spatial_shapes, level_start_index,
                                     reference_points, merged[..., :split], merged[..., split:], width, grad_output,
                                     grad_merged[..., :split], grad_merged[..., split:], grad_ref)
    return (grad_value, grad_merged) + ((grad_ref,) if ref_grad else ())


def dwconv_supported(x, weight, H, W):
    """True when the token-layout depth-wise 3x3 kernel applies (else the module runs the reference's op sequence)."""
    return (x.is_cuda and x.dtype in _ADAPTER_DTYPES and weight.dtype == x.dtype and x.dim() == 3 and H % 2 == 0 and W % 2 == 0
            and x.shape[1] == 21 * (H // 2) * (W // 2) and x.shape[2] <= 1024 and tuple(weight.shape) == (x.shape[2], 1, 3, 3))


def dwconv_forward(x, weight, bias, H, W):
    lib = load()
    dev = _check_cuda(x=x, weight=weight) if bias is None else _check_cuda(x=x, weight=weight, bias=bias)
    B, n, C = x.shape
    with _on(dev):
        y = torch.empty_like(x)
        rc = lib.adapter_dwconv_forward(_ADAPTER_DTYPES[x.dtype], x.data_ptr(), weight.data_ptr(),
                                        bias.data_ptr() if bias is not None else None, y.data_ptr(), B, n, C, H, W, _stream())
    if rc != 0:
        _raise(rc, 'adapter_dwconv_forward')
    return y


def dwconv_backward(x, weight, grad_y, H, W, need_input=True, need_weight=True):
    """(grad_x or None, grad_weight [C,1,3,3] or None, grad_bias [C] or None) in x.dtype."""
    lib = load()
    dev = _check_cuda(x=x, weight=weight, grad_y=grad_y)
    B, n, C = x.shape
    code = _ADAPTER_DTYPES[x.dtype]
    gx = gw = gb = None
    with _on(dev):
        if need_input:
            gx = torch.empty_like(x)
            rc = lib.adapter_dwconv_backward_input(code, grad_y.data_ptr(), weight.data_ptr(), gx.data_ptr(), B, n, C, H, W, _stream())
            if rc != 0:
                _raise(rc, 'adapter_dwconv_backward_input')
        if need_weight:
            adt = torch.float64 if x.dtype == torch.float64 else torch.float32
            gw = torch.empty((C, 1, 3, 3), dtype=adt, device=dev)
            gb = torch.empty((C,), dtype=adt, device=dev)
            ws_bytes = lib.adapter_dwconv_backward_weight_workspace_bytes(code, B, n, C, H, W)
            ws, ws_ptr = _workspace(ws_bytes, dev)
            rc = lib.adapter_dwconv_backward_weight(code, x.data_ptr(), grad_y.data_ptr(), gw.data_ptr(), gb.data_ptr(),
                                                    B, n, C, H, W, ws_ptr, ws_bytes, _stream())
            if rc != 0:
                _raise(rc, 'adapter_dwconv_backward_weight')
            gw, gb = gw.to(weight.dtype), gb.to(weight.dtype)
    return gx, gw, gb


def debug_point_index(spatial_shapes, level_start_index, sampling_loc, num_heads, channels):
    """[N*Lq*M*L*P, 4] int32: (h_low, w_low, corner mask, corner-1 element offset) per point."""
    lib = load()
    dev = _check_cuda(spatial_shapes=spatial_shapes, level_start_index=level_start_index,
                      sampling_loc=sampling_loc)
    _check_meta(spatial_shapes, level_start_index)
    N, Lq, M, L, P, _ = sampling_loc.shape
    if sampling_loc.dtype != torch.float32 or M != num_heads:
        raise RuntimeError('debug_point_index: float32 sampling_loc [N,Lq,M,L,P,2] expected')
    S = int((spatial_shapes[:, 0] * spatial_shapes[:, 1]).sum().item())
    dims = MsdaDims(N, S, M, channels, L, Lq, P)
    with _on(dev):
        idx = torch.empty((N * Lq * M * L * P, 4), dtype=torch.int32, device=dev)
        rc = lib.msda_debug_point_index(ctypes.byref(dims), spatial_shapes.data_ptr(),
                                        level_start_index.data_ptr(), sampling_loc.data_ptr(),
                                        idx.data_ptr(), _stream())
    if rc != 0:
        _raise(rc, 'msda_debug_point_index')
    return idx


def launch_count():
    return int(load().msda_launch_count())


def set_tuning(**kv):
    """Benchmark knobs, e.g. set_tuning(fwd_chunk=64, fwd_smem=1); value 0 restores the heuristic.
    Keys: fwd_chunk, bwd_chunk, fwd_min_ctas, bwd_min_ctas, fwd_smem, fwd_smem_threads, fwd_smem_chunks, fwd_wide,
    bwd_cell (2 = the cell-bucketed backward), bwd_cell_chunk, bwd_packed16 (2 = packed 16-bit reductions into grad_value), bwd_sorted (slab-sorted backward: 0 = where it measured faster, 1 = never, 2 = wherever it applies). The knobs are process-wide (see include/msda_b200.h)."""
    global _WANT_HOST_SHAPES
    lib = load()
    for k, v in kv.items():
        if lib.msda_set_tuning(k.encode(), int(v)) != 0:
            _raise(-1, 'msda_set_tuning')
        if k == 'fwd_smem':
            _WANT_HOST_SHAPES = int(v) == 2


# --- adapter LayerNorm prologues (SURVEY §8(f) N2) ---------------------------------------------------------------------
_LN_COMBOS = {(torch.float32, torch.float32), (torch.float32, torch.bfloat16), (torch.bfloat16, torch.bfloat16),
              (torch.float32, torch.float16), (torch.float16, torch.float16)}


def layernorm_supported(x, weight, bias, out_dtype):
    """True when the row kernel applies; otherwise the module calls torch's LayerNorm (the reference's op)."""
    C = x.shape[-1]
    return (x.is_cuda and (x.dtype, out_dtype) in _LN_COMBOS and weight is not None and weight.dtype == torch.float32
            and (bias is None or bias.dtype == torch.float32) and C % 4 == 0 and C <= 1024 and x.numel() > 0)


def layernorm_forward(x, weight, bias, eps, out_dtype):
    """(y in out_dtype, mean, rstd) for x [..., C] (contiguous)."""
    lib = load()
    dev = _check_cuda(x=x, weight=weight) if bias is None else _check_cuda(x=x, weight=weight, bias=bias)
    C = x.shape[-1]
    rows = x.numel() // C
    with _on(dev):
        y = torch.empty(x.shape, dtype=out_dtype, device=dev)
        stats = torch.empty((2, rows), dtype=torch.float32, device=dev)
        rc = lib.adapter_layernorm_forward(_ADAPTER_DTYPES[x.dtype], _ADAPTER_DTYPES[out_dtype], x.data_ptr(), weight.data_ptr(),
                                           bias.data_ptr() if bias is not None else None, y.data_ptr(), stats[0].data_ptr(),
                                           stats[1].data_ptr(), rows, C, float(eps), _stream())
    if rc != 0:
        _raise(rc, 'adapter_layernorm_forward')
    return y, stats


def layernorm_backward(grad_y, x, weight, stats, grad_residual=None):
    """(grad_x in x.dtype, grad_weight fp32 [C], grad_bias fp32 [C]); grad_residual (x's shape and dtype, contiguous) is
    added into grad_x."""
    gx, gwb = layernorm_backward_stacked(grad_y, x, weight, stats, grad_residual)
    return gx, gwb[0], gwb[1]


def layernorm_backward_stacked(grad_y, x, weight, stats, grad_residual=None):
    """layernorm_backward with grad_weight and grad_bias returned as the one fp32 [2, C] buffer the kernel writes."""
    lib = load()
    dev = _check_cuda(grad_y=grad_y, x=x, weight=weight)
    if grad_residual is not None:
        _check_cuda(grad_residual=grad_residual)
        if grad_residual.dtype != x.dtype or grad_residual.shape != x.shape:
            raise RuntimeError('layernorm_backward: grad_residual must have the shape and dtype of x')
    C = x.shape[-1]
    rows = x.numel() // C
    with _on(dev):
        gx = torch.empty_like(x)
        gwb = torch.empty((2, C), dtype=torch.float32, device=dev)
        ws_bytes = lib.adapter_layernorm_backward_workspace_bytes(rows, C)
        ws = torch.empty((ws_bytes,), dtype=torch.uint8, device=dev)
        rc = lib.adapter_layernorm_backward(_ADAPTER_DTYPES[x.dtype], _ADAPTER_DTYPES[grad_y.dtype], grad_y.data_ptr(), x.data_ptr(), weight.data_ptr(),
                                            stats[0].data_ptr(), stats[1].data_ptr(),
                                            grad_residual.data_ptr() if grad_residual is not None else None,
                                            gx.data_ptr(), gwb[0].data_ptr(), gwb[1].data_ptr(),
                                            rows, C, ws.data_ptr(), ws_bytes, _stream())
    if rc != 0:
        _raise(rc, 'adapter_layernorm_backward')
    return gx, gwb


# --- bias gradient of the adapter's Linears (SURVEY §8(f) N1) ------------------------------------------------------------
def colsum_supported(x):
    """x: [..., C] contiguous CUDA f32 (C % 4 == 0, C <= 1024) or bf16 / f16 (C % 8 == 0, C <= 2048)."""
    if not (x.is_cuda and x.dim() >= 2 and x.numel() > 0 and x.is_contiguous()):
        return False
    C = x.shape[-1]
    if x.dtype == torch.float32:
        return C % 4 == 0 and C <= 1024
    if x.dtype in (torch.bfloat16, torch.float16):
        return C % 8 == 0 and C <= 2048
    return False


def colsum(x):
    """fp32 [C] = sum of x over all leading dimensions (deterministic two-stage reduction)."""
    lib = load()
    dev = _check_cuda(x=x)
    C = x.shape[-1]
    rows = x.numel() // C
    code = _ADAPTER_DTYPES[x.dtype]
    with _on(dev):
        out = torch.empty((C,), dtype=torch.float32, device=dev)
        ws_bytes = lib.adapter_colsum_workspace_bytes(code, rows, C)
        ws = torch.empty((ws_bytes,), dtype=torch.uint8, device=dev)
        rc = lib.adapter_colsum(code, x.data_ptr(), rows, C, out.data_ptr(), ws.data_ptr(), ws_bytes, _stream())
    if rc != 0:
        _raise(rc, 'adapter_colsum')
    return out


# --- residual epilogue (SURVEY §8(f) N2) ----------------------------------------------------------------------------------
def residual_add_layout_supported(res, branch):
    """residual_add_supported without its pointer-alignment test (which compiled code defers to run time)."""
    return (res.is_cuda and branch.is_cuda and res.dtype == torch.float32 and branch.dtype in (torch.float32, torch.bfloat16, torch.float16)
            and res.shape == branch.shape and res.is_contiguous() and branch.is_contiguous() and res.numel() > 0
            and res.numel() % 8 == 0)


def residual_add_supported(res, branch):
    return residual_add_layout_supported(res, branch) and res.data_ptr() % 16 == 0 and branch.data_ptr() % 16 == 0


def residual_add(res, branch):
    """fp32 res + (f32 | bf16) branch -> fp32, one pass with 16-byte accesses on every operand."""
    lib = load()
    dev = _check_cuda(res=res, branch=branch)
    with _on(dev):
        out = torch.empty_like(res)
        rc = lib.adapter_residual_add(_ADAPTER_DTYPES[branch.dtype], res.data_ptr(), branch.data_ptr(), out.data_ptr(), res.numel(), _stream())
    if rc != 0:
        _raise(rc, 'adapter_residual_add')
    return out
