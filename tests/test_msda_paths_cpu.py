"""CPU checks for the launch paths of the plain sampling op (msda_forward / msda_backward): pointers at sub-element
offsets are refused before any CUDA call, and every plain-path kernel the library compiles is named by a case of
tests/test_msda_paths_gpu.py. The fake device pointers are never dereferenced."""
import ctypes
import glob
import os
import re
import shutil
import subprocess

import pytest

from conftest import ROOT
from vit_adapter_b200 import _cabi

import test_msda_paths_gpu as paths

E_ALIGN = -4
P = 0x10000  # a 16-byte aligned fake device address
DTYPES = [_cabi.MSDA_F32, _cabi.MSDA_BF16, _cabi.MSDA_F16, _cabi.MSDA_F64]
FWD_PTRS = ('value', 'spatial_shapes', 'level_start_index', 'sampling_loc', 'attn_weight', 'out')
BWD_PTRS = ('value', 'spatial_shapes', 'level_start_index', 'sampling_loc', 'attn_weight', 'grad_out', 'grad_value',
            'grad_sampling_loc', 'grad_attn_weight')


def _alignment(name, dtype):
    if name in ('spatial_shapes', 'level_start_index'):
        return 8
    if name in ('value', 'out', 'grad_out', 'grad_value'):
        return {_cabi.MSDA_F32: 4, _cabi.MSDA_BF16: 2, _cabi.MSDA_F16: 2, _cabi.MSDA_F64: 8}[dtype]
    return 8 if dtype == _cabi.MSDA_F64 else 4


@pytest.mark.parametrize('dtype', DTYPES, ids=['f32', 'bf16', 'f16', 'f64'])
def test_plain_entries_refuse_sub_element_offsets(dtype):
    lib = _cabi.load()
    d = _cabi.MsdaDims(2, 84, 3, 32, 3, 16, 4)
    for entry, names in (('forward', FWD_PTRS), ('backward', BWD_PTRS)):
        for name in names:
            for k in range(1, _alignment(name, dtype)):
                ptrs = [P + k if n == name else P for n in names]
                if entry == 'forward':
                    rc = lib.msda_forward(ctypes.byref(d), dtype, *ptrs, None)
                else:
                    rc = lib.msda_backward(ctypes.byref(d), dtype, *ptrs, P, 1 << 30, None)
                assert rc == E_ALIGN, (entry, name, k, rc, lib.msda_last_error())
                assert b'aligned' in lib.msda_last_error()


@pytest.mark.parametrize('dtype', [_cabi.MSDA_BF16, _cabi.MSDA_F16], ids=['bf16', 'f16'])
def test_fused_backward_refuses_an_odd_16bit_grad_value(dtype):
    """The fused backward converts into a 16-bit grad_value at any element offset, but not at an odd address."""
    lib = _cabi.load()
    d = _cabi.MsdaDims(2, 84, 3, 32, 3, 16, 4)
    ws = lib.msda_backward_fused_workspace_bytes(ctypes.byref(d), dtype, 1, 1, 2, 0)
    assert ws > 0
    rc = lib.msda_backward_fused(ctypes.byref(d), dtype, P, P, P, P, 1, 1, P, P, 0, 0, P, P + 1, P, P, P, ws, None)
    assert rc == E_ALIGN, (rc, lib.msda_last_error())
    rc = lib.msda_backward_fused_ref(ctypes.byref(d), dtype, P, P, P, P, 1, 1, 2, P, P, 0, 0, P, P + 3, P, P, None, P, ws, None)
    assert rc == E_ALIGN, (rc, lib.msda_last_error())


# --- every compiled plain-path kernel has a GPU case -----------------------------------------------------------------------
PLAIN = ('msda_fwd_vec_kernel', 'msda_bwd_vec_kernel', 'msda_fwd_generic_kernel', 'msda_bwd_generic_kernel',
         'msda_cvt_f32_bf16_kernel', 'msda_cvt_f32_bf16_scalar_kernel')


def _normalise(args):
    """cu++filt's template arguments ('(int)8', '(bool)0') in the profiler's spelling ('8', 'false')."""
    out = []
    for a in args.split(','):
        a = a.strip()
        a = {'(bool)0': 'false', '(bool)1': 'true'}.get(a, a)
        out.append(re.sub(r'^\(int\)', '', a))
    return tuple(out)


def _compiled_plain_kernels():
    objs = sorted(glob.glob(os.path.join(ROOT, 'vit-adapter_b200', 'lib', 'obj', 'msda_fwd*.o')) +
                  glob.glob(os.path.join(ROOT, 'vit-adapter_b200', 'lib', 'obj', 'msda_bwd*.o')))
    if not objs:
        pytest.skip('the library objects are not built')
    syms = set()
    for o in objs:
        out = subprocess.run(['cuobjdump', '-symbols', o], stdout=subprocess.PIPE, text=True, check=True).stdout
        syms.update(l.split()[-1] for l in out.splitlines() if 'STT_FUNC' in l)
    names = subprocess.run(['cu++filt'], input='\n'.join(sorted(syms)), stdout=subprocess.PIPE, text=True, check=True).stdout
    found = set()
    for line in names.splitlines():
        m = re.search(r'\bmsda::(\w+)<(.*)>\(', line)
        if not m or m.group(1) not in PLAIN:
            continue
        args = _normalise(m.group(2))
        if m.group(1) == 'msda_fwd_vec_kernel' and args[6] != 'false':
            continue    # fused forward
        if m.group(1) == 'msda_bwd_vec_kernel' and (args[5], args[6]) != ('false', 'false'):
            continue    # fused or packed 16-bit backward
        found.add((m.group(1), args))
    return found


def _named_kernels():
    named = set()
    for case in paths.CASES:
        named.update(paths.case_kernels(case))
    for case in paths.ALIGN_CASES:
        named.update(k for k in case[-1] if isinstance(k, tuple))
    return {(name, tuple(str(a) for a in args)) for name, args in named
            if name in PLAIN and not (name == 'msda_bwd_vec_kernel' and args[6] == 'true')}


@pytest.mark.skipif(not (shutil.which('cuobjdump') and shutil.which('cu++filt')), reason='needs cuobjdump and cu++filt')
def test_every_compiled_plain_kernel_has_a_case():
    """81 16-byte-lane forwards, 99 backwards, 15 32-byte-lane forwards, 8 generic kernels and 4 converts (vector and
    scalar stores, bf16 and f16)."""
    compiled, named = _compiled_plain_kernels(), _named_kernels()
    assert compiled - named == set(), 'compiled but not launched by any case: %s' % sorted(compiled - named)
    assert named - compiled == set(), 'named by a case but not compiled: %s' % sorted(named - compiled)
    count = {}
    for name, args in compiled:
        key = name + ('-wide' if name == 'msda_fwd_vec_kernel' and args[5] == '32' else '')
        count[key] = count.get(key, 0) + 1
    assert count == {'msda_fwd_vec_kernel': 81, 'msda_bwd_vec_kernel': 99, 'msda_fwd_vec_kernel-wide': 15,
                     'msda_fwd_generic_kernel': 4, 'msda_bwd_generic_kernel': 4, 'msda_cvt_f32_bf16_kernel': 2,
                     'msda_cvt_f32_bf16_scalar_kernel': 2}, count
