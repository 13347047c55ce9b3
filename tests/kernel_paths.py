"""Helpers shared by the kernel launch-path suites (tests/test_adapter_paths_gpu.py, tests/test_msda_paths_gpu.py):
inputs placed at byte offsets, the CUDA kernels a call launched, and elementwise rounding bounds against an fp64
reference."""
import math
import re

import torch


def at_offset(t, byte_offset):
    """A contiguous copy of `t` that starts `byte_offset` bytes into a larger (allocator-aligned) buffer."""
    es = t.element_size()
    assert byte_offset % es == 0
    k = byte_offset // es
    buf = torch.empty(t.numel() + k + 16, dtype=t.dtype, device=t.device)
    out = buf[k:k + t.numel()].view(t.shape)
    out.copy_(t)
    assert out.is_contiguous() and out.data_ptr() % 16 == byte_offset % 16, (out.data_ptr(), byte_offset)
    return out


def kernels_launched(fn, attempts=3):
    """(fn's result, names of the CUDA kernels fn launched, in launch order). Memsets and copies are left out.

    After other GPU tests have run in the same process, a profiler session can lose the first records it collects. So
    each session opens with a run of filler kernels and then one marker kernel (torch.cuda._sleep, which fn does not
    call), and only the kernels after the marker count. A session that lost the marker is repeated (fn again, so fn
    must be repeatable), and after `attempts` such sessions the call fails instead of reporting a short list."""
    from torch.autograd import DeviceType
    from torch.profiler import ProfilerActivity, profile
    filler = torch.zeros(1, device='cuda')
    for _ in range(attempts):
        torch.cuda.synchronize()
        with profile(activities=[ProfilerActivity.CPU, ProfilerActivity.CUDA]) as prof:
            for _ in range(64):
                filler.add_(1)
            torch.cuda.synchronize()
            torch.cuda._sleep(1000)
            torch.cuda.synchronize()
            out = fn()
            torch.cuda.synchronize()
        events = sorted((e for e in prof.profiler.kineto_results.events() if e.device_type() == DeviceType.CUDA),
                        key=lambda e: e.start_ns())
        names = [e.name() for e in events if not e.name().startswith(('Memset', 'Memcpy', 'memset', 'memcpy'))]
        marks = [i for i, n in enumerate(names) if 'spin_kernel' in n]
        if marks:
            return out, names[marks[-1] + 1:]
    raise AssertionError('%d profiler sessions lost the marker kernel; the last one recorded %s' % (attempts, names))


def kernel(name, *args):
    """Regex for a kernel by template name and arguments, tolerant of the demangler's spacing."""
    if not args:
        return re.compile(r'\b%s\s*\(' % name)
    return re.compile(r'\b%s\s*<\s*%s\s*>' % (name, r'\s*,\s*'.join(re.escape(str(a)) for a in args)))


def unit_roundoff(dtype):
    return {torch.float32: 0.0, torch.float64: 0.0, torch.bfloat16: 2.0 ** -8, torch.float16: 2.0 ** -11}[dtype]


def assert_within(out, ref, acc, what):
    """|out - ref| <= u_out |ref| + (1 + u_out) acc + floor, elementwise, in fp64."""
    fi = torch.finfo(out.dtype)
    uo = unit_roundoff(out.dtype)
    err = (out.double() - ref).abs()
    bound = uo * ref.abs() + (1.0 + uo) * acc + fi.smallest_normal * fi.eps / 2
    bad = ~(err <= bound)
    if bad.any():
        ratio = torch.where(bound > 0, err / bound, torch.full_like(err, math.inf))
        i = int(ratio.flatten().argmax())
        raise AssertionError('%s: %d of %d elements outside the bound; worst at flat index %d: out %r ref %r err %.3e bound %.3e'
                             % (what, int(bad.sum()), err.numel(), i, float(out.flatten()[i]), float(ref.flatten()[i]),
                                float(err.flatten()[i]), float(bound.flatten()[i])))
