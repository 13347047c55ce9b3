"""bench.py --dump-outputs: what the timed path computed in its last step, as float32 .npy files that two builds can be
compared on (fixed sample positions, at most 64 MB in all)."""
import json
import os
import subprocess
import sys
import tempfile

import numpy as np
import pytest
import torch

from conftest import ROOT

import bench

ARRAYS = ('out', 'grad_value', 'grad_loc', 'grad_aw')


def test_dump_writes_small_arrays_whole_and_samples_one_element_per_stretch(tmp_path):
    g = torch.Generator().manual_seed(1)
    n = 3 * bench.DUMP_ELEMS + 12345
    big = torch.randn(n, generator=g).bfloat16()
    small = torch.randn(3, 4, generator=g)
    bench.dump_outputs(str(tmp_path), ['injector'], [(big, small, small.double(), small.half())])
    assert sorted(os.listdir(tmp_path)) == sorted('injector_%s.npy' % a for a in ARRAYS)
    for a in ARRAYS:
        assert np.load(tmp_path / ('injector_%s.npy' % a)).dtype == np.float32
    np.testing.assert_array_equal(np.load(tmp_path / 'injector_grad_value.npy'), small.numpy().reshape(-1))
    np.testing.assert_array_equal(np.load(tmp_path / 'injector_grad_aw.npy'), small.half().float().numpy().reshape(-1))
    pos = bench.dump_positions(n)
    k = torch.arange(bench.DUMP_ELEMS)
    assert pos.shape == (bench.DUMP_ELEMS,)
    assert ((pos >= k * n // bench.DUMP_ELEMS) & (pos < (k + 1) * n // bench.DUMP_ELEMS)).all()
    assert len(set((pos - k * n // bench.DUMP_ELEMS).tolist())) > 2   # not a fixed stride
    np.testing.assert_array_equal(np.load(tmp_path / 'injector_out.npy'), big.float()[pos].numpy())


def test_dump_positions_are_the_same_in_a_fresh_process(tmp_path):
    n = 5 * bench.DUMP_ELEMS + 7
    torch.manual_seed(123)
    torch.rand(11)   # the global generator's state must not matter
    here = bench.dump_positions(n).numpy()
    f = str(tmp_path / 'pos.npy')
    code = 'import sys; sys.path.insert(0, %r)\nimport numpy, bench\nnumpy.save(%r, bench.dump_positions(%d).numpy())' % (ROOT, f, n)
    subprocess.run([sys.executable, '-c', code], check=True, timeout=300)
    np.testing.assert_array_equal(np.load(f), here)


def test_dump_outputs_needs_the_gpu_path():
    r = subprocess.run([sys.executable, os.path.join(ROOT, 'bench.py'), '--impl', 'reference', '--dump-outputs', 'x'],
                       stdout=subprocess.PIPE, stderr=subprocess.PIPE, text=True, timeout=300)
    assert r.returncode == 2 and '--dump-outputs' in r.stderr


@pytest.mark.gpu
def test_bench_runs_the_steps_asked_for_and_dumps_what_the_last_one_computed():
    """bench.py at ViT-Adapter-B, 1 image, 2 timed steps: the launches of exactly 2 steps, and a dump that matches the C
    oracle on the inputs bench.py draws for that run (Injector seed 0, Extractor seed 1)."""
    from oracle import c_oracle
    from vit_adapter_b200 import _cabi
    with tempfile.TemporaryDirectory() as d:
        cmd = [sys.executable, os.path.join(ROOT, 'bench.py'), '--gpus', '1', '--steps', '2', '--warmup', '3', '--batch', '1',
               '--no-cpu-baseline', '--no-ref-cuda', '--no-other-shapes', '--no-step', '--dump-outputs', d]
        r = subprocess.run(cmd, stdout=subprocess.PIPE, stderr=subprocess.PIPE, text=True, timeout=900)
        assert r.returncode == 0, r.stderr[-3000:]
        line = json.loads(r.stdout.strip().splitlines()[-1])
        assert sorted(os.listdir(d)) == sorted('%s_%s.npy' % (c, a) for c in ('injector', 'extractor') for a in ARRAYS)
        assert sum(os.path.getsize(os.path.join(d, f)) for f in os.listdir(d)) <= 64e6
        dumped = {f[:-4]: np.load(os.path.join(d, f)) for f in os.listdir(d)}
    calls = [bench.adapter_inputs(name, N, M, D, Lq, shapes, seed=i, dtype=torch.float32)
             for i, (name, N, M, D, Lq, shapes) in enumerate(bench.call_shapes('B', 1))]
    # one step of the same calls in this process gives the launches per step
    n0 = _cabi.launch_count()
    for c in calls:
        g = {k: v.cuda() for k, v in c.items()}
        _cabi.forward(g['value'], g['shapes'], g['lsi'], g['loc'], g['aw'], 64)
        _cabi.backward(g['value'], g['shapes'], g['lsi'], g['loc'], g['aw'], g['grad_out'], 64)
    torch.cuda.synchronize()
    assert line['steps'] == 2 and line['gpu_launches'] == 2 * (_cabi.launch_count() - n0)
    for (name, *_), c in zip(bench.call_shapes('B', 1), calls):
        out = c_oracle.forward(c['value'], c['shapes'], c['lsi'], c['loc'], c['aw'])
        grads = c_oracle.backward(c['value'], c['shapes'], c['lsi'], c['loc'], c['aw'], c['grad_out'])
        for what, want, tol in zip(ARRAYS, (out,) + tuple(grads), (1e-5, 1e-4, 1e-4, 1e-4)):
            want = want.reshape(-1)
            if want.numel() > bench.DUMP_ELEMS:
                want = want[bench.dump_positions(want.numel())]
            got = torch.from_numpy(dumped['%s_%s' % (name, what)])
            torch.testing.assert_close(got, want, rtol=tol, atol=tol * float(want.abs().max()), msg='%s_%s' % (name, what))
