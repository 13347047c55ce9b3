#!/usr/bin/env python
"""bench.py — headline benchmark of the MSDeformAttn hot path (BASELINE.json metric).

    python bench.py --gpus N --steps K --warmup W          (N>1: launched by torch.distributed.run)
    python bench.py --impl reference ...                   (the reference's CPU path on the host cores)
    python bench.py ... --dump-outputs DIR                 (also writes the last timed step's results as .npy files)

One "step" = one pass of the hot path over one batch: Injector (n_levels=3) forward+backward and
Extractor (n_levels=1) forward+backward at the ViT-Adapter shape named in `config.workload`
(BASELINE.json configs[1]: ViT-Adapter-B, 512x512, 16 images per GPU, fp32 by default).
metric = sampled points per second (Gsamples/s), pts = N*Lq*M*L*P, whole job over all GPUs.
--steps K sets the timed region of that metric: exactly K steps on device-resident inputs. The informational arms clamp
it: `e2e` times 5 passes of min(max(K, 4), 50) steps and `ref_cuda` min(max(K, 2), 10) steps; both report their count.

Printed: ONE JSON line on stdout (rank 0). Keys follow the driver contract plus `roofline`,
`cpu_baseline`, `e2e`, `clocks`, `gpu_launches`, and informational `kernels` / `ref_cuda`.
"""
import argparse
import json
import os
import statistics
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

import torch  # noqa: E402

# ---------------------------------------------------------------------------------------------------
# workloads (SURVEY.md App. B). (M, D) per variant; levels derived from the image side.
# ---------------------------------------------------------------------------------------------------
VARIANTS = {
    # name: (heads, channels/head, image side, default images per GPU)
    'B': (12, 32, 512, 16),    # ViT-Adapter-B  (upernet_deit_adapter_base_512_160k_ade20k.py:14,21,23)
    'S': (6, 64, 512, 16),     # ViT-Adapter-S
    'T': (6, 32, 512, 16),     # ViT-Adapter-T
    'L': (16, 32, 896, 1),     # ViT-Adapter-L as configured by the reference (deform_ratio 0.5 -> 32 ch)
    'L64': (16, 64, 896, 1),   # ViT-Adapter-L as BASELINE.json words it (16 x 64)
    'HTC': (16, 32, 1024, 1),  # HTC++ inference shape (21 504 value tokens)
    'M2F': (32, 32, 896, 1),   # Mask2Former pixel decoder's deformable encoder (SURVEY §8(f) N4; ..._large_896_...ss.py:50-61)
}
P = 4


def call_shapes(variant, batch):
    """The two operator calls of one adapter interaction: (name, N, M, D, Lq, level shapes)."""
    M, D, side, _ = VARIANTS[variant]
    l8, l16, l32 = side // 8, side // 16, side // 32
    if variant == 'M2F':  # one self-attention call over the three levels' tokens
        return [('encoder', batch, M, D, l8 * l8 + l16 * l16 + l32 * l32, [(l8, l8), (l16, l16), (l32, l32)])]
    inj = ('injector', batch, M, D, l16 * l16, [(l8, l8), (l16, l16), (l32, l32)])
    ext = ('extractor', batch, M, D, l8 * l8 + l16 * l16 + l32 * l32, [(l16, l16)])
    return [inj, ext]


def n_points(N, M, Lq, L):
    return N * Lq * M * L * P


def algorithmic_bytes(N, M, D, Lq, shapes, esize):
    """SURVEY.md §8(d): every tensor touched once; loc/aw fp32 (12 B per point)."""
    S = sum(h * w for h, w in shapes)
    L = len(shapes)
    b_val = esize * N * S * M * D
    b_out = esize * N * Lq * M * D
    b_la = 12 * n_points(N, M, Lq, L)
    return {'fwd': b_val + b_la + b_out, 'bwd': b_out + 2 * b_val + 2 * b_la}


def adapter_inputs(name, N, M, D, Lq, shapes, seed, dtype):
    """Distribution A of SURVEY.md §8(d): reference-point grid (adapter_modules.py:13-25) + the module's
    initial offset ring (ms_deform_attn.py:66-75) + N(0, 1 px) noise; softmax(N(0,1)) weights; value and
    grad_out ~ N(0,1). Drawn on the CPU generator, like detection/ops/test.py."""
    import math
    g = torch.Generator().manual_seed(seed)
    shapes_t = torch.as_tensor(shapes, dtype=torch.long)
    L = len(shapes)
    S = int(shapes_t.prod(1).sum())
    lsi = torch.cat((shapes_t.new_zeros((1,)), shapes_t.prod(1).cumsum(0)[:-1]))
    # reference points: the query grid(s) — injector queries are the H/16 grid, extractor queries the 3 levels
    if name == 'injector':
        grids = [shapes[1]]
    elif name == 'encoder':
        grids = list(shapes)
    else:
        h, w = shapes[0]
        grids = [(2 * h, 2 * w), (h, w), (h // 2, w // 2)]
    refs = []
    for (h, w) in grids:
        ys = (torch.arange(h, dtype=torch.float32) + 0.5) / h
        xs = (torch.arange(w, dtype=torch.float32) + 0.5) / w
        yy, xx = torch.meshgrid(ys, xs, indexing='ij')
        refs.append(torch.stack([xx.reshape(-1), yy.reshape(-1)], -1))
    ref = torch.cat(refs, 0)
    assert ref.shape[0] == Lq
    theta = torch.arange(M, dtype=torch.float32) * (2.0 * math.pi / M)
    ray = torch.stack([theta.cos(), theta.sin()], -1)
    ray = ray / ray.abs().max(-1, keepdim=True)[0]
    off = ray.view(1, 1, M, 1, 1, 2) * torch.arange(1, P + 1, dtype=torch.float32).view(1, 1, 1, 1, P, 1)
    off = off + torch.randn(N, Lq, M, L, P, 2, generator=g)
    wh = torch.stack([shapes_t[:, 1], shapes_t[:, 0]], -1).float()
    loc = (ref.view(1, Lq, 1, 1, 1, 2) + off / wh.view(1, 1, 1, L, 1, 2)).contiguous()
    aw = torch.softmax(torch.randn(N, Lq, M, L * P, generator=g), -1).view(N, Lq, M, L, P).contiguous()
    value = torch.randn(N, S, M, D, generator=g).to(dtype)
    grad_out = torch.randn(N, Lq, M * D, generator=g).to(dtype)
    return dict(value=value, shapes=shapes_t, lsi=lsi, loc=loc, aw=aw, grad_out=grad_out)


# ---------------------------------------------------------------------------------------------------
# clocks sampling during the timed region (B200_PROFILING.md recipe)
# ---------------------------------------------------------------------------------------------------
class ClockSampler:
    """SM clock + throttle reasons sampled DURING the timed region. NVML polled from a thread every ~2 ms
    (the timed region is tens of ms); falls back to `nvidia-smi -lms` when pynvml is unavailable."""
    SMI_FIELDS = ('clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,'
                  'clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap')

    def __init__(self, gpu_index):
        self.gpu = gpu_index
        self.samples = []   # (time, sm_mhz, reasons bitmask or None)
        self.max_mhz = None
        self.stop_flag = False
        self.thread = None
        self.proc = None
        self.nvml = None

    def start(self):
        try:
            import pynvml
            pynvml.nvmlInit()
            self.nvml = pynvml
            self.handle = pynvml.nvmlDeviceGetHandleByIndex(self.gpu)
            self.max_mhz = float(pynvml.nvmlDeviceGetMaxClockInfo(self.handle, pynvml.NVML_CLOCK_SM))
            self.thread = threading.Thread(target=self._poll_nvml, daemon=True)
            self.thread.start()
            return
        except Exception:
            self.nvml = None
        try:
            self.proc = subprocess.Popen(
                ['nvidia-smi', '-i', str(self.gpu), '--query-gpu=' + self.SMI_FIELDS, '--format=csv,noheader,nounits',
                 '-lms', '20'], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.thread = threading.Thread(target=self._read_smi, daemon=True)
            self.thread.start()
        except OSError:
            self.proc = None

    def _poll_nvml(self):
        n = self.nvml
        while not self.stop_flag:
            try:
                mhz = float(n.nvmlDeviceGetClockInfo(self.handle, n.NVML_CLOCK_SM))
                try:
                    reasons = int(n.nvmlDeviceGetCurrentClocksEventReasons(self.handle))
                except Exception:
                    reasons = int(n.nvmlDeviceGetCurrentClocksThrottleReasons(self.handle))
                self.samples.append((time.time(), mhz, reasons))
            except Exception:
                pass
            time.sleep(0.002)

    def _read_smi(self):
        names = ['hw_slowdown', 'hw_thermal_slowdown', 'sw_thermal_slowdown', 'sw_power_cap']
        for line in self.proc.stdout:
            parts = [x.strip() for x in line.split(',')]
            if len(parts) < 6:
                continue
            try:
                mhz = float(parts[0])
                self.max_mhz = float(parts[1])
            except ValueError:
                continue
            self.samples.append((time.time(), mhz, [n for n, v in zip(names, parts[2:6]) if v.lower().startswith('active')]))

    def stop(self, t0, t1):
        self.stop_flag = True
        if self.proc is not None:
            time.sleep(0.05)
            self.proc.terminate()
        if self.thread is not None:
            self.thread.join(timeout=2)
        if not self.samples:
            return {'sm_mhz': None, 'sm_max_mhz': self.max_mhz, 'reasons': ['no clock samples'], 'samples': 0}
        inside = [s for s in self.samples if t0 <= s[0] <= t1] or self.samples[-3:]
        reasons = set()
        for _, _, r in inside:
            if isinstance(r, list):
                reasons.update(r)
            elif r is not None and self.nvml is not None:
                n = self.nvml
                for name, bit in (('hw_slowdown', 0x8), ('sw_thermal_slowdown', 0x20), ('hw_thermal_slowdown', 0x40),
                                  ('sw_power_cap', 0x4)):
                    if r & bit:
                        reasons.add(name)
        return {'sm_mhz': statistics.median([s[1] for s in inside]), 'sm_max_mhz': self.max_mhz,
                'reasons': sorted(reasons), 'samples': len(inside), 'source': 'nvml' if self.nvml else 'nvidia-smi'}


# ---------------------------------------------------------------------------------------------------
# CPU arm: the reference's CPU path (oracle/core_pytorch.py restates ms_deform_attn_core_pytorch)
# ---------------------------------------------------------------------------------------------------
def cpu_reference_pass(variant, sample_batch, threads, steps, warmup):
    """Time fwd+bwd of Injector+Extractor on the host cores for `sample_batch` images. Returns
    (Gsamples/s, seconds per step, points per step)."""
    from oracle import core_pytorch  # the ONLY place bench.py executes oracle/ code
    torch.set_num_threads(threads)
    calls = []
    pts = 0
    for i, (name, N, M, D, Lq, shapes) in enumerate(call_shapes(variant, sample_batch)):
        calls.append(adapter_inputs(name, N, M, D, Lq, shapes, seed=i, dtype=torch.float32))
        pts += n_points(N, M, Lq, len(shapes))
    times = []
    for it in range(warmup + steps):
        t0 = time.perf_counter()
        for c in calls:
            core_pytorch.forward_backward(c['value'], c['shapes'], c['loc'], c['aw'], c['grad_out'])
        dt = time.perf_counter() - t0
        if it >= warmup:
            times.append(dt)
    mean = sum(times) / len(times)
    return pts / mean / 1e9, mean, pts


def run_reference_arm(args):
    rank = int(os.environ.get('RANK', '0'))
    if rank != 0:
        return 0
    variant = args.variant
    _, _, _, default_batch = VARIANTS[variant]
    batch = args.batch or default_batch
    sample_batch = min(batch, 2)
    threads = os.cpu_count() or 1
    value, sec, pts = cpu_reference_pass(variant, sample_batch, threads, args.steps, max(1, args.warmup))
    M, D, side, _ = VARIANTS[variant]
    line = {
        'impl': 'reference', 'metric': 'msdeformattn_fwd_bwd_gsamples_per_s', 'value': value, 'unit': 'Gsamples/s',
        'n_gpus': args.gpus, 'steps': args.steps, 'warmup': max(1, args.warmup), 'ms_per_step': sec * 1e3,
        'higher_is_better': True, 'scaling': 'weak', 'vs_baseline': None, 'dtype': 'f32', 'data': 'synthetic',
        'config': workload_config(variant, batch, 'f32'),
        'cpu_baseline': {'value': value, 'unit': 'Gsamples/s', 'cores': threads, 'kind': 'port',
                         'sample': '%d of %d images per step at this workload\'s own shape (ViT-Adapter-%s: %d heads x %d ch, '
                                   '%dx%d; BASELINE cfg 1 is the same call sequence at variant S), Injector+Extractor fwd+bwd via '
                                   'oracle/core_pytorch.py (restatement of ms_deform_attn_core_pytorch, F.grid_sample '
                                   '+ autograd), torch %d threads' % (sample_batch, batch, variant, M, D, side, side, threads)},
        'e2e': {'value': value, 'unit': 'Gsamples/s', 'h2d_bytes_per_step': 0, 'd2h_bytes_per_step': 0},
        'gpu_launches': 0,
    }
    emit(line)
    return 0


def workload_config(variant, batch, dtype):
    M, D, side, _ = VARIANTS[variant]
    return {
        'workload': 'ViT-Adapter-%s MSDeformAttn fwd+bwd: Injector(n_levels=3)+Extractor(n_levels=1), %dx%d, '
                    '%d images per GPU, %d heads x %d ch, 4 points' % (variant, side, side, batch, M, D),
        'variant': variant, 'image': side, 'batch_per_gpu': batch, 'heads': M, 'channels': D, 'points': P,
        'io_dtype': dtype, 'inputs': 'distribution A (adapter reference grid + init ring + N(0,1px))',
        'l2': 'working set per step is larger than L2 (no explicit flush)', 'parallelism': 'batch-sharded, no collective',
    }


DUMP_ELEMS = 1 << 20   # per array: the 8 float32 arrays of an Injector+Extractor step stay below 64 MB in all


def dump_positions(n):
    """The flattened positions dump_outputs writes of an array of n > DUMP_ELEMS elements: one at a seeded random place in
    each of DUMP_ELEMS equal stretches, in order. They depend on n alone, so every run with the same arguments samples the
    same elements."""
    lo = torch.arange(DUMP_ELEMS + 1, dtype=torch.int64) * n // DUMP_ELEMS
    u = torch.rand(DUMP_ELEMS, generator=torch.Generator().manual_seed(0), dtype=torch.float64)
    return lo[:-1] + (u * (lo[1:] - lo[:-1])).long()


def dump_outputs(directory, names, results):
    """Write each call's (out, grad_value, grad_loc, grad_aw) as <directory>/<call>_<array>.npy in float32: the whole
    flattened array, or for one of more than DUMP_ELEMS elements its elements at dump_positions(), so that two builds can
    be compared output for output."""
    import numpy as np
    os.makedirs(directory, exist_ok=True)
    for name, arrays in zip(names, results):
        for what, t in zip(('out', 'grad_value', 'grad_loc', 'grad_aw'), arrays):
            flat = t.detach().reshape(-1)
            if flat.numel() > DUMP_ELEMS:
                flat = flat[dump_positions(flat.numel()).to(flat.device)]
            np.save(os.path.join(directory, '%s_%s.npy' % (name, what)), flat.float().cpu().numpy())


# ---------------------------------------------------------------------------------------------------
# GPU arm
# ---------------------------------------------------------------------------------------------------
def run_ours(args):
    import torch.distributed as dist
    import vit_adapter_b200 as vab
    from vit_adapter_b200 import _cabi
    from vit_adapter_b200.sharding import batch_shard, max_over_ranks

    world = int(os.environ.get('WORLD_SIZE', '1'))
    rank = int(os.environ.get('RANK', '0'))
    local_rank = int(os.environ.get('LOCAL_RANK', '0'))
    if not torch.cuda.is_available():
        raise RuntimeError('bench.py needs a CUDA device: the product path has no CPU fallback '
                           '(use --impl reference for the CPU arm)')
    torch.cuda.set_device(local_rank)
    dev = torch.device('cuda', local_rank)
    all_cpus = os.sched_getaffinity(0)
    numa = bind_host_thread_to_gpu(dev)
    if world > 1:
        os.environ.setdefault('MASTER_ADDR', '127.0.0.1')
        if not args.no_step:
            # the training-step block captures DDP's all-reduce in a CUDA graph: captured NCCL work has no watchdog-visible events
            os.environ.setdefault('TORCH_NCCL_ASYNC_ERROR_HANDLING', '0')
        dist.init_process_group('nccl', device_id=dev)
    _cabi.load()

    variant = args.variant
    M, D, side, default_batch = VARIANTS[variant]
    batch = args.batch or default_batch
    dtype = {'f32': torch.float32, 'bf16': torch.bfloat16}[args.dtype]
    esize = 4 if dtype == torch.float32 else 2

    # ---- inputs: host (pinned) master copies + device-resident copies -----------------------------------
    # weak scaling: the job holds world * batch images; this rank owns the contiguous slice batch_shard() gives it and
    # draws exactly those samples (the seed is the first global sample index of the shard)
    shard_begin, shard_end = batch_shard(world * batch, world, rank)
    assert shard_end - shard_begin == batch
    calls = []
    pts_step = 0
    for i, (name, N, Mh, Dh, Lq, shapes) in enumerate(call_shapes(variant, shard_end - shard_begin)):
        host = adapter_inputs(name, N, Mh, Dh, Lq, shapes, seed=1000 * shard_begin + i, dtype=dtype)
        pinned = {k: v.pin_memory() for k, v in host.items()}
        devt = {k: v.to(dev, non_blocking=True) for k, v in pinned.items()}
        calls.append({'name': name, 'dims': (N, Mh, Dh, Lq, shapes), 'host': pinned, 'dev': devt,
                      'pts': n_points(N, Mh, Lq, len(shapes)), 'bytes': algorithmic_bytes(N, Mh, Dh, Lq, shapes, esize)})
        pts_step += calls[-1]['pts']
    torch.cuda.synchronize()

    def step_device(events=None, keep=False):
        """One step on device-resident inputs, straight through the C-ABI binding. With keep, returns per call what a
        caller of the binding receives: [out, grad_value, grad_loc, grad_aw]; otherwise every result is freed as soon as
        it is returned, so its memory serves the next allocation of the step."""
        results = []
        for ci, c in enumerate(calls):
            d = c['dev']
            if events is not None:
                events[ci][0].record()
            out = _cabi.forward(d['value'], d['shapes'], d['lsi'], d['loc'], d['aw'], 64)
            if keep:
                results.append([out])
            del out
            if events is not None:
                events[ci][1].record()
            grads = _cabi.backward(d['value'], d['shapes'], d['lsi'], d['loc'], d['aw'], d['grad_out'], 64)
            if keep:
                results[-1].extend(grads)
            del grads
            if events is not None:
                events[ci][2].record()
        return results

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    # ---- warm-up -------------------------------------------------------------------------------------------
    # --dump-outputs keeps the results of the last timed step; the last warm-up step keeps its own too, so the caching
    # allocator already holds the memory that step needs and the timed region allocates none
    dumping = bool(args.dump_outputs)
    for w in range(args.warmup):
        step_device(keep=dumping and w == args.warmup - 1)
    barrier()

    # ---- timed region: exactly K steps, CUDA events, per-kernel events inside ------------------------------
    K = args.steps
    ev = [[[torch.cuda.Event(enable_timing=True) for _ in range(3)] for _ in calls] for _ in range(K)]
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    sampler = ClockSampler(local_rank) if rank == 0 else None
    if sampler:
        sampler.start()
        time.sleep(0.05)
    launches0 = _cabi.launch_count()
    barrier()
    t0 = time.time()
    e0.record()
    for k in range(K):
        last = step_device(ev[k], keep=dumping and k == K - 1)
    e1.record()
    barrier()
    t1 = time.time()
    launches = _cabi.launch_count() - launches0
    elapsed_ms = e0.elapsed_time(e1)
    clocks = sampler.stop(t0, t1) if sampler else None
    if rank == 0 and dumping:
        dump_outputs(args.dump_outputs, [c['name'] for c in calls], last)
    del last

    # per-kernel average durations (fwd: events 0->1, bwd: events 1->2; bwd includes its grad_value zero-fill)
    kernels = []
    for ci, c in enumerate(calls):
        fwd = sum(ev[k][ci][0].elapsed_time(ev[k][ci][1]) for k in range(K)) / K
        bwd = sum(ev[k][ci][1].elapsed_time(ev[k][ci][2]) for k in range(K)) / K
        kernels.append({'name': c['name'] + '_fwd', 'ms': fwd, 'alg_bytes': c['bytes']['fwd'], 'pts': c['pts']})
        kernels.append({'name': c['name'] + '_bwd', 'ms': bwd, 'alg_bytes': c['bytes']['bwd'], 'pts': c['pts']})

    # ---- max over ranks -----------------------------------------------------------------------------------
    elapsed_ms = max_over_ranks(elapsed_ms, dev)
    ms_per_step = elapsed_ms / K
    value = world * pts_step / (ms_per_step * 1e-3) / 1e9

    # ---- e2e: public API (MSDeformAttnFunction.apply + autograd) from pinned HOST buffers -------------------
    # Every step copies ITS inputs host->device and ITS results (out + 3 gradients) device->host. The three
    # phases run on three streams (copy-in / compute / copy-out) with double-buffered device inputs and pinned
    # host result buffers, so step k+1's upload and step k-1's download overlap step k's kernels (full-duplex
    # PCIe). Steady-state throughput; all bytes of every step are inside the timed region.
    s_in, s_cmp, s_out = torch.cuda.Stream(), torch.cuda.Stream(), torch.cuda.Stream()
    in_keys = ('value', 'loc', 'aw', 'grad_out', 'shapes', 'lsi')
    dev_in = [[{k: torch.empty_like(c['host'][k], device=dev) for k in in_keys} for c in calls] for _ in range(2)]
    host_out = [[[torch.empty(c['host']['grad_out'].shape, dtype=dtype).pin_memory(),
                  torch.empty(c['host']['value'].shape, dtype=dtype).pin_memory(),
                  torch.empty(c['host']['loc'].shape, dtype=torch.float32).pin_memory(),
                  torch.empty(c['host']['aw'].shape, dtype=torch.float32).pin_memory()] for c in calls] for _ in range(2)]
    ev_in = [torch.cuda.Event() for _ in range(2)]
    ev_free = [torch.cuda.Event() for _ in range(2)]     # compute finished reading dev_in[slot]
    ev_outfree = [torch.cuda.Event() for _ in range(2)]  # copy-out finished with host_out[slot]
    keep = [None, None]

    def run_e2e(nsteps):
        for k in range(nsteps):
            slot = k & 1
            with torch.cuda.stream(s_in):
                if k >= 2:
                    s_in.wait_event(ev_free[slot])
                for ci, c in enumerate(calls):
                    for key in in_keys:
                        dev_in[slot][ci][key].copy_(c['host'][key], non_blocking=True)
                ev_in[slot].record(s_in)
            with torch.cuda.stream(s_cmp):
                s_cmp.wait_event(ev_in[slot])
                results = []
                for ci, c in enumerate(calls):
                    d = dev_in[slot][ci]
                    v = d['value'].detach().requires_grad_()
                    loc = d['loc'].detach().requires_grad_()
                    aw = d['aw'].detach().requires_grad_()
                    out = vab.MSDeformAttnFunction.apply(v, d['shapes'], d['lsi'], loc, aw, 64)
                    out.backward(d['grad_out'])
                    results.append((out.detach(), v.grad, loc.grad, aw.grad))
                ev_free[slot].record(s_cmp)
            with torch.cuda.stream(s_out):
                s_out.wait_event(ev_free[slot])
                # the pinned result buffers of this slot were last written two steps ago ON THIS STREAM: stream order
                # already keeps the new copy behind the old one, so the host never has to block here
                for ci, res in enumerate(results):
                    for dst, src in zip(host_out[slot][ci], res):
                        src.record_stream(s_out)
                        dst.copy_(src, non_blocking=True)
                ev_outfree[slot].record(s_out)
            keep[slot] = results
        for st in (s_in, s_cmp, s_out):
            st.synchronize()

    h2d = sum(sum(c['host'][k].numel() * c['host'][k].element_size() for k in in_keys) for c in calls)
    d2h = sum(sum(t.numel() * t.element_size() for t in bufs) for bufs in host_out[0])
    e2e_steps = max(4, min(K, 50))   # per pass; each pass includes the pipeline's fill and drain, five passes are timed
    # warm-up: W steps, then one full untimed pass of the same length as the timed ones (the first pass after the
    # device-resident phase was 3.5x slower than the following ones in round 1: pinned result buffers touched for the first
    # time by the DMA engine and the copy streams' first use all land in it)
    run_e2e(max(4, args.warmup))
    run_e2e(e2e_steps)
    # the host link is noisy from one pass to the next (8.6 - 12 ms per step seen on one box): five passes of K steps
    # each, every pass timed on the device as the max over ranks; the MEDIAN pass is reported and all five are listed
    e2e_runs = []
    for _ in range(5):
        barrier()
        a0, a1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a0.record()
        run_e2e(e2e_steps)
        a1.record()
        barrier()
        t_ms = max_over_ranks(a0.elapsed_time(a1), dev)  # device clock: a1 is recorded after run_e2e synchronised all three streams
        e2e_runs.append(t_ms)
    e2e_ms = statistics.median(e2e_runs)
    e2e_value = world * pts_step / (e2e_ms / e2e_steps * 1e-3) / 1e9
    del dev_in, keep

    # ---- reference CUDA kernel on the same GPU, same inputs (fp32 only; informational) ---------------------
    ref_cuda = None
    if rank == 0 and not args.no_ref_cuda:
        try:
            from oracle import refcuda
            if refcuda.available():
                f32 = [{k: (v.float() if v.is_floating_point() else v) for k, v in c['dev'].items()} for c in calls]

                def step_ref():
                    for d in f32:
                        refcuda.forward(d['value'], d['shapes'], d['lsi'], d['loc'], d['aw'])
                        refcuda.backward(d['value'], d['shapes'], d['lsi'], d['loc'], d['aw'], d['grad_out'])
                for _ in range(2):
                    step_ref()
                torch.cuda.synchronize()
                r0, r1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                nref = max(2, min(K, 10))
                r0.record()
                for _ in range(nref):
                    step_ref()
                r1.record()
                torch.cuda.synchronize()
                rms = r0.elapsed_time(r1) / nref
                ref_cuda = {'what': "reference's own CUDA kernels (ms_deform_im2col_cuda.cuh) recompiled for sm_100a, fp32, "
                                    'same inputs, 1 GPU', 'ms_per_step': rms, 'value': pts_step / (rms * 1e-3) / 1e9,
                            'unit': 'Gsamples/s', 'steps': nref}
                del f32
        except Exception as e:  # informational only
            ref_cuda = {'error': repr(e)}

    # ---- the other BASELINE shapes, rank 0. The north star's target configuration is ViT-Adapter-L at 896^2 in bf16
    #      (16 heads x 32 channels as the reference configures it, and 16 x 64 as BASELINE.json words it): those two get a
    #      roofline-grade block of their own (per-kernel CUDA events, L2 flushed before every launch, median of 30, HBM
    #      traffic per launch from the committed ncu capture in profiles/traffic.json) ---------------------------------
    other = None
    north_star = None
    if rank == 0 and not args.no_other_shapes:
        other = []
        north_star = []
        peak_o = (float(json.load(open(os.path.join(ROOT, 'MEASURED_PEAKS.json')))['hbm_gbs'])
                  if os.path.exists(os.path.join(ROOT, 'MEASURED_PEAKS.json')) else 6650.0)
        try:
            traffic_all = json.load(open(os.path.join(ROOT, 'profiles', 'traffic.json')))
        except Exception:
            traffic_all = {}
        flushbuf = torch.empty(256 << 20, dtype=torch.uint8, device=dev)
        for ov, odt in (('L', 'bf16'), ('L64', 'bf16'), ('L', 'f32'), ('B', 'bf16'), ('HTC', 'f32'), ('M2F', 'bf16'), ('M2F', 'f32')):
            if ov == variant and odt == args.dtype:
                continue
            oM, oD, oside, ob = VARIANTS[ov]
            tdt = torch.float32 if odt == 'f32' else torch.bfloat16
            reps = 30 if ov in ('L', 'L64') else 10
            tot_ms, tot_pts, tot_bytes, per_kernel = 0.0, 0, 0, []
            for ci, (name, N_, M_, D_, Lq_, shp) in enumerate(call_shapes(ov, ob)):
                hin = adapter_inputs(name, N_, M_, D_, Lq_, shp, seed=77 + ci, dtype=tdt)
                din = {k: v.to(dev) for k, v in hin.items()}
                ab = algorithmic_bytes(N_, M_, D_, Lq_, shp, 4 if odt == 'f32' else 2)
                fw = lambda: _cabi.forward(din['value'], din['shapes'], din['lsi'], din['loc'], din['aw'], 64)
                bw = lambda: _cabi.backward(din['value'], din['shapes'], din['lsi'], din['loc'], din['aw'], din['grad_out'], 64)
                for fn, key in ((fw, 'fwd'), (bw, 'bwd')):
                    if ov == 'HTC' and key == 'bwd':
                        continue  # inference shape
                    for _ in range(3):
                        fn()
                    ts = []
                    for _ in range(reps):
                        flushbuf.zero_()
                        x0, x1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                        x0.record()
                        fn()
                        x1.record()
                        torch.cuda.synchronize()
                        ts.append(x0.elapsed_time(x1))
                    ts.sort()
                    med = ts[len(ts) // 2]
                    tot_ms += med
                    tot_bytes += ab[key]
                    kname = '%s_%s' % (name, key)
                    per_kernel.append({'name': kname, 'us': med * 1e3, 'min_us': ts[0] * 1e3, 'alg_bytes': ab[key],
                                       'gbs': ab[key] / (med * 1e-3) / 1e9, 'frac': ab[key] / (med * 1e-3) / 1e9 / peak_o,
                                       'gsamples_s': n_points(N_, M_, Lq_, len(shp)) / (med * 1e-3) / 1e9,
                                       'traffic': traffic_all.get('%s_%s_%s' % (ov, odt, kname))})
                tot_pts += n_points(N_, M_, Lq_, len(shp))
            entry = {'variant': ov, 'dtype': odt, 'image': oside, 'batch': ob, 'heads': oM, 'channels': oD,
                     'what': ('encoder self-attention ' if ov == 'M2F' else 'Injector+Extractor ') + ('fwd' if ov == 'HTC' else 'fwd+bwd')
                             + ', L2 flushed before every launch, median of %d' % reps,
                     'us': tot_ms * 1e3, 'gsamples_s': tot_pts / (tot_ms * 1e-3) / 1e9,
                     'hbm_frac': tot_bytes / (tot_ms * 1e-3) / 1e9 / peak_o, 'kernels': per_kernel}
            if ov in ('L', 'L64') and odt == 'bf16':
                dom_o = max(per_kernel, key=lambda k: k['us'])
                entry['roofline'] = {'bound': 'hbm', 'kernel': dom_o['name'], 'achieved': dom_o['gbs'], 'peak': peak_o, 'unit': 'GB/s',
                                     'frac': dom_o['frac'], 'traffic': dom_o['traffic'], 'step_frac': entry['hbm_frac']}
                entry['target'] = 'north star: fwd+bwd at >= 0.60 of the HBM roofline (step_frac)'
                north_star.append(entry)
            else:
                other.append(entry)
        del flushbuf

    # ---- informational: the adapter-side kernels around the op (SURVEY §8(f) N1-N3), B 16 x 512^2 bf16-autocast shapes ----
    adapter_kernels = None
    if rank == 0 and not args.no_other_shapes:
        try:
            adapter_kernels = time_adapter_kernels(dev)
        except Exception as exc:  # never let an informational block cost the bench line
            adapter_kernels = {'error': repr(exc)[:200]}

    # ---- roofline of the dominant kernel ------------------------------------------------------------------
    peaks_path = os.path.join(ROOT, 'MEASURED_PEAKS.json')
    if os.path.exists(peaks_path):
        peak = float(json.load(open(peaks_path))['hbm_gbs'])
        peak_src = 'measured (MEASURED_PEAKS.json hbm_gbs)'
    else:
        peak, peak_src = 6650.0, 'fallback (B200_PROFILING.md)'
    dom = max(kernels, key=lambda k: k['ms'])
    for k in kernels:
        k['gbs'] = k['alg_bytes'] / (k['ms'] * 1e-3) / 1e9
        k['frac'] = k['gbs'] / peak
        k['gsamples_s'] = k['pts'] / (k['ms'] * 1e-3) / 1e9
    traffic = None
    tpath = os.path.join(ROOT, 'profiles', 'traffic.json')
    if os.path.exists(tpath):
        try:
            traffic = json.load(open(tpath)).get('%s_%s_%s' % (variant, args.dtype, dom['name']))
        except Exception:
            traffic = None
    roofline = {'bound': 'hbm', 'kernel': dom['name'], 'achieved': dom['gbs'], 'peak': peak, 'unit': 'GB/s',
                'frac': dom['frac'], 'traffic': traffic, 'peak_source': peak_src,
                'step_frac': sum(k['alg_bytes'] for k in kernels) / (sum(k['ms'] for k in kernels) * 1e-3) / 1e9 / peak}

    # ---- CPU baseline (rank 0, N=1 only; bounded sample) ----------------------------------------------------
    cpu_baseline = None
    if rank == 0 and world == 1 and not args.no_cpu_baseline:
        os.sched_setaffinity(0, all_cpus)   # the CPU arm gets every host core again (the GPU arm was pinned to its NUMA node)
        threads = os.cpu_count() or 1
        sb = min(batch, 2)
        cv, csec, cpts = cpu_reference_pass(variant, sb, threads, steps=3, warmup=1)
        cv1, _, _ = cpu_reference_pass(variant, sb, 1, steps=1, warmup=1)   # SURVEY §8(d): "... and also 1 thread"
        cpu_baseline = {'value': cv, 'unit': 'Gsamples/s', 'cores': threads, 'kind': 'port', 'value_1_thread': cv1,
                        'sample': '%d of %d images, Injector+Extractor fwd+bwd, oracle/core_pytorch.py (restatement of the '
                                  "reference's ms_deform_attn_core_pytorch), %.0f ms per pass" % (sb, batch, csec * 1e3)}

    # ---- the batch-sharded TRAINING STEP (BASELINE.json configs[2] / [3]; north star: "near-linear 1->8-GPU images/s on
    #      the adapter training step", NCCL only for DDP's gradient all-reduce). Every rank takes part. -----------------
    step_block = None
    used_graph_ddp = False
    if not args.no_step:
        from bench_step import step_bench
        step_block = {}
        plans = [('B_512_train_bf16_2img_eager', dict(variant='B', image=512, batch=2, amp=True, graph=False, steps=10, warmup=5)),
                 # the same eager step with vit_adapter_b200.adapter.SyncBatchNormNoHostSync in the SPM / output norms (identical
                 # statistics and results; torch's SyncBatchNorm synchronises the host 3x per layer and forward)
                 ('B_512_train_bf16_2img_eager_nosync_bn', dict(variant='B', image=512, batch=2, amp=True, graph=False, steps=10, warmup=5, bn='nosync')),
                 ('B_512_train_bf16_2img_graph', dict(variant='B', image=512, batch=2, amp=True, graph=True, steps=20, warmup=5)),
                 ('L_896_train_bf16_1img_cp_eager', dict(variant='L', image=896, batch=1, amp=True, with_cp=True, graph=False, steps=5, warmup=3)),
                 ('L_896_train_bf16_1img_cp_graph', dict(variant='L', image=896, batch=1, amp=True, with_cp=True, graph=True, steps=10, warmup=3))]
        for key, kw in plans:
            try:
                r = step_bench(mode='train', **kw)
                used_graph_ddp = used_graph_ddp or (kw['graph'] and world > 1)
                step_block[key] = {'img_per_s': r['value'], 'ms_per_step': r['ms_per_step'], 'n_gpus': r['n_gpus'],
                                   'allreduce_bytes': r['allreduce_bytes'], 'allreduce_ms_exposed': r['allreduce_ms_exposed'],
                                   'cuda_graph': r['cuda_graph'], 'batchnorm': r['batchnorm'], 'msda_kernel_launches': r['msda_kernel_launches'],
                                   'params_total': r['config']['params_total'], 'params_adapter': r['config']['params_adapter'],
                                   'workload': r['config']['workload'], 'parallelism': r['config']['parallelism']}
            except Exception as exc:  # a failing model-level block must not cost the operator bench line
                step_block[key] = {'error': repr(exc)[:300]}
                if world > 1:
                    break   # the ranks may no longer be in step: do not start another collective workload
        step_block['note'] = ('ViT trunk and head are minimal stand-ins (mmcv / mmseg / timm absent); the adapter path (SPM, Injector, '
                              'Extractor, MSDeformAttn) is the drop-in code. allreduce_ms_exposed = eager step time minus the same '
                              'steps under DDP.no_sync(). Weak scaling: images per GPU fixed.')

    if rank == 0:
        line = {
            'metric': 'msdeformattn_fwd_bwd_gsamples_per_s', 'value': value, 'unit': 'Gsamples/s', 'n_gpus': world,
            'steps': K, 'warmup': args.warmup, 'ms_per_step': ms_per_step, 'higher_is_better': True, 'scaling': 'weak',
            'vs_baseline': None, 'dtype': args.dtype, 'data': 'synthetic',
            'config': workload_config(variant, batch, args.dtype),
            'roofline': roofline, 'cpu_baseline': cpu_baseline,
            'e2e': {'value': e2e_value, 'unit': 'Gsamples/s', 'h2d_bytes_per_step': h2d, 'd2h_bytes_per_step': d2h,
                    'ms_per_step': e2e_ms / e2e_steps, 'steps': e2e_steps, 'passes_ms_per_step': [r / e2e_steps for r in e2e_runs], 'reported': 'median of the passes', 'api': 'MSDeformAttnFunction.apply + autograd backward; pinned host buffers; copy-in / compute / copy-out on 3 streams, double-buffered'},
            'gpu_launches': launches, 'clocks': clocks, 'kernels': kernels, 'ref_cuda': ref_cuda,
            'points_per_step_per_gpu': pts_step, 'north_star': north_star, 'other_shapes': other, 'adapter_kernels': adapter_kernels,
            'step': step_block, 'shard': {'global_batch': world * batch, 'samples': [shard_begin, shard_end]},
            'host_affinity': numa,
        }
        emit(line)
    if world > 1:
        dist.barrier()
        if used_graph_ddp:
            # tearing the NCCL communicator down after its collectives were captured in a CUDA graph hung on the test box:
            # the line is out, every rank has passed the barrier - leave without the destructor
            torch.cuda.synchronize()
            sys.stdout.flush()
            sys.stderr.flush()
            os._exit(0)
        dist.destroy_process_group()
    return 0


def bind_host_thread_to_gpu(dev):
    """Pin this process to the CPUs NVML reports as local to its GPU, BEFORE any pinned host buffer is allocated, so the
    e2e arm's staging buffers are first-touched on the GPU's own NUMA node (with one rank per GPU and no binding, half
    of the ranks copy across the socket interconnect). Returns a short description for the JSON line, or None."""
    try:
        import pynvml
        import torch
        pynvml.nvmlInit()
        h = None
        try:
            uuid = str(torch.cuda.get_device_properties(dev).uuid)
            for cand in ('GPU-' + uuid, uuid):
                try:
                    h = pynvml.nvmlDeviceGetHandleByUUID(cand.encode() if hasattr(cand, 'encode') else cand)
                    break
                except Exception:
                    h = None
        except Exception:
            h = None
        if h is None:
            vis = os.environ.get('CUDA_VISIBLE_DEVICES')
            idx = int(vis.split(',')[dev.index]) if vis and vis.split(',')[dev.index].isdigit() else dev.index
            h = pynvml.nvmlDeviceGetHandleByIndex(idx)
        words = (os.cpu_count() + 63) // 64
        mask = pynvml.nvmlDeviceGetCpuAffinity(h, words)
        cpus = [w * 64 + b for w, m in enumerate(mask) for b in range(64) if (int(m) >> b) & 1]
        allowed = sorted(set(cpus) & set(os.sched_getaffinity(0)))
        if not allowed:
            return None
        os.sched_setaffinity(0, allowed)
        return {'cpus': '%d-%d' % (allowed[0], allowed[-1]), 'n': len(allowed)}
    except Exception:
        return None


def time_adapter_kernels(dev):
    """LayerNorm fwd / bwd (+ folded residual gradient), DWConv fwd / grad_x / grad_w, bias-gradient column sum and residual
    add, each alone through the C ABI binding at the ViT-Adapter-B 16 x 512^2 shapes (86 016 tokens x 768 / 192 channels,
    fp32 stream, bf16 branches). CUDA events around back-to-back calls that rotate through > 512 MB of distinct inputs;
    HBM fraction on the compulsory bytes of each kernel."""
    import torch
    from vit_adapter_b200 import _cabi
    peaks_path = os.path.join(ROOT, 'MEASURED_PEAKS.json')
    peak = float(json.load(open(peaks_path))['hbm_gbs']) if os.path.exists(peaks_path) else 6650.0
    B, n, C, H = 16, 5376, 768, 32
    rows = B * n
    nset = 3
    xs = [torch.randn(B, n, C, device=dev) for _ in range(nset)]
    gys = [torch.randn(B, n, C, device=dev).bfloat16() for _ in range(nset)]
    w, b = 1 + 0.1 * torch.randn(C, device=dev), 0.1 * torch.randn(C, device=dev)
    stats = [_cabi.layernorm_forward(x, w, b, 1e-6, torch.bfloat16)[1] for x in xs]
    hid = C // 4
    hx = [torch.randn(B, n, hid, device=dev).bfloat16() for _ in range(2 * nset)]
    dw, db = torch.randn(hid, 1, 3, 3, device=dev).bfloat16(), torch.randn(hid, device=dev).bfloat16()
    e32, e16 = 4 * rows * C, 2 * rows * C
    h16 = 2 * rows * hid
    cases = [
        ('layernorm_fwd f32->bf16', lambda i: _cabi.layernorm_forward(xs[i % nset], w, b, 1e-6, torch.bfloat16), e32 + e16),
        ('layernorm_bwd (+residual grad)', lambda i: _cabi.layernorm_backward(gys[i % nset], xs[i % nset], w, stats[i % nset], xs[(i + 1) % nset]),
         3 * e32 + e16),
        ('dwconv_fwd bf16', lambda i: _cabi.dwconv_forward(hx[i % (2 * nset)], dw, db, H, H), 2 * h16),
        ('dwconv_bwd bf16 (grad_x + grad_w)', lambda i: _cabi.dwconv_backward(hx[i % (2 * nset)], dw, hx[(i + 1) % (2 * nset)], H, H), 4 * h16),
        ('colsum bf16 [86016, 768]', lambda i: _cabi.colsum(gys[i % nset]), e16),
        ('residual_add f32 + bf16', lambda i: _cabi.residual_add(xs[i % nset], gys[i % nset]), 2 * e32 + e16),
    ]
    out = []
    for name, fn, nbytes in cases:
        for i in range(3):
            fn(i)
        torch.cuda.synchronize()
        reps = 12
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for i in range(reps):
            fn(i)
        e1.record()
        torch.cuda.synchronize()
        us = e0.elapsed_time(e1) * 1e3 / reps
        out.append({'name': name, 'us': us, 'alg_bytes': nbytes, 'gbs': nbytes / us / 1e3, 'hbm_frac': nbytes / us / 1e3 / peak})
    return out


class _StdoutGuard:
    """Keep stdout clean: everything any library prints to fd 1 while we run (NCCL prints its version banner
    there) goes to stderr; only emit() writes to the real stdout — exactly one JSON line."""

    def __init__(self):
        sys.stdout.flush()
        self.real = os.dup(1)
        os.dup2(2, 1)

    def emit(self, line):
        sys.stdout.flush()
        os.write(self.real, (line + '\n').encode())


_GUARD = None


def emit(obj):
    line = json.dumps(obj)
    if _GUARD is not None:
        _GUARD.emit(line)
    else:
        print(line, flush=True)


def main():
    global _GUARD
    _GUARD = _StdoutGuard()
    ap = argparse.ArgumentParser()
    ap.add_argument('--gpus', type=int, default=1)
    ap.add_argument('--steps', type=int, default=20,
                    help='timed steps of the headline metric (the e2e arm clamps to 4..50 per pass, ref_cuda to 2..10)')
    ap.add_argument('--warmup', type=int, default=5)
    ap.add_argument('--impl', default='ours', choices=['ours', 'reference'])
    ap.add_argument('--variant', default='B', choices=sorted(VARIANTS))
    ap.add_argument('--dtype', default='f32', choices=['f32', 'bf16'])
    ap.add_argument('--batch', type=int, default=0, help='images per GPU (0 = the variant default)')
    ap.add_argument('--no-cpu-baseline', action='store_true')
    ap.add_argument('--no-ref-cuda', action='store_true')
    ap.add_argument('--no-other-shapes', action='store_true')
    ap.add_argument('--no-step', action='store_true', help='skip the model-level training-step block (bench_step.step_bench)')
    ap.add_argument('--dump-outputs', metavar='DIR', default=None,
                    help='after the timed steps, write what the last one computed (rank 0) as DIR/<call>_<array>.npy')
    args = ap.parse_args()
    if args.steps < 1:
        ap.error('--steps must be at least 1')
    if args.dump_outputs and args.impl != 'ours':
        ap.error('--dump-outputs records the GPU path (--impl ours)')
    if args.warmup < 3 and args.impl == 'ours':
        args.warmup = 3
    if args.impl == 'reference':
        return run_reference_arm(args)  # each step: a bounded 2-image sample, ~0.2-1 s of CPU work
    return run_ours(args)


if __name__ == '__main__':
    sys.exit(main())
