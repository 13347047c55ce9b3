#!/usr/bin/env python
"""One ViT-Adapter-B interaction, forward + backward in bf16 autocast: eager vs torch.compile vs
torch.compile(mode="reduce-overhead") vs GraphedStep (whole-step CUDA graph).

    python tools/bench_compile.py --images 2 16 --out profiles/r3_compile_interaction.jsonl

The interaction is the model's first one: Injector -> 3 ViT blocks (bench_step.ViTBlock) -> Extractor, d=768, 12 heads,
deform_ratio 0.5, ConvFFN ratio 0.25, 512x512 input (a 32x32 ViT grid), the bf16 sampling kernels under autocast
(set_amp_value_dtype(bfloat16), as bench_step.py --amp). Every arm runs the same step on its own copy of the module and
inputs, built from the same seed: zero the gradients, forward, loss = mean(x^2) + mean(c^2), backward.

Method: each arm is warmed up (the compile arms' first calls compile; their wall time is reported as compile_s), then
`--rounds` rounds each time every arm for `--steps` steps with CUDA events, the arms' order rotating from round to round;
ms_per_step is the median over rounds. The first and last loss of each arm are reported so the arms can be checked to
compute the same thing. One JSON line per (images, arm), with the card name and power limit.
"""
import argparse
import json
import os
import statistics
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

import torch  # noqa: E402


def card():
    q = subprocess.run(['nvidia-smi', '--query-gpu=name,power.limit,clocks.max.sm', '--format=csv,noheader'],
                       capture_output=True, text=True)
    fields = [f.strip() for f in q.stdout.splitlines()[torch.cuda.current_device()].split(',')] if q.returncode == 0 else []
    return {'gpu': torch.cuda.get_device_name(), 'power_limit': fields[1] if len(fields) > 1 else None,
            'max_sm_clock': fields[2] if len(fields) > 2 else None}


def build(images, dim=768, heads=12):
    from bench_step import ViTBlock
    from vit_adapter_b200.adapter import InteractionBlock, deform_inputs
    torch.manual_seed(0)
    dev = torch.device('cuda')
    blk = InteractionBlock(dim=dim, num_heads=heads, n_points=4, init_values=0., drop_path=0., with_cffn=True,
                           cffn_ratio=0.25, deform_ratio=0.5, extra_extractor=False).to(dev)
    vit = torch.nn.ModuleList([ViTBlock(dim, heads) for _ in range(3)]).to(dev)
    params = list(blk.parameters()) + list(vit.parameters())
    h = 512 // 16
    di1, di2 = deform_inputs(torch.zeros(images, 3, 512, 512, device=dev))
    x = (0.5 * torch.randn(images, h * h, dim, device=dev)).requires_grad_()
    c = (0.5 * torch.randn(images, 21 * (h // 2) ** 2, dim, device=dev)).requires_grad_()
    for t in params + [x, c]:
        t.grad = torch.zeros_like(t)
    grads = [t.grad for t in params + [x, c]]

    def forward(x, c):
        return blk(x, c, vit, di1, di2, h, h)
    return forward, x, c, grads


def make_step(forward, x, c, grads, mark_step=False):
    def step():
        if mark_step:
            torch.compiler.cudagraph_mark_step_begin()
        torch._foreach_zero_(grads)
        with torch.autocast('cuda', dtype=torch.bfloat16):
            xo, co = forward(x, c)
        loss = xo.float().square().mean() + co.float().square().mean()
        loss.backward()
        return loss.detach()
    return step


def wall(fn, n=1):
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    out = None
    for _ in range(n):
        out = fn()
    torch.cuda.synchronize()
    return time.perf_counter() - t0, out


def bench(images, rounds, steps, warmup):
    import vit_adapter_b200 as vab
    from vit_adapter_b200.graphs import GraphedStep
    torch._dynamo.reset()
    arms, info = {}, {}

    eager = make_step(*build(images))
    t, loss = wall(eager, warmup)
    arms['eager'], info['eager'] = eager, {'first_loss': float(loss)}

    forward, x, c, grads = build(images)
    default = make_step(torch.compile(forward, fullgraph=True, dynamic=False), x, c, grads)
    t, loss = wall(default)
    info['compile'] = {'compile_s': t, 'first_loss': float(loss)}
    wall(default, warmup)
    arms['compile'] = default

    forward, x, c, grads = build(images)
    ro = make_step(torch.compile(forward, mode='reduce-overhead', fullgraph=True, dynamic=False), x, c, grads, mark_step=True)
    t, loss = wall(ro)
    t2, _ = wall(ro, 2)   # cudagraph trees: the first call runs the compiled code, the next records, then replays
    info['compile_reduce_overhead'] = {'compile_s': t, 'record_s': t2, 'first_loss': float(loss)}
    wall(ro, warmup)
    arms['compile_reduce_overhead'] = ro

    t0 = time.perf_counter()
    gs = GraphedStep(make_step(*build(images)), warmup=warmup)
    torch.cuda.synchronize()
    info['graphed_step'] = {'capture_s': time.perf_counter() - t0}
    _, loss = wall(gs)
    info['graphed_step']['first_loss'] = float(loss)
    arms['graphed_step'] = gs

    names = list(arms)
    per_round = {k: [] for k in names}
    last = {}
    for r in range(rounds):
        for k in names[r % len(names):] + names[:r % len(names)]:
            torch.cuda.synchronize()
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            for _ in range(steps):
                out = arms[k]()
            e1.record()
            torch.cuda.synchronize()
            per_round[k].append(e0.elapsed_time(e1) / steps)
            last[k] = float(out)
    vab.set_amp_value_dtype(torch.float32)
    res = []
    for k in names:
        ms = statistics.median(per_round[k])
        res.append(dict(images=images, arm=k, ms_per_step=ms, img_per_s=images / (ms * 1e-3),
                        ms_min=min(per_round[k]), ms_max=max(per_round[k]), last_loss=last[k], **info[k]))
    del arms, gs, default, ro
    torch._dynamo.reset()
    torch.cuda.synchronize()
    torch.cuda.empty_cache()
    return res


def main():
    ap = argparse.ArgumentParser(description=__doc__.split('\n')[0])
    ap.add_argument('--images', type=int, nargs='+', default=[2, 16])
    ap.add_argument('--rounds', type=int, default=15)
    ap.add_argument('--steps', type=int, default=10, help='steps per arm per round')
    ap.add_argument('--warmup', type=int, default=3)
    ap.add_argument('--out', default=None, help='JSONL file to write (default: print only)')
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit('bench_compile.py needs a CUDA device')
    import vit_adapter_b200 as vab
    vab.set_amp_value_dtype(torch.bfloat16)
    meta = dict(workload='ViT-Adapter-B interaction (Injector + 3 ViT blocks + Extractor), 512x512, fwd+bwd, bf16 autocast',
                torch=torch.__version__, rounds=args.rounds, steps_per_round=args.steps, **card())
    lines = []
    for images in args.images:
        vab.set_amp_value_dtype(torch.bfloat16)
        for row in bench(images, args.rounds, args.steps, args.warmup):
            row.update(meta)
            lines.append(json.dumps(row))
            print(lines[-1], flush=True)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, 'w') as f:
            f.write('\n'.join(lines) + '\n')


if __name__ == '__main__':
    main()
