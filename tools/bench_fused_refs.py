#!/usr/bin/env python
"""tools/bench_fused_refs.py — MSDeformAttn module forward + backward, fused=True against fused=False (the reference's op
sequence), at Deformable-DETR shapes: the 4-level encoder, decoders with box / learned reference points, and the adapter's
Extractor call for comparison.

Every case runs in fp32 and under bf16 autocast with the 16-bit value kernels (set_amp_value_dtype(torch.bfloat16)).
Method: CUDA events around each step; the configurations (and fused / unfused within each) are alternated round by round
in one process, and the median over rounds is reported. Before every timed step the L2 is overwritten by writing a
256 MB buffer (twice the B200's 126 MB L2), outside the timed events, so each step starts from a cold L2. The card's name
and power limit are read in the same run and printed in the first line. Writes JSON lines to stdout and, with --out,
to a file."""
import argparse
import json
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

import torch  # noqa: E402

import vit_adapter_b200 as vab  # noqa: E402
from vit_adapter_b200.adapter import deform_inputs  # noqa: E402

# 800 x 1344 input at strides 8 / 16 / 32 / 64 (Deformable-DETR's 4 encoder levels): S = 22 323
DETR_SHAPES = [(100, 168), (50, 84), (25, 42), (13, 21)]


def _card():
    info = {'device': torch.cuda.get_device_name(0)}
    try:
        out = subprocess.run(['nvidia-smi', '--query-gpu=power.limit,clocks.max.sm', '--format=csv,noheader', '-i', '0'],
                             stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True, timeout=60).stdout.strip()
        info['power_limit_and_max_sm_clock'] = out
    except (OSError, subprocess.SubprocessError) as e:
        info['power_limit_and_max_sm_clock'] = 'not read: %s' % e
    return info


def _module(d_model, L, heads, ratio, dev):
    torch.manual_seed(0)
    m = vab.MSDeformAttn(d_model, L, heads, 4, ratio).to(dev)
    with torch.no_grad():
        for p in m.parameters():
            p.add_(torch.randn_like(p) * 0.02)
    return m


def _detr_cases(dev, N):
    shapes = torch.as_tensor(DETR_SHAPES, dtype=torch.long, device=dev)
    lsi = torch.cat((shapes.new_zeros((1,)), shapes.prod(1).cumsum(0)[:-1]))
    S = int(shapes.prod(1).sum())
    m = _module(256, 4, 8, 1.0, dev)
    memory = torch.randn(N, S, 256, device=dev, requires_grad=True)
    g = torch.Generator(device=dev).manual_seed(1)
    cases = []
    # encoder: every token queries the 4 levels around its own (constant) reference point
    cases.append(('encoder N=%d Lq=S=%d ref[N,S,4,2] no grad' % (N, S), m, memory, torch.rand(N, S, 4, 2, device=dev, generator=g),
                  False, shapes, lsi, memory))
    for Lq in (300, 900):
        q = torch.randn(N, Lq, 256, device=dev, requires_grad=True)
        box = torch.rand(N, Lq, 4, 4, device=dev, generator=g)
        box[..., 2:] *= 0.3
        pts = torch.rand(N, Lq, 4, 2, device=dev, generator=g)
        cases.append(('decoder Lq=%d box ref[N,Lq,4,4] no grad' % Lq, m, q, box, False, shapes, lsi, memory))
        cases.append(('decoder Lq=%d box ref[N,Lq,4,4] with grad' % Lq, m, q, box, True, shapes, lsi, memory))
        cases.append(('decoder Lq=%d learned ref[N,Lq,4,2] with grad' % Lq, m, q, pts, True, shapes, lsi, memory))
    return cases


def _extractor_case(dev, batch, image):
    # ViT-Adapter-B Extractor: d_model 768, 12 heads, ratio 0.5 (D = 32), one level, constant 2-d reference grid
    _, di2 = deform_inputs(torch.zeros(batch, 3, image, image, device=dev))
    h = image // 16
    nq, nf = (2 * h) ** 2 + h * h + (h // 2) ** 2, h * h
    m = _module(768, 1, 12, 0.5, dev)
    q = torch.randn(batch, nq, 768, device=dev, requires_grad=True)
    f = torch.randn(batch, nf, 768, device=dev, requires_grad=True)
    return ('adapter Extractor ViT-Adapter-B bs %d %dpx' % (batch, image), m, q, di2[0], False, di2[1], di2[2], f)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument('--rounds', type=int, default=15)
    ap.add_argument('--warmup', type=int, default=3)
    ap.add_argument('--batch', type=int, default=2, help='N of the Deformable-DETR cases')
    ap.add_argument('--out', default=None)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit('bench_fused_refs.py needs a CUDA device')
    dev = torch.device('cuda', 0)
    lines = [dict(_card(), method='CUDA events per step, median of %d alternated rounds, L2 overwritten (256 MB) before '
                                  'every timed step' % args.rounds)]
    print(json.dumps(lines[0]), flush=True)
    cases = _detr_cases(dev, args.batch) + [_extractor_case(dev, 16, 512)]
    flush = torch.empty(256 << 20, dtype=torch.uint8, device=dev)

    def step(case, amp, fused):
        _, m, q, ref, grad_ref, shapes, lsi, feat = case
        m.fused = fused
        r = ref.detach().requires_grad_(grad_ref)
        with torch.autocast('cuda', dtype=torch.bfloat16, enabled=amp):
            out = m(q, r, feat, shapes, lsi)
        out.float().backward(torch.ones(out.shape, device=out.device))
        return out

    arms = [(i, amp) for i in range(len(cases)) for amp in (False, True)]
    times = {(i, amp, f): [] for i, amp in arms for f in (True, False)}
    try:
        for rnd in range(args.warmup + args.rounds):
            for i, amp in arms:
                vab.set_amp_value_dtype(torch.bfloat16 if amp else torch.float32)
                for fused in (True, False):
                    flush.zero_()
                    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                    e0.record()
                    step(cases[i], amp, fused)
                    e1.record()
                    torch.cuda.synchronize()
                    if rnd >= args.warmup:
                        times[(i, amp, fused)].append(e0.elapsed_time(e1))
    finally:
        vab.set_amp_value_dtype(torch.float32)
    for i, amp in arms:
        med = {}
        for fused in (True, False):
            ts = sorted(times[(i, amp, fused)])
            med[fused] = ts[len(ts) // 2]
        rec = {'case': cases[i][0], 'precision': 'bf16-autocast' if amp else 'fp32', 'fused_ms': round(med[True], 4),
               'unfused_ms': round(med[False], 4), 'speedup': round(med[False] / med[True], 3)}
        lines.append(rec)
        print(json.dumps(rec), flush=True)
    if args.out:
        with open(args.out, 'w') as fh:
            fh.write('\n'.join(json.dumps(x) for x in lines) + '\n')


if __name__ == '__main__':
    main()
