"""CUDA-event timing of the self-loop GEMM at the two shapes of bench.py's step, old and new kernel alternated in one process.

    python tools/bench_selfloop.py [--launches 400] [--json OUT]

Layer 1: 34483 rows gathered (with repeats) from the 23033-row entity table; layer 2: 8573 distinct rows of the layer-1
output.  Engine 2 is the packed tcgen05 kernel, engine 1 the persistent self-loop kernel.  As in bench.py, every step is a
new weight generation and makes two calls per shape (the two directions), so the first call of a step includes the
packing launch; each engine has its own weight buffers, so each pays its own packing.  Index arrays rotate over 8 seeds.
"""
import argparse
import json
import os
import subprocess
import sys

import numpy as np
import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from renet_b200 import _lib  # noqa: E402

H = 200
SHAPES = (('layer1', 34483, 23033, True), ('layer2', 8573, 34483, False))   # name, rows, source rows, repeated ids
HBM_GBS = 7700.0        # HGX B200 data sheet, one GPU
TF32_TFLOPS = 1125.0    # HGX B200 data sheet, dense TF32, one GPU (3xTF32 issues 3 products per fp32 multiply-add)


def card():
    try:
        q = subprocess.run(['nvidia-smi', '--query-gpu=name,power.limit,clocks.max.sm', '--format=csv,noheader'],
                           capture_output=True, text=True, timeout=30).stdout.strip().splitlines()[0]
        return q
    except Exception as ex:
        return 'unknown (%s)' % ex


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument('--launches', type=int, default=400, help='timed launches per shape and engine (>= 200)')
    ap.add_argument('--warmup', type=int, default=20)
    ap.add_argument('--json', default=None)
    args = ap.parse_args()
    L = _lib.lib()
    dev = 'cuda:0'
    torch.manual_seed(0)
    stream = _lib.stream()
    P = _lib.ptr
    data = {}
    for name, M, src_rows, repeats in SHAPES:
        src = torch.randn(src_rows, H, device=dev) * 0.3
        idx = []
        for s in range(8):
            g = torch.Generator(device='cpu').manual_seed(100 + s)
            ids = torch.randint(0, src_rows, (M,), generator=g) if repeats else torch.randperm(src_rows, generator=g)[:M]
            idx.append(ids.to(torch.int32).to(dev))
        w = torch.randn(H, H, device=dev) * 0.1
        data[name] = {'M': M, 'src': src, 'idx': idx, 'W': {1: w.clone(), 2: w.clone()},
                      'out': {1: torch.empty(M, H, device=dev), 2: torch.empty(M, H, device=dev)}}

    def step(gen, eng, i):
        L.renet_set_gemm_engine(eng)
        L.renet_set_weight_generation(gen)
        for name, _, _, _ in SHAPES:
            d = data[name]
            for call in range(2):
                _lib.check(L.renet_selfloop_gemm(P(d['src']), P(d['idx'][(2 * i + call) % 8]), P(d['W'][eng]), P(d['out'][eng]),
                                                 d['M'], H, H, stream), 'selfloop')
        L.renet_set_weight_generation(-1)

    gen = 0
    for i in range(args.warmup):
        for eng in (2, 1):
            gen += 1
            step(gen, eng, i)
    torch.cuda.synchronize()
    # timed: per step and engine, two calls per shape, each between its own pair of events
    times = {(n, e): [] for n, _, _, _ in SHAPES for e in (1, 2)}
    n_steps = max(1, args.launches // 2)
    pending = []
    for i in range(n_steps):
        for eng in ((2, 1) if i % 2 == 0 else (1, 2)):
            gen += 1
            L.renet_set_gemm_engine(eng)
            L.renet_set_weight_generation(gen)
            for name, _, _, _ in SHAPES:
                d = data[name]
                for call in range(2):
                    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                    a.record()
                    _lib.check(L.renet_selfloop_gemm(P(d['src']), P(d['idx'][(2 * i + call) % 8]), P(d['W'][eng]),
                                                     P(d['out'][eng]), d['M'], H, H, stream), 'selfloop')
                    b.record()
                    pending.append(((name, eng), a, b))
            L.renet_set_weight_generation(-1)
    torch.cuda.synchronize()
    for key, a, b in pending:
        times[key].append(a.elapsed_time(b) * 1e3)
    # same inputs through both engines: outputs of the last call are compared
    diffs = {}
    for name, _, _, _ in SHAPES:
        d = data[name]
        for eng in (2, 1):
            L.renet_set_gemm_engine(eng)
            _lib.check(L.renet_selfloop_gemm(P(d['src']), P(d['idx'][0]), P(d['W'][eng]), P(d['out'][eng]), d['M'], H, H, stream),
                       'selfloop')
        torch.cuda.synchronize()
        diffs[name] = float((d['out'][1] - d['out'][2]).abs().max().item())
    L.renet_set_gemm_engine(1)
    res = {'card': card(), 'launches_per_engine_and_shape': len(times[(SHAPES[0][0], 1)]), 'shapes': {}}
    for name, M, _, _ in SHAPES:
        flops3 = 3 * 2.0 * M * H * H
        bytes_ = M * (H * 4 * 2 + 4) + H * H * 4
        tensor_floor_us = flops3 / (TF32_TFLOPS * 1e12) * 1e6
        hbm_floor_us = bytes_ / (HBM_GBS * 1e9) * 1e6
        row = {'rows': M, 'max_abs_new_minus_old': diffs[name]}
        for eng, label in ((2, 'old_packed'), (1, 'new_persistent')):
            t = np.array(times[(name, eng)])
            us = float(np.mean(t))
            row[label] = {'us_per_launch': us, 'median_us': float(np.median(t)), 'p10_us': float(np.percentile(t, 10)),
                          'p90_us': float(np.percentile(t, 90)), 'tflops_3xtf32': flops3 / (us * 1e-6) / 1e12,
                          'frac_tensor_floor': tensor_floor_us / us, 'frac_hbm_floor': hbm_floor_us / us}
        row['tensor_floor_us'] = tensor_floor_us
        row['hbm_floor_us'] = hbm_floor_us
        row['speedup'] = row['old_packed']['us_per_launch'] / row['new_persistent']['us_per_launch']
        res['shapes'][name] = row
    res['floors'] = 'tensor: 3xTF32 products at %.0f TFLOP/s dense TF32; hbm: rows in + rows out + weight at %.0f GB/s ' \
                    '(data-sheet figures; the gathered rows are L2-resident at these sizes)' % (TF32_TFLOPS, HBM_GBS)
    print(json.dumps(res, indent=1))
    if args.json:
        with open(args.json, 'w') as fh:
            json.dump(res, fh, indent=1)


if __name__ == '__main__':
    main()
