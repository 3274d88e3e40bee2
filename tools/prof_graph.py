"""Time the graph build alone: 8 synthetic 20 000-point frames per call through gen_multi_level_local_graph_v3 with the
car_auto_T3 graph kwargs (the graph stage of bench.py's default workload).

    python tools/prof_graph.py [--frames 8] [--reps 40] [--rounds 5] [--variant NAME=lib.so ...] [--out FILE]

A variant is a build of libpointgnn_b200.so; the build in the tree is always measured, as "tree".  Each round times
`reps` calls of every variant in turn, in one process, so that two builds are compared under the same conditions.
Every call starts with L2 flushed (as in bench.py) and is timed between CUDA events; the wall clock includes the
call's one host round trip.  A separate torch.profiler pass per variant then lists the kernels of `reps` calls: their
summed device time against the event time shows how much of the stage the GPU spends waiting for the host."""
import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
from oracle import synth  # noqa: E402
from pointgnn_b200 import _lib  # noqa: E402
from pointgnn_b200.models import graph_gen  # noqa: E402


def use(lib_path):
    """Point pointgnn_b200._lib at another build (loaded once, then switched)."""
    _lib._lib = None
    _lib.LIB_PATH = lib_path
    return _lib.load()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument('--frames', type=int, default=8)
    ap.add_argument('--reps', type=int, default=40)
    ap.add_argument('--rounds', type=int, default=5)
    ap.add_argument('--variant', action='append', default=[], help='NAME=path of another libpointgnn_b200.so')
    ap.add_argument('--out', default=None, help='also write the report (JSON) here')
    args = ap.parse_args()
    variants = {'tree': os.path.join(ROOT, 'point-gnn_b200', 'libpointgnn_b200.so')}
    for v in args.variant:
        name, path = v.split('=', 1)
        variants[name] = os.path.abspath(path)
    libs = {name: use(path) for name, path in variants.items()}

    cfg = json.load(open(os.path.join(ROOT, 'tests/golden/config_car_auto_T3_train.json')))
    gkw = cfg['runtime_graph_gen_kwargs']
    n = 20000
    batches = []
    for b in range(4):
        pts = np.vstack([synth.lidar_frame(100 + b * args.frames + i, n)[0] for i in range(args.frames)])
        batches.append(torch.from_numpy(pts).cuda())
    fp = torch.arange(args.frames + 1, dtype=torch.int32, device='cuda') * n
    flush = torch.empty(256 << 20, dtype=torch.uint8, device='cuda')      # > 126 MB L2

    def call(r):
        return graph_gen.gen_multi_level_local_graph_v3(batches[r % 4], frame_ptr=fp, **gkw)

    # outputs must agree between the builds before their times mean anything
    ref = None
    for name, lib in libs.items():
        _lib._lib = lib
        for r in range(8):
            call(r)
        coords, kp, edges = call(0)
        out = [kp[0].cpu(), edges[0].cpu(), edges[1].cpu()]
        if ref is None:
            ref = out
        assert all(torch.equal(a, b) for a, b in zip(out, ref)), '%s computes a different graph' % name
    torch.cuda.synchronize()

    ev_ms = {name: [] for name in libs}
    wall_ms = {name: [] for name in libs}
    for rnd in range(args.rounds):
        for name, lib in libs.items():
            _lib._lib = lib
            for r in range(args.reps):
                flush.zero_()
                torch.cuda.synchronize()
                a, z = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                t0 = time.perf_counter()
                a.record()
                call(r)
                z.record()
                z.synchronize()
                wall_ms[name].append((time.perf_counter() - t0) * 1e3)
                ev_ms[name].append(a.elapsed_time(z))

    kernels = {}
    for name, lib in libs.items():
        _lib._lib = lib
        per = {}
        with torch.profiler.profile(activities=[torch.profiler.ProfilerActivity.CUDA]) as prof:
            for r in range(args.reps):
                flush.zero_()
                torch.cuda.synchronize()
                call(r)
        for e in prof.key_averages():
            t = getattr(e, 'self_device_time_total', None)
            if t is None:
                t = e.self_cuda_time_total
            if t > 0 and 'zero_' not in e.key and 'fill' not in e.key.lower():
                per[e.key[:90]] = (t / 1e3 / args.reps, e.count / args.reps)
        kernels[name] = per

    smi = subprocess.run(['nvidia-smi', '--query-gpu=name,power.limit,clocks.max.sm', '--format=csv,noheader'],
                         capture_output=True, text=True).stdout.strip()
    report = {'gpu': smi, 'frames_per_call': args.frames, 'points_per_frame': n, 'reps': args.reps,
              'rounds': args.rounds, 'variants': {}}
    for name in libs:
        ev = np.array(ev_ms[name]).reshape(args.rounds, args.reps)
        per = kernels[name]
        ksum = sum(t for t, _ in per.values())
        report['variants'][name] = {
            'event_ms_median': float(np.median(ev)), 'event_ms_round_medians': np.median(ev, axis=1).round(4).tolist(),
            'wall_ms_median': float(np.median(wall_ms[name])),
            'kernel_ms_sum_per_call': ksum, 'launches_per_call': sum(c for _, c in per.values()),
            'kernels_ms_per_call': {k: round(t, 4) for k, (t, _) in sorted(per.items(), key=lambda kv: -kv[1][0])}}
    print('gpu: %s' % smi)
    for name, v in report['variants'].items():
        print('%-8s event %.3f ms/call (round medians %s), wall %.3f ms, kernels %.3f ms/call in %.1f launches '
              '-> host gaps %.3f ms' % (name, v['event_ms_median'], v['event_ms_round_medians'], v['wall_ms_median'],
                                        v['kernel_ms_sum_per_call'], v['launches_per_call'],
                                        v['event_ms_median'] - v['kernel_ms_sum_per_call']))
        for k, t in list(v['kernels_ms_per_call'].items())[:14]:
            print('    %8.4f  %s' % (t, k))
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, 'w') as f:
            json.dump(report, f, indent=1)


if __name__ == '__main__':
    main()
