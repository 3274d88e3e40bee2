#!/usr/bin/env python
"""bench.py - KITTI-shape frames/s of the Point-GNN message-passing hot path on B200.

    python bench.py --gpus N --steps K --warmup W [--impl reference] [--workload NAME] [--precision P]
                    [--dump-outputs DIR]

A *step* is one pass of the hot path (GPU graph construction + car_auto_T3 forward, real
trained weights) over one batch of synthetic 20k-point KITTI-crop frames per GPU.  One JSON line is
printed by rank 0 (contract: project brief, "Measurement").

value      whole-job frames/s, inputs resident in HBM, timed with CUDA events per step (max over ranks)
e2e        the same metric through the reference-shaped public API with host (pinned) inputs:
           H2D of points+intensity and D2H of class probabilities + box encodings inside the timing
roofline   dominant kernel = the fused edge-MLP/segment-max kernel of the GNN iterations, timed live
           with CUDA events; achieved = algorithmic FLOPs (E1 * 361 800 per launch, SURVEY 8d) / time
cpu_baseline  the CPU oracle (a port: TF-1.15 cannot be installed) on one frame of the same workload
--impl reference   times that CPU port alone, all host threads, one frame per step
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)
GOLDEN = os.path.join(ROOT, 'tests', 'golden')

WORKLOADS = {
    # name: (config, points per frame, full_360, frames per step per GPU)
    'car_auto_T3_20k': ('car_auto_T3_train', 20000, False, 8),
    'car_auto_T3_120k': ('car_auto_T3_train', 120000, True, 2),
    'ped_cyl_auto_T3_20k_b8': ('ped_cyl_auto_T3_trainval', 20000, False, 8),
}
METRIC = 'KITTI-shape frames/sec (car_auto_T3, graph build + GNN forward)'
UNIT = 'frames/s'
FRAME_POOL = 6     # distinct step inputs the timed loop cycles through (L2 is flushed between steps)
# `ncu --set full` summaries of the dominant kernel, newest first (tools/ncu_summary.py output, committed under
# profiles/): roofline.traffic = dram__bytes_read.sum + dram__bytes_write.sum of one launch is parsed from the first
# one that exists - a measurement taken under the profiler at the default workload, named in the JSON line
NCU_SUMMARIES = ('profiles/r2_seg_tc_ncu_summary.txt', 'profiles/r1_seg_tc_ncu_summary.txt')


def edge_kernel_dram_traffic():
    """-> (bytes per launch or None, file it came from)."""
    for rel in NCU_SUMMARIES:
        path = os.path.join(ROOT, rel)
        if not os.path.isfile(path):
            continue
        total, seen = 0.0, 0
        scale = {'byte': 1.0, 'Kbyte': 1e3, 'Mbyte': 1e6, 'Gbyte': 1e9}
        with open(path) as f:
            for line in f:
                parts = line.split()
                if len(parts) >= 3 and parts[0] in ('dram__bytes_read.sum', 'dram__bytes_write.sum') and parts[1] in scale:
                    total += float(parts[2]) * scale[parts[1]]
                    seen += 1
        if seen == 2:
            return total, rel
    return None, None


def load_config(name):
    with open(os.path.join(GOLDEN, 'config_%s.json' % name)) as f:
        config = json.load(f)
    weights = dict(np.load(os.path.join(GOLDEN, 'weights_%s.npz' % name)))
    return config, weights


def algorithmic_flops(config, k, e0, e1):
    """SURVEY 8d: 2*M*K*N per fully-connected layer; bias / ReLU / max not counted."""
    layers = config['model_kwargs']['layer_configs']
    total = 0
    edge_flops_per_edge = 0
    for lc in layers[:-1]:
        kw = lc['kwargs']
        if lc['type'] == 'scatter_max_point_set_pooling':
            dims = [4] + kw['point_MLP_depth_list']
            total += e0 * sum(2 * a * b for a, b in zip(dims[:-1], dims[1:]))
            dims = [dims[-1]] + kw['output_MLP_depth_list']
            total += k * sum(2 * a * b for a, b in zip(dims[:-1], dims[1:]))
        else:
            d = kw['edge_MLP_depth_list']
            dims = [d[0] + 3] + d
            edge_flops_per_edge = sum(2 * a * b for a, b in zip(dims[:-1], dims[1:]))
            total += e1 * edge_flops_per_edge
            dims = [d[-1]] + kw['update_MLP_depth_list']
            total += k * sum(2 * a * b for a, b in zip(dims[:-1], dims[1:]))
            if kw.get('auto_offset'):
                dims = [d[-1]] + kw['auto_offset_MLP_depth_list']
                total += k * sum(2 * a * b for a, b in zip(dims[:-1], dims[1:]))
    c = config['num_classes']
    dlast = layers[-2]['kwargs']['update_MLP_depth_list'][-1]
    total += k * (2 * dlast * 64 + 2 * 64 * c + c * (2 * dlast * 64 + 2 * 64 * 64 + 2 * 64 * 7))
    return total, edge_flops_per_edge


# ---------------------------------------------------------------------------------------------
# CPU baseline (oracle port) - also the --impl reference arm
# ---------------------------------------------------------------------------------------------
def cpu_frame_seconds(config, weights, frame_idx, num_points, full_360):
    """One frame through the reference's CPU path: sklearn graph build (graph_gen.py, n_jobs=1 as pinned
    there) + the torch-CPU restatement of the TF-1.15 forward on all host cores (oracle/cpu_reference.py)."""
    import warnings
    from oracle import cpu_reference
    from oracle import synth
    xyz, intensity = synth.lidar_frame(frame_idx, num_points, full_360)
    with warnings.catch_warnings():
        warnings.simplefilter('ignore')
        t0 = time.perf_counter()
        coords, kp, edges = cpu_reference.gen_graph(xyz, **config['runtime_graph_gen_kwargs'])
        t1 = time.perf_counter()
        cpu_reference.predict(weights, config['model_kwargs']['layer_configs'], config['num_classes'], 7,
                              intensity, coords, kp, edges, num_threads=cpu_threads())
        t2 = time.perf_counter()
    return t1 - t0, t2 - t1


def cpu_model_name():
    try:
        with open('/proc/cpuinfo') as f:
            for line in f:
                if line.startswith('model name'):
                    return line.split(':', 1)[1].strip()
    except OSError:
        pass
    return 'unknown'


def static_config(args, cfg_name, num_points, frames_per_step, world):
    """The part of `config` that does not depend on the run: identical for the GPU arm and the reference arm."""
    return {'workload': args.workload, 'model': cfg_name, 'frames_per_step_per_gpu': frames_per_step,
            'points_per_frame': num_points, 'weights': 'reference checkpoint ' + cfg_name,
            'frames': 'oracle/synth.py lidar_frame(seed = utils.sharding.frame_seed(step, frame, rank))',
            'l2': 'flushed between timed steps (256 MB write) + distinct frames per step',
            'parallelism': 'dp%d (frames sharded, counters all-gathered)' % world}


def cpu_threads():
    """Threads of the CPU arms: all host cores, capped at 64 (beyond that the gather / segment-max stages of the
    port stop scaling and oversubscription made round 1's numbers vary 4.5x between boxes)."""
    return max(1, min(os.cpu_count() or 1, 64))


def run_reference(args, rank):
    """The reference's own CPU path (oracle port of TF-1.15 graph mode + the reference's scikit-learn graph
    builder) on the SAME frames as the GPU arm: step s times frame 0 of the GPU arm's step s on rank 0 (a bounded
    sample of the step's 8 frames: the unit, frames/s, is per frame)."""
    if rank != 0:
        return
    import torch
    from pointgnn_b200.utils import sharding
    cfg_name, num_points, full_360, frames_per_step = WORKLOADS[args.workload]
    if args.frames_per_step:
        frames_per_step = args.frames_per_step
    config, weights = load_config(cfg_name)
    cores = cpu_threads()
    torch.set_num_threads(cores)
    warm = max(args.warmup, 3)                       # the GPU arm's minimum warm-up: keeps the step -> frame map equal
    pool = min(warm + args.steps, FRAME_POOL)        # the GPU arm cycles through this many distinct step inputs
    for i in range(args.warmup):
        cpu_frame_seconds(config, weights, sharding.frame_seed(i % pool, 0, 0, frames_per_step), num_points, full_360)
    t_graph = t_gnn = 0.0
    for i in range(args.steps):
        a, b = cpu_frame_seconds(config, weights, sharding.frame_seed((warm + i) % pool, 0, 0, frames_per_step),
                                 num_points, full_360)
        t_graph += a
        t_gnn += b
    total = t_graph + t_gnn
    value = args.steps / total
    line = {
        'impl': 'reference', 'metric': METRIC, 'value': value, 'unit': UNIT, 'n_gpus': args.gpus,
        'steps': args.steps, 'warmup': args.warmup, 'ms_per_step': 1e3 * total / args.steps,
        'higher_is_better': True, 'scaling': 'weak', 'vs_baseline': None, 'dtype': 'f32', 'data': 'synthetic',
        'config': static_config(args, cfg_name, num_points, frames_per_step, max(args.gpus, 1)),
        'cpu_baseline': {'value': value, 'unit': UNIT, 'cores': cores, 'kind': 'port',
                         'sample': 'each step = frame 0 of the GPU arm\'s step (1 of %d frames) of %s; gen graph %.3f s + '
                                   'gnn inference %.3f s per frame; sklearn graph (n_jobs=1 as the reference pins) + '
                                   'torch-CPU fp32 GNN on %d threads; %s' % (
                                       frames_per_step, args.workload, t_graph / args.steps, t_gnn / args.steps, cores,
                                       cpu_model_name())},
        'e2e': {'value': value, 'unit': UNIT, 'h2d_bytes_per_step': 0, 'd2h_bytes_per_step': 0},
        'gpu_launches': 0,
    }
    print(json.dumps(line), flush=True)


# ---------------------------------------------------------------------------------------------
# GPU arm
# ---------------------------------------------------------------------------------------------
class ClockSampler(object):
    QUERY = ('index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,'
             'clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,'
             'clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap')

    def __init__(self, gpu_index):
        self.gpu = gpu_index
        self.rows = []
        self.proc = None
        self.thread = None

    def start(self):
        try:
            self.proc = subprocess.Popen(
                ['nvidia-smi', '--query-gpu=' + self.QUERY, '--format=csv,noheader,nounits', '-lms', '20',
                 '-i', str(self.gpu)], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
        except OSError:
            self.proc = None
            return
        self.thread = threading.Thread(target=self._read, daemon=True)
        self.thread.start()

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append((time.perf_counter(), [c.strip() for c in line.split(',')]))

    def stop(self, t0, t1):
        if self.proc is None:
            return {'sm_mhz': None, 'sm_max_mhz': None, 'reasons': ['nvidia-smi unavailable']}
        self.proc.terminate()
        try:
            self.proc.wait(timeout=5)
        except subprocess.TimeoutExpired:
            self.proc.kill()
        rows = [r for t, r in self.rows if t0 <= t <= t1 and len(r) >= 9] or [r for _, r in self.rows if len(r) >= 9]
        if not rows:
            return {'sm_mhz': None, 'sm_max_mhz': None, 'reasons': ['no samples']}
        sm = sorted(float(r[1]) for r in rows)
        reasons = set()
        for r in rows:
            for name, col in (('hw_slowdown', 5), ('hw_thermal_slowdown', 6), ('sw_thermal_slowdown', 7),
                              ('sw_power_cap', 8)):
                if r[col].lower().startswith('active'):
                    reasons.add(name)
        return {'sm_mhz': sm[len(sm) // 2], 'sm_max_mhz': float(rows[0][2]), 'reasons': sorted(reasons),
                'samples': len(rows), 'power_w_max': max(float(r[3]) for r in rows)}


def run_gpu(args, rank, world):
    import torch
    import torch.distributed as dist
    import pointgnn_b200
    from oracle import synth                      # synthetic input generator only
    from pointgnn_b200 import _lib
    from pointgnn_b200.models import graph_gen, models
    from pointgnn_b200.utils import sharding

    local_rank = int(os.environ.get('LOCAL_RANK', 0))
    torch.cuda.set_device(local_rank)
    dev = torch.device('cuda', local_rank)
    if world > 1:
        dist.init_process_group('nccl', device_id=dev)
    cfg_name, num_points, full_360, frames_per_step = WORKLOADS[args.workload]
    if args.frames_per_step:
        frames_per_step = args.frames_per_step
    config, weights = load_config(cfg_name)
    precision = args.precision or ('bf16x3' if _lib.tc_available() else 'fp32')
    pointgnn_b200.set_precision(precision)
    model = models.get_model(config['model_name'])(num_classes=config['num_classes'], box_encoding_len=7,
                                                   mode='test', **config['model_kwargs'])
    model.load_weights(weights)
    graph_fn = graph_gen.get_graph_generate_fn(config['graph_gen_method'])
    gkw = config['runtime_graph_gen_kwargs']

    # a pool of distinct frames; every step sees different frames (rank-disjoint), inputs pinned on the host
    total_steps = args.warmup + args.steps
    pool = min(total_steps, FRAME_POOL)
    host_steps = []
    for s in range(pool):
        pts, inten = [], []
        for f in range(frames_per_step):
            x, it = synth.lidar_frame(sharding.frame_seed(s, f, rank, frames_per_step), num_points, full_360)
            pts.append(x)
            inten.append(it)
        fp = np.arange(frames_per_step + 1, dtype=np.int32) * num_points
        host_steps.append((torch.from_numpy(np.vstack(pts)).pin_memory(), torch.from_numpy(np.vstack(inten)).pin_memory(),
                           torch.from_numpy(fp).pin_memory()))
    dev_steps = [(a.to(dev), b.to(dev), c.to(dev)) for a, b, c in host_steps]
    flush = torch.empty(256 << 20, dtype=torch.uint8, device=dev)      # > 126 MB L2

    stage_ms = {'gen graph': 0.0, 'gnn inference': 0.0, 'edge kernel': 0.0}
    counters = {'edges1': 0, 'edges0': 0, 'keypoints': 0, 'edge_launches': 0}

    def step_device(xyz, inten, fp, instrument=False):
        if instrument:
            ev = [torch.cuda.Event(enable_timing=True) for _ in range(3)]
            ev[0].record()
        coords, kp, edges = graph_fn(xyz, frame_ptr=fp, **gkw)
        if instrument:
            ev[1].record()
        logits, boxes = model.predict(inten, coords, kp, edges, is_training=True)
        probs = model.postprocess(logits)
        if instrument:
            ev[2].record()
            torch.cuda.synchronize()
            stage_ms['gen graph'] += ev[0].elapsed_time(ev[1])
            stage_ms['gnn inference'] += ev[1].elapsed_time(ev[2])
        outputs = {'probs': probs, 'boxes': boxes, 'keypoint_indices': kp[0], 'keypoint_xyz': coords[1],
                   'edges0': edges[0], 'edges1': edges[1]}
        return probs, boxes, kp[0].shape[0], edges[0].shape[0], edges[1].shape[0], outputs

    # end-to-end arm: pinned host buffers on both sides (inputs above; outputs here, sized for the worst case of
    # one keypoint per point), asynchronous copies on the compute stream, ONE synchronisation per step
    n_cls = config['num_classes']
    out_probs = torch.empty((frames_per_step * num_points, n_cls), dtype=torch.float32).pin_memory()
    out_boxes = torch.empty((frames_per_step * num_points, n_cls, 7), dtype=torch.float32).pin_memory()

    def step_e2e(hx, hi, hfp):
        xyz = hx.to(dev, non_blocking=True)
        inten = hi.to(dev, non_blocking=True)
        fp = hfp.to(dev, non_blocking=True)
        probs, boxes, k, e0, e1, _ = step_device(xyz, inten, fp)
        hp, hb = out_probs[:k], out_boxes[:k]
        hp.copy_(probs, non_blocking=True)
        hb.copy_(boxes, non_blocking=True)
        torch.cuda.current_stream().synchronize()
        return hp, hb

    # the same end-to-end work with the NEXT batch's copy + graph build on a side stream while the model runs
    # the current batch (utils/prefetch.py = the role of the reference's DataProvider worker pool, train.py:419-483)
    from pointgnn_b200.utils.prefetch import GraphPrefetcher
    prefetcher = GraphPrefetcher(graph_fn, gkw, dev)

    def loop_e2e_pipelined(batches):
        last = None
        ticket = prefetcher.submit(*batches[0])
        for i in range(len(batches)):
            inten, coords, kp, edges = prefetcher.collect(ticket)
            logits, boxes = model.predict(inten, coords, kp, edges, is_training=True)
            probs = model.postprocess(logits)
            k = kp[0].shape[0]
            hp, hb = out_probs[:k], out_boxes[:k]
            hp.copy_(probs, non_blocking=True)
            hb.copy_(boxes, non_blocking=True)
            done = torch.cuda.Event()
            done.record()
            if i + 1 < len(batches):
                ticket = prefetcher.submit(*batches[i + 1])      # overlaps with the predict + copies queued above
            done.synchronize()                                   # results of batch i are on the host
            last = (hp, hb)
        return last

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    # ---- warm-up ---------------------------------------------------------------------------
    for s in range(args.warmup):
        step_device(*dev_steps[s % pool])
        step_e2e(*host_steps[s % pool])
    loop_e2e_pipelined([host_steps[s % pool] for s in range(args.warmup)])
    barrier()

    # ---- timed: device-resident inputs -------------------------------------------------------
    sampler = ClockSampler(local_rank)
    if rank == 0:
        sampler.start()
        time.sleep(0.25)
    launches0 = _lib.launch_count()
    barrier()
    t_wall0 = time.perf_counter()
    elapsed_ms = 0.0
    frames = 0
    for s in range(args.steps):
        flush.zero_()                                   # L2 flush between timed iterations (untimed)
        torch.cuda.synchronize()
        a = torch.cuda.Event(enable_timing=True)
        b = torch.cuda.Event(enable_timing=True)
        a.record()
        probs, boxes, k, e0, e1, outputs = step_device(*dev_steps[(args.warmup + s) % pool])
        b.record()
        b.synchronize()
        elapsed_ms += a.elapsed_time(b)
        frames += frames_per_step
        counters['keypoints'] += k
        counters['edges0'] += e0
        counters['edges1'] += e1
        if s + 1 < args.steps:
            outputs = None          # the graph of step s is not kept alive while step s + 1 allocates its own
    barrier()
    t_wall1 = time.perf_counter()
    launches = _lib.launch_count() - launches0
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, outputs)
    del outputs

    # ---- timed: end to end through the public API with host buffers ---------------------------
    barrier()
    e2e_t0 = time.perf_counter()
    d2h = 0
    for s in range(args.steps):
        p, bx = step_e2e(*host_steps[(args.warmup + s) % pool])
        d2h = p.numel() * 4 + bx.numel() * 4
    torch.cuda.synchronize()
    e2e_serial_s = time.perf_counter() - e2e_t0
    barrier()
    e2e_t0 = time.perf_counter()
    loop_e2e_pipelined([host_steps[(args.warmup + s) % pool] for s in range(args.steps)])
    torch.cuda.synchronize()
    e2e_pipelined_s = time.perf_counter() - e2e_t0
    barrier()
    # the two modes do the same work through the same public calls; which one is faster depends on the host (the
    # prefetcher hides launch latency and the size round trip, but its side-stream kernels also interleave with the
    # forward pass): report both, headline = the faster one
    e2e_s = min(e2e_serial_s, e2e_pipelined_s)
    clocks = sampler.stop(t_wall0, time.perf_counter()) if rank == 0 else None
    h2d = sum(t.numel() * t.element_size() for t in host_steps[0])

    # ---- instrumented pass: stage split + the dominant kernel under CUDA events ---------------
    n_instr = min(args.steps, 3)
    for s in range(n_instr):
        step_device(*dev_steps[(args.warmup + s) % pool], instrument=True)
    edge_ms, edge_flops, edge_launches = time_edge_kernel(model, graph_fn, gkw, dev_steps[args.warmup % pool], config)
    sm_ms, sm_bytes = (0.0, 0.0)
    if rank == 0:
        d_model = [l for l in config['model_kwargs']['layer_configs'] if 'edge_MLP_depth_list' in l['kwargs']]
        if d_model:
            sm_ms, sm_bytes = time_scatter_max(graph_fn, gkw, dev_steps[args.warmup % pool],
                                               d_model[0]['kwargs']['edge_MLP_depth_list'][-1])

    # ---- reduce over ranks: the only collective of the job is this all-gather of counters --------
    _, summary = sharding.gather_counters(
        {'frames': frames, 'device_ms': elapsed_ms, 'e2e_ms': e2e_s * 1e3, 'edges0': counters['edges0'],
         'edges1': counters['edges1'], 'keypoints': counters['keypoints']}, device=dev)
    max_ms, max_e2e_ms = summary['device_ms'], summary['e2e_ms']
    total_frames = summary['frames']

    if rank == 0:
        peaks = {}
        try:
            with open(os.path.join(ROOT, 'MEASURED_PEAKS.json')) as f:
                peaks = json.load(f)
        except OSError:
            pass
        # the kernel is timed in isolation (a handful of back-to-back launches): the BURST peak is the denominator
        peak_tf = peaks.get('bf16_tflops', 1590.0)
        peak_src = 'measured (MEASURED_PEAKS.json bf16_tflops, burst)' if peaks else 'fallback 1.59 PFLOP/s burst'
        traffic, traffic_src = edge_kernel_dram_traffic()
        hbm = peaks.get('hbm_gbs', 6650.0)
        hbm_src = 'measured (MEASURED_PEAKS.json hbm_gbs)' if peaks else 'fallback 6.65 TB/s'
        achieved = edge_flops / (edge_ms * 1e-3) / 1e12 if edge_ms > 0 else 0.0
        k_avg = counters['keypoints'] / args.steps / frames_per_step
        e0_avg = counters['edges0'] / args.steps / frames_per_step
        e1_avg = counters['edges1'] / args.steps / frames_per_step
        flops_frame, _ = algorithmic_flops(config, k_avg, e0_avg, e1_avg)
        cpu = None
        if not args.no_cpu_baseline:
            seeds = [sharding.frame_seed((args.warmup + i) % pool, 0, 0, frames_per_step) for i in range(4)]
            cpu_frame_seconds(config, weights, seeds[0], num_points, full_360)          # warm-up frame
            reps = [cpu_frame_seconds(config, weights, sd, num_points, full_360) for sd in seeds[1:]]
            g, n = min(reps, key=lambda r: r[0] + r[1])
            cpu = {'value': 1.0 / (g + n), 'unit': UNIT, 'cores': cpu_threads(), 'kind': 'port',
                   'sample': 'fastest of 3 frames (frame 0 of timed steps 1-3) of %s after 1 warm-up (gen graph %.3f s + '
                             'gnn inference %.3f s); sklearn graph n_jobs=1 + torch-CPU fp32 GNN on %d threads; %s' % (
                                 args.workload, g, n, cpu_threads(), cpu_model_name())}
        line = {
            'metric': METRIC, 'value': total_frames / (max_ms * 1e-3), 'unit': UNIT, 'n_gpus': world,
            'steps': args.steps, 'warmup': args.warmup, 'ms_per_step': max_ms / args.steps,
            'higher_is_better': True, 'scaling': 'weak', 'vs_baseline': None,
            'dtype': 'bf16x3(f32-class)' if precision == 'bf16x3' else 'f32', 'data': 'synthetic',
            'config': static_config(args, cfg_name, num_points, frames_per_step, world),
            'workload_stats': {'keypoints_per_frame': k_avg, 'edges0_per_frame': e0_avg, 'edges1_per_frame': e1_avg,
                               'algorithmic_gflop_per_frame': flops_frame / 1e9, 'precision': precision},
            # through the public API with host buffers, two modes: `serial_value` one batch at a time, `prefetch_value`
            # the next batch's copy + graph build on a side stream (utils.prefetch.GraphPrefetcher); `value` = the faster
            # (per-rank values; the headline is all ranks' frames / the slowest rank's time)
            'e2e': {'value': total_frames / (max_e2e_ms * 1e-3), 'unit': UNIT, 'h2d_bytes_per_step': h2d,
                    'd2h_bytes_per_step': d2h,
                    'mode': ('prefetch: graph build of batch i+1 on a side stream during the forward pass of batch i'
                             if e2e_pipelined_s < e2e_serial_s else 'serial: one batch at a time') +
                            ' (rank 0; one host synchronisation per batch; value = the faster of the two modes)',
                    'serial_value': frames / e2e_serial_s, 'prefetch_value': frames / e2e_pipelined_s},
            'gpu_launches': launches,
            'clocks': clocks,
            'stages_ms_per_step': {k: v / n_instr for k, v in stage_ms.items() if k != 'edge kernel'},
            'roofline': {'bound': 'tensor', 'kernel': 'seg_gemm_tc_kernel (fused GNN edge layer: gather + edge MLP + '
                                                      'segment max; timed as the prepared pg_layer_edge_mlp_max call = '
                                                      'hoisted per-vertex GEMM + output fill + the fused kernel)',
                         'achieved': achieved, 'peak': peak_tf, 'unit': 'TFLOP/s', 'frac': achieved / peak_tf,
                         'traffic': traffic, 'traffic_source': traffic_src, 'peak_source': peak_src,
                         'launch_ms': edge_ms / max(edge_launches, 1),
                         'algorithmic_flops_per_launch': edge_flops / max(edge_launches, 1),
                         # the kernel executes 3 BF16 MMAs per product (BF16x3 split) on the padded 304x304 second
                         # layer only (the first layer is hoisted to a per-vertex GEMM): executed tensor FLOP/s
                         'executed_tensor_tflops': achieved * (2 * 3 * 304 * 304) / 361800.0
                         if cfg_name.startswith('car') else None},
            # BASELINE.json's "scatter-max GB/s vs roofline": the stand-alone segment-max op (the fused path above
            # never materialises its [E, D] input; this is the op as the reference calls it)
            'roofline_scatter_max': {
                'bound': 'hbm', 'kernel': 'scatter_max_kernel (pg_scatter_max = graph_scatter_max_fn, stand-alone)',
                'achieved': (sm_bytes / (sm_ms * 1e-3) / 1e9) if sm_ms > 0 else None,
                'peak': hbm, 'unit': 'GB/s',
                'frac': (sm_bytes / (sm_ms * 1e-3) / 1e9 / hbm) if sm_ms > 0 else None,
                'peak_source': hbm_src,
                'launch_ms': sm_ms, 'algorithmic_bytes_per_launch': sm_bytes, 'traffic': None},
            # the graph build (keypoints + both radius graphs, pg_multi_level_graph): HBM / L2-latency bound integer
            # and fp64-predicate work.  Algorithmic bytes per step (SURVEY 8d, minimum traffic): keypoints N*12 + K*4;
            # level 0: N*12 + K*12 + 4(K+1) + 8*E0; level 1: K*12 + K*12 + 4(K+1) + 8*E1 (src and dst columns, 4 B each)
            'roofline_graph': graph_roofline(stage_ms['gen graph'] / n_instr, frames_per_step * num_points,
                                             k_avg * frames_per_step, e0_avg * frames_per_step,
                                             e1_avg * frames_per_step, hbm, hbm_src),
            'cpu_baseline': cpu,
        }
        print(json.dumps(line), flush=True)
    if world > 1:
        dist.destroy_process_group()


DUMP_MAX_ARRAY_BYTES = 8 << 20     # 6 arrays: at most 48 MB written


def dump_outputs(out_dir, outputs):
    """Write what one timed step returned as <out_dir>/<name>.npy: floating point as float32 / float64, integer
    indices as float64 (exact).  An array larger than DUMP_MAX_ARRAY_BYTES is replaced by a fixed sample of its rows
    (seed 0, ascending row order; the edge lists at the default workload); <name>_rows.npy then holds the sampled row
    numbers, so two builds that return the same number of rows are compared on the same rows."""
    os.makedirs(out_dir, exist_ok=True)
    for name, t in outputs.items():
        a = np.ascontiguousarray(t.detach().cpu().numpy())
        a = a.astype(np.float64 if a.dtype.kind in 'iu' or a.dtype == np.float64 else np.float32)
        row_bytes = a[:1].nbytes or 1
        if a.nbytes > DUMP_MAX_ARRAY_BYTES:
            m = DUMP_MAX_ARRAY_BYTES // (row_bytes + 8)
            rows = np.sort(np.random.default_rng(0).choice(a.shape[0], m, replace=False))
            a = a[rows]
            np.save(os.path.join(out_dir, name + '_rows.npy'), rows.astype(np.float64))
        np.save(os.path.join(out_dir, name + '.npy'), a)


def graph_roofline(ms, n, k, e0, e1, hbm, hbm_src):
    b = (n * 12 + k * 4) + (n * 12 + k * 12 + 4 * (k + 1) + 8 * e0) + (k * 12 + k * 12 + 4 * (k + 1) + 8 * e1)
    achieved = b / (ms * 1e-3) / 1e9 if ms > 0 else None
    return {'bound': 'hbm', 'kernel': 'pg_multi_level_graph (grid build, voxel keypoints, radius count / fill, CSR row sort)',
            'achieved': achieved, 'peak': hbm, 'unit': 'GB/s', 'frac': achieved / hbm if achieved else None,
            'peak_source': hbm_src, 'step_ms': ms, 'algorithmic_bytes_per_step': b, 'traffic': None}


def time_edge_kernel(model, graph_fn, gkw, dev_step, config):
    """CUDA-event time of the dominant kernel (fused edge MLP + segment max of one GNN iteration)."""
    import torch
    import pointgnn_b200
    from pointgnn_b200 import _lib
    from pointgnn_b200.models import gnn
    xyz, inten, fp = dev_step
    coords, kp, edges = graph_fn(xyz, frame_ptr=fp, **gkw)
    lc = [l for l in config['model_kwargs']['layer_configs'] if l['type'] == 'scatter_max_graph_auto_center_net']
    if not lc:
        return 0.0, 0.0, 0
    lc = lc[0]
    d = lc['kwargs']['edge_MLP_depth_list']
    k = coords[1].shape[0]
    feats = torch.rand((k, d[-1]), device=xyz.device) * 0.5
    store = model._store
    with gnn.variable_session(store), gnn.variable_scope(lc['scope']), gnn.variable_scope('extract_vertex_features'):
        ws, bs = gnn._take_mlp_weights(len(d))
    src, dst = edges[1][:, 0].contiguous(), edges[1][:, 1].contiguous()
    reps = 5
    prec = pointgnn_b200.get_precision()
    layer = _lib.PreparedLayer(_lib.PG_LAYER_EDGE_GNN, ws, bs, [d[0] + 3] + list(d), prec)
    for _ in range(2):
        layer.edge_mlp_max(feats, coords[1], coords[1], None, src, dst, k, trusted=True)
    torch.cuda.synchronize()
    a = torch.cuda.Event(enable_timing=True)
    b = torch.cuda.Event(enable_timing=True)
    a.record()
    for _ in range(reps):
        layer.edge_mlp_max(feats, coords[1], coords[1], None, src, dst, k, trusted=True)
    b.record()
    b.synchronize()
    dims = [d[0] + 3] + d
    per_edge = sum(2 * x * y for x, y in zip(dims[:-1], dims[1:]))
    return a.elapsed_time(b), float(src.numel()) * per_edge * reps, reps


def time_scatter_max(graph_fn, gkw, dev_step, channels):
    """BASELINE.json's second roofline: the stand-alone graph_scatter_max_fn op (gnn.py:106-109) on the [E1, D]
    edge-feature tensor the reference materialises, against the measured HBM copy bandwidth.  Algorithmic bytes
    (SURVEY 8d) = E*C*4 (features) + E*4 (ids) + K*C*4 (output).  Returns (ms per call, bytes per call)."""
    import torch
    from pointgnn_b200 import _lib
    xyz, inten, fp = dev_step
    coords, kp, edges = graph_fn(xyz, frame_ptr=fp, **gkw)
    dst = edges[1][:, 1].contiguous()
    e, k = int(dst.numel()), int(coords[1].shape[0])
    feats = torch.rand((e, channels), device=xyz.device)          # 4.7 GB at the default workload: >> L2
    for _ in range(2):
        _lib.scatter_max(feats, dst, k)
    torch.cuda.synchronize()
    reps = 5
    a = torch.cuda.Event(enable_timing=True)
    b = torch.cuda.Event(enable_timing=True)
    a.record()
    for _ in range(reps):
        _lib.scatter_max(feats, dst, k)
    b.record()
    b.synchronize()
    del feats
    return a.elapsed_time(b) / reps, float(e) * channels * 4 + float(e) * 4 + float(k) * channels * 4


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument('--gpus', type=int, default=1)
    ap.add_argument('--steps', type=int, default=100)
    ap.add_argument('--warmup', type=int, default=3)
    ap.add_argument('--impl', default='ours', choices=['ours', 'reference'])
    ap.add_argument('--workload', default='car_auto_T3_20k', choices=sorted(WORKLOADS))
    ap.add_argument('--precision', default=None, choices=['fp32', 'bf16x3'])
    ap.add_argument('--frames-per-step', type=int, default=0)
    ap.add_argument('--no-cpu-baseline', action='store_true')
    ap.add_argument('--dump-outputs', metavar='DIR', default=None,
                    help='after the timed steps, write the outputs of the last one as DIR/<name>.npy')
    args = ap.parse_args()
    if args.steps < 1:
        ap.error('--steps must be at least 1')
    if args.dump_outputs and args.impl != 'ours':
        ap.error('--dump-outputs writes the outputs of the GPU path (--impl ours)')
    args.warmup = max(args.warmup, 3) if args.impl == 'ours' else args.warmup
    rank = int(os.environ.get('RANK', 0))
    world = int(os.environ.get('WORLD_SIZE', 1))
    if args.impl == 'reference':
        run_reference(args, rank)
        return
    run_gpu(args, rank, world)


if __name__ == '__main__':
    main()
