"""CPU checks of bench.py's metric definitions (no GPU, no library calls)."""
import importlib.util
import json
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _bench():
    spec = importlib.util.spec_from_file_location('bench_module', os.path.join(ROOT, 'bench.py'))
    mod = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(mod)
    return mod


def test_algorithmic_flops_match_survey_formulas(car, ped):
    """SURVEY.md 8d: 2*M*K*N per fully-connected layer, bias / ReLU / max not counted."""
    bench = _bench()
    k, e0, e1 = 4051, 848749, 940343
    total, per_edge = bench.algorithmic_flops(car.config, k, e0, e1)
    assert per_edge == 361800                              # 2*303*300 + 2*300*300
    want = e0 * 97536 + k * 360000 + 3 * (e1 * 361800 + k * (360000 + 38784)) + k * 228864
    assert total == want
    total_p, per_edge_p = bench.algorithmic_flops(ped.config, k, e0, e1)
    assert per_edge_p == 263680                            # 2*259*256 + 2*256*256
    want_p = e0 * 348416 + k * 393216 + 3 * (e1 * 263680 + k * (262144 + 33152)) + k * 284672
    assert total_p == want_p


def test_workloads_name_baseline_configs():
    bench = _bench()
    assert bench.WORKLOADS['car_auto_T3_20k'][:3] == ('car_auto_T3_train', 20000, False)
    assert bench.WORKLOADS['car_auto_T3_120k'][:3] == ('car_auto_T3_train', 120000, True)
    assert bench.WORKLOADS['ped_cyl_auto_T3_20k_b8'][3] == 8
    assert bench.UNIT == 'frames/s'


def test_reference_arm_rank_nonzero_is_silent():
    """Under torchrun only rank 0 runs the CPU reference arm; the other ranks exit 0 without output."""
    env = dict(os.environ, RANK='1', WORLD_SIZE='2')
    out = subprocess.run([sys.executable, os.path.join(ROOT, 'bench.py'), '--impl', 'reference', '--gpus', '2',
                          '--steps', '1', '--warmup', '0'], env=env, capture_output=True, text=True, timeout=120)
    assert out.returncode == 0 and out.stdout.strip() == ''


def test_committed_bench_line_has_the_contract_keys():
    path = os.path.join(ROOT, 'profiles', 'r1_bench_line.json')
    line = [l for l in open(path).read().splitlines() if l.startswith('{')][-1]
    d = json.loads(line)
    for key in ('metric', 'value', 'unit', 'n_gpus', 'steps', 'warmup', 'ms_per_step', 'higher_is_better', 'scaling',
                'vs_baseline', 'dtype', 'data', 'config', 'e2e', 'gpu_launches', 'clocks', 'roofline', 'cpu_baseline'):
        assert key in d, key
    assert d['config']['workload'] == 'car_auto_T3_20k'
    for key in ('bound', 'achieved', 'peak', 'unit', 'frac', 'traffic'):
        assert key in d['roofline'], key
    assert d['e2e']['h2d_bytes_per_step'] > 0 and d['e2e']['d2h_bytes_per_step'] > 0
    assert d['gpu_launches'] > 0 and d['warmup'] >= 3


def test_dump_outputs_float_arrays_fixed_sample(tmp_path):
    """--dump-outputs: float32 / float64 .npy files, integer indices exact, a large array replaced by the same seeded
    sample of rows on every run, within the 64 MB budget."""
    import numpy as np
    import torch
    bench = _bench()
    edges = torch.arange(2 * 3000000, dtype=torch.int32).reshape(3000000, 2)
    probs = torch.rand(1000, 4)
    for run in ('a', 'b'):
        bench.dump_outputs(str(tmp_path / run), {'probs': probs, 'edges1': edges})
    files = sorted(os.listdir(tmp_path / 'a'))
    assert files == ['edges1.npy', 'edges1_rows.npy', 'probs.npy']
    assert sum(os.path.getsize(tmp_path / 'a' / f) for f in files) <= 64 << 20
    for f in files:
        a, b = np.load(tmp_path / 'a' / f), np.load(tmp_path / 'b' / f)
        assert a.dtype in (np.float32, np.float64) and np.array_equal(a, b)
    assert np.array_equal(np.load(tmp_path / 'a' / 'probs.npy'), probs.numpy())
    rows = np.load(tmp_path / 'a' / 'edges1_rows.npy').astype(np.int64)
    assert 0 < len(rows) < 3000000 and np.all(np.diff(rows) > 0)
    assert np.array_equal(np.load(tmp_path / 'a' / 'edges1.npy'), edges.numpy()[rows].astype(np.float64))
