"""GPU tests of the graph build's row sort and cell keys, bit-exact against the CPU oracle.

- Row-length boundaries: one warp sorts a row of up to 1 024 entries in registers, padded to a power of two; longer
  rows go to a block pass that merges 1 024-entry chunks, in shared memory up to 8 192 entries.  Every size class
  edge is hit, through the one-call multi-level graph and through the stand-alone radius graph.
- Key width: cell keys are 32 bits when the cell indices fit (frame bits first, the rest split across the axes) and
  the call is redone with 64-bit keys when one does not.
"""
import numpy as np
import pytest
import torch

from oracle import graph, synth

pytestmark = pytest.mark.gpu

ROW_LENGTHS = [0, 1, 31, 32, 33, 63, 64, 1023, 1024, 1025, 2047, 2048, 2049, 8192, 8193]
CFG = [dict(graph_level=0, graph_scale=1.0, graph_gen_method='disjointed_rnn_local_graph_v3',
            graph_gen_kwargs=dict(radius=1.0, num_neighbors=-1)),
       dict(graph_level=1, graph_scale=1.0, graph_gen_method='disjointed_rnn_local_graph_v3',
            graph_gen_kwargs=dict(radius=4.0, num_neighbors=-1))]


def _blobs(lengths, seed):
    """Tight blobs (radius 0.1) of the given sizes 10 m apart, points shuffled so that no row arrives sorted, and
    one centre per blob (a size-0 blob is a centre with no point near it)."""
    rng = np.random.default_rng(seed)
    pts, ctr = [], []
    for i, n in enumerate(lengths):
        c = np.array([10.0 * i, 0.5 * (i % 3), 3.0 + 0.25 * (i % 2)])
        d = rng.normal(size=(n, 3))
        d *= (0.1 * rng.random((n, 1)) ** (1 / 3)) / np.maximum(np.linalg.norm(d, axis=1, keepdims=True), 1e-9)
        pts.append(c + d)
        ctr.append(c)
    pts = np.vstack(pts).astype(np.float32)
    return pts[rng.permutation(pts.shape[0])], np.array(ctr, np.float32)


def _frames(lengths, num_frames, seed):
    return [_blobs(lengths[f::num_frames], seed + f) for f in range(num_frames)]


def _row_lengths(edges, num_rows):
    return np.bincount(np.asarray(edges)[:, 1], minlength=num_rows)


def _assert_multi_level(clouds, kwargs):
    from pointgnn_b200.models import graph_gen
    frames = []
    for c in clouds:
        co, kp, ed = graph.gen_multi_level_local_graph_v3(c, **kwargs)
        frames.append((np.zeros((c.shape[0], 1), np.float32), co, kp, ed))
    _, bc, bk, be = graph.batch_graphs(frames)
    fp = np.cumsum([0] + [c.shape[0] for c in clouds]).astype(np.int32)
    coords, kp, edges = graph_gen.gen_multi_level_local_graph_v3(np.vstack(clouds), frame_ptr=fp, **kwargs)
    for a, b in zip(kp, bk):
        assert a.shape == b.shape and np.array_equal(a, b)
    for a, b in zip(edges, be):
        assert a.shape == b.shape and np.array_equal(a, b)
    return coords, kp, edges


@pytest.mark.parametrize('num_frames', [1, 3])
def test_row_length_boundaries_multi_level(num_frames):
    clouds = [p for p, _ in _frames([n for n in ROW_LENGTHS if n > 0], num_frames, 7)]
    _, kp, edges = _assert_multi_level(clouds, dict(base_voxel_size=1.0, level_configs=CFG))
    lengths = set(_row_lengths(edges[0], kp[1].shape[0]).tolist())
    assert {n for n in ROW_LENGTHS if n > 0} <= lengths


@pytest.mark.parametrize('num_frames', [1, 3])
def test_row_length_boundaries_radius_graph(num_frames):
    from pointgnn_b200 import _lib
    from pointgnn_b200.models import graph_gen
    parts = _frames(ROW_LENGTHS, num_frames, 11)
    if num_frames == 1:
        pts, ctr = parts[0]
        e = graph_gen.gen_disjointed_rnn_local_graph_v3(pts, ctr, 1.0, -1)
        assert np.array_equal(e, graph.radius_graph(pts, ctr, 1.0))
        assert sorted(_row_lengths(e, ctr.shape[0]).tolist()) == sorted(ROW_LENGTHS)
    want, p_off, c_off = [], 0, 0
    for pts, ctr in parts:
        w = graph.radius_graph(pts, ctr, 1.0)
        want.append(w + [p_off, c_off])
        p_off, c_off = p_off + pts.shape[0], c_off + ctr.shape[0]
    want = np.vstack(want)
    t = lambda a: torch.from_numpy(np.ascontiguousarray(a)).cuda()
    pfp = t(np.cumsum([0] + [p.shape[0] for p, _ in parts]).astype(np.int32))
    cfp = t(np.cumsum([0] + [c.shape[0] for _, c in parts]).astype(np.int32))
    pts, ctr = t(np.vstack([p for p, _ in parts])), t(np.vstack([c for _, c in parts]))
    _, e1 = _lib.radius_graph(pts, pfp, ctr, cfp, 1.0)
    _, e2 = _lib.radius_graph_two_pass(pts, pfp, ctr, cfp, 1.0)     # the fill half runs on 64-bit keys
    for e in (e1, e2):
        assert np.array_equal(e.t().cpu().numpy().astype(np.int64), want)


def _launches(xyz, fp, voxel, r0, r1):
    """Launches of one pg_multi_level_graph call (the second of two, so that the buffer sizes are settled)."""
    from pointgnn_b200 import _lib
    xyz, fp = torch.from_numpy(xyz).cuda(), torch.from_numpy(fp).cuda()
    _lib.multi_level_graph(xyz, fp, voxel, r0, r1)
    a = _lib.launch_count()
    out = _lib.multi_level_graph(xyz, fp, voxel, r0, r1)
    return out, _lib.launch_count() - a


def _frame_ptr(clouds):
    return np.cumsum([0] + [c.shape[0] for c in clouds]).astype(np.int32)


def test_key_width_fallback():
    """8 frames leave 10 bits (1 024 cells) for x in the compact key: a 2 km cloud at 0.4 m voxels overflows it but
    fits 16 bits per axis, so the call is redone with 64-bit keys."""
    rng = np.random.default_rng(3)
    far = np.vstack([rng.random((800, 3)) * [4.0, 1.0, 4.0],
                     rng.random((800, 3)) * [4.0, 1.0, 4.0] + [1996.0, 0.0, 0.0]]).astype(np.float32)
    near = [synth.lidar_frame(40 + i, 1500)[0] for i in range(7)]
    kwargs = dict(base_voxel_size=0.4, level_configs=CFG)
    _assert_multi_level([far] + near, kwargs)
    _assert_multi_level([near[0]] + near, kwargs)
    _, wide = _launches(np.vstack([far] + near), _frame_ptr([far] + near), (0.4,) * 3, 1.0, 4.0)
    _, compact = _launches(np.vstack([near[0]] + near), _frame_ptr([near[0]] + near), (0.4,) * 3, 1.0, 4.0)
    # the retry repeats the whole call
    assert wide > 1.5 * compact


def test_key_width_boundary():
    """For 8 frames, x cell 1 023 is the last one the compact key holds and 1 024 the first it does not: both clouds
    give the oracle's result, the second through the 64-bit retry."""
    rest = [synth.lidar_frame(60 + i, 1000)[0] for i in range(7)]
    counts = []
    for last_cell in (1023, 1024):
        # voxel 1.0, origin = frame minimum - 0.5: x = last_cell - 0.25 lies in cell last_cell
        line = np.zeros((64, 3), np.float32)
        line[:, 0] = np.linspace(0.0, last_cell - 0.25, 64, dtype=np.float32)
        line[:, 2] = 5.0
        _assert_multi_level([line] + rest, dict(base_voxel_size=1.0, level_configs=CFG))
        _, n = _launches(np.vstack([line] + rest), _frame_ptr([line] + rest), (1.0,) * 3, 1.0, 4.0)
        counts.append(n)
    assert counts[1] > 1.5 * counts[0]


def test_many_frames():
    """64 frames -> 7 frame bits, 9 | 7 | 9 bits for x | y | z."""
    clouds = [synth.lidar_frame(200 + i, 2000)[0] for i in range(64)]
    _assert_multi_level(clouds, dict(base_voxel_size=0.8, level_configs=[
        dict(graph_level=0, graph_scale=0.5, graph_gen_method='disjointed_rnn_local_graph_v3',
             graph_gen_kwargs=dict(radius=1.0, num_neighbors=-1)),
        dict(graph_level=1, graph_scale=0.5, graph_gen_method='disjointed_rnn_local_graph_v3',
             graph_gen_kwargs=dict(radius=4.0, num_neighbors=-1))]))
