"""GPU tests of the training-time graph path (train.py:88-90 with configs/*_train_config: downsample_method='random',
add_rnd3d, num_neighbors 256 on the keypoint graph): pg_random_keypoints and pg_cap_neighbors behind
graph_gen._downsampling_random and graph_gen._radius_edges.

* Keypoints are exact once the random numbers are fixed: fed the numbers recorded in tests/golden/graph_random.npz
  (the reference's own multi_layer_downsampling_random), the kernels return the reference's keypoints; batched frames
  equal the oracle frame by frame.
* The add_rnd3d grid shifts are drawn frame-major, so a batch of F frames equals F one-frame calls.
* The neighbour cap is random by design: it is checked through invariants that do not depend on the draw
  (oracle.graph.check_neighbor_cap against the oracle's radius graph), on hand-built rows that force priority ties,
  and statistically over seeds.
"""
import collections
import json
import os

import numpy as np
import pytest
import torch
from scipy import stats

from oracle import graph, synth

pytestmark = pytest.mark.gpu

GOLDEN = os.path.join(os.path.dirname(__file__), 'golden')


def _level_configs(scales, radii):
    return [{'graph_gen_kwargs': {'num_neighbors': -1, 'radius': r}, 'graph_gen_method': 'disjointed_rnn_local_graph_v3',
             'graph_level': i, 'graph_scale': s} for i, (s, r) in enumerate(zip(scales, radii))]


def _gpu_random(xyz, voxel, levels, add_rnd3d, shifts=None, uniforms=None, frame_ptr=None):
    """graph_gen._downsampling_random with explicit random numbers -> device (coords, keypoint idx, frame_ptr) lists."""
    from pointgnn_b200.models import graph_gen
    cloud = graph_gen._Cloud(xyz, frame_ptr)
    u = None
    if uniforms is not None:
        u = [None if a is None else torch.from_numpy(np.ascontiguousarray(a, dtype=np.float32)).cuda() for a in uniforms]
    return graph_gen._downsampling_random(cloud, voxel, levels, add_rnd3d, uniform=u, shifts=shifts)


def _np(ts):
    return [t.cpu().numpy() for t in ts]


def _frame_ptr(clouds):
    return np.concatenate([[0], np.cumsum([len(c) for c in clouds])]).astype(np.int32)


def _cube(seed, n, side, origin=(0.0, 0.0, 0.0)):
    rng = np.random.default_rng(seed)
    return (rng.random((n, 3)) * side + np.asarray(origin)).astype(np.float32)


# ---------------------------------------------------------------------------------------------------------------------
# keypoints, exact given the random numbers
# ---------------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize('tag', graph.RANDOM_GOLDEN_CASES)
def test_random_keypoints_match_reference_golden(tag):
    """Same keypoint indices in the same order and the same vertices as the reference's own function fed the same
    numbers: a repeated scale (plain, rnd3d), a second distinct scale on the ORIGINAL cloud's grid (ms_*) and an array
    voxel size with points where float32 and float64 floor-division disagree (arr, with its radius graphs)."""
    from pointgnn_b200.models import graph_gen
    c = graph.random_golden_case(np.load(os.path.join(GOLDEN, 'graph_random.npz')), tag)
    vc, kp, fp = _gpu_random(c['xyz'], c['voxel'], c['levels'], c['add_rnd3d'],
                             c['shifts'] if c['add_rnd3d'] else None, c['uniforms'])
    for li in range(len(c['levels'])):
        assert np.array_equal(kp[li][:, 0].cpu().numpy(), c['kp'][li]), li
        assert np.array_equal(vc[li + 1].cpu().numpy(), c['coords'][li]), li
        assert int(fp[li + 1][-1]) == len(c['kp'][li]), li
    if c['edges'] is not None:
        for lvl, r in enumerate(c['radii']):
            e = graph_gen._radius_edges(vc[lvl], fp[lvl], vc[lvl + 1], fp[lvl + 1], r, -1)
            assert np.array_equal(e.cpu().numpy(), c['edges'][lvl]), lvl


def _batch_case(levels, add_rnd3d, seed):
    """Frames of different sizes (one of a single point), per-frame random numbers and the oracle's per-frame result,
    and the same numbers laid out for one batched call: uniforms by global voxel rank, shifts stacked [F,3]."""
    clouds = [synth.lidar_frame(50, 3000)[0], np.array([[2.5, -1.0, 9.0]], np.float32), synth.lidar_frame(51, 1500)[0],
              _cube(52, 2000, 6.0, origin=(-20.0, -3.0, -7.5))]
    rng = np.random.default_rng(seed)
    per_frame = []
    for cl in clouds:
        shifts = [rng.random((1, 3)) for _ in levels]
        uniforms = [rng.random(len(cl)).astype(np.float32) for _ in levels]
        co, ko = graph.multi_layer_downsampling_random(cl, 0.8, levels, add_rnd3d, shifts=shifts, uniforms=uniforms)
        per_frame.append((shifts, uniforms, co, ko))
    b_shifts, b_uniforms = [], []
    for li in range(len(levels)):
        b_shifts.append(np.vstack([f[0][li] for f in per_frame]))
        u = np.concatenate([f[1][li][:len(f[3][li])] for f in per_frame])       # voxel o of frame f -> its own u
        n_base = sum(len(f[2][li]) for f in per_frame)
        b_uniforms.append(np.concatenate([u, rng.random(n_base - len(u)).astype(np.float32)]))
    return clouds, per_frame, b_shifts, b_uniforms


@pytest.mark.parametrize('levels', [[1, 1], [1, 2]])
@pytest.mark.parametrize('add_rnd3d', [False, True])
def test_batched_random_keypoints_equal_oracle_per_frame(levels, add_rnd3d):
    """frame_ptr batching: the batched call equals the oracle frame by frame with the batch_data offsets
    (train.py:135-171), each frame voxelised on its own grid."""
    clouds, per_frame, b_shifts, b_uniforms = _batch_case(levels, add_rnd3d, seed=len(levels) + 10 * add_rnd3d)
    vc, kp, fps = _gpu_random(np.vstack(clouds), 0.8, levels, add_rnd3d, b_shifts if add_rnd3d else None, b_uniforms,
                              frame_ptr=_frame_ptr(clouds))
    vc, kp, fps = _np(vc), [k[:, 0].astype(np.int64) for k in _np(kp)], _np(fps)
    for li in range(len(levels)):
        want_kp, want_co, base_off = [], [], 0
        for shifts, uniforms, co, ko in per_frame:
            want_kp.append(ko[li][:, 0] + base_off)
            want_co.append(co[li + 1])
            base_off += len(co[li])
        assert np.array_equal(kp[li], np.concatenate(want_kp)), li
        assert np.array_equal(vc[li + 1], np.vstack(want_co)), li
        assert np.array_equal(fps[li + 1], _frame_ptr([c for c in want_co])), li
    assert len(per_frame[1][3][0]) == 1                       # the one-point frame keeps its point


@pytest.mark.parametrize('base_voxel_size', [0.8, [0.8, 0.8, 0.8], [0.6, 0.9, 0.7]])
@pytest.mark.parametrize('add_rnd3d', [False, True])
def test_public_random_graph_edges_equal_oracle(base_voxel_size, add_rnd3d):
    """gen_multi_level_local_graph_v3(..., downsample_method='random', num_neighbors=-1) on a batch: every keypoint is a
    point of its frame's previous level, and the edge lists equal the oracle's radius graph on the GPU's own vertices."""
    from pointgnn_b200.models import graph_gen
    clouds = [synth.lidar_frame(60, 4000)[0], _cube(61, 1500, 5.0), np.array([[0.0, 0.0, 30.0]], np.float32)]
    cfg = _level_configs([1, 2, 2], [1.0, 2.0, 4.0])
    np.random.seed(5)
    graph_gen.set_seed(5)
    coords, kp, edges, fps = graph_gen.gen_multi_level_local_graph_v3(
        np.vstack(clouds), base_voxel_size, cfg, add_rnd3d=add_rnd3d, downsample_method='random',
        frame_ptr=_frame_ptr(clouds), return_frame_ptr=True)
    for lvl in range(len(cfg)):
        src, dst = coords[lvl], coords[lvl + 1]
        assert np.array_equal(dst, src[kp[lvl][:, 0]])
        want = []
        for f in range(len(clouds)):
            s0, s1, d0, d1 = fps[lvl][f], fps[lvl][f + 1], fps[lvl + 1][f], fps[lvl + 1][f + 1]
            assert np.all((kp[lvl][d0:d1, 0] >= s0) & (kp[lvl][d0:d1, 0] < s1))        # keypoints stay in the frame
            want.append(graph.radius_graph(src[s0:s1], dst[d0:d1], cfg[lvl]['graph_gen_kwargs']['radius'])
                        + np.array([[s0, d0]]))
        assert np.array_equal(edges[lvl], np.vstack(want)), lvl
    assert len(kp[1]) < len(kp[0])                                         # the second scale did pool


# ---------------------------------------------------------------------------------------------------------------------
# draw order of the add_rnd3d shifts
# ---------------------------------------------------------------------------------------------------------------------
DRAW_ORDER_CLOUDS = ((70, 2500), (71, 1800), (72, 3100))


@pytest.mark.parametrize('scales', [[1, 1], [1, 2, 2]])
def test_rnd3d_draw_order_batch_equals_per_frame_calls(scales):
    """The reference builds one frame per call and each call draws np.random.random((1, 3)) once per new scale.  Seeded
    alike, one batched call and F one-frame calls must partition every frame into the same voxels.  Random method with
    every uniform 0 (the lowest-index point of each voxel: the partition itself), and the centroid method (deterministic
    given the shifts)."""
    from pointgnn_b200.models import graph_gen
    clouds = [synth.lidar_frame(s, n)[0] for s, n in DRAW_ORDER_CLOUDS]
    fp = _frame_ptr(clouds)
    zeros = [np.zeros(fp[-1], np.float32) for _ in scales]
    np.random.seed(11)
    _, b_kp, b_fp = _gpu_random(np.vstack(clouds), 0.8, scales, True, uniforms=zeros, frame_ptr=fp)
    b_kp, b_fp = [k[:, 0] for k in _np(b_kp)], _np(b_fp)
    np.random.seed(11)
    for f, cl in enumerate(clouds):
        _, kp, _ = _gpu_random(cl, 0.8, scales, True, uniforms=zeros)
        for li in range(len(scales)):
            mine = b_kp[li][b_fp[li + 1][f]:b_fp[li + 1][f + 1]] - b_fp[li][f]
            assert np.array_equal(mine, kp[li][:, 0].cpu().numpy()), (f, li)

    cfg = _level_configs(scales, [1.0] + [4.0] * (len(scales) - 1))
    np.random.seed(12)
    co, b_kp, b_e, b_fp = graph_gen.gen_multi_level_local_graph_v3(np.vstack(clouds), 0.8, cfg, add_rnd3d=True,
                                                                   frame_ptr=fp, return_frame_ptr=True)
    np.random.seed(12)
    for f, cl in enumerate(clouds):
        _, kp, e = graph_gen.gen_multi_level_local_graph_v3(cl, 0.8, cfg, add_rnd3d=True)
        for li in range(len(scales)):
            d0, d1, s0 = b_fp[li + 1][f], b_fp[li + 1][f + 1], b_fp[li][f]
            assert np.array_equal(b_kp[li][d0:d1, 0] - s0, kp[li][:, 0]), (f, li)
            rows = (b_e[li][:, 1] >= d0) & (b_e[li][:, 1] < d1)
            assert np.array_equal(b_e[li][rows] - np.array([[s0, d0]]), e[li]), (f, li)

    # the public random method (the per-voxel choice from the CUDA generator): same voxel count per frame at the first
    # scale (a later scale voxelises the first one's random picks, which batching draws differently)
    np.random.seed(13)
    _, b_kp, _, b_fp = graph_gen.gen_multi_level_local_graph_v3(
        np.vstack(clouds), 0.8, cfg, add_rnd3d=True, downsample_method='random', frame_ptr=fp, return_frame_ptr=True)
    np.random.seed(13)
    for f, cl in enumerate(clouds):
        _, kp, _ = graph_gen.gen_multi_level_local_graph_v3(cl, 0.8, cfg, add_rnd3d=True, downsample_method='random')
        assert b_fp[1][f + 1] - b_fp[1][f] == len(kp[0]), f


# ---------------------------------------------------------------------------------------------------------------------
# neighbour cap: invariants that do not depend on the draw
# ---------------------------------------------------------------------------------------------------------------------
def _assert_canonical(edges):
    """Rows grouped by ascending destination, ascending source inside a row (a capped row included)."""
    assert np.all(np.diff(edges[:, 1]) >= 0)
    same = edges[1:, 1] == edges[:-1, 1]
    assert np.all(edges[1:, 0][same] > edges[:-1, 0][same])


def _cluster(rng, center, n, spread=0.3):
    d = rng.normal(size=(n, 3))
    d *= (spread * rng.random((n, 1)) ** (1 / 3)) / np.linalg.norm(d, axis=1, keepdims=True)
    return (np.asarray(center) + d).astype(np.float32)


@pytest.mark.parametrize('cap', [1, 7, 256])
def test_neighbor_cap_rows_of_every_length(cap):
    """Rows that are empty, shorter than the cap, exactly the cap, cap + 1, a few times the cap and far longer than a
    warp's 32 lanes (a 9 000-point blob, also as two identical rows), through the public API."""
    from pointgnn_b200.models import graph_gen
    rng = np.random.default_rng(cap)
    sizes = [max(cap - 1, 0), cap, cap + 1, 3 * cap + 5, 9000]
    pts = np.vstack([_cluster(rng, (10.0 * i, 0.0, 20.0), n) for i, n in enumerate(sizes)])
    centers = np.array([(10.0 * i, 0.0, 20.0) for i in range(len(sizes))] + [(10.0 * 4, 0.0, 20.0), (0.0, 50.0, 20.0)],
                       np.float32)
    full = graph.radius_graph(pts, centers, 1.0)
    assert np.array_equal(np.bincount(full[:, 1], minlength=len(centers)), sizes + [9000, 0])
    graph_gen.set_seed(cap)
    capped = graph_gen.gen_disjointed_rnn_local_graph_v3(pts, centers, 1.0, cap)
    assert capped.dtype == np.int64 and capped.shape[1] == 2
    _assert_canonical(capped)
    n_long = sum(1 for n in sizes + [9000] if n > cap)
    assert graph.check_neighbor_cap(full, capped, cap) == n_long
    blob = capped[capped[:, 1] == 4, 0], capped[capped[:, 1] == 5, 0]
    assert not np.array_equal(*blob)            # identical rows are drawn independently


def test_neighbor_cap_with_scale():
    """num_neighbors > 0 together with the per-axis scale (graph_gen.py:203-214)."""
    from pointgnn_b200.models import graph_gen
    pts = _cube(80, 6000, 6.0)
    centers = pts[::37].copy()
    scale = [1.0, 0.5, 1.3]
    full = graph.gen_disjointed_rnn_local_graph_v3(pts, centers, 0.9, -1, scale=scale)
    graph_gen.set_seed(80)
    capped = graph_gen.gen_disjointed_rnn_local_graph_v3(pts, centers, 0.9, 40, scale=scale)
    _assert_canonical(capped)
    n_capped = graph.check_neighbor_cap(full, capped, 40)
    assert 0 < n_capped < len(centers)


def test_shipped_train_config_on_a_batch():
    """The graph_gen_kwargs of car_auto_T3_train (random keypoints, add_rnd3d, num_neighbors 256 at radius 4 m) on a
    batch of a dense volumetric cloud and a LiDAR frame: level 0 exact against the oracle, level 1 capped, with capped
    rows actually present (a LiDAR frame alone never reaches 256 neighbours)."""
    from pointgnn_b200.models import graph_gen
    with open(os.path.join(GOLDEN, 'config_car_auto_T3_train.json')) as f:
        kw = json.load(f)['graph_gen_kwargs']
    assert kw['downsample_method'] == 'random' and kw['add_rnd3d']
    assert kw['level_configs'][1]['graph_gen_kwargs']['num_neighbors'] == 256
    clouds = [_cube(90, 12000, 8.0), synth.lidar_frame(91, 6000)[0]]
    fp = _frame_ptr(clouds)
    np.random.seed(9)
    graph_gen.set_seed(9)
    coords, kp, edges, fps = graph_gen.gen_multi_level_local_graph_v3(np.vstack(clouds), frame_ptr=fp,
                                                                      return_frame_ptr=True, **kw)
    full = []
    for lvl, lc in enumerate(kw['level_configs']):
        want = []
        for f in range(len(clouds)):
            s0, s1, d0, d1 = fps[lvl][f], fps[lvl][f + 1], fps[lvl + 1][f], fps[lvl + 1][f + 1]
            want.append(graph.radius_graph(coords[lvl][s0:s1], coords[lvl + 1][d0:d1], lc['graph_gen_kwargs']['radius'])
                        + np.array([[s0, d0]]))
        full.append(np.vstack(want))
    assert np.array_equal(edges[0], full[0])
    _assert_canonical(edges[1])
    n_capped = graph.check_neighbor_cap(full[1], edges[1], 256)
    assert n_capped > 100
    rows = np.bincount(edges[1][:, 1], minlength=len(coords[1]))
    assert rows[fps[1][1]:].max() < 256                     # the LiDAR frame's rows are all below the cap


# ---------------------------------------------------------------------------------------------------------------------
# neighbour cap: ties
# ---------------------------------------------------------------------------------------------------------------------
def test_cap_neighbors_ties_keep_a_sub_multiset():
    """Hand-built CSR rows with repeated sources.  Equal sources have equal priorities, so a row of one repeated source
    ties everywhere (for distinct sources the hash is a bijection and cannot tie).  Every row keeps exactly
    min(length, cap) entries, a sub-multiset of the row, in ascending source order."""
    from pointgnn_b200 import _lib
    cap = 7
    rows = [[5] * 40, [9] * 8, [3] * 7, [], [2] * 100, [1, 1, 1, 1, 6, 6, 6, 6, 6, 8, 8, 8], [4, 4, 4, 4, 4, 4, 4, 4, 12],
            list(range(30)) + [29] * 30, [0, 1, 2], [7] * 33]
    row_ptr = np.concatenate([[0], np.cumsum([len(r) for r in rows])]).astype(np.int32)
    src = np.concatenate([np.asarray(r, np.int32) for r in rows])
    dst = np.repeat(np.arange(len(rows), dtype=np.int32), [len(r) for r in rows])
    rp_t = torch.from_numpy(row_ptr).cuda()
    e_t = torch.from_numpy(np.stack([src, dst])).cuda()
    for seed in (0, 1, 12345, 2 ** 31 - 2, 0xdeadbeef):
        out_rp, out = _lib.cap_neighbors(rp_t, e_t, cap, seed)
        out_rp, out = out_rp.cpu().numpy(), out.cpu().numpy()
        assert np.array_equal(np.diff(out_rp), [min(len(r), cap) for r in rows]), seed
        for i, r in enumerate(rows):
            kept = out[0, out_rp[i]:out_rp[i + 1]]
            assert np.all(out[1, out_rp[i]:out_rp[i + 1]] == i)
            assert np.all(np.diff(kept) >= 0), (seed, i)
            assert not collections.Counter(kept.tolist()) - collections.Counter(r), (seed, i)
            if len(r) <= cap:
                assert kept.tolist() == r


# ---------------------------------------------------------------------------------------------------------------------
# neighbour cap and keypoint choice: distribution over seeds
# ---------------------------------------------------------------------------------------------------------------------
CAP_SEEDS = range(1000, 2000)


def _cap_distribution_scene():
    """Clusters whose members are consecutive point indices: A (20 points from index 0, two identical centres),
    B (cap + 1 = 8 points), D (20 points from index 4 124, behind 4 096 far-away filler points)."""
    rng = np.random.default_rng(3)
    a = _cluster(rng, (0.0, 0.0, 10.0), 20)
    b = _cluster(rng, (5.0, 0.0, 10.0), 8)
    filler = _cube(4, 4096, 20.0, origin=(100.0, 100.0, 100.0))
    d = _cluster(rng, (10.0, 0.0, 10.0), 20)
    pts = np.vstack([a, b, filler, d])
    centers = np.array([(0.0, 0.0, 10.0), (0.0, 0.0, 10.0), (5.0, 0.0, 10.0), (10.0, 0.0, 10.0)], np.float32)
    members = [np.arange(20), np.arange(20), np.arange(20, 28), np.arange(4124, 4144)]
    full = graph.radius_graph(pts, centers, 1.0)
    for i, m in enumerate(members):
        assert np.array_equal(full[full[:, 1] == i, 0], m)
    return pts, centers, members


def test_neighbor_cap_distribution_over_seeds():
    """Seeds as the product draws them (set_seed(k) before each call).  Every member of a capped row is kept with
    probability cap / L (within 5 binomial sigma, consecutive sources included); for L = cap + 1 the dropped member is
    uniform (chi-square); two identical rows get independent subsets; a seed reproduces its output and different
    seeds give different outputs."""
    from pointgnn_b200.models import graph_gen
    cap = 7
    pts, centers, members = _cap_distribution_scene()
    counts = [np.zeros(len(m)) for m in members]
    subsets_a, same_dup = set(), 0
    for k in CAP_SEEDS:
        graph_gen.set_seed(k)
        e = graph_gen.gen_disjointed_rnn_local_graph_v3(pts, centers, 1.0, cap)
        kept = [e[e[:, 1] == i, 0] for i in range(len(centers))]
        for i, m in enumerate(members):
            assert len(kept[i]) == cap
            counts[i][np.searchsorted(m, kept[i])] += 1
        same_dup += int(np.array_equal(kept[0], kept[1]))
        subsets_a.add(tuple(kept[0]))
    n = len(CAP_SEEDS)
    for i, m in enumerate(members):
        p = cap / len(m)
        z = np.abs(counts[i] - n * p) / np.sqrt(n * p * (1 - p))
        assert z.max() < 5.0, (i, z.max())
    dropped = n - counts[2]                                # L = cap + 1: which member was left out
    assert stats.chisquare(dropped).pvalue > 1e-6, dropped
    assert same_dup < n // 100                             # identical rows are not capped identically
    assert len(subsets_a) > 0.95 * n                       # C(20, 7) = 77 520 subsets: repeats are rare
    graph_gen.set_seed(CAP_SEEDS[0])
    e1 = graph_gen.gen_disjointed_rnn_local_graph_v3(pts, centers, 1.0, cap)
    graph_gen.set_seed(CAP_SEEDS[0])
    e2 = graph_gen.gen_disjointed_rnn_local_graph_v3(pts, centers, 1.0, cap)
    assert np.array_equal(e1, e2)


def test_random_keypoint_choice_distribution_over_seeds():
    """Every pick is a member of its voxel, voxels come in first-appearance order, and over seeds the pick inside a
    voxel of m points is uniform (chi-square per voxel)."""
    from pointgnn_b200.models import graph_gen
    rng = np.random.default_rng(21)
    sizes = [1, 2, 3, 5, 8, 13]
    cells = [(i % 3, i // 3, 0) for i in range(len(sizes))]
    pts = [np.zeros((1, 3), np.float32)]          # the grid origin: cell (0, 0, 0) begins at this point
    for cell, m in zip(cells, sizes):
        pts.append(((np.asarray(cell) + 0.1 + 0.6 * rng.random((m - (cell == (0, 0, 0)), 3))) * 0.8).astype(np.float32))
    xyz = np.vstack(pts)
    xyz = xyz[rng.permutation(len(xyz))]          # members of a voxel are not consecutive
    vox = (xyz - xyz.min(axis=0)) // np.float32(0.8)
    keys = [tuple(v) for v in vox.astype(int).tolist()]
    order = list(dict.fromkeys(keys))             # first-appearance order of the voxels (graph_gen.py:133-144)
    members = [np.flatnonzero([k == key for k in keys]) for key in order]
    assert sorted(len(m) for m in members) == sorted(sizes)
    counts = [collections.Counter() for _ in members]
    for k in range(2000, 2600):
        graph_gen.set_seed(k)
        _, kp = graph_gen.multi_layer_downsampling_random(xyz, 0.8, [1])
        assert len(kp[0]) == len(members)
        for o, m in enumerate(members):
            assert kp[0][o, 0] in m, (k, o)
            counts[o][int(kp[0][o, 0])] += 1
    for o, m in enumerate(members):
        if len(m) > 1:
            assert stats.chisquare([counts[o][int(j)] for j in m]).pvalue > 1e-6, (o, counts[o])
