"""CPU tests: the oracle against the committed golden vectors, which hold what the reference's own code computed
(tools/make_golden.py)."""
import os

import numpy as np
import pytest

from oracle import gnn, graph, synth

GOLDEN = os.path.join(os.path.dirname(__file__), 'golden')


def test_synth_is_seeded_and_kitti_shaped():
    a, ia = synth.lidar_frame(3, 2000)
    b, ib = synth.lidar_frame(3, 2000)
    assert a.dtype == np.float32 and a.shape == (2000, 3) and ia.shape == (2000, 1)
    assert np.array_equal(a, b) and np.array_equal(ia, ib)
    c, _ = synth.lidar_frame(4, 2000)
    assert not np.array_equal(a, c)
    assert 0 <= ia.min() and ia.max() < 1
    assert a[:, 2].min() > 0 and a[:, 2].max() < 80.5          # front crop, max range


@pytest.mark.parametrize('name', ['car', 'ped'])
def test_oracle_graph_matches_reference_golden(name, request):
    g = request.getfixturevalue(name)
    coords, keypoints, edges = graph.gen_multi_level_local_graph_v3(g.graph['xyz'], **g.graph_kwargs)
    assert np.array_equal(keypoints[0][:, 0], g.graph['keypoint_idx'])
    # golden edges come from the reference's gen_disjointed_rnn_local_graph_v3 (sklearn ball tree)
    assert np.array_equal(edges[0], g.graph['edges0'])
    assert np.array_equal(edges[1], g.graph['edges1'])
    assert np.array_equal(keypoints[1][:, 0], np.arange(len(keypoints[0])))
    assert np.array_equal(coords[1], g.graph['xyz'][keypoints[0][:, 0]])
    assert coords[2] is coords[1] or np.array_equal(coords[2], coords[1])


def test_oracle_graph_invariants(car):
    e0, e1 = car.graph['edges0'], car.graph['edges1']
    k = len(car.graph['keypoint_idx'])
    for e in (e0, e1):
        assert np.all(np.diff(e[:, 1]) >= 0)                  # grouped by destination (fact 5)
        same = e[1:, 1] == e[:-1, 1]
        assert np.all(e[1:, 0][same] > e[:-1, 0][same])       # canonical: ascending src in a row
    # every vertex has a self loop in the keypoint graph (radius query includes the query point)
    loops = e1[e1[:, 0] == e1[:, 1]]
    assert len(np.unique(loops[:, 1])) == k
    # every keypoint is in its own point set (distance 0 <= r)
    kp = car.graph['keypoint_idx']
    own = set(map(tuple, e0.tolist()))
    assert all((int(kp[j]), j) in own for j in range(0, k, 17))


def test_brute_and_tree_radius_paths_agree():
    xyz, _ = synth.lidar_frame(5, 1500)
    centers = xyz[::7]
    a = graph.radius_graph(xyz, centers, 1.0, method='brute')
    b = graph.radius_graph(xyz, centers, 1.0, method='tree')
    assert np.array_equal(a, b)


def test_voxel_keys_canonical_order():
    xyz, _ = synth.lidar_frame(6, 1200)
    keys, dims = graph.voxel_keys(xyz, 0.4)
    cent = graph.voxel_down_sample(xyz, 0.4)
    assert len(cent) == len(np.unique(keys))
    # centroid j belongs to the j-th smallest key
    ck, _ = graph.voxel_keys(np.vstack([xyz.astype(np.float64), cent]), 0.4)
    # (adding centroids never moves the bounding-box minimum, so keys are comparable)
    assert np.array_equal(np.sort(np.unique(keys)), ck[len(xyz):])


def test_oracle_against_live_reference_graph_gen():
    """tests/golden/graph_live.npz: the edge lists the reference's own gen_disjointed_rnn_local_graph_v3 returned, and
    scikit-learn's kd-tree 1-NN of the voxel centroids, on one frame at two scales."""
    g = np.load(os.path.join(GOLDEN, 'graph_live.npz'))
    xyz = g['xyz']
    for i in range(2):
        voxel, r0, r1 = (float(v) for v in g['params_%d' % i])
        cent = graph.voxel_down_sample(xyz, voxel)
        kp = graph.nearest_point(xyz, cent)
        kxyz = xyz[kp]
        for lvl, (pts, ctr, r) in enumerate(((xyz, kxyz, r0), (kxyz, kxyz, r1))):
            e_ref = g['edges_%d_%d' % (i, lvl)].astype(np.int64)
            assert np.array_equal(graph.canonical_edges(e_ref), graph.radius_graph(pts, ctr, r))
        # kd-tree snap: identical except on exact distance ties (two-point voxels), where the
        # oracle's rule is "lowest index" and sklearn's is traversal order
        idx = g['knn_%d' % i].astype(np.int64)
        assert len(idx) == len(kp)
        diff = np.flatnonzero(idx != kp)
        x64 = xyz.astype(np.float64)
        for j in diff:
            da, db = cent[j] - x64[idx[j]], cent[j] - x64[kp[j]]
            assert (da[0] * da[0] + da[1] * da[1]) + da[2] * da[2] == (db[0] * db[0] + db[1] * db[1]) + db[2] * db[2]
            assert kp[j] < idx[j]


@pytest.mark.parametrize('name', ['car', 'ped'])
def test_oracle_gnn_matches_golden(name, request):
    g = request.getfixturevalue(name)
    coords, keypoints, edges = g.graph_tuple()
    logits, boxes, feats = gnn.predict(g.weights, g.layer_configs, g.config['num_classes'], 7,
                                       g.graph['intensity'], coords, keypoints, edges, return_features=True)
    # same code, same BLAS -> near bit-equal; the tolerance only absorbs BLAS threading differences
    assert np.abs(logits - g.gnn['logits']).max() < 2e-5
    assert np.abs(boxes - g.gnn['boxes']).max() < 2e-5
    assert np.abs(feats[1] - g.gnn['features_pool']).max() < 2e-5
    assert np.abs(feats[-1] - g.gnn['features_last']).max() < 2e-5
    probs = gnn.postprocess(logits)
    assert np.allclose(probs.sum(axis=1), 1.0, atol=1e-5)


def test_oracle_fp32_close_to_fp64(car):
    coords, keypoints, edges = car.graph_tuple()
    l32, b32 = gnn.predict(car.weights, car.layer_configs, 4, 7, car.graph['intensity'], coords, keypoints, edges)
    l64, b64 = gnn.predict(car.weights, car.layer_configs, 4, 7, car.graph['intensity'], coords, keypoints, edges,
                           dtype=np.float64)
    assert np.abs(l32 - l64).max() < 1e-4 and np.abs(b32 - b64).max() < 1e-4


def test_scatter_max_semantics():
    f = np.array([[1., -5.], [3., -7.], [-2., -1.], [9., 9.]], dtype=np.float32)
    out = gnn.graph_scatter_max_fn(f, np.array([2, 0, 2, 0]), 4)       # unsorted ids
    lowest = np.finfo(np.float32).min
    assert np.array_equal(out, np.array([[9., 9.], [lowest, lowest], [1., -1.], [lowest, lowest]], np.float32))


def test_batch_graphs_offsets(car):
    coords, keypoints, edges = car.graph_tuple()
    frame = (car.graph['intensity'], coords, keypoints, edges)
    inp, bc, bk, be = graph.batch_graphs([frame, frame])
    n, k = coords[0].shape[0], coords[1].shape[0]
    assert inp.shape[0] == 2 * n and bc[0].shape[0] == 2 * n and bc[1].shape[0] == 2 * k
    e0 = edges[0]
    assert np.array_equal(be[0][len(e0):], e0 + np.array([[n, k]]))
    assert np.array_equal(be[1][len(edges[1]):], edges[1] + np.array([[k, k]]))
    assert np.array_equal(bk[0][k:], keypoints[0] + n)


def test_checkpoint_reader_matches_golden_weights(car, tmp_path):
    """The reference's car_auto_T3_train checkpoint, rebuilt byte for byte (oracle/golden_checkpoint.py)."""
    from oracle import golden_checkpoint
    from pointgnn_b200.utils import tf_checkpoint
    w = tf_checkpoint.load_checkpoint(golden_checkpoint.rebuild('car_auto_T3_train', str(tmp_path)))
    assert w['Variable'] == 1400000
    for k, v in car.weights.items():
        assert np.array_equal(w[k], v)
    assert w['layer2/extract_vertex_features/fully_connected/weights'].shape == (303, 300)


def test_cpu_reference_baseline_matches_oracle(car):
    """bench.py's CPU baseline (sklearn graph + torch-CPU GNN) computes the same thing as the oracle."""
    from oracle import cpu_reference
    xyz, intensity = car.graph['xyz'], car.graph['intensity']
    coords, kp, edges = cpu_reference.gen_graph(xyz, **car.graph_kwargs)
    co, ko, eo = car.graph_tuple()
    for a, b in zip(edges, eo):
        # keypoints may differ on exact 1-NN ties (sklearn traversal order) -> compare on the oracle's vertices
        pass
    e_lvl1 = cpu_reference.gen_graph.__globals__['ograph'].canonical_edges(edges[1])
    if np.array_equal(kp[0], ko[0]):
        assert np.array_equal(e_lvl1, eo[1])
    logits, boxes, probs = cpu_reference.predict(car.weights, car.layer_configs, 4, 7, intensity, co, ko, eo)
    assert np.abs(logits - car.gnn['logits']).max() < 5e-5
    assert np.abs(boxes - car.gnn['boxes']).max() < 5e-5
    assert np.abs(probs - gnn.postprocess(car.gnn['logits'])).max() < 1e-5


def test_all_shipped_checkpoints_load_and_run_through_the_oracle(tmp_path):
    """Every checkpoint the reference ships (T0..T3, fixed / auto offset, car / ped; rebuilt byte for byte by
    oracle/golden_checkpoint.py) parses with the TF-free reader, names every variable its frozen config asks for, and
    runs through the oracle forward on a small graph - i.e. the restatement covers all shipped layer stacks, not just
    the two golden configurations."""
    import json
    from oracle import golden_checkpoint
    from pointgnn_b200.utils import tf_checkpoint
    xyz, inten = synth.lidar_frame(5, 1500)
    seen = 0
    for name in golden_checkpoint.names():
        with open(os.path.join(GOLDEN, 'config_%s.json' % name)) as f:
            config = json.load(f)
        w = tf_checkpoint.load_checkpoint(golden_checkpoint.rebuild(name, str(tmp_path / name)))
        coords, kp, edges = graph.gen_multi_level_local_graph_v3(xyz, **config['runtime_graph_gen_kwargs'])
        layers = config['model_kwargs']['layer_configs']
        logits, boxes = gnn.predict(w, layers, config['num_classes'], 7, inten, coords, kp, edges)
        k = len(kp[0])
        assert logits.shape == (k, config['num_classes']) and boxes.shape == (k, config['num_classes'], 7)
        assert np.isfinite(logits).all() and np.isfinite(boxes).all()
        n_gnn = sum(1 for lc in layers if lc['type'] == 'scatter_max_graph_auto_center_net')
        assert ('T%d' % n_gnn) in name                       # T0..T3 = number of GNN iterations
        probs = gnn.postprocess(logits)
        assert np.allclose(probs.sum(axis=1), 1.0, atol=1e-5)
        seen += 1
    assert seen == 7


def test_oracle_multiscale_matches_reference_golden():
    """Several distinct downsampling scales (graph_gen.py:17-23, 76-88): tests/golden/graph_multiscale.npz is the
    reference's own multi_layer_downsampling_select (unspecified orders canonicalised, tools/make_golden.py)."""
    import os
    g = np.load(os.path.join(os.path.dirname(__file__), 'golden', 'graph_multiscale.npz'))
    levels = [float(v) for v in g['levels']]
    coords, kp = graph.multi_layer_downsampling_select(g['xyz'], float(g['base_voxel_size']), levels)
    cents = graph.multi_layer_downsampling(g['xyz'], float(g['base_voxel_size']), levels)
    assert int(g['tie_rows']) > 0          # the fixture does exercise the tie rule
    for i in range(len(levels)):
        assert np.array_equal(kp[i][:, 0], g['kp_%d' % i])
        assert np.array_equal(np.asarray(coords[i + 1], dtype=np.float32), g['coords_%d' % (i + 1)])
        assert np.array_equal(np.asarray(cents[i + 1], dtype=np.float64), g['centroids_%d' % (i + 1)])
    # level 2 repeats level 1's scale: identity (graph_gen.py:76-81)
    assert np.array_equal(kp[2][:, 0], np.arange(len(kp[1])))


def test_oracle_scaled_radius_graph_matches_reference_golden():
    """The per-axis `scale` of gen_disjointed_rnn_local_graph_v3 (graph_gen.py:203-206) against edge lists produced by
    the reference's own function (tests/golden/graph_scale.npz)."""
    import os
    g = np.load(os.path.join(os.path.dirname(__file__), 'golden', 'graph_scale.npz'))
    for i in range(3):
        e = graph.gen_disjointed_rnn_local_graph_v3(g['xyz'], g['centers'], float(g['radius']), -1, scale=list(g['scale_%d' % i]))
        assert np.array_equal(e, g['edges_%d' % i])
    assert not np.array_equal(g['edges_0'], g['edges_1'])


def test_oracle_rnd3d_centroids_match_reference_golden():
    """add_rnd3d with the centroid method (graph_gen.py:24-39): tests/golden/graph_rnd3d.npz holds the reference's own
    output for a seeded NumPy generator; the oracle makes the same NumPy calls and must reproduce the centroids bit for
    bit and the snapped indices wherever the nearest vertex is unique."""
    import os
    g = np.load(os.path.join(os.path.dirname(__file__), 'golden', 'graph_rnd3d.npz'))
    levels = [float(v) for v in g['levels']]
    np.random.seed(int(g['seed']))
    cents = graph.multi_layer_downsampling(g['xyz'], float(g['base_voxel_size']), levels, add_rnd3d=True)
    np.random.seed(int(g['seed']))
    coords, kp = graph.multi_layer_downsampling_select(g['xyz'], float(g['base_voxel_size']), levels, add_rnd3d=True)
    for i in range(len(levels)):
        assert np.array_equal(np.asarray(cents[i + 1], dtype=np.float64), g['centroids_%d' % (i + 1)])
        assert (kp[i][:, 0] == g['kp_%d' % i]).mean() > 0.97
    assert np.array_equal(kp[1][:, 0], np.arange(len(kp[0])))


@pytest.mark.parametrize('tag', graph.RANDOM_GOLDEN_CASES)
def test_oracle_random_downsampling_matches_reference_golden(tag):
    """The training-time keypoint choice (graph_gen.py:92-153): tests/golden/graph_random.npz holds the reference's own
    multi_layer_downsampling_random with its random sources patched to recorded numbers.  Fed the same numbers, the
    oracle's restatement must return the same keypoints and vertices - at a repeated scale, at a second distinct scale
    (grid origin = the ORIGINAL cloud's minimum) and with an array voxel size (float64 floor-division)."""
    c = graph.random_golden_case(np.load(os.path.join(GOLDEN, 'graph_random.npz')), tag)
    coords, kp = graph.multi_layer_downsampling_random(c['xyz'], c['voxel'], c['levels'], c['add_rnd3d'],
                                                       shifts=c['shifts'], uniforms=c['uniforms'])
    assert len(kp) == len(c['levels'])
    for li in range(len(c['levels'])):
        assert np.array_equal(kp[li][:, 0], c['kp'][li]), li
        assert coords[li + 1].dtype == np.float32 and np.array_equal(coords[li + 1], c['coords'][li]), li
    if c['edges'] is not None:
        for lvl, r in enumerate(c['radii']):
            assert np.array_equal(graph.radius_graph(coords[lvl], coords[lvl + 1], r), c['edges'][lvl]), lvl


def test_random_golden_discriminates_the_divergences():
    """The fixture's cases would catch a grid origin taken from the previous level and a float32 division for an array
    voxel size: those rules give different keypoints on the same recorded numbers."""
    g = np.load(os.path.join(GOLDEN, 'graph_random.npz'))
    for tag in ('ms_plain', 'ms_rnd3d'):
        c = graph.random_golden_case(g, tag)
        li = 1                                  # the second scale, voxelised on its own minimum
        _, kp = graph.multi_layer_downsampling_random(c['coords'][0], c['voxel'], [c['levels'][li]], c['add_rnd3d'],
                                                      shifts=[c['shifts'][li]], uniforms=[c['uniforms'][li]])
        assert not np.array_equal(kp[0][:, 0], c['kp'][li]), tag
    c = graph.random_golden_case(g, 'arr')
    assert isinstance(c['voxel'], np.ndarray) and c['voxel'].shape == (3,)
    _, kp = graph.multi_layer_downsampling_random(c['xyz'], float(c['voxel'][0]), c['levels'],
                                                  uniforms=c['uniforms'])
    assert len(kp[0]) != len(c['kp'][0])


def _cap_fixture():
    """Radius graph with a long row (dst 0: 6 members), a short one (dst 1: 2), one of exactly the cap (dst 2: 3),
    an empty one (dst 3) and another long one (dst 4: 4); cap 3."""
    full = np.array([[s, 0] for s in (1, 2, 4, 5, 7, 9)] + [[3, 1], [8, 1]] + [[0, 2], [6, 2], [9, 2]] +
                    [[2, 4], [3, 4], [5, 4], [6, 4]], dtype=np.int64)
    capped = np.array([[2, 0], [5, 0], [9, 0], [3, 1], [8, 1], [0, 2], [6, 2], [9, 2], [2, 4], [3, 4], [6, 4]],
                      dtype=np.int64)
    return full, capped


def test_check_neighbor_cap_accepts_a_valid_cap():
    full, capped = _cap_fixture()
    assert graph.check_neighbor_cap(full, capped, 3) == 2
    other = capped.copy()
    other[:3, 0] = (1, 4, 7)                   # any other subset of the long row is as valid
    assert graph.check_neighbor_cap(full, other, 3) == 2
    assert graph.check_neighbor_cap(full, full, 6) == 0


@pytest.mark.parametrize('breakage', ['duplicate', 'outside', 'short_row', 'long_short', 'long_long', 'exact_row',
                                      'moved_dst'])
def test_check_neighbor_cap_rejects_a_broken_cap(breakage):
    """The checker behind the neighbour-cap GPU tests must be able to fail."""
    full, capped = _cap_fixture()
    bad = capped.copy()
    if breakage == 'duplicate':                # a long row keeps one member twice
        bad[1, 0] = bad[0, 0]
    elif breakage == 'outside':                # a long row keeps a point that is not its neighbour
        bad[1, 0] = 3
    elif breakage == 'short_row':              # a short row loses a member for a neighbour of another row
        bad[3, 0] = 6
    elif breakage == 'long_short':             # a long row keeps cap - 1 members
        bad = np.delete(bad, 0, axis=0)
    elif breakage == 'long_long':              # a long row keeps cap + 1 members
        bad = np.vstack([bad, [[1, 0]]])
    elif breakage == 'exact_row':              # a row of exactly the cap loses a member
        bad = np.delete(bad, 6, axis=0)
    else:                                      # an edge changes rows
        bad[10, 1] = 0
    with pytest.raises(AssertionError):
        graph.check_neighbor_cap(full, bad, 3)
