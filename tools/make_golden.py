"""Generate tests/golden/* (run in the BUILD container, where /root/reference exists).

* weights_<cfg>.npz / config_<cfg>.json : the reference's trained checkpoints
  (checkpoints/<cfg>/model-*.{index,data}) decoded with utils/tf_checkpoint.py, and the frozen
  JSON config saved beside them (train.py:591-592).  Data, not code.
* graph_<cfg>.npz : a seeded synthetic frame, the keypoints of the oracle's voxel restatement,
  and the edge lists produced by the REFERENCE's own models/graph_gen.py
  (gen_disjointed_rnn_local_graph_v3, scikit-learn ball tree) on those vertices, in canonical
  (dst, src) order -> pins oracle/graph.py and the CUDA radius kernels to the reference.
* gnn_<cfg>.npz : logits / box encodings / class probabilities / per-layer features obtained by
  executing the REFERENCE'S OWN saved TensorFlow graph (checkpoints/<cfg>/model-N.meta, the
  MetaGraphDef train.py wrote) with the NumPy GraphDef interpreter oracle/graphdef.py on that
  frame with the real weights -> pins oracle/gnn.py and the CUDA kernels to the graph the
  reference built (op order, concat order, gather indices, segment ids), for all seven shipped
  checkpoints.  The script asserts that oracle/gnn.py reproduces those vectors to <= 1e-5.
"""
import glob
import json
import os
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

from oracle import gnn, graph, graphdef, reference_graph, synth  # noqa: E402
from pointgnn_b200.utils import tf_checkpoint  # noqa: E402

GOLDEN = os.path.join(ROOT, 'tests', 'golden')
CONFIGS = {
    'car_auto_T3_train': dict(num_points=3000, frame=7, graph='car_auto_T3_train'),
    'ped_cyl_auto_T3_trainval': dict(num_points=3000, frame=8, graph='ped_cyl_auto_T3_trainval'),
    # the other shipped checkpoints share car_auto_T3_train's graph settings (and its graph fixture)
    'car_auto_T0_train': dict(num_points=3000, frame=7, graph='car_auto_T3_train'),
    'car_auto_T1_train': dict(num_points=3000, frame=7, graph='car_auto_T3_train'),
    'car_auto_T2_train': dict(num_points=3000, frame=7, graph='car_auto_T3_train'),
    'car_auto_T3_trainval': dict(num_points=3000, frame=7, graph='car_auto_T3_train'),
    'car_fixed_T3_train': dict(num_points=3000, frame=7, graph='car_auto_T3_train'),
}


def main():
    os.makedirs(GOLDEN, exist_ok=True)
    ref = reference_graph.load()
    for name, spec in CONFIGS.items():
        ckpt_dir = os.path.join(reference_graph.REFERENCE_ROOT, 'checkpoints', name)
        with open(os.path.join(ckpt_dir, 'config')) as f:
            config = json.load(f)
        with open(os.path.join(GOLDEN, 'config_%s.json' % name), 'w') as f:
            json.dump(config, f, indent=1, sort_keys=True)
        weights = {k: v for k, v in tf_checkpoint.load_checkpoint(ckpt_dir).items()
                   if k.endswith('/weights') or k.endswith('/biases')}
        np.savez(os.path.join(GOLDEN, 'weights_%s.npz' % name), **weights)

        xyz, intensity = synth.lidar_frame(spec['frame'], spec['num_points'])
        kw = config['runtime_graph_gen_kwargs']
        coords, keypoints, edges = graph.gen_multi_level_local_graph_v3(xyz, **kw)
        ref_edges = []
        for lvl, cfg in enumerate(kw['level_configs']):
            e = ref.gen_disjointed_rnn_local_graph_v3(coords[lvl], coords[lvl + 1], **cfg['graph_gen_kwargs'])
            assert np.all(np.diff(e[:, 1]) >= 0), 'reference edges are not grouped by destination'
            e = graph.canonical_edges(e)
            assert np.array_equal(e, edges[lvl]), 'oracle radius graph != reference graph_gen'
            ref_edges.append(e.astype(np.int32))
        if spec['graph'] == name:
            np.savez_compressed(
                os.path.join(GOLDEN, 'graph_%s.npz' % name), xyz=xyz, intensity=intensity,
                keypoint_idx=keypoints[0][:, 0].astype(np.int32),
                edges0=ref_edges[0], edges1=ref_edges[1])
        # the reference's own saved graph, interpreted op by op
        meta = sorted(glob.glob(os.path.join(ckpt_dir, 'model-*.meta')))[-1]
        nodes = graphdef.load_meta_graph(meta)
        pool_node = 'layer1/combined_features/fully_connected_1/Relu'
        last_node = nodes['output/predictor/cls/fully_connected/MatMul'].inputs[0]
        all_vars = tf_checkpoint.load_checkpoint(ckpt_dir)
        out = graphdef.run_forward(meta, all_vars, intensity, coords, keypoints, edges,
                                   extra_nodes=(pool_node, last_node))
        np.savez_compressed(os.path.join(GOLDEN, 'gnn_%s.npz' % name), logits=out['logits'], boxes=out['boxes'],
                            probs=out['probs'], features_pool=out[pool_node], features_last=out[last_node])
        with open(os.path.join(GOLDEN, 'graphdef_ops_%s.json' % name), 'w') as f:
            json.dump({'meta': os.path.basename(meta), 'nodes_total': len(nodes), 'ops_executed': out['ops']},
                      f, indent=1, sort_keys=True)
        logits, boxes, feats = gnn.predict(weights, config['model_kwargs']['layer_configs'],
                                           config['num_classes'], 7, intensity, coords, keypoints, edges,
                                           return_features=True)
        err = max(np.abs(logits - out['logits']).max(), np.abs(boxes - out['boxes']).max(),
                  np.abs(feats[1] - out[pool_node]).max(), np.abs(feats[-1] - out[last_node]).max())
        assert err <= 1e-5, 'oracle/gnn.py differs from the reference graph by %g' % err
        print(name, 'K=%d E0=%d E1=%d' % (len(keypoints[0]), len(edges[0]), len(edges[1])),
              'logits', logits.shape, float(np.abs(logits).max()), 'restatement-vs-graphdef %g' % err)


POST_CASES = [   # (name, label_method, num_classes, nms_overlapped_thres of the shipped config, seed)
    ('car', 'Car', 4, 0.01, 11),
    ('ped', 'Pedestrian_and_Cyclist', 6, 0.2, 12),
]


def post_goldens():
    """tests/golden/post_<case>.npz: run.py:265-325 executed with the reference's own box_encoding.py and nms.py
    (shapely replaced by the convex-polygon stand-in of oracle/postprocess.py) on seeded synthetic network outputs."""
    from oracle import postprocess as pp
    be, nms = pp.reference_modules()
    for name, method, c, thres, seed in POST_CASES:
        pts, enc, probs = pp.synthetic_outputs(seed, num_classes=c)
        out = {'points_xyz': pts, 'box_encodings': enc, 'probs': probs, 'thres': np.float64(thres)}
        for variant in ('uncertainty', 'merge_only', 'score_only', 'plain'):
            r = pp.reference_postprocess_frame(be, nms, probs.copy(), enc.copy(), pts.copy(), method, thres, variant)
            for k in ('label', 'box', 'score', 'nms_index'):
                out['%s_%s' % (variant, k)] = r[k]
            out['cand_index'] = r['cand_index']
            out['decoded'] = r['decoded']
        np.savez_compressed(os.path.join(GOLDEN, 'post_%s.npz' % name), **out)
        print('post', name, 'candidates', len(out['cand_index']), 'kept', len(out['uncertainty_label']))


def kitti_goldens():
    """tests/golden/kitti_io.npz + kitti_result_car.txt: the reference's own dataset/kitti_dataset.py (Open3D stubbed)
    on a synthetic KITTI-format frame - calibration matrices, camera points in image with colours - and run.py:361-429
    (label conversion + file text) assembled from the reference's functions on the post_car detections."""
    import tempfile
    import cv2
    from oracle import kitti as ok
    from oracle import postprocess as pp
    ref = ok.reference_dataset_module()
    be, nms = pp.reference_modules()
    root = tempfile.mkdtemp()
    ok.write_synthetic_kitti(root, [5], 6000)
    ds = ref.KittiDataset(os.path.join(root, 'image/testing/image_2'), os.path.join(root, 'velodyne/testing/velodyne/'),
                          os.path.join(root, 'calib/testing/calib/'), '', num_classes=4, is_training=False)
    calib = ds.get_calib(0)
    pts = ds.get_cam_points_in_image_with_rgb(0, None)
    velo = np.fromfile(os.path.join(root, 'velodyne/testing/velodyne/000000.bin'), dtype=np.float32).reshape(-1, 4)
    image = cv2.imread(os.path.join(root, 'image/testing/image_2/000000.png'))
    # run.py:361-429 with the reference's functions, on the car post-processing fixture
    g = dict(np.load(os.path.join(GOLDEN, 'post_car.npz')))
    labels, boxes, scores = g['uncertainty_label'], g['uncertainty_box'], g['uncertainty_score']
    cand_xyz = g['points_xyz'][g['cand_index'] // 4]

    def occlusion(label, xyz):            # run.py:88-100
        if xyz.shape[0] == 0:
            return 0
        normals, lower, upper = ds.box3d_to_normals(label)
        projected = np.matmul(xyz, np.transpose(normals))
        rates = [(np.max(projected[:, i]) - np.min(projected[:, i])) / (upper[i] - lower[i]) for i in range(3)]
        return rates[0] * rates[1] * rates[2]

    corners_all = nms.boxes_3d_to_corners(boxes)
    names = ['Background', 'Car', 'Car', 'DontCare']
    text = ''
    for i in range(len(corners_all)):
        corners_xy = ds.cam_points_to_image(ref.Points(xyz=corners_all[i], attr=None), calib).xyz[:, :2]
        xmin, ymin = np.amin(corners_xy, axis=0)
        xmax, ymax = np.amax(corners_xy, axis=0)
        clip_xmin, clip_ymin, clip_xmax, clip_ymax = max(xmin, 0.0), max(ymin, 0.0), min(xmax, 1242.0), min(ymax, 375.0)
        truncation_rate = 1.0 - (clip_ymax - clip_ymin) * (clip_xmax - clip_xmin) / ((ymax - ymin) * (xmax - xmin))
        if truncation_rate > 0.4:
            continue
        x3d, y3d, z3d, l, h, w, yaw = boxes[i]
        tmp_label = {"x3d": x3d, "y3d": y3d, "z3d": z3d, "yaw": yaw, "height": h, "width": w, "length": l}
        inside_mask = ds.sel_xyz_in_box3d(tmp_label, cand_xyz)
        score = (1 + occlusion(tmp_label, cand_xyz[inside_mask])) * scores[i]
        for field in (names[labels[i]], -1, -1, 0, clip_xmin, clip_ymin, clip_xmax, clip_ymax, h, w, l, x3d, y3d, z3d, yaw, score):
            text += str(field) + ' '
        text += '\n'
    text += '\n'
    with open(os.path.join(GOLDEN, 'kitti_result_car.txt'), 'w') as f:
        f.write(text)
    np.savez_compressed(os.path.join(GOLDEN, 'kitti_io.npz'), velo=velo, image=image, xyz=pts.xyz, attr=pts.attr,
                        **{'calib_' + k: np.asarray(calib[k]) for k in ('velo_to_cam', 'cam_to_image', 'cam_to_velo', 'P2')})
    with open(os.path.join(GOLDEN, 'kitti_calib.txt'), 'w') as f:
        f.write(ok.CALIB_TEXT)
    print('kitti: points in image', pts.xyz.shape, 'result lines', text.count('\n') - 1)


def _with_recorded_draws(fn, shifts, uniforms):
    """Call fn() - which runs the reference's multi_layer_downsampling_random - with its two random sources patched to
    recorded numbers.  The level a draw belongs to is read from the reference's own loop: li = the number of levels it
    has finished (len(keypoint_indices_list)).  np.random.random((1, 3)) -> shifts[li]; random.choice(seq) for the o-th
    voxel of level li -> seq[floor(uniforms[li][o] * len(seq))].  -> (fn(), {li: number of voxels drawn})."""
    import random as _random
    drawn = {}

    def level_of_caller():
        return len(sys._getframe(2).f_locals['keypoint_indices_list'])

    def fake_choice(seq):
        li = level_of_caller()
        o = drawn.get(li, 0)
        drawn[li] = o + 1
        return seq[min(int(np.float32(uniforms[li][o]) * np.float32(len(seq))), len(seq) - 1)]

    def fake_random(size=None):
        assert size == (1, 3)
        return np.array(shifts[level_of_caller()], dtype=np.float64).reshape(1, 3)

    orig_choice, orig_rand = _random.choice, np.random.random
    _random.choice, np.random.random = fake_choice, fake_random
    try:
        return fn(), drawn
    finally:
        _random.choice, np.random.random = orig_choice, orig_rand


def _floor_divide_boundary_pairs(xyz, voxel):
    """Two points per axis that the float32 and the float64 voxel rule partition differently.  A sits where
    floor_divide(p - min, voxel) in float32 and in float64 disagree on that axis (float32(0.8) > 0.8, so e.g.
    min + 29.6f is voxel 36 in float32 and 37 in float64), B in the middle of the higher of the two voxels; on the other
    two axes both sit in the middle of a voxel beyond the cloud.  One rule puts A and B in one voxel, the other in two."""
    mn, mx = xyz.min(axis=0), xyz.max(axis=0)
    v32 = np.float32(voxel)
    pairs = []
    for a in range(3):
        found = None
        for k in range(20, 400):
            c = np.float32(mn[a] + k * voxel)
            for step in range(-8, 9):
                p = (c.view(np.int32) + np.int32(step)).view(np.float32)
                d = np.float32(p - mn[a])
                i32, i64 = int(np.floor_divide(d, v32)), int(np.floor_divide(np.float64(d), voxel))
                if i32 != i64:
                    found = (p, max(i32, i64))
                    break
            if found:
                break
        assert found, 'no float32/float64 floor-divide disagreement on axis %d' % a
        p, hi = found
        pt = np.empty(3, dtype=np.float32)
        for b in range(3):
            if b != a:         # a voxel of its own beyond the cloud, different for every axis' pair
                pt[b] = np.float32(mn[b] + (np.floor((mx[b] - mn[b]) / voxel) + 3 + 2 * a + 0.5) * voxel)
        pt_a, pt_b = pt.copy(), pt.copy()
        pt_a[a] = p
        pt_b[a] = np.float32(mn[a] + (hi + 0.5) * voxel)
        pairs += [pt_a, pt_b]
    return np.asarray(pairs, dtype=np.float32)


RANDOM_LEVEL_CONFIGS = [   # the structure of configs/*_train_config without the neighbour cap, so edges are exact
    {'graph_gen_kwargs': {'num_neighbors': -1, 'radius': 1.0}, 'graph_gen_method': 'disjointed_rnn_local_graph_v3',
     'graph_level': 0, 'graph_scale': 1},
    {'graph_gen_kwargs': {'num_neighbors': -1, 'radius': 4.0}, 'graph_gen_method': 'disjointed_rnn_local_graph_v3',
     'graph_level': 1, 'graph_scale': 1}]


def graph_random_goldens():
    """tests/golden/graph_random.npz: the reference's OWN multi_layer_downsampling_random (graph_gen.py:92-153) with its
    two random sources patched to recorded numbers (_with_recorded_draws): one grid shift and one uniform array per new
    scale, the uniforms indexed by voxel rank in first-appearance order, which is how the CUDA path consumes them.  The
    CUDA path gets the same numbers as arguments and must return the same keypoints.

    * ``plain`` / ``rnd3d``: levels [1, 1], scalar voxel 0.8, without / with add_rnd3d (keys <kind>_<tag>).
    * ``ms_plain`` / ``ms_rnd3d``: levels [1, 2, 2]: the second scale voxelises level 1's vertices on the grid of the
      ORIGINAL cloud's minimum (:107-110, 123-128), which differs from level 1's own minimum here.
    * ``arr``: voxel np.array([0.8] * 3) through gen_multi_level_local_graph_v3(downsample_method='random') with
      num_neighbors -1, on a cloud with points where float32 and float64 floor-division disagree: an array voxel size
      divides in float64 (:123-124), a scalar one in float32.  The edge lists are the reference's ball tree, canonical.
    Cases after the first two: keys <kind>_<tag>_<level index>; levels_<tag>, voxel_<tag>, add_<tag>, radii_<tag> with
    the edge lists, and xyz_<tag> where the cloud is not ``xyz``.  oracle.graph.random_golden_case reads them back."""
    ref = reference_graph.load()
    xyz, _ = synth.lidar_frame(3, 8000)
    rng = np.random.default_rng(0)
    out = {'xyz': xyz}
    for add in (False, True):
        shift = rng.random((1, 3))
        u = rng.random(len(xyz)).astype(np.float32)
        (vc, kp), _ = _with_recorded_draws(lambda: ref.multi_layer_downsampling_random(xyz, 0.8, [1, 1], add_rnd3d=add),
                                           [shift, None], [u, None])
        tag = 'rnd3d' if add else 'plain'
        out['shift_' + tag] = shift
        out['u_' + tag] = u
        out['kp_' + tag] = kp[0][:, 0].astype(np.int32)
        vc2, kp2 = graph.multi_layer_downsampling_random(xyz, 0.8, [1, 1], add_rnd3d=add, shifts=[shift, None],
                                                         uniforms=[u, None])
        assert np.array_equal(kp[0], kp2[0]) and np.array_equal(vc[1], vc2[1]), 'oracle restatement != reference'
        print('graph_random', tag, 'keypoints', len(kp[0]))

    rng = np.random.default_rng(2)      # a draw for which level 1's minimum differs from the cloud's in both cases
    cases = []
    levels = [1, 2, 2]
    for add in (False, True):
        tag = 'ms_rnd3d' if add else 'ms_plain'
        shifts = [rng.random((1, 3)), rng.random((1, 3)), None]
        uniforms = [rng.random(len(xyz)).astype(np.float32), rng.random(len(xyz)).astype(np.float32), None]
        (vc, kp), drawn = _with_recorded_draws(
            lambda: ref.multi_layer_downsampling_random(xyz, 0.8, levels, add_rnd3d=add), shifts, uniforms)
        uniforms[1] = uniforms[1][:len(vc[1])]         # one per point of the level it voxelises
        vo, ko = graph.multi_layer_downsampling_random(xyz, 0.8, levels, add_rnd3d=add, shifts=shifts, uniforms=uniforms)
        for li in range(len(levels)):
            assert np.array_equal(kp[li], ko[li]) and np.array_equal(vc[li + 1], vo[li + 1]), 'oracle != reference'
        # the fixture tells the grid origins apart: level 1's own minimum partitions level 2 differently
        _, k_own = graph.multi_layer_downsampling_random(vc[1], 0.8, [2], add_rnd3d=add, shifts=[shifts[1]],
                                                         uniforms=[uniforms[1]])
        assert not np.array_equal(k_own[0], kp[1]), 'the second scale does not depend on the grid origin'
        cases.append((tag, xyz, levels, np.float64(0.8), add, shifts, uniforms, vc, kp, None))
        print('graph_random', tag, 'keypoints', [len(k) for k in kp], 'voxels drawn', drawn)

    cloud, _ = synth.lidar_frame(5, 3000)
    cloud = np.vstack([cloud, _floor_divide_boundary_pairs(cloud, 0.8)])
    voxel = np.array([0.8, 0.8, 0.8])
    u = rng.random(len(cloud)).astype(np.float32)
    (vc, kp, edges), _ = _with_recorded_draws(
        lambda: ref.gen_multi_level_local_graph_v3(cloud, voxel, RANDOM_LEVEL_CONFIGS, downsample_method='random'),
        [None, None], [u, None])
    (_, kp_scalar), _ = _with_recorded_draws(lambda: ref.multi_layer_downsampling_random(cloud, 0.8, [1, 1]),
                                             [None, None], [u, None])
    assert len(kp_scalar[0]) != len(kp[0]), 'array and scalar voxel sizes partition this cloud alike'
    vo, ko = graph.multi_layer_downsampling_random(cloud, voxel, [1, 1], shifts=[None, None], uniforms=[u, None])
    edges = [graph.canonical_edges(e) for e in edges]
    for li in range(2):
        assert np.array_equal(kp[li], ko[li]) and np.array_equal(vc[li + 1], vo[li + 1]), 'oracle != reference'
        cfg = RANDOM_LEVEL_CONFIGS[li]
        assert np.array_equal(edges[li], graph.radius_graph(vo[li], vo[li + 1], cfg['graph_gen_kwargs']['radius']))
    cases.append(('arr', cloud, [1, 1], voxel, False, [None, None], [u, None], vc, kp, edges))
    print('graph_random arr keypoints', len(kp[0]), 'with a scalar voxel', len(kp_scalar[0]))

    for tag, pts, lv, vox, add, shifts, uniforms, vc, kp, edges in cases:
        if pts is not xyz:
            out['xyz_' + tag] = pts
        out['levels_' + tag] = np.asarray(lv, dtype=np.float64)
        out['voxel_' + tag] = np.asarray(vox, dtype=np.float64)
        out['add_' + tag] = np.bool_(add)
        for li in range(len(lv)):
            if shifts[li] is not None and add:
                out['shift_%s_%d' % (tag, li)] = shifts[li]
            if uniforms[li] is not None:
                out['u_%s_%d' % (tag, li)] = uniforms[li]
            out['kp_%s_%d' % (tag, li)] = np.asarray(kp[li])[:, 0].astype(np.int32)
            out['coords_%s_%d' % (tag, li + 1)] = np.asarray(vc[li + 1], dtype=np.float32)
        for lvl, e in enumerate(edges or []):
            out['edges_%s_%d' % (tag, lvl)] = e.astype(np.int32)
        if edges:
            out['radii_' + tag] = np.array([c['graph_gen_kwargs']['radius'] for c in RANDOM_LEVEL_CONFIGS])
    out['cases'] = np.array([c[0] for c in cases])
    np.savez_compressed(os.path.join(GOLDEN, 'graph_random.npz'), **out)


def graph_multiscale_goldens():
    """tests/golden/graph_multiscale.npz: the reference's OWN multi_layer_downsampling_select (graph_gen.py:49-90, with
    multi_layer_downsampling :11-47) for SEVERAL distinct scales - which cloud is voxelised, which level is searched,
    the index layout are the reference running.  Two calls inside it have an UNSPECIFIED order upstream and are
    canonicalised: (1) open3d.voxel_down_sample (:41-45; Open3D 0.7 is not installable) is served by the oracle's
    restated voxel rule (ascending voxel key); (2) the kd_tree 1-NN (:84-86) is scikit-learn's own query, but where
    several base vertices are EXACTLY equidistant in fp64 - every voxel with two points: its centroid is their
    midpoint - scikit-learn returns whichever its tree visits first (version dependent); the wrapper returns the
    lowest index among those exact minimisers.  The fixture records how many rows needed (2)."""
    import sys as _sys
    from sklearn.neighbors import NearestNeighbors as _SkNN
    ref = reference_graph.load()
    o3d = _sys.modules['open3d']

    class _Pcd(object):
        points = None
    o3d.PointCloud = _Pcd
    o3d.Vector3dVector = lambda a: np.asarray(a)
    o3d.voxel_down_sample = lambda pcd, voxel_size: type('R', (), {'points': graph.voxel_down_sample(pcd.points, voxel_size)})()
    stats = {'queries': 0, 'ties': 0}

    class _CanonicalTies(object):
        def __init__(self, n_neighbors=1, algorithm='kd_tree', n_jobs=1):
            assert n_neighbors == 1 and algorithm == 'kd_tree'
            self._nn = _SkNN(n_neighbors=1, algorithm=algorithm, n_jobs=n_jobs)

        def fit(self, x):
            self._x = np.asarray(x, dtype=np.float64)
            self._nn.fit(x)
            return self

        def kneighbors(self, q, return_distance=False):
            assert not return_distance
            dist, idx = self._nn.kneighbors(q, return_distance=True)
            q64 = np.asarray(q, dtype=np.float64)
            out = idx.copy()
            for j in range(len(q64)):
                c = self._nn.radius_neighbors(q64[j:j + 1], radius=dist[j, 0] * (1 + 1e-9) + 1e-12,
                                              return_distance=False)[0]
                d = self._x[c] - q64[j]
                d2 = (d[:, 0] * d[:, 0] + d[:, 1] * d[:, 1]) + d[:, 2] * d[:, 2]
                best = np.sort(c[d2 == d2.min()])
                assert idx[j, 0] in best, 'scikit-learn returned a non-minimiser'
                stats['queries'] += 1
                stats['ties'] += int(len(best) > 1)
                out[j, 0] = best[0]
            return out

    xyz, _ = synth.lidar_frame(11, 12000)
    levels = [1, 2, 2, 4.5]
    orig = ref.NearestNeighbors
    ref.NearestNeighbors = _CanonicalTies
    try:
        vc, kp = ref.multi_layer_downsampling_select(xyz, 0.4, levels)
    finally:
        ref.NearestNeighbors = orig
    vo, ko = graph.multi_layer_downsampling_select(xyz, 0.4, levels)
    out = {'xyz': xyz, 'levels': np.asarray(levels, dtype=np.float64), 'base_voxel_size': np.float64(0.4),
           'tie_rows': np.int64(stats['ties']), 'query_rows': np.int64(stats['queries'])}
    for i in range(len(levels)):
        assert np.array_equal(np.asarray(vc[i + 1]), np.asarray(vo[i + 1])), 'oracle coordinates != reference (level %d)' % i
        assert np.array_equal(np.asarray(kp[i]), np.asarray(ko[i])), 'oracle index != reference (level %d)' % i
        out['coords_%d' % (i + 1)] = np.asarray(vc[i + 1], dtype=np.float32)
        out['kp_%d' % i] = np.asarray(kp[i])[:, 0].astype(np.int32)
        print('graph_multiscale level', i, 'scale', levels[i], 'vertices', len(kp[i]))
    print('graph_multiscale: %d of %d 1-NN queries had exactly tied minimisers' % (stats['ties'], stats['queries']))
    cents = ref.multi_layer_downsampling(xyz, 0.4, levels)
    for i in range(len(levels)):
        out['centroids_%d' % (i + 1)] = np.asarray(cents[i + 1], dtype=np.float64)
    np.savez_compressed(os.path.join(GOLDEN, 'graph_multiscale.npz'), **out)


def graph_scale_goldens():
    """tests/golden/graph_scale.npz: the reference's OWN gen_disjointed_rnn_local_graph_v3 with the per-axis `scale`
    argument (graph_gen.py:203-206; float64 division before the ball tree), rows in canonical order."""
    ref = reference_graph.load()
    xyz, _ = synth.lidar_frame(21, 3000)
    centers = xyz[::7].copy()
    out = {'xyz': xyz, 'centers': centers, 'radius': np.float64(1.0)}
    for i, scale in enumerate(([1.0, 0.7, 1.3], [0.3, 1.0, 1.9], [2.0, 2.0, 2.0])):
        e = ref.gen_disjointed_rnn_local_graph_v3(xyz, centers, 1.0, -1, scale=scale)
        e = e[np.lexsort((e[:, 0], e[:, 1]))]
        assert np.array_equal(e, graph.gen_disjointed_rnn_local_graph_v3(xyz, centers, 1.0, -1, scale=scale)), 'oracle != reference'
        out['scale_%d' % i] = np.asarray(scale, dtype=np.float64)
        out['edges_%d' % i] = e.astype(np.int32)
        print('graph_scale', scale, 'edges', len(e))
    np.savez_compressed(os.path.join(GOLDEN, 'graph_scale.npz'), **out)


def graph_rnd3d_goldens():
    """tests/golden/graph_rnd3d.npz: the reference's OWN multi_layer_downsampling / multi_layer_downsampling_select with
    add_rnd3d=True and the centroid method (graph_gen.py:24-39, 82-88), NumPy's global generator seeded; the oracle,
    seeded the same way, must return the same arrays bit for bit (it makes the same NumPy calls)."""
    ref = reference_graph.load()
    xyz, _ = synth.lidar_frame(17, 9000)
    levels = [1, 1, 2.5]
    np.random.seed(7)
    cents = ref.multi_layer_downsampling(xyz, 0.4, levels, add_rnd3d=True)
    np.random.seed(7)
    co = graph.multi_layer_downsampling(xyz, 0.4, levels, add_rnd3d=True)
    np.random.seed(7)
    vc, kp = ref.multi_layer_downsampling_select(xyz, 0.4, levels, add_rnd3d=True)
    np.random.seed(7)
    vo, ko = graph.multi_layer_downsampling_select(xyz, 0.4, levels, add_rnd3d=True)
    out = {'xyz': xyz, 'levels': np.asarray(levels, dtype=np.float64), 'base_voxel_size': np.float64(0.4), 'seed': np.int64(7)}
    exact = 0
    for i in range(len(levels)):
        assert np.array_equal(np.asarray(cents[i + 1]), np.asarray(co[i + 1])), 'oracle centroids != reference'
        # the kd-tree tie rule (lowest index among exact minimisers) only matters for exact ties; with float32-summed
        # centroids there are hardly any, but identical base rows (level 3) still tie
        same = np.asarray(kp[i])[:, 0] == np.asarray(ko[i])[:, 0]
        exact += int(same.sum())
        out['centroids_%d' % (i + 1)] = np.asarray(cents[i + 1], dtype=np.float64)
        out['kp_%d' % i] = np.asarray(kp[i])[:, 0].astype(np.int32)
        out['coords_%d' % (i + 1)] = np.asarray(vc[i + 1], dtype=np.float32)
        print('graph_rnd3d level', i, 'vertices', len(kp[i]), 'oracle index == reference:', int(same.sum()))
    np.savez_compressed(os.path.join(GOLDEN, 'graph_rnd3d.npz'), **out)


def graph_live_goldens():
    """tests/golden/graph_live.npz: the reference's OWN gen_disjointed_rnn_local_graph_v3 (rows as it returns them,
    int16: the frame has 2500 points) on the voxel keypoints of a seeded frame at two scales, and scikit-learn's kd-tree
    1-NN of the voxel centroids."""
    from sklearn.neighbors import NearestNeighbors
    ref = reference_graph.load()
    xyz, _ = synth.lidar_frame(11, 2500)
    out = {'xyz': xyz}
    for i, (voxel, r0, r1) in enumerate(((0.4, 1.0, 4.0), (0.2, 0.4, 1.6))):
        cent = graph.voxel_down_sample(xyz, voxel)
        kxyz = xyz[graph.nearest_point(xyz, cent)]
        for lvl, (pts, ctr, r) in enumerate(((xyz, kxyz, r0), (kxyz, kxyz, r1))):
            out['edges_%d_%d' % (i, lvl)] = ref.gen_disjointed_rnn_local_graph_v3(pts, ctr, r, -1).astype(np.int16)
        out['knn_%d' % i] = NearestNeighbors(n_neighbors=1, algorithm='kd_tree', n_jobs=1).fit(xyz).kneighbors(
            cent, return_distance=False)[:, 0].astype(np.int32)
        out['params_%d' % i] = np.asarray([voxel, r0, r1], dtype=np.float64)
    np.savez_compressed(os.path.join(GOLDEN, 'graph_live.npz'), **out)


def checkpoint_goldens():
    """tests/golden/checkpoints/<cfg>/: each shipped checkpoint in a form small enough to commit - its `checkpoint`
    state file and `.index` table verbatim, and data.json, the byte layout of its `.data` file (tensor name, offset,
    size, the bytes of the non-weight tensors, sha256 of the whole file).  oracle/golden_checkpoint.py rebuilds the
    `.data` file from weights_<cfg>.npz and checks the sha256.  For the checkpoints in FORWARD_META the `.meta` is
    kept too (gzipped), cut down to the forward sub-graph oracle/graphdef.run_forward executes (plus every
    placeholder)."""
    import gzip
    import hashlib
    import shutil
    for name in CONFIGS:
        src = os.path.join(reference_graph.REFERENCE_ROOT, 'checkpoints', name)
        dst = os.path.join(GOLDEN, 'checkpoints', name)
        os.makedirs(dst, exist_ok=True)
        prefix = tf_checkpoint.latest_checkpoint(src)
        base = os.path.basename(prefix)
        shutil.copyfile(os.path.join(src, 'checkpoint'), os.path.join(dst, 'checkpoint'))
        shutil.copyfile(prefix + '.index', os.path.join(dst, base + '.index'))
        with open(prefix + '.data-00000-of-00001', 'rb') as f:
            blob = f.read()
        weights = dict(np.load(os.path.join(GOLDEN, 'weights_%s.npz' % name)))
        tensors, extra = [], {}
        for key, e in sorted(tf_checkpoint.read_index(prefix + '.index').items(), key=lambda kv: kv[1]['offset']):
            assert e['shard'] == 0
            tensors.append([key, e['offset'], e['size']])
            raw = blob[e['offset']:e['offset'] + e['size']]
            if key in weights:
                assert weights[key].astype('<f4').tobytes() == raw, key
            else:
                extra[key] = raw.hex()
        layout = {'data_file': base + '.data-00000-of-00001', 'size': len(blob),
                  'sha256': hashlib.sha256(blob).hexdigest(), 'tensors': tensors, 'extra_hex': extra}
        with open(os.path.join(dst, 'data.json'), 'w') as f:
            json.dump(layout, f, indent=0)
        if name in FORWARD_META:
            meta = sorted(glob.glob(os.path.join(src, 'model-*.meta')))[-1]
            with gzip.open(os.path.join(dst, os.path.basename(meta) + '.gz'), 'wb') as f:
                f.write(forward_meta_graph(meta))
        print('checkpoint', name, len(tensors), 'tensors', sorted(extra))


FORWARD_META = ('car_auto_T1_train', 'car_fixed_T3_train')


def forward_meta_graph(meta_path):
    """-> a MetaGraphDef (bytes) holding only the NodeDefs run_forward reads, each copied byte for byte."""
    def ld(num, payload):
        head, n = b'', len(payload)
        tag = num << 3 | 2
        for v in (tag, n):
            while True:
                b, v = v & 0x7F, v >> 7
                head += bytes([b | 0x80]) if v else bytes([b])
                if not v:
                    break
        return head + payload

    nodes = graphdef.load_meta_graph(meta_path)
    keep = graphdef._closure(nodes, [graphdef.LOGITS_NODE, graphdef.BOXES_NODE, graphdef.PROBS_NODE])
    keep |= {n for n in nodes if nodes[n].op == 'Placeholder'}
    with open(meta_path, 'rb') as f:
        buf = memoryview(f.read())
    body = b''
    for num, _, val in graphdef.fields(buf):
        if num == 2:
            for n2, _, v2 in graphdef.fields(val):
                if n2 == 1 and graphdef._node(v2).name in keep:
                    body += ld(1, bytes(v2))
    return ld(2, body)


if __name__ == '__main__':
    which = sys.argv[1] if len(sys.argv) > 1 else 'all'
    if which in ('all', 'graph_live'):
        graph_live_goldens()
    if which in ('all', 'graph_random'):
        graph_random_goldens()
    if which in ('all', 'graph_multiscale'):
        graph_multiscale_goldens()
    if which in ('all', 'graph_scale'):
        graph_scale_goldens()
    if which in ('all', 'graph_rnd3d'):
        graph_rnd3d_goldens()
    if which in ('all', 'gnn'):
        main()
    if which in ('all', 'post'):
        post_goldens()
    if which in ('all', 'kitti'):
        kitti_goldens()
    if which in ('all', 'checkpoints'):     # after 'gnn': rebuilt from the weights_<cfg>.npz it writes
        checkpoint_goldens()
