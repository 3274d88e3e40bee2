"""CPU oracle for graph construction (reference models/graph_gen.py).

TEST INFRASTRUCTURE (see oracle/__init__.py).

* ``voxel_down_sample``      restates ``open3d.voxel_down_sample`` as called at
  reference graph_gen.py:41-45 (Open3D 0.7 is not installable here; semantics
  recalled: grid origin = min_bound - voxel/2, index = floor((p-origin)/voxel),
  fp64 centroid).  Open3D's output order is an unordered_map iteration order,
  i.e. unspecified; the oracle DEFINES the canonical order = ascending linear
  voxel key ix + iy*dimx + iz*dimx*dimy (same key formula as reference
  graph_gen.py:30-31).
* ``nearest_point``          restates the kd_tree 1-NN snap of
  graph_gen.py:84-87 (fp64 squared distances, ties -> lowest index).
* ``multi_layer_downsampling_select`` / ``gen_multi_level_local_graph_v3`` /
  ``gen_disjointed_rnn_local_graph_v3`` follow graph_gen.py:49-90, 155-195,
  197-220 with the same signatures and return layouts.
* ``radius_graph``           restates the ball_tree radius query of
  graph_gen.py:207-220: predicate ((dx*dx + dy*dy) + dz*dz) <= r*r evaluated in
  fp64 on float32-valued coordinates (sklearn _binary_tree leaf test), boundary
  inclusive; rows grouped by ascending destination (centre) index.  sklearn's
  intra-row order is its tree traversal order (unspecified), so the oracle's
  canonical intra-row order is ascending source index.
"""
import numpy as np


def voxel_keys(points_xyz, voxel_size):
    """fp64 voxel index + linear key of every point -> (keys int64 [N], dims int64 [3])."""
    p = np.asarray(points_xyz, dtype=np.float64)
    voxel = np.broadcast_to(np.asarray(voxel_size, dtype=np.float64), (3,))
    origin = p.min(axis=0) - voxel * 0.5
    idx = np.floor((p - origin[None, :]) / voxel[None, :]).astype(np.int64)
    dims = idx.max(axis=0) + 1
    keys = idx[:, 0] + idx[:, 1] * dims[0] + idx[:, 2] * dims[0] * dims[1]
    return keys, dims


def voxel_down_sample(points_xyz, voxel_size):
    """-> fp64 centroids [K,3], ascending linear voxel key; sums in ascending point order."""
    p = np.asarray(points_xyz, dtype=np.float64)
    keys, _ = voxel_keys(points_xyz, voxel_size)
    order = np.argsort(keys, kind='stable')
    sk = keys[order]
    starts = np.flatnonzero(np.concatenate([[True], sk[1:] != sk[:-1]]))
    counts = np.diff(np.concatenate([starts, [len(sk)]]))
    sp = p[order]
    cent = np.empty((len(starts), 3), dtype=np.float64)
    # sequential fp64 accumulation in ascending point index (np.add.reduceat is
    # pairwise for long runs, so accumulate explicitly to keep the order defined)
    maxc = int(counts.max())
    acc = np.zeros((len(starts), 3), dtype=np.float64)
    for j in range(maxc):
        live = counts > j
        acc[live] += sp[starts[live] + j]
    cent[:] = acc / counts[:, None].astype(np.float64)
    return cent


def nearest_point(base_points, queries, chunk=512):
    """argmin_j ((dx*dx+dy*dy)+dz*dz) in fp64, ties -> lowest j.  -> int64 [Q]."""
    b = np.asarray(base_points, dtype=np.float64)
    q = np.asarray(queries, dtype=np.float64)
    out = np.empty(q.shape[0], dtype=np.int64)
    for s in range(0, q.shape[0], chunk):
        d = q[s:s + chunk, None, :] - b[None, :, :]
        d2 = (d[..., 0] * d[..., 0] + d[..., 1] * d[..., 1]) + d[..., 2] * d[..., 2]
        out[s:s + chunk] = np.argmin(d2, axis=1)
    return out


def multi_layer_downsampling(points_xyz, base_voxel_size, levels=[1], add_rnd3d=False):
    """reference graph_gen.py:11-47.  add_rnd3d=True (:24-39) draws np.random.random((1, 3)) exactly where the
    reference does and uses the same NumPy calls (float32 reduceat sums in argsort order), so with the same generator
    state it returns the reference's arrays bit for bit."""
    points_xyz = np.asarray(points_xyz)
    xmin, ymin, zmin = np.amin(points_xyz, axis=0)
    xyz_offset = np.asarray([[xmin, ymin, zmin]])
    downsampled_list = [points_xyz]
    last_level = 0
    for level in levels:
        if np.isclose(last_level, level):
            downsampled_list.append(np.copy(downsampled_list[-1]))
        elif add_rnd3d:
            xyz_idx = (points_xyz - xyz_offset + base_voxel_size * level * np.random.random((1, 3))) // \
                (base_voxel_size * level)
            xyz_idx = xyz_idx.astype(np.int32)
            dim_x, dim_y, dim_z = np.amax(xyz_idx, axis=0) + 1
            keys = xyz_idx[:, 0] + xyz_idx[:, 1] * dim_x + xyz_idx[:, 2] * dim_y * dim_x
            sorted_order = np.argsort(keys)
            sorted_keys = keys[sorted_order]
            sorted_points_xyz = points_xyz[sorted_order]
            _, lens = np.unique(sorted_keys, return_counts=True)
            indices = np.hstack([[0], lens[:-1]]).cumsum()
            downsampled_list.append(np.array(np.add.reduceat(sorted_points_xyz, indices, axis=0) / lens[:, np.newaxis]))
        else:
            downsampled_list.append(
                voxel_down_sample(points_xyz, np.asarray(base_voxel_size) * level))
        last_level = level
    return downsampled_list


def multi_layer_downsampling_select(points_xyz, base_voxel_size, levels=[1], add_rnd3d=False):
    """reference graph_gen.py:49-90."""
    vertex_coord_list = multi_layer_downsampling(points_xyz, base_voxel_size, levels, add_rnd3d)
    num_levels = len(vertex_coord_list)
    keypoint_indices_list = []
    last_level = 0
    for i in range(1, num_levels):
        current_level = levels[i - 1]
        base_points = vertex_coord_list[i - 1]
        current_points = vertex_coord_list[i]
        if np.isclose(current_level, last_level):
            vertex_coord_list[i] = base_points
            keypoint_indices_list.append(np.expand_dims(np.arange(base_points.shape[0]), axis=1))
        else:
            indices = nearest_point(base_points, current_points)[:, None]
            vertex_coord_list[i] = base_points[indices[:, 0], :]
            keypoint_indices_list.append(indices)
        last_level = current_level
    return vertex_coord_list, keypoint_indices_list


def _within(points, centers_chunk, r2):
    d = centers_chunk[:, None, :] - points[None, :, :]
    d2 = (d[..., 0] * d[..., 0] + d[..., 1] * d[..., 1]) + d[..., 2] * d[..., 2]
    return d2 <= r2


def radius_graph(points_xyz, center_xyz, radius, method='auto', chunk=256):
    """-> edges [E,2] int64 rows (point_idx, center_idx); dst ascending, src ascending in a row."""
    p = np.asarray(points_xyz, dtype=np.float64)
    c = np.asarray(center_xyz, dtype=np.float64)
    r2 = float(radius) * float(radius)
    if method == 'auto':
        method = 'brute' if p.shape[0] * c.shape[0] <= (1 << 24) else 'tree'
    src, dst = [], []
    if method == 'brute':
        for s in range(0, c.shape[0], chunk):
            ci, pi = np.nonzero(_within(p, c[s:s + chunk], r2))
            src.append(pi)
            dst.append(ci + s)
    else:
        # candidate superset from a kd-tree with an inflated radius, then the
        # exact fp64 predicate decides (so the tree's own rounding never matters)
        from scipy.spatial import cKDTree
        tree = cKDTree(p)
        cand = tree.query_ball_point(c, float(radius) * (1.0 + 1e-6) + 1e-9, return_sorted=True)
        lens = np.fromiter((len(x) for x in cand), dtype=np.int64, count=len(cand))
        pi = np.fromiter((j for x in cand for j in x), dtype=np.int64, count=int(lens.sum()))
        ci = np.repeat(np.arange(c.shape[0], dtype=np.int64), lens)
        d = c[ci] - p[pi]
        d2 = (d[:, 0] * d[:, 0] + d[:, 1] * d[:, 1]) + d[:, 2] * d[:, 2]
        ok = d2 <= r2
        src.append(pi[ok])
        dst.append(ci[ok])
    src = np.concatenate(src) if src else np.zeros(0, np.int64)
    dst = np.concatenate(dst) if dst else np.zeros(0, np.int64)
    return np.stack([src, dst], axis=1).astype(np.int64)


def gen_disjointed_rnn_local_graph_v3(points_xyz, center_xyz, radius, num_neighbors,
                                      neighbors_downsample_method='random', scale=None):
    """reference graph_gen.py:197-220 (inference path: num_neighbors <= 0, no random cap)."""
    if scale is not None:
        scale = np.array(scale)
        points_xyz = points_xyz / scale
        center_xyz = center_xyz / scale
    assert num_neighbors <= 0, 'random neighbour cap is training-only (non-deterministic)'
    return radius_graph(points_xyz, center_xyz, radius)


def canonical_edges(edges):
    """Sort an [E,2] (src,dst) list by (dst, src) - the parity form of SURVEY 8c."""
    e = np.asarray(edges).astype(np.int64)
    order = np.lexsort((e[:, 0], e[:, 1]))
    return e[order]


def gen_multi_level_local_graph_v3(points_xyz, base_voxel_size, level_configs,
                                   add_rnd3d=False, downsample_method='center'):
    """reference graph_gen.py:155-195, downsample_method='center'."""
    assert downsample_method == 'center'
    if isinstance(base_voxel_size, list):
        base_voxel_size = np.array(base_voxel_size)
    scales = [config['graph_scale'] for config in level_configs]
    vertex_coord_list, keypoint_indices_list = multi_layer_downsampling_select(
        points_xyz, base_voxel_size, scales, add_rnd3d=add_rnd3d)
    edges_list = []
    for config in level_configs:
        graph_level = config['graph_level']
        assert config['graph_gen_method'] == 'disjointed_rnn_local_graph_v3'
        edges_list.append(gen_disjointed_rnn_local_graph_v3(
            vertex_coord_list[graph_level], vertex_coord_list[graph_level + 1],
            **config['graph_gen_kwargs']))
    return vertex_coord_list, keypoint_indices_list, edges_list


def batch_graphs(frames):
    """reference train.py:135-171 (batch_data) restricted to the graph tuple.

    frames: list of (input_v, vertex_coord_list, keypoint_indices_list, edges_list).
    """
    n_in, n_coord, n_kp, n_edges = zip(*frames)
    level_num = len(n_coord[0])
    b_kp, b_edges = [], []
    for lvl in range(level_num - 1):
        centers, vertices = [], []
        point_counter = 0
        center_counter = 0
        for b in range(len(frames)):
            centers.append(n_kp[b][lvl] + point_counter)
            e = n_edges[b][lvl]
            vertices.append(np.hstack([e[:, [0]] + point_counter, e[:, [1]] + center_counter]))
            point_counter += n_coord[b][lvl].shape[0]
            center_counter += n_kp[b][lvl].shape[0]
        b_kp.append(np.vstack(centers))
        b_edges.append(np.vstack(vertices))
    b_coord = [np.vstack([n_coord[b][lvl] for b in range(len(frames))]) for lvl in range(level_num)]
    return np.vstack(n_in), b_coord, b_kp, b_edges


# ---------------------------------------------------------------------------------------------
# training-time path (graph_gen.py:92-153, 210-214) with the randomness made explicit
# ---------------------------------------------------------------------------------------------
def multi_layer_downsampling_random(points_xyz, base_voxel_size, levels=(1,), add_rnd3d=False, shifts=None,
                                    uniforms=None):
    """graph_gen.py:92-153 with its two random sources as arguments: ``shifts[i]`` = the np.random.random((1,3))
    draw of level i (add_rnd3d), ``uniforms[i][o]`` in [0,1) picks the point of the o-th voxel (first-appearance
    order) as seq[floor(u * len(seq))] - what random.choice does with its own generator.  Same arithmetic as the
    reference: float32 floor-division without the shift, float64 with it.
    -> (vertex_coord_list, keypoint_indices_list)."""
    points_xyz = np.asarray(points_xyz)
    xyz_offset = np.asarray([np.amin(points_xyz, axis=0)])
    vertex_coord_list = [points_xyz]
    keypoint_indices_list = []
    last_level = 0
    for li, level in enumerate(levels):
        last = vertex_coord_list[-1]
        if np.isclose(last_level, level):
            vertex_coord_list.append(np.copy(last))
            keypoint_indices_list.append(np.expand_dims(np.arange(len(last)), axis=1))
        else:
            if not add_rnd3d:
                xyz_idx = (last - xyz_offset) // (base_voxel_size * level)
            else:
                xyz_idx = (last - xyz_offset + base_voxel_size * level * np.asarray(shifts[li]).reshape(1, 3)) \
                    // (base_voxel_size * level)
            xyz_idx = xyz_idx.astype(np.int32)
            dim_x, dim_y, _ = np.amax(xyz_idx, axis=0) + 1
            keys = xyz_idx[:, 0] + xyz_idx[:, 1] * dim_x + xyz_idx[:, 2] * dim_y * dim_x
            voxels = {}
            for pidx, key in enumerate(keys.tolist()):
                voxels.setdefault(key, []).append(pidx)
            chosen = []
            for o, key in enumerate(voxels):
                seq = voxels[key]
                pick = min(int(np.float32(uniforms[li][o]) * np.float32(len(seq))), len(seq) - 1)
                chosen.append(seq[pick])
            vertex_coord_list.append(last[chosen])
            keypoint_indices_list.append(np.expand_dims(np.array(chosen), axis=1))
        last_level = level
    return vertex_coord_list, keypoint_indices_list


RANDOM_GOLDEN_CASES = ('plain', 'rnd3d', 'ms_plain', 'ms_rnd3d', 'arr')


def random_golden_case(g, tag):
    """One case of tests/golden/graph_random.npz (written by tools/make_golden.py::graph_random_goldens) ->
    dict(xyz, levels, voxel, add_rnd3d, shifts, uniforms, kp, coords, radii, edges).  shifts / uniforms / kp / coords
    are per level (None where a level draws nothing); kp[i] indexes level i's input, coords[i] = level i + 1's vertices;
    voxel is a Python float for a scalar voxel size and a float64 array for an array one; radii / edges: the radius
    graph of each level where the case pins it, else None."""
    files = set(g.files)
    if tag in ('plain', 'rnd3d'):          # levels [1, 1], scalar voxel 0.8
        add, xyz, kp0 = tag == 'rnd3d', g['xyz'], g['kp_' + tag]
        return dict(xyz=xyz, levels=[1, 1], voxel=0.8, add_rnd3d=add,
                    shifts=[g['shift_' + tag] if add else None, None], uniforms=[g['u_' + tag], None],
                    kp=[kp0, np.arange(len(kp0))], coords=[xyz[kp0], xyz[kp0]], radii=None, edges=None)
    levels = [float(v) for v in g['levels_' + tag]]
    voxel = g['voxel_' + tag]

    def per_level(kind, shift_by=0):
        keys = ['%s_%s_%d' % (kind, tag, li + shift_by) for li in range(len(levels))]
        return [g[k] if k in files else None for k in keys]
    edges = None
    if 'radii_' + tag in files:
        edges = [g['edges_%s_%d' % (tag, lvl)] for lvl in range(len(g['radii_' + tag]))]
    return dict(xyz=g['xyz_' + tag] if 'xyz_' + tag in files else g['xyz'], levels=levels,
                voxel=float(voxel) if voxel.ndim == 0 else voxel, add_rnd3d=bool(g['add_' + tag]),
                shifts=per_level('shift'), uniforms=per_level('u'), kp=per_level('kp'), coords=per_level('coords', 1),
                radii=[float(r) for r in g['radii_' + tag]] if edges is not None else None, edges=edges)


def check_neighbor_cap(full_edges, capped_edges, num_neighbors):
    """Invariants of graph_gen.py:210-214 that do not depend on the draw: per destination, rows of at most
    num_neighbors entries are unchanged, longer rows keep exactly num_neighbors DISTINCT members of the row."""
    full_edges, capped_edges = np.asarray(full_edges), np.asarray(capped_edges)
    ndst = int(max(full_edges[:, 1].max(), capped_edges[:, 1].max())) + 1 if len(full_edges) else 0
    f_cnt = np.bincount(full_edges[:, 1], minlength=ndst)
    c_cnt = np.bincount(capped_edges[:, 1], minlength=ndst)
    assert np.array_equal(c_cnt, np.minimum(f_cnt, num_neighbors)), 'row lengths'
    full_set = set(map(tuple, full_edges.tolist()))
    cap_list = list(map(tuple, capped_edges.tolist()))
    assert len(set(cap_list)) == len(cap_list), 'duplicate edge'
    assert all(e in full_set for e in cap_list), 'edge outside the radius graph'
    short = f_cnt <= num_neighbors
    keep = short[full_edges[:, 1]]
    want = set(map(tuple, full_edges[keep].tolist()))
    got = set(e for e in cap_list if short[e[1]])
    assert want == got, 'an uncapped row changed'
    return int((~short).sum())
