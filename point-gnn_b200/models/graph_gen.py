"""Graph generation on the GPU - same names / signatures / return layout as the reference's
``models/graph_gen.py`` (/root/reference/models/graph_gen.py).

* ``get_graph_generate_fn``              graph_gen.py:222-227
* ``gen_multi_level_local_graph_v3``     graph_gen.py:155-195
* ``gen_disjointed_rnn_local_graph_v3``  graph_gen.py:197-220
* ``multi_layer_downsampling``           graph_gen.py:11-47  (voxel centroids, any list of scales)
* ``multi_layer_downsampling_select``    graph_gen.py:49-90  (any list of scales)

Inputs may be NumPy arrays (the reference's calling convention, run.py:219-222: arrays are
copied to the GPU, results copied back as NumPy) or torch CUDA tensors (results stay on the
device).  Built: the deterministic inference path (``add_rnd3d=False``, ``downsample_method='center'``,
``num_neighbors <= 0``) and the training-time path of train.py:88-90 with configs/*_train_config
(``downsample_method='random'`` with or without ``add_rnd3d``, ``num_neighbors > 0``,
graph_gen.py:92-153, 210-214).  The random path takes its randomness from NumPy's global generator for
the per-frame grid shift - the same ``np.random.random((1, 3))`` draws as the reference, frame-major: a batch of
F frames gets the draws of F one-frame calls - and from this module's CUDA generator (``set_seed``) for the
per-voxel choice and the neighbour cap, where the reference uses Python's ``random`` / ``np.random.choice``:
results are equal in distribution, not draw by draw.  Everything else is the reference's arithmetic: every level's
grid starts at the minimum of the original cloud (graph_gen.py:107-110), and the voxel index is a float32
floor-division for a scalar voxel size and float64 for an array one or with ``add_rnd3d``, as NumPy promotes.
Given the same random numbers (``_downsampling_random(..., uniform=, shifts=)``) the keypoints are the reference's
bit for bit (tests/test_graph_random_gpu.py against tests/golden/graph_random.npz).  A capped neighbour row keeps
its members in ascending source order where the reference keeps ``np.random.choice``'s random order; the model
only reduces a row with a segment max, which does not depend on the order.  ``add_rnd3d`` with the centroid method
(graph_gen.py:24-39) draws the same ``np.random.random((1, 3))`` per frame and new scale; its centroids equal the
reference's to float32 summation accuracy (the reference sums in float32 in ``argsort`` order).  The per-axis
``scale`` of ``gen_disjointed_rnn_local_graph_v3`` (graph_gen.py:203-206) is divided in float64 inside the
kernels, as ``points_xyz / np.array(scale)`` does.

Extra, backwards-compatible keyword ``frame_ptr``: a [F+1] int array batching F frames in one
call; the result is then exactly what the reference's ``batch_data`` (train.py:135-171) builds
from F per-frame graphs (indices offset per level).

Canonical orders (the reference leaves both unspecified, SURVEY facts 5 and 7): keypoints in
ascending linear voxel key, edges grouped by destination with ascending source inside a group.
"""
import numpy as np
import torch

from .. import _lib


_rng = {'gen': None}


def set_seed(seed):
    """Seed of the generator behind the random keypoint choice and the random neighbour cap."""
    g = torch.Generator(device=_device())
    g.manual_seed(int(seed))
    _rng['gen'] = g


def _generator():
    if _rng['gen'] is None:
        set_seed(torch.initial_seed() & 0x7fffffff)
    return _rng['gen']


def _device():
    if not torch.cuda.is_available():
        raise RuntimeError('point-gnn_b200 needs a CUDA device (no CPU fallback)')
    return torch.device('cuda', torch.cuda.current_device())


class _Cloud(object):
    """points + frame partition on the device, remembering the caller's array type."""

    def __init__(self, points_xyz, frame_ptr=None):
        self.numpy_io = not isinstance(points_xyz, torch.Tensor)
        dev = _device()
        if self.numpy_io:
            pts = torch.from_numpy(np.ascontiguousarray(points_xyz, dtype=np.float32)).to(dev)
        else:
            pts = points_xyz.to(device=dev, dtype=torch.float32).contiguous()
        assert pts.dim() == 2 and pts.shape[1] == 3, 'points_xyz must be [N, 3]'
        if frame_ptr is None:
            fp = torch.tensor([0, pts.shape[0]], dtype=torch.int32, device=dev)
        elif isinstance(frame_ptr, torch.Tensor):
            fp = frame_ptr.to(device=dev, dtype=torch.int32).contiguous()
        else:
            fp = torch.from_numpy(np.asarray(frame_ptr, dtype=np.int32)).to(dev)
        self.xyz = pts
        self.frame_ptr = fp


def _voxel_vector(base_voxel_size, level):
    v = np.asarray(base_voxel_size, dtype=np.float64) * level      # graph_gen.py:44
    return np.broadcast_to(v, (3,)).astype(np.float64)


def _divides_in_float64(base_voxel_size, level):
    """graph_gen.py:123-124 floor-divides float32 coordinates by ``base_voxel_size*level``: NumPy keeps float32 for a
    Python float and promotes to float64 for a float64 array (what gen_multi_level_local_graph_v3 makes of a list,
    :172-173).  Probe the promotion instead of restating it."""
    if isinstance(base_voxel_size, list):
        base_voxel_size = np.array(base_voxel_size)
    return (np.zeros((1, 3), dtype=np.float32) // (base_voxel_size * level)).dtype == np.float64


def _new_scales(levels):
    """Per level: True where it voxelises (a scale different from the previous level's), False for a repeated scale."""
    flags, last_level = [], 0
    for level in levels:
        flags.append(not np.isclose(level, last_level))
        last_level = level
    return flags


def _rnd3d_shifts(levels, num_frames):
    """The add_rnd3d grid shifts of F frames, one np.random.random((1, 3)) per frame and new scale, drawn frame-major:
    the reference builds one frame per call (train.py:88-90), and each call draws its scales in turn (graph_gen.py:24-27,
    126-128), so frame f gets the draws F separate calls would give it.  -> per level: [F,3] float64 or None."""
    new = [li for li, is_new in enumerate(_new_scales(levels)) if is_new]
    draws = [[np.random.random((1, 3)) for _ in new] for _ in range(num_frames)]
    shifts = [None] * len(levels)
    for j, li in enumerate(new):
        shifts[li] = np.vstack([draws[f][j] for f in range(num_frames)])
    return shifts


def multi_layer_downsampling(points_xyz, base_voxel_size, levels=[1], add_rnd3d=False):
    """graph_gen.py:11-47 (Open3D branch).  -> list: the cloud, then per level the fp64 voxel centroids of the
    ORIGINAL cloud at that scale (a level with the previous level's scale repeats the previous entry, :21-22).
    Centroid order: ascending linear voxel key per frame (Open3D's own order is unspecified)."""
    cloud = _Cloud(points_xyz)
    downsampled_list = [cloud.xyz]
    last_level = 0
    for level in levels:
        if np.isclose(last_level, level):
            downsampled_list.append(downsampled_list[-1].clone())
        elif add_rnd3d:      # graph_gen.py:24-39: grid shifted by one np.random.random((1, 3)) draw per level
            _, _, cent = _lib.voxel_keypoints_rnd3d(cloud.xyz, cloud.frame_ptr, _voxel_vector(base_voxel_size, level),
                                                    np.random.random((1, 3)), want_centroids=True)
            downsampled_list.append(cent)
        else:
            cent, _ = _lib.voxel_centroids(cloud.xyz, cloud.frame_ptr, _voxel_vector(base_voxel_size, level))
            downsampled_list.append(cent)
        last_level = level
    if cloud.numpy_io:
        downsampled_list = [np.asarray(points_xyz)] + [d.cpu().numpy() for d in downsampled_list[1:]]
    return downsampled_list


def multi_layer_downsampling_select(points_xyz, base_voxel_size, levels=[1], add_rnd3d=False):
    """graph_gen.py:49-90.  -> (vertex_coord_list, keypoint_indices_list)."""
    cloud = _Cloud(points_xyz)
    vertex_coord_list, keypoint_indices_list, _ = _downsampling_select(cloud, base_voxel_size, levels, add_rnd3d)
    if cloud.numpy_io:
        vertex_coord_list = [v.cpu().numpy() for v in vertex_coord_list]
        keypoint_indices_list = [k.cpu().numpy().astype(np.int64) for k in keypoint_indices_list]
    return vertex_coord_list, keypoint_indices_list


def _downsampling_select(cloud, base_voxel_size, levels, add_rnd3d):
    """Device-side body of multi_layer_downsampling_select, also tracking each level's frame_ptr."""
    num_frames = cloud.frame_ptr.numel() - 1
    vertex_coord_list = [cloud.xyz]
    frame_ptr_list = [cloud.frame_ptr]
    keypoint_indices_list = []
    # graph_gen.py:24-39: random grid shift, one np.random.random((1, 3)) per frame and new scale (frame-major)
    shifts = _rnd3d_shifts(levels, num_frames) if add_rnd3d else None
    for li, (level, is_new) in enumerate(zip(levels, _new_scales(levels))):
        base_points = vertex_coord_list[-1]
        if not is_new:
            # same scale (a gnn layer): identity, graph_gen.py:76-81
            vertex_coord_list.append(base_points)
            frame_ptr_list.append(frame_ptr_list[-1])
            kidx = torch.arange(base_points.shape[0], dtype=torch.int32, device=base_points.device)[:, None]
            kidx._pg_trusted = (int(base_points.shape[0]), kidx._version)
            keypoint_indices_list.append(kidx)
        else:
            # graph_gen.py:41-45 voxelises the ORIGINAL cloud, :84-88 snaps to the previous level.
            voxel = _voxel_vector(base_voxel_size, level)
            if add_rnd3d:
                idx, kp_fp, _ = _lib.voxel_keypoints_rnd3d(cloud.xyz, cloud.frame_ptr, voxel, shifts[li], base_points,
                                                           frame_ptr_list[-1])
            elif base_points is cloud.xyz:
                # every shipped config: one distinct scale, previous level == original cloud (one grid, one kernel)
                idx, kp_fp = _lib.voxel_keypoints(cloud.xyz, cloud.frame_ptr, voxel)
            else:
                # a second distinct scale (graph_gen.py:17-23, 76-88): nearest vertex of the previous level
                idx, kp_fp = _lib.voxel_keypoints_select(cloud.xyz, cloud.frame_ptr, voxel, base_points,
                                                         frame_ptr_list[-1])
            vertex_coord_list.append(_lib.gather_rows(base_points, idx))
            frame_ptr_list.append(kp_fp)
            kidx = idx[:, None]
            kidx._pg_trusted = (int(base_points.shape[0]), kidx._version)    # rows of the level it was snapped to
            keypoint_indices_list.append(kidx)
    return vertex_coord_list, keypoint_indices_list, frame_ptr_list


def multi_layer_downsampling_random(points_xyz, base_voxel_size, levels=[1], add_rnd3d=False):
    """graph_gen.py:92-153.  -> (vertex_coord_list, keypoint_indices_list)."""
    cloud = _Cloud(points_xyz)
    vertex_coord_list, keypoint_indices_list, _ = _downsampling_random(cloud, base_voxel_size, levels, add_rnd3d)
    if cloud.numpy_io:
        vertex_coord_list = [v.cpu().numpy() for v in vertex_coord_list]
        keypoint_indices_list = [k.cpu().numpy().astype(np.int64) for k in keypoint_indices_list]
    return vertex_coord_list, keypoint_indices_list


def _downsampling_random(cloud, base_voxel_size, levels, add_rnd3d, uniform=None, shifts=None):
    """Device-side body of multi_layer_downsampling_random.  ``uniform`` / ``shifts`` (tests): explicit random
    numbers per level instead of draws from the generators - ``uniform[li]`` one float32 in [0,1) per voxel of level li
    in first-appearance order (at least one per point of the previous level), ``shifts[li]`` the [F,3] grid shifts."""
    vertex_coord_list = [cloud.xyz]
    frame_ptr_list = [cloud.frame_ptr]
    keypoint_indices_list = []
    num_frames = cloud.frame_ptr.numel() - 1
    if add_rnd3d and shifts is None:
        shifts = _rnd3d_shifts(levels, num_frames)
    for li, (level, is_new) in enumerate(zip(levels, _new_scales(levels))):
        base_points = vertex_coord_list[-1]
        if not is_new:
            vertex_coord_list.append(base_points)
            frame_ptr_list.append(frame_ptr_list[-1])
            kidx = torch.arange(base_points.shape[0], dtype=torch.int32, device=base_points.device)[:, None]
            kidx._pg_trusted = (int(base_points.shape[0]), kidx._version)
            keypoint_indices_list.append(kidx)
        else:
            # graph_gen.py:115: the PREVIOUS level is voxelised (not the original cloud as in the centroid method), on the
            # grid whose origin is the minimum of the ORIGINAL cloud (:107-110) at every level
            if add_rnd3d:
                shift = shifts[li]
            elif _divides_in_float64(base_voxel_size, level):
                shift = np.zeros((num_frames, 3))       # a zero shift takes the kernel's exact float64 quotient
            else:
                shift = None
            u = uniform[li] if uniform is not None else torch.rand(base_points.shape[0], generator=_generator(),
                                                                   device=base_points.device, dtype=torch.float32)
            idx, kp_fp = _lib.random_keypoints(cloud.xyz, cloud.frame_ptr, _voxel_vector(base_voxel_size, level), shift,
                                               base_points, frame_ptr_list[-1], u)
            vertex_coord_list.append(_lib.gather_rows(base_points, idx))
            frame_ptr_list.append(kp_fp)
            kidx = idx[:, None]
            kidx._pg_trusted = (int(base_points.shape[0]), kidx._version)
            keypoint_indices_list.append(kidx)
    return vertex_coord_list, keypoint_indices_list, frame_ptr_list


def _radius_edges(points, point_fp, centers, center_fp, radius, num_neighbors,
                  neighbors_downsample_method='random', scale=None, cap_seed=None):
    if num_neighbors > 0 and neighbors_downsample_method != 'random':
        raise NotImplementedError('only neighbors_downsample_method="random" exists in the reference (graph_gen.py:211)')
    sc = None
    if scale is not None:
        # graph_gen.py:203-206: points_xyz / np.array(scale) is a float64 division; it is done inside the kernels
        sc = np.broadcast_to(np.asarray(scale, dtype=np.float64), (3,))
        if np.any(sc <= 0):
            raise ValueError('scale must be positive')
    row_ptr, edges = _lib.radius_graph(points, point_fp, centers, center_fp, radius, scale=sc)
    if num_neighbors > 0:
        # graph_gen.py:210-214: rows longer than num_neighbors keep a random subset of that size
        seed = cap_seed if cap_seed is not None else int(torch.randint(0, 2 ** 31 - 1, (1,), generator=_generator(),
                                                                      device=points.device))
        _, edges = _lib.cap_neighbors(row_ptr, edges, num_neighbors, seed)
    edges = edges.t()     # [E,2] view whose columns (src, dst) are contiguous
    # index ranges are guaranteed by construction: lets model.predict skip the per-layer range check
    edges._pg_trusted = (int(points.shape[0]), int(centers.shape[0]), edges._version)
    return edges


def _is_two_level(level_configs, add_rnd3d):
    """level 0: cloud -> keypoints of one scale, level 1: the same keypoints -> themselves (configs/*_config)."""
    if add_rnd3d or len(level_configs) != 2:
        return False
    a, b = level_configs
    if a['graph_level'] != 0 or b['graph_level'] != 1 or not np.isclose(a['graph_scale'], b['graph_scale']):
        return False
    for c in (a, b):
        kw = c['graph_gen_kwargs']
        if kw.get('num_neighbors', -1) > 0 or kw.get('scale') is not None:
            return False
    return True


def _two_level_graph(cloud, base_voxel_size, level_configs):
    a, b = level_configs
    idx, kp_fp, kp_xyz, e0, e1 = _lib.multi_level_graph(
        cloud.xyz, cloud.frame_ptr, _voxel_vector(base_voxel_size, a['graph_scale']),
        a['graph_gen_kwargs']['radius'], b['graph_gen_kwargs']['radius'])
    n, k = int(cloud.xyz.shape[0]), int(kp_xyz.shape[0])
    kidx0 = idx[:, None]
    kidx0._pg_trusted = (n, kidx0._version)
    kidx1 = torch.arange(k, dtype=torch.int32, device=kp_xyz.device)[:, None]
    kidx1._pg_trusted = (k, kidx1._version)
    edges0, edges1 = e0.t(), e1.t()
    edges0._pg_trusted = (n, k, edges0._version)
    edges1._pg_trusted = (k, k, edges1._version)
    return ([cloud.xyz, kp_xyz, kp_xyz], [kidx0, kidx1], [edges0, edges1], [cloud.frame_ptr, kp_fp, kp_fp])


def gen_disjointed_rnn_local_graph_v3(points_xyz, center_xyz, radius, num_neighbors,
                                      neighbors_downsample_method='random', scale=None):
    """graph_gen.py:197-220.  -> [E,2] (point_idx, center_idx)."""
    pc = _Cloud(points_xyz)
    cc = _Cloud(center_xyz)
    edges = _radius_edges(pc.xyz, pc.frame_ptr, cc.xyz, cc.frame_ptr, radius, num_neighbors,
                          neighbors_downsample_method, scale)
    if pc.numpy_io:
        return np.ascontiguousarray(edges.cpu().numpy()).astype(np.int64)
    return edges


def gen_multi_level_local_graph_v3(points_xyz, base_voxel_size, level_configs, add_rnd3d=False,
                                   downsample_method='center', frame_ptr=None, return_frame_ptr=False):
    """graph_gen.py:155-195.  -> (vertex_coord_list, keypoint_indices_list, edges_list)."""
    if isinstance(base_voxel_size, list):
        base_voxel_size = np.array(base_voxel_size)
    if downsample_method not in ('center', 'random'):
        raise KeyError(downsample_method)
    cloud = _Cloud(points_xyz, frame_ptr)
    scales = [config['graph_scale'] for config in level_configs]
    for config in level_configs:
        if config['graph_gen_method'] != 'disjointed_rnn_local_graph_v3':
            raise KeyError(config['graph_gen_method'])
    if downsample_method == 'center' and _is_two_level(level_configs, add_rnd3d) and cloud.xyz.shape[0] > 0:
        # the structure of every shipped config: ONE library call, one host round trip
        vertex_coord_list, keypoint_indices_list, edges_list, frame_ptr_list = _two_level_graph(
            cloud, base_voxel_size, level_configs)
    else:
        if downsample_method == 'center':
            vertex_coord_list, keypoint_indices_list, frame_ptr_list = _downsampling_select(
                cloud, base_voxel_size, scales, add_rnd3d)
        else:       # graph_gen.py:179-181
            vertex_coord_list, keypoint_indices_list, frame_ptr_list = _downsampling_random(
                cloud, base_voxel_size, scales, add_rnd3d)
        edges_list = []
        for config in level_configs:
            graph_level = config['graph_level']
            edges_list.append(_radius_edges(vertex_coord_list[graph_level], frame_ptr_list[graph_level],
                                            vertex_coord_list[graph_level + 1], frame_ptr_list[graph_level + 1],
                                            **config['graph_gen_kwargs']))
    if cloud.numpy_io:
        vertex_coord_list = [v.cpu().numpy() for v in vertex_coord_list]
        keypoint_indices_list = [k.cpu().numpy().astype(np.int64) for k in keypoint_indices_list]
        edges_list = [np.ascontiguousarray(e.cpu().numpy()).astype(np.int64) for e in edges_list]
        frame_ptr_list = [f.cpu().numpy() for f in frame_ptr_list]
    if return_frame_ptr:
        return vertex_coord_list, keypoint_indices_list, edges_list, frame_ptr_list
    return vertex_coord_list, keypoint_indices_list, edges_list


def get_graph_generate_fn(method_name):
    """graph_gen.py:222-227."""
    method_map = {
        'disjointed_rnn_local_graph_v3': gen_disjointed_rnn_local_graph_v3,
        'multi_level_local_graph_v3': gen_multi_level_local_graph_v3,
    }
    return method_map[method_name]
