"""ctypes binding of libpointgnn_b200.so (C ABI: include/pointgnn_b200.h).

The library is loaded on first use and the import fails loudly when it is
missing or lacks a symbol - there is no CPU or PyTorch fallback behind these
wrappers.  Arguments are torch CUDA tensors; only their device pointers, sizes
and the current CUDA stream cross the boundary.
"""
import ctypes
import os

import torch

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, 'libpointgnn_b200.so')

PG_ERR_CAPACITY = -3

c_i32p = ctypes.c_void_p
c_f32p = ctypes.c_void_p
c_i64 = ctypes.c_int64
c_i32 = ctypes.c_int32

# name -> (restype, argtypes); must list every symbol include/pointgnn_b200.h declares
SIGNATURES = {
    'pg_version': (ctypes.c_int, []),
    'pg_last_error': (ctypes.c_char_p, []),
    'pg_device_is_sm100': (ctypes.c_int, []),
    'pg_launch_count': (c_i64, []),
    'pg_tc_available': (ctypes.c_int, []),
    'pg_tc_launch_count': (c_i64, [c_i32]),
    'pg_voxel_keypoints': (ctypes.c_int, [c_f32p, c_i32p, c_i32, c_i64, ctypes.POINTER(ctypes.c_double),
                                          c_i32p, c_i64, c_i32p, ctypes.POINTER(c_i64), ctypes.c_void_p]),
    'pg_voxel_centroids': (ctypes.c_int, [c_f32p, c_i32p, c_i32, c_i64, ctypes.POINTER(ctypes.c_double),
                                          ctypes.c_void_p, c_i64, c_i32p, ctypes.POINTER(c_i64), ctypes.c_void_p]),
    'pg_voxel_keypoints_select': (ctypes.c_int, [c_f32p, c_i32p, c_i32, c_i64, ctypes.POINTER(ctypes.c_double),
                                                 c_f32p, c_i32p, c_i64, c_i32p, c_i64, c_i32p,
                                                 ctypes.POINTER(c_i64), ctypes.c_void_p]),
    'pg_voxel_keypoints_rnd3d': (ctypes.c_int, [c_f32p, c_i32p, c_i32, c_i64, ctypes.POINTER(ctypes.c_double),
                                                ctypes.POINTER(ctypes.c_double), c_f32p, c_i32p, c_i64, c_i32p,
                                                ctypes.c_void_p, c_i64, c_i32p, ctypes.POINTER(c_i64), ctypes.c_void_p]),
    'pg_radius_graph_count': (ctypes.c_int, [c_f32p, c_i32p, c_f32p, c_i32p, c_i32, c_i64, c_i64,
                                             ctypes.c_double, c_i32p, ctypes.POINTER(c_i64), ctypes.c_void_p]),
    'pg_radius_graph_fill': (ctypes.c_int, [c_f32p, c_i32p, c_f32p, c_i32p, c_i32, c_i64, c_i64,
                                            ctypes.c_double, c_i32p, c_i64, c_i32p, c_i32p, ctypes.c_void_p]),
    'pg_radius_graph': (ctypes.c_int, [c_f32p, c_i32p, c_f32p, c_i32p, c_i32, c_i64, c_i64, ctypes.c_double,
                                       c_i32p, c_i32p, c_i32p, c_i64, ctypes.POINTER(c_i64), ctypes.c_void_p]),
    'pg_radius_graph_scaled': (ctypes.c_int, [c_f32p, c_i32p, c_f32p, c_i32p, c_i32, c_i64, c_i64, ctypes.c_double,
                                              ctypes.POINTER(ctypes.c_double), c_i32p, c_i32p, c_i32p, c_i64,
                                              ctypes.POINTER(c_i64), ctypes.c_void_p]),
    'pg_multi_level_graph': (ctypes.c_int, [c_f32p, c_i32p, c_i32, c_i64, ctypes.POINTER(ctypes.c_double),
                                            ctypes.c_double, ctypes.c_double, c_i32p, c_i64, c_i32p, c_f32p,
                                            c_i32p, c_i32p, c_i32p, c_i64, c_i32p, c_i32p, c_i32p, c_i64,
                                            ctypes.POINTER(c_i64), ctypes.c_void_p]),
    'pg_random_keypoints': (ctypes.c_int, [c_f32p, c_i32p, c_i32, c_i64, ctypes.POINTER(ctypes.c_double),
                                           ctypes.POINTER(ctypes.c_double), c_f32p, c_i32p, c_i64, c_f32p, c_i32p,
                                           c_i64, c_i32p, ctypes.POINTER(c_i64), ctypes.c_void_p]),
    'pg_cap_neighbors': (ctypes.c_int, [c_i32p, c_i32p, c_i64, c_i32, ctypes.c_uint32, c_i32p, c_i32p, c_i32p, c_i64,
                                        ctypes.POINTER(c_i64), ctypes.c_void_p]),
    'pg_scatter_max': (ctypes.c_int, [c_f32p, c_i32p, c_i64, c_i32, c_i64, c_f32p, ctypes.c_void_p]),
    'pg_scatter_sum': (ctypes.c_int, [c_f32p, c_i32p, c_i64, c_i32, c_i64, c_f32p, ctypes.c_void_p]),
    'pg_scatter_mean': (ctypes.c_int, [c_f32p, c_i32p, c_i64, c_i32, c_i64, c_f32p, ctypes.c_void_p]),
    'pg_gather_rows': (ctypes.c_int, [c_f32p, c_i64, c_i32, c_i32p, c_i64, c_f32p, ctypes.c_void_p]),
    'pg_fully_connected': (ctypes.c_int, [c_f32p, c_i64, c_i32, c_f32p, c_f32p, c_i32, c_i32, c_f32p, c_f32p,
                                          c_i32, ctypes.c_void_p]),
    'pg_edge_mlp_max': (ctypes.c_int, [c_i32, c_f32p, c_i32, c_f32p, c_f32p, c_i32p, c_i32p, c_i32p, c_i64, c_i64,
                                       c_i64, ctypes.POINTER(ctypes.c_void_p), ctypes.POINTER(ctypes.c_void_p),
                                       ctypes.POINTER(c_i32), c_i32, c_f32p, c_i32, ctypes.c_void_p]),
    'pg_softmax_rows': (ctypes.c_int, [c_f32p, c_i64, c_i32, c_f32p, ctypes.c_void_p]),
    'pg_check_edges': (ctypes.c_int, [c_i32p, c_i32p, c_i64, c_i64, c_i64, ctypes.c_void_p]),
    'pg_cam_points_in_image': (ctypes.c_int, [c_f32p, c_i32p, c_i32, c_i64, ctypes.POINTER(ctypes.c_float),
                                              ctypes.POINTER(ctypes.c_double), ctypes.POINTER(c_i32), ctypes.c_void_p,
                                              ctypes.POINTER(c_i64), c_f32p, c_f32p, c_i32, c_i64, c_i32p,
                                              ctypes.POINTER(c_i64), ctypes.c_void_p]),
    'pg_decode_boxes': (ctypes.c_int, [c_f32p, c_f32p, c_i64, c_i32, ctypes.POINTER(ctypes.c_float), c_f32p,
                                       ctypes.c_void_p]),
    'pg_postprocess': (ctypes.c_int, [c_f32p, c_f32p, c_f32p, c_i32p, c_i32, c_i64, c_i32,
                                      ctypes.POINTER(ctypes.c_float), ctypes.c_double, c_i32, c_i64, c_i32p, c_f32p,
                                      c_f32p, c_i32p, c_i64, c_i32p, c_i32p, c_i32p, ctypes.POINTER(c_i64),
                                      ctypes.c_void_p]),
    'pg_nms_boxes_3d': (ctypes.c_int, [c_i32p, c_f32p, c_f32p, c_i32p, c_i32, c_i64, ctypes.c_double,
                                       ctypes.c_double, c_i32, c_i64, c_i32p, c_f32p, c_f32p, c_i32p, c_i64, c_i32p,
                                       ctypes.POINTER(c_i64), ctypes.c_void_p]),
    'pg_layer_create': (ctypes.c_int, [c_i32, ctypes.POINTER(ctypes.c_void_p), ctypes.POINTER(ctypes.c_void_p),
                                       ctypes.POINTER(c_i32), c_i32, c_i32, ctypes.c_void_p,
                                       ctypes.POINTER(ctypes.c_void_p)]),
    'pg_layer_destroy': (ctypes.c_int, [ctypes.c_void_p]),
    'pg_layer_mlp': (ctypes.c_int, [ctypes.c_void_p, c_f32p, c_i64, c_i32, c_f32p, c_f32p, ctypes.c_void_p]),
    'pg_layer_edge_mlp_max': (ctypes.c_int, [ctypes.c_void_p, c_f32p, c_f32p, c_f32p, c_i32p, c_i32p, c_i32p, c_i64,
                                             c_i64, c_i64, c_f32p, c_i32, ctypes.c_void_p]),
    'pg_layer_predictor': (ctypes.c_int, [ctypes.c_void_p, c_f32p, c_i64, c_f32p, c_f32p, c_f32p, ctypes.c_void_p]),
}
PG_LAYER_MLP, PG_LAYER_EDGE_POOL, PG_LAYER_EDGE_GNN, PG_LAYER_PREDICTOR = 0, 1, 2, 3
PG_FLAG_TRUSTED_INDICES = 0x100

_lib = None


class PointGNNError(RuntimeError):
    """A C-ABI call returned a negative status."""

    def __init__(self, code, message):
        super().__init__('libpointgnn_b200 error %d: %s' % (code, message))
        self.code = code


def load():
    """Load (once) and type the shared library; raise if it is absent or incomplete."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.isfile(LIB_PATH):
        raise ImportError(
            'libpointgnn_b200.so not found at %s - build it with `python -c "import __graft_entry__ as g; '
            'g.build()"` or `make -C point-gnn_b200/csrc`; there is no CPU fallback' % LIB_PATH)
    lib = ctypes.CDLL(LIB_PATH)
    for name, (restype, argtypes) in SIGNATURES.items():
        fn = getattr(lib, name)      # AttributeError if the symbol is missing
        fn.restype = restype
        fn.argtypes = argtypes
    _lib = lib
    return lib


def _check(code):
    if code < 0:
        raise PointGNNError(code, load().pg_last_error().decode())
    return code


def _stream():
    return ctypes.c_void_p(torch.cuda.current_stream().cuda_stream)


def _ptr(t, dtype, name):
    if t is None:
        return None
    if not isinstance(t, torch.Tensor) or not t.is_cuda:
        raise TypeError('%s must be a CUDA tensor (there is no CPU path)' % name)
    if t.dtype != dtype:
        raise TypeError('%s must be %s, got %s' % (name, dtype, t.dtype))
    if not t.is_contiguous():
        raise ValueError('%s must be contiguous' % name)
    return ctypes.c_void_p(t.data_ptr())


def launch_count():
    return int(load().pg_launch_count())


def device_is_sm100():
    return bool(load().pg_device_is_sm100())


def tc_launch_count(which=0):
    """tcgen05 launches so far: which=0 fused edge kernel, 1 dense-layer kernel."""
    return int(load().pg_tc_launch_count(int(which)))


def tc_available():
    """True when the tcgen05 (precision=1) kernels are compiled in and the device is sm_100."""
    return bool(load().pg_tc_available())


# ---------------------------------------------------------------------------------------------
# graph construction
# ---------------------------------------------------------------------------------------------

def voxel_keypoints(xyz, frame_ptr, voxel_size):
    """-> (keypoint_idx [K] int32 global point rows, kp_frame_ptr [F+1] int32)."""
    lib = load()
    n = xyz.shape[0]
    num_frames = frame_ptr.numel() - 1
    out_idx = torch.empty(n, dtype=torch.int32, device=xyz.device)
    out_fp = torch.empty(num_frames + 1, dtype=torch.int32, device=xyz.device)
    vs = (ctypes.c_double * 3)(*[float(v) for v in voxel_size])
    k = c_i64(0)
    _check(lib.pg_voxel_keypoints(_ptr(xyz, torch.float32, 'xyz'), _ptr(frame_ptr, torch.int32, 'frame_ptr'),
                                  num_frames, n, vs, _ptr(out_idx, torch.int32, 'out'), n,
                                  _ptr(out_fp, torch.int32, 'out_fp'), ctypes.byref(k), _stream()))
    return out_idx[:k.value], out_fp


def voxel_centroids(xyz, frame_ptr, voxel_size):
    """pg_voxel_centroids -> (centroids [K,3] float64, frame_ptr [F+1] int32)."""
    lib = load()
    n = xyz.shape[0]
    num_frames = frame_ptr.numel() - 1
    out = torch.empty((n, 3), dtype=torch.float64, device=xyz.device)
    out_fp = torch.empty(num_frames + 1, dtype=torch.int32, device=xyz.device)
    vs = (ctypes.c_double * 3)(*[float(v) for v in voxel_size])
    k = c_i64(0)
    _check(lib.pg_voxel_centroids(_ptr(xyz, torch.float32, 'xyz'), _ptr(frame_ptr, torch.int32, 'frame_ptr'),
                                  num_frames, n, vs, _ptr(out, torch.float64, 'out'), n,
                                  _ptr(out_fp, torch.int32, 'out_fp'), ctypes.byref(k), _stream()))
    return out[:k.value], out_fp


def voxel_keypoints_select(xyz, frame_ptr, voxel_size, base_xyz, base_frame_ptr):
    """pg_voxel_keypoints_select -> (keypoint_idx [K] int32 rows of base_xyz, kp_frame_ptr [F+1] int32)."""
    lib = load()
    n = xyz.shape[0]
    num_frames = frame_ptr.numel() - 1
    out_idx = torch.empty(n, dtype=torch.int32, device=xyz.device)
    out_fp = torch.empty(num_frames + 1, dtype=torch.int32, device=xyz.device)
    vs = (ctypes.c_double * 3)(*[float(v) for v in voxel_size])
    k = c_i64(0)
    _check(lib.pg_voxel_keypoints_select(_ptr(xyz, torch.float32, 'xyz'), _ptr(frame_ptr, torch.int32, 'frame_ptr'),
                                         num_frames, n, vs, _ptr(base_xyz, torch.float32, 'base_xyz'),
                                         _ptr(base_frame_ptr, torch.int32, 'base_frame_ptr'), base_xyz.shape[0],
                                         _ptr(out_idx, torch.int32, 'out'), n, _ptr(out_fp, torch.int32, 'out_fp'),
                                         ctypes.byref(k), _stream()))
    return out_idx[:k.value], out_fp


def voxel_keypoints_rnd3d(xyz, frame_ptr, voxel_size, shift, base_xyz=None, base_frame_ptr=None, want_centroids=False):
    """pg_voxel_keypoints_rnd3d.  shift: [F,3] float64 host array.  -> (keypoint_idx [K] int32 rows of base_xyz or None,
    kp_frame_ptr [F+1] int32, centroids [K,3] float64 or None)."""
    import numpy as np
    lib = load()
    n = xyz.shape[0]
    num_frames = frame_ptr.numel() - 1
    out_idx = torch.empty(n, dtype=torch.int32, device=xyz.device) if base_xyz is not None else None
    cent = torch.empty((n, 3), dtype=torch.float64, device=xyz.device) if want_centroids else None
    out_fp = torch.empty(num_frames + 1, dtype=torch.int32, device=xyz.device)
    vs = (ctypes.c_double * 3)(*[float(v) for v in voxel_size])
    sh_arr = np.ascontiguousarray(shift, dtype=np.float64).reshape(num_frames, 3)
    k = c_i64(0)
    _check(lib.pg_voxel_keypoints_rnd3d(
        _ptr(xyz, torch.float32, 'xyz'), _ptr(frame_ptr, torch.int32, 'frame_ptr'), num_frames, n, vs,
        sh_arr.ctypes.data_as(ctypes.POINTER(ctypes.c_double)), _ptr(base_xyz, torch.float32, 'base_xyz'),
        _ptr(base_frame_ptr, torch.int32, 'base_frame_ptr'), 0 if base_xyz is None else base_xyz.shape[0],
        _ptr(out_idx, torch.int32, 'out'), _ptr(cent, torch.float64, 'centroids'), n,
        _ptr(out_fp, torch.int32, 'out_fp'), ctypes.byref(k), _stream()))
    return (None if out_idx is None else out_idx[:k.value]), out_fp, (None if cent is None else cent[:k.value])


def random_keypoints(xyz, frame_ptr, voxel_size, shift, base_xyz, base_frame_ptr, uniform):
    """pg_random_keypoints.  xyz / frame_ptr: the original cloud (grid origin); base_xyz / base_frame_ptr: the points
    voxelised; shift: None or [F,3] float64 host array; uniform: [len(base_xyz)] CUDA fp32 in [0,1).
    -> (keypoint_idx [K] int32 rows of base_xyz, kp_frame_ptr [F+1] int32)."""
    import numpy as np
    lib = load()
    n = base_xyz.shape[0]
    num_frames = frame_ptr.numel() - 1
    if base_frame_ptr.numel() != num_frames + 1:
        raise ValueError('base_frame_ptr has %d entries, expected %d' % (base_frame_ptr.numel(), num_frames + 1))
    if uniform.numel() < n:
        raise ValueError('uniform has %d entries, need one per base point (%d)' % (uniform.numel(), n))
    out_idx = torch.empty(n, dtype=torch.int32, device=xyz.device)
    out_fp = torch.empty(num_frames + 1, dtype=torch.int32, device=xyz.device)
    vs = (ctypes.c_double * 3)(*[float(v) for v in voxel_size])
    sh = None
    if shift is not None:
        sh_arr = np.ascontiguousarray(shift, dtype=np.float64).reshape(num_frames, 3)
        sh = sh_arr.ctypes.data_as(ctypes.POINTER(ctypes.c_double))
    k = c_i64(0)
    _check(lib.pg_random_keypoints(_ptr(xyz, torch.float32, 'xyz'), _ptr(frame_ptr, torch.int32, 'frame_ptr'), num_frames,
                                   xyz.shape[0], vs, sh, _ptr(base_xyz, torch.float32, 'base_xyz'),
                                   _ptr(base_frame_ptr, torch.int32, 'base_frame_ptr'), n,
                                   _ptr(uniform, torch.float32, 'uniform'), _ptr(out_idx, torch.int32, 'out'), n,
                                   _ptr(out_fp, torch.int32, 'out_fp'), ctypes.byref(k), _stream()))
    return out_idx[:k.value], out_fp


def cap_neighbors(row_ptr, edges, num_neighbors, seed):
    """pg_cap_neighbors on the (row_ptr, [2,E] edges) pair of radius_graph.  -> (row_ptr', [2,E'] edges)."""
    lib = load()
    num_rows = row_ptr.numel() - 1
    e = edges.shape[1]
    out_rp = torch.empty_like(row_ptr)
    buf = torch.empty((2, max(e, 1)), dtype=torch.int32, device=edges.device)
    n = c_i64(0)
    src = edges[0].contiguous() if e else edges.new_zeros(1)
    _check(lib.pg_cap_neighbors(_ptr(row_ptr, torch.int32, 'row_ptr'), _ptr(src, torch.int32, 'src'), num_rows,
                                int(num_neighbors), ctypes.c_uint32(int(seed) & 0xffffffff),
                                _ptr(out_rp, torch.int32, 'out_rp'), ctypes.c_void_p(buf[0].data_ptr()),
                                ctypes.c_void_p(buf[1].data_ptr()), buf.shape[1], ctypes.byref(n), _stream()))
    return out_rp, buf[:, :n.value]


_edge_capacity = {}


def radius_graph(points, point_frame_ptr, centers, center_frame_ptr, radius, scale=None):
    """-> (row_ptr [K+1] int32, edges [2,E] int32 with row 0 = src, row 1 = dst).  scale: None or 3 positive
    per-axis divisors (graph_gen.py:203-206, float64 division inside the kernels)."""
    lib = load()
    sc = None if scale is None else (ctypes.c_double * 3)(*[float(v) for v in scale])
    p, k = points.shape[0], centers.shape[0]
    num_frames = point_frame_ptr.numel() - 1
    row_ptr = torch.empty(k + 1, dtype=torch.int32, device=points.device)
    key = (points.device.index, float(radius), None if scale is None else tuple(float(v) for v in scale))
    cap = max(_edge_capacity.get(key, 0), 64 * k, 1 << 16)
    e = c_i64(0)
    while True:
        buf = torch.empty((2, cap), dtype=torch.int32, device=points.device)
        code = lib.pg_radius_graph_scaled(_ptr(points, torch.float32, 'points'),
                                          _ptr(point_frame_ptr, torch.int32, 'point_frame_ptr'),
                                          _ptr(centers, torch.float32, 'centers'),
                                          _ptr(center_frame_ptr, torch.int32, 'center_frame_ptr'), num_frames, p, k,
                                          float(radius), sc, _ptr(row_ptr, torch.int32, 'row_ptr'),
                                          ctypes.c_void_p(buf[0].data_ptr()), ctypes.c_void_p(buf[1].data_ptr()), cap,
                                          ctypes.byref(e), _stream())
        if code == PG_ERR_CAPACITY:
            cap = int(e.value * 1.25) + 1024
            continue
        _check(code)
        break
    _edge_capacity[key] = max(_edge_capacity.get(key, 0), int(e.value * 1.25) + 1024)
    # rows of buf are src / dst; the [E,2] transpose view of this slice has contiguous columns
    return row_ptr, buf[:, :e.value]


_graph_capacity = {}


def multi_level_graph(xyz, frame_ptr, voxel_size, radius0, radius1):
    """pg_multi_level_graph: keypoints + both radius graphs in one call with one host round trip.
    -> (kp_idx [K] int32, kp_frame_ptr [F+1] int32, kp_xyz [K,3], edges0 [2,E0], edges1 [2,E1])."""
    lib = load()
    n = xyz.shape[0]
    num_frames = frame_ptr.numel() - 1
    dev = xyz.device
    key = (dev.index, int(n), tuple(float(v) for v in voxel_size), float(radius0), float(radius1))
    # buffer sizes: 1.25 x the largest result seen for this problem shape (first call: generous guesses)
    kcap, cap0, cap1 = _graph_capacity.get(key, (min(n, max(4096, n // 4)), 32 * n, 48 * n))
    vs = (ctypes.c_double * 3)(*[float(v) for v in voxel_size])
    sizes = (c_i64 * 3)()
    while True:
        kcap = min(int(kcap), n)
        kp_idx = torch.empty(kcap, dtype=torch.int32, device=dev)
        kp_fp = torch.empty(num_frames + 1, dtype=torch.int32, device=dev)
        kp_xyz = torch.empty((kcap, 3), dtype=torch.float32, device=dev)
        rp0 = torch.empty(kcap + 1, dtype=torch.int32, device=dev)
        rp1 = torch.empty(kcap + 1, dtype=torch.int32, device=dev)
        e0 = torch.empty((2, int(cap0)), dtype=torch.int32, device=dev)
        e1 = torch.empty((2, int(cap1)), dtype=torch.int32, device=dev)
        code = lib.pg_multi_level_graph(
            _ptr(xyz, torch.float32, 'xyz'), _ptr(frame_ptr, torch.int32, 'frame_ptr'), num_frames, n, vs,
            float(radius0), float(radius1), _ptr(kp_idx, torch.int32, 'kp_idx'), kcap,
            _ptr(kp_fp, torch.int32, 'kp_fp'), _ptr(kp_xyz, torch.float32, 'kp_xyz'),
            _ptr(rp0, torch.int32, 'rp0'), ctypes.c_void_p(e0[0].data_ptr()), ctypes.c_void_p(e0[1].data_ptr()), int(cap0),
            _ptr(rp1, torch.int32, 'rp1'), ctypes.c_void_p(e1[0].data_ptr()), ctypes.c_void_p(e1[1].data_ptr()), int(cap1),
            sizes, _stream())
        k, n0, n1 = int(sizes[0]), int(sizes[1]), int(sizes[2])
        if code == PG_ERR_CAPACITY:
            if k > kcap:      # the edge counts were computed on a truncated keypoint set: scale them up too
                cap0, cap1 = max(cap0, int(n0 * 1.3 * k / kcap) + 1024), max(cap1, int(n1 * 1.7 * k / kcap) + 1024)
                kcap = int(k * 1.25) + 64
            elif n0 > cap0 or n1 > cap1:
                cap0, cap1 = max(cap0, int(n0 * 1.25) + 1024), max(cap1, int(n1 * 1.25) + 1024)
            else:             # the internal hit-parking buffer (10 x the edge capacity) overflowed
                cap0, cap1 = 2 * int(cap0), 2 * int(cap1)
            continue
        _check(code)
        break
    old = _graph_capacity.get(key, (0, 0, 0))
    _graph_capacity[key] = (max(old[0], int(k * 1.25) + 64), max(old[1], int(n0 * 1.25) + 1024),
                            max(old[2], int(n1 * 1.25) + 1024))
    return kp_idx[:k], kp_fp, kp_xyz[:k], e0[:, :n0], e1[:, :n1]


def radius_graph_two_pass(points, point_frame_ptr, centers, center_frame_ptr, radius):
    """The count / fill pair of the ABI (caller-allocated exact edge buffer)."""
    lib = load()
    p, k = points.shape[0], centers.shape[0]
    num_frames = point_frame_ptr.numel() - 1
    row_ptr = torch.empty(k + 1, dtype=torch.int32, device=points.device)
    e = c_i64(0)
    args = (_ptr(points, torch.float32, 'points'), _ptr(point_frame_ptr, torch.int32, 'point_frame_ptr'),
            _ptr(centers, torch.float32, 'centers'), _ptr(center_frame_ptr, torch.int32, 'center_frame_ptr'),
            num_frames, p, k, float(radius))
    _check(lib.pg_radius_graph_count(*args, _ptr(row_ptr, torch.int32, 'row_ptr'), ctypes.byref(e), _stream()))
    out = torch.empty((2, e.value), dtype=torch.int32, device=points.device)
    _check(lib.pg_radius_graph_fill(*args, _ptr(row_ptr, torch.int32, 'row_ptr'), e.value,
                                    ctypes.c_void_p(out[0].data_ptr()), ctypes.c_void_p(out[1].data_ptr()),
                                    _stream()))
    return row_ptr, out


# ---------------------------------------------------------------------------------------------
# GNN ops
# ---------------------------------------------------------------------------------------------

def scatter_max(features, centers, num_centers):
    lib = load()
    e, c = features.shape
    out = torch.empty((int(num_centers), c), dtype=torch.float32, device=features.device)
    _check(lib.pg_scatter_max(_ptr(features, torch.float32, 'features'), _ptr(centers, torch.int32, 'centers'), e, c,
                              int(num_centers), _ptr(out, torch.float32, 'out'), _stream()))
    return out


def scatter_sum(features, centers, num_centers, mean=False):
    lib = load()
    e, c = features.shape
    out = torch.empty((int(num_centers), c), dtype=torch.float32, device=features.device)
    fn = lib.pg_scatter_mean if mean else lib.pg_scatter_sum
    _check(fn(_ptr(features, torch.float32, 'features'), _ptr(centers, torch.int32, 'centers'), e, c,
              int(num_centers), _ptr(out, torch.float32, 'out'), _stream()))
    return out


def gather_rows(params, indices):
    lib = load()
    r, c = params.shape
    n = indices.numel()
    out = torch.empty((n, c), dtype=torch.float32, device=params.device)
    _check(lib.pg_gather_rows(_ptr(params, torch.float32, 'params'), r, c, _ptr(indices, torch.int32, 'indices'), n,
                              _ptr(out, torch.float32, 'out'), _stream()))
    return out


def fully_connected(x, w, b, relu, residual=None, precision=0):
    lib = load()
    m, k = x.shape
    if w.shape[0] != k:
        raise ValueError('fully_connected: input width %d != weight rows %d' % (k, w.shape[0]))
    n = w.shape[1]
    if b.numel() != n:
        raise ValueError('fully_connected: bias has %d entries, layer width is %d' % (b.numel(), n))
    if residual is not None and tuple(residual.shape) != (m, n):
        # the reference's tf add raises a shape error here (gnn.py:346, 372)
        raise ValueError('fully_connected: residual shape %s != output shape (%d, %d)' % (tuple(residual.shape), m, n))
    out = torch.empty((m, n), dtype=torch.float32, device=x.device)
    _check(lib.pg_fully_connected(_ptr(x, torch.float32, 'x'), m, k, _ptr(w, torch.float32, 'w'),
                                  _ptr(b, torch.float32, 'b'), n, 1 if relu else 0,
                                  _ptr(residual, torch.float32, 'residual'), _ptr(out, torch.float32, 'out'),
                                  int(precision), _stream()))
    return out


def check_edges(src, dst, num_src, num_dst):
    """Raise PointGNNError unless 0 <= src < num_src and 0 <= dst < num_dst (one synchronising kernel)."""
    lib = load()
    _check(lib.pg_check_edges(_ptr(src, torch.int32, 'src'), _ptr(dst, torch.int32, 'dst'), src.numel(),
                              int(num_src), int(num_dst), _stream()))


def edge_mlp_max(mode, features, xyz_src, xyz_dst, dst_index, src, dst, num_dst, weights, biases, precision=0,
                 trusted=False):
    """trusted=True: the caller vouches for the index ranges (graph_gen output / check_edges passed); the call
    then does not read the range-error flag back and does not synchronise the stream."""
    lib = load()
    num_layers = len(weights)
    dims = [weights[0].shape[0]] + [w.shape[1] for w in weights]
    wp = (ctypes.c_void_p * num_layers)(*[_ptr(w, torch.float32, 'weight').value for w in weights])
    bp = (ctypes.c_void_p * num_layers)(*[_ptr(b, torch.float32, 'bias').value for b in biases])
    dm = (c_i32 * (num_layers + 1))(*dims)
    out = torch.empty((int(num_dst), dims[-1]), dtype=torch.float32, device=features.device)
    _check(lib.pg_edge_mlp_max(int(mode), _ptr(features, torch.float32, 'features'), features.shape[1],
                               _ptr(xyz_src, torch.float32, 'xyz_src'), _ptr(xyz_dst, torch.float32, 'xyz_dst'),
                               _ptr(dst_index, torch.int32, 'dst_index'), _ptr(src, torch.int32, 'src'),
                               _ptr(dst, torch.int32, 'dst'), src.numel(), features.shape[0], int(num_dst), wp, bp,
                               dm, num_layers, _ptr(out, torch.float32, 'out'),
                               int(precision) | (PG_FLAG_TRUSTED_INDICES if trusted else 0), _stream()))
    return out


def softmax_rows(logits):
    lib = load()
    out = torch.empty_like(logits)
    _check(lib.pg_softmax_rows(_ptr(logits, torch.float32, 'logits'), logits.shape[0], logits.shape[1],
                               _ptr(out, torch.float32, 'out'), _stream()))
    return out


# ---------------------------------------------------------------------------------------------
# prepared layers (weights packed once; the calls below launch compute kernels only)
# ---------------------------------------------------------------------------------------------
class PreparedLayer(object):
    """Owner of one ``pg_layer`` handle.  Keeps the weight tensors alive: the C side stores their pointers."""

    def __init__(self, kind, weights, biases, dims, precision=0):
        lib = load()
        n = len(weights)
        self.kind = int(kind)
        self.dims = [int(d) for d in dims]
        self._keep = (list(weights), list(biases))
        wp = (ctypes.c_void_p * n)(*[_ptr(w, torch.float32, 'weight').value for w in weights])
        bp = (ctypes.c_void_p * n)(*[_ptr(b, torch.float32, 'bias').value for b in biases])
        dm = (c_i32 * len(self.dims))(*self.dims)
        handle = ctypes.c_void_p()
        self._handle = None
        _check(lib.pg_layer_create(self.kind, wp, bp, dm, n, int(precision), _stream(), ctypes.byref(handle)))
        self._handle = handle

    def __del__(self):
        if getattr(self, '_handle', None) is not None and _lib is not None:
            _lib.pg_layer_destroy(self._handle)
            self._handle = None

    # multi_layer_neural_network_fn / multi_layer_fc_fn (gnn.py:34-104)
    def mlp(self, x, last_linear, residual=None):
        m, k = x.shape
        if k != self.dims[0]:
            raise ValueError('fully_connected: input width %d != weight rows %d' % (k, self.dims[0]))
        n = self.dims[-1]
        if residual is not None and tuple(residual.shape) != (m, n):
            raise ValueError('fully_connected: residual shape %s != output shape (%d, %d)'
                             % (tuple(residual.shape), m, n))
        out = torch.empty((m, n), dtype=torch.float32, device=x.device)
        _check(load().pg_layer_mlp(self._handle, _ptr(x, torch.float32, 'x'), m, 1 if last_linear else 0,
                                   _ptr(residual, torch.float32, 'residual'), _ptr(out, torch.float32, 'out'),
                                   _stream()))
        return out

    # fused gather -> edge MLP -> segment max (gnn.py:256-277, 338-365)
    def edge_mlp_max(self, features, xyz_src, xyz_dst, dst_index, src, dst, num_dst, trusted=False):
        if features.shape[1] + 3 != self.dims[0]:
            raise ValueError('edge layer: %d feature channels + 3 != first weight rows %d'
                             % (features.shape[1], self.dims[0]))
        out = torch.empty((int(num_dst), self.dims[-1]), dtype=torch.float32, device=features.device)
        _check(load().pg_layer_edge_mlp_max(
            self._handle, _ptr(features, torch.float32, 'features'), _ptr(xyz_src, torch.float32, 'xyz_src'),
            _ptr(xyz_dst, torch.float32, 'xyz_dst'), _ptr(dst_index, torch.int32, 'dst_index'),
            _ptr(src, torch.int32, 'src'), _ptr(dst, torch.int32, 'dst'), src.numel(), features.shape[0],
            int(num_dst), _ptr(out, torch.float32, 'out'), PG_FLAG_TRUSTED_INDICES if trusted else 0, _stream()))
        return out

    # ClassAwarePredictor (gnn.py:133-163) + softmax (models.py:165-168)
    def predictor(self, x):
        d, h, c, box = self.dims
        m = x.shape[0]
        if x.shape[1] != d:
            raise ValueError('predictor: input width %d != %d' % (x.shape[1], d))
        logits = torch.empty((m, c), dtype=torch.float32, device=x.device)
        probs = torch.empty((m, c), dtype=torch.float32, device=x.device)
        boxes = torch.empty((m, c, box), dtype=torch.float32, device=x.device)
        _check(load().pg_layer_predictor(self._handle, _ptr(x, torch.float32, 'x'), m,
                                         _ptr(logits, torch.float32, 'logits'), _ptr(boxes, torch.float32, 'boxes'),
                                         _ptr(probs, torch.float32, 'probs'), _stream()))
        return logits, boxes, probs


# ---------------------------------------------------------------------------------------------
# post-processing (box decoding + NMS)
# ---------------------------------------------------------------------------------------------
PG_NMS_MERGE, PG_NMS_RESCORE, PG_NMS_INT_CORNERS = 1, 2, 4
MAX_CANDIDATES_PER_FRAME = 16384


def _class_table(table):
    flat = [float(v) for row in table for v in row]
    return (ctypes.c_float * len(flat))(*flat)


def decode_boxes(box_encodings, xyz, class_table):
    """[K, C, 7] encodings at the K vertices -> [K, C, 7] boxes (box_encoding.py:265-299)."""
    k, c, _ = box_encodings.shape
    out = torch.empty_like(box_encodings)
    _check(load().pg_decode_boxes(_ptr(box_encodings, torch.float32, 'box_encodings'), _ptr(xyz, torch.float32, 'xyz'),
                                  k, c, _class_table(class_table), _ptr(out, torch.float32, 'out'), _stream()))
    return out


def postprocess(probs, box_encodings, xyz, frame_ptr, class_table, overlapped_thres, merge=True, rescore=True,
                want_candidates=False):
    """run.py:265-325 for a batch of frames on the device.
    -> dict(label [D] int32, box [D,7], score [D], index [D] int32, frame_ptr [F+1] int32
            [, cand_index [B] int32, cand_frame_ptr [F+1] int32])."""
    lib = load()
    k, c = probs.shape
    num_frames = frame_ptr.numel() - 1
    dev = probs.device
    cap = max(1024, k)
    flags = (PG_NMS_MERGE if merge else 0) | (PG_NMS_RESCORE if rescore else 0)
    sizes = (c_i64 * 2)()
    cand_index = torch.empty(k * max(c - 2, 1), dtype=torch.int32, device=dev) if want_candidates else None
    cand_fp = torch.empty(num_frames + 1, dtype=torch.int32, device=dev) if want_candidates else None
    while True:
        label = torch.empty(cap, dtype=torch.int32, device=dev)
        box = torch.empty((cap, 7), dtype=torch.float32, device=dev)
        score = torch.empty(cap, dtype=torch.float32, device=dev)
        index = torch.empty(cap, dtype=torch.int32, device=dev)
        det_fp = torch.empty(num_frames + 1, dtype=torch.int32, device=dev)
        code = lib.pg_postprocess(
            _ptr(probs, torch.float32, 'probs'), _ptr(box_encodings, torch.float32, 'box_encodings'),
            _ptr(xyz, torch.float32, 'xyz'), _ptr(frame_ptr, torch.int32, 'frame_ptr'), num_frames, k, c,
            _class_table(class_table), float(overlapped_thres), flags, MAX_CANDIDATES_PER_FRAME,
            _ptr(label, torch.int32, 'label'), _ptr(box, torch.float32, 'box'), _ptr(score, torch.float32, 'score'),
            _ptr(index, torch.int32, 'index'), cap, _ptr(det_fp, torch.int32, 'det_fp'),
            _ptr(cand_index, torch.int32, 'cand_index'), _ptr(cand_fp, torch.int32, 'cand_fp'), sizes, _stream())
        if code == PG_ERR_CAPACITY and int(sizes[0]) > cap:
            cap = int(sizes[0])
            continue
        _check(code)
        break
    d, b = int(sizes[0]), int(sizes[1])
    out = dict(label=label[:d], box=box[:d], score=score[:d], index=index[:d], frame_ptr=det_fp)
    if want_candidates:
        out['cand_index'] = cand_index[:b]
        out['cand_frame_ptr'] = cand_fp
    return out


def nms_boxes_3d(class_labels, boxes, scores, frame_ptr, overlapped_thres, merge, rescore, appr_factor=0.0,
                 int_corners=False):
    """models/nms.py's entry points on caller-provided boxes.  -> (label, box, score, index, det_frame_ptr)."""
    lib = load()
    n = boxes.shape[0]
    num_frames = frame_ptr.numel() - 1
    dev = boxes.device
    flags = (PG_NMS_MERGE if merge else 0) | (PG_NMS_RESCORE if rescore else 0) | (PG_NMS_INT_CORNERS if int_corners else 0)
    sizes = (c_i64 * 2)()
    label = torch.empty(n, dtype=torch.int32, device=dev)
    box = torch.empty((n, 7), dtype=torch.float32, device=dev)
    score = torch.empty(n, dtype=torch.float32, device=dev)
    index = torch.empty(n, dtype=torch.int32, device=dev)
    det_fp = torch.empty(num_frames + 1, dtype=torch.int32, device=dev)
    _check(lib.pg_nms_boxes_3d(_ptr(class_labels, torch.int32, 'class_labels'), _ptr(boxes, torch.float32, 'boxes'),
                               _ptr(scores, torch.float32, 'scores'), _ptr(frame_ptr, torch.int32, 'frame_ptr'),
                               num_frames, n, float(overlapped_thres), float(appr_factor), flags,
                               MAX_CANDIDATES_PER_FRAME, _ptr(label, torch.int32, 'label'),
                               _ptr(box, torch.float32, 'box'), _ptr(score, torch.float32, 'score'),
                               _ptr(index, torch.int32, 'index'), n, _ptr(det_fp, torch.int32, 'det_fp'), sizes,
                               _stream()))
    d = int(sizes[0])
    return label[:d], box[:d], score[:d], index[:d], det_fp


# ---------------------------------------------------------------------------------------------
# input stage
# ---------------------------------------------------------------------------------------------
def cam_points_in_image(velo, frame_ptr, velo_to_cam, cam_to_image, image_sizes, images=None, image_offsets=None):
    """pg_cam_points_in_image.  velo [M,4] CUDA fp32, frame_ptr [F+1] CUDA int32, velo_to_cam [F,4,4] / cam_to_image
    [F,3,4] / image_sizes [F,2] host arrays; images: optional CUDA uint8 buffer (+ byte offsets per frame).
    -> (xyz [N,3], attr [N,1 or 4], out_frame_ptr [F+1])."""
    import numpy as np
    lib = load()
    m = velo.shape[0]
    num_frames = frame_ptr.numel() - 1
    vtc = np.ascontiguousarray(velo_to_cam, dtype=np.float32).reshape(num_frames, 16)
    cti = np.ascontiguousarray(cam_to_image, dtype=np.float64).reshape(num_frames, 12)
    wh = np.ascontiguousarray(image_sizes, dtype=np.int32).reshape(num_frames, 2)
    channels = 4 if images is not None else 1
    out_xyz = torch.empty((m, 3), dtype=torch.float32, device=velo.device)
    out_attr = torch.empty((m, channels), dtype=torch.float32, device=velo.device)
    out_fp = torch.empty(num_frames + 1, dtype=torch.int32, device=velo.device)
    n = c_i64(0)
    offs = None
    if images is not None:
        offs = np.ascontiguousarray(image_offsets, dtype=np.int64)
        if images.dtype != torch.uint8 or not images.is_cuda:
            raise TypeError('images must be a CUDA uint8 tensor')
    _check(lib.pg_cam_points_in_image(
        _ptr(velo, torch.float32, 'velo'), _ptr(frame_ptr, torch.int32, 'frame_ptr'), num_frames, m,
        vtc.ctypes.data_as(ctypes.POINTER(ctypes.c_float)), cti.ctypes.data_as(ctypes.POINTER(ctypes.c_double)),
        wh.ctypes.data_as(ctypes.POINTER(c_i32)), None if images is None else ctypes.c_void_p(images.data_ptr()),
        None if offs is None else offs.ctypes.data_as(ctypes.POINTER(c_i64)), _ptr(out_xyz, torch.float32, 'out_xyz'),
        _ptr(out_attr, torch.float32, 'out_attr'), channels, m, _ptr(out_fp, torch.int32, 'out_fp'), ctypes.byref(n),
        _stream()))
    return out_xyz[:n.value], out_attr[:n.value], out_fp
