// Graph construction on the GPU: voxel keypoint selection and radius-neighbour CSR graphs.
//
// Replaces /root/reference/models/graph_gen.py:
//   multi_layer_downsampling (:11-47, open3d.voxel_down_sample branch :41-45)
//   multi_layer_downsampling_select (:49-90, kd-tree 1-NN snap :84-88)
//   gen_disjointed_rnn_local_graph_v3 (:197-220, ball-tree radius query)
//
// Design: every spatial query runs on a sorted-key uniform grid.  A point's 64-bit key is
//   frame(16) | iz(16) | iy(16) | ix(16)
// so one radix sort groups points by (frame, cell) and, because ix is the low field, the three
// x-adjacent cells of a (frame, iz, iy) row are one contiguous range of the sorted array: a
// 3x3x3 neighbourhood costs 9 binary searches.  There is no dense grid, so memory is O(N)
// whatever the extent of the cloud.  All predicates that decide membership (voxel index,
// nearest point, radius test) are evaluated in fp64 with explicitly rounded mul/add
// (no FMA contraction), which is what makes the edge lists bit-exact against the reference's
// scikit-learn float64 trees.
#include <cub/cub.cuh>

#include "pg_common.cuh"

namespace pg {
namespace {

constexpr int kAxisBits = 16;
constexpr int kAxisMax = (1 << kAxisBits) - 1;
constexpr double kCellSlack = 1.0001;  // cell edge = radius * slack, keeps +-1 cell search exact
// device-side error word of one graph call (read back once, together with the result size)
constexpr int kErrRange = 1;       // cloud extent exceeds the key bits
constexpr int kErrFramePtr = 2;    // point frame_ptr does not run from 0 to N
constexpr int kErrCenterPtr = 4;   // centre frame_ptr does not run from 0 to K
constexpr int kErrParking = 8;     // pg_multi_level_graph: hit parking buffer too small (retry with larger edge capacity)

__host__ __device__ inline uint64_t make_key(uint32_t frame, uint32_t iz, uint32_t iy, uint32_t ix) {
  return (uint64_t(frame) << 48) | (uint64_t(iz) << 32) | (uint64_t(iy) << 16) | uint64_t(ix);
}

// float <-> order-preserving uint (for atomicMin on floats)
__device__ inline uint32_t float_to_ordered(float f) {
  uint32_t b = __float_as_uint(f);
  return (b & 0x80000000u) ? ~b : (b | 0x80000000u);
}
__device__ inline float ordered_to_float(uint32_t u) {
  uint32_t b = (u & 0x80000000u) ? (u & 0x7fffffffu) : ~u;
  return __uint_as_float(b);
}

__device__ inline int find_frame(const int32_t* __restrict__ frame_ptr, int num_frames, int64_t row) {
  int lo = 0, hi = num_frames;  // invariant: frame_ptr[lo] <= row < frame_ptr[hi]
  while (hi - lo > 1) {
    int mid = (lo + hi) >> 1;
    if (frame_ptr[mid] <= row) lo = mid; else hi = mid;
  }
  return lo;
}

// ---- per-frame bounding-box minimum ---------------------------------------------------------
__global__ void init_bounds_kernel(uint32_t* __restrict__ bounds, int n) {
  int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i < n) bounds[i] = 0xffffffffu;
}

__global__ void frame_min_kernel(const float* __restrict__ xyz, const int32_t* __restrict__ frame_ptr, int64_t n,
                                 uint32_t* __restrict__ bounds) {
  const int f = blockIdx.y;
  // clamped: a malformed partition is reported through the error word, it must not read out of bounds
  const int64_t begin = max(int64_t(frame_ptr[f]), int64_t(0)), end = min(int64_t(frame_ptr[f + 1]), n);
  float mx = FLT_MAX, my = FLT_MAX, mz = FLT_MAX;
  for (int64_t i = begin + blockIdx.x * blockDim.x + threadIdx.x; i < end;
       i += int64_t(gridDim.x) * blockDim.x) {
    mx = fminf(mx, xyz[3 * i + 0]);
    my = fminf(my, xyz[3 * i + 1]);
    mz = fminf(mz, xyz[3 * i + 2]);
  }
  for (int o = 16; o > 0; o >>= 1) {
    mx = fminf(mx, __shfl_xor_sync(0xffffffffu, mx, o));
    my = fminf(my, __shfl_xor_sync(0xffffffffu, my, o));
    mz = fminf(mz, __shfl_xor_sync(0xffffffffu, mz, o));
  }
  if ((threadIdx.x & 31) == 0 && begin < end) {
    atomicMin(&bounds[3 * f + 0], float_to_ordered(mx));
    atomicMin(&bounds[3 * f + 1], float_to_ordered(my));
    atomicMin(&bounds[3 * f + 2], float_to_ordered(mz));
  }
}

// Grid description shared by key generation and queries.
struct GridSpec {
  double cell[3];     // cell edge per axis
  double origin_off;  // origin = frame_min - cell * origin_off   (0.5 for Open3D voxels, 0 for radius grids)
  // gen_disjointed_rnn_local_graph_v3's `scale` (graph_gen.py:203-206): every coordinate is DIVIDED by scale[axis] in
  // float64 before anything else (points_xyz / np.array(scale) -> float64).  scaled == 0: coordinates as they are.
  int scaled;
  double scale[3];
  // multi_layer_downsampling with add_rnd3d (graph_gen.py:24-31): cell = floor_divide((p - frame_min)[float32] +
  // cell * shift[frame], cell) in float64, shift = the np.random.random((1, 3)) draw of the frame.  shift == nullptr:
  // the rule of cell_of below.
  const double* shift;
};

// coordinate of axis a as the reference sees it: float32 value -> float64, divided by the scale if there is one
__device__ __forceinline__ double coord(const GridSpec& g, float v, int a) {
  return g.scaled ? __ddiv_rn(double(v), g.scale[a]) : double(v);
}

__device__ inline void cell_of(const GridSpec& g, const uint32_t* __restrict__ bounds, int f, float x,
                               float y, float z, long long* ix, long long* iy, long long* iz) {
  const double ox = __dsub_rn(coord(g, ordered_to_float(bounds[3 * f + 0]), 0), __dmul_rn(g.cell[0], g.origin_off));
  const double oy = __dsub_rn(coord(g, ordered_to_float(bounds[3 * f + 1]), 1), __dmul_rn(g.cell[1], g.origin_off));
  const double oz = __dsub_rn(coord(g, ordered_to_float(bounds[3 * f + 2]), 2), __dmul_rn(g.cell[2], g.origin_off));
  *ix = (long long)floor(__ddiv_rn(__dsub_rn(coord(g, x, 0), ox), g.cell[0]));
  *iy = (long long)floor(__ddiv_rn(__dsub_rn(coord(g, y, 1), oy), g.cell[1]));
  *iz = (long long)floor(__ddiv_rn(__dsub_rn(coord(g, z, 2), oz), g.cell[2]));
}

// graph_gen.py:24-31 (defined next to the random keypoint path further down)
__device__ void shifted_cell_of(const GridSpec& g, const uint32_t* __restrict__ bounds, int f, float x, float y, float z,
                                long long* ix, long long* iy, long long* iz);

// `n_valid` (optional, device): only rows [0, *n_valid) of the n-row buffer hold points (a point set whose size is
// still on the device, e.g. the keypoints of the same call); the others get the key of frame `num_frames`, which
// sorts behind every real cell and is never looked up.
__global__ void point_keys_kernel(const float* __restrict__ xyz, const int32_t* __restrict__ frame_ptr,
                                  int num_frames, int64_t n, const int32_t* __restrict__ n_valid, GridSpec g,
                                  const uint32_t* __restrict__ bounds, uint64_t* __restrict__ keys,
                                  int32_t* __restrict__ vals, int* __restrict__ range_error) {
  int64_t i = int64_t(blockIdx.x) * blockDim.x + threadIdx.x;
  if (i >= n) return;
  const int64_t nv = n_valid ? int64_t(*n_valid) : n;
  // the caller's frame partition must run from 0 to n (checked here instead of with a host round trip)
  if (i == 0 && (frame_ptr[0] != 0 || int64_t(frame_ptr[num_frames]) != nv)) atomicOr(range_error, kErrFramePtr);
  if (i >= nv) {
    keys[i] = make_key(uint32_t(num_frames), 0, 0, 0);
    vals[i] = int32_t(i);
    return;
  }
  const int f = find_frame(frame_ptr, num_frames, i);
  long long ix, iy, iz;
  if (g.shift != nullptr) shifted_cell_of(g, bounds, f, xyz[3 * i], xyz[3 * i + 1], xyz[3 * i + 2], &ix, &iy, &iz);
  else cell_of(g, bounds, f, xyz[3 * i], xyz[3 * i + 1], xyz[3 * i + 2], &ix, &iy, &iz);
  if (ix < 0 || iy < 0 || iz < 0 || ix > kAxisMax || iy > kAxisMax || iz > kAxisMax) {
    atomicOr(range_error, kErrRange);
    ix = iy = iz = 0;
  }
  keys[i] = make_key(uint32_t(f), uint32_t(iz), uint32_t(iy), uint32_t(ix));
  vals[i] = int32_t(i);
}

// sorted point record (coalesced candidate reads) + head flag of each run of equal keys
__global__ void gather_sorted_kernel(const float* __restrict__ xyz, const uint64_t* __restrict__ keys,
                                     const int32_t* __restrict__ order, int64_t n,
                                     float4* __restrict__ sorted_pts, int32_t* __restrict__ head) {
  int64_t i = int64_t(blockIdx.x) * blockDim.x + threadIdx.x;
  if (i >= n) return;
  const int32_t j = order[i];
  sorted_pts[i] = make_float4(xyz[3 * j], xyz[3 * j + 1], xyz[3 * j + 2], __int_as_float(j));
  head[i] = (i == 0 || keys[i] != keys[i - 1]) ? 1 : 0;
}

// cell table: cell_key[c], cell_start[c] for every non-empty cell c (ascending key)
__global__ void cell_table_kernel(const uint64_t* __restrict__ keys, const int32_t* __restrict__ head_scan,
                                  int64_t n, uint64_t* __restrict__ cell_key,
                                  int32_t* __restrict__ cell_start) {
  int64_t i = int64_t(blockIdx.x) * blockDim.x + threadIdx.x;
  if (i >= n) return;
  const int32_t c = head_scan[i] - 1;  // inclusive scan of head flags
  const bool is_head = (i == 0) || (head_scan[i] != head_scan[i - 1]);
  if (is_head) {
    cell_key[c] = keys[i];
    cell_start[c] = int32_t(i);
  }
  if (i == n - 1) cell_start[c + 1] = int32_t(n);
}

__device__ inline int lower_bound_u64(const uint64_t* __restrict__ a, int n, uint64_t v) {
  int lo = 0, hi = n;
  while (lo < hi) {
    int mid = (lo + hi) >> 1;
    if (a[mid] < v) lo = mid + 1; else hi = mid;
  }
  return lo;
}

struct SortedGrid {
  const uint64_t* cell_key;   // [num_cells]
  const int32_t* cell_start;  // [num_cells+1]
  const float4* pts;          // [n] sorted (x,y,z,orig idx)
  const int32_t* num_cells;   // device scalar (= last element of the head-flag scan): no host round trip
};

// point range covering cells (f, iz, iy, ix_lo..ix_hi); indices already clamped to [0, kAxisMax]
__device__ inline void row_range(const SortedGrid& g, uint32_t f, uint32_t iz, uint32_t iy, uint32_t ix_lo,
                                 uint32_t ix_hi, int* begin, int* end) {
  const int nc = __ldg(g.num_cells);
  const int a = lower_bound_u64(g.cell_key, nc, make_key(f, iz, iy, ix_lo));
  const int b = lower_bound_u64(g.cell_key, nc, make_key(f, iz, iy, ix_hi) + 1ull);
  *begin = g.cell_start[a];
  *end = g.cell_start[b];
}

__device__ inline double dist2_rn(double ax, double ay, double az, float bx, float by, float bz) {
  const double dx = __dsub_rn(ax, double(bx));
  const double dy = __dsub_rn(ay, double(by));
  const double dz = __dsub_rn(az, double(bz));
  return __dadd_rn(__dadd_rn(__dmul_rn(dx, dx), __dmul_rn(dy, dy)), __dmul_rn(dz, dz));
}

// ---- voxel keypoints: centroid (fp64, ascending point order) + exact nearest original point ----
__global__ void voxel_keypoint_kernel(SortedGrid g, GridSpec spec, const uint32_t* __restrict__ bounds,
                                      int32_t* __restrict__ out_idx, int64_t capacity) {
  const int v = blockIdx.x * blockDim.x + threadIdx.x;
  if (v >= __ldg(g.num_cells)) return;
  const int s = g.cell_start[v], e = g.cell_start[v + 1];
  double sx = 0.0, sy = 0.0, sz = 0.0;
  for (int i = s; i < e; ++i) {  // sorted by (key, original index): ascending point order
    const float4 p = g.pts[i];
    sx = __dadd_rn(sx, double(p.x));
    sy = __dadd_rn(sy, double(p.y));
    sz = __dadd_rn(sz, double(p.z));
  }
  const double cnt = double(e - s);
  const double cx = __ddiv_rn(sx, cnt), cy = __ddiv_rn(sy, cnt), cz = __ddiv_rn(sz, cnt);
  // best candidate inside the own voxel
  double best = DBL_MAX;
  int best_idx = 0x7fffffff;
  for (int i = s; i < e; ++i) {
    const float4 p = g.pts[i];
    const double d = dist2_rn(cx, cy, cz, p.x, p.y, p.z);
    const int idx = __float_as_int(p.w);
    if (d < best || (d == best && idx < best_idx)) { best = d; best_idx = idx; }
  }
  // every point closer than sqrt(best) lies in a cell overlapping the box centroid +- reach
  const uint64_t key = g.cell_key[v];
  const uint32_t f = uint32_t(key >> 48);
  const double reach = sqrt(best) * (1.0 + 1e-9) + 1e-12;
  const double ox = double(ordered_to_float(bounds[3 * f + 0])) - spec.cell[0] * spec.origin_off;
  const double oy = double(ordered_to_float(bounds[3 * f + 1])) - spec.cell[1] * spec.origin_off;
  const double oz = double(ordered_to_float(bounds[3 * f + 2])) - spec.cell[2] * spec.origin_off;
  // reach is inflated by 1e-9 relative, far above the fp64 rounding of the corner cells
  long long x0 = (long long)floor((cx - reach - ox) / spec.cell[0]), x1 = (long long)floor((cx + reach - ox) / spec.cell[0]);
  long long y0 = (long long)floor((cy - reach - oy) / spec.cell[1]), y1 = (long long)floor((cy + reach - oy) / spec.cell[1]);
  long long z0 = (long long)floor((cz - reach - oz) / spec.cell[2]), z1 = (long long)floor((cz + reach - oz) / spec.cell[2]);
  x0 = max(x0, 0ll); y0 = max(y0, 0ll); z0 = max(z0, 0ll);
  x1 = min(x1, (long long)kAxisMax); y1 = min(y1, (long long)kAxisMax); z1 = min(z1, (long long)kAxisMax);
  for (long long iz = z0; iz <= z1; ++iz) {
    for (long long iy = y0; iy <= y1; ++iy) {
      int b, en;
      row_range(g, f, uint32_t(iz), uint32_t(iy), uint32_t(x0), uint32_t(x1), &b, &en);
      for (int i = b; i < en; ++i) {
        const float4 p = g.pts[i];
        const double d = dist2_rn(cx, cy, cz, p.x, p.y, p.z);
        const int idx = __float_as_int(p.w);
        if (d < best || (d == best && idx < best_idx)) { best = d; best_idx = idx; }
      }
    }
  }
  if (v < capacity) out_idx[v] = best_idx;
}

// ---- general multi-scale keypoints (graph_gen.py:11-47 + :49-90 with more than one distinct scale) -------------
// multi_layer_downsampling voxelises the ORIGINAL cloud at every scale; multi_layer_downsampling_select then snaps
// each centroid to the nearest vertex of the PREVIOUS level (kd_tree 1-NN on base_points).  Two kernels: the fp64
// centroid of every occupied voxel, and an exact nearest-point query against a second grid built over the base
// points.
__global__ void voxel_centroid_kernel(SortedGrid g, double* __restrict__ out_centroid, int32_t* __restrict__ out_frame,
                                      int64_t capacity) {
  const int v = blockIdx.x * blockDim.x + threadIdx.x;
  if (v >= __ldg(g.num_cells) || v >= capacity) return;
  const int s = g.cell_start[v], e = g.cell_start[v + 1];
  double sx = 0.0, sy = 0.0, sz = 0.0;
  for (int i = s; i < e; ++i) {  // ascending point order (stable sort)
    const float4 p = g.pts[i];
    sx = __dadd_rn(sx, double(p.x));
    sy = __dadd_rn(sy, double(p.y));
    sz = __dadd_rn(sz, double(p.z));
  }
  const double cnt = double(e - s);
  out_centroid[3 * int64_t(v) + 0] = __ddiv_rn(sx, cnt);
  out_centroid[3 * int64_t(v) + 1] = __ddiv_rn(sy, cnt);
  out_centroid[3 * int64_t(v) + 2] = __ddiv_rn(sz, cnt);
  if (out_frame) out_frame[v] = int32_t(g.cell_key[v] >> 48);
}

// nearest base point (fp64 squared distance, ties -> lowest index) of query q inside its own frame.
// Growing boxes of cells until one holds a point, then ONE exact pass over every cell the ball of that radius touches.
__global__ void nearest_point_kernel(SortedGrid g, GridSpec spec, const uint32_t* __restrict__ bounds,
                                     const int32_t* __restrict__ base_frame_ptr, const double* __restrict__ q_xyz,
                                     const int32_t* __restrict__ q_frame, const int32_t* __restrict__ num_q,
                                     int64_t capacity, int32_t* __restrict__ out_idx, int* __restrict__ err) {
  const int64_t q = int64_t(blockIdx.x) * blockDim.x + threadIdx.x;
  if (q >= int64_t(__ldg(num_q)) || q >= capacity) return;
  const uint32_t f = uint32_t(q_frame[q]);
  if (base_frame_ptr[f + 1] == base_frame_ptr[f]) {   // a frame with voxels but no base vertex
    atomicOr(err, kErrCenterPtr);
    out_idx[q] = 0;
    return;
  }
  const double cx = q_xyz[3 * q], cy = q_xyz[3 * q + 1], cz = q_xyz[3 * q + 2];
  const double ox = double(ordered_to_float(bounds[3 * f + 0])) - spec.cell[0] * spec.origin_off;
  const double oy = double(ordered_to_float(bounds[3 * f + 1])) - spec.cell[1] * spec.origin_off;
  const double oz = double(ordered_to_float(bounds[3 * f + 2])) - spec.cell[2] * spec.origin_off;
  double best = DBL_MAX;
  int best_idx = 0x7fffffff;
  auto scan = [&](long long x0, long long x1, long long y0, long long y1, long long z0, long long z1) {
    x0 = max(x0, 0ll); y0 = max(y0, 0ll); z0 = max(z0, 0ll);
    x1 = min(x1, (long long)kAxisMax); y1 = min(y1, (long long)kAxisMax); z1 = min(z1, (long long)kAxisMax);
    if (x0 > x1) return;
    for (long long iz = z0; iz <= z1; ++iz)
      for (long long iy = y0; iy <= y1; ++iy) {
        int b, en;
        row_range(g, f, uint32_t(iz), uint32_t(iy), uint32_t(x0), uint32_t(x1), &b, &en);
        for (int i = b; i < en; ++i) {
          const float4 p = g.pts[i];
          const double d = dist2_rn(cx, cy, cz, p.x, p.y, p.z);
          const int idx = __float_as_int(p.w);
          if (d < best || (d == best && idx < best_idx)) { best = d; best_idx = idx; }
        }
      }
  };
  const long long ix = (long long)floor((cx - ox) / spec.cell[0]);
  const long long iy = (long long)floor((cy - oy) / spec.cell[1]);
  const long long iz = (long long)floor((cz - oz) / spec.cell[2]);
  // the frame is not empty, so a box that covers the whole key space terminates the loop
  for (long long r = 1; best == DBL_MAX; r *= 2) {
    scan(ix - r, ix + r, iy - r, iy + r, iz - r, iz + r);
    if (r > 4ll * (kAxisMax + 1) + llabs(ix) + llabs(iy) + llabs(iz)) break;
  }
  if (best == DBL_MAX) {
    atomicOr(err, kErrRange);
    out_idx[q] = 0;
    return;
  }
  // every point closer than sqrt(best) lies in a cell overlapping the box centroid +- reach
  const double reach = sqrt(best) * (1.0 + 1e-9) + 1e-12;
  scan((long long)floor((cx - reach - ox) / spec.cell[0]), (long long)floor((cx + reach - ox) / spec.cell[0]),
       (long long)floor((cy - reach - oy) / spec.cell[1]), (long long)floor((cy + reach - oy) / spec.cell[1]),
       (long long)floor((cz - reach - oz) / spec.cell[2]), (long long)floor((cz + reach - oz) / spec.cell[2]));
  out_idx[q] = best_idx;
}

__global__ void frame_ranges_kernel(const uint64_t* __restrict__ cell_key, const int32_t* __restrict__ num_cells,
                                    int num_frames, int32_t* __restrict__ out_frame_ptr) {
  const int f = blockIdx.x * blockDim.x + threadIdx.x;
  if (f > num_frames) return;
  out_frame_ptr[f] = lower_bound_u64(cell_key, __ldg(num_cells), uint64_t(f) << 48);
}

// ---- radius graph ----------------------------------------------------------------------------
struct CenterCell {
  uint32_t f;
  long long ix, iy, iz;
};

// One warp per centre.  kFill=false: count neighbours.  kFill=true: write source indices at
// row_ptr[c] + rank (rank from a warp ballot prefix, traversal order; rows are sorted afterwards).
template <bool kFill>
__global__ void __launch_bounds__(256) radius_query_kernel(
    SortedGrid g, GridSpec spec, const uint32_t* __restrict__ bounds, const float* __restrict__ centers,
    const int32_t* __restrict__ center_frame_ptr, int num_frames, int64_t num_centers_cap,
    const int32_t* __restrict__ num_centers_dev, double r2, int32_t* __restrict__ counts,
    const int32_t* __restrict__ row_ptr, int32_t* __restrict__ out_src, int64_t capacity, int* __restrict__ err,
    unsigned long long* __restrict__ total64) {
  const int lane = threadIdx.x & 31;
  const int64_t c = (int64_t(blockIdx.x) * blockDim.x + threadIdx.x) >> 5;
  // the number of centres may still be on the device (keypoints of the same call): launch for the capacity
  const int64_t num_centers = num_centers_dev ? int64_t(*num_centers_dev) : num_centers_cap;
  if (c >= num_centers || c >= num_centers_cap) return;
  if (kFill && int64_t(row_ptr[min(num_centers, num_centers_cap)]) > capacity) return;   // edge buffer too small: reported by the host
  if (!kFill && c == 0 && lane == 0 &&
      (center_frame_ptr[0] != 0 || int64_t(center_frame_ptr[num_frames]) != num_centers))
    atomicOr(err, kErrCenterPtr);
  const int f = find_frame(center_frame_ptr, num_frames, c);
  const float cxf = centers[3 * c], cyf = centers[3 * c + 1], czf = centers[3 * c + 2];
  const double cx = coord(spec, cxf, 0), cy = coord(spec, cyf, 1), cz = coord(spec, czf, 2);
  long long ix, iy, iz;
  cell_of(spec, bounds, f, cxf, cyf, czf, &ix, &iy, &iz);
  const long long x0 = max(ix - 1, 0ll), x1 = min(ix + 1, (long long)kAxisMax);
  int total = 0;
  int base = kFill ? row_ptr[c] : 0;
  if (x0 <= x1) {
    for (long long zz = iz - 1; zz <= iz + 1; ++zz) {
      if (zz < 0 || zz > kAxisMax) continue;
      for (long long yy = iy - 1; yy <= iy + 1; ++yy) {
        if (yy < 0 || yy > kAxisMax) continue;
        int b, e;
        row_range(g, uint32_t(f), uint32_t(zz), uint32_t(yy), uint32_t(x0), uint32_t(x1), &b, &e);
        for (int i0 = b; i0 < e; i0 += 32) {
          const int i = i0 + lane;
          bool hit = false;
          int idx = 0;
          if (i < e) {
            const float4 p = g.pts[i];
            if (spec.scaled) {
              const double dx = __dsub_rn(cx, coord(spec, p.x, 0)), dy = __dsub_rn(cy, coord(spec, p.y, 1));
              const double dz = __dsub_rn(cz, coord(spec, p.z, 2));
              hit = __dadd_rn(__dadd_rn(__dmul_rn(dx, dx), __dmul_rn(dy, dy)), __dmul_rn(dz, dz)) <= r2;
            } else {
              hit = dist2_rn(cx, cy, cz, p.x, p.y, p.z) <= r2;
            }
            idx = __float_as_int(p.w);
          }
          const uint32_t m = __ballot_sync(0xffffffffu, hit);
          if (kFill && hit) out_src[base + total + __popc(m & ((1u << lane) - 1u))] = idx;
          total += __popc(m);
        }
      }
    }
  }
  if (!kFill && lane == 0) {
    counts[c] = total;
    atomicAdd(total64, (unsigned long long)total);   // 64-bit edge total: the int32 row_ptr scan may wrap
  }
}

// ---- single-traversal variant (pg_multi_level_graph) -------------------------------------------------------------
// Pass A, one THREAD per centre: the nine sorted-point ranges of its 3 x 3 x 3 cell neighbourhood (18 ints) and
// their total length = an upper bound of the row length.  No point is touched.
__global__ void radius_candidates_kernel(SortedGrid g, GridSpec spec, const uint32_t* __restrict__ bounds,
                                         const float* __restrict__ centers, const int32_t* __restrict__ center_frame_ptr,
                                         int num_frames, int64_t num_centers_cap, const int32_t* __restrict__ num_centers_dev,
                                         int32_t* __restrict__ ranges, int32_t* __restrict__ cand, int* __restrict__ err) {
  const int64_t c = int64_t(blockIdx.x) * blockDim.x + threadIdx.x;
  if (c > num_centers_cap) return;
  const int64_t num_centers = min(int64_t(*num_centers_dev), num_centers_cap);
  if (c >= num_centers) {
    cand[c] = 0;
    return;
  }
  if (c == 0 && (center_frame_ptr[0] != 0 || int64_t(center_frame_ptr[num_frames]) != int64_t(*num_centers_dev)))
    atomicOr(err, kErrCenterPtr);
  const int f = find_frame(center_frame_ptr, num_frames, c);
  long long ix, iy, iz;
  cell_of(spec, bounds, f, centers[3 * c], centers[3 * c + 1], centers[3 * c + 2], &ix, &iy, &iz);
  const long long x0 = max(ix - 1, 0ll), x1 = min(ix + 1, (long long)kAxisMax);
  int total = 0, k = 0;
  for (long long zz = iz - 1; zz <= iz + 1; ++zz) {
    for (long long yy = iy - 1; yy <= iy + 1; ++yy, ++k) {
      int b = 0, e = 0;
      if (x0 <= x1 && zz >= 0 && zz <= kAxisMax && yy >= 0 && yy <= kAxisMax)
        row_range(g, uint32_t(f), uint32_t(zz), uint32_t(yy), uint32_t(x0), uint32_t(x1), &b, &e);
      ranges[c * 18 + 2 * k] = b;
      ranges[c * 18 + 2 * k + 1] = e;
      total += e - b;
    }
  }
  cand[c] = total;
}

// Pass B, one WARP per centre: the only traversal of the points.  Hits are parked, compacted in traversal order, at
// tmp[cand_off[c] ...] (cand_off = exclusive scan of the candidate counts, so the slots never overlap); counts[c]
// = row length.  The row sort then reads the parked hits and writes the final CSR row.
__global__ void __launch_bounds__(256) radius_collect_kernel(SortedGrid g, const float* __restrict__ centers,
                                                             int64_t num_centers_cap,
                                                             const int32_t* __restrict__ num_centers_dev, double r2,
                                                             const int32_t* __restrict__ ranges,
                                                             const int32_t* __restrict__ cand_off, int64_t tmp_capacity,
                                                             int32_t* __restrict__ tmp, int32_t* __restrict__ counts,
                                                             unsigned long long* __restrict__ total64, int* __restrict__ err) {
  const int lane = threadIdx.x & 31;
  const int64_t c = (int64_t(blockIdx.x) * blockDim.x + threadIdx.x) >> 5;
  const int64_t num_centers = min(int64_t(*num_centers_dev), num_centers_cap);
  if (c >= num_centers) return;
  if (int64_t(cand_off[num_centers_cap]) > tmp_capacity) {     // the parking buffer is too small: reported by the host
    if (c == 0 && lane == 0) atomicOr(err, kErrParking);
    return;
  }
  const double cx = double(centers[3 * c]), cy = double(centers[3 * c + 1]), cz = double(centers[3 * c + 2]);
  const int base = cand_off[c];
  int total = 0;
  int rb = 0, re = 0;
  if (lane < 18) rb = ranges[c * 18 + lane];
  for (int k = 0; k < 9; ++k) {
    const int b = __shfl_sync(0xffffffffu, rb, 2 * k), e = __shfl_sync(0xffffffffu, rb, 2 * k + 1);
    (void)re;
    for (int i0 = b; i0 < e; i0 += 32) {
      const int i = i0 + lane;
      bool hit = false;
      int idx = 0;
      if (i < e) {
        const float4 p = g.pts[i];
        hit = dist2_rn(cx, cy, cz, p.x, p.y, p.z) <= r2;
        idx = __float_as_int(p.w);
      }
      const uint32_t m = __ballot_sync(0xffffffffu, hit);
      if (hit) tmp[base + total + __popc(m & ((1u << lane) - 1u))] = idx;
      total += __popc(m);
    }
  }
  if (lane == 0) {
    counts[c] = total;
    atomicAdd(total64, (unsigned long long)total);
  }
}

// Sort every CSR row ascending (canonical order) and expand the destination index.
// Bitonic network in its "all comparators ascending" form (flip stage i^(k-1), then half-cleaners
// i^j): with every comparator ascending, virtual +inf padding at the tail never moves, so rows of
// any length sort in place.
constexpr int kRowSortMax = 8192;
constexpr int kWarpRowMax = 1024;   // rows up to this length are sorted by one warp (sort_rows_warp_kernel)

// One warp per CSR row: classic bitonic network in the warp's private slice of shared memory, padded with
// INT_MAX to a power of two, __syncwarp between stages (no block barrier: KITTI-shape rows have ~100-600
// entries, and the block-per-row version spent its time in 36+ __syncthreads per row).  Also expands dst.
// `in` / `in_off` (optional): the unsorted hits of row r sit at in[in_off[r] ...] (radius_collect_kernel) instead of
// in src[row_ptr[r] ...]; the sorted row is always written to src.
__global__ void __launch_bounds__(256) sort_rows_warp_kernel(const int32_t* __restrict__ row_ptr, int64_t num_rows,
                                                              int32_t* __restrict__ src, int32_t* __restrict__ dst,
                                                              int* __restrict__ has_long_rows, int64_t capacity,
                                                              const int32_t* __restrict__ in = nullptr,
                                                              const int32_t* __restrict__ in_off = nullptr) {
  __shared__ int32_t srows[8][kWarpRowMax];
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  if (int64_t(row_ptr[num_rows]) > capacity) return;      // the edge buffer was too small: nothing was filled
  int32_t* a = srows[warp];
  for (int64_t r = int64_t(blockIdx.x) * 8 + warp; r < num_rows; r += int64_t(gridDim.x) * 8) {
    const int b = row_ptr[r], e = row_ptr[r + 1];
    const int len = e - b;
    if (dst != nullptr)
      for (int i = lane; i < len; i += 32) dst[b + i] = int32_t(r);
    if (len > kWarpRowMax && lane == 0) *has_long_rows = 1;   // tells sort_rows_kernel there is work for it
    if (len > kWarpRowMax) continue;                  // long rows: sort_rows_kernel
    const int32_t* rin = in ? in + in_off[r] : src + b;
    if (len <= 1) {
      if (in && len == 1 && lane == 0) src[b] = rin[0];
      continue;
    }
    int n = 2;
    while (n < len) n <<= 1;
    __syncwarp();
    for (int i = lane; i < n; i += 32) a[i] = i < len ? rin[i] : 0x7fffffff;
    __syncwarp();
    for (int k = 2; k <= n; k <<= 1) {
      for (int j = k >> 1; j > 0; j >>= 1) {
        for (int t = lane; t < (n >> 1); t += 32) {
          const int i = 2 * t - (t & (j - 1));          // lower index of the pair (bit j clear)
          const int x = a[i], y = a[i + j];
          const bool up = (i & k) == 0;                 // ascending block of the bitonic merge
          if ((x > y) == up) { a[i] = y; a[i + j] = x; }
        }
        __syncwarp();
      }
    }
    for (int i = lane; i < len; i += 32) src[b + i] = a[i];
  }
}

__global__ void __launch_bounds__(256) sort_rows_kernel(const int32_t* __restrict__ row_ptr, int64_t num_rows,
                                                         int32_t* __restrict__ src, int32_t* __restrict__ dst,
                                                         const int* __restrict__ has_long_rows, int64_t capacity,
                                                         const int32_t* __restrict__ in = nullptr,
                                                         const int32_t* __restrict__ in_off = nullptr) {
  extern __shared__ int32_t srow[];
  if (*has_long_rows == 0 || int64_t(row_ptr[num_rows]) > capacity) return;                      // the usual case: every row was sorted by a warp
  for (int64_t r = blockIdx.x; r < num_rows; r += gridDim.x) {
    const int b = row_ptr[r], e = row_ptr[r + 1];
    const int len = e - b;
    if (len <= kWarpRowMax) continue;                   // sorted (and dst expanded) by sort_rows_warp_kernel

    int n = 1;
    while (n < len) n <<= 1;
    const bool in_smem = len <= kRowSortMax;
    int32_t* a = in_smem ? srow : src + b;
    const int32_t* rin = in ? in + in_off[r] : src + b;
    if (in_smem) {
      for (int i = threadIdx.x; i < len; i += blockDim.x) srow[i] = rin[i];
    } else if (in) {
      for (int i = threadIdx.x; i < len; i += blockDim.x) src[b + i] = rin[i];     // sorted in place in global memory
    }
    __syncthreads();
    for (int k = 2; k <= n; k <<= 1) {
      for (int j = k >> 1; j > 0; j >>= 1) {
        const bool flip = (j == (k >> 1));
        for (int i = threadIdx.x; i < len; i += blockDim.x) {
          const int p = flip ? (i ^ (k - 1)) : (i ^ j);
          if (p > i && p < len) {
            const int x = a[i], y = a[p];
            if (x > y) { a[i] = y; a[p] = x; }
          }
        }
        __syncthreads();
      }
    }
    if (in_smem) {
      for (int i = threadIdx.x; i < len; i += blockDim.x) src[b + i] = srow[i];
    }
    __syncthreads();
  }
}

// coordinates of the selected keypoints (count still on the device)
__global__ void gather_keypoints_kernel(const float* __restrict__ xyz, const int32_t* __restrict__ kp_idx,
                                        const int32_t* __restrict__ num_kp, int64_t capacity, float* __restrict__ out) {
  const int64_t v = int64_t(blockIdx.x) * blockDim.x + threadIdx.x;
  if (v >= capacity || v >= *num_kp) return;
  const int64_t j = kp_idx[v];
  out[3 * v + 0] = xyz[3 * j + 0];
  out[3 * v + 1] = xyz[3 * j + 1];
  out[3 * v + 2] = xyz[3 * j + 2];
}

// ---- host-side building blocks ----------------------------------------------------------------
struct BuiltGrid {
  Temp bounds, keys_a, keys_b, vals_a, vals_b, sorted_pts, head, head_scan, cell_key, cell_start, cub_tmp, err;
  SortedGrid view{};
};

int build_grid(const float* xyz, const int32_t* frame_ptr, int num_frames, int64_t n, const GridSpec& spec,
               cudaStream_t s, BuiltGrid* out, const int32_t* n_valid = nullptr) {
  PG_REQUIRE(num_frames >= 1 && num_frames <= 65534, "num_frames=%d out of range [1,65534]", num_frames);
  PG_REQUIRE(n >= 1 && n < (int64_t(1) << 31), "num_points=%lld out of range", (long long)n);
  PG_CUDA_OK(out->bounds.alloc(sizeof(uint32_t) * 3 * num_frames, s));
  PG_CUDA_OK(out->keys_a.alloc(sizeof(uint64_t) * n, s));
  PG_CUDA_OK(out->keys_b.alloc(sizeof(uint64_t) * n, s));
  PG_CUDA_OK(out->vals_a.alloc(sizeof(int32_t) * n, s));
  PG_CUDA_OK(out->vals_b.alloc(sizeof(int32_t) * n, s));
  PG_CUDA_OK(out->sorted_pts.alloc(sizeof(float4) * n, s));
  PG_CUDA_OK(out->head.alloc(sizeof(int32_t) * n, s));
  PG_CUDA_OK(out->head_scan.alloc(sizeof(int32_t) * n, s));
  PG_CUDA_OK(out->cell_key.alloc(sizeof(uint64_t) * n, s));
  PG_CUDA_OK(out->cell_start.alloc(sizeof(int32_t) * (n + 1), s));
  PG_CUDA_OK(out->err.alloc(sizeof(int), s));
  PG_CUDA_OK(cudaMemsetAsync(out->err.ptr, 0, sizeof(int), s));

  uint32_t* bounds = out->bounds.as<uint32_t>();
  init_bounds_kernel<<<ceil_div(3 * num_frames, 256), 256, 0, s>>>(bounds, 3 * num_frames);
  PG_LAUNCH_CHECK();
  const int blocks_per_frame = int(std::min<int64_t>(std::max<int64_t>(1, ceil_div(n / num_frames, 1024)), 64));
  frame_min_kernel<<<dim3(blocks_per_frame, num_frames), 256, 0, s>>>(xyz, frame_ptr, n, bounds);
  PG_LAUNCH_CHECK();
  point_keys_kernel<<<ceil_div(n, 256), 256, 0, s>>>(xyz, frame_ptr, num_frames, n, n_valid, spec, bounds,
                                                      out->keys_a.as<uint64_t>(), out->vals_a.as<int32_t>(),
                                                      out->err.as<int>());
  PG_LAUNCH_CHECK();
  // radix sort (key, original index); stable, so equal keys keep ascending point index
  int frame_bits = 1;
  while ((1 << frame_bits) < num_frames + 1) ++frame_bits;     // + 1: the key of rows beyond n_valid
  const int end_bit = 48 + frame_bits;
  size_t tmp_bytes = 0;
  PG_CUDA_OK(cub::DeviceRadixSort::SortPairs(nullptr, tmp_bytes, out->keys_a.as<uint64_t>(), out->keys_b.as<uint64_t>(),
                                             out->vals_a.as<int32_t>(), out->vals_b.as<int32_t>(), int(n), 0, end_bit, s));
  size_t scan_bytes = 0;
  PG_CUDA_OK(cub::DeviceScan::InclusiveSum(nullptr, scan_bytes, out->head.as<int32_t>(), out->head_scan.as<int32_t>(), int(n), s));
  PG_CUDA_OK(out->cub_tmp.alloc(std::max(tmp_bytes, scan_bytes), s));
  PG_CUDA_OK(cub::DeviceRadixSort::SortPairs(out->cub_tmp.ptr, tmp_bytes, out->keys_a.as<uint64_t>(), out->keys_b.as<uint64_t>(),
                                             out->vals_a.as<int32_t>(), out->vals_b.as<int32_t>(), int(n), 0, end_bit, s));
  count_launch(4);
  gather_sorted_kernel<<<ceil_div(n, 256), 256, 0, s>>>(xyz, out->keys_b.as<uint64_t>(), out->vals_b.as<int32_t>(), n,
                                                         out->sorted_pts.as<float4>(), out->head.as<int32_t>());
  PG_LAUNCH_CHECK();
  PG_CUDA_OK(cub::DeviceScan::InclusiveSum(out->cub_tmp.ptr, scan_bytes, out->head.as<int32_t>(), out->head_scan.as<int32_t>(), int(n), s));
  count_launch(2);
  cell_table_kernel<<<ceil_div(n, 256), 256, 0, s>>>(out->keys_b.as<uint64_t>(), out->head_scan.as<int32_t>(), n,
                                                      out->cell_key.as<uint64_t>(), out->cell_start.as<int32_t>());
  PG_LAUNCH_CHECK();
  // no host round trip here: the cell count stays on the device, the error word is read back by the caller
  // together with the size of its result
  out->view.cell_key = out->cell_key.as<uint64_t>();
  out->view.cell_start = out->cell_start.as<int32_t>();
  out->view.pts = out->sorted_pts.as<float4>();
  out->view.num_cells = out->head_scan.as<int32_t>() + (n - 1);
  return PG_OK;
}

// Decode the device-side error word of a graph call.
int graph_error(int err) {
  if (err & kErrFramePtr) {
    set_error("point frame_ptr must run from 0 to the number of points");
    return PG_ERR_INVALID_ARGUMENT;
  }
  if (err & kErrCenterPtr) {
    set_error("center frame_ptr must run from 0 to the number of centers");
    return PG_ERR_INVALID_ARGUMENT;
  }
  if (err & kErrRange) {
    set_error("point cloud extent exceeds %d grid cells per axis", kAxisMax + 1);
    return PG_ERR_RANGE;
  }
  if (err & kErrParking) {
    set_error("radius graph: hit parking buffer too small for this cloud; repeat with a larger edge capacity");
    return PG_ERR_CAPACITY;
  }
  return PG_OK;
}

struct RadiusPlan {
  BuiltGrid grid;
  GridSpec spec{};
  double r2;
};

int radius_prepare(const float* points, const int32_t* point_frame_ptr, int num_frames, int64_t num_points,
                   double radius, cudaStream_t s, RadiusPlan* plan, const double* scale_host = nullptr) {
  PG_REQUIRE(radius > 0.0, "radius must be positive");
  plan->spec = GridSpec{};
  plan->spec.cell[0] = plan->spec.cell[1] = plan->spec.cell[2] = radius * kCellSlack;
  plan->spec.origin_off = 0.0;
  plan->spec.scale[0] = plan->spec.scale[1] = plan->spec.scale[2] = 1.0;
  if (scale_host != nullptr) {
    PG_REQUIRE(scale_host[0] > 0 && scale_host[1] > 0 && scale_host[2] > 0, "scale must be positive");
    plan->spec.scaled = 1;
    for (int a = 0; a < 3; ++a) plan->spec.scale[a] = scale_host[a];
  }
  plan->r2 = radius * radius;
  return build_grid(points, point_frame_ptr, num_frames, num_points, plan->spec, s, &plan->grid);
}

}  // namespace
}  // namespace pg

using namespace pg;

extern "C" int pg_voxel_keypoints(const float* xyz, const int32_t* frame_ptr, int32_t num_frames, int64_t num_points,
                                  const double* voxel_size_host, int32_t* out_keypoint_idx, int64_t capacity,
                                  int32_t* out_kp_frame_ptr, int64_t* out_num_keypoints_host, void* stream) {
  cudaStream_t s = static_cast<cudaStream_t>(stream);
  PG_REQUIRE(xyz && frame_ptr && voxel_size_host && out_keypoint_idx && out_kp_frame_ptr && out_num_keypoints_host,
             "pg_voxel_keypoints: null argument");
  PG_REQUIRE(voxel_size_host[0] > 0 && voxel_size_host[1] > 0 && voxel_size_host[2] > 0, "voxel size must be positive");
  GridSpec spec{};
  spec.cell[0] = voxel_size_host[0];
  spec.cell[1] = voxel_size_host[1];
  spec.cell[2] = voxel_size_host[2];
  spec.origin_off = 0.5;  // Open3D: voxel_min_bound = min_bound - voxel_size * 0.5
  BuiltGrid grid;
  if (int rc = build_grid(xyz, frame_ptr, num_frames, num_points, spec, s, &grid)) return rc;
  // K = number of occupied voxels <= N is only known on the device: launch for N, surplus threads exit;
  // a keypoint is only written when it fits the caller's buffer
  voxel_keypoint_kernel<<<ceil_div(num_points, 128), 128, 0, s>>>(grid.view, spec, grid.bounds.as<uint32_t>(),
                                                                    out_keypoint_idx, capacity);
  PG_LAUNCH_CHECK();
  frame_ranges_kernel<<<ceil_div(num_frames + 1, 128), 128, 0, s>>>(grid.view.cell_key, grid.view.num_cells, num_frames,
                                                                     out_kp_frame_ptr);
  PG_LAUNCH_CHECK();
  int32_t h[2] = {0, 0};   // the one host round trip of this call: K and the error word
  PG_CUDA_OK(cudaMemcpyAsync(&h[0], grid.view.num_cells, sizeof(int32_t), cudaMemcpyDeviceToHost, s));
  PG_CUDA_OK(cudaMemcpyAsync(&h[1], grid.err.ptr, sizeof(int32_t), cudaMemcpyDeviceToHost, s));
  PG_CUDA_OK(cudaStreamSynchronize(s));
  if (int rc = graph_error(h[1])) return rc;
  *out_num_keypoints_host = h[0];
  if (h[0] > capacity) {
    set_error("keypoint buffer too small: need %d, capacity %lld", h[0], (long long)capacity);
    return PG_ERR_CAPACITY;
  }
  return PG_OK;
}

// multi_layer_downsampling for one scale (graph_gen.py:41-45): the fp64 voxel centroids themselves.
extern "C" int pg_voxel_centroids(const float* xyz, const int32_t* frame_ptr, int32_t num_frames, int64_t num_points,
                                  const double* voxel_size_host, double* out_centroids, int64_t capacity,
                                  int32_t* out_frame_ptr, int64_t* out_num_host, void* stream) {
  cudaStream_t s = static_cast<cudaStream_t>(stream);
  PG_REQUIRE(xyz && frame_ptr && voxel_size_host && out_centroids && out_frame_ptr && out_num_host,
             "pg_voxel_centroids: null argument");
  PG_REQUIRE(voxel_size_host[0] > 0 && voxel_size_host[1] > 0 && voxel_size_host[2] > 0, "voxel size must be positive");
  GridSpec spec{};
  spec.cell[0] = voxel_size_host[0];
  spec.cell[1] = voxel_size_host[1];
  spec.cell[2] = voxel_size_host[2];
  spec.origin_off = 0.5;
  BuiltGrid grid;
  if (int rc = build_grid(xyz, frame_ptr, num_frames, num_points, spec, s, &grid)) return rc;
  voxel_centroid_kernel<<<ceil_div(num_points, 128), 128, 0, s>>>(grid.view, out_centroids, nullptr, capacity);
  PG_LAUNCH_CHECK();
  frame_ranges_kernel<<<ceil_div(num_frames + 1, 128), 128, 0, s>>>(grid.view.cell_key, grid.view.num_cells, num_frames,
                                                                     out_frame_ptr);
  PG_LAUNCH_CHECK();
  int32_t h[2] = {0, 0};
  PG_CUDA_OK(cudaMemcpyAsync(&h[0], grid.view.num_cells, sizeof(int32_t), cudaMemcpyDeviceToHost, s));
  PG_CUDA_OK(cudaMemcpyAsync(&h[1], grid.err.ptr, sizeof(int32_t), cudaMemcpyDeviceToHost, s));
  PG_CUDA_OK(cudaStreamSynchronize(s));
  if (int rc = graph_error(h[1])) return rc;
  *out_num_host = h[0];
  if (h[0] > capacity) {
    set_error("centroid buffer too small: need %d, capacity %lld", h[0], (long long)capacity);
    return PG_ERR_CAPACITY;
  }
  return PG_OK;
}

// multi_layer_downsampling_select for a scale that differs from the previous level's (graph_gen.py:82-88):
// voxel centroids of the ORIGINAL cloud, each snapped to the nearest vertex of the previous level `base_xyz`.
extern "C" int pg_voxel_keypoints_select(const float* xyz, const int32_t* frame_ptr, int32_t num_frames, int64_t num_points,
                                         const double* voxel_size_host, const float* base_xyz,
                                         const int32_t* base_frame_ptr, int64_t num_base, int32_t* out_keypoint_idx,
                                         int64_t capacity, int32_t* out_kp_frame_ptr, int64_t* out_num_keypoints_host,
                                         void* stream) {
  cudaStream_t s = static_cast<cudaStream_t>(stream);
  PG_REQUIRE(xyz && frame_ptr && voxel_size_host && base_xyz && base_frame_ptr && out_keypoint_idx && out_kp_frame_ptr &&
                 out_num_keypoints_host,
             "pg_voxel_keypoints_select: null argument");
  PG_REQUIRE(voxel_size_host[0] > 0 && voxel_size_host[1] > 0 && voxel_size_host[2] > 0, "voxel size must be positive");
  GridSpec spec{};
  spec.cell[0] = voxel_size_host[0];
  spec.cell[1] = voxel_size_host[1];
  spec.cell[2] = voxel_size_host[2];
  spec.origin_off = 0.5;
  BuiltGrid grid, base;
  if (int rc = build_grid(xyz, frame_ptr, num_frames, num_points, spec, s, &grid)) return rc;
  Temp cent, cframe;
  PG_CUDA_OK(cent.alloc(sizeof(double) * 3 * num_points, s));
  PG_CUDA_OK(cframe.alloc(sizeof(int32_t) * num_points, s));
  voxel_centroid_kernel<<<ceil_div(num_points, 128), 128, 0, s>>>(grid.view, cent.as<double>(), cframe.as<int32_t>(),
                                                                    num_points);
  PG_LAUNCH_CHECK();
  frame_ranges_kernel<<<ceil_div(num_frames + 1, 128), 128, 0, s>>>(grid.view.cell_key, grid.view.num_cells, num_frames,
                                                                     out_kp_frame_ptr);
  PG_LAUNCH_CHECK();
  GridSpec bspec = spec;       // search grid over the base vertices, same cell size
  bspec.origin_off = 0.0;
  if (int rc = build_grid(base_xyz, base_frame_ptr, num_frames, num_base, bspec, s, &base)) return rc;
  nearest_point_kernel<<<ceil_div(num_points, 128), 128, 0, s>>>(base.view, bspec, base.bounds.as<uint32_t>(), base_frame_ptr,
                                                                   cent.as<double>(), cframe.as<int32_t>(),
                                                                   grid.view.num_cells, capacity, out_keypoint_idx,
                                                                   base.err.as<int>());
  PG_LAUNCH_CHECK();
  int32_t h[3] = {0, 0, 0};
  PG_CUDA_OK(cudaMemcpyAsync(&h[0], grid.view.num_cells, sizeof(int32_t), cudaMemcpyDeviceToHost, s));
  PG_CUDA_OK(cudaMemcpyAsync(&h[1], grid.err.ptr, sizeof(int32_t), cudaMemcpyDeviceToHost, s));
  PG_CUDA_OK(cudaMemcpyAsync(&h[2], base.err.ptr, sizeof(int32_t), cudaMemcpyDeviceToHost, s));
  PG_CUDA_OK(cudaStreamSynchronize(s));
  if (int rc = graph_error(h[1])) return rc;
  if (int rc = graph_error(h[2])) return rc;
  *out_num_keypoints_host = h[0];
  if (h[0] > capacity) {
    set_error("keypoint buffer too small: need %d, capacity %lld", h[0], (long long)capacity);
    return PG_ERR_CAPACITY;
  }
  return PG_OK;
}

// multi_layer_downsampling / multi_layer_downsampling_select with add_rnd3d (graph_gen.py:24-39 + :82-88): the voxel
// grid of every frame is shifted by its random fraction, a voxel's centroid is the mean of its points, and (when
// base_xyz is given) each centroid is snapped to the nearest base vertex.  The reference sums a voxel's points in
// float32 in argsort order (np.add.reduceat); here the sum is fp64 in ascending point order - equal to ~1e-6 relative.
extern "C" int pg_voxel_keypoints_rnd3d(const float* xyz, const int32_t* frame_ptr, int32_t num_frames, int64_t num_points,
                                        const double* voxel_size_host, const double* shift_host, const float* base_xyz,
                                        const int32_t* base_frame_ptr, int64_t num_base, int32_t* out_keypoint_idx,
                                        double* out_centroids, int64_t capacity, int32_t* out_kp_frame_ptr,
                                        int64_t* out_num_keypoints_host, void* stream) {
  cudaStream_t s = static_cast<cudaStream_t>(stream);
  PG_REQUIRE(xyz && frame_ptr && voxel_size_host && shift_host && out_kp_frame_ptr && out_num_keypoints_host,
             "pg_voxel_keypoints_rnd3d: null argument");
  PG_REQUIRE((base_xyz != nullptr) == (out_keypoint_idx != nullptr), "pg_voxel_keypoints_rnd3d: base_xyz and out_keypoint_idx go together");
  PG_REQUIRE(base_xyz == nullptr || base_frame_ptr != nullptr, "pg_voxel_keypoints_rnd3d: base_frame_ptr is null");
  PG_REQUIRE(voxel_size_host[0] > 0 && voxel_size_host[1] > 0 && voxel_size_host[2] > 0, "voxel size must be positive");
  Temp shift;
  PG_CUDA_OK(shift.alloc(sizeof(double) * 3 * num_frames, s));
  PG_CUDA_OK(cudaMemcpyAsync(shift.ptr, shift_host, sizeof(double) * 3 * num_frames, cudaMemcpyHostToDevice, s));
  GridSpec spec{};
  spec.cell[0] = voxel_size_host[0];
  spec.cell[1] = voxel_size_host[1];
  spec.cell[2] = voxel_size_host[2];
  spec.shift = shift.as<double>();
  BuiltGrid grid, base;
  if (int rc = build_grid(xyz, frame_ptr, num_frames, num_points, spec, s, &grid)) return rc;
  Temp cent, cframe;
  double* cent_ptr = out_centroids;
  const int64_t cent_cap = out_centroids ? capacity : num_points;
  if (cent_ptr == nullptr) {
    PG_CUDA_OK(cent.alloc(sizeof(double) * 3 * num_points, s));
    cent_ptr = cent.as<double>();
  }
  PG_CUDA_OK(cframe.alloc(sizeof(int32_t) * num_points, s));
  voxel_centroid_kernel<<<ceil_div(num_points, 128), 128, 0, s>>>(grid.view, cent_ptr, cframe.as<int32_t>(), cent_cap);
  PG_LAUNCH_CHECK();
  frame_ranges_kernel<<<ceil_div(num_frames + 1, 128), 128, 0, s>>>(grid.view.cell_key, grid.view.num_cells, num_frames,
                                                                     out_kp_frame_ptr);
  PG_LAUNCH_CHECK();
  int32_t h[3] = {0, 0, 0};
  if (base_xyz != nullptr) {
    GridSpec bspec{};
    bspec.cell[0] = voxel_size_host[0];
    bspec.cell[1] = voxel_size_host[1];
    bspec.cell[2] = voxel_size_host[2];
    if (int rc = build_grid(base_xyz, base_frame_ptr, num_frames, num_base, bspec, s, &base)) return rc;
    nearest_point_kernel<<<ceil_div(num_points, 128), 128, 0, s>>>(base.view, bspec, base.bounds.as<uint32_t>(),
                                                                     base_frame_ptr, cent_ptr, cframe.as<int32_t>(),
                                                                     grid.view.num_cells, std::min(capacity, cent_cap),
                                                                     out_keypoint_idx, base.err.as<int>());
    PG_LAUNCH_CHECK();
    PG_CUDA_OK(cudaMemcpyAsync(&h[2], base.err.ptr, sizeof(int32_t), cudaMemcpyDeviceToHost, s));
  }
  PG_CUDA_OK(cudaMemcpyAsync(&h[0], grid.view.num_cells, sizeof(int32_t), cudaMemcpyDeviceToHost, s));
  PG_CUDA_OK(cudaMemcpyAsync(&h[1], grid.err.ptr, sizeof(int32_t), cudaMemcpyDeviceToHost, s));
  PG_CUDA_OK(cudaStreamSynchronize(s));
  if (int rc = graph_error(h[1])) return rc;
  if (int rc = graph_error(h[2])) return rc;
  *out_num_keypoints_host = h[0];
  if (h[0] > capacity) {
    set_error("keypoint buffer too small: need %d, capacity %lld", h[0], (long long)capacity);
    return PG_ERR_CAPACITY;
  }
  return PG_OK;
}

static int radius_count_impl(RadiusPlan& plan, const float* centers, const int32_t* center_frame_ptr, int num_frames,
                             int64_t num_centers, int32_t* out_row_ptr, int64_t* out_num_edges_host, cudaStream_t s) {
  Temp counts, tmp, total;
  PG_CUDA_OK(counts.alloc(sizeof(int32_t) * (num_centers + 1), s));
  PG_CUDA_OK(cudaMemsetAsync(counts.ptr, 0, sizeof(int32_t) * (num_centers + 1), s));
  PG_CUDA_OK(total.alloc(sizeof(unsigned long long), s));
  PG_CUDA_OK(cudaMemsetAsync(total.ptr, 0, sizeof(unsigned long long), s));
  radius_query_kernel<false><<<ceil_div(num_centers * 32, 256), 256, 0, s>>>(
      plan.grid.view, plan.spec, plan.grid.bounds.as<uint32_t>(), centers, center_frame_ptr, num_frames, num_centers,
      nullptr, plan.r2, counts.as<int32_t>(), nullptr, nullptr, 0, plan.grid.err.as<int>(),
      total.as<unsigned long long>());
  PG_LAUNCH_CHECK();
  size_t bytes = 0;
  PG_CUDA_OK(cub::DeviceScan::ExclusiveSum(nullptr, bytes, counts.as<int32_t>(), out_row_ptr, int(num_centers + 1), s));
  PG_CUDA_OK(tmp.alloc(bytes, s));
  PG_CUDA_OK(cub::DeviceScan::ExclusiveSum(tmp.ptr, bytes, counts.as<int32_t>(), out_row_ptr, int(num_centers + 1), s));
  count_launch(2);
  unsigned long long h_total = 0;   // the one host round trip of the graph build: E (64 bit) and the error word
  int32_t h_err = 0;
  PG_CUDA_OK(cudaMemcpyAsync(&h_total, total.ptr, sizeof(h_total), cudaMemcpyDeviceToHost, s));
  PG_CUDA_OK(cudaMemcpyAsync(&h_err, plan.grid.err.ptr, sizeof(int32_t), cudaMemcpyDeviceToHost, s));
  PG_CUDA_OK(cudaStreamSynchronize(s));
  if (int rc = graph_error(h_err)) return rc;
  *out_num_edges_host = int64_t(h_total);
  if (h_total > 0x7fffffffull) {    // row_ptr is int32 (the reference's int32 edge arrays, train.py:131)
    set_error("radius graph has %llu edges: more than int32 row_ptr can index; split the batch", h_total);
    return PG_ERR_RANGE;
  }
  return PG_OK;
}

static int radius_fill_impl(RadiusPlan& plan, const float* centers, const int32_t* center_frame_ptr, int num_frames,
                            int64_t num_centers, const int32_t* row_ptr, int32_t* out_src, int32_t* out_dst,
                            cudaStream_t s) {
  radius_query_kernel<true><<<ceil_div(num_centers * 32, 256), 256, 0, s>>>(
      plan.grid.view, plan.spec, plan.grid.bounds.as<uint32_t>(), centers, center_frame_ptr, num_frames, num_centers,
      nullptr, plan.r2, nullptr, row_ptr, out_src, int64_t(1) << 40, nullptr, nullptr);
  PG_LAUNCH_CHECK();
  const int wblocks = int(std::min<int64_t>(ceil_div(num_centers, 8), int64_t(num_sms()) * 6));
  Temp has_long;
  PG_CUDA_OK(has_long.alloc(sizeof(int), s));
  PG_CUDA_OK(cudaMemsetAsync(has_long.ptr, 0, sizeof(int), s));
  sort_rows_warp_kernel<<<wblocks, 256, 0, s>>>(row_ptr, num_centers, out_src, out_dst, has_long.as<int>(),
                                                int64_t(1) << 40);
  PG_LAUNCH_CHECK();
  // rows longer than kWarpRowMax (dense full-360 clouds): one block per row
  const int blocks = int(std::min<int64_t>(num_centers, int64_t(num_sms()) * 4));
  sort_rows_kernel<<<blocks, 256, kRowSortMax * sizeof(int32_t), s>>>(row_ptr, num_centers, out_src, out_dst,
                                                                      has_long.as<int>(), int64_t(1) << 40);
  PG_LAUNCH_CHECK();
  return PG_OK;
}

extern "C" int pg_radius_graph_count(const float* points, const int32_t* point_frame_ptr, const float* centers,
                                     const int32_t* center_frame_ptr, int32_t num_frames, int64_t num_points,
                                     int64_t num_centers, double radius, int32_t* out_row_ptr,
                                     int64_t* out_num_edges_host, void* stream) {
  cudaStream_t s = static_cast<cudaStream_t>(stream);
  PG_REQUIRE(points && point_frame_ptr && centers && center_frame_ptr && out_row_ptr && out_num_edges_host,
             "pg_radius_graph_count: null argument");
  PG_REQUIRE(num_centers >= 1 && num_centers < (int64_t(1) << 31) - 1, "num_centers out of range");
  RadiusPlan plan;
  if (int rc = radius_prepare(points, point_frame_ptr, num_frames, num_points, radius, s, &plan)) return rc;
  return radius_count_impl(plan, centers, center_frame_ptr, num_frames, num_centers, out_row_ptr, out_num_edges_host, s);
}

extern "C" int pg_radius_graph_fill(const float* points, const int32_t* point_frame_ptr, const float* centers,
                                    const int32_t* center_frame_ptr, int32_t num_frames, int64_t num_points,
                                    int64_t num_centers, double radius, const int32_t* row_ptr, int64_t num_edges,
                                    int32_t* out_src, int32_t* out_dst, void* stream) {
  cudaStream_t s = static_cast<cudaStream_t>(stream);
  PG_REQUIRE(points && point_frame_ptr && centers && center_frame_ptr && row_ptr && (out_src || num_edges == 0),
             "pg_radius_graph_fill: null argument");
  if (num_edges == 0) return PG_OK;
  RadiusPlan plan;
  if (int rc = radius_prepare(points, point_frame_ptr, num_frames, num_points, radius, s, &plan)) return rc;
  return radius_fill_impl(plan, centers, center_frame_ptr, num_frames, num_centers, row_ptr, out_src, out_dst, s);
}

extern "C" int pg_radius_graph(const float* points, const int32_t* point_frame_ptr, const float* centers,
                               const int32_t* center_frame_ptr, int32_t num_frames, int64_t num_points,
                               int64_t num_centers, double radius, int32_t* out_row_ptr, int32_t* out_src,
                               int32_t* out_dst, int64_t capacity, int64_t* out_num_edges_host, void* stream) {
  return pg_radius_graph_scaled(points, point_frame_ptr, centers, center_frame_ptr, num_frames, num_points, num_centers,
                                radius, nullptr, out_row_ptr, out_src, out_dst, capacity, out_num_edges_host, stream);
}

extern "C" int pg_radius_graph_scaled(const float* points, const int32_t* point_frame_ptr, const float* centers,
                                      const int32_t* center_frame_ptr, int32_t num_frames, int64_t num_points,
                                      int64_t num_centers, double radius, const double* scale_host,
                                      int32_t* out_row_ptr, int32_t* out_src, int32_t* out_dst, int64_t capacity,
                                      int64_t* out_num_edges_host, void* stream) {
  cudaStream_t s = static_cast<cudaStream_t>(stream);
  PG_REQUIRE(points && point_frame_ptr && centers && center_frame_ptr && out_row_ptr && out_num_edges_host,
             "pg_radius_graph: null argument");
  PG_REQUIRE(num_centers >= 1 && num_centers < (int64_t(1) << 31) - 1, "num_centers out of range");
  RadiusPlan plan;
  if (int rc = radius_prepare(points, point_frame_ptr, num_frames, num_points, radius, s, &plan, scale_host)) return rc;
  if (int rc = radius_count_impl(plan, centers, center_frame_ptr, num_frames, num_centers, out_row_ptr,
                                 out_num_edges_host, s))
    return rc;
  if (*out_num_edges_host > capacity) {
    set_error("edge buffer too small: need %lld, capacity %lld", (long long)*out_num_edges_host, (long long)capacity);
    return PG_ERR_CAPACITY;
  }
  if (*out_num_edges_host == 0) return PG_OK;
  PG_REQUIRE(out_src != nullptr, "pg_radius_graph: out_src is null");
  return radius_fill_impl(plan, centers, center_frame_ptr, num_frames, num_centers, out_row_ptr, out_src, out_dst, s);
}


// One radius level of pg_multi_level_graph: count -> scan -> fill -> row sort, the number of centres and the number
// of edges staying on the device (`num_centers_dev`; E = out_row_ptr[kp_capacity]).
static int radius_level_device(RadiusPlan& plan, const float* centers, const int32_t* center_frame_ptr, int num_frames,
                               int64_t kp_capacity, const int32_t* num_centers_dev, int32_t* out_row_ptr,
                               int32_t* out_src, int32_t* out_dst, int64_t capacity, unsigned long long* total64,
                               cudaStream_t s) {
  // candidates per row are ~6.5x the hits (27 cells of edge r against the ball of radius r); the parking buffer is
  // sized from the caller's edge capacity and its overflow is reported like an edge-buffer overflow
  const int64_t tmp_capacity = std::min<int64_t>(capacity * 10 + 4096, (int64_t(1) << 31) - 1);
  Temp counts, cand, cand_off, ranges, parked, tmp, has_long;
  PG_CUDA_OK(counts.alloc(sizeof(int32_t) * (kp_capacity + 1), s));
  PG_CUDA_OK(cudaMemsetAsync(counts.ptr, 0, sizeof(int32_t) * (kp_capacity + 1), s));
  PG_CUDA_OK(cand.alloc(sizeof(int32_t) * (kp_capacity + 1), s));
  PG_CUDA_OK(cand_off.alloc(sizeof(int32_t) * (kp_capacity + 1), s));
  PG_CUDA_OK(ranges.alloc(sizeof(int32_t) * 18 * kp_capacity, s));
  PG_CUDA_OK(parked.alloc(sizeof(int32_t) * tmp_capacity, s));
  radius_candidates_kernel<<<ceil_div(kp_capacity + 1, 128), 128, 0, s>>>(
      plan.grid.view, plan.spec, plan.grid.bounds.as<uint32_t>(), centers, center_frame_ptr, num_frames, kp_capacity,
      num_centers_dev, ranges.as<int32_t>(), cand.as<int32_t>(), plan.grid.err.as<int>());
  PG_LAUNCH_CHECK();
  size_t bytes = 0;
  PG_CUDA_OK(cub::DeviceScan::ExclusiveSum(nullptr, bytes, cand.as<int32_t>(), cand_off.as<int32_t>(), int(kp_capacity + 1), s));
  PG_CUDA_OK(tmp.alloc(bytes, s));
  PG_CUDA_OK(cub::DeviceScan::ExclusiveSum(tmp.ptr, bytes, cand.as<int32_t>(), cand_off.as<int32_t>(), int(kp_capacity + 1), s));
  count_launch(2);
  radius_collect_kernel<<<ceil_div(kp_capacity * 32, 256), 256, 0, s>>>(
      plan.grid.view, centers, kp_capacity, num_centers_dev, plan.r2, ranges.as<int32_t>(), cand_off.as<int32_t>(),
      tmp_capacity, parked.as<int32_t>(), counts.as<int32_t>(), total64, plan.grid.err.as<int>());
  PG_LAUNCH_CHECK();
  PG_CUDA_OK(cub::DeviceScan::ExclusiveSum(tmp.ptr, bytes, counts.as<int32_t>(), out_row_ptr, int(kp_capacity + 1), s));
  count_launch(2);
  // rows beyond the real number of centres are empty, so row_ptr[c] == E for every c >= K
  PG_CUDA_OK(has_long.alloc(sizeof(int), s));
  PG_CUDA_OK(cudaMemsetAsync(has_long.ptr, 0, sizeof(int), s));
  const int wblocks = int(std::min<int64_t>(ceil_div(kp_capacity, 8), int64_t(num_sms()) * 6));
  sort_rows_warp_kernel<<<wblocks, 256, 0, s>>>(out_row_ptr, kp_capacity, out_src, out_dst, has_long.as<int>(), capacity,
                                                parked.as<int32_t>(), cand_off.as<int32_t>());
  PG_LAUNCH_CHECK();
  const int blocks = int(std::min<int64_t>(kp_capacity, int64_t(num_sms()) * 4));
  sort_rows_kernel<<<blocks, 256, kRowSortMax * sizeof(int32_t), s>>>(out_row_ptr, kp_capacity, out_src, out_dst,
                                                                      has_long.as<int>(), capacity, parked.as<int32_t>(),
                                                                      cand_off.as<int32_t>());
  PG_LAUNCH_CHECK();
  return PG_OK;
}

extern "C" int pg_multi_level_graph(const float* xyz, const int32_t* frame_ptr, int32_t num_frames, int64_t num_points,
                                    const double* voxel_size_host, double radius0, double radius1,
                                    int32_t* out_keypoint_idx, int64_t kp_capacity, int32_t* out_kp_frame_ptr,
                                    float* out_kp_xyz, int32_t* out_row_ptr0, int32_t* out_src0, int32_t* out_dst0,
                                    int64_t capacity0, int32_t* out_row_ptr1, int32_t* out_src1, int32_t* out_dst1,
                                    int64_t capacity1, int64_t* out_sizes_host, void* stream) {
  cudaStream_t s = static_cast<cudaStream_t>(stream);
  PG_REQUIRE(xyz && frame_ptr && voxel_size_host && out_keypoint_idx && out_kp_frame_ptr && out_kp_xyz && out_row_ptr0 &&
                 out_row_ptr1 && out_sizes_host,
             "pg_multi_level_graph: null argument");
  PG_REQUIRE(out_src0 && out_dst0 && out_src1 && out_dst1 && capacity0 >= 1 && capacity1 >= 1,
             "pg_multi_level_graph: edge buffers are required");
  PG_REQUIRE(kp_capacity >= 1 && kp_capacity <= num_points, "pg_multi_level_graph: keypoint capacity out of range");
  PG_REQUIRE(voxel_size_host[0] > 0 && voxel_size_host[1] > 0 && voxel_size_host[2] > 0, "voxel size must be positive");
  // ---- keypoints (multi_layer_downsampling_select, graph_gen.py:49-90) ---------------------------
  GridSpec vspec{};
  vspec.cell[0] = voxel_size_host[0];
  vspec.cell[1] = voxel_size_host[1];
  vspec.cell[2] = voxel_size_host[2];
  vspec.origin_off = 0.5;
  BuiltGrid vgrid;
  if (int rc = build_grid(xyz, frame_ptr, num_frames, num_points, vspec, s, &vgrid)) return rc;
  voxel_keypoint_kernel<<<ceil_div(num_points, 128), 128, 0, s>>>(vgrid.view, vspec, vgrid.bounds.as<uint32_t>(),
                                                                    out_keypoint_idx, kp_capacity);
  PG_LAUNCH_CHECK();
  frame_ranges_kernel<<<ceil_div(num_frames + 1, 128), 128, 0, s>>>(vgrid.view.cell_key, vgrid.view.num_cells, num_frames,
                                                                     out_kp_frame_ptr);
  PG_LAUNCH_CHECK();
  const int32_t* k_dev = vgrid.view.num_cells;      // K = number of occupied voxels, on the device
  gather_keypoints_kernel<<<ceil_div(kp_capacity, 256), 256, 0, s>>>(xyz, out_keypoint_idx, k_dev, kp_capacity, out_kp_xyz);
  PG_LAUNCH_CHECK();
  Temp totals;
  PG_CUDA_OK(totals.alloc(2 * sizeof(unsigned long long), s));
  PG_CUDA_OK(cudaMemsetAsync(totals.ptr, 0, 2 * sizeof(unsigned long long), s));
  // ---- level 0: original points -> keypoints (graph_gen.py:186-194, graph_level 0) -----------------
  RadiusPlan plan0;
  if (int rc = radius_prepare(xyz, frame_ptr, num_frames, num_points, radius0, s, &plan0)) return rc;
  if (int rc = radius_level_device(plan0, out_kp_xyz, out_kp_frame_ptr, num_frames, kp_capacity, k_dev, out_row_ptr0,
                                   out_src0, out_dst0, capacity0, totals.as<unsigned long long>(), s))
    return rc;
  // ---- level 1: keypoints -> keypoints (same scale: graph_gen.py:76-81 makes level 2 = level 1) ------
  RadiusPlan plan1;
  PG_REQUIRE(radius1 > 0.0, "radius must be positive");
  plan1.spec.cell[0] = plan1.spec.cell[1] = plan1.spec.cell[2] = radius1 * kCellSlack;
  plan1.spec.origin_off = 0.0;
  plan1.r2 = radius1 * radius1;
  if (int rc = build_grid(out_kp_xyz, out_kp_frame_ptr, num_frames, kp_capacity, plan1.spec, s, &plan1.grid, k_dev)) return rc;
  if (int rc = radius_level_device(plan1, out_kp_xyz, out_kp_frame_ptr, num_frames, kp_capacity, k_dev, out_row_ptr1,
                                   out_src1, out_dst1, capacity1, totals.as<unsigned long long>() + 1, s))
    return rc;
  // ---- the ONE host round trip: K, E0, E1 and the error words ---------------------------------------
  int32_t h_k = 0, h_err[3] = {0, 0, 0};
  unsigned long long h_tot[2] = {0, 0};
  PG_CUDA_OK(cudaMemcpyAsync(&h_k, k_dev, sizeof(int32_t), cudaMemcpyDeviceToHost, s));
  PG_CUDA_OK(cudaMemcpyAsync(h_tot, totals.ptr, sizeof(h_tot), cudaMemcpyDeviceToHost, s));
  PG_CUDA_OK(cudaMemcpyAsync(&h_err[0], vgrid.err.ptr, sizeof(int32_t), cudaMemcpyDeviceToHost, s));
  PG_CUDA_OK(cudaMemcpyAsync(&h_err[1], plan0.grid.err.ptr, sizeof(int32_t), cudaMemcpyDeviceToHost, s));
  PG_CUDA_OK(cudaMemcpyAsync(&h_err[2], plan1.grid.err.ptr, sizeof(int32_t), cudaMemcpyDeviceToHost, s));
  PG_CUDA_OK(cudaStreamSynchronize(s));
  out_sizes_host[0] = h_k;
  out_sizes_host[1] = int64_t(h_tot[0]);
  out_sizes_host[2] = int64_t(h_tot[1]);
  if (h_k > kp_capacity) {
    // the downstream levels only saw the first kp_capacity keypoints: everything must be redone with a larger buffer
    set_error("keypoint buffer too small: need %d, capacity %lld", h_k, (long long)kp_capacity);
    return PG_ERR_CAPACITY;
  }
  for (int i = 0; i < 3; ++i)
    if (int rc = graph_error(h_err[i])) return rc;
  if (h_tot[0] > 0x7fffffffull || h_tot[1] > 0x7fffffffull) {
    set_error("radius graph has more edges than int32 row_ptr can index; split the batch");
    return PG_ERR_RANGE;
  }
  if (int64_t(h_tot[0]) > capacity0 || int64_t(h_tot[1]) > capacity1) {
    set_error("edge buffer too small: need %llu / %llu, capacity %lld / %lld", h_tot[0], h_tot[1], (long long)capacity0,
              (long long)capacity1);
    return PG_ERR_CAPACITY;
  }
  return PG_OK;
}

// =================================================================================================
// Training-time graph path (SURVEY 8a-3 / 8f-4): random voxel keypoints and the random neighbour cap.
// The reference draws from Python's / NumPy's global generators (graph_gen.py:92-153, 210-214), so parity is
// statistical; everything that is NOT random is reproduced exactly: the voxel index arithmetic (float32
// floor-division for a scalar voxel size without the random shift, float64 with it or for an array voxel size; the
// grid origin is the minimum of the original cloud at every level), the set of occupied voxels, the first-appearance
// output order of the keypoints, "one point of its own voxel per keypoint", and for the cap "rows of at most
// num_neighbors entries keep every neighbour, longer rows keep exactly num_neighbors distinct neighbours".
// =================================================================================================
namespace pg {
namespace {

// NumPy's floor_divide for floats (npy_floor_divide / npy_divmod): Python semantics
template <typename T>
__device__ inline T np_floor_divide(T a, T b) {
  T mod = fmod(a, b);
  T div = (a - mod) / b;
  if (mod != T(0) && ((b < T(0)) != (mod < T(0)))) div -= T(1);
  if (div != T(0)) {
    T fl = floor(div);
    if (div - fl > T(0.5)) fl += T(1);
    return fl;
  }
  return copysign(T(0), a / b);
}

__device__ void shifted_cell_of(const GridSpec& g, const uint32_t* __restrict__ bounds, int f, float x, float y, float z,
                                long long* ix, long long* iy, long long* iz) {
  const float p[3] = {x, y, z};
  long long idx[3];
  for (int a = 0; a < 3; ++a) {
    const float d = __fsub_rn(p[a], ordered_to_float(bounds[3 * f + a]));            // float32, as points_xyz - xyz_offset
    const double t = __dadd_rn(double(d), __dmul_rn(g.cell[a], g.shift[3 * f + a]));
    idx[a] = (long long)np_floor_divide<double>(t, g.cell[a]);
  }
  *ix = idx[0];
  *iy = idx[1];
  *iz = idx[2];
}

// graph_gen.py:124-131 voxel index of every point; shift == nullptr: float32 arithmetic (add_rnd3d False),
// else float64 with the per-frame random shift fractions (add_rnd3d True; a zero shift gives the exact float64
// quotient of an array voxel size).  `bounds` holds the per-frame minimum of the ORIGINAL cloud (origin_frame_ptr,
// num_origin rows), which fixes the grid origin of every level (graph_gen.py:107-110).
__global__ void random_voxel_keys_kernel(const float* __restrict__ xyz, const int32_t* __restrict__ frame_ptr, int num_frames,
                                         int64_t n, const int32_t* __restrict__ origin_frame_ptr, int64_t num_origin,
                                         double vx, double vy, double vz, const double* __restrict__ shift,
                                         const uint32_t* __restrict__ bounds, uint64_t* __restrict__ keys,
                                         int32_t* __restrict__ vals, int* __restrict__ err) {
  const int64_t i = int64_t(blockIdx.x) * blockDim.x + threadIdx.x;
  if (i >= n) return;
  if (i == 0 && (frame_ptr[0] != 0 || int64_t(frame_ptr[num_frames]) != n || origin_frame_ptr[0] != 0 ||
                 int64_t(origin_frame_ptr[num_frames]) != num_origin))
    atomicOr(err, kErrFramePtr);
  const int f = find_frame(frame_ptr, num_frames, i);
  const float mn[3] = {ordered_to_float(bounds[3 * f]), ordered_to_float(bounds[3 * f + 1]), ordered_to_float(bounds[3 * f + 2])};
  const double v[3] = {vx, vy, vz};
  long long idx[3];
  for (int a = 0; a < 3; ++a) {
    const float d = __fsub_rn(xyz[3 * i + a], mn[a]);
    if (shift == nullptr) {
      idx[a] = (long long)np_floor_divide<float>(d, float(v[a]));
    } else {
      const double t = __dadd_rn(double(d), __dmul_rn(v[a], shift[3 * f + a]));
      idx[a] = (long long)np_floor_divide<double>(t, v[a]);
    }
    if (idx[a] < 0 || idx[a] > kAxisMax) {
      atomicOr(err, kErrRange);
      idx[a] = 0;
    }
  }
  keys[i] = make_key(uint32_t(f), uint32_t(idx[2]), uint32_t(idx[1]), uint32_t(idx[0]));
  vals[i] = int32_t(i);
}

__global__ void head_flags_kernel(const uint64_t* __restrict__ keys, int64_t n, int32_t* __restrict__ head) {
  const int64_t i = int64_t(blockIdx.x) * blockDim.x + threadIdx.x;
  if (i < n) head[i] = (i == 0 || keys[i] != keys[i - 1]) ? 1 : 0;
}

// second sort key of every voxel: (frame, smallest original point index) = dict insertion order of graph_gen.py:133-139
__global__ void voxel_first_keys_kernel(const uint64_t* __restrict__ cell_key, const int32_t* __restrict__ cell_start,
                                        const int32_t* __restrict__ sorted_idx, const int32_t* __restrict__ num_cells,
                                        int64_t n, int num_frames, uint64_t* __restrict__ keys2, int32_t* __restrict__ vals2) {
  const int64_t v = int64_t(blockIdx.x) * blockDim.x + threadIdx.x;
  if (v >= n) return;
  vals2[v] = int32_t(v);
  if (v < *num_cells) keys2[v] = ((cell_key[v] >> 48) << 32) | uint64_t(uint32_t(sorted_idx[cell_start[v]]));
  else keys2[v] = uint64_t(num_frames) << 32;     // behind every real voxel
}

__global__ void random_pick_kernel(const int32_t* __restrict__ order, const int32_t* __restrict__ cell_start,
                                   const int32_t* __restrict__ sorted_idx, const int32_t* __restrict__ num_cells,
                                   const float* __restrict__ uniform, int64_t capacity, int32_t* __restrict__ out_idx) {
  const int64_t o = int64_t(blockIdx.x) * blockDim.x + threadIdx.x;
  if (o >= *num_cells || o >= capacity) return;
  const int c = order[o];
  const int s = cell_start[c], cnt = cell_start[c + 1] - s;
  int pick = int(uniform[o] * float(cnt));          // random.choice(seq) = seq[floor(u * len)], u in [0, 1)
  pick = min(max(pick, 0), cnt - 1);
  out_idx[o] = sorted_idx[s + pick];
}

__global__ void random_frame_ranges_kernel(const uint64_t* __restrict__ keys2_sorted, const int32_t* __restrict__ num_cells,
                                           int num_frames, int32_t* __restrict__ out_frame_ptr) {
  const int f = blockIdx.x * blockDim.x + threadIdx.x;
  if (f > num_frames) return;
  out_frame_ptr[f] = lower_bound_u64(keys2_sorted, *num_cells, uint64_t(f) << 32);
}

// ---- random neighbour cap ------------------------------------------------------------------------
__device__ inline uint32_t mix32(uint32_t x) {     // integer hash (murmur3 finaliser)
  x ^= x >> 16; x *= 0x85ebca6bu; x ^= x >> 13; x *= 0xc2b2ae35u; x ^= x >> 16;
  return x;
}
__device__ inline uint32_t edge_priority(uint32_t seed, uint32_t row, uint32_t src) {
  return mix32(mix32(seed ^ (row * 0x9e3779b9u)) ^ (src * 0x7f4a7c15u));
}

__global__ void capped_counts_kernel(const int32_t* __restrict__ row_ptr, int64_t num_rows, int cap, int32_t* __restrict__ counts) {
  const int64_t r = int64_t(blockIdx.x) * blockDim.x + threadIdx.x;
  if (r > num_rows) return;
  counts[r] = r < num_rows ? min(row_ptr[r + 1] - row_ptr[r], cap) : 0;
}

// One warp per row.  Rows longer than `cap` keep the `cap` entries with the smallest hash priority (a uniformly random
// subset for a random seed), found by a bitwise search for the cap-th smallest priority; ascending source order is kept.
__global__ void __launch_bounds__(256) cap_rows_kernel(const int32_t* __restrict__ row_ptr, const int32_t* __restrict__ src,
                                                       int64_t num_rows, int cap, uint32_t seed,
                                                       const int32_t* __restrict__ new_row_ptr, int32_t* __restrict__ out_src,
                                                       int32_t* __restrict__ out_dst) {
  const int lane = threadIdx.x & 31;
  const int64_t r = (int64_t(blockIdx.x) * blockDim.x + threadIdx.x) >> 5;
  if (r >= num_rows) return;
  const int b = row_ptr[r], len = row_ptr[r + 1] - b, ob = new_row_ptr[r];
  if (len <= cap) {
    for (int i = lane; i < len; i += 32) {
      out_src[ob + i] = src[b + i];
      out_dst[ob + i] = int32_t(r);
    }
    return;
  }
  // largest threshold t with count(priority < t) <= cap, built bit by bit
  uint32_t t = 0;
  for (int bit = 31; bit >= 0; --bit) {
    const uint32_t cand = t | (1u << bit);
    int cnt = 0;
    for (int i = lane; i < len; i += 32) cnt += edge_priority(seed, uint32_t(r), uint32_t(src[b + i])) < cand ? 1 : 0;
    for (int o = 16; o > 0; o >>= 1) cnt += __shfl_xor_sync(0xffffffffu, cnt, o);
    if (cnt <= cap) t = cand;
  }
  // entries with priority < t are kept; ties at t fill the remaining slots in source order
  int below = 0;
  for (int i = lane; i < len; i += 32) below += edge_priority(seed, uint32_t(r), uint32_t(src[b + i])) < t ? 1 : 0;
  for (int o = 16; o > 0; o >>= 1) below += __shfl_xor_sync(0xffffffffu, below, o);
  int need_ties = cap - below, written = 0;
  for (int i0 = 0; i0 < len; i0 += 32) {
    const int i = i0 + lane;
    bool keep = false, tie = false;
    int s = 0;
    if (i < len) {
      s = src[b + i];
      const uint32_t pr = edge_priority(seed, uint32_t(r), uint32_t(s));
      keep = pr < t;
      tie = pr == t;
    }
    const uint32_t tm = __ballot_sync(0xffffffffu, tie);
    const int tie_rank = __popc(tm & ((1u << lane) - 1u));
    if (tie && tie_rank < need_ties) keep = true;
    need_ties -= min(need_ties, __popc(tm));
    const uint32_t km = __ballot_sync(0xffffffffu, keep);
    if (keep) {
      const int o = ob + written + __popc(km & ((1u << lane) - 1u));
      out_src[o] = s;
      out_dst[o] = int32_t(r);
    }
    written += __popc(km);
  }
}

}  // namespace
}  // namespace pg

extern "C" int pg_random_keypoints(const float* xyz, const int32_t* frame_ptr, int32_t num_frames, int64_t num_points,
                                   const double* voxel_size_host, const double* shift_host, const float* base_xyz,
                                   const int32_t* base_frame_ptr, int64_t num_base, const float* uniform,
                                   int32_t* out_keypoint_idx, int64_t capacity, int32_t* out_kp_frame_ptr,
                                   int64_t* out_num_keypoints_host, void* stream) {
  cudaStream_t s = static_cast<cudaStream_t>(stream);
  PG_REQUIRE(xyz && frame_ptr && voxel_size_host && base_xyz && base_frame_ptr && uniform && out_keypoint_idx &&
                 out_kp_frame_ptr && out_num_keypoints_host,
             "pg_random_keypoints: null argument");
  PG_REQUIRE(voxel_size_host[0] > 0 && voxel_size_host[1] > 0 && voxel_size_host[2] > 0, "voxel size must be positive");
  PG_REQUIRE(num_frames >= 1 && num_frames <= 65534, "num_frames=%d out of range [1,65534]", num_frames);
  PG_REQUIRE(num_points >= 1 && num_points < (int64_t(1) << 31), "num_points=%lld out of range", (long long)num_points);
  const int64_t n = num_base;      // the points that are voxelised; xyz only sets the grid origin
  PG_REQUIRE(n >= 1 && n < (int64_t(1) << 31), "num_base=%lld out of range", (long long)n);
  Temp bounds, keys_a, keys_b, vals_a, vals_b, head, head_scan, cell_key, cell_start, keys2a, keys2b, vals2a, vals2b, tmp, err,
      shift;
  PG_CUDA_OK(bounds.alloc(sizeof(uint32_t) * 3 * num_frames, s));
  PG_CUDA_OK(keys_a.alloc(sizeof(uint64_t) * n, s));
  PG_CUDA_OK(keys_b.alloc(sizeof(uint64_t) * n, s));
  PG_CUDA_OK(vals_a.alloc(sizeof(int32_t) * n, s));
  PG_CUDA_OK(vals_b.alloc(sizeof(int32_t) * n, s));
  PG_CUDA_OK(head.alloc(sizeof(int32_t) * n, s));
  PG_CUDA_OK(head_scan.alloc(sizeof(int32_t) * n, s));
  PG_CUDA_OK(cell_key.alloc(sizeof(uint64_t) * n, s));
  PG_CUDA_OK(cell_start.alloc(sizeof(int32_t) * (n + 1), s));
  PG_CUDA_OK(keys2a.alloc(sizeof(uint64_t) * n, s));
  PG_CUDA_OK(keys2b.alloc(sizeof(uint64_t) * n, s));
  PG_CUDA_OK(vals2a.alloc(sizeof(int32_t) * n, s));
  PG_CUDA_OK(vals2b.alloc(sizeof(int32_t) * n, s));
  PG_CUDA_OK(err.alloc(sizeof(int), s));
  PG_CUDA_OK(cudaMemsetAsync(err.ptr, 0, sizeof(int), s));
  const double* shift_dev = nullptr;
  if (shift_host != nullptr) {
    PG_CUDA_OK(shift.alloc(sizeof(double) * 3 * num_frames, s));
    PG_CUDA_OK(cudaMemcpyAsync(shift.ptr, shift_host, sizeof(double) * 3 * num_frames, cudaMemcpyHostToDevice, s));
    shift_dev = shift.as<double>();
  }
  init_bounds_kernel<<<ceil_div(3 * num_frames, 256), 256, 0, s>>>(bounds.as<uint32_t>(), 3 * num_frames);
  PG_LAUNCH_CHECK();
  const int blocks_per_frame = int(std::min<int64_t>(std::max<int64_t>(1, ceil_div(num_points / num_frames, 1024)), 64));
  frame_min_kernel<<<dim3(blocks_per_frame, num_frames), 256, 0, s>>>(xyz, frame_ptr, num_points, bounds.as<uint32_t>());
  PG_LAUNCH_CHECK();
  random_voxel_keys_kernel<<<ceil_div(n, 256), 256, 0, s>>>(base_xyz, base_frame_ptr, num_frames, n, frame_ptr, num_points,
                                                            voxel_size_host[0], voxel_size_host[1], voxel_size_host[2],
                                                            shift_dev, bounds.as<uint32_t>(), keys_a.as<uint64_t>(),
                                                            vals_a.as<int32_t>(), err.as<int>());
  PG_LAUNCH_CHECK();
  int frame_bits = 1;
  while ((1 << frame_bits) < num_frames + 1) ++frame_bits;
  size_t b1 = 0, b2 = 0, b3 = 0;
  PG_CUDA_OK(cub::DeviceRadixSort::SortPairs(nullptr, b1, keys_a.as<uint64_t>(), keys_b.as<uint64_t>(), vals_a.as<int32_t>(),
                                             vals_b.as<int32_t>(), int(n), 0, 48 + frame_bits, s));
  PG_CUDA_OK(cub::DeviceScan::InclusiveSum(nullptr, b2, head.as<int32_t>(), head_scan.as<int32_t>(), int(n), s));
  PG_CUDA_OK(cub::DeviceRadixSort::SortPairs(nullptr, b3, keys2a.as<uint64_t>(), keys2b.as<uint64_t>(), vals2a.as<int32_t>(),
                                             vals2b.as<int32_t>(), int(n), 0, 32 + frame_bits, s));
  PG_CUDA_OK(tmp.alloc(std::max(b1, std::max(b2, b3)), s));
  PG_CUDA_OK(cub::DeviceRadixSort::SortPairs(tmp.ptr, b1, keys_a.as<uint64_t>(), keys_b.as<uint64_t>(), vals_a.as<int32_t>(),
                                             vals_b.as<int32_t>(), int(n), 0, 48 + frame_bits, s));
  count_launch(4);
  head_flags_kernel<<<ceil_div(n, 256), 256, 0, s>>>(keys_b.as<uint64_t>(), n, head.as<int32_t>());
  PG_LAUNCH_CHECK();
  PG_CUDA_OK(cub::DeviceScan::InclusiveSum(tmp.ptr, b2, head.as<int32_t>(), head_scan.as<int32_t>(), int(n), s));
  count_launch(2);
  cell_table_kernel<<<ceil_div(n, 256), 256, 0, s>>>(keys_b.as<uint64_t>(), head_scan.as<int32_t>(), n, cell_key.as<uint64_t>(),
                                                      cell_start.as<int32_t>());
  PG_LAUNCH_CHECK();
  const int32_t* num_cells = head_scan.as<int32_t>() + (n - 1);
  voxel_first_keys_kernel<<<ceil_div(n, 256), 256, 0, s>>>(cell_key.as<uint64_t>(), cell_start.as<int32_t>(), vals_b.as<int32_t>(),
                                                            num_cells, n, num_frames, keys2a.as<uint64_t>(), vals2a.as<int32_t>());
  PG_LAUNCH_CHECK();
  PG_CUDA_OK(cub::DeviceRadixSort::SortPairs(tmp.ptr, b3, keys2a.as<uint64_t>(), keys2b.as<uint64_t>(), vals2a.as<int32_t>(),
                                             vals2b.as<int32_t>(), int(n), 0, 32 + frame_bits, s));
  count_launch(4);
  random_pick_kernel<<<ceil_div(n, 256), 256, 0, s>>>(vals2b.as<int32_t>(), cell_start.as<int32_t>(), vals_b.as<int32_t>(),
                                                       num_cells, uniform, capacity, out_keypoint_idx);
  PG_LAUNCH_CHECK();
  random_frame_ranges_kernel<<<ceil_div(num_frames + 1, 128), 128, 0, s>>>(keys2b.as<uint64_t>(), num_cells, num_frames,
                                                                            out_kp_frame_ptr);
  PG_LAUNCH_CHECK();
  int32_t h[2] = {0, 0};
  PG_CUDA_OK(cudaMemcpyAsync(&h[0], num_cells, sizeof(int32_t), cudaMemcpyDeviceToHost, s));
  PG_CUDA_OK(cudaMemcpyAsync(&h[1], err.ptr, sizeof(int32_t), cudaMemcpyDeviceToHost, s));
  PG_CUDA_OK(cudaStreamSynchronize(s));
  if (int rc = graph_error(h[1])) return rc;
  *out_num_keypoints_host = h[0];
  if (h[0] > capacity) {
    set_error("keypoint buffer too small: need %d, capacity %lld", h[0], (long long)capacity);
    return PG_ERR_CAPACITY;
  }
  return PG_OK;
}

extern "C" int pg_cap_neighbors(const int32_t* row_ptr, const int32_t* src, int64_t num_rows, int32_t num_neighbors,
                                uint32_t seed, int32_t* out_row_ptr, int32_t* out_src, int32_t* out_dst, int64_t capacity,
                                int64_t* out_num_edges_host, void* stream) {
  cudaStream_t s = static_cast<cudaStream_t>(stream);
  PG_REQUIRE(row_ptr && out_row_ptr && out_num_edges_host && num_rows >= 1 && num_neighbors >= 1,
             "pg_cap_neighbors: bad argument");
  Temp counts, tmp;
  PG_CUDA_OK(counts.alloc(sizeof(int32_t) * (num_rows + 1), s));
  capped_counts_kernel<<<ceil_div(num_rows + 1, 256), 256, 0, s>>>(row_ptr, num_rows, num_neighbors, counts.as<int32_t>());
  PG_LAUNCH_CHECK();
  size_t bytes = 0;
  PG_CUDA_OK(cub::DeviceScan::ExclusiveSum(nullptr, bytes, counts.as<int32_t>(), out_row_ptr, int(num_rows + 1), s));
  PG_CUDA_OK(tmp.alloc(bytes, s));
  PG_CUDA_OK(cub::DeviceScan::ExclusiveSum(tmp.ptr, bytes, counts.as<int32_t>(), out_row_ptr, int(num_rows + 1), s));
  count_launch(2);
  int32_t h_e = 0;
  PG_CUDA_OK(cudaMemcpyAsync(&h_e, out_row_ptr + num_rows, sizeof(int32_t), cudaMemcpyDeviceToHost, s));
  PG_CUDA_OK(cudaStreamSynchronize(s));
  *out_num_edges_host = h_e;
  if (h_e > capacity) {
    set_error("edge buffer too small: need %d, capacity %lld", h_e, (long long)capacity);
    return PG_ERR_CAPACITY;
  }
  if (h_e == 0) return PG_OK;
  PG_REQUIRE(src && out_src && out_dst, "pg_cap_neighbors: null edge buffer");
  cap_rows_kernel<<<ceil_div(num_rows * 32, 256), 256, 0, s>>>(row_ptr, src, num_rows, num_neighbors, seed, out_row_ptr, out_src,
                                                               out_dst);
  PG_LAUNCH_CHECK();
  return PG_OK;
}
