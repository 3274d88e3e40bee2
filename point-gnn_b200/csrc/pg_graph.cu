// Graph construction on the GPU: voxel keypoint selection and radius-neighbour CSR graphs.
//
// Replaces /root/reference/models/graph_gen.py:
//   multi_layer_downsampling (:11-47, open3d.voxel_down_sample branch :41-45)
//   multi_layer_downsampling_select (:49-90, kd-tree 1-NN snap :84-88)
//   gen_disjointed_rnn_local_graph_v3 (:197-220, ball-tree radius query)
//
// Design: every spatial query runs on a sorted-key uniform grid.  A point's key packs
//   frame | iz | iy | ix
// (KeyLayout: 32 bits when the cell indices fit, 64 bits with 16 bits per axis otherwise), so one radix sort groups
// points by (frame, cell) and, because ix is the low field, the three x-adjacent cells of a (frame, iz, iy) row are one
// contiguous range of the sorted array: a 3x3x3 neighbourhood costs 9 binary searches.  There is no dense grid, so
// memory is O(N) whatever the extent of the cloud.  All predicates that decide membership (voxel index, nearest
// point, radius test) are evaluated in fp64 with explicitly rounded mul/add (no FMA contraction), which is what makes
// the edge lists bit-exact against the reference's scikit-learn float64 trees.
#include <cub/cub.cuh>

#include "pg_common.cuh"

namespace pg {
namespace {

constexpr int kAxisBits = 16;
constexpr int kAxisMax = (1 << kAxisBits) - 1;
constexpr double kCellSlack = 1.0001;  // cell edge = radius * slack, keeps +-1 cell search exact
// device-side error word of one graph call (read back once, together with the result size)
constexpr int kErrRange = 1;       // cloud extent exceeds 16 bits per axis
constexpr int kErrFramePtr = 2;    // point frame_ptr does not run from 0 to N
constexpr int kErrCenterPtr = 4;   // centre frame_ptr does not run from 0 to K
constexpr int kErrParking = 8;     // pg_multi_level_graph: hit parking buffer too small (retry with larger edge capacity)
constexpr int kErrKeyWidth = 16;   // a cell index fits 16 bits but not the compact 32-bit key: redo the call with 64 bits
// internal return code (never leaves the library): the call ran on compact keys and must be redone on 64-bit keys
constexpr int kRetryWide = 1;

// Bit layout of a cell key: frame | iz | iy | ix, ix in the low bits.  Both widths keep this field order, so cells
// sort identically and the keypoint order (= cell order) does not depend on the width.
template <typename Key>
struct KeyLayout {
  using KeyType = Key;
  int sy, sz, sf;   // bit offsets of iy, iz and the frame (ix starts at bit 0)
  uint32_t max[3];  // largest cell index per axis (x, y, z)
  int end_bit;      // bits the radix sort looks at
  __host__ __device__ Key make(uint32_t f, uint32_t iz, uint32_t iy, uint32_t ix) const {
    return (Key(f) << sf) | (Key(iz) << sz) | (Key(iy) << sy) | Key(ix);
  }
  __host__ __device__ uint32_t frame(Key k) const { return uint32_t(k >> sf); }
};

// + 1: the frame field also holds `num_frames`, the key of padding rows beyond n_valid
int frame_bits(int num_frames) {
  int bits = 1;
  while ((1 << bits) < num_frames + 1) ++bits;
  return bits;
}

KeyLayout<uint64_t> wide_layout(int num_frames) {
  return {16, 32, 48, {kAxisMax, kAxisMax, kAxisMax}, 48 + frame_bits(num_frames)};
}

// The bits the frame field leaves are split between the axes; y (the camera frame's vertical axis, a few metres of
// extent) gets the fewest.  8 frames: 10 | 8 | 10 bits for x | y | z, 410 x 102 x 410 m at 0.4 m cells; 64 frames:
// 9 | 7 | 9 bits.
KeyLayout<uint32_t> compact_layout(int num_frames) {
  const int axis = 32 - frame_bits(num_frames);
  const int by = axis / 3 - 1, bx = (axis - by + 1) / 2, bz = axis - by - bx;
  return {bx, bx + by, axis, {(1u << bx) - 1, (1u << by) - 1, (1u << bz) - 1}, 32};
}

// Runs `body` on compact keys and, when a cell index did not fit them, once more on 64-bit keys.
template <typename Body>
int with_cell_keys(int num_frames, Body&& body) {
  const int rc = body(compact_layout(num_frames));
  return rc == kRetryWide ? body(wide_layout(num_frames)) : rc;
}

// All temporaries of a call live in one stream-ordered allocation.  `carve` takes the call's slices in a fixed order;
// it runs once on an empty arena to add up the sizes and once on the allocated block.
struct Arena {
  char* base = nullptr;
  size_t used = 0;
  template <typename T>
  T* take(size_t count) {
    const size_t at = (used + 255) & ~size_t(255);
    used = at + sizeof(T) * std::max<size_t>(count, 1);
    return base ? reinterpret_cast<T*>(base + at) : nullptr;
  }
};

template <typename Carve>
int alloc_workspace(Temp& ws, cudaStream_t s, Carve&& carve) {
  Arena probe;
  carve(probe);
  PG_CUDA_OK(ws.alloc(probe.used, s));
  Arena real;
  real.base = ws.as<char>();
  carve(real);
  return PG_OK;
}

// The words a call clears before its first kernel (one memset): edge totals, error word, long-row counters.
struct CallHeader {
  unsigned long long totals[2];
  int err;
  int num_long[2];
};

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

// ---- per-frame bounding-box minimum (bounds start as 0xff bytes: the largest ordered value) ----------------------
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

GridSpec voxel_spec(const double* voxel_size_host, double origin_off) {
  GridSpec spec{};
  for (int a = 0; a < 3; ++a) spec.cell[a] = voxel_size_host[a];
  spec.origin_off = origin_off;
  return spec;
}

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

// Key of a cell.  An index beyond 16 bits per axis is an error of the call (kErrRange); one that only overflows the
// compact layout asks for the 64-bit retry (kErrKeyWidth).  Either way the key stays inside the layout.
template <typename Key>
__device__ inline Key checked_key(const KeyLayout<Key>& L, uint32_t f, long long ix, long long iy, long long iz,
                                  int* __restrict__ err) {
  if (ix < 0 || iy < 0 || iz < 0 || ix > kAxisMax || iy > kAxisMax || iz > kAxisMax) {
    atomicOr(err, kErrRange);
    return L.make(f, 0, 0, 0);
  }
  if (ix > L.max[0] || iy > L.max[1] || iz > L.max[2]) {
    atomicOr(err, kErrKeyWidth);
    return L.make(f, 0, 0, 0);
  }
  return L.make(f, uint32_t(iz), uint32_t(iy), uint32_t(ix));
}

// `n_valid` (optional, device): only rows [0, *n_valid) of the n-row buffer hold points (a point set whose size is
// still on the device, e.g. the keypoints of the same call); the others get the key of frame `num_frames`, which
// sorts behind every real cell and is never looked up.
template <typename Key>
__global__ void point_keys_kernel(const float* __restrict__ xyz, const int32_t* __restrict__ frame_ptr,
                                  int num_frames, int64_t n, const int32_t* __restrict__ n_valid, GridSpec g,
                                  KeyLayout<Key> L, const uint32_t* __restrict__ bounds, Key* __restrict__ keys,
                                  int32_t* __restrict__ vals, int* __restrict__ err) {
  int64_t i = int64_t(blockIdx.x) * blockDim.x + threadIdx.x;
  if (i >= n) return;
  const int64_t nv = n_valid ? int64_t(*n_valid) : n;
  // the caller's frame partition must run from 0 to n (checked here instead of with a host round trip)
  if (i == 0 && (frame_ptr[0] != 0 || int64_t(frame_ptr[num_frames]) != nv)) atomicOr(err, kErrFramePtr);
  vals[i] = int32_t(i);
  if (i >= nv) {
    keys[i] = L.make(uint32_t(num_frames), 0, 0, 0);
    return;
  }
  const int f = find_frame(frame_ptr, num_frames, i);
  long long ix, iy, iz;
  if (g.shift != nullptr) shifted_cell_of(g, bounds, f, xyz[3 * i], xyz[3 * i + 1], xyz[3 * i + 2], &ix, &iy, &iz);
  else cell_of(g, bounds, f, xyz[3 * i], xyz[3 * i + 1], xyz[3 * i + 2], &ix, &iy, &iz);
  keys[i] = checked_key(L, uint32_t(f), ix, iy, iz, err);
}

// sorted point record (coalesced candidate reads) + head flag of each run of equal keys
template <typename Key>
__global__ void gather_sorted_kernel(const float* __restrict__ xyz, const Key* __restrict__ keys,
                                     const int32_t* __restrict__ order, int64_t n,
                                     float4* __restrict__ sorted_pts, int32_t* __restrict__ head) {
  int64_t i = int64_t(blockIdx.x) * blockDim.x + threadIdx.x;
  if (i >= n) return;
  const int32_t j = order[i];
  sorted_pts[i] = make_float4(xyz[3 * j], xyz[3 * j + 1], xyz[3 * j + 2], __int_as_float(j));
  head[i] = (i == 0 || keys[i] != keys[i - 1]) ? 1 : 0;
}

// cell table: cell_key[c], cell_start[c] for every non-empty cell c (ascending key)
template <typename Key>
__global__ void cell_table_kernel(const Key* __restrict__ keys, const int32_t* __restrict__ head_scan,
                                  int64_t n, Key* __restrict__ cell_key, int32_t* __restrict__ cell_start) {
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

template <typename Key>
__device__ inline int lower_bound_key(const Key* __restrict__ a, int n, Key v) {
  int lo = 0, hi = n;
  while (lo < hi) {
    int mid = (lo + hi) >> 1;
    if (a[mid] < v) lo = mid + 1; else hi = mid;
  }
  return lo;
}

template <typename Key>
struct SortedGrid {
  KeyLayout<Key> layout;
  const Key* cell_key;        // [num_cells]
  const int32_t* cell_start;  // [num_cells+1]
  const float4* pts;          // [n] sorted (x,y,z,orig idx)
  const int32_t* num_cells;   // device scalar (= last element of the head-flag scan): no host round trip
};

// point range covering cells (f, iz, iy, ix_lo..ix_hi); indices already clamped to the layout
template <typename Key>
__device__ inline void row_range(const SortedGrid<Key>& g, uint32_t f, uint32_t iz, uint32_t iy, uint32_t ix_lo,
                                 uint32_t ix_hi, int* begin, int* end) {
  const int nc = __ldg(g.num_cells);
  const int a = lower_bound_key(g.cell_key, nc, g.layout.make(f, iz, iy, ix_lo));
  const int b = lower_bound_key(g.cell_key, nc, Key(g.layout.make(f, iz, iy, ix_hi) + 1));
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
template <typename Key>
__global__ void voxel_keypoint_kernel(SortedGrid<Key> g, GridSpec spec, const uint32_t* __restrict__ bounds,
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
  const uint32_t f = g.layout.frame(g.cell_key[v]);
  const double reach = sqrt(best) * (1.0 + 1e-9) + 1e-12;
  const double ox = double(ordered_to_float(bounds[3 * f + 0])) - spec.cell[0] * spec.origin_off;
  const double oy = double(ordered_to_float(bounds[3 * f + 1])) - spec.cell[1] * spec.origin_off;
  const double oz = double(ordered_to_float(bounds[3 * f + 2])) - spec.cell[2] * spec.origin_off;
  // reach is inflated by 1e-9 relative, far above the fp64 rounding of the corner cells
  long long x0 = (long long)floor((cx - reach - ox) / spec.cell[0]), x1 = (long long)floor((cx + reach - ox) / spec.cell[0]);
  long long y0 = (long long)floor((cy - reach - oy) / spec.cell[1]), y1 = (long long)floor((cy + reach - oy) / spec.cell[1]);
  long long z0 = (long long)floor((cz - reach - oz) / spec.cell[2]), z1 = (long long)floor((cz + reach - oz) / spec.cell[2]);
  x0 = max(x0, 0ll); y0 = max(y0, 0ll); z0 = max(z0, 0ll);
  x1 = min(x1, (long long)g.layout.max[0]); y1 = min(y1, (long long)g.layout.max[1]); z1 = min(z1, (long long)g.layout.max[2]);
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
template <typename Key>
__global__ void voxel_centroid_kernel(SortedGrid<Key> g, double* __restrict__ out_centroid, int32_t* __restrict__ out_frame,
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
  if (out_frame) out_frame[v] = int32_t(g.layout.frame(g.cell_key[v]));
}

// nearest base point (fp64 squared distance, ties -> lowest index) of query q inside its own frame.
// Growing boxes of cells until one holds a point, then ONE exact pass over every cell the ball of that radius touches.
template <typename Key>
__global__ void nearest_point_kernel(SortedGrid<Key> g, GridSpec spec, const uint32_t* __restrict__ bounds,
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
  const KeyLayout<Key>& L = g.layout;
  double best = DBL_MAX;
  int best_idx = 0x7fffffff;
  auto scan = [&](long long x0, long long x1, long long y0, long long y1, long long z0, long long z1) {
    x0 = max(x0, 0ll); y0 = max(y0, 0ll); z0 = max(z0, 0ll);
    x1 = min(x1, (long long)L.max[0]); y1 = min(y1, (long long)L.max[1]); z1 = min(z1, (long long)L.max[2]);
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

template <typename Key>
__global__ void frame_ranges_kernel(SortedGrid<Key> g, int num_frames, int32_t* __restrict__ out_frame_ptr) {
  const int f = blockIdx.x * blockDim.x + threadIdx.x;
  if (f > num_frames) return;
  out_frame_ptr[f] = lower_bound_key(g.cell_key, __ldg(g.num_cells), g.layout.make(uint32_t(f), 0, 0, 0));
}

// ---- radius graph ----------------------------------------------------------------------------
// One warp per centre.  kFill=false: count neighbours.  kFill=true: write source indices at
// row_ptr[c] + rank (rank from a warp ballot prefix, traversal order; rows are sorted afterwards).
template <bool kFill, typename Key>
__global__ void __launch_bounds__(256) radius_query_kernel(
    SortedGrid<Key> g, GridSpec spec, const uint32_t* __restrict__ bounds, const float* __restrict__ centers,
    const int32_t* __restrict__ center_frame_ptr, int num_frames, int64_t num_centers,
    double r2, int32_t* __restrict__ counts, const int32_t* __restrict__ row_ptr, int32_t* __restrict__ out_src,
    int* __restrict__ err, unsigned long long* __restrict__ total64) {
  const int lane = threadIdx.x & 31;
  const int64_t c = (int64_t(blockIdx.x) * blockDim.x + threadIdx.x) >> 5;
  if (c >= num_centers) return;
  if (!kFill && c == 0 && lane == 0 &&
      (center_frame_ptr[0] != 0 || int64_t(center_frame_ptr[num_frames]) != num_centers))
    atomicOr(err, kErrCenterPtr);
  const KeyLayout<Key>& L = g.layout;
  const int f = find_frame(center_frame_ptr, num_frames, c);
  const float cxf = centers[3 * c], cyf = centers[3 * c + 1], czf = centers[3 * c + 2];
  const double cx = coord(spec, cxf, 0), cy = coord(spec, cyf, 1), cz = coord(spec, czf, 2);
  long long ix, iy, iz;
  cell_of(spec, bounds, f, cxf, cyf, czf, &ix, &iy, &iz);
  const long long x0 = max(ix - 1, 0ll), x1 = min(ix + 1, (long long)L.max[0]);
  int total = 0;
  int base = kFill ? row_ptr[c] : 0;
  if (x0 <= x1) {
    for (long long zz = iz - 1; zz <= iz + 1; ++zz) {
      if (zz < 0 || zz > L.max[2]) continue;
      for (long long yy = iy - 1; yy <= iy + 1; ++yy) {
        if (yy < 0 || yy > L.max[1]) continue;
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
// their total length = an upper bound of the row length.  No point is touched.  It also clears the row lengths that
// pass B fills (rows beyond the real number of centres stay empty).
template <typename Key>
__global__ void radius_candidates_kernel(SortedGrid<Key> g, GridSpec spec, const uint32_t* __restrict__ bounds,
                                         const float* __restrict__ centers, const int32_t* __restrict__ center_frame_ptr,
                                         int num_frames, int64_t num_centers_cap, const int32_t* __restrict__ num_centers_dev,
                                         int32_t* __restrict__ ranges, int32_t* __restrict__ cand,
                                         int32_t* __restrict__ counts, int* __restrict__ err) {
  const int64_t c = int64_t(blockIdx.x) * blockDim.x + threadIdx.x;
  if (c > num_centers_cap) return;
  counts[c] = 0;
  const int64_t num_centers = min(int64_t(*num_centers_dev), num_centers_cap);
  if (c >= num_centers) {
    cand[c] = 0;
    return;
  }
  if (c == 0 && (center_frame_ptr[0] != 0 || int64_t(center_frame_ptr[num_frames]) != int64_t(*num_centers_dev)))
    atomicOr(err, kErrCenterPtr);
  const KeyLayout<Key>& L = g.layout;
  const int f = find_frame(center_frame_ptr, num_frames, c);
  long long ix, iy, iz;
  cell_of(spec, bounds, f, centers[3 * c], centers[3 * c + 1], centers[3 * c + 2], &ix, &iy, &iz);
  const long long x0 = max(ix - 1, 0ll), x1 = min(ix + 1, (long long)L.max[0]);
  int total = 0, k = 0;
  for (long long zz = iz - 1; zz <= iz + 1; ++zz) {
    for (long long yy = iy - 1; yy <= iy + 1; ++yy, ++k) {
      int b = 0, e = 0;
      if (x0 <= x1 && zz >= 0 && zz <= L.max[2] && yy >= 0 && yy <= L.max[1])
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
__global__ void __launch_bounds__(256) radius_collect_kernel(const float4* __restrict__ pts, const float* __restrict__ centers,
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
  int rb = 0;
  if (lane < 18) rb = ranges[c * 18 + lane];
  for (int k = 0; k < 9; ++k) {
    const int b = __shfl_sync(0xffffffffu, rb, 2 * k), e = __shfl_sync(0xffffffffu, rb, 2 * k + 1);
    for (int i0 = b; i0 < e; i0 += 32) {
      const int i = i0 + lane;
      bool hit = false;
      int idx = 0;
      if (i < e) {
        const float4 p = pts[i];
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

// ---- CSR row sort ------------------------------------------------------------------------------------------------
// Every row ascending (canonical order), dst expanded.  The unsorted entries of row r sit at in[in_off[r] ...] (the
// parked hits); the sorted row is written to src[row_ptr[r] ...].  A row holds distinct point indices.
constexpr int kWarpRowMax = 1024;    // one warp sorts rows up to this length in registers (32 entries per lane)
constexpr int kLongRowSmem = 8192;   // longer rows up to this length keep their sorted chunks in shared memory

// Bitonic sort of the warp's 32 * E values, entry e * 32 + lane in v[e] of that lane: strides of 32 and more are
// compare-exchanges inside a lane, shorter ones a __shfl_xor_sync.  Ascending.
template <int E>
__device__ __forceinline__ void warp_bitonic(int32_t (&v)[E], int lane) {
#pragma unroll
  for (int k = 2; k <= 32 * E; k <<= 1) {
#pragma unroll
    for (int j = k >> 1; j > 0; j >>= 1) {
      if (j >= 32) {
#pragma unroll
        for (int e = 0; e < E; ++e) {
          const int p = e ^ (j >> 5);
          if (p > e) {
            const bool up = ((e * 32) & k) == 0;
            const int32_t x = v[e], y = v[p];
            v[e] = up ? min(x, y) : max(x, y);
            v[p] = up ? max(x, y) : min(x, y);
          }
        }
      } else {
        const bool lower = (lane & j) == 0;
#pragma unroll
        for (int e = 0; e < E; ++e) {
          const bool up = ((e * 32 + lane) & k) == 0;
          const int32_t y = __shfl_xor_sync(0xffffffffu, v[e], j);
          v[e] = (lower == up) ? min(v[e], y) : max(v[e], y);
        }
      }
    }
  }
}

// sort in[0, len) (len <= 32 * E) into out[0, len); padding INT_MAX stays behind every point index
template <int E>
__device__ __forceinline__ void warp_sort_run(const int32_t* in, int len, int32_t* out, int lane) {
  int32_t v[E];
#pragma unroll
  for (int e = 0; e < E; ++e) v[e] = e * 32 + lane < len ? in[e * 32 + lane] : 0x7fffffff;
  warp_bitonic<E>(v, lane);
#pragma unroll
  for (int e = 0; e < E; ++e)
    if (e * 32 + lane < len) out[e * 32 + lane] = v[e];
}

// One warp per row, dispatched by the row's power-of-two size class.  Longer rows are listed for row_sort_long_kernel.
__global__ void __launch_bounds__(256, 2) row_sort_warp_kernel(const int32_t* __restrict__ row_ptr, int64_t num_rows,
                                                             const int32_t* __restrict__ in, const int32_t* __restrict__ in_off,
                                                             int32_t* __restrict__ src, int32_t* __restrict__ dst,
                                                             int64_t capacity, int32_t* __restrict__ long_rows,
                                                             int* __restrict__ num_long) {
  const int lane = threadIdx.x & 31;
  const int64_t r = (int64_t(blockIdx.x) * blockDim.x + threadIdx.x) >> 5;
  if (r >= num_rows || int64_t(row_ptr[num_rows]) > capacity) return;   // edge buffer too small: nothing was filled
  const int b = row_ptr[r], len = row_ptr[r + 1] - b;
  if (dst != nullptr)
    for (int i = lane; i < len; i += 32) dst[b + i] = int32_t(r);
  if (len > kWarpRowMax) {
    if (lane == 0) long_rows[atomicAdd(num_long, 1)] = int32_t(r);
    return;
  }
  const int32_t* rin = in + in_off[r];
  int32_t* out = src + b;
  if (len <= 1) {
    if (len == 1 && lane == 0) out[0] = rin[0];
  } else if (len <= 32) {
    warp_sort_run<1>(rin, len, out, lane);
  } else if (len <= 64) {
    warp_sort_run<2>(rin, len, out, lane);
  } else if (len <= 128) {
    warp_sort_run<4>(rin, len, out, lane);
  } else if (len <= 256) {
    warp_sort_run<8>(rin, len, out, lane);
  } else if (len <= 512) {
    warp_sort_run<16>(rin, len, out, lane);
  } else {
    warp_sort_run<32>(rin, len, out, lane);
  }
}

// One block per listed long row.  Each warp sorts 1024-entry chunks in registers; an entry's place in the row is then
// its place in its chunk plus the number of entries below it in every other chunk (binary searches; the entries are
// distinct).  Two block barriers per row, whatever its length.  Rows longer than kLongRowSmem keep their sorted
// chunks in place in `in`.
__global__ void __launch_bounds__(256) row_sort_long_kernel(const int32_t* __restrict__ row_ptr, int64_t num_rows,
                                                             int32_t* in, const int32_t* __restrict__ in_off,
                                                             int32_t* __restrict__ src, int64_t capacity,
                                                             const int32_t* __restrict__ long_rows,
                                                             const int* __restrict__ num_long) {
  __shared__ int32_t chunks[kLongRowSmem];
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31, num_warps = blockDim.x >> 5;
  if (int64_t(row_ptr[num_rows]) > capacity) return;
  const int count = *num_long;
  for (int l = blockIdx.x; l < count; l += gridDim.x) {
    const int r = long_rows[l];
    const int b = row_ptr[r], len = row_ptr[r + 1] - b;
    int32_t* rin = in + in_off[r];
    int32_t* sorted = len <= kLongRowSmem ? chunks : rin;
    const int num_chunks = (len + kWarpRowMax - 1) / kWarpRowMax;
    for (int c = warp; c < num_chunks; c += num_warps) {
      const int cb = c * kWarpRowMax;
      warp_sort_run<kWarpRowMax / 32>(rin + cb, min(kWarpRowMax, len - cb), sorted + cb, lane);
    }
    __syncthreads();
    for (int i = threadIdx.x; i < len; i += blockDim.x) {
      const int32_t x = sorted[i];
      const int own = i / kWarpRowMax;
      int rank = i - own * kWarpRowMax;
      for (int c = 0; c < num_chunks; ++c) {
        if (c == own) continue;
        int lo = c * kWarpRowMax, hi = min(lo + kWarpRowMax, len);
        const int cb = lo;
        while (lo < hi) {
          const int mid = (lo + hi) >> 1;
          if (sorted[mid] < x) lo = mid + 1; else hi = mid;
        }
        rank += lo - cb;
      }
      src[b + rank] = x;
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
// CUB's onesweep radix sort: an upfront histogram, its scan, then one pass per 8 key bits
int radix_sort_launches(int end_bit) { return 2 + (end_bit + 7) / 8; }

// per-frame minimum of xyz into bounds (which the caller set to 0xff bytes)
int frame_min(const float* xyz, const int32_t* frame_ptr, int num_frames, int64_t n, uint32_t* bounds, cudaStream_t s) {
  const int blocks_per_frame = int(std::min<int64_t>(std::max<int64_t>(1, ceil_div(n / num_frames, 1024)), 64));
  frame_min_kernel<<<dim3(blocks_per_frame, num_frames), 256, 0, s>>>(xyz, frame_ptr, n, bounds);
  PG_LAUNCH_CHECK();
  return PG_OK;
}

int check_grid_args(int num_frames, int64_t n) {
  PG_REQUIRE(num_frames >= 1 && num_frames <= 65534, "num_frames=%d out of range [1,65534]", num_frames);
  PG_REQUIRE(n >= 1 && n < (int64_t(1) << 31), "num_points=%lld out of range", (long long)n);
  return PG_OK;
}

// CUB scratch of one grid build (radix sort, head-flag scan)
template <typename Key>
int grid_cub_bytes(int64_t n, const KeyLayout<Key>& L, size_t* bytes) {
  size_t sort = 0, scan = 0;
  PG_CUDA_OK(cub::DeviceRadixSort::SortPairs(nullptr, sort, (const Key*)nullptr, (Key*)nullptr, (const int32_t*)nullptr,
                                             (int32_t*)nullptr, int(n), 0, L.end_bit));
  PG_CUDA_OK(cub::DeviceScan::InclusiveSum(nullptr, scan, (const int32_t*)nullptr, (int32_t*)nullptr, int(n)));
  *bytes = std::max(*bytes, std::max(sort, scan));
  return PG_OK;
}

int exclusive_sum_bytes(int64_t n, size_t* bytes) {
  size_t scan = 0;
  PG_CUDA_OK(cub::DeviceScan::ExclusiveSum(nullptr, scan, (const int32_t*)nullptr, (int32_t*)nullptr, int(n)));
  *bytes = std::max(*bytes, scan);
  return PG_OK;
}

template <typename Key>
struct GridBufs {
  int64_t n = 0;
  Key *keys_a, *keys_b, *cell_key;
  int32_t *vals_a, *vals_b, *head, *head_scan, *cell_start;
  float4* pts;
  void carve(Arena& a, int64_t num) {
    n = num;
    keys_a = a.take<Key>(n);
    keys_b = a.take<Key>(n);
    cell_key = a.take<Key>(n);
    vals_a = a.take<int32_t>(n);
    vals_b = a.take<int32_t>(n);
    head = a.take<int32_t>(n);
    head_scan = a.take<int32_t>(n);
    cell_start = a.take<int32_t>(n + 1);
    pts = a.take<float4>(n);
  }
};

// Keys -> stable radix sort -> sorted points + cell table.  `bounds` holds the per-frame minimum (frame_min).
// No host round trip: the cell count stays on the device, the error word is read back by the caller together with
// the size of its result.
template <typename Key>
int build_grid(const float* xyz, const int32_t* frame_ptr, int num_frames, const GridSpec& spec, const KeyLayout<Key>& L,
               const uint32_t* bounds, GridBufs<Key>& b, void* cub_tmp, size_t cub_bytes, int* err, cudaStream_t s,
               SortedGrid<Key>* out, const int32_t* n_valid = nullptr) {
  const int64_t n = b.n;
  point_keys_kernel<Key><<<ceil_div(n, 256), 256, 0, s>>>(xyz, frame_ptr, num_frames, n, n_valid, spec, L, bounds,
                                                         b.keys_a, b.vals_a, err);
  PG_LAUNCH_CHECK();
  // radix sort (key, original index); stable, so equal keys keep ascending point index
  size_t bytes = cub_bytes;
  PG_CUDA_OK(cub::DeviceRadixSort::SortPairs(cub_tmp, bytes, b.keys_a, b.keys_b, b.vals_a, b.vals_b, int(n), 0,
                                             L.end_bit, s));
  count_launch(radix_sort_launches(L.end_bit));
  gather_sorted_kernel<Key><<<ceil_div(n, 256), 256, 0, s>>>(xyz, b.keys_b, b.vals_b, n, b.pts, b.head);
  PG_LAUNCH_CHECK();
  bytes = cub_bytes;
  PG_CUDA_OK(cub::DeviceScan::InclusiveSum(cub_tmp, bytes, b.head, b.head_scan, int(n), s));
  count_launch(2);
  cell_table_kernel<Key><<<ceil_div(n, 256), 256, 0, s>>>(b.keys_b, b.head_scan, n, b.cell_key, b.cell_start);
  PG_LAUNCH_CHECK();
  out->layout = L;
  out->cell_key = b.cell_key;
  out->cell_start = b.cell_start;
  out->pts = b.pts;
  out->num_cells = b.head_scan + (n - 1);
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
  if (err & kErrKeyWidth) return kRetryWide;
  if (err & kErrParking) {
    set_error("radius graph: hit parking buffer too small for this cloud; repeat with a larger edge capacity");
    return PG_ERR_CAPACITY;
  }
  return PG_OK;
}

int radius_spec(double radius, const double* scale_host, GridSpec* spec) {
  PG_REQUIRE(radius > 0.0, "radius must be positive");
  *spec = GridSpec{};
  spec->cell[0] = spec->cell[1] = spec->cell[2] = radius * kCellSlack;
  spec->origin_off = 0.0;
  spec->scale[0] = spec->scale[1] = spec->scale[2] = 1.0;
  if (scale_host != nullptr) {
    PG_REQUIRE(scale_host[0] > 0 && scale_host[1] > 0 && scale_host[2] > 0, "scale must be positive");
    spec->scaled = 1;
    for (int a = 0; a < 3; ++a) spec->scale[a] = scale_host[a];
  }
  return PG_OK;
}

// Sort the rows (in -> src) and expand dst; long_rows [num_rows] and *num_long (cleared) list the long rows.
int sort_rows(const int32_t* row_ptr, int64_t num_rows, int32_t* in, const int32_t* in_off, int32_t* src, int32_t* dst,
              int64_t capacity, int32_t* long_rows, int* num_long, cudaStream_t s) {
  row_sort_warp_kernel<<<ceil_div(num_rows * 32, 256), 256, 0, s>>>(row_ptr, num_rows, in, in_off, src, dst, capacity,
                                                                    long_rows, num_long);
  PG_LAUNCH_CHECK();
  const int blocks = int(std::min<int64_t>(num_rows, int64_t(num_sms()) * 4));
  row_sort_long_kernel<<<blocks, 256, 0, s>>>(row_ptr, num_rows, in, in_off, src, capacity, long_rows, num_long);
  PG_LAUNCH_CHECK();
  return PG_OK;
}

// ---- one-grid entries ---------------------------------------------------------------------------------------------
// pg_voxel_keypoints (keypoint indices) and pg_voxel_centroids (fp64 centroids): one voxel grid, one round trip.
template <typename Key>
int voxel_grid_call(const KeyLayout<Key>& L, const float* xyz, const int32_t* frame_ptr, int num_frames, int64_t n,
                    const double* voxel_size_host, int32_t* out_keypoint_idx, double* out_centroids, int64_t capacity,
                    int32_t* out_frame_ptr, int64_t* out_num_host, cudaStream_t s) {
  const GridSpec spec = voxel_spec(voxel_size_host, 0.5);  // Open3D: voxel_min_bound = min_bound - voxel_size * 0.5
  size_t cub_bytes = 0;
  if (int rc = grid_cub_bytes(n, L, &cub_bytes)) return rc;
  CallHeader* hdr;
  uint32_t* bounds;
  GridBufs<Key> gb;
  void* cub_tmp;
  Temp ws;
  if (int rc = alloc_workspace(ws, s, [&](Arena& a) {
        hdr = a.take<CallHeader>(1);
        bounds = a.take<uint32_t>(3 * num_frames);
        gb.carve(a, n);
        cub_tmp = a.take<char>(cub_bytes);
      }))
    return rc;
  PG_CUDA_OK(cudaMemsetAsync(hdr, 0, sizeof(CallHeader), s));
  PG_CUDA_OK(cudaMemsetAsync(bounds, 0xff, sizeof(uint32_t) * 3 * num_frames, s));
  if (int rc = frame_min(xyz, frame_ptr, num_frames, n, bounds, s)) return rc;
  SortedGrid<Key> g;
  if (int rc = build_grid(xyz, frame_ptr, num_frames, spec, L, bounds, gb, cub_tmp, cub_bytes, &hdr->err, s, &g)) return rc;
  // K = number of occupied voxels <= N is only known on the device: launch for N, surplus threads exit;
  // a result is only written when it fits the caller's buffer
  if (out_keypoint_idx != nullptr)
    voxel_keypoint_kernel<Key><<<ceil_div(n, 128), 128, 0, s>>>(g, spec, bounds, out_keypoint_idx, capacity);
  else
    voxel_centroid_kernel<Key><<<ceil_div(n, 128), 128, 0, s>>>(g, out_centroids, nullptr, capacity);
  PG_LAUNCH_CHECK();
  frame_ranges_kernel<Key><<<ceil_div(num_frames + 1, 128), 128, 0, s>>>(g, num_frames, out_frame_ptr);
  PG_LAUNCH_CHECK();
  int32_t h[2] = {0, 0};   // the one host round trip of this call: K and the error word
  PG_CUDA_OK(cudaMemcpyAsync(&h[0], g.num_cells, sizeof(int32_t), cudaMemcpyDeviceToHost, s));
  PG_CUDA_OK(cudaMemcpyAsync(&h[1], &hdr->err, sizeof(int32_t), cudaMemcpyDeviceToHost, s));
  PG_CUDA_OK(cudaStreamSynchronize(s));
  if (int rc = graph_error(h[1])) return rc;
  *out_num_host = h[0];
  if (h[0] > capacity) {
    set_error("%s buffer too small: need %d, capacity %lld", out_keypoint_idx ? "keypoint" : "centroid", h[0],
              (long long)capacity);
    return PG_ERR_CAPACITY;
  }
  return PG_OK;
}

// voxel centroids of the ORIGINAL cloud (`spec`, shift optional), each snapped to the nearest vertex of `base_xyz`
// when it is given: pg_voxel_keypoints_select and pg_voxel_keypoints_rnd3d.
template <typename Key>
int voxel_select_call(const KeyLayout<Key>& L, const float* xyz, const int32_t* frame_ptr, int num_frames, int64_t n,
                      const double* voxel_size_host, const double* shift_host, const float* base_xyz,
                      const int32_t* base_frame_ptr, int64_t num_base, int32_t* out_keypoint_idx, double* out_centroids,
                      int64_t capacity, int32_t* out_kp_frame_ptr, int64_t* out_num_keypoints_host, cudaStream_t s) {
  GridSpec spec = voxel_spec(voxel_size_host, shift_host ? 0.0 : 0.5);
  // search grid over the base vertices, same cell size
  const GridSpec bspec = voxel_spec(voxel_size_host, 0.0);
  if (base_xyz != nullptr)
    if (int rc = check_grid_args(num_frames, num_base)) return rc;
  size_t cub_bytes = 0;
  if (int rc = grid_cub_bytes(n, L, &cub_bytes)) return rc;
  if (base_xyz != nullptr)
    if (int rc = grid_cub_bytes(num_base, L, &cub_bytes)) return rc;
  const int64_t cent_cap = out_centroids ? capacity : n;
  CallHeader* hdr;
  uint32_t* bounds;
  double *shift = nullptr, *cent = out_centroids;
  int32_t* cframe;
  GridBufs<Key> gb, bb;
  void* cub_tmp;
  Temp ws;
  if (int rc = alloc_workspace(ws, s, [&](Arena& a) {
        hdr = a.take<CallHeader>(1);
        bounds = a.take<uint32_t>(6 * num_frames);   // the cloud's and the base vertices' per-frame minimum
        if (shift_host) shift = a.take<double>(3 * num_frames);
        if (!out_centroids) cent = a.take<double>(3 * n);
        cframe = a.take<int32_t>(n);
        gb.carve(a, n);
        if (base_xyz) bb.carve(a, num_base);
        cub_tmp = a.take<char>(cub_bytes);
      }))
    return rc;
  PG_CUDA_OK(cudaMemsetAsync(hdr, 0, sizeof(CallHeader), s));
  PG_CUDA_OK(cudaMemsetAsync(bounds, 0xff, sizeof(uint32_t) * 6 * num_frames, s));
  if (shift_host) {
    PG_CUDA_OK(cudaMemcpyAsync(shift, shift_host, sizeof(double) * 3 * num_frames, cudaMemcpyHostToDevice, s));
    spec.shift = shift;
  }
  if (int rc = frame_min(xyz, frame_ptr, num_frames, n, bounds, s)) return rc;
  SortedGrid<Key> g;
  if (int rc = build_grid(xyz, frame_ptr, num_frames, spec, L, bounds, gb, cub_tmp, cub_bytes, &hdr->err, s, &g)) return rc;
  voxel_centroid_kernel<Key><<<ceil_div(n, 128), 128, 0, s>>>(g, cent, cframe, cent_cap);
  PG_LAUNCH_CHECK();
  frame_ranges_kernel<Key><<<ceil_div(num_frames + 1, 128), 128, 0, s>>>(g, num_frames, out_kp_frame_ptr);
  PG_LAUNCH_CHECK();
  if (base_xyz != nullptr) {
    uint32_t* bbounds = bounds + 3 * num_frames;
    if (int rc = frame_min(base_xyz, base_frame_ptr, num_frames, num_base, bbounds, s)) return rc;
    SortedGrid<Key> bg;
    if (int rc = build_grid(base_xyz, base_frame_ptr, num_frames, bspec, L, bbounds, bb, cub_tmp, cub_bytes, &hdr->err,
                            s, &bg))
      return rc;
    nearest_point_kernel<Key><<<ceil_div(n, 128), 128, 0, s>>>(bg, bspec, bbounds, base_frame_ptr, cent, cframe,
                                                               g.num_cells, std::min(capacity, cent_cap),
                                                               out_keypoint_idx, &hdr->err);
    PG_LAUNCH_CHECK();
  }
  int32_t h[2] = {0, 0};
  PG_CUDA_OK(cudaMemcpyAsync(&h[0], g.num_cells, sizeof(int32_t), cudaMemcpyDeviceToHost, s));
  PG_CUDA_OK(cudaMemcpyAsync(&h[1], &hdr->err, sizeof(int32_t), cudaMemcpyDeviceToHost, s));
  PG_CUDA_OK(cudaStreamSynchronize(s));
  if (int rc = graph_error(h[1])) return rc;
  *out_num_keypoints_host = h[0];
  if (h[0] > capacity) {
    set_error("keypoint buffer too small: need %d, capacity %lld", h[0], (long long)capacity);
    return PG_ERR_CAPACITY;
  }
  return PG_OK;
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
  if (int rc = check_grid_args(num_frames, num_points)) return rc;
  return with_cell_keys(num_frames, [&](auto L) {
    return voxel_grid_call(L, xyz, frame_ptr, num_frames, num_points, voxel_size_host, out_keypoint_idx, nullptr,
                           capacity, out_kp_frame_ptr, out_num_keypoints_host, s);
  });
}

// multi_layer_downsampling for one scale (graph_gen.py:41-45): the fp64 voxel centroids themselves.
extern "C" int pg_voxel_centroids(const float* xyz, const int32_t* frame_ptr, int32_t num_frames, int64_t num_points,
                                  const double* voxel_size_host, double* out_centroids, int64_t capacity,
                                  int32_t* out_frame_ptr, int64_t* out_num_host, void* stream) {
  cudaStream_t s = static_cast<cudaStream_t>(stream);
  PG_REQUIRE(xyz && frame_ptr && voxel_size_host && out_centroids && out_frame_ptr && out_num_host,
             "pg_voxel_centroids: null argument");
  PG_REQUIRE(voxel_size_host[0] > 0 && voxel_size_host[1] > 0 && voxel_size_host[2] > 0, "voxel size must be positive");
  if (int rc = check_grid_args(num_frames, num_points)) return rc;
  return with_cell_keys(num_frames, [&](auto L) {
    return voxel_grid_call(L, xyz, frame_ptr, num_frames, num_points, voxel_size_host, nullptr, out_centroids, capacity,
                           out_frame_ptr, out_num_host, s);
  });
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
  if (int rc = check_grid_args(num_frames, num_points)) return rc;
  return with_cell_keys(num_frames, [&](auto L) {
    return voxel_select_call(L, xyz, frame_ptr, num_frames, num_points, voxel_size_host, nullptr, base_xyz,
                             base_frame_ptr, num_base, out_keypoint_idx, nullptr, capacity, out_kp_frame_ptr,
                             out_num_keypoints_host, s);
  });
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
  if (int rc = check_grid_args(num_frames, num_points)) return rc;
  return with_cell_keys(num_frames, [&](auto L) {
    return voxel_select_call(L, xyz, frame_ptr, num_frames, num_points, voxel_size_host, shift_host, base_xyz,
                             base_frame_ptr, num_base, out_keypoint_idx, out_centroids, capacity, out_kp_frame_ptr,
                             out_num_keypoints_host, s);
  });
}

namespace pg {
namespace {

// The radius graph of the stand-alone entries.  Count pass (row lengths, one round trip for E), then, when `fill`,
// the fill pass parks every row's hits in traversal order and the row sort writes the CSR rows.
template <typename Key>
int radius_call(const KeyLayout<Key>& L, const float* points, const int32_t* point_frame_ptr, const float* centers,
                const int32_t* center_frame_ptr, int num_frames, int64_t num_points, int64_t num_centers, double radius,
                const double* scale_host, int32_t* out_row_ptr, bool fill, int64_t num_edges, int32_t* out_src,
                int32_t* out_dst, int64_t capacity, int64_t* out_num_edges_host, cudaStream_t s) {
  GridSpec spec;
  if (int rc = radius_spec(radius, scale_host, &spec)) return rc;
  if (int rc = check_grid_args(num_frames, num_points)) return rc;
  const bool count = out_num_edges_host != nullptr;
  size_t cub_bytes = 0;
  if (int rc = grid_cub_bytes(num_points, L, &cub_bytes)) return rc;
  if (int rc = exclusive_sum_bytes(num_centers + 1, &cub_bytes)) return rc;
  CallHeader* hdr;
  uint32_t* bounds;
  int32_t *counts = nullptr, *long_rows = nullptr;
  GridBufs<Key> gb;
  void* cub_tmp;
  Temp ws;
  if (int rc = alloc_workspace(ws, s, [&](Arena& a) {
        hdr = a.take<CallHeader>(1);
        bounds = a.take<uint32_t>(3 * num_frames);
        if (count) counts = a.take<int32_t>(num_centers + 1);
        if (fill) long_rows = a.take<int32_t>(num_centers);
        gb.carve(a, num_points);
        cub_tmp = a.take<char>(cub_bytes);
      }))
    return rc;
  PG_CUDA_OK(cudaMemsetAsync(hdr, 0, sizeof(CallHeader), s));
  PG_CUDA_OK(cudaMemsetAsync(bounds, 0xff, sizeof(uint32_t) * 3 * num_frames, s));
  if (int rc = frame_min(points, point_frame_ptr, num_frames, num_points, bounds, s)) return rc;
  SortedGrid<Key> g;
  if (int rc = build_grid(points, point_frame_ptr, num_frames, spec, L, bounds, gb, cub_tmp, cub_bytes, &hdr->err, s, &g))
    return rc;
  const double r2 = radius * radius;
  if (count) {
    PG_CUDA_OK(cudaMemsetAsync(counts + num_centers, 0, sizeof(int32_t), s));
    radius_query_kernel<false, Key><<<ceil_div(num_centers * 32, 256), 256, 0, s>>>(
        g, spec, bounds, centers, center_frame_ptr, num_frames, num_centers, r2, counts, nullptr, nullptr, &hdr->err,
        hdr->totals);
    PG_LAUNCH_CHECK();
    size_t bytes = cub_bytes;
    PG_CUDA_OK(cub::DeviceScan::ExclusiveSum(cub_tmp, bytes, counts, out_row_ptr, int(num_centers + 1), s));
    count_launch(2);
    unsigned long long h_total = 0;   // the one host round trip of the graph build: E (64 bit) and the error word
    int32_t h_err = 0;
    PG_CUDA_OK(cudaMemcpyAsync(&h_total, hdr->totals, sizeof(h_total), cudaMemcpyDeviceToHost, s));
    PG_CUDA_OK(cudaMemcpyAsync(&h_err, &hdr->err, sizeof(int32_t), cudaMemcpyDeviceToHost, s));
    PG_CUDA_OK(cudaStreamSynchronize(s));
    if (int rc = graph_error(h_err)) return rc;
    *out_num_edges_host = int64_t(h_total);
    if (h_total > 0x7fffffffull) {    // row_ptr is int32 (the reference's int32 edge arrays, train.py:131)
      set_error("radius graph has %llu edges: more than int32 row_ptr can index; split the batch", h_total);
      return PG_ERR_RANGE;
    }
    if (!fill) return PG_OK;
    num_edges = int64_t(h_total);
    if (num_edges > capacity) {
      set_error("edge buffer too small: need %lld, capacity %lld", (long long)num_edges, (long long)capacity);
      return PG_ERR_CAPACITY;
    }
    if (num_edges == 0) return PG_OK;
    PG_REQUIRE(out_src != nullptr, "pg_radius_graph: out_src is null");
  }
  Temp parked;
  PG_CUDA_OK(parked.alloc(sizeof(int32_t) * num_edges, s));
  radius_query_kernel<true, Key><<<ceil_div(num_centers * 32, 256), 256, 0, s>>>(
      g, spec, bounds, centers, center_frame_ptr, num_frames, num_centers, r2, nullptr, out_row_ptr,
      parked.as<int32_t>(), nullptr, nullptr);
  PG_LAUNCH_CHECK();
  return sort_rows(out_row_ptr, num_centers, parked.as<int32_t>(), out_row_ptr, out_src, out_dst, num_edges, long_rows,
                   &hdr->num_long[0], s);
}

}  // namespace
}  // namespace pg

extern "C" int pg_radius_graph_count(const float* points, const int32_t* point_frame_ptr, const float* centers,
                                     const int32_t* center_frame_ptr, int32_t num_frames, int64_t num_points,
                                     int64_t num_centers, double radius, int32_t* out_row_ptr,
                                     int64_t* out_num_edges_host, void* stream) {
  cudaStream_t s = static_cast<cudaStream_t>(stream);
  PG_REQUIRE(points && point_frame_ptr && centers && center_frame_ptr && out_row_ptr && out_num_edges_host,
             "pg_radius_graph_count: null argument");
  PG_REQUIRE(num_centers >= 1 && num_centers < (int64_t(1) << 31) - 1, "num_centers out of range");
  if (int rc = check_grid_args(num_frames, num_points)) return rc;
  return with_cell_keys(num_frames, [&](auto L) {
    return radius_call(L, points, point_frame_ptr, centers, center_frame_ptr, num_frames, num_points, num_centers,
                       radius, nullptr, out_row_ptr, false, 0, nullptr, nullptr, 0, out_num_edges_host, s);
  });
}

// The fill half has no host round trip in which a compact-key overflow could be seen, so it always uses 64-bit keys.
extern "C" int pg_radius_graph_fill(const float* points, const int32_t* point_frame_ptr, const float* centers,
                                    const int32_t* center_frame_ptr, int32_t num_frames, int64_t num_points,
                                    int64_t num_centers, double radius, const int32_t* row_ptr, int64_t num_edges,
                                    int32_t* out_src, int32_t* out_dst, void* stream) {
  cudaStream_t s = static_cast<cudaStream_t>(stream);
  PG_REQUIRE(points && point_frame_ptr && centers && center_frame_ptr && row_ptr && (out_src || num_edges == 0),
             "pg_radius_graph_fill: null argument");
  if (num_edges == 0) return PG_OK;
  if (int rc = check_grid_args(num_frames, num_points)) return rc;
  return radius_call(wide_layout(num_frames), points, point_frame_ptr, centers, center_frame_ptr, num_frames, num_points,
                     num_centers, radius, nullptr, const_cast<int32_t*>(row_ptr), true, num_edges, out_src, out_dst,
                     num_edges, nullptr, s);
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
  if (int rc = check_grid_args(num_frames, num_points)) return rc;
  return with_cell_keys(num_frames, [&](auto L) {
    return radius_call(L, points, point_frame_ptr, centers, center_frame_ptr, num_frames, num_points, num_centers,
                       radius, scale_host, out_row_ptr, true, 0, out_src, out_dst, capacity, out_num_edges_host, s);
  });
}

namespace pg {
namespace {

// Buffers of one radius level of pg_multi_level_graph.
struct LevelBufs {
  int64_t parking;   // capacity of the hit parking buffer
  int32_t *cand, *cand_off, *counts, *ranges, *parked, *long_rows;
  void carve(Arena& a, int64_t kp_capacity, int64_t edge_capacity) {
    // candidates per row are ~6.5x the hits (27 cells of edge r against the ball of radius r); the parking buffer is
    // sized from the caller's edge capacity and its overflow is reported like an edge-buffer overflow
    parking = std::min<int64_t>(edge_capacity * 10 + 4096, (int64_t(1) << 31) - 1);
    cand = a.take<int32_t>(kp_capacity + 1);
    cand_off = a.take<int32_t>(kp_capacity + 1);
    counts = a.take<int32_t>(kp_capacity + 1);
    ranges = a.take<int32_t>(18 * kp_capacity);
    parked = a.take<int32_t>(parking);
    long_rows = a.take<int32_t>(kp_capacity);
  }
};

// One radius level of pg_multi_level_graph: candidates -> scan -> collect -> scan -> row sort, the number of centres
// and the number of edges staying on the device (`num_centers_dev`; E = out_row_ptr[kp_capacity]).
template <typename Key>
int radius_level_device(const SortedGrid<Key>& g, const GridSpec& spec, const uint32_t* bounds, double r2,
                        const float* centers, const int32_t* center_frame_ptr, int num_frames, int64_t kp_capacity,
                        const int32_t* num_centers_dev, LevelBufs& lb, void* cub_tmp, size_t cub_bytes,
                        int32_t* out_row_ptr, int32_t* out_src, int32_t* out_dst, int64_t capacity,
                        unsigned long long* total64, int* num_long, int* err, cudaStream_t s) {
  radius_candidates_kernel<Key><<<ceil_div(kp_capacity + 1, 128), 128, 0, s>>>(
      g, spec, bounds, centers, center_frame_ptr, num_frames, kp_capacity, num_centers_dev, lb.ranges, lb.cand,
      lb.counts, err);
  PG_LAUNCH_CHECK();
  size_t bytes = cub_bytes;
  PG_CUDA_OK(cub::DeviceScan::ExclusiveSum(cub_tmp, bytes, lb.cand, lb.cand_off, int(kp_capacity + 1), s));
  count_launch(2);
  radius_collect_kernel<<<ceil_div(kp_capacity * 32, 256), 256, 0, s>>>(
      g.pts, centers, kp_capacity, num_centers_dev, r2, lb.ranges, lb.cand_off, lb.parking, lb.parked, lb.counts, total64,
      err);
  PG_LAUNCH_CHECK();
  bytes = cub_bytes;
  PG_CUDA_OK(cub::DeviceScan::ExclusiveSum(cub_tmp, bytes, lb.counts, out_row_ptr, int(kp_capacity + 1), s));
  count_launch(2);
  // rows beyond the real number of centres are empty, so row_ptr[c] == E for every c >= K
  return sort_rows(out_row_ptr, kp_capacity, lb.parked, lb.cand_off, out_src, out_dst, capacity, lb.long_rows, num_long, s);
}

template <typename Key>
int multi_level_call(const KeyLayout<Key>& L, const float* xyz, const int32_t* frame_ptr, int num_frames,
                     int64_t num_points, const double* voxel_size_host, double radius0, double radius1,
                     int32_t* out_keypoint_idx, int64_t kp_capacity, int32_t* out_kp_frame_ptr, float* out_kp_xyz,
                     int32_t* out_row_ptr0, int32_t* out_src0, int32_t* out_dst0, int64_t capacity0,
                     int32_t* out_row_ptr1, int32_t* out_src1, int32_t* out_dst1, int64_t capacity1,
                     int64_t* out_sizes_host, cudaStream_t s) {
  const GridSpec vspec = voxel_spec(voxel_size_host, 0.5);
  GridSpec spec0, spec1;
  if (int rc = radius_spec(radius0, nullptr, &spec0)) return rc;
  if (int rc = radius_spec(radius1, nullptr, &spec1)) return rc;
  size_t cub_bytes = 0;
  if (int rc = grid_cub_bytes(num_points, L, &cub_bytes)) return rc;
  if (int rc = grid_cub_bytes(kp_capacity, L, &cub_bytes)) return rc;
  if (int rc = exclusive_sum_bytes(kp_capacity + 1, &cub_bytes)) return rc;
  CallHeader* hdr;
  uint32_t* bounds;   // per-frame minimum of the points (keypoint grid and level 0), then of the keypoints (level 1)
  GridBufs<Key> vb, b0, b1;
  LevelBufs lb0, lb1;
  void* cub_tmp;
  Temp ws;
  if (int rc = alloc_workspace(ws, s, [&](Arena& a) {
        hdr = a.take<CallHeader>(1);
        bounds = a.take<uint32_t>(6 * num_frames);
        vb.carve(a, num_points);
        b0.carve(a, num_points);
        b1.carve(a, kp_capacity);
        lb0.carve(a, kp_capacity, capacity0);
        lb1.carve(a, kp_capacity, capacity1);
        cub_tmp = a.take<char>(cub_bytes);
      }))
    return rc;
  uint32_t* kp_bounds = bounds + 3 * num_frames;
  PG_CUDA_OK(cudaMemsetAsync(hdr, 0, sizeof(CallHeader), s));
  PG_CUDA_OK(cudaMemsetAsync(bounds, 0xff, sizeof(uint32_t) * 6 * num_frames, s));
  if (int rc = frame_min(xyz, frame_ptr, num_frames, num_points, bounds, s)) return rc;
  // ---- keypoints (multi_layer_downsampling_select, graph_gen.py:49-90) ---------------------------
  SortedGrid<Key> vg;
  if (int rc = build_grid(xyz, frame_ptr, num_frames, vspec, L, bounds, vb, cub_tmp, cub_bytes, &hdr->err, s, &vg))
    return rc;
  voxel_keypoint_kernel<Key><<<ceil_div(num_points, 128), 128, 0, s>>>(vg, vspec, bounds, out_keypoint_idx, kp_capacity);
  PG_LAUNCH_CHECK();
  frame_ranges_kernel<Key><<<ceil_div(num_frames + 1, 128), 128, 0, s>>>(vg, num_frames, out_kp_frame_ptr);
  PG_LAUNCH_CHECK();
  const int32_t* k_dev = vg.num_cells;      // K = number of occupied voxels, on the device
  gather_keypoints_kernel<<<ceil_div(kp_capacity, 256), 256, 0, s>>>(xyz, out_keypoint_idx, k_dev, kp_capacity, out_kp_xyz);
  PG_LAUNCH_CHECK();
  // ---- level 0: original points -> keypoints (graph_gen.py:186-194, graph_level 0) -----------------
  SortedGrid<Key> g0;
  if (int rc = build_grid(xyz, frame_ptr, num_frames, spec0, L, bounds, b0, cub_tmp, cub_bytes, &hdr->err, s, &g0))
    return rc;
  if (int rc = radius_level_device(g0, spec0, bounds, radius0 * radius0, out_kp_xyz, out_kp_frame_ptr, num_frames,
                                   kp_capacity, k_dev, lb0, cub_tmp, cub_bytes, out_row_ptr0, out_src0, out_dst0,
                                   capacity0, &hdr->totals[0], &hdr->num_long[0], &hdr->err, s))
    return rc;
  // ---- level 1: keypoints -> keypoints (same scale: graph_gen.py:76-81 makes level 2 = level 1) ------
  if (int rc = frame_min(out_kp_xyz, out_kp_frame_ptr, num_frames, kp_capacity, kp_bounds, s)) return rc;
  SortedGrid<Key> g1;
  if (int rc = build_grid(out_kp_xyz, out_kp_frame_ptr, num_frames, spec1, L, kp_bounds, b1, cub_tmp, cub_bytes,
                          &hdr->err, s, &g1, k_dev))
    return rc;
  if (int rc = radius_level_device(g1, spec1, kp_bounds, radius1 * radius1, out_kp_xyz, out_kp_frame_ptr, num_frames,
                                   kp_capacity, k_dev, lb1, cub_tmp, cub_bytes, out_row_ptr1, out_src1, out_dst1,
                                   capacity1, &hdr->totals[1], &hdr->num_long[1], &hdr->err, s))
    return rc;
  // ---- the ONE host round trip: K, E0, E1 and the error word ---------------------------------------
  int32_t h_k = 0;
  CallHeader h;
  PG_CUDA_OK(cudaMemcpyAsync(&h_k, k_dev, sizeof(int32_t), cudaMemcpyDeviceToHost, s));
  PG_CUDA_OK(cudaMemcpyAsync(&h, hdr, sizeof(CallHeader), cudaMemcpyDeviceToHost, s));
  PG_CUDA_OK(cudaStreamSynchronize(s));
  if (h.err & kErrKeyWidth && !(h.err & (kErrFramePtr | kErrCenterPtr | kErrRange))) return kRetryWide;
  out_sizes_host[0] = h_k;
  out_sizes_host[1] = int64_t(h.totals[0]);
  out_sizes_host[2] = int64_t(h.totals[1]);
  if (h_k > kp_capacity) {
    // the downstream levels only saw the first kp_capacity keypoints: everything must be redone with a larger buffer
    set_error("keypoint buffer too small: need %d, capacity %lld", h_k, (long long)kp_capacity);
    return PG_ERR_CAPACITY;
  }
  if (int rc = graph_error(h.err)) return rc;
  if (h.totals[0] > 0x7fffffffull || h.totals[1] > 0x7fffffffull) {
    set_error("radius graph has more edges than int32 row_ptr can index; split the batch");
    return PG_ERR_RANGE;
  }
  if (int64_t(h.totals[0]) > capacity0 || int64_t(h.totals[1]) > capacity1) {
    set_error("edge buffer too small: need %llu / %llu, capacity %lld / %lld", h.totals[0], h.totals[1],
              (long long)capacity0, (long long)capacity1);
    return PG_ERR_CAPACITY;
  }
  return PG_OK;
}

}  // namespace
}  // namespace pg

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
  if (int rc = check_grid_args(num_frames, num_points)) return rc;
  return with_cell_keys(num_frames, [&](auto L) {
    return multi_level_call(L, xyz, frame_ptr, num_frames, num_points, voxel_size_host, radius0, radius1,
                            out_keypoint_idx, kp_capacity, out_kp_frame_ptr, out_kp_xyz, out_row_ptr0, out_src0,
                            out_dst0, capacity0, out_row_ptr1, out_src1, out_dst1, capacity1, out_sizes_host, s);
  });
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
template <typename Key>
__global__ void random_voxel_keys_kernel(const float* __restrict__ xyz, const int32_t* __restrict__ frame_ptr, int num_frames,
                                         int64_t n, const int32_t* __restrict__ origin_frame_ptr, int64_t num_origin,
                                         double vx, double vy, double vz, const double* __restrict__ shift,
                                         const uint32_t* __restrict__ bounds, KeyLayout<Key> L, Key* __restrict__ keys,
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
  }
  keys[i] = checked_key(L, uint32_t(f), idx[0], idx[1], idx[2], err);
  vals[i] = int32_t(i);
}

template <typename Key>
__global__ void head_flags_kernel(const Key* __restrict__ keys, int64_t n, int32_t* __restrict__ head) {
  const int64_t i = int64_t(blockIdx.x) * blockDim.x + threadIdx.x;
  if (i < n) head[i] = (i == 0 || keys[i] != keys[i - 1]) ? 1 : 0;
}

// second sort key of every voxel: (frame, smallest original point index) = dict insertion order of graph_gen.py:133-139
template <typename Key>
__global__ void voxel_first_keys_kernel(const Key* __restrict__ cell_key, KeyLayout<Key> L,
                                        const int32_t* __restrict__ cell_start, const int32_t* __restrict__ sorted_idx,
                                        const int32_t* __restrict__ num_cells, int64_t n, int num_frames,
                                        uint64_t* __restrict__ keys2, int32_t* __restrict__ vals2) {
  const int64_t v = int64_t(blockIdx.x) * blockDim.x + threadIdx.x;
  if (v >= n) return;
  vals2[v] = int32_t(v);
  if (v < *num_cells) keys2[v] = (uint64_t(L.frame(cell_key[v])) << 32) | uint64_t(uint32_t(sorted_idx[cell_start[v]]));
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
  out_frame_ptr[f] = lower_bound_key(keys2_sorted, *num_cells, uint64_t(f) << 32);
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

namespace pg {
namespace {

template <typename Key>
int random_keypoints_call(const KeyLayout<Key>& L, const float* xyz, const int32_t* frame_ptr, int num_frames,
                          int64_t num_points, const double* voxel_size_host, const double* shift_host,
                          const float* base_xyz, const int32_t* base_frame_ptr, int64_t n, const float* uniform,
                          int32_t* out_keypoint_idx, int64_t capacity, int32_t* out_kp_frame_ptr,
                          int64_t* out_num_keypoints_host, cudaStream_t s) {
  const int key2_bits = 32 + frame_bits(num_frames);
  size_t cub_bytes = 0, sort2 = 0;
  if (int rc = grid_cub_bytes(n, L, &cub_bytes)) return rc;
  PG_CUDA_OK(cub::DeviceRadixSort::SortPairs(nullptr, sort2, (const uint64_t*)nullptr, (uint64_t*)nullptr,
                                             (const int32_t*)nullptr, (int32_t*)nullptr, int(n), 0, key2_bits));
  cub_bytes = std::max(cub_bytes, sort2);
  CallHeader* hdr;
  uint32_t* bounds;
  double* shift = nullptr;
  GridBufs<Key> gb;   // keys, head flags and cell table of the voxel grid (its sorted point records stay unused)
  uint64_t *keys2a, *keys2b;
  int32_t *vals2a, *vals2b;
  void* cub_tmp;
  Temp ws;
  if (int rc = alloc_workspace(ws, s, [&](Arena& a) {
        hdr = a.take<CallHeader>(1);
        bounds = a.take<uint32_t>(3 * num_frames);
        if (shift_host) shift = a.take<double>(3 * num_frames);
        gb.carve(a, n);
        keys2a = a.take<uint64_t>(n);
        keys2b = a.take<uint64_t>(n);
        vals2a = a.take<int32_t>(n);
        vals2b = a.take<int32_t>(n);
        cub_tmp = a.take<char>(cub_bytes);
      }))
    return rc;
  PG_CUDA_OK(cudaMemsetAsync(hdr, 0, sizeof(CallHeader), s));
  PG_CUDA_OK(cudaMemsetAsync(bounds, 0xff, sizeof(uint32_t) * 3 * num_frames, s));
  if (shift_host != nullptr)
    PG_CUDA_OK(cudaMemcpyAsync(shift, shift_host, sizeof(double) * 3 * num_frames, cudaMemcpyHostToDevice, s));
  if (int rc = frame_min(xyz, frame_ptr, num_frames, num_points, bounds, s)) return rc;
  random_voxel_keys_kernel<Key><<<ceil_div(n, 256), 256, 0, s>>>(base_xyz, base_frame_ptr, num_frames, n, frame_ptr,
                                                                num_points, voxel_size_host[0], voxel_size_host[1],
                                                                voxel_size_host[2], shift, bounds, L, gb.keys_a,
                                                                gb.vals_a, &hdr->err);
  PG_LAUNCH_CHECK();
  size_t bytes = cub_bytes;
  PG_CUDA_OK(cub::DeviceRadixSort::SortPairs(cub_tmp, bytes, gb.keys_a, gb.keys_b, gb.vals_a, gb.vals_b, int(n), 0,
                                             L.end_bit, s));
  count_launch(radix_sort_launches(L.end_bit));
  head_flags_kernel<Key><<<ceil_div(n, 256), 256, 0, s>>>(gb.keys_b, n, gb.head);
  PG_LAUNCH_CHECK();
  bytes = cub_bytes;
  PG_CUDA_OK(cub::DeviceScan::InclusiveSum(cub_tmp, bytes, gb.head, gb.head_scan, int(n), s));
  count_launch(2);
  cell_table_kernel<Key><<<ceil_div(n, 256), 256, 0, s>>>(gb.keys_b, gb.head_scan, n, gb.cell_key, gb.cell_start);
  PG_LAUNCH_CHECK();
  const int32_t* num_cells = gb.head_scan + (n - 1);
  voxel_first_keys_kernel<Key><<<ceil_div(n, 256), 256, 0, s>>>(gb.cell_key, L, gb.cell_start, gb.vals_b, num_cells, n,
                                                               num_frames, keys2a, vals2a);
  PG_LAUNCH_CHECK();
  bytes = cub_bytes;
  PG_CUDA_OK(cub::DeviceRadixSort::SortPairs(cub_tmp, bytes, keys2a, keys2b, vals2a, vals2b, int(n), 0, key2_bits, s));
  count_launch(radix_sort_launches(key2_bits));
  random_pick_kernel<<<ceil_div(n, 256), 256, 0, s>>>(vals2b, gb.cell_start, gb.vals_b, num_cells, uniform, capacity,
                                                       out_keypoint_idx);
  PG_LAUNCH_CHECK();
  random_frame_ranges_kernel<<<ceil_div(num_frames + 1, 128), 128, 0, s>>>(keys2b, num_cells, num_frames,
                                                                            out_kp_frame_ptr);
  PG_LAUNCH_CHECK();
  int32_t h[2] = {0, 0};
  PG_CUDA_OK(cudaMemcpyAsync(&h[0], num_cells, sizeof(int32_t), cudaMemcpyDeviceToHost, s));
  PG_CUDA_OK(cudaMemcpyAsync(&h[1], &hdr->err, sizeof(int32_t), cudaMemcpyDeviceToHost, s));
  PG_CUDA_OK(cudaStreamSynchronize(s));
  if (int rc = graph_error(h[1])) return rc;
  *out_num_keypoints_host = h[0];
  if (h[0] > capacity) {
    set_error("keypoint buffer too small: need %d, capacity %lld", h[0], (long long)capacity);
    return PG_ERR_CAPACITY;
  }
  return PG_OK;
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
  if (int rc = check_grid_args(num_frames, num_points)) return rc;
  // the points that are voxelised; xyz only sets the grid origin
  PG_REQUIRE(num_base >= 1 && num_base < (int64_t(1) << 31), "num_base=%lld out of range", (long long)num_base);
  return with_cell_keys(num_frames, [&](auto L) {
    return random_keypoints_call(L, xyz, frame_ptr, num_frames, num_points, voxel_size_host, shift_host, base_xyz,
                                 base_frame_ptr, num_base, uniform, out_keypoint_idx, capacity, out_kp_frame_ptr,
                                 out_num_keypoints_host, s);
  });
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
