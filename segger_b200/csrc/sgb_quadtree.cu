// Quadtree tiling: QuadTreeTiling (/root/reference/src/segger/data/tiling.py:198-235, cuSpatial quadtree leaves of
// <= max_tile_size points) and the per-node tile label / training mask of TileFitDataset (data/tile_dataset.py:13-153),
// without cuSpatial.  The rules (restated in oracle/quadtree_ref.py, which the tests compare against bit for bit):
//
//   root    xmin, ymin = minimum over the points; side = max(xmax - xmin, ymax - ymin) (1 if 0); scale = side / 2^D.
//   edges   edge(c) = xmin + c * scale in fp64 (no FMA contraction), the ONE formula for every cell edge at every level,
//           so neighbouring leaves share bit-identical edges.
//   cell    ix = floor((x - xmin) / scale), corrected by +-1 so that edge(ix) <= x < edge(ix + 1), clamped to
//           [0, 2^D - 1]; key = Morton interleave of (ix, iy) with x in the even bits (2D <= 30 bits).
//   leaves  a quadrant at level L is split iff it holds > max_tile_size points and L < D; tiles are the non-empty
//           unsplit quadrants in Morton order.
//
// Build: key kernel -> stable radix sort of (key, id) over 2D bits -> level-synchronous split of a frontier of quadrant
// ranges over the sorted keys (each quadrant finds its 4 children by binary search inside its own range; children with
// > max_tile_size points form the next frontier, the others become leaves).  Frontier quadrants are disjoint, so a level
// holds at most F = floor(N / (max_tile_size + 1)) of them and the buffers are sized on the host without a per-level
// sync.  Every leaf covers one contiguous range of the sorted keys: flag its first position, and an exclusive scan of the
// flags numbers the leaves in Morton order and labels every sorted position at once.
#include <algorithm>

#include "sgb_api_internal.cuh"
#include "sgb_sort.cuh"

namespace sgb {
namespace {

constexpr int kT = 256;
constexpr int kBoundBlocks = 1024;    // partial min / max per block of the bounds pass

struct Quad {
  int32_t prefix, start, end;
};
struct Leaf {
  int32_t prefix, level, start, count;
};

__device__ __forceinline__ double edge_at(double lo, int64_t c, double scale) {
  return __dadd_rn(lo, __dmul_rn(static_cast<double>(c), scale));
}

__device__ __forceinline__ int32_t cell_of(double v, double lo, double scale, int D) {
  const int64_t nc = int64_t(1) << D;
  double f = floor(__ddiv_rn(__dsub_rn(v, lo), scale));
  f = fmin(fmax(f, -1.0), static_cast<double>(nc));
  int64_t c = static_cast<int64_t>(f);
  if (v < edge_at(lo, c, scale)) c -= 1;
  else if (v >= edge_at(lo, c + 1, scale)) c += 1;
  return static_cast<int32_t>(c < 0 ? 0 : (c > nc - 1 ? nc - 1 : c));
}

__device__ __forceinline__ uint32_t spread_bits(uint32_t v) {   // 16 bits -> even bit positions
  v &= 0xFFFFu;
  v = (v | (v << 8)) & 0x00FF00FFu;
  v = (v | (v << 4)) & 0x0F0F0F0Fu;
  v = (v | (v << 2)) & 0x33333333u;
  v = (v | (v << 1)) & 0x55555555u;
  return v;
}
__device__ __forceinline__ uint32_t compact_bits(uint32_t v) {  // even bit positions -> 16 bits
  v &= 0x55555555u;
  v = (v | (v >> 1)) & 0x33333333u;
  v = (v | (v >> 2)) & 0x0F0F0F0Fu;
  v = (v | (v >> 4)) & 0x00FF00FFu;
  v = (v | (v >> 8)) & 0x0000FFFFu;
  return v;
}

template <typename PT>
__device__ __forceinline__ uint32_t point_key(const PT* pos, int64_t i, const double* root, int D) {
  const int32_t ix = cell_of(static_cast<double>(pos[2 * i]), root[0], root[2], D);
  const int32_t iy = cell_of(static_cast<double>(pos[2 * i + 1]), root[1], root[2], D);
  return spread_bits(static_cast<uint32_t>(ix)) | (spread_bits(static_cast<uint32_t>(iy)) << 1);
}

// per-block (xmin, ymin, -xmax, -ymax) over a grid-stride slice of the points
template <typename PT>
__global__ void __launch_bounds__(kT) bounds_kernel(const PT* __restrict__ pos, int64_t n, double* __restrict__ part) {
  double v[4] = {INFINITY, INFINITY, INFINITY, INFINITY};
  for (int64_t i = static_cast<int64_t>(blockIdx.x) * blockDim.x + threadIdx.x; i < n; i += static_cast<int64_t>(gridDim.x) * blockDim.x) {
    const double x = static_cast<double>(pos[2 * i]), y = static_cast<double>(pos[2 * i + 1]);
    v[0] = fmin(v[0], x); v[1] = fmin(v[1], y); v[2] = fmin(v[2], -x); v[3] = fmin(v[3], -y);
  }
  __shared__ double s[4][kT / kWarp];
#pragma unroll
  for (int k = 0; k < 4; ++k) {
    for (int o = kWarp / 2; o > 0; o >>= 1) v[k] = fmin(v[k], __shfl_xor_sync(kFull, v[k], o));
    if ((threadIdx.x & (kWarp - 1)) == 0) s[k][threadIdx.x / kWarp] = v[k];
  }
  __syncthreads();
  if (threadIdx.x < 4) {
    double m = INFINITY;
    for (int w = 0; w < kT / kWarp; ++w) m = fmin(m, s[threadIdx.x][w]);
    part[4 * blockIdx.x + threadIdx.x] = m;
  }
}

// root = (xmin, ymin, scale)
__global__ void root_kernel(const double* __restrict__ part, int nparts, int D, double* __restrict__ root) {
  if (threadIdx.x != 0) return;
  double v[4] = {INFINITY, INFINITY, INFINITY, INFINITY};
  for (int b = 0; b < nparts; ++b)
    for (int k = 0; k < 4; ++k) v[k] = fmin(v[k], part[4 * b + k]);
  double xmin = 0.0, ymin = 0.0, side = 1.0;
  if (nparts > 0) {
    xmin = v[0]; ymin = v[1];
    side = fmax(__dsub_rn(-v[2], xmin), __dsub_rn(-v[3], ymin));
    if (!(side > 0.0)) side = 1.0;
  }
  root[0] = xmin; root[1] = ymin; root[2] = ldexp(side, -D);
}

// the root quadrant is the first frontier (> max_tile_size points) or the only leaf
__global__ void seed_kernel(int64_t n, int64_t max_tile, Quad* __restrict__ frontier, int32_t* __restrict__ fcount,
                            Leaf* __restrict__ leaves, int32_t* __restrict__ leaf_count, int32_t* __restrict__ flags) {
  if (threadIdx.x != 0) return;
  if (n > max_tile) {
    frontier[0] = Quad{0, 0, static_cast<int32_t>(n)};
    *fcount = 1;
  } else {
    leaves[0] = Leaf{0, 0, 0, static_cast<int32_t>(n)};
    *leaf_count = 1;
    flags[0] = 1;
  }
}

template <typename PT>
__global__ void __launch_bounds__(kT) key_kernel(const PT* __restrict__ pos, int64_t n, const double* __restrict__ root, int D,
                                                 uint32_t* __restrict__ keys) {
  const int64_t i = static_cast<int64_t>(blockIdx.x) * blockDim.x + threadIdx.x;
  if (i < n) keys[i] = point_key(pos, i, root, D);
}

__device__ __forceinline__ int32_t lower_bound_u32(const uint32_t* __restrict__ a, int32_t lo, int32_t hi, uint32_t v) {
  while (lo < hi) {
    const int32_t mid = lo + ((hi - lo) >> 1);
    if (__ldg(a + mid) < v) lo = mid + 1; else hi = mid;
  }
  return lo;
}

// one thread per frontier quadrant of level L: children at level L + 1
__global__ void __launch_bounds__(kT) split_kernel(const uint32_t* __restrict__ skeys, const Quad* __restrict__ in,
                                                   const int32_t* __restrict__ in_count, Quad* __restrict__ out,
                                                   int32_t* __restrict__ out_count, Leaf* __restrict__ leaves,
                                                   int32_t* __restrict__ leaf_count, int64_t leaf_cap,
                                                   int32_t* __restrict__ flags, int L, int D, int64_t max_tile) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= *in_count) return;
  const Quad q = in[i];
  const int shift = 2 * (D - L - 1);
  int32_t b[5];
  b[0] = q.start; b[4] = q.end;
  for (int c = 1; c < 4; ++c)
    b[c] = lower_bound_u32(skeys, b[c - 1], q.end, (static_cast<uint32_t>(q.prefix) * 4u + c) << shift);
  for (int c = 0; c < 4; ++c) {
    const int32_t cnt = b[c + 1] - b[c];
    if (cnt == 0) continue;
    const int32_t prefix = q.prefix * 4 + c;
    if (cnt > max_tile && L + 1 < D) {
      out[atomicAdd(out_count, 1)] = Quad{prefix, b[c], b[c + 1]};
    } else {
      const int32_t k = atomicAdd(leaf_count, 1);
      if (k < leaf_cap) leaves[k] = Leaf{prefix, L + 1, b[c], cnt};
      flags[b[c]] = 1;
    }
  }
}

// labels[perm[s]] = (inclusive scan of the leaf-start flags)[s] - 1
__global__ void __launch_bounds__(kT) fill_labels_kernel(const uint32_t* __restrict__ perm, const int32_t* __restrict__ flags,
                                                         const int32_t* __restrict__ scan, int64_t n, int32_t* __restrict__ labels,
                                                         int32_t* __restrict__ n_leaves) {
  const int64_t s = static_cast<int64_t>(blockIdx.x) * blockDim.x + threadIdx.x;
  if (s == 0) *n_leaves = scan[n];
  if (s < n) labels[perm[s]] = scan[s] + flags[s] - 1;
}

// leaf table in Morton order: id = number of leaves starting before this one
__global__ void __launch_bounds__(kT) leaf_table_kernel(const Leaf* __restrict__ leaves, const int32_t* __restrict__ leaf_count,
                                                        const int32_t* __restrict__ scan, const double* __restrict__ root, int D,
                                                        int32_t* __restrict__ meta, double* __restrict__ box) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= *leaf_count) return;
  const Leaf lf = leaves[i];
  const int id = scan[lf.start];
  const int64_t span = int64_t(1) << (D - lf.level);
  const int64_t qx = compact_bits(static_cast<uint32_t>(lf.prefix)), qy = compact_bits(static_cast<uint32_t>(lf.prefix) >> 1);
  meta[3 * id] = lf.prefix;
  meta[3 * id + 1] = lf.level;
  meta[3 * id + 2] = lf.count;
  box[4 * id] = edge_at(root[0], qx * span, root[2]);
  box[4 * id + 1] = edge_at(root[1], qy * span, root[2]);
  box[4 * id + 2] = edge_at(root[0], (qx + 1) * span, root[2]);
  box[4 * id + 3] = edge_at(root[1], (qy + 1) * span, root[2]);
}

// leaf whose quadrant contains the point's cell, or -1 (a cell of an empty quadrant)
template <typename PT>
__global__ void __launch_bounds__(kT) label_kernel(const PT* __restrict__ pts, int64_t n, const double* __restrict__ root, int D,
                                                   const int32_t* __restrict__ meta, int P, int32_t* __restrict__ labels) {
  const int64_t i = static_cast<int64_t>(blockIdx.x) * blockDim.x + threadIdx.x;
  if (i >= n) return;
  const uint64_t key = point_key(pts, i, root, D);
  int lo = 0, hi = P;                 // first leaf whose key range starts after `key`
  while (lo < hi) {
    const int mid = (lo + hi) >> 1;
    const uint64_t start = static_cast<uint64_t>(static_cast<uint32_t>(__ldg(meta + 3 * mid))) << (2 * (D - __ldg(meta + 3 * mid + 1)));
    if (start <= key) lo = mid + 1; else hi = mid;
  }
  int32_t out = -1;
  if (lo > 0) {
    const int l = lo - 1;
    const int sh = 2 * (D - meta[3 * l + 1]);
    const uint64_t end = (static_cast<uint64_t>(static_cast<uint32_t>(meta[3 * l])) + 1) << sh;
    if (key < end) out = l;
  }
  labels[i] = out;
}

// inside the own tile's box shrunk by that tile's margin (closed)
template <typename PT>
__global__ void __launch_bounds__(kT) fit_mask_kernel(const PT* __restrict__ pos, int64_t n, const int32_t* __restrict__ labels,
                                                      const double* __restrict__ box, const double* __restrict__ margins, int P,
                                                      uint8_t* __restrict__ mask) {
  const int64_t i = static_cast<int64_t>(blockIdx.x) * blockDim.x + threadIdx.x;
  if (i >= n) return;
  const int32_t l = labels[i];
  bool in = false;
  if (l >= 0 && l < P) {
    const double x = static_cast<double>(pos[2 * i]), y = static_cast<double>(pos[2 * i + 1]), m = margins[l];
    const double* b = box + 4 * l;
    in = x >= __dadd_rn(b[0], m) && x <= __dsub_rn(b[2], m) && y >= __dadd_rn(b[1], m) && y <= __dsub_rn(b[3], m);
  }
  mask[i] = in ? 1 : 0;
}

inline unsigned blocks_for(int64_t n) { return static_cast<unsigned>(ceil_div(n > 0 ? n : 1, kT)); }

int64_t frontier_cap(int64_t n, int64_t max_tile) { return n / (max_tile + 1); }

struct QtWs {
  double* part;
  uint32_t *keys, *skeys, *perm;
  int32_t *scan, *counts;   // counts: [0, D] frontier sizes per level, [D + 1] leaves emitted
  Quad *fa, *fb;
  Leaf* leaves;
  void *sort_ws, *scan_ws;
  size_t total;
};
QtWs carve(void* ws, int64_t n, int64_t max_tile, int D) {
  QtWs w{};
  const int64_t nn = n > 0 ? n : 1, F = frontier_cap(n, max_tile) > 0 ? frontier_cap(n, max_tile) : 1;
  char* p = static_cast<char*>(ws);
  size_t o = 0;
  auto take = [&](size_t bytes) { char* r = p + o; o += align_up(bytes); return r; };
  w.part = reinterpret_cast<double*>(take(sizeof(double) * 4 * kBoundBlocks));
  w.keys = reinterpret_cast<uint32_t*>(take(4 * nn));          // reused as the leaf-start flags after the sort
  w.skeys = reinterpret_cast<uint32_t*>(take(4 * nn));
  w.perm = reinterpret_cast<uint32_t*>(take(4 * nn));
  w.scan = reinterpret_cast<int32_t*>(take(4 * (nn + 1)));
  w.counts = reinterpret_cast<int32_t*>(take(4 * (D + 2)));
  w.fa = reinterpret_cast<Quad*>(take(sizeof(Quad) * F));
  w.fb = reinterpret_cast<Quad*>(take(sizeof(Quad) * F));
  w.leaves = reinterpret_cast<Leaf*>(take(sizeof(Leaf) * std::max<int64_t>(1, sgb_quadtree_max_leaves(n, max_tile, D))));
  w.sort_ws = take(sort_pairs_workspace_bytes(n));
  w.scan_ws = take(scan_workspace_bytes(n));
  w.total = o;
  return w;
}

}  // namespace
}  // namespace sgb

using namespace sgb;

extern "C" int64_t sgb_quadtree_max_leaves(int64_t n, int64_t max_tile_size, int max_depth) {
  if (n <= 0 || max_tile_size < 1 || max_depth < 1) return 0;
  return std::min<int64_t>(n, 1 + 3 * int64_t(max_depth) * frontier_cap(n, max_tile_size));
}

extern "C" size_t sgb_quadtree_workspace_bytes(int64_t n, int64_t max_tile_size, int max_depth) {
  if (n < 0 || max_tile_size < 1 || max_depth < 1 || max_depth > 15) return 0;
  return carve(nullptr, n, max_tile_size, max_depth).total;
}

extern "C" int sgb_quadtree_build(const void* pos, int pos_f64, int64_t n, int64_t max_tile_size, int max_depth, int32_t* labels,
                                  double* root, int32_t* leaf_meta, double* leaf_box, int64_t leaf_cap, int32_t* n_leaves,
                                  void* ws, size_t ws_bytes, void* stream_) {
  cudaStream_t stream = static_cast<cudaStream_t>(stream_);
  SGB_REQUIRE(n >= 0 && n < (int64_t(1) << 31) - 1, SGB_ERR_RANGE, "quadtree_build: n=%lld out of range", (long long)n);
  SGB_REQUIRE(max_depth >= 1 && max_depth <= 15 && max_tile_size >= 1, SGB_ERR_ARG,
              "quadtree_build: max_depth=%d (1..15), max_tile_size=%lld (>= 1)", max_depth, (long long)max_tile_size);
  SGB_REQUIRE(root && n_leaves && (n == 0 || (pos && labels && leaf_meta && leaf_box)), SGB_ERR_ARG, "quadtree_build: null argument");
  SGB_REQUIRE(leaf_cap >= sgb_quadtree_max_leaves(n, max_tile_size, max_depth), SGB_ERR_ARG,
              "quadtree_build: leaf_cap=%lld < sgb_quadtree_max_leaves=%lld", (long long)leaf_cap,
              (long long)sgb_quadtree_max_leaves(n, max_tile_size, max_depth));
  SGB_REQUIRE(ws && ws_bytes >= sgb_quadtree_workspace_bytes(n, max_tile_size, max_depth), SGB_ERR_WORKSPACE,
              "quadtree_build: workspace too small");
  const int D = max_depth;
  QtWs w = carve(ws, n, max_tile_size, D);
  int32_t* leaf_count = w.counts + D + 1;
  cudaMemsetAsync(w.counts, 0, sizeof(int32_t) * (D + 2), stream);
  const int nparts = n > 0 ? static_cast<int>(std::min<int64_t>(kBoundBlocks, ceil_div(n, kT))) : 0;
  if (nparts > 0) {
    if (pos_f64) bounds_kernel<double><<<nparts, kT, 0, stream>>>(static_cast<const double*>(pos), n, w.part);
    else bounds_kernel<float><<<nparts, kT, 0, stream>>>(static_cast<const float*>(pos), n, w.part);
  }
  root_kernel<<<1, 32, 0, stream>>>(w.part, nparts, D, root);
  if (n == 0) {
    cudaMemsetAsync(n_leaves, 0, sizeof(int32_t), stream);
    return check_launch("quadtree_build(empty)");
  }
  if (pos_f64) key_kernel<double><<<blocks_for(n), kT, 0, stream>>>(static_cast<const double*>(pos), n, root, D, w.keys);
  else key_kernel<float><<<blocks_for(n), kT, 0, stream>>>(static_cast<const float*>(pos), n, root, D, w.keys);
  int rc = sort_pairs(w.keys, nullptr, w.skeys, w.perm, n, 2 * D, w.sort_ws, sort_pairs_workspace_bytes(n), stream);
  if (rc != SGB_OK) return rc;
  int32_t* flags = reinterpret_cast<int32_t*>(w.keys);       // the unsorted keys are dead after the sort
  cudaMemsetAsync(flags, 0, sizeof(int32_t) * n, stream);
  seed_kernel<<<1, 32, 0, stream>>>(n, max_tile_size, w.fa, w.counts, w.leaves, leaf_count, flags);
  const int64_t F = frontier_cap(n, max_tile_size);
  const int64_t cap = sgb_quadtree_max_leaves(n, max_tile_size, D);
  if (F > 0) {
    for (int L = 0; L < D; ++L) {
      const Quad* in = (L & 1) ? w.fb : w.fa;
      Quad* out = (L & 1) ? w.fa : w.fb;
      split_kernel<<<L == 0 ? 1u : blocks_for(F), kT, 0, stream>>>(w.skeys, in, w.counts + L, out, w.counts + L + 1, w.leaves,
                                                                 leaf_count, cap, flags, L, D, max_tile_size);
    }
  }
  rc = exclusive_scan_i32(flags, w.scan, n, w.scan_ws, scan_workspace_bytes(n), stream);
  if (rc != SGB_OK) return rc;
  fill_labels_kernel<<<blocks_for(n), kT, 0, stream>>>(w.perm, flags, w.scan, n, labels, n_leaves);
  leaf_table_kernel<<<blocks_for(cap), kT, 0, stream>>>(w.leaves, leaf_count, w.scan, root, D, leaf_meta, leaf_box);
  return check_launch("quadtree_build");
}

extern "C" int sgb_quadtree_label(const void* pts, int pos_f64, int64_t n, const double* root, int max_depth, const int32_t* leaf_meta,
                                  int n_leaves, int32_t* labels, void* stream_) {
  cudaStream_t stream = static_cast<cudaStream_t>(stream_);
  SGB_REQUIRE(n >= 0 && n < (int64_t(1) << 31) && n_leaves >= 0, SGB_ERR_RANGE, "quadtree_label: n=%lld out of range", (long long)n);
  SGB_REQUIRE(max_depth >= 1 && max_depth <= 15, SGB_ERR_ARG, "quadtree_label: max_depth=%d (1..15)", max_depth);
  if (n == 0) return SGB_OK;
  SGB_REQUIRE(pts && root && labels && (n_leaves == 0 || leaf_meta), SGB_ERR_ARG, "quadtree_label: null argument");
  if (pos_f64)
    label_kernel<double><<<blocks_for(n), kT, 0, stream>>>(static_cast<const double*>(pts), n, root, max_depth, leaf_meta, n_leaves, labels);
  else
    label_kernel<float><<<blocks_for(n), kT, 0, stream>>>(static_cast<const float*>(pts), n, root, max_depth, leaf_meta, n_leaves, labels);
  return check_launch("quadtree_label");
}

extern "C" int sgb_quadtree_fit_mask(const void* pos, int pos_f64, int64_t n, const int32_t* labels, const double* leaf_box,
                                     const double* margins, int n_leaves, uint8_t* mask, void* stream_) {
  cudaStream_t stream = static_cast<cudaStream_t>(stream_);
  SGB_REQUIRE(n >= 0 && n < (int64_t(1) << 31) && n_leaves >= 0, SGB_ERR_RANGE, "quadtree_fit_mask: n=%lld out of range", (long long)n);
  if (n == 0) return SGB_OK;
  SGB_REQUIRE(pos && labels && mask && (n_leaves == 0 || (leaf_box && margins)), SGB_ERR_ARG, "quadtree_fit_mask: null argument");
  if (pos_f64)
    fit_mask_kernel<double><<<blocks_for(n), kT, 0, stream>>>(static_cast<const double*>(pos), n, labels, leaf_box, margins, n_leaves, mask);
  else
    fit_mask_kernel<float><<<blocks_for(n), kT, 0, stream>>>(static_cast<const float*>(pos), n, labels, leaf_box, margins, n_leaves, mask);
  return check_launch("quadtree_fit_mask");
}
