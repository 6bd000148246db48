// Points-in-polygons spatial join (SURVEY 8f row N2): which transcripts lie strictly inside which (buffered) cell
// outlines -- the tx-neighbors-bd candidate edges the scoring kernel consumes.
//
// Replaces cuspatial.quadtree_point_in_polygon behind
//   points_in_polygons(..., predicate='contains')   /root/reference/src/segger/geometry/query.py:21-100
//   setup_prediction_graph (shape modes)            /root/reference/src/segger/data/utils/neighbors.py:226-238
// The buffered variant (sgb_pip_buffered_count / _fill) takes the raw outlines plus one distance per ring and decides
// membership in the exact Minkowski sum of the ring with a disc (or its erosion for a negative distance) instead of
// asking geopandas .buffer (neighbors.py:229-231) for a grown polygon; sgb_polygon_props supplies the ring areas
// those distances are derived from.  Outlines with holes and several parts (sgb_pip_multi_count / _fill,
// sgb_polygon_props_multi) come in the GeoArrow / cuSpatial layout (ring_off, part_off, geom_off): one CTA per
// geometry, the even-odd rule over all of its rings.
//
// Layout: points are binned into a uniform grid over the polygons' bounding box (cell ~ a polygon's extent) and
// radix-sorted by cell (stable), so a polygon's bounding box covers a few contiguous ranges of the sorted point
// array (one per grid row).  One CTA per polygon keeps its ring in shared memory and streams those ranges; the
// inside test is the even-odd crossing rule evaluated in fp64 with explicitly rounded operations (the CPU oracle
// performs the same operations in the same order, so decisions agree bit for bit, boundary cases included).
// Two passes (count, exclusive scan, fill) and one stable sort by point id give a deterministic point-major,
// polygon-ascending edge list.
#include "sgb_api_internal.cuh"
#include "sgb_sort.cuh"

namespace sgb {
namespace {

constexpr int kPipThreads = 128;
constexpr int kPipMaxSmemVerts = 1024;          // rings longer than this are read from global memory
constexpr int kPipMaxSmemRings = 64;            // multi-ring geometries: ring descriptors beyond this come from global

struct PipGrid {
  double xmin, ymin, inv_cell;
  int nx, ny;
};

__device__ __forceinline__ int pip_cell(double v, double lo, double inv, int n) {
  const double c = floor((v - lo) * inv);
  if (!(c >= 0.0) || c >= static_cast<double>(n)) return -1;
  return static_cast<int>(c);
}

template <typename T>
__global__ void pip_cell_ids_kernel(const T* __restrict__ pts, int64_t n, PipGrid g, uint32_t* __restrict__ cell) {
  const int64_t i = static_cast<int64_t>(blockIdx.x) * blockDim.x + threadIdx.x;
  if (i >= n) return;
  const int cx = pip_cell(static_cast<double>(pts[2 * i]), g.xmin, g.inv_cell, g.nx);
  const int cy = pip_cell(static_cast<double>(pts[2 * i + 1]), g.ymin, g.inv_cell, g.ny);
  cell[i] = (cx < 0 || cy < 0) ? static_cast<uint32_t>(g.nx) * g.ny : static_cast<uint32_t>(cy) * g.nx + cx;
}

template <typename T>
__global__ void pip_gather_kernel(const T* __restrict__ pts, const uint32_t* __restrict__ perm, int64_t n,
                                  double2* __restrict__ sorted) {
  const int64_t i = static_cast<int64_t>(blockIdx.x) * blockDim.x + threadIdx.x;
  if (i >= n) return;
  const int64_t p = perm[i];
  sorted[i] = make_double2(static_cast<double>(pts[2 * p]), static_cast<double>(pts[2 * p + 1]));
}

// even-odd rule; an edge (a -> b) is crossed by the ray to +x iff exactly one endpoint is strictly above py and
// px < a.x + (py - a.y) * (b.x - a.x) / (b.y - a.y).  Operation order is part of the contract (see oracle).
__device__ __forceinline__ bool pip_inside(const double2* __restrict__ v, int nv, double px, double py) {
  bool in = false;
  double2 a = v[nv - 1];
  for (int e = 0; e < nv; ++e) {
    const double2 b = v[e];
    if ((a.y > py) != (b.y > py)) {
      const double t = __ddiv_rn(__dmul_rn(__dsub_rn(py, a.y), __dsub_rn(b.x, a.x)), __dsub_rn(b.y, a.y));
      if (px < __dadd_rn(a.x, t)) in = !in;
    }
    a = b;
  }
  return in;
}

// Squared distance from p to the ring: minimum over the edges a -> b of the point-to-segment distance, with
//   dx, dy = b - a;  ex, ey = p - a;  L = dx^2 + dy^2;  t = L > 0 ? clamp((ex dx + ey dy) / L, 0, 1) : 0
//   d2 = (ex - t dx)^2 + (ey - t dy)^2.
// Every operation is rounded explicitly in this order (the oracle evaluates the same text in numpy).  The loop stops
// early once the comparison with dd is decided: d2 < dd when `below`, d2 <= dd otherwise; the decision, not the
// returned value, is the contract.
__device__ __forceinline__ bool pip_ring_dist2_below(const double2* __restrict__ v, int nv, double px, double py, double dd,
                                                     bool strict) {
  double2 a = v[nv - 1];
  for (int e = 0; e < nv; ++e) {
    const double2 b = v[e];
    const double dx = __dsub_rn(b.x, a.x), dy = __dsub_rn(b.y, a.y);
    const double ex = __dsub_rn(px, a.x), ey = __dsub_rn(py, a.y);
    const double L = __dadd_rn(__dmul_rn(dx, dx), __dmul_rn(dy, dy));
    double t = 0.0;
    if (L > 0.0) t = fmin(fmax(__ddiv_rn(__dadd_rn(__dmul_rn(ex, dx), __dmul_rn(ey, dy)), L), 0.0), 1.0);
    const double qx = __dsub_rn(ex, __dmul_rn(t, dx)), qy = __dsub_rn(ey, __dmul_rn(t, dy));
    const double d2 = __dadd_rn(__dmul_rn(qx, qx), __dmul_rn(qy, qy));
    if (strict ? d2 < dd : d2 <= dd) return true;
    a = b;
  }
  return false;
}

// One ring of a multi-ring geometry: its first vertex relative to the geometry's first vertex, its vertex count
// after dropping a closing duplicate, and its box (empty for rings of fewer than 3 vertices, which match nothing).
struct PipRing {
  double4 box;
  int start, nv;
};

__device__ __forceinline__ PipRing pip_ring_info(const double2* __restrict__ verts, const int64_t* __restrict__ ring_off,
                                                 int64_t r, int64_t v0) {
  PipRing R;
  const int64_t s = ring_off[r];
  R.start = static_cast<int>(s - v0);
  R.nv = static_cast<int>(ring_off[r + 1] - s);
  if (R.nv >= 2) {
    const double2 f = verts[s], l = verts[s + R.nv - 1];
    if (f.x == l.x && f.y == l.y) --R.nv;
  }
  R.box = make_double4(INFINITY, INFINITY, -INFINITY, -INFINITY);
  if (R.nv >= 3)
    for (int i = 0; i < R.nv; ++i) {
      const double2 p = verts[s + i];
      R.box.x = fmin(R.box.x, p.x); R.box.y = fmin(R.box.y, p.y);
      R.box.z = fmax(R.box.z, p.x); R.box.w = fmax(R.box.w, p.y);
    }
  return R;
}

// Ring i of the geometry: from shared memory for the first kPipMaxSmemRings rings, recomputed from global memory
// beyond (an outline with that many holes or parts is rare).
__device__ __forceinline__ PipRing pip_ring_at(const PipRing* __restrict__ sring, int i, const double2* __restrict__ verts,
                                               const int64_t* __restrict__ ring_off, int64_t r0, int64_t v0) {
  return i < kPipMaxSmemRings ? sring[i] : pip_ring_info(verts, ring_off, r0 + i, v0);
}

// Membership of p in a multi-ring geometry: inside = XOR over its rings of the single-ring decision (ring box, then the
// even-odd test) -- the even-odd rule over all rings; with BUF the distance is the minimum over all rings, decided
// ring by ring with the same early exit as one ring.
template <bool BUF>
__device__ __forceinline__ bool pip_multi_hit(const PipRing* __restrict__ sring, int nring, const double2* __restrict__ vbase,
                                              const double2* __restrict__ verts, const int64_t* __restrict__ ring_off,
                                              int64_t r0, int64_t v0, double px, double py, double d, double dd) {
  bool inside = false;
  for (int i = 0; i < nring; ++i) {
    const PipRing R = pip_ring_at(sring, i, verts, ring_off, r0, v0);
    if (R.nv < 3 || px < R.box.x || px > R.box.z || py < R.box.y || py > R.box.w) continue;
    if (pip_inside(vbase + R.start, R.nv, px, py)) inside = !inside;
  }
  if (!BUF || d == 0.0) return inside;
  if (d > 0.0 && inside) return true;
  if (d < 0.0 && !inside) return false;
  for (int i = 0; i < nring; ++i) {
    const PipRing R = pip_ring_at(sring, i, verts, ring_off, r0, v0);
    if (R.nv >= 3 && pip_ring_dist2_below(vbase + R.start, R.nv, px, py, dd, d > 0.0)) return d > 0.0;
  }
  return d < 0.0;
}

// FILL == false: counts[poly] = number of points strictly inside;  FILL == true: writes (point, poly) at offsets[poly] + i
// BUF == true: ring `poly` is grown by dist[poly] (d > 0: inside or squared distance < d^2; d < 0: inside and squared
// distance > d^2; d == 0: inside); its box, and so the candidate range, grows by |d| (1 + 2^-20).  BUF == false is the
// plain join and compiles to the same code as before the buffered variant existed.
// MULTI == true: `poly` is geometry g of the polygon layout (rings part_off[geom_off[g]] .. part_off[geom_off[g + 1]],
// their vertices one contiguous range), tested with pip_multi_hit against the union of its ring boxes.  The geometry's
// vertices are staged in shared memory while they total at most kPipMaxSmemVerts, the first kPipMaxSmemRings ring
// descriptors always.  MULTI == false compiles to the same code as before the multi-ring variant existed.
template <bool FILL, bool BUF, bool MULTI = false>
__global__ void __launch_bounds__(kPipThreads)
pip_polygon_kernel(const double2* __restrict__ verts, const int64_t* __restrict__ ring_off, const double* __restrict__ dist,
                   int64_t n_poly, const double2* __restrict__ sorted, const uint32_t* __restrict__ perm,
                   const int32_t* __restrict__ cell_start, PipGrid g, int32_t* __restrict__ counts,
                   const int32_t* __restrict__ offsets, uint32_t* __restrict__ out_point, uint32_t* __restrict__ out_poly,
                   const int64_t* __restrict__ part_off = nullptr, const int64_t* __restrict__ geom_off = nullptr) {
  __shared__ double2 sv[kPipMaxSmemVerts];
  __shared__ double sbox[4];
  __shared__ int scount;
  __shared__ PipRing sring[MULTI ? kPipMaxSmemRings : 1];
  const int64_t poly = blockIdx.x;
  if (poly >= n_poly) return;
  int64_t v0, r0 = 0;
  int nv, nring = 0;
  if constexpr (MULTI) {
    r0 = part_off[geom_off[poly]];
    const int64_t r1 = part_off[geom_off[poly + 1]];
    nring = static_cast<int>(r1 - r0);
    v0 = ring_off[r0];
    nv = static_cast<int>(ring_off[r1] - v0);
  } else {
    v0 = ring_off[poly];
    nv = static_cast<int>(ring_off[poly + 1] - v0);
    // a closed ring that repeats its first vertex at the end: drop the duplicate (zero-length edge)
    if (nv >= 2) {
      const double2 f = verts[v0], l = verts[v0 + nv - 1];
      if (f.x == l.x && f.y == l.y) --nv;
    }
  }
  const bool in_smem = nv <= kPipMaxSmemVerts;
  if (threadIdx.x == 0) { scount = 0; sbox[0] = INFINITY; sbox[1] = INFINITY; sbox[2] = -INFINITY; sbox[3] = -INFINITY; }
  __syncthreads();
  if (in_smem)
    for (int i = threadIdx.x; i < nv; i += kPipThreads) sv[i] = verts[v0 + i];
  if constexpr (MULTI) {
    const int nstage = nring < kPipMaxSmemRings ? nring : kPipMaxSmemRings;
    for (int i = threadIdx.x; i < nstage; i += kPipThreads) sring[i] = pip_ring_info(verts, ring_off, r0 + i, v0);
    __syncthreads();
    // the geometry's box: the union of its ring boxes
    if (threadIdx.x == 0) {
      for (int i = 0; i < nring; ++i) {
        const double4 b = pip_ring_at(sring, i, verts, ring_off, r0, v0).box;
        sbox[0] = fmin(sbox[0], b.x); sbox[1] = fmin(sbox[1], b.y);
        sbox[2] = fmax(sbox[2], b.z); sbox[3] = fmax(sbox[3], b.w);
      }
    }
    __syncthreads();
    if (!(sbox[0] <= sbox[2])) {                        // no ring of 3 or more vertices: matches nothing
      if (!FILL && threadIdx.x == 0) counts[poly] = 0;
      return;
    }
  } else {
    // bounding box: one thread (rings are tens of vertices)
    if (threadIdx.x == 0) {
      for (int i = 0; i < nv; ++i) {
        const double2 p = verts[v0 + i];
        sbox[0] = fmin(sbox[0], p.x); sbox[1] = fmin(sbox[1], p.y);
        sbox[2] = fmax(sbox[2], p.x); sbox[3] = fmax(sbox[3], p.y);
      }
    }
    __syncthreads();
    if (nv < 3) {
      if (!FILL && threadIdx.x == 0) counts[poly] = 0;
      return;
    }
  }
  const double2* v = in_smem ? sv : verts + v0;
  const double d = BUF ? dist[poly] : 0.0;
  const double dd = __dmul_rn(d, d);
  const double grow = BUF ? __dmul_rn(fabs(d), 1.0 + 0x1p-20) : 0.0;
  const double bx0 = BUF ? __dsub_rn(sbox[0], grow) : sbox[0], by0 = BUF ? __dsub_rn(sbox[1], grow) : sbox[1];
  const double bx1 = BUF ? __dadd_rn(sbox[2], grow) : sbox[2], by1 = BUF ? __dadd_rn(sbox[3], grow) : sbox[3];
  int cx0 = pip_cell(bx0, g.xmin, g.inv_cell, g.nx), cx1 = pip_cell(bx1, g.xmin, g.inv_cell, g.nx);
  int cy0 = pip_cell(by0, g.ymin, g.inv_cell, g.ny), cy1 = pip_cell(by1, g.ymin, g.inv_cell, g.ny);
  // the grid covers the union of all (grown) polygon boxes, so the clamps only guard rounding at the upper edge
  cx0 = cx0 < 0 ? 0 : cx0; cy0 = cy0 < 0 ? 0 : cy0;
  cx1 = cx1 < 0 ? g.nx - 1 : cx1; cy1 = cy1 < 0 ? g.ny - 1 : cy1;
  const int base = FILL ? offsets[poly] : 0;
  int mine = 0;
  for (int cy = cy0; cy <= cy1; ++cy) {
    const int beg = cell_start[static_cast<int64_t>(cy) * g.nx + cx0];
    const int end = cell_start[static_cast<int64_t>(cy) * g.nx + cx1 + 1];
    for (int s = beg + threadIdx.x; s < end; s += kPipThreads) {
      const double2 p = sorted[s];
      bool hit;
      if constexpr (MULTI) {
        if (p.x < bx0 || p.x > bx1 || p.y < by0 || p.y > by1) continue;
        hit = pip_multi_hit<BUF>(sring, nring, v, verts, ring_off, r0, v0, p.x, p.y, d, dd);
      } else if (BUF) {
        if (p.x < bx0 || p.x > bx1 || p.y < by0 || p.y > by1) continue;
        const bool inside = !(p.x < sbox[0] || p.x > sbox[2] || p.y < sbox[1] || p.y > sbox[3]) && pip_inside(v, nv, p.x, p.y);
        if (d > 0.0) hit = inside || pip_ring_dist2_below(v, nv, p.x, p.y, dd, true);
        else if (d < 0.0) hit = inside && !pip_ring_dist2_below(v, nv, p.x, p.y, dd, false);
        else hit = inside;
      } else {
        if (p.x < sbox[0] || p.x > sbox[2] || p.y < sbox[1] || p.y > sbox[3]) continue;
        hit = pip_inside(v, nv, p.x, p.y);
      }
      if (hit) {
        if (FILL) {
          const int slot = atomicAdd(&scount, 1);
          out_point[base + slot] = perm[s];
          out_poly[base + slot] = static_cast<uint32_t>(poly);
        } else {
          ++mine;
        }
      }
    }
  }
  if (!FILL) {
    atomicAdd(&scount, mine);
    __syncthreads();
    if (threadIdx.x == 0) counts[poly] = scount;
  }
}

// One thread per ring, sequential and in a fixed order (the oracle repeats it in numpy):
//   area (signed, counter-clockwise > 0): x taken relative to the first vertex as GEOS's ring-area routine does,
//     A = 0.5 * sum_{i=1..n-1} (x_i - x_0) * (y_{i+1} - y_{i-1}),  y_n = y_0;
//   centroid: triangle fan from the first vertex, c_i = a_i x b_i with a_i = p_i - p_0, b_i = p_{i+1} - p_0,
//     centroid = p_0 + sum c_i (a_i + b_i) / (3 sum c_i);  a ring whose fan area is 0 reports its first vertex;
//   box: (xmin, ymin, xmax, ymax);  dist = sqrt(|A| / pi) * ratio.
// An empty ring has area 0, a NaN centroid and the empty box (+inf, +inf, -inf, -inf).
__global__ void polygon_props_kernel(const double2* __restrict__ verts, const int64_t* __restrict__ ring_off, int64_t n_poly,
                                     double ratio, double* __restrict__ area, double2* __restrict__ centroid,
                                     double4* __restrict__ box, double* __restrict__ dist) {
  const int64_t r = static_cast<int64_t>(blockIdx.x) * blockDim.x + threadIdx.x;
  if (r >= n_poly) return;
  const double2* v = verts + ring_off[r];
  int64_t n = ring_off[r + 1] - ring_off[r];
  if (n >= 2 && v[0].x == v[n - 1].x && v[0].y == v[n - 1].y) --n;
  double4 b = make_double4(INFINITY, INFINITY, -INFINITY, -INFINITY);
  double s = 0.0, a2 = 0.0, sx = 0.0, sy = 0.0;
  if (n > 0) {
    const double2 p0 = v[0];
    for (int64_t i = 0; i < n; ++i) {
      const double2 p = v[i];
      b.x = fmin(b.x, p.x); b.y = fmin(b.y, p.y); b.z = fmax(b.z, p.x); b.w = fmax(b.w, p.y);
    }
    if (n >= 3) {
      for (int64_t i = 1; i < n; ++i) {
        const double yn = v[i + 1 < n ? i + 1 : 0].y;
        s = __dadd_rn(s, __dmul_rn(__dsub_rn(v[i].x, p0.x), __dsub_rn(yn, v[i - 1].y)));
      }
      for (int64_t i = 1; i + 1 < n; ++i) {
        const double ax = __dsub_rn(v[i].x, p0.x), ay = __dsub_rn(v[i].y, p0.y);
        const double bx = __dsub_rn(v[i + 1].x, p0.x), by = __dsub_rn(v[i + 1].y, p0.y);
        const double c = __dsub_rn(__dmul_rn(ax, by), __dmul_rn(ay, bx));
        a2 = __dadd_rn(a2, c);
        sx = __dadd_rn(sx, __dmul_rn(c, __dadd_rn(ax, bx)));
        sy = __dadd_rn(sy, __dmul_rn(c, __dadd_rn(ay, by)));
      }
    }
  }
  const double A = __dmul_rn(s, 0.5);
  if (area) area[r] = A;
  if (box) box[r] = b;
  if (centroid) {
    double2 c = make_double2(NAN, NAN);
    if (n > 0) {
      c = v[0];
      if (a2 != 0.0) {
        const double den = __dmul_rn(3.0, a2);
        c = make_double2(__dadd_rn(c.x, __ddiv_rn(sx, den)), __dadd_rn(c.y, __ddiv_rn(sy, den)));
      }
    }
    centroid[r] = c;
  }
  if (dist) dist[r] = __dmul_rn(__dsqrt_rn(__ddiv_rn(fabs(A), 3.141592653589793)), ratio);
}

// One ring of polygon_props_kernel, in its operation order: signed area A, fan centroid c (the first vertex when the fan
// area is 0), box; returns the vertex count after dropping a closing duplicate (0: A = 0 and the box empty, c
// untouched).  polygon_props_kernel keeps its own copy of these lines so that its code stays what it was.
__device__ __forceinline__ int64_t ring_props(const double2* __restrict__ v, int64_t n, double& A, double2& c, double4& b) {
  if (n >= 2 && v[0].x == v[n - 1].x && v[0].y == v[n - 1].y) --n;
  b = make_double4(INFINITY, INFINITY, -INFINITY, -INFINITY);
  double s = 0.0, a2 = 0.0, sx = 0.0, sy = 0.0;
  if (n > 0) {
    const double2 p0 = v[0];
    for (int64_t i = 0; i < n; ++i) {
      const double2 p = v[i];
      b.x = fmin(b.x, p.x); b.y = fmin(b.y, p.y); b.z = fmax(b.z, p.x); b.w = fmax(b.w, p.y);
    }
    if (n >= 3) {
      for (int64_t i = 1; i < n; ++i) {
        const double yn = v[i + 1 < n ? i + 1 : 0].y;
        s = __dadd_rn(s, __dmul_rn(__dsub_rn(v[i].x, p0.x), __dsub_rn(yn, v[i - 1].y)));
      }
      for (int64_t i = 1; i + 1 < n; ++i) {
        const double ax = __dsub_rn(v[i].x, p0.x), ay = __dsub_rn(v[i].y, p0.y);
        const double bx = __dsub_rn(v[i + 1].x, p0.x), by = __dsub_rn(v[i + 1].y, p0.y);
        const double cr = __dsub_rn(__dmul_rn(ax, by), __dmul_rn(ay, bx));
        a2 = __dadd_rn(a2, cr);
        sx = __dadd_rn(sx, __dmul_rn(cr, __dadd_rn(ax, bx)));
        sy = __dadd_rn(sy, __dmul_rn(cr, __dadd_rn(ay, by)));
      }
    }
    c = p0;
    if (a2 != 0.0) {
      const double den = __dmul_rn(3.0, a2);
      c = make_double2(__dadd_rn(c.x, __ddiv_rn(sx, den)), __dadd_rn(c.y, __ddiv_rn(sy, den)));
    }
  }
  A = __dmul_rn(s, 0.5);
  return n;
}

// One thread per geometry of the polygon layout, rings in layout order (the oracle repeats it in numpy).  Ring r has
// the area A_r, centroid c_r and box of polygon_props_kernel and the weight w_r = |A_r| for the first ring of a part
// (its exterior) and -|A_r| for the others (its holes); empty rings are skipped.  With c_f the centroid of the first
// non-empty ring:
//   area W = sum w_r (left to right from 0);  centroid = c_f + (sum w_r (c_r - c_f)) / W, or c_f when W == 0;
//   box = union of the ring boxes;  dist = sqrt(|W| / pi) * ratio.
// A geometry with one non-empty ring so reproduces polygon_props_kernel bit for bit (|A|, c, box, dist); one with no
// vertices has area 0, a NaN centroid and the empty box.
__global__ void polygon_props_multi_kernel(const double2* __restrict__ verts, const int64_t* __restrict__ ring_off,
                                           const int64_t* __restrict__ part_off, const int64_t* __restrict__ geom_off,
                                           int64_t n_geom, double ratio, double* __restrict__ area,
                                           double2* __restrict__ centroid, double4* __restrict__ box, double* __restrict__ dist) {
  const int64_t gi = static_cast<int64_t>(blockIdx.x) * blockDim.x + threadIdx.x;
  if (gi >= n_geom) return;
  double4 b = make_double4(INFINITY, INFINITY, -INFINITY, -INFINITY);
  double W = 0.0, nx = 0.0, ny = 0.0;
  double2 cf = make_double2(NAN, NAN);
  bool any = false;
  for (int64_t q = geom_off[gi]; q < geom_off[gi + 1]; ++q) {
    for (int64_t r = part_off[q]; r < part_off[q + 1]; ++r) {
      double A;
      double2 c;
      double4 rb;
      if (ring_props(verts + ring_off[r], ring_off[r + 1] - ring_off[r], A, c, rb) == 0) continue;
      if (!any) { any = true; cf = c; }
      const double w = r == part_off[q] ? fabs(A) : -fabs(A);
      b.x = fmin(b.x, rb.x); b.y = fmin(b.y, rb.y); b.z = fmax(b.z, rb.z); b.w = fmax(b.w, rb.w);
      W = __dadd_rn(W, w);
      nx = __dadd_rn(nx, __dmul_rn(w, __dsub_rn(c.x, cf.x)));
      ny = __dadd_rn(ny, __dmul_rn(w, __dsub_rn(c.y, cf.y)));
    }
  }
  if (area) area[gi] = W;
  if (box) box[gi] = b;
  if (centroid) centroid[gi] = W != 0.0 ? make_double2(__dadd_rn(cf.x, __ddiv_rn(nx, W)), __dadd_rn(cf.y, __ddiv_rn(ny, W))) : cf;
  if (dist) dist[gi] = __dmul_rn(__dsqrt_rn(__ddiv_rn(fabs(W), 3.141592653589793)), ratio);
}

__global__ void pip_emit_kernel(const uint32_t* __restrict__ point, const uint32_t* __restrict__ poly, int64_t E,
                                int32_t* __restrict__ out, int64_t ld) {
  const int64_t i = static_cast<int64_t>(blockIdx.x) * blockDim.x + threadIdx.x;
  if (i >= E) return;
  out[i] = static_cast<int32_t>(point[i]);
  out[ld + i] = static_cast<int32_t>(poly[i]);
}

struct PipWs {
  uint32_t *cell, *skey, *perm;
  int32_t* cell_start;
  double2* sorted;
  int32_t *counts, *offsets;
  void* sort_ws;
  size_t sort_bytes, total;
};

PipWs pip_carve(void* ws, int64_t n, int64_t ncell, int64_t n_poly) {
  PipWs w{};
  char* p = static_cast<char*>(ws);
  const size_t nb = align_up(static_cast<size_t>(n > 0 ? n : 1) * 4);
  w.cell = reinterpret_cast<uint32_t*>(p); p += nb;
  w.skey = reinterpret_cast<uint32_t*>(p); p += nb;
  w.perm = reinterpret_cast<uint32_t*>(p); p += nb;
  w.cell_start = reinterpret_cast<int32_t*>(p); p += align_up(static_cast<size_t>(ncell + 2) * 4);
  w.sorted = reinterpret_cast<double2*>(p); p += align_up(static_cast<size_t>(n > 0 ? n : 1) * sizeof(double2));
  w.counts = reinterpret_cast<int32_t*>(p); p += align_up(static_cast<size_t>(n_poly + 1) * 4);
  w.offsets = reinterpret_cast<int32_t*>(p); p += align_up(static_cast<size_t>(n_poly + 2) * 4);
  w.sort_ws = p;
  const size_t s1 = sort_pairs_workspace_bytes(n), s2 = scan_workspace_bytes(n_poly + 1);
  w.sort_bytes = s1 > s2 ? s1 : s2;
  w.total = static_cast<size_t>(p - static_cast<char*>(ws)) + w.sort_bytes;
  return w;
}

PipGrid make_grid(double xmin, double ymin, double cell, int nx, int ny) { return PipGrid{xmin, ymin, 1.0 / cell, nx, ny}; }

}  // namespace
}  // namespace sgb

using namespace sgb;

extern "C" size_t sgb_pip_workspace_bytes(int64_t n_points, int64_t n_poly, int nx, int ny) {
  return pip_carve(nullptr, n_points, static_cast<int64_t>(nx) * ny, n_poly).total;
}

extern "C" size_t sgb_pip_fill_scratch_bytes(int64_t E) {
  return 4 * align_up(static_cast<size_t>(E > 0 ? E : 1) * 4) + sort_pairs_workspace_bytes(E);
}

namespace sgb {
namespace {

int pip_count_impl(const char* what, const void* points, int points_f64, int64_t n_points, const double* verts,
                   const int64_t* ring_off, const int64_t* part_off, const int64_t* geom_off, const double* dist, int64_t n_poly,
                   double xmin, double ymin, double cell, int nx, int ny, int32_t* total, void* ws, size_t ws_bytes,
                   cudaStream_t stream) {
  SGB_REQUIRE(n_points >= 0 && n_points < (int64_t(1) << 31) && n_poly >= 0 && n_poly < (int64_t(1) << 31), SGB_ERR_RANGE,
              "%s: size out of range", what);
  SGB_REQUIRE(nx >= 1 && ny >= 1 && static_cast<int64_t>(nx) * ny < (int64_t(1) << 28) && cell > 0.0, SGB_ERR_ARG, "%s: bad grid", what);
  SGB_REQUIRE(total && ws && (n_points == 0 || points) && (n_poly == 0 || (verts && ring_off && (!geom_off || part_off))),
              SGB_ERR_ARG, "%s: null tensor", what);
  SGB_REQUIRE(ws_bytes >= sgb_pip_workspace_bytes(n_points, n_poly, nx, ny), SGB_ERR_WORKSPACE, "%s: workspace too small", what);
  if (n_points == 0 || n_poly == 0) { cudaMemsetAsync(total, 0, sizeof(int32_t), stream); return check_launch(what); }
  const int64_t ncell = static_cast<int64_t>(nx) * ny;
  PipWs w = pip_carve(ws, n_points, ncell, n_poly);
  const PipGrid g = make_grid(xmin, ymin, cell, nx, ny);
  const unsigned nb = static_cast<unsigned>(ceil_div(n_points, 256));
  if (points_f64) pip_cell_ids_kernel<double><<<nb, 256, 0, stream>>>(static_cast<const double*>(points), n_points, g, w.cell);
  else pip_cell_ids_kernel<float><<<nb, 256, 0, stream>>>(static_cast<const float*>(points), n_points, g, w.cell);
  int rc = sort_pairs(w.cell, nullptr, w.skey, w.perm, n_points, bits_for(ncell + 1), w.sort_ws, w.sort_bytes, stream, true);
  if (rc != SGB_OK) return rc;
  rc = rowptr_from_sorted(w.skey, n_points, w.cell_start, ncell + 1, stream);     // cell_start[ncell] = first out-of-grid point
  if (rc != SGB_OK) return rc;
  if (points_f64) pip_gather_kernel<double><<<nb, 256, 0, stream>>>(static_cast<const double*>(points), w.perm, n_points, w.sorted);
  else pip_gather_kernel<float><<<nb, 256, 0, stream>>>(static_cast<const float*>(points), w.perm, n_points, w.sorted);
  if (geom_off && dist)
    pip_polygon_kernel<false, true, true><<<static_cast<unsigned>(n_poly), kPipThreads, 0, stream>>>(
        reinterpret_cast<const double2*>(verts), ring_off, dist, n_poly, w.sorted, w.perm, w.cell_start, g, w.counts, nullptr,
        nullptr, nullptr, part_off, geom_off);
  else if (geom_off)
    pip_polygon_kernel<false, false, true><<<static_cast<unsigned>(n_poly), kPipThreads, 0, stream>>>(
        reinterpret_cast<const double2*>(verts), ring_off, nullptr, n_poly, w.sorted, w.perm, w.cell_start, g, w.counts, nullptr,
        nullptr, nullptr, part_off, geom_off);
  else if (dist)
    pip_polygon_kernel<false, true><<<static_cast<unsigned>(n_poly), kPipThreads, 0, stream>>>(
        reinterpret_cast<const double2*>(verts), ring_off, dist, n_poly, w.sorted, w.perm, w.cell_start, g, w.counts, nullptr,
        nullptr, nullptr);
  else
    pip_polygon_kernel<false, false><<<static_cast<unsigned>(n_poly), kPipThreads, 0, stream>>>(
        reinterpret_cast<const double2*>(verts), ring_off, nullptr, n_poly, w.sorted, w.perm, w.cell_start, g, w.counts, nullptr,
        nullptr, nullptr);
  rc = exclusive_scan_i32(w.counts, w.offsets, n_poly, w.sort_ws, w.sort_bytes, stream);
  if (rc != SGB_OK) return rc;
  cudaMemcpyAsync(total, w.offsets + n_poly, sizeof(int32_t), cudaMemcpyDeviceToDevice, stream);
  return check_launch(what);
}

int pip_fill_impl(const char* what, const double* verts, const int64_t* ring_off, const int64_t* part_off, const int64_t* geom_off,
                  const double* dist, int64_t n_points, int64_t n_poly, double xmin, double ymin, double cell, int nx, int ny,
                  int64_t E, int32_t* edge_index, int64_t ld, void* ws, size_t ws_bytes, void* scratch, size_t scratch_bytes,
                  cudaStream_t stream) {
  SGB_REQUIRE(E >= 0 && E < (int64_t(1) << 31), SGB_ERR_RANGE, "%s: E out of range", what);
  if (E == 0) return SGB_OK;
  SGB_REQUIRE(verts && ring_off && (!geom_off || part_off) && edge_index && ws && scratch && ld >= E, SGB_ERR_ARG,
              "%s: null tensor", what);
  SGB_REQUIRE(ws_bytes >= sgb_pip_workspace_bytes(n_points, n_poly, nx, ny), SGB_ERR_WORKSPACE, "%s: workspace too small", what);
  SGB_REQUIRE(scratch_bytes >= sgb_pip_fill_scratch_bytes(E), SGB_ERR_WORKSPACE, "%s: scratch too small", what);
  const int64_t ncell = static_cast<int64_t>(nx) * ny;
  PipWs w = pip_carve(ws, n_points, ncell, n_poly);
  const PipGrid g = make_grid(xmin, ymin, cell, nx, ny);
  char* p = static_cast<char*>(scratch);
  const size_t eb = align_up(static_cast<size_t>(E) * 4);
  uint32_t* pt = reinterpret_cast<uint32_t*>(p); p += eb;
  uint32_t* pl = reinterpret_cast<uint32_t*>(p); p += eb;
  uint32_t* spt = reinterpret_cast<uint32_t*>(p); p += eb;
  uint32_t* spl = reinterpret_cast<uint32_t*>(p); p += eb;
  if (geom_off && dist)
    pip_polygon_kernel<true, true, true><<<static_cast<unsigned>(n_poly), kPipThreads, 0, stream>>>(
        reinterpret_cast<const double2*>(verts), ring_off, dist, n_poly, w.sorted, w.perm, w.cell_start, g, nullptr, w.offsets, pt,
        pl, part_off, geom_off);
  else if (geom_off)
    pip_polygon_kernel<true, false, true><<<static_cast<unsigned>(n_poly), kPipThreads, 0, stream>>>(
        reinterpret_cast<const double2*>(verts), ring_off, nullptr, n_poly, w.sorted, w.perm, w.cell_start, g, nullptr, w.offsets, pt,
        pl, part_off, geom_off);
  else if (dist)
    pip_polygon_kernel<true, true><<<static_cast<unsigned>(n_poly), kPipThreads, 0, stream>>>(
        reinterpret_cast<const double2*>(verts), ring_off, dist, n_poly, w.sorted, w.perm, w.cell_start, g, nullptr, w.offsets, pt, pl);
  else
    pip_polygon_kernel<true, false><<<static_cast<unsigned>(n_poly), kPipThreads, 0, stream>>>(
        reinterpret_cast<const double2*>(verts), ring_off, nullptr, n_poly, w.sorted, w.perm, w.cell_start, g, nullptr, w.offsets, pt,
        pl);
  // pairs are grouped by polygon (ascending) with arbitrary order inside a group; a stable sort by point id makes the
  // list point-major with polygons ascending per point -- independent of the order the atomics handed out slots
  int rc = sort_pairs(pt, pl, spt, spl, E, bits_for(n_points), p, sort_pairs_workspace_bytes(E), stream);
  if (rc != SGB_OK) return rc;
  pip_emit_kernel<<<static_cast<unsigned>(ceil_div(E, 256)), 256, 0, stream>>>(spt, spl, E, edge_index, ld);
  return check_launch(what);
}

}  // namespace
}  // namespace sgb

// Pass 1: bins the points, counts the contained points of every polygon, scans.  total[0] (device int32) = number of
// (point, polygon) pairs; the caller reads it back to size the output of sgb_pip_fill (same workspace, untouched between).
extern "C" int sgb_pip_count(const void* points, int points_f64, int64_t n_points, const double* verts, const int64_t* ring_off,
                             int64_t n_poly, double xmin, double ymin, double cell, int nx, int ny, int32_t* total, void* ws,
                             size_t ws_bytes, void* stream) {
  return pip_count_impl("pip_count", points, points_f64, n_points, verts, ring_off, nullptr, nullptr, nullptr, n_poly, xmin, ymin,
                        cell, nx, ny, total, ws, ws_bytes, static_cast<cudaStream_t>(stream));
}

// Pass 2: edge_index [2, E] int32 (row 0 = point index, row 1 = polygon index), point-major, polygon ascending.
// scratch: 4 * E uint32 (pairs + sorted pairs) + sort workspace for E keys: sgb_pip_fill_scratch_bytes(E).
extern "C" int sgb_pip_fill(const double* verts, const int64_t* ring_off, int64_t n_points, int64_t n_poly, double xmin, double ymin,
                            double cell, int nx, int ny, int64_t E, int32_t* edge_index, int64_t ld, void* ws, size_t ws_bytes,
                            void* scratch, size_t scratch_bytes, void* stream) {
  return pip_fill_impl("pip_fill", verts, ring_off, nullptr, nullptr, nullptr, n_points, n_poly, xmin, ymin, cell, nx, ny, E,
                       edge_index, ld, ws, ws_bytes, scratch, scratch_bytes, static_cast<cudaStream_t>(stream));
}

// The same two passes against rings grown by dist[poly] (device fp64, one per ring); the grid must cover the union of
// the boxes grown by |dist| (1 + 2^-20).
extern "C" int sgb_pip_buffered_count(const void* points, int points_f64, int64_t n_points, const double* verts,
                                      const int64_t* ring_off, const double* dist, int64_t n_poly, double xmin, double ymin,
                                      double cell, int nx, int ny, int32_t* total, void* ws, size_t ws_bytes, void* stream) {
  SGB_REQUIRE(n_poly <= 0 || dist, SGB_ERR_ARG, "pip_buffered_count: null dist");
  return pip_count_impl("pip_buffered_count", points, points_f64, n_points, verts, ring_off, nullptr, nullptr, dist, n_poly, xmin,
                        ymin, cell, nx, ny, total, ws, ws_bytes, static_cast<cudaStream_t>(stream));
}

extern "C" int sgb_pip_buffered_fill(const double* verts, const int64_t* ring_off, const double* dist, int64_t n_points,
                                     int64_t n_poly, double xmin, double ymin, double cell, int nx, int ny, int64_t E,
                                     int32_t* edge_index, int64_t ld, void* ws, size_t ws_bytes, void* scratch,
                                     size_t scratch_bytes, void* stream) {
  SGB_REQUIRE(E == 0 || dist, SGB_ERR_ARG, "pip_buffered_fill: null dist");
  return pip_fill_impl("pip_buffered_fill", verts, ring_off, nullptr, nullptr, dist, n_points, n_poly, xmin, ymin, cell, nx, ny,
                       E, edge_index, ld, ws, ws_bytes, scratch, scratch_bytes, static_cast<cudaStream_t>(stream));
}

// Per-ring area / centroid / box and, when `dist` is given, the buffer distance sqrt(|area| / pi) * ratio.
// area [n_poly], centroid [n_poly, 2], box [n_poly, 4] = (xmin, ymin, xmax, ymax), dist [n_poly]: fp64, each may be NULL.
extern "C" int sgb_polygon_props(const double* verts, const int64_t* ring_off, int64_t n_poly, double ratio, double* area,
                                 double* centroid, double* box, double* dist, void* stream_) {
  cudaStream_t stream = static_cast<cudaStream_t>(stream_);
  SGB_REQUIRE(n_poly >= 0 && n_poly < (int64_t(1) << 31), SGB_ERR_RANGE, "polygon_props: size out of range");
  if (n_poly == 0) return SGB_OK;
  SGB_REQUIRE(verts && ring_off, SGB_ERR_ARG, "polygon_props: null tensor");
  polygon_props_kernel<<<static_cast<unsigned>(ceil_div(n_poly, 128)), 128, 0, stream>>>(
      reinterpret_cast<const double2*>(verts), ring_off, n_poly, ratio, area, reinterpret_cast<double2*>(centroid),
      reinterpret_cast<double4*>(box), dist);
  return check_launch("polygon_props");
}

// The polygon layout (GeoArrow / cuSpatial): ring_off [R+1] vertices of ring r, part_off [Q+1] rings of part q (its
// exterior, then its holes), geom_off [n_geom+1] parts of geometry g.  Per geometry: net area (exteriors minus holes),
// centroid, box (union of the ring boxes) and, when `dist` is given, sqrt(|area| / pi) * ratio.  Outputs as
// sgb_polygon_props, each may be NULL.
extern "C" int sgb_polygon_props_multi(const double* verts, const int64_t* ring_off, const int64_t* part_off,
                                       const int64_t* geom_off, int64_t n_geom, double ratio, double* area, double* centroid,
                                       double* box, double* dist, void* stream_) {
  cudaStream_t stream = static_cast<cudaStream_t>(stream_);
  SGB_REQUIRE(n_geom >= 0 && n_geom < (int64_t(1) << 31), SGB_ERR_RANGE, "polygon_props_multi: size out of range");
  if (n_geom == 0) return SGB_OK;
  SGB_REQUIRE(verts && ring_off && part_off && geom_off, SGB_ERR_ARG, "polygon_props_multi: null tensor");
  polygon_props_multi_kernel<<<static_cast<unsigned>(ceil_div(n_geom, 128)), 128, 0, stream>>>(
      reinterpret_cast<const double2*>(verts), ring_off, part_off, geom_off, n_geom, ratio, area,
      reinterpret_cast<double2*>(centroid), reinterpret_cast<double4*>(box), dist);
  return check_launch("polygon_props_multi");
}

// The join of sgb_pip_count / _fill (same grid, workspace, scratch and output, with geometries in place of rings)
// against geometries of the polygon layout: a point is inside geometry g iff the even-odd rule over all rings of g
// says so.  `dist` [n_geom] (device fp64) or NULL: with it, geometry g is grown by dist[g] as sgb_pip_buffered_count
// grows one ring, the squared distance taken to the nearest edge of any of its rings; the grid must then cover the
// geometry boxes grown by |dist| (1 + 2^-20).
extern "C" int sgb_pip_multi_count(const void* points, int points_f64, int64_t n_points, const double* verts,
                                   const int64_t* ring_off, const int64_t* part_off, const int64_t* geom_off, const double* dist,
                                   int64_t n_geom, double xmin, double ymin, double cell, int nx, int ny, int32_t* total,
                                   void* ws, size_t ws_bytes, void* stream) {
  SGB_REQUIRE(n_geom <= 0 || (part_off && geom_off), SGB_ERR_ARG, "pip_multi_count: null offsets");
  return pip_count_impl("pip_multi_count", points, points_f64, n_points, verts, ring_off, part_off, geom_off, dist, n_geom,
                        xmin, ymin, cell, nx, ny, total, ws, ws_bytes, static_cast<cudaStream_t>(stream));
}

extern "C" int sgb_pip_multi_fill(const double* verts, const int64_t* ring_off, const int64_t* part_off, const int64_t* geom_off,
                                  const double* dist, int64_t n_points, int64_t n_geom, double xmin, double ymin, double cell,
                                  int nx, int ny, int64_t E, int32_t* edge_index, int64_t ld, void* ws, size_t ws_bytes,
                                  void* scratch, size_t scratch_bytes, void* stream) {
  SGB_REQUIRE(E == 0 || (part_off && geom_off), SGB_ERR_ARG, "pip_multi_fill: null offsets");
  return pip_fill_impl("pip_multi_fill", verts, ring_off, part_off, geom_off, dist, n_points, n_geom, xmin, ymin, cell, nx, ny,
                       E, edge_index, ld, ws, ws_bytes, scratch, scratch_bytes, static_cast<cudaStream_t>(stream));
}
