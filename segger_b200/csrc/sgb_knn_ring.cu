// 2-D k-nearest-neighbour search for any 1 <= k <= 1024 and any radius in (0, +inf]: exact ring search on a grid.
// Serves the inputs the register kernel of sgb_knn.cu does not hold (k > 32, no radius cap), with the same outputs,
// arithmetic contract and order: d^2 = fl(fl(dx*dx) + fl(dy*dy)) in float64, accepted iff d^2 < max_dist^2, rows by
// (d^2, original index), padded with n_points.  Kept in its own translation unit so the register kernel compiles
// to the same instructions as before.
//
// Layout: the grid spans the points only and its cell is sized from their mean density; the points are binned and
// sorted by cell exactly as for the register kernel (sgb_knn.cuh).  A warp per query visits square rings of cells
// around the query's cell, keeps its top-k in shared memory and stops as soon as no unscanned point can enter it.
#include "sgb_knn.cuh"

namespace sgb {
namespace {
// ---- ring search: 1 <= k <= 1024, max_dist in (0, +inf] ----
constexpr int kRingMaxK = 1024;

struct RingGrid {
  Grid g;
  double cell;   // cell edge
  double slack;  // absolute error bound of the binning and of the cell-edge positions (see ring_bound)
};

// warps per CTA: the lists of one CTA total at most 2,048 entries (24 KB of shared memory)
constexpr int ring_warps(int K) { return K <= 256 ? 8 : 2048 / K; }

// A lower bound on the d^2 the kernel computes for any point outside the scanned square [cx - rho, cx + rho] x
// [cy - rho, cy + rho] of cells, +inf once the square covers the grid.  Such a point lies beyond a side of the square
// that is not on the grid border, so at least `gap` from the query, where gap is measured to the cell edges (not from
// the clamped cell index: the query may lie outside the points' box).  cell_key_kernel rounds floor((v - lo) * inv)
// and the edges xmin + c * cell are rounded too, a few ulps of the coordinates' magnitude in all; `slack` and the
// 2^-40 factors cover that and the rounding of d^2 with a wide margin.  Too small a bound only costs another ring.
__device__ __forceinline__ double ring_bound(const RingGrid& rg, double qx, double qy, int cx, int cy, int rho) {
  double gap = INFINITY;
  if (cx - rho > 0) gap = fmin(gap, qx - (rg.g.xmin + static_cast<double>(cx - rho) * rg.cell));
  if (cx + rho < rg.g.nx - 1) gap = fmin(gap, rg.g.xmin + static_cast<double>(cx + rho + 1) * rg.cell - qx);
  if (cy - rho > 0) gap = fmin(gap, qy - (rg.g.ymin + static_cast<double>(cy - rho) * rg.cell));
  if (cy + rho < rg.g.ny - 1) gap = fmin(gap, rg.g.ymin + static_cast<double>(cy + rho + 1) * rg.cell - qy);
  if (gap == INFINITY) return INFINITY;
  const double gl = gap * (1.0 - 0x1p-40) - (rg.slack + (fabs(qx) + fabs(qy)) * 0x1p-40);
  return gl > 0.0 ? gl * gl * (1.0 - 0x1p-40) : 0.0;
}

// One warp's top-k list in shared memory, sorted by (d^2, idx): entries [0, cnt), cnt <= k.  kd / ki is the k-th
// entry once the list is full, else +inf / INT_MAX, so a candidate enters iff it is below it.
struct RingList {
  double* d;
  int* i;
  double* bd;   // the sorted survivors of one 32-candidate batch
  int* bi;
  int cnt;
  double kd;
  int ki;
};

// Scans sorted[beg, end) 32 candidates at a time: a ballot keeps those below the k-th key (and inside the radius),
// a bitonic sort across the warp orders them, and they are merged into the list.
__device__ __forceinline__ void ring_scan(RingList& L, const double2* __restrict__ sorted, const uint32_t* __restrict__ perm,
                                          int beg, int end, double qx, double qy, double r2, int k, int lane) {
  for (int b = beg; b < end; b += 32) {
    const int s = b + lane;
    double d2 = INFINITY;
    int idx = 0x7fffffff;
    bool take = false;
    if (s < end) {
      const double2 p = sorted[s];
      const double dx = __dsub_rn(p.x, qx), dy = __dsub_rn(p.y, qy);
      d2 = __dadd_rn(__dmul_rn(dx, dx), __dmul_rn(dy, dy));
      if (d2 < r2 && d2 <= L.kd) {
        idx = static_cast<int>(perm[s]);
        take = knn_less(d2, idx, L.kd, L.ki);
      }
    }
    const unsigned mask = __ballot_sync(kFull, take);
    if (mask == 0) continue;
    if (!take) { d2 = INFINITY; idx = 0x7fffffff; }
#pragma unroll
    for (int size = 2; size <= 32; size <<= 1) {
#pragma unroll
      for (int stride = size >> 1; stride > 0; stride >>= 1) {
        const double od = __shfl_xor_sync(kFull, d2, stride);
        const int oi = __shfl_xor_sync(kFull, idx, stride);
        const bool keep_min = ((lane & stride) == 0) == ((lane & size) == 0);
        const bool other_less = knn_less(od, oi, d2, idx);
        if (keep_min ? other_less : !other_less) { d2 = od; idx = oi; }
      }
    }
    const int m = __popc(mask), cnt = L.cnt;
    // survivor `lane` goes to lane + (number of list entries below it)
    int pos = lane;
    if (lane < m) {
      L.bd[lane] = d2; L.bi[lane] = idx;
      int lo = 0, hi = cnt;
      while (lo < hi) {
        const int mid = (lo + hi) >> 1;
        if (knn_less(L.d[mid], L.i[mid], d2, idx)) lo = mid + 1; else hi = mid;
      }
      pos += lo;
    }
    __syncwarp();
    // list entry e moves up by the number of survivors below it; chunks of 32 from the top down, so an entry is read
    // before anything lands on it.  The shift grows with the position: a chunk whose lowest entry stays ends the loop.
    for (int base = (cnt - 1) & ~31; base >= 0; base -= 32) {
      const int e = base + lane;
      double ed = 0.0;
      int ei = 0, sh = 0;
      if (e < cnt) {
        ed = L.d[e]; ei = L.i[e];
        int hi = m;
        while (sh < hi) {
          const int mid = (sh + hi) >> 1;
          if (knn_less(L.bd[mid], L.bi[mid], ed, ei)) sh = mid + 1; else hi = mid;
        }
      }
      __syncwarp();
      if (sh > 0 && e + sh < k) { L.d[e + sh] = ed; L.i[e + sh] = ei; }
      __syncwarp();
      if (__shfl_sync(kFull, sh, 0) == 0) break;
    }
    if (lane < m && pos < k) { L.d[pos] = d2; L.i[pos] = idx; }
    L.cnt = min(cnt + m, k);
    __syncwarp();
    if (L.cnt == k) { L.kd = L.d[k - 1]; L.ki = L.i[k - 1]; }
  }
}

// K = shared-memory list capacity (k <= K); one warp per query
template <int K, typename T>
__global__ void __launch_bounds__(32 * ring_warps(K))
knn_ring_kernel(const double2* __restrict__ sorted, const uint32_t* __restrict__ perm, const int32_t* __restrict__ cell_start,
                RingGrid rg, const T* __restrict__ query, int64_t n_query, int64_t n_points, int k, double r2,
                int64_t* __restrict__ table, int32_t* __restrict__ count) {
  constexpr int W = ring_warps(K);
  __shared__ double s_d[W][K];
  __shared__ int s_i[W][K];
  __shared__ double s_bd[W][32];
  __shared__ int s_bi[W][32];
  const int lane = threadIdx.x & 31, w = threadIdx.x >> 5;
  const int64_t t = static_cast<int64_t>(blockIdx.x) * W + w;
  if (t >= n_query) return;
  double qx, qy;
  int64_t qrow;
  if (query) {
    qx = static_cast<double>(query[2 * t]); qy = static_cast<double>(query[2 * t + 1]); qrow = t;
  } else {
    const double2 q = sorted[t];
    qx = q.x; qy = q.y; qrow = perm[t];
  }
  RingList L{s_d[w], s_i[w], s_bd[w], s_bi[w], 0, INFINITY, 0x7fffffff};
  const Grid& g = rg.g;
  const int cx = cell_coord(qx, g.xmin, g.inv_cell, g.nx);
  const int cy = cell_coord(qy, g.ymin, g.inv_cell, g.ny);
  const int rho_max = max(max(cx, g.nx - 1 - cx), max(cy, g.ny - 1 - cy));
  for (int rho = 0; rho <= rho_max; ++rho) {
    // the ring: rows cy - rho and cy + rho over [cx - rho, cx + rho] (one contiguous range each), then the cells of
    // columns cx - rho and cx + rho strictly between those rows
    const int x0 = max(cx - rho, 0), x1 = min(cx + rho, g.nx - 1);
    for (int side = 0; side < (rho > 0 ? 2 : 1); ++side) {
      const int yy = side ? cy + rho : cy - rho;
      if (yy < 0 || yy >= g.ny) continue;
      const int64_t row = static_cast<int64_t>(yy) * g.nx;
      ring_scan(L, sorted, perm, cell_start[row + x0], cell_start[row + x1 + 1], qx, qy, r2, k, lane);
    }
    if (rho > 0) {
      const int y0 = max(cy - rho + 1, 0), y1 = min(cy + rho - 1, g.ny - 1);
      for (int side = 0; side < 2; ++side) {
        const int xx = side ? cx + rho : cx - rho;
        if (xx < 0 || xx >= g.nx) continue;
        for (int yy = y0; yy <= y1; ++yy) {
          const int64_t c = static_cast<int64_t>(yy) * g.nx + xx;
          ring_scan(L, sorted, perm, cell_start[c], cell_start[c + 1], qx, qy, r2, k, lane);
        }
      }
    }
    // every unscanned point has d^2 >= bound: none is inside the radius, or none can displace the k-th entry
    // (strictly below: a tie at the k-th distance would be decided by the index)
    const double bound = ring_bound(rg, qx, qy, cx, cy, rho);
    if (bound >= r2 || (L.cnt == k && L.kd < bound)) break;
  }
  for (int j = lane; j < k; j += 32) table[qrow * k + j] = j < L.cnt ? static_cast<int64_t>(L.i[j]) : n_points;
  if (count && lane == 0) count[qrow] = L.cnt;
}

template <typename T>
int run_knn_ring(const sgb_knn_plan* plan, const T* points, const T* query, int64_t* table, int32_t* count, void* ws,
                 cudaStream_t stream) {
  const int64_t n = plan->n_points, nq = plan->n_query;
  KnnWs w = knn_carve(ws, n, plan->nx * plan->ny);
  Grid g{plan->xmin, plan->ymin, 1.0 / plan->cell, static_cast<int>(plan->nx), static_cast<int>(plan->ny)};
  const int rc = bin_points<T>(plan, points, w, g, stream);
  if (rc != SGB_OK) return rc;
  // magnitude bound of every coordinate and cell edge of the grid, times 2^-40
  const double span = fabs(plan->xmin) + fabs(plan->ymin) + static_cast<double>(plan->nx + plan->ny + 2) * plan->cell;
  const RingGrid rg{g, plan->cell, span * 0x1p-40};
  const double r2 = plan->max_dist * plan->max_dist;
  const int k = plan->k;
#define SGB_RING_LAUNCH(KK)                                                                                       \
  knn_ring_kernel<KK, T><<<static_cast<unsigned>(ceil_div(nq, ring_warps(KK))), 32 * ring_warps(KK), 0, stream>>>( \
      w.sorted, w.perm, w.cell_start, rg, query, nq, n, k, r2, table, count)
  if (k <= 64) SGB_RING_LAUNCH(64);
  else if (k <= 128) SGB_RING_LAUNCH(128);
  else if (k <= 256) SGB_RING_LAUNCH(256);
  else if (k <= 512) SGB_RING_LAUNCH(512);
  else SGB_RING_LAUNCH(1024);
#undef SGB_RING_LAUNCH
  return check_launch("knn2d_ring");
}

}  // namespace
}  // namespace sgb

using namespace sgb;

extern "C" int sgb_knn2d_ring_plan(const void* points, int is_f64, int64_t n_points, const void* query, int64_t n_query,
                                   int k, double max_dist, sgb_knn_plan* plan, void* ws64, void* stream_) {
  cudaStream_t stream = static_cast<cudaStream_t>(stream_);
  SGB_REQUIRE(plan, SGB_ERR_ARG, "knn2d_ring_plan: null plan");
  SGB_REQUIRE(n_points >= 0 && n_points < (int64_t(1) << 31) && n_query >= 0 && n_query < (int64_t(1) << 31), SGB_ERR_RANGE,
              "knn2d_ring_plan: point count out of range");
  SGB_REQUIRE(k >= 1 && k <= kRingMaxK, SGB_ERR_ARG, "knn2d_ring_plan: k=%d unsupported (1..%d)", k, kRingMaxK);
  SGB_REQUIRE(max_dist > 0.0, SGB_ERR_ARG, "knn2d_ring_plan: max_dist must be > 0 (+inf for no radius cap), got %g", max_dist);
  plan->n_points = n_points; plan->n_query = query ? n_query : n_points; plan->k = k; plan->max_dist = max_dist;
  plan->xmin = plan->ymin = 0.0; plan->cell = 1.0; plan->nx = plan->ny = 1;
  if (n_points == 0) return SGB_OK;
  SGB_REQUIRE(points && ws64, SGB_ERR_ARG, "knn2d_ring_plan: null tensor");
  // the grid spans the points only (a query far outside must not dilute the density); box[4..8) checks the queries
  double* box = static_cast<double*>(ws64);
  enqueue_bbox(points, n_points, nullptr, 0, is_f64, box, stream);
  const bool has_q = query && n_query > 0;
  if (has_q) enqueue_bbox(query, n_query, nullptr, 0, is_f64, box + 4, stream);
  double h[8];
  cudaError_t e = cudaMemcpyAsync(h, box, (has_q ? 8 : 4) * sizeof(double), cudaMemcpyDeviceToHost, stream);
  if (e == cudaSuccess) e = cudaStreamSynchronize(stream);
  if (e != cudaSuccess) return set_error(SGB_ERR_CUDA, "knn2d_ring_plan: %s", cudaGetErrorString(e));
  SGB_REQUIRE(box_finite(h) && (!has_q || box_finite(h + 4)), SGB_ERR_ARG, "knn2d_ring_plan: non-finite coordinates");
  // cell from the mean density: about 4k points in a 3 x 3 window (at least 8 points a cell), so the first ring
  // usually holds the k nearest; no larger than max_dist, since rings stop once the gap reaches it
  const double wx = h[2] - h[0], wy = h[3] - h[1], np = static_cast<double>(n_points);
  const double per_cell = fmax(4.0 * k / 9.0, 8.0);
  double cell = (wx > 0.0 && wy > 0.0) ? sqrt(per_cell * wx * wy / np) : fmax(wx, wy) * per_cell / np;
  cell = fmin(cell, max_dist * (1.0 + 1e-9));
  if (!(cell > 0.0) || !(1.0 / cell < INFINITY)) cell = fmax(fmax(wx, wy), 1.0);   // all points in one spot
  double nx = floor(wx / cell) + 1.0, ny = floor(wy / cell) + 1.0;
  if (nx * ny > static_cast<double>(kMaxCells)) {
    cell = sqrt((wx + cell) * (wy + cell) / static_cast<double>(kMaxCells)) * 1.01;
    nx = floor(wx / cell) + 1.0; ny = floor(wy / cell) + 1.0;
    while (nx * ny > static_cast<double>(kMaxCells)) { cell *= 1.5; nx = floor(wx / cell) + 1.0; ny = floor(wy / cell) + 1.0; }
  }
  plan->xmin = h[0]; plan->ymin = h[1]; plan->cell = cell;
  plan->nx = static_cast<int64_t>(nx); plan->ny = static_cast<int64_t>(ny);
  return SGB_OK;
}

extern "C" size_t sgb_knn2d_ring_workspace_bytes(const sgb_knn_plan* plan) { return sgb_knn2d_workspace_bytes(plan); }

extern "C" int sgb_knn2d_ring(const sgb_knn_plan* plan, const void* points, int is_f64, const void* query, int64_t* table,
                              int32_t* count, void* ws, size_t ws_bytes, void* stream_) {
  cudaStream_t stream = static_cast<cudaStream_t>(stream_);
  SGB_REQUIRE(plan, SGB_ERR_ARG, "knn2d_ring: null plan");
  SGB_REQUIRE(plan->k >= 1 && plan->k <= kRingMaxK && plan->max_dist > 0.0, SGB_ERR_ARG,
              "knn2d_ring: plan with k=%d, max_dist=%g (needs 1 <= k <= %d, max_dist > 0)", plan->k, plan->max_dist, kRingMaxK);
  if (plan->n_query == 0) return SGB_OK;
  SGB_REQUIRE(table, SGB_ERR_ARG, "knn2d_ring: null table");
  if (plan->n_points == 0) {
    cudaMemsetAsync(table, 0, static_cast<size_t>(plan->n_query) * plan->k * sizeof(int64_t), stream);
    if (count) cudaMemsetAsync(count, 0, static_cast<size_t>(plan->n_query) * sizeof(int32_t), stream);
    return check_launch("knn2d_ring(empty)");
  }
  SGB_REQUIRE(points && ws && ws_bytes >= sgb_knn2d_ring_workspace_bytes(plan), SGB_ERR_WORKSPACE,
              "knn2d_ring: workspace too small");
  if (is_f64)
    return run_knn_ring<double>(plan, static_cast<const double*>(points), static_cast<const double*>(query), table, count, ws, stream);
  return run_knn_ring<float>(plan, static_cast<const float*>(points), static_cast<const float*>(query), table, count, ws, stream);
}

