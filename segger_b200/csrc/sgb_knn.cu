// 2-D k-nearest-neighbour search with a radius cap on a uniform grid, and neighbour-table -> COO.
// Replaces scipy.spatial.KDTree(points, leafsize=100).query(q, k, distance_upper_bound, workers=-1)
// as called by kdtree_neighbors (/root/reference/src/segger/data/utils/neighbors.py:139-150) and the
// ATen nonzero/index plumbing of knn_to_edge_index (:54-92).
//
// Arithmetic contract (SURVEY.md Appendix A.5): coordinates are widened to float64 exactly; the
// squared distance is fl(fl(dx*dx) + fl(dy*dy)) with explicit round-to-nearest multiplies/adds (no
// FMA contraction) -- the value cKDTree compares; a neighbour is accepted iff d^2 < max_dist^2
// (strict); rows are ordered by (d^2, original index) and padded with n_points.
//
// Layout: points are binned into square cells of edge >= max_dist (slightly enlarged so rounding can
// never push a true neighbour two cells away), sorted by cell with the stable radix sort, and the
// sorted float64 coordinates are streamed; a query scans 3 rows of 3 adjacent cells, which are 3
// contiguous ranges of the sorted array.  One thread per query keeps its top-k in registers.
// That kernel holds k <= 32 and needs a finite radius; sgb_knn_ring.cu serves every other k <= 1024 and radius.
#include "sgb_knn.cuh"

namespace sgb {
namespace {

// K = compile-time capacity of the register top-k (k <= K)
template <int K, typename T>
__global__ void __launch_bounds__(128)
knn_query_kernel(const double2* __restrict__ sorted, const uint32_t* __restrict__ perm, const int32_t* __restrict__ cell_start,
                 Grid g, const T* __restrict__ query, int64_t n_query, int64_t n_points, int k, double r2,
                 int64_t* __restrict__ table, int32_t* __restrict__ count) {
  const int64_t t = static_cast<int64_t>(blockIdx.x) * blockDim.x + threadIdx.x;
  if (t >= n_query) return;
  double qx, qy;
  int64_t qrow;
  if (query) {
    qx = static_cast<double>(query[2 * t]); qy = static_cast<double>(query[2 * t + 1]); qrow = t;
  } else {
    const double2 q = sorted[t];
    qx = q.x; qy = q.y; qrow = perm[t];
  }
  double bd[K];
  int bi[K];
#pragma unroll
  for (int j = 0; j < K; ++j) { bd[j] = INFINITY; bi[j] = 0x7fffffff; }
  const int cx = cell_coord(qx, g.xmin, g.inv_cell, g.nx);
  const int cy = cell_coord(qy, g.ymin, g.inv_cell, g.ny);
  const int x0 = max(cx - 1, 0), x1 = min(cx + 1, g.nx - 1);
  for (int yy = max(cy - 1, 0); yy <= min(cy + 1, g.ny - 1); ++yy) {
    const int beg = cell_start[static_cast<int64_t>(yy) * g.nx + x0];
    const int end = cell_start[static_cast<int64_t>(yy) * g.nx + x1 + 1];
    for (int s = beg; s < end; ++s) {
      const double2 pnt = sorted[s];
      const double dx = __dsub_rn(pnt.x, qx), dy = __dsub_rn(pnt.y, qy);
      const double d2 = __dadd_rn(__dmul_rn(dx, dx), __dmul_rn(dy, dy));
      if (d2 < r2) {
        const int idx = static_cast<int>(perm[s]);
        // top-K (K >= k, compile-time) kept sorted by (d2, idx): replace the worst, bubble up with
        // branch-free compare-swaps so the list stays in registers
        if (knn_less(d2, idx, bd[K - 1], bi[K - 1])) {
          bd[K - 1] = d2;
          bi[K - 1] = idx;
#pragma unroll
          for (int j = K - 1; j > 0; --j) {
            const bool sw = knn_less(bd[j], bi[j], bd[j - 1], bi[j - 1]);
            const double lo_d = sw ? bd[j] : bd[j - 1], hi_d = sw ? bd[j - 1] : bd[j];
            const int lo_i = sw ? bi[j] : bi[j - 1], hi_i = sw ? bi[j - 1] : bi[j];
            bd[j - 1] = lo_d; bd[j] = hi_d;
            bi[j - 1] = lo_i; bi[j] = hi_i;
          }
        }
      }
    }
  }
  int cnt = 0;
#pragma unroll
  for (int j = 0; j < K; ++j) {
    if (j < k) {
      const bool ok = bd[j] < INFINITY;
      table[qrow * k + j] = ok ? static_cast<int64_t>(bi[j]) : n_points;
      cnt += ok ? 1 : 0;
    }
  }
  if (count) count[qrow] = cnt;
}

__global__ void count_valid_kernel(const int64_t* __restrict__ table, int64_t n, int k, int64_t pad, int32_t* __restrict__ count) {
  const int64_t r = static_cast<int64_t>(blockIdx.x) * blockDim.x + threadIdx.x;
  if (r >= n) return;
  int c = 0;
  for (int j = 0; j < k; ++j) c += table[r * k + j] != pad ? 1 : 0;
  count[r] = c;
}
__global__ void table_to_coo_kernel(const int64_t* __restrict__ table, const int64_t* __restrict__ index_ptr, int64_t n,
                                    int k, int64_t pad, int64_t row_offset, int64_t E, int64_t* __restrict__ ei) {
  const int64_t r = static_cast<int64_t>(blockIdx.x) * blockDim.x + threadIdx.x;
  if (r >= n) return;
  int64_t o = index_ptr[r];
  for (int j = 0; j < k; ++j) {
    const int64_t v = table[r * k + j];
    if (v != pad) {
      ei[o] = r + row_offset;
      ei[E + o] = v;
      ++o;
    }
  }
}

template <typename T>
int run_knn(const sgb_knn_plan* plan, const T* points, const T* query, int64_t* table, int32_t* count, void* ws,
            cudaStream_t stream) {
  const int64_t n = plan->n_points, nq = plan->n_query;
  KnnWs w = knn_carve(ws, n, plan->nx * plan->ny);
  Grid g{plan->xmin, plan->ymin, 1.0 / plan->cell, static_cast<int>(plan->nx), static_cast<int>(plan->ny)};
  const int rc = bin_points<T>(plan, points, w, g, stream);
  if (rc != SGB_OK) return rc;
  const unsigned qb = static_cast<unsigned>(ceil_div(nq, 128));
  const double r2 = plan->max_dist * plan->max_dist;
  const int k = plan->k;
#define SGB_KNN_LAUNCH(KK) \
  knn_query_kernel<KK, T><<<qb, 128, 0, stream>>>(w.sorted, w.perm, w.cell_start, g, query, nq, n, k, r2, table, count)
  // register top-K capacity = smallest instantiation >= k: every accepted candidate costs K - 1 compare-swaps, and the
  // register footprint (3 per slot) sets the occupancy (k = 20 on K = 32: 204 registers, 2 CTAs/SM)
  if (k <= 4) SGB_KNN_LAUNCH(4);
  else if (k <= 5) SGB_KNN_LAUNCH(5);
  else if (k <= 6) SGB_KNN_LAUNCH(6);
  else if (k <= 8) SGB_KNN_LAUNCH(8);
  else if (k <= 10) SGB_KNN_LAUNCH(10);
  else if (k <= 12) SGB_KNN_LAUNCH(12);
  else if (k <= 16) SGB_KNN_LAUNCH(16);
  else if (k <= 20) SGB_KNN_LAUNCH(20);
  else if (k <= 24) SGB_KNN_LAUNCH(24);
  else SGB_KNN_LAUNCH(32);
#undef SGB_KNN_LAUNCH
  return check_launch("knn2d");
}

}  // namespace
}  // namespace sgb

using namespace sgb;

extern "C" int sgb_knn2d_plan(const void* points, int is_f64, int64_t n_points, const void* query, int64_t n_query,
                              int k, double max_dist, sgb_knn_plan* plan, void* ws64, void* stream_) {
  cudaStream_t stream = static_cast<cudaStream_t>(stream_);
  SGB_REQUIRE(plan, SGB_ERR_ARG, "knn2d_plan: null plan");
  SGB_REQUIRE(n_points >= 0 && n_points < (int64_t(1) << 31) && n_query >= 0 && n_query < (int64_t(1) << 31), SGB_ERR_RANGE,
              "knn2d_plan: point count out of range");
  SGB_REQUIRE(k >= 1 && k <= 32, SGB_ERR_ARG, "knn2d_plan: k=%d unsupported (1..32)", k);
  SGB_REQUIRE(max_dist > 0.0 && max_dist < INFINITY, SGB_ERR_ARG, "knn2d_plan: max_dist must be finite and > 0");
  plan->n_points = n_points; plan->n_query = query ? n_query : n_points; plan->k = k; plan->max_dist = max_dist;
  plan->xmin = plan->ymin = 0.0; plan->cell = max_dist; plan->nx = plan->ny = 1;
  if (n_points == 0) return SGB_OK;
  SGB_REQUIRE(points && ws64, SGB_ERR_ARG, "knn2d_plan: null tensor");
  double* box = static_cast<double*>(ws64);
  enqueue_bbox(points, n_points, query, n_query, is_f64, box, stream);
  double h[4];
  cudaError_t e = cudaMemcpyAsync(h, box, sizeof(h), cudaMemcpyDeviceToHost, stream);
  if (e == cudaSuccess) e = cudaStreamSynchronize(stream);
  if (e != cudaSuccess) return set_error(SGB_ERR_CUDA, "knn2d_plan: %s", cudaGetErrorString(e));
  SGB_REQUIRE(box_finite(h), SGB_ERR_ARG, "knn2d_plan: non-finite coordinates");
  // enlarge the cell a hair so floor((v - lo) / cell) can never separate true neighbours by 2 cells
  double cell = max_dist * (1.0 + 1e-9);
  const double wx = h[2] - h[0], wy = h[3] - h[1];
  double nx = floor(wx / cell) + 1.0, ny = floor(wy / cell) + 1.0;
  if (nx * ny > static_cast<double>(kMaxCells)) {
    cell = sqrt((wx + cell) * (wy + cell) / static_cast<double>(kMaxCells)) * 1.01;
    if (cell < max_dist * (1.0 + 1e-9)) cell = max_dist * (1.0 + 1e-9);
    nx = floor(wx / cell) + 1.0; ny = floor(wy / cell) + 1.0;
    while (nx * ny > static_cast<double>(kMaxCells)) { cell *= 1.5; nx = floor(wx / cell) + 1.0; ny = floor(wy / cell) + 1.0; }
  }
  plan->xmin = h[0]; plan->ymin = h[1]; plan->cell = cell;
  plan->nx = static_cast<int64_t>(nx); plan->ny = static_cast<int64_t>(ny);
  return SGB_OK;
}

extern "C" size_t sgb_knn2d_workspace_bytes(const sgb_knn_plan* plan) {
  if (!plan) return 0;
  return knn_carve(nullptr, plan->n_points, plan->nx * plan->ny).total;
}

extern "C" int sgb_knn2d(const sgb_knn_plan* plan, const void* points, int is_f64, const void* query, int64_t* table,
                         int32_t* count, void* ws, size_t ws_bytes, void* stream_) {
  cudaStream_t stream = static_cast<cudaStream_t>(stream_);
  SGB_REQUIRE(plan, SGB_ERR_ARG, "knn2d: null plan");
  if (plan->n_query == 0) return SGB_OK;
  SGB_REQUIRE(table, SGB_ERR_ARG, "knn2d: null table");
  if (plan->n_points == 0) {
    // nothing to find: the table is all padding (= 0 == n_points)
    cudaMemsetAsync(table, 0, static_cast<size_t>(plan->n_query) * plan->k * sizeof(int64_t), stream);
    if (count) cudaMemsetAsync(count, 0, static_cast<size_t>(plan->n_query) * sizeof(int32_t), stream);
    return check_launch("knn2d(empty)");
  }
  SGB_REQUIRE(points && ws && ws_bytes >= sgb_knn2d_workspace_bytes(plan), SGB_ERR_WORKSPACE, "knn2d: workspace too small");
  if (is_f64) return run_knn<double>(plan, static_cast<const double*>(points), static_cast<const double*>(query), table, count, ws, stream);
  return run_knn<float>(plan, static_cast<const float*>(points), static_cast<const float*>(query), table, count, ws, stream);
}

extern "C" int sgb_knn_count_valid(const int64_t* table, int64_t n, int k, int64_t pad_value, int32_t* count, void* stream) {
  SGB_REQUIRE(n >= 0 && k >= 1, SGB_ERR_ARG, "knn_count_valid: bad size");
  if (n == 0) return SGB_OK;
  SGB_REQUIRE(table && count, SGB_ERR_ARG, "knn_count_valid: null tensor");
  count_valid_kernel<<<static_cast<unsigned>(ceil_div(n, 256)), 256, 0, static_cast<cudaStream_t>(stream)>>>(table, n, k, pad_value, count);
  return check_launch("knn_count_valid");
}

extern "C" size_t sgb_knn_coo_workspace_bytes(int64_t n_query) { return scan_i64_workspace_bytes(n_query); }

extern "C" int sgb_knn_count_edges(const int32_t* count, int64_t n_query, int64_t* index_ptr, int64_t* n_edges_host,
                                   void* ws, size_t ws_bytes, void* stream_) {
  cudaStream_t stream = static_cast<cudaStream_t>(stream_);
  SGB_REQUIRE(n_query >= 0 && index_ptr && ws, SGB_ERR_ARG, "knn_count_edges: bad argument");
  SGB_REQUIRE(ws_bytes >= sgb_knn_coo_workspace_bytes(n_query), SGB_ERR_WORKSPACE, "knn_count_edges: workspace too small");
  if (n_query == 0) {
    cudaMemsetAsync(index_ptr, 0, sizeof(int64_t), stream);
  } else {
    SGB_REQUIRE(count, SGB_ERR_ARG, "knn_count_edges: null count");
    // int64 sums: the offsets stay exact when the edge count reaches 2^31 (k = 1024 does at 2.1M queries)
    int rc = exclusive_scan_i64(count, index_ptr, n_query, ws, ws_bytes, stream);
    if (rc != SGB_OK) return rc;
  }
  if (n_edges_host) {
    cudaError_t e = cudaMemcpyAsync(n_edges_host, index_ptr + n_query, sizeof(int64_t), cudaMemcpyDeviceToHost, stream);
    if (e == cudaSuccess) e = cudaStreamSynchronize(stream);
    if (e != cudaSuccess) return set_error(SGB_ERR_CUDA, "knn_count_edges: %s", cudaGetErrorString(e));
  }
  return check_launch("knn_count_edges");
}

extern "C" int sgb_knn_table_to_coo(const int64_t* table, const int64_t* index_ptr, int64_t n_query, int k,
                                    int64_t pad_value, int64_t row_offset, int64_t E, int64_t* edge_index, void* stream) {
  SGB_REQUIRE(n_query >= 0 && k >= 1 && E >= 0, SGB_ERR_ARG, "knn_table_to_coo: bad size");
  if (n_query == 0 || E == 0) return SGB_OK;
  SGB_REQUIRE(table && index_ptr && edge_index, SGB_ERR_ARG, "knn_table_to_coo: null tensor");
  table_to_coo_kernel<<<static_cast<unsigned>(ceil_div(n_query, 256)), 256, 0, static_cast<cudaStream_t>(stream)>>>(
      table, index_ptr, n_query, k, pad_value, row_offset, E, edge_index);
  return check_launch("knn_table_to_coo");
}
