// Shared by the two 2-D kNN searches (sgb_knn.cu: register top-k, k <= 32 with a radius; sgb_knn_ring.cu: ring
// search, any k <= 1024 and any radius): bounding box, uniform grid, cell binning and the cell-sorted point array.
#pragma once
#include "sgb_api_internal.cuh"
#include "sgb_sort.cuh"

namespace sgb {
namespace {

constexpr int64_t kMaxCells = int64_t(1) << 26;

template <typename T>
__global__ void __launch_bounds__(256) bbox_kernel(const T* __restrict__ pts, int64_t n, double* __restrict__ box) {
  // box = [minx, miny, maxx, maxy] pre-initialised; one atomic per CTA via ordered-int trick on doubles
  __shared__ double sm[4][8];
  double mnx = INFINITY, mny = INFINITY, mxx = -INFINITY, mxy = -INFINITY;
  for (int64_t i = static_cast<int64_t>(blockIdx.x) * blockDim.x + threadIdx.x; i < n;
       i += static_cast<int64_t>(gridDim.x) * blockDim.x) {
    const double x = static_cast<double>(pts[2 * i]), y = static_cast<double>(pts[2 * i + 1]);
    mnx = fmin(mnx, x); mny = fmin(mny, y); mxx = fmax(mxx, x); mxy = fmax(mxy, y);
  }
#pragma unroll
  for (int o = 16; o >= 1; o >>= 1) {
    mnx = fmin(mnx, __shfl_xor_sync(kFull, mnx, o)); mny = fmin(mny, __shfl_xor_sync(kFull, mny, o));
    mxx = fmax(mxx, __shfl_xor_sync(kFull, mxx, o)); mxy = fmax(mxy, __shfl_xor_sync(kFull, mxy, o));
  }
  const int lane = threadIdx.x & 31, w = threadIdx.x >> 5;
  if (lane == 0) { sm[0][w] = mnx; sm[1][w] = mny; sm[2][w] = mxx; sm[3][w] = mxy; }
  __syncthreads();
  if (threadIdx.x == 0) {
    for (int i = 1; i < 8; ++i) {
      mnx = fmin(mnx, sm[0][i]); mny = fmin(mny, sm[1][i]); mxx = fmax(mxx, sm[2][i]); mxy = fmax(mxy, sm[3][i]);
    }
    // order-preserving double <-> signed 64-bit
    auto enc = [](double d) { long long v = __double_as_longlong(d); return v >= 0 ? v : v ^ 0x7fffffffffffffffLL; };
    long long* b = reinterpret_cast<long long*>(box);
    atomicMin(b + 0, enc(mnx)); atomicMin(b + 1, enc(mny)); atomicMax(b + 2, enc(mxx)); atomicMax(b + 3, enc(mxy));
  }
}
__global__ void bbox_init_kernel(double* box) {
  auto enc = [](double d) { long long v = __double_as_longlong(d); return v >= 0 ? v : v ^ 0x7fffffffffffffffLL; };
  long long* b = reinterpret_cast<long long*>(box);
  b[0] = enc(INFINITY); b[1] = enc(INFINITY); b[2] = enc(-INFINITY); b[3] = enc(-INFINITY);
}
__global__ void bbox_decode_kernel(double* box) {
  long long* b = reinterpret_cast<long long*>(box);
  for (int i = 0; i < 4; ++i) {
    long long v = b[i];
    v = v >= 0 ? v : v ^ 0x7fffffffffffffffLL;
    box[i] = __longlong_as_double(v);
  }
}

struct Grid {
  double xmin, ymin, inv_cell;
  int nx, ny;
};
__device__ __forceinline__ int cell_coord(double v, double lo, double inv, int n) {
  int c = static_cast<int>(floor((v - lo) * inv));
  return c < 0 ? 0 : (c >= n ? n - 1 : c);
}

template <typename T>
__global__ void cell_key_kernel(const T* __restrict__ pts, int64_t n, Grid g, uint32_t* __restrict__ keys) {
  const int64_t i = static_cast<int64_t>(blockIdx.x) * blockDim.x + threadIdx.x;
  if (i >= n) return;
  const int cx = cell_coord(static_cast<double>(pts[2 * i]), g.xmin, g.inv_cell, g.nx);
  const int cy = cell_coord(static_cast<double>(pts[2 * i + 1]), g.ymin, g.inv_cell, g.ny);
  keys[i] = static_cast<uint32_t>(cy) * static_cast<uint32_t>(g.nx) + static_cast<uint32_t>(cx);
}

template <typename T>
__global__ void gather_sorted_kernel(const T* __restrict__ pts, const uint32_t* __restrict__ perm, int64_t n,
                                     double2* __restrict__ sorted) {
  const int64_t i = static_cast<int64_t>(blockIdx.x) * blockDim.x + threadIdx.x;
  if (i >= n) return;
  const int64_t j = perm[i];
  sorted[i] = make_double2(static_cast<double>(pts[2 * j]), static_cast<double>(pts[2 * j + 1]));
}

__device__ __forceinline__ bool knn_less(double d1, int i1, double d2, int i2) {
  return d1 < d2 || (d1 == d2 && i1 < i2);
}

struct KnnWs {
  uint32_t *keys, *skeys, *perm;
  double2* sorted;
  int32_t* cell_start;
  void* sort_ws;
  size_t sort_bytes, total;
};
KnnWs knn_carve(void* ws, int64_t n, int64_t ncells) {
  KnnWs k{};
  const size_t nb = align_up(static_cast<size_t>(n > 0 ? n : 1) * 4);
  char* p = static_cast<char*>(ws);
  k.keys = reinterpret_cast<uint32_t*>(p); p += nb;
  k.skeys = reinterpret_cast<uint32_t*>(p); p += nb;
  k.perm = reinterpret_cast<uint32_t*>(p); p += nb;
  k.sorted = reinterpret_cast<double2*>(p); p += align_up(static_cast<size_t>(n > 0 ? n : 1) * 16);
  k.cell_start = reinterpret_cast<int32_t*>(p); p += align_up(static_cast<size_t>(ncells + 1) * 4);
  k.sort_ws = p;
  k.sort_bytes = sort_pairs_workspace_bytes(n);
  k.total = static_cast<size_t>(p - static_cast<char*>(ws)) + k.sort_bytes;
  return k;
}

// bins the points into the plan's grid, sorts them by cell and gathers the sorted fp64 coordinates
template <typename T>
int bin_points(const sgb_knn_plan* plan, const T* points, const KnnWs& w, const Grid& g, cudaStream_t stream) {
  const int64_t n = plan->n_points;
  const int64_t ncells = plan->nx * plan->ny;
  const unsigned nb = static_cast<unsigned>(ceil_div(n, 256));
  cell_key_kernel<T><<<nb, 256, 0, stream>>>(points, n, g, w.keys);
  int rc = sort_pairs(w.keys, nullptr, w.skeys, w.perm, n, bits_for(ncells), w.sort_ws, w.sort_bytes, stream);
  if (rc != SGB_OK) return rc;
  rc = rowptr_from_sorted(w.skeys, n, w.cell_start, ncells, stream);
  if (rc != SGB_OK) return rc;
  gather_sorted_kernel<T><<<nb, 256, 0, stream>>>(points, w.perm, n, w.sorted);
  return SGB_OK;
}

// Enqueues the bounding box of a[0, na) and b[0, nb) (b may be NULL) into box[0..4) = [minx, miny, maxx, maxy].
void enqueue_bbox(const void* a, int64_t na, const void* b, int64_t nb, int is_f64, double* box, cudaStream_t stream) {
  bbox_init_kernel<<<1, 1, 0, stream>>>(box);
  const int blocks = sm_count() * 4;
  if (is_f64) {
    bbox_kernel<double><<<blocks, 256, 0, stream>>>(static_cast<const double*>(a), na, box);
    if (b && nb > 0) bbox_kernel<double><<<blocks, 256, 0, stream>>>(static_cast<const double*>(b), nb, box);
  } else {
    bbox_kernel<float><<<blocks, 256, 0, stream>>>(static_cast<const float*>(a), na, box);
    if (b && nb > 0) bbox_kernel<float><<<blocks, 256, 0, stream>>>(static_cast<const float*>(b), nb, box);
  }
  bbox_decode_kernel<<<1, 1, 0, stream>>>(box);
}

bool box_finite(const double* h) {
  return h[0] == h[0] && h[2] == h[2] && h[0] > -INFINITY && h[2] < INFINITY && h[1] > -INFINITY && h[3] < INFINITY;
}

}  // namespace
}  // namespace sgb
