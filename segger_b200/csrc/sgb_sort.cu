// Stable LSD radix sort (8-bit digits), exclusive scan and sorted-key -> rowptr, hand-written.
// Used by the CSR builder (dst-sorted + src-sorted edge lists), the candidate CSR of the scoring
// kernel and the cell binning of the grid kNN.  All of it is HBM-bound integer work; the keys are
// streamed with coalesced loads, digit ranks are computed with warp match/ballot so the sort is
// stable without atomics on the output order (deterministic edge order => deterministic fp sums).
#include "sgb_sort.cuh"

namespace sgb {

namespace {

__global__ void __launch_bounds__(kRsThreads)
rs_hist_kernel(const uint32_t* __restrict__ keys, int64_t n, int shift, int32_t* __restrict__ hist,
               int nblk, const int32_t* __restrict__ skip) {
  if (skip && *skip) return;   // keys already sorted: presorted_copy_kernel produces the output
  __shared__ int cnt[kRadix];
  cnt[threadIdx.x] = 0;
  __syncthreads();
  const int64_t base = static_cast<int64_t>(blockIdx.x) * kRsTile;
#pragma unroll
  for (int i = 0; i < kRsItems; ++i) {
    const int64_t idx = base + i * kRsThreads + threadIdx.x;
    if (idx < n) atomicAdd(&cnt[(keys[idx] >> shift) & (kRadix - 1)], 1);
  }
  __syncthreads();
  hist[static_cast<int64_t>(threadIdx.x) * nblk + blockIdx.x] = cnt[threadIdx.x];
}

__global__ void __launch_bounds__(kRsThreads)
rs_scatter_kernel(const uint32_t* __restrict__ keys_in, const uint32_t* __restrict__ vals_in,
                  uint32_t* __restrict__ keys_out, uint32_t* __restrict__ vals_out, int64_t n,
                  int shift, const int32_t* __restrict__ offs, int nblk, const int32_t* __restrict__ skip) {
  if (skip && *skip) return;
  constexpr int kWarps = kRsThreads / 32;
  constexpr int kPerWarp = kRsTile / kWarps;  // 512 consecutive keys per warp
  __shared__ int cnt[kWarps][kRadix];
  const int w = threadIdx.x >> 5, lane = threadIdx.x & 31;
  for (int i = threadIdx.x; i < kWarps * kRadix; i += kRsThreads) (&cnt[0][0])[i] = 0;
  __syncthreads();

  const int64_t wbase = static_cast<int64_t>(blockIdx.x) * kRsTile + static_cast<int64_t>(w) * kPerWarp;
  uint32_t k[kRsItems];
  int rank[kRsItems];
#pragma unroll
  for (int r = 0; r < kRsItems; ++r) {
    const int64_t idx = wbase + r * 32 + lane;
    const bool valid = idx < n;
    k[r] = valid ? keys_in[idx] : 0u;
    rank[r] = 0;
    const unsigned act = __ballot_sync(kFull, valid);
    if (valid) {
      const int d = (k[r] >> shift) & (kRadix - 1);
      const unsigned peers = __match_any_sync(act, d);
      const int leader = __ffs(peers) - 1;
      int old = 0;
      if (lane == leader) {
        old = cnt[w][d];
        cnt[w][d] = old + __popc(peers);
      }
      old = __shfl_sync(act, old, leader);
      rank[r] = old + __popc(peers & ((1u << lane) - 1u));
    }
    __syncwarp();
  }
  __syncthreads();
  {  // digit t: exclusive prefix over the warps of this CTA, seeded with the global offset
    const int t = threadIdx.x;
    int base = offs[static_cast<int64_t>(t) * nblk + blockIdx.x];
#pragma unroll
    for (int ww = 0; ww < kWarps; ++ww) {
      const int c = cnt[ww][t];
      cnt[ww][t] = base;
      base += c;
    }
  }
  __syncthreads();
#pragma unroll
  for (int r = 0; r < kRsItems; ++r) {
    const int64_t idx = wbase + r * 32 + lane;
    if (idx < n) {
      const int d = (k[r] >> shift) & (kRadix - 1);
      const int dst = cnt[w][d] + rank[r];
      keys_out[dst] = k[r];
      vals_out[dst] = vals_in ? vals_in[idx] : static_cast<uint32_t>(idx);
    }
  }
}

// ---- scan ----
constexpr int kScanThreads = 256;
constexpr int kScanItems = 8;
constexpr int kScanTile = kScanThreads * kScanItems;

// A = accumulator / output type: int (the 32-bit scan) or long long (kNN edge offsets that may pass 2^31)
template <typename A>
__device__ __forceinline__ A block_exclusive_scan(A v, A* total) {
  __shared__ A wsum[kScanThreads / 32];
  __shared__ A wtot;
  const int lane = threadIdx.x & 31, w = threadIdx.x >> 5;
  A inc = v;
#pragma unroll
  for (int o = 1; o < 32; o <<= 1) {
    const A t = __shfl_up_sync(kFull, inc, o);
    if (lane >= o) inc += t;
  }
  if (lane == 31) wsum[w] = inc;
  __syncthreads();
  if (w == 0) {
    A s = lane < kScanThreads / 32 ? wsum[lane] : 0;
    A sinc = s;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
      const A t = __shfl_up_sync(kFull, sinc, o);
      if (lane >= o) sinc += t;
    }
    if (lane < kScanThreads / 32) wsum[lane] = sinc - s;
    if (lane == 31) wtot = sinc;
  }
  __syncthreads();
  const A res = wsum[w] + inc - v;
  *total = wtot;
  __syncthreads();
  return res;
}

template <typename A>
__global__ void __launch_bounds__(kScanThreads)
scan_tile_sum_kernel(const int32_t* __restrict__ in, int64_t n, A* __restrict__ bsum) {
  const int64_t base = static_cast<int64_t>(blockIdx.x) * kScanTile + threadIdx.x * kScanItems;
  A s = 0;
#pragma unroll
  for (int j = 0; j < kScanItems; ++j)
    if (base + j < n) s += in[base + j];
  A tot;
  block_exclusive_scan<A>(s, &tot);
  if (threadIdx.x == 0) bsum[blockIdx.x] = tot;
}

// single CTA: in-place exclusive scan of bsum[0..nb), bsum[nb] = total
template <typename A>
__global__ void __launch_bounds__(kScanThreads)
scan_block_sums_kernel(A* __restrict__ bsum, int64_t nb) {
  A carry = 0;
  for (int64_t base = 0; base < nb; base += kScanThreads) {
    const int64_t i = base + threadIdx.x;
    const A v = i < nb ? bsum[i] : 0;
    A tot;
    const A ex = block_exclusive_scan<A>(v, &tot);
    if (i < nb) bsum[i] = carry + ex;
    carry += tot;
  }
  if (threadIdx.x == 0) bsum[nb] = carry;
}

template <typename A>
__global__ void __launch_bounds__(kScanThreads)
scan_apply_kernel(const int32_t* __restrict__ in, A* __restrict__ out, int64_t n,
                  const A* __restrict__ bsum, int64_t nb) {
  const int64_t base = static_cast<int64_t>(blockIdx.x) * kScanTile + threadIdx.x * kScanItems;
  int v[kScanItems];
  A s = 0;
#pragma unroll
  for (int j = 0; j < kScanItems; ++j) {
    v[j] = base + j < n ? in[base + j] : 0;
    s += v[j];
  }
  A tot;
  A ex = block_exclusive_scan<A>(s, &tot) + bsum[blockIdx.x];
#pragma unroll
  for (int j = 0; j < kScanItems; ++j) {
    if (base + j < n) out[base + j] = ex;
    ex += v[j];
  }
  if (blockIdx.x == 0 && threadIdx.x == 0) out[n] = bsum[nb];
}

__global__ void rowptr_kernel(const uint32_t* __restrict__ keys, int64_t n, int32_t* __restrict__ rowptr,
                              int64_t n_rows) {
  const int64_t r = static_cast<int64_t>(blockIdx.x) * blockDim.x + threadIdx.x;
  if (r > n_rows) return;
  int64_t lo = 0, hi = n;  // first position with key >= r
  while (lo < hi) {
    const int64_t mid = (lo + hi) >> 1;
    if (static_cast<int64_t>(keys[mid]) < r) lo = mid + 1; else hi = mid;
  }
  rowptr[r] = static_cast<int32_t>(lo);
}

// flag[0] starts at 1 and is cleared by any adjacent pair out of order (under the key mask)
__global__ void sorted_flag_init_kernel(int32_t* flag) { *flag = 1; }
__global__ void sorted_check_kernel(const uint32_t* __restrict__ keys, int64_t n, uint32_t mask, int32_t* __restrict__ flag) {
  const int64_t i = static_cast<int64_t>(blockIdx.x) * blockDim.x + threadIdx.x;
  if (i + 1 < n && (keys[i] & mask) > (keys[i + 1] & mask)) *flag = 0;
}
__global__ void presorted_copy_kernel(const uint32_t* __restrict__ keys_in, const uint32_t* __restrict__ vals_in,
                                      uint32_t* __restrict__ keys_out, uint32_t* __restrict__ vals_out, int64_t n,
                                      const int32_t* __restrict__ flag) {
  if (!*flag) return;
  const int64_t i = static_cast<int64_t>(blockIdx.x) * blockDim.x + threadIdx.x;
  if (i < n) {
    keys_out[i] = keys_in[i];
    vals_out[i] = vals_in ? vals_in[i] : static_cast<uint32_t>(i);
  }
}

template <typename A>
size_t scan_ws_bytes(int64_t n) {
  const int64_t nb = ceil_div(n > 0 ? n : 1, kScanTile);
  return align_up(static_cast<size_t>(nb + 1) * sizeof(A));
}

template <typename A>
int exclusive_scan(const int32_t* in, A* out, int64_t n, void* ws, size_t ws_bytes, cudaStream_t stream) {
  SGB_REQUIRE(n >= 0 && in && out && ws, SGB_ERR_ARG, "exclusive_scan: null argument");
  SGB_REQUIRE(ws_bytes >= scan_ws_bytes<A>(n), SGB_ERR_WORKSPACE, "exclusive_scan: workspace too small");
  if (n == 0) {
    cudaMemsetAsync(out, 0, sizeof(A), stream);
    return check_launch("exclusive_scan(memset)");
  }
  const int64_t nb = ceil_div(n, kScanTile);
  A* bsum = static_cast<A*>(ws);
  scan_tile_sum_kernel<A><<<static_cast<unsigned>(nb), kScanThreads, 0, stream>>>(in, n, bsum);
  scan_block_sums_kernel<A><<<1, kScanThreads, 0, stream>>>(bsum, nb);
  scan_apply_kernel<A><<<static_cast<unsigned>(nb), kScanThreads, 0, stream>>>(in, out, n, bsum, nb);
  return check_launch("exclusive_scan");
}

}  // namespace

size_t scan_workspace_bytes(int64_t n) { return scan_ws_bytes<int>(n); }
int exclusive_scan_i32(const int32_t* in, int32_t* out, int64_t n, void* ws, size_t ws_bytes, cudaStream_t stream) {
  return exclusive_scan<int>(in, out, n, ws, ws_bytes, stream);
}
size_t scan_i64_workspace_bytes(int64_t n) { return scan_ws_bytes<long long>(n); }
int exclusive_scan_i64(const int32_t* in, int64_t* out, int64_t n, void* ws, size_t ws_bytes, cudaStream_t stream) {
  static_assert(sizeof(long long) == sizeof(int64_t), "int64_t is long long");
  return exclusive_scan<long long>(in, reinterpret_cast<long long*>(out), n, ws, ws_bytes, stream);
}

size_t sort_pairs_workspace_bytes(int64_t n) {
  const int64_t nn = n > 0 ? n : 1;
  const int64_t nblk = ceil_div(nn, kRsTile);
  const int64_t nh = nblk * kRadix;
  return 2 * align_up(static_cast<size_t>(nn) * 4)        // tmp keys, tmp vals
         + 2 * align_up(static_cast<size_t>(nh + 1) * 4)  // histogram + scanned offsets
         + scan_workspace_bytes(nh) + 256;                 // + presorted flag
}

int sort_pairs(const uint32_t* keys_in, const uint32_t* vals_in, uint32_t* keys_out,
               uint32_t* vals_out, int64_t n, int key_bits, void* ws, size_t ws_bytes,
               cudaStream_t stream, bool detect_presorted) {
  SGB_REQUIRE(n >= 0 && n < (int64_t(1) << 31), SGB_ERR_RANGE, "sort_pairs: n=%lld out of range", (long long)n);
  SGB_REQUIRE(keys_out && vals_out && ws, SGB_ERR_ARG, "sort_pairs: null argument");
  SGB_REQUIRE(keys_in != keys_out, SGB_ERR_ARG, "sort_pairs: in-place sort is not supported");
  SGB_REQUIRE(ws_bytes >= sort_pairs_workspace_bytes(n), SGB_ERR_WORKSPACE, "sort_pairs: workspace too small");
  if (n == 0) return SGB_OK;
  SGB_REQUIRE(keys_in, SGB_ERR_ARG, "sort_pairs: null keys");
  if (key_bits < 1) key_bits = 1;
  if (key_bits > 32) key_bits = 32;
  const int passes = (key_bits + 7) / 8;
  const int nblk = static_cast<int>(ceil_div(n, kRsTile));
  const int64_t nh = static_cast<int64_t>(nblk) * kRadix;

  char* p = static_cast<char*>(ws);
  uint32_t* tk = reinterpret_cast<uint32_t*>(p); p += align_up(static_cast<size_t>(n) * 4);
  uint32_t* tv = reinterpret_cast<uint32_t*>(p); p += align_up(static_cast<size_t>(n) * 4);
  int32_t* hist = reinterpret_cast<int32_t*>(p); p += align_up(static_cast<size_t>(nh + 1) * 4);
  int32_t* offs = reinterpret_cast<int32_t*>(p); p += align_up(static_cast<size_t>(nh + 1) * 4);
  void* scan_ws = p;
  const size_t scan_bytes = scan_workspace_bytes(nh);
  p += scan_bytes;
  // Presorted inputs (the src-major edge lists kNN and setup_heterodata emit): one check pass sets a device flag,
  // the histogram / scatter passes return at once and a single copy produces the (identical) stable result.
  int32_t* flag = nullptr;
  const bool detect = detect_presorted && keys_in != keys_out && vals_in != vals_out;
  if (detect) {
    flag = reinterpret_cast<int32_t*>(p);
    const uint32_t mask = key_bits >= 32 ? 0xFFFFFFFFu : ((1u << key_bits) - 1u);
    sorted_flag_init_kernel<<<1, 1, 0, stream>>>(flag);
    sorted_check_kernel<<<static_cast<unsigned>(ceil_div(n, 256)), 256, 0, stream>>>(keys_in, n, mask, flag);
  }

  const uint32_t* sk = keys_in;
  const uint32_t* sv = vals_in;
  for (int ps = 0; ps < passes; ++ps) {
    const bool to_out = ((passes - 1 - ps) % 2) == 0;
    uint32_t* dk = to_out ? keys_out : tk;
    uint32_t* dv = to_out ? vals_out : tv;
    rs_hist_kernel<<<nblk, kRsThreads, 0, stream>>>(sk, n, ps * 8, hist, nblk, flag);
    int rc = exclusive_scan_i32(hist, offs, nh, scan_ws, scan_bytes, stream);
    if (rc != SGB_OK) return rc;
    rs_scatter_kernel<<<nblk, kRsThreads, 0, stream>>>(sk, sv, dk, dv, n, ps * 8, offs, nblk, flag);
    sk = dk;
    sv = dv;
  }
  if (detect)
    presorted_copy_kernel<<<static_cast<unsigned>(ceil_div(n, 256)), 256, 0, stream>>>(keys_in, vals_in, keys_out, vals_out, n, flag);
  return check_launch("sort_pairs");
}

int rowptr_from_sorted(const uint32_t* sorted_keys, int64_t n, int32_t* rowptr, int64_t n_rows,
                       cudaStream_t stream) {
  SGB_REQUIRE(rowptr && (n == 0 || sorted_keys), SGB_ERR_ARG, "rowptr_from_sorted: null argument");
  const int64_t blocks = ceil_div(n_rows + 1, 256);
  rowptr_kernel<<<static_cast<unsigned>(blocks), 256, 0, stream>>>(sorted_keys, n, rowptr, n_rows);
  return check_launch("rowptr_from_sorted");
}

}  // namespace sgb
