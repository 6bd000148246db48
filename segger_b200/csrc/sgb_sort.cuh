// Stable LSD radix sort of (u32 key, u32 value) pairs + exclusive scan, hand-written (no CUB).
#pragma once
#include "sgb_common.cuh"

namespace sgb {

constexpr int kRsThreads = 256;
constexpr int kRsItems = 16;                       // items per thread
constexpr int kRsTile = kRsThreads * kRsItems;     // 4096 keys per CTA
constexpr int kRadix = 256;

// bytes of scratch for sorting n pairs (double buffers + per-tile digit histograms)
size_t sort_pairs_workspace_bytes(int64_t n);

// Sorts n pairs by the low `key_bits` bits of the key, stable.  keys_in/vals_in are preserved
// unless they alias the outputs.  Result lands in keys_out/vals_out.
// vals_in == nullptr means "values are 0..n-1".
// detect_presorted: check on the device whether the keys are already non-decreasing; if so the radix passes
// return immediately and one copy writes the result (bit-identical to what the stable sort would produce).
int sort_pairs(const uint32_t* keys_in, const uint32_t* vals_in, uint32_t* keys_out,
               uint32_t* vals_out, int64_t n, int key_bits, void* ws, size_t ws_bytes,
               cudaStream_t stream, bool detect_presorted = false);

// out[i] = sum_{j<i} in[j] for i in [0, n]; out has n+1 entries (out[n] = total).  in may alias out+0..n-1? no.
size_t scan_workspace_bytes(int64_t n);
int exclusive_scan_i32(const int32_t* in, int32_t* out, int64_t n, void* ws, size_t ws_bytes,
                       cudaStream_t stream);
// the same scan with int64 sums and output: exact for totals of 2^31 and more
size_t scan_i64_workspace_bytes(int64_t n);
int exclusive_scan_i64(const int32_t* in, int64_t* out, int64_t n, void* ws, size_t ws_bytes,
                       cudaStream_t stream);

// rowptr[r] = lower_bound(sorted_keys, r) for r in [0, n_rows]
int rowptr_from_sorted(const uint32_t* sorted_keys, int64_t n, int32_t* rowptr, int64_t n_rows,
                       cudaStream_t stream);

static inline int bits_for(int64_t n) {  // bits needed to represent values in [0, n)
  int b = 1;
  while (b < 32 && (int64_t(1) << b) < n) ++b;
  return b;
}

}  // namespace sgb
