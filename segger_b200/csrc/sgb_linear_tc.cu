// Error-compensated split-TF32 GEMM on Blackwell 5th-gen tensor cores (tcgen05.mma, accumulators in TMEM)
// with the fp32 accumulation finished OUTSIDE the tensor core.
//
//   C[m,n] = sum_k A(m,k) * B(n,k)            fp32 in, fp32 out
//
// Each fp32 operand x is split into x_hi = rn_tf32(x) and x_lo = rn_tf32(x - x_hi) (x = hi + lo to 2^-24) and
//   A*B ~= A_lo*B_lo + A_lo*B_hi + A_hi*B_lo + A_hi*B_hi   (3 or 4 kind::tf32 MMAs per K=8 step, small terms first).
// The tensor core adds every MMA into its fp32 accumulator with ROUND-TOWARD-ZERO: a biased error that grows
// with the number of accumulations (measured 4.3e-6 relative at K=256) and that the attention backward of the
// following GATv2 layer amplifies ~10^3x (DESIGN.md "GEMM precision").  So the reduction is cut into CHUNKS of
// `kc` K=8 steps: each chunk is accumulated in TMEM from zero, read back with tcgen05.ld and added into a
// register accumulator with round-to-nearest FADDs (the scheme of Ootomo & Yokota for mma.sync, here with TMEM
// double-buffered per chunk so the read-back overlaps the next chunk's MMAs).  kc = 1 leaves one truncation per
// 8 products; kc = 4 (one 32-deep stage) is the fast setting for gradients.
//
// Persistent, warp-specialised CTA (one per SM, 288 threads):
//   warps 0-3   producers: cp.async (LDGSTS) of the raw A (and, for wgrad, B) k-slab straight into the stage slot
//               S-1 slabs ahead, then an in-place hi/lo split with swizzle-128B stores into the UMMA canonical shared-memory layout (K-major or
//               MN-major, so x W^T, dy W and dy^T x all run without a transpose), fence.proxy.async + mbarrier
//               arrive.  Weights (forward / dgrad B operand) are split and laid out ONCE per call by
//               pack_b_kernel in the exact shared-memory image, and a stage's B tile is one cp.async.bulk
//               (UBLKCP) completing on the same mbarrier -- no per-tile re-conversion of the weights.
//   warp  4     MMA issuer: one elected lane issues tcgen05.mma (M=128, N=BN, K=8); tcgen05.commit releases the
//               smem stage / publishes the chunk accumulator; owns TMEM alloc/dealloc.
//   warps 5-8   epilogue: per chunk tcgen05.ld (32 lanes x 32 columns) -> acc += chunk (FADD.RN); per tile
//               bias / activation / act' / accumulate -> 128-bit global stores.
// Split-K over the reduction (wgrad: reduction = number of rows) writes per-split partials that a
// fixed-order reduce kernel sums -> deterministic.
//
// Replaces cuBLAS SGEMM reached from PyG Linear / torch.nn.Linear
// (/root/reference/src/segger/models/ist_encoder.py:43-47,111-131,261,282-286).
#include "sgb_api_internal.cuh"
#include "sgb_linear.cuh"

namespace sgb {
namespace {

constexpr int BM = 128;            // UMMA M (cta_group::1)
constexpr int BK = 32;             // fp32 per 128-byte swizzle row = reduction elements per stage
constexpr int kProducerWarps = 4;   // warpgroup 0
constexpr int kProducerThreads = kProducerWarps * 32;
constexpr int kEpiWarp0 = kProducerWarps;      // warpgroups 1-2
constexpr int kEpiWarps = 8;       // two per TMEM lane quarter, each owning half of the tile's columns
constexpr int kMmaWarp = kEpiWarp0 + kEpiWarps;   // warpgroup 3: MMA issuer, packed-weight loader, two idle warps
constexpr int kBLoadWarp = kMmaWarp + 1;
constexpr int kHelperWarp0 = kMmaWarp + 2;      // wgrad: the two otherwise idle warps of warpgroup 3 stage + split half of B
constexpr int kHelperThreads = 64;
constexpr int kThreads = 16 * 32;  // 512: four whole warpgroups, so setmaxnreg can move registers between the roles
// Register budget (64K per SM, 128 per thread at launch): warpgroup 3 gives up 72 per thread, the producers take them.
constexpr int kRegsProducer = 184, kRegsControl = 72;   // 128 x 184 + 256 x 128 + 128 x 72 = 64K
constexpr int kMaxStages = 4;
// epilogue transpose buffer: per warp 32 rows x (PW + 4) floats, PW = columns written out per pass
constexpr int kPW = 16;            // 64-byte row segments per write-out pass: leaves shared memory for a third 64 KB stage
constexpr size_t stg_bytes(int pw) { return static_cast<size_t>(kEpiWarps) * 32 * (pw + 4) * sizeof(float); }
constexpr int kAccBufs = 4;        // TMEM chunk accumulators in flight (4 x BN columns <= 512)

struct TcParams {
  const float *A, *B;
  int64_t lda, ldb;
  int64_t M, N, K;          // MN extent of A, MN extent of B, reduction extent
  int splits;
  int64_t k_per_split;      // multiple of BK
  float* C;                 // output, or split-K partials [splits][M][N] (ldc = N)
  int64_t ldc;
  const float* bias;
  int act;
  float* C_act;
  int64_t ldca;
  int accumulate;
  const float* act_pre;
  int64_t ld_pre;
  int stages;
  int terms;                // 3: hi*hi + lo*hi + hi*lo (~2^-22);  4: + lo*lo (fp32-exact products)
  int kc;                   // K=8 steps per TMEM chunk (1, 2 or 4): accumulations done inside the tensor core
  int ks;                   // SS kernel, kc == BK/8 only: k-STAGES per TMEM chunk (wgrad: the chunk read-back, not the
                            // tensor core, paced the 32-deep chunks of a reduction over 10^6 rows); 0 / 1 = one stage
  float* colsum;            // wgrad only: column sums of A's source (db = sum_m dy[m, :]): [splits][M] partials, or db itself
  int colsum_accumulate;    // splits == 1: add into db
  int dbg;                  // timing experiments only (SEGGER_B200_TC_DBG bitmask): results are wrong when set
  const float* Bp;          // B_PACKED: pre-split weights in the shared-memory tile image [n-tile][k-stage][hi|lo]
  // forward only: C[m, :] += gtab[gids[m], :] -- the part of the product that depends on the row only through a small
  // integer id (the gene-embedding half of ISTEncoder's first projection) is a table lookup, not a GEMM
  const void* gids;
  int gid_bytes;
  const float* gtab;
  int64_t ld_gtab;
};

// Timing knock-outs (SEGGER_B200_TC_DBG, scripts/gemm_knockouts*.sh) exist only in -DSGB_TC_DEBUG builds: the flag
// tests sat in the hottest loops of warp roles whose instruction count is the critical path.
__device__ __forceinline__ int tc_dbg(const TcParams& p) {
#ifdef SGB_TC_DEBUG
  return p.dbg;
#else
  (void)p;
  return 0;
#endif
}

// ---- PTX wrappers ---------------------------------------------------------------------------
__device__ __forceinline__ uint32_t smem_u32(const void* p) { return static_cast<uint32_t>(__cvta_generic_to_shared(p)); }
__device__ __forceinline__ void mbar_init(uint32_t bar, uint32_t count) {
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(bar), "r"(count) : "memory");
}
__device__ __forceinline__ void mbar_arrive(uint32_t bar) {
  asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(bar) : "memory");
}
__device__ __forceinline__ void mbar_wait(uint32_t bar, uint32_t parity) {
  uint32_t ok;
  do {
    asm volatile(
        "{\n\t.reg .pred p;\n\t"
        "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\t"
        "selp.u32 %0, 1, 0, p;\n\t}"
        : "=r"(ok) : "r"(bar), "r"(parity) : "memory");
  } while (!ok);
}
__device__ __forceinline__ void mbar_arrive_expect_tx(uint32_t bar, uint32_t bytes) {
  asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(bar), "r"(bytes) : "memory");
}
__device__ __forceinline__ void bulk_g2s(uint32_t dst, const void* src, uint32_t bytes, uint32_t bar) {
  asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];"
               ::"r"(dst), "l"(src), "r"(bytes), "r"(bar) : "memory");
}
__device__ __forceinline__ void fence_barrier_init() { asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory"); }
__device__ __forceinline__ void fence_proxy_async() { asm volatile("fence.proxy.async.shared::cta;" ::: "memory"); }
__device__ __forceinline__ void tc_fence_before() { asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void tc_fence_after() { asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void tc_commit(uint32_t bar) {
  asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(bar) : "memory");
}
__device__ __forceinline__ void tc_mma_tf32(uint32_t tmem_d, uint64_t adesc, uint64_t bdesc, uint32_t idesc, uint32_t accum) {
  asm volatile(
      "{\n\t.reg .pred p;\n\t"
      "setp.ne.b32 p, %4, 0;\n\t"
      "tcgen05.mma.cta_group::1.kind::tf32 [%0], %1, %2, %3, {%5, %5, %5, %5}, p;\n\t}"
      ::"r"(tmem_d), "l"(adesc), "l"(bdesc), "r"(idesc), "r"(accum), "r"(0u) : "memory");
}
__device__ __forceinline__ void tc_ld32(uint32_t taddr, uint32_t (&r)[32]) {
  asm volatile(
      "tcgen05.ld.sync.aligned.32x32b.x32.b32 "
      "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, "
      "%16, %17, %18, %19, %20, %21, %22, %23, %24, %25, %26, %27, %28, %29, %30, %31}, [%32];"
      : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]),
        "=r"(r[8]), "=r"(r[9]), "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15]),
        "=r"(r[16]), "=r"(r[17]), "=r"(r[18]), "=r"(r[19]), "=r"(r[20]), "=r"(r[21]), "=r"(r[22]), "=r"(r[23]),
        "=r"(r[24]), "=r"(r[25]), "=r"(r[26]), "=r"(r[27]), "=r"(r[28]), "=r"(r[29]), "=r"(r[30]), "=r"(r[31])
      : "r"(taddr) : "memory");
}
__device__ __forceinline__ void tc_ld16(uint32_t taddr, uint32_t (&r)[16]) {
  asm volatile(
      "tcgen05.ld.sync.aligned.32x32b.x16.b32 "
      "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15}, [%16];"
      : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]),
        "=r"(r[8]), "=r"(r[9]), "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15])
      : "r"(taddr) : "memory");
}
__device__ __forceinline__ void tc_wait_ld() { asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory"); }

// ---- descriptors (cute/arch/mma_sm100_desc.hpp bit layout) -----------------------------------
// instruction descriptor: c=F32, a=b=TF32, majors, N>>3 at bit 17, M>>4 at bit 24
__host__ __device__ constexpr uint32_t make_idesc(int n, bool a_mn, bool b_mn) {
  return (1u << 4) | (2u << 7) | (2u << 10) | (static_cast<uint32_t>(a_mn) << 15) | (static_cast<uint32_t>(b_mn) << 16) |
         (static_cast<uint32_t>(n >> 3) << 17) | (static_cast<uint32_t>(BM >> 4) << 24);
}
// shared-memory matrix descriptor, version 1 (Blackwell).  layout_type: 2 = SWIZZLE_128B (K-major
// operands), 1 = SWIZZLE_128B_BASE32B (the only layout tcgen05 accepts for MN-major tf32 operands).
__device__ __forceinline__ uint64_t make_sdesc(uint32_t saddr, uint32_t lbo_bytes, uint32_t sbo_bytes, uint32_t layout_type) {
  const uint64_t lo = static_cast<uint64_t>((saddr >> 4) & 0x3FFFu) | (static_cast<uint64_t>((lbo_bytes >> 4) & 0x3FFFu) << 16);
  const uint64_t hi = static_cast<uint64_t>((sbo_bytes >> 4) & 0x3FFFu) | (1ull << 14) | (static_cast<uint64_t>(layout_type) << 29);
  return lo | (hi << 32);
}

__device__ __forceinline__ float act_apply(float x, int act) {
  if (act == SGB_ACT_GELU) return gelu_erf(x);
  if (act == SGB_ACT_SILU) return x / (1.0f + __expf(-x));
  return x;
}
__device__ __forceinline__ float act_grad(float x, int act) {
  if (act == SGB_ACT_GELU) return gelu_erf_grad(x);
  if (act == SGB_ACT_SILU) {
    const float s = 1.0f / (1.0f + __expf(-x));
    return s * (1.0f + x * (1.0f - s));
  }
  return 1.0f;
}

// Round-to-nearest to the 11 significant bits of TF32 (low 13 mantissa bits cleared, so the tensor
// core's own truncation is a no-op).  x = hi + lo with hi = rn(x), lo = rn(x - hi) represents x to
// 2^-24 relative -- i.e. the split itself loses nothing of an fp32 value.
__device__ __forceinline__ float rn_tf32(float x) {
  return __uint_as_float((__float_as_uint(x) + 0x1000u) & 0xFFFFE000u);
}
// The low half of a split is only ever a tensor-core operand: kind::tf32 ignores the 13 low mantissa bits of its
// operands, so rounding to nearest needs the carry (+ 2^12 ulp) but not the mask.  (The high half keeps the mask: it is
// also subtracted from x, which needs the exact tf32 value.)  SEGGER_B200-internal: parity tests compare bit-identical
// error figures with and without this shortcut.
__device__ __forceinline__ float rn_tf32_operand(float x) { return __uint_as_float(__float_as_uint(x) + 0x1000u); }

// Operand slab staging: EXT rows of the MN dimension x BK reduction elements starting at (mn0, k0).
// Every producer thread owns NV 16-byte chunks of the slab: it copies them global -> shared with cp.async
// (LDGSTS, zero-filled out of range) into a RAW ring several slabs ahead of the converter, later reads the same
// chunks back, splits them into hi / lo and stores both into the stage's UMMA tiles.  Raw, hi and lo tiles use
// the same canonical swizzle-128B offsets, so a thread only ever touches its own chunks (no cross-thread
// synchronisation: cp.async.wait_group suffices) and the accesses stay bank-conflict free.
//   K-major  (MN == false): element (mn, k) at src[mn * ld + k]; smem row = one mn, 128 B of k.
//   MN-major (MN == true) : element (mn, k) at src[k * ld + mn]; smem row = one k, 128 B of mn;
//                           512-byte atoms (4 k-rows, Swizzle<2,5,2>: 32-byte chunk ^= k % 4)
//                           ordered [k-group of 4][mn-block of 32].
template <int EXT, bool MN>
__device__ __forceinline__ uint32_t chunk_offset(int ri, int chunk) {
  if (!MN) return (ri >> 3) * 1024 + (ri & 7) * 128 + ((chunk ^ (ri & 7)) << 4);
  const int kk = ri & 31, blk = ri >> 5;
  const int c16 = ((((chunk >> 1) ^ (kk & 3)) << 1) | (chunk & 1));
  return ((kk >> 2) * (EXT / 32) + blk) * 512 + (kk & 3) * 128 + (c16 << 4);
}

__device__ __forceinline__ void cp_async16_zfill(uint32_t saddr, const void* g, uint32_t src_bytes) {
  asm volatile("cp.async.cg.shared.global [%0], [%1], 16, %2;" ::"r"(saddr), "l"(g), "r"(src_bytes) : "memory");
}
__device__ __forceinline__ void cp_async_commit() { asm volatile("cp.async.commit_group;" ::: "memory"); }
template <int N>
__device__ __forceinline__ void cp_async_wait() { asm volatile("cp.async.wait_group %0;" ::"n"(N) : "memory"); }

template <int EXT, bool MN>
__device__ __forceinline__ void stage_raw(const float* __restrict__ src, int64_t ld, int64_t mn0, int64_t mn_end, int64_t k0,
                                          int64_t k_end, uint32_t raw_tile, int t) {
  constexpr int NV = EXT * 8 / kProducerThreads;
  const int chunk = t & 7;
#pragma unroll
  for (int i = 0; i < NV; ++i) {
    const int ri = (t >> 3) + (kProducerThreads / 8) * i;       // 0 .. EXT-1 (K-major) or 0 .. 32*(EXT/32)-1
    const float* g = src;
    bool ok;
    if (!MN) {
      const int64_t mn = mn0 + ri, k = k0 + chunk * 4;
      ok = mn < mn_end && k < k_end;                               // K % 4 == 0 guaranteed by the dispatcher
      if (ok) g = src + mn * ld + k;
    } else {
      const int kk = ri & 31, blk = ri >> 5;
      const int64_t k = k0 + kk, mn = mn0 + blk * 32 + chunk * 4;
      ok = k < k_end && mn < mn_end;                               // MN % 4 == 0 guaranteed
      if (ok) g = src + k * ld + mn;
    }
    cp_async16_zfill(raw_tile + chunk_offset<EXT, MN>(ri, chunk), g, ok ? 16u : 0u);
  }
}

// MN-major staging with everything that depends on the tile only hoisted out of the per-slab path (wgrad: both operands
// stream through here): `base` = src + mn0 + chunk * 4, `mn_ok` bit b = this thread's columns of 32-wide block b exist,
// `raw0` = slot address + this thread's first chunk offset.  Row r0 + 16 i of the slab is reduction row r0 + 16 (i & 1) of
// block i >> 1, whose shared-memory offset differs from the first by a compile-time constant.
template <int EXT, int NVL = EXT * 8 / kProducerThreads>
__device__ __forceinline__ void stage_raw_mn_fast(const float* __restrict__ base, int64_t ld, uint32_t mn_ok, int64_t k0,
                                                  int64_t k_end, uint32_t raw0, int r0) {
  constexpr int NV = NVL;
  const int64_t k = k0 + r0;
  const float* g0 = base + k * ld;
  const int64_t half = 16 * ld;
  const bool k_ok0 = k < k_end, k_ok1 = k + 16 < k_end;
#pragma unroll
  for (int i = 0; i < NV; ++i) {
    const bool ok = ((i & 1) ? k_ok1 : k_ok0) && ((mn_ok >> (i >> 1)) & 1u);
    // src-size 0 reads nothing (pure zero fill): the address of an out-of-range chunk is never dereferenced, so it is
    // not replaced by a safe one -- the two row pointers then serve all chunks with immediate offsets
    const float* g = ((i & 1) ? g0 + half : g0) + (i >> 1) * 32;
    cp_async16_zfill(raw0 + static_cast<uint32_t>((4 * (i & 1) * (EXT / 32) + (i >> 1)) * 512), g, ok ? 16u : 0u);
  }
}

// wgrad helpers (64 threads, ht = 0..63): the upper half of B's 32-wide MN blocks (blk >= EXT / 64), all 32 reduction
// rows: thread ht owns chunk ht & 7 of rows (ht >> 3) + 8 j, j < 4, of each of those blocks.  `base` / `mn_ok` as above.
template <int EXT>
__device__ __forceinline__ uint32_t helper_off0(int ht) {
  return chunk_offset<EXT, true>((EXT / 64) * 32 + (ht >> 3), ht & 7);
}
template <int EXT>
__device__ __forceinline__ void stage_raw_mn_helper(const float* __restrict__ base, int64_t ld, uint32_t mn_ok, int64_t k0,
                                                    int64_t k_end, uint32_t raw0, int ht) {
  const int64_t k = k0 + (ht >> 3);
  const float* g0 = base + k * ld + (EXT / 64) * 32;
  const int64_t step = 8 * ld;
#pragma unroll
  for (int j = 0; j < 4; ++j) {
    const bool kok = k + 8 * j < k_end;
#pragma unroll
    for (int b = 0; b < EXT / 64; ++b) {
      const bool ok = kok && ((mn_ok >> (EXT / 64 + b)) & 1u);
      cp_async16_zfill(raw0 + static_cast<uint32_t>((2 * j * (EXT / 32) + b) * 512), g0 + j * step + b * 32, ok ? 16u : 0u);
    }
  }
}
template <int EXT>
__device__ __forceinline__ void split_slab_helper(uint8_t* hi_tile, uint8_t* lo_tile, int ht) {
  const uint32_t off0 = helper_off0<EXT>(ht);
#pragma unroll
  for (int j = 0; j < 4; ++j) {
#pragma unroll
    for (int b = 0; b < EXT / 64; ++b) {
      const uint32_t off = off0 + static_cast<uint32_t>((2 * j * (EXT / 32) + b) * 512);
      const float4 v = *reinterpret_cast<const float4*>(hi_tile + off);
      float4 h, l;
      h.x = rn_tf32(v.x); l.x = rn_tf32_operand(v.x - h.x);
      h.y = rn_tf32(v.y); l.y = rn_tf32_operand(v.y - h.y);
      h.z = rn_tf32(v.z); l.z = rn_tf32_operand(v.z - h.z);
      h.w = rn_tf32(v.w); l.w = rn_tf32_operand(v.w - h.w);
      *reinterpret_cast<float4*>(hi_tile + off) = h;
      *reinterpret_cast<float4*>(lo_tile + off) = l;
    }
  }
}

// SUM (MN-major only): also accumulate the raw values per 32-wide MN block into cs[] -- thread t sees, for every
// block, the same 4 columns (chunk t & 7) of two reduction rows per slab, so cs[blk] is a partial column sum.
template <int EXT, bool MN, bool SUM = false, int NVL = EXT * 8 / kProducerThreads>
__device__ __forceinline__ void split_slab(const uint8_t* raw_tile, uint8_t* hi_tile, uint8_t* lo_tile, int t, float4* cs = nullptr) {
  constexpr int NV = NVL;
  const int chunk = t & 7;
#pragma unroll
  for (int i = 0; i < NV; ++i) {
    const int ri = (t >> 3) + (kProducerThreads / 8) * i;
    const uint32_t off = chunk_offset<EXT, MN>(ri, chunk);
    const float4 v = *reinterpret_cast<const float4*>(raw_tile + off);
    if constexpr (SUM) {
      float4& c = cs[(kProducerThreads / 8) * i / 32];     // blk = ri >> 5 (t >> 3 < 16)
      c.x += v.x; c.y += v.y; c.z += v.z; c.w += v.w;
    }
    float4 h, l;
    h.x = rn_tf32(v.x); l.x = rn_tf32_operand(v.x - h.x);
    h.y = rn_tf32(v.y); l.y = rn_tf32_operand(v.y - h.y);
    h.z = rn_tf32(v.z); l.z = rn_tf32_operand(v.z - h.z);
    h.w = rn_tf32(v.w); l.w = rn_tf32_operand(v.w - h.w);
    *reinterpret_cast<float4*>(hi_tile + off) = h;
    *reinterpret_cast<float4*>(lo_tile + off) = l;
  }
}

// Weight pre-pack: B(n, k) for n < N, k < K (zero padded) -> per (n-tile, k-stage) block of 2*BN*128 bytes holding
// the hi tile then the lo tile in the K-major SWIZZLE_128B image the MMA descriptors expect.
//   src_mn == 0: B(n, k) = w[n * ldw + k]  (forward: w is [N, K])
//   src_mn == 1: B(n, k) = w[k * ldw + n]  (dgrad: B(k_out, n_in) = w[n_in, k_out])
template <int BN>
__global__ void pack_b_kernel(const float* __restrict__ w, int64_t ldw, int64_t N, int64_t K, int src_mn, int num_n, int num_ks,
                              float* __restrict__ out) {
  const int64_t idx = static_cast<int64_t>(blockIdx.x) * blockDim.x + threadIdx.x;   // one 16-byte chunk (4 k) of one row n
  const int64_t total = static_cast<int64_t>(num_n) * BN * num_ks * 8;
  if (idx >= total) return;
  const int c = static_cast<int>(idx & 7);
  const int64_t t = idx >> 3;
  const int ks = static_cast<int>(t % num_ks);
  const int64_t nrow = t / num_ks;                 // global padded row
  const int nb = static_cast<int>(nrow / BN), r = static_cast<int>(nrow % BN);
  float v[4];
#pragma unroll
  for (int e = 0; e < 4; ++e) {
    const int64_t k = static_cast<int64_t>(ks) * BK + c * 4 + e;
    v[e] = (nrow < N && k < K) ? (src_mn ? __ldg(w + k * ldw + nrow) : __ldg(w + nrow * ldw + k)) : 0.f;
  }
  float4 h, l;
  h.x = rn_tf32(v[0]); l.x = rn_tf32(v[0] - h.x);
  h.y = rn_tf32(v[1]); l.y = rn_tf32(v[1] - h.y);
  h.z = rn_tf32(v[2]); l.z = rn_tf32(v[2] - h.z);
  h.w = rn_tf32(v[3]); l.w = rn_tf32(v[3] - h.w);
  const uint32_t off = (r >> 3) * 1024 + (r & 7) * 128 + ((c ^ (r & 7)) << 4);
  uint8_t* blk = reinterpret_cast<uint8_t*>(out) + (static_cast<size_t>(nb) * num_ks + ks) * (2 * BN * 128);
  *reinterpret_cast<float4*>(blk + off) = h;
  *reinterpret_cast<float4*>(blk + BN * 128 + off) = l;
}

template <int BN, bool A_MN, bool B_MN, bool B_PACKED, int S>
__global__ void __launch_bounds__(kThreads, 1) gemm_tf32x3_kernel(const TcParams p) {
  extern __shared__ uint8_t smem_raw[];
  constexpr uint32_t kATile = BM * 128;            // bytes of one hi (or lo) A tile
  constexpr uint32_t kBTile = BN * 128;
  constexpr uint32_t kStageBytes = 2 * kATile + 2 * kBTile;
  constexpr uint32_t kTmemCols = kAccBufs * BN;    // 256 or 512: a power of two >= 32
  static_assert(BN <= 128, "the register accumulator holds one row x BN/2 columns per epilogue thread");
  constexpr int CW = BN / 2;                        // columns per epilogue warp
  constexpr int PW = kPW;                           // columns per write-out pass
  constexpr int kStgLd = PW + 4;
  static_assert(!(B_PACKED && B_MN), "packed weights are always K-major in shared memory");

  uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~static_cast<uintptr_t>(1023));
  __shared__ uint64_t bar_full[kMaxStages], bar_empty[kMaxStages], bar_tfull[kAccBufs], bar_tempty[kAccBufs];
  __shared__ uint32_t tmem_base_holder;

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  constexpr int stages = S;
  // wgrad (both operands streamed, MN-major): the producers were the busiest role (ncu source view: 82 % of their
  // cycles issuing); the two idle warps of warpgroup 3 take the upper half of B's columns off them
  constexpr bool kHelp = A_MN && B_MN && !B_PACKED;
  constexpr int kNvB = BN * 8 / kProducerThreads / (kHelp ? 2 : 1);     // B row slots per main producer thread

  if (threadIdx.x == 0) {
    for (int s = 0; s < stages; ++s) {
      mbar_init(smem_u32(&bar_full[s]), kProducerThreads + (B_PACKED ? 1 : 0) + (kHelp ? kHelperThreads : 0));
      mbar_init(smem_u32(&bar_empty[s]), 1);
    }
    for (int a = 0; a < kAccBufs; ++a) {
      mbar_init(smem_u32(&bar_tfull[a]), 1);
      mbar_init(smem_u32(&bar_tempty[a]), kEpiWarps * 32);
    }
    fence_barrier_init();
  }
  if (warp == kMmaWarp) {
    asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(&tmem_base_holder)), "r"(kTmemCols) : "memory");
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
  }
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = tmem_base_holder;

  const int64_t num_m = (p.M + BM - 1) / BM, num_n = (p.N + BN - 1) / BN;
  const int64_t tiles = num_m * num_n * p.splits;
  const int64_t num_ks = (p.K + BK - 1) / BK;      // k-stages of the whole reduction (packed-B block index)

  // tile / k-slab cursor shared by the producer, loader and (implicitly) MMA / epilogue loops: tiles are dealt
  // round-robin to the persistent CTAs, a tile's reduction range is cut into BK-deep slabs
  struct Cur { int64_t tile, k0, ke, mb, nb; bool live; const float *a_base, *b_base; uint32_t a_ok, b_ok; };
  const int st_chunk = threadIdx.x & 7;              // producers: 16-byte chunk this thread stages (MN-major fast path)
  auto tile_range = [&](Cur& c) {
    const int64_t sp = c.tile / (num_n * num_m);
    c.nb = c.tile % num_n;
    c.mb = (c.tile / num_n) % num_m;
    c.k0 = sp * p.k_per_split;
    c.ke = min(p.K, c.k0 + p.k_per_split);
    if constexpr (A_MN) {
      const int64_t mn = c.mb * BM + st_chunk * 4;
      c.a_base = p.A + mn;
      c.a_ok = 0;
#pragma unroll
      for (int b = 0; b < BM / 32; ++b) c.a_ok |= (mn + 32 * b < p.M) ? (1u << b) : 0u;
    }
    if constexpr (B_MN && !B_PACKED) {
      const int64_t mn = c.nb * BN + st_chunk * 4;
      c.b_base = p.B + mn;
      c.b_ok = 0;
#pragma unroll
      for (int b = 0; b < BN / 32; ++b) c.b_ok |= (mn + 32 * b < p.N) ? (1u << b) : 0u;
    }
  };
  auto init = [&](Cur& c) {
    c.tile = blockIdx.x;
    c.live = c.tile < tiles;
    if (c.live) tile_range(c);
  };
  auto advance = [&](Cur& c) {
    c.k0 += BK;
    if (c.k0 >= c.ke) {
      c.tile += gridDim.x;
      c.live = c.tile < tiles;
      if (c.live) tile_range(c);
    }
  };

  if (warp < kProducerWarps) {
    // ===================================== producers =====================================
    asm volatile("setmaxnreg.inc.sync.aligned.u32 %0;" ::"n"(kRegsProducer));
    const int t = threadIdx.x;
    // A stage slot is filled in place: cp.async lands the RAW fp32 slab(s) in the slot's hi tiles as soon as the
    // MMAs of the slot's previous use retire (S-1 slabs ahead of the split), the same threads later read their
    // own chunks back, write hi over them and lo beside them.  Packed weights (forward / dgrad) arrive through
    // the loader warp instead.  (A register-staged variant -- global loads held in registers four slabs ahead,
    // slots written the moment they free up -- measured no faster: these GEMMs are bound by shared-memory
    // bandwidth, which the tensor core's own operand reads nearly saturate at N = 128; profiles/r1c_gemm_knockouts.txt.)
    int istage = 0, cstage = 0;
    uint32_t iphase = 0;
    const int st_r0 = t >> 3;
    const uint32_t st_offa = chunk_offset<BM, true>(st_r0, st_chunk), st_offb = chunk_offset<BN, true>(st_r0, st_chunk);
    auto issue = [&](const Cur& c) {
      mbar_wait(smem_u32(&bar_empty[istage]), iphase ^ 1u);
      uint8_t* st = smem + static_cast<size_t>(istage) * kStageBytes;
      if constexpr (A_MN) stage_raw_mn_fast<BM>(c.a_base, p.lda, c.a_ok, c.k0, c.ke, smem_u32(st) + st_offa, st_r0);
      else stage_raw<BM, false>(p.A, p.lda, c.mb * BM, p.M, c.k0, c.ke, smem_u32(st), t);
      if constexpr (!B_PACKED) {
        if constexpr (B_MN) stage_raw_mn_fast<BN, kNvB>(c.b_base, p.ldb, c.b_ok, c.k0, c.ke, smem_u32(st + 2 * kATile) + st_offb, st_r0);
        else stage_raw<BN, false>(p.B, p.ldb, c.nb * BN, p.N, c.k0, c.ke, smem_u32(st + 2 * kATile), t);
      }
      if (++istage == S) { istage = 0; iphase ^= 1u; }
    };
    // fused bias gradient (wgrad): column sums of dy, accumulated while its slabs pass through the producers
    constexpr bool kColsum = A_MN;
    float4 cs[kColsum ? BM / 32 : 1];
#pragma unroll
    for (int i = 0; i < (kColsum ? BM / 32 : 1); ++i) cs[i] = make_float4(0.f, 0.f, 0.f, 0.f);
    float* red = reinterpret_cast<float*>(smem + static_cast<size_t>(S) * kStageBytes + stg_bytes(kPW));
    auto flush_colsum = [&](int64_t tl) {
      if constexpr (kColsum) {
        const int64_t nb = tl % num_n, mb = (tl / num_n) % num_m, sp = tl / (num_n * num_m);
        if (p.colsum && nb == 0) {                   // one n-tile per (m-block, split) owns the sum
#pragma unroll
          for (int i = 0; i < BM / 32; ++i) *reinterpret_cast<float4*>(red + t * (BM / 8) + i * 4) = cs[i];
          asm volatile("bar.sync 1, %0;" ::"n"(kProducerThreads) : "memory");
          if (t < BM / 4) {
            const int blk = t >> 3, chunk = t & 7;
            float4 a = make_float4(0.f, 0.f, 0.f, 0.f);
            for (int j = 0; j < kProducerThreads / 8; ++j) {     // fixed order: deterministic
              const float4 v = *reinterpret_cast<const float4*>(red + ((j << 3) | chunk) * (BM / 8) + blk * 4);
              a.x += v.x; a.y += v.y; a.z += v.z; a.w += v.w;
            }
            const int64_t n = mb * BM + blk * 32 + chunk * 4;
            float* dst = p.colsum + (p.splits > 1 ? sp * p.M : 0) + n;
            const float o[4] = {a.x, a.y, a.z, a.w};
#pragma unroll
            for (int e = 0; e < 4; ++e)
              if (n + e < p.M) dst[e] = (p.splits == 1 && p.colsum_accumulate) ? dst[e] + o[e] : o[e];
          }
          asm volatile("bar.sync 1, %0;" ::"n"(kProducerThreads) : "memory");
        }
#pragma unroll
        for (int i = 0; i < BM / 32; ++i) cs[i] = make_float4(0.f, 0.f, 0.f, 0.f);
      }
    };
    Cur pi, ci;
    init(pi);
    init(ci);
#pragma unroll
    for (int i = 0; i < S - 1; ++i) {
      if (pi.live) { issue(pi); advance(pi); }
      cp_async_commit();
    }
    while (ci.live) {
      cp_async_wait<S - 2>();                       // this thread's chunks of slab `ci` have landed
      uint8_t* st = smem + static_cast<size_t>(cstage) * kStageBytes;
      if (!(tc_dbg(p) & 2)) split_slab<BM, A_MN, kColsum>(st, st, st + kATile, t, cs);
      if constexpr (!B_PACKED) if (!(tc_dbg(p) & 2)) split_slab<BN, B_MN, false, kNvB>(st + 2 * kATile, st + 2 * kATile, st + 2 * kATile + kBTile, t);
      fence_proxy_async();
      mbar_arrive(smem_u32(&bar_full[cstage]));
      if (++cstage == S) cstage = 0;
      const int64_t done_tile = ci.tile;
      advance(ci);
      if (!ci.live || ci.tile != done_tile) flush_colsum(done_tile);
      if (pi.live) { issue(pi); advance(pi); }      // refill the slot the tensor core finished with
      cp_async_commit();
    }
    cp_async_wait<0>();
  } else if (warp >= kMmaWarp) {
    asm volatile("setmaxnreg.dec.sync.aligned.u32 %0;" ::"n"(kRegsControl));
    if (B_PACKED && warp == kBLoadWarp && lane == 0) {
      // ===================================== packed-weight loader =====================================
      // one bulk copy (hi tile + lo tile of the slot's k-slab, pre-split by pack_b_kernel) per stage slot, issued
      // the moment the tensor core frees the slot: S-1 slots ahead of the MMAs.
      Cur b;
      init(b);
      int stage = 0;
      uint32_t phase = 0;
      while (b.live) {
        mbar_wait(smem_u32(&bar_empty[stage]), phase ^ 1u);
        uint8_t* st = smem + static_cast<size_t>(stage) * kStageBytes;
        const int64_t blk = b.nb * num_ks + b.k0 / BK;
        mbar_arrive_expect_tx(smem_u32(&bar_full[stage]), 2 * kBTile);
        bulk_g2s(smem_u32(st + 2 * kATile), p.Bp + static_cast<size_t>(blk) * (2 * BN * 32), 2 * kBTile, smem_u32(&bar_full[stage]));
        if (++stage == S) { stage = 0; phase ^= 1u; }
        advance(b);
      }
    }
    if constexpr (kHelp) {
      if (warp >= kHelperWarp0) {
        // ===================================== wgrad helpers =====================================
        // same protocol as the producers (stage S-1 slabs ahead into the slot, later split the very same chunks in
        // place, arrive on the slot's full barrier), on the upper half of B's column blocks
        const int ht = threadIdx.x - kHelperWarp0 * 32;
        const uint32_t hoff = helper_off0<BN>(ht);
        int istage = 0, cstage = 0;
        uint32_t iphase = 0;
        auto issue = [&](const Cur& c) {
          mbar_wait(smem_u32(&bar_empty[istage]), iphase ^ 1u);
          uint8_t* st = smem + static_cast<size_t>(istage) * kStageBytes;
          stage_raw_mn_helper<BN>(c.b_base, p.ldb, c.b_ok, c.k0, c.ke, smem_u32(st + 2 * kATile) + hoff, ht);
          if (++istage == S) { istage = 0; iphase ^= 1u; }
        };
        Cur pi, ci;
        init(pi);
        init(ci);
#pragma unroll
        for (int i = 0; i < S - 1; ++i) {
          if (pi.live) { issue(pi); advance(pi); }
          cp_async_commit();
        }
        while (ci.live) {
          cp_async_wait<S - 2>();
          uint8_t* st = smem + static_cast<size_t>(cstage) * kStageBytes;
          if (!(tc_dbg(p) & 2)) split_slab_helper<BN>(st + 2 * kATile, st + 2 * kATile + kBTile, ht);
          fence_proxy_async();
          mbar_arrive(smem_u32(&bar_full[cstage]));
          if (++cstage == S) cstage = 0;
          advance(ci);
          if (pi.live) { issue(pi); advance(pi); }
          cp_async_commit();
        }
        cp_async_wait<0>();
      }
    }
    // ===================================== MMA issuer =====================================
    if (warp == kMmaWarp && lane == 0) {
      constexpr uint32_t idesc = make_idesc(BN, A_MN, B_MN);
      // K-major: LBO unused (1 -> encoded 16 B), SBO = 1024 B between 8-row groups, +32 B per k-step.
      // MN-major: LBO = 512 B between 32-wide MN blocks, SBO = (EXT/32)*512 B between 4-deep k groups;
      //           one K=8 MMA spans two k groups -> +2*SBO per k-step.
      constexpr uint32_t a_lbo = A_MN ? 512u : 16u, a_sbo = A_MN ? (BM / 32) * 512u : 1024u, a_step = A_MN ? 2 * a_sbo : 32u;
      constexpr uint32_t b_lbo = B_MN ? 512u : 16u, b_sbo = B_MN ? (BN / 32) * 512u : 1024u, b_step = B_MN ? 2 * b_sbo : 32u;
      constexpr uint32_t a_lt = A_MN ? 1u : 2u, b_lt = B_MN ? 1u : 2u;
      const int kc = p.kc;
      const int ks = (p.kc == BK / 8 && p.ks > 1) ? p.ks : 1;
      int in_chunk = 0;              // stages already accumulated into the current chunk (ks > 1)
      int stage = 0;
      uint32_t phase = 0;
      uint32_t cc = 0;               // chunk counter: TMEM buffer = cc % kAccBufs
      for (int64_t tile = blockIdx.x; tile < tiles; tile += gridDim.x) {
        const int64_t sp = tile / (num_n * num_m);
        const int64_t kb = sp * p.k_per_split, ke = min(p.K, kb + p.k_per_split);
        for (int64_t k0 = kb; k0 < ke; k0 += BK) {
          mbar_wait(smem_u32(&bar_full[stage]), phase);
          tc_fence_after();
          const uint32_t st = smem_u32(smem + static_cast<size_t>(stage) * kStageBytes);
          const uint32_t a_hi = st, a_lo = st + kATile, b_hi = st + 2 * kATile, b_lo = b_hi + kBTile;
          if (ks > 1) {           // a chunk spans ks stages (the last chunk of a split may be shorter)
            const uint32_t buf = cc % kAccBufs;
            if (in_chunk == 0) {
              mbar_wait(smem_u32(&bar_tempty[buf]), ((cc / kAccBufs) & 1u) ^ 1u);
              tc_fence_after();
            }
            const uint32_t d_tmem = tmem_base + buf * BN;
            uint32_t accum = in_chunk == 0 ? 0u : 1u;
            for (int term = ((tc_dbg(p) & 4) ? 3 : (p.terms >= 4 ? 0 : 1)); term < 4; ++term) {
              const uint32_t ab = (term == 3 || term == 2) ? a_hi : a_lo;
              const uint32_t bb = (term == 3 || term == 1) ? b_hi : b_lo;
              for (int j = 0; j < BK / 8; ++j) {
                tc_mma_tf32(d_tmem, make_sdesc(ab + j * a_step, a_lbo, a_sbo, a_lt), make_sdesc(bb + j * b_step, b_lbo, b_sbo, b_lt),
                            idesc, accum);
                accum = 1u;
              }
            }
            if (++in_chunk == ks || k0 + BK >= ke) {
              tc_commit(smem_u32(&bar_tfull[buf]));
              ++cc;
              in_chunk = 0;
            }
          } else
          for (int j0 = 0; j0 < BK / 8; j0 += kc, ++cc) {
            const uint32_t buf = cc % kAccBufs;
            mbar_wait(smem_u32(&bar_tempty[buf]), ((cc / kAccBufs) & 1u) ^ 1u);
            tc_fence_after();
            const uint32_t d_tmem = tmem_base + buf * BN;
            uint32_t accum = 0;
            // small terms first: the truncating accumulator then sees the big hi*hi products last
            for (int term = ((tc_dbg(p) & 4) ? 3 : (p.terms >= 4 ? 0 : 1)); term < 4; ++term) {
              const uint32_t ab = (term == 3 || term == 2) ? a_hi : a_lo;      // 0: lo*lo  1: lo*hi  2: hi*lo  3: hi*hi
              const uint32_t bb = (term == 3 || term == 1) ? b_hi : b_lo;
              for (int j = j0; j < j0 + kc; ++j) {
                tc_mma_tf32(d_tmem, make_sdesc(ab + j * a_step, a_lbo, a_sbo, a_lt), make_sdesc(bb + j * b_step, b_lbo, b_sbo, b_lt),
                            idesc, accum);
                accum = 1u;
              }
            }
            tc_commit(smem_u32(&bar_tfull[buf]));             // chunk accumulator complete
          }
          tc_commit(smem_u32(&bar_empty[stage]));             // frees this smem stage when the MMAs retire
          if (++stage == stages) { stage = 0; phase ^= 1u; }
        }
      }
    }
  } else {
    // ===================================== epilogue =====================================
    const int q = warp & 3;                                  // TMEM lane quarter this warp may access
    const int half = (warp - kEpiWarp0) >> 2;                // which half of the tile's columns
    float* stg = reinterpret_cast<float*>(smem + static_cast<size_t>(stages) * kStageBytes) +
                 (warp - kEpiWarp0) * (32 * kStgLd);
    const uint32_t lane_base = tmem_base + (static_cast<uint32_t>(q * 32) << 16) + static_cast<uint32_t>(half * CW);
    const int chunks_per_stage = (BK / 8) / p.kc;
    uint32_t cc = 0;
    for (int64_t tile = blockIdx.x; tile < tiles; tile += gridDim.x) {
      const int64_t nb = tile % num_n, mb = (tile / num_n) % num_m, sp = tile / (num_n * num_m);
      const int64_t n0 = nb * BN + half * CW;
      const int64_t kb = sp * p.k_per_split, ke = min(p.K, kb + p.k_per_split);
      const int64_t nstages = (ke - kb + BK - 1) / BK;
      const int64_t nchunks = (p.kc == BK / 8 && p.ks > 1) ? (nstages + p.ks - 1) / p.ks : nstages * chunks_per_stage;
      float acc[CW];
#pragma unroll
      for (int i = 0; i < CW; ++i) acc[i] = 0.f;
      for (int64_t c = 0; c < nchunks; ++c, ++cc) {
        const uint32_t buf = cc % kAccBufs;
        mbar_wait(smem_u32(&bar_tfull[buf]), (cc / kAccBufs) & 1u);
        tc_fence_after();
        // 13 warps put four on one SM sub-partition (16K registers): 128 registers per thread, so one
        // 32-column read-back is in flight per warp; two epilogue warps per sub-partition interleave
#pragma unroll
        for (int c0 = 0; c0 < CW; c0 += 32) {
          if (tc_dbg(p) & 1) break;
          uint32_t r0[32];
          tc_ld32(lane_base + buf * BN + c0, r0);
          tc_wait_ld();
#pragma unroll
          for (int j = 0; j < 32; ++j) acc[c0 + j] += __uint_as_float(r0[j]);
        }
        tc_fence_before();
        mbar_arrive(smem_u32(&bar_tempty[buf]));
      }
      // ---- tile write-out through a per-warp shared-memory transpose (32 rows x 32 columns at a time): the
      // accumulator of a thread is one ROW, but global memory wants a warp instruction to cover whole 128-byte
      // row segments.  Keeping the element-wise epilogue in a rolled loop also keeps the kernel's code small
      // (a fully unrolled per-register epilogue was 25k SASS instructions and ran out of the instruction cache).
      float* C = p.C + (p.splits > 1 ? sp * p.M * p.N : 0);
      constexpr int LR = PW / 4;                      // lanes per row in the write-out pass
      const int sub = lane / LR, c4 = (lane % LR) * 4;
      const bool vec_c = (p.ldc % 4 == 0) && aligned16(C) && (n0 % 4 == 0);
      const bool vec_a = p.C_act && (p.ldca % 4 == 0) && aligned16(p.C_act) && (n0 % 4 == 0);
      const bool vec_p = p.act_pre && (p.ld_pre % 4 == 0) && aligned16(p.act_pre) && (n0 % 4 == 0);
      // One ROLLED loop over the write-out passes: the body below (bias / accumulate / table gather / activation, each
      // behind a run-time flag) is emitted once instead of CW/PW times -- unrolled it was over half of the kernel's SASS
      // and the instruction cache, not the LSU, bounded the write-out.  Only the register -> staging copy is selected
      // per pass (compile-time register indices under `pass == k`).
#pragma unroll 1
      for (int pass = 0; pass < CW / PW; ++pass) {
        const int c0 = pass * PW;
        if (tc_dbg(p) & 8) break;
        __syncwarp();
#pragma unroll
        for (int k = 0; k < CW / PW; ++k) {
          if (pass == k) {
#pragma unroll
            for (int j = 0; j < PW; j += 4)
              *reinterpret_cast<float4*>(stg + lane * kStgLd + j) =
                  make_float4(acc[k * PW + j], acc[k * PW + j + 1], acc[k * PW + j + 2], acc[k * PW + j + 3]);
          }
        }
        __syncwarp();
        const int64_t n = n0 + c0 + c4;
        if (n < p.N) {
          const bool whole = n + 4 <= p.N;
          float b4[4] = {0.f, 0.f, 0.f, 0.f};
          if (p.bias) {
#pragma unroll
            for (int e = 0; e < 4; ++e) if (n + e < p.N) b4[e] = __ldg(p.bias + n + e);
          }
#pragma unroll 1
          for (int it = 0; it < LR; ++it) {
            const int r = it * (32 / LR) + sub;
            const int64_t grow = mb * BM + q * 32 + r;
            if (grow >= p.M) continue;
            const float4 t4 = *reinterpret_cast<const float4*>(stg + r * kStgLd + c4);
            float v[4] = {t4.x + b4[0], t4.y + b4[1], t4.z + b4[2], t4.w + b4[3]};
            float* dst = C + grow * p.ldc + n;
            if (p.accumulate) {
              if (whole && vec_c) {
                const float4 o = *reinterpret_cast<const float4*>(dst);
                v[0] += o.x; v[1] += o.y; v[2] += o.z; v[3] += o.w;
              } else {
#pragma unroll
                for (int e = 0; e < 4; ++e) if (n + e < p.N) v[e] += dst[e];
              }
            }
            if (p.gtab) {
              const int64_t id = p.gid_bytes == 8 ? static_cast<const int64_t*>(p.gids)[grow]
                                                  : static_cast<int64_t>(static_cast<const int32_t*>(p.gids)[grow]);
              const float* tp = p.gtab + id * p.ld_gtab + n;
              if (whole && (p.ld_gtab % 4 == 0) && aligned16(p.gtab) && (n % 4 == 0)) {
                const float4 o = ldg4(tp);
                v[0] += o.x; v[1] += o.y; v[2] += o.z; v[3] += o.w;
              } else {
#pragma unroll
                for (int e = 0; e < 4; ++e) if (n + e < p.N) v[e] += __ldg(tp + e);
              }
            }
            if (p.act_pre) {
              const float* pp = p.act_pre + grow * p.ld_pre + n;
              float u[4] = {0.f, 0.f, 0.f, 0.f};
              if (whole && vec_p) {
                const float4 o = ldg4(pp);
                u[0] = o.x; u[1] = o.y; u[2] = o.z; u[3] = o.w;
              } else {
#pragma unroll
                for (int e = 0; e < 4; ++e) if (n + e < p.N) u[e] = __ldg(pp + e);
              }
#pragma unroll
              for (int e = 0; e < 4; ++e) v[e] *= act_grad(u[e], p.act);
            }
            if (whole && vec_c) {
              st4(dst, make_float4(v[0], v[1], v[2], v[3]));
            } else {
#pragma unroll
              for (int e = 0; e < 4; ++e) if (n + e < p.N) dst[e] = v[e];
            }
            if (p.C_act) {
              float* da = p.C_act + grow * p.ldca + n;
              if (whole && vec_a) {
                st4(da, make_float4(act_apply(v[0], p.act), act_apply(v[1], p.act), act_apply(v[2], p.act), act_apply(v[3], p.act)));
              } else {
#pragma unroll
                for (int e = 0; e < 4; ++e) if (n + e < p.N) da[e] = act_apply(v[e], p.act);
              }
            }
          }
        }
      }
    }
  }

  tc_fence_before();
  __syncthreads();
  if (warp == kMmaWarp) {
    tc_fence_after();
    asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem_base), "r"(kTmemCols) : "memory");
  }
}

// ================================================================================================
// Forward / dgrad kernel, third generation: the activation operand travels through TENSOR MEMORY.
//
// gemm_tf32x3_kernel keeps hi and lo of BOTH operands in shared memory, so every K=8 MMA reads 8 KB of it and the
// producers write 32 KB per slab on top of the 16 KB cp.async landing: shared-memory bandwidth, not the tensor
// pipe, sets the pace (profiles/r1c_gemm_knockouts.txt).  Here
//   * a producer thread owns one ROW of the 128-row tile: it reads its 32 raw fp32 of the slab from the (swizzled)
//     cp.async landing zone, splits them in registers and stores hi | lo with tcgen05.st straight into 64 TMEM
//     columns of its lane -- the A operand of `tcgen05.mma ... [d], [a_tmem], b_desc` (TS form).  Shared memory no
//     longer holds a split copy of A, and the tensor core reads only B from it (4 KB per MMA instead of 8);
//   * the freed 32 KB per stage buy a fourth pipeline stage (4 x 32 KB of packed weights + 4 x 16 KB raw A);
//   * B_RES: when the whole packed weight panel of an n-tile (hi + lo, all k-stages) fits in 128 KB (K <= 128 at
//     BN = 128) it is loaded ONCE per CTA -- the grid is a multiple of the n-tile count, so a persistent CTA keeps
//     its n-tile -- and the per-tile re-streaming of the weights through L2 (2/3 of the kernel's L2->SM traffic)
//     disappears.
// TMEM: [0, 2*BN) two chunk accumulators, [256, 512) four A slots of 64 columns (hi 32 | lo 32).
// ================================================================================================
constexpr int kTsAcc = 2;
// register budget of the TS kernel (512 threads, 64K registers): 128 x 120 + 256 x 176 + 128 x 40 = 65536
constexpr int kTsRegsProducer = 120, kTsRegsEpilogue = 176, kTsRegsControl = 40;
constexpr int kTsRaw = 4;          // raw-A landing ring (16 KB slots), filled kTsRaw-1 slabs ahead
constexpr int kTsASlots = 4;       // TMEM A slots
constexpr uint32_t kTsACol0 = 256;

__device__ __forceinline__ void tc_st32(uint32_t taddr, const uint32_t (&r)[32]) {
  asm volatile(
      "tcgen05.st.sync.aligned.32x32b.x32.b32 [%0], "
      "{%1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, %16, "
      "%17, %18, %19, %20, %21, %22, %23, %24, %25, %26, %27, %28, %29, %30, %31, %32};"
      ::"r"(taddr), "r"(r[0]), "r"(r[1]), "r"(r[2]), "r"(r[3]), "r"(r[4]), "r"(r[5]), "r"(r[6]), "r"(r[7]),
        "r"(r[8]), "r"(r[9]), "r"(r[10]), "r"(r[11]), "r"(r[12]), "r"(r[13]), "r"(r[14]), "r"(r[15]),
        "r"(r[16]), "r"(r[17]), "r"(r[18]), "r"(r[19]), "r"(r[20]), "r"(r[21]), "r"(r[22]), "r"(r[23]),
        "r"(r[24]), "r"(r[25]), "r"(r[26]), "r"(r[27]), "r"(r[28]), "r"(r[29]), "r"(r[30]), "r"(r[31])
      : "memory");
}
__device__ __forceinline__ void tc_wait_st() { asm volatile("tcgen05.wait::st.sync.aligned;" ::: "memory"); }
__device__ __forceinline__ void tc_mma_tf32_ts(uint32_t tmem_d, uint32_t tmem_a, uint64_t bdesc, uint32_t idesc, uint32_t accum) {
  asm volatile(
      "{\n\t.reg .pred p;\n\t"
      "setp.ne.b32 p, %4, 0;\n\t"
      "tcgen05.mma.cta_group::1.kind::tf32 [%0], [%1], %2, %3, {%5, %5, %5, %5}, p;\n\t}"
      ::"r"(tmem_d), "r"(tmem_a), "l"(bdesc), "r"(idesc), "r"(accum), "r"(0u) : "memory");
}

// Specialised write-out of one staged pass (32 rows x PW columns of a warp) for the common epilogues: the general body
// below carries every option behind run-time flags (bias, accumulate, table gather, activation and its derivative, scalar
// tails) and is ~1.4k SASS instructions of which ~40 execute; ncu's source view put 44 % of an epilogue warp's life in
// that loop at ~7 cycles per instruction (branches, address arithmetic, one exposed shared-memory load per row group).
// MODE 0: C = acc + bias.  1: + table[gid[row]].  2: + C_act = act(C).  3: C += acc + bias.  All need whole, 16-byte
// aligned float4 columns; the four row groups of the pass are unrolled so their loads overlap.
template <int MODE, int PW, bool PRELOADED = false>
__device__ __forceinline__ void ts_write_rows(const float* __restrict__ stg_lane /* stg + sub * ld + c4 */, float* __restrict__ dst,
                                              int64_t row_step /* floats between row groups */, int rows_left /* - sub */,
                                              const float4 b, float* __restrict__ dst_act, int64_t act_step, int act,
                                              const float* const (&trow)[PW / 4], const float4* pre = nullptr) {
  constexpr int LR = PW / 4;
  constexpr int kStgLd = PW + 4;
  // MODE 1: the table chunks of all row groups are requested up front, so their (L2) latencies overlap each other and
  // the shared-memory reads instead of being exposed once per row group inside the loop (the gather epilogue cost the
  // first-layer projection 2x the plain one).  Kept inside this instantiation: hoisting the loads above the register ->
  // staging copy of the caller made every OTHER epilogue mode 20 % slower (16 more live registers in the pass loop), and a
  // register-free prefetch.global.L1 there cost the plain mode 10 % as well (the pass loop is instruction-fetch bound).
  // (PRELOADED: the WM = 1 kernel requested them even earlier, before the register -> staging copy)
  float4 tabv[LR];
  if (MODE == 1) {
#pragma unroll
    for (int it = 0; it < LR; ++it)
      tabv[it] = PRELOADED ? pre[it] : (it * (32 / LR) < rows_left ? ldg4(trow[it]) : make_float4(0.f, 0.f, 0.f, 0.f));
  }
  float4 t[LR];
#pragma unroll
  for (int it = 0; it < LR; ++it) t[it] = *reinterpret_cast<const float4*>(stg_lane + it * (32 / LR) * kStgLd);
#pragma unroll
  for (int it = 0; it < LR; ++it) {
    if (it * (32 / LR) >= rows_left) break;
    float4 v = make_float4(t[it].x + b.x, t[it].y + b.y, t[it].z + b.z, t[it].w + b.w);
    float* d = dst + it * row_step;
    if (MODE == 3) {
      const float4 o = *reinterpret_cast<const float4*>(d);
      v.x += o.x; v.y += o.y; v.z += o.z; v.w += o.w;
    }
    if (MODE == 1) {
      const float4 o = tabv[it];
      v.x += o.x; v.y += o.y; v.z += o.z; v.w += o.w;
    }
    st4(d, v);
    if (MODE == 2)
      st4(dst_act + it * act_step, make_float4(act_apply(v.x, act), act_apply(v.y, act), act_apply(v.z, act), act_apply(v.w, act)));
  }
}

// WM: write-out class compiled into this instantiation -- 0 plain, 1 + table gather, 2 + activated copy (the host
// checked their alignment preconditions), 4 every option behind run-time flags.  The epilogue warps run one or two to a
// scheduler and their pass loop is bound by instruction fetch and live registers, so the ~1.4k-instruction general body
// is only compiled into the WM = 4 kernels.
template <int BN, int S, bool B_RES, bool PP, int WM>
__global__ void __launch_bounds__(kThreads, 1) gemm_tf32x3_ts_kernel(const TcParams p) {
  extern __shared__ uint8_t smem_raw[];
  constexpr uint32_t kBTile = BN * 128;            // bytes of one hi (or lo) B tile of a k-stage
  constexpr uint32_t kBStage = 2 * kBTile;
  constexpr uint32_t kRawTile = BM * 128;          // 16 KB: raw fp32 A slab
  // PP: two epilogue groups alternate tiles (a thread owns one row x all BN columns); else all eight warps share a
  // tile (one row x BN/2 columns per thread)
  constexpr int CW = PP ? BN : BN / 2;
  constexpr int PW = kPW;
  constexpr int kStgLd = PW + 4;
  static_assert(kTsAcc * BN <= static_cast<int>(kTsACol0), "accumulators overlap the A slots");

  uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~static_cast<uintptr_t>(1023));
  uint8_t* smem_b = smem;                                              // S stages (ring) or S resident k-stages
  uint8_t* smem_rawa = smem + static_cast<size_t>(S) * kBStage;        // kTsRaw landing slots
  uint8_t* smem_stg = smem_rawa + static_cast<size_t>(kTsRaw) * kRawTile;
  __shared__ uint64_t bar_full[kTsASlots], bar_empty[kTsASlots], bar_tfull[kTsAcc], bar_tempty[kTsAcc], bar_bres, bar_turn[2];
  __shared__ uint32_t tmem_base_holder;

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  // the A slots and (streamed) B stages advance together: ring depth = kTsASlots; B_RES keeps S k-stages resident
  constexpr int R = kTsASlots;
  static_assert(B_RES || S == R, "streamed weights share the ring of the A slots");

  if (threadIdx.x == 0) {
    for (int s = 0; s < R; ++s) {
      mbar_init(smem_u32(&bar_full[s]), kProducerThreads + (B_RES ? 0 : 1));
      mbar_init(smem_u32(&bar_empty[s]), 1);
    }
    for (int a = 0; a < kTsAcc; ++a) {
      mbar_init(smem_u32(&bar_tfull[a]), 1);
      mbar_init(smem_u32(&bar_tempty[a]), (PP ? kEpiWarps / 2 : kEpiWarps) * 32);   // the epilogue warps that own the tile
    }
    mbar_init(smem_u32(&bar_bres), 1);
    mbar_init(smem_u32(&bar_turn[0]), (kEpiWarps / 2) * 32);
    mbar_init(smem_u32(&bar_turn[1]), (kEpiWarps / 2) * 32);
    fence_barrier_init();
  }
  if (warp == kMmaWarp) {
    asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(&tmem_base_holder)), "r"(512u) : "memory");
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
  }
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = tmem_base_holder;

  const int64_t num_m = (p.M + BM - 1) / BM, num_n = (p.N + BN - 1) / BN;
  const int64_t tiles = num_m * num_n;
  const int64_t num_ks = (p.K + BK - 1) / BK;

  if (warp < kProducerWarps) {
    // ===================================== producers =====================================
    asm volatile("setmaxnreg.dec.sync.aligned.u32 %0;" ::"n"(kTsRegsProducer));
    const int t = threadIdx.x;                        // = row of the tile this thread owns in the split
    // flattened slab sequence of this CTA: (tile, ks).  Everything that depends on the tile only -- the 64-bit tile ->
    // row-block division, this thread's first source row, which of its 8 rows exist -- is computed when the cursor
    // enters a tile, so a slab costs 8 LDGSTS with immediate shared-memory offsets (ncu: the generic stage_raw was 256
    // of the producers' ~720 instructions per slab, the division another ~100, and the producers were 70 % busy).
    struct Cur { int64_t tile, ks; bool live; const float* rowbase; uint32_t rows_ok; };
    const int chunk = t & 7, r0 = t >> 3;                       // 16-byte chunk / first row this thread copies
    const uint32_t soff0 = chunk_offset<BM, false>(r0, chunk);  // row r0 + 16 i lands 2048 i bytes further on
    auto enter = [&](Cur& c) {
      c.live = c.tile < tiles;
      if (!c.live) return;
      const int64_t mb = static_cast<int64_t>(static_cast<uint32_t>(c.tile) / static_cast<uint32_t>(num_n));   // tiles < 2^31
      const int64_t row = mb * BM + r0;
      c.rowbase = p.A + row * p.lda + chunk * 4;
      uint32_t m = 0;
#pragma unroll
      for (int i = 0; i < 8; ++i) m |= (row + 16 * i < p.M) ? (1u << i) : 0u;
      c.rows_ok = m;
    };
    auto init = [&](Cur& c) { c.tile = blockIdx.x; c.ks = 0; enter(c); };
    auto adv = [&](Cur& c) {
      if (++c.ks == num_ks) { c.ks = 0; c.tile += gridDim.x; enter(c); }
    };
    auto issue_raw = [&](const Cur& c, int rslot) {
      const int64_t k = c.ks * BK + chunk * 4;
      const bool kok = k < p.K;                                   // K % 4 == 0 guaranteed by the dispatcher
      const float* g = c.rowbase + c.ks * BK;
      const uint32_t dst = smem_u32(smem_rawa + static_cast<size_t>(rslot) * kRawTile) + soff0;
#pragma unroll
      for (int i = 0; i < 8; ++i) {
        const bool ok = kok && ((c.rows_ok >> i) & 1u);
        cp_async16_zfill(dst + 2048u * i, ok ? static_cast<const void*>(g + static_cast<int64_t>(16 * i) * p.lda) : static_cast<const void*>(p.A),
                         ok ? 16u : 0u);
      }
    };
    Cur pi, ci;
    init(pi); init(ci);
    int prslot = 0, crslot = 0, aslot = 0;
    uint32_t aphase = 0;
#pragma unroll
    for (int i = 0; i < kTsRaw - 1; ++i) {
      if (pi.live) { issue_raw(pi, prslot); adv(pi); }
      cp_async_commit();
      prslot = (prslot + 1 == kTsRaw) ? 0 : prslot + 1;
    }
    const uint32_t lane_field = static_cast<uint32_t>((warp & 3) * 32) << 16;
    while (ci.live) {
      cp_async_wait<kTsRaw - 2>();                    // this thread's chunks of the slab have landed ...
      asm volatile("bar.sync 1, %0;" ::"n"(kProducerThreads) : "memory");   // ... and everybody else's; all are also done
                                                                          // reading the slot refilled below
      if (pi.live) { issue_raw(pi, prslot); adv(pi); }
      cp_async_commit();
      prslot = (prslot + 1 == kTsRaw) ? 0 : prslot + 1;
      // this thread's row of the slab: 8 x 16 B at the swizzled chunk positions
      const uint8_t* rt = smem_rawa + static_cast<size_t>(crslot) * kRawTile;
      uint32_t hi[32], lo[32];
      if (tc_dbg(p) & 2) {
#pragma unroll
        for (int e = 0; e < 32; ++e) { hi[e] = 0u; lo[e] = 0u; }
      } else
#pragma unroll
      for (int c = 0; c < 8; ++c) {
        const float4 v = *reinterpret_cast<const float4*>(rt + chunk_offset<BM, false>(t, c));
        const float x[4] = {v.x, v.y, v.z, v.w};
#pragma unroll
        for (int e = 0; e < 4; ++e) {
          const float h = rn_tf32(x[e]);
          hi[c * 4 + e] = __float_as_uint(h);
          lo[c * 4 + e] = __float_as_uint(rn_tf32_operand(x[e] - h));
        }
      }
      crslot = (crslot + 1 == kTsRaw) ? 0 : crslot + 1;
      mbar_wait(smem_u32(&bar_empty[aslot]), aphase ^ 1u);             // the MMAs that read this A slot have retired
      tc_fence_after();
      const uint32_t a_addr = tmem_base + lane_field + kTsACol0 + static_cast<uint32_t>(aslot) * 64u;
      if (!(tc_dbg(p) & 16)) {
        tc_st32(a_addr, hi);
        tc_st32(a_addr + 32u, lo);
        tc_wait_st();
      }
      tc_fence_before();
      mbar_arrive(smem_u32(&bar_full[aslot]));
      if (++aslot == R) { aslot = 0; aphase ^= 1u; }
      adv(ci);
    }
    cp_async_wait<0>();
  } else if (warp >= kMmaWarp) {
    asm volatile("setmaxnreg.dec.sync.aligned.u32 %0;" ::"n"(kTsRegsControl));
    if (warp == kBLoadWarp && lane == 0) {
      // ===================================== packed-weight loader =====================================
      if constexpr (B_RES) {
        const int64_t nb = blockIdx.x % num_n;        // grid is a multiple of num_n: every tile of this CTA has this nb
        if (blockIdx.x < tiles) {
          mbar_arrive_expect_tx(smem_u32(&bar_bres), static_cast<uint32_t>(num_ks) * kBStage);
          for (int64_t ks = 0; ks < num_ks; ++ks)
            bulk_g2s(smem_u32(smem_b + static_cast<size_t>(ks) * kBStage), p.Bp + static_cast<size_t>(nb * num_ks + ks) * (2 * BN * 32),
                     kBStage, smem_u32(&bar_bres));
        }
      } else {
        int stage = 0;
        uint32_t phase = 0;
        for (int64_t tile = blockIdx.x; tile < tiles; tile += gridDim.x) {
          const int64_t nb = tile % num_n;
          for (int64_t ks = 0; ks < num_ks; ++ks) {
            mbar_wait(smem_u32(&bar_empty[stage]), phase ^ 1u);
            mbar_arrive_expect_tx(smem_u32(&bar_full[stage]), kBStage);
            bulk_g2s(smem_u32(smem_b + static_cast<size_t>(stage) * kBStage), p.Bp + static_cast<size_t>(nb * num_ks + ks) * (2 * BN * 32),
                     kBStage, smem_u32(&bar_full[stage]));
            if (++stage == R) { stage = 0; phase ^= 1u; }
          }
        }
      }
    }
    // ===================================== MMA issuer =====================================
    if (warp == kMmaWarp && lane == 0) {
      constexpr uint32_t idesc = make_idesc(BN, false, false);
      int stage = 0;
      uint32_t phase = 0;
      uint32_t cc = 0;
      if constexpr (B_RES) {
        if (blockIdx.x < tiles) mbar_wait(smem_u32(&bar_bres), 0);
      }
      const int cks = p.ks > 1 ? p.ks : 1;          // k-stages per TMEM chunk
      for (int64_t tile = blockIdx.x; tile < tiles; tile += gridDim.x) {
        int in_chunk = 0;                             // (no division on this thread: it paces the tensor core)
        for (int64_t ks = 0; ks < num_ks; ++ks) {
          mbar_wait(smem_u32(&bar_full[stage]), phase);
          tc_fence_after();
          const uint32_t b_hi = smem_u32(smem_b + static_cast<size_t>(B_RES ? ks : stage) * kBStage), b_lo = b_hi + kBTile;
          const uint32_t a_hi = tmem_base + kTsACol0 + static_cast<uint32_t>(stage) * 64u, a_lo = a_hi + 32u;
          const uint32_t buf = cc % kTsAcc;
          const bool first = in_chunk == 0;
          const bool last = ++in_chunk == cks || ks + 1 == num_ks;
          if (last) in_chunk = 0;
          if (first) {
            mbar_wait(smem_u32(&bar_tempty[buf]), ((cc / kTsAcc) & 1u) ^ 1u);
            tc_fence_after();
          }
          const uint32_t d_tmem = tmem_base + buf * BN;
          uint32_t accum = first ? 0u : 1u;
          // small terms first: lo*hi, hi*lo, then hi*hi (terms >= 4 adds lo*lo in front)
          for (int term = ((tc_dbg(p) & 4) ? 3 : (p.terms >= 4 ? 0 : 1)); term < 4; ++term) {
            const uint32_t ab = (term == 3 || term == 2) ? a_hi : a_lo;
            const uint32_t bb = (term == 3 || term == 1) ? b_hi : b_lo;
            for (int j = 0; j < BK / 8; ++j) {
              tc_mma_tf32_ts(d_tmem, ab + static_cast<uint32_t>(j) * 8u, make_sdesc(bb + j * 32u, 16u, 1024u, 2u), idesc, accum);
              accum = 1u;
            }
          }
          if (last) {
            tc_commit(smem_u32(&bar_tfull[buf]));
            ++cc;
          }
          tc_commit(smem_u32(&bar_empty[stage]));
          if (++stage == R) { stage = 0; phase ^= 1u; }
        }
      }
    }
  } else {
    // ===================================== epilogue =====================================
    // Two groups of four warps alternate TILES: while one group transposes and writes its finished tile out, the other
    // one drains the chunk accumulators of the next tile, so the tensor core never waits for a write-out (with both
    // halves of one tile on all eight warps the write-out cost 40 % of the K = 128 GEMMs: knock-out 8).
    asm volatile("setmaxnreg.inc.sync.aligned.u32 %0;" ::"n"(kTsRegsEpilogue));
    const int q = warp & 3;
    const int grp = (warp - kEpiWarp0) >> 2;          // PP: tile parity this group serves; else: column half
    float* stg = reinterpret_cast<float*>(smem_stg) + (warp - kEpiWarp0) * (32 * kStgLd);
    const uint32_t lane_base = tmem_base + (static_cast<uint32_t>(q * 32) << 16) + (PP ? 0u : static_cast<uint32_t>(grp * CW));
    for (int64_t ti = PP ? grp : 0; blockIdx.x + ti * gridDim.x < tiles; ti += PP ? 2 : 1) {
      const int64_t tile = blockIdx.x + ti * gridDim.x;
      const int64_t nb = tile % num_n, mb = tile / num_n;
      const int64_t n0 = nb * BN + (PP ? 0 : grp * CW);
      const int64_t nchunk = p.ks > 1 ? (num_ks + p.ks - 1) / p.ks : num_ks;
      uint32_t cc = static_cast<uint32_t>(ti * nchunk);
      // The chunk barriers carry one parity bit: a group may only start waiting for its tile's chunks once the other
      // group has drained the previous tile, otherwise the wait would match a completion two phases early.  The
      // hand-over is a barrier per group ("your turn"), completed by the 128 threads of the other group.
      if (PP && ti > 0) mbar_wait(smem_u32(&bar_turn[grp]), static_cast<uint32_t>(((ti >> 1) - (grp == 0 ? 1 : 0)) & 1));
      float acc[CW];
#pragma unroll
      for (int i = 0; i < CW; ++i) acc[i] = 0.f;
      for (int64_t c = 0; c < nchunk; ++c, ++cc) {
        const uint32_t buf = cc % kTsAcc;
        mbar_wait(smem_u32(&bar_tfull[buf]), (cc / kTsAcc) & 1u);
        tc_fence_after();
#pragma unroll
        for (int c0 = 0; c0 < CW; c0 += 32) {
          if (tc_dbg(p) & 1) break;
          uint32_t r0[32];
          tc_ld32(lane_base + buf * BN + c0, r0);
          tc_wait_ld();
#pragma unroll
          for (int j = 0; j < 32; ++j) acc[c0 + j] += __uint_as_float(r0[j]);
        }
        tc_fence_before();
        mbar_arrive(smem_u32(&bar_tempty[buf]));
      }
      if (PP) mbar_arrive(smem_u32(&bar_turn[grp ^ 1]));      // the other group may now wait for the next tile's chunks
      float* C = p.C;
      constexpr int LR = PW / 4;
      const int sub = lane / LR, c4 = (lane % LR) * 4;
      const bool vec_c = (p.ldc % 4 == 0) && aligned16(C) && (n0 % 4 == 0);
      const bool vec_a = p.C_act && (p.ldca % 4 == 0) && aligned16(p.C_act) && (n0 % 4 == 0);
      const bool vec_p = p.act_pre && (p.ld_pre % 4 == 0) && aligned16(p.act_pre) && (n0 % 4 == 0);
      const bool vec_g = p.gtab && (p.ld_gtab % 4 == 0) && aligned16(p.gtab) && (n0 % 4 == 0);
      // epilogue class of this launch (uniform): 0 plain, 1 + table gather, 2 + activated copy, 3 accumulate, 4 general
      const int wmode = WM < 4 ? WM
                        : (!vec_c || p.act_pre) ? 4
                        : p.gtab ? ((vec_g && !p.accumulate && !p.C_act) ? 1 : 4)
                        : p.C_act ? ((vec_a && !p.accumulate) ? 2 : 4)
                        : p.accumulate ? 3 : 0;
      // per-tile addressing of the specialised paths: this lane's first destination row (row group 0) and column chunk
      const int64_t fast_row = mb * BM + q * 32 + sub;
      const int fast_rows = static_cast<int>(min(static_cast<int64_t>(32), p.M - (mb * BM + q * 32))) - sub;   // row group `it` exists iff it * 8 < fast_rows
      float* fast_dst = C + fast_row * p.ldc + n0 + c4;
      const int64_t fast_step = static_cast<int64_t>(32 / LR) * p.ldc;
      float* fast_dst_act = p.C_act ? p.C_act + fast_row * p.ldca + n0 + c4 : nullptr;
      const int64_t fast_act_step = static_cast<int64_t>(32 / LR) * p.ldca;
      const float* fast_trow[LR];
#pragma unroll
      for (int it = 0; it < LR; ++it) {
        fast_trow[it] = nullptr;
        if (wmode == 1 && it * (32 / LR) < fast_rows) {
          const int64_t grow = fast_row + it * (32 / LR);
          const int64_t id = p.gid_bytes == 8 ? static_cast<const int64_t*>(p.gids)[grow]
                                              : static_cast<int64_t>(static_cast<const int32_t*>(p.gids)[grow]);
          fast_trow[it] = p.gtab + id * p.ld_gtab + n0 + c4;
        }
      }
      // One ROLLED loop over the write-out passes: the body below (bias / accumulate / table gather / activation, each
      // behind a run-time flag) is emitted once instead of CW/PW times -- unrolled it was over half of the kernel's SASS
      // and the instruction cache, not the LSU, bounded the write-out.  Only the register -> staging copy is selected
      // per pass (compile-time register indices under `pass == k`).
#pragma unroll 1
      for (int pass = 0; pass < CW / PW; ++pass) {
        const int c0 = pass * PW;
        if (tc_dbg(p) & 8) break;
        // WM = 1 (this instantiation only gathers): the pass's table chunks are requested before the register -> staging
        // copy so their L2 latency overlaps it.  Columns at or past N are not read: in the tail n-tile they would lie
        // past the end of a table row (past the table itself for its last row when ld_gtab == N).
        float4 pre[WM == 1 ? LR : 1];
        if constexpr (WM == 1) {
          const bool col_in = n0 + c0 + c4 < p.N;
#pragma unroll
          for (int it = 0; it < LR; ++it)
            pre[it] = (col_in && fast_trow[it] != nullptr) ? ldg4(fast_trow[it] + c0) : make_float4(0.f, 0.f, 0.f, 0.f);
        }
        __syncwarp();
#pragma unroll
        for (int k = 0; k < CW / PW; ++k) {
          if (pass == k) {
#pragma unroll
            for (int j = 0; j < PW; j += 4)
              *reinterpret_cast<float4*>(stg + lane * kStgLd + j) =
                  make_float4(acc[k * PW + j], acc[k * PW + j + 1], acc[k * PW + j + 2], acc[k * PW + j + 3]);
          }
        }
        __syncwarp();
        const int64_t n = n0 + c0 + c4;
        if (n < p.N) {
          const bool whole = WM < 4 || n + 4 <= p.N;      // (WM < 4: N % 4 == 0, checked by the host)
          float b4[4] = {0.f, 0.f, 0.f, 0.f};
          if (p.bias) {
#pragma unroll
            for (int e = 0; e < 4; ++e) if (WM < 4 || n + e < p.N) b4[e] = __ldg(p.bias + n + e);
          }
          if (whole && wmode != 4) {
            const float4 bv = make_float4(b4[0], b4[1], b4[2], b4[3]);
            const float* sl = stg + sub * kStgLd + c4;
            float* d = fast_dst + c0;
            if (wmode == 0) ts_write_rows<0, PW>(sl, d, fast_step, fast_rows, bv, nullptr, 0, 0, fast_trow);
            else if (wmode == 1) {
              if constexpr (WM == 1) {
                ts_write_rows<1, PW, true>(sl, d, fast_step, fast_rows, bv, nullptr, 0, 0, fast_trow, pre);
              } else {
                const float* tr[LR];
#pragma unroll
                for (int it = 0; it < LR; ++it) tr[it] = fast_trow[it] + c0;
                ts_write_rows<1, PW>(sl, d, fast_step, fast_rows, bv, nullptr, 0, 0, tr);
              }
            } else if (wmode == 2) ts_write_rows<2, PW>(sl, d, fast_step, fast_rows, bv, fast_dst_act + c0, fast_act_step, p.act, fast_trow);
            else ts_write_rows<3, PW>(sl, d, fast_step, fast_rows, bv, nullptr, 0, 0, fast_trow);
            continue;
          }
          if constexpr (WM == 4) {
#pragma unroll 1
          for (int it = 0; it < LR; ++it) {
            const int r = it * (32 / LR) + sub;
            const int64_t grow = mb * BM + q * 32 + r;
            if (grow >= p.M) continue;
            const float4 t4 = *reinterpret_cast<const float4*>(stg + r * kStgLd + c4);
            float v[4] = {t4.x + b4[0], t4.y + b4[1], t4.z + b4[2], t4.w + b4[3]};
            float* dst = C + grow * p.ldc + n;
            if (p.accumulate) {
              if (whole && vec_c) {
                const float4 o = *reinterpret_cast<const float4*>(dst);
                v[0] += o.x; v[1] += o.y; v[2] += o.z; v[3] += o.w;
              } else {
#pragma unroll
                for (int e = 0; e < 4; ++e) if (n + e < p.N) v[e] += dst[e];
              }
            }
            if (p.gtab) {
              const int64_t id = p.gid_bytes == 8 ? static_cast<const int64_t*>(p.gids)[grow]
                                                  : static_cast<int64_t>(static_cast<const int32_t*>(p.gids)[grow]);
              const float* tp = p.gtab + id * p.ld_gtab + n;
              if (whole && vec_g) {
                const float4 o = ldg4(tp);
                v[0] += o.x; v[1] += o.y; v[2] += o.z; v[3] += o.w;
              } else {
#pragma unroll
                for (int e = 0; e < 4; ++e) if (n + e < p.N) v[e] += __ldg(tp + e);
              }
            }
            if (p.act_pre) {
              const float* pp = p.act_pre + grow * p.ld_pre + n;
              float u[4] = {0.f, 0.f, 0.f, 0.f};
              if (whole && vec_p) {
                const float4 o = ldg4(pp);
                u[0] = o.x; u[1] = o.y; u[2] = o.z; u[3] = o.w;
              } else {
#pragma unroll
                for (int e = 0; e < 4; ++e) if (n + e < p.N) u[e] = __ldg(pp + e);
              }
#pragma unroll
              for (int e = 0; e < 4; ++e) v[e] *= act_grad(u[e], p.act);
            }
            if (whole && vec_c) {
              st4(dst, make_float4(v[0], v[1], v[2], v[3]));
            } else {
#pragma unroll
              for (int e = 0; e < 4; ++e) if (n + e < p.N) dst[e] = v[e];
            }
            if (p.C_act) {
              float* da = p.C_act + grow * p.ldca + n;
              if (whole && vec_a) {
                st4(da, make_float4(act_apply(v[0], p.act), act_apply(v[1], p.act), act_apply(v[2], p.act), act_apply(v[3], p.act)));
              } else {
#pragma unroll
                for (int e = 0; e < 4; ++e) if (n + e < p.N) da[e] = act_apply(v[e], p.act);
              }
            }
          }
          }   // WM == 4
        }
      }
    }
  }

  tc_fence_before();
  __syncthreads();
  if (warp == kMmaWarp) {
    tc_fence_after();
    asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem_base), "r"(512u) : "memory");
  }
}

__global__ void tc_splitk_reduce_kernel(const float* __restrict__ part, int splits, int64_t MN, int64_t N,
                                        float* __restrict__ out, int64_t ldo, int accumulate) {
  const int64_t i = static_cast<int64_t>(blockIdx.x) * blockDim.x + threadIdx.x;
  if (i >= MN) return;
  float s = 0.f;
  for (int z = 0; z < splits; ++z) s += part[static_cast<int64_t>(z) * MN + i];
  float* dst = out + (i / N) * ldo + (i % N);
  *dst = accumulate ? *dst + s : s;
}

int env_int(const char* name, int lo, int hi, int dflt) {
  const char* e = getenv(name);
  if (!e) return dflt;
  const int v = atoi(e);
  return (v < lo || v > hi) ? dflt : v;
}

__global__ void tc_colsum_reduce_kernel(const float* __restrict__ part, int splits, int64_t N, float* __restrict__ db, int accumulate) {
  const int64_t n = static_cast<int64_t>(blockIdx.x) * blockDim.x + threadIdx.x;
  if (n >= N) return;
  float s = 0.f;
  for (int z = 0; z < splits; ++z) s += part[static_cast<int64_t>(z) * N + n];
  db[n] = accumulate ? db[n] + s : s;
}

template <int BN>
constexpr size_t stage_bytes() { return static_cast<size_t>(2 * BM * 128 + 2 * BN * 128); }

template <int BN, bool A_MN, bool B_MN, bool B_PACKED, int S>
int launch_tc_s(TcParams p, cudaStream_t stream) {
  constexpr size_t kStgBytes = stg_bytes(kPW);
  static_assert(S <= kMaxStages, "stage count");
  p.stages = S;
  p.dbg = env_int("SEGGER_B200_TC_DBG", 0, 255, 0);
  constexpr size_t kRedBytes = A_MN ? kProducerThreads * (BM / 8) * sizeof(float) : 0;   // fused column sums
  const size_t smem = S * stage_bytes<BN>() + kStgBytes + kRedBytes + 1024;
  static_assert(S * stage_bytes<BN>() + kStgBytes + kRedBytes + 1024 + 256 <= 227 * 1024, "shared memory budget");
  static bool configured = false;   // per instantiation
  if (!configured) {
    cudaError_t e = cudaFuncSetAttribute(gemm_tf32x3_kernel<BN, A_MN, B_MN, B_PACKED, S>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                         static_cast<int>(smem));
    if (e != cudaSuccess) return set_error(SGB_ERR_CUDA, "tc gemm: cudaFuncSetAttribute: %s", cudaGetErrorString(e));
    configured = true;
  }
  const int64_t tiles = ceil_div(p.M, BM) * ceil_div(p.N, BN) * p.splits;
  const int grid = static_cast<int>(tiles < sm_count() ? tiles : sm_count());
  gemm_tf32x3_kernel<BN, A_MN, B_MN, B_PACKED, S><<<grid, kThreads, smem, stream>>>(p);
  return check_launch("gemm_tf32x3");
}

template <int BN, bool A_MN, bool B_MN, bool B_PACKED>
int launch_tc(TcParams p, cudaStream_t stream) {
  // 3 x 64 KB or 4 x 48 KB stage slots: all the shared memory there is.  One slot fewer costs 17-24 % on the
  // BN = 128 kernels and on wgrad, nothing on the packed BN = 64 kernels (profiles/r1d_gemm_stage_depth.txt).
  constexpr int S = (BN == 128) ? 3 : 4;
  return launch_tc_s<BN, A_MN, B_MN, B_PACKED, S>(p, stream);
}

int pick_bn(int64_t N) { return N <= 64 ? 64 : 128; }

// packed-weight GEMM (forward / dgrad): B is split + laid out once by pack_b_kernel into `ws`
size_t packed_b_bytes(int64_t N, int64_t K) {
  const int bn = pick_bn(N);
  return align_up(static_cast<size_t>(ceil_div(N, bn)) * ceil_div(K, BK) * (2 * bn * 128));
}

template <int BN, int S, bool B_RES, bool PP, int WM>
int launch_ts_wm(TcParams p, cudaStream_t stream) {
  p.stages = S;
  p.dbg = env_int("SEGGER_B200_TC_DBG", 0, 255, 0);
  constexpr size_t smem = static_cast<size_t>(S) * (2 * BN * 128) + static_cast<size_t>(kTsRaw) * (BM * 128) + stg_bytes(kPW) + 1024;
  static_assert(smem + 512 <= 227 * 1024, "shared memory budget");
  static bool configured = false;
  if (!configured) {
    cudaError_t e = cudaFuncSetAttribute(gemm_tf32x3_ts_kernel<BN, S, B_RES, PP, WM>, cudaFuncAttributeMaxDynamicSharedMemorySize, static_cast<int>(smem));
    if (e != cudaSuccess) return set_error(SGB_ERR_CUDA, "tc gemm (ts): cudaFuncSetAttribute: %s", cudaGetErrorString(e));
    configured = true;
  }
  const int64_t num_n = ceil_div(p.N, BN);
  const int64_t tiles = ceil_div(p.M, BM) * num_n;
  int64_t grid = tiles < sm_count() ? tiles : sm_count();
  if (B_RES) {                         // a persistent CTA keeps its n-tile: grid multiple of num_n
    grid = grid / num_n * num_n;
    if (grid < num_n) grid = num_n < tiles ? num_n : tiles;
  }
  gemm_tf32x3_ts_kernel<BN, S, B_RES, PP, WM><<<static_cast<unsigned>(grid), kThreads, smem, stream>>>(p);
  return check_launch("gemm_tf32x3_ts");
}

// write-out class of a launch (the kernel's own rule, evaluated once on the host): see gemm_tf32x3_ts_kernel's WM
static int ts_write_mode(const TcParams& p) {
  static int force_general = env_int("SEGGER_B200_GEMM_WM", 0, 1, 1) == 0;     // SEGGER_B200_GEMM_WM=0: general kernels only
  const bool vec_c = p.ldc % 4 == 0 && aligned16(p.C) && p.N % 4 == 0;
  if (force_general || !vec_c || p.act_pre || p.accumulate) return 4;
  if (p.gtab) return (p.ld_gtab % 4 == 0 && aligned16(p.gtab) && !p.C_act) ? 1 : 4;
  if (p.C_act) return (p.ldca % 4 == 0 && aligned16(p.C_act)) ? 2 : 4;
  return 0;
}

template <int BN, int S, bool B_RES, bool PP>
int launch_ts_pp(TcParams p, cudaStream_t stream) {
  switch (ts_write_mode(p)) {
    case 0: return launch_ts_wm<BN, S, B_RES, PP, 0>(p, stream);
    case 1: return launch_ts_wm<BN, S, B_RES, PP, 1>(p, stream);
    case 2: return launch_ts_wm<BN, S, B_RES, PP, 2>(p, stream);
    default: return launch_ts_wm<BN, S, B_RES, PP, 4>(p, stream);
  }
}

// Epilogue mode, chosen from scripts/bench_gemm.py on B200 (profiles/r2_gemm_epilogue_modes.md): alternating tile groups
// hide a tile's write-out behind the next tile's MMAs whenever a tile has at least three k-stages of MMA work to hide
// it behind; on shallower tiles all eight warps share one tile.  SEGGER_B200_GEMM_PP=0|1 forces a mode.
template <int BN, int S, bool B_RES>
int launch_ts(TcParams p, cudaStream_t stream) {
  static int force = env_int("SEGGER_B200_GEMM_PP", 0, 1, -1);
  const int64_t num_ks = ceil_div(p.K, BK);
  const bool pp = force >= 0 ? force == 1 : num_ks >= 3;
  return pp ? launch_ts_pp<BN, S, B_RES, true>(p, stream) : launch_ts_pp<BN, S, B_RES, false>(p, stream);
}

// SEGGER_B200_GEMM_TS=0 keeps the second-generation kernel (A/B of the two designs)
static bool ts_enabled() {
  static int flag = -1;
  if (flag < 0) {
    const char* e = getenv("SEGGER_B200_GEMM_TS");
    flag = (e && e[0] == '0') ? 0 : 1;
  }
  return flag == 1;
}

int run_packed(TcParams p, const float* w, int64_t ldw, int src_mn, void* ws, cudaStream_t stream) {
  const int bn = pick_bn(p.N);
  const int num_n = static_cast<int>(ceil_div(p.N, bn)), num_ks = static_cast<int>(ceil_div(p.K, BK));
  const int64_t chunks = static_cast<int64_t>(num_n) * bn * num_ks * 8;
  float* out = static_cast<float*>(ws);
  if (bn == 64) pack_b_kernel<64><<<static_cast<unsigned>(ceil_div(chunks, 256)), 256, 0, stream>>>(w, ldw, p.N, p.K, src_mn, num_n, num_ks, out);
  else pack_b_kernel<128><<<static_cast<unsigned>(ceil_div(chunks, 256)), 256, 0, stream>>>(w, ldw, p.N, p.K, src_mn, num_n, num_ks, out);
  int rc = check_launch("pack_b");
  if (rc != SGB_OK) return rc;
  p.Bp = out;
  if (ts_enabled() && p.splits == 1) {
    // resident weights when every k-stage of an n-tile's packed panel fits in 128 KB beside the raw-A ring
    if (bn == 128) {
      if (num_ks <= 4 && num_n <= sm_count()) {
        if (num_ks <= 2) return launch_ts<128, 2, true>(p, stream);
        return launch_ts<128, 4, true>(p, stream);
      }
      return launch_ts<128, 4, false>(p, stream);
    }
    if (num_ks <= 8 && num_n <= sm_count()) {
      if (num_ks <= 2) return launch_ts<64, 2, true>(p, stream);
      if (num_ks <= 4) return launch_ts<64, 4, true>(p, stream);
      return launch_ts<64, 8, true>(p, stream);
    }
    return launch_ts<64, 4, false>(p, stream);
  }
  return bn == 64 ? launch_tc<64, false, false, true>(p, stream) : launch_tc<128, false, false, true>(p, stream);
}

bool is_blackwell() {
  static int cached = -1;
  if (cached < 0) {
    int dev = 0, major = 0;
    if (cudaGetDevice(&dev) != cudaSuccess || cudaDeviceGetAttribute(&major, cudaDevAttrComputeCapabilityMajor, dev) != cudaSuccess)
      return false;
    cached = (major == 10) ? 1 : 0;
  }
  return cached == 1;
}

bool ok_ptr(const float* p, int64_t ld) { return aligned16(p) && ld % 4 == 0; }


}  // namespace

bool tc_enabled() {
  static int flag = -1;
  if (flag < 0) {
    const char* e = getenv("SEGGER_B200_GEMM");
    flag = (e && (e[0] == 's' || e[0] == 'S')) ? 0 : 1;    // SEGGER_B200_GEMM=simt forces the fp32 SIMT path
  }
  return flag == 1 && is_blackwell();
}

// Number of TF32 products per fp32 product and K=8 steps accumulated inside the tensor core per chunk.
//   3 terms (hi*hi + lo*hi + hi*lo), kc = 4 for every GEMM.  The dropped lo*lo term is <= 2^-24 |a||b| per product
//   (|lo| <= 2^-12 |x| after the round-to-nearest split), i.e. below the fp32 rounding of the product itself:
//   measured on the encoder parity case (scripts/debug_param_err.py) the worst parameter gradient is 8.2e-7 from
//   the fp64 oracle with 3 terms and 9.7e-7 with 4, outputs 3.5e-7 vs 2.9e-7 -- while the fourth MMA pass costs
//   8-18 % of every forward GEMM (shared-memory operand reads are the binding resource).  What matters for the
//   attention backward is the ROUNDING of the accumulation, which the 32-deep chunks fix (kc = 1, 2, 4 alike
//   within 1e-6; un-chunked TMEM accumulation: 5e-3).
// SEGGER_B200_TF32_TERMS=4 restores the fourth term for `exact` calls; SEGGER_B200_TC_KC / _KC_EXACT override kc.
static int tc_terms(bool exact) {
  static int env = env_int("SEGGER_B200_TF32_TERMS", 3, 4, 3);
  return (exact && env == 4) ? 4 : 3;
}
// k-stages per TMEM chunk (read per call: A/B runs in one process)
static int tc_env_ks(const char* name, int dflt) {
  const char* e = getenv(name);
  const int v = e ? atoi(e) : dflt;
  return v < 1 ? 1 : (v > 16 ? 16 : v);
}
static int tc_kc(bool exact) {
  static int fast = env_int("SEGGER_B200_TC_KC", 1, 4, 4), ex = env_int("SEGGER_B200_TC_KC_EXACT", 1, 4, 4);
  const int v = exact ? ex : fast;
  return v == 3 ? 2 : v;
}

size_t tc_linear_workspace_bytes(int64_t N, int64_t K) { return packed_b_bytes(N, K); }

bool tc_linear_fwd_ok(const float* x, int64_t ldx, const float* w, int64_t ldw, int64_t M, int64_t N, int64_t K) {
  (void)w; (void)ldw;
  return tc_enabled() && M >= 1 && N >= 8 && K >= 8 && K % 4 == 0 && ok_ptr(x, ldx);
}
int tc_linear_fwd(const float* x, int64_t ldx, const float* w, int64_t ldw, const float* b, int64_t M, int64_t N, int64_t K,
                  float* y, int64_t ldy, int act, float* y_act, int64_t ldya, int exact, void* ws, cudaStream_t stream,
                  const void* gids, int gid_bytes, const float* gtab, int64_t ld_gtab) {
  TcParams p{};
  p.gids = gids; p.gid_bytes = gid_bytes; p.gtab = gtab; p.ld_gtab = ld_gtab;
  p.A = x; p.lda = ldx; p.B = w; p.ldb = ldw; p.M = M; p.N = N; p.K = K; p.splits = 1;
  p.k_per_split = ceil_div(K, BK) * BK;
  p.C = y; p.ldc = ldy; p.bias = b; p.act = act; p.C_act = y_act; p.ldca = ldya;
  p.terms = tc_terms(exact != 0);
  p.kc = tc_kc(exact != 0);
  // forward projections keep 32-deep chunks: 64-deep ones are 3-12 % faster (1M x 128 -> 384: 0.92 -> 0.81 ms) but raise
  // the output error from 2.4e-7 to 5.2e-7 of the row scale, which the attention backward amplifies
  // (test_istencoder_forward_backward_vs_oracle[cfg1] fails with SEGGER_B200_TC_FWD_KS=2)
  p.ks = tc_env_ks("SEGGER_B200_TC_FWD_KS", 1);
  return run_packed(p, w, ldw, 0, ws, stream);
}

bool tc_linear_dgrad_ok(const float* dy, int64_t ldy, const float* w, int64_t ldw, int64_t M, int64_t N, int64_t K) {
  // dx[M,K] = dy[M,N] w[N,K]: A = dy (K-major over n), B(k', n) = w[n, k'] (transposed by the pre-pack)
  (void)w; (void)ldw;
  return tc_enabled() && M >= 1 && K >= 8 && N >= 8 && N % 4 == 0 && ok_ptr(dy, ldy);
}
int tc_linear_dgrad(const float* dy, int64_t ldy, const float* w, int64_t ldw, int64_t M, int64_t N, int64_t K, float* dx,
                    int64_t ldx, int accumulate, int act, const float* act_pre, int64_t ld_pre, void* ws, cudaStream_t stream) {
  TcParams p{};
  p.A = dy; p.lda = ldy; p.B = w; p.ldb = ldw; p.M = M; p.N = K; p.K = N; p.splits = 1;
  p.k_per_split = ceil_div(N, BK) * BK;
  p.C = dx; p.ldc = ldx; p.accumulate = accumulate; p.act = act; p.act_pre = act_pre; p.ld_pre = ld_pre;
  p.terms = tc_terms(false);
  p.kc = tc_kc(false);
  p.ks = tc_env_ks("SEGGER_B200_TC_DGRAD_KS", 2);   // feature gradients: 64-deep chunks (-3..5 %, error 2e-7 -> 4.5e-7 of the row scale)
  return run_packed(p, w, ldw, 1, ws, stream);
}

// k-stages per TMEM chunk of the weight-gradient GEMM (SEGGER_B200_TC_WGRAD_KS, read per call for A/B runs).
// Measured on B200 (scripts/bench_gemm.py --only wgrad; error = max |dw - fp64| / max |fp64| over 10^6-row reductions):
//   ks   1M x 384 x 256   1M x 256 x 128   2M x 64 x 64     error
//   1       1.81 ms          0.61 ms          0.57 ms       5.0 .. 7.4e-7
//   2       1.49             0.50             0.43          5.1 .. 6.8e-7
//   4       1.45             0.49             0.42          0.9 .. 1.1e-6
//   8       1.45             0.49             0.42          1.7 .. 2.0e-6
// 64-deep chunks take the read-back hand-over off the critical path at no measurable cost in accuracy; deeper ones buy
// 2 % more and start to show the tensor core's truncating accumulation.
static int tc_wgrad_ks() {
  const char* e = getenv("SEGGER_B200_TC_WGRAD_KS");
  const int v = e ? atoi(e) : 2;
  return v < 1 ? 1 : (v > 16 ? 16 : v);
}
static int tc_wgrad_splits(int64_t M, int64_t N, int64_t K) {
  const int64_t bn = pick_bn(K);
  const int64_t tiles = ceil_div(N, BM) * ceil_div(K, bn);
  int64_t s = sm_count() / tiles;
  const int64_t max_by_rows = ceil_div(M, 8 * BK);     // at least 8 k-stages per split
  if (s > max_by_rows) s = max_by_rows;
  if (s < 1) s = 1;
  return static_cast<int>(s);
}
bool tc_linear_wgrad_ok(const float* dy, int64_t ldy, const float* x, int64_t ldx, int64_t M, int64_t N, int64_t K) {
  // dw[N,K] = dy^T x: A(n, m) = dy[m, n] (MN-major), B(k, m) = x[m, k] (MN-major), reduction over m
  return tc_enabled() && M >= 256 && N >= 8 && K >= 8 && N % 4 == 0 && K % 4 == 0 && ok_ptr(dy, ldy) && ok_ptr(x, ldx);
}
size_t tc_linear_wgrad_workspace_bytes(int64_t M, int64_t N, int64_t K) {
  const size_t sp = static_cast<size_t>(tc_wgrad_splits(M, N, K));
  return align_up(sp * N * K * sizeof(float)) + align_up(sp * N * sizeof(float));
}
// db (optional) = column sums of dy, produced by the same kernel (its producers see every dy element anyway)
int tc_linear_wgrad(const float* dy, int64_t ldy, const float* x, int64_t ldx, int64_t M, int64_t N, int64_t K, float* dw,
                    int64_t lddw, float* db, int accumulate, void* ws, cudaStream_t stream) {
  TcParams p{};
  const int splits0 = tc_wgrad_splits(M, N, K);
  p.A = dy; p.lda = ldy; p.B = x; p.ldb = ldx; p.M = N; p.N = K; p.K = M; p.splits = splits0;
  p.k_per_split = ceil_div(ceil_div(M, splits0), BK) * BK;
  p.terms = tc_terms(false);
  p.kc = tc_kc(false);
  p.ks = tc_wgrad_ks();
  // every split must own at least one k-stage
  while (p.splits > 1 && static_cast<int64_t>(p.splits - 1) * p.k_per_split >= M) --p.splits;
  const bool narrow = pick_bn(K) == 64;
  float* db_part = reinterpret_cast<float*>(static_cast<char*>(ws) + align_up(static_cast<size_t>(splits0) * N * K * sizeof(float)));
  if (p.splits == 1) {
    p.C = dw; p.ldc = lddw; p.accumulate = accumulate;
    p.colsum = db; p.colsum_accumulate = accumulate;
    return narrow ? launch_tc<64, true, true, false>(p, stream) : launch_tc<128, true, true, false>(p, stream);
  }
  p.C = static_cast<float*>(ws); p.ldc = K;
  p.colsum = db ? db_part : nullptr;
  int rc = narrow ? launch_tc<64, true, true, false>(p, stream) : launch_tc<128, true, true, false>(p, stream);
  if (rc != SGB_OK) return rc;
  const int64_t MN = N * K;
  tc_splitk_reduce_kernel<<<static_cast<unsigned>(ceil_div(MN, 256)), 256, 0, stream>>>(static_cast<const float*>(ws), p.splits, MN, K,
                                                                                       dw, lddw, accumulate);
  if (db) tc_colsum_reduce_kernel<<<static_cast<unsigned>(ceil_div(N, 128)), 128, 0, stream>>>(db_part, p.splits, N, db, accumulate);
  return check_launch("tc_splitk_reduce");
}

}  // namespace sgb
