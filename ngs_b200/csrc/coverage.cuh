// K9 — resolve one contig's int32 difference array into what CoverageFacet::teardown
// computes with an O(L) scalar sweep over a Vec<usize> (coverage.rs:182-262):
//   * depth histogram over positions 0..=L, capped at 2048 (deeper -> pileup_too_large),
//   * per-50 kb running sums: bin 0 = {0}, bin k = (50000(k-1), 50000k], partial tail bin.
// The depth array itself is never materialised, and the difference array is read ONCE: the sum of
// every 4096-position tile is maintained by the kernels that scatter into the array (two more reductions
// per record into an L2-resident int32 table), so the resolve needs only the scan of those sums
// (cov_scan_tiles) and one streaming pass (cov_resolve: per tile a local scan fused with the run-length
// aggregated, shared-memory privatised histogram and the bin sums).  HBM-bound: 4 B/position.
//
// cov_resolve_kernel: each 16 KB tile reaches the CTA by one cp.async.bulk (TMA 1-D bulk copy, SASS UBLKCP)
// into a double-buffered shared-memory stage, completion on an mbarrier.  Against per-thread 128-bit loads
// it removes the long-scoreboard stall and is 2.6 % faster on a B200 (profiles/round2_coverage_bulk_ab.md).
#pragma once
#include <cstdint>
#include <cuda_runtime.h>

#include "facets.cuh"

namespace ngsq {

constexpr int kCovThreads = 256;
constexpr int kCovPerThread = 16;
constexpr int kCovTile = kCovThreads * kCovPerThread;  // 4096 positions < bin size
constexpr uint32_t kCovBin = 50000;
constexpr uint32_t kCovTileShift = 12;
static_assert((1u << kCovTileShift) == (uint32_t)kCovTile, "tile size");

// depth -> slot of the CTA-private histogram; [2049] collects depths beyond the reference's 2048 cap.  A negative running depth
// cannot come from the facet kernel's scatter (+1 at a start precedes its -1); should the int32 array ever wrap, stay in bounds.
__device__ __forceinline__ uint32_t cov_hist_slot(int64_t d) { return (d > 2048 || d < 0) ? 2049u : (uint32_t)d; }

// exclusive scan of one contig's int32 tile sums into int64 tile bases (single CTA)
__global__ void __launch_bounds__(1024)
cov_scan_tiles_kernel(const int32_t* __restrict__ tile_sum, int64_t* __restrict__ tile_base, uint32_t n_tiles, const uint64_t* __restrict__ touched) {
  if (!*touched) return;
  __shared__ int64_t warp_sums[32];
  __shared__ int64_t carry_s;
  if (threadIdx.x == 0) carry_s = 0;
  __syncthreads();
  const uint32_t lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
  for (uint32_t start = 0; start < n_tiles; start += blockDim.x) {
    uint32_t i = start + threadIdx.x;
    int64_t v = i < n_tiles ? (int64_t)tile_sum[i] : 0, x = v;
    for (int o = 1; o < 32; o <<= 1) {
      int64_t y = __shfl_up_sync(0xFFFFFFFFu, x, o);
      if ((int)lane >= o) x += y;
    }
    if (lane == 31) warp_sums[wid] = x;
    __syncthreads();
    if (wid == 0) {
      int64_t s = lane < (blockDim.x >> 5) ? warp_sums[lane] : 0;
      for (int o = 1; o < 32; o <<= 1) {
        int64_t y = __shfl_up_sync(0xFFFFFFFFu, s, o);
        if ((int)lane >= o) s += y;
      }
      warp_sums[lane] = s;
    }
    __syncthreads();
    int64_t carry = carry_s;
    int64_t wbase = wid ? warp_sums[wid - 1] : 0;
    if (i < n_tiles) tile_base[i] = carry + wbase + x - v;
    __syncthreads();
    if (threadIdx.x == blockDim.x - 1) carry_s = carry + wbase + x;
    __syncthreads();
  }
}

__device__ __forceinline__ uint32_t smem_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }

__device__ __forceinline__ void mbar_init(uint64_t* bar, uint32_t count) {
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count) : "memory");
}
__device__ __forceinline__ void mbar_expect_tx(uint64_t* bar, uint32_t bytes) {
  asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)), "r"(bytes) : "memory");
}
__device__ __forceinline__ void mbar_wait(uint64_t* bar, uint32_t parity) {
  asm volatile(
      "{\n\t.reg .pred p;\n\t"
      "WAIT_%=:\n\t"
      "mbarrier.try_wait.parity.shared::cta.b64 p, [%0], %1;\n\t"
      "@!p bra WAIT_%=;\n\t}" ::"r"(smem_u32(bar)), "r"(parity) : "memory");
}
// 1-D bulk copy global -> shared (addresses and size multiples of 16 bytes), completion counted in bytes on `bar`
__device__ __forceinline__ void bulk_g2s(void* dst_smem, const void* src_gmem, uint32_t bytes, uint64_t* bar) {
  asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(smem_u32(dst_smem)), "l"(src_gmem),
               "r"(bytes), "r"(smem_u32(bar))
               : "memory");
}

// Persistent CTAs loop over tiles; slot = this contig's [touched, too_large, hist[2049], bins[]].
__global__ void __launch_bounds__(kCovThreads)
cov_resolve_kernel(const int32_t* __restrict__ diff, uint32_t n, const int64_t* __restrict__ tile_base, uint32_t n_tiles,
                   uint64_t* __restrict__ slot) {
  if (!slot[COV_TOUCHED]) return;
  __shared__ uint32_t hist[2050];  // [2049] = deeper than 2048
  __shared__ int64_t ws[kCovThreads / 32];
  __shared__ unsigned long long bsum[2];
  __shared__ __align__(128) int32_t stage[2][kCovTile];
  __shared__ __align__(8) uint64_t bar[2];
  for (uint32_t i = threadIdx.x; i < 2050; i += blockDim.x) hist[i] = 0;
  if (threadIdx.x == 0) {
    mbar_init(&bar[0], 1);
    mbar_init(&bar[1], 1);
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  }
  __syncthreads();
  const uint32_t lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
  // bytes of tile t in the array, rounded up to the 16 bytes a bulk copy moves (the array is padded: engine.cu)
  auto tile_bytes = [&](uint32_t t) { const uint32_t left = n - t * kCovTile; return ((left < (uint32_t)kCovTile ? left : (uint32_t)kCovTile) * 4u + 15u) & ~15u; };
  if (threadIdx.x == 0 && blockIdx.x < n_tiles) {
    mbar_expect_tx(&bar[0], tile_bytes(blockIdx.x));
    bulk_g2s(stage[0], diff + (size_t)blockIdx.x * kCovTile, tile_bytes(blockIdx.x), &bar[0]);
  }
  uint32_t it = 0;
  for (uint32_t t = blockIdx.x; t < n_tiles; t += gridDim.x, ++it) {
    const uint32_t p0 = t * kCovTile + threadIdx.x * kCovPerThread;  // first position of this thread
    int32_t v[kCovPerThread];
    const uint32_t buf = it & 1;
    // the next tile streams into the other stage while this one is consumed (every thread left that stage at the
    // __syncthreads() that closed the previous iteration)
    const uint32_t tn = t + gridDim.x;
    if (threadIdx.x == 0 && tn < n_tiles) {
      mbar_expect_tx(&bar[buf ^ 1], tile_bytes(tn));
      bulk_g2s(stage[buf ^ 1], diff + (size_t)tn * kCovTile, tile_bytes(tn), &bar[buf ^ 1]);
    }
    mbar_wait(&bar[buf], (it >> 1) & 1);
    const int4* sp = reinterpret_cast<const int4*>(&stage[buf][threadIdx.x * kCovPerThread]);
#pragma unroll
    for (int k = 0; k < kCovPerThread; k += 4) {
      const int4 q = sp[k / 4];
      const uint32_t i = p0 + k;
      v[k] = i < n ? q.x : 0; v[k + 1] = i + 1 < n ? q.y : 0; v[k + 2] = i + 2 < n ? q.z : 0; v[k + 3] = i + 3 < n ? q.w : 0;
    }
    int64_t tsum = 0;
#pragma unroll
    for (int k = 0; k < kCovPerThread; ++k) tsum += v[k];
    // exclusive scan of thread sums across the CTA
    int64_t x = tsum;
    for (int o = 1; o < 32; o <<= 1) {
      int64_t y = __shfl_up_sync(0xFFFFFFFFu, x, o);
      if ((int)lane >= o) x += y;
    }
    if (threadIdx.x < 2) bsum[threadIdx.x] = 0;
    if (lane == 31) ws[wid] = x;
    __syncthreads();
    int64_t wbase = 0;
    for (uint32_t w = 0; w < wid; ++w) wbase += ws[w];
    int64_t depth = tile_base[t] + wbase + x - tsum;
    // positions -> depth; run-length aggregated histogram; bin sums
    const uint32_t k0 = (t * kCovTile + kCovBin - 1) / kCovBin;  // bin of the tile's first position (0 for position 0)
    const uint32_t bin_last = k0 * kCovBin;                       // last position of that bin: bin k = (50000(k-1), 50000k]
    unsigned long long s0 = 0, s1 = 0;
    int64_t run_d = -1;
    uint32_t run_n = 0;
#pragma unroll
    for (int k = 0; k < kCovPerThread; ++k) {
      uint32_t i = p0 + k;
      depth += v[k];
      if (i < n) {
        if (i <= bin_last) s0 += (unsigned long long)depth; else s1 += (unsigned long long)depth;  // a tile meets at most two bins
        if (depth == run_d) ++run_n;
        else {
          if (run_n) atomicAdd(&hist[cov_hist_slot(run_d)], run_n);
          run_d = depth;
          run_n = 1;
        }
      }
    }
    if (run_n) atomicAdd(&hist[cov_hist_slot(run_d)], run_n);
    // 64-bit butterfly: two independent 32-bit reductions of the halves would drop the carry out of the low words once the
    // 32 lanes' sums pass 2^32 (depth of a few million over the warp's 512 positions: amplicon / rRNA data)
#pragma unroll
    for (int o = 16; o; o >>= 1) {
      s0 += __shfl_down_sync(0xFFFFFFFFu, s0, o);
      s1 += __shfl_down_sync(0xFFFFFFFFu, s1, o);
    }
    if (lane == 0) {
      if (s0) atomicAdd(&bsum[0], s0);
      if (s1) atomicAdd(&bsum[1], s1);
    }
    __syncthreads();
    if (threadIdx.x == 0) {
      if (bsum[0]) atomicAdd((unsigned long long*)&slot[COV_BINS + k0], bsum[0]);
      if (bsum[1]) atomicAdd((unsigned long long*)&slot[COV_BINS + k0 + 1], bsum[1]);
    }
    __syncthreads();
  }
  for (uint32_t i = threadIdx.x; i <= 2048; i += blockDim.x)
    if (hist[i]) atomicAdd((unsigned long long*)&slot[COV_HIST + i], (unsigned long long)hist[i]);
  if (threadIdx.x == 0 && hist[2049]) atomicAdd((unsigned long long*)&slot[COV_TOO_LARGE], (unsigned long long)hist[2049]);
}

}  // namespace ngsq
