// Two building blocks shared by mesh.cu (region filter, vertex / face compaction) and components.cu (connected-component
// labelling of masks):
//   * an in-place exclusive scan of uint32 words (three launches: per-tile sums, one-block scan of the sums, apply);
//   * a union-find over an int parent array whose union always hooks the larger root under the smaller.  Every parent
//     pointer then points at a smaller index, so the root of a set is its minimum element whatever order concurrent
//     unions resolve in.  The pointers may live in global or shared memory (generic addressing).
#pragma once
#include <cuda_runtime.h>

#include <cstdint>

#include "api_common.h"

namespace oai {
namespace {

// ------------------------------------------------------------------------------------------------ exclusive scan (uint32)
constexpr int kScanBlock = 256, kScanItems = 4, kScanTile = kScanBlock * kScanItems;

__device__ __forceinline__ uint32_t block_exclusive_scan(uint32_t v, uint32_t* total) {
  __shared__ uint32_t warp_sums[kScanBlock / 32];
  const int lane = threadIdx.x & 31, wrp = threadIdx.x >> 5;
  uint32_t incl = v;
#pragma unroll
  for (int d = 1; d < 32; d <<= 1) {
    const uint32_t n = __shfl_up_sync(0xffffffffu, incl, d);
    if (lane >= d) incl += n;
  }
  if (lane == 31) warp_sums[wrp] = incl;
  __syncthreads();
  if (wrp == 0) {
    uint32_t s = lane < kScanBlock / 32 ? warp_sums[lane] : 0;
#pragma unroll
    for (int d = 1; d < kScanBlock / 32; d <<= 1) {
      const uint32_t n = __shfl_up_sync(0xffffffffu, s, d);
      if (lane >= d) s += n;
    }
    if (lane < kScanBlock / 32) warp_sums[lane] = s;
  }
  __syncthreads();
  const uint32_t before = wrp ? warp_sums[wrp - 1] : 0;
  if (total) *total = warp_sums[kScanBlock / 32 - 1];
  __syncthreads();
  return before + incl - v;
}

__global__ void __launch_bounds__(kScanBlock) scan_reduce_kernel(const uint32_t* __restrict__ in, long long n,
                                                                uint32_t* __restrict__ block_sums) {
  const long long base = static_cast<long long>(blockIdx.x) * kScanTile + threadIdx.x * kScanItems;
  uint32_t s = 0;
#pragma unroll
  for (int k = 0; k < kScanItems; ++k) if (base + k < n) s += in[base + k];
  uint32_t total;
  block_exclusive_scan(s, &total);
  if (threadIdx.x == 0) block_sums[blockIdx.x] = total;
}

// single block: exclusive scan of the block sums in place; the grand total lands in sums[nblocks]
__global__ void __launch_bounds__(kScanBlock) scan_sums_kernel(uint32_t* sums, int nblocks) {
  __shared__ uint32_t carry_s;
  if (threadIdx.x == 0) carry_s = 0;
  __syncthreads();
  for (int b0 = 0; b0 < nblocks; b0 += kScanBlock) {
    const int i = b0 + threadIdx.x;
    const uint32_t v = i < nblocks ? sums[i] : 0;
    uint32_t total;
    const uint32_t ex = block_exclusive_scan(v, &total);
    const uint32_t carry = carry_s;
    if (i < nblocks) sums[i] = carry + ex;
    __syncthreads();
    if (threadIdx.x == 0) carry_s = carry + total;
    __syncthreads();
  }
  if (threadIdx.x == 0) sums[nblocks] = carry_s;
}

__global__ void __launch_bounds__(kScanBlock) scan_apply_kernel(uint32_t* __restrict__ data, long long n,
                                                               const uint32_t* __restrict__ block_sums) {
  const long long base = static_cast<long long>(blockIdx.x) * kScanTile + threadIdx.x * kScanItems;
  uint32_t v[kScanItems], s = 0;
#pragma unroll
  for (int k = 0; k < kScanItems; ++k) { v[k] = base + k < n ? data[base + k] : 0; s += v[k]; }
  uint32_t run = block_exclusive_scan(s, nullptr) + block_sums[blockIdx.x];
#pragma unroll
  for (int k = 0; k < kScanItems; ++k) {
    if (base + k < n) data[base + k] = run;
    run += v[k];
  }
}

int scan_blocks(long long n) { return static_cast<int>((n + kScanTile - 1) / kScanTile); }

// in-place exclusive scan of data[n]; sums: scan_blocks(n) + 1 words; the total ends in sums[scan_blocks(n)]
int exclusive_scan(uint32_t* data, long long n, uint32_t* sums, cudaStream_t st) {
  const int nb = scan_blocks(n);
  scan_reduce_kernel<<<nb, kScanBlock, 0, st>>>(data, n, sums);
  if (int rc = launched("scan_reduce_kernel")) return rc;
  scan_sums_kernel<<<1, kScanBlock, 0, st>>>(sums, nb);
  if (int rc = launched("scan_sums_kernel")) return rc;
  scan_apply_kernel<<<nb, kScanBlock, 0, st>>>(data, n, sums);
  return launched("scan_apply_kernel");
}

// ------------------------------------------------------------------------------------------------ min-root union-find
__device__ __forceinline__ int uf_find(int* parent, int x) {
  while (true) {
    const int px = parent[x];
    if (px == x) return x;
    const int ppx = parent[px];
    if (ppx != px) parent[x] = ppx;   // path halving (benign race: any ancestor is a valid parent)
    x = px;
  }
}
__device__ __forceinline__ void uf_union(int* parent, int a, int b) {
  while (true) {
    a = uf_find(parent, a);
    b = uf_find(parent, b);
    if (a == b) return;
    if (a < b) { const int t = a; a = b; b = t; }   // the larger root is hooked under the smaller
    if (atomicCAS(&parent[a], a, b) == a) return;
  }
}

}  // namespace
}  // namespace oai
