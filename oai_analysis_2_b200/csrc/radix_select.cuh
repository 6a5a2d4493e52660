// Exact order statistics of float32 keys on the device: a three-pass radix select (11 + 11 + 10 bits of the
// order-preserving integer image of the keys) for up to kTargets ranks at once.  The caller zeroes the histograms and
// sets n and the ranks (select_reset plus its own rank computation), then runs
//   select_hist_kernel<0>, select_pick_kernel<0>, <1>, <1>, <2>, <2>
// after which key_float(prefix[k]) is the key of the rank the caller set in rank[k].  Histograms are integer atomics, so the result does
// not depend on the order in which the keys are visited.  Used by preproc.cu (np.percentile of a volume) and
// seg_quality.cu (np.percentile of the surface distances).
#pragma once
#include <cuda_runtime.h>

#include "api_common.h"

namespace oai {
namespace {

constexpr int kTargets = 4;
struct SelectState {
  long long n;                         // number of keys read by the histogram passes
  unsigned long long rank[kTargets];   // remaining rank inside the surviving prefix
  unsigned int prefix[kTargets];       // selected high bits so far
  unsigned int hist1[2048];
  unsigned int hist2[kTargets][2048];
  unsigned int hist3[kTargets][1024];
  float frac[2];                       // preproc.cu: interpolation weights (numpy's gamma) of the two percentiles
  double window[2];                    // preproc.cu: result, window_min and window_max
};

__device__ __forceinline__ unsigned int float_key(float v) {
  const unsigned int u = __float_as_uint(v);
  return (u & 0x80000000u) ? ~u : (u | 0x80000000u);  // monotone: key order == float order
}
__device__ __forceinline__ float key_float(unsigned int k) {
  return __uint_as_float((k & 0x80000000u) ? (k & 0x7fffffffu) : ~k);
}

// zero the histograms and the prefixes; every thread of the block takes part
__device__ __forceinline__ void select_reset(SelectState* s) {
  for (int i = threadIdx.x; i < 2048; i += blockDim.x) {
    s->hist1[i] = 0;
    for (int k = 0; k < kTargets; ++k) s->hist2[k][i] = 0;
    if (i < 1024)
      for (int k = 0; k < kTargets; ++k) s->hist3[k][i] = 0;
  }
  if (threadIdx.x < kTargets) s->prefix[threadIdx.x] = 0;
}

// PASS 0: top 11 bits of every key; PASS 1 / 2: next 11 / last 10 bits of the keys whose higher bits match a target.
// `in` is 16-byte aligned.
template <int PASS>
__global__ void __launch_bounds__(512) select_hist_kernel(const float* __restrict__ in, SelectState* s) {
  constexpr int BINS = PASS == 2 ? 1024 : 2048;
  constexpr int NH = PASS == 0 ? 1 : kTargets;
  __shared__ unsigned int sh[NH][BINS];
  for (int i = threadIdx.x; i < NH * BINS; i += blockDim.x) (&sh[0][0])[i] = 0;
  unsigned int pre[kTargets] = {0, 0, 0, 0};
  if (PASS > 0) {
#pragma unroll
    for (int k = 0; k < kTargets; ++k) pre[k] = s->prefix[k];
  }
  const long long n = s->n;
  __syncthreads();
  const long long n4 = n / 4;
  auto visit = [&](float v) {
    const unsigned int key = float_key(v);
    if (PASS == 0) {
      // smooth volumes put most keys of a warp into a handful of bins: one atomic per distinct bin of the warp
      const unsigned int bin = key >> 21, act = __activemask();
      const unsigned int same = __match_any_sync(act, bin);
      if ((__ffs(same) - 1) == static_cast<int>(threadIdx.x & 31)) atomicAdd(&sh[0][bin], __popc(same));
    } else {
      const unsigned int hi = PASS == 1 ? key >> 21 : key >> 10;
      const unsigned int bin = PASS == 1 ? (key >> 10) & 2047u : key & 1023u;
#pragma unroll
      for (int k = 0; k < kTargets; ++k)
        if (hi == pre[k]) atomicAdd(&sh[PASS == 0 ? 0 : k][bin], 1u);
    }
  };
  for (long long i = blockIdx.x * static_cast<long long>(blockDim.x) + threadIdx.x; i < n4;
       i += static_cast<long long>(gridDim.x) * blockDim.x) {
    const float4 v = __ldg(reinterpret_cast<const float4*>(in) + i);
    visit(v.x); visit(v.y); visit(v.z); visit(v.w);
  }
  if (blockIdx.x == 0)
    for (long long i = 4 * n4 + threadIdx.x; i < n; i += blockDim.x) visit(__ldg(in + i));
  __syncthreads();
  unsigned int* g = PASS == 0 ? s->hist1 : (PASS == 1 ? &s->hist2[0][0] : &s->hist3[0][0]);
  for (int i = threadIdx.x; i < NH * BINS; i += blockDim.x) {
    const unsigned int c = (&sh[0][0])[i];
    if (c) atomicAdd(g + i, c);
  }
}

// one warp per target: find the bin holding the remaining rank, extend the prefix
template <int PASS>
__global__ void __launch_bounds__(32 * kTargets) select_pick_kernel(SelectState* s) {
  constexpr int BINS = PASS == 2 ? 1024 : 2048;
  constexpr int BITS = PASS == 2 ? 10 : 11;
  const int k = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const unsigned int* h = PASS == 0 ? s->hist1 : (PASS == 1 ? s->hist2[k] : s->hist3[k]);
  unsigned long long rank = s->rank[k], base = 0;
  int found = -1;
  for (int b0 = 0; b0 < BINS && found < 0; b0 += 32) {
    const unsigned int c = h[b0 + lane];
    unsigned long long incl = c;  // inclusive scan over the warp
#pragma unroll
    for (int d = 1; d < 32; d <<= 1) {
      const unsigned long long o = __shfl_up_sync(0xffffffffu, incl, d);
      if (lane >= d) incl += o;
    }
    const bool here = base + incl > rank;
    const unsigned int m = __ballot_sync(0xffffffffu, here);
    if (m) {
      const int l = __ffs(m) - 1;
      const unsigned long long before = base + __shfl_sync(0xffffffffu, incl, l) - __shfl_sync(0xffffffffu, (unsigned long long)c, l);
      found = b0 + l;
      rank -= before;
    } else {
      base += __shfl_sync(0xffffffffu, incl, 31);
    }
  }
  if (found < 0) found = BINS - 1;  // unreachable for rank < n
  if (lane == 0) {
    s->rank[k] = rank;
    s->prefix[k] = (s->prefix[k] << BITS) | static_cast<unsigned int>(found);
  }
}

// the six launches of the select on `stream`, after the caller has reset the state and set n and the ranks
inline int select_launch(const float* in, SelectState* s, unsigned grid, cudaStream_t st) {
  select_hist_kernel<0><<<grid, 512, 0, st>>>(in, s);
  if (int rc = launched("select_hist_kernel<0>")) return rc;
  select_pick_kernel<0><<<1, 32 * kTargets, 0, st>>>(s);
  if (int rc = launched("select_pick_kernel<0>")) return rc;
  select_hist_kernel<1><<<grid, 512, 0, st>>>(in, s);
  if (int rc = launched("select_hist_kernel<1>")) return rc;
  select_pick_kernel<1><<<1, 32 * kTargets, 0, st>>>(s);
  if (int rc = launched("select_pick_kernel<1>")) return rc;
  select_hist_kernel<2><<<grid, 512, 0, st>>>(in, s);
  if (int rc = launched("select_hist_kernel<2>")) return rc;
  select_pick_kernel<2><<<1, 32 * kTargets, 0, st>>>(s);
  return launched("select_pick_kernel<2>");
}

}  // namespace
}  // namespace oai
