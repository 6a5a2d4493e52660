// Segmentation quality on the device: Dice, volumes and the surface distances (ASSD, HD95, HD) of two masks, over an
// exact separable Euclidean distance transform with per-axis spacing (Felzenszwalb & Huttenlocher, "Distance
// Transforms of Sampled Functions", 2012).  Two channels travel through the same three passes: channel 0 is the EDT to
// the surface of B, channel 1 the EDT to the surface of A.
//   * pass 1 (edt_x_kernel)        : one warp per x line.  The 6-neighbour border test of both masks and the mask
//                                    counts, then the 1-D nearest feature along x by a warp scan; the squared distance
//                                    in mm^2 goes to tmp[channel][D][H][W] (float32) through a shared-memory row, so
//                                    loads and stores stay coalesced.
//   * pass 2 (edt_envelope<false>) : lower envelope of the parabolas tmp(y') + ((y - y') sy)^2 along y, one thread per
//                                    line with x across the warp (coalesced), the envelope stack in shared memory;
//                                    written back in place.
//   * pass 3 (edt_envelope<true>)  : the same along z; the square root is the distance.  A voxel is a feature of a
//                                    channel iff its value there is exactly 0 after pass 2, so the surface of the other
//                                    mask is read off the other channel without materialising it.  Count, fp64 sum and
//                                    max of the distances at those voxels become per-block partials; the distances
//                                    themselves are appended to a list for the HD95 order statistic.
// HD95 is numpy's linear percentile of the pooled list: the exact radix select of radix_select.cuh finds the two
// order statistics, the lerp runs in fp64.  Every float reduction is fixed-order (per-block partials, one finishing
// kernel); the integer atomics (list slots, select histograms) do not change any result.  Nothing allocates or
// synchronises, so the launches can be captured in a CUDA graph.
#include "../../include/oai_b200.h"
#include "api_common.h"
#include "radix_select.cuh"

#include <cmath>
#include <cstdint>

namespace oai {
namespace {

constexpr int kMaxLen = 512;     // longest supported axis; the envelope stack indexes fit uint16
constexpr int kRows = 8;         // pass 1: x lines (warps) per block
constexpr int kFar = 1 << 20;    // "no feature on this side" in pass 1
constexpr size_t kEnvelopeSmemMax = static_cast<size_t>(kMaxLen) * 32 * (sizeof(float) + sizeof(uint16_t));

struct SurfaceState {
  SelectState sel;
  unsigned long long list_n;     // pooled surface distances written so far
  double gamma;                  // numpy's interpolation weight of the 95th percentile
};

struct EdtParams {
  const uint8_t* a;              // surface mode: the two masks
  const uint8_t* b;
  const uint8_t* feature;        // distance-transform mode: the feature set (a, b unused, one channel)
  int D, H, W, nch;
  double sx, sy, sz;
  float* tmp;                    // [nch][D][H][W]
  float* map[2];                 // pass 3 output per channel, optional
  long long* mask_partials;      // pass 1: [3][blocks] = |A|, |B|, |A & B| (surface mode)
  long long* cnt_partials;       // pass 3: [2][blocks] surface voxels seen (surface mode)
  double* sum_partials;          // pass 3: [2][blocks]
  float* max_partials;           // pass 3: [2][blocks]
  float* list;                   // pooled distances, room for 2 * nvox
  SurfaceState* st;
};

__global__ void __launch_bounds__(32 * kRows) edt_x_kernel(const EdtParams p) {
  __shared__ uint8_t flags[kRows][kMaxLen];
  __shared__ float row_out[kRows][kMaxLen];
  __shared__ int warp_counts[3][kRows];
  const int w = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int y = blockIdx.x * kRows + w, z = blockIdx.y;
  const int D = p.D, H = p.H, W = p.W;
  const long long hw = static_cast<long long>(H) * W, nvox = hw * D;
  int cA = 0, cB = 0, cAB = 0;
  if (y < H) {  // warp-uniform
    const long long row = (static_cast<long long>(z) * H + y) * W;
    for (int x = lane; x < W; x += 32) {
      uint8_t f;
      if (p.feature) {
        f = __ldg(p.feature + row + x) != 0;
      } else {
        // bit 0: feature of channel 0 (surface of B), bit 1: feature of channel 1 (surface of A)
        const bool face = x == 0 || x == W - 1 || y == 0 || y == H - 1 || z == 0 || z == D - 1;
        auto surface = [&](const uint8_t* m, bool& inside) {
          const uint8_t* c = m + row + x;
          inside = __ldg(c) != 0;
          return inside && (face || !__ldg(c - 1) || !__ldg(c + 1) || !__ldg(c - W) || !__ldg(c + W) ||
                            !__ldg(c - hw) || !__ldg(c + hw));
        };
        bool inA, inB;
        const bool sA = surface(p.a, inA), sB = surface(p.b, inB);
        cA += inA;
        cB += inB;
        cAB += inA && inB;
        f = (sB ? 1 : 0) | (sA ? 2 : 0);
      }
      flags[w][x] = f;
    }
    __syncwarp();
    // lane l owns the chunk [x0, x1); nearest feature to the left / right from a warp max / min scan of the chunks
    const int C = (W + 31) / 32, x0 = lane * C, x1 = min(x0 + C, W);
    for (int c = 0; c < p.nch; ++c) {
      int last = -kFar, first = kFar;
      for (int x = x0; x < x1; ++x)
        if ((flags[w][x] >> c) & 1) {
          first = min(first, x);
          last = x;
        }
      int lsc = last, rsc = first;
#pragma unroll
      for (int d = 1; d < 32; d <<= 1) {
        const int l = __shfl_up_sync(0xffffffffu, lsc, d), r = __shfl_down_sync(0xffffffffu, rsc, d);
        if (lane >= d) lsc = max(lsc, l);
        if (lane + d < 32) rsc = min(rsc, r);
      }
      int left = __shfl_up_sync(0xffffffffu, lsc, 1), right = __shfl_down_sync(0xffffffffu, rsc, 1);
      if (lane == 0) left = -kFar;
      if (lane == 31) right = kFar;
      int* nearest_right = reinterpret_cast<int*>(row_out[w]);
      for (int x = x1 - 1; x >= x0; --x) {
        if ((flags[w][x] >> c) & 1) right = x;
        nearest_right[x] = right;
      }
      for (int x = x0; x < x1; ++x) {
        if ((flags[w][x] >> c) & 1) left = x;
        const int dist = min(x - left, nearest_right[x] - x);
        const double d = dist * p.sx;
        row_out[w][x] = dist >= kFar / 2 ? INFINITY : static_cast<float>(d * d);
      }
      __syncwarp();
      float* dst = p.tmp + c * nvox + row;
      for (int x = lane; x < W; x += 32) dst[x] = row_out[w][x];
      __syncwarp();
    }
  }
  if (p.mask_partials) {
    const int v[3] = {__reduce_add_sync(0xffffffffu, cA), __reduce_add_sync(0xffffffffu, cB),
                      __reduce_add_sync(0xffffffffu, cAB)};
    if (lane == 0)
      for (int k = 0; k < 3; ++k) warp_counts[k][w] = v[k];
    __syncthreads();
    if (threadIdx.x < 3) {
      long long s = 0;
      for (int i = 0; i < kRows; ++i) s += warp_counts[threadIdx.x][i];
      const long long blocks = static_cast<long long>(gridDim.x) * gridDim.y;
      p.mask_partials[threadIdx.x * blocks + static_cast<long long>(blockIdx.y) * gridDim.x + blockIdx.x] = s;
    }
  }
}

// boundary between parabola i (height fi) and parabola j > i (height fj) of f(i) + ((q - i) s)^2, in voxels
__device__ __forceinline__ double parabola_sep(int i, float fi, int j, float fj, double s2) {
  return (static_cast<double>(fj) - static_cast<double>(fi) + s2 * (static_cast<double>(j) * j -
                                                                      static_cast<double>(i) * i)) /
         (2.0 * s2 * (j - i));
}

// One warp per block: 32 consecutive x of one line set and one channel (blockIdx.z).  LAST = false: lines along y of
// plane z = blockIdx.y, in place.  LAST = true: lines along z of row y = blockIdx.y, distances and reductions.
template <bool LAST>
__global__ void __launch_bounds__(32) edt_envelope_kernel(const EdtParams p) {
  extern __shared__ __align__(16) unsigned char smem[];
  const int n = LAST ? p.D : p.H;
  float* sf = reinterpret_cast<float*>(smem);                  // [n][32] parabola heights
  uint16_t* sv = reinterpret_cast<uint16_t*>(sf + n * 32);      // [n][32] parabola apexes
  const int lane = threadIdx.x, x = blockIdx.x * 32 + lane, c = blockIdx.z, o = blockIdx.y;
  const bool valid = x < p.W;
  const long long hw = static_cast<long long>(p.H) * p.W, nvox = hw * p.D;
  const long long stride = LAST ? hw : p.W;
  const long long off = (LAST ? static_cast<long long>(o) * p.W : static_cast<long long>(o) * hw) + x;
  float* line = p.tmp + c * nvox + off;
  const double s = LAST ? p.sz : p.sy, s2 = s * s;
  // lower envelope: stack of parabolas (apex, height); ztop = left boundary of the top one
  int k = -1;
  double ztop = -INFINITY;
  for (int q = 0; q < n; ++q) {
    const float fq = valid ? line[q * stride] : INFINITY;
    if (!(fq < INFINITY)) continue;
    double zq = -INFINITY;
    while (k >= 0) {
      zq = parabola_sep(sv[k * 32 + lane], sf[k * 32 + lane], q, fq, s2);
      if (zq > ztop) break;
      --k;
      ztop = k >= 1 ? parabola_sep(sv[(k - 1) * 32 + lane], sf[(k - 1) * 32 + lane], sv[k * 32 + lane],
                                   sf[k * 32 + lane], s2)
                    : -INFINITY;
      zq = -INFINITY;
    }
    ++k;
    sv[k * 32 + lane] = static_cast<uint16_t>(q);
    sf[k * 32 + lane] = fq;
    ztop = zq;
  }
  if (!LAST && k < 0) return;  // no feature on this line: it stays +inf
  const bool reduce = LAST && p.list != nullptr;
  long long cnt = 0;
  double sum = 0.0;
  float mx = 0.f;
  int j = 0, vj = 0;
  float fj = 0.f;
  double zn = INFINITY;  // right boundary of parabola j
  if (k >= 0) {
    vj = sv[lane];
    fj = sf[lane];
    if (k > 0) zn = parabola_sep(vj, fj, sv[32 + lane], sf[32 + lane], s2);
  }
  for (int q = 0; q < n; ++q) {
    double val = INFINITY;
    if (k >= 0) {
      while (zn < q) {
        ++j;
        vj = sv[j * 32 + lane];
        fj = sf[j * 32 + lane];
        zn = j < k ? parabola_sep(vj, fj, sv[(j + 1) * 32 + lane], sf[(j + 1) * 32 + lane], s2) : INFINITY;
      }
      const double dq = static_cast<double>(q - vj) * s;
      val = static_cast<double>(fj) + dq * dq;
    }
    if (!LAST) {
      if (valid) line[q * stride] = static_cast<float>(val);
      continue;
    }
    const double dist = sqrt(val);
    const float df = static_cast<float>(dist);
    const long long v = q * stride + off;
    if (valid && p.map[c]) p.map[c][v] = df;
    if (reduce) {
      const bool surf = valid && p.tmp[(1 - c) * nvox + v] == 0.f;
      if (surf) {
        ++cnt;
        sum += dist;
        mx = fmaxf(mx, df);
      }
      const unsigned m = __ballot_sync(0xffffffffu, surf);
      if (m) {
        unsigned long long base = 0;
        if (lane == __ffs(m) - 1) base = atomicAdd(&p.st->list_n, static_cast<unsigned long long>(__popc(m)));
        base = __shfl_sync(0xffffffffu, base, __ffs(m) - 1);
        if (surf) p.list[base + __popc(m & ((1u << lane) - 1u))] = df;
      }
    }
  }
  if (reduce) {
#pragma unroll
    for (int d = 16; d > 0; d >>= 1) {
      cnt += __shfl_down_sync(0xffffffffu, cnt, d);
      sum += __shfl_down_sync(0xffffffffu, sum, d);
      mx = fmaxf(mx, __shfl_down_sync(0xffffffffu, mx, d));
    }
    if (lane == 0) {
      const long long blocks = static_cast<long long>(gridDim.x) * gridDim.y;
      const long long i = c * blocks + static_cast<long long>(blockIdx.y) * gridDim.x + blockIdx.x;
      p.cnt_partials[i] = cnt;
      p.sum_partials[i] = sum;
      p.max_partials[i] = mx;
    }
  }
}

__global__ void __launch_bounds__(256) surface_init_kernel(SurfaceState* st) {
  if (threadIdx.x == 0) st->list_n = 0;
}

// numpy's linear percentile 95 of the n pooled distances: ranks floor(vi), floor(vi) + 1 with vi = (n - 1) * 0.95
__global__ void __launch_bounds__(256) surface_rank_kernel(SurfaceState* st) {
  select_reset(&st->sel);
  if (threadIdx.x == 0) {
    const long long n = static_cast<long long>(st->list_n);
    st->sel.n = n;
    unsigned long long k0 = 0, k1 = 0;
    double gamma = 0.0;
    if (n > 0) {
      const double vi = static_cast<double>(n - 1) * 0.95;
      if (vi >= static_cast<double>(n - 1)) {
        k0 = k1 = static_cast<unsigned long long>(n - 1);
      } else {
        const double f = floor(vi);
        k0 = static_cast<unsigned long long>(f);
        k1 = k0 + 1;
        gamma = vi - f;
      }
    }
    st->sel.rank[0] = st->sel.rank[2] = k0;
    st->sel.rank[1] = st->sel.rank[3] = k1;
    st->gamma = gamma;
  }
}

// fixed-order reduction of n values over the 256-thread block; every thread gets the result
template <class T, class Op>
__device__ T reduce_partials(const T* p, long long n, T init, Op op) {
  __shared__ T s[256];
  T v = init;
  for (long long i = threadIdx.x; i < n; i += 256) v = op(v, p[i]);
  s[threadIdx.x] = v;
  __syncthreads();
  for (int o = 128; o > 0; o >>= 1) {
    if (threadIdx.x < o) s[threadIdx.x] = op(s[threadIdx.x], s[threadIdx.x + o]);
    __syncthreads();
  }
  const T r = s[0];
  __syncthreads();
  return r;
}

__global__ void __launch_bounds__(256) surface_finish_kernel(const EdtParams p, int nb1, int nb3, double* terms,
                                                             long long* counts) {
  auto add_ll = [](long long a, long long b) { return a + b; };
  auto add_d = [](double a, double b) { return a + b; };
  auto max_f = [](float a, float b) { return fmaxf(a, b); };
  long long m[3], sc[2];
  double sum[2];
  float mx[2];
#pragma unroll
  for (int i = 0; i < 3; ++i) m[i] = reduce_partials(p.mask_partials + static_cast<long long>(i) * nb1, nb1, 0ll, add_ll);
#pragma unroll
  for (int c = 0; c < 2; ++c) {
    const long long o = static_cast<long long>(c) * nb3;
    sc[c] = reduce_partials(p.cnt_partials + o, nb3, 0ll, add_ll);
    sum[c] = reduce_partials(p.sum_partials + o, nb3, 0.0, add_d);
    mx[c] = reduce_partials(p.max_partials + o, nb3, 0.f, max_f);
  }
  if (threadIdx.x == 0) {
    const long long nA = m[0], nB = m[1], nAB = m[2];
    // sc[0]: voxels of the surface of A (where channel 0, the EDT to the surface of B, was read) and vice versa
    counts[0] = nA;
    counts[1] = nB;
    counts[2] = nAB;
    counts[3] = sc[0];
    counts[4] = sc[1];
    terms[0] = nA + nB > 0 ? static_cast<double>(2 * nAB) / static_cast<double>(nA + nB) : NAN;
    if (nA > 0 && nB > 0) {
      const double mean_ab = sum[0] / static_cast<double>(sc[0]), mean_ba = sum[1] / static_cast<double>(sc[1]);
      // numpy _lerp in fp64 of the two order statistics: a + (b - a) * t, taken from the other end for t >= 0.5
      const double a = key_float(p.st->sel.prefix[0]), b = key_float(p.st->sel.prefix[1]), t = p.st->gamma;
      const double d = __dsub_rn(b, a);
      terms[1] = (mean_ab + mean_ba) / 2.0;
      terms[2] = t >= 0.5 ? __dsub_rn(b, __dmul_rn(d, __dsub_rn(1.0, t))) : __dadd_rn(a, __dmul_rn(d, t));
      terms[3] = fmax(static_cast<double>(mx[0]), static_cast<double>(mx[1]));
      terms[4] = mean_ab;
      terms[5] = mean_ba;
      terms[6] = mx[0];
      terms[7] = mx[1];
    } else {
      for (int i = 1; i < 8; ++i) terms[i] = NAN;
    }
  }
}

size_t align256(size_t v) { return (v + 255) & ~static_cast<size_t>(255); }

struct Layout {
  size_t tmp, list, state, mask, cnt, sum, mx, total;
  int nb1, nb3;
};

Layout layout(const int* d) {
  Layout l;
  const size_t nvox = static_cast<size_t>(d[0]) * d[1] * d[2];
  l.nb1 = ((d[1] + kRows - 1) / kRows) * d[0];
  l.nb3 = ((d[2] + 31) / 32) * d[1];
  size_t o = 0;
  l.tmp = o;   o = align256(o + 2 * nvox * sizeof(float));
  l.list = o;  o = align256(o + 2 * nvox * sizeof(float));
  l.state = o; o = align256(o + sizeof(SurfaceState));
  l.mask = o;  o = align256(o + 3 * static_cast<size_t>(l.nb1) * sizeof(long long));
  l.cnt = o;   o = align256(o + 2 * static_cast<size_t>(l.nb3) * sizeof(long long));
  l.sum = o;   o = align256(o + 2 * static_cast<size_t>(l.nb3) * sizeof(double));
  l.mx = o;    o = align256(o + 2 * static_cast<size_t>(l.nb3) * sizeof(float));
  l.total = o;
  return l;
}

int check_grid(const char* what, const int* dims, const double* spacing_xyz) {
  OAI_REQUIRE(dims && spacing_xyz, "%s: null pointer", what);
  for (int i = 0; i < 3; ++i)
    OAI_REQUIRE(dims[i] >= 1 && dims[i] <= kMaxLen, "%s: every axis needs 1 to %d voxels (got %d x %d x %d)", what,
                kMaxLen, dims[0], dims[1], dims[2]);
  for (int i = 0; i < 3; ++i)
    OAI_REQUIRE(std::isfinite(spacing_xyz[i]) && spacing_xyz[i] > 0.0,
                "%s: spacing must be positive and finite (got %g, %g, %g)", what, spacing_xyz[0], spacing_xyz[1],
                spacing_xyz[2]);
  return 0;
}

// passes 1-3 of the transform for the channels of p
int edt_launch(const EdtParams& p, cudaStream_t st) {
  static bool attr_set[64] = {false};   // the opt-in covers the longest axis once per device, before any capture
  int dev = 0;
  if (int rc = check_cuda(cudaGetDevice(&dev), "seg_quality: device")) return rc;
  if (dev < 0 || dev >= 64 || !attr_set[dev]) {
    if (int rc = check_cuda(cudaFuncSetAttribute(edt_envelope_kernel<false>,
                                                 cudaFuncAttributeMaxDynamicSharedMemorySize,
                                                 static_cast<int>(kEnvelopeSmemMax)),
                            "seg_quality: shared memory opt-in"))
      return rc;
    if (int rc = check_cuda(cudaFuncSetAttribute(edt_envelope_kernel<true>,
                                                 cudaFuncAttributeMaxDynamicSharedMemorySize,
                                                 static_cast<int>(kEnvelopeSmemMax)),
                            "seg_quality: shared memory opt-in"))
      return rc;
    if (dev >= 0 && dev < 64) attr_set[dev] = true;
  }
  const unsigned bx = static_cast<unsigned>((p.W + 31) / 32);
  edt_x_kernel<<<dim3((p.H + kRows - 1) / kRows, p.D), 32 * kRows, 0, st>>>(p);
  if (int rc = launched("edt_x_kernel")) return rc;
  const size_t per = 32 * (sizeof(float) + sizeof(uint16_t));
  edt_envelope_kernel<false><<<dim3(bx, p.D, p.nch), 32, per * p.H, st>>>(p);
  if (int rc = launched("edt_envelope_kernel<y>")) return rc;
  edt_envelope_kernel<true><<<dim3(bx, p.H, p.nch), 32, per * p.D, st>>>(p);
  return launched("edt_envelope_kernel<z>");
}

EdtParams make_params(const int* dims, const double* spacing_xyz, void* workspace, const Layout& l) {
  EdtParams p{};
  char* ws = static_cast<char*>(workspace);
  p.D = dims[0];
  p.H = dims[1];
  p.W = dims[2];
  p.sx = spacing_xyz[0];
  p.sy = spacing_xyz[1];
  p.sz = spacing_xyz[2];
  p.tmp = reinterpret_cast<float*>(ws + l.tmp);
  return p;
}

}  // namespace
}  // namespace oai

using namespace oai;

extern "C" size_t oai_seg_quality_workspace_bytes(const int* dims) {
  if (!dims) return 0;
  for (int i = 0; i < 3; ++i)
    if (dims[i] < 1 || dims[i] > kMaxLen) return 0;
  return layout(dims).total;
}

extern "C" int oai_distance_transform(const uint8_t* feature, const int* dims, const double* spacing_xyz, float* out,
                                      void* workspace, size_t workspace_bytes, void* stream) {
  if (int rc = check_grid("distance_transform", dims, spacing_xyz)) return rc;
  OAI_REQUIRE(feature && out && workspace, "distance_transform: null pointer");
  const Layout l = layout(dims);
  OAI_REQUIRE(workspace_bytes >= l.total && (reinterpret_cast<uintptr_t>(workspace) & 255) == 0,
              "distance_transform: workspace of %zu bytes (256-byte aligned) required, got %zu", l.total,
              workspace_bytes);
  EdtParams p = make_params(dims, spacing_xyz, workspace, l);
  p.feature = feature;
  p.nch = 1;
  p.map[0] = out;
  return edt_launch(p, static_cast<cudaStream_t>(stream));
}

extern "C" int oai_surface_metrics(const uint8_t* mask_a, const uint8_t* mask_b, const int* dims,
                                   const double* spacing_xyz, double* terms, long long* counts, float* dist_to_B,
                                   float* dist_to_A, void* workspace, size_t workspace_bytes, void* stream) {
  if (int rc = check_grid("surface_metrics", dims, spacing_xyz)) return rc;
  OAI_REQUIRE(mask_a && mask_b && terms && counts && workspace, "surface_metrics: null pointer");
  const Layout l = layout(dims);
  OAI_REQUIRE(workspace_bytes >= l.total && (reinterpret_cast<uintptr_t>(workspace) & 255) == 0,
              "surface_metrics: workspace of %zu bytes (256-byte aligned) required, got %zu", l.total,
              workspace_bytes);
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  char* ws = static_cast<char*>(workspace);
  EdtParams p = make_params(dims, spacing_xyz, workspace, l);
  p.a = mask_a;
  p.b = mask_b;
  p.nch = 2;
  p.map[0] = dist_to_B;
  p.map[1] = dist_to_A;
  p.list = reinterpret_cast<float*>(ws + l.list);
  p.st = reinterpret_cast<SurfaceState*>(ws + l.state);
  p.mask_partials = reinterpret_cast<long long*>(ws + l.mask);
  p.cnt_partials = reinterpret_cast<long long*>(ws + l.cnt);
  p.sum_partials = reinterpret_cast<double*>(ws + l.sum);
  p.max_partials = reinterpret_cast<float*>(ws + l.mx);
  surface_init_kernel<<<1, 32, 0, st>>>(p.st);
  if (int rc = launched("surface_init_kernel")) return rc;
  if (int rc = edt_launch(p, st)) return rc;
  surface_rank_kernel<<<1, 256, 0, st>>>(p.st);
  if (int rc = launched("surface_rank_kernel")) return rc;
  if (int rc = select_launch(p.list, &p.st->sel, static_cast<unsigned>(num_sms()) * 2, st)) return rc;
  surface_finish_kernel<<<1, 256, 0, st>>>(p, l.nb1, l.nb3, terms, counts);
  return launched("surface_finish_kernel");
}
