// Connected components of a 3-D mask on the device, numbered exactly like scipy.ndimage.label with the structuring
// element generate_binary_structure(3, r): r = 1, 2, 3 for 6-, 18- and 26-connectivity.  Block-based union-find
// (Playne & Hawick, TPDS 2018; Allegretti, Bolelli & Grana, TPDS 2020), with the labels buffer as the parent array:
//   * cc_local_kernel   : one CTA per 4 x 8 x 32 brick.  Union-find in shared memory over the brick's own edges, then
//                         every voxel gets the *global* linear index of its local root.  Raster order inside a brick is
//                         global linear order, so that root is the minimum global index of its local piece.
//   * cc_merge_kernel   : unions across brick faces, edges and corners in global memory (uf_union of
//                         scan_union_find.cuh, larger root hooked under the smaller), so each final root is the minimum
//                         linear index of its component whatever order the races resolve in.
//   * cc_flatten_kernel : every voxel's label becomes its root; roots (label == index) are flagged.
//   * exclusive scan of the flags -> rank of each root in raster order of first voxels.
//   * cc_relabel_kernel : label = 1 + rank of its root (scipy's numbering; background 0); sizes by warp-aggregated
//                         atomics (__match_any_sync, one atomic per group of equal labels), which keeps the largest
//                         component from serialising millions of atomics on one address.
// Labels and sizes are exact integers and the roots do not depend on scheduling, so equal inputs give bitwise-equal
// outputs.  Nothing allocates or synchronises: the launches can be captured in a CUDA graph.
#include "../../include/oai_b200.h"
#include "api_common.h"
#include "scan_union_find.cuh"

#include <cstdint>

namespace oai {
namespace {

constexpr int kBX = 32, kBY = 8, kBZ = 4, kBrick = kBX * kBY * kBZ;  // one thread per brick voxel
constexpr int kKeepThreads = 1024;

// the 13 offsets (dz, dy, dx) that precede the centre in raster order; offset k belongs to the structuring element of
// rank r iff |dz| + |dy| + |dx| <= r
__constant__ int8_t c_back[13][3] = {{-1, -1, -1}, {-1, -1, 0}, {-1, -1, 1}, {-1, 0, -1}, {-1, 0, 0},
                                     {-1, 0, 1},   {-1, 1, -1}, {-1, 1, 0},  {-1, 1, 1},  {0, -1, -1},
                                     {0, -1, 0},   {0, -1, 1},  {0, 0, -1}};

struct CcGeom {
  int D, H, W, rank;   // rank = 1, 2, 3 for connectivity 6, 18, 26
  int nbx, nby;        // bricks along x and y
};

__device__ __forceinline__ void brick_coords(const CcGeom& g, int& lx, int& ly, int& lz, int& x0, int& y0, int& z0) {
  const int l = threadIdx.x;
  lx = l % kBX;
  ly = (l / kBX) % kBY;
  lz = l / (kBX * kBY);
  const int b = blockIdx.x;
  x0 = (b % g.nbx) * kBX;
  y0 = ((b / g.nbx) % g.nby) * kBY;
  z0 = (b / (g.nbx * g.nby)) * kBZ;
}

__device__ __forceinline__ bool back_offset(const CcGeom& g, int k, int& dz, int& dy, int& dx) {
  dz = c_back[k][0];
  dy = c_back[k][1];
  dx = c_back[k][2];
  return abs(dz) + abs(dy) + abs(dx) <= g.rank;
}

__global__ void __launch_bounds__(kBrick) cc_local_kernel(const uint8_t* __restrict__ mask, int* __restrict__ labels,
                                                          const CcGeom g) {
  __shared__ int par[kBrick];
  int lx, ly, lz, x0, y0, z0;
  brick_coords(g, lx, ly, lz, x0, y0, z0);
  const int x = x0 + lx, y = y0 + ly, z = z0 + lz, l = threadIdx.x;
  const bool inside = x < g.W && y < g.H && z < g.D;
  const int gi = inside ? (z * g.H + y) * g.W + x : 0;
  const bool fg = inside && __ldg(mask + gi) != 0;
  par[l] = fg ? l : -1;
  __syncthreads();
  if (fg) {
    for (int k = 0; k < 13; ++k) {
      int dz, dy, dx;
      if (!back_offset(g, k, dz, dy, dx)) continue;
      const int nx = lx + dx, ny = ly + dy, nz = lz + dz;
      if (nx < 0 || nx >= kBX || ny < 0 || ny >= kBY || nz < 0) continue;   // nz < kBZ always holds (dz <= 0)
      const int nl = (nz * kBY + ny) * kBX + nx;
      if (par[nl] >= 0) uf_union(par, l, nl);   // a background slot stays -1, a foreground one never becomes -1
    }
  }
  __syncthreads();
  if (fg) {
    const int r = uf_find(par, l);
    const int rx = r % kBX, ry = (r / kBX) % kBY, rz = r / (kBX * kBY);
    labels[gi] = ((z0 + rz) * g.H + y0 + ry) * g.W + x0 + rx;
  } else if (inside) {
    labels[gi] = -1;
  }
}

// the edges the local pass could not see: a foreground voxel and a preceding neighbour in another brick
__global__ void __launch_bounds__(kBrick) cc_merge_kernel(const uint8_t* __restrict__ mask, int* labels,
                                                          const CcGeom g) {
  int lx, ly, lz, x0, y0, z0;
  brick_coords(g, lx, ly, lz, x0, y0, z0);
  // only the brick's low faces and (for rank >= 2) its x = 31 and y = 7 edges have such neighbours
  if (lz != 0 && ly != 0 && lx != 0 && lx != kBX - 1 && ly != kBY - 1) return;
  const int x = x0 + lx, y = y0 + ly, z = z0 + lz;
  if (x >= g.W || y >= g.H || z >= g.D) return;
  const int gi = (z * g.H + y) * g.W + x;
  if (!__ldg(mask + gi)) return;
  for (int k = 0; k < 13; ++k) {
    int dz, dy, dx;
    if (!back_offset(g, k, dz, dy, dx)) continue;
    const int nx = lx + dx, ny = ly + dy, nz = lz + dz;
    if (nx >= 0 && nx < kBX && ny >= 0 && ny < kBY && nz >= 0) continue;   // same brick: done by the local pass
    if (x + dx < 0 || x + dx >= g.W || y + dy < 0 || y + dy >= g.H || z + dz < 0) continue;
    const int gn = gi + (dz * g.H + dy) * g.W + dx;
    if (__ldg(mask + gn)) uf_union(labels, gi, gn);
  }
}

// The root chase does not compress paths: a path-halving write by another thread could land on labels[i] after this
// thread stored the root there and leave a non-root ancestor behind.  The only write is labels[i] = root.
__global__ void __launch_bounds__(256) cc_flatten_kernel(int* labels, uint32_t* __restrict__ root_flag, int n) {
  for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < n; i += gridDim.x * blockDim.x) {
    bool root = false;
    int r = labels[i];
    if (r >= 0) {
      for (int p = labels[r]; p != r; p = labels[r]) r = p;
      labels[i] = r;
      root = r == i;
    }
    root_flag[i] = root ? 1u : 0u;
  }
}

// rank: exclusive scan of the root flags.  The loop bound is warp-uniform so __match_any_sync sees whole warps.  Each
// warp carries the count of one label in a register (the largest group it last saw, usually the giant component) and
// adds it once at the end; the other groups take one atomic each.  One atomic per warp and step on the giant
// component's counter would otherwise serialise about N / 32 atomics on one address.
__global__ void __launch_bounds__(256) cc_relabel_kernel(int* labels, const uint32_t* __restrict__ rank, int n,
                                                         int* __restrict__ sizes, const uint32_t* __restrict__ total,
                                                         long long* count) {
  if (blockIdx.x == 0 && threadIdx.x == 0) *count = *total;
  const int lane = threadIdx.x & 31;
  int carried = 0;         // warp-uniform label whose count lives in `held`; 0 = none
  unsigned held = 0;
  for (int base = blockIdx.x * blockDim.x; base < n; base += gridDim.x * blockDim.x) {
    const int i = base + threadIdx.x;
    int lab = 0;
    if (i < n) {
      const int r = labels[i];
      lab = r >= 0 ? static_cast<int>(__ldg(rank + r)) + 1 : 0;
      labels[i] = lab;
    }
    const unsigned grp = __match_any_sync(0xffffffffu, lab);
    const unsigned same = __ballot_sync(0xffffffffu, carried > 0 && lab == carried);
    held += __popc(same);
    if (lab > 0 && lab != carried && lane == __ffs(grp) - 1) atomicAdd(sizes + lab - 1, __popc(grp));
    if (!same) {   // the carried label is absent here: flush it and carry the largest group of this step instead
      if (carried > 0 && lane == 0) atomicAdd(sizes + carried - 1, static_cast<int>(held));
      const unsigned key = __reduce_max_sync(0xffffffffu, lab > 0 ? (__popc(grp) << 5) | lane : 0u);
      carried = key ? __shfl_sync(0xffffffffu, lab, key & 31) : 0;
      held = 0;
    }
  }
  if (carried > 0 && lane == 0 && held) atomicAdd(sizes + carried - 1, static_cast<int>(held));
}

// min_voxels < 0: keep the largest component (lowest label on a tie: numpy's argmax); otherwise every component of at
// least min_voxels voxels.  Every block finds the largest itself from the sizes (cheap next to the volume pass for any
// real count), so the policy needs neither a second launch nor scratch memory.
__global__ void __launch_bounds__(kKeepThreads) cc_keep_kernel(const int* __restrict__ labels,
                                                               const int* __restrict__ sizes,
                                                               const long long* __restrict__ count, long long nvox,
                                                               int min_voxels, uint8_t* keep, float* values) {
  __shared__ unsigned long long warp_best[kKeepThreads / 32];
  int keep_label = 0;
  if (min_voxels < 0) {
    const int n = static_cast<int>(*count);
    // key: size in the high word, ~index in the low word, so the max is the largest size with the lowest index
    unsigned long long best = 0;
    for (int k = threadIdx.x; k < n; k += kKeepThreads) {
      const unsigned long long key =
          (static_cast<unsigned long long>(static_cast<uint32_t>(__ldg(sizes + k))) << 32) | (0xffffffffu - k);
      best = key > best ? key : best;
    }
#pragma unroll
    for (int d = 16; d > 0; d >>= 1) {
      const unsigned long long o = __shfl_down_sync(0xffffffffu, best, d);
      best = o > best ? o : best;
    }
    if ((threadIdx.x & 31) == 0) warp_best[threadIdx.x >> 5] = best;
    __syncthreads();
    best = 0;
    for (int w = 0; w < kKeepThreads / 32; ++w) best = warp_best[w] > best ? warp_best[w] : best;
    keep_label = best ? static_cast<int>(0xffffffffu - static_cast<uint32_t>(best)) + 1 : 0;
  }
  for (long long i = blockIdx.x * static_cast<long long>(kKeepThreads) + threadIdx.x; i < nvox;
       i += static_cast<long long>(gridDim.x) * kKeepThreads) {
    const int lab = labels[i];
    const bool k = lab > 0 && (min_voxels < 0 ? lab == keep_label : __ldg(sizes + lab - 1) >= min_voxels);
    if (keep) keep[i] = k ? 1 : 0;
    if (values && !k) values[i] = 0.f;
  }
}

size_t align256(size_t v) { return (v + 255) & ~static_cast<size_t>(255); }

int conn_rank(int connectivity) {
  return connectivity == 6 ? 1 : connectivity == 18 ? 2 : connectivity == 26 ? 3 : 0;
}

// D*H*W as long long, or -1 when an axis is < 1 or the volume does not fit int32 labels
long long voxel_count(const int* dims) {
  if (!dims || dims[0] < 1 || dims[1] < 1 || dims[2] < 1) return -1;
  const long long n = static_cast<long long>(dims[0]) * dims[1] * dims[2];
  return n < (1ll << 31) ? n : -1;
}

struct CcLayout {
  size_t rank, sums, total;
};

CcLayout cc_layout(long long n) {
  CcLayout l;
  size_t o = 0;
  l.rank = o; o = align256(o + static_cast<size_t>(n) * sizeof(uint32_t));
  l.sums = o; o = align256(o + static_cast<size_t>(scan_blocks(n) + 1) * sizeof(uint32_t));
  l.total = o;
  return l;
}

int check_dims(const char* what, const int* dims) {
  OAI_REQUIRE(dims, "%s: null pointer", what);
  OAI_REQUIRE(dims[0] >= 1 && dims[1] >= 1 && dims[2] >= 1, "%s: every axis needs at least 1 voxel (got %d x %d x %d)",
              what, dims[0], dims[1], dims[2]);
  OAI_REQUIRE(voxel_count(dims) > 0, "%s: D*H*W must be below 2^31 for int32 labels (got %d x %d x %d)", what,
              dims[0], dims[1], dims[2]);
  return 0;
}

int grid_for(long long n, int threads) {
  const long long b = (n + threads - 1) / threads, cap = static_cast<long long>(num_sms()) * (2048 / threads);
  return static_cast<int>(b < cap ? b : cap);
}

}  // namespace
}  // namespace oai

using namespace oai;

extern "C" size_t oai_components_workspace_bytes(const int* dims) {
  const long long n = voxel_count(dims);
  return n > 0 ? cc_layout(n).total : 0;
}

extern "C" long long oai_components_max(const int* dims, int connectivity) {
  const long long n = voxel_count(dims);
  if (n <= 0 || !conn_rank(connectivity)) return 0;
  // One voxel picked per component gives pairwise non-adjacent voxels.  26: at most one per 2x2x2 cell, whose voxels
  // are mutually adjacent.  6 and 18: a serpentine path visits every voxel through 6-adjacent steps, and no two
  // consecutive voxels on it can both be picked.
  if (connectivity == 26)
    return static_cast<long long>((dims[0] + 1) / 2) * ((dims[1] + 1) / 2) * ((dims[2] + 1) / 2);
  return (n + 1) / 2;
}

extern "C" int oai_connected_components(const uint8_t* mask, const int* dims, int connectivity, int* labels,
                                        int* sizes, long long* count, void* workspace, size_t workspace_bytes,
                                        void* stream) {
  OAI_REQUIRE(conn_rank(connectivity), "connected_components: connectivity must be 6, 18 or 26 (got %d)",
              connectivity);
  if (int rc = check_dims("connected_components", dims)) return rc;
  OAI_REQUIRE(mask && labels && sizes && count && workspace, "connected_components: null pointer");
  const long long n = voxel_count(dims);
  const CcLayout l = cc_layout(n);
  OAI_REQUIRE(workspace_bytes >= l.total && (reinterpret_cast<uintptr_t>(workspace) & 255) == 0,
              "connected_components: workspace of %zu bytes (256-byte aligned) required, got %zu", l.total,
              workspace_bytes);
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  char* ws = static_cast<char*>(workspace);
  uint32_t* rank = reinterpret_cast<uint32_t*>(ws + l.rank);
  uint32_t* sums = reinterpret_cast<uint32_t*>(ws + l.sums);
  CcGeom g;
  g.D = dims[0];
  g.H = dims[1];
  g.W = dims[2];
  g.rank = conn_rank(connectivity);
  g.nbx = (g.W + kBX - 1) / kBX;
  g.nby = (g.H + kBY - 1) / kBY;
  const long long bricks = static_cast<long long>(g.nbx) * g.nby * ((g.D + kBZ - 1) / kBZ);
  const size_t max_n = static_cast<size_t>(oai_components_max(dims, connectivity));
  if (int rc = check_cuda(cudaMemsetAsync(sizes, 0, max_n * sizeof(int), st), "connected_components: clear sizes"))
    return rc;
  cc_local_kernel<<<static_cast<unsigned>(bricks), kBrick, 0, st>>>(mask, labels, g);
  if (int rc = launched("cc_local_kernel")) return rc;
  cc_merge_kernel<<<static_cast<unsigned>(bricks), kBrick, 0, st>>>(mask, labels, g);
  if (int rc = launched("cc_merge_kernel")) return rc;
  const int ni = static_cast<int>(n);
  cc_flatten_kernel<<<grid_for(n, 256), 256, 0, st>>>(labels, rank, ni);
  if (int rc = launched("cc_flatten_kernel")) return rc;
  if (int rc = exclusive_scan(rank, n, sums, st)) return rc;
  cc_relabel_kernel<<<grid_for(n, 256), 256, 0, st>>>(labels, rank, ni, sizes, sums + scan_blocks(n), count);
  return launched("cc_relabel_kernel");
}

extern "C" int oai_keep_components(const int* labels, const int* sizes, const long long* count, const int* dims,
                                   int min_voxels, uint8_t* keep_mask, float* values, void* stream) {
  if (int rc = check_dims("keep_components", dims)) return rc;
  OAI_REQUIRE(labels && sizes && count, "keep_components: null pointer");
  OAI_REQUIRE(keep_mask || values, "keep_components: neither a keep mask nor values to write");
  const long long n = voxel_count(dims);
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  cc_keep_kernel<<<grid_for(n, kKeepThreads), kKeepThreads, 0, st>>>(labels, sizes, count, n, min_voxels, keep_mask,
                                                                      values);
  return launched("cc_keep_kernel");
}
