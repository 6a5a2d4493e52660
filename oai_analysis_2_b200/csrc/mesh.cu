// Iso-surface extraction of the atlas-space probability maps straight from HBM (SURVEY §8f-2).
//
// Replaces skimage.measure.marching_cubes(level=0.5, spacing, step_size=1, gradient_direction="ascent") of
// oai_analysis/mesh_processing.py:325-340 (get_mesh) and the vtkPolyDataConnectivityFilter region filter of
// mesh_processing.py:102-146 (get_vtk_mesh: regions with more than 3000 cells are kept).
//
//   * one vertex per lattice edge the iso-level crosses (linear interpolation, shared between the cells around it);
//   * the polygon table is GENERATED at first use: for each of the 256 corner-sign patterns and each resolution of the
//     pattern's ambiguous faces, the crossed edges are chained face by face into closed oriented loops and fanned;
//   * ambiguous faces (two diagonal corners inside) are resolved per cell with the asymptotic decider (bilinear saddle
//     value against the level, evaluated in fp64), which depends only on the face's four values, so neighbouring cells
//     agree and the surface is watertight;
//   * regions: lock-free union-find over the vertices, faces counted per root, small regions dropped, vertices compacted.
//
// Data flow (all device side, caller-owned workspace): classify (per voxel: crossed owned edges, per cell: pattern +
// face bits + triangle count) -> two exclusive scans -> vertex emit -> face emit.
#include "../../include/oai_b200.h"
#include "api_common.h"
#include "scan_union_find.cuh"

#include <algorithm>
#include <cstdint>
#include <cstring>
#include <mutex>
#include <vector>

namespace oai {
namespace {

// ------------------------------------------------------------------------------------------------ cube topology
// corner c = dx + 2 dy + 4 dz; edge e = 4 * axis + (u + 2 v), (u, v) = offsets along the two other axes in increasing
// axis order; the edge runs from its base corner to base + 1 along `axis`
constexpr int kMaxTris = 10;
constexpr int kEntryBytes = 32;   // count + 10 x 3 edge ids (+ 1 pad)

struct Topology {
  int edge_c0[12], edge_c1[12];
  int face_corner[6][4];     // cyclic order
  int face_edge[6][4];       // edge between cyclic corner i and i+1
  int face_axis[6], face_side[6];
};

int corner_of(int x, int y, int z) { return x + 2 * y + 4 * z; }

Topology make_topology() {
  Topology t;
  for (int e = 0; e < 12; ++e) {
    const int axis = e / 4, uv = e % 4;
    int o[2], k = 0;
    for (int a = 0; a < 3; ++a) if (a != axis) o[k++] = a;
    int b[3] = {0, 0, 0};
    b[o[0]] = uv & 1;
    b[o[1]] = uv >> 1;
    t.edge_c0[e] = corner_of(b[0], b[1], b[2]);
    t.edge_c1[e] = t.edge_c0[e] + (1 << axis);
  }
  int f = 0;
  for (int axis = 0; axis < 3; ++axis) {
    int o[2], k = 0;
    for (int a = 0; a < 3; ++a) if (a != axis) o[k++] = a;
    for (int side = 0; side < 2; ++side, ++f) {
      const int uv[4][2] = {{0, 0}, {1, 0}, {1, 1}, {0, 1}};
      for (int i = 0; i < 4; ++i) {
        int p[3];
        p[axis] = side; p[o[0]] = uv[i][0]; p[o[1]] = uv[i][1];
        t.face_corner[f][i] = corner_of(p[0], p[1], p[2]);
      }
      t.face_axis[f] = axis;
      t.face_side[f] = side;
    }
  }
  for (f = 0; f < 6; ++f)
    for (int i = 0; i < 4; ++i) {
      const int a = t.face_corner[f][i], b = t.face_corner[f][(i + 1) % 4];
      t.face_edge[f][i] = -1;
      for (int e = 0; e < 12; ++e)
        if ((t.edge_c0[e] == a && t.edge_c1[e] == b) || (t.edge_c0[e] == b && t.edge_c1[e] == a)) t.face_edge[f][i] = e;
    }
  return t;
}

bool face_ambiguous(const Topology& t, int mask, int f) {
  int s[4];
  for (int i = 0; i < 4; ++i) s[i] = (mask >> t.face_corner[f][i]) & 1;
  return s[0] == s[2] && s[1] == s[3] && s[0] != s[1];
}

// Triangles (edge-id triples) of one (pattern, face-resolution) pair.  Integer geometry: coordinates doubled so edge
// midpoints are integral.  Orientation: loop normals point from the inside corners outwards ("descent").
int cell_triangles(const Topology& t, int mask, int bits, uint8_t* tris) {
  int nxt[12];
  for (int e = 0; e < 12; ++e) nxt[e] = -1;
  auto mid2 = [&](int e, int p[3]) {
    for (int a = 0; a < 3; ++a) p[a] = ((t.edge_c0[e] >> a) & 1) + ((t.edge_c1[e] >> a) & 1);
  };
  for (int f = 0; f < 6; ++f) {
    int s[4], k = 0;
    for (int i = 0; i < 4; ++i) { s[i] = (mask >> t.face_corner[f][i]) & 1; k += s[i]; }
    if (k == 0 || k == 4) continue;
    struct Seg { int ea, eb, ref; bool ref_inside; } segs[2];
    int nseg = 0;
    const int* e = t.face_edge[f];
    if (k == 1 || k == 3) {
      int odd = 0;
      for (int i = 0; i < 4; ++i) if (s[i] == (k == 1 ? 1 : 0)) odd = i;
      segs[nseg++] = Seg{e[(odd + 3) % 4], e[odd], t.face_corner[f][odd], k == 1};
    } else if (s[0] == s[1] || s[1] == s[2]) {
      int i0 = 0;
      for (int i = 0; i < 4; ++i) if (s[i] && s[(i + 1) % 4]) i0 = i;
      segs[nseg++] = Seg{e[(i0 + 3) % 4], e[(i0 + 1) % 4], t.face_corner[f][i0], true};
    } else {
      const bool cut_inside = !((bits >> f) & 1);
      for (int i = 0; i < 4; ++i)
        if ((s[i] != 0) == cut_inside) segs[nseg++] = Seg{e[(i + 3) % 4], e[i], t.face_corner[f][i], cut_inside};
    }
    for (int q = 0; q < nseg; ++q) {
      int a[3], b[3], p[3];
      mid2(segs[q].ea, a);
      mid2(segs[q].eb, b);
      for (int ax = 0; ax < 3; ++ax) p[ax] = 2 * ((segs[q].ref >> ax) & 1);
      const int u[3] = {b[0] - a[0], b[1] - a[1], b[2] - a[2]}, v[3] = {p[0] - a[0], p[1] - a[1], p[2] - a[2]};
      const int cr[3] = {u[1] * v[2] - u[2] * v[1], u[2] * v[0] - u[0] * v[2], u[0] * v[1] - u[1] * v[0]};
      const int left = cr[t.face_axis[f]] * (t.face_side[f] ? 1 : -1);   // > 0: ref corner left of a -> b from outside
      const bool forward = (left < 0) == segs[q].ref_inside;             // inside region on the right
      const int src = forward ? segs[q].ea : segs[q].eb, dst = forward ? segs[q].eb : segs[q].ea;
      nxt[src] = dst;
    }
  }
  auto coplanar = [&](int e0, int e1) {
    for (int f = 0; f < 6; ++f) {
      bool h0 = false, h1 = false;
      for (int i = 0; i < 4; ++i) { h0 |= t.face_edge[f][i] == e0; h1 |= t.face_edge[f][i] == e1; }
      if (h0 && h1) return true;
    }
    return false;
  };
  bool seen[12] = {false};
  int ntri = 0;
  for (int start = 0; start < 12; ++start) {
    if (nxt[start] < 0 || seen[start]) continue;
    int loop[12], n = 0;
    for (int cur = start; !seen[cur]; cur = nxt[cur]) { seen[cur] = true; loop[n++] = cur; }
    int best = 0;
    for (int apex = 0; apex < n; ++apex) {   // first apex whose fan has no diagonal lying in a cube face
      bool bad = false;
      for (int k2 = 2; k2 < n - 1; ++k2) bad |= coplanar(loop[apex], loop[(apex + k2) % n]);
      if (!bad) { best = apex; break; }
    }
    for (int i = 1; i < n - 1; ++i) {
      tris[3 * ntri] = static_cast<uint8_t>(loop[best]);
      tris[3 * ntri + 1] = static_cast<uint8_t>(loop[(best + i) % n]);
      tris[3 * ntri + 2] = static_cast<uint8_t>(loop[(best + i + 1) % n]);
      ++ntri;
    }
  }
  return ntri;
}

// table[(mask << 6 | bits)] = {count, 30 edge ids, pad}
const std::vector<uint8_t>& host_table() {
  static std::vector<uint8_t> tab;
  static std::once_flag once;
  std::call_once(once, [] {
    const Topology t = make_topology();
    tab.assign(256 * 64 * kEntryBytes, 0);
    for (int mask = 0; mask < 256; ++mask)
      for (int bits = 0; bits < 64; ++bits) {
        int eff = 0;   // only ambiguous faces' bits matter
        for (int f = 0; f < 6; ++f) if (face_ambiguous(t, mask, f) && ((bits >> f) & 1)) eff |= 1 << f;
        uint8_t* ent = tab.data() + static_cast<size_t>(mask * 64 + bits) * kEntryBytes;
        if (eff != bits) {   // alias of the canonical entry (filled earlier: eff < bits)
          memcpy(ent, tab.data() + static_cast<size_t>(mask * 64 + eff) * kEntryBytes, kEntryBytes);
          continue;
        }
        ent[0] = static_cast<uint8_t>(cell_triangles(t, mask, bits, ent + 1));
      }
  });
  return tab;
}

struct DevTable {
  uint8_t* table = nullptr;
};

int device_table(const uint8_t** out) {
  static DevTable dev[64];
  static std::mutex mu;
  int d = 0;
  cudaGetDevice(&d);
  OAI_REQUIRE(d >= 0 && d < 64, "marching cubes: device index %d", d);
  std::lock_guard<std::mutex> lock(mu);
  if (!dev[d].table) {
    const std::vector<uint8_t>& t = host_table();
    if (int rc = check_cuda(cudaMalloc(&dev[d].table, t.size()), "marching cubes: table cudaMalloc")) return rc;
    if (int rc = check_cuda(cudaMemcpy(dev[d].table, t.data(), t.size(), cudaMemcpyHostToDevice), "marching cubes: table copy"))
      return rc;
  }
  *out = dev[d].table;
  return 0;
}

// ------------------------------------------------------------------------------------------------ device helpers
struct McParams {
  const float* vol;     // [D][H][W]
  int D, H, W;
  float level;
  const uint8_t* table;
  uint32_t* vword;      // per voxel: vertex base (29 bits, after the scan) | crossed owned edges x,y,z << 29
  uint32_t* vcnt;       // per voxel: crossed owned edges (scan input) / exclusive scan (vertex base)
  uint32_t* tcnt;       // per voxel (= cell at its low corner): triangles (scan input) / exclusive scan (face base)
  uint16_t* cinfo;      // per cell: corner mask | face bits << 8
  double sx, sy, sz;
  int ascent;
  float* verts;
  int* faces;
};

__device__ __forceinline__ bool inside(float v, float level) { return v > level; }

__global__ void __launch_bounds__(256) mc_classify_kernel(const McParams p) {
  const long long nvox = static_cast<long long>(p.D) * p.H * p.W;
  for (long long i = blockIdx.x * static_cast<long long>(blockDim.x) + threadIdx.x; i < nvox;
       i += static_cast<long long>(gridDim.x) * blockDim.x) {
    const int x = static_cast<int>(i % p.W), y = static_cast<int>((i / p.W) % p.H), z = static_cast<int>(i / (static_cast<long long>(p.W) * p.H));
    const bool hx = x + 1 < p.W, hy = y + 1 < p.H, hz = z + 1 < p.D;
    float v[8];
#pragma unroll
    for (int c = 0; c < 8; ++c) {
      const int dx = c & 1, dy = (c >> 1) & 1, dz = c >> 2;
      const bool ok = (!dx || hx) && (!dy || hy) && (!dz || hz);
      v[c] = ok ? __ldg(p.vol + i + dx + static_cast<long long>(dy) * p.W + static_cast<long long>(dz) * p.W * p.H) : 0.f;
    }
    const bool in0 = inside(v[0], p.level);
    uint32_t flags = 0;
    if (hx && inside(v[1], p.level) != in0) flags |= 1u;
    if (hy && inside(v[2], p.level) != in0) flags |= 2u;
    if (hz && inside(v[4], p.level) != in0) flags |= 4u;
    uint32_t ntri = 0, info = 0;
    if (hx && hy && hz) {
      uint32_t mask = 0;
#pragma unroll
      for (int c = 0; c < 8; ++c) mask |= (inside(v[c], p.level) ? 1u : 0u) << c;
      if (mask != 0 && mask != 255) {
        uint32_t bits = 0;
        // faces in table order: (axis 0: x = 0, x = 1), (axis 1), (axis 2); cyclic corners (0,0),(1,0),(1,1),(0,1) in the
        // two other axes
#pragma unroll
        for (int f = 0; f < 6; ++f) {
          const int axis = f >> 1, side = f & 1;
          const int o0 = axis == 0 ? 1 : 0, o1 = axis == 2 ? 1 : 2;
          int cc[4];
#pragma unroll
          for (int q = 0; q < 4; ++q) {
            const int u = (q == 1 || q == 2) ? 1 : 0, w = q >> 1;
            cc[q] = (side << axis) | (u << o0) | (w << o1);
          }
          const bool s0 = (mask >> cc[0]) & 1, s1 = (mask >> cc[1]) & 1, s2 = (mask >> cc[2]) & 1, s3 = (mask >> cc[3]) & 1;
          if (s0 == s2 && s1 == s3 && s0 != s1) {
            // asymptotic decider: bilinear saddle value (a c - b d) / (a + c - b - d) relative to the level, in fp64
            const double a = static_cast<double>(v[cc[0]]) - p.level, b = static_cast<double>(v[cc[1]]) - p.level,
                         c = static_cast<double>(v[cc[2]]) - p.level, d = static_cast<double>(v[cc[3]]) - p.level;
            if ((a * c - b * d) / (a + c - b - d) > 0.0) bits |= 1u << f;
          }
        }
        info = mask | (bits << 8);
        ntri = p.table[(mask * 64 + bits) * kEntryBytes];
      }
    }
    p.vword[i] = flags << 29;
    p.vcnt[i] = __popc(flags);
    p.tcnt[i] = ntri;
    p.cinfo[i] = static_cast<uint16_t>(info);
  }
}

__global__ void __launch_bounds__(256) mc_vertex_kernel(const McParams p) {
  const long long nvox = static_cast<long long>(p.D) * p.H * p.W;
  for (long long i = blockIdx.x * static_cast<long long>(blockDim.x) + threadIdx.x; i < nvox;
       i += static_cast<long long>(gridDim.x) * blockDim.x) {
    const uint32_t flags = p.vword[i] >> 29;
    const uint32_t base = p.vcnt[i];
    p.vword[i] = (flags << 29) | base;
    if (!flags) continue;
    const int x = static_cast<int>(i % p.W), y = static_cast<int>((i / p.W) % p.H), z = static_cast<int>(i / (static_cast<long long>(p.W) * p.H));
    const double a = static_cast<double>(__ldg(p.vol + i)) - p.level;
    uint32_t k = base;
    const long long step[3] = {1, p.W, static_cast<long long>(p.W) * p.H};
#pragma unroll
    for (int axis = 0; axis < 3; ++axis) {
      if (!((flags >> axis) & 1u)) continue;
      const double b = static_cast<double>(__ldg(p.vol + i + step[axis])) - p.level;
      const double t = a / (a - b);
      double pos[3] = {static_cast<double>(x), static_cast<double>(y), static_cast<double>(z)};
      pos[axis] += t;
      p.verts[3 * static_cast<size_t>(k)] = static_cast<float>(pos[0] * p.sx);
      p.verts[3 * static_cast<size_t>(k) + 1] = static_cast<float>(pos[1] * p.sy);
      p.verts[3 * static_cast<size_t>(k) + 2] = static_cast<float>(pos[2] * p.sz);
      ++k;
    }
  }
}

__global__ void __launch_bounds__(256) mc_face_kernel(const McParams p) {
  const long long nvox = static_cast<long long>(p.D) * p.H * p.W;
  for (long long i = blockIdx.x * static_cast<long long>(blockDim.x) + threadIdx.x; i < nvox;
       i += static_cast<long long>(gridDim.x) * blockDim.x) {
    const uint32_t info = p.cinfo[i];
    if (!info) continue;
    const uint8_t* ent = p.table + ((info & 255u) * 64 + (info >> 8)) * kEntryBytes;
    const int ntri = ent[0];
    size_t out = static_cast<size_t>(p.tcnt[i]) * 3;
    for (int t = 0; t < ntri; ++t) {
      int ids[3];
#pragma unroll
      for (int k = 0; k < 3; ++k) {
        const int e = ent[1 + 3 * t + k];
        const int axis = e >> 2, uv = e & 3;
        const int o0 = axis == 0 ? 1 : 0, o1 = axis == 2 ? 1 : 2;
        int off[3] = {0, 0, 0};
        off[o0] = uv & 1;
        off[o1] = uv >> 1;
        const long long owner = i + off[0] + static_cast<long long>(off[1]) * p.W + static_cast<long long>(off[2]) * p.W * p.H;
        const uint32_t w = p.vword[owner];
        ids[k] = static_cast<int>((w & 0x1FFFFFFFu) + __popc((w >> 29) & ((1u << axis) - 1u)));
      }
      if (p.ascent) { const int tmp = ids[0]; ids[0] = ids[2]; ids[2] = tmp; }
      p.faces[out] = ids[0]; p.faces[out + 1] = ids[1]; p.faces[out + 2] = ids[2];
      out += 3;
    }
  }
}

size_t align_up(size_t v) { return (v + 255) & ~size_t(255); }

struct McLayout {
  size_t vword, vcnt, tcnt, cinfo, sums_v, sums_t, total;
};

McLayout mc_layout(long long nvox) {
  McLayout l;
  size_t off = 0;
  l.vword = off; off += align_up(nvox * 4);
  l.vcnt = off; off += align_up(nvox * 4);
  l.tcnt = off; off += align_up(nvox * 4);
  l.cinfo = off; off += align_up(nvox * 2);
  l.sums_v = off; off += align_up((scan_blocks(nvox) + 1) * 4);
  l.sums_t = off; off += align_up((scan_blocks(nvox) + 1) * 4);
  l.total = off;
  return l;
}

int grid_for_n(long long n) {
  long long b = (n + 255) / 256;
  const long long cap = static_cast<long long>(num_sms()) * 16;
  return static_cast<int>(b < cap ? (b < 1 ? 1 : b) : cap);
}

// ------------------------------------------------------------------------------------------------ regions (union-find)
__global__ void uf_init_kernel(int* parent, int* count, int n) {
  for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < n; i += gridDim.x * blockDim.x) { parent[i] = i; count[i] = 0; }
}
__global__ void uf_union_kernel(int* parent, const int* __restrict__ faces, int nf) {
  for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < nf; i += gridDim.x * blockDim.x) {
    uf_union(parent, faces[3 * i], faces[3 * i + 1]);
    uf_union(parent, faces[3 * i + 1], faces[3 * i + 2]);
  }
}
__global__ void uf_count_kernel(int* parent, int* count, const int* __restrict__ faces, int nf) {
  for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < nf; i += gridDim.x * blockDim.x)
    atomicAdd(&count[uf_find(parent, faces[3 * i])], 1);
}
// keep[f] = 1 if the face's region has more than min_cells faces; used[v] = 1 for the vertices of kept faces
__global__ void uf_mark_kernel(int* parent, const int* __restrict__ count, const int* __restrict__ faces, int nf,
                               int min_cells, uint32_t* keep, uint32_t* used) {
  for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < nf; i += gridDim.x * blockDim.x) {
    const bool k = count[uf_find(parent, faces[3 * i])] > min_cells;
    keep[i] = k ? 1u : 0u;
    if (k) { used[faces[3 * i]] = 1u; used[faces[3 * i + 1]] = 1u; used[faces[3 * i + 2]] = 1u; }
  }
}
__global__ void zero_u32_kernel(uint32_t* p, long long n) {
  for (long long i = blockIdx.x * static_cast<long long>(blockDim.x) + threadIdx.x; i < n; i += static_cast<long long>(gridDim.x) * blockDim.x) p[i] = 0;
}
// flags were replaced by their exclusive scans; an element is kept iff scan[i+1] != scan[i] (last one: total != scan)
__global__ void compact_kernel(const float* __restrict__ verts, int nv, const int* __restrict__ faces, int nf,
                               const uint32_t* __restrict__ vscan, const uint32_t* __restrict__ vtotal,
                               const uint32_t* __restrict__ fscan, const uint32_t* __restrict__ ftotal,
                               float* out_verts, int* out_faces) {
  const int n = nv > nf ? nv : nf;
  for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < n; i += gridDim.x * blockDim.x) {
    if (i < nv) {
      const uint32_t nx = i + 1 < nv ? vscan[i + 1] : *vtotal;
      if (nx != vscan[i]) {
        const size_t o = 3 * static_cast<size_t>(vscan[i]);
        out_verts[o] = verts[3 * static_cast<size_t>(i)];
        out_verts[o + 1] = verts[3 * static_cast<size_t>(i) + 1];
        out_verts[o + 2] = verts[3 * static_cast<size_t>(i) + 2];
      }
    }
    if (i < nf) {
      const uint32_t nx = i + 1 < nf ? fscan[i + 1] : *ftotal;
      if (nx != fscan[i]) {
        const size_t o = 3 * static_cast<size_t>(fscan[i]);
        out_faces[o] = static_cast<int>(vscan[faces[3 * i]]);
        out_faces[o + 1] = static_cast<int>(vscan[faces[3 * i + 1]]);
        out_faces[o + 2] = static_cast<int>(vscan[faces[3 * i + 2]]);
      }
    }
  }
}

}  // namespace
}  // namespace oai

using namespace oai;

extern "C" int oai_mc_table(uint8_t* table, size_t bytes) {
  const std::vector<uint8_t>& t = host_table();
  OAI_REQUIRE(table != nullptr && bytes >= t.size(), "mc_table: need %zu bytes", t.size());
  memcpy(table, t.data(), t.size());
  return 0;
}

extern "C" size_t oai_mc_workspace_bytes(const int* dims) {
  if (!dims || dims[0] < 1 || dims[1] < 1 || dims[2] < 1) return 0;
  return mc_layout(static_cast<long long>(dims[0]) * dims[1] * dims[2]).total;
}

static int mc_params(const float* vol, const int* dims, float level, void* ws, size_t ws_bytes, McParams* p,
                     McLayout* lay) {
  OAI_REQUIRE(vol && dims && ws, "marching cubes: null pointer");
  OAI_REQUIRE(dims[0] >= 2 && dims[1] >= 2 && dims[2] >= 2, "marching cubes: every axis needs at least 2 samples");
  const long long nvox = static_cast<long long>(dims[0]) * dims[1] * dims[2];
  OAI_REQUIRE(3 * nvox < (1ll << 29), "marching cubes: volume too large for 29-bit vertex ids");
  *lay = mc_layout(nvox);
  OAI_REQUIRE(ws_bytes >= lay->total && (reinterpret_cast<uintptr_t>(ws) & 255) == 0,
              "marching cubes: workspace needs %zu bytes, 256-byte aligned", lay->total);
  uint8_t* w = static_cast<uint8_t*>(ws);
  memset(p, 0, sizeof(*p));
  p->vol = vol; p->D = dims[0]; p->H = dims[1]; p->W = dims[2]; p->level = level;
  if (device_table(&p->table)) return 1;
  p->vword = reinterpret_cast<uint32_t*>(w + lay->vword);
  p->vcnt = reinterpret_cast<uint32_t*>(w + lay->vcnt);
  p->tcnt = reinterpret_cast<uint32_t*>(w + lay->tcnt);
  p->cinfo = reinterpret_cast<uint16_t*>(w + lay->cinfo);
  return 0;
}

extern "C" int oai_mc_count(const float* vol, const int* dims, float level, void* workspace, size_t workspace_bytes,
                            long long* counts_host, void* stream) {
  OAI_REQUIRE(counts_host != nullptr, "mc_count: null pointer");
  McParams p;
  McLayout lay;
  if (mc_params(vol, dims, level, workspace, workspace_bytes, &p, &lay)) return 1;
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  const long long nvox = static_cast<long long>(p.D) * p.H * p.W;
  mc_classify_kernel<<<grid_for_n(nvox), 256, 0, st>>>(p);
  if (int rc = launched("mc_classify_kernel")) return rc;
  uint8_t* w = static_cast<uint8_t*>(workspace);
  uint32_t* sv = reinterpret_cast<uint32_t*>(w + lay.sums_v);
  uint32_t* stt = reinterpret_cast<uint32_t*>(w + lay.sums_t);
  if (exclusive_scan(p.vcnt, nvox, sv, st) || exclusive_scan(p.tcnt, nvox, stt, st)) return 1;
  uint32_t tot[2] = {0, 0};
  const int nb = scan_blocks(nvox);
  if (int rc = check_cuda(cudaMemcpyAsync(&tot[0], sv + nb, 4, cudaMemcpyDeviceToHost, st), "mc_count: copy")) return rc;
  if (int rc = check_cuda(cudaMemcpyAsync(&tot[1], stt + nb, 4, cudaMemcpyDeviceToHost, st), "mc_count: copy")) return rc;
  if (int rc = check_cuda(cudaStreamSynchronize(st), "mc_count: sync")) return rc;
  counts_host[0] = tot[0];
  counts_host[1] = tot[1];
  return 0;
}

extern "C" int oai_mc_emit(const float* vol, const int* dims, float level, const double* spacing_xyz, int ascent,
                           void* workspace, size_t workspace_bytes, float* verts, int* faces, void* stream) {
  OAI_REQUIRE(spacing_xyz && verts && faces, "mc_emit: null pointer");
  McParams p;
  McLayout lay;
  if (mc_params(vol, dims, level, workspace, workspace_bytes, &p, &lay)) return 1;
  p.sx = spacing_xyz[0]; p.sy = spacing_xyz[1]; p.sz = spacing_xyz[2];
  p.ascent = ascent; p.verts = verts; p.faces = faces;
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  const long long nvox = static_cast<long long>(p.D) * p.H * p.W;
  mc_vertex_kernel<<<grid_for_n(nvox), 256, 0, st>>>(p);
  if (int rc = launched("mc_vertex_kernel")) return rc;
  mc_face_kernel<<<grid_for_n(nvox), 256, 0, st>>>(p);
  return launched("mc_face_kernel");
}

extern "C" size_t oai_mesh_regions_workspace_bytes(long long n_verts, long long n_faces) {
  if (n_verts < 0 || n_faces < 0) return 0;
  return align_up(n_verts * 4) * 3 + align_up(n_faces * 4) + align_up((scan_blocks(n_verts) + 1) * 4) +
         align_up((scan_blocks(n_faces) + 1) * 4);
}

extern "C" int oai_mesh_keep_large_regions(const float* verts, long long n_verts, const int* faces, long long n_faces,
                                           int min_cells, void* workspace, size_t workspace_bytes, float* out_verts,
                                           int* out_faces, long long* counts_host, void* stream) {
  OAI_REQUIRE(counts_host != nullptr, "keep_large_regions: null pointer");
  counts_host[0] = counts_host[1] = 0;
  if (n_verts == 0 || n_faces == 0) return 0;
  OAI_REQUIRE(verts && faces && workspace && out_verts && out_faces, "keep_large_regions: null pointer");
  OAI_REQUIRE(n_verts < (1ll << 31) && n_faces < (1ll << 31), "keep_large_regions: mesh too large");
  OAI_REQUIRE(workspace_bytes >= oai_mesh_regions_workspace_bytes(n_verts, n_faces) &&
                  (reinterpret_cast<uintptr_t>(workspace) & 255) == 0,
              "keep_large_regions: workspace needs %zu bytes, 256-byte aligned",
              oai_mesh_regions_workspace_bytes(n_verts, n_faces));
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  const int nv = static_cast<int>(n_verts), nf = static_cast<int>(n_faces);
  uint8_t* w = static_cast<uint8_t*>(workspace);
  int* parent = reinterpret_cast<int*>(w); w += align_up(n_verts * 4);
  int* count = reinterpret_cast<int*>(w); w += align_up(n_verts * 4);
  uint32_t* used = reinterpret_cast<uint32_t*>(w); w += align_up(n_verts * 4);
  uint32_t* keep = reinterpret_cast<uint32_t*>(w); w += align_up(n_faces * 4);
  uint32_t* sums_v = reinterpret_cast<uint32_t*>(w); w += align_up((scan_blocks(n_verts) + 1) * 4);
  uint32_t* sums_f = reinterpret_cast<uint32_t*>(w);
  uf_init_kernel<<<grid_for_n(nv), 256, 0, st>>>(parent, count, nv);
  if (int rc = launched("uf_init_kernel")) return rc;
  zero_u32_kernel<<<grid_for_n(nv), 256, 0, st>>>(used, nv);
  if (int rc = launched("zero_u32_kernel")) return rc;
  uf_union_kernel<<<grid_for_n(nf), 256, 0, st>>>(parent, faces, nf);
  if (int rc = launched("uf_union_kernel")) return rc;
  uf_count_kernel<<<grid_for_n(nf), 256, 0, st>>>(parent, count, faces, nf);
  if (int rc = launched("uf_count_kernel")) return rc;
  uf_mark_kernel<<<grid_for_n(nf), 256, 0, st>>>(parent, count, faces, nf, min_cells, keep, used);
  if (int rc = launched("uf_mark_kernel")) return rc;
  if (exclusive_scan(used, nv, sums_v, st) || exclusive_scan(keep, nf, sums_f, st)) return 1;
  compact_kernel<<<grid_for_n(nv > nf ? nv : nf), 256, 0, st>>>(verts, nv, faces, nf, used, sums_v + scan_blocks(nv), keep,
                                                               sums_f + scan_blocks(nf), out_verts, out_faces);
  if (int rc = launched("compact_kernel")) return rc;
  uint32_t tot[2] = {0, 0};
  if (int rc = check_cuda(cudaMemcpyAsync(&tot[0], sums_v + scan_blocks(nv), 4, cudaMemcpyDeviceToHost, st), "regions: copy")) return rc;
  if (int rc = check_cuda(cudaMemcpyAsync(&tot[1], sums_f + scan_blocks(nf), 4, cudaMemcpyDeviceToHost, st), "regions: copy")) return rc;
  if (int rc = check_cuda(cudaStreamSynchronize(st), "regions: sync")) return rc;
  counts_host[0] = tot[0];
  counts_host[1] = tot[1];
  return 0;
}
