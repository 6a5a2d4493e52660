// Stage-level C ABI of the registration stage: icon_registration's register_pair on the GradICON knee model
// (reference call sites: oai_analysis/registration.py:20,25, oai_analysis/dask_processing.py:77,85; arithmetic in the
// un-vendored icon_registration==1.1.2: pretrained_models.OAI_knees_gradICON_model, networks.tallUNet2,
// network_wrappers.{TwoStepRegistration, DownsampleRegistration, FunctionFromVectorField}, itk_wrapper.register_pair)
// behind three calls --
//   oai_reg_create   : takes the regis_net state dict with icon's own key paths, derives the module tree from them
//                      (strict: every tensor must belong to a complete tallUNet2), folds BatchNorm(eval), packs the
//                      weights for the kernels of reg_kernels.cu and uploads them; plans the workspace;
//   oai_reg_forward  : trilinear resize of both images to the network shape, both directions batched through every
//                      tallUNet2 of the cascade, the TwoStep warps, the final composition on the identity map and
//                      (optionally) create_itk_transform's displacement fields;
//   oai_reg_destroy.
// Layer order, concatenation buffers, scratch and the cascade's intermediate images are laid out here; the caller owns
// the images, the outputs, the workspace and the stream.
#include "../../include/oai_b200.h"
#include "api_common.h"
#include "reg_kernels.cuh"

#include <nvtx3/nvToolsExt.h>

#include <algorithm>
#include <array>
#include <cmath>
#include <cstring>
#include <map>
#include <set>
#include <string>
#include <vector>

using namespace oai;

namespace {

// networks.tallUNet2: UNet2(num_layers=5, channels=[[2,16,32,64,256,512],[16,32,64,128,256]], dimension=3)
constexpr int kDown[6] = {2, 16, 32, 64, 256, 512};
constexpr int kUpOut[5] = {16, 32, 64, 128, 256};
constexpr int up_in(int d) { return kDown[d + 1] + (d + 1 < 5 ? kUpOut[d + 1] : 0); }
constexpr int cat_channels(int d) { return kUpOut[d] + kDown[d]; }
constexpr int kBatch = 2;   // direction 0 registers A -> B, direction 1 B -> A

struct Node {
  char kind;       // 'T' TwoStepRegistration(netPhi, netPsi) | 'D' DownsampleRegistration(net) | 'F' FFVF(tallUNet2)
  int a = -1, b = -1;
  int leaf = -1;
};

typedef std::map<std::string, const oai_tensor*> TensorGroup;

struct Parsed {
  std::vector<Node> nodes;
  int root = -1;
  std::vector<std::string> leaf_paths;
  std::vector<TensorGroup> leaf_tensors;
};

bool ends_with(const std::string& s, const char* tail) {
  const size_t n = strlen(tail);
  return s.size() >= n && s.compare(s.size() - n, n, tail) == 0;
}

std::string join(const std::vector<std::string>& v, const char* sep) {
  std::string s;
  for (size_t i = 0; i < v.size(); ++i) s += (i ? sep : "") + v[i];
  return s;
}

typedef std::vector<std::string> Path;

// The module tree from the UNets' key paths: 'netPhi' / 'netPsi' are the children of a TwoStepRegistration, 'net' is
// FunctionFromVectorField.net when it ends a path and DownsampleRegistration.net otherwise.
int build_tree(const Path& prefix, const std::vector<Path>& rel, const std::map<std::string, int>& leaf_of,
               Parsed* out, int* node) {
  const std::string where = prefix.empty() ? "<root>" : join(prefix, ".");
  if (rel.size() == 1 && rel[0].size() == 1 && rel[0][0] == "net") {
    Path p = prefix;
    p.push_back("net");
    Node n;
    n.kind = 'F';
    n.leaf = leaf_of.at(join(p, "."));
    out->nodes.push_back(n);
    *node = static_cast<int>(out->nodes.size()) - 1;
    return 0;
  }
  std::set<std::string> firsts;
  for (const Path& r : rel) {
    if (r.empty()) return fail("GradICON checkpoint: malformed module path under %s", where.c_str());
    firsts.insert(r[0]);
  }
  if (firsts.empty()) return fail("GradICON checkpoint: malformed module path under %s", where.c_str());
  auto tails = [&](const char* head) {
    std::vector<Path> t;
    for (const Path& r : rel)
      if (r[0] == head) t.emplace_back(r.begin() + 1, r.end());
    return t;
  };
  auto child = [&](const char* head, int* id) {
    Path p = prefix;
    p.push_back(head);
    return build_tree(p, tails(head), leaf_of, out, id);
  };
  if (firsts.size() == 1 && firsts.count("net")) {
    int c = -1;
    if (int rc = child("net", &c)) return rc;
    Node n;
    n.kind = 'D';
    n.a = c;
    out->nodes.push_back(n);
    *node = static_cast<int>(out->nodes.size()) - 1;
    return 0;
  }
  if (firsts.size() == 2 && firsts.count("netPhi") && firsts.count("netPsi")) {
    int a = -1, b = -1;
    if (int rc = child("netPhi", &a)) return rc;
    if (int rc = child("netPsi", &b)) return rc;
    Node n;
    n.kind = 'T';
    n.a = a;
    n.b = b;
    out->nodes.push_back(n);
    *node = static_cast<int>(out->nodes.size()) - 1;
    return 0;
  }
  std::vector<std::string> f(firsts.begin(), firsts.end());
  return fail("GradICON checkpoint: cannot interpret children [%s] under %s (expected netPhi+netPsi, or net)",
              join(f, ", ").c_str(), where.c_str());
}

struct Expected {
  std::string key;
  int ndim;
  long long shape[5];
};

std::vector<Expected> unet_template() {
  std::vector<Expected> t;
  auto add = [&](const std::string& k, std::initializer_list<long long> s) {
    Expected e;
    e.key = k;
    e.ndim = static_cast<int>(s.size());
    int i = 0;
    for (long long v : s) e.shape[i++] = v;
    t.push_back(e);
  };
  for (int d = 0; d < 5; ++d) {
    const std::string D = std::to_string(d);
    add("downConvs." + D + ".weight", {kDown[d + 1], kDown[d], 3, 3, 3});
    add("downConvs." + D + ".bias", {kDown[d + 1]});
    add("upConvs." + D + ".weight", {up_in(d), kUpOut[d], 4, 4, 4});
    add("upConvs." + D + ".bias", {kUpOut[d]});
    for (const char* k : {"weight", "bias", "running_mean", "running_var"})
      add("batchNorms." + D + "." + k, {kUpOut[d]});
  }
  add("lastConv.weight", {3, 18, 3, 3, 3});
  add("lastConv.bias", {3});
  return t;
}

// split_checkpoint + parse_tree + the per-UNet strict load of the Python loader, on the state dict's names and shapes.
int parse_state_dict(const oai_tensor* sd, int n, Parsed* out) {
  static const char* kHeads[] = {"downConvs.", "upConvs.", "batchNorms.", "lastConv."};
  std::map<std::string, TensorGroup> groups;
  int unknown = 0;
  std::string example;
  for (int i = 0; i < n; ++i) {
    if (!sd[i].name) return fail("GradICON state dict: entry %d has no name", i);
    std::string key = sd[i].name;
    if (key.rfind("regis_net.", 0) == 0) key = key.substr(10);
    if (ends_with(key, "identity_map")) continue;   // older icon versions saved these buffers
    size_t cut = std::string::npos;
    for (const char* h : kHeads) cut = std::min(cut, key.find(h));
    bool ok = cut != std::string::npos && cut > 0;
    std::string path;
    if (ok) {
      path = key.substr(0, cut);
      while (!path.empty() && path.back() == '.') path.pop_back();
      ok = !path.empty();
      size_t pos = 0;
      while (ok && pos <= path.size()) {
        const size_t dot = std::min(path.find('.', pos), path.size());
        const std::string tok = path.substr(pos, dot - pos);
        ok = tok == "netPhi" || tok == "netPsi" || tok == "net";
        pos = dot + 1;
      }
    }
    if (!ok) {
      if (!unknown++) example = sd[i].name;
      continue;
    }
    groups[path][key.substr(cut)] = &sd[i];
  }
  if (unknown)
    return fail("GradICON checkpoint has %d key(s) outside any tallUNet2 of the registration tree, e.g. %s", unknown,
                example.c_str());
  if (groups.empty()) return fail("GradICON checkpoint holds no tallUNet2 weights");
  std::map<std::string, int> leaf_of;
  std::vector<Path> paths;
  for (const auto& g : groups) {
    leaf_of[g.first] = static_cast<int>(out->leaf_paths.size());
    out->leaf_paths.push_back(g.first);
    out->leaf_tensors.push_back(g.second);
    Path p;
    size_t pos = 0;
    while (pos <= g.first.size()) {
      const size_t dot = std::min(g.first.find('.', pos), g.first.size());
      p.push_back(g.first.substr(pos, dot - pos));
      pos = dot + 1;
    }
    paths.push_back(p);
  }
  if (int rc = build_tree(Path(), paths, leaf_of, out, &out->root)) return rc;
  // every UNet complete, nothing stray, shapes as networks.tallUNet2 builds them
  const std::vector<Expected> tmpl = unet_template();
  for (size_t l = 0; l < out->leaf_paths.size(); ++l) {
    const TensorGroup& g = out->leaf_tensors[l];
    std::vector<std::string> missing, unexpected;
    for (const Expected& e : tmpl)
      if (!g.count(e.key)) missing.push_back(e.key);
    for (const auto& kv : g) {
      if (ends_with(kv.first, "num_batches_tracked")) continue;
      if (std::none_of(tmpl.begin(), tmpl.end(), [&](const Expected& e) { return e.key == kv.first; }))
        unexpected.push_back(kv.first);
    }
    if (!missing.empty() || !unexpected.empty())
      return fail("tallUNet2 %s: missing keys [%s], unexpected keys [%s]", out->leaf_paths[l].c_str(),
                  join(missing, ", ").c_str(), join(unexpected, ", ").c_str());
    for (const Expected& e : tmpl) {
      const oai_tensor* t = g.at(e.key);
      bool same = t->ndim == e.ndim;
      for (int a = 0; same && a < e.ndim; ++a) same = t->shape[a] == e.shape[a];
      if (!same)
        return fail("tallUNet2 %s: size mismatch for %s", out->leaf_paths[l].c_str(), e.key.c_str());
      if (!t->data) return fail("tallUNet2 %s: %s has no data", out->leaf_paths[l].c_str(), e.key.c_str());
    }
  }
  return 0;
}

std::string describe(const Parsed& p, int node) {
  const Node& n = p.nodes[node];
  if (n.kind == 'F') return "FFVF";
  if (n.kind == 'D') return "Down(" + describe(p, n.a) + ")";
  return "TwoStep(" + describe(p, n.a) + ", " + describe(p, n.b) + ")";
}

struct UNetWeights {
  float *dw[5], *db[5];            // down step d: [cin][27][cout], [cout]
  void* du[5];                     // weight blocks of the tcgen05 down step (levels with 16+ input channels)
  int dexp[5];
  float *uw[5], *ub[5];            // up step d: [cin][64][cout], [cout]
  float *bs[5], *bt[5];            // folded BatchNorm(eval): scale, shift
  uint4* uq[5];                    // split-fp16 B fragments of uw for the mma.sync path
  void* uu[5];                     // weight blocks of the tcgen05 path (levels with 16 - 128 output channels)
  int uexp[5];
  float *lw, *lb;                  // lastConv: [18][27][4] (3 channels padded to 4), [3]
};

struct FieldRef {
  size_t off;     // byte offset inside the arena part of the workspace: [kBatch][3][d][h][w] float32
  int dims[3];
  int leaf;
};

size_t align256(size_t v) { return (v + 255) & ~size_t(255); }
size_t voxels(const int* d) { return static_cast<size_t>(d[0]) * d[1] * d[2]; }

struct Geo {
  int lv[6][3];
  float* cat[5];
  float* x5;
};

// One pass over the cascade.  With dry = true nothing is launched: the pass only walks the allocation sequence (the
// workspace plan made at create time); a real pass repeats exactly the same sequence over the caller's workspace.
struct Ctx {
  const oai_reg_handle* h;
  cudaStream_t st;
  bool dry;
  char* arena;          // base of the bump-allocated part of the workspace
  size_t off = 0;
  void* scratch;        // split-K partial sums / hi-lo split layer input: one region, the kernels using it are
  size_t scratch_bytes; //   serialised by the stream
  size_t scratch_need = 0;
  std::map<std::array<int, 3>, Geo> geos;
  std::vector<FieldRef> fields;   // every leaf's displacement field, evaluation order
  size_t pair_off = 0;            // arena offset of the resized pair [A, B] (Slots::src)

  void* alloc(size_t bytes) {
    off = align256(off);
    void* p = arena + off;
    off += bytes;
    return p;
  }
  Geo& geo(const int* dims) {
    const std::array<int, 3> key = {dims[0], dims[1], dims[2]};
    auto it = geos.find(key);
    if (it != geos.end()) return it->second;
    Geo g;
    for (int a = 0; a < 3; ++a) g.lv[0][a] = dims[a];
    for (int l = 1; l < 6; ++l)
      for (int a = 0; a < 3; ++a) g.lv[l][a] = (g.lv[l - 1][a] + 1) / 2;
    for (int d = 0; d < 5; ++d)
      g.cat[d] = static_cast<float*>(alloc(sizeof(float) * kBatch * cat_channels(d) * voxels(g.lv[d])));
    g.x5 = static_cast<float*>(alloc(sizeof(float) * kBatch * kDown[5] * voxels(g.lv[5])));
    return geos.emplace(key, g).first->second;
  }
};

struct Field {
  float* p;   // [kBatch][3][d][h][w]
  int dims[3];
};

}  // namespace

struct oai_reg_handle {
  int device = 0;
  int dims[3] = {0, 0, 0};
  Parsed tree;                        // leaf_tensors point into the caller's state dict: cleared after create
  std::vector<UNetWeights> leaves;
  std::vector<void*> allocs;
  std::string description;
  size_t scratch_bytes = 0, arena_bytes = 0;
  std::vector<FieldRef> fields;       // application order of the whole cascade (first applied first)
  size_t pair_off = 0;                // arena offset of the resized pair [A, B] at the network shape
  bool forwarded = false;             // oai_reg_forward has run at least once (the loss reads its results)
};

namespace {

#define RC(expr)                \
  do {                          \
    if (int rc_ = (expr)) return rc_; \
  } while (0)

int copy_plane(Ctx& c, float* dst, const float* src, size_t n) {
  if (c.dry) return 0;
  return check_cuda(cudaMemcpyAsync(dst, src, n * sizeof(float), cudaMemcpyDeviceToDevice, c.st), "reg: image copy");
}

// networks.UNet2.forward on the batched pair: x = cat(src, tgt); five strided down steps with avg-pool residuals; five
// transposed-conv up steps with upsampled residuals, BatchNorm and skip concatenation; lastConv / 10.
int unet_forward(Ctx& c, const UNetWeights& w, const float* src, const float* tgt, const int* dims, float* u) {
  Geo& g = c.geo(dims);
  size_t vol[6];
  for (int l = 0; l < 6; ++l) vol[l] = voxels(g.lv[l]);
  for (int n = 0; n < kBatch; ++n) {
    float* slot = g.cat[0] + (static_cast<size_t>(n) * cat_channels(0) + kUpOut[0]) * vol[0];
    RC(copy_plane(c, slot, src + n * vol[0], vol[0]));
    RC(copy_plane(c, slot + vol[0], tgt + n * vol[0], vol[0]));
  }
  for (int d = 0; d < 5; ++d) {
    Conv3Params p{};
    p.in = g.cat[d] + kUpOut[d] * vol[d];
    p.in_nstride = static_cast<long long>(cat_channels(d) * vol[d]);
    p.in_cstride = static_cast<long long>(vol[d]);
    p.cin = kDown[d];
    p.Di = g.lv[d][0]; p.Hi = g.lv[d][1]; p.Wi = g.lv[d][2];
    p.w = w.dw[d]; p.bias = w.db[d];
    if (d < 4) {
      p.out = g.cat[d + 1] + kUpOut[d + 1] * vol[d + 1];
      p.out_nstride = static_cast<long long>(cat_channels(d + 1) * vol[d + 1]);
    } else {
      p.out = g.x5;
      p.out_nstride = static_cast<long long>(kDown[5] * vol[5]);
    }
    p.out_cstride = static_cast<long long>(vol[d + 1]);
    p.cout = kDown[d + 1]; p.cout_pad = kDown[d + 1];
    p.Do = g.lv[d + 1][0]; p.Ho = g.lv[d + 1][1]; p.Wo = g.lv[d + 1][2];
    p.N = kBatch; p.stride = 2; p.leaky_in = 1; p.residual = 1; p.out_scale = 1.0f;
    const size_t need = conv3_splitk_bytes(p);
    c.scratch_need = std::max(c.scratch_need, need);
    p.splitk_ws = need ? static_cast<float*>(c.scratch) : nullptr;
    p.splitk_bytes = need ? c.scratch_bytes : 0;
    p.wumma = w.du[d]; p.wexp = w.dexp[d];
    if (p.wumma && conv3_umma_eligible(p)) {
      c.scratch_need = std::max(c.scratch_need, conv3_umma_workspace(p));
      p.xsplit = c.scratch;
      p.xsplit_bytes = c.scratch_bytes;
    }
    if (!c.dry) RC(conv3_launch(p, c.st));
  }
  for (int d = 4; d >= 0; --d) {
    ConvT4Params p{};
    p.in = d == 4 ? g.x5 : g.cat[d + 1];
    p.in_nstride = static_cast<long long>((d == 4 ? kDown[5] : cat_channels(d + 1)) * vol[d + 1]);
    p.in_cstride = static_cast<long long>(vol[d + 1]);
    p.cin = up_in(d);
    p.Di = g.lv[d + 1][0]; p.Hi = g.lv[d + 1][1]; p.Wi = g.lv[d + 1][2];
    p.w = w.uw[d]; p.bias = w.ub[d]; p.bn_scale = w.bs[d]; p.bn_shift = w.bt[d];
    p.out = g.cat[d];
    p.out_nstride = static_cast<long long>(cat_channels(d) * vol[d]);
    p.out_cstride = static_cast<long long>(vol[d]);
    p.cout = kUpOut[d];
    p.Do = g.lv[d][0]; p.Ho = g.lv[d][1]; p.Wo = g.lv[d][2];
    p.N = kBatch;
    p.wpk = w.uq[d]; p.wexp = w.uexp[d]; p.wumma = w.uu[d];
    const int in_dims[3] = {p.Di, p.Hi, p.Wi};
    c.scratch_need = std::max(c.scratch_need, oai_reg_convt4_mma_workspace(p.cin, p.cout, in_dims, kBatch));
    p.xsplit = static_cast<uint32_t*>(c.scratch);
    p.xsplit_bytes = c.scratch_bytes;
    if (!c.dry) RC(convt4_launch(p, c.st));
  }
  Conv3Params p{};
  p.in = g.cat[0];
  p.in_nstride = static_cast<long long>(cat_channels(0) * vol[0]);
  p.in_cstride = static_cast<long long>(vol[0]);
  p.cin = cat_channels(0);
  p.Di = p.Do = dims[0]; p.Hi = p.Ho = dims[1]; p.Wi = p.Wo = dims[2];
  p.w = w.lw; p.bias = w.lb;
  p.out = u;
  p.out_nstride = static_cast<long long>(3 * vol[0]);
  p.out_cstride = static_cast<long long>(vol[0]);
  p.cout = 3; p.cout_pad = 4;
  p.N = kBatch; p.stride = 1; p.leaky_in = 0; p.residual = 0; p.out_scale = 0.1f;   // FunctionFromVectorField: net(x) / 10
  const size_t need = conv3_splitk_bytes(p);
  c.scratch_need = std::max(c.scratch_need, need);
  p.splitk_ws = need ? static_cast<float*>(c.scratch) : nullptr;
  p.splitk_bytes = need ? c.scratch_bytes : 0;
  if (!c.dry) RC(conv3_launch(p, c.st));
  return 0;
}

// c <- c + S(fields[k], c) over `fields` (application order) starting from the identity map of `grid`, then either the
// map itself or an image sampled at it (network_wrappers' closures; FunctionFromVectorField adds its field without
// interpolation when it is handed the identity map of its own shape).
int compose(Ctx& c, const std::vector<Field>& fields, int k, const int* grid, const float* img, const int* img_dims,
            float* phi_out, float* img_out) {
  if (fields.size() > 4) return fail("registration trees with more than four cascaded fields are not supported");
  if (grid[0] < 2 || grid[1] < 2 || grid[2] < 2) return fail("compose: grid axes must have at least 2 samples");
  ChainParams p{};
  p.D = grid[0]; p.H = grid[1]; p.W = grid[2];
  p.nfields = static_cast<int>(fields.size());
  for (int f = 0; f < p.nfields; ++f) {
    p.u[f] = fields[f].p + static_cast<size_t>(k) * 3 * voxels(fields[f].dims);
    p.ud[f] = fields[f].dims[0]; p.uh[f] = fields[f].dims[1]; p.uw[f] = fields[f].dims[2];
  }
  p.shortcut_first = !fields.empty() && fields[0].dims[0] == grid[0] && fields[0].dims[1] == grid[1] &&
                     fields[0].dims[2] == grid[2];
  p.img = img_out ? img : nullptr;
  if (img_out) { p.id = img_dims[0]; p.ih = img_dims[1]; p.iw = img_dims[2]; }
  p.phi_out = phi_out; p.img_out = img_out;
  if (c.dry) return 0;
  return chain_launch(p, c.st);
}

// One node on the batched pair (src -> tgt), both [kBatch][dims].  `out` receives the displacement fields of its
// leaves in APPLICATION order (first applied first): TwoStep(phi, psi) maps c -> phi(psi(c)).
int eval(Ctx& c, int node, const float* src, const float* tgt, const int* dims, std::vector<Field>* out) {
  const Node& n = c.h->tree.nodes[node];
  if (n.kind == 'F') {
    Field f;
    const size_t before = align256(c.off);
    f.p = static_cast<float*>(c.alloc(sizeof(float) * kBatch * 3 * voxels(dims)));
    for (int a = 0; a < 3; ++a) f.dims[a] = dims[a];
    FieldRef r;
    r.off = before;
    r.leaf = n.leaf;
    for (int a = 0; a < 3; ++a) r.dims[a] = dims[a];
    c.fields.push_back(r);
    RC(unet_forward(c, c.h->leaves[n.leaf], src, tgt, dims, f.p));
    out->assign(1, f);
    return 0;
  }
  if (n.kind == 'D') {   // DownsampleRegistration: F.avg_pool3d(x, 2, ceil_mode=True) on both images
    int lo[3];
    for (int a = 0; a < 3; ++a) lo[a] = (dims[a] + 1) / 2;
    float* lo_src = static_cast<float*>(c.alloc(sizeof(float) * kBatch * voxels(lo)));
    float* lo_tgt = static_cast<float*>(c.alloc(sizeof(float) * kBatch * voxels(lo)));
    if (!c.dry) {
      RC(avgpool2_ceil_launch(src, kBatch, dims[0], dims[1], dims[2], lo_src, c.st));
      RC(avgpool2_ceil_launch(tgt, kBatch, dims[0], dims[1], dims[2], lo_tgt, c.st));
    }
    return eval(c, n.a, lo_src, lo_tgt, lo, out);
  }
  std::vector<Field> f_phi, f_psi;
  RC(eval(c, n.a, src, tgt, dims, &f_phi));
  float* warped = static_cast<float*>(c.alloc(sizeof(float) * kBatch * voxels(dims)));   // as_function(image_A)(phi(identity_map))
  for (int k = 0; k < kBatch; ++k)
    RC(compose(c, f_phi, k, dims, src + k * voxels(dims), dims, nullptr, warped + k * voxels(dims)));
  RC(eval(c, n.b, warped, tgt, dims, &f_psi));
  *out = f_psi;
  out->insert(out->end(), f_phi.begin(), f_phi.end());
  return 0;
}

struct Slots {
  float *src, *tgt, *phi;
};

// the allocation sequence shared by the planning pass and the real pass
int run(Ctx& c, const float* A, const int* dims_A, const float* B, const int* dims_B, float* phi_AB, float* phi_BA,
        float* disp_AB, float* disp_BA, std::vector<FieldRef>* order) {
  const int* dims = c.h->dims;
  const size_t vol = voxels(dims);
  Slots s;
  s.src = static_cast<float*>(c.alloc(sizeof(float) * kBatch * vol));
  s.tgt = static_cast<float*>(c.alloc(sizeof(float) * kBatch * vol));
  s.phi = static_cast<float*>(c.alloc(sizeof(float) * kBatch * 3 * vol));
  c.pair_off = static_cast<size_t>(reinterpret_cast<char*>(s.src) - c.arena);
  if (!c.dry) {   // itk_wrapper.register_pair: F.interpolate(size=shape, mode="trilinear", align_corners=False)
    RC(resize_trilinear_launch(A, dims_A[0], dims_A[1], dims_A[2], s.src, dims[0], dims[1], dims[2], c.st));
    RC(resize_trilinear_launch(B, dims_B[0], dims_B[1], dims_B[2], s.src + vol, dims[0], dims[1], dims[2], c.st));
    RC(copy_plane(c, s.tgt, s.src + vol, vol));
    RC(copy_plane(c, s.tgt + vol, s.src, vol));
  }
  std::vector<Field> fields;
  RC(eval(c, c.h->tree.root, s.src, s.tgt, dims, &fields));
  if (fields.size() > 4) return fail("registration trees with more than four cascaded fields are not supported");
  if (order) {
    order->clear();
    for (const Field& f : fields) {
      const size_t off = static_cast<size_t>(reinterpret_cast<char*>(f.p) - c.arena);
      for (const FieldRef& r : c.fields)
        if (r.off == off) order->push_back(r);
    }
  }
  float* phi[2] = {phi_AB ? phi_AB : s.phi, phi_BA ? phi_BA : s.phi + 3 * vol};
  float* disp[2] = {disp_AB, disp_BA};
  for (int k = 0; k < kBatch; ++k) {
    if (c.dry) break;
    if (!(k == 0 ? (phi_AB || disp_AB) : (phi_BA || disp_BA))) continue;
    RC(compose(c, fields, k, dims, nullptr, nullptr, phi[k], nullptr));
    if (disp[k]) RC(disp_field_launch(phi[k], dims[0], dims[1], dims[2], disp[k], c.st));
  }
  return 0;
}

int upload(oai_reg_handle* h, const void* host, size_t bytes, void** dev) {
  RC(check_cuda(cudaMalloc(dev, bytes), "reg_create: cudaMalloc"));
  h->allocs.push_back(*dev);
  return check_cuda(cudaMemcpy(*dev, host, bytes, cudaMemcpyHostToDevice), "reg_create: upload");
}

int upload_unet(oai_reg_handle* h, const TensorGroup& g, UNetWeights* w) {
  std::vector<float> buf;
  for (int d = 0; d < 5; ++d) {
    const std::string D = std::to_string(d);
    {   // Conv3d weight [cout][cin][27] -> [cin][27][cout]
      const int cin = kDown[d], cout = kDown[d + 1];
      const float* src = g.at("downConvs." + D + ".weight")->data;
      buf.assign(static_cast<size_t>(cin) * 27 * cout, 0.f);
      for (int co = 0; co < cout; ++co)
        for (int ci = 0; ci < cin; ++ci)
          for (int t = 0; t < 27; ++t)
            buf[(static_cast<size_t>(ci) * 27 + t) * cout + co] = src[(static_cast<size_t>(co) * cin + ci) * 27 + t];
      RC(upload(h, buf.data(), buf.size() * 4, reinterpret_cast<void**>(&w->dw[d])));
      RC(upload(h, g.at("downConvs." + D + ".bias")->data, sizeof(float) * cout, reinterpret_cast<void**>(&w->db[d])));
      w->du[d] = nullptr;
      w->dexp[d] = 0;
      if (const size_t nb = conv3_umma_wbytes(cin, cout)) {
        float wmax = 0.f;
        for (float v : buf) wmax = std::max(wmax, std::fabs(v));
        int wexp = wmax == 0.f ? 0 : static_cast<int>(13 - std::floor(std::log2(static_cast<double>(wmax))));
        w->dexp[d] = std::max(-14, std::min(30, wexp));
        RC(check_cuda(cudaMalloc(&w->du[d], nb), "reg_create: cudaMalloc"));
        h->allocs.push_back(w->du[d]);
        RC(reg_pack_conv3_umma_launch(w->dw[d], cin, cout, cout, w->dexp[d], w->du[d], nullptr));
      }
    }
    {   // ConvTranspose3d weight [cin][cout][64] -> [cin][64][cout]
      const int cin = up_in(d), cout = kUpOut[d];
      const float* src = g.at("upConvs." + D + ".weight")->data;
      buf.assign(static_cast<size_t>(cin) * 64 * cout, 0.f);
      float wmax = 0.f;
      for (int ci = 0; ci < cin; ++ci)
        for (int co = 0; co < cout; ++co)
          for (int t = 0; t < 64; ++t) {
            const float v = src[(static_cast<size_t>(ci) * cout + co) * 64 + t];
            buf[(static_cast<size_t>(ci) * 64 + t) * cout + co] = v;
            wmax = std::max(wmax, std::fabs(v));
          }
      RC(upload(h, buf.data(), buf.size() * 4, reinterpret_cast<void**>(&w->uw[d])));
      RC(upload(h, g.at("upConvs." + D + ".bias")->data, sizeof(float) * cout, reinterpret_cast<void**>(&w->ub[d])));
      // scale so that max|w| * 2^wexp lies in [2^13, 2^14): the lo halves stay clear of fp16 subnormals
      int wexp = wmax == 0.f ? 0 : static_cast<int>(13 - std::floor(std::log2(static_cast<double>(wmax))));
      wexp = std::max(-14, std::min(30, wexp));
      w->uexp[d] = wexp;
      void* q = nullptr;
      RC(check_cuda(cudaMalloc(&q, static_cast<size_t>(cin) * 64 * cout * 4), "reg_create: cudaMalloc"));
      h->allocs.push_back(q);
      w->uq[d] = static_cast<uint4*>(q);
      RC(reg_pack_convt4_launch(w->uw[d], cin, cout, wexp, w->uq[d], nullptr));
      w->uu[d] = nullptr;
      if (cout <= 128) {
        RC(check_cuda(cudaMalloc(&w->uu[d], convt4_umma_wbytes(cin, cout)), "reg_create: cudaMalloc"));
        h->allocs.push_back(w->uu[d]);
        RC(reg_pack_convt4_umma_launch(w->uw[d], cin, cout, wexp, w->uu[d], nullptr));
      }
      // BatchNorm3d(eval) folded in float64
      const float* gamma = g.at("batchNorms." + D + ".weight")->data;
      const float* beta = g.at("batchNorms." + D + ".bias")->data;
      const float* mean = g.at("batchNorms." + D + ".running_mean")->data;
      const float* var = g.at("batchNorms." + D + ".running_var")->data;
      std::vector<float> sc(cout), sh(cout);
      for (int co = 0; co < cout; ++co) {
        const double s = static_cast<double>(gamma[co]) / std::sqrt(static_cast<double>(var[co]) + 1e-5);
        sc[co] = static_cast<float>(s);
        sh[co] = static_cast<float>(static_cast<double>(beta[co]) - static_cast<double>(mean[co]) * s);
      }
      RC(upload(h, sc.data(), sizeof(float) * cout, reinterpret_cast<void**>(&w->bs[d])));
      RC(upload(h, sh.data(), sizeof(float) * cout, reinterpret_cast<void**>(&w->bt[d])));
    }
  }
  const float* src = g.at("lastConv.weight")->data;   // [3][18][27] -> [18][27][4]
  buf.assign(18 * 27 * 4, 0.f);
  for (int co = 0; co < 3; ++co)
    for (int ci = 0; ci < 18; ++ci)
      for (int t = 0; t < 27; ++t) buf[(ci * 27 + t) * 4 + co] = src[(co * 18 + ci) * 27 + t];
  RC(upload(h, buf.data(), buf.size() * 4, reinterpret_cast<void**>(&w->lw)));
  RC(upload(h, g.at("lastConv.bias")->data, sizeof(float) * 3, reinterpret_cast<void**>(&w->lb)));
  return check_cuda(cudaDeviceSynchronize(), "reg_create: weight packing");
}

}  // namespace

extern "C" int oai_reg_parse_tree(const oai_tensor* state_dict, int n_tensors, char* description,
                                  size_t description_bytes) {
  OAI_REQUIRE(state_dict || n_tensors == 0, "reg_parse_tree: null state dict");
  Parsed p;
  RC(parse_state_dict(state_dict, n_tensors, &p));
  if (description && description_bytes) snprintf(description, description_bytes, "%s", describe(p, p.root).c_str());
  return 0;
}

extern "C" int oai_reg_create(const oai_tensor* state_dict, int n_tensors, const int* net_dims, oai_reg_t* handle) {
  OAI_REQUIRE(handle && net_dims && (state_dict || n_tensors == 0), "reg_create: null pointer");
  *handle = nullptr;
  for (int a = 0; a < 3; ++a)
    OAI_REQUIRE(net_dims[a] >= 2, "reg_create: network axis %d has %d samples (at least 2 needed)", a, net_dims[a]);
  oai_reg_handle* h = new oai_reg_handle();
  auto bail = [&](int rc) {
    oai_reg_destroy(h);
    return rc;
  };
  if (int rc = parse_state_dict(state_dict, n_tensors, &h->tree)) return bail(rc);
  if (int rc = check_cuda(cudaGetDevice(&h->device), "reg_create: cudaGetDevice")) return bail(rc);
  for (int a = 0; a < 3; ++a) h->dims[a] = net_dims[a];
  h->description = describe(h->tree, h->tree.root);
  h->leaves.resize(h->tree.leaf_paths.size());
  for (size_t l = 0; l < h->leaves.size(); ++l)
    if (int rc = upload_unet(h, h->tree.leaf_tensors[l], &h->leaves[l])) return bail(rc);
  h->tree.leaf_tensors.clear();   // the caller's state dict is not referenced after this call
  // workspace plan: the allocation sequence of one forward, walked without launching anything
  Ctx c{h, nullptr, true, reinterpret_cast<char*>(uintptr_t(1) << 40), 0, nullptr, 0};
  if (int rc = run(c, nullptr, h->dims, nullptr, h->dims, nullptr, nullptr, nullptr, nullptr, &h->fields))
    return bail(rc);
  h->scratch_bytes = align256(std::max<size_t>(c.scratch_need, 256));
  h->arena_bytes = align256(c.off);
  h->pair_off = c.pair_off;
  *handle = h;
  return 0;
}

extern "C" int oai_reg_destroy(oai_reg_t h) {
  if (!h) return 0;
  for (void* p : h->allocs) cudaFree(p);
  delete h;
  return 0;
}

extern "C" int oai_reg_describe(oai_reg_t h, char* description, size_t description_bytes) {
  OAI_REQUIRE(h && description && description_bytes, "reg_describe: null pointer");
  snprintf(description, description_bytes, "%s", h->description.c_str());
  return 0;
}

extern "C" size_t oai_reg_workspace_bytes(oai_reg_t h) { return h ? h->scratch_bytes + h->arena_bytes : 0; }

extern "C" int oai_reg_num_fields(oai_reg_t h) { return h ? static_cast<int>(h->fields.size()) : 0; }

extern "C" int oai_reg_field(oai_reg_t h, int index, size_t* workspace_offset, int* dims) {
  OAI_REQUIRE(h && workspace_offset && dims, "reg_field: null pointer");
  OAI_REQUIRE(index >= 0 && index < static_cast<int>(h->fields.size()), "reg_field: index %d out of range", index);
  *workspace_offset = h->scratch_bytes + h->fields[index].off;
  for (int a = 0; a < 3; ++a) dims[a] = h->fields[index].dims[a];
  return 0;
}

namespace {
int check_workspace(oai_reg_t h, const void* ws, size_t ws_bytes, const char* who) {
  OAI_REQUIRE(h, "%s: null handle", who);
  OAI_REQUIRE(ws && (reinterpret_cast<uintptr_t>(ws) & 255) == 0 && ws_bytes >= oai_reg_workspace_bytes(h),
              "%s: workspace of %zu bytes, 256-byte aligned, required", who, oai_reg_workspace_bytes(h));
  int dev = -1;
  cudaGetDevice(&dev);
  OAI_REQUIRE(dev == h->device, "%s: handle was created on device %d, current device is %d", who, h->device, dev);
  return 0;
}
}  // namespace

extern "C" int oai_reg_forward(oai_reg_t h, const float* image_A, const int* dims_A, const float* image_B,
                               const int* dims_B, float* phi_AB, float* phi_BA, float* disp_AB, float* disp_BA,
                               void* workspace, size_t workspace_bytes, void* stream) {
  RC(check_workspace(h, workspace, workspace_bytes, "reg_forward"));
  OAI_REQUIRE(image_A && dims_A && image_B && dims_B, "reg_forward: null image");
  for (int a = 0; a < 3; ++a)
    OAI_REQUIRE(dims_A[a] >= 1 && dims_B[a] >= 1, "reg_forward: empty image axis %d", a);
  nvtxRangePushA("oai.reg_forward");
  Ctx c{h, static_cast<cudaStream_t>(stream), false, static_cast<char*>(workspace) + h->scratch_bytes, 0, workspace,
        h->scratch_bytes};
  const int rc = run(c, image_A, dims_A, image_B, dims_B, phi_AB, phi_BA, disp_AB, disp_BA, nullptr);
  nvtxRangePop();
  if (rc) return rc;
  OAI_REQUIRE(align256(c.off) == h->arena_bytes && c.scratch_need <= h->scratch_bytes,
              "reg_forward: workspace plan mismatch (%zu vs %zu bytes)", align256(c.off), h->arena_bytes);
  h->forwarded = true;
  return 0;
}

extern "C" int oai_reg_warp_image(oai_reg_t h, const float* image, const int* dims, int direction, float* out,
                                  void* workspace, size_t workspace_bytes, void* stream) {
  RC(check_workspace(h, workspace, workspace_bytes, "reg_warp_image"));
  OAI_REQUIRE(image && dims && out, "reg_warp_image: null pointer");
  OAI_REQUIRE(direction == 0 || direction == 1, "reg_warp_image: direction must be 0 (phi_AB) or 1 (phi_BA)");
  Ctx c{h, static_cast<cudaStream_t>(stream), false, static_cast<char*>(workspace) + h->scratch_bytes, 0, workspace,
        h->scratch_bytes};
  std::vector<Field> fields;
  for (const FieldRef& r : h->fields) {
    Field f;
    f.p = reinterpret_cast<float*>(c.arena + r.off);
    for (int a = 0; a < 3; ++a) f.dims[a] = r.dims[a];
    fields.push_back(f);
  }
  return compose(c, fields, direction, dims, image, dims, nullptr, out);
}

// ---- registration quality (GradientICON.forward's ICONLoss terms) on the last forward's workspace
namespace {

struct LossPlan {
  size_t phi, warped, tag, wtag, zb, g, s, m, count, total;   // byte offsets inside the loss workspace
  int ng, ns, nm;
};

LossPlan loss_plan(const oai_reg_handle* h, const oai_icon_loss_cfg& cfg) {
  const int D = h->dims[0], H = h->dims[1], W = h->dims[2];
  const size_t vol = voxels(h->dims);
  const bool ssd = cfg.similarity == OAI_SIM_SSD_ONLY_INTERPOLATED;
  LossPlan p{};
  size_t off = 0;
  auto take = [&](size_t bytes) {
    const size_t at = align256(off);
    off = at + bytes;
    return at;
  };
  p.ng = gradicon_blocks(D, H, W);
  p.ns = ssd ? ssd_blocks(D, H, W) : lncc_blocks(D, H, W);
  p.nm = jacobian_blocks(D, H, W);
  p.phi = take(sizeof(float) * kBatch * 3 * vol);    // phi_AB, phi_BA on the identity map
  p.warped = take(sizeof(float) * kBatch * vol);     // S(A, phi_AB), S(B, phi_BA)
  if (ssd) {
    p.tag = take(sizeof(float) * vol);
    p.wtag = take(sizeof(float) * kBatch * vol);
  } else {
    p.zb = take(sizeof(float) * 5 * vol);
  }
  p.g = take(sizeof(double) * p.ng);
  p.s = take(sizeof(double) * kBatch * 2 * p.ns);
  p.m = take(sizeof(double) * p.nm);
  p.count = take(sizeof(unsigned long long));
  p.total = align256(off);
  return p;
}

int check_loss_cfg(const oai_icon_loss_cfg* cfg) {
  OAI_REQUIRE(cfg, "reg_icon_loss: null configuration");
  OAI_REQUIRE(cfg->similarity == OAI_SIM_LNCC || cfg->similarity == OAI_SIM_SSD_ONLY_INTERPOLATED,
              "reg_icon_loss: unknown similarity %d (0 = LNCC, 1 = ssd_only_interpolated)", cfg->similarity);
  if (cfg->similarity == OAI_SIM_LNCC)
    OAI_REQUIRE(cfg->sigma > 0 && lncc_radius(cfg->sigma) <= kLnccMaxRadius,
                "reg_icon_loss: LNCC sigma %g outside (0, 12.5)", cfg->sigma);
  OAI_REQUIRE(std::isfinite(cfg->delta) && cfg->delta > 0, "reg_icon_loss: delta %g must be positive", cfg->delta);
  OAI_REQUIRE(std::isfinite(cfg->lmbda), "reg_icon_loss: lmbda must be finite");
  return 0;
}

}  // namespace

extern "C" size_t oai_reg_loss_workspace_bytes(oai_reg_t h, const oai_icon_loss_cfg* cfg) {
  if (!h || check_loss_cfg(cfg)) return 0;
  return loss_plan(h, *cfg).total;
}

extern "C" int oai_reg_icon_loss(oai_reg_t h, const oai_icon_loss_cfg* cfg, const float* noise, double* terms,
                                 float* jac_det_BA, void* loss_ws, size_t loss_ws_bytes, const void* reg_ws,
                                 size_t reg_ws_bytes, void* stream) {
  RC(check_loss_cfg(cfg));
  OAI_REQUIRE(h, "reg_icon_loss: null handle");
  OAI_REQUIRE(noise && terms, "reg_icon_loss: null noise / terms");
  OAI_REQUIRE(h->forwarded, "reg_icon_loss: no oai_reg_forward has run on this handle");
  const LossPlan lp = loss_plan(h, *cfg);
  OAI_REQUIRE(loss_ws && (reinterpret_cast<uintptr_t>(loss_ws) & 255) == 0 && loss_ws_bytes >= lp.total,
              "reg_icon_loss: loss workspace of %zu bytes, 256-byte aligned, required (got %zu)", lp.total,
              loss_ws_bytes);
  RC(check_workspace(h, reg_ws, reg_ws_bytes, "reg_icon_loss"));
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  const int* dims = h->dims;
  const int D = dims[0], H = dims[1], W = dims[2];
  const size_t vol = voxels(dims);
  char* lw = static_cast<char*>(loss_ws);
  char* arena = const_cast<char*>(static_cast<const char*>(reg_ws)) + h->scratch_bytes;
  const float* pair = reinterpret_cast<const float*>(arena + h->pair_off);   // [A, B] at the network shape
  float* phi = reinterpret_cast<float*>(lw + lp.phi);
  float* warped = reinterpret_cast<float*>(lw + lp.warped);
  double* g = reinterpret_cast<double*>(lw + lp.g);
  double* s = reinterpret_cast<double*>(lw + lp.s);
  double* m = reinterpret_cast<double*>(lw + lp.m);
  auto* count = reinterpret_cast<unsigned long long*>(lw + lp.count);
  const bool ssd = cfg->similarity == OAI_SIM_SSD_ONLY_INTERPOLATED;
  nvtxRangePushA("oai.reg_icon_loss");
  auto body = [&]() -> int {
    Ctx c{h, st, false, arena, 0, nullptr, 0};
    std::vector<Field> fields;
    for (const FieldRef& r : h->fields) {
      Field f;
      f.p = reinterpret_cast<float*>(arena + r.off);
      for (int a = 0; a < 3; ++a) f.dims[a] = r.dims[a];
      fields.push_back(f);
    }
    if (ssd) RC(inbounds_tag_launch(reinterpret_cast<float*>(lw + lp.tag), D, H, W, st));
    // phi_AB / phi_BA on the identity map and the warped images: direction k warps pair[k] onto pair[1 - k]
    for (int k = 0; k < kBatch; ++k) {
      RC(compose(c, fields, k, dims, pair + k * vol, dims, phi + k * 3 * vol, warped + k * vol));
      if (ssd)
        RC(compose(c, fields, k, dims, reinterpret_cast<const float*>(lw + lp.tag), dims, nullptr,
                   reinterpret_cast<float*>(lw + lp.wtag) + k * vol));
    }
    for (int k = 0; k < kBatch; ++k) {
      double* sk = s + static_cast<size_t>(k) * 2 * lp.ns;
      if (ssd) {
        RC(ssd_launch(warped + k * vol, reinterpret_cast<const float*>(lw + lp.wtag) + k * vol,
                      pair + (1 - k) * vol, D, H, W, sk, sk + lp.ns, st));
      } else {
        LnccParams q{};
        q.D = D; q.H = H; q.W = W;
        q.I = warped + k * vol;
        q.J = pair + (1 - k) * vol;
        q.radius = lncc_radius(cfg->sigma);
        double wsum = 0.0, w[2 * kLnccMaxRadius + 1];
        for (int i = -q.radius; i <= q.radius; ++i) wsum += w[i + q.radius] = std::exp(-(i * i) / (2.0 * cfg->sigma * cfg->sigma));
        for (int i = 0; i <= 2 * q.radius; ++i) q.taps[i] = static_cast<float>(w[i] / wsum);
        q.zb = reinterpret_cast<float*>(lw + lp.zb);
        q.partials = sk;
        RC(lncc_launch(q, st));
      }
    }
    GradIconParams gp{};
    gp.D = D; gp.H = H; gp.W = W;
    gp.noise = noise;
    gp.delta = static_cast<float>(cfg->delta);
    for (int dir = 0; dir < 2; ++dir) {   // phi_BA's fields (direction 1 of the batch) first, then phi_AB's
      const int k = 1 - dir;
      gp.nf[dir] = static_cast<int>(fields.size());
      for (size_t f = 0; f < fields.size(); ++f) {
        gp.u[dir][f] = fields[f].p + static_cast<size_t>(k) * 3 * voxels(fields[f].dims);
        gp.ud[dir][f] = fields[f].dims[0]; gp.uh[dir][f] = fields[f].dims[1]; gp.uw[dir][f] = fields[f].dims[2];
      }
    }
    gp.partials = g;
    RC(gradicon_launch(gp, st));
    JacobianParams jp{};
    jp.D = D; jp.H = H; jp.W = W;
    jp.phi_jac = phi + 3 * vol;   // losses.flips(phi_BA_vectorfield), as GradientICON.forward counts it
    jp.phi_mag = phi;             // mean((identity_map - phi_AB_vectorfield) ** 2)
    jp.det_out = jac_det_BA;
    jp.count = count;
    jp.mag_partials = m;
    RC(jacobian_launch(jp, st));
    LossFinishParams fp{};
    fp.g = g; fp.ng = lp.ng;
    fp.s = s; fp.ns = lp.ns; fp.ssd = ssd ? 1 : 0;
    fp.m = m; fp.nm = lp.nm;
    fp.count = count;
    fp.nvox = static_cast<double>(vol);
    fp.lmbda = cfg->lmbda;
    fp.terms = terms;
    return loss_finish_launch(fp, st);
  };
  const int rc = body();
  nvtxRangePop();
  return rc;
}

extern "C" int oai_jacobian_flips(const float* phi, const int* dims, float* det_out, long long* count_out,
                                  void* stream) {
  OAI_REQUIRE(phi && dims && count_out, "jacobian_flips: null pointer");
  for (int a = 0; a < 3; ++a)
    OAI_REQUIRE(dims[a] >= 2, "jacobian_flips: axis %d has %d samples (at least 2 needed)", a, dims[a]);
  OAI_REQUIRE(static_cast<long long>((dims[2] + 31) / 32) * ((dims[1] + 7) / 8) * dims[0] < (1ll << 31),
              "jacobian_flips: map too large");
  JacobianParams jp{};
  jp.D = dims[0]; jp.H = dims[1]; jp.W = dims[2];
  jp.phi_jac = phi;
  jp.det_out = det_out;
  jp.count = reinterpret_cast<unsigned long long*>(count_out);
  return jacobian_launch(jp, static_cast<cudaStream_t>(stream));
}
