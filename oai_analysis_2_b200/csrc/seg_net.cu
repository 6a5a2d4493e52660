// Stage-level C ABI of the segmentation stage: the whole of Segmenter3DInPatchClassWise.segment
// (reference: oai_analysis/segmentation/segmenter.py:100-131) behind three calls --
//   oai_seg_create   : UNet.__init__ + initialize_model's load_state_dict (networks.py:39-66, utils.py:20-41): takes the
//                      reference's state-dict tensors, folds BatchNorm(eval), re-orients the transposed convolutions,
//                      packs every layer for the tcgen05 kernel and uploads the result;
//   oai_seg_forward  : Partition.__call__ + UNet.forward over all tiles + sigmoid (+ >0.5) + Partition.assemble
//                      (image_transforms.py:395-519, networks.py:109-149, segmenter.py:109-129);
//   oai_seg_destroy.
// Layer order, skip wiring, dead-halo regions, precision plan and the activation workspace layout all live here, so a
// host language with a C FFI needs nothing else.  The caller owns the input / output volumes, the activation
// workspace and the stream; the handle owns only the packed weights.
#include "../../include/oai_b200.h"
#include "api_common.h"
#include "conv_api.h"
#include "seg_misc.cuh"

#include <nvtx3/nvToolsExt.h>

#include <algorithm>
#include <cmath>
#include <cstdlib>
#include <cstring>
#include <map>
#include <set>
#include <string>
#include <vector>

using namespace oai;

namespace {

struct LayerDef {
  const char* name;
  char kind;    // 'c' Conv3d k3 p1 | 't' ConvTranspose3d k3 s1 p1 | 'u' ConvTranspose3d k2 s2
  int cin, cout;
  int level;    // resolution level of the layer's INPUT grid (tile >> level)
  int c_first;  // channels of the first source when the input is cat((upsampled, skip)) (networks.py:127,134,141)
};

// networks.py:43-66 (ec0 is evaluated by the stem kernel, dc0 by the fused head)
const LayerDef kLayers[] = {
    {"ec0", 'c', 1, 32, 0, 0},     {"ec1", 'c', 32, 64, 0, 0},    {"ec2", 'c', 64, 64, 1, 0},
    {"ec3", 'c', 64, 128, 1, 0},   {"ec4", 'c', 128, 128, 2, 0},  {"ec5", 'c', 128, 256, 2, 0},
    {"ec6", 'c', 256, 256, 3, 0},  {"ec7", 'c', 256, 512, 3, 0},  {"dc9", 'u', 512, 512, 3, 0},
    {"dc8", 't', 768, 256, 2, 512}, {"dc7", 't', 256, 256, 2, 0}, {"dc6", 'u', 256, 256, 2, 0},
    {"dc5", 't', 384, 128, 1, 256}, {"dc4", 't', 128, 128, 1, 0}, {"dc3", 'u', 128, 128, 1, 0},
    {"dc2", 't', 192, 64, 0, 128},  {"dc1", 't', 64, 64, 0, 0},
};
constexpr int kNumLayers = 17;
enum { EC0, EC1, EC2, EC3, EC4, EC5, EC6, EC7, DC9, DC8, DC7, DC6, DC5, DC4, DC3, DC2, DC1 };

// activation tensors of one tile batch, in creation order
enum { T_E0, T_SYN0, T_P0, T_E2, T_SYN1, T_P1, T_E4, T_SYN2, T_P2, T_E6, T_E7, T_D9, T_D8, T_D7, T_D6, T_D5, T_D4,
       T_D3, T_D2, kNumTensors };
struct TensorDef {
  int level, channels, birth, last_use;  // steps as numbered in forward()
  int consumers[2];                       // layers reading it through the tensor pipe (-1: none / pooled)
};
const TensorDef kTensors[kNumTensors] = {
    {0, 32, 0, 1, {EC1, -1}},    {0, 64, 1, 18, {DC2, -1}},    {1, 64, 2, 3, {EC2, -1}},    {1, 64, 3, 4, {EC3, -1}},
    {1, 128, 4, 15, {DC5, -1}},  {2, 128, 5, 6, {EC4, -1}},    {2, 128, 6, 7, {EC5, -1}},   {2, 256, 7, 12, {DC8, -1}},
    {3, 256, 8, 9, {EC6, -1}},   {3, 256, 9, 10, {EC7, -1}},   {3, 512, 10, 11, {DC9, -1}}, {2, 512, 11, 12, {DC8, -1}},
    {2, 256, 12, 13, {DC7, -1}}, {2, 256, 13, 14, {DC6, -1}},  {1, 256, 14, 15, {DC5, -1}}, {1, 128, 15, 16, {DC4, -1}},
    {1, 128, 16, 17, {DC3, -1}}, {0, 128, 17, 18, {DC2, -1}},  {0, 64, 18, 19, {DC1, -1}},
};
// the pooled copies feed ec2 / ec4 / ec6: a skip tensor is pooled through whichever planes its pooled consumer needs
const int kPoolOf[3][3] = {{T_SYN0, T_P0, EC2}, {T_SYN1, T_P1, EC4}, {T_SYN2, T_P2, EC6}};

struct PackedLayer {
  ConvSpec spec;
  void* w = nullptr;   // device, packed
  size_t w_bytes = 0;
  float* bias = nullptr;  // device [cout]
};

struct Box {
  int lo[3], hi[3];
};

}  // namespace

struct oai_seg_handle {
  oai_seg_config cfg;
  int device;
  int tile[3], overlap[3];   // z,y,x
  int terms[kNumLayers];
  int split[kNumTensors];
  int lo8[kNumTensors];      // the tensor is a plain 16-bit hi tensor followed by an e4m3 lo plane (terms 6 / 7)
  PackedLayer layers[kNumLayers];
  float* stem_w = nullptr;   // [27][32]
  float* head_w = nullptr;   // [ncls][64]
  float* head_b = nullptr;   // [ncls]
  bool has_region = false;
  Box region[kNumLayers];    // dead-halo elimination: output sub-box each decoder layer must compute
};

namespace {

int dims_at(const oai_seg_handle* h, int level, int a) { return h->tile[a] >> level; }

// bytes of the 16-bit part of a tensor ([hi | lo] planes when split); a lo8 tensor's e4m3 plane follows it
size_t tensor_hi_bytes(const oai_seg_handle* h, int t, int NT) {
  const TensorDef& d = kTensors[t];
  size_t n = static_cast<size_t>(NT) * dims_at(h, d.level, 0) * dims_at(h, d.level, 1) * dims_at(h, d.level, 2) *
             d.channels * 2 * (h->split[t] ? 2 : 1);
  return (n + 255) & ~size_t(255);
}

size_t tensor_bytes(const oai_seg_handle* h, int t, int NT) {
  const size_t hi = tensor_hi_bytes(h, t, NT);
  return h->lo8[t] ? hi + (((hi / 2) + 255) & ~size_t(255)) : hi;   // 2 B + 1 B per channel and voxel
}

// First-fit offsets for the batch's activation tensors from their lifetimes; returns the peak.
size_t plan_workspace(const oai_seg_handle* h, int NT, size_t* offs) {
  struct Live { size_t off, size; int last; };
  std::vector<Live> live;
  size_t peak = 0;
  for (int t = 0; t < kNumTensors; ++t) {
    const int birth = kTensors[t].birth;
    live.erase(std::remove_if(live.begin(), live.end(), [&](const Live& l) { return l.last < birth; }), live.end());
    std::sort(live.begin(), live.end(), [](const Live& a, const Live& b) { return a.off < b.off; });
    const size_t size = tensor_bytes(h, t, NT);
    size_t off = 0;
    for (const Live& l : live) {
      if (off + size <= l.off) break;
      off = std::max(off, l.off + l.size);
    }
    offs[t] = off;
    live.push_back(Live{off, size, kTensors[t].last_use});
    peak = std::max(peak, off + size);
  }
  return peak;
}

// image_transforms.py:404-406
void tiling(const oai_seg_handle* h, const int* vol, int* eff, int* grid) {
  for (int a = 0; a < 3; ++a) {
    eff[a] = h->tile[a] - 2 * h->overlap[a];
    grid[a] = (vol[a] + eff[a] - 1) / eff[a];
  }
}

// Output sub-boxes the kept tile interior depends on, per decoder layer.  The reference computes every layer on the
// whole tile and crops afterwards (image_transforms.py:497-503); a k3 conv widens the needed box by 1, a k2s2 up-conv
// halves it.  Boxes of the up-convs are on their INPUT grid.
void needed_regions(const int* tile, const int* overlap, Box* region) {
  auto clampbox = [&](Box b, int lvl) {
    for (int a = 0; a < 3; ++a) {
      b.lo[a] = std::max(b.lo[a], 0);
      b.hi[a] = std::min(b.hi[a], (tile[a] >> lvl) - 1);
    }
    return b;
  };
  auto dil = [&](Box b, int k, int lvl) {
    for (int a = 0; a < 3; ++a) { b.lo[a] -= k; b.hi[a] += k; }
    return clampbox(b, lvl);
  };
  auto half = [&](Box b, int lvl) {
    for (int a = 0; a < 3; ++a) { b.lo[a] /= 2; b.hi[a] /= 2; }
    return clampbox(b, lvl);
  };
  for (int l = 0; l < kNumLayers; ++l)
    for (int a = 0; a < 3; ++a) { region[l].lo[a] = 0; region[l].hi[a] = (tile[a] >> kLayers[l].level) - 1; }
  Box n0;
  for (int a = 0; a < 3; ++a) { n0.lo[a] = overlap[a]; n0.hi[a] = tile[a] - overlap[a] - 1; }
  n0 = clampbox(n0, 0);
  region[DC1] = n0;
  region[DC2] = dil(n0, 1, 0);
  Box need = dil(n0, 2, 0);
  const int ups[2][3] = {{DC3, DC4, DC5}, {DC6, DC7, DC8}};
  for (int i = 0; i < 2; ++i) {
    const int lvl = i + 1;
    const Box q = half(need, lvl);
    region[ups[i][0]] = q;
    region[ups[i][1]] = q;
    region[ups[i][2]] = dil(q, 1, lvl);
    need = dil(q, 2, lvl);
  }
  region[DC9] = half(need, 3);
}

struct NamedTensor {
  const float* data;
  std::vector<long long> shape;
  long long numel;
};

// OAI_B200_SEG_W_HALO=0 keeps dc2 and dc1 in row-shared mode (whole 128-wide rows, the w halo computed and dropped)
bool w_halo_skip_disabled() {
  const char* e = getenv("OAI_B200_SEG_W_HALO");
  return e && e[0] == '0';
}

// OAI_B200_SEG_LO8=0 keeps the mixed plan's lo terms as fp16 planes (codes 4 / 2 instead of 6 / 7)
bool lo8_disabled() {
  const char* e = getenv("OAI_B200_SEG_LO8");
  return e && e[0] == '0';
}

int device_copy(const void* host, size_t bytes, void** dev) {
  if (int rc = check_cuda(cudaMalloc(dev, bytes), "seg_create: cudaMalloc")) return rc;
  return check_cuda(cudaMemcpy(*dev, host, bytes, cudaMemcpyHostToDevice), "seg_create: cudaMemcpy");
}

}  // namespace

extern "C" int oai_seg_needed_regions(const int* tile_zyx, const int* overlap_zyx, int* boxes) {
  OAI_REQUIRE(tile_zyx && overlap_zyx && boxes, "seg_needed_regions: null pointer");
  Box region[kNumLayers];
  needed_regions(tile_zyx, overlap_zyx, region);
  for (int l = 0; l < kNumLayers; ++l)
    for (int a = 0; a < 3; ++a) {
      boxes[l * 6 + a] = region[l].lo[a];
      boxes[l * 6 + 3 + a] = region[l].hi[a];
    }
  return 0;
}

extern "C" int oai_seg_layer_terms(int precision, int* terms17) {
  OAI_REQUIRE(terms17 != nullptr, "seg_layer_terms: null pointer");
  OAI_REQUIRE(precision >= OAI_SEG_PRECISION_FP16 && precision <= OAI_SEG_PRECISION_FP16X3,
              "seg_layer_terms: unknown precision %d", precision);
  for (int l = 0; l < kNumLayers; ++l) terms17[l] = 1;
  if (precision == OAI_SEG_PRECISION_MIXED) {
    // Where the logit error comes from was measured plan by plan on the golden fixtures (scripts/dice_plans.py,
    // profiles/r02_dice_plans.jsonl; mask flips summed over the three fixtures, noise about +-3): all-fp16 30;
    // dc2 reading both inputs as fp16 hi + lo pairs 17; only its skip input (ec1's output, the largest activations
    // of the network) 22; only its upsampled input 25; the skip input AND dc1's input 11; dc2 + dc1 entirely 5.
    // The default spends the split where it pays: dc2's skip source (code 4: 64 of its 192 input channels) and dc1
    // -- +9 ms per knee over all-fp16 instead of +20 ms for all of dc2, with fewer flips (min Dice 0.99932).
    // The lo terms carry ~2^-11 of the activation, so they are stored as e4m3 planes and issued as block-scaled 8-bit
    // MMAs at twice the fp16 rate (codes 6 / 7; adds ~2^-14 relative, 8x below the hi term's fp16 rounding);
    // OAI_B200_SEG_LO8=0 keeps them as fp16 planes.
    const bool lo8 = !lo8_disabled();
    terms17[DC2] = lo8 ? 6 : 4;
    terms17[DC1] = lo8 ? 7 : 2;
  } else if (precision == OAI_SEG_PRECISION_FP16X2 || precision == OAI_SEG_PRECISION_FP16X3) {
    for (int l = 1; l < kNumLayers; ++l) terms17[l] = precision == OAI_SEG_PRECISION_FP16X2 ? 2 : 3;
  }
  return 0;
}

extern "C" int oai_seg_create(const oai_seg_config* cfg, const oai_tensor* state_dict, int n_tensors,
                              oai_seg_t* handle) {
  OAI_REQUIRE(cfg && state_dict && handle, "seg_create: null pointer");
  OAI_REQUIRE(cfg->in_channels == 1, "seg_create: the fused stem kernel supports in_channels == 1 (got %d)",
              cfg->in_channels);
  OAI_REQUIRE(cfg->n_classes >= 1 && cfg->n_classes <= 8, "seg_create: n_classes=%d unsupported", cfg->n_classes);
  OAI_REQUIRE(cfg->ab_format == 0 || cfg->ab_format == 1, "seg_create: ab_format=%d", cfg->ab_format);
  std::map<std::string, NamedTensor> sd;
  for (int i = 0; i < n_tensors; ++i) {
    const oai_tensor& t = state_dict[i];
    OAI_REQUIRE(t.name && t.ndim >= 0 && t.ndim <= 5, "seg_create: bad tensor %d", i);
    NamedTensor nt;
    nt.data = t.data;
    nt.numel = 1;
    for (int d = 0; d < t.ndim; ++d) { nt.shape.push_back(t.shape[d]); nt.numel *= t.shape[d]; }
    OAI_REQUIRE(sd.emplace(t.name, nt).second, "seg_create: duplicate key %s", t.name);
  }
  oai_seg_handle* h = new oai_seg_handle();
  struct Guard {
    oai_seg_handle* h;
    ~Guard() { if (h) oai_seg_destroy(h); }
  } guard{h};
  h->cfg = *cfg;
  cudaGetDevice(&h->device);
  for (int a = 0; a < 3; ++a) {   // x,y,z -> z,y,x (image_transforms.py:389-391)
    h->tile[a] = cfg->patch_xyz[2 - a];
    h->overlap[a] = cfg->overlap_xyz[2 - a];
    OAI_REQUIRE(h->tile[a] > 0 && h->tile[a] % 8 == 0, "seg_create: tile size %d must be a positive multiple of 8",
                h->tile[a]);
    OAI_REQUIRE(h->overlap[a] >= 0 && 2 * h->overlap[a] < h->tile[a],
                "seg_create: overlap_size must be smaller than half the patch size");
  }
  if (cfg->precision == OAI_SEG_PRECISION_CUSTOM) {
    for (int l = 0; l < kNumLayers; ++l) {
      h->terms[l] = l == 0 ? 1 : cfg->layer_terms[l];
      const int tm = h->terms[l];
      // 4 / 5 / 6 on concatenating layers only; 7 on one-source 3x3x3 layers whose input a conv writes
      const bool conv_input = l == EC3 || l == EC5 || l == EC7 || l == DC7 || l == DC4 || l == DC1;
      OAI_REQUIRE(tm >= 1 && tm <= 7 && ((tm != 4 && tm != 5 && tm != 6) || kLayers[l].c_first > 0) &&
                      (tm != 7 || conv_input),
                  "seg_create: layer_terms[%d]=%d", l, h->terms[l]);
    }
  } else if (oai_seg_layer_terms(cfg->precision, h->terms)) {
    return 1;
  }
  for (int t = 0; t < kNumTensors; ++t) {
    // a tensor carries [hi | lo] planes when the layer reading it splits that source (terms 4 / 5: only the skip / only
    // the upsampled source of a concatenating layer)
    const int c = kTensors[t].consumers[0];
    const bool is_skip = t == T_SYN0 || t == T_SYN1 || t == T_SYN2;
    const int tm = c >= 0 ? h->terms[c] : 1;
    h->split[t] = tm == 2 || tm == 3 || (tm == 4 && is_skip) || (tm == 5 && !is_skip);
    h->lo8[t] = (tm == 6 && is_skip) || tm == 7;
  }
  for (int i = 0; i < 3; ++i) {  // a skip tensor must also carry both planes when its pooled consumer wants them
    if (h->split[kPoolOf[i][1]]) h->split[kPoolOf[i][0]] = 1;
    // the pool reads the 16-bit part only, so a lo8 skip tensor pools like a plain one; a skip tensor cannot be both
    OAI_REQUIRE(!(h->split[kPoolOf[i][0]] && h->lo8[kPoolOf[i][0]]),
                "seg_create: layer_terms: %s reads its skip input with an e4m3 lo plane while %s needs it as fp16 hi + lo",
                kLayers[kTensors[kPoolOf[i][0]].consumers[0]].name, kLayers[kPoolOf[i][2]].name);
  }
  needed_regions(h->tile, h->overlap, h->region);
  h->has_region = h->overlap[0] || h->overlap[1] || h->overlap[2];
  // dc2 and dc1 (full resolution, 64 output channels) compute only their needed (h, w) box: kh-shared M tiles skip the
  // dead w halo that row-shared tiles (one whole 128-wide row each) compute and throw away
  const bool skip_w_halo = h->has_region && !w_halo_skip_disabled();

  // ---- consume the state dict (strict: every expected key present with the right shape, nothing left over)
  std::set<std::string> consumed;
  auto take = [&](const std::string& key, std::initializer_list<long long> shape, const NamedTensor** out) -> int {
    auto it = sd.find(key);
    OAI_REQUIRE(it != sd.end(), "seg_create: missing key %s in state_dict", key.c_str());
    const NamedTensor& t = it->second;
    bool ok = t.shape.size() == shape.size() && t.data != nullptr;
    size_t i = 0;
    for (long long s : shape) ok = ok && t.shape[i++] == s;
    OAI_REQUIRE(ok, "seg_create: size mismatch for %s", key.c_str());
    *out = &t;
    consumed.insert(key);
    return 0;
  };
  const int ncls = cfg->n_classes;
  for (int l = 0; l < kNumLayers; ++l) {
    const LayerDef& L = kLayers[l];
    const std::string nm = L.name;
    const int k = L.kind == 'u' ? 2 : 3, taps = k * k * k, ci = L.cin, co = L.cout;
    const NamedTensor *w, *b = nullptr, *g = nullptr, *beta = nullptr, *mean = nullptr, *var = nullptr;
    if (L.kind == 'c') {
      if (take(nm + ".0.weight", {co, ci, k, k, k}, &w)) return 1;
    } else {
      if (take(nm + ".0.weight", {ci, co, k, k, k}, &w)) return 1;
    }
    if (cfg->bias && take(nm + ".0.bias", {co}, &b)) return 1;
    if (cfg->BN) {
      if (take(nm + ".1.weight", {co}, &g) || take(nm + ".1.bias", {co}, &beta) ||
          take(nm + ".1.running_mean", {co}, &mean) || take(nm + ".1.running_var", {co}, &var))
        return 1;
      consumed.insert(nm + ".1.num_batches_tracked");   // integer bookkeeping of BatchNorm; callers may omit it
    }
    // conv orientation [co][ci][tap] with BatchNorm(eval) folded in float64 (networks.py:85-86, 99-100; eps 1e-5)
    std::vector<float> wf(static_cast<size_t>(co) * ci * taps), bf(co);
    for (int o = 0; o < co; ++o) {
      double s = 1.0, shift = b ? static_cast<double>(b->data[o]) : 0.0;
      if (cfg->BN) {
        s = static_cast<double>(g->data[o]) / std::sqrt(static_cast<double>(var->data[o]) + 1e-5);
        shift = (shift - mean->data[o]) * s + beta->data[o];
      }
      bf[o] = static_cast<float>(shift);
      for (int i = 0; i < ci; ++i)
        for (int t = 0; t < taps; ++t) {
          // ConvTranspose stores [ci][co]; a stride-1 transposed conv is a conv with the spatially flipped filter
          const size_t src = L.kind == 'c' ? (static_cast<size_t>(o) * ci + i) * taps + t
                                           : (static_cast<size_t>(i) * co + o) * taps + (L.kind == 't' ? taps - 1 - t : t);
          wf[(static_cast<size_t>(o) * ci + i) * taps + t] = static_cast<float>(static_cast<double>(w->data[src]) * s);
        }
    }
    PackedLayer& P = h->layers[l];
    if (device_copy(bf.data(), bf.size() * sizeof(float), reinterpret_cast<void**>(&P.bias))) return 1;
    if (l == EC0) {
      std::vector<float> w27(27 * co);
      for (int t = 0; t < 27; ++t)
        for (int o = 0; o < co; ++o) w27[t * co + o] = wf[static_cast<size_t>(o) * 27 + t];
      if (device_copy(w27.data(), w27.size() * sizeof(float), reinterpret_cast<void**>(&h->stem_w))) return 1;
      continue;
    }
    ConvSpec& s = P.spec;
    s.D = dims_at(h, L.level, 0); s.H = dims_at(h, L.level, 1); s.W = dims_at(h, L.level, 2);
    s.c0 = L.c_first ? L.c_first : ci;
    s.c1 = ci - s.c0;
    s.cout = co;
    s.kind = L.kind == 'u' ? 2 : 0;
    s.terms = h->terms[l];
    s.fmt = cfg->ab_format;
    // (where the tile is narrower than 128 these layers run per-tap tiles of whole rows, and stay so)
    s.flags = (skip_w_halo && (l == DC2 || l == DC1) && s.W % 128 == 0) ? kConvFlagKhShared : 0;
    s.split0 = s.split1 = 0;   // filled per launch from the tensors actually bound
    ConvSpec ps = s;            // the packer only needs the terms' split pattern (lo8 sources are plain hi tensors)
    ps.split0 = s.terms == 2 || s.terms == 3 || s.terms == 5;
    ps.split1 = (s.terms == 2 || s.terms == 3 || s.terms == 4) && s.c1 > 0;
    P.w_bytes = conv_wpack_bytes(ps);
    OAI_REQUIRE(P.w_bytes > 0, "seg_create: layer %s: %s", L.name, oai_last_error());
    std::vector<uint8_t> img(P.w_bytes);
    if (conv_pack_weights(ps, wf.data(), img.data(), img.size())) return 1;
    if (device_copy(img.data(), img.size(), &P.w)) return 1;
  }
  {
    const NamedTensor *w0, *b0 = nullptr;
    if (take("dc0.weight", {ncls, 64, 1, 1, 1}, &w0)) return 1;
    if (cfg->bias && take("dc0.bias", {ncls}, &b0)) return 1;
    std::vector<float> hb(ncls, 0.f);
    if (b0) std::copy(b0->data, b0->data + ncls, hb.begin());
    if (device_copy(w0->data, static_cast<size_t>(ncls) * 64 * sizeof(float), reinterpret_cast<void**>(&h->head_w)) ||
        device_copy(hb.data(), ncls * sizeof(float), reinterpret_cast<void**>(&h->head_b)))
      return 1;
  }
  for (const auto& kv : sd)
    OAI_REQUIRE(consumed.count(kv.first), "seg_create: unexpected key %s in state_dict", kv.first.c_str());
  guard.h = nullptr;
  *handle = h;
  return 0;
}

extern "C" int oai_seg_destroy(oai_seg_t h) {
  if (!h) return 0;
  for (int l = 0; l < kNumLayers; ++l) {
    cudaFree(h->layers[l].w);
    cudaFree(h->layers[l].bias);
  }
  cudaFree(h->stem_w);
  cudaFree(h->head_w);
  cudaFree(h->head_b);
  delete h;
  return 0;
}

extern "C" int oai_seg_num_tiles(oai_seg_t h, const int* vol_dims) {
  if (!h || !vol_dims) return -1;
  int eff[3], grid[3];
  tiling(h, vol_dims, eff, grid);
  return grid[0] * grid[1] * grid[2];
}

extern "C" size_t oai_seg_workspace_bytes(oai_seg_t h, const int* vol_dims, int tiles_per_batch) {
  if (!h || !vol_dims) return 0;
  const int T = oai_seg_num_tiles(h, vol_dims);
  const int nb = tiles_per_batch <= 0 ? T : std::min(T, tiles_per_batch);
  size_t offs[kNumTensors];
  return plan_workspace(h, nb, offs);
}

extern "C" int oai_seg_forward(oai_seg_t h, const float* vol, const int* vol_dims, float* out, int out_mode,
                               int tiles_per_batch, void* workspace, size_t workspace_bytes, void* stream) {
  OAI_REQUIRE(h && vol && vol_dims && out && workspace, "seg_forward: null pointer");
  OAI_REQUIRE(out_mode >= 0 && out_mode <= 2, "seg_forward: out_mode=%d", out_mode);
  OAI_REQUIRE((reinterpret_cast<uintptr_t>(workspace) & 255) == 0, "seg_forward: workspace must be 256-byte aligned");
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  int eff[3], grid[3];
  tiling(h, vol_dims, eff, grid);
  for (int a = 0; a < 3; ++a) {
    const int padded = eff[a] * grid[a] + 2 * h->overlap[a] - vol_dims[a];
    OAI_REQUIRE(vol_dims[a] >= 1 && !(vol_dims[a] < 2 && padded > 0),
                "seg_forward: reflect padding needs at least 2 samples along a padded axis");
  }
  const int T = grid[0] * grid[1] * grid[2];
  const int nb = tiles_per_batch <= 0 ? T : std::min(T, tiles_per_batch);
  size_t offs[kNumTensors];
  const size_t need = plan_workspace(h, nb, offs);
  OAI_REQUIRE(workspace_bytes >= need, "seg_forward: workspace holds %zu bytes, %d tiles per batch need %zu",
              workspace_bytes, nb, need);
  uint8_t* ws = static_cast<uint8_t*>(workspace);
  auto buf = [&](int t) { return static_cast<void*>(ws + offs[t]); };
  auto lo8buf = [&](int t) { return h->lo8[t] ? static_cast<void*>(ws + offs[t] + tensor_hi_bytes(h, t, nb)) : nullptr; };
  const int geom[12] = {h->tile[0], h->tile[1], h->tile[2], eff[0], eff[1], eff[2],
                        h->overlap[0], h->overlap[1], h->overlap[2], grid[0], grid[1], grid[2]};
  // assemble's crop_size indexing: crop_size (x,y,z) is read as [2], [0], [1] for z, y, x (image_transforms.py:511)
  const int crop_zyx[3] = {h->cfg.overlap_xyz[2], h->cfg.overlap_xyz[0], h->cfg.overlap_xyz[1]};
  const int fmt = h->cfg.ab_format;

  auto conv = [&](int l, int NT, int t0, int t1, int tout) -> int {
    const LayerDef& L = kLayers[l];
    const PackedLayer& P = h->layers[l];
    ConvSpec s = P.spec;
    s.split0 = h->split[t0];
    s.split1 = t1 >= 0 ? h->split[t1] : 0;
    ConvLaunch a;
    a.src0 = buf(t0);
    a.src1 = t1 >= 0 ? buf(t1) : nullptr;
    a.NT = NT; a.wpack = P.w; a.wpack_bytes = P.w_bytes; a.bias = P.bias; a.relu = 1;
    a.out = buf(tout);
    a.out_lo8 = lo8buf(tout);
    a.src_lo8 = lo8buf(s.terms == 6 ? t1 : t0);
    a.obase = 0;
    a.out_split = h->split[tout];
    a.out_lo_off = L.cout;
    const long long cp = (a.out_split ? 2ll : 1ll) * L.cout;
    if (L.kind == 'u') {
      a.osN = 8ll * s.D * s.H * s.W * cp; a.osD = 8ll * s.H * s.W * cp; a.osH = 4ll * s.W * cp; a.osW = 2 * cp;
    } else {
      a.osN = 1ll * s.D * s.H * s.W * cp; a.osD = 1ll * s.H * s.W * cp; a.osH = 1ll * s.W * cp; a.osW = cp;
    }
    int region[4];
    a.region = nullptr;
    if (h->has_region && l >= DC9) {
      const Box& b = h->region[l];
      region[0] = b.lo[0]; region[1] = b.hi[0] - b.lo[0] + 1; region[2] = b.lo[1]; region[3] = b.hi[1] - b.lo[1] + 1;
      a.region = region;
    }
    a.head = nullptr;
    if (a.region && (s.flags & kConvFlagKhShared)) return conv_run_w_box(s, a, h->region[l].lo[2], h->region[l].hi[2], st);
    return conv_run(s, a, st);
  };
  auto pool = [&](int i, int NT) -> int {
    const int tin = kPoolOf[i][0], tout = kPoolOf[i][1];
    const TensorDef& d = kTensors[tin];
    return maxpool2_launch(buf(tin), buf(tout), NT, dims_at(h, d.level, 0), dims_at(h, d.level, 1),
                           dims_at(h, d.level, 2), d.channels, h->split[tin], h->split[tout], fmt, st);
  };

  nvtxRangePushA("oai.seg_forward");
  int rc = 0;
  for (int t0 = 0; t0 < T && !rc; t0 += nb) {
    const int NT = std::min(nb, T - t0);
    StemParams sp;
    sp.vol = vol; sp.VD = vol_dims[0]; sp.VH = vol_dims[1]; sp.VW = vol_dims[2];
    sp.td = geom[0]; sp.th = geom[1]; sp.tw = geom[2];
    sp.ed = geom[3]; sp.eh = geom[4]; sp.ew = geom[5];
    sp.od = geom[6]; sp.oh = geom[7]; sp.ow = geom[8];
    sp.gh = geom[10]; sp.gw = geom[11];
    sp.tile0 = t0; sp.ntiles = NT; sp.c0 = 32; sp.w = h->stem_w; sp.b = h->layers[EC0].bias; sp.out = buf(T_E0);
    sp.fmt = fmt; sp.out_split = h->split[T_E0];
    // networks.py:110-144
    rc = stem_launch(sp, st)                                  // step 0: Partition + ec0
         || conv(EC1, NT, T_E0, -1, T_SYN0)                   // 1
         || pool(0, NT)                                       // 2
         || conv(EC2, NT, T_P0, -1, T_E2)                     // 3
         || conv(EC3, NT, T_E2, -1, T_SYN1)                   // 4
         || pool(1, NT)                                       // 5
         || conv(EC4, NT, T_P1, -1, T_E4)                     // 6
         || conv(EC5, NT, T_E4, -1, T_SYN2)                   // 7
         || pool(2, NT)                                       // 8
         || conv(EC6, NT, T_P2, -1, T_E6)                     // 9
         || conv(EC7, NT, T_E6, -1, T_E7)                     // 10
         || conv(DC9, NT, T_E7, -1, T_D9)                     // 11
         || conv(DC8, NT, T_D9, T_SYN2, T_D8)                 // 12: cat((dc9, syn2))
         || conv(DC7, NT, T_D8, -1, T_D7)                     // 13
         || conv(DC6, NT, T_D7, -1, T_D6)                     // 14
         || conv(DC5, NT, T_D6, T_SYN1, T_D5)                 // 15: cat((dc6, syn1))
         || conv(DC4, NT, T_D5, -1, T_D4)                     // 16
         || conv(DC3, NT, T_D4, -1, T_D3)                     // 17
         || conv(DC2, NT, T_D3, T_SYN0, T_D2);                // 18: cat((dc3, syn0))
    if (rc) break;
    // step 19: dc1 + dc0 + sigmoid (+ >0.5) + assemble, one launch (networks.py:145-148, segmenter.py:121-129)
    const PackedLayer& P = h->layers[DC1];
    ConvSpec s = P.spec;
    s.split0 = h->split[T_D2];
    HeadFuse hd = make_head_fuse(h->cfg.n_classes, h->head_w, h->head_b, out, vol_dims, geom, t0, crop_zyx, out_mode);
    const int region[4] = {geom[6], geom[3], geom[7], geom[4]};   // only the tile interior is ever written
    ConvLaunch a;
    a.src0 = buf(T_D2); a.src1 = nullptr; a.NT = NT; a.wpack = P.w; a.wpack_bytes = P.w_bytes; a.bias = P.bias;
    a.relu = 1; a.out = nullptr; a.obase = a.osN = a.osD = a.osH = a.osW = 0; a.out_split = 0; a.out_lo_off = 0;
    a.region = region; a.head = &hd; a.src_lo8 = lo8buf(T_D2);
    rc = (s.flags & kConvFlagKhShared) ? conv_run_w_box(s, a, geom[8], geom[8] + geom[5] - 1, st) : conv_run(s, a, st);
  }
  nvtxRangePop();
  return rc;
}
