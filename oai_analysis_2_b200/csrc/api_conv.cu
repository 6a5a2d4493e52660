// C-ABI entry points of the tcgen05 implicit-GEMM conv: geometry planner, weight packer, launcher.
#include "../../include/oai_b200.h"
#include "api_common.h"
#include "conv_api.h"
#include "conv_igemm.cuh"

#include <cuda_bf16.h>
#include <cuda_fp16.h>

#include <cstring>
#include <vector>

namespace oai {

cudaError_t conv_igemm_launch(const ConvIgemmParams& p, const CUtensorMap& tm0, const CUtensorMap& tm1, int num_sms,
                              cudaStream_t stream);
cudaError_t conv_overflow_count(unsigned int* count, bool reset, cudaStream_t stream);

namespace {

constexpr int kFlagForcePerTap = 1;
constexpr int kFlagBaseOffFormula = 2;  // debug: descriptor base_offset = (addr>>7)&7 (measured WRONG on B200)
constexpr int kFlagForceKd1 = 4;
constexpr int kFlagNoFastPath = 8;
constexpr int kFlagWideN = 16;     // A/B: keep 256-wide N tiles for 3x3x3 layers with cout >= 256 (one kd per weight block)
constexpr int kFlagWideRows = 32;  // A/B: keep 128-byte rows (zero-filled upper half) for a 32-channel source
constexpr int kFlagNoPingPong = 128;  // A/B: k2s2 units use every TMEM column (no accumulator ping-pong)
constexpr int kFlagOneKhRow = 64;  // A/B: one kh row per A stage even where the three-row stage applies
constexpr size_t kSmemBudget = 232448 - 1024 - 48 * 8 - 2112 - 2048;  // 227 KB minus alignment slack, barriers, head weights, bias

// One K chunk of the implicit GEMM: a TMA box of 64 (32) channels starting at channel cc of source `src`.
// wsel picks the weight image multiplied with it: 0 = 16-bit weights rounded with error feedback, 1 = plain hi half,
// 2 = lo half (w - hi); dup: the chunk runs over the [hi | lo] planes of a split tensor (virtual channel v < 2C maps
// to input channel v mod C), otherwise over the first C channels only.
struct Chunk {
  int src, cc, wsel, dup;
};

struct Plan {
  int mode, kd_per_block, R, Rd, up_groups, nhalf, cph, nblk, nch, k16, row_bytes, TW, TH, n_wbuf, n_astage;
  int nkh;   // kh rows per A stage at launch (the packed image is the same: three consecutive kh blocks form one)
  int pingpong;  // kModeUp2: accumulator halves alternate between consecutive units
  int stationary;  // one shared-memory buffer per weight block of a (N split, tap group); units ordered group-major
  uint32_t wblock_bytes, astage_bytes, astage_stride;
  Chunk chunks[kMaxChunks];
};

// which sources a term code reads as fp16 hi + lo pairs: 2 / 3 both, 4 the second (the decoder's skip connection) only,
// 5 the first only
inline bool split_src(int terms, int src) {
  return terms == 2 || terms == 3 || (terms == 4 && src == 1) || (terms == 5 && src == 0);
}

int build_chunks(const ConvSpec& s, Plan* pl) {
  int n = 0;
  const int cs[2] = {s.c0, s.c1};
  for (int src = 0; src < 2; ++src) {
    const int c = cs[src];
    if (c == 0) continue;
    const bool spl = split_src(s.terms, src);
    const int wide = spl ? 2 * c : c;
    for (int j = 0; j * 64 < wide; ++j) {
      OAI_REQUIRE(n < kMaxChunks, "conv plan: more than %d K chunks", kMaxChunks);
      pl->chunks[n++] = Chunk{src, j * 64, s.terms == 3 ? 1 : 0, spl ? 1 : 0};
    }
    if (s.terms == 3)
      for (int j = 0; j * 64 < c; ++j) {
        OAI_REQUIRE(n < kMaxChunks, "conv plan: more than %d K chunks", kMaxChunks);
        pl->chunks[n++] = Chunk{src, j * 64, 2, 0};
      }
  }
  pl->nch = n;
  return 0;
}

// tw: M tile width of a kh-shared layer (8, 16 or 32); the packed weights do not depend on it
int make_plan(const ConvSpec& s, Plan* pl, int d_cnt = 0, int tw = 32) {
  const int D = s.D, H = s.H, W = s.W, c0 = s.c0, c1 = s.c1, cout = s.cout, pointwise = s.kind, flags = s.flags;
  OAI_REQUIRE(D > 0 && H > 0 && W > 0 && c0 > 0 && c1 >= 0 && cout > 0, "conv plan: bad dims");
  OAI_REQUIRE(c0 % 8 == 0 && c1 % 8 == 0, "conv plan: channel counts must be multiples of 8 (got %d,%d)", c0, c1);
  OAI_REQUIRE(s.terms >= 1 && s.terms <= 5,
              "conv plan: terms=%d (1 = 16-bit, 2 = split activations, 3 = split both, 4 / 5 = split the second / first "
              "source's activations only)", s.terms);
  OAI_REQUIRE((!split_src(s.terms, 0) || s.split0) && (!split_src(s.terms, 1) || c1 == 0 || s.split1),
              "conv plan: terms=%d needs the split sources stored as [hi | lo] planes", s.terms);
  OAI_REQUIRE(s.terms < 4 || c1 > 0, "conv plan: terms=%d is for two-source layers", s.terms);
  OAI_REQUIRE((!s.split0 || c0 % 32 == 0) && (!s.split1 || c1 % 64 == 0) && (c1 == 0 || c0 % 64 == 0),
              "conv plan: split / concatenated sources need 64-channel multiples (got %d,%d)", c0, c1);
  pl->TW = W < 128 ? W : 128;
  pl->TH = 128 / pl->TW;
  if (!(flags & kConvFlagKhShared)) {
    OAI_REQUIRE(128 % pl->TW == 0 && W % pl->TW == 0, "conv plan: W=%d must divide or be a multiple of 128", W);
    OAI_REQUIRE(H % pl->TH == 0, "conv plan: H=%d not a multiple of the %d-row M tile", H, pl->TH);
  }
  // 3x3x3 layers split cout into 128-wide N tiles: each tile then stacks the three kd taps of an input slice (N = 256 +
  // 128) and keeps R = 4 accumulators, which halves the weight bytes streamed per output compared with a 256-wide
  // tile limited to R = 2 by the 512 TMEM columns.  Pointwise layers keep 256-wide tiles.
  const int ntile = (!pointwise && cout > 128 && !(flags & kFlagWideN)) ? 128 : 256;
  pl->nhalf = (cout + ntile - 1) / ntile;
  OAI_REQUIRE(cout % pl->nhalf == 0, "conv plan: cout=%d not divisible into %d N splits", cout, pl->nhalf);
  pl->cph = cout / pl->nhalf;
  OAI_REQUIRE(pl->cph % 32 == 0, "conv plan: cout per split (%d) must be a multiple of 32", pl->cph);
  OAI_REQUIRE(cout <= 512, "conv plan: cout=%d exceeds the 512-float bias staging area", cout);
  if (d_cnt <= 0) d_cnt = D;
  // as many accumulators as TMEM holds; the last d-group of a region may be partial
  int R = 512 / pl->cph < 8 ? 512 / pl->cph : 8;
  if (R > d_cnt) R = d_cnt;
  pl->R = R;
  pl->Rd = R;
  pl->up_groups = 1;
  pl->pingpong = 0;
  if (build_chunks(s, pl)) return 1;
  const int c0v = split_src(s.terms, 0) ? 2 * c0 : c0;  // channels the first source's chunks run over
  pl->k16 = (c1 == 0 && c0v <= 32) ? (c0v <= 16 ? 1 : 2) : 4;
  // a single 32-channel source keeps 64-byte rows (SWIZZLE_64B): half the TMA / shared-memory bytes per voxel
  pl->row_bytes = (c1 == 0 && c0v == 32 && !(flags & kFlagWideRows)) ? 64 : 128;
  const int rb = pl->row_bytes;
  const int nch = pl->nch;
  if (pointwise == 2) {
    // ConvTranspose3d(k2,s2): the unit's accumulators are taps of one M tile
    pl->mode = kModeUp2;
    pl->kd_per_block = 1;
    pl->R = 512 / pl->cph < 8 ? 512 / pl->cph : 8;
    // All accumulators of a k2s2 unit complete together (one K pass over the input channels), so with every TMEM
    // column in use the next unit's first MMA waits for the whole epilogue.  Half the taps per unit and alternating
    // accumulator halves let the tensor pipe run through the epilogue of the previous unit.
    if (pl->R >= 2 && !(flags & (kFlagNoFastPath | kFlagBaseOffFormula | kFlagNoPingPong))) {
      pl->R /= 2;
      pl->pingpong = 1;
    }
    pl->Rd = 1;
    pl->up_groups = 8 / pl->R;
    pl->wblock_bytes = pl->R * pl->cph * rb;
    pl->nblk = nch;
    pl->n_wbuf = 2;
  } else if (pointwise) {
    pl->mode = kModePointwise;
    pl->kd_per_block = 1;
    pl->wblock_bytes = pl->cph * rb;
    pl->nblk = nch;
    pl->n_wbuf = 3;
  } else if (flags & kConvFlagKhShared) {
    OAI_REQUIRE(pl->cph <= 64 && rb == 128 && (tw == 8 || tw == 16 || tw == 32) && W >= tw && H >= 128 / tw,
                "conv plan: kh-shared mode needs cout <= 64, 64-channel chunks and a grid of at least one %d-wide tile "
                "(cout=%d, %dx%d)", tw, cout, H, W);
    pl->mode = kModeKhShared;
    pl->kd_per_block = 3;
    pl->wblock_bytes = 9 * pl->cph * rb;
    pl->nblk = nch * 3;
    pl->n_wbuf = 2;
    pl->TW = tw;
    pl->TH = 128 / tw;
  } else if (pl->TW == 128 && pl->cph <= 64 && !(flags & kFlagForcePerTap)) {
    pl->mode = kModeRowShared;
    pl->kd_per_block = 3;
    pl->wblock_bytes = 9 * pl->cph * rb;
    pl->nblk = nch * 3;
    pl->n_wbuf = 2;
  } else {
    pl->mode = kModePerTap;
    pl->kd_per_block = (pl->cph <= 128 && !(flags & kFlagForceKd1)) ? 3 : 1;
    pl->wblock_bytes = pl->kd_per_block * pl->cph * rb;
    pl->nblk = nch * (pl->kd_per_block == 3 ? 9 : 27);
    pl->n_wbuf = pl->kd_per_block == 3 ? 2 : 3;
  }
  // A 32-channel row-shared layer (ec1) issues only six MMAs per one-row stage, fewer tensor clocks than the issuing
  // thread needs instructions (DESIGN 4.1): there the stage holds the three kh rows of a slice (18 MMAs) and the whole
  // 27-tap weight image (three consecutive kh blocks of the packed layout, 110 KB) stays resident in shared memory.
  pl->nkh = 1;
  if (pl->mode == kModeRowShared && rb == 64 && nch == 1 &&
      !(flags & (kFlagOneKhRow | kFlagNoFastPath | kFlagBaseOffFormula))) {
    pl->nkh = 3;
    pl->n_wbuf = 1;
  }
  pl->astage_bytes = (pl->mode == kModeRowShared ? 130 : pl->mode == kModeKhShared ? 128 + 2 * pl->TW : 128) * rb * pl->nkh;
  pl->astage_stride = (pl->astage_bytes + 1023u) & ~1023u;
  const size_t wstride = (static_cast<size_t>(pl->wblock_bytes) * pl->nkh + 1023u) & ~size_t(1023);
  // Stationary weights: a k2s2 unit is one K pass over a 128-voxel tile, so streaming its weight blocks per unit costs
  // ~64 B/clk/SM of L2 bandwidth (dc6: 128 KB per 2048-clock unit); when all blocks of a tap group fit beside four A
  // stages they get one buffer each and stay put while the CTA walks its tiles.  The three-row ec1 plan is the same
  // thing with a single group.
  pl->stationary = 0;
  if (pl->nkh == 3) pl->stationary = 1;
  if (pl->mode == kModeUp2 && pl->pingpong && pl->nblk <= 4 && pl->nblk * wstride + 4 * pl->astage_stride <= kSmemBudget) {
    pl->stationary = 1;
    pl->n_wbuf = pl->nblk;
  }
  const size_t left = kSmemBudget - pl->n_wbuf * wstride;
  int ns = static_cast<int>(left / pl->astage_stride);
  if (ns > 8) ns = 8;
  OAI_REQUIRE(ns >= 2, "conv plan: shared memory budget leaves %d A stages", ns);
  pl->n_astage = ns;
  return 0;
}

size_t plan_wpack_bytes(const Plan& pl) {
  return static_cast<size_t>(pl.nhalf) * pl.up_groups * pl.nblk * pl.wblock_bytes;
}

typedef CUresult (*EncodeTiledFn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*,
                                  const cuuint64_t*, const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave,
                                  CUtensorMapSwizzle, CUtensorMapL2promotion, CUtensorMapFloatOOBfill);

EncodeTiledFn encode_fn() {
  static EncodeTiledFn fn = nullptr;
  if (!fn) {
    void* p = nullptr;
    cudaDriverEntryPointQueryResult q;
    if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &p, cudaEnableDefault, &q) == cudaSuccess &&
        q == cudaDriverEntryPointSuccess)
      fn = reinterpret_cast<EncodeTiledFn>(p);
  }
  return fn;
}

// NDHWC 16-bit activation tensor viewed as a rank-5 TMA tensor (C, W, H, D, N); box = (64, bw, bh, 1, 1).
int make_act_tmap(CUtensorMap* tm, const void* base, int C, int W, int H, int D, int N, int bw, int bh, int fmt,
                  int row_bytes = 128) {
  EncodeTiledFn fn = encode_fn();
  OAI_REQUIRE(fn != nullptr, "cuTensorMapEncodeTiled not available from the driver");
  cuuint64_t dims[5] = {(cuuint64_t)C, (cuuint64_t)W, (cuuint64_t)H, (cuuint64_t)D, (cuuint64_t)N};
  cuuint64_t strides[4] = {(cuuint64_t)C * 2, (cuuint64_t)W * C * 2, (cuuint64_t)H * W * C * 2,
                           (cuuint64_t)D * H * W * C * 2};
  cuuint32_t box[5] = {(cuuint32_t)(row_bytes / 2), (cuuint32_t)bw, (cuuint32_t)bh, 1, 1};
  cuuint32_t estr[5] = {1, 1, 1, 1, 1};
  CUresult r = fn(tm, fmt == 0 ? CU_TENSOR_MAP_DATA_TYPE_FLOAT16 : CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 5,
                  const_cast<void*>(base), dims, strides, box, estr, CU_TENSOR_MAP_INTERLEAVE_NONE,
                  row_bytes == 128 ? CU_TENSOR_MAP_SWIZZLE_128B : CU_TENSOR_MAP_SWIZZLE_64B,
                  CU_TENSOR_MAP_L2_PROMOTION_L2_256B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  OAI_REQUIRE(r == CUDA_SUCCESS, "cuTensorMapEncodeTiled failed with %d (C=%d W=%d H=%d D=%d N=%d box %dx%d)", (int)r,
              C, W, H, D, N, bw, bh);
  return 0;
}

inline uint16_t to16(float x, int fmt) {
  if (fmt == 0) {
    __half h = __float2half_rn(x);
    uint16_t u;
    memcpy(&u, &h, 2);
    return u;
  }
  __nv_bfloat16 h = __float2bfloat16_rn(x);
  uint16_t u;
  memcpy(&u, &h, 2);
  return u;
}

// byte offset of element j (16-bit) of row r in a K-major swizzled block: 16-byte chunks are XOR-ed with the row index
// (SWIZZLE_128B: chunk ^= r & 7 over 128-byte rows; SWIZZLE_64B: chunk ^= (r >> 1) & 3 over 64-byte rows)
inline size_t swz_off(int r, int j, int row_bytes) {
  const int chunk = j >> 3;
  const int sw = row_bytes == 128 ? (chunk ^ (r & 7)) : (chunk ^ ((r >> 1) & 3));
  return static_cast<size_t>(r) * row_bytes + (static_cast<size_t>(sw) << 4) + (j & 7) * 2;
}

inline float from16(uint16_t u, int fmt) {
  if (fmt == 0) {
    __half h;
    memcpy(&h, &u, 2);
    return __half2float(h);
  }
  __nv_bfloat16 h;
  memcpy(&h, &u, 2);
  return __bfloat162float(h);
}

// Optional per-launch timing of the conv kernel (CUDA events on the launch stream) for bench.py's roofline line.
struct ProfEntry {
  cudaEvent_t a, b;
  double flops;       // algorithmic: every MAC the reference executes for this layer
  double exec_flops;  // MACs actually issued to the tensor pipe (dead-halo rows skipped, split-precision terms counted)
};

// Inside a stream capture (the per-knee CUDA graph) the profiling events become external event-record nodes: every
// replay re-records them, so oai_profile_end reports the conv launches of the most recent replay.
inline void prof_record(cudaEvent_t ev, cudaStream_t st) {
  cudaStreamCaptureStatus cs = cudaStreamCaptureStatusNone;
  cudaStreamIsCapturing(st, &cs);
  cudaEventRecordWithFlags(ev, st, cs == cudaStreamCaptureStatusActive ? cudaEventRecordExternal : cudaEventRecordDefault);
}
std::vector<ProfEntry> g_prof;
size_t g_prof_used = 0;
bool g_prof_on = false;

}  // namespace

size_t conv_wpack_bytes(const ConvSpec& s) {
  Plan pl;
  if (make_plan(s, &pl)) return 0;
  return plan_wpack_bytes(pl);
}

// w: float32 in conv orientation [cout][c0+c1][taps] with taps = 27 (kind 0), 1 (kind 1) or 8 (kind 2, tap = a*4+b*2+c).
int conv_pack_weights(const ConvSpec& s, const float* w, void* dst, size_t dst_bytes) {
  Plan pl;
  if (make_plan(s, &pl)) return 1;
  const size_t need = plan_wpack_bytes(pl);
  OAI_REQUIRE(dst_bytes >= need, "pack: dst holds %zu bytes, need %zu", dst_bytes, need);
  const int cout = s.cout, cin = s.c0 + s.c1, fmt = s.fmt;
  const int ktaps = s.kind == 0 ? 27 : (s.kind == 1 ? 1 : 8);
  uint8_t* out = static_cast<uint8_t*>(dst);
  memset(out, 0, need);
  // Three 16-bit images of the weights.
  //  q[0]: rounded with error feedback along the taps of each (co, ci) filter: the rounding residual of one tap is
  //        carried into the next, so the 27 rounding errors of a filter sum to (almost) zero.  On smooth inputs -- where
  //        all taps see nearly the same activation -- this cancels the systematic part of the weight-quantisation error.
  //        (The taps of a k2s2 transposed conv feed different outputs: plain rounding there.)
  //  q[1], q[2]: hi = rn16(w) and lo = rn16(w - hi) of the three-term split (hi + lo carries ~22 mantissa bits).
  const size_t nw = static_cast<size_t>(cout) * cin * ktaps;
  std::vector<uint16_t> q[3];
  q[0].resize(nw);
  if (s.terms == 3) { q[1].resize(nw); q[2].resize(nw); }
  for (size_t f = 0; f < static_cast<size_t>(cout) * cin; ++f) {
    double carry = 0.0;
    for (int t = 0; t < ktaps; ++t) {
      const double v = static_cast<double>(w[f * ktaps + t]) + (s.kind == 2 ? 0.0 : carry);
      const uint16_t h = to16(static_cast<float>(v), fmt);
      q[0][f * ktaps + t] = h;
      carry = v - static_cast<double>(from16(h, fmt));
      if (s.terms == 3) {
        const float wf = w[f * ktaps + t];
        const uint16_t hi = to16(wf, fmt);
        q[1][f * ktaps + t] = hi;
        q[2][f * ktaps + t] = to16(wf - from16(hi, fmt), fmt);
      }
    }
  }
  const int cs[2] = {s.c0, s.c1};
  const int ngroups = pl.up_groups;
  for (int nh = 0; nh < pl.nhalf; ++nh)
    for (int tg = 0; tg < ngroups; ++tg)
      for (int b = 0; b < pl.nblk; ++b) {
        uint8_t* blk = out + ((static_cast<size_t>(nh) * ngroups + tg) * pl.nblk + b) * pl.wblock_bytes;
        // decode the block exactly as the kernel does: chunk c, and the taps whose rows are stacked in it
        int c, kh = 0, kw0 = 0, nkw = 1, kdlo = 0, nkd = 1;
        const bool kh_inner = pl.mode == kModeKhShared;   // the three sub-blocks step kh instead of kw
        if (pl.mode == kModeRowShared) {
          c = b / 3; kh = b % 3; nkw = 3; nkd = 3;
        } else if (kh_inner) {
          c = b / 3; kw0 = b % 3; nkw = 3; nkd = 3;
        } else if (pl.mode == kModePerTap && pl.kd_per_block == 3) {
          c = b / 9; const int r = b % 9; kh = r / 3; kw0 = r % 3; nkd = 3;
        } else if (pl.mode == kModePerTap) {
          c = b / 27; const int r = b % 27; kh = r / 9; kw0 = (r / 3) % 3; kdlo = r % 3;
        } else {
          c = b;
        }
        const Chunk& ck = pl.chunks[c];
        const int csrc = cs[ck.src], cbase = ck.src == 0 ? 0 : s.c0;
        const std::vector<uint16_t>& qq = q[ck.wsel];
        const int nstack = pl.mode == kModeUp2 ? pl.R : nkd;
        for (int kwi = 0; kwi < nkw; ++kwi)
          for (int ti = 0; ti < nstack; ++ti) {
            int tap;
            if (pl.mode == kModeUp2) tap = tg * pl.R + ti;
            else if (s.kind == 1) tap = 0;
            else if (kh_inner) tap = ((kdlo + nkd - 1 - ti) * 3 + kh + kwi) * 3 + kw0;
            else tap = ((kdlo + nkd - 1 - ti) * 3 + kh) * 3 + kw0 + kwi;
            for (int co = 0; co < pl.cph; ++co) {
              const int r = (kwi * nstack + ti) * pl.cph + co;
              const uint16_t* wrow = qq.data() + (static_cast<size_t>(nh * pl.cph + co) * cin) * ktaps;
              for (int j = 0; j < 64 && j * 2 < pl.row_bytes; ++j) {
                const int v = ck.cc + j;
                if (v >= (ck.dup ? 2 * csrc : csrc)) break;
                const int ci = cbase + (ck.dup ? v % csrc : v);
                const uint16_t h = wrow[static_cast<size_t>(ci) * ktaps + tap];
                memcpy(blk + swz_off(r, j, pl.row_bytes), &h, 2);
              }
            }
          }
      }
  return 0;
}

int conv_run(const ConvSpec& s, const ConvLaunch& a, cudaStream_t st) {
  const int D = s.D, H = s.H, W = s.W, c0 = s.c0, c1 = s.c1, cout = s.cout;
  // region = {d_lo, d_cnt, h_lo, h_cnt} (+ a.w_lo, a.w_cnt): the output sub-box to compute.  Everything outside is dead
  // halo the caller never reads.  Without a w range, rows are computed whole and the h range is widened to whole
  // M-tile rows; a kh-shared layer places its tiles from (h_lo, w_lo) instead.
  const bool kh_shared = (s.flags & kConvFlagKhShared) != 0;
  int d_lo = 0, d_cnt = D, h_lo = 0, h_cnt = H, w_lo = 0, w_cnt = W;
  if (a.region) {
    d_lo = a.region[0]; d_cnt = a.region[1]; h_lo = a.region[2]; h_cnt = a.region[3];
    OAI_REQUIRE(d_lo >= 0 && d_cnt >= 1 && d_lo + d_cnt <= D && h_lo >= 0 && h_cnt >= 1 && h_lo + h_cnt <= H,
                "conv: region [%d,+%d)x[%d,+%d) outside %dx%d", d_lo, d_cnt, h_lo, h_cnt, D, H);
  }
  if (a.w_cnt) {
    w_lo = a.w_lo; w_cnt = a.w_cnt;
    OAI_REQUIRE(kh_shared, "conv: a w range needs a layer packed for kh-shared mode");
    OAI_REQUIRE(w_lo >= 0 && w_cnt >= 1 && w_lo + w_cnt <= W, "conv: w range [%d,+%d) outside W=%d", w_lo, w_cnt, W);
  }
  // kh-shared tile width: the fewest M tiles over the box, the widest on a tie (dc1's 96 x 96 box: 72 tiles at every
  // width; 32 x 4 and 8 x 16 tiles measured the same, 7.98 / 7.90 ms, though the 8-wide box is 25 % fewer bytes)
  int tw = 32, ntile = 0;
  if (kh_shared)
    for (int t = 32; t >= 8; t /= 2) {
      if (t > W || 128 / t > H) continue;
      const int n = ((w_cnt + t - 1) / t) * ((h_cnt + 128 / t - 1) / (128 / t));
      if (ntile == 0 || n < ntile) { ntile = n; tw = t; }
    }
  Plan pl;
  if (make_plan(s, &pl, d_cnt, tw)) return 1;
  int tile_h_lo = h_lo, nph = (h_cnt + pl.TH - 1) / pl.TH, npw = (w_cnt + pl.TW - 1) / pl.TW;
  if (!kh_shared) {   // whole M-tile rows of whole-row (or whole-grid-aligned) tiles
    tile_h_lo = h_lo / pl.TH * pl.TH;
    nph = (h_lo + h_cnt + pl.TH - 1) / pl.TH - h_lo / pl.TH;
    npw = W / pl.TW;
  }
  const HeadFuse* head = a.head;
  OAI_REQUIRE(a.src0 && a.wpack && a.bias, "conv: null pointer");
  OAI_REQUIRE(!head || (pl.cph == 64 && pl.nhalf == 1), "conv head: the fused head needs a 64-channel layer");
  OAI_REQUIRE((c1 == 0) == (a.src1 == nullptr), "conv: src1/c1 mismatch");
  const size_t need = plan_wpack_bytes(pl);
  OAI_REQUIRE(a.wpack_bytes == need, "conv: packed weights are %zu bytes, geometry needs %zu", a.wpack_bytes, need);
  OAI_REQUIRE(a.obase % 16 == 0 && a.osN % 16 == 0 && a.osD % 16 == 0 && a.osH % 16 == 0 && a.osW % 16 == 0 &&
                  a.out_lo_off % 16 == 0 && (head || (reinterpret_cast<uintptr_t>(a.out) & 31) == 0),
              "conv: output base and strides must keep 32-byte alignment");
  OAI_REQUIRE(!(head && a.out_split), "conv head: the fused head writes class maps, not a split activation");

  ConvIgemmParams p;
  memset(&p, 0, sizeof(p));
  p.NT = a.NT; p.D = D; p.H = H; p.W = W;
  p.TW = pl.TW; p.TH = pl.TH; p.R = pl.R;
  p.cout = pl.cph; p.nhalf = pl.nhalf;
  p.nchunks = pl.nch; p.k16_steps = pl.k16; p.row_bytes = pl.row_bytes;
  for (int c = 0; c < pl.nch; ++c) {
    p.chunk_src[c] = static_cast<uint8_t>(pl.chunks[c].src);
    p.chunk_cc[c] = static_cast<uint16_t>(pl.chunks[c].cc);
  }
  p.mode = pl.mode; p.kd_per_block = pl.kd_per_block; p.nblk = pl.nblk / pl.nkh;
  p.wblock_bytes = pl.wblock_bytes * pl.nkh; p.n_wbuf = pl.n_wbuf; p.n_astage = pl.n_astage;
  p.nkh = pl.nkh;
  p.acc_pingpong = pl.pingpong;
  p.w_stationary = pl.stationary;
  p.astage_bytes = pl.astage_bytes; p.astage_stride = pl.astage_stride;
  p.ab_format = s.fmt; p.relu = a.relu;
  p.base_off_mode = (s.flags & kFlagBaseOffFormula) ? 1 : 0;
  p.no_fast_path = (s.flags & kFlagNoFastPath) ? 1 : 0;
  p.wpack = static_cast<const uint8_t*>(a.wpack);
  p.bias = a.bias;
  p.out = a.out;
  p.obase = a.obase; p.osN = a.osN; p.osD = a.osD; p.osH = a.osH; p.osW = a.osW;
  p.out_split = a.out_split; p.out_lo_off = a.out_lo_off;
  p.d_lo = d_lo; p.d_cnt = d_cnt; p.h_lo = tile_h_lo; p.nph = nph; p.w_lo = kh_shared ? w_lo : 0; p.npw = npw;
  p.Rd = pl.Rd; p.up_groups = pl.up_groups;
  p.nunits = a.NT * ((d_cnt + pl.Rd - 1) / pl.Rd) * (nph * npw) * pl.up_groups * pl.nhalf;
  if (pl.mode == kModeUp2) {
    // tap (a,b,c) lands on voxel (2z+a, 2y+b, 2x+c): osW is the element pitch of TWO output voxels (set by the caller)
    const long long vox = a.osW / 2;
    for (int t = 0; t < 8; ++t)
      p.tap_off[t] = ((static_cast<long long>(t >> 2) * 2 * H + ((t >> 1) & 1)) * 2 * W + (t & 1)) * vox;
  }
  if (head) p.head = *head;

  OAI_REQUIRE(pl.mode != kModeUp2 || (c1 == 0 && !head), "conv: up2 mode takes one source and no fused head");
  const int bw = pl.mode == kModeRowShared ? 130 : pl.TW;
  const int bh = pl.mode == kModeKhShared ? pl.TH + 2 : pl.TH * pl.nkh;
  CUtensorMap tm0, tm1;
  if (make_act_tmap(&tm0, a.src0, s.split0 ? 2 * c0 : c0, W, H, D, a.NT, bw, bh, s.fmt, pl.row_bytes)) return 1;
  if (a.src1) {
    if (make_act_tmap(&tm1, a.src1, s.split1 ? 2 * c1 : c1, W, H, D, a.NT, bw, bh, s.fmt)) return 1;
  } else {
    tm1 = tm0;
  }
  ProfEntry* pe = nullptr;
  if (g_prof_on) {
    if (g_prof_used == g_prof.size()) {
      ProfEntry ne;
      if (cudaEventCreate(&ne.a) != cudaSuccess || cudaEventCreate(&ne.b) != cudaSuccess)
        return fail("conv profile: cannot create events");
      g_prof.push_back(ne);
    }
    pe = &g_prof[g_prof_used++];
    const double taps = s.kind == 0 ? 27.0 : (s.kind == 1 ? 1.0 : 8.0);
    pe->flops = 2.0 * a.NT * D * H * W * static_cast<double>(cout) * (c0 + c1) * taps * a.flop_share;
    // issued to the tensor pipe: computed M tiles x every K chunk listed (split-precision terms included)
    pe->exec_flops = 2.0 * a.NT * static_cast<double>(d_cnt) * nph * npw * 128 * static_cast<double>(cout) * taps *
                     (static_cast<double>(pl.nch) * pl.k16 * 16);
    prof_record(pe->a, st);
  }
  cudaError_t e = conv_igemm_launch(p, tm0, tm1, num_sms(), st);
  if (pe) prof_record(pe->b, st);
  g_launches.fetch_add(1, std::memory_order_relaxed);
  return check_cuda(e, "conv_igemm launch");
}

}  // namespace oai

using namespace oai;

namespace {
ConvSpec spec_of(int D, int H, int W, int c0, int c1, int cout, int pointwise, int ab_format, int flags) {
  ConvSpec s;
  s.D = D; s.H = H; s.W = W; s.c0 = c0; s.c1 = c1; s.split0 = 0; s.split1 = 0; s.cout = cout; s.kind = pointwise;
  s.terms = 1; s.fmt = ab_format; s.flags = flags;
  return s;
}
}  // namespace

extern "C" int oai_conv3d_igemm_plan(int D, int H, int W, int c0, int c1, int cout, int pointwise, int flags,
                                     int* plan) {
  int full[10];
  if (oai_conv3d_igemm_plan_ex(D, H, W, c0, c1, cout, pointwise, 1, flags, full)) return 1;
  for (int i = 0; i < 9; ++i) plan[i] = full[i];
  return 0;
}

extern "C" int oai_conv3d_igemm_plan_ex(int D, int H, int W, int c0, int c1, int cout, int pointwise, int terms,
                                        int flags, int* plan) {
  Plan pl;
  ConvSpec s = spec_of(D, H, W, c0, c1, cout, pointwise, 0, flags);
  s.terms = terms;
  s.split0 = terms > 1;
  s.split1 = terms > 1 && c1 > 0;
  if (make_plan(s, &pl)) return 1;
  plan[0] = pl.mode;
  plan[1] = pl.mode == kModeUp2 ? pl.up_groups : pl.kd_per_block;
  plan[2] = pl.R;
  plan[3] = pl.nhalf;
  plan[4] = pl.cph;
  plan[5] = pl.nblk;
  plan[6] = static_cast<int>(pl.wblock_bytes);
  plan[7] = pl.nch;
  plan[8] = pl.row_bytes;
  plan[9] = static_cast<int>(plan_wpack_bytes(pl) >> 4);  // total packed size in 16-byte units
  return 0;
}

extern "C" int oai_pack_conv_weights(const float* w, int cout, int c0, int c1, int D, int H, int W, int pointwise,
                                     int ab_format, int flags, void* dst, size_t dst_bytes) {
  return conv_pack_weights(spec_of(D, H, W, c0, c1, cout, pointwise, ab_format, flags), w, dst, dst_bytes);
}

extern "C" int oai_pack_conv_weights_ex(const float* w, int cout, int c0, int c1, int D, int H, int W, int pointwise,
                                        int terms, int ab_format, int flags, void* dst, size_t dst_bytes) {
  ConvSpec s = spec_of(D, H, W, c0, c1, cout, pointwise, ab_format, flags);
  s.terms = terms;
  s.split0 = terms > 1;
  s.split1 = terms > 1 && c1 > 0;
  return conv_pack_weights(s, w, dst, dst_bytes);
}

static int conv_common(const void* src0, int c0, const void* src1, int c1, int NT, int D, int H, int W,
                       const void* wpack, size_t wpack_bytes, const float* bias, int cout, int pointwise, int relu,
                       int ab_format, void* out, long long obase, long long osN, long long osD, long long osH,
                       long long osW, int flags, const HeadFuse* head, const int* region, void* stream) {
  ConvLaunch a;
  a.src0 = src0; a.src1 = src1; a.NT = NT; a.wpack = wpack; a.wpack_bytes = wpack_bytes; a.bias = bias; a.relu = relu;
  a.out = out; a.obase = obase; a.osN = osN; a.osD = osD; a.osH = osH; a.osW = osW; a.out_split = 0; a.out_lo_off = 0;
  a.region = region; a.head = head;
  return conv_run(spec_of(D, H, W, c0, c1, cout, pointwise, ab_format, flags), a, static_cast<cudaStream_t>(stream));
}

extern "C" int oai_conv3d_igemm(const void* src0, int c0, const void* src1, int c1, int NT, int D, int H, int W,
                                const void* wpack, size_t wpack_bytes, const float* bias, int cout, int pointwise,
                                int relu, int ab_format, void* out, long long obase, long long osN, long long osD,
                                long long osH, long long osW, int flags, void* stream) {
  OAI_REQUIRE(out != nullptr, "conv: null output");
  return conv_common(src0, c0, src1, c1, NT, D, H, W, wpack, wpack_bytes, bias, cout, pointwise, relu, ab_format, out,
                     obase, osN, osD, osH, osW, flags, nullptr, nullptr, stream);
}

extern "C" int oai_conv3d_igemm_region(const void* src0, int c0, const void* src1, int c1, int NT, int D, int H, int W,
                                       const void* wpack, size_t wpack_bytes, const float* bias, int cout,
                                       int pointwise, int relu, int ab_format, void* out, long long obase,
                                       long long osN, long long osD, long long osH, long long osW, int flags,
                                       const int* region, void* stream) {
  OAI_REQUIRE(out != nullptr && region != nullptr, "conv region: null pointer");
  return conv_common(src0, c0, src1, c1, NT, D, H, W, wpack, wpack_bytes, bias, cout, pointwise, relu, ab_format, out,
                     obase, osN, osD, osH, osW, flags, nullptr, region, stream);
}

// Split-precision form: sources stored as [hi | lo] planes (in_split), `terms` K-concatenated products, optional
// [hi | lo] output.  The output tensor is dense NDHWC with cout (or 2*cout when out_split) channels per voxel.
extern "C" int oai_conv3d_igemm_ex(const void* src0, int c0, const void* src1, int c1, int in_split, int NT, int D,
                                   int H, int W, const void* wpack, size_t wpack_bytes, const float* bias, int cout,
                                   int pointwise, int relu, int ab_format, int terms, void* out, int out_split,
                                   int flags, const int* region, void* stream) {
  OAI_REQUIRE(out != nullptr, "conv: null output");
  OAI_REQUIRE(pointwise == 0 || pointwise == 1 || pointwise == 2, "conv: pointwise=%d", pointwise);
  ConvSpec s = spec_of(D, H, W, c0, c1, cout, pointwise, ab_format, flags);
  s.terms = terms;
  s.split0 = in_split;
  s.split1 = in_split && c1 > 0;
  const long long cp = out_split ? 2ll * cout : cout;
  ConvLaunch a;
  a.src0 = src0; a.src1 = src1; a.NT = NT; a.wpack = wpack; a.wpack_bytes = wpack_bytes; a.bias = bias; a.relu = relu;
  a.out = out; a.obase = 0; a.out_split = out_split; a.out_lo_off = cout; a.region = region; a.head = nullptr;
  if (pointwise == 2) {
    a.osN = 8ll * D * H * W * cp; a.osD = 8ll * H * W * cp; a.osH = 4ll * W * cp; a.osW = 2 * cp;
  } else {
    a.osN = 1ll * D * H * W * cp; a.osD = 1ll * H * W * cp; a.osH = 1ll * W * cp; a.osW = cp;
  }
  return conv_run(s, a, static_cast<cudaStream_t>(stream));
}

extern "C" int oai_conv3d_igemm_head(const void* src0, int c0, const void* src1, int c1, int NT, int D, int H, int W,
                                     const void* wpack, size_t wpack_bytes, const float* bias, int ab_format,
                                     int ncls, const float* head_w, const float* head_b, float* out,
                                     const int* vol_dims, const int* geom, int tile0, const int* crop_zyx,
                                     int out_mode, int flags, void* stream) {
  OAI_REQUIRE(head_w && head_b && out && vol_dims && geom && crop_zyx, "conv head: null pointer");
  OAI_REQUIRE(ncls >= 1 && ncls <= 8, "conv head: ncls=%d unsupported", ncls);
  OAI_REQUIRE(geom[0] == D && geom[1] == H && geom[2] == W, "conv head: tile geometry does not match the layer");
  // only the tile interior is ever written, so only the interior rows are computed
  const int region[4] = {geom[6], geom[3], geom[7], geom[4]};
  HeadFuse hd = make_head_fuse(ncls, head_w, head_b, out, vol_dims, geom, tile0, crop_zyx, out_mode);
  return conv_common(src0, c0, src1, c1, NT, D, H, W, wpack, wpack_bytes, bias, 64, 0, 1, ab_format, nullptr, 0, 0, 0,
                     0, 0, flags, &hd, region, stream);
}

extern "C" int oai_conv_overflow_count(long long* count, int reset, void* stream) {
  OAI_REQUIRE(count != nullptr, "conv_overflow_count: null pointer");
  unsigned int c = 0;
  if (int rc = check_cuda(conv_overflow_count(&c, reset != 0, static_cast<cudaStream_t>(stream)), "conv_overflow_count"))
    return rc;
  *count = c;
  return 0;
}

extern "C" int oai_profile_begin(void) {
  g_prof_used = 0;
  g_prof_on = true;
  return 0;
}

extern "C" int oai_profile_end(double* conv_ms, long long* conv_launches, double* conv_flops,
                               double* conv_exec_flops) {
  g_prof_on = false;
  double ms = 0, fl = 0, xfl = 0;
  for (size_t i = 0; i < g_prof_used; ++i) {
    if (int rc = check_cuda(cudaEventSynchronize(g_prof[i].b), "conv profile: event sync")) return rc;
    float t = 0;
    if (int rc = check_cuda(cudaEventElapsedTime(&t, g_prof[i].a, g_prof[i].b), "conv profile: elapsed")) return rc;
    ms += t;
    fl += g_prof[i].flops;
    xfl += g_prof[i].exec_flops;
  }
  if (conv_ms) *conv_ms = ms;
  if (conv_launches) *conv_launches = static_cast<long long>(g_prof_used);
  if (conv_flops) *conv_flops = fl;
  if (conv_exec_flops) *conv_exec_flops = xfl;
  g_prof_used = 0;
  return 0;
}

/* per-launch detail of the same profile (call before oai_profile_end): ms / flops / exec_flops of launch i */
extern "C" int oai_profile_entry(int i, double* ms, double* flops, double* exec_flops) {
  OAI_REQUIRE(i >= 0 && static_cast<size_t>(i) < g_prof_used, "conv profile: entry %d of %zu", i, g_prof_used);
  if (int rc = check_cuda(cudaEventSynchronize(g_prof[i].b), "conv profile: event sync")) return rc;
  float t = 0;
  if (int rc = check_cuda(cudaEventElapsedTime(&t, g_prof[i].a, g_prof[i].b), "conv profile: elapsed")) return rc;
  if (ms) *ms = t;
  if (flops) *flops = g_prof[i].flops;
  if (exec_flops) *exec_flops = g_prof[i].exec_flops;
  return 0;
}


// ---------------------------------------------------------------------------------------------- ConvTranspose3d k2 s2
extern "C" int oai_pack_convt2_weights(const float* w, int cout, int cin, int D, int H, int W, int ab_format,
                                       void* dst, size_t dst_bytes) {
  return conv_pack_weights(spec_of(D, H, W, cin, 0, cout, 2, ab_format, 0), w, dst, dst_bytes);
}

extern "C" int oai_convt2_igemm(const void* src, int cin, int NT, int D, int H, int W, const void* wpack,
                                size_t wpack_bytes, const float* bias, int cout, int relu, int ab_format, void* out,
                                const int* region, void* stream) {
  OAI_REQUIRE(out != nullptr, "convt2: null output");
  const long long c = cout;
  return conv_common(src, cin, nullptr, 0, NT, D, H, W, wpack, wpack_bytes, bias, cout, 2, relu, ab_format, out, 0,
                     8ll * D * H * W * c, 8ll * H * W * c, 4ll * W * c, 2 * c, 0, nullptr, region, stream);
}
