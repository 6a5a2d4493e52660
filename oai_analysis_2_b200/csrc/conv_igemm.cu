// tcgen05 implicit-GEMM 3-D convolution for sm_100a (B200).
//
// Replaces the cuDNN/oneDNN calls behind nn.Conv3d(k3,p1), nn.ConvTranspose3d(k3,s1,p1) (== conv with flipped
// weights) and nn.ConvTranspose3d(k2,s2) (== 8 pointwise GEMMs + pixel shuffle) of the reference segmentation UNet
// (reference: oai_analysis/segmentation/networks.py:80-107 layer builders, :109-149 forward).
//
// Design (input-tile stationary, taps stacked along N):
//   * activations are NDHWC 16-bit; one M tile = 128 voxels of one d-slice (TH x TW patch);
//   * a unit owns R consecutive output d-slices of one patch: R accumulators of [128 x cout] fp32 in TMEM
//     (R*cout <= 512 columns);
//   * an input tile (slice d') feeds the outputs d'-1, d', d'+1 through the taps kd = 2,1,0, whose weight rows sit
//     next to each other in shared memory, so ONE tcgen05.mma with N = 3*cout (<=256) updates three adjacent
//     accumulators while reading the A tile from shared memory once;
//   * in row-shared mode (full-resolution level, TW = W = 128) the A tile is a 130-voxel row (w halo, TMA zero fill)
//     and the three kw taps are the same buffer shifted by one 128-byte row;
//   * kh-shared mode swaps the roles of kh and kw: the M tile is a TH x TW sub-box placed anywhere in the slice, the
//     A tile of one kw is a (TH + 2) x TW box and the three kh taps are the same buffer shifted by TW rows;
//   * weights arrive as pre-swizzled blocks by cp.async.bulk and stay resident while the unit walks its input
//     slices; the K loop can read two sources (decoder skip connection) so torch.cat is never materialised;
//   * warp roles: 0 = TMA producer (activations), 1 = bulk producer (weights), 2 = MMA issuer + TMEM owner,
//     4..7 = epilogue (TMEM -> registers -> bias/ReLU -> 16-bit NDHWC store, overlapped per accumulator).
#include "conv_igemm.cuh"
#include "ptx.cuh"

#include <cuda_bf16.h>
#include <cuda_fp16.h>

namespace oai {

namespace {

constexpr int kThreads = 384;   // warps 0-2: producers + MMA issuer, 3: idle, 4-11: two epilogue groups
constexpr int kEpiGroups = 2;  // epilogue group g (warps 4+4g .. 7+4g) drains the accumulators a = g, g+2, ...
constexpr int kTmemCols = 512;

// activations that left the fp16 range (|x| > 65504 before rounding) since the last reset: a real checkpoint with large
// folded-BatchNorm scales would otherwise turn into inf / NaN silently
__device__ unsigned int g_fp16_overflow = 0;

struct BlockInfo {
  int c, kh, kw, kdlo, nkd;
  int ns;  // taps stacked along N in this block's weight rows (== nkd except kModeUp2)
};

__device__ __forceinline__ BlockInfo decode_block(const ConvIgemmParams& p, int b) {
  BlockInfo bi;
  if (p.mode == kModeRowShared) {
    bi.c = p.nkh == 3 ? b : b / 3;
    bi.kh = p.nkh == 3 ? 0 : b % 3;   // three-row stages start at row h - 1 and hold kh = 0, 1, 2
    bi.kw = 0;
    bi.kdlo = 0;
    bi.nkd = 3;
  } else if (p.mode == kModeKhShared) {
    bi.c = b / 3;
    bi.kh = 0;   // the box starts at row h0 - 1 and holds kh = 0, 1, 2
    bi.kw = b % 3;
    bi.kdlo = 0;
    bi.nkd = 3;
  } else if (p.mode == kModePerTap) {
    if (p.kd_per_block == 3) {
      bi.c = b / 9;
      const int r = b % 9;
      bi.kh = r / 3;
      bi.kw = r % 3;
      bi.kdlo = 0;
      bi.nkd = 3;
    } else {
      bi.c = b / 27;
      const int r = b % 27;
      bi.kh = r / 9;
      bi.kw = (r / 3) % 3;
      bi.kdlo = r % 3;
      bi.nkd = 1;
    }
  } else {
    bi.c = b;
    bi.kh = 1;
    bi.kw = 1;
    bi.kdlo = 1;
    bi.nkd = 1;
  }
  bi.ns = (p.mode == kModeUp2) ? p.R : bi.nkd;
  return bi;
}

struct UnitInfo {
  int n, d0, h0, w0, nh;
  int tg;  // kModeUp2: tap group
  int rd;  // output d-slices of this unit (the last group of a region may be partial)
  int ra;  // accumulators used by this unit (== rd, or the tap count in kModeUp2)
};

__device__ __forceinline__ UnitInfo decode_unit(const ConvIgemmParams& p, int u) {
  UnitInfo ui;
  const int npw = p.npw;
  const int np = npw * p.nph, ndg = (p.d_cnt + p.Rd - 1) / p.Rd;
  if (p.w_stationary) {   // (N split, tap group) slowest: consecutive units of a CTA share their weight blocks
    const int per_key = np * ndg * p.NT;
    const int key = u / per_key;
    u -= key * per_key;
    ui.tg = key % p.up_groups;
    ui.nh = key / p.up_groups;
  } else {
    ui.nh = u % p.nhalf;
    u /= p.nhalf;
    ui.tg = u % p.up_groups;
    u /= p.up_groups;
  }
  const int patch = u % np;
  u /= np;
  ui.d0 = p.d_lo + (u % ndg) * p.Rd;
  ui.n = u / ndg;
  ui.h0 = min(p.h_lo + (patch / npw) * p.TH, p.H - p.TH);   // the last tile of a range may overlap its neighbour
  ui.w0 = min(p.w_lo + (patch % npw) * p.TW, p.W - p.TW);
  ui.rd = min(p.Rd, p.d_lo + p.d_cnt - ui.d0);
  ui.ra = (p.mode == kModeUp2) ? p.R : ui.rd;
  return ui;
}

template <int FMT>
__device__ __forceinline__ uint32_t pack2(float a, float b) {
  if (FMT == 0) {
    __half2 h = __floats2half2_rn(a, b);
    return *reinterpret_cast<uint32_t*>(&h);
  }
  __nv_bfloat162 h = __floats2bfloat162_rn(a, b);
  return *reinterpret_cast<uint32_t*>(&h);
}

// one 32-byte global store (sm_100: STG.256); p must be 32-byte aligned
__device__ __forceinline__ void st_global_256(void* p, const uint32_t* v) {
  asm volatile("st.global.v8.b32 [%0], {%1,%2,%3,%4,%5,%6,%7,%8};" ::"l"(p), "r"(v[0]), "r"(v[1]), "r"(v[2]), "r"(v[3]),
               "r"(v[4]), "r"(v[5]), "r"(v[6]), "r"(v[7])
               : "memory");
}

// rn16(x - hi) for the pair whose rounded hi halves are already packed in `hi`
template <int FMT>
__device__ __forceinline__ uint32_t pack2_residual(float a, float b, uint32_t hi) {
  if (FMT == 0) {
    const float2 h = __half22float2(*reinterpret_cast<const __half2*>(&hi));
    return pack2<FMT>(a - h.x, b - h.y);
  }
  const float2 h = __bfloat1622float2(*reinterpret_cast<const __nv_bfloat162*>(&hi));
  return pack2<FMT>(a - h.x, b - h.y);
}

// rn(satfinite(e4m3)) of (a, b) scaled by 2^S, a in the low byte
__device__ __forceinline__ uint32_t pack2_e4m3(float a, float b) {
  uint16_t v;
  asm("cvt.rn.satfinite.e4m3x2.f32 %0, %1, %2;" : "=h"(v) : "f"(b), "f"(a));
  return v;
}

// Epilogue of one 32-column chunk held in registers: + bias (from shared memory), ReLU, 16-bit rounding, two 32-byte
// stores per thread (a thread owns one voxel's channel row, so every L2 sector is written whole by one instruction).
// LO == 1 also writes the rounding residual lo = rn16(x - hi) lo_off elements further, so hi + lo carries ~22 bits;
// LO == 2 writes it to the 8-bit plane dst8 instead, as e4m3(lo * 2^S) (one 32-byte store).
template <int FMT, bool RELU, int LO>
__device__ __forceinline__ void epi_store_chunk(uint32_t (&v)[32], uint32_t sbias, uint16_t* dst, long long lo_off,
                                                uint8_t* dst8, float& amax) {
  uint32_t o[16];
#pragma unroll
  for (int i = 0; i < 8; ++i) {
    const float4 b4 = lds_f4(sbias + 16 * i);
    float x0 = __uint_as_float(v[4 * i]) + b4.x, x1 = __uint_as_float(v[4 * i + 1]) + b4.y;
    float x2 = __uint_as_float(v[4 * i + 2]) + b4.z, x3 = __uint_as_float(v[4 * i + 3]) + b4.w;
    if (RELU) {
      x0 = fmaxf(x0, 0.f); x1 = fmaxf(x1, 0.f); x2 = fmaxf(x2, 0.f); x3 = fmaxf(x3, 0.f);
    }
    amax = fmaxf(amax, fmaxf(fmaxf(fabsf(x0), fabsf(x1)), fmaxf(fabsf(x2), fabsf(x3))));
    o[2 * i] = pack2<FMT>(x0, x1);
    o[2 * i + 1] = pack2<FMT>(x2, x3);
    if (LO) {
      v[4 * i] = __float_as_uint(x0); v[4 * i + 1] = __float_as_uint(x1);
      v[4 * i + 2] = __float_as_uint(x2); v[4 * i + 3] = __float_as_uint(x3);
    }
  }
  st_global_256(dst, o);
  st_global_256(dst + 16, o + 8);
  if (LO == 1) {
#pragma unroll
    for (int i = 0; i < 16; ++i)
      o[i] = pack2_residual<FMT>(__uint_as_float(v[2 * i]), __uint_as_float(v[2 * i + 1]), o[i]);
    st_global_256(dst + lo_off, o);
    st_global_256(dst + lo_off + 16, o + 8);
  } else if (LO == 2) {
    constexpr float kScale = FMT == 0 ? 2048.f : 256.f;   // 2^lo8_shift(FMT)
    uint32_t q[8];
#pragma unroll
    for (int i = 0; i < 8; ++i) {
      float2 h0, h1;
      if (FMT == 0) {
        h0 = __half22float2(*reinterpret_cast<const __half2*>(&o[2 * i]));
        h1 = __half22float2(*reinterpret_cast<const __half2*>(&o[2 * i + 1]));
      } else {
        h0 = __bfloat1622float2(*reinterpret_cast<const __nv_bfloat162*>(&o[2 * i]));
        h1 = __bfloat1622float2(*reinterpret_cast<const __nv_bfloat162*>(&o[2 * i + 1]));
      }
      const uint32_t lo01 = pack2_e4m3((__uint_as_float(v[4 * i]) - h0.x) * kScale,
                                       (__uint_as_float(v[4 * i + 1]) - h0.y) * kScale);
      const uint32_t lo23 = pack2_e4m3((__uint_as_float(v[4 * i + 2]) - h1.x) * kScale,
                                       (__uint_as_float(v[4 * i + 3]) - h1.y) * kScale);
      q[i] = lo01 | (lo23 << 16);
    }
    st_global_256(dst8, q);
  }
}

// All 32-column chunks of one accumulator (this warp's 32 TMEM lanes).  The accumulator is handed back to the MMA warp
// as soon as its last columns sit in registers, before the conversion and the global stores of that batch.
template <int FMT, bool RELU, int LO>
__device__ __forceinline__ void epi_store_acc(uint32_t t_acc, int nb, uint32_t sbias, uint16_t* dst, long long lo_off,
                                              uint8_t* dst8, uint64_t* acc_empty_bar, int lane, float& amax) {
  for (int j = 0; j < nb; ++j) {
    uint32_t v[32];
    tmem_ld_32x32(t_acc + j * 32, v);
    tmem_ld_wait();
    if (j + 1 == nb) {
      tc_fence_before();
      __syncwarp();
      if (lane == 0) mbar_arrive(acc_empty_bar);
    }
    epi_store_chunk<FMT, RELU, LO>(v, sbias + j * 128, dst + j * 32, lo_off, dst8 + j * 32, amax);
  }
}

// acc[k] += sum_i relu(v[i] + bias[i]) * w[k][i] over one 32-column chunk; bias and the head filter (rows 64 floats
// apart) are read from shared memory, four columns per load
template <int NC>
__device__ __forceinline__ void head_dot(const uint32_t (&v)[32], uint32_t sbias, uint32_t sw, float (&acc)[8],
                                         int ncls = NC) {
#pragma unroll
  for (int i = 0; i < 8; ++i) {
    const float4 b4 = lds_f4(sbias + 16 * i);
    const float f0 = fmaxf(__uint_as_float(v[4 * i]) + b4.x, 0.f), f1 = fmaxf(__uint_as_float(v[4 * i + 1]) + b4.y, 0.f);
    const float f2 = fmaxf(__uint_as_float(v[4 * i + 2]) + b4.z, 0.f), f3 = fmaxf(__uint_as_float(v[4 * i + 3]) + b4.w, 0.f);
#pragma unroll
    for (int k = 0; k < NC; ++k)
      if (k < ncls) {
        const float4 w4 = lds_f4(sw + k * 256 + 16 * i);
        acc[k] = fmaf(f3, w4.w, fmaf(f2, w4.z, fmaf(f1, w4.y, fmaf(f0, w4.x, acc[k]))));
      }
  }
}


// ---------------------------------------------------------------------------------------------- MMA issue
// The single thread that feeds the tensor pipe is the critical resource of the kernel: a lone warp retires one
// instruction every ~7 clocks (dependent integer chains, branch resolution; ncu source counters of the ec1 launch,
// profiles/r02_ncu_ec1_issuer.txt), so every instruction of the per-stage loop costs more than one K=16 step of a
// small MMA is worth.  Two loops therefore exist:
//   * mma_issuer_fast<NKW, K16N, PER>: compile-time (kw taps per A stage, K=16 steps per chunk, accumulators one MMA may
//     span = 256 / cout); per stage it does one mbarrier poll, five integer ops for the accumulator span, descriptor
//     adds and the MMAs; accumulators seeing their first MMA of the unit (first weight block) take a short side path;
//   * mma_issuer_general: run-time trip counts and descriptors rebuilt per MMA (debug / A-B flags, uncommon shapes).
// The whole warp walks the (warp-uniform) schedule so the compiler keeps the descriptor arithmetic in uniform
// registers; one lane, elected once, issues every tcgen05.mma / tcgen05.commit.
struct IssueConsts {
  uint32_t kw_step, b_kw, desc_hi32, idesc_1, idesc_step, tap16, cout;
  uint32_t kh_a, kh_b;   // three-row stages: descriptor units between the kh rows of the A stage / the kh sub-blocks of B
  uint32_t sfa, sfb;     // F8 stages: TMEM addresses of the block scales
};

// one MMA of a stage: kind::f16, or (F8) the block-scaled e4m3 kind with K = 32 over the same 32 bytes per row
template <bool F8>
__device__ __forceinline__ void issue_mma(const IssueConsts& c, uint32_t d, uint32_t a_lo, uint32_t b_lo, uint32_t idesc,
                                          uint32_t acc) {
  if (F8) umma_mxf8_ss_lohi(d, a_lo, b_lo, c.desc_hi32, idesc, c.sfa, c.sfb, acc);
  else umma_f16_ss_lohi(d, a_lo, b_lo, c.desc_hi32, idesc, acc);
}

// shared-memory row pitch (128 or 64 bytes) and its K steps: every field of IssueConsts that depends on them
__device__ __forceinline__ IssueConsts make_issue_consts(const ConvIgemmParams& p, uint32_t rowb, bool f8, int ns,
                                                         uint32_t tmem_base) {
  IssueConsts c;
  const uint32_t sbo = 8u * rowb, lay = rowb == 128u ? 2u : 4u;
  c.cout = static_cast<uint32_t>(p.cout);
  c.tap16 = (c.cout * rowb) >> 4;                               // one tap's weight rows, in descriptor units
  // descriptor units between the taps of one A stage: one voxel row (row-shared kw), TW rows (kh-shared kh)
  c.kw_step = (p.mode == kModeKhShared ? static_cast<uint32_t>(p.TW) * rowb : rowb) >> 4;
  c.desc_hi32 = (sbo >> 4) | (1u << 14) | (lay << 29);          // SBO, version = 1, swizzle mode
  c.idesc_1 = f8 ? umma_idesc_mxf8_e4m3(128, c.cout) : umma_idesc_f16(128, c.cout, p.ab_format);
  c.idesc_step = (c.cout >> 3) << 17;                           // +1 tap in the N field
  c.b_kw = static_cast<uint32_t>(ns) * c.tap16;
  c.kh_a = (130u * rowb) >> 4;
  c.kh_b = 3u * c.b_kw;
  c.sfa = tmem_base + kSfaCol;
  c.sfb = tmem_base + kSfbCol;
  return c;
}

// every (kw, k16) step of one A stage onto the accumulators [d_addr, +nt*cout), all accumulating; skip_first leaves out
// the (0, 0) step (already issued by issue_first with per-accumulator overwrite flags)
template <int NKW, int K16N, int PER, int NKH, bool F8>
__device__ __forceinline__ void issue_stage(const IssueConsts& c, uint32_t d_addr, uint32_t a_lo, uint32_t b_lo, int nt,
                                            bool skip_first) {
  for (int g0 = 0; g0 < nt; g0 += PER) {
    const int ng = min(PER, nt - g0);
    const uint32_t idesc = c.idesc_1 + static_cast<uint32_t>(ng - 1) * c.idesc_step;
    const uint32_t d = d_addr + static_cast<uint32_t>(g0) * c.cout;
    const uint32_t bl = b_lo + static_cast<uint32_t>(g0) * c.tap16;
#pragma unroll
    for (int kh = 0; kh < NKH; ++kh)
#pragma unroll
      for (int kw = 0; kw < NKW; ++kw)
#pragma unroll
        for (int k16 = 0; k16 < K16N; ++k16) {
          if (kh == 0 && kw == 0 && k16 == 0) {
            if (!skip_first) issue_mma<F8>(c, d, a_lo, bl, idesc, 1u);
          } else {
            issue_mma<F8>(c, d, a_lo + kh * c.kh_a + kw * c.kw_step + k16 * 2, bl + kh * c.kh_b + kw * c.b_kw + k16 * 2,
                          idesc, 1u);
          }
        }
  }
}

// the (kw = 0, k16 = 0) step of a stage whose span [acc0, acc0 + nt) holds partial sums below accumulator f0 and is
// fresh (first MMA of the unit: overwrite) from f0 on
template <int PER, bool F8>
__device__ __forceinline__ void issue_first(const IssueConsts& c, uint32_t tmem_base, int acc0, int nt, int f0,
                                            uint32_t a_lo, uint32_t b_lo) {
  for (int g0 = 0; g0 < nt; g0 += PER) {
    const int ng = min(PER, nt - g0);
    const int ag = acc0 + g0;
    const int keep = min(max(f0 - ag, 0), ng);  // leading accumulators of the group that accumulate
    const uint32_t bl = b_lo + static_cast<uint32_t>(g0) * c.tap16;
    if (keep > 0)
      issue_mma<F8>(c, tmem_base + static_cast<uint32_t>(ag) * c.cout, a_lo, bl,
                    c.idesc_1 + static_cast<uint32_t>(keep - 1) * c.idesc_step, 1u);
    if (keep < ng)
      issue_mma<F8>(c, tmem_base + static_cast<uint32_t>(ag + keep) * c.cout, a_lo,
                    bl + static_cast<uint32_t>(keep) * c.tap16,
                    c.idesc_1 + static_cast<uint32_t>(ng - keep - 1) * c.idesc_step, 0u);
  }
}

// chunk of weight block b (the block order of decode_block)
__device__ __forceinline__ int block_chunk(const ConvIgemmParams& p, int b) {
  if (p.mode == kModeRowShared) return p.nkh == 3 ? b : b / 3;
  if (p.mode == kModeKhShared) return b / 3;
  if (p.mode == kModePerTap) return p.kd_per_block == 3 ? b / 9 : b / 27;
  return b;
}

// LO8: the layer lists e4m3 lo-plane chunks; their stages take the second, 8-bit form of the loop body (one uniform
// branch per stage, block-scaled MMAs with K = 32, 64-byte rows)
template <int NKW, int K16N, int PER, int NKH, bool LO8>
__device__ __forceinline__ void mma_issuer_fast(const ConvIgemmParams& p, const uint32_t tmem_base0, uint8_t* abuf,
                                                uint8_t* wbuf, const uint32_t wstride, uint64_t* full_a,
                                                uint64_t* empty_a, uint64_t* full_w, uint64_t* empty_w,
                                                uint64_t* acc_full0, uint64_t* acc_empty0) {
  const int mode = p.mode, R_acc = p.R, nblk = p.nblk, nst = p.n_astage, nwb = p.n_wbuf, Dm1 = p.D - 1;
  const uint32_t a_lo0 = ((smem_u32(abuf) & 0x3FFFF) >> 4) | (1u << 16), a_step = p.astage_stride >> 4;
  const uint32_t w_lo0 = ((smem_u32(wbuf) & 0x3FFFF) >> 4) | (1u << 16), w_step = wstride >> 4;
  const bool up2 = mode == kModeUp2;
  const bool one_kd = mode == kModePointwise || up2;
  const bool kd_cycle = mode == kModePerTap && p.kd_per_block == 1;
  const int ns = up2 ? R_acc : ((one_kd || kd_cycle) ? 1 : 3);  // taps stacked along N in every weight block
  const int a_inc = up2 ? 0 : 1;
  const IssueConsts c = make_issue_consts(p, static_cast<uint32_t>(p.row_bytes), false, ns, tmem_base0);
  const IssueConsts c8 = make_issue_consts(p, 64u, true, ns, tmem_base0);
  const bool stationary = p.w_stationary != 0;
  int prev_key = -1;
  const bool leader = elect_one();
  int stage = 0, wb = 0;
  uint32_t aphase = 0, wphase = 0;
  uint32_t ub0 = 0, ub1 = 0;                      // per-accumulator mbarrier phase (flips per use), per TMEM half
  uint32_t a_lo = a_lo0;                          // descriptor low word of the current A stage
  int half = 0;
  for (int u = blockIdx.x; u < p.nunits; u += gridDim.x) {
    const UnitInfo ui = decode_unit(p, u);
    const int d0 = ui.d0, ra = ui.ra, rd = ui.rd;
    const uint32_t all_acc = (1u << ra) - 1u;
    // accumulator ping-pong (kModeUp2): this unit's accumulators are the half `half` of TMEM / of the barrier arrays
    const int ab = half * R_acc;
    const uint32_t tmem_base = tmem_base0 + static_cast<uint32_t>(ab) * c.cout;
    uint64_t* const acc_full = acc_full0 + ab;
    uint64_t* const acc_empty = acc_empty0 + ab;
    const int this_half = half;
    const uint32_t use_bits = this_half ? ub1 : ub0;
    if (p.acc_pingpong) half ^= 1;
    uint32_t touched = 0, signaled = 0;
    int kd_it = 0;  // kd counter of the one-kd-per-block schedule (fastest block index there)
    // stationary weights: wait for the blocks only when this unit's group differs from the previous unit's, release
    // them only when the next unit's does (the weight producer applies the same rule)
    const int key = ui.nh * p.up_groups + ui.tg;
    const bool reload = !(stationary && key == prev_key);
    prev_key = key;
    bool release = true;
    if (stationary && u + static_cast<int>(gridDim.x) < p.nunits) {
      const UnitInfo un = decode_unit(p, u + static_cast<int>(gridDim.x));
      release = un.nh * p.up_groups + un.tg != key;
    }
    for (int b = 0; b < nblk; ++b) {
      int kdlo = 0, kdhi = 2;
      if (one_kd) { kdlo = 1; kdhi = 1; }
      else if (kd_cycle) { kdlo = kdhi = kd_it; kd_it = kd_it == 2 ? 0 : kd_it + 1; }
      const int dlo = max(0, d0 + kdlo - 1);
      const int dhi = min(Dm1, d0 + rd - 1 + kdhi - 1);
      const bool last_blk = b == nblk - 1;
      if (reload) mbar_wait(&full_w[wb], wphase, 300 + wb);
      const bool f8 = LO8 && p.chunk_src[block_chunk(p, b)] == kSrcLo8;
      const uint32_t w_lo = w_lo0 + static_cast<uint32_t>(wb) * w_step;
      int a_first = up2 ? 0 : dlo - kdhi + 1 - d0;  // accumulator hit by the first stacked tap
      for (int dp = dlo; dp <= dhi; ++dp, a_first += a_inc) {
        mbar_wait(&full_a[stage], aphase, 400 + stage);
        tc_fence_after();
        const int acc0 = max(a_first, 0);
        const int acc1 = min(a_first + ns - 1, ra - 1);
        const int nt = acc1 - acc0 + 1;
        const uint32_t d_addr = tmem_base + static_cast<uint32_t>(acc0) * c.cout;
        const uint32_t b_lo = w_lo + static_cast<uint32_t>(acc0 - a_first) * (f8 ? c8.tap16 : c.tap16);
        int f0 = -1;
        if (touched != all_acc) {
          // first weight block of the unit (and, in the one-kd schedule at the volume's first slice, the second):
          // accumulators seeing their first MMA wait until the epilogue has drained their previous contents
          const uint32_t span = ((2u << (acc1 - acc0)) - 1u) << acc0;
          const uint32_t fresh = span & ~touched;
          touched |= span;
          if (fresh) {
            f0 = __ffs(fresh) - 1;  // the fresh accumulators are always the top of the span
            for (int a = f0; a <= acc1; ++a) mbar_wait(&acc_empty[a], ((use_bits >> a) & 1u) ^ 1u, 500 + a);
            tc_fence_after();
          }
        }
        const bool publish = last_blk && a_first >= 0 && a_first < ra;
        if (leader) {
          if (f8) {
            if (f0 >= 0) issue_first<PER, true>(c8, tmem_base, acc0, nt, f0, a_lo, b_lo);
            issue_stage<NKW, 2, PER, 1, true>(c8, d_addr, a_lo, b_lo, nt, f0 >= 0);
          } else {
            if (f0 >= 0) issue_first<PER, false>(c, tmem_base, acc0, nt, f0, a_lo, b_lo);
            issue_stage<NKW, K16N, PER, NKH, false>(c, d_addr, a_lo, b_lo, nt, f0 >= 0);
          }
          // release the A stage; the last block's last tap of an accumulator also publishes it to the epilogue
          umma_commit(&empty_a[stage]);
          if (publish) umma_commit(&acc_full[a_first]);
        }
        if (publish) signaled |= 1u << a_first;
        a_lo += a_step;
        if (++stage == nst) {
          stage = 0;
          aphase ^= 1u;
          a_lo = a_lo0;
        }
      }
      if (release && leader) umma_commit(&empty_w[wb]);
      if (++wb == nwb) {
        wb = 0;
        if (reload) wphase ^= 1u;   // one phase per (re)load of the buffers
      }
    }
    if (leader && signaled != all_acc) {
      for (int a = 0; a < ra; ++a)
        if (!((signaled >> a) & 1u)) umma_commit(&acc_full[a]);
    }
    if (this_half) ub1 = use_bits ^ all_acc;
    else ub0 = use_bits ^ all_acc;
  }
  __syncwarp();
}

__device__ __forceinline__ void mma_issuer_general(const ConvIgemmParams& p, const uint32_t tmem_base, uint8_t* abuf,
                                                   uint8_t* wbuf, const uint32_t wstride, uint64_t* full_a,
                                                   uint64_t* empty_a, uint64_t* full_w, uint64_t* empty_w,
                                                   uint64_t* acc_full, uint64_t* acc_empty) {
  const int mode = p.mode, R_acc = p.R, cout = p.cout, nblk = p.nblk, nst = p.n_astage, nwb = p.n_wbuf, Dm1 = p.D - 1,
            kpb = p.kd_per_block;
  const int nkw = (mode == kModeRowShared || mode == kModeKhShared) ? 3 : 1;
  const bool up2 = mode == kModeUp2;
  const bool leader = elect_one();
  int stage = 0, wb = 0;
  uint32_t aphase = 0, wphase = 0, use_bits = 0;  // use_bits: per-accumulator mbarrier phase (flips per use)
  for (int u = blockIdx.x; u < p.nunits; u += gridDim.x) {
    const UnitInfo ui = decode_unit(p, u);
    const int d0 = ui.d0, ra = ui.ra, rd = ui.rd;
    const uint32_t all_acc = (1u << ra) - 1u;
    uint32_t touched = 0, signaled = 0;
    int kd_it = 0;  // kd counter of the one-kd-per-block schedule (fastest block index there)
    for (int b = 0; b < nblk; ++b) {
      const bool f8 = p.chunk_src[block_chunk(p, b)] == kSrcLo8;   // e4m3 lo-plane chunk: 64-byte rows, K = 32 steps
      const uint32_t rowb = f8 ? 64u : static_cast<uint32_t>(p.row_bytes), sbo = 8u * rowb, lay = rowb == 128u ? 2u : 4u;
      const uint32_t a_tap = mode == kModeKhShared ? static_cast<uint32_t>(p.TW) * rowb : rowb;
      const uint32_t cout128 = static_cast<uint32_t>(cout) * rowb;    // bytes of one tap's weight rows
      const int k16n = f8 ? 2 : p.k16_steps;
      // taps stacked in this block and the input slices it walks (same arithmetic as decode_block, by counters)
      int kdlo = 0, nkd = 3;
      if (mode == kModePointwise || up2) { kdlo = 1; nkd = 1; }
      else if (mode == kModePerTap && kpb == 1) { kdlo = kd_it; nkd = 1; kd_it = kd_it == 2 ? 0 : kd_it + 1; }
      const int ns = up2 ? R_acc : nkd;
      const int kdhi = kdlo + nkd - 1;
      const int dlo = max(0, d0 + kdlo - 1);
      const int dhi = min(Dm1, d0 + rd - 1 + kdhi - 1);
      const bool last_blk = b == nblk - 1;
      mbar_wait(&full_w[wb], wphase, 300 + wb);
      int a_first = up2 ? 0 : dlo - kdhi + 1 - d0;  // accumulator hit by the first stacked tap
      for (int dp = dlo; dp <= dhi; ++dp, a_first += (up2 ? 0 : 1)) {
        mbar_wait(&full_a[stage], aphase, 400 + stage);
        tc_fence_after();
        const int acc0 = max(a_first, 0);
        const int ti_lo = acc0 - a_first;
        const int nt = min(ns - 1, ra - 1 - a_first) - ti_lo + 1;
        // one group per run of equal accumulator state, descriptors rebuilt per MMA
        const uint32_t a_base = smem_u32(abuf + static_cast<size_t>(stage) * p.astage_stride);
        const uint32_t w_base = smem_u32(wbuf + static_cast<size_t>(wb) * wstride);
        const int ti_hi = ti_lo + nt - 1;
        for (int kw = 0; kw < nkw; ++kw) {
          int ti = ti_lo;
          while (ti <= ti_hi) {
            const int a0 = a_first + ti;
            const uint32_t f = (touched >> a0) & 1u;
            int len = 1;
            while (ti + len <= ti_hi && ((touched >> (a0 + len)) & 1u) == f && (len + 1) * cout <= 256) ++len;
            if (!f) {
              for (int j = 0; j < len; ++j)
                mbar_wait(&acc_empty[a0 + j], ((use_bits >> (a0 + j)) & 1u) ^ 1u, 500 + a0 + j);
              tc_fence_after();
            }
            const uint32_t idesc = f8 ? umma_idesc_mxf8_e4m3(128, static_cast<uint32_t>(len * cout))
                                      : umma_idesc_f16(128, static_cast<uint32_t>(len * cout), p.ab_format);
            const uint32_t a_addr = a_base + static_cast<uint32_t>(kw) * a_tap;
            const uint32_t b_addr = w_base + static_cast<uint32_t>(kw * ns + ti) * cout128;
            const uint32_t boff = p.base_off_mode ? ((a_addr >> 7) & 7u) : 0u;
            const uint32_t d_addr = tmem_base + static_cast<uint32_t>(a0 * cout);
            if (leader) {
              for (int k16 = 0; k16 < k16n; ++k16) {
                const uint64_t adesc = umma_desc_kmajor(a_addr + k16 * 32, sbo, boff, lay);
                const uint64_t bdesc = umma_desc_kmajor(b_addr + k16 * 32, sbo, 0, lay);
                if (f8) umma_mxf8_ss(d_addr, adesc, bdesc, idesc, tmem_base + kSfaCol, tmem_base + kSfbCol,
                                     (f | (k16 > 0)) ? 1u : 0u);
                else umma_f16_ss(d_addr, adesc, bdesc, idesc, (f | (k16 > 0)) ? 1u : 0u);
              }
            }
            touched |= ((1u << len) - 1u) << a0;
            ti += len;
          }
        }
        // release the A stage; the last block's last tap of an accumulator also publishes it to the epilogue
        const bool publish = last_blk && a_first >= 0 && a_first < ra;
        if (leader) {
          umma_commit(&empty_a[stage]);
          if (publish) umma_commit(&acc_full[a_first]);
        }
        if (publish) signaled |= 1u << a_first;
        if (++stage == nst) {
          stage = 0;
          aphase ^= 1u;
        }
      }
      if (leader) umma_commit(&empty_w[wb]);
      if (++wb == nwb) {
        wb = 0;
        wphase ^= 1u;
      }
    }
    if (leader) {
      for (int a = 0; a < ra; ++a)
        if (!((signaled >> a) & 1u)) umma_commit(&acc_full[a]);
    }
    use_bits ^= all_acc;
  }
  __syncwarp();
}

}  // namespace

__global__ void __launch_bounds__(kThreads, 1)
conv_igemm_kernel(const __grid_constant__ CUtensorMap tm0, const __grid_constant__ CUtensorMap tm1,
                  const __grid_constant__ CUtensorMap tm2, const __grid_constant__ ConvIgemmParams p) {
  extern __shared__ uint8_t smem_raw[];
  uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~uintptr_t(1023));
  const uint32_t wstride = (p.wblock_bytes + 1023u) & ~1023u;
  uint8_t* wbuf = smem;
  uint8_t* abuf = wbuf + static_cast<size_t>(p.n_wbuf) * wstride;
  uint64_t* bars = reinterpret_cast<uint64_t*>(abuf + static_cast<size_t>(p.n_astage) * p.astage_stride);
  uint64_t* full_a = bars;        // [8]
  uint64_t* empty_a = bars + 8;   // [8]
  uint64_t* full_w = bars + 16;   // [4]
  uint64_t* empty_w = bars + 20;  // [4]
  uint64_t* acc_full = bars + 24;   // [8]
  uint64_t* acc_empty = bars + 32;  // [8]
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(bars + 40);
  float* s_head = reinterpret_cast<float*>(bars + 48);  // [ncls*64 + ncls] when the head is fused (2112 B reserved)
  float* s_bias = s_head + 528;                          // [nhalf*cout] (<= 512 floats)

  const int warp = threadIdx.x >> 5;
  const int lane = threadIdx.x & 31;

  if (threadIdx.x == 0) {
    for (int i = 0; i < 8; ++i) {
      mbar_init(&full_a[i], 1);
      mbar_init(&empty_a[i], 1);
      mbar_init(&acc_full[i], 1);
      mbar_init(&acc_empty[i], 4);
    }
    for (int i = 0; i < 4; ++i) {
      mbar_init(&full_w[i], 1);
      mbar_init(&empty_w[i], 1);
    }
    fence_mbar_init();
    tma_prefetch_desc(&tm0);
    tma_prefetch_desc(&tm1);
    if (p.lo8_sf_off) tma_prefetch_desc(&tm2);
  }
  if (warp == 2) {
    tmem_alloc(tmem_slot, kTmemCols);
    tmem_relinquish();
  }
  for (int i = threadIdx.x; i < p.nhalf * p.cout; i += blockDim.x) s_bias[i] = p.bias[i];
  if (p.head.enabled) {
    for (int i = threadIdx.x; i < p.head.ncls * 64; i += blockDim.x) s_head[i] = p.head.w[i];
    for (int i = threadIdx.x; i < p.head.ncls; i += blockDim.x) s_head[p.head.ncls * 64 + i] = p.head.b[i];
  }
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_slot;
  if (p.lo8_sf_off) {
    // block scales of the e4m3 chunks: every scale of A is 2^-S and every scale of B 2^-T, so whatever the hardware's
    // scale-factor layout, two uniformly filled 32-column regions serve every MMA
    if (warp >= 4 && warp < 8) {
      const uint32_t* sf = reinterpret_cast<const uint32_t*>(p.wpack + p.lo8_sf_off);
      const uint32_t lane_base = tmem_base + (static_cast<uint32_t>((warp & 3) * 32) << 16);
      tmem_st_32x32_fill(lane_base + kSfaCol, __ldg(sf));
      tmem_st_32x32_fill(lane_base + kSfbCol, __ldg(sf + 1));
      tmem_st_wait();
    }
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
  }

  if (warp == 0) {
    // ------------------------------------------------------------ activation producer
    if (lane == 0) {
      int stage = 0;
      uint32_t phase = 0;
      for (int u = blockIdx.x; u < p.nunits; u += gridDim.x) {
        const UnitInfo ui = decode_unit(p, u);
        for (int b = 0; b < p.nblk; ++b) {
          const BlockInfo bi = decode_block(p, b);
          const int csrc = p.chunk_src[bi.c];
          const CUtensorMap* tm = csrc == 0 ? &tm0 : csrc == 1 ? &tm1 : &tm2;
          const uint32_t bytes = csrc == kSrcLo8 ? p.astage_bytes / 2 : p.astage_bytes;   // e4m3: 64-byte rows
          const int cc = p.chunk_cc[bi.c];
          const int kdhi = bi.kdlo + bi.nkd - 1;
          const int dlo = max(0, ui.d0 + bi.kdlo - 1);
          const int dhi = min(p.D - 1, ui.d0 + ui.rd - 1 + kdhi - 1);
          const int cw = (p.mode == kModeRowShared) ? ui.w0 - 1 : ui.w0 + bi.kw - 1;
          const int ch = ui.h0 + bi.kh - 1;
          for (int dp = dlo; dp <= dhi; ++dp) {
            mbar_wait(&empty_a[stage], phase ^ 1u, 100 + stage);
            mbar_arrive_expect_tx(&full_a[stage], bytes);
            tma_load_5d(abuf + static_cast<size_t>(stage) * p.astage_stride, tm, &full_a[stage], cc, cw, ch, dp, ui.n);
            if (++stage == p.n_astage) {
              stage = 0;
              phase ^= 1u;
            }
          }
        }
      }
    }
  } else if (warp == 1) {
    // ------------------------------------------------------------ weight producer
    if (lane == 0) {
      int wb = 0, prev_key = -1;
      uint32_t phase = 0;
      for (int u = blockIdx.x; u < p.nunits; u += gridDim.x) {
        const UnitInfo ui = decode_unit(p, u);
        const uint8_t* src = p.wpack + static_cast<size_t>(ui.nh * p.up_groups + ui.tg) * p.nblk * p.wblock_bytes;
        const int key = ui.nh * p.up_groups + ui.tg;
        if (p.w_stationary && key == prev_key) continue;   // this group's blocks are still in shared memory
        prev_key = key;
        for (int b = 0; b < p.nblk; ++b) {
          // the e4m3 rows of a lo-plane chunk fill the first half of its block
          const uint32_t bytes = p.chunk_src[block_chunk(p, b)] == kSrcLo8 ? p.wblock_bytes / 2 : p.wblock_bytes;
          mbar_wait(&empty_w[wb], phase ^ 1u, 200 + wb);
          mbar_arrive_expect_tx(&full_w[wb], bytes);
          bulk_load(wbuf + static_cast<size_t>(wb) * wstride, src + static_cast<size_t>(b) * p.wblock_bytes, bytes,
                    &full_w[wb]);
          if (++wb == p.n_wbuf) {
            wb = 0;
            phase ^= 1u;
          }
        }
      }
    }
  } else if (warp == 2) {
    // ------------------------------------------------------------ MMA issuer
    // The single thread that feeds the tensor pipe is the critical resource of the kernel: an ncu source-level profile
    // (profiles/r02_ncu_ec1_issuer.txt) showed the previous loop executing ~245 warp instructions per A stage -- about
    // 1300 clocks for a lone warp -- against 6 x 96 clocks of MMAs for a 32-channel stage.  The loop body is therefore
    // specialised at compile time on (kw taps per stage, K=16 steps per chunk) and kept to descriptor adds.
    const bool general = p.base_off_mode || p.no_fast_path;
    const int nkw_rt = (p.mode == kModeRowShared || p.mode == kModeKhShared) ? 3 : 1;
    const int per_rt = max(1, 256 / p.cout);
#define OAI_ISSUE_LO8(NKW, K16N, PER, LO8) \
  mma_issuer_fast<NKW, K16N, PER, 1, LO8>(p, tmem_base, abuf, wbuf, wstride, full_a, empty_a, full_w, empty_w, acc_full, \
                                          acc_empty)
#define OAI_ISSUE(NKW, K16N, PER) OAI_ISSUE_LO8(NKW, K16N, PER, false)
#define OAI_ISSUE_GENERAL() \
  mma_issuer_general(p, tmem_base, abuf, wbuf, wstride, full_a, empty_a, full_w, empty_w, acc_full, acc_empty)
    const bool lo8 = p.lo8_sf_off != 0;
    if (general) OAI_ISSUE_GENERAL();
    else if (lo8) {
      if (nkw_rt == 3 && p.k16_steps == 4 && per_rt == 4) OAI_ISSUE_LO8(3, 4, 4, true);
      else if (nkw_rt == 1 && p.k16_steps == 4 && per_rt == 4) OAI_ISSUE_LO8(1, 4, 4, true);
      else OAI_ISSUE_GENERAL();
    } else if (nkw_rt == 3 && p.k16_steps == 4 && per_rt == 4) OAI_ISSUE(3, 4, 4);
    else if (nkw_rt == 3 && p.k16_steps == 2 && per_rt == 4 && p.nkh == 3)
      mma_issuer_fast<3, 2, 4, 3, false>(p, tmem_base, abuf, wbuf, wstride, full_a, empty_a, full_w, empty_w, acc_full, acc_empty);
    else if (nkw_rt == 3 && p.k16_steps == 2 && per_rt == 4) OAI_ISSUE(3, 2, 4);
    else if (nkw_rt == 1 && p.k16_steps == 4 && per_rt == 4) OAI_ISSUE(1, 4, 4);
    else if (nkw_rt == 1 && p.k16_steps == 4 && per_rt == 2) OAI_ISSUE(1, 4, 2);
    else if (nkw_rt == 1 && p.k16_steps == 4 && per_rt == 1) OAI_ISSUE(1, 4, 1);
    else OAI_ISSUE_GENERAL();
#undef OAI_ISSUE_GENERAL
#undef OAI_ISSUE
#undef OAI_ISSUE_LO8
  } else if (warp >= 4) {
    // ------------------------------------------------------------ epilogue
    const int q = warp & 3;                 // TMEM lane quadrant this warp may read
    const int eg = (warp - 4) >> 2;         // epilogue group: drains the accumulators a = eg, eg + kEpiGroups, ...
    const int epi_variant = (p.ab_format ? 6 : 0) + (p.out_lo8 ? 4 : p.out_split ? 2 : 0) + (p.relu ? 1 : 0);
    const uint32_t s_bias_addr = smem_u32(s_bias), s_head_addr = smem_u32(s_head);
    const int m = q * 32 + lane;
    const int th = m / p.TW, tw = m % p.TW;
    uint32_t ub0 = 0, ub1 = 0;
    int half = 0;
    const uint32_t tmem_base0 = tmem_base;
    uint64_t* const acc_full0 = acc_full;
    uint64_t* const acc_empty0 = acc_empty;
    uint16_t* out = reinterpret_cast<uint16_t*>(p.out);
    float amax = 0.f;   // largest |activation| this thread rounded to 16 bits
    for (int u = blockIdx.x; u < p.nunits; u += gridDim.x) {
      const UnitInfo ui = decode_unit(p, u);
      // accumulator ping-pong (kModeUp2): same half selection as the MMA warp
      const int ab = half * p.R;
      const uint32_t tmem_base = tmem_base0 + static_cast<uint32_t>(ab * p.cout);
      uint64_t* const acc_full = acc_full0 + ab;
      uint64_t* const acc_empty = acc_empty0 + ab;
      const int this_half = half;
      const uint32_t use_bits = this_half ? ub1 : ub0;
      if (p.acc_pingpong) half ^= 1;
      const long long off0 = p.obase + ui.n * p.osN + (ui.h0 + th) * p.osH + (ui.w0 + tw) * p.osW +
                             static_cast<long long>(ui.nh) * p.cout;
      for (int a = 0; a < ui.ra; ++a) {
        if (((ab + a) % kEpiGroups) != eg) continue;   // the groups share the PHYSICAL accumulators round-robin
        mbar_wait(&acc_full[a], (use_bits >> a) & 1u, 600 + a);
        tc_fence_after();
        if (p.head.enabled) {
          // fused dc0 + sigmoid + crop-and-place: only interior voxels of the tile are ever written
          const HeadFuse& hd = p.head;
          const int z = ui.d0 + a - hd.od, y = ui.h0 + th - hd.oh, x = ui.w0 + tw - hd.ow;
          const bool row_in = z >= 0 && z < hd.ed;  // warp-uniform when TH == 1
          const bool mine = row_in && y >= 0 && y < hd.eh && x >= 0 && x < hd.ew;
          if (__any_sync(0xffffffffu, mine)) {
            float acc[8];
#pragma unroll
            for (int k = 0; k < 8; ++k) acc[k] = 0.f;
            for (int j = 0; j < 2; ++j) {
              uint32_t v[32];
              tmem_ld_32x32(tmem_base + (static_cast<uint32_t>(q * 32) << 16) +
                                static_cast<uint32_t>(a * p.cout + j * 32), v);
              tmem_ld_wait();
              const uint32_t sbj = s_bias_addr + static_cast<uint32_t>(ui.nh * p.cout + j * 32) * 4u;
              const uint32_t swj = s_head_addr + static_cast<uint32_t>(j * 32) * 4u;
              switch (hd.ncls) {
                case 1: head_dot<1>(v, sbj, swj, acc); break;
                case 2: head_dot<2>(v, sbj, swj, acc); break;
                case 3: head_dot<3>(v, sbj, swj, acc); break;
                case 4: head_dot<4>(v, sbj, swj, acc); break;
                default: head_dot<8>(v, sbj, swj, acc, hd.ncls); break;
              }
            }
            if (mine) {
              const int tile = hd.tile0 + ui.n;
              const int tk = tile % hd.gw, tj = (tile / hd.gw) % hd.gh, ti = tile / (hd.gw * hd.gh);
              const int gz = ti * hd.ed + z, gy = tj * hd.eh + y, gx = tk * hd.ew + x;
              if (gz < hd.VD && gy < hd.VH && gx < hd.VW) {
                const bool shell = gz < hd.cz || gz >= hd.VD - hd.cz || gy < hd.cy || gy >= hd.VH - hd.cy ||
                                   gx < hd.cx || gx >= hd.VW - hd.cx;
                const size_t o = (static_cast<size_t>(gz) * hd.VH + gy) * hd.VW + gx;
                const size_t cls_stride = static_cast<size_t>(hd.VD) * hd.VH * hd.VW;
#pragma unroll
                for (int k = 0; k < 8; ++k) {
                  if (k >= hd.ncls) break;
                  float r = 0.f;
                  if (!shell) {
                    const float logit = acc[k] + s_head[hd.ncls * 64 + k];
                    r = hd.out_mode == 2 ? logit : 1.f / (1.f + __expf(-logit));
                    if (hd.out_mode == 1) r = r > 0.5f ? 1.f : 0.f;
                  }
                  hd.out[k * cls_stride + o] = r;
                }
              }
            }
          }
        } else {
          uint16_t* dst = (p.mode == kModeUp2) ? out + off0 + ui.d0 * p.osD + p.tap_off[ui.tg * p.R + a]
                                               : out + off0 + (ui.d0 + a) * p.osD;
          const uint32_t sb = s_bias_addr + static_cast<uint32_t>(ui.nh * p.cout) * 4u;
          const uint32_t t_acc = tmem_base + (static_cast<uint32_t>(q * 32) << 16) + static_cast<uint32_t>(a * p.cout);
          const int nb = p.cout / 32;
          uint8_t* dst8 = p.out_lo8 + (dst - out);
#define OAI_EPI(FMT, RELU, LO) \
  epi_store_acc<FMT, RELU, LO>(t_acc, nb, sb, dst, p.out_lo_off, dst8, &acc_empty[a], lane, amax)
          switch (epi_variant) {
            case 0: OAI_EPI(0, false, 0); break;
            case 1: OAI_EPI(0, true, 0); break;
            case 2: OAI_EPI(0, false, 1); break;
            case 3: OAI_EPI(0, true, 1); break;
            case 4: OAI_EPI(0, false, 2); break;
            case 5: OAI_EPI(0, true, 2); break;
            case 6: OAI_EPI(1, false, 0); break;
            case 7: OAI_EPI(1, true, 0); break;
            case 8: OAI_EPI(1, false, 1); break;
            case 9: OAI_EPI(1, true, 1); break;
            case 10: OAI_EPI(1, false, 2); break;
            default: OAI_EPI(1, true, 2); break;
          }
#undef OAI_EPI
          continue;  // accumulator already released
        }
        tc_fence_before();
        __syncwarp();
        if (lane == 0) mbar_arrive(&acc_empty[a]);
      }
      if (this_half) ub1 = use_bits ^ ((1u << ui.ra) - 1u);
      else ub0 = use_bits ^ ((1u << ui.ra) - 1u);
    }
    if (p.ab_format == 0 && !(amax <= 65504.f)) atomicAdd(&g_fp16_overflow, 1u);   // also catches NaN
  }

  tc_fence_before();
  __syncthreads();
  if (warp == 2) {
    tc_fence_after();
    tmem_dealloc(tmem_base, kTmemCols);
  }
}

// ---------------------------------------------------------------------------------------------- host side

static size_t conv_igemm_smem_bytes(const ConvIgemmParams& p) {
  const size_t wstride = (p.wblock_bytes + 1023u) & ~size_t(1023);
  return 1024 + p.n_wbuf * wstride + static_cast<size_t>(p.n_astage) * p.astage_stride + 48 * 8 + 2112 + 2048;
}

cudaError_t conv_overflow_count(unsigned int* count, bool reset, cudaStream_t stream) {
  cudaError_t e = cudaMemcpyFromSymbolAsync(count, g_fp16_overflow, sizeof(unsigned int), 0, cudaMemcpyDeviceToHost, stream);
  if (e != cudaSuccess) return e;
  e = cudaStreamSynchronize(stream);
  if (e != cudaSuccess || !reset) return e;
  const unsigned int zero = 0;
  return cudaMemcpyToSymbolAsync(g_fp16_overflow, &zero, sizeof(unsigned int), 0, cudaMemcpyHostToDevice, stream);
}

cudaError_t conv_igemm_launch(const ConvIgemmParams& p, const CUtensorMap& tm0, const CUtensorMap& tm1,
                              const CUtensorMap& tm2, int num_sms, cudaStream_t stream) {
  const size_t smem = conv_igemm_smem_bytes(p);
  // the attribute is per device: cache what has been configured for each device of this process
  static size_t configured[64] = {0};
  int dev = 0;
  cudaGetDevice(&dev);
  if (dev < 0 || dev >= 64 || smem > configured[dev]) {
    cudaError_t e = cudaFuncSetAttribute(conv_igemm_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                         static_cast<int>(smem));
    if (e != cudaSuccess) return e;
    if (dev >= 0 && dev < 64) configured[dev] = smem;
  }
  const int grid = p.nunits < num_sms ? p.nunits : num_sms;
  conv_igemm_kernel<<<grid, kThreads, smem, stream>>>(tm0, tm1, tm2, p);
  return cudaGetLastError();
}

}  // namespace oai
