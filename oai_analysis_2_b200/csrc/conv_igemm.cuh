// Parameter block shared by the tcgen05 implicit-GEMM conv kernel and its host launcher.
#pragma once
#include <cstdint>
#include <cuda.h>
#include <cuda_runtime.h>

namespace oai {

constexpr int kMaxChunks = 48;

enum ConvMode : int {
  kModeRowShared = 0,  // 3x3x3, M tile = one full 128-wide row; w halo loaded once, kw taps = smem row shifts
  kModePerTap = 1,     // 3x3x3, one TMA box per (kh,kw) shift; M tile = TH x TW patch
  kModePointwise = 2,  // 1x1x1
  kModeUp2 = 3,        // ConvTranspose3d(k=2, s=2): the accumulators of a unit are sub-filters (taps) of ONE input
                       // M tile, stacked along N; the epilogue scatters each tap into the 2x output grid
  kModeKhShared = 4,   // 3x3x3, M tile = TH x TW sub-box at any (h0, w0); one (TH+2) x TW box per kw, the kh taps are
                       // the same buffer shifted by TW rows (a multiple of the 1024-byte swizzle atom)
};

// Optional fused epilogue of the last decoder layer: dc0 (1x1x1, C->ncls) + sigmoid (+ >0.5) + Partition.assemble
// crop-and-place, computed from the fp32 accumulators so the layer's activation is never written.
struct HeadFuse {
  int enabled;
  int ncls, out_mode;             // 0 probability, 1 mask, 2 logit
  const float* w;                 // [ncls][64]
  const float* b;                 // [ncls]
  float* out;                     // [ncls][VD][VH][VW]
  int VD, VH, VW;
  int ed, eh, ew, od, oh, ow, gh, gw, tile0;
  int cz, cy, cx;
};

struct ConvIgemmParams {
  // activation grid (identical for input and output: stride-1 "same" conv or pointwise)
  int NT, D, H, W;
  int TW, TH;       // M tile = TH x TW voxels in one d-slice (TH*TW == 128)
  int R;            // accumulators per unit = consecutive output d-slices (R*cout <= 512; the last group of a region may be partial)
  int Rd;           // d-slices per unit (== R except kModeUp2, where R counts taps and Rd == 1)
  int up_groups;    // kModeUp2: tap groups per M tile (8 / R)
  long long tap_off[8];  // kModeUp2: output element offset of tap (a,b,c) = ((a*2H + b)*2W + c)*cout
  int d_lo, d_cnt;  // output region computed: slices [d_lo, d_lo+d_cnt) ...
  int h_lo, nph;     // ... and M tiles with origins (min(h_lo + i*TH, H-TH), min(w_lo + j*TW, W-TW)), i < nph, j < npw;
  int w_lo, npw;    // the rest is dead halo
  int cout;         // N per accumulator (multiple of 16, <= 256)
  int nhalf;        // N splits (cout_total = nhalf*cout)
  int nchunks;      // K chunks (one TMA box of 64 channels each, 32 when row_bytes == 64) per tap set
  // chunk c reads channels [chunk_cc[c], +64) of tensor map chunk_src[c].  A plain layer lists source 0's channels then
  // source 1's (the decoder's torch.cat).  Split-precision layers (terms 2 / 3) read tensors stored as [hi | lo] fp16
  // planes (2C channels per voxel) and list more chunks: K-concatenation of a_hi*w, a_lo*w (and a_hi*w_lo).
  uint16_t chunk_cc[kMaxChunks];
  uint8_t chunk_src[kMaxChunks];
  int k16_steps;    // K=16 MMA steps per chunk: 4 (64 channels) or 2 (32 channels)
  int row_bytes;    // shared-memory row pitch of one voxel's K slice: 128 (64 ch, SWIZZLE_128B) or 64 (32 ch, SWIZZLE_64B)
  int mode;         // ConvMode
  int kd_per_block; // 3: weights block stacks kd=2,1,0 ; 1: one kd per block
  int nblk;         // weight blocks per (unit, nhalf)
  uint32_t wblock_bytes;
  int n_wbuf;       // weight buffers in smem
  int nkh;          // row-shared mode: kh rows of an input slice held by ONE A stage (1, or 3 for a 32-channel source:
                    // the stage is a 3 x 130-voxel box and the weight block is the whole 27-tap image)
  int w_stationary; // every weight block of a (N split, tap group) has its own shared-memory buffer (n_wbuf == nblk) and the
                    // units are ordered split / tap-group major: the blocks are (re)loaded only when a CTA's next unit
                    // belongs to another group -- once per kernel for a single-group layer (ec1), eight times for dc6
  int acc_pingpong; // kModeUp2: a unit uses R of the 2R accumulators TMEM holds, consecutive units of a CTA alternate
                    // between the two halves, so the MMAs of one unit overlap the epilogue of the previous one
  int n_astage;     // A ring depth
  uint32_t astage_bytes;  // bytes landed per A stage (expect_tx)
  uint32_t astage_stride; // smem stride between A stages (1024-aligned)
  int ab_format;    // 0 fp16, 1 bf16
  int relu;
  int no_fast_path;   // debug/A-B: always take the general MMA grouping path
  int base_off_mode;  // row-shared mode: 0 (correct on B200: the swizzle XOR uses absolute smem address bits) or
                      // 1 = descriptor base_offset = (addr>>7)&7 (kept for the bring-up test; gives wrong results)
  const uint8_t* wpack;   // [nhalf][nblk][wblock_bytes] pre-swizzled smem images
  const float* bias;      // [nhalf*cout]
  // output addressing (element units, 16-bit elements): off = obase + n*osN + d*osD + h*osH + w*osW + nh*cout + c
  void* out;
  long long obase, osN, osD, osH, osW;
  // split output: besides hi = rn16(x) also write lo = rn16(x - hi) out_lo_off elements further (the [hi | lo] layout
  // split-precision consumers read); the os* strides then address the 2*C-channel voxel rows
  int out_split;
  long long out_lo_off;
  int nunits;
  HeadFuse head;
};

}  // namespace oai
