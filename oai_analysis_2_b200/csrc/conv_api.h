// Internal (library-private) interface of the tcgen05 implicit-GEMM conv: layer spec, weight packer, launcher.
// The C-ABI entry points of api_conv.cu and the stage-level segmentation network (seg_net.cu) both sit on top of it.
#pragma once
#include <cstddef>
#include <cuda_runtime.h>

#include "conv_igemm.cuh"

namespace oai {

// ConvSpec::flags bit: pack and run a 3x3x3 layer in kh-shared mode (conv_igemm.cuh), whose M tiles may cover any
// (h, w) box; the weight blocks are ordered (chunk, kw) with the 3 kh x 3 kd taps inside.
constexpr int kConvFlagKhShared = 256;

struct ConvSpec {
  int D, H, W;         // layer grid (the INPUT grid for kind 2)
  int c0, c1;          // logical channels of source 0 / source 1 (skip connection; 0 if absent)
  int split0, split1;  // the source tensor holds [hi | lo] 16-bit planes (2*c channels per voxel)
  int cout;
  int kind;            // 0 = 3x3x3 p1, 1 = 1x1x1, 2 = ConvTranspose3d(k2,s2)
  int terms;           // 1: a*w (16-bit operands) | 2: (a_hi + a_lo)*w | 3: a_hi*w_hi + a_lo*w_hi + a_hi*w_lo
                       // 4 / 5: as 2, but only source 1 / only source 0 is read as hi + lo
                       // 6 / 7: as 4 / 2 (7: one-source layers), the source a plain fp16 hi tensor plus an e4m3 lo
                       //        plane (ConvLaunch::src_lo8) multiplied by block-scaled 8-bit MMAs
  int fmt;             // 0 fp16, 1 bf16
  int flags;
};

struct ConvLaunch {
  const void* src0;
  const void* src1;
  int NT;
  const void* wpack;
  size_t wpack_bytes;
  const float* bias;
  int relu;
  void* out;
  long long obase, osN, osD, osH, osW;  // element offsets of the output voxel rows
  int out_split;                        // also write the lo plane out_lo_off elements after the hi plane
  long long out_lo_off;
  const int* region;                    // {d_lo, d_cnt, h_lo, h_cnt} or nullptr
  int w_lo = 0, w_cnt = 0;              // w range of the region (kConvFlagKhShared layers only; 0: full rows)
  double flop_share = 1.0;              // part of the layer's algorithmic MACs the profile books on this launch
  const HeadFuse* head;                 // fused dc0 + sigmoid + assemble epilogue or nullptr
  const void* src_lo8 = nullptr;        // terms 6 / 7: e4m3 lo plane of the lo8 source (C bytes per voxel)
  void* out_lo8 = nullptr;              // also write the output's e4m3 lo plane (cout bytes per voxel) here
};

size_t conv_wpack_bytes(const ConvSpec& s);
int conv_pack_weights(const ConvSpec& s, const float* w, void* dst, size_t dst_bytes);
int conv_run(const ConvSpec& s, const ConvLaunch& a, cudaStream_t st);
// A kh-shared launch (kConvFlagKhShared) over the w range [w_lo, w_hi] of a.region: 32-wide M tiles over the largest
// multiple of 32 columns, and a second launch of 8-wide tiles over the last columns when the width is not a multiple of
// 32 (dc2: 98 = 96 + 2, the strip covers the last 8 and overlaps the main tiles, which write the same values there).
int conv_run_w_box(const ConvSpec& s, ConvLaunch a, int w_lo, int w_hi, cudaStream_t st);

inline HeadFuse make_head_fuse(int ncls, const float* head_w, const float* head_b, float* out, const int* vol_dims,
                               const int* geom, int tile0, const int* crop_zyx, int out_mode) {
  HeadFuse hd;
  hd.enabled = 1; hd.ncls = ncls; hd.out_mode = out_mode; hd.w = head_w; hd.b = head_b; hd.out = out;
  hd.VD = vol_dims[0]; hd.VH = vol_dims[1]; hd.VW = vol_dims[2];
  hd.ed = geom[3]; hd.eh = geom[4]; hd.ew = geom[5];
  hd.od = geom[6]; hd.oh = geom[7]; hd.ow = geom[8];
  hd.gh = geom[10]; hd.gw = geom[11]; hd.tile0 = tile0;
  hd.cz = crop_zyx[0]; hd.cy = crop_zyx[1]; hd.cx = crop_zyx[2];
  return hd;
}

}  // namespace oai
