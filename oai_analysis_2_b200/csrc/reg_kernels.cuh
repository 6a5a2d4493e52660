// Parameter blocks of the registration-stage kernels (reg_kernels.cu) shared with their C-ABI wrappers.
#pragma once
#include <cuda_runtime.h>

#include <cstddef>
#include <cstdint>

namespace oai {

// Direct fp32 convolution, kernel 3, pad 1, stride 1 or 2, planar NCDHW tensors with explicit channel strides so a
// layer can read / write a channel slice of a concatenation buffer in place.
struct Conv3Params {
  const float* in;   // [N][cin] planes of Di*Hi*Wi
  long long in_nstride, in_cstride;
  int cin, Di, Hi, Wi;
  const float* w;    // packed [cin][27][cout_pad]
  const float* bias; // [cout]
  float* out;        // [N][cout] planes of Do*Ho*Wo
  long long out_nstride, out_cstride;
  int cout, cout_pad, Do, Ho, Wo;
  int N, stride;
  int leaky_in;      // apply leaky_relu(0.01) to the input on load
  int residual;      // 1: add pad_or_crop(avg_pool3d(in, 2, ceil_mode=True)) (zero-padded IN FRONT to cout channels)
  float out_scale;   // multiplies (acc + bias [+ residual])
  float* splitk_ws;  // optional workspace for the split-K path of the deep levels (conv3_splitk_bytes)
  size_t splitk_bytes;
  // optional tcgen05 path of the strided down steps (reg_umma_down.cu): weight blocks, their scale exponent and a
  // workspace of conv3_umma_workspace() bytes for the space-to-depth hi / lo copy of the layer input
  const void* wumma = nullptr;
  int wexp = 0;
  void* xsplit = nullptr;
  size_t xsplit_bytes = 0;
};

// Direct fp32 transposed convolution, kernel 4, stride 2, pad 1 (output = 2x input), fused with the icon UNet2 up-path:
//   out = BN( convT(leaky_relu(in)) + bias + upsample2x_trilinear(in[:, :cout]) ), cropped to (Do,Ho,Wo).
struct ConvT4Params {
  const float* in;   // [N][cin] planes of Di*Hi*Wi
  long long in_nstride, in_cstride;
  int cin, Di, Hi, Wi;
  const float* w;    // packed [cin][64][cout]
  const float* bias, *bn_scale, *bn_shift;  // [cout]
  float* out;
  long long out_nstride, out_cstride;
  int cout, Do, Ho, Wo;  // Do <= 2*Di etc. (crop)
  int N;
  // optional split-fp16 weights for the mma.sync path (reg_pack_convt4_launch): [cout/16][cin/16][64 taps in visit order][2][32] uint4 of
  // B fragments (hi k0-7, hi k8-15, lo k0-7, lo k8-15), scaled by 2^wexp
  const uint4* wpk;
  int wexp;
  int debug;         // development switches (OAI_CONVT4_DEBUG): 1 no residual, 2 no MMAs, 4 no staging, 8 no stores
  int res_planes_per_n;  // filled by the launcher: in_nstride / in_cstride
  size_t xsplit_bytes;
  uint32_t* xsplit;  // workspace of N*cin*Di*Hi*Wi words for the tensor paths: the layer input as hi / lo fp16
  const void* wumma = nullptr;  // optional weight blocks of the tcgen05 path (reg_pack_convt4_umma_launch)
};

struct ChainParams {
  int D, H, W;             // grid of the coordinate map being built
  int nfields;
  const float* u[4];       // displacement tensors [3][ud][uh][uw] (components z,y,x in [0,1] units), applied in order
  int ud[4], uh[4], uw[4];
  int shortcut_first;      // first field has the grid's shape and is added without interpolation
  const float* img;        // optional image [id][ih][iw] sampled at the final coordinates
  int id, ih, iw;
  float* phi_out;          // optional [3][D][H][W]
  float* img_out;          // optional [D][H][W]
};

struct Affine3 {
  double m[9];
  double t[3];
};

struct WarpVolumeParams {
  const float* src;  // [C][SD][SH][SW] image being resampled (prob maps, on image A's grid)
  int C, SD, SH, SW;
  const float* disp; // [FD][FH][FW][3] displacement (x,y,z components, network-voxel units)
  int FD, FH, FW;
  Affine3 out_index_to_net;   // output index (x,y,z) -> network lattice coordinate (x,y,z)
  Affine3 net_to_src_index;   // displaced lattice coordinate -> continuous index (x,y,z) of src
  float* out;        // [C][OD][OH][OW]
  int OD, OH, OW;
  float default_value;
  double fhi[3], shi[3];  // filled by warp_volume_launch: upper inside bounds n - 0.5 of the field / source lattices (x,y,z)
};

struct WarpPointsParams {
  const double* pts;  // [n][3] physical x,y,z
  double* out;        // [n][3]
  long long n;
  const float* disp;
  int FD, FH, FW;
  Affine3 phys_to_net, net_to_phys;
};

int conv3_launch(const Conv3Params& p, cudaStream_t st);
size_t conv3_splitk_bytes(const Conv3Params& p);
size_t convt4_splitk_bytes(const ConvT4Params& p);
int convt4_launch(const ConvT4Params& p, cudaStream_t st);
int reg_pack_convt4_launch(const float* w, int cin, int cout, int wexp, uint4* wpk, cudaStream_t st);
// tcgen05 path of the up step (reg_umma.cu): cout in {16, 32, 64, 128}, cin a multiple of 16, lattice at least 8 x 8
bool convt4_umma_eligible(const ConvT4Params& p);
size_t convt4_umma_wbytes(int cin, int cout);
int reg_pack_convt4_umma_launch(const float* w, int cin, int cout, int wexp, void* dst, cudaStream_t st);
int convt4_umma_launch(const ConvT4Params& p, cudaStream_t st);
// tcgen05 path of the down step (reg_umma_down.cu): stride 2, leaky input, residual, cin % 16 == 0, cout 32 or a
// multiple of 64, output lattice at least 8 x 8
bool conv3_umma_eligible(const Conv3Params& p);
size_t conv3_umma_wbytes(int cin, int cout);
size_t conv3_umma_workspace(const Conv3Params& p);
int reg_pack_conv3_umma_launch(const float* w, int cin, int cout, int cout_pad, int wexp, void* dst, cudaStream_t st);
int conv3_umma_launch(const Conv3Params& p, cudaStream_t st);
int chain_launch(const ChainParams& p, cudaStream_t st);
int resize_trilinear_launch(const float* in, int Di, int Hi, int Wi, float* out, int Do, int Ho, int Wo,
                            cudaStream_t st);
int avgpool2_ceil_launch(const float* in, int C, int Di, int Hi, int Wi, float* out, cudaStream_t st);
int disp_field_launch(const float* phi, int D, int H, int W, float* disp, cudaStream_t st);
int warp_volume_launch(const WarpVolumeParams& p, cudaStream_t st);
int warp_points_launch(const WarpPointsParams& p, cudaStream_t st);

// ---- registration-quality terms of GradientICON.forward (reg_loss.cu)
struct GradIconParams {
  int D, H, W;               // grid of the noisy identity map Ie = identity + noise / W
  const float* noise;        // [3][D][H][W] N(0, 1)
  float delta;               // finite-difference step along each coordinate channel
  int nf[2];                 // fields of the two maps: [0] applied first (phi_BA), [1] then (phi_AB)
  const float* u[2][4];      // [3][ud][uh][uw] displacement fields in application order
  int ud[2][4], uh[2][4], uw[2][4];
  double* partials;          // [gradicon_blocks]
};

struct JacobianParams {
  int D, H, W;
  const float* phi_jac;      // [3][D][H][W] map whose dV / folds are counted
  const float* phi_mag;      // optional [3][D][H][W] map of mean((identity - phi)^2)
  float* det_out;            // optional dV map [D-1][H-1][W-1]
  unsigned long long* count; // device counter of dV < 0 (reset by jacobian_launch)
  double* mag_partials;      // [jacobian_blocks] when phi_mag is set
};

constexpr int kLnccMaxRadius = 24;   // taps 2R + 1 with R = floor(2 sigma): sigma < 12.5
struct LnccParams {
  int D, H, W;
  const float* I;            // warped image
  const float* J;            // target
  int radius;
  float taps[2 * kLnccMaxRadius + 1];   // normalised Gaussian, 2 * radius + 1 used
  float* zb;                 // scratch [5][D][H][W]: the moments blurred along z
  double* partials;          // [lncc_blocks]: sums of 1 - NCC
};

struct LossFinishParams {
  const double* g;           // gradicon partials
  int ng;
  const double* s;           // similarity partials [2 directions][2][ns]: LNCC uses [d][0]; SSD numerator, divisor
  int ns, ssd;
  const double* m;           // transform-magnitude partials
  int nm;
  const unsigned long long* count;
  double nvox, lmbda;
  double* terms;             // ICONLoss order: all, inverse consistency, similarity, transform magnitude, flips
};

int gradicon_blocks(int D, int H, int W);
int jacobian_blocks(int D, int H, int W);
int lncc_blocks(int D, int H, int W);
int ssd_blocks(int D, int H, int W);
int lncc_radius(double sigma);
size_t lncc_tile_smem(int radius);
int gradicon_launch(const GradIconParams& p, cudaStream_t st);
int jacobian_launch(const JacobianParams& p, cudaStream_t st);
int lncc_launch(const LnccParams& p, cudaStream_t st);
int ssd_launch(const float* warped, const float* tag, const float* target, int D, int H, int W, double* num,
               double* den, cudaStream_t st);
int inbounds_tag_launch(float* tag, int D, int H, int W, cudaStream_t st);
int loss_finish_launch(const LossFinishParams& p, cudaStream_t st);

}  // namespace oai
