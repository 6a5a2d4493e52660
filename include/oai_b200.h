/* liboai_b200 -- C ABI of the B200-native per-knee inference hot path of OAI Analysis 2.
 *
 * The reference (uncbiag/OAI_analysis_2) is pure Python and has no FFI of its own: its hot path calls
 * torch / ITK / icon_registration library ops.  Each entry point below names the reference call it replaces
 * (paths relative to the reference repository root).  INTEGRATION.md shows the ctypes stub a maintainer adds on the
 * reference side.
 *
 * Conventions
 *   - every function returns 0 on success, non-zero on failure; oai_last_error() returns a message for the calling
 *     thread's last failure;
 *   - the caller owns every device buffer and the CUDA stream (passed as void* == cudaStream_t); nothing here
 *     allocates caller-visible memory, synchronises the device, or keeps a pointer after returning;
 *   - "act16" tensors are channels-last NDHWC, 16-bit (fp16 when ab_format == 0, bf16 when 1);
 *   - volumes are dense z,y,x (numpy order of the reference, image_transforms.py:376-379) float32.
 */
#ifndef OAI_B200_H_
#define OAI_B200_H_

#include <stddef.h>
#include <stdint.h>

#if defined(__GNUC__)
#define OAI_API __attribute__((visibility("default")))
#else
#define OAI_API
#endif

#ifdef __cplusplus
extern "C" {
#endif

OAI_API const char* oai_last_error(void);
OAI_API int oai_version(void);
/* number of kernels launched through this library since load (bench.py reports it as gpu_launches) */
OAI_API long long oai_launch_count(void);

/* ------------------------------------------------------------------------------------------------------------
 * Segmentation UNet layers  (reference: oai_analysis/segmentation/networks.py:38-149)
 * ------------------------------------------------------------------------------------------------------------ */

/* 3x3x3 stride-1 "same" convolution or pointwise convolution as a tcgen05 implicit GEMM.
 * Replaces nn.Conv3d(k=3,p=1) / nn.ConvTranspose3d(k=3,s=1,p=1) [+BatchNorm3d(eval)+ReLU folded]
 * (networks.py:80-107) and, with pointwise=1, each of the 8 sub-filters of nn.ConvTranspose3d(k=2,s=2).
 *
 *   src0/src1 : act16 [NT, D, H, W, c0] / [NT, D, H, W, c1]  (src1 may be NULL with c1 == 0; the K loop runs over
 *               src0's channels then src1's, which is torch.cat((src0, src1), dim=1) of networks.py:127,134,141)
 *   wpack     : weights packed by oai_pack_conv_weights() for the same geometry
 *   bias      : float32 [cout]
 *   out       : act16, element offset of voxel (n,d,h,w) channel c is
 *               obase + n*osN + d*osD + h*osH + w*osW + c   (lets a k2s2 transposed conv scatter its 8 sub-grids)
 */
OAI_API int oai_conv3d_igemm(const void* src0, int c0, const void* src1, int c1, int NT, int D, int H, int W,
                     const void* wpack, size_t wpack_bytes, const float* bias, int cout, int pointwise, int relu,
                     int ab_format, void* out, long long obase, long long osN, long long osD, long long osH,
                     long long osW, int flags, void* stream);

/* oai_conv3d_igemm restricted to the output sub-box region = {d_lo, d_cnt, h_lo, h_cnt} (full rows in w).  The
 * reference computes every decoder layer on the whole tile and then keeps only the tile interior
 * (image_transforms.py:497-503); outputs no kept voxel depends on ("dead halo") need not be computed.  Results inside
 * the region are identical to the full-layer call; memory outside it is left untouched. */
OAI_API int oai_conv3d_igemm_region(const void* src0, int c0, const void* src1, int c1, int NT, int D, int H, int W,
                                    const void* wpack, size_t wpack_bytes, const float* bias, int cout, int pointwise,
                                    int relu, int ab_format, void* out, long long obase, long long osN, long long osD,
                                    long long osH, long long osW, int flags, const int* region, void* stream);

/* nn.ConvTranspose3d(k=2, s=2) [+BN+ReLU folded] (networks.py:56,59,62) in one launch: out[co, 2z+a, 2y+b, 2x+c] =
 * sum_ci in[ci,z,y,x] * w[co][ci][a][b][c] + bias[co].  Each input M tile is loaded once and multiplied with the 8
 * sub-filters stacked along N; the epilogue scatters every tap into the 2x grid.  src: act16 [NT,D,H,W,cin];
 * out: act16 [NT,2D,2H,2W,cout]; w for the packer: float32 [cout][cin][2][2][2] (conv orientation);
 * region (may be NULL) = {d_lo, d_cnt, h_lo, h_cnt} on the INPUT grid. */
OAI_API int oai_pack_convt2_weights(const float* w, int cout, int cin, int D, int H, int W, int ab_format, void* dst,
                                    size_t dst_bytes);
OAI_API int oai_convt2_igemm(const void* src, int cin, int NT, int D, int H, int W, const void* wpack,
                             size_t wpack_bytes, const float* bias, int cout, int relu, int ab_format, void* out,
                             const int* region, void* stream);

/* The last decoder layer fused with the network head and the assembler: dc1 = ConvTranspose3d(64->64,k3,s1,p1)+BN+ReLU
 * (networks.py:64) feeding dc0 = Conv3d(64->ncls,k1) (networks.py:66,148), torch.sigmoid (segmenter.py:121)
 * [out_mode 1: ">0.5", segmenter.py:123-124; 2: raw logits] and Partition.assemble's crop-and-place with the zeroed
 * border shell (image_transforms.py:492-513).  dc0 is evaluated on the fp32 accumulators, the 64-channel activation is
 * never written.  out: float32 [ncls][vol_dims]; geom / vol_dims / crop_zyx as for oai_seg_head. */
OAI_API int oai_conv3d_igemm_head(const void* src0, int c0, const void* src1, int c1, int NT, int D, int H, int W,
                                  const void* wpack, size_t wpack_bytes, const float* bias, int ab_format, int ncls,
                                  const float* head_w, const float* head_b, float* out, const int* vol_dims,
                                  const int* geom, int tile0, const int* crop_zyx, int out_mode, int flags,
                                  void* stream);

/* Geometry the kernel will use for (D,H,W,cin,cout,pointwise): fills plan[9] =
 * {mode, kd_per_block (tap groups when pointwise == 2), R, nhalf, cout_per_half, nblk, wblock_bytes, nchunks,
 *  row_bytes}.
 * pointwise: 0 = 3x3x3, 1 = 1x1x1, 2 = ConvTranspose3d(k2,s2).  Pure host arithmetic (no GPU). */
OAI_API int oai_conv3d_igemm_plan(int D, int H, int W, int c0, int c1, int cout, int pointwise, int flags, int* plan);

/* Pack float32 conv weights [cout][cin][3][3][3] (or [cout][cin] when pointwise) into the pre-swizzled
 * shared-memory block images the kernel streams with cp.async.bulk.  Host function (no GPU).
 * dst must hold oai_conv3d_igemm_plan()'s nhalf*nblk*wblock_bytes bytes. */
OAI_API int oai_pack_conv_weights(const float* w, int cout, int c0, int c1, int D, int H, int W, int pointwise, int ab_format,
                          int flags, void* dst, size_t dst_bytes);

/* Split-precision forms.  fp16 carries 11 significant bits (what the reference's cuDNN path gets from TF32); where the
 * north-star Dice bar needs more, a tensor is stored as two 16-bit planes per voxel, [hi | lo] with hi = rn16(x) and
 * lo = rn16(x - hi) (2*C channels, ~22 bits), and a layer K-concatenates `terms` products in the same accumulator:
 *   terms 1: a*w                       (sources may still be split tensors: only their hi plane is read)
 *   terms 2: (a_hi + a_lo) * w         (sources must be split)
 *   terms 3: a_hi*w_hi + a_lo*w_hi + a_hi*w_lo   (fp32-faithful; weights packed as hi + lo too)
 * in_split: the sources are [hi | lo] tensors; out_split: write the output as a [hi | lo] tensor (dense NDHWC with
 * 2*cout channels).  pointwise as above (2 = ConvTranspose3d(k2,s2), out on the 2x grid); region may be NULL.
 * plan[10]: the 9 values of oai_conv3d_igemm_plan + the packed size in 16-byte units. */
OAI_API int oai_conv3d_igemm_plan_ex(int D, int H, int W, int c0, int c1, int cout, int pointwise, int terms, int flags,
                                     int* plan);
OAI_API int oai_pack_conv_weights_ex(const float* w, int cout, int c0, int c1, int D, int H, int W, int pointwise,
                                     int terms, int ab_format, int flags, void* dst, size_t dst_bytes);
OAI_API int oai_conv3d_igemm_ex(const void* src0, int c0, const void* src1, int c1, int in_split, int NT, int D, int H,
                                int W, const void* wpack, size_t wpack_bytes, const float* bias, int cout,
                                int pointwise, int relu, int ab_format, int terms, void* out, int out_split, int flags,
                                const int* region, void* stream);

/* fp16 saturation guard: how many epilogue threads of the conv kernel (on the current device, since the last reset) saw
 * an activation outside the fp16 range (|x| > 65504, or NaN) before rounding it.  Non-zero means the 16-bit tensors hold
 * inf: re-run with ab_format = 1 (bf16).  Synchronises `stream`. */
OAI_API int oai_conv_overflow_count(long long* count, int reset, void* stream);

/* Per-launch timing of oai_conv3d_igemm with CUDA events on the launch stream (bench.py's roofline numbers):
 * between begin and end every conv launch is bracketed by an event pair; end waits for them and returns the summed
 * kernel time, the number of launches, their algorithmic FLOPs (2*voxels*cout*cin*taps over the whole layer, i.e. what
 * the reference executes) and the FLOPs actually issued (dead-halo rows skipped, see oai_conv3d_igemm_region). */
OAI_API int oai_profile_begin(void);
OAI_API int oai_profile_end(double* conv_ms, long long* conv_launches, double* conv_flops, double* conv_exec_flops);
/* launch i of the current profile (call before oai_profile_end): kernel ms, algorithmic and issued FLOPs */
OAI_API int oai_profile_entry(int i, double* ms, double* flops, double* exec_flops);

/* Tiling geometry arrays used below (all z,y,x): geom[12] = {tile[3], effective[3], overlap[3], grid[3]} exactly as
 * Partition computes them (image_transforms.py:389-391,404-406); vol_dims[3] = image size. */

/* Partition.__call__ (image_transforms.py:408-446: reflect pad + overlap tiling) fused with the first UNet layer
 * ec0 = Conv3d(1->c0,k3,p1)[+BN]+ReLU (networks.py:43,84-86).  Reads the float32 volume in place (tiles are never
 * materialised), writes act16 [ntiles, td, th, tw, c0] for tiles tile0 .. tile0+ntiles-1 (i-major tile order).
 * w27c: folded weights [27][c0] (tap = (kd*3+kh)*3+kw), bias [c0]. */
OAI_API int oai_seg_stem(const float* vol, const int* vol_dims, const int* geom, int tile0, int ntiles,
                         const float* w27c, const float* bias, int c0, void* out, int ab_format, void* stream);

/* nn.MaxPool3d(2) (networks.py:52-54) on act16 [N,D,H,W,C] -> [N,D/2,H/2,W/2,C]. */
OAI_API int oai_maxpool3d_2(const void* in, void* out, int N, int D, int H, int W, int C, int ab_format, void* stream);
/* Same on split tensors: in_split: the input is [hi | lo] (2C channels per voxel); out_split: the output too (the
 * winner is chosen by hi + lo and both halves are kept); in_split without out_split pools the hi plane only. */
OAI_API int oai_maxpool3d_2_ex(const void* in, void* out, int N, int D, int H, int W, int C, int in_split, int out_split,
                               int ab_format, void* stream);
/* oai_seg_stem writing a [hi | lo] tensor [ntiles, td, th, tw, 2*c0] when out_split != 0. */
OAI_API int oai_seg_stem_ex(const float* vol, const int* vol_dims, const int* geom, int tile0, int ntiles,
                            const float* w27c, const float* bias, int c0, void* out, int ab_format, int out_split,
                            void* stream);

/* dc0 = Conv3d(C->ncls,k1) (networks.py:66,148) + torch.sigmoid (segmenter.py:121) [+ ">0.5" when out_mode==1,
 * segmenter.py:123-124; out_mode==2 writes raw logits] + Partition.assemble (image_transforms.py:492-513): each tile's interior is written to its
 * place in out[ncls][VD][VH][VW] (float32), trimmed to the image, with the crop_zyx border shell set to 0. */
OAI_API int oai_seg_head(const void* act, int C, int ncls, const float* w, const float* b, float* out,
                         const int* vol_dims, const int* geom, int tile0, int ntiles, const int* crop_zyx, int out_mode,
                         int ab_format, void* stream);

/* ------------------------------------------------------------------------------------------------------------
 * Stage-level segmentation  (reference: Segmenter3DInPatchClassWise.segment, oai_analysis/segmentation/
 * segmenter.py:100-131, with pred_setup :51-62): two calls segment a volume; layer order, skip wiring, BatchNorm
 * folding, weight packing, dead-halo regions and the workspace layout live inside the library.
 * ------------------------------------------------------------------------------------------------------------ */
enum {
  OAI_SEG_PRECISION_FP16 = 0,    /* 16-bit operands everywhere (TF32-class mantissa, the reference's cuDNN default) */
  OAI_SEG_PRECISION_MIXED = 1,   /* default: dc2's skip input (ec1's output) and dc1's input are read as fp16 hi+lo */
  OAI_SEG_PRECISION_FP16X2 = 2,  /* every layer reads fp16 hi+lo activations (terms 2) */
  OAI_SEG_PRECISION_FP16X3 = 3,  /* fp32-faithful: activations and weights both hi+lo (terms 3) */
  OAI_SEG_PRECISION_CUSTOM = 4   /* layer_terms[] below */
};

typedef struct {
  int in_channels, n_classes, bias, BN;   /* training-config "model_setting" (segmenter.py:56) */
  int patch_xyz[3];                       /* training-config "patch_size" (x,y,z; segmenter.py:53) */
  int overlap_xyz[3];                     /* segmenter_config "overlap_size" (x,y,z; analysis_object.py:23) */
  int ab_format;                          /* 0 fp16, 1 bf16 */
  int precision;                          /* OAI_SEG_PRECISION_* */
  int layer_terms[17];                    /* CUSTOM only: terms of ec0..ec7, dc9..dc1 (ec0 is always exact): 1..3 as above;
                                           * 4 / 5 on a concatenating layer (dc8, dc5, dc2): only the skip / only the
                                           * upsampled source is read as hi+lo */
} oai_seg_config;

/* one entry of the reference's state_dict: float32, contiguous, host memory, torch layout */
typedef struct {
  const char* name;
  const float* data;
  int ndim;
  long long shape[5];
} oai_tensor;

typedef struct oai_seg_handle* oai_seg_t;

/* Dead-halo elimination (host arithmetic, no GPU): boxes[17][6] = inclusive {lo z,y,x, hi z,y,x} of the output
 * sub-box each layer ec0..ec7, dc9..dc1 must compute for the kept tile interior (the reference computes whole tiles
 * and crops afterwards, image_transforms.py:497-503); up-convs are boxed on their input grid, encoder layers whole. */
OAI_API int oai_seg_needed_regions(const int* tile_zyx, const int* overlap_zyx, int* boxes);
/* the per-layer terms a precision preset expands to (terms17[0] = ec0 ... terms17[16] = dc1) */
OAI_API int oai_seg_layer_terms(int precision, int* terms17);
/* UNet(in_channels, n_classes, bias, BN) + load_state_dict(strict=True) (networks.py:39-66, utils.py:20-41) on the
 * current device.  state_dict uses the reference's keys ("ec0.0.weight", "dc9.1.running_var", "dc0.bias", ...);
 * missing, mis-shaped or unexpected keys fail.  The handle owns the packed weights (about 40 MB). */
OAI_API int oai_seg_create(const oai_seg_config* cfg, const oai_tensor* state_dict, int n_tensors, oai_seg_t* handle);
OAI_API int oai_seg_destroy(oai_seg_t handle);
/* tiles Partition cuts the volume into (image_transforms.py:404-406) and the device workspace one forward needs when
 * tiles_per_batch tiles (<= 0: all) go through the network together */
OAI_API int oai_seg_num_tiles(oai_seg_t handle, const int* vol_dims);
OAI_API size_t oai_seg_workspace_bytes(oai_seg_t handle, const int* vol_dims, int tiles_per_batch);
/* vol: float32 [D][H][W] on the device; out: float32 [n_classes][D][H][W] (class 0 = FC, 1 = TC), out_mode 0 = sigmoid
 * probabilities, 1 = (p > 0.5) masks, 2 = logits.  workspace: 256-byte aligned device memory of at least
 * oai_seg_workspace_bytes(); asynchronous on `stream`. */
OAI_API int oai_seg_forward(oai_seg_t handle, const float* vol, const int* vol_dims, float* out, int out_mode,
                            int tiles_per_batch, void* workspace, size_t workspace_bytes, void* stream);

/* ------------------------------------------------------------------------------------------------------------
 * ICON / GradICON registration  (reference call sites: oai_analysis/registration.py:20,25,
 * oai_analysis/dask_processing.py:77,85; arithmetic in the un-vendored icon_registration==1.1.2, pyproject.toml:35)
 * All tensors float32, planar [N][C][D][H][W] with explicit batch / channel strides (elements) so a layer reads and
 * writes channel slices of the UNet's concatenation buffers in place.  dims arrays are z,y,x.
 * ------------------------------------------------------------------------------------------------------------ */

/* icon networks.UNet2 down step / lastConv: Conv3d(k3, p1, stride 1|2) on leaky_relu(in) (when leaky_in)
 * [+ pad_or_crop(avg_pool3d(in, 2, ceil_mode=True)) when residual], times out_scale.
 * w packed [cin][27][cout_pad] (tap = (kd*3+kh)*3+kw), bias [cout]. */
OAI_API int oai_reg_conv3(const float* in, long long in_nstride, long long in_cstride, int cin, const int* in_dims,
                          const float* w, const float* bias, float* out, long long out_nstride, long long out_cstride,
                          int cout, int cout_pad, int N, int stride, int leaky_in, int residual, float out_scale,
                          void* workspace, size_t workspace_bytes, void* stream);

/* The strided down step (stride 2, leaky input, avg-pool residual, out_scale 1) on the 5th-generation tensor cores
 * (tcgen05.mma, accumulator in TMEM, split-fp16 operands: fp32-level accuracy) for cin a multiple of 16, cout 32 or a
 * multiple of 64 (<= 512), cout >= cin and an output lattice of at least 8 x 8.  oai_reg_pack_conv3_umma turns
 * w [cin][27][cout_pad] fp32 (device) into the kernel's pre-swizzled weight blocks (oai_reg_conv3_umma_wbytes bytes,
 * 16-byte aligned; wexp chosen as for oai_reg_pack_convt4).  workspace: oai_reg_conv3_umma_workspace bytes, 128-byte
 * aligned (the layer input as eight parity planes, channels-last hi / lo fp16). */
OAI_API size_t oai_reg_conv3_umma_wbytes(int cin, int cout);
OAI_API size_t oai_reg_conv3_umma_workspace(int cin, const int* in_dims, int N);
OAI_API int oai_reg_pack_conv3_umma(const float* w, int cin, int cout, int cout_pad, int wexp, void* dst, void* stream);
OAI_API int oai_reg_conv3_umma(const float* in, long long in_nstride, long long in_cstride, int cin,
                               const int* in_dims, const void* wumma, int wexp, const float* bias, float* out,
                               long long out_nstride, long long out_cstride, int cout, int N, void* workspace,
                               size_t workspace_bytes, void* stream);

/* Optional device scratch for oai_reg_conv3 (may be NULL / 0): with oai_reg_conv3_workspace(...) bytes the deep
 * levels (stride 2, cin >= 64, at most 4096 output voxels over the batch: weight-streaming GEMMs) run split-K over
 * blocks with a fixed-order (deterministic) reduction; returns 0 for layers that do not use it. */
OAI_API size_t oai_reg_conv3_workspace(int cin, int cout, const int* in_dims, int N, int stride, int leaky_in);

/* icon networks.UNet2 up step: BatchNorm3d(eval)( ConvTranspose3d(k4,s2,p1)(leaky_relu(in)) +
 * F.interpolate(in[:, :cout], scale_factor=2, trilinear, align_corners=False) ), cropped to out_dims.
 * w packed [cin][64][cout] (tap = (kd*4+kh)*4+kw); bn_scale = gamma/sqrt(var+eps), bn_shift = beta - mean*bn_scale. */
OAI_API int oai_reg_convt4(const float* in, long long in_nstride, long long in_cstride, int cin, const int* in_dims,
                           const float* w, const float* bias, const float* bn_scale, const float* bn_shift, float* out,
                           long long out_nstride, long long out_cstride, int cout, const int* out_dims, int N,
                           void* stream);

/* Split-fp16 weights for oai_reg_convt4_mma: w [cin][64][cout] fp32 (device) -> wpk (device, cin*64*cout*4 bytes,
 * 16-byte aligned): mma.sync.m16n8k16 B fragments [cout/16][cin/16][64 taps, kernel visit order][2 n-tiles][32 lanes] x (hi k0-7, hi k8-15,
 * lo k0-7, lo k8-15), each weight scaled by 2^wexp before the hi/lo fp16 split (choose wexp so that
 * max|w| * 2^wexp is in [2^13, 2^14): lo then stays clear of fp16 subnormals).  cin, cout multiples of 16. */
OAI_API int oai_reg_pack_convt4(const float* w, int cin, int cout, int wexp, void* wpk, void* stream);

/* Same operator as oai_reg_convt4 (icon networks.UNet2 up step) on the tensor path: implicit GEMM with
 * mma.sync.m16n8k16, operands split into fp16 hi + lo pairs (hi*hi + lo*hi + hi*lo, fp32 accumulate: fp32-level
 * accuracy).  Levels narrower than 12 input points run as split-K fp32 GEMMs on w (deterministic reduction);
 * workspace: see
 * oai_reg_convt4_mma_workspace (16-byte aligned). */
OAI_API int oai_reg_convt4_mma(const float* in, long long in_nstride, long long in_cstride, int cin,
                               const int* in_dims, const float* w, const void* wpk, int wexp, const float* bias,
                               const float* bn_scale, const float* bn_shift, float* out, long long out_nstride,
                               long long out_cstride, int cout, const int* out_dims, int N, void* workspace,
                               size_t workspace_bytes, void* stream);

/* The same up step on the 5th-generation tensor cores (tcgen05.mma, accumulators in TMEM) for the wide levels:
 * cout in {16, 32, 64, 128}, cin a multiple of 16, cout <= cin, lattice at least 8 x 8.  Split-fp16 operands as above
 * (fp32-level accuracy).  oai_reg_pack_convt4_umma turns w [cin][64][cout] fp32 (device) into the kernel's pre-swizzled
 * weight blocks (oai_reg_convt4_umma_wbytes(cin, cout) bytes, 16-byte aligned; wexp as for oai_reg_pack_convt4).
 * workspace: N * cin * D * H * W * 4 bytes, 128-byte aligned (the layer input as channels-last hi / lo fp16). */
OAI_API size_t oai_reg_convt4_umma_wbytes(int cin, int cout);
OAI_API int oai_reg_pack_convt4_umma(const float* w, int cin, int cout, int wexp, void* dst, void* stream);
OAI_API int oai_reg_convt4_umma(const float* in, long long in_nstride, long long in_cstride, int cin,
                                const int* in_dims, const void* wumma, int wexp, const float* bias,
                                const float* bn_scale, const float* bn_shift, float* out, long long out_nstride,
                                long long out_cstride, int cout, const int* out_dims, int N, void* workspace,
                                size_t workspace_bytes, void* stream);

/* Bytes of caller-owned device scratch oai_reg_convt4_mma needs: the layer input rewritten once as leaky-ReLU'd
 * hi / lo fp16 channel pairs (N * cin * D * H * W * 4), or, for levels narrower than 12 points, the split-K partial
 * sums of their fp32 GEMM form. */
OAI_API size_t oai_reg_convt4_mma_workspace(int cin, int cout, const int* in_dims, int N);

/* Composition of displacement maps and image warp, fused (icon network_wrappers.TwoStepRegistration /
 * FunctionFromVectorField closures; mermaidlite.compute_warped_image_multiNC == F.grid_sample(bilinear, border,
 * align_corners=True) at 2c-1).  Starting from the identity map of grid_dims (coordinates in [0,1], channel order
 * z,y,x), applies c <- c + S(fields[k], c) for k = 0..nfields-1 (fields[k] is [3][field_dims[3k..3k+2]]); with
 * shortcut_first the first field is added without interpolation (FunctionFromVectorField's identity shortcut).
 * Writes the map to phi_out [3][D][H][W] and/or S(img, c) to img_out [D][H][W] (either may be NULL). */
OAI_API int oai_compose(const int* grid_dims, int nfields, const float* const* fields, const int* field_dims,
                        int shortcut_first, const float* img, const int* img_dims, float* phi_out, float* img_out,
                        void* stream);

/* itk_wrapper.register_pair's F.interpolate(size=..., mode="trilinear", align_corners=False), one channel. */
OAI_API int oai_resize_trilinear(const float* in, const int* in_dims, float* out, const int* out_dims, void* stream);

/* DownsampleRegistration's F.avg_pool3d(x, 2, ceil_mode=True) on [C][D][H][W]. */
OAI_API int oai_avgpool3d_2_ceil(const float* in, int C, const int* in_dims, float* out, void* stream);

/* itk_wrapper.create_itk_transform: disp[z][y][x][(x,y,z)] = (phi - identity)[(2,1,0)] * (N - 1), float32. */
OAI_API int oai_displacement_field(const float* phi, const int* dims, float* disp, void* stream);

/* ------------------------------------------------------------------------------------------------------------
 * Stage-level registration  (reference: ICON_Registration.__init__ / register, oai_analysis/registration.py:18-27,
 * i.e. icon_registration.pretrained_models.OAI_knees_gradICON_model + itk_wrapper.register_pair; worker-side call
 * sites oai_analysis/dask_processing.py:77,85): two calls register a pair in both directions; the module tree, the
 * tallUNet2 layer order, concatenation buffers, BatchNorm folding, weight packing, the TwoStep / Downsample closures
 * and the workspace layout live inside the library.
 * ------------------------------------------------------------------------------------------------------------ */
typedef struct oai_reg_handle* oai_reg_t;

/* Host arithmetic only (no GPU): validates a regis_net state dict exactly as oai_reg_create does and writes the module
 * tree it encodes, e.g. "TwoStep(TwoStep(Down(TwoStep(FFVF, FFVF)), FFVF), FFVF)".  Keys are icon's own paths
 * ("regis_net." prefix optional): netPhi / netPsi = TwoStepRegistration children, net = DownsampleRegistration.net or,
 * at the end of a path, FunctionFromVectorField.net (a tallUNet2: downConvs.N / upConvs.N / batchNorms.N / lastConv).
 * "identity_map" buffers and "num_batches_tracked" counters are skipped; any other tensor outside a tallUNet2, an
 * incomplete or mis-shaped tallUNet2, or a TwoStep with one child fails (nothing ever "loads" partially). */
OAI_API int oai_reg_parse_tree(const oai_tensor* state_dict, int n_tensors, char* description,
                               size_t description_bytes);
/* pretrained_models.OAI_knees_gradICON_model's regis_net + assign_identity_map([1,1,*net_dims]) on the current device
 * (net_dims z,y,x; the knee model uses 80,192,192).  The handle owns the packed weights (about 150 MB per tallUNet2);
 * the state dict is not referenced after the call. */
OAI_API int oai_reg_create(const oai_tensor* state_dict, int n_tensors, const int* net_dims, oai_reg_t* handle);
OAI_API int oai_reg_destroy(oai_reg_t handle);
OAI_API int oai_reg_describe(oai_reg_t handle, char* description, size_t description_bytes);
OAI_API size_t oai_reg_workspace_bytes(oai_reg_t handle);
/* itk_wrapper.register_pair(model, image_A, image_B) on device-resident float32 volumes [dims] (z,y,x) of any size:
 * both are resized to net_dims (F.interpolate trilinear, align_corners=False), both directions run batched through
 * the cascade.  Outputs, each optional (NULL): phi_AB / phi_BA = model.phi_AB(identity_map) / phi_BA(...), float32
 * [3][net_dims] in [0,1] coordinates (channels z,y,x); disp_AB / disp_BA = create_itk_transform's displacement
 * fields, float32 [net_dims][3] (x,y,z components, network-voxel units) as oai_warp_volume / oai_warp_points take
 * them.  workspace: 256-byte aligned device memory of at least oai_reg_workspace_bytes(); asynchronous on `stream`.
 * The cascade's own displacement fields stay in the workspace until the next forward (oai_reg_field). */
OAI_API int oai_reg_forward(oai_reg_t handle, const float* image_A, const int* dims_A, const float* image_B,
                            const int* dims_B, float* phi_AB, float* phi_BA, float* disp_AB, float* disp_BA,
                            void* workspace, size_t workspace_bytes, void* stream);
/* The cascade's displacement fields in application order (first applied first): field `index` is float32
 * [2 directions][3][dims] at workspace + *workspace_offset (valid after oai_reg_forward on that workspace). */
OAI_API int oai_reg_num_fields(oai_reg_t handle);
OAI_API int oai_reg_field(oai_reg_t handle, int index, size_t* workspace_offset, int* dims);
/* as_function(image)(phi(identity_map)) for the last pair registered on `workspace`: image [dims] (any size) warped
 * by phi_AB (direction 0) or phi_BA (1), fused with the composition (no map is materialised). */
OAI_API int oai_reg_warp_image(oai_reg_t handle, const float* image, const int* dims, int direction, float* out,
                               void* workspace, size_t workspace_bytes, void* stream);

/* Registration quality: the terms of icon_registration's GradientICON.forward(A, B), i.e. its ICONLoss tuple, for the
 * last pair oai_reg_forward registered on reg_workspace (read only; nothing is written into it).  At the network shape:
 *   similarity          = sim(S(A, phi_AB), B) + sim(S(B, phi_BA), A) on the resized pair, sim = LNCC(sigma) (Gaussian
 *                         of 2*floor(2*sigma)+1 taps, zero padding) or ssd_only_interpolated (in-bounds tag warped
 *                         with the image);
 *   inverse consistency = sum_d mean(((e(Ie) - e(Ie + delta*e_d)) / delta)^2), e(c) = c - phi_AB(phi_BA(c)),
 *                         Ie = identity + noise / W, noise: device float32 [3][net_dims] of N(0, 1) values;
 *   transform magnitude = mean((identity - phi_AB)^2);  flips = #{dV < 0} of phi_BA (losses.flips);
 *   all                 = lmbda * inverse consistency + similarity.
 * terms: device double[5] in ICONLoss order (all, inverse consistency, similarity, transform magnitude, flips).
 * jac_det_BA (optional): device float32 [D-1][H-1][W-1], the dV map of phi_BA.  loss_workspace: 256-byte aligned
 * device memory of oai_reg_loss_workspace_bytes(handle, cfg) bytes (oai_reg_workspace_bytes is unaffected).
 * Fixed-order reductions (equal inputs give bitwise equal terms); no host synchronisation, no allocation. */
#define OAI_SIM_LNCC 0
#define OAI_SIM_SSD_ONLY_INTERPOLATED 1
typedef struct {
  int similarity;   /* OAI_SIM_LNCC or OAI_SIM_SSD_ONLY_INTERPOLATED */
  double sigma;     /* LNCC Gaussian sigma in voxels, 0 < sigma < 12.5 (ignored by ssd_only_interpolated) */
  double lmbda;     /* weight of the inverse-consistency term in `all` */
  double delta;     /* finite-difference step of the gradient-ICON term (icon: 1e-3) */
} oai_icon_loss_cfg;
OAI_API size_t oai_reg_loss_workspace_bytes(oai_reg_t handle, const oai_icon_loss_cfg* cfg);
OAI_API int oai_reg_icon_loss(oai_reg_t handle, const oai_icon_loss_cfg* cfg, const float* noise, double* terms,
                              float* jac_det_BA, void* loss_workspace, size_t loss_workspace_bytes,
                              const void* reg_workspace, size_t reg_workspace_bytes, void* stream);
/* losses.flips on any map phi: device float32 [3][dims] (z,y,x channels): dV = ((a x b) . c) with forward differences
 * a, b, c along z, y, x at cells [1:, 1:, 1:]; *count_out (device int64) = #{dV < 0}, exact; det_out (optional) =
 * device float32 [D-1][H-1][W-1].  Every axis needs at least 2 samples. */
OAI_API int oai_jacobian_flips(const float* phi, const int* dims, float* det_out, long long* count_out, void* stream);

/* Segmentation quality: overlap and surface distances of two masks A and B on one grid dims = {D, H, W} (z, y, x),
 * every axis 1 to 512 voxels; spacing_xyz = {sx, sy, sz} in mm, positive and finite.  The definitions are medpy's
 * dc / assd / hd / hd95:
 *   surface  dM = M & ~binary_erosion(M, 6-connected cross, border_value=0): mask voxels on a volume face are surface;
 *   d_AB     = EDT to dB at the voxels of dA, d_BA likewise, in mm between voxel centres;
 *   dice     = 2|A & B| / (|A| + |B|);  assd = (mean d_AB + mean d_BA) / 2;  hd = max(max d_AB, max d_BA);
 *   hd95     = np.percentile(np.hstack((d_AB, d_BA)), 95), numpy's linear interpolation (an exact order statistic).
 * dice is NaN when both masks are empty; assd, hd, hd95 and the means and maxima are NaN when either is empty.
 * workspace: 256-byte aligned device memory of oai_seg_quality_workspace_bytes(dims) bytes (0 for unsupported dims);
 * it serves both calls.  Fixed-order reductions (equal inputs give bitwise equal terms); no host synchronisation, no
 * allocation. */
OAI_API size_t oai_seg_quality_workspace_bytes(const int* dims);
/* scipy.ndimage.distance_transform_edt(~feature, sampling=(sz, sy, sx)): out[v] = distance in mm from voxel v to the
 * nearest voxel with feature[v] != 0 (+inf everywhere when there is none).  feature: device uint8 [dims]; out: device
 * float32 [dims]. */
OAI_API int oai_distance_transform(const uint8_t* feature, const int* dims, const double* spacing_xyz, float* out,
                                   void* workspace, size_t workspace_bytes, void* stream);
/* mask_a, mask_b: device uint8 [dims], non-zero = inside.
 * terms: device double[8] = {dice, assd, hd95, hd, mean d_AB, mean d_BA, max d_AB, max d_BA};
 * counts: device int64[5] = {|A|, |B|, |A & B|, |dA|, |dB|};
 * dist_to_B / dist_to_A (optional, NULL to skip): device float32 [dims], the EDT maps to dB and to dA in mm. */
OAI_API int oai_surface_metrics(const uint8_t* mask_a, const uint8_t* mask_b, const int* dims,
                                const double* spacing_xyz, double* terms, long long* counts, float* dist_to_B,
                                float* dist_to_A, void* workspace, size_t workspace_bytes, void* stream);

/* Connected components of a mask on dims = {D, H, W} (z, y, x): every axis at least 1 voxel and D*H*W < 2^31.
 * connectivity 6, 18 or 26 is scipy.ndimage.generate_binary_structure(3, 1 / 2 / 3).  labels equal
 * scipy.ndimage.label(mask, structure)[0] bit for bit: background 0, components 1..n in raster (C) order of their first
 * voxel.  The workspace (256-byte aligned, oai_components_workspace_bytes(dims) bytes, 0 for unsupported dims) holds
 * the rank map and the scan partials; the labels buffer doubles as the union-find parent array.  Integer results only
 * (equal inputs give bitwise equal outputs); no host synchronisation, no allocation. */
OAI_API size_t oai_components_workspace_bytes(const int* dims);
/* Host-only upper bound on n, the length of the sizes buffer: ceil(D/2) ceil(H/2) ceil(W/2) for 26 (tight),
 * ceil(D*H*W / 2) for 6 (tight: the checkerboard) and 18.  0 for unsupported dims or connectivity. */
OAI_API long long oai_components_max(const int* dims, int connectivity);
/* mask: device uint8 [dims], non-zero = inside; labels: device int32 [dims];
 * sizes: device int32 [oai_components_max(dims, connectivity)], sizes[k - 1] = voxels of label k, zero past n;
 * count: device int64, n. */
OAI_API int oai_connected_components(const uint8_t* mask, const int* dims, int connectivity, int* labels, int* sizes,
                                     long long* count, void* workspace, size_t workspace_bytes, void* stream);
/* Keep policy on a labelled volume (labels, sizes, count of oai_connected_components): min_voxels < 0 keeps the largest
 * component only (the lowest label on a tie, numpy's argmax), min_voxels >= 0 every component of at least min_voxels
 * voxels.  The policy is read from the device-side sizes.  keep_mask (optional): device uint8 [dims], 1 = kept;
 * values (optional): device float32 [dims], zeroed in place outside the kept components.  At least one is needed. */
OAI_API int oai_keep_components(const int* labels, const int* sizes, const long long* count, const int* dims,
                                int min_voxels, uint8_t* keep_mask, float* values, void* stream);

/* ------------------------------------------------------------------------------------------------------------
 * ITK-semantics warps  (reference: oai_analysis/dask_processing.py:95-111 deform_probmap_delayed,
 * test/test_all.py:42-52; transform = R_A o DisplacementFieldTransform o R_B^-1 built by create_itk_transform)
 * Affines are row-major 3x4 [M | t] in float64 acting on (x,y,z).
 * ------------------------------------------------------------------------------------------------------------ */

/* itk.resample_image_filter(src, transform, LinearInterpolateImageFunction, output grid, default pixel):
 * out[c][j] = trilinear(src[c], net_to_src_index( q + D(q) )), q = out_index_to_net(j); D = identity outside the
 * field buffer; neighbours clamped to the edge; default_value outside [-0.5, N-0.5). */
OAI_API int oai_warp_volume(const float* src, int C, const int* src_dims, const float* disp, const int* field_dims,
                            const double* out_index_to_net, const double* net_to_src_index, float* out,
                            const int* out_dims, float default_value, void* stream);

/* itk CompositeTransform::TransformPoint on n physical points (float64 x,y,z): out = net_to_phys(q + D(q)),
 * q = phys_to_net(p).  (Mesh-vertex warp, reference README.md:34 / SURVEY 3.4.) */
OAI_API int oai_warp_points(const double* pts, long long n, const float* disp, const int* field_dims,
                            const double* phys_to_net, const double* net_to_phys, double* out, void* stream);

/* ------------------------------------------------------------------------------------------------------------
 * Intensity pre-normalisation (SURVEY 8f-1; oai_analysis/dask_processing.py:10-26 image_normalize, called at :75 and
 * :177 right before registration and segmentation):
 *   wmin, wmax = np.percentile(volume, perc_lo), np.percentile(volume, perc_hi)      (numpy "linear" method)
 *   out = itk.IntensityWindowingImageFilter(window [wmin, wmax] -> [out_min, out_max])
 * in / out: n float32 voxels on the device (in 16-byte aligned; out may alias in).  The order statistics come from an
 * exact three-pass radix select on the device, no host synchronisation.  workspace: oai_intensity_window_workspace()
 * bytes of device memory, 8-byte aligned; afterwards it holds the window, readable with oai_intensity_window_result
 * (copies {wmin, wmax} to the host and synchronises the stream).
 * ------------------------------------------------------------------------------------------------------------ */
OAI_API size_t oai_intensity_window_workspace(void);
OAI_API int oai_intensity_window(const float* in, long long n, double perc_lo, double perc_hi, float out_min,
                                 float out_max, float* out, void* workspace, size_t workspace_bytes, void* stream);
OAI_API int oai_intensity_window_result(const void* workspace, double* window_host, void* stream);

/* ------------------------------------------------------------------------------------------------------------
 * Iso-surface extraction of the atlas-space probability maps (SURVEY 8f-2): skimage.measure.marching_cubes(level,
 * spacing, step_size=1, gradient_direction) of oai_analysis/mesh_processing.py:325-340 (get_mesh) and the
 * vtkPolyDataConnectivityFilter region filter of mesh_processing.py:102-146 (get_vtk_mesh keeps regions with more than
 * 3000 cells).  vol: float32 [D][H][W] on the device (z,y,x, the array the reference swaps to x,y,z before the call);
 * vertices come out as (x*sx, y*sy, z*sz) float32, one per crossed lattice edge; faces are int32 vertex triples wound so
 * that normals point to ascending values when ascent != 0.  Ambiguous faces use the asymptotic decider.
 * Two calls: oai_mc_count classifies, scans and returns {n_verts, n_faces} on the host (synchronises the stream);
 * oai_mc_emit writes them into caller buffers of that size using the SAME workspace (oai_mc_workspace_bytes, 256-byte
 * aligned, untouched in between).
 * ------------------------------------------------------------------------------------------------------------ */
OAI_API size_t oai_mc_workspace_bytes(const int* dims);
OAI_API int oai_mc_count(const float* vol, const int* dims, float level, void* workspace, size_t workspace_bytes,
                         long long* counts_host, void* stream);
OAI_API int oai_mc_emit(const float* vol, const int* dims, float level, const double* spacing_xyz, int ascent,
                        void* workspace, size_t workspace_bytes, float* verts, int* faces, void* stream);
/* the generated polygon table (host, no GPU): 256 corner patterns x 64 face resolutions x 32 bytes
 * {n_triangles, 3 edge ids per triangle ...}; edge id = 4*axis + (u + 2v) */
OAI_API int oai_mc_table(uint8_t* table, size_t bytes);
/* get_vtk_mesh's region filter: connected components of the faces over shared vertices; components with MORE than
 * min_cells faces are kept, vertices compacted and faces re-indexed.  out_verts / out_faces must hold n_verts / n_faces
 * entries; counts_host receives {kept verts, kept faces} (synchronises the stream). */
OAI_API size_t oai_mesh_regions_workspace_bytes(long long n_verts, long long n_faces);
OAI_API int oai_mesh_keep_large_regions(const float* verts, long long n_verts, const int* faces, long long n_faces,
                                        int min_cells, void* workspace, size_t workspace_bytes, float* out_verts,
                                        int* out_faces, long long* counts_host, void* stream);

/* ------------------------------------------------------------------------------------------------------------
 * Mesh post-processing (SURVEY 8f-3; oai_analysis/mesh_processing.py).  Meshes are (verts float32 [n][3], faces int32
 * [m][3]) on the device; workspaces are caller-owned, 256-byte aligned.
 * ------------------------------------------------------------------------------------------------------------ */
/* smooth_mesh (mesh_processing.py:298-306): vtkSmoothPolyDataFilter(NumberOfIterations, RelaxationFactor = 0.01 by
 * default, feature-edge smoothing off): x <- x + f * (mean(unique edge neighbours) - x), positions float32 between
 * iterations.  Jacobi sweeps (VTK sweeps in place); vertices on open boundary edges stay fixed. */
OAI_API size_t oai_mesh_smooth_workspace_bytes(long long n_verts, long long n_faces);
OAI_API int oai_mesh_smooth(const float* verts, long long n_verts, const int* faces, long long n_faces, int iterations,
                            float relaxation, void* workspace, size_t workspace_bytes, float* out_verts, void* stream);
/* get_cell_normals / get_cell_centroid (mesh_processing.py:25-47): unit face normals (right-hand rule, zero for a
 * degenerate face) and face centroids, float32 [m][3] each. */
OAI_API int oai_mesh_face_features(const float* verts, const int* faces, long long n_faces, float* normals,
                                   float* centroids, void* stream);
/* get_distance (mesh_processing.py:310-321, vtkDistancePolyDataFilter, unsigned): for every point the distance to the
 * closest point ON the target mesh's triangles. */
OAI_API int oai_mesh_distance(const float* points, long long n_points, const float* verts, const int* faces,
                              long long n_faces, float* dist, void* stream);
/* KMeans(n_clusters = 2, algorithm = "lloyd") of split_*_cartilage_surface (mesh_processing.py:197-294) on float32
 * features [n][dim], dim <= 16: Lloyd iterations from a deterministic farthest-point initialisation until no label
 * changes (or max_iter).  labels int32 [n] in {0, 1}; which cluster is 0 is arbitrary, as with sklearn (the callers
 * re-orient by the normals).  Synchronises the stream; iterations_host (may be NULL) receives the sweeps done. */
OAI_API size_t oai_kmeans2_workspace_bytes(int dim);
OAI_API int oai_kmeans2(const float* features, long long n, int dim, int max_iter, int* labels, void* workspace,
                        size_t workspace_bytes, int* iterations_host, void* stream);

/* ---- atlas attribute mapping and 2-D projection of the thickness maps (SURVEY 8f-4) ------------------------------------ */
/* map_attributes (mesh_processing.py:398-406): vtkPointInterpolator with its default vtkLinearKernel (footprint RADIUS,
 * radius 1.0 in the reference) and SetNullPointsStrategyToClosestPoint: out[t] = mean of source_attr over the source
 * points within `radius` of target point t (distance <= radius), or the attribute of the closest source point when
 * none is in range.  source_attr / out are float32 [n][n_attr], n_attr <= 4. */
OAI_API int oai_mesh_map_attributes(const float* source_points, const float* source_attr, long long n_source,
                                    int n_attr, const float* target_points, long long n_target, float radius,
                                    float* out, void* stream);
/* 256-byte device scratch (256-byte aligned) of the two projection helpers below. */
OAI_API size_t oai_mesh_project_workspace_bytes(void);
/* compute_least_square_circle (mesh_processing.py:409-443, scipy.optimize.leastsq from the centroid): least-squares
 * circle through coordinates (coord_x, coord_y) of the float32 points [.,3] selected by `index` (int32 [n], or NULL for
 * the first n points).  Gauss-Newton on the same residual and Jacobian; the sums run on the device, the 2x2 solves on
 * the host, so the call synchronises the stream.  center_host[2], radius_host / iterations_host (may be NULL). */
OAI_API int oai_circle_fit(const float* points, const int* index, long long n, int coord_x, int coord_y,
                           double* center_host, double* radius_host, int* iterations_host, void* workspace,
                           size_t workspace_bytes, void* stream);
/* get_projection_from_circle_and_vertice (mesh_processing.py:455-476): angle[i] = atan2(p[coord_y] - center_y,
 * p[coord_x] - center_x), height[i] = p[coord_z]; float64 [n] device outputs. */
OAI_API int oai_cylinder_project(const float* points, long long n, int coord_x, int coord_y, int coord_z,
                                 double center_x, double center_y, double* angle, double* height, void* stream);
/* The tibial branch of project_thickness (mesh_processing.py:497-534) for one plateau: sklearn KernelPCA(n_components=2)
 * with its default linear kernel = the first two principal-component scores of the selected points (each column signed
 * so its largest-magnitude entry is positive), then rotate_embedded(rotate_deg), optional x mirror, offset.  float64 [n]
 * device outputs in the order of `index` (NULL: the first n points).  Synchronises the stream (3x3 eigenproblem on the
 * host). */
OAI_API int oai_pca2_project(const float* points, const int* index, long long n, double rotate_deg, int mirror_x,
                             double offset_x, double offset_y, double* out_x, double* out_y, void* workspace,
                             size_t workspace_bytes, void* stream);

#ifdef __cplusplus
}
#endif
#endif /* OAI_B200_H_ */
