// Registration-stage kernels (fp32 / fp64, CUDA cores -- these ops are bandwidth- or latency-bound, no tensor cores):
//   * conv3 / convt4      : the layers of icon_registration's tallUNet2 (networks.UNet2.forward) with its residual
//                           avg-pool / trilinear-upsample shortcuts, BatchNorm(eval), leaky-ReLU and crops fused in
//   * chain               : composition of displacement maps  c <- c + S(u_k, c)  and the final image warp
//                           (network_wrappers.TwoStepRegistration closures + mermaidlite.compute_warped_image_multiNC
//                            == F.grid_sample(bilinear, border, align_corners=True))
//   * resize / avgpool    : register_pair's F.interpolate(trilinear, align_corners=False) and
//                           DownsampleRegistration's avg_pool3d(2, ceil_mode=True)
//   * disp_field          : itk_wrapper.create_itk_transform's (phi - id) * (N - 1), components reversed to x,y,z
//   * warp_volume/points  : itk.resample_image_filter / TransformPoint through R_A o DisplacementField o R_B^-1
//                           (oai_analysis/dask_processing.py:100-109), float64 coordinate arithmetic
#include <cuda_fp16.h>

#include <type_traits>

#include <cuda.h>

#include "api_common.h"
#include "ptx.cuh"
#include "reg_kernels.cuh"
#include "reg_sample.cuh"

#include <cmath>
#include <cstdlib>

namespace oai {

namespace {

__device__ __forceinline__ float leaky(float v) { return v > 0.f ? v : 0.01f * v; }

__device__ __forceinline__ void cp_async_4(float* smem_dst, const float* gsrc, bool valid) {
  const uint32_t d = static_cast<uint32_t>(__cvta_generic_to_shared(smem_dst));
  const int sz = valid ? 4 : 0;  // src-size 0 -> zero fill
  asm volatile("cp.async.ca.shared.global [%0], [%1], 4, %2;" ::"r"(d), "l"(gsrc), "r"(sz) : "memory");
}
__device__ __forceinline__ void cp_async_16(float* smem_dst, const float* gsrc) {
  const uint32_t d = static_cast<uint32_t>(__cvta_generic_to_shared(smem_dst));
  asm volatile("cp.async.cg.shared.global [%0], [%1], 16;" ::"r"(d), "l"(gsrc) : "memory");
}
__device__ __forceinline__ void cp_async_commit() { asm volatile("cp.async.commit_group;" ::: "memory"); }
template <int N>
__device__ __forceinline__ void cp_async_wait() { asm volatile("cp.async.wait_group %0;" ::"n"(N) : "memory"); }


// ------------------------------------------------------------------------------------------------ conv k3
// Register-tiled direct convolution: a thread produces XS x-adjacent outputs for CO_T output channels, so every
// weight vector read from shared memory feeds XS FMAs per channel and every input value feeds up to 3*CO_T.
// KS > 1 splits the input channels of each chunk over KS thread groups (reduced through shared memory at the end):
// the deep levels have few voxels and hundreds of channels, so the serial chain per thread is what limits them.
template <int CO_T, int XS, int STRIDE, int KS>
__global__ void __launch_bounds__(128) conv3_kernel(const Conv3Params p) {
  constexpr int CI_CHUNK = KS > 1 ? 16 : 8;
  constexpr int NIN = (XS - 1) * STRIDE + 3;
  constexpr int NV = 128 / KS;
  constexpr int CO_S = CO_T == 3 ? 4 : CO_T;   // shared-memory stride of a tap's weights: three channels padded to one
                                               // 16-byte vector (lastConv is bound by the L1 / shared-memory pipe)
  __shared__ __align__(16) float s_w[CI_CHUNK * 27 * CO_S];
  __shared__ float s_red[KS > 1 ? (KS - 1) * NV * XS * CO_T : 1];
  const int co0 = blockIdx.y * CO_T;
  const int n = blockIdx.z;
  const int nsx = (p.Wo + XS - 1) / XS;
  const long long nthr = static_cast<long long>(p.Do) * p.Ho * nsx;
  const int ks = threadIdx.x / NV, lv = threadIdx.x % NV;
  const long long v = blockIdx.x * static_cast<long long>(NV) + lv;
  const bool active = v < nthr;
  int sx = 0, yo = 0, zo = 0;
  if (active) {
    sx = static_cast<int>(v % nsx);
    yo = static_cast<int>((v / nsx) % p.Ho);
    zo = static_cast<int>(v / (static_cast<long long>(nsx) * p.Ho));
  }
  const int xo0 = sx * XS;
  const int xi0 = xo0 * STRIDE - 1, yi0 = yo * STRIDE - 1, zi0 = zo * STRIDE - 1;
  const bool vec_ok = (p.Wi & 3) == 0 && (p.in_cstride & 3) == 0 && (p.in_nstride & 3) == 0 &&
                      (reinterpret_cast<uintptr_t>(p.in) & 15) == 0;
  float acc[XS][CO_T];
#pragma unroll
  for (int i = 0; i < XS; ++i)
#pragma unroll
    for (int j = 0; j < CO_T; ++j) acc[i][j] = 0.f;
  const float* in_n = p.in + n * p.in_nstride;
  for (int ci0 = 0; ci0 < p.cin; ci0 += CI_CHUNK) {
    const int nci = min(CI_CHUNK, p.cin - ci0);
    __syncthreads();
    for (int i = threadIdx.x; i < nci * 27 * CO_S; i += blockDim.x) {
      const int j = i % CO_S, k = (i / CO_S) % 27, c = i / (CO_S * 27);
      const int co = co0 + j;
      s_w[i] = (j < CO_T && co < p.cout_pad) ? p.w[(static_cast<size_t>(ci0 + c) * 27 + k) * p.cout_pad + co] : 0.f;
    }
    __syncthreads();
    if (!active) continue;
    for (int c = ks; c < nci; c += KS) {
      const float* plane = in_n + (ci0 + c) * p.in_cstride;
      const float* wc = s_w + c * 27 * CO_S;
      // one (kd, kh) input row: NIN x-adjacent samples (zeros outside the volume), leaky ReLU applied on load
      auto load_row = [&](int r, float (&xin)[NIN]) {
        const int z = zi0 + r / 3, y = yi0 + r % 3;
        if (z < 0 || z >= p.Di || y < 0 || y >= p.Hi) {
#pragma unroll
          for (int i = 0; i < NIN; ++i) xin[i] = 0.f;
          return;
        }
        const float* row = plane + (static_cast<size_t>(z) * p.Hi + y) * p.Wi;
        if (XS * STRIDE % 4 == 0 && vec_ok) {
          // xi0 + 1 is a multiple of 4: aligned float4 loads for the body, scalars for the two halo samples
          xin[0] = xi0 >= 0 ? __ldg(row + xi0) : 0.f;
#pragma unroll
          for (int i = 0; i < (NIN - 1) / 4; ++i) {
            const float4 m = (xi0 + 1 + 4 * i < p.Wi) ? __ldg(reinterpret_cast<const float4*>(row + xi0 + 1) + i)
                                                      : make_float4(0.f, 0.f, 0.f, 0.f);
            xin[1 + 4 * i] = m.x; xin[2 + 4 * i] = m.y; xin[3 + 4 * i] = m.z; xin[4 + 4 * i] = m.w;
          }
#pragma unroll
          for (int i = 1 + 4 * ((NIN - 1) / 4); i < NIN; ++i) xin[i] = (xi0 + i < p.Wi) ? __ldg(row + xi0 + i) : 0.f;
        } else {
#pragma unroll
          for (int i = 0; i < NIN; ++i) {
            const int x = xi0 + i;
            xin[i] = (x >= 0 && x < p.Wi) ? __ldg(row + x) : 0.f;
          }
        }
        if (p.leaky_in) {
#pragma unroll
          for (int i = 0; i < NIN; ++i) xin[i] = leaky(xin[i]);
        }
      };
      // The nine rows are software-pipelined: row r + 1 is in flight while row r feeds its 3 * XS * CO_T FMAs.  Loading
      // and consuming one row at a time left every warp waiting a full L2 round trip per row (the 18 -> 3 last conv of
      // tallUNet2 ran at a third of the FMA rate).
      float xr[2][NIN];
      load_row(0, xr[0]);
#pragma unroll
      for (int r = 0; r < 9; ++r) {
        if (r + 1 < 9) load_row(r + 1, xr[(r + 1) & 1]);
        const float (&xin)[NIN] = xr[r & 1];
#pragma unroll
        for (int kw = 0; kw < 3; ++kw) {
          const float* wk = wc + (r * 3 + kw) * CO_S;
          float wv[CO_S];
          if (CO_S % 4 == 0) {   // one 16-byte shared-memory load per four channels
#pragma unroll
            for (int j = 0; j < CO_S / 4; ++j) {
              const float4 w4 = reinterpret_cast<const float4*>(wk)[j];
              wv[4 * j] = w4.x; wv[4 * j + 1] = w4.y; wv[4 * j + 2] = w4.z; wv[4 * j + 3] = w4.w;
            }
          } else {
#pragma unroll
            for (int j = 0; j < CO_T; ++j) wv[j] = wk[j];
          }
#pragma unroll
          for (int i = 0; i < XS; ++i)
#pragma unroll
            for (int j = 0; j < CO_T; ++j) acc[i][j] = fmaf(xin[i * STRIDE + kw], wv[j], acc[i][j]);
        }
      }
    }
  }
  if (KS > 1) {
    if (ks > 0) {
#pragma unroll
      for (int i = 0; i < XS; ++i)
#pragma unroll
        for (int j = 0; j < CO_T; ++j) s_red[((ks - 1) * NV + lv) * XS * CO_T + i * CO_T + j] = acc[i][j];
    }
    __syncthreads();
    if (ks > 0) return;
#pragma unroll
    for (int k = 1; k < KS; ++k)
#pragma unroll
      for (int i = 0; i < XS; ++i)
#pragma unroll
        for (int j = 0; j < CO_T; ++j) acc[i][j] += s_red[((k - 1) * NV + lv) * XS * CO_T + i * CO_T + j];
  }
  if (!active) return;
  float* out_n = p.out + n * p.out_nstride;
#pragma unroll
  for (int i = 0; i < XS; ++i) {
    const int xo = xo0 + i;
    if (xo >= p.Wo) break;
    const long long ovox = (static_cast<long long>(zo) * p.Ho + yo) * p.Wo + xo;
#pragma unroll
    for (int j = 0; j < CO_T; ++j) {
      const int co = co0 + j;
      if (co >= p.cout) break;
      float r = acc[i][j] + p.bias[co];
      if (p.residual) {
        const int cs = co - (p.cout - p.cin);  // zero padding sits in front of the pooled channels
        if (cs >= 0) {
          const float* plane = in_n + cs * p.in_cstride;
          float s = 0.f;
          int cnt = 0;
          for (int dz = 0; dz < 2; ++dz)
            for (int dy = 0; dy < 2; ++dy)
              for (int dx = 0; dx < 2; ++dx) {
                const int z = 2 * zo + dz, y = 2 * yo + dy, x = 2 * xo + dx;
                if (z < p.Di && y < p.Hi && x < p.Wi) {
                  s += plane[(static_cast<size_t>(z) * p.Hi + y) * p.Wi + x];
                  ++cnt;
                }
              }
          r += s / static_cast<float>(cnt);
        }
      }
      out_n[co * p.out_cstride + ovox] = r * p.out_scale;
    }
  }
}

// ------------------------------------------------------------------------------------------------ convT k4 s2 p1
// A thread produces XP x-adjacent output PAIRS (2*XP outputs) of one (zo, yo) row for CO_T channels.
// o = 2 i - 1 + k  =>  per axis two taps: k = (o+1)%2 + 2 t, i = (o + 1 - k)/2, t in {0,1}.
// Along x, output 2j uses (kx=1, ix=j), (kx=3, ix=j-1); output 2j+1 uses (kx=0, ix=j+1), (kx=2, ix=j).
template <int CO_T, int XP, int KS>
__global__ void __launch_bounds__(128) convt4_kernel(const ConvT4Params p) {
  constexpr int CI_CHUNK = KS > 1 ? 16 : 4;
  constexpr int NV = 128 / KS;
  __shared__ __align__(16) float s_w[CI_CHUNK * 64 * CO_T];
  __shared__ float s_red[KS > 1 ? (KS - 1) * NV * 2 * XP * CO_T : 1];
  const int co0 = blockIdx.y * CO_T;
  const int n = blockIdx.z;
  const int Wp = (p.Wo + 1) / 2;
  const int nsx = (Wp + XP - 1) / XP;
  const long long nthr = static_cast<long long>(p.Do) * p.Ho * nsx;
  const int ks = threadIdx.x / NV, lv = threadIdx.x % NV;
  const long long v = blockIdx.x * static_cast<long long>(NV) + lv;
  const bool active = v < nthr;
  int sx = 0, yo = 0, zo = 0;
  if (active) {
    sx = static_cast<int>(v % nsx);
    yo = static_cast<int>((v / nsx) % p.Ho);
    zo = static_cast<int>(v / (static_cast<long long>(nsx) * p.Ho));
  }
  const int j0 = sx * XP;
  const bool vec_ok = (p.Wi & 3) == 0 && (p.in_cstride & 3) == 0 && (p.in_nstride & 3) == 0 &&
                      (reinterpret_cast<uintptr_t>(p.in) & 15) == 0;
  int kz[2], iz[2], ky[2], iy[2];
#pragma unroll
  for (int t = 0; t < 2; ++t) {
    kz[t] = ((zo + 1) & 1) + 2 * t;
    iz[t] = (zo + 1 - kz[t]) / 2;
    ky[t] = ((yo + 1) & 1) + 2 * t;
    iy[t] = (yo + 1 - ky[t]) / 2;
  }
  float acc0[XP][CO_T], acc1[XP][CO_T];
#pragma unroll
  for (int i = 0; i < XP; ++i)
#pragma unroll
    for (int c = 0; c < CO_T; ++c) acc0[i][c] = acc1[i][c] = 0.f;
  const float* in_n = p.in + n * p.in_nstride;
  for (int ci0 = 0; ci0 < p.cin; ci0 += CI_CHUNK) {
    const int nci = min(CI_CHUNK, p.cin - ci0);
    __syncthreads();
    for (int i = threadIdx.x; i < nci * 64 * CO_T; i += blockDim.x) {
      const int c = i % CO_T, k = (i / CO_T) % 64, ci = i / (CO_T * 64);
      const int co = co0 + c;
      s_w[i] = co < p.cout ? p.w[(static_cast<size_t>(ci0 + ci) * 64 + k) * p.cout + co] : 0.f;
    }
    __syncthreads();
    if (!active) continue;
    for (int ci = ks; ci < nci; ci += KS) {
      const float* plane = in_n + (ci0 + ci) * p.in_cstride;
      const float* wc = s_w + ci * 64 * CO_T;
      // issue the loads of all four (tz, ty) input rows first (memory-level parallelism), then the FMAs
      float xin[4][XP + 2];
#pragma unroll
      for (int tz = 0; tz < 2; ++tz)
#pragma unroll
        for (int ty = 0; ty < 2; ++ty) {
          const int z = iz[tz], y = iy[ty];
          float* xr = xin[tz * 2 + ty];
          if (z < 0 || z >= p.Di || y < 0 || y >= p.Hi) {
#pragma unroll
            for (int i = 0; i < XP + 2; ++i) xr[i] = 0.f;
            continue;
          }
          const float* row = plane + (static_cast<size_t>(z) * p.Hi + y) * p.Wi;
          if (XP == 4 && vec_ok) {
            const float4 m = (j0 < p.Wi) ? __ldg(reinterpret_cast<const float4*>(row + j0))
                                         : make_float4(0.f, 0.f, 0.f, 0.f);
            xr[0] = j0 > 0 ? __ldg(row + j0 - 1) : 0.f;
            xr[1] = m.x; xr[2] = m.y; xr[3] = m.z; xr[4] = m.w;
            xr[XP + 1] = (j0 + 4 < p.Wi) ? __ldg(row + j0 + 4) : 0.f;
          } else {
#pragma unroll
            for (int i = 0; i < XP + 2; ++i) {
              const int x = j0 - 1 + i;
              xr[i] = (x >= 0 && x < p.Wi) ? __ldg(row + x) : 0.f;
            }
          }
        }
#pragma unroll
      for (int tz = 0; tz < 2; ++tz)
#pragma unroll
        for (int ty = 0; ty < 2; ++ty) {
          float* xr = xin[tz * 2 + ty];
#pragma unroll
          for (int i = 0; i < XP + 2; ++i) xr[i] = leaky(xr[i]);
          const float* wk = wc + ((kz[tz] * 4 + ky[ty]) * 4) * CO_T;
          float w0[CO_T], w1[CO_T], w2[CO_T], w3[CO_T];
#pragma unroll
          for (int c = 0; c < CO_T; ++c) {
            w0[c] = wk[c]; w1[c] = wk[CO_T + c]; w2[c] = wk[2 * CO_T + c]; w3[c] = wk[3 * CO_T + c];
          }
#pragma unroll
          for (int i = 0; i < XP; ++i)
#pragma unroll
            for (int c = 0; c < CO_T; ++c) {
              acc0[i][c] = fmaf(xr[i + 1], w1[c], acc0[i][c]);
              acc0[i][c] = fmaf(xr[i], w3[c], acc0[i][c]);
              acc1[i][c] = fmaf(xr[i + 2], w0[c], acc1[i][c]);
              acc1[i][c] = fmaf(xr[i + 1], w2[c], acc1[i][c]);
            }
        }
    }
  }
  if (KS > 1) {
    if (ks > 0) {
#pragma unroll
      for (int i = 0; i < XP; ++i)
#pragma unroll
        for (int c = 0; c < CO_T; ++c) {
          s_red[((ks - 1) * NV + lv) * 2 * XP * CO_T + (2 * i) * CO_T + c] = acc0[i][c];
          s_red[((ks - 1) * NV + lv) * 2 * XP * CO_T + (2 * i + 1) * CO_T + c] = acc1[i][c];
        }
    }
    __syncthreads();
    if (ks > 0) return;
#pragma unroll
    for (int k = 1; k < KS; ++k)
#pragma unroll
      for (int i = 0; i < XP; ++i)
#pragma unroll
        for (int c = 0; c < CO_T; ++c) {
          acc0[i][c] += s_red[((k - 1) * NV + lv) * 2 * XP * CO_T + (2 * i) * CO_T + c];
          acc1[i][c] += s_red[((k - 1) * NV + lv) * 2 * XP * CO_T + (2 * i + 1) * CO_T + c];
        }
  }
  if (!active) return;
  // residual: F.interpolate(in[:, :cout], scale_factor=2, trilinear, align_corners=False) on the RAW input
  int z0, z1, y0, y1;
  float lz, ly;
  {
    float s = fmaxf(0.5f * (zo + 0.5f) - 0.5f, 0.f);
    z0 = static_cast<int>(s); z1 = z0 + (z0 < p.Di - 1 ? 1 : 0); lz = s - z0;
    s = fmaxf(0.5f * (yo + 0.5f) - 0.5f, 0.f);
    y0 = static_cast<int>(s); y1 = y0 + (y0 < p.Hi - 1 ? 1 : 0); ly = s - y0;
  }
  float* out_n = p.out + n * p.out_nstride;
#pragma unroll
  for (int i = 0; i < XP; ++i) {
#pragma unroll
    for (int xx = 0; xx < 2; ++xx) {
      const int xo = 2 * (j0 + i) + xx;
      if (xo >= p.Wo) break;
      const float s = fmaxf(0.5f * (xo + 0.5f) - 0.5f, 0.f);
      const int x0 = static_cast<int>(s), x1 = x0 + (x0 < p.Wi - 1 ? 1 : 0);
      const float lx = s - x0;
      const long long ovox = (static_cast<long long>(zo) * p.Ho + yo) * p.Wo + xo;
#pragma unroll
      for (int c = 0; c < CO_T; ++c) {
        const int co = co0 + c;
        if (co >= p.cout) break;
        const float* pl = in_n + co * p.in_cstride;
        auto at = [&](int z, int y, int x) { return pl[(static_cast<size_t>(z) * p.Hi + y) * p.Wi + x]; };
        const float r = (1.f - lz) * ((1.f - ly) * ((1.f - lx) * at(z0, y0, x0) + lx * at(z0, y0, x1)) +
                                      ly * ((1.f - lx) * at(z0, y1, x0) + lx * at(z0, y1, x1))) +
                        lz * ((1.f - ly) * ((1.f - lx) * at(z1, y0, x0) + lx * at(z1, y0, x1)) +
                              ly * ((1.f - lx) * at(z1, y1, x0) + lx * at(z1, y1, x1)));
        const float a = (xx == 0 ? acc0[i][c] : acc1[i][c]) + p.bias[co] + r;
        out_n[co * p.out_cstride + ovox] = a * p.bn_scale[co] + p.bn_shift[co];
      }
    }
  }
}

// ---- shared-memory tiled variant for the large levels -----------------------------------------------------------
// Block = 128 threads = one output tile of 2 (z) x 8 (y) x 64 (x) voxels; per chunk of 8 input channels the
// 3 x 6 x 34 input neighbourhood and the [8][64][CO_T] weight slice are staged with cp.async (double buffered), so the
// FMA loop reads shared memory only and the next chunk's global loads are in flight while the current one computes.
constexpr int kTileCI = 8, kTileSX = 36, kTileIn = 3 * 6 * kTileSX;  // input tile floats per channel (x padded 34 -> 36)

template <int CO_T>
__global__ void __launch_bounds__(128) convt4_tile_kernel(const ConvT4Params p) {
  constexpr int XP = 4;
  extern __shared__ __align__(16) float s_tile[];
  float* s_in = s_tile;                                  // [2][kTileCI][3][6][kTileSX]
  float* s_w = s_tile + 2 * kTileCI * kTileIn;           // [2][kTileCI][64][CO_T]
  const int co0 = blockIdx.y * CO_T;
  const int n = blockIdx.z;
  const int ntx = ((p.Wo + 1) / 2 + 31) / 32, nty = ((p.Ho + 1) / 2 + 3) / 4;
  const int x0 = (blockIdx.x % ntx) * 32, y0 = ((blockIdx.x / ntx) % nty) * 4, z0 = blockIdx.x / (ntx * nty);
  const int tid = threadIdx.x;
  const int strip = tid & 7, yl = (tid >> 3) & 7, zl = tid >> 6;
  const int zo = 2 * z0 + zl, yo = 2 * y0 + yl, j0 = x0 + 4 * strip;
  const float* in_n = p.in + n * p.in_nstride;

  auto stage = [&](int chunk, int buf) {
    const int ci0 = chunk * kTileCI;
    float* din = s_in + buf * kTileCI * kTileIn;
    for (int i = tid; i < kTileCI * 3 * 6 * 34; i += 128) {
      const int sx = i % 34, sy = (i / 34) % 6, sz = (i / (34 * 6)) % 3, c = i / (34 * 6 * 3);
      const int x = x0 - 1 + sx, y = y0 - 1 + sy, z = z0 - 1 + sz, ci = ci0 + c;
      const bool ok = ci < p.cin && x >= 0 && x < p.Wi && y >= 0 && y < p.Hi && z >= 0 && z < p.Di;
      const float* src = ok ? in_n + ci * p.in_cstride + (static_cast<size_t>(z) * p.Hi + y) * p.Wi + x : in_n;
      cp_async_4(din + c * kTileIn + (sz * 6 + sy) * kTileSX + sx, src, ok);
    }
    float* dw = s_w + buf * kTileCI * 64 * CO_T;
    for (int i = tid; i < kTileCI * 64 * CO_T / 4; i += 128) {
      const int q4 = i % (CO_T / 4), k = (i / (CO_T / 4)) % 64, c = i / (64 * CO_T / 4);
      const int ci = min(ci0 + c, p.cin - 1);  // channels past cin read a valid row; their inputs are zero-filled
      cp_async_16(dw + (c * 64 + k) * CO_T + 4 * q4, p.w + (static_cast<size_t>(ci) * 64 + k) * p.cout + co0 + 4 * q4);
    }
    cp_async_commit();
  };

  int kz[2], sz[2], ky[2], sy[2];
#pragma unroll
  for (int t = 0; t < 2; ++t) {
    kz[t] = ((zo + 1) & 1) + 2 * t;
    sz[t] = (zo + 1 - kz[t]) / 2 - (z0 - 1);
    ky[t] = ((yo + 1) & 1) + 2 * t;
    sy[t] = (yo + 1 - ky[t]) / 2 - (y0 - 1);
  }
  float acc0[XP][CO_T], acc1[XP][CO_T];
#pragma unroll
  for (int i = 0; i < XP; ++i)
#pragma unroll
    for (int c = 0; c < CO_T; ++c) acc0[i][c] = acc1[i][c] = 0.f;

  const int nchunks = (p.cin + kTileCI - 1) / kTileCI;
  stage(0, 0);
  for (int ch = 0; ch < nchunks; ++ch) {
    const int buf = ch & 1;
    if (ch + 1 < nchunks) {
      stage(ch + 1, buf ^ 1);
      cp_async_wait<1>();
    } else {
      cp_async_wait<0>();
    }
    __syncthreads();
    const float* tin = s_in + buf * kTileCI * kTileIn;
    const float* tw = s_w + buf * kTileCI * 64 * CO_T;
#pragma unroll 2
    for (int c = 0; c < kTileCI; ++c) {
#pragma unroll
      for (int tz = 0; tz < 2; ++tz)
#pragma unroll
        for (int ty = 0; ty < 2; ++ty) {
          const float* row = tin + c * kTileIn + (sz[tz] * 6 + sy[ty]) * kTileSX + 4 * strip;
          const float4 m = *reinterpret_cast<const float4*>(row);
          const float2 e = *reinterpret_cast<const float2*>(row + 4);
          const float xr[XP + 2] = {leaky(m.x), leaky(m.y), leaky(m.z), leaky(m.w), leaky(e.x), leaky(e.y)};
          const float* wk = tw + (c * 64 + (kz[tz] * 4 + ky[ty]) * 4) * CO_T;
          float w0[CO_T], w1[CO_T], w2[CO_T], w3[CO_T];
#pragma unroll
          for (int k = 0; k < CO_T; ++k) {
            w0[k] = wk[k]; w1[k] = wk[CO_T + k]; w2[k] = wk[2 * CO_T + k]; w3[k] = wk[3 * CO_T + k];
          }
#pragma unroll
          for (int i = 0; i < XP; ++i)
#pragma unroll
            for (int k = 0; k < CO_T; ++k) {
              acc0[i][k] = fmaf(xr[i + 1], w1[k], acc0[i][k]);
              acc0[i][k] = fmaf(xr[i], w3[k], acc0[i][k]);
              acc1[i][k] = fmaf(xr[i + 2], w0[k], acc1[i][k]);
              acc1[i][k] = fmaf(xr[i + 1], w2[k], acc1[i][k]);
            }
        }
    }
    __syncthreads();
  }
  if (zo >= p.Do || yo >= p.Ho) return;
  // residual: F.interpolate(in[:, :cout], scale_factor=2, trilinear, align_corners=False) on the RAW input
  int zz0, zz1, yy0, yy1;
  float lz, ly;
  {
    float sc = fmaxf(0.5f * (zo + 0.5f) - 0.5f, 0.f);
    zz0 = static_cast<int>(sc); zz1 = zz0 + (zz0 < p.Di - 1 ? 1 : 0); lz = sc - zz0;
    sc = fmaxf(0.5f * (yo + 0.5f) - 0.5f, 0.f);
    yy0 = static_cast<int>(sc); yy1 = yy0 + (yy0 < p.Hi - 1 ? 1 : 0); ly = sc - yy0;
  }
  float* out_n = p.out + n * p.out_nstride;
#pragma unroll
  for (int i = 0; i < XP; ++i) {
#pragma unroll
    for (int xx = 0; xx < 2; ++xx) {
      const int xo = 2 * (j0 + i) + xx;
      if (xo >= p.Wo) break;
      const float sc = fmaxf(0.5f * (xo + 0.5f) - 0.5f, 0.f);
      const int xx0 = static_cast<int>(sc), xx1 = xx0 + (xx0 < p.Wi - 1 ? 1 : 0);
      const float lx = sc - xx0;
      const long long ovox = (static_cast<long long>(zo) * p.Ho + yo) * p.Wo + xo;
#pragma unroll
      for (int c = 0; c < CO_T; ++c) {
        const int co = co0 + c;
        if (co >= p.cout) break;
        const float* pl = in_n + co * p.in_cstride;
        auto at = [&](int z, int y, int x) { return __ldg(pl + (static_cast<size_t>(z) * p.Hi + y) * p.Wi + x); };
        const float r = (1.f - lz) * ((1.f - ly) * ((1.f - lx) * at(zz0, yy0, xx0) + lx * at(zz0, yy0, xx1)) +
                                      ly * ((1.f - lx) * at(zz0, yy1, xx0) + lx * at(zz0, yy1, xx1))) +
                        lz * ((1.f - ly) * ((1.f - lx) * at(zz1, yy0, xx0) + lx * at(zz1, yy0, xx1)) +
                              ly * ((1.f - lx) * at(zz1, yy1, xx0) + lx * at(zz1, yy1, xx1)));
        const float a = (xx == 0 ? acc0[i][c] : acc1[i][c]) + p.bias[co] + r;
        out_n[co * p.out_cstride + ovox] = a * p.bn_scale[co] + p.bn_shift[co];
      }
    }
  }
}

// Deep levels of the up path (few voxels, hundreds of channels): one block serves ONE output parity class
// (zo%2, yo%2, xo%2), which uses only 8 of the 64 taps, so the weight tile staged in shared memory is 8x smaller than
// in the strip kernel and is amortised over the whole block; the channel loop is split KS ways across thread groups.
template <int CO_T, int KS>
__global__ void __launch_bounds__(128) convt4_par_kernel(const ConvT4Params p) {
  constexpr int CI_CHUNK = 16;
  constexpr int NV = 128 / KS;
  __shared__ __align__(16) float s_w[CI_CHUNK * 8 * CO_T];
  __shared__ float s_red[KS > 1 ? (KS - 1) * NV * CO_T : 1];
  const int co0 = blockIdx.y * CO_T;
  const int cls = blockIdx.z & 7, n = blockIdx.z >> 3;
  const int pz = cls >> 2, py = (cls >> 1) & 1, px = cls & 1;
  const int Dq = (p.Do - pz + 1) / 2, Hq = (p.Ho - py + 1) / 2, Wq = (p.Wo - px + 1) / 2;
  const long long nthr = static_cast<long long>(Dq) * Hq * Wq;
  const int ks = threadIdx.x / NV, lv = threadIdx.x % NV;
  const long long v = blockIdx.x * static_cast<long long>(NV) + lv;
  const bool active = v < nthr;
  int zo = pz, yo = py, xo = px;
  if (active) {
    xo = 2 * static_cast<int>(v % Wq) + px;
    yo = 2 * static_cast<int>((v / Wq) % Hq) + py;
    zo = 2 * static_cast<int>(v / (static_cast<long long>(Wq) * Hq)) + pz;
  }
  // o = 2 i - 1 + k: taps k = (o+1)%2 + 2t, input i = (o + 1 - k)/2 (block-uniform k, per-thread i)
  const int kz0 = (pz + 1) & 1, ky0 = (py + 1) & 1, kx0 = (px + 1) & 1;
  int off[8];
  bool ok[8];
#pragma unroll
  for (int t = 0; t < 8; ++t) {
    const int tz = t >> 2, ty = (t >> 1) & 1, tx = t & 1;
    const int z = (zo + 1 - (kz0 + 2 * tz)) / 2, y = (yo + 1 - (ky0 + 2 * ty)) / 2, x = (xo + 1 - (kx0 + 2 * tx)) / 2;
    ok[t] = active && z >= 0 && z < p.Di && y >= 0 && y < p.Hi && x >= 0 && x < p.Wi;
    off[t] = ok[t] ? (z * p.Hi + y) * p.Wi + x : 0;
  }
  float acc[CO_T];
#pragma unroll
  for (int c = 0; c < CO_T; ++c) acc[c] = 0.f;
  const float* in_n = p.in + n * p.in_nstride;
  for (int ci0 = 0; ci0 < p.cin; ci0 += CI_CHUNK) {
    const int nci = min(CI_CHUNK, p.cin - ci0);
    __syncthreads();
    for (int i = threadIdx.x; i < nci * 8 * CO_T; i += blockDim.x) {
      const int c = i % CO_T, t = (i / CO_T) % 8, ci = i / (CO_T * 8);
      const int k = ((kz0 + 2 * (t >> 2)) * 4 + (ky0 + 2 * ((t >> 1) & 1))) * 4 + (kx0 + 2 * (t & 1));
      const int co = co0 + c;
      s_w[i] = co < p.cout ? p.w[(static_cast<size_t>(ci0 + ci) * 64 + k) * p.cout + co] : 0.f;
    }
    __syncthreads();
    for (int ci = ks; ci < nci; ci += KS) {
      const float* plane = in_n + (ci0 + ci) * p.in_cstride;
      const float* wc = s_w + ci * 8 * CO_T;
      float x[8];
#pragma unroll
      for (int t = 0; t < 8; ++t) x[t] = ok[t] ? leaky(__ldg(plane + off[t])) : 0.f;
#pragma unroll
      for (int t = 0; t < 8; ++t)
#pragma unroll
        for (int c = 0; c < CO_T; ++c) acc[c] = fmaf(x[t], wc[t * CO_T + c], acc[c]);
    }
  }
  if (KS > 1) {
    if (ks > 0) {
#pragma unroll
      for (int c = 0; c < CO_T; ++c) s_red[((ks - 1) * NV + lv) * CO_T + c] = acc[c];
    }
    __syncthreads();
    if (ks > 0) return;
#pragma unroll
    for (int k = 1; k < KS; ++k)
#pragma unroll
      for (int c = 0; c < CO_T; ++c) acc[c] += s_red[((k - 1) * NV + lv) * CO_T + c];
  }
  if (!active) return;
  // residual: F.interpolate(in[:, :cout], scale_factor=2, trilinear, align_corners=False) on the RAW input
  int i0[3], i1[3];
  float l[3];
  {
    const int o[3] = {zo, yo, xo}, nd[3] = {p.Di, p.Hi, p.Wi};
#pragma unroll
    for (int a = 0; a < 3; ++a) {
      const float s = fmaxf(0.5f * (o[a] + 0.5f) - 0.5f, 0.f);
      i0[a] = static_cast<int>(s);
      i1[a] = i0[a] + (i0[a] < nd[a] - 1 ? 1 : 0);
      l[a] = s - i0[a];
    }
  }
  float* out_n = p.out + n * p.out_nstride;
  const long long ovox = (static_cast<long long>(zo) * p.Ho + yo) * p.Wo + xo;
#pragma unroll
  for (int c = 0; c < CO_T; ++c) {
    const int co = co0 + c;
    if (co >= p.cout) break;
    const float* pl = in_n + co * p.in_cstride;
    auto at = [&](int z, int y, int x) { return pl[(static_cast<size_t>(z) * p.Hi + y) * p.Wi + x]; };
    const float lz = l[0], ly = l[1], lx = l[2];
    const float r = (1.f - lz) * ((1.f - ly) * ((1.f - lx) * at(i0[0], i0[1], i0[2]) + lx * at(i0[0], i0[1], i1[2])) +
                                  ly * ((1.f - lx) * at(i0[0], i1[1], i0[2]) + lx * at(i0[0], i1[1], i1[2]))) +
                    lz * ((1.f - ly) * ((1.f - lx) * at(i1[0], i0[1], i0[2]) + lx * at(i1[0], i0[1], i1[2])) +
                          ly * ((1.f - lx) * at(i1[0], i1[1], i0[2]) + lx * at(i1[0], i1[1], i1[2])));
    out_n[co * p.out_cstride + ovox] = (acc[c] + p.bias[co] + r) * p.bn_scale[co] + p.bn_shift[co];
  }
}

// ------------------------------------------------------------------------------------------------ convT k4 s2 p1, MMA
// The up path of tallUNet2 holds 79 % of the registration FLOPs with 48..512 input channels: it runs as an implicit
// GEMM on the warp-level tensor path (mma.sync m16n8k16, fp16 operands, fp32 accumulate) with fp32-level accuracy:
// every operand is split x = hi + lo into two fp16 values (22 mantissa bits) and hi*hi + lo*hi + hi*lo is accumulated
// (the dropped lo*lo term is ~2^-22 relative; products of two fp16 values are exact in fp32).  Weights are pre-split,
// pre-scaled by 2^wexp (so lo never falls into fp16 subnormals) and stored in B-fragment order by
// reg_pack_convt4_kernel.
//   GEMM view per output parity class (pz,py,px): M = input lattice points q, K = 8 taps x Cin, N = Cout.
//   o = 2 i - 1 + k: class p = 0 uses (k = 1, i = q), (k = 3, i = q - 1); p = 1 uses (k = 2, i = q), (k = 0, i = q + 1).
// reg_split_kernel first rewrites the layer input once as leaky-ReLU'd hi / lo fp16 channel pairs (one 32-bit word =
// one A-fragment register).  A block owns TX x TY x 1 lattice points (all 8 classes = 2TX x 2TY x 2 outputs) and 16
// output channels; per chunk of 16 input channels the 3 x (TY+2) x (TX+8) neighbourhood of both arrays arrives as two
// TMA boxes issued by one thread (zero fill outside the volume = the conv's padding; double buffered: chunk c+1 flies
// while chunk c computes), so the kernel spends no instructions on staging.  Each of the 27 neighbour shifts loads its A fragments once and feeds
// every (class, tap) pair that maps to it: 64 weight taps x 2 m-tiles x 2 n-tiles x 3 split terms = 768 MMAs per warp
// per chunk against 432 shared-memory loads.  The residual (2x trilinear upsample of the raw input channels, fixed
// 0.25 / 0.75 weights), bias and BatchNorm are applied in the epilogue from the 16 raw residual channels, which one
// more TMA box brings into the free buffer during the last chunk's MMAs (the epilogue clamps its neighbour indices =
// the interpolation's replicate border).
__device__ __forceinline__ void mma16816(float (&c)[4], const uint32_t (&a)[4], uint32_t b0, uint32_t b1) {
  asm volatile(
      "mma.sync.aligned.m16n8k16.row.col.f32.f16.f16.f32 {%0,%1,%2,%3}, {%4,%5,%6,%7}, {%8,%9}, {%0,%1,%2,%3};"
      : "+f"(c[0]), "+f"(c[1]), "+f"(c[2]), "+f"(c[3])
      : "r"(a[0]), "r"(a[1]), "r"(a[2]), "r"(a[3]), "r"(b0), "r"(b1));
}
__device__ __forceinline__ void split_pack(float x0, float x1, uint32_t& hi, uint32_t& lo) {
  const __half2 h = __floats2half2_rn(x0, x1);
  const float2 hf = __half22float2(h);
  const __half2 l = __floats2half2_rn(x0 - hf.x, x1 - hf.y);
  hi = *reinterpret_cast<const uint32_t*>(&h);
  lo = *reinterpret_cast<const uint32_t*>(&l);
}
// (class parity, tap) pairs served by neighbour shift s in {0,1,2} (input i = q + s - 1) along one axis
__host__ __device__ constexpr int sh_ncomb(int s) { return s == 1 ? 2 : 1; }
__host__ __device__ constexpr int sh_par(int s, int i) { return s == 0 ? 0 : (s == 2 ? 1 : i); }
__host__ __device__ constexpr int sh_tap(int s, int i) { return s == 0 ? 3 : (s == 2 ? 0 : (i == 0 ? 1 : 2)); }

// The kernel visits the 64 weight taps in the order of its shift loops; the packed weights are stored in that order so
// the B-fragment stream of a chunk is read front to back (register double buffering + L1 prefetch a few visits ahead).
__host__ __device__ constexpr int visit_tap(int v) {
  int c = 0;
  for (int sz = 0; sz < 3; ++sz)
    for (int sy = 0; sy < 3; ++sy)
      for (int sx = 0; sx < 3; ++sx)
        for (int iz = 0; iz < sh_ncomb(sz); ++iz)
          for (int iy = 0; iy < sh_ncomb(sy); ++iy)
            for (int ix = 0; ix < sh_ncomb(sx); ++ix) {
              if (c == v) return (sh_tap(sz, iz) * 4 + sh_tap(sy, iy)) * 4 + sh_tap(sx, ix);
              ++c;
            }
  return -1;
}
__device__ __forceinline__ void prefetch_l1(const void* ptr) { asm volatile("prefetch.global.L1 [%0];" ::"l"(ptr)); }
__device__ __forceinline__ void prefetch_l2(const void* ptr) { asm volatile("prefetch.global.L2 [%0];" ::"l"(ptr)); }

template <int TX>
struct ConvT4MmaCfg {
  static constexpr int TY = 128 / TX;             // 4 / 8 lattice rows per block for TX = 32 / 16
  // shared-memory row = one TMA box row.  The innermost start coordinate of a TMA box must be 16-byte aligned
  // (measured: scripts/micro/tma_probe.cu -- x = qx0 - 1 raises "illegal instruction", qx0 - 4 works), so the box
  // starts 4 words left of the tile: col 3 = left halo, cols 4 .. TX+3 = the tile, col TX+4 = right halo
  static constexpr int SX = TX + 8, SY = TY + 2;
  static constexpr int PS = 3 * SY * SX;          // words per channel pair (720: pairs t and t+2 share banks, 2-way)
  static constexpr int BUF = 16 * PS;             // words per buffer: (hi, lo) x 8 pairs = two TMA boxes
  static constexpr size_t smem_bytes = 2 * BUF * 4 + 128;       // + alignment slack
};

template <int TX>
__global__ void __launch_bounds__(128, 2) convt4_mma_kernel(const __grid_constant__ CUtensorMap tm_x,
                                                            const __grid_constant__ CUtensorMap tm_res,
                                                            const ConvT4Params p) {
  using Cfg = ConvT4MmaCfg<TX>;
  constexpr int TY = Cfg::TY, SX = Cfg::SX, SY = Cfg::SY, PS = Cfg::PS, BUF = Cfg::BUF;
  extern __shared__ uint8_t s_mma_raw[];
  uint32_t* s_mma = reinterpret_cast<uint32_t*>((reinterpret_cast<uintptr_t>(s_mma_raw) + 127) & ~uintptr_t(127));
  __shared__ uint64_t full_bar[2];                   // TMA completion of buffer 0 / 1
  const int tid = threadIdx.x, lane = tid & 31, wrp = tid >> 5, g = lane >> 2, t = lane & 3;
  const int ntx = (p.Wi + TX - 1) / TX, nty = (p.Hi + TY - 1) / TY;
  const int qx0 = static_cast<int>(blockIdx.x % ntx) * TX, qy0 = static_cast<int>((blockIdx.x / ntx) % nty) * TY;
  const int qz = static_cast<int>(blockIdx.x / (ntx * nty));
  const int coblk = blockIdx.y, co0 = coblk * 16, n = blockIdx.z;
  const float* in_n = p.in + n * p.in_nstride;
  const int nchunks = p.cin / 16;
  const long long vol = static_cast<long long>(p.Di) * p.Hi * p.Wi;
  // rows g and g + 8 (h = 0, 1) of m-tile j of this warp <-> lattice point (ty[j][h], tx[j][h]) of the block tile
  // (an m-tile is 16 x-adjacent points)
  int ty[2][2], tx[2][2];
#pragma unroll
  for (int j = 0; j < 2; ++j)
#pragma unroll
    for (int h = 0; h < 2; ++h) {
      ty[j][h] = TX == 32 ? wrp : 2 * wrp + j;
      tx[j][h] = TX == 32 ? 16 * j + g + 8 * h : g + 8 * h;
    }
  float acc[8][2][2][4];
#pragma unroll
  for (int c = 0; c < 8; ++c)
#pragma unroll
    for (int j = 0; j < 2; ++j)
#pragma unroll
      for (int nt = 0; nt < 2; ++nt) acc[c][j][nt][0] = acc[c][j][nt][1] = acc[c][j][nt][2] = acc[c][j][nt][3] = 0.f;

  // ---- one chunk = two TMA boxes (hi, lo) of 8 channel pairs x 3 x SY x (TX + 4) words of the pre-split input
  // (reg_split_kernel); coordinates outside the volume are zero-filled by TMA = the transposed conv's implicit padding
  const int planes_n = p.cin / 2;                    // channel pairs per sample
  // the descriptors must be addressed in parameter space: take the addresses here, not inside a capturing lambda
  const CUtensorMap* const ptm_x = &tm_x;
  const CUtensorMap* const ptm_res = &tm_res;
  auto fetch_chunk = [&](int ch, int b) {            // one elected thread
    uint32_t* dbuf = s_mma + b * BUF;
    mbar_arrive_expect_tx(&full_bar[b], BUF * 4);
    tma_load_5d(dbuf, ptm_x, &full_bar[b], qx0 - 4, qy0 - 1, qz - 1, n * planes_n + ch * 8, 0);
    tma_load_5d(dbuf + 8 * PS, ptm_x, &full_bar[b], qx0 - 4, qy0 - 1, qz - 1, (p.N + n) * planes_n + ch * 8, 0);
  };
  // ---- the 16 raw fp32 residual channels co0 .. co0+15: one TMA box into the buffer the last chunk does not use
  // (zero-filled outside the volume; the epilogue clamps its neighbour indices = the upsample's replicate border)
  auto fetch_res = [&](int b) {                      // one elected thread
    mbar_arrive_expect_tx(&full_bar[b], BUF * 4);
    tma_load_5d(s_mma + b * BUF, ptm_res, &full_bar[b], qx0 - 4, qy0 - 1, qz - 1, n * p.res_planes_per_n + co0, 0);
  };
  const int rb = nchunks & 1;  // buffer the last chunk does not use: the residual channels land there
  if (tid == 0) {
    mbar_init(&full_bar[0], 1);
    mbar_init(&full_bar[1], 1);
    fence_mbar_init();
  }
  __syncthreads();
  if (tid == 0 && !(p.debug & 4)) fetch_chunk(0, 0);
  uint32_t phase[2] = {0u, 0u};
  for (int ch = 0; ch < nchunks; ++ch) {
    fence_proxy_async_smem();   // this thread's reads of the buffer refilled below are ordered before the TMA writes
    __syncthreads();            // every warp is done with chunk ch - 1
    if (!(p.debug & 4)) {
      if (tid == 0) {
        if (ch + 1 < nchunks) fetch_chunk(ch + 1, (ch + 1) & 1);
        else fetch_res(rb);
      }
      mbar_wait(&full_bar[ch & 1], phase[ch & 1], 40 + ch);
      phase[ch & 1] ^= 1u;
    }
    const uint32_t* sHi = s_mma + (ch & 1) * BUF;
    const uint32_t* sLo = sHi + 8 * PS;
    // ---- MMAs: 27 neighbour shifts, A fragments loaded once per shift
    const uint4* wq = p.wpk + (static_cast<size_t>(coblk) * nchunks + ch) * (64 * 2 * 32) + lane;
    if (ch + 1 < nchunks) {
      // next chunk's weights (64 KB) towards L2 while this chunk computes
      const char* wn = reinterpret_cast<const char*>(wq - lane + 64 * 2 * 32);
#pragma unroll
      for (int i = 0; i < 4; ++i) prefetch_l2(wn + (tid + 128 * i) * 128);
    }
    constexpr int kAhead = 8;  // L1 prefetch distance in B-fragment visits (one visit = 512 B = 6 MMAs)
#pragma unroll
    for (int i = 0; i < kAhead; ++i) prefetch_l1(wq + i * 32);
    if (p.debug & 2) continue;
    uint4 bnext[2] = {__ldg(wq), __ldg(wq + 32)};
    int v = 0;  // visit counter (tap): compile-time after unrolling
#pragma unroll
    for (int sz = 0; sz < 3; ++sz)
#pragma unroll
      for (int sy = 0; sy < 3; ++sy)
#pragma unroll
        for (int sx = 0; sx < 3; ++sx) {
          uint32_t ah[2][4], al[2][4];
#pragma unroll
          for (int j = 0; j < 2; ++j) {
            const int b0 = (sz * SY + ty[j][0] + sy) * SX + tx[j][0] + sx + 3;
            const int b1 = (sz * SY + ty[j][1] + sy) * SX + tx[j][1] + sx + 3;
            ah[j][0] = sHi[t * PS + b0];       ah[j][1] = sHi[t * PS + b1];
            ah[j][2] = sHi[(t + 4) * PS + b0]; ah[j][3] = sHi[(t + 4) * PS + b1];
            al[j][0] = sLo[t * PS + b0];       al[j][1] = sLo[t * PS + b1];
            al[j][2] = sLo[(t + 4) * PS + b0]; al[j][3] = sLo[(t + 4) * PS + b1];
          }
#pragma unroll
          for (int iz = 0; iz < sh_ncomb(sz); ++iz)
#pragma unroll
            for (int iy = 0; iy < sh_ncomb(sy); ++iy)
#pragma unroll
              for (int ix = 0; ix < sh_ncomb(sx); ++ix) {
                const int cls = sh_par(sz, iz) * 4 + sh_par(sy, iy) * 2 + sh_par(sx, ix);
                const uint4 b[2] = {bnext[0], bnext[1]};
                if (v + 1 < 64) {
                  bnext[0] = __ldg(wq + (2 * v + 2) * 32);
                  bnext[1] = __ldg(wq + (2 * v + 3) * 32);
                }
                if (2 * v + kAhead < 128) {
                  prefetch_l1(wq + (2 * v + kAhead) * 32);
                  prefetch_l1(wq + (2 * v + kAhead + 1) * 32);
                }
                ++v;
                // term-major order: the three split terms of one accumulator are 4 MMAs apart (mma.sync on the same
                // accumulator serialises on the previous result)
#pragma unroll
                for (int term = 0; term < 3; ++term)
#pragma unroll
                  for (int nt = 0; nt < 2; ++nt)
#pragma unroll
                    for (int j = 0; j < 2; ++j)
                      mma16816(acc[cls][j][nt], term == 1 ? al[j] : ah[j], term == 2 ? b[nt].z : b[nt].x,
                               term == 2 ? b[nt].w : b[nt].y);
              }
        }
  }
  if (!(p.debug & 4)) mbar_wait(&full_bar[rb], phase[rb], 39);   // raw residual channels have landed in buffer rb
  const float* sRaw = reinterpret_cast<const float*>(s_mma + rb * BUF);
  const int rz[3] = {max(qz - 1, 0) - (qz - 1), 1, min(qz + 1, p.Di - 1) - (qz - 1)};  // replicate-clamped planes

  // ---- epilogue: out = BN( acc * 2^-wexp + bias + upsample2x(raw in[co]) ), cropped to (Do, Ho, Wo)
  const float inv = exp2f(static_cast<float>(-p.wexp));
  float* out_n = p.out + n * p.out_nstride;
#pragma unroll
  for (int nt = 0; nt < 2; ++nt)
#pragma unroll
    for (int cb = 0; cb < 2; ++cb) {
      const int cl = 8 * nt + 2 * t + cb, co = co0 + cl;
      const float bias = __ldg(p.bias + co), bs = __ldg(p.bn_scale + co), bt = __ldg(p.bn_shift + co);
      float* out_c = out_n + co * p.out_cstride;
#pragma unroll
      for (int j = 0; j < 2; ++j)
#pragma unroll
        for (int h = 0; h < 2; ++h) {
          const int xl = tx[j][h], yl = ty[j][h];
          const int qx = qx0 + xl, qy = qy0 + yl;
          if (qx >= p.Wi || qy >= p.Hi || (p.debug & 8)) continue;
          // separable 0.25 / 0.75 interpolation of the 3x3x3 raw neighbourhood (replicate-clamped) -> 8 class values
          const int ry[3] = {max(qy - 1, 0) - (qy0 - 1), yl + 1, min(qy + 1, p.Hi - 1) - (qy0 - 1)};
          const int rx[3] = {max(qx - 1, 0) - (qx0 - 4), xl + 4, min(qx + 1, p.Wi - 1) - (qx0 - 4)};
          float ax[3][3][2];
#pragma unroll
          for (int dz = 0; dz < 3; ++dz)
#pragma unroll
            for (int dy = 0; dy < 3; ++dy) {
              const float* row = sRaw + cl * PS + (rz[dz] * SY + ry[dy]) * SX;
              const float v0 = row[rx[0]], v1 = row[rx[1]], v2 = row[rx[2]];
              ax[dz][dy][0] = 0.25f * v0 + 0.75f * v1;
              ax[dz][dy][1] = 0.75f * v1 + 0.25f * v2;
            }
          float ay[3][2][2];
#pragma unroll
          for (int dz = 0; dz < 3; ++dz)
#pragma unroll
            for (int px = 0; px < 2; ++px) {
              ay[dz][0][px] = 0.25f * ax[dz][0][px] + 0.75f * ax[dz][1][px];
              ay[dz][1][px] = 0.75f * ax[dz][1][px] + 0.25f * ax[dz][2][px];
            }
#pragma unroll
          for (int pz = 0; pz < 2; ++pz)
#pragma unroll
            for (int py = 0; py < 2; ++py) {
              const int zo = 2 * qz + pz, yo = 2 * qy + py, xo = 2 * qx;
              if (zo >= p.Do || yo >= p.Ho || xo >= p.Wo) continue;
              float v[2];
#pragma unroll
              for (int px = 0; px < 2; ++px) {
                const float r = pz == 0 ? 0.25f * ay[0][py][px] + 0.75f * ay[1][py][px]
                                        : 0.75f * ay[1][py][px] + 0.25f * ay[2][py][px];
                v[px] = (acc[pz * 4 + py * 2 + px][j][nt][2 * h + cb] * inv + bias + r) * bs + bt;
              }
              float* dst = out_c + (static_cast<long long>(zo) * p.Ho + yo) * p.Wo + xo;
              if (xo + 1 < p.Wo && (reinterpret_cast<uintptr_t>(dst) & 7) == 0) {
                *reinterpret_cast<float2*>(dst) = make_float2(v[0], v[1]);
              } else {
                dst[0] = v[0];
                if (xo + 1 < p.Wo) dst[1] = v[1];
              }
            }
        }
    }
}

// Layer input [N][cin] planes (explicit strides) -> xsplit [2 (hi, lo)][N][cin/2][vol] words: leaky_relu, then the
// hi / lo fp16 split of channels (2c, 2c+1) packed into one word each.
__global__ void __launch_bounds__(256) reg_split_kernel(const float* __restrict__ in, long long in_nstride,
                                                        long long in_cstride, int N, int cin, long long vol,
                                                        uint32_t* __restrict__ xs) {
  const long long per_n = static_cast<long long>(cin / 2) * vol, total = N * per_n;
  for (long long i = blockIdx.x * static_cast<long long>(blockDim.x) + threadIdx.x; i < total;
       i += static_cast<long long>(gridDim.x) * blockDim.x) {
    const long long n = i / per_n, r = i - n * per_n;
    const long long c = r / vol, v = r - c * vol;
    const float* src = in + n * in_nstride + 2 * c * in_cstride + v;
    uint32_t hi, lo;
    split_pack(leaky(__ldg(src)), leaky(__ldg(src + in_cstride)), hi, lo);
    xs[i] = hi;
    xs[total + i] = lo;
  }
}

// w [cin][64][cout] fp32 -> B fragments of mma.sync.m16n8k16 (col-major B: k = input channel within the chunk,
// n = output channel within the 8-wide n-tile), split into hi / lo fp16 after scaling by 2^wexp; taps in the
// kernel's visit order (visit_tap).
__global__ void reg_pack_convt4_kernel(const float* __restrict__ w, int cin, int cout, int wexp, uint4* __restrict__ wpk) {
  const long long total = static_cast<long long>(cout / 16) * (cin / 16) * 64 * 2 * 32;
  const float sc = exp2f(static_cast<float>(wexp));
  for (long long i = blockIdx.x * static_cast<long long>(blockDim.x) + threadIdx.x; i < total;
       i += static_cast<long long>(gridDim.x) * blockDim.x) {
    long long r = i;
    const int lane = r % 32; r /= 32;
    const int nt = r % 2; r /= 2;
    const int k = visit_tap(static_cast<int>(r % 64)); r /= 64;
    const int ch = r % (cin / 16);
    const int coblk = static_cast<int>(r / (cin / 16));
    const int g = lane >> 2, t = lane & 3;
    const int co = coblk * 16 + nt * 8 + g;
    auto at = [&](int ci) { return w[(static_cast<size_t>(ch * 16 + ci) * 64 + k) * cout + co] * sc; };
    uint4 o;
    split_pack(at(2 * t), at(2 * t + 1), o.x, o.z);
    split_pack(at(2 * t + 8), at(2 * t + 9), o.y, o.w);
    wpk[i] = o;
  }
}

// ------------------------------------------------------------------------------------------------ deep levels, split-K
// The deepest levels of tallUNet2 have a few hundred output voxels and up to 512 channels: they are weight-streaming
// GEMMs (M = N x voxels <= a few thousand, K = taps x Cin up to 13 824, 14 - 34 MB of weights) that the direct kernels
// above run at ~0.1 TB/s because one block walks the whole K range.  Here K is split over blocks: block
// (m-tile, co-tile, ks) computes a 64 x 64 partial over one tap and one range of input channels with a register-tiled
// fp32 SGEMM whose A operand is gathered on the fly (leaky-ReLU applied), and writes it to a caller-owned workspace
// [ks][class][M][cout]; a second kernel adds the partials IN FIXED ORDER (deterministic, unlike atomics) and applies
// the layer's epilogue (bias + residual [+ BatchNorm]).
//   MODE 0: Conv3d k3 s2 p1: m = (n, zo, yo, xo), tap (kd, kh, kw), input (2 zo - 1 + kd, ...)
//   MODE 1: ConvTranspose3d k4 s2 p1, one output parity class per grid.y slice: m = (n, q), tap t in {0,1}^3,
//           k = k0 + 2 t, input q + (p + 1 - k0) / 2 - t per axis (k0 = (p + 1) & 1)
struct DeepGemmParams {
  const float* in;
  long long in_nstride, in_cstride;
  int cin, Di, Hi, Wi;
  const float* w;      // [cin][taps_total][wld]
  int taps_total, wld; // 27 / 64; leading dimension of the co axis
  int cout;
  int N, Mo_d, Mo_h, Mo_w;  // m-space: (n, d, h, w) with these extents
  int ntaps;           // taps per block-group: 27 (conv) or 8 (one parity class)
  int ci_per_split, nsplit;
  float* ws;           // [ntaps * nsplit][ncls][M][cout]
  int ncls;
};

template <int MODE>
__global__ void __launch_bounds__(256) deep_gemm_kernel(const DeepGemmParams p) {
  constexpr int BM = 64, BN = 64, BK = 16;
  __shared__ __align__(16) float sA[2][BK][BM];
  __shared__ __align__(16) float sW[2][BK][BN];
  const int tid = threadIdx.x;
  const long long M = static_cast<long long>(p.N) * p.Mo_d * p.Mo_h * p.Mo_w;
  const int mtiles = static_cast<int>((M + BM - 1) / BM);
  const int m0 = (blockIdx.x % mtiles) * BM, co0 = (blockIdx.x / mtiles) * BN;
  const int cls = blockIdx.y;
  const int ks = blockIdx.z, tap = ks / p.nsplit, split = ks % p.nsplit;
  const int ci_begin = split * p.ci_per_split, ci_end = min(p.cin, ci_begin + p.ci_per_split);
  // ---- A gather set-up: this thread always loads row m = m0 + tid % 64 (4 channels per chunk)
  const int am = tid & 63, ac = tid >> 6;
  long long a_off = -1;
  {
    const long long m = m0 + am;
    if (m < M) {
      long long r = m;
      const int x = r % p.Mo_w; r /= p.Mo_w;
      const int y = r % p.Mo_h; r /= p.Mo_h;
      const int z = r % p.Mo_d; r /= p.Mo_d;
      const int n = static_cast<int>(r);
      int iz, iy, ix;
      if (MODE == 0) {
        iz = 2 * z - 1 + tap / 9; iy = 2 * y - 1 + (tap / 3) % 3; ix = 2 * x - 1 + tap % 3;
      } else {
        const int pz = cls >> 2, py = (cls >> 1) & 1, px = cls & 1;
        const int tz = tap >> 2, ty = (tap >> 1) & 1, tx = tap & 1;
        iz = z + (pz ? 1 : 0) - tz; iy = y + (py ? 1 : 0) - ty; ix = x + (px ? 1 : 0) - tx;
      }
      if (iz >= 0 && iz < p.Di && iy >= 0 && iy < p.Hi && ix >= 0 && ix < p.Wi)
        a_off = n * p.in_nstride + (static_cast<long long>(iz) * p.Hi + iy) * p.Wi + ix;
    }
  }
  // ---- W set-up: tap index into the [taps_total] axis
  int wtap = tap;
  if (MODE == 1) {
    const int pz = cls >> 2, py = (cls >> 1) & 1, px = cls & 1;
    const int kz = ((pz + 1) & 1) + 2 * (tap >> 2), ky = ((py + 1) & 1) + 2 * ((tap >> 1) & 1),
              kx = ((px + 1) & 1) + 2 * (tap & 1);
    wtap = (kz * 4 + ky) * 4 + kx;
  }
  const int wc = tid >> 4, wn = (tid & 15) * 4;   // this thread loads W[ci = wc][co0 + wn .. +3]
  const bool wvec = (p.wld & 3) == 0 && co0 + wn + 3 < p.wld;
  float ra[4];
  float4 rw;
  auto gload = [&](int ci0) {
#pragma unroll
    for (int j = 0; j < 4; ++j) {
      const int ci = ci0 + ac + 4 * j;
      ra[j] = (a_off >= 0 && ci < ci_end) ? leaky(__ldg(p.in + a_off + ci * p.in_cstride)) : 0.f;
    }
    const int ci = ci0 + wc;
    rw = make_float4(0.f, 0.f, 0.f, 0.f);
    if (ci < ci_end) {
      const float* wp = p.w + (static_cast<size_t>(ci) * p.taps_total + wtap) * p.wld + co0 + wn;
      if (wvec) {
        rw = __ldg(reinterpret_cast<const float4*>(wp));
      } else {
        rw.x = co0 + wn < p.wld ? __ldg(wp) : 0.f;
        rw.y = co0 + wn + 1 < p.wld ? __ldg(wp + 1) : 0.f;
        rw.z = co0 + wn + 2 < p.wld ? __ldg(wp + 2) : 0.f;
        rw.w = co0 + wn + 3 < p.wld ? __ldg(wp + 3) : 0.f;
      }
    }
  };
  auto sstore = [&](int b) {
#pragma unroll
    for (int j = 0; j < 4; ++j) sA[b][ac + 4 * j][am] = ra[j];
    *reinterpret_cast<float4*>(&sW[b][wc][wn]) = rw;
  };
  const int tm = (tid & 15) * 4, tn = (tid >> 4) * 4;
  float acc[4][4];
#pragma unroll
  for (int i = 0; i < 4; ++i)
#pragma unroll
    for (int j = 0; j < 4; ++j) acc[i][j] = 0.f;
  gload(ci_begin);
  sstore(0);
  __syncthreads();
  int b = 0;
  for (int ci0 = ci_begin; ci0 < ci_end; ci0 += BK) {
    const bool more = ci0 + BK < ci_end;
    if (more) gload(ci0 + BK);
#pragma unroll
    for (int kk = 0; kk < BK; ++kk) {
      const float4 a = *reinterpret_cast<const float4*>(&sA[b][kk][tm]);
      const float4 w = *reinterpret_cast<const float4*>(&sW[b][kk][tn]);
      const float av[4] = {a.x, a.y, a.z, a.w}, wv[4] = {w.x, w.y, w.z, w.w};
#pragma unroll
      for (int i = 0; i < 4; ++i)
#pragma unroll
        for (int j = 0; j < 4; ++j) acc[i][j] = fmaf(av[i], wv[j], acc[i][j]);
    }
    if (more) sstore(b ^ 1);
    __syncthreads();
    b ^= 1;
  }
  float* dst = p.ws + (static_cast<size_t>(ks) * p.ncls + cls) * M * p.cout;
#pragma unroll
  for (int i = 0; i < 4; ++i) {
    const long long m = m0 + tm + i;
    if (m >= M) break;
#pragma unroll
    for (int j = 0; j < 4; ++j)
      if (co0 + tn + j < p.cout) dst[m * p.cout + co0 + tn + j] = acc[i][j];
  }
}

// out = (sum_ks partial + bias [+ pad_or_crop(avg_pool3d(in, 2, ceil_mode=True))]) * out_scale   (conv3 epilogue)
__global__ void __launch_bounds__(256) deep_reduce_conv3_kernel(const Conv3Params p, const float* __restrict__ ws,
                                                                int nks) {
  const long long vol = static_cast<long long>(p.Do) * p.Ho * p.Wo, M = p.N * vol, total = M * p.cout;
  for (long long i = blockIdx.x * static_cast<long long>(blockDim.x) + threadIdx.x; i < total;
       i += static_cast<long long>(gridDim.x) * blockDim.x) {
    const int co = static_cast<int>(i % p.cout);
    const long long m = i / p.cout;
    float r = 0.f;
    for (int k = 0; k < nks; ++k) r += ws[(static_cast<size_t>(k) * M + m) * p.cout + co];
    r += p.bias[co];
    const long long v = m % vol;
    const int n = static_cast<int>(m / vol);
    const int xo = static_cast<int>(v % p.Wo), yo = static_cast<int>((v / p.Wo) % p.Ho),
              zo = static_cast<int>(v / (static_cast<long long>(p.Wo) * p.Ho));
    if (p.residual) {
      const int cs = co - (p.cout - p.cin);
      if (cs >= 0) {
        const float* plane = p.in + n * p.in_nstride + cs * p.in_cstride;
        float sum = 0.f;
        int cnt = 0;
        for (int dz = 0; dz < 2; ++dz)
          for (int dy = 0; dy < 2; ++dy)
            for (int dx = 0; dx < 2; ++dx) {
              const int z = 2 * zo + dz, y = 2 * yo + dy, x = 2 * xo + dx;
              if (z < p.Di && y < p.Hi && x < p.Wi) {
                sum += plane[(static_cast<size_t>(z) * p.Hi + y) * p.Wi + x];
                ++cnt;
              }
            }
        r += sum / static_cast<float>(cnt);
      }
    }
    p.out[n * p.out_nstride + co * p.out_cstride + v] = r * p.out_scale;
  }
}

// out = BN( sum_ks partial[class of o][q = o / 2] + bias + upsample2x_trilinear(in[:, :cout]) )   (convT4 epilogue)
__global__ void __launch_bounds__(256) deep_reduce_convt4_kernel(const ConvT4Params p, const float* __restrict__ ws,
                                                                 int nks) {
  const long long ovol = static_cast<long long>(p.Do) * p.Ho * p.Wo, total = p.N * ovol * p.cout;
  const long long qvol = static_cast<long long>(p.Di) * p.Hi * p.Wi, M = p.N * qvol;
  for (long long i = blockIdx.x * static_cast<long long>(blockDim.x) + threadIdx.x; i < total;
       i += static_cast<long long>(gridDim.x) * blockDim.x) {
    const int co = static_cast<int>(i % p.cout);
    long long r0 = i / p.cout;
    const int xo = static_cast<int>(r0 % p.Wo); r0 /= p.Wo;
    const int yo = static_cast<int>(r0 % p.Ho); r0 /= p.Ho;
    const int zo = static_cast<int>(r0 % p.Do);
    const int n = static_cast<int>(r0 / p.Do);
    const int cls = ((zo & 1) << 2) | ((yo & 1) << 1) | (xo & 1);
    const long long m = n * qvol + (static_cast<long long>(zo >> 1) * p.Hi + (yo >> 1)) * p.Wi + (xo >> 1);
    float acc = 0.f;
    for (int k = 0; k < nks; ++k) acc += ws[((static_cast<size_t>(k) * 8 + cls) * M + m) * p.cout + co];
    int i0[3], i1[3];
    float l[3];
    const int o[3] = {zo, yo, xo}, nd[3] = {p.Di, p.Hi, p.Wi};
#pragma unroll
    for (int a = 0; a < 3; ++a) {
      const float sc = fmaxf(0.5f * (o[a] + 0.5f) - 0.5f, 0.f);
      i0[a] = static_cast<int>(sc);
      i1[a] = i0[a] + (i0[a] < nd[a] - 1 ? 1 : 0);
      l[a] = sc - i0[a];
    }
    const float* pl = p.in + n * p.in_nstride + co * p.in_cstride;
    auto at = [&](int z, int y, int x) { return pl[(static_cast<size_t>(z) * p.Hi + y) * p.Wi + x]; };
    const float lz = l[0], ly = l[1], lx = l[2];
    const float res = (1.f - lz) * ((1.f - ly) * ((1.f - lx) * at(i0[0], i0[1], i0[2]) + lx * at(i0[0], i0[1], i1[2])) +
                                    ly * ((1.f - lx) * at(i0[0], i1[1], i0[2]) + lx * at(i0[0], i1[1], i1[2]))) +
                      lz * ((1.f - ly) * ((1.f - lx) * at(i1[0], i0[1], i0[2]) + lx * at(i1[0], i0[1], i1[2])) +
                            ly * ((1.f - lx) * at(i1[0], i1[1], i0[2]) + lx * at(i1[0], i1[1], i1[2])));
    const long long ovox = (static_cast<long long>(zo) * p.Ho + yo) * p.Wo + xo;
    p.out[n * p.out_nstride + co * p.out_cstride + ovox] = (acc + p.bias[co] + res) * p.bn_scale[co] + p.bn_shift[co];
  }
}

// Thread mapping: a warp owns 32 x-adjacent grid points of one row, so every gather and every store of the warp
// touches a few 128-byte lines; a block owns 8 consecutive rows; a thread carries kChainVZ z-adjacent points through
// the whole chain (independent gather sequences in flight; the z+1 plane of point i is the z plane of point i+1).
template <int kChainVZ, int kMinBlocks>
__global__ void __launch_bounds__(256, kMinBlocks) chain_kernel(const ChainParams p) {
  const long long nvox = static_cast<long long>(p.D) * p.H * p.W;
  const double sz = 1.0 / (p.D - 1), sy = 1.0 / (p.H - 1), sx = 1.0 / (p.W - 1);
  const int nbx = (p.W + 31) / 32, nby = (p.H + 7) / 8, nbz = (p.D + kChainVZ - 1) / kChainVZ;
  const long long ntiles = static_cast<long long>(nbx) * nby * nbz;
  const int lane = threadIdx.x & 31, wrp = threadIdx.x >> 5;
  for (long long tile = blockIdx.x; tile < ntiles; tile += gridDim.x) {
    const int x = static_cast<int>(tile % nbx) * 32 + lane;
    const int y = static_cast<int>((tile / nbx) % nby) * 8 + wrp;
    const int z0 = static_cast<int>(tile / (static_cast<long long>(nbx) * nby)) * kChainVZ;
    if (x >= p.W || y >= p.H) continue;
    float cz[kChainVZ], cy[kChainVZ], cx[kChainVZ];
    const long long v0 = (static_cast<long long>(z0) * p.H + y) * p.W + x, zs = static_cast<long long>(p.H) * p.W;
    auto vof = [&](int i) { return v0 + min(i, p.D - 1 - z0) * zs; };
#pragma unroll
    for (int i = 0; i < kChainVZ; ++i) {
      const int z = min(z0 + i, p.D - 1);
      cz[i] = static_cast<float>(z * sz);
      cy[i] = static_cast<float>(y * sy);
      cx[i] = static_cast<float>(x * sx);
    }
    for (int f = 0; f < p.nfields; ++f) {
      const float* u = p.u[f];
      const size_t plane = static_cast<size_t>(p.ud[f]) * p.uh[f] * p.uw[f];
      if (f == 0 && p.shortcut_first) {
#pragma unroll
        for (int i = 0; i < kChainVZ; ++i) {
          const long long v = vof(i);
          cz[i] += __ldg(u + v); cy[i] += __ldg(u + plane + v); cx[i] += __ldg(u + 2 * plane + v);
        }
      } else {
        Tri q[kChainVZ];
        const int fsx = p.uw[f] > 1 ? 1 : 0;
        const long long fsy = p.uh[f] > 1 ? p.uw[f] : 0;
        const long long fsz = p.ud[f] > 1 ? static_cast<long long>(p.uh[f]) * p.uw[f] : 0;
#pragma unroll
        for (int i = 0; i < kChainVZ; ++i) q[i] = tri_setup(cz[i], cy[i], cx[i], p.ud[f], p.uh[f], p.uw[f]);
#pragma unroll
        for (int i = 0; i < kChainVZ; ++i) {
          const float dz = tri_sample(u, q[i], fsy, fsz, fsx);
          const float dy = tri_sample(u + plane, q[i], fsy, fsz, fsx);
          const float dx = tri_sample(u + 2 * plane, q[i], fsy, fsz, fsx);
          cz[i] += dz; cy[i] += dy; cx[i] += dx;
        }
      }
    }
    float img[kChainVZ];
    if (p.img_out) {
#pragma unroll
      for (int i = 0; i < kChainVZ; ++i) {
        const Tri q = tri_setup(cz[i], cy[i], cx[i], p.id, p.ih, p.iw);
        img[i] = tri_sample(p.img, q, p.ih > 1 ? p.iw : 0, p.id > 1 ? static_cast<long long>(p.ih) * p.iw : 0,
                            p.iw > 1 ? 1 : 0);
      }
    }
#pragma unroll
    for (int i = 0; i < kChainVZ; ++i) {
      if (z0 + i >= p.D) break;
      const long long v = v0 + i * zs;
      if (p.phi_out) {
        p.phi_out[v] = cz[i]; p.phi_out[nvox + v] = cy[i]; p.phi_out[2 * nvox + v] = cx[i];
      }
      if (p.img_out) p.img_out[v] = img[i];
    }
  }
}

// F.interpolate(mode="trilinear", align_corners=False, size=(Do,Ho,Wo)) of a single-channel volume
__global__ void __launch_bounds__(256) resize_trilinear_kernel(const float* __restrict__ in, int Di, int Hi, int Wi,
                                                               float* __restrict__ out, int Do, int Ho, int Wo) {
  const long long nvox = static_cast<long long>(Do) * Ho * Wo;
  const float rz = static_cast<float>(Di) / Do, ry = static_cast<float>(Hi) / Ho, rx = static_cast<float>(Wi) / Wo;
  for (long long v = blockIdx.x * static_cast<long long>(blockDim.x) + threadIdx.x; v < nvox;
       v += static_cast<long long>(gridDim.x) * blockDim.x) {
    const int x = static_cast<int>(v % Wo), y = static_cast<int>((v / Wo) % Ho),
              z = static_cast<int>(v / (static_cast<long long>(Wo) * Ho));
    const float fz = fmaxf(rz * (z + 0.5f) - 0.5f, 0.f), fy = fmaxf(ry * (y + 0.5f) - 0.5f, 0.f),
                fx = fmaxf(rx * (x + 0.5f) - 0.5f, 0.f);
    const int z0 = min(static_cast<int>(fz), Di - 1), y0 = min(static_cast<int>(fy), Hi - 1),
              x0 = min(static_cast<int>(fx), Wi - 1);
    const int z1 = z0 + (z0 < Di - 1), y1 = y0 + (y0 < Hi - 1), x1 = x0 + (x0 < Wi - 1);
    const float lz = fz - z0, ly = fy - y0, lx = fx - x0;
    auto at = [&](int zz, int yy, int xx) { return __ldg(in + (static_cast<size_t>(zz) * Hi + yy) * Wi + xx); };
    out[v] = (1.f - lz) * ((1.f - ly) * ((1.f - lx) * at(z0, y0, x0) + lx * at(z0, y0, x1)) +
                           ly * ((1.f - lx) * at(z0, y1, x0) + lx * at(z0, y1, x1))) +
             lz * ((1.f - ly) * ((1.f - lx) * at(z1, y0, x0) + lx * at(z1, y0, x1)) +
                   ly * ((1.f - lx) * at(z1, y1, x0) + lx * at(z1, y1, x1)));
  }
}

__global__ void __launch_bounds__(256) avgpool2_ceil_kernel(const float* __restrict__ in, int C, int Di, int Hi,
                                                            int Wi, float* __restrict__ out) {
  const int Do = (Di + 1) / 2, Ho = (Hi + 1) / 2, Wo = (Wi + 1) / 2;
  const long long n = static_cast<long long>(C) * Do * Ho * Wo;
  for (long long v = blockIdx.x * static_cast<long long>(blockDim.x) + threadIdx.x; v < n;
       v += static_cast<long long>(gridDim.x) * blockDim.x) {
    long long r = v;
    const int x = r % Wo; r /= Wo;
    const int y = r % Ho; r /= Ho;
    const int z = r % Do; r /= Do;
    const float* pl = in + r * (static_cast<size_t>(Di) * Hi * Wi);
    float s = 0.f;
    int cnt = 0;
    for (int dz = 0; dz < 2; ++dz)
      for (int dy = 0; dy < 2; ++dy)
        for (int dx = 0; dx < 2; ++dx) {
          const int zz = 2 * z + dz, yy = 2 * y + dy, xx = 2 * x + dx;
          if (zz < Di && yy < Hi && xx < Wi) {
            s += __ldg(pl + (static_cast<size_t>(zz) * Hi + yy) * Wi + xx);
            ++cnt;
          }
        }
    out[v] = s / static_cast<float>(cnt);
  }
}

// disp[z][y][x][(x,y,z)] = (phi - identity)[(2,1,0)] * (N - 1)
__global__ void __launch_bounds__(256) disp_field_kernel(const float* __restrict__ phi, int D, int H, int W,
                                                         float* __restrict__ disp) {
  const long long nvox = static_cast<long long>(D) * H * W;
  const double sz = 1.0 / (D - 1), sy = 1.0 / (H - 1), sx = 1.0 / (W - 1);
  for (long long v = blockIdx.x * static_cast<long long>(blockDim.x) + threadIdx.x; v < nvox;
       v += static_cast<long long>(gridDim.x) * blockDim.x) {
    const int x = static_cast<int>(v % W), y = static_cast<int>((v / W) % H),
              z = static_cast<int>(v / (static_cast<long long>(W) * H));
    const float iz = static_cast<float>(z * sz), iy = static_cast<float>(y * sy), ix = static_cast<float>(x * sx);
    disp[3 * v + 0] = (phi[2 * nvox + v] - ix) * static_cast<float>(W - 1);
    disp[3 * v + 1] = (phi[nvox + v] - iy) * static_cast<float>(H - 1);
    disp[3 * v + 2] = (phi[v] - iz) * static_cast<float>(D - 1);
  }
}

// ------------------------------------------------------------------------------------------------ ITK-style warps
__device__ __forceinline__ void affine_apply(const Affine3& a, const double in[3], double out[3]) {
#pragma unroll
  for (int r = 0; r < 3; ++r) out[r] = a.m[3 * r] * in[0] + a.m[3 * r + 1] * in[1] + a.m[3 * r + 2] * in[2] + a.t[r];
}
__device__ __forceinline__ bool affine_is_diagonal(const Affine3& a) {
  return a.m[1] == 0.0 && a.m[2] == 0.0 && a.m[3] == 0.0 && a.m[5] == 0.0 && a.m[6] == 0.0 && a.m[7] == 0.0;
}
// the same map with the axis-aligned case (a third of the fp64 work) as one fused multiply-add per axis; both volume
// warp kernels go through this function so that they round identically
__device__ __forceinline__ void affine_apply_fast(const Affine3& a, bool diagonal, const double in[3], double out[3]) {
  if (diagonal) {
#pragma unroll
    for (int r = 0; r < 3; ++r) out[r] = fma(a.m[4 * r], in[r], a.t[r]);
  } else {
    affine_apply(a, in, out);
  }
}

// q (x,y,z lattice coordinate) += trilinear(disp, q) when q is inside the field buffer [-0.5, n-0.5)
__device__ __forceinline__ void displace(const float* __restrict__ disp, int FD, int FH, int FW, double q[3]) {
  const int n[3] = {FW, FH, FD};
  bool inside = true;
#pragma unroll
  for (int a = 0; a < 3; ++a) inside = inside && q[a] >= -0.5 && q[a] < n[a] - 0.5;
  if (!inside) return;
  int i0[3], i1[3];
  double t[3];
#pragma unroll
  for (int a = 0; a < 3; ++a) {
    const double f = floor(q[a]);
    t[a] = q[a] - f;
    const int b = static_cast<int>(f);
    i0[a] = min(max(b, 0), n[a] - 1);
    i1[a] = min(max(b + 1, 0), n[a] - 1);
  }
  double d[3] = {0, 0, 0};
#pragma unroll
  for (int c = 0; c < 8; ++c) {
    const int ix = (c & 1) ? i1[0] : i0[0], iy = (c & 2) ? i1[1] : i0[1], iz = (c & 4) ? i1[2] : i0[2];
    const double w = ((c & 1) ? t[0] : 1.0 - t[0]) * ((c & 2) ? t[1] : 1.0 - t[1]) * ((c & 4) ? t[2] : 1.0 - t[2]);
    const float* e = disp + ((static_cast<size_t>(iz) * FH + iy) * FW + ix) * 3;
    d[0] += w * __ldg(e); d[1] += w * __ldg(e + 1); d[2] += w * __ldg(e + 2);
  }
  q[0] += d[0]; q[1] += d[1]; q[2] += d[2];
}

// Trilinear sample set-up for one continuous index (x,y,z) with ITK semantics: clamped neighbours, fp32 weights
// derived from the fp64 fractional parts.
struct TriF {
  int i0[3], i1[3];
  float t[3];
};
// floor / fractional split of a lattice coordinate without the slow fp64 conversion instructions (FRND, F2I, I2F):
// adding 1.5 * 2^52 leaves round-to-nearest(s) in the low mantissa word (|s| < 2^31); the remainder s - rn(s) is exact
// in fp64, lies in [-0.5, 0.5] and is folded back to [0, 1) in fp32.
__device__ __forceinline__ TriF trif_setup(const double s[3], const int n[3]) {
  TriF r;
  const double magic = 6755399441055744.0;
#pragma unroll
  for (int a = 0; a < 3; ++a) {
    const double m = s[a] + magic;
    int b = __double2loint(m);
    float d = static_cast<float>(s[a] - (m - magic));
    if (d < 0.f) { d += 1.f; b -= 1; }
    r.t[a] = d;
    r.i0[a] = min(max(b, 0), n[a] - 1);
    r.i1[a] = min(max(b + 1, 0), n[a] - 1);
  }
  return r;
}

// Tile = 32 (x) x 8 (y) output voxels of one z-slice per block; lane <-> x, so the gathers and stores of a warp fall in
// a few 128-byte lines and neighbouring warps (rows) share them through L1.  One voxel per thread.  The kernel is
// issue-bound, not DRAM-bound (profiles/r01_warp_variants.txt: ~420 instructions per voxel in the first version), so
// the structure below is about instruction count: the eight neighbour offsets (32-bit, relative to the channel plane)
// and the eight interpolation weights are computed ONCE per voxel and reused by every channel -- the channel loop is
// eight loads, eight FMAs and a store -- and the displacement gather uses 32-bit element offsets as well.  Staging the
// tile's field footprint in shared memory was measured again in round 2 and is slower (the cooperative copy costs more
// than the L1 gathers it replaces), and so are two further variants built on an axis-aligned output grid -- a block-wide
// staged field box with threads walking z columns, and a warp-cooperative coalesced fetch of the four field rows a
// 32-voxel row touches (fewer L1 wavefronts, but more integer instructions): profiles/r02_warp_variants.json.
// Coordinates stay fp64 (ITK computes in double); interpolation weights and sums are fp32.
template <int kMinBlocks>
__global__ void __launch_bounds__(256, kMinBlocks) warp_volume_kernel(const WarpVolumeParams p) {
  const long long nvox = static_cast<long long>(p.OD) * p.OH * p.OW;
  const size_t splane = static_cast<size_t>(p.SD) * p.SH * p.SW;
  const int nf[3] = {p.FW, p.FH, p.FD}, ns[3] = {p.SW, p.SH, p.SD};
  const int nbx = (p.OW + 31) / 32, nby = (p.OH + 7) / 8;
  const int lane = threadIdx.x & 31, wrp = threadIdx.x >> 5;
  const int x = static_cast<int>(blockIdx.x % nbx) * 32 + lane, y = static_cast<int>((blockIdx.x / nbx) % nby) * 8 + wrp;
  const int z = static_cast<int>(blockIdx.x / (nbx * nby));
  if (x >= p.OW || y >= p.OH) return;
  // ---- lattice coordinate of the output voxel and the displacement there
  double q[3];
  {
    const double j[3] = {static_cast<double>(x), static_cast<double>(y), static_cast<double>(z)};
    affine_apply_fast(p.out_index_to_net, affine_is_diagonal(p.out_index_to_net), j, q);
  }
  bool fin = true;
#pragma unroll
  for (int a = 0; a < 3; ++a) fin = fin && q[a] >= -0.5 && q[a] < p.fhi[a];
  float dx = 0.f, dy = 0.f, dz = 0.f;
  if (fin) {
    const TriF tf = trif_setup(q, nf);
    const int r00 = (tf.i0[2] * p.FH + tf.i0[1]) * p.FW, r01 = (tf.i0[2] * p.FH + tf.i1[1]) * p.FW;
    const int r10 = (tf.i1[2] * p.FH + tf.i0[1]) * p.FW, r11 = (tf.i1[2] * p.FH + tf.i1[1]) * p.FW;
    const float tx = tf.t[0], ty = tf.t[1], tz = tf.t[2];
    const float wy0 = (1.f - ty) * (1.f - tz), wy1 = ty * (1.f - tz), wy2 = (1.f - ty) * tz, wy3 = ty * tz;
    const int rows[4] = {r00, r01, r10, r11};
    const float wr[4] = {wy0, wy1, wy2, wy3};
#pragma unroll
    for (int k = 0; k < 4; ++k) {
      const float* e0 = p.disp + 3 * (rows[k] + tf.i0[0]);
      const float* e1 = p.disp + 3 * (rows[k] + tf.i1[0]);
      const float w0 = wr[k] * (1.f - tx), w1 = wr[k] * tx;
      dx = fmaf(w0, __ldg(e0), dx); dy = fmaf(w0, __ldg(e0 + 1), dy); dz = fmaf(w0, __ldg(e0 + 2), dz);
      dx = fmaf(w1, __ldg(e1), dx); dy = fmaf(w1, __ldg(e1 + 1), dy); dz = fmaf(w1, __ldg(e1 + 2), dz);
    }
  }
  // ---- source index, inside test, interpolation set-up (once per voxel, shared by every channel)
  const double qd[3] = {q[0] + dx, q[1] + dy, q[2] + dz};
  double sidx[3];
  affine_apply_fast(p.net_to_src_index, affine_is_diagonal(p.net_to_src_index), qd, sidx);
  bool sin = true;
#pragma unroll
  for (int a = 0; a < 3; ++a) sin = sin && sidx[a] >= -0.5 && sidx[a] < p.shi[a];
  const long long v = (static_cast<long long>(z) * p.OH + y) * p.OW + x;
  if (!sin) {
    for (int c = 0; c < p.C; ++c) p.out[c * nvox + v] = p.default_value;
    return;
  }
  const TriF ts = trif_setup(sidx, ns);
  int off[8];
  float w[8];
  {
    const int r00 = (ts.i0[2] * p.SH + ts.i0[1]) * p.SW, r01 = (ts.i0[2] * p.SH + ts.i1[1]) * p.SW;
    const int r10 = (ts.i1[2] * p.SH + ts.i0[1]) * p.SW, r11 = (ts.i1[2] * p.SH + ts.i1[1]) * p.SW;
    const float tx = ts.t[0], ty = ts.t[1], tz = ts.t[2];
    const float a0 = (1.f - ty) * (1.f - tz), a1 = ty * (1.f - tz), a2 = (1.f - ty) * tz, a3 = ty * tz;
    off[0] = r00 + ts.i0[0]; off[1] = r00 + ts.i1[0]; off[2] = r01 + ts.i0[0]; off[3] = r01 + ts.i1[0];
    off[4] = r10 + ts.i0[0]; off[5] = r10 + ts.i1[0]; off[6] = r11 + ts.i0[0]; off[7] = r11 + ts.i1[0];
    w[0] = a0 * (1.f - tx); w[1] = a0 * tx; w[2] = a1 * (1.f - tx); w[3] = a1 * tx;
    w[4] = a2 * (1.f - tx); w[5] = a2 * tx; w[6] = a3 * (1.f - tx); w[7] = a3 * tx;
  }
  const float* src = p.src;
  float* dst = p.out + v;
  for (int c = 0; c < p.C; ++c, src += splane, dst += nvox) {
    float acc = 0.f;
#pragma unroll
    for (int k = 0; k < 8; ++k) acc = fmaf(w[k], __ldg(src + off[k]), acc);
    *dst = acc;
  }
}

// ---- the same resampling with neighbours at fixed strides
// The gather kernel above spends most of its ~380 (C = 1) to ~550 (C = 8) instructions per voxel on address arithmetic:
// every one of its 24 + 8 C loads carries its own clamped 32-bit offset and a three- or four-instruction 64-bit address
// (profiles/r02_warp_sass_notes.txt).  Here the clamping is folded into the interpolation fraction instead: a lattice
// coordinate whose lower / upper neighbour would be clamped (s in [-0.5, 0) or [n-1, n-0.5)) takes the base index 0 /
// n-2 with fraction 0 / 1 -- the same value, v[0] or v[n-1] -- so the eight corners of EVERY voxel sit at the same
// offsets {0, 1} + {0, W} + {0, H W} from one base pointer.  Per voxel and channel that is one 64-bit pointer bump,
// three row pointers and eight loads with immediate offsets.  Needs every lattice dimension >= 2 (else the gather kernel).
struct Tri1 {
  int b[3];
  float t[3];
};
__device__ __forceinline__ Tri1 tri1_setup(const double s[3], const int n[3]) {
  Tri1 r;
  const double magic = 6755399441055744.0;
#pragma unroll
  for (int a = 0; a < 3; ++a) {
    const double m = s[a] + magic;
    int b = __double2loint(m);
    float d = static_cast<float>(s[a] - (m - magic));
    if (d < 0.f) { d += 1.f; b -= 1; }
    if (b < 0) { b = 0; d = 0.f; }
    if (b > n[a] - 2) { b = n[a] - 2; d = 1.f; }
    r.b[a] = b;
    r.t[a] = d;
  }
  return r;
}

// A block owns a 32 (x) x 8 (y) tile over kWarpZ consecutive output slices and walks them in order: the upper
// neighbour planes (field and source) of slice z are the lower ones of slice z + 1 and are still in L1.  With one slice
// per block every corner plane came from L2 twice; the sweep was bound by L2 -> SM traffic (~24 B per voxel and channel
// against 8 B algorithmic), which is why trimming instructions alone did not move it.
constexpr int kWarpZ = 4;
template <int kMinBlocks>
__global__ void __launch_bounds__(256, kMinBlocks) warp_volume_fast_kernel(const WarpVolumeParams p) {
  const long long nvox = static_cast<long long>(p.OD) * p.OH * p.OW;
  const long long splane = static_cast<long long>(p.SD) * p.SH * p.SW;
  const int nf[3] = {p.FW, p.FH, p.FD}, ns[3] = {p.SW, p.SH, p.SD};
  const int nbx = (p.OW + 31) / 32, nby = (p.OH + 7) / 8;
  const int lane = threadIdx.x & 31, wrp = threadIdx.x >> 5;
  const int xl = static_cast<int>(blockIdx.x % nbx) * 32 + lane, y = static_cast<int>((blockIdx.x / nbx) % nby) * 8 + wrp;
  const int z0 = static_cast<int>(blockIdx.x / (nbx * nby)) * kWarpZ;
  if (y >= p.OH) return;                 // whole warp
  const bool live = xl < p.OW;           // lanes past the row's end shadow its last voxel and store nothing
  const int x = min(xl, p.OW - 1);
  const bool diag1 = affine_is_diagonal(p.out_index_to_net), diag2 = affine_is_diagonal(p.net_to_src_index);
  const long long frow = 3ll * p.FW, fslice = frow * p.FH;
  const long long srow = p.SW, sslice = static_cast<long long>(p.SW) * p.SH;
  const int z1 = min(z0 + kWarpZ, p.OD);
  for (int z = z0; z < z1; ++z) {
    double q[3];
    {
      const double j[3] = {static_cast<double>(x), static_cast<double>(y), static_cast<double>(z)};
      affine_apply_fast(p.out_index_to_net, diag1, j, q);
    }
    bool fin = true;
#pragma unroll
    for (int a = 0; a < 3; ++a) fin = fin && q[a] >= -0.5 && q[a] < p.fhi[a];
    float dx = 0.f, dy = 0.f, dz = 0.f;
    if (fin) {
      const Tri1 tf = tri1_setup(q, nf);
      const float* e00 = p.disp + 3 * ((tf.b[2] * p.FH + tf.b[1]) * p.FW + tf.b[0]);
      const float* e01 = e00 + frow;
      const float* e10 = e00 + fslice;
      const float* e11 = e10 + frow;
      const float tx = tf.t[0], ty = tf.t[1], tz = tf.t[2];
      const float wr[4] = {(1.f - ty) * (1.f - tz), ty * (1.f - tz), (1.f - ty) * tz, ty * tz};
      const float* rows[4] = {e00, e01, e10, e11};
#pragma unroll
      for (int k = 0; k < 4; ++k) {
        const float* e = rows[k];
        const float w0 = wr[k] * (1.f - tx), w1 = wr[k] * tx;
        dx = fmaf(w0, __ldg(e), dx); dy = fmaf(w0, __ldg(e + 1), dy); dz = fmaf(w0, __ldg(e + 2), dz);
        dx = fmaf(w1, __ldg(e + 3), dx); dy = fmaf(w1, __ldg(e + 4), dy); dz = fmaf(w1, __ldg(e + 5), dz);
      }
    }
    const double qd[3] = {q[0] + dx, q[1] + dy, q[2] + dz};
    double sidx[3];
    affine_apply_fast(p.net_to_src_index, diag2, qd, sidx);
    bool sin = true;
#pragma unroll
    for (int a = 0; a < 3; ++a) sin = sin && sidx[a] >= -0.5 && sidx[a] < p.shi[a];
    float* dst = p.out + (static_cast<long long>(z) * p.OH + y) * p.OW + x;
    if (!sin) {
      if (live)
        for (int c = 0; c < p.C; ++c, dst += nvox) *dst = p.default_value;
      continue;
    }
    const Tri1 ts = tri1_setup(sidx, ns);
    float w[8];
    {
      const float tx = ts.t[0], ty = ts.t[1], tz = ts.t[2];
      const float a0 = (1.f - ty) * (1.f - tz), a1 = ty * (1.f - tz), a2 = (1.f - ty) * tz, a3 = ty * tz;
      w[0] = a0 * (1.f - tx); w[1] = a0 * tx; w[2] = a1 * (1.f - tx); w[3] = a1 * tx;
      w[4] = a2 * (1.f - tx); w[5] = a2 * tx; w[6] = a3 * (1.f - tx); w[7] = a3 * tx;
    }
    const int sbase = (ts.b[2] * p.SH + ts.b[1]) * p.SW + ts.b[0];
    {
      const float* s00 = p.src + sbase;
      // one channel per trip: the eight loads are issued back to back, then consumed (an unrolled loop at this register
      // budget interleaves each load with its use and serialises on the load latency: 2x slower for C >= 4)
#pragma unroll 1
      for (int c = 0; c < p.C; ++c, s00 += splane, dst += nvox) {
        const float* s01 = s00 + srow;
        const float* s10 = s00 + sslice;
        const float* s11 = s10 + srow;
        const float v0 = __ldg(s00), v1 = __ldg(s00 + 1), v2 = __ldg(s01), v3 = __ldg(s01 + 1);
        const float v4 = __ldg(s10), v5 = __ldg(s10 + 1), v6 = __ldg(s11), v7 = __ldg(s11 + 1);
        float acc = w[0] * v0;
        acc = fmaf(w[1], v1, acc);
        acc = fmaf(w[2], v2, acc);
        acc = fmaf(w[3], v3, acc);
        acc = fmaf(w[4], v4, acc);
        acc = fmaf(w[5], v5, acc);
        acc = fmaf(w[6], v6, acc);
        acc = fmaf(w[7], v7, acc);
        if (live) *dst = acc;
      }
    }
  }
}

__global__ void __launch_bounds__(128) warp_points_kernel(const WarpPointsParams p) {
  for (long long i = blockIdx.x * static_cast<long long>(blockDim.x) + threadIdx.x; i < p.n;
       i += static_cast<long long>(gridDim.x) * blockDim.x) {
    const double pt[3] = {p.pts[3 * i], p.pts[3 * i + 1], p.pts[3 * i + 2]};
    double q[3], o[3];
    affine_apply(p.phys_to_net, pt, q);
    displace(p.disp, p.FD, p.FH, p.FW, q);
    affine_apply(p.net_to_phys, q, o);
    p.out[3 * i] = o[0]; p.out[3 * i + 1] = o[1]; p.out[3 * i + 2] = o[2];
  }
}

inline unsigned grid_for(long long n, int block, int per_sm) {
  long long b = (n + block - 1) / block;
  const long long cap = static_cast<long long>(num_sms()) * per_sm;
  if (b > cap) b = cap;
  if (b < 1) b = 1;
  return static_cast<unsigned>(b);
}

}  // namespace

template <int CO_T, int XS, int KS>
static void conv3_dispatch(const Conv3Params& p, cudaStream_t st) {
  const long long nthr = static_cast<long long>(p.Do) * p.Ho * ((p.Wo + XS - 1) / XS);
  constexpr int NV = 128 / KS;
  dim3 g(static_cast<unsigned>((nthr + NV - 1) / NV), (p.cout + CO_T - 1) / CO_T, p.N);
  if (p.stride == 1) conv3_kernel<CO_T, XS, 1, KS><<<g, 128, 0, st>>>(p);
  else conv3_kernel<CO_T, XS, 2, KS><<<g, 128, 0, st>>>(p);
}

// ci range per block so that the grid has a few hundred blocks
static int deep_ci_split(int cin, long long blocks_per_split) {
  int nsplit = 1;
  while (blocks_per_split * nsplit < 592 && cin / (nsplit * 2) >= 64) nsplit *= 2;
  return nsplit;
}

size_t conv3_splitk_bytes(const Conv3Params& p) {
  const long long M = static_cast<long long>(p.N) * p.Do * p.Ho * p.Wo;
  if (p.stride != 2 || !p.leaky_in || p.cin < 64 || M > 4096) return 0;
  const long long tiles = ((M + 63) / 64) * ((p.cout + 63) / 64) * 27;
  return static_cast<size_t>(27) * deep_ci_split(p.cin, tiles) * M * p.cout * sizeof(float);
}

size_t convt4_splitk_bytes(const ConvT4Params& p) {
  if (p.Wi >= 12) return 0;
  const long long M = static_cast<long long>(p.N) * p.Di * p.Hi * p.Wi;
  const long long tiles = ((M + 63) / 64) * ((p.cout + 63) / 64) * 64;
  return static_cast<size_t>(8) * deep_ci_split(p.cin, tiles) * 8 * M * p.cout * sizeof(float);
}

int conv3_launch(const Conv3Params& p, cudaStream_t st) {
  const long long nvox = static_cast<long long>(p.Do) * p.Ho * p.Wo;
  // tcgen05 path (reg_umma_down.cu): the strided levels with 16+ input channels; OAI_B200_CONV3_UMMA=0 is the A/B switch
  if (p.wumma && p.xsplit && conv3_umma_eligible(p) && p.xsplit_bytes >= conv3_umma_workspace(p))
    return conv3_umma_launch(p, st);
  const size_t need = conv3_splitk_bytes(p);
  if (need && p.splitk_ws && p.splitk_bytes >= need) {
    DeepGemmParams g;
    g.in = p.in; g.in_nstride = p.in_nstride; g.in_cstride = p.in_cstride; g.cin = p.cin;
    g.Di = p.Di; g.Hi = p.Hi; g.Wi = p.Wi;
    g.w = p.w; g.taps_total = 27; g.wld = p.cout_pad; g.cout = p.cout;
    g.N = p.N; g.Mo_d = p.Do; g.Mo_h = p.Ho; g.Mo_w = p.Wo;
    g.ntaps = 27; g.ncls = 1; g.ws = p.splitk_ws;
    const long long M = static_cast<long long>(p.N) * nvox;
    const long long tiles = ((M + 63) / 64) * ((p.cout + 63) / 64);
    g.nsplit = deep_ci_split(p.cin, tiles * 27);
    g.ci_per_split = (p.cin + g.nsplit - 1) / g.nsplit;
    deep_gemm_kernel<0><<<dim3(static_cast<unsigned>(tiles), 1, 27 * g.nsplit), 256, 0, st>>>(g);
    if (int rc = launched("deep_gemm_kernel (conv3)")) return rc;
    deep_reduce_conv3_kernel<<<grid_for(M * p.cout, 256, 8), 256, 0, st>>>(p, p.splitk_ws, 27 * g.nsplit);
    return launched("deep_reduce_conv3_kernel");
  }
  if (p.cout == 3) conv3_dispatch<3, 8, 1>(p, st);              // lastConv: 18 -> 3 at full resolution: no FMAs on a
                                                                 // padding channel (a row-walking variant with lanes along x
                                                                 // and 8 output rows per thread measured 2x slower:
                                                                 // 1.31 vs 0.65 ms at 80x192x192, latency-bound; a
                                                                 // 4-outputs-per-thread variant with lanes 16 bytes apart and
                                                                 // the halo samples by shuffle: 0.86 ms, bit-identical;
                                                                 // shuffled halos inside this kernel's pipelined row loads:
                                                                 // 1.13 ms -- the shuffle waits for the load it forwards.
                                                                 // ncu: L1 pipe 85 %, FMA pipe 43 %)
  else if (p.cout <= 4) conv3_dispatch<4, 8, 1>(p, st);
  else if (nvox * ((p.cout + 7) / 8) >= (1 << 16)) conv3_dispatch<8, 4, 1>(p, st);
  else if (p.cin >= 32) conv3_dispatch<8, 1, 4>(p, st);          // deep levels: few voxels, many channels
  else conv3_dispatch<8, 1, 1>(p, st);
  return launched("conv3_kernel");
}

template <int CO_T, int XP, int KS>
static void convt4_dispatch(const ConvT4Params& p, cudaStream_t st) {
  const int Wp = (p.Wo + 1) / 2;
  const long long nthr = static_cast<long long>(p.Do) * p.Ho * ((Wp + XP - 1) / XP);
  constexpr int NV = 128 / KS;
  dim3 g(static_cast<unsigned>((nthr + NV - 1) / NV), (p.cout + CO_T - 1) / CO_T, p.N);
  convt4_kernel<CO_T, XP, KS><<<g, 128, 0, st>>>(p);
}

// `planes` dense planes of Di x Hi x Wi 32-bit words as a rank-5 TMA tensor (W, H, D, plane, 1);
// box = (bx, by, 3, box_planes, 1) words, no swizzle, zero fill outside
static int make_plane_tmap(CUtensorMap* tm, void* base, unsigned long long planes, int box_planes,
                           const ConvT4Params& p, int bx, int by) {
  typedef CUresult (*EncodeTiledFn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*,
                                    const cuuint64_t*, const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave,
                                    CUtensorMapSwizzle, CUtensorMapL2promotion, CUtensorMapFloatOOBfill);
  static EncodeTiledFn fn = nullptr;
  if (!fn) {
    void* q = nullptr;
    cudaDriverEntryPointQueryResult r;
    if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &q, cudaEnableDefault, &r) == cudaSuccess &&
        r == cudaDriverEntryPointSuccess)
      fn = reinterpret_cast<EncodeTiledFn>(q);
  }
  if (!fn) return fail("convt4_mma: cuTensorMapEncodeTiled not available from the driver");
  cuuint64_t dims[5] = {(cuuint64_t)p.Wi, (cuuint64_t)p.Hi, (cuuint64_t)p.Di, planes, 1};
  cuuint64_t strides[4] = {(cuuint64_t)p.Wi * 4, (cuuint64_t)p.Hi * p.Wi * 4, (cuuint64_t)p.Di * p.Hi * p.Wi * 4,
                           planes * p.Di * p.Hi * p.Wi * 4};
  cuuint32_t box[5] = {(cuuint32_t)bx, (cuuint32_t)by, 3, (cuuint32_t)box_planes, 1};
  cuuint32_t estr[5] = {1, 1, 1, 1, 1};
  const CUresult r = fn(tm, CU_TENSOR_MAP_DATA_TYPE_UINT32, 5, base, dims, strides, box, estr,
                        CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_NONE, CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
                        CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  if (r != CUDA_SUCCESS)
    return fail("convt4_mma: cuTensorMapEncodeTiled failed with %d (W=%d H=%d D=%d planes=%llu box %dx%d)", (int)r, p.Wi,
                p.Hi, p.Di, (unsigned long long)planes, bx, by);
  return 0;
}

template <int TX>
static int convt4_mma_dispatch(const ConvT4Params& p, cudaStream_t st) {
  using Cfg = ConvT4MmaCfg<TX>;
  static bool configured[64] = {false};   // the attribute is per device
  int dev = 0;
  cudaGetDevice(&dev);
  if (dev < 0 || dev >= 64 || !configured[dev]) {
    if (int rc = check_cuda(cudaFuncSetAttribute(convt4_mma_kernel<TX>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                                 static_cast<int>(Cfg::smem_bytes)),
                            "convt4_mma: cudaFuncSetAttribute"))
      return rc;
    if (dev >= 0 && dev < 64) configured[dev] = true;
  }
  CUtensorMap tm, tm_res;
  if (int rc = make_plane_tmap(&tm, p.xsplit, static_cast<unsigned long long>(2) * p.N * (p.cin / 2), 8, p, Cfg::SX,
                               Cfg::SY))
    return rc;
  // raw fp32 input planes for the residual: sample n, channel c = plane n * (in_nstride / in_cstride) + c
  const unsigned long long ratio = static_cast<unsigned long long>(p.in_nstride / p.in_cstride);
  if (int rc = make_plane_tmap(&tm_res, const_cast<float*>(p.in), (p.N - 1) * ratio + p.cin, 16, p, Cfg::SX, Cfg::SY))
    return rc;
  const long long vol = static_cast<long long>(p.Di) * p.Hi * p.Wi;
  reg_split_kernel<<<grid_for(p.N * (p.cin / 2) * vol, 256, 16), 256, 0, st>>>(p.in, p.in_nstride, p.in_cstride, p.N,
                                                                              p.cin, vol, p.xsplit);
  if (int rc = launched("reg_split_kernel")) return rc;
  const int ntx = (p.Wi + TX - 1) / TX, nty = (p.Hi + Cfg::TY - 1) / Cfg::TY;
  dim3 g(static_cast<unsigned>(ntx) * nty * p.Di, p.cout / 16, p.N);
  static const int dbg = getenv("OAI_CONVT4_DEBUG") ? atoi(getenv("OAI_CONVT4_DEBUG")) : 0;
  ConvT4Params q = p;
  q.debug = dbg;
  q.res_planes_per_n = static_cast<int>(ratio);
  convt4_mma_kernel<TX><<<g, 128, Cfg::smem_bytes, st>>>(tm, tm_res, q);
  return 0;
}

int reg_pack_convt4_launch(const float* w, int cin, int cout, int wexp, uint4* wpk, cudaStream_t st) {
  const long long total = static_cast<long long>(cout / 16) * (cin / 16) * 64 * 2 * 32;
  reg_pack_convt4_kernel<<<grid_for(total, 256, 8), 256, 0, st>>>(w, cin, cout, wexp, wpk);
  return launched("reg_pack_convt4_kernel");
}

static bool convt4_umma_disabled() {
  const char* e = getenv("OAI_B200_CONVT4_UMMA");
  return e && e[0] == '0';
}

int convt4_launch(const ConvT4Params& p, cudaStream_t st) {
  const long long nout = static_cast<long long>(p.Do) * p.Ho * p.Wo;
  // levels narrower than 12 lattice points (the two deepest): 3x3 / 6x6 planes fill too little of an MMA tile; with a
  // workspace they run as split-K fp32 GEMMs, otherwise on the parity-class kernel below
  if (const size_t need = convt4_splitk_bytes(p); need && p.xsplit && p.xsplit_bytes >= need) {
    DeepGemmParams g;
    g.in = p.in; g.in_nstride = p.in_nstride; g.in_cstride = p.in_cstride; g.cin = p.cin;
    g.Di = p.Di; g.Hi = p.Hi; g.Wi = p.Wi;
    g.w = p.w; g.taps_total = 64; g.wld = p.cout; g.cout = p.cout;
    g.N = p.N; g.Mo_d = p.Di; g.Mo_h = p.Hi; g.Mo_w = p.Wi;
    g.ntaps = 8; g.ncls = 8; g.ws = reinterpret_cast<float*>(p.xsplit);
    const long long M = static_cast<long long>(p.N) * p.Di * p.Hi * p.Wi;
    const long long tiles = ((M + 63) / 64) * ((p.cout + 63) / 64);
    g.nsplit = deep_ci_split(p.cin, tiles * 64);
    g.ci_per_split = (p.cin + g.nsplit - 1) / g.nsplit;
    deep_gemm_kernel<1><<<dim3(static_cast<unsigned>(tiles), 8, 8 * g.nsplit), 256, 0, st>>>(g);
    if (int rc = launched("deep_gemm_kernel (convt4)")) return rc;
    deep_reduce_convt4_kernel<<<grid_for(static_cast<long long>(p.N) * nout * p.cout, 256, 8), 256, 0, st>>>(
        p, reinterpret_cast<const float*>(p.xsplit), 8 * g.nsplit);
    return launched("deep_reduce_convt4_kernel");
  }
  // tcgen05 path (reg_umma.cu): the wide levels with 16 - 64 output channels; OAI_B200_CONVT4_UMMA=0 is the A/B switch
  if (p.wumma && p.xsplit && convt4_umma_eligible(p) && !convt4_umma_disabled() &&
      p.xsplit_bytes >= static_cast<size_t>(p.N) * p.cin * p.Di * p.Hi * p.Wi * 4)
    return convt4_umma_launch(p, st);
  // tensor path: rows must be 16-byte multiples for the TMA boxes (every tallUNet2 level that is wide enough is)
  if (p.wpk && p.xsplit && p.cin % 16 == 0 && p.cout % 16 == 0 && p.Wi >= 12 && p.Wi % 4 == 0 &&
      p.in_cstride == static_cast<long long>(p.Di) * p.Hi * p.Wi && p.in_nstride % p.in_cstride == 0 &&
      (reinterpret_cast<uintptr_t>(p.in) & 15) == 0 &&
      p.xsplit_bytes >= static_cast<size_t>(p.N) * p.cin * p.Di * p.Hi * p.Wi * 4) {
    if (int rc = p.Wi > 16 ? convt4_mma_dispatch<32>(p, st) : convt4_mma_dispatch<16>(p, st)) return rc;
    return launched("convt4_mma_kernel");
  }
  if (nout * ((p.cout + 7) / 8) >= (1 << 17) && p.cout % 8 == 0) {
    // large levels: shared-memory tiled kernel (2 x 8 x 64 output voxels per block)
    constexpr int CO_T = 8;
    constexpr size_t smem = (2 * kTileCI * kTileIn + 2 * kTileCI * 64 * CO_T) * sizeof(float);
    static bool configured[64] = {false};   // the attribute is per device
    int dev = 0;
    cudaGetDevice(&dev);
    if (dev < 0 || dev >= 64 || !configured[dev]) {
      if (int rc = check_cuda(cudaFuncSetAttribute(convt4_tile_kernel<CO_T>,
                                                   cudaFuncAttributeMaxDynamicSharedMemorySize, static_cast<int>(smem)),
                              "convt4_tile: cudaFuncSetAttribute"))
        return rc;
      if (dev >= 0 && dev < 64) configured[dev] = true;
    }
    const int ntx = ((p.Wo + 1) / 2 + 31) / 32, nty = ((p.Ho + 1) / 2 + 3) / 4, ntz = (p.Do + 1) / 2;
    dim3 g(static_cast<unsigned>(ntx) * nty * ntz, p.cout / CO_T, p.N);
    convt4_tile_kernel<CO_T><<<g, 128, smem, st>>>(p);
  } else if (nout * ((p.cout + 7) / 8) >= (1 << 17)) {
    convt4_dispatch<8, 4, 1>(p, st);
  } else {
    // deep levels: one block per output parity class, channel loop split 4 ways
    constexpr int CO_T = 16, KS = 4, NV = 128 / KS;
    const long long ncls = static_cast<long long>((p.Do + 1) / 2) * ((p.Ho + 1) / 2) * ((p.Wo + 1) / 2);
    dim3 g(static_cast<unsigned>((ncls + NV - 1) / NV), (p.cout + CO_T - 1) / CO_T, p.N * 8);
    convt4_par_kernel<CO_T, KS><<<g, 128, 0, st>>>(p);
  }
  return launched("convt4_kernel");
}

int chain_launch(const ChainParams& p, cudaStream_t st) {
  constexpr int vz = 2;
  const long long tiles = static_cast<long long>((p.W + 31) / 32) * ((p.H + 7) / 8) * ((p.D + vz - 1) / vz);
  chain_kernel<vz, 4><<<grid_for(tiles * 256, 256, 64), 256, 0, st>>>(p);
  return launched("chain_kernel");
}

int resize_trilinear_launch(const float* in, int Di, int Hi, int Wi, float* out, int Do, int Ho, int Wo,
                            cudaStream_t st) {
  const long long n = static_cast<long long>(Do) * Ho * Wo;
  resize_trilinear_kernel<<<grid_for(n, 256, 16), 256, 0, st>>>(in, Di, Hi, Wi, out, Do, Ho, Wo);
  return launched("resize_trilinear_kernel");
}

int avgpool2_ceil_launch(const float* in, int C, int Di, int Hi, int Wi, float* out, cudaStream_t st) {
  const long long n = static_cast<long long>(C) * ((Di + 1) / 2) * ((Hi + 1) / 2) * ((Wi + 1) / 2);
  avgpool2_ceil_kernel<<<grid_for(n, 256, 16), 256, 0, st>>>(in, C, Di, Hi, Wi, out);
  return launched("avgpool2_ceil_kernel");
}

int disp_field_launch(const float* phi, int D, int H, int W, float* disp, cudaStream_t st) {
  const long long n = static_cast<long long>(D) * H * W;
  disp_field_kernel<<<grid_for(n, 256, 16), 256, 0, st>>>(phi, D, H, W, disp);
  return launched("disp_field_kernel");
}

// A/B and test switch: OAI_B200_WARP_GATHER=1 forces the general gather kernel
static bool warp_force_gather() {
  const char* e = getenv("OAI_B200_WARP_GATHER");
  return e && e[0] == '1';
}

int warp_volume_launch(const WarpVolumeParams& p, cudaStream_t st) {
  const long long tiles = static_cast<long long>((p.OW + 31) / 32) * ((p.OH + 7) / 8) * p.OD;
  if (tiles <= 0 || tiles > 0x7fffffffLL) return fail("warp_volume: output too large");
  if (static_cast<long long>(p.SD) * p.SH * p.SW >= (1ll << 31) || 3ll * p.FD * p.FH * p.FW >= (1ll << 31))
    return fail("warp_volume: source / field planes must stay below 2^31 elements (32-bit gather offsets)");
  WarpVolumeParams q = p;
  const int nf[3] = {p.FW, p.FH, p.FD}, ns[3] = {p.SW, p.SH, p.SD};
  for (int a = 0; a < 3; ++a) { q.fhi[a] = nf[a] - 0.5; q.shi[a] = ns[a] - 0.5; }
  if (p.FW >= 2 && p.FH >= 2 && p.FD >= 2 && p.SW >= 2 && p.SH >= 2 && p.SD >= 2 && !warp_force_gather()) {
    const long long ftiles = static_cast<long long>((p.OW + 31) / 32) * ((p.OH + 7) / 8) * ((p.OD + kWarpZ - 1) / kWarpZ);
    warp_volume_fast_kernel<5><<<static_cast<unsigned>(ftiles), 256, 0, st>>>(q);
    return launched("warp_volume_fast_kernel");
  }
  warp_volume_kernel<5><<<static_cast<unsigned>(tiles), 256, 0, st>>>(q);
  return launched("warp_volume_kernel");
}

int warp_points_launch(const WarpPointsParams& p, cudaStream_t st) {
  warp_points_kernel<<<grid_for(p.n, 128, 8), 128, 0, st>>>(p);
  return launched("warp_points_kernel");
}

}  // namespace oai
