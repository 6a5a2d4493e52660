// Registration-quality terms of icon_registration's GradientICON.forward (the ICONLoss tuple) on the maps and fields
// oai_reg_forward leaves in its workspace:
//   * gradicon  : the gradient inverse-consistency term, four chains (Ie and Ie + delta * e_d) per point through
//                 phi_BA's then phi_AB's fields, finite differences and squares in registers
//   * jacobian  : losses.flips' dV = ((a x b) . c) on forward differences, the fold count, mean((id - phi)^2)
//   * lncc      : LNCC(sigma) -- moments I, J, I^2, J^2, IJ blurred along z (pass 1, five planes to memory), then along
//                 y and x inside a shared-memory tile with the per-voxel NCC (pass 2)
//   * ssd       : ssd_only_interpolated -- one streaming pass over the warped image, the warped in-bounds tag and the
//                 target
// Every reduction is fixed-order: per-block partial sums in fp64 (one block per tile, no grid-stride loop), then one
// finishing kernel, so equal inputs give bitwise equal terms.  The fold count is an integer sum.  Nothing here
// allocates or synchronises, so the launches can be captured in a CUDA graph.
#include "api_common.h"
#include "reg_kernels.cuh"
#include "reg_sample.cuh"

#include <algorithm>
#include <cmath>

namespace oai {

namespace {

constexpr int kTX = 32, kTY = 8;          // gradicon / jacobian thread tile: a warp per row, 8 rows per block
constexpr int kLZ = 8;                    // lncc pass 1: z outputs per thread
constexpr int kLTX = 64, kLTY = 16;       // lncc pass 2: output tile of one block (one z plane)
constexpr int kSsdPerThread = 8;

// Sum of one double per thread over a 256-thread block in a fixed order; the result is valid on thread 0.
__device__ __forceinline__ double block_sum(double v) {
  __shared__ double warp_sums[8];
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v += __shfl_down_sync(0xffffffffu, v, o);
  if ((threadIdx.x & 31) == 0) warp_sums[threadIdx.x >> 5] = v;
  __syncthreads();
  double r = 0.0;
  if (threadIdx.x == 0)
    for (int i = 0; i < 8; ++i) r += warp_sums[i];
  return r;
}

__global__ void __launch_bounds__(256) gradicon_kernel(const GradIconParams p) {
  const int nbx = (p.W + kTX - 1) / kTX, nby = (p.H + kTY - 1) / kTY;
  const int x = (blockIdx.x % nbx) * kTX + (threadIdx.x & 31);
  const int y = ((blockIdx.x / nbx) % nby) * kTY + (threadIdx.x >> 5);
  const int z = blockIdx.x / (nbx * nby);
  double acc = 0.0;
  if (x < p.W && y < p.H) {
    const long long nvox = static_cast<long long>(p.D) * p.H * p.W;
    const long long v = (static_cast<long long>(z) * p.H + y) * p.W + x;
    const double sz = 1.0 / (p.D - 1), sy = 1.0 / (p.H - 1), sx = 1.0 / (p.W - 1);
    const float id[3] = {static_cast<float>(z * sz), static_cast<float>(y * sy), static_cast<float>(x * sx)};
    // Iepsilon = identity_map + randn / W; the three shifted starts add delta to one coordinate channel each
    float s[4][3], c[4][3];
#pragma unroll
    for (int a = 0; a < 3; ++a) s[0][a] = id[a] + __ldg(p.noise + a * nvox + v) / static_cast<float>(p.W);
#pragma unroll
    for (int d = 0; d < 3; ++d)
#pragma unroll
      for (int a = 0; a < 3; ++a) s[d + 1][a] = a == d ? s[0][a] + p.delta : s[0][a];
#pragma unroll
    for (int i = 0; i < 4; ++i)
#pragma unroll
      for (int a = 0; a < 3; ++a) c[i][a] = s[i][a];
    // phi_AB(phi_BA(c)): direction 0 holds phi_BA's fields, direction 1 phi_AB's, each in application order
    for (int dir = 0; dir < 2; ++dir) {
      for (int f = 0; f < p.nf[dir]; ++f) {
        const float* u = p.u[dir][f];
        const int ud = p.ud[dir][f], uh = p.uh[dir][f], uw = p.uw[dir][f];
        const size_t plane = static_cast<size_t>(ud) * uh * uw;
        const int fsx = uw > 1 ? 1 : 0;
        const long long fsy = uh > 1 ? uw : 0;
        const long long fsz = ud > 1 ? static_cast<long long>(uh) * uw : 0;
        Tri q[4];
#pragma unroll
        for (int i = 0; i < 4; ++i) q[i] = tri_setup(c[i][0], c[i][1], c[i][2], ud, uh, uw);
#pragma unroll
        for (int i = 0; i < 4; ++i) {
          const float dz = tri_sample(u, q[i], fsy, fsz, fsx);
          const float dy = tri_sample(u + plane, q[i], fsy, fsz, fsx);
          const float dx = tri_sample(u + 2 * plane, q[i], fsy, fsz, fsx);
          c[i][0] += dz; c[i][1] += dy; c[i][2] += dx;
        }
      }
    }
    // ((Ie - phi(Ie)) - (Ie_d - phi(Ie_d))) / delta, squared, summed over the channels and the three directions
#pragma unroll
    for (int d = 1; d < 4; ++d)
#pragma unroll
      for (int a = 0; a < 3; ++a) {
        const float g = ((s[0][a] - c[0][a]) - (s[d][a] - c[d][a])) / p.delta;
        acc += static_cast<double>(g) * g;
      }
  }
  const double total = block_sum(acc);
  if (threadIdx.x == 0) p.partials[blockIdx.x] = total;
}

// dV of losses.flips at every cell (z, y, x >= 1) of phi_jac, and (id - phi_mag)^2 at every voxel of phi_mag
__global__ void __launch_bounds__(256) jacobian_kernel(const JacobianParams p) {
  const int nbx = (p.W + kTX - 1) / kTX, nby = (p.H + kTY - 1) / kTY;
  const int x = (blockIdx.x % nbx) * kTX + (threadIdx.x & 31);
  const int y = ((blockIdx.x / nbx) % nby) * kTY + (threadIdx.x >> 5);
  const int z = blockIdx.x / (nbx * nby);
  const long long nvox = static_cast<long long>(p.D) * p.H * p.W, hw = static_cast<long long>(p.H) * p.W;
  const long long v = (static_cast<long long>(z) * p.H + y) * p.W + x;
  const bool in = x < p.W && y < p.H;
  double mag = 0.0;
  if (in && p.phi_mag) {
    const double sz = 1.0 / (p.D - 1), sy = 1.0 / (p.H - 1), sx = 1.0 / (p.W - 1);
    const float id[3] = {static_cast<float>(z * sz), static_cast<float>(y * sy), static_cast<float>(x * sx)};
#pragma unroll
    for (int a = 0; a < 3; ++a) {
      const float e = id[a] - __ldg(p.phi_mag + a * nvox + v);
      mag += static_cast<double>(e * e);
    }
  }
  int neg = 0;
  if (in && z >= 1 && y >= 1 && x >= 1) {
    float a[3], b[3], c[3];
#pragma unroll
    for (int ch = 0; ch < 3; ++ch) {
      const float* q = p.phi_jac + ch * nvox + v;
      const float here = __ldg(q);
      a[ch] = __fsub_rn(here, __ldg(q - hw));
      b[ch] = __fsub_rn(here, __ldg(q - p.W));
      c[ch] = __fsub_rn(here, __ldg(q - 1));
    }
    // torch.cross(a, b, 1) * c summed over the channel axis, without contraction into FMAs
    const float x0 = __fsub_rn(__fmul_rn(a[1], b[2]), __fmul_rn(a[2], b[1]));
    const float x1 = __fsub_rn(__fmul_rn(a[2], b[0]), __fmul_rn(a[0], b[2]));
    const float x2 = __fsub_rn(__fmul_rn(a[0], b[1]), __fmul_rn(a[1], b[0]));
    const float dV = __fadd_rn(__fadd_rn(__fmul_rn(x0, c[0]), __fmul_rn(x1, c[1])), __fmul_rn(x2, c[2]));
    neg = dV < 0.f;
    if (p.det_out)
      p.det_out[(static_cast<long long>(z - 1) * (p.H - 1) + (y - 1)) * (p.W - 1) + (x - 1)] = dV;
  }
  const int nneg = __syncthreads_count(neg);
  if (threadIdx.x == 0 && nneg) atomicAdd(p.count, static_cast<unsigned long long>(nneg));
  if (p.mag_partials) {
    const double total = block_sum(mag);
    if (threadIdx.x == 0) p.mag_partials[blockIdx.x] = total;
  }
}

// LNCC pass 1: the five moment volumes of (I, J) blurred along z with zero padding, written as zb[5][D][H][W].
// A thread owns one (y, x) column and kLZ consecutive z outputs, and scatters each input plane into the outputs it
// reaches (kLZ + 2R loads of I and J for kLZ outputs instead of 2R + 1 per output).
__global__ void __launch_bounds__(256) lncc_zblur_kernel(const LnccParams p) {
  const int nbx = (p.W + kTX - 1) / kTX, nby = (p.H + kTY - 1) / kTY;
  const int x = (blockIdx.x % nbx) * kTX + (threadIdx.x & 31);
  const int y = ((blockIdx.x / nbx) % nby) * kTY + (threadIdx.x >> 5);
  const int z0 = blockIdx.y * kLZ;
  if (x >= p.W || y >= p.H) return;
  const long long hw = static_cast<long long>(p.H) * p.W, nvox = hw * p.D;
  const long long col = static_cast<long long>(y) * p.W + x;
  const int R = p.radius;
  float acc[kLZ][5];
#pragma unroll
  for (int o = 0; o < kLZ; ++o)
#pragma unroll
    for (int m = 0; m < 5; ++m) acc[o][m] = 0.f;
  const int zlo = max(z0 - R, 0), zhi = min(z0 + kLZ - 1 + R, p.D - 1);
  for (int zi = zlo; zi <= zhi; ++zi) {
    const float I = __ldg(p.I + zi * hw + col), J = __ldg(p.J + zi * hw + col);
    const float mo[5] = {I, J, I * I, J * J, I * J};
#pragma unroll
    for (int o = 0; o < kLZ; ++o) {
      const int k = zi - (z0 + o) + R;
      if (k >= 0 && k <= 2 * R) {
        const float w = p.taps[k];
#pragma unroll
        for (int m = 0; m < 5; ++m) acc[o][m] += w * mo[m];
      }
    }
  }
#pragma unroll
  for (int o = 0; o < kLZ; ++o) {
    if (z0 + o >= p.D) break;
#pragma unroll
    for (int m = 0; m < 5; ++m) p.zb[m * nvox + (z0 + o) * hw + col] = acc[o][m];
  }
}

// LNCC pass 2: one kLTY x kLTX output tile of one z plane.  The five z-blurred moments of the tile and its R-halo go
// to shared memory (zero outside the volume), are blurred along y into a second buffer and along x on the way to the
// per-voxel 1 - NCC, whose block sum is the partial.
__global__ void __launch_bounds__(256) lncc_tile_kernel(const LnccParams p) {
  extern __shared__ float smem[];
  const int R = p.radius, K = 2 * R + 1;
  const int SX = kLTX + 2 * R, SY = kLTY + 2 * R;
  float* taps = smem;                               // [K] (padded to 64)
  float* tin = smem + 64;                           // [5][SY][SX]
  float* tmid = tin + 5 * SY * SX;                  // [5][kLTY][SX]
  const int nbx = (p.W + kLTX - 1) / kLTX;
  const int x0 = (blockIdx.x % nbx) * kLTX, y0 = (blockIdx.x / nbx) * kLTY, z = blockIdx.y;
  const long long hw = static_cast<long long>(p.H) * p.W, nvox = hw * p.D;
  for (int i = threadIdx.x; i < K; i += blockDim.x) taps[i] = p.taps[i];
  for (int i = threadIdx.x; i < 5 * SY * SX; i += blockDim.x) {
    const int m = i / (SY * SX), r = (i / SX) % SY, cc = i % SX;
    const int gy = y0 - R + r, gx = x0 - R + cc;
    tin[i] = (gy >= 0 && gy < p.H && gx >= 0 && gx < p.W) ? __ldg(p.zb + m * nvox + z * hw + gy * p.W + gx) : 0.f;
  }
  __syncthreads();
  for (int i = threadIdx.x; i < 5 * kLTY * SX; i += blockDim.x) {
    const int m = i / (kLTY * SX), r = (i / SX) % kLTY, cc = i % SX;
    const float* src = tin + (m * SY + r) * SX + cc;
    float s = 0.f;
    for (int k = 0; k < K; ++k) s += taps[k] * src[k * SX];
    tmid[i] = s;
  }
  __syncthreads();
  double acc = 0.0;
  for (int i = threadIdx.x; i < kLTY * kLTX; i += blockDim.x) {
    const int r = i / kLTX, cx = i % kLTX;
    if (y0 + r >= p.H || x0 + cx >= p.W) continue;
    float b[5];
#pragma unroll
    for (int m = 0; m < 5; ++m) {
      const float* src = tmid + (m * kLTY + r) * SX + cx;
      float s = 0.f;
      for (int k = 0; k < K; ++k) s += taps[k] * src[k];
      b[m] = s;
    }
    const float cross = b[4] - b[0] * b[1];
    const float var_i = fmaxf(b[2] - b[0] * b[0], 0.f) + 1e-5f, var_j = fmaxf(b[3] - b[1] * b[1], 0.f) + 1e-5f;
    acc += static_cast<double>(1.f - cross / sqrtf(var_i * var_j));
  }
  const double total = block_sum(acc);
  if (threadIdx.x == 0) p.partials[static_cast<size_t>(blockIdx.y) * gridDim.x + blockIdx.x] = total;
}

// ssd_only_interpolated of one direction: sum(tag * (warped - target)^2) and sum(tag) per block
__global__ void __launch_bounds__(256) ssd_kernel(const float* __restrict__ warped, const float* __restrict__ tag,
                                                  const float* __restrict__ target, long long n, double* num,
                                                  double* den) {
  double s = 0.0, t = 0.0;
  const long long base = static_cast<long long>(blockIdx.x) * 256 * kSsdPerThread + threadIdx.x;
#pragma unroll
  for (int i = 0; i < kSsdPerThread; ++i) {
    const long long v = base + i * 256;
    if (v < n) {
      const float w = __ldg(tag + v), d = __ldg(warped + v) - __ldg(target + v);
      s += static_cast<double>(w * (d * d));
      t += static_cast<double>(w);
    }
  }
  const double ts = block_sum(s);
  __syncthreads();
  const double tt = block_sum(t);
  if (threadIdx.x == 0) {
    num[blockIdx.x] = ts;
    den[blockIdx.x] = tt;
  }
}

// icon's inbounds_tag: 1 on [1:-1]^3, 0 on the outer shell
__global__ void __launch_bounds__(256) inbounds_tag_kernel(float* tag, int D, int H, int W) {
  const long long n = static_cast<long long>(D) * H * W;
  for (long long v = blockIdx.x * 256ll + threadIdx.x; v < n; v += static_cast<long long>(gridDim.x) * 256) {
    const int x = static_cast<int>(v % W), y = static_cast<int>((v / W) % H), z = static_cast<int>(v / W / H);
    tag[v] = (z >= 1 && z <= D - 2 && y >= 1 && y <= H - 2 && x >= 1 && x <= W - 2) ? 1.f : 0.f;
  }
}

// Fixed-order sum of n doubles over the block; every thread gets the result.
__device__ double sum_partials(const double* p, int n) {
  __shared__ double s[256];
  double v = 0.0;
  for (int i = threadIdx.x; i < n; i += 256) v += p[i];
  s[threadIdx.x] = v;
  __syncthreads();
  for (int o = 128; o > 0; o >>= 1) {
    if (threadIdx.x < o) s[threadIdx.x] += s[threadIdx.x + o];
    __syncthreads();
  }
  const double r = s[0];
  __syncthreads();
  return r;
}

__global__ void __launch_bounds__(256) loss_finish_kernel(const LossFinishParams p) {
  const double ic = sum_partials(p.g, p.ng) / (3.0 * p.nvox);
  double sim = 0.0;
  for (int dir = 0; dir < 2; ++dir) {
    const double* s = p.s + static_cast<size_t>(dir) * 2 * p.ns;
    const double a = sum_partials(s, p.ns);
    sim += p.ssd ? a / sum_partials(s + p.ns, p.ns) : a / p.nvox;
  }
  const double tm = sum_partials(p.m, p.nm) / (3.0 * p.nvox);
  if (threadIdx.x == 0) {
    p.terms[0] = p.lmbda * ic + sim;
    p.terms[1] = ic;
    p.terms[2] = sim;
    p.terms[3] = tm;
    p.terms[4] = static_cast<double>(*p.count);
  }
}

}  // namespace

int gradicon_blocks(int D, int H, int W) { return ((W + kTX - 1) / kTX) * ((H + kTY - 1) / kTY) * D; }
int jacobian_blocks(int D, int H, int W) { return gradicon_blocks(D, H, W); }
int lncc_blocks(int D, int H, int W) { return ((W + kLTX - 1) / kLTX) * ((H + kLTY - 1) / kLTY) * D; }
int ssd_blocks(int D, int H, int W) {
  const long long n = static_cast<long long>(D) * H * W;
  return static_cast<int>((n + 256 * kSsdPerThread - 1) / (256 * kSsdPerThread));
}

int lncc_radius(double sigma) { return static_cast<int>(std::floor(2.0 * sigma)); }

int gradicon_launch(const GradIconParams& p, cudaStream_t st) {
  gradicon_kernel<<<gradicon_blocks(p.D, p.H, p.W), 256, 0, st>>>(p);
  return launched("gradicon_kernel");
}

int jacobian_launch(const JacobianParams& p, cudaStream_t st) {
  if (int rc = check_cuda(cudaMemsetAsync(p.count, 0, sizeof(unsigned long long), st), "jacobian: count reset"))
    return rc;
  jacobian_kernel<<<jacobian_blocks(p.D, p.H, p.W), 256, 0, st>>>(p);
  return launched("jacobian_kernel");
}

size_t lncc_tile_smem(int radius) {
  const int SX = kLTX + 2 * radius, SY = kLTY + 2 * radius;
  return sizeof(float) * (64 + 5 * SY * SX + 5 * kLTY * SX);
}

int lncc_launch(const LnccParams& p, cudaStream_t st) {
  if (p.radius > kLnccMaxRadius) return fail("lncc: blur radius %d above %d", p.radius, kLnccMaxRadius);
  const int nbx = (p.W + kTX - 1) / kTX, nby = (p.H + kTY - 1) / kTY;
  lncc_zblur_kernel<<<dim3(nbx * nby, (p.D + kLZ - 1) / kLZ), 256, 0, st>>>(p);
  if (int rc = launched("lncc_zblur_kernel")) return rc;
  static bool attr_set = false;   // the opt-in covers the largest radius once, before any capture
  if (!attr_set) {
    if (int rc = check_cuda(cudaFuncSetAttribute(lncc_tile_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                                 static_cast<int>(lncc_tile_smem(kLnccMaxRadius))),
                            "lncc: shared memory opt-in"))
      return rc;
    attr_set = true;
  }
  const int tiles = ((p.W + kLTX - 1) / kLTX) * ((p.H + kLTY - 1) / kLTY);
  lncc_tile_kernel<<<dim3(tiles, p.D), 256, lncc_tile_smem(p.radius), st>>>(p);
  return launched("lncc_tile_kernel");
}

int ssd_launch(const float* warped, const float* tag, const float* target, int D, int H, int W, double* num,
               double* den, cudaStream_t st) {
  const long long n = static_cast<long long>(D) * H * W;
  ssd_kernel<<<ssd_blocks(D, H, W), 256, 0, st>>>(warped, tag, target, n, num, den);
  return launched("ssd_kernel");
}

int inbounds_tag_launch(float* tag, int D, int H, int W, cudaStream_t st) {
  const long long n = static_cast<long long>(D) * H * W;
  const long long blocks = std::min<long long>((n + 255) / 256, static_cast<long long>(num_sms()) * 16);
  inbounds_tag_kernel<<<static_cast<unsigned>(blocks), 256, 0, st>>>(tag, D, H, W);
  return launched("inbounds_tag_kernel");
}

int loss_finish_launch(const LossFinishParams& p, cudaStream_t st) {
  loss_finish_kernel<<<1, 256, 0, st>>>(p);
  return launched("loss_finish_kernel");
}

}  // namespace oai
