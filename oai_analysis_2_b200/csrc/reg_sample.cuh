// Trilinear sampling shared by the composition / warp kernels (reg_kernels.cu) and the loss kernels (reg_loss.cu).
#pragma once
#include <cuda_runtime.h>

namespace oai {
namespace {

// ------------------------------------------------------------------------------------------------ sampling helpers
// F.grid_sample(bilinear, border, align_corners=True) at normalised coordinate g = 2c-1 along each axis.
// The neighbour pair of every axis is (b, b + 1) with b <= n - 2: at the clamped upper border (pix == n - 1, where
// grid_sample reads v[n-1] twice with weights 1 and 0) the base steps back to n - 2 and the fraction becomes 1 -- the
// same value -- so the eight corners of every sample sit at fixed offsets {0,1} + {0,W} + {0,HW} from one base
// pointer and the loads take immediate / row-pointer offsets instead of eight separate 64-bit address computations.
// An axis of extent 1 keeps b = 0, t = 0 and a zero stride.
struct Tri {
  long long base;   // element offset of corner (b_z, b_y, b_x) inside one component plane
  float t[3];
};
__device__ __forceinline__ Tri tri_setup(float cz, float cy, float cx, int D, int H, int W) {
  Tri r;
  const float c[3] = {cz, cy, cx};
  const int n[3] = {D, H, W};
  int b[3];
#pragma unroll
  for (int a = 0; a < 3; ++a) {
    const float g = c[a] * 2.f - 1.f;
    float pix = ((g + 1.f) / 2.f) * static_cast<float>(n[a] - 1);
    pix = fminf(fmaxf(pix, 0.f), static_cast<float>(n[a] - 1));
    const float f = floorf(pix);
    int i0 = static_cast<int>(f);
    float t = pix - f;
    if (i0 > n[a] - 2) {   // pix == n - 1 exactly (t == 0): read (n-2, n-1) with weights (0, 1)
      i0 = max(n[a] - 2, 0);
      t = n[a] > 1 ? 1.f : 0.f;
    }
    b[a] = i0;
    r.t[a] = t;
  }
  r.base = (static_cast<long long>(b[0]) * H + b[1]) * W + b[2];
  return r;
}
// sx / sy / sz: element strides of the three axes (0 for an axis of extent 1)
__device__ __forceinline__ float tri_sample(const float* __restrict__ v, const Tri& q, long long sy, long long sz,
                                            int sx) {
  const float* r00 = v + q.base;
  const float* r01 = r00 + sy;
  const float* r10 = r00 + sz;
  const float* r11 = r10 + sy;
  const float v000 = __ldg(r00), v001 = __ldg(r00 + sx);
  const float v010 = __ldg(r01), v011 = __ldg(r01 + sx);
  const float v100 = __ldg(r10), v101 = __ldg(r10 + sx);
  const float v110 = __ldg(r11), v111 = __ldg(r11 + sx);
  const float tz = q.t[0], ty = q.t[1], tx = q.t[2];
  return (1.f - tz) * ((1.f - ty) * ((1.f - tx) * v000 + tx * v001) + ty * ((1.f - tx) * v010 + tx * v011)) +
         tz * ((1.f - ty) * ((1.f - tx) * v100 + tx * v101) + ty * ((1.f - tx) * v110 + tx * v111));
}

}  // namespace
}  // namespace oai
