// Intensity pre-normalisation on the device: oai_analysis/dask_processing.py:10-26 (image_normalize) =
//   window_min/max = np.percentile(volume, p_lo / p_hi)          (numpy "linear" method: lerp of two order statistics)
//   itk.IntensityWindowingImageFilter: x < wmin -> out_min, x > wmax -> out_max, else x * factor + offset (in double)
// The reference sorts (partitions) 23.6 M voxels on the host; here the four order statistics come from an exact
// three-pass radix select (11 + 11 + 10 bits of the order-preserving integer image of the float keys), with no host
// round trip: histogram -> pick bin -> histogram of the surviving prefix ... -> window -> apply.  HBM-bound: the volume
// is read four times and written once (20 B / voxel).
#include "../../include/oai_b200.h"
#include "api_common.h"
#include "radix_select.cuh"

namespace oai {
namespace {

__global__ void __launch_bounds__(256) window_init_kernel(SelectState* s, long long n, double p_lo, double p_hi) {
  const int t = threadIdx.x;
  select_reset(s);
  if (t == 0) s->n = n;
  if (t < 2) {
    // numpy >= 2 on a float32 array (NEP 50: the Python-float percentile and the integer count are "weak" and take the
    // array's dtype): q = float32(p) / float32(100); virtual index = float32(n - 1) * q; previous = floor, next =
    // previous + 1, both the last element once the virtual index reaches n - 1; gamma = virtual - previous, in float32
    // (numpy/lib/_function_base_impl.py::_quantile, _get_indexes, _get_gamma).
    const float q = __fdiv_rn(static_cast<float>(t == 0 ? p_lo : p_hi), 100.f);
    const float vi = __fmul_rn(static_cast<float>(n - 1), q);
    unsigned long long k0, k1;
    float gamma;
    if (vi >= static_cast<float>(n - 1)) {
      k0 = k1 = static_cast<unsigned long long>(n - 1);
      gamma = 0.f;
    } else {
      const float f = fmaxf(floorf(vi), 0.f);
      k0 = static_cast<unsigned long long>(f);
      k1 = k0 + 1;
      gamma = __fsub_rn(vi, f);
    }
    s->rank[2 * t] = k0;
    s->rank[2 * t + 1] = k1;
    s->frac[t] = gamma;
  }
}

// numpy _lerp in float32 of percentile i from the selected order statistics: a + (b - a) * t, taken from the other end
// for t >= 0.5
__device__ __forceinline__ float window_bound(const SelectState* s, int i) {
  const float a = key_float(s->prefix[2 * i]), b = key_float(s->prefix[2 * i + 1]);
  const float t = s->frac[i], d = __fsub_rn(b, a);
  return t >= 0.5f ? __fsub_rn(b, __fmul_rn(d, __fsub_rn(1.f, t))) : __fadd_rn(a, __fmul_rn(d, t));
}

__global__ void __launch_bounds__(256) window_apply_kernel(const float* __restrict__ in, long long n,
                                                           SelectState* __restrict__ s, float out_min,
                                                           float out_max, float* __restrict__ out) {
  const float wmin = window_bound(s, 0), wmax = window_bound(s, 1);
  if (blockIdx.x == 0 && threadIdx.x == 0) {
    s->window[0] = static_cast<double>(wmin);
    s->window[1] = static_cast<double>(wmax);
  }
  // itk::Functor::IntensityWindowingTransform: factor / offset in RealType (double)
  const double factor = (static_cast<double>(out_max) - static_cast<double>(out_min)) /
                        (static_cast<double>(wmax) - static_cast<double>(wmin));
  const double offset = static_cast<double>(out_min) - static_cast<double>(wmin) * factor;
  auto f = [&](float x) {
    if (x < wmin) return out_min;
    if (x > wmax) return out_max;
    return static_cast<float>(static_cast<double>(x) * factor + offset);
  };
  const long long n4 = n / 4;
  const bool vec = ((reinterpret_cast<uintptr_t>(in) | reinterpret_cast<uintptr_t>(out)) & 15) == 0;
  if (vec) {
    for (long long i = blockIdx.x * static_cast<long long>(blockDim.x) + threadIdx.x; i < n4;
         i += static_cast<long long>(gridDim.x) * blockDim.x) {
      const float4 v = __ldg(reinterpret_cast<const float4*>(in) + i);
      reinterpret_cast<float4*>(out)[i] = make_float4(f(v.x), f(v.y), f(v.z), f(v.w));
    }
    if (blockIdx.x == 0)
      for (long long i = 4 * n4 + threadIdx.x; i < n; i += blockDim.x) out[i] = f(__ldg(in + i));
  } else {
    for (long long i = blockIdx.x * static_cast<long long>(blockDim.x) + threadIdx.x; i < n;
         i += static_cast<long long>(gridDim.x) * blockDim.x)
      out[i] = f(__ldg(in + i));
  }
}

}  // namespace
}  // namespace oai

using namespace oai;

extern "C" size_t oai_intensity_window_workspace(void) { return sizeof(SelectState); }

extern "C" int oai_intensity_window(const float* in, long long n, double perc_lo, double perc_hi, float out_min,
                                    float out_max, float* out, void* workspace, size_t workspace_bytes,
                                    void* stream) {
  OAI_REQUIRE(in && out && workspace, "intensity_window: null pointer");
  OAI_REQUIRE(n > 0, "intensity_window: empty volume");
  OAI_REQUIRE(perc_lo >= 0.0 && perc_hi <= 100.0 && perc_lo <= perc_hi,
              "intensity_window: percentiles must satisfy 0 <= lo <= hi <= 100 (got %g, %g)", perc_lo, perc_hi);
  OAI_REQUIRE(workspace_bytes >= sizeof(SelectState) && (reinterpret_cast<uintptr_t>(workspace) & 7) == 0,
              "intensity_window: workspace of %zu bytes (8-byte aligned) required", sizeof(SelectState));
  OAI_REQUIRE((reinterpret_cast<uintptr_t>(in) & 15) == 0, "intensity_window: input must be 16-byte aligned");
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  SelectState* s = static_cast<SelectState*>(workspace);
  const unsigned grid = static_cast<unsigned>(num_sms()) * 4;
  window_init_kernel<<<1, 256, 0, st>>>(s, n, perc_lo, perc_hi);
  if (int rc = launched("window_init_kernel")) return rc;
  if (int rc = select_launch(in, s, grid, st)) return rc;
  window_apply_kernel<<<grid * 2, 256, 0, st>>>(in, n, s, out_min, out_max, out);
  return launched("window_apply_kernel");
}

extern "C" int oai_intensity_window_result(const void* workspace, double* window_host, void* stream) {
  OAI_REQUIRE(workspace && window_host, "intensity_window_result: null pointer");
  const SelectState* s = static_cast<const SelectState*>(workspace);
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  if (int rc = check_cuda(cudaMemcpyAsync(window_host, s->window, 2 * sizeof(double), cudaMemcpyDeviceToHost, st),
                          "intensity_window_result: copy"))
    return rc;
  return check_cuda(cudaStreamSynchronize(st), "intensity_window_result: sync");
}
