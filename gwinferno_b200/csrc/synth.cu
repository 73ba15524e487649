// Synthetic found-injection set of SURVEY.md section 8d, generated ON THE DEVICE (benchmarks and tests; the reference has no
// counterpart: its injections come from files, gwinferno/preprocess/selection.py).  Uniform over the support
//   m1 in [3, 100], q in [3/m1, 1], a1, a2 in [0, 1], cos tilt 1, 2 in [-1, 1], z in [1e-3, 1.9],
// `prior` = the analytic density of that draw.  Counter-based: injection i takes its seven uniforms from Philox4x32-10 blocks
// with counter (i_lo, i_hi, block, 0) and key (seed_lo, seed_hi), so any index range is generated independently -- a rank
// generates exactly its shard, nothing crosses PCIe -- and gwinferno_b200/synthetic.py: make_injections_philox reproduces every
// value bit for bit on the host (the arithmetic below uses explicitly rounded operations: no FMA contraction).
#include <cuda_runtime.h>

#include <cstdint>
#include <string>

#include "dev_structs.h"
#include "philox.h"

namespace gwi {
namespace {

#ifdef GWI_HOST_EMULATION
inline double mul_rn(double a, double b) { return a * b; }
inline double add_rn(double a, double b) { return a + b; }
#else
__device__ inline double mul_rn(double a, double b) { return __dmul_rn(a, b); }
__device__ inline double add_rn(double a, double b) { return __dadd_rn(a, b); }
#endif

struct SynthCols {
  double* c[9];  // mass_1, mass_ratio, mass_2, a_1, a_2, cos_tilt_1, cos_tilt_2, redshift, prior
};

__global__ void __launch_bounds__(256) synth_injections_kernel(SynthCols out, uint64_t seed, int64_t first, int64_t count) {
  const int64_t j = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (j >= count) return;
  const uint64_t i = (uint64_t)(first + j);
  const uint32_t k0 = (uint32_t)seed, k1 = (uint32_t)(seed >> 32);
  double u[8];
  for (uint32_t b = 0; b < 4; ++b) {
    const U4 r = philox4x32_10(U4{(uint32_t)i, (uint32_t)(i >> 32), b, 0u}, k0, k1);
    u[2 * b] = u01(r.x, r.y);
    u[2 * b + 1] = u01(r.z, r.w);
  }
  const double MMIN = 3.0, MMAX = 100.0, ZLO = 1e-3, ZHI = 1.9;
  const double m1 = add_rn(MMIN, mul_rn(MMAX - MMIN, u[0]));
  const double qlo = MMIN / m1;
  const double q = add_rn(qlo, mul_rn(1.0 - qlo, u[1]));
  const double z = add_rn(ZLO, mul_rn(ZHI - ZLO, u[6]));
  out.c[0][j] = m1;
  out.c[1][j] = q;
  out.c[2][j] = mul_rn(m1, q);
  out.c[3][j] = u[2];
  out.c[4][j] = u[3];
  out.c[5][j] = add_rn(-1.0, mul_rn(2.0, u[4]));
  out.c[6][j] = add_rn(-1.0, mul_rn(2.0, u[5]));
  out.c[7][j] = z;
  out.c[8][j] = 1.0 / (MMAX - MMIN) / (1.0 - qlo) / 4.0 / (ZHI - ZLO);  // density of the draw
}

// order-encoded doubles so that integer atomics give min / max
__device__ inline unsigned long long enc(double x) {
  unsigned long long b = (unsigned long long)__double_as_longlong(x);
  return (b >> 63) ? ~b : (b | 0x8000000000000000ull);
}
__global__ void __launch_bounds__(256) minmax_kernel(const double* __restrict__ x, int64_t n, unsigned long long* __restrict__ out) {
  unsigned long long mn = ~0ull, mx = 0ull;
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x) {
    const double v = x[i];
    if (v == v) {
      const unsigned long long e = enc(v);
      mn = e < mn ? e : mn;
      mx = e > mx ? e : mx;
    }
  }
  for (int o = 16; o > 0; o >>= 1) {
    const unsigned long long a = __shfl_xor_sync(0xffffffffu, mn, o), b = __shfl_xor_sync(0xffffffffu, mx, o);
    mn = a < mn ? a : mn;
    mx = b > mx ? b : mx;
  }
  if ((threadIdx.x & 31) == 0) {
    atomicMin(out, mn);
    atomicMax(out + 1, mx);
  }
}

}  // namespace
}  // namespace gwi

using namespace gwi;

extern "C" {

int gwi_synth_injections(int32_t device, uint64_t seed, int64_t first, int64_t count, double* const* columns_dev, void* stream) {
  if (!columns_dev || first < 0 || count < 0) {
    set_error("gwi_synth_injections: bad arguments");
    return GWI_ERR_INVALID;
  }
  SynthCols C{};
  for (int k = 0; k < 9; ++k) {
    if (!columns_dev[k] && count > 0) {
      set_error("gwi_synth_injections: null column pointer");
      return GWI_ERR_INVALID;
    }
    C.c[k] = columns_dev[k];
  }
  if (cudaSetDevice(device) != cudaSuccess) {
    set_error("gwi_synth_injections: bad device ordinal");
    return GWI_ERR_CUDA;
  }
  if (count > 0) GWI_LAUNCH(synth_injections_kernel, dim3((unsigned)((count + 255) / 256)), dim3(256), 0, (cudaStream_t)stream)(C, seed, first, count);
  const cudaError_t e = cudaGetLastError();
  if (e != cudaSuccess) {
    set_error(std::string("gwi_synth_injections: launch failed: ") + cudaGetErrorString(e));
    return GWI_ERR_CUDA;
  }
  return GWI_OK;
}

int gwi_device_minmax(int32_t device, const double* x_dev, int64_t n, double* out_host) {
  if (!out_host || (n > 0 && !x_dev) || n < 0) {
    set_error("gwi_device_minmax: bad arguments");
    return GWI_ERR_INVALID;
  }
  if (cudaSetDevice(device) != cudaSuccess) return GWI_ERR_CUDA;
  unsigned long long h[2] = {~0ull, 0ull}, *d = nullptr;
  if (cudaMalloc((void**)&d, sizeof(h)) != cudaSuccess) return GWI_ERR_ALLOC;
  cudaMemcpy(d, h, sizeof(h), cudaMemcpyHostToDevice);
  if (n > 0) GWI_LAUNCH(minmax_kernel, dim3((unsigned)std::min<int64_t>(1184, (n + 255) / 256)), dim3(256), 0, 0)(x_dev, n, d);
  const cudaError_t e = cudaMemcpy(h, d, sizeof(h), cudaMemcpyDeviceToHost);
  cudaFree(d);
  if (e != cudaSuccess) {
    set_error(std::string("gwi_device_minmax failed: ") + cudaGetErrorString(e));
    return GWI_ERR_CUDA;
  }
  auto dec = [](unsigned long long v) {
    const unsigned long long b = (v >> 63) ? (v & 0x7fffffffffffffffull) : ~v;
    double x;
    memcpy(&x, &b, 8);
    return x;
  };
  out_host[0] = h[0] == ~0ull ? (double)NAN : dec(h[0]);
  out_host[1] = h[1] == 0ull ? (double)NAN : dec(h[1]);
  return GWI_OK;
}

}  // extern "C"
