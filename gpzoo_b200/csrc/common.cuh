// Shared device/host helpers for the gpzoo_b200 CUDA kernels (sm_100a only).
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>

#define GPZ_OK 0
#define GPZ_ERR_BADARG (-1000)
#define GPZ_ERR_UNSUPPORTED (-1001)

// after every kernel launch: count it (gpz_launch_count) and surface launch errors
extern "C" void gpz_count_launch_(void);
#define GPZ_CHECK_LAUNCH()                                  \
  do {                                                      \
    gpz_count_launch_();                                    \
    cudaError_t e__ = cudaGetLastError();                   \
    if (e__ != cudaSuccess) return -(int)e__;               \
  } while (0)

#define GPZ_CUDA(call)                                      \
  do {                                                      \
    cudaError_t e__ = (call);                               \
    if (e__ != cudaSuccess) return -(int)e__;               \
  } while (0)

namespace gpz {

__host__ __device__ inline int64_t cdiv(int64_t a, int64_t b) { return (a + b - 1) / b; }

// the split-TF32 lo plane of x: x - tf32(x), tf32(x) being x with the 13 low mantissa bits cleared
__device__ __forceinline__ float tf32_lo_part(float v) { return v - __uint_as_float(__float_as_uint(v) & 0xFFFFE000u); }

template <typename T> struct Num;
template <> struct Num<float> {
  __device__ static float exp(float x) { return expf(x); }
  __device__ static float exp2(float x) { return exp2f(x); }
  __device__ static float log(float x) { return logf(x); }
  __device__ static float sqrt(float x) { return sqrtf(x); }
  __device__ static float rsqrt(float x) { return rsqrtf(x); }
  __device__ static float pow(float x, float y) { return powf(x, y); }
  __device__ static float log1p(float x) { return log1pf(x); }
  __device__ static float lgamma(float x) { return lgammaf(x); }
};
template <> struct Num<double> {
  __device__ static double exp(double x) { return ::exp(x); }
  __device__ static double exp2(double x) { return ::exp2(x); }
  __device__ static double log(double x) { return ::log(x); }
  __device__ static double sqrt(double x) { return ::sqrt(x); }
  __device__ static double rsqrt(double x) { return 1.0 / ::sqrt(x); }
  __device__ static double pow(double x, double y) { return ::pow(x, y); }
  __device__ static double log1p(double x) { return ::log1p(x); }
  __device__ static double lgamma(double x) { return ::lgamma(x); }
};

// fast-math variants for the HBM-bound fp32 kernels (MUFU-based, ~2 ulp): used where the value only enters sums whose
// parity tolerance is 1e-4; fp64 keeps the exact functions
#ifdef GPZ_EXACT_EXP
__device__ inline float fast_exp(float x) { return expf(x); }
#else
__device__ inline float fast_exp(float x) { return __expf(x); }
#endif
__device__ inline double fast_exp(double x) { return ::exp(x); }
__device__ inline float fast_log(float x) { return __logf(x); }
__device__ inline double fast_log(double x) { return ::log(x); }
__device__ inline float fast_div(float a, float b) { return __fdividef(a, b); }
__device__ inline double fast_div(double a, double b) { return a / b; }

// softplus with torch's threshold (=20): softplus(x) = x for x > 20   (torch.nn.functional.softplus)
template <typename T> __device__ inline T softplus(T x) {
  return x > T(20) ? x : Num<T>::log1p(Num<T>::exp(x));
}
template <typename T> __device__ inline T sigmoid(T x) { return T(1) / (T(1) + Num<T>::exp(-x)); }
// d softplus / dx with the same threshold rule
template <typename T> __device__ inline T softplus_grad(T x) { return x > T(20) ? T(1) : sigmoid(x); }

// 16-byte vector loads of an FMAX-long shared-memory row (FMAX is a multiple of 4, rows are 16-byte aligned)
template <int FMAX> __device__ __forceinline__ void load_row(const float* p, float (&o)[FMAX]) {
#pragma unroll
  for (int i = 0; i < FMAX / 4; ++i) {
    const float4 v = reinterpret_cast<const float4*>(p)[i];
    o[4 * i] = v.x; o[4 * i + 1] = v.y; o[4 * i + 2] = v.z; o[4 * i + 3] = v.w;
  }
}
template <int FMAX> __device__ __forceinline__ void load_row(const double* p, double (&o)[FMAX]) {
#pragma unroll
  for (int i = 0; i < FMAX / 2; ++i) {
    const double2 v = reinterpret_cast<const double2*>(p)[i];
    o[2 * i] = v.x; o[2 * i + 1] = v.y;
  }
}

template <typename T> __device__ inline T warp_sum(T v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  return v;
}

// Block-wide sum; result valid in thread 0.  `red` must hold >= 32 elements of T.
template <typename T> __device__ inline T block_sum(T v, T* red) {
  const int lane = threadIdx.x & 31, w = threadIdx.x >> 5, nw = (blockDim.x + 31) >> 5;
  v = warp_sum(v);
  __syncthreads();
  if (lane == 0) red[w] = v;
  __syncthreads();
  if (w == 0) {
    v = lane < nw ? red[lane] : T(0);
    v = warp_sum(v);
  }
  return v;
}

}  // namespace gpz
