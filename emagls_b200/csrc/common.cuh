// Shared device helpers for libemagls_cuda (sm_100a only).
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>
#include <math.h>
#include <map>
#include <mutex>
#include <utility>

namespace emagls {

// ---------------------------------------------------------------- complex (FP64) helpers
struct __align__(16) cplx {
  double x, y;
};
__host__ __device__ __forceinline__ cplx mk(double r, double i) { cplx c; c.x = r; c.y = i; return c; }
__device__ __forceinline__ cplx cadd(cplx a, cplx b) { return mk(a.x + b.x, a.y + b.y); }
__device__ __forceinline__ cplx csub(cplx a, cplx b) { return mk(a.x - b.x, a.y - b.y); }
__device__ __forceinline__ cplx cmul(cplx a, cplx b) {
  return mk(fma(a.x, b.x, -a.y * b.y), fma(a.x, b.y, a.y * b.x));
}
// a * conj(b)
__device__ __forceinline__ cplx cmulc(cplx a, cplx b) {
  return mk(fma(a.x, b.x, a.y * b.y), fma(a.y, b.x, -a.x * b.y));
}
// acc += a * b
__device__ __forceinline__ void cfma(cplx& acc, cplx a, cplx b) {
  acc.x = fma(a.x, b.x, acc.x); acc.x = fma(-a.y, b.y, acc.x);
  acc.y = fma(a.x, b.y, acc.y); acc.y = fma(a.y, b.x, acc.y);
}
// acc += conj(a) * b
__device__ __forceinline__ void cfmac(cplx& acc, cplx a, cplx b) {
  acc.x = fma(a.x, b.x, acc.x); acc.x = fma(a.y, b.y, acc.x);
  acc.y = fma(a.x, b.y, acc.y); acc.y = fma(-a.y, b.x, acc.y);
}
// acc -= a * b
__device__ __forceinline__ void cfms(cplx& acc, cplx a, cplx b) {
  acc.x = fma(-a.x, b.x, acc.x); acc.x = fma(a.y, b.y, acc.x);
  acc.y = fma(-a.x, b.y, acc.y); acc.y = fma(-a.y, b.x, acc.y);
}
__device__ __forceinline__ cplx cconj(cplx a) { return mk(a.x, -a.y); }
__device__ __forceinline__ cplx cscale(cplx a, double s) { return mk(a.x * s, a.y * s); }
__device__ __forceinline__ double cabs2(cplx a) { return fma(a.x, a.x, a.y * a.y); }
__device__ __forceinline__ cplx cdiv(cplx a, cplx b) {  // Smith's algorithm
  if (fabs(b.x) >= fabs(b.y)) {
    double r = b.y / b.x, d = b.x + b.y * r;
    return mk((a.x + a.y * r) / d, (a.y - a.x * r) / d);
  } else {
    double r = b.x / b.y, d = b.x * r + b.y;
    return mk((a.x * r + a.y) / d, (a.y * r - a.x) / d);
  }
}

// getFadeWindow(len) (dependencies/getFadeWindow.m:9-16): half-Hann fade over round(0.15 len) taps
// at both ends, hann(2n) symmetric with zero end points.
__host__ __device__ inline double fade_window(int tp, int len) {
  const int nf = (int)floor(0.15 * (double)len + 0.5);
  if (nf <= 0) return 1.0;
  const double den = (double)(2 * nf - 1);
  if (tp < nf) return 0.5 * (1.0 - cos(2.0 * 3.141592653589793 * (double)tp / den));
  if (tp >= len - nf) {
    const int q = tp - (len - nf) + nf;  // index into hann(2*nf), second half
    return 0.5 * (1.0 - cos(2.0 * 3.141592653589793 * (double)q / den));
  }
  return 1.0;
}

// ---------------------------------------------------------------- warp helpers
__device__ __forceinline__ double shfl_xor_d(double v, int m, unsigned mask = 0xffffffffu) {
  return __shfl_xor_sync(mask, v, m);
}
template <int WIDTH>
__device__ __forceinline__ double group_sum(double v) {  // all-reduce over aligned groups of WIDTH lanes
#pragma unroll
  for (int m = WIDTH / 2; m > 0; m >>= 1) v += __shfl_xor_sync(0xffffffffu, v, m);
  return v;
}
template <int WIDTH>
__device__ __forceinline__ cplx group_sum(cplx v) {
  v.x = group_sum<WIDTH>(v.x);
  v.y = group_sum<WIDTH>(v.y);
  return v;
}

// ---------------------------------------------------------------- FP64 tensor core (DMMA)
// D(8x8) += A(8x4, row) * B(4x8, col).  Lane l holds A[l/4][l%4], B[l%4][l/4],
// C[l/4][2*(l%4)+{0,1}].  SASS: DMMA.8x8x4 (the only native FP64 MMA shape on sm_100a).
__device__ __forceinline__ void dmma884(double& c0, double& c1, double a, double b) {
  asm volatile("mma.sync.aligned.m8n8k4.row.col.f64.f64.f64.f64 {%0,%1}, {%2}, {%3}, {%0,%1};\n"
               : "+d"(c0), "+d"(c1)
               : "d"(a), "d"(b));
}

// ---------------------------------------------------------------- cp.async (LDGSTS)
__device__ __forceinline__ void cp_async16(void* smem, const void* gmem, bool pred) {
  unsigned s = (unsigned)__cvta_generic_to_shared(smem);
  int sz = pred ? 16 : 0;  // src-size 0 => zero fill
  asm volatile("cp.async.cg.shared.global [%0], [%1], 16, %2;\n" ::"r"(s), "l"(gmem), "r"(sz));
}
__device__ __forceinline__ void cp_async8(void* smem, const void* gmem, bool pred) {
  unsigned s = (unsigned)__cvta_generic_to_shared(smem);
  int sz = pred ? 8 : 0;
  asm volatile("cp.async.ca.shared.global [%0], [%1], 8, %2;\n" ::"r"(s), "l"(gmem), "r"(sz));
}
__device__ __forceinline__ void cp_async_commit() { asm volatile("cp.async.commit_group;\n" ::); }
template <int N>
__device__ __forceinline__ void cp_async_wait() { asm volatile("cp.async.wait_group %0;\n" ::"n"(N)); }

// ---------------------------------------------------------------- host: per-device launch state
// Handles on several devices may launch from several host threads at once (include/emagls_cuda.h), so what the
// launchers remember is kept per device, behind one lock.  The statics of these inline functions are shared by all
// translation units of the library.
inline std::mutex& launch_state_mutex() {
  static std::mutex m;
  return m;
}

// Lets `kernel` launch with `bytes` of dynamic shared memory on the current device.  The attribute belongs to one
// device; it is set when `bytes` exceeds the largest value set so far for this (device, kernel).  Up to 48 KB needs
// no opt-in.
inline cudaError_t allow_dynamic_smem(const void* kernel, size_t bytes) {
  if (bytes <= 48 * 1024) return cudaSuccess;
  int dev = 0;
  cudaError_t e = cudaGetDevice(&dev);
  if (e != cudaSuccess) return e;
  static std::map<std::pair<int, const void*>, size_t> set_to;
  std::lock_guard<std::mutex> lock(launch_state_mutex());
  size_t& cur = set_to[{dev, kernel}];
  if (bytes <= cur) return cudaSuccess;
  e = cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)bytes);
  if (e == cudaSuccess) cur = bytes;
  return e;
}
template <class... Args>
inline cudaError_t allow_dynamic_smem(void (*kernel)(Args...), size_t bytes) {
  return allow_dynamic_smem(reinterpret_cast<const void*>(kernel), bytes);
}

// Number of SMs of the current device.
inline int sm_count() {
  int dev = 0;
  cudaGetDevice(&dev);
  static std::map<int, int> count;
  std::lock_guard<std::mutex> lock(launch_state_mutex());
  int& n = count[dev];
  if (!n) cudaDeviceGetAttribute(&n, cudaDevAttrMultiProcessorCount, dev);
  return n;
}

}  // namespace emagls
