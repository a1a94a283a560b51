// Stand-alone check + timing of the int8-sliced FP64 GEMM (emagls_b200/csrc/ozaki.cuh) against a plain
// FP64 reference kernel.  build: nvcc -gencode arch=compute_100a,code=sm_100a -O3 -std=c++17 -lineinfo
//   -o tools/microbench/bin/ozaki_test tools/microbench/ozaki_test.cu ; run on a B200.
#include <cstdio>
#include <cstdlib>
#include <cmath>
#include <vector>
#include <random>
#include "../../emagls_b200/csrc/ozaki.cuh"

using namespace emagls::oz;

#define CK(x) do { cudaError_t e_ = (x); if (e_ != cudaSuccess) { printf("CUDA error %s at %s:%d\n", cudaGetErrorString(e_), __FILE__, __LINE__); exit(2); } } while (0)

__global__ void ref_gemm(const double* A, const double* B, int M, int N, int K, double* C, double* nrm) {
  int n = blockIdx.x * blockDim.x + threadIdx.x, m = blockIdx.y;
  if (n >= N) return;
  double acc = 0.0, na = 0.0, nb = 0.0;
  for (int k = 0; k < K; ++k) {
    double a = A[(size_t)m * K + k], b = B[(size_t)n * K + k];
    acc = fma(a, b, acc); na = fma(a, a, na); nb = fma(b, b, nb);
  }
  C[(size_t)m * N + n] = acc;
  nrm[(size_t)m * N + n] = sqrt(na * nb);
}

template <class Cfg>
int run_cfg(int M, int N, int K, int T, int reps, int grade, int dbg) {
  const int Kpad = (K + 31) & ~31;
  std::mt19937_64 rng(1234 + M + N + K);
  std::normal_distribution<double> nd(0.0, 1.0);
  std::vector<double> hA((size_t)M * K), hB((size_t)N * K);
  for (size_t i = 0; i < hA.size(); ++i) hA[i] = nd(rng);
  for (size_t i = 0; i < hB.size(); ++i) {
    double g = grade ? std::pow(10.0, -(double)grade * (double)(i % K) / K) : 1.0;  // graded along k
    hB[i] = nd(rng) * g * std::pow(2.0, (double)((i / K) % 7) - 3.0);
  }
  double *dA, *dB, *dC, *dR, *dNrm, *sA, *sB;
  int8_t *qA, *qB;
  CK(cudaMalloc(&dA, hA.size() * 8)); CK(cudaMalloc(&dB, hB.size() * 8));
  CK(cudaMalloc(&dC, (size_t)M * N * 8)); CK(cudaMalloc(&dR, (size_t)M * N * 8)); CK(cudaMalloc(&dNrm, (size_t)M * N * 8));
  CK(cudaMalloc(&sA, (size_t)M * 8)); CK(cudaMalloc(&sB, (size_t)N * 8));
  CK(cudaMalloc(&qA, (size_t)T * M * Kpad)); CK(cudaMalloc(&qB, (size_t)T * N * Kpad));
  CK(cudaMemcpy(dA, hA.data(), hA.size() * 8, cudaMemcpyHostToDevice));
  CK(cudaMemcpy(dB, hB.data(), hB.size() * 8, cudaMemcpyHostToDevice));
  CK(cudaMemset(dC, 0xff, (size_t)M * N * 8));
  auto slice = [&](const double* d, int R, int8_t* q, double* sc) {
    if (T == 4) slice_rows_kernel<4><<<(R + 7) / 8, 256>>>(d, K, 1, R, K, Kpad, q, sc);
    else slice_rows_kernel<6><<<(R + 7) / 8, 256>>>(d, K, 1, R, K, Kpad, q, sc);
  };
  slice(dA, M, qA, sA);
  slice(dB, N, qB, sB);
  CK(cudaGetLastError());
  ref_gemm<<<dim3((N + 127) / 128, M), 128>>>(dA, dB, M, N, K, dR, dNrm);
  CK(cudaGetLastError());
  CK(cudaDeviceSynchronize());
  int sms = 0;
  CK(cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, 0));
  EpiStoreF64 epi{dC, N};
  CK((launch_ozaki_gemm<EpiStoreF64, Cfg>(0, qA, sA, qB, sB, M, N, Kpad, T, epi, sms)));
  cudaError_t e = cudaDeviceSynchronize();
  if (e != cudaSuccess) { printf("M=%d N=%d K=%d T=%d: kernel failed: %s\n", M, N, K, T, cudaGetErrorString(e)); return 1; }
  std::vector<double> hC((size_t)M * N), hR((size_t)M * N), hN((size_t)M * N);
  CK(cudaMemcpy(hC.data(), dC, hC.size() * 8, cudaMemcpyDeviceToHost));
  CK(cudaMemcpy(hR.data(), dR, hR.size() * 8, cudaMemcpyDeviceToHost));
  CK(cudaMemcpy(hN.data(), dNrm, hN.size() * 8, cudaMemcpyDeviceToHost));
  double emax = 0.0, erel = 0.0; size_t bad = 0, where = 0;
  for (size_t i = 0; i < hC.size(); ++i) {
    double d = std::fabs(hC[i] - hR[i]);
    if (!(d == d)) { ++bad; continue; }
    double en = d / (hN[i] + 1e-300);
    if (en > emax) { emax = en; where = i; }
    if (std::fabs(hR[i]) > 0.1 * hN[i] / std::sqrt((double)K)) erel = std::max(erel, d / std::fabs(hR[i]));
  }
  float ms = 0.f;
  if (reps > 0) {
    cudaEvent_t a, b; cudaEventCreate(&a); cudaEventCreate(&b);
    for (int i = 0; i < 2; ++i) launch_ozaki_gemm<EpiStoreF64, Cfg>(0, qA, sA, qB, sB, M, N, Kpad, T, epi, sms, dbg);
    cudaEventRecord(a);
    for (int i = 0; i < reps; ++i) launch_ozaki_gemm<EpiStoreF64, Cfg>(0, qA, sA, qB, sB, M, N, Kpad, T, epi, sms, dbg);
    cudaEventRecord(b);
    CK(cudaDeviceSynchronize());
    cudaEventElapsedTime(&ms, a, b); ms /= reps;
  }
  const double flop = 2.0 * M * N * K;
  const double iops = 2.0 * M * (double)((N + Cfg::NT - 1) / Cfg::NT * Cfg::NT) * Kpad * (T * (T + 1) / 2);
  printf("NT=%d M=%5d N=%5d K=%4d T=%d grade=%d: err/(|a||b|) max %.2e (at m=%zu n=%zu: got %.15g want %.15g)  rel(typical) %.2e  nan %zu",
         Cfg::NT, M, N, K, T, grade, emax, where / N, where % N, hC[where], hR[where], erel, bad);
  if (reps > 0) printf("  dbg=%d %.3f ms  %.1f TFLOP/s fp64-equivalent  %.0f int8 TOP/s", dbg, ms, flop / ms / 1e9, iops / ms / 1e9);
  printf("\n");
  fflush(stdout);
  cudaFree(dA); cudaFree(dB); cudaFree(dC); cudaFree(dR); cudaFree(dNrm); cudaFree(sA); cudaFree(sB); cudaFree(qA); cudaFree(qB);
  return (bad == 0 && emax < (T >= 6 ? 1e-9 : 1e-6)) ? 0 : 1;
}

int run(int M, int N, int K, int T, int reps, int grade, int dbg = 0) { return run_cfg<TileDefault>(M, N, K, T, reps, grade, dbg); }

int main(int argc, char** argv) {
  int fails = 0;
  if (argc >= 5) {
    fails += run(atoi(argv[1]), atoi(argv[2]), atoi(argv[3]), atoi(argv[4]), argc > 5 ? atoi(argv[5]) : 5, argc > 6 ? atoi(argv[6]) : 0);
    return fails;
  }
  fails += run(128, 64, 64, 6, 0, 0);
  fails += run(300, 200, 400, 6, 0, 4);
  fails += run(1000, 400, 2702, 4, 0, 0);
  for (int dbg = 0; dbg < 4; ++dbg) {
    fails += run(2702, 14400, 400, 6, 10, 0, dbg);
    fails += run(14400, 400, 2702, 6, 10, 0, dbg);
  }
  fails += run_cfg<TileWide>(300, 200, 400, 6, 0, 4, 0);
  fails += run_cfg<TileWide>(1000, 400, 2702, 6, 0, 0, 0);
  for (int dbg = 0; dbg < 4; ++dbg) fails += run_cfg<TileWide>(14400, 400, 2702, 6, 10, 0, dbg);
  fails += run_cfg<TileWide>(2702, 14400, 400, 6, 10, 0, 0);
  fails += run_cfg<TileCfg<80, 2, 20>>(1000, 400, 2702, 6, 0, 0, 0);     // 20 epilogue warps: two chunks per warp
  fails += run_cfg<TileCfg<80, 2, 20>>(14400, 400, 2702, 6, 10, 0, 0);
  fails += run_cfg<TileCfg<80, 2, 20>>(1800, 400, 2702, 6, 10, 0, 0);
  fails += run_cfg<TileWide>(1800, 400, 2702, 6, 10, 0, 0);
  fails += run_cfg<TileCfg<48, 3>>(1800, 400, 2702, 6, 10, 0, 0);
  fails += run_cfg<TileCfg<48, 3, 12>>(1800, 400, 2702, 6, 10, 0, 0);    // six chunks: 12 warps take two each
  fails += run(2702, 14400, 400, 4, 10, 0);
  fails += run_cfg<TileWide>(14400, 400, 2702, 4, 10, 0, 0);
  printf("%s (%d failing)\n", fails ? "FAIL" : "PASS", fails);
  return fails != 0;
}
