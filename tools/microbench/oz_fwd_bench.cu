// Timing + digit checksum of the forward direction-grid product of the MagLS recursion (launch_oz_fwd:
// int8 tensor-core GEMM with the fused phase continuation / digit slicing epilogue) on synthetic digits of the
// BASELINE config-2 shape.  Every epilogue variant launch_oz_fwd can take runs in turn: its digits are compared with
// those of the FP64 functor (raw), and it is timed whole and in parts (GemmArgs::dbg).  Then, for six digits, synthetic
// functors of one kind of work each run against the MMAs (interference study).
// usage: oz_fwd_bench [P [sets [reps [T = 4 | 6 [variant: run it alone for about five seconds]]]]]
// build: nvcc -gencode arch=compute_100a,code=sm_100a -O3 -std=c++17 -lineinfo -o tools/microbench/bin/oz_fwd_bench
//        tools/microbench/oz_fwd_bench.cu -lcuda ; run on a B200.
#include <cstdio>
#include <cstdlib>
#include <cmath>
#include <vector>
#include <random>
#include "../../emagls_b200/csrc/ozaki_kernels.cu"

#define CK(x) do { cudaError_t e_ = (x); if (e_ != cudaSuccess) { printf("CUDA error %s at %s:%d\n", cudaGetErrorString(e_), __FILE__, __LINE__); exit(2); } } while (0)

__global__ void unused_fnv_kernel(const uint8_t* p, size_t n, unsigned long long* out) {
  // order-independent checksum: sum of byte * (index hash)
  unsigned long long acc = 0;
  for (size_t i = blockIdx.x * (size_t)blockDim.x + threadIdx.x; i < n; i += (size_t)gridDim.x * blockDim.x)
    acc += (unsigned long long)p[i] * ((i * 0x9E3779B97F4A7C15ull) >> 17 | 1ull);
  atomicAdd(out, acc);
}


// ---- synthetic epilogue functors (interference study): the accumulators are drained as usual, then each epilogue
// thread runs one kind of work only, sized like the real functor (about 1.3 us per 8-column chunk when run alone)
template <int KIND>
struct EpiSynthetic {
  static constexpr bool raw = true;
  int8_t* Tq; long long slice_stride; int Kpad; double* sink; const double* src; int iters;
  struct TileState { int dummy; };
  __device__ __forceinline__ TileState begin_tile(int, int, int, int) const { return TileState{0}; }
  __device__ __forceinline__ void apply(TileState&, int m, int n0, const double (&v)[8], int M, int N) const {
    if (KIND == 0) {            // integer ALU chain
      unsigned x = (unsigned)__double2loint(v[0]) | 1u;
      for (int i = 0; i < iters; ++i) x = x * 1664525u + 1013904223u;
      if (x == 0x12345678u) sink[m] = 1.0;
    } else if (KIND == 1) {     // FP64 chain (4 independent)
      double a = v[0], b = v[1], c = v[2], d = v[3];
      for (int i = 0; i < iters; ++i) { a = fma(a, 1.0000001, 1e-9); b = fma(b, 0.9999999, 1e-9); c = fma(c, 1.0000002, 1e-9); d = fma(d, 0.9999998, 1e-9); }
      if (a + b + c + d == 12345.678) sink[m] = a;
    } else if (KIND == 2) {     // byte stores like the digit stores: 8 columns x 6 planes x 2 (re / im)
      int8_t* p = Tq + (long long)n0 * Kpad + m;
      const int q = __double2loint(v[0]);
#pragma unroll
      for (int c = 0; c < 8; ++c)
#pragma unroll
        for (int s_ = 0; s_ < 6; ++s_) p[(long long)s_ * slice_stride + (long long)c * Kpad] = (int8_t)(q + c + s_);
    } else {                    // dependent global loads (L2 hits)
      const double* p = src + (m & 1023);
      double acc = 0.0;
      for (int i = 0; i < iters; ++i) acc += p[(long long)((i * 977 + n0) & 4095) * 1024];
      if (acc == 12345.678) sink[m] = acc;
    }
  }
};

int main(int argc, char** argv) {
  const int P = argc > 1 ? atoi(argv[1]) : 3600, sets = argc > 2 ? atoi(argv[2]) : 1, reps = argc > 3 ? atoi(argv[3]) : 20;
  const int long_mode = argc > 5 ? atoi(argv[5]) : -1;   // >= 0: run this variant for about five seconds (clock sampling)
  const int T = argc > 4 ? atoi(argv[4]) : 6;
  if (T != 4 && T != 6) { printf("T=%d: the forward product takes 4 or 6 digits\n", T); return 1; }
  const int D = 2702, S = 400, K = 8;
  const int rows = 4 * P * sets, KpS = emagls::oz_pad32(S), KpD = emagls::oz_pad32(D);
  std::mt19937_64 rng(7);
  std::normal_distribution<double> nd(0.0, 1.0);
  std::vector<double> hY((size_t)D * S), hC((size_t)rows * S), hAbs((size_t)sets * 2 * K * D);
  for (auto& x : hY) x = nd(rng);
  for (size_t i = 0; i < hC.size(); ++i) hC[i] = nd(rng) * std::pow(2.0, (double)((i / S) % 9) - 4.0);
  for (auto& x : hAbs) x = std::fabs(nd(rng)) + 0.01;
  double *dY, *dC, *dAbs, *sY, *sC, *sT, *up, *sc;
  int8_t *qY, *qC, *qT;
  CK(cudaMalloc(&dY, hY.size() * 8)); CK(cudaMalloc(&dC, hC.size() * 8)); CK(cudaMalloc(&dAbs, hAbs.size() * 8));
  CK(cudaMalloc(&sY, D * 8)); CK(cudaMalloc(&sC, (size_t)rows * 8)); CK(cudaMalloc(&sT, (size_t)rows * 8));
  CK(cudaMalloc(&up, (size_t)sets * 2 * K * 8)); CK(cudaMalloc(&sc, (size_t)sets * 2 * K * 8));
  CK(cudaMalloc(&qY, (size_t)T * D * KpS)); CK(cudaMalloc(&qC, (size_t)T * rows * KpS)); CK(cudaMalloc(&qT, (size_t)T * rows * KpD));
  CK(cudaMemcpy(dY, hY.data(), hY.size() * 8, cudaMemcpyHostToDevice));
  CK(cudaMemcpy(dC, hC.data(), hC.size() * 8, cudaMemcpyHostToDevice));
  CK(cudaMemcpy(dAbs, hAbs.data(), hAbs.size() * 8, cudaMemcpyHostToDevice));
  CK(emagls::launch_slice_rows(0, dY, S, 1, D, S, KpS, T, qY, sY));
  CK(emagls::launch_slice_rows(0, dC, S, 1, rows, S, KpS, T, qC, sC));
  CK(emagls::launch_row_scale(0, dAbs, (long long)sets * 2 * K, D, up, sc));
  CK(cudaMemset(qT, 0, (size_t)T * rows * KpD));
  const int kb = 3;
  emagls::OzFwdArgs fa{qY, sY, D, KpS, qC, sC, rows, T, qT, KpD, sT, dAbs + (size_t)kb * D, 2LL * K * D, (long long)K * D,
                       up + kb, sc + kb, K, P, 0};
  using namespace emagls;
  // the forward epilogues the library launches: raw (the only one for four digits; for six digits the reference of
  // EMAGLS_OZ_FWD=raw), and for six digits the integer functor on 128 x 64 tiles and on 128 x 80 tiles with 20 warps
  auto run = [&](int mode) -> cudaError_t {
    if (T == 4) return oz_fwd_t<4, EpiPhaseSliceRaw<4>>(0, fa);
    if (mode == 0) return oz_fwd_t<6, EpiPhaseSliceRaw<6>>(0, fa);
    if (mode == 1) return oz_fwd_t<6, EpiPhaseSliceFix<6>>(0, fa);
    return oz_fwd_t<6, EpiPhaseSliceFix<6>, oz::TileCfg<80, 2, 20>>(0, fa);
  };
  const char* names[3] = {"raw", "fix", "fix80e20"};
  const int n_modes = T == 6 ? 3 : 1;
  if (long_mode >= n_modes) { printf("variant %d: not run for T=%d\n", long_mode, T); return 1; }
  std::vector<int8_t> fixref;
  const size_t nq = (size_t)T * rows * KpD;
  std::vector<int8_t> ref(nq), got(nq);
  std::vector<double> sref(rows), sgot(rows);
  cudaEvent_t e0, e1;
  CK(cudaEventCreate(&e0)); CK(cudaEventCreate(&e1));
  if (long_mode >= 0) {
    for (int i = 0; i < 12000; ++i) CK(run(long_mode));
    CK(cudaDeviceSynchronize());
    CK(cudaEventRecord(e0));
    for (int i = 0; i < 2000; ++i) CK(run(long_mode));
    CK(cudaEventRecord(e1));
    CK(cudaDeviceSynchronize());
    float msl = 0;
    CK(cudaEventElapsedTime(&msl, e0, e1));
    printf("long run %s: %.4f ms per launch after 12000 launches\n", names[long_mode], msl / 2000);
    return 0;
  }
  for (int mode = 0; mode < n_modes; ++mode) {
    CK(cudaMemset(qT, 0, nq));
    CK(cudaMemset(sT, 0, (size_t)rows * 8));
    CK(run(mode));
    CK(cudaDeviceSynchronize());
    CK(cudaMemcpy(got.data(), qT, nq, cudaMemcpyDeviceToHost));
    CK(cudaMemcpy(sgot.data(), sT, (size_t)rows * 8, cudaMemcpyDeviceToHost));
    size_t bad = 0, bad_s = 0, shown = 0;
    double maxdiff = 0.0;
    if (mode == 1) fixref = got;
    if (mode > 1) {                                  // every variant of the integer functor writes the same bytes
      size_t nb = 0;
      for (size_t i = 0; i < nq; ++i) nb += (got[i] != fixref[i]);
      printf("   %-9s vs fix: %zu of %zu bytes differ\n", names[mode], nb, nq);
    }
    if (mode == 0) { ref = got; sref = sgot; }   // the raw functor: the bytes of oz::slice_digits
    else {
      for (int r = 0; r < rows; ++r) {
        bad_s += (sgot[r] != sref[r]);
        for (int m = 0; m < KpD; ++m) {
          double va = 0, vb = 0; bool neq = false;
          for (int s = 0; s < T; ++s) {
            const size_t i = ((size_t)s * rows + r) * KpD + m;
            va += ref[i] * std::pow(256.0, -s); vb += got[i] * std::pow(256.0, -s);
            neq |= ref[i] != got[i];
          }
          if (neq) {
            ++bad; maxdiff = std::max(maxdiff, std::fabs(va - vb));
            if (shown < 2) { printf("   mismatch row %d col %d: ref %.17g got %.17g\n", r, m, va, vb); ++shown; }
          }
        }
      }
    }
    for (int dbg : {1, 4}) {   // decomposition: 1 no epilogue, 2 no MMAs, 3 operand ring only, 4 drain only, 6 drain only without MMAs
      oz_fwd_debug = dbg;
      CK(run(mode));
      CK(cudaEventRecord(e0));
      for (int i = 0; i < reps; ++i) CK(run(mode));
      CK(cudaEventRecord(e1));
      CK(cudaDeviceSynchronize());
      float msd = 0;
      CK(cudaEventElapsedTime(&msd, e0, e1));
      printf("   %-9s dbg=%d: %.4f ms\n", names[mode], dbg, msd / reps);
    }
    oz_fwd_debug = 0;
    for (int i = 0; i < 3; ++i) CK(run(mode));
    CK(cudaEventRecord(e0));
    for (int i = 0; i < reps; ++i) CK(run(mode));
    CK(cudaEventRecord(e1));
    CK(cudaDeviceSynchronize());
    float ms = 0;
    CK(cudaEventElapsedTime(&ms, e0, e1));
    const double ops = 2.0 * D * (double)rows * KpS * (T * (T + 1) / 2);
    printf("oz_fwd %-9s P=%d sets=%d T=%d: %.4f ms per launch, %.0f int8 TOP/s; vs raw: %zu of %zu values differ (max %.3g in units of the leading digit), %zu scales differ\n",
           names[mode], P, sets, T, ms / reps, ops / (ms / reps * 1e-3) / 1e12, bad, (size_t)rows * KpD, maxdiff, bad_s);
  }

  {
    double *sink, *srcb;
    CK(cudaMalloc(&sink, 1 << 20)); CK(cudaMalloc(&srcb, (size_t)4096 * 1024 * 8 + 8192)); CK(cudaMemset(srcb, 0, (size_t)4096 * 1024 * 8 + 8192));
    CUtensorMap tmA, tmB;
    if (!oz::make_operand_map(&tmA, qY, D, KpS, T, oz::TILE_M) || !oz::make_operand_map(&tmB, qC, rows, KpS, T, oz::TILE_N)) return 3;
    auto run_syn = [&](int kind, int iters, int dbg) -> cudaError_t {
      oz::GemmArgs g{D, rows, KpS, sY, sC, dbg, 0, oz::TILE_N};
      if (kind == 0) return oz::launch_ozaki_gemm_t<6, EpiSynthetic<0>>(0, tmA, tmB, g, EpiSynthetic<0>{qT, (long long)rows * KpD, KpD, sink, srcb, iters}, 148);
      if (kind == 1) return oz::launch_ozaki_gemm_t<6, EpiSynthetic<1>>(0, tmA, tmB, g, EpiSynthetic<1>{qT, (long long)rows * KpD, KpD, sink, srcb, iters}, 148);
      if (kind == 2) return oz::launch_ozaki_gemm_t<6, EpiSynthetic<2>>(0, tmA, tmB, g, EpiSynthetic<2>{qT, (long long)rows * KpD, KpD, sink, srcb, iters}, 148);
      return oz::launch_ozaki_gemm_t<6, EpiSynthetic<3>>(0, tmA, tmB, g, EpiSynthetic<3>{qT, (long long)rows * KpD, KpD, sink, srcb, iters}, 148);
    };
    const char* kn[4] = {"int-alu", "fp64", "byte-stores", "global-loads"};
    const int its[4] = {600, 150, 1, 4};
    if (T == 6)
      for (int kind = 0; kind < 4; ++kind)
        for (int dbg : {0, 2}) {
          CK(run_syn(kind, its[kind], dbg));
          CK(cudaEventRecord(e0));
          for (int i = 0; i < reps; ++i) CK(run_syn(kind, its[kind], dbg));
          CK(cudaEventRecord(e1));
          CK(cudaDeviceSynchronize());
          float msd = 0;
          CK(cudaEventElapsedTime(&msd, e0, e1));
          printf("synthetic functor %-12s %s: %.4f ms\n", kn[kind], dbg == 2 ? "without MMAs" : "with MMAs   ", msd / reps);
        }
  }
  return 0;
}
