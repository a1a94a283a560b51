// The two direction-grid contractions of the MagLS recursion on the int8 tensor cores (see ozaki.cuh):
//   forward : y = Y_h c  (D x 4P, contraction over the S simulation harmonics) with the phase
//             continuation t = |H_k| y / |y| (lib/getEMagLs2Filters.m:95-103) fused into the epilogue,
//             which also slices t into the int8 digits the backward product consumes;
//   backward: t^T Y_h (or t^T Q)  (4P x S, contraction over the D directions), FP64 out.
#include <cstdlib>
#include <string>
#include "kernels.h"
#include "ozaki.cuh"
#include "phase_fixed.cuh"

namespace emagls {

namespace {

// Epilogue of the forward product on the unscaled integer results (oz::epi_raw): y / |y| does not depend on a common
// scale, so the row scale of Y_h and the weight of the digit planes are not applied (only the scales of the re and the
// im row of c, which differ); |H_k|, its power-of-two scale and the 256^(T-4) of the digit split are one factor per
// (set, ear, direction), fetched before the accumulators are waited for; the digits come out of the FP64 / integer
// pipes (oz::slice_words) instead of F2I / I2F.  Bitwise the same digits as oz::slice_digits of the scaled phase
// continuation (every factor that moved is a power of two).
template <int T>
struct EpiPhaseSliceRaw {
  static constexpr bool raw = true;
  int8_t* Tq; long long slice_stride; int Kpad;   // [T][rows][Kpad], element (n, m) at n * Kpad + m
  double* sT;                                     // [rows] scale of row n (written by the m == 0 lanes)
  const double* absH; long long abs_set_stride, abs_ear_stride;   // this bin: [set][ear][dir]
  const double* up; const double* sc; int scale_stride;           // 2^(6-e), 2^(e-6) at [(set*2+ear)*scale_stride]
  int orient_per_set; int nyquist;
  const double* sB;                               // [rows] scales of the rows of c (the B operand)
  struct TileState { double mu[2]; int set; };
  __device__ __forceinline__ void load_set(TileState& ts, int set, int m) const {
    constexpr double split = (double)(1 << (8 * (T - 4)));
    ts.set = set;
#pragma unroll
    for (int ear = 0; ear < 2; ++ear)
      ts.mu[ear] = absH[(long long)set * abs_set_stride + (long long)ear * abs_ear_stride + m] *
                   (up[(set * 2 + ear) * scale_stride] * split);
  }
  __device__ __forceinline__ TileState begin_tile(int m, int n, int M, int N) const {
    TileState ts;
    load_set(ts, (min(n, N - 1) >> 2) / orient_per_set, m);   // a chunk past the last column is never applied
    return ts;
  }
  // digit j of a column goes to plane T-1-j (j < 3: bytes of zl; j >= 3: bytes of zh)
  __device__ __forceinline__ void put_digits(int8_t* p, uint32_t zl, uint32_t zh) const {
    p[(T - 1) * slice_stride] = (int8_t)zl;
    p[(T - 2) * slice_stride] = (int8_t)(zl >> 8);
    p[(T - 3) * slice_stride] = (int8_t)(zl >> 16);
    p[(T - 4) * slice_stride] = (int8_t)zh;
    if (T >= 5) p[(T - 5) * slice_stride] = (int8_t)(zh >> 8);
    if (T >= 6) p[(T - 6) * slice_stride] = (int8_t)(zh >> 16);
  }
  // columns n0..n0+7 are the (re, im) pairs of four consecutive (problem, ear) indices j = n / 2 (n0 is a multiple
  // of 8, so the ear is (q >> 1) & 1); the HRTF set of a problem is found with one division per call and then
  // tracked incrementally.
  __device__ __forceinline__ void apply(TileState& ts, int m, int n0, const double (&v)[8], int M, int N) const {
    int8_t* p = Tq + (long long)n0 * Kpad + m;
    const int prob = n0 >> 2;
    int set = prob / orient_per_set;
    int left = (set + 1) * orient_per_set - prob;     // problems left in this set, >= 1
    if (m == 0) {                                     // scale of the output rows (one writer per row)
      int s2 = set, l2 = left;
      for (int q = 0; q < 8 && n0 + q < N; q += 2) {
        const int e = (q >> 1) & 1;
        const double s_ = sc[(s2 * 2 + e) * scale_stride];
        sT[n0 + q] = s_; sT[n0 + q + 1] = s_;
        if (e == 1 && --l2 == 0) { ++s2; l2 = orient_per_set; }
      }
    }
#pragma unroll
    for (int q = 0; q < 8; q += 2) {
      if (n0 + q >= N) break;
      const int e = (q >> 1) & 1;
      if (set != ts.set) load_set(ts, set, m);        // warp-uniform: a tile rarely straddles two HRTF sets
      const double mu = ts.mu[e];
      const double2 sb = *reinterpret_cast<const double2*>(sB + n0 + q);   // warp-uniform, 16-byte aligned
      const double re = v[q] * sb.x, im = v[q + 1] * sb.y;
      const double a2 = fma(re, re, im * im);         // zero only if y == 0
      double tr = mu, ti = 0.0;                       // angle(0) = 0
      if (a2 > 0.0) {
        const double inv = mu * rsqrt(a2);
        tr = re * inv; ti = im * inv;
      }
      if (nyquist) ti = 0.0;
      uint32_t zl, zh;                                // |tr|, |ti| <= 64 * 256^(T-4)
      oz::slice_words<T>(tr, zl, zh);
      put_digits(p + (long long)q * Kpad, zl, zh);
      oz::slice_words<T>(ti, zl, zh);
      put_digits(p + (long long)(q + 1) * Kpad, zl, zh);
      if (e == 1 && --left == 0) { ++set; left = orient_per_set; }   // next pair belongs to the next problem
    }
  }
};
// The same epilogue without FP64 instructions in the functor (phase_fixed.cuh): FP64 work does not overlap with the
// tcgen05 MMAs of the next tile on this part, integer work does.  The drain hands over the exact 64-bit integers
// (int64_values: the kernel instance then contains no FP64 instruction at all), they are normalised by
// count-leading-zeros and shifts, |y|^-1 comes from a 22-bit MUFU seed and one third-order correction in 64-bit
// fixed point, and the digits are those of rn(t 2^24) formed in integer arithmetic.  Against EpiPhaseSliceRaw the last digit may differ by one unit
// (|Z - exact| <= 0.6 instead of <= 0.53; tests/test_phase_fixed.py on the host, tests/test_gpu_ozaki.py on the device).
// Stores: the digit bytes of four columns are packed per plane, transposed across groups of four lanes (two shuffles
// and two byte permutes per word) and leave as 4-byte stores: lane l writes rows l & ~3 .. (l & ~3) + 3 of column
// l & 3: a quarter of the store instructions (and of their address arithmetic) of byte stores.  The whole warp enters
// apply() (lanes past the last row contribute zero bytes, which land in the row padding), so N must be a multiple of 4.
template <int T>
struct EpiPhaseSliceFix {
  static constexpr bool raw = true;
  static constexpr bool all_lanes = true;
  static constexpr bool int64_values = true;      // the drain hands over exact 64-bit integers (no FP64 at all)
  int8_t* Tq; long long slice_stride; int Kpad;   // [T][rows][Kpad], element (n, m) at n * Kpad + m
  double* sT;                                     // [rows] scale of row n (written by the m == 0 lanes)
  const double* absH; long long abs_set_stride, abs_ear_stride;   // this bin: [set][ear][dir]
  const double* up; const double* sc; int scale_stride;           // 2^(6-e), 2^(e-6) at [(set*2+ear)*scale_stride]
  int orient_per_set; int nyquist;
  const double* sB;                               // [rows] scales of the rows of c (the B operand)
  struct TileState { uint64_t mu[2]; int set; };
  __device__ __forceinline__ void load_set(TileState& ts, int set, int m) const {
    ts.set = set;
#pragma unroll
    for (int ear = 0; ear < 2; ++ear)
      ts.mu[ear] = pfx::magnitude_fixed<T>(absH[(long long)set * abs_set_stride + (long long)ear * abs_ear_stride + m],
                                           up[(set * 2 + ear) * scale_stride]);
  }
  // the same out of line: a tile rarely straddles two HRTF sets, and twelve inlined copies of the conversion made the
  // epilogue's straight-line code a third longer (instruction-cache footprint)
  static __device__ __noinline__ uint64_t mu_cold(const double* x, const double* u) { return pfx::magnitude_fixed<T>(*x, *u); }
  __device__ __forceinline__ void load_set_cold(TileState& ts, int set, int m) const {
    ts.set = set;
#pragma unroll
    for (int ear = 0; ear < 2; ++ear)
      ts.mu[ear] = mu_cold(absH + ((long long)set * abs_set_stride + (long long)ear * abs_ear_stride + m),
                           up + (set * 2 + ear) * scale_stride);
  }
  __device__ __forceinline__ TileState begin_tile(int m, int n, int M, int N) const {
    TileState ts;
    load_set(ts, (min(n, N - 1) >> 2) / orient_per_set, m);   // a chunk past the last column is never applied
    return ts;
  }
  // scale of the output rows n0 .. n0+7 (one writer per row: the m == 0 lane)
  __device__ __forceinline__ void put_scales(int n0, int N, int set, int left) const {
    for (int q = 0; q < 8 && n0 + q < N; q += 2) {
      const int e = (q >> 1) & 1;
      const double s_ = sc[(set * 2 + e) * scale_stride];
      sT[n0 + q] = s_; sT[n0 + q + 1] = s_;
      if (e == 1 && --left == 0) { ++set; left = orient_per_set; }
    }
  }
  // digit words (zl, zh) of the (re, im) columns n0 + q, n0 + q + 1
  __device__ __forceinline__ void pair_digits(const TileState& ts, int n0, int q, long long vr, long long vi, uint32_t& rl,
                                              uint32_t& rh, uint32_t& il, uint32_t& ih) const {
    const int4 sb = *reinterpret_cast<const int4*>(sB + n0 + q);   // warp-uniform: two powers of two
    const int dexp = ((sb.y >> 20) & 0x7FF) - ((sb.w >> 20) & 0x7FF);
    int64_t Zr, Zi;
    pfx::phase_fixed_i64(vr, vi, dexp, ts.mu[(q >> 1) & 1], Zr, Zi);
    if (nyquist) Zi = 0;
    pfx::split_words<T>(Zr, rl, rh);
    pfx::split_words<T>(Zi, il, ih);
  }
  __device__ __forceinline__ void apply(TileState& ts, int m, int n0, const long long (&v)[8], int M, int N) const {
    const int prob = n0 >> 2;
    int set = prob / orient_per_set;
    int left = (set + 1) * orient_per_set - prob;     // problems left in this set, >= 1
    if (m == 0) put_scales(n0, N, set, left);
    const int lane = threadIdx.x & 31, g = lane & 3;
    const uint32_t selA = (lane & 2) ? 0x3276u : 0x5410u, selB = (lane & 1) ? 0x3715u : 0x6240u;
    const uint32_t keep = m < M ? 0xFFFFFFFFu : 0u;
    const bool writer = m - g < M;                  // the group's first row exists (then all four lie below Kpad)
    const int mc = min(m, M - 1);
    // this lane's word: column n0 + g (+ 4), rows m - g .. m - g + 3; the plane / column-group offsets are uniform
    int8_t* const pw = Tq + ((long long)(n0 + g) * Kpad + (m - g));
    const long long col4 = 4ll * Kpad;
#pragma unroll
    for (int h = 0; h < 2; ++h) {                   // four columns = both ears of one problem
      if (n0 + 4 * h >= N) break;
      if (set != ts.set) load_set_cold(ts, set, mc);   // warp-uniform: a tile rarely straddles two HRTF sets
      uint32_t zl[4], zh[4];
      pair_digits(ts, n0, 4 * h, v[4 * h], v[4 * h + 1], zl[0], zh[0], zl[1], zh[1]);
      pair_digits(ts, n0, 4 * h + 2, v[4 * h + 2], v[4 * h + 3], zl[2], zh[2], zl[3], zh[3]);
      if (--left == 0) { ++set; left = orient_per_set; }
      uint32_t w[6];                                // w[j]: digit T-1-j of the four columns
      oz::transpose4x3(zl[0], zl[1], zl[2], zl[3], w[0], w[1], w[2]);
      oz::transpose4x3(zh[0], zh[1], zh[2], zh[3], w[3], w[4], w[5]);
#pragma unroll
      for (int j = 0; j < T; ++j) {
        uint32_t x = w[j] & keep;
        x = __byte_perm(x, __shfl_xor_sync(0xffffffffu, x, 2), selA);
        x = __byte_perm(x, __shfl_xor_sync(0xffffffffu, x, 1), selB);
        if (writer) *reinterpret_cast<uint32_t*>(pw + ((long long)(T - 1 - j) * slice_stride + h * col4)) = x;
      }
    }
  }
};

// one warp per row: 2^e > max_d |x(row, d)|  ->  up = 2^(6-e), sc = 2^(e-6)
__global__ void row_scale_kernel(const double* __restrict__ x, long long rows, int D, double* __restrict__ up,
                                 double* __restrict__ sc) {
  const int lane = threadIdx.x & 31;
  const long long r = (long long)blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
  if (r >= rows) return;
  double mx = 0.0;
  for (int d = lane; d < D; d += 32) mx = fmax(mx, fabs(x[r * D + d]));
#pragma unroll
  for (int m = 16; m > 0; m >>= 1) mx = fmax(mx, __shfl_xor_sync(0xffffffffu, mx, m));
  int e = 0;
  if (mx > 0.0 && mx < 1e300) frexp(mx, &e);
  if (lane == 0) { up[r] = scalbn(1.0, 6 - e); sc[r] = scalbn(1.0, e - 6); }
}

int sm_count() {
  static int n = 0;
  if (!n) {
    int dev = 0;
    cudaGetDevice(&dev);
    cudaDeviceGetAttribute(&n, cudaDevAttrMultiProcessorCount, dev);
  }
  return n;
}

}  // namespace

int oz_pad32(int k) { return (k + 31) & ~31; }
bool oz_contraction_fits(int Kpad, int T) { return oz::contraction_fits(Kpad, T); }

cudaError_t launch_slice_rows(cudaStream_t st, const double* src, long long rs, long long cs, int R, int K, int Kpad,
                              int T, int8_t* out, double* scale) {
  const dim3 grid((R + 7) / 8), block(256);
  switch (T) {
    case 4: oz::slice_rows_kernel<4><<<grid, block, 0, st>>>(src, rs, cs, R, K, Kpad, out, scale); break;
    case 6: oz::slice_rows_kernel<6><<<grid, block, 0, st>>>(src, rs, cs, R, K, Kpad, out, scale); break;
    default: return cudaErrorInvalidValue;
  }
  return cudaGetLastError();
}

cudaError_t launch_row_scale(cudaStream_t st, const double* x, long long rows, int D, double* up, double* sc) {
  row_scale_kernel<<<(unsigned)((rows + 7) / 8), 256, 0, st>>>(x, rows, D, up, sc);
  return cudaGetLastError();
}

int oz_fwd_debug = 0;   // GemmArgs::dbg of the forward launches (tools/microbench/oz_fwd_bench.cu)

template <int T, class Epi, class Cfg = oz::TileDefault>
static cudaError_t oz_fwd_t(cudaStream_t st, const OzFwdArgs& a) {
  CUtensorMap tmA, tmB;
  if (!oz::make_operand_map(&tmA, a.YhA_q, a.D, a.KpS, T, oz::TILE_M) ||
      !oz::make_operand_map(&tmB, a.Cv_q, a.rows, a.KpS, T, Cfg::NT))
    return cudaErrorInvalidValue;
  oz::GemmArgs g{a.D, a.rows, a.KpS, a.sYhA, a.sCv, oz_fwd_debug, 0, Cfg::NT};   // m fastest: the 42 MB of Cv digits are the shared operand
  Epi epi{a.Tt_q, (long long)a.rows * a.KpD, a.KpD, a.sT, a.absH, a.abs_set_stride, a.abs_ear_stride,
          a.up, a.sc, a.scale_stride, a.orient_per_set, a.nyquist, a.sCv};
  return oz::launch_ozaki_gemm_t<T, Epi, Cfg>(st, tmA, tmB, g, epi, sm_count());
}

cudaError_t launch_oz_fwd(cudaStream_t st, const OzFwdArgs& a) {
  if (!oz::contraction_fits(a.KpS, a.T)) return cudaErrorInvalidValue;
  // Six digits: the FP64-free functor (EpiPhaseSliceFix: its integer work overlaps with the MMAs of the next tile, FP64
  // work does not; 0.34 against 0.425 ms per launch, profiles/r02_v40_fwd_fix.txt) on 128 x 80 tiles when that takes
  // fewer rounds of tiles.  With four digits the MMAs of a tile are too short to hide the longer integer functor, so
  // the FP64 functor on the raw accumulators stays (0.076 against 0.078 ms).
  // EMAGLS_OZ_FWD=raw runs that FP64 functor for six digits too: the reference the integer functor is tested against
  // (it may differ from it by one unit of the last digit, phase_fixed.cuh).
  static const bool raw = [] {
    const char* e = getenv("EMAGLS_OZ_FWD");
    return e && std::string(e) == "raw";
  }();
  if (a.T == 4) return oz_fwd_t<4, EpiPhaseSliceRaw<4>>(st, a);
  if (a.T != 6) return cudaErrorInvalidValue;
  if (raw) return oz_fwd_t<6, EpiPhaseSliceRaw<6>>(st, a);
  if (a.rows & 3) return cudaErrorInvalidValue;   // the integer functor's 4-byte stores span four rows
  // Contractions over more than 2016 harmonics (simulation order 44 and up) may carry |y| beyond the range of the
  // integer functor's 64-bit drain: the FP64 functor rounds once instead of wrapping.
  if (!oz::drain_i64_fits(a.KpS, a.T)) return oz_fwd_t<6, EpiPhaseSliceRaw<6>>(st, a);
  // 80 columns = ten chunks per lane group: 20 epilogue warps take two each (16 leave 3 + 3 + 2 + 2; 0.321 against
  // 0.334 ms per launch, profiles/r02_v46_cluster.txt)
  using Wide20 = oz::TileCfg<80, 2, 20>;
  const int sms = sm_count();
  const long long m_tiles = (a.D + oz::TILE_M - 1) / oz::TILE_M;
  auto cost = [&](int nt) { return ((m_tiles * ((a.rows + nt - 1) / nt) + sms - 1) / sms) * (long long)(128 + nt); };
  if (cost(Wide20::NT) < cost(oz::TILE_N)) return oz_fwd_t<6, EpiPhaseSliceFix<6>, Wide20>(st, a);
  return oz_fwd_t<6, EpiPhaseSliceFix<6>>(st, a);
}

cudaError_t launch_oz_bwd(cudaStream_t st, const int8_t* Tt_q, const double* sT, int rows, const int8_t* B_q,
                          const double* sB, int S, int KpD, int T, double* tq) {
  // Tile width by shape: a k-step costs (128 + NT) operand bytes per slice (TMA traffic and the shared-memory reads of
  // the MMAs), and the launch takes ceil(tiles / SMs) rounds of tiles.  80 columns for the 3600-orientation batch
  // (S = 400 = 5 x 80: no padded columns, the A operand passes through L2 5 instead of 7 times); 48 columns when that
  // brings an otherwise half-empty grid to one full round (450 orientations per GPU: 135 tiles instead of 75).
  const int sms = sm_count();
  const int m_tiles = (rows + oz::TILE_M - 1) / oz::TILE_M;
  auto cost = [&](int nt) {
    const long long tiles = (long long)m_tiles * ((S + nt - 1) / nt);
    return ((tiles + sms - 1) / sms) * (long long)(128 + nt);
  };
  int nt = 64;
  if (cost(80) <= cost(nt)) nt = 80;
  if (cost(48) < cost(nt)) nt = 48;
  const oz::EpiStoreF64 epi{tq, (long long)S};
  if (nt == 80) return oz::launch_ozaki_gemm<oz::EpiStoreF64, oz::TileWide>(st, Tt_q, sT, B_q, sB, rows, S, KpD, T, epi, sms);
  if (nt == 48) return oz::launch_ozaki_gemm<oz::EpiStoreF64, oz::TileCfg<48, 3>>(st, Tt_q, sT, B_q, sB, rows, S, KpD, T, epi, sms);
  return oz::launch_ozaki_gemm(st, Tt_q, sT, B_q, sB, rows, S, KpD, T, epi, sms);
}

}  // namespace emagls
