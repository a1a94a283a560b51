// FP64 tensor-core GEMM used by every dense contraction of the design path:
//   C[m][n] = epi( sum_k A(m,k) * B(n,k) )
// DMMA.8x8x4 is the only FP64 MMA shape sm_100a executes natively (m16n8k{4,8,16} lower to it), so
// the kernel is built from 8x8x4 tiles: CTA tile BM x BN x 16, 8 warps, multi-stage cp.async
// (LDGSTS) ring.  Two configurations: 128x128 (2x4 warps of 64x32, 4 stages) for the wide
// contractions and 128x80 (4x2 warps of 32x40, 3 stages, 2 CTAs/SM) for N = S = 400 and friends,
// where 128-wide tiles would waste 22 % of the tensor work.  A and B may be K-contiguous ([m][k])
// or K-strided ([k][m]); tiles are staged in their global orientation (padding chosen so both
// fragment patterns are bank-conflict free), so no transposes are materialised in HBM.  The
// cp.async traffic of the next stage is issued between the four k4 steps of the current one, so the
// warps never leave the DMMA stream for a synchronised load phase.  Optional split-K (grid.z):
// every split writes its own partial C (deterministic; the consumer adds the partials).
#pragma once
#include "common.cuh"

namespace emagls {

constexpr int GM_BK = 16, GM_THREADS = 256;
constexpr int GM_LDK = GM_BK + 4;    // [row][k] orientation: row stride 20 doubles

struct GemmOperand {
  const double* p;
  long long ld;      // stride (doubles) of the non-contiguous index
  int kcontig;       // 1: element (row,k) at p[row*ld + k];  0: at p[k*ld + row]
};

struct GemmShape { int M, N, K; };

// ---- epilogues (z = split-K index) -----------------------------------------------------------
struct EpiStore {
  double* C; long long ldc; double alpha; long long split_stride = 0;
  __device__ __forceinline__ void operator()(int m, int n, double v0, double v1, int M, int N, int z) const {
    if (m >= M) return;
    double* q = C + (long long)z * split_stride + (long long)m * ldc + n;
    if (n + 1 < N) {
      if ((((uintptr_t)q) & 15) == 0) { *reinterpret_cast<double2*>(q) = make_double2(alpha * v0, alpha * v1); }
      else { q[0] = alpha * v0; q[1] = alpha * v1; }
    } else if (n < N) q[0] = alpha * v0;
  }
};

// MagLS phase continuation, lib/getEMagLs2Filters.m:95-103: columns (2j, 2j+1) hold (re, im)
// of y = W(k-1,:) * pwGrid for direction m and problem/ear j; the target written back is
// abs(H(k,m)) * exp(1i*angle(y)) (real part only for the Nyquist bin).
struct EpiPhase {
  double* T; long long ldt;
  const double* absH;        // [set][ear][dir] for this bin
  long long abs_set_stride;  // doubles between sets
  long long abs_ear_stride;  // doubles between ears
  int orient_per_set;
  int nyquist;
  __device__ __forceinline__ void operator()(int m, int n, double re, double im, int M, int N, int) const {
    if (m >= M || n >= N) return;
    int j = n >> 1;                 // problem*2 + ear
    int ear = j & 1, prob = j >> 1;
    int set = prob / orient_per_set;
    double mag = absH[(long long)set * abs_set_stride + (long long)ear * abs_ear_stride + m];
    double a2 = fma(re, re, im * im);
    double tr, ti;
    if (a2 > 1e-290 && a2 < 1e290) {
      const double inv = mag * rsqrt(a2);   // |H| / |y|: rsqrt (<= 1 ulp) instead of sqrt + divide
      tr = re * inv; ti = im * inv;
    } else if (a2 > 0.0) {                  // denormal / huge |y|^2: the slow exact route
      const double inv = mag / sqrt(a2);
      tr = re * inv; ti = im * inv;
    } else { tr = mag; ti = 0.0; }          // angle(0) = 0
    if (nyquist) ti = 0.0;
    double* q = T + (long long)m * ldt + n;
    *reinterpret_cast<double2*>(q) = make_double2(tr, ti);  // n even, ldt even, T 16B aligned
  }
};

// ---- tile configuration ----------------------------------------------------------------------
template <int WM_, int WN_, int WARPS_M_, int WARPS_N_, int STAGES_, int MINB_>
struct GemmCfg {
  static constexpr int WM = WM_, WN = WN_, WARPS_M = WARPS_M_, WARPS_N = WARPS_N_, STAGES = STAGES_, MINB = MINB_;
  static constexpr int BM = WARPS_M * WM * 8, BN = WARPS_N * WN * 8;
  static constexpr int LDMA = BM + 4, LDMB = BN + 4;   // [k][row] orientation strides (== 4 mod 16)
  static constexpr int TILE_A = (BM * GM_LDK > GM_BK * LDMA) ? BM * GM_LDK : GM_BK * LDMA;
  static constexpr int TILE_B = (BN * GM_LDK > GM_BK * LDMB) ? BN * GM_LDK : GM_BK * LDMB;
  static constexpr size_t SMEM = (size_t)STAGES * (TILE_A + TILE_B) * sizeof(double);
  static_assert(WARPS_M * WARPS_N * 32 == GM_THREADS, "8 warps");
  static_assert(LDMA % 16 == 4 && LDMB % 16 == 4, "k-strided tiles need a row stride of 4 mod 16 doubles");
};
using GemmWide = GemmCfg<8, 4, 2, 4, 4, 1>;    // 128 x 128, 160 KB, 1 CTA / SM
using GemmNarrow = GemmCfg<4, 5, 4, 2, 3, 2>;  // 128 x 80,   98 KB, 2 CTAs / SM
using GemmTall = GemmCfg<8, 5, 4, 2, 3, 1>;    // 256 x 80,  158 KB, 1 CTA / SM (4x2 warps of 64x40)

// ---- tile loader -----------------------------------------------------------------------------
// Issues the part `part` of `nparts` of the cp.async traffic of a [ROWS x BK] operand tile
// (zero-filled out of range).  LDM: row stride of the [k][row] orientation.  KC: operand is
// K-contiguous; VEC: 16-byte chunks are legal.  Both are compile-time so the main loop of the GEMM is
// straight-line code the scheduler can software-pipeline.
template <int ROWS, int LDM, bool KC, bool VEC>
__device__ __forceinline__ void load_tile_part(double* s, const GemmOperand& op, int row0, int k0, int nrows,
                                               int kend, int tid, int part, int nparts) {
  constexpr int E = VEC ? 2 : 1;                                 // doubles per chunk
  constexpr int TOTAL = ROWS * GM_BK / E;
  constexpr int PER = (TOTAL + GM_THREADS - 1) / GM_THREADS;     // chunks per thread
#pragma unroll
  for (int i = 0; i < PER; ++i) {
    if (i % nparts != part) continue;
    const int c = tid + i * GM_THREADS;
    if (TOTAL % GM_THREADS != 0 && c >= TOTAL) break;
    int r, kk, soff;
    if (KC) { r = c / (GM_BK / E); kk = (c % (GM_BK / E)) * E; soff = r * GM_LDK + kk; }
    else { kk = c / (ROWS / E); r = (c % (ROWS / E)) * E; soff = kk * LDM + r; }
    const int gr = row0 + r, gk = k0 + kk;
    const bool ok = (gr < nrows) && (gk < kend);
    const double* g = KC ? op.p + (long long)(ok ? gr : 0) * op.ld + (ok ? gk : 0)
                         : op.p + (long long)(ok ? gk : 0) * op.ld + (ok ? gr : 0);
    if (VEC) cp_async16(s + soff, g, ok);
    else cp_async8(s + soff, g, ok);
  }
}

template <class Cfg, class Epi, bool AKC, bool BKC, bool VEC>
__global__ void __launch_bounds__(GM_THREADS, Cfg::MINB)
gemm_f64_kernel(GemmOperand A, GemmOperand B, GemmShape sh, int ksplit, Epi epi) {
  extern __shared__ __align__(16) double gsm[];
  constexpr int WM = Cfg::WM, WN = Cfg::WN, STAGES = Cfg::STAGES, NK4 = GM_BK / 4;
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const int wm = warp / Cfg::WARPS_N, wn = warp % Cfg::WARPS_N;
  const int m0 = blockIdx.y * Cfg::BM, n0 = blockIdx.x * Cfg::BN;
  // split-K: this CTA contracts k in [kbeg, kend)
  const int kbeg = blockIdx.z * ksplit;
  const int kend = min(sh.K, kbeg + ksplit);
  const int ktiles = (kend - kbeg + GM_BK - 1) / GM_BK;

  double acc[WM][WN][2];
#pragma unroll
  for (int i = 0; i < WM; ++i)
#pragma unroll
    for (int j = 0; j < WN; ++j) { acc[i][j][0] = 0.0; acc[i][j][1] = 0.0; }

  auto stageA = [&](int s) { return gsm + (size_t)s * (Cfg::TILE_A + Cfg::TILE_B); };
  auto stageB = [&](int s) { return gsm + (size_t)s * (Cfg::TILE_A + Cfg::TILE_B) + Cfg::TILE_A; };

#pragma unroll
  for (int s = 0; s < STAGES - 1; ++s) {
    if (s < ktiles) {
      load_tile_part<Cfg::BM, Cfg::LDMA, AKC, VEC>(stageA(s), A, m0, kbeg + s * GM_BK, sh.M, kend, tid, 0, 1);
      load_tile_part<Cfg::BN, Cfg::LDMB, BKC, VEC>(stageB(s), B, n0, kbeg + s * GM_BK, sh.N, kend, tid, 0, 1);
    }
    cp_async_commit();
  }

  // fragment addresses of this lane (doubles): element (row, kk) of the staged tiles
  const int lr = lane >> 2, lk = lane & 3;
  const int a_off = AKC ? (wm * (WM * 8) + lr) * GM_LDK + lk : lk * Cfg::LDMA + wm * (WM * 8) + lr;
  const int b_off = BKC ? (wn * (WN * 8) + lr) * GM_LDK + lk : lk * Cfg::LDMB + wn * (WN * 8) + lr;
  constexpr int a_row = AKC ? 8 * GM_LDK : 8, a_k4 = AKC ? 4 : 4 * Cfg::LDMA;
  constexpr int b_row = BKC ? 8 * GM_LDK : 8, b_k4 = BKC ? 4 : 4 * Cfg::LDMB;

  for (int kt = 0; kt < ktiles; ++kt) {
    cp_async_wait<STAGES - 2>();
    __syncthreads();
    // tile kt + STAGES - 1 goes into the slot freed by iteration kt - 1; its cp.async traffic is
    // spread over the four k4 steps below
    const int nk = kt + STAGES - 1;
    const bool pre = nk < ktiles;
    double* nA = stageA(nk % STAGES);
    double* nB = stageB(nk % STAGES);
    const double* As = stageA(kt % STAGES) + a_off;
    const double* Bs = stageB(kt % STAGES) + b_off;
    double a[2][WM], b[2][WN];
#pragma unroll
    for (int i = 0; i < WM; ++i) a[0][i] = As[i * a_row];
#pragma unroll
    for (int j = 0; j < WN; ++j) b[0][j] = Bs[j * b_row];
#pragma unroll
    for (int k4 = 0; k4 < NK4; ++k4) {
      const int cur = k4 & 1, nxt = cur ^ 1;
      if (k4 + 1 < NK4) {   // fragments of the next k4 step are in flight while this one multiplies
#pragma unroll
        for (int i = 0; i < WM; ++i) a[nxt][i] = As[(k4 + 1) * a_k4 + i * a_row];
#pragma unroll
        for (int j = 0; j < WN; ++j) b[nxt][j] = Bs[(k4 + 1) * b_k4 + j * b_row];
      }
      if (pre) {
        load_tile_part<Cfg::BM, Cfg::LDMA, AKC, VEC>(nA, A, m0, kbeg + nk * GM_BK, sh.M, kend, tid, k4, NK4);
        load_tile_part<Cfg::BN, Cfg::LDMB, BKC, VEC>(nB, B, n0, kbeg + nk * GM_BK, sh.N, kend, tid, k4, NK4);
      }
#pragma unroll
      for (int i = 0; i < WM; ++i)
#pragma unroll
        for (int j = 0; j < WN; ++j) dmma884(acc[i][j][0], acc[i][j][1], a[cur][i], b[cur][j]);
    }
    cp_async_commit();
  }
  cp_async_wait<0>();

#pragma unroll
  for (int i = 0; i < WM; ++i)
#pragma unroll
    for (int j = 0; j < WN; ++j) {
      int m = m0 + wm * (WM * 8) + i * 8 + lr;
      int n = n0 + wn * (WN * 8) + j * 8 + 2 * lk;
      epi(m, n, acc[i][j][0], acc[i][j][1], sh.M, sh.N, (int)blockIdx.z);
    }
}

// vec16 is legal when the contiguous extent, the stride and the base pointer are all even/aligned
inline int gemm_vec_ok(const GemmOperand& op, int rows, int K) {
  bool aligned = (((uintptr_t)op.p) & 15) == 0 && (op.ld % 2 == 0);
  int contig_extent = op.kcontig ? K : rows;
  return aligned && (contig_extent % 2 == 0);
}

// Number of K splits that fills the 148 SMs best for a grid of `tiles` CTAs (1 = no split).
inline int gemm_pick_splits(int tiles, int K, int ctas_per_sm, int max_splits) {
  const int slots = 148 * ctas_per_sm;
  int best = 1; double best_eff = 0.0;
  for (int s = 1; s <= max_splits; ++s) {
    if (s > 1 && K / s < 256) break;
    const long long t = (long long)tiles * s;
    const double eff = (double)t / (double)(((t + slots - 1) / slots) * slots);
    if (eff > best_eff + 0.05) { best_eff = eff; best = s; }
  }
  return best;
}

template <class Cfg, class Epi, bool AKC, bool BKC, bool VEC>
inline cudaError_t launch_gemm_inst(cudaStream_t st, GemmOperand A, GemmOperand B, GemmShape sh, Epi epi, dim3 grid,
                                    int ksplit) {
  auto kern = gemm_f64_kernel<Cfg, Epi, AKC, BKC, VEC>;
  const cudaError_t e = allow_dynamic_smem(kern, Cfg::SMEM);
  if (e != cudaSuccess) return e;
  kern<<<grid, GM_THREADS, Cfg::SMEM, st>>>(A, B, sh, ksplit, epi);
  return cudaGetLastError();
}

template <class Cfg, class Epi>
inline cudaError_t launch_gemm_cfg(cudaStream_t st, GemmOperand A, GemmOperand B, GemmShape sh, Epi epi, int splits) {
  if (splits < 1) splits = 1;
  int ksplit = (sh.K + splits - 1) / splits;
  ksplit = (ksplit + GM_BK - 1) / GM_BK * GM_BK;      // splits start on a k-tile (keeps 16-byte chunks aligned)
  splits = (sh.K + ksplit - 1) / ksplit;
  dim3 grid((sh.N + Cfg::BN - 1) / Cfg::BN, (sh.M + Cfg::BM - 1) / Cfg::BM, splits);
  const bool vec = gemm_vec_ok(A, sh.M, sh.K) && gemm_vec_ok(B, sh.N, sh.K);
  const int key = (A.kcontig ? 4 : 0) | (B.kcontig ? 2 : 0) | (vec ? 1 : 0);
  switch (key) {
    case 7: return launch_gemm_inst<Cfg, Epi, true, true, true>(st, A, B, sh, epi, grid, ksplit);
    case 6: return launch_gemm_inst<Cfg, Epi, true, true, false>(st, A, B, sh, epi, grid, ksplit);
    case 5: return launch_gemm_inst<Cfg, Epi, true, false, true>(st, A, B, sh, epi, grid, ksplit);
    case 4: return launch_gemm_inst<Cfg, Epi, true, false, false>(st, A, B, sh, epi, grid, ksplit);
    case 3: return launch_gemm_inst<Cfg, Epi, false, true, true>(st, A, B, sh, epi, grid, ksplit);
    case 2: return launch_gemm_inst<Cfg, Epi, false, true, false>(st, A, B, sh, epi, grid, ksplit);
    case 1: return launch_gemm_inst<Cfg, Epi, false, false, true>(st, A, B, sh, epi, grid, ksplit);
    default: return launch_gemm_inst<Cfg, Epi, false, false, false>(st, A, B, sh, epi, grid, ksplit);
  }
}

// Tile choice by estimated efficiency = useful fraction of the padded tile grid x wave occupancy x the
// sustained DMMA rate of the configuration measured on B200 (tools/microbench/gemm_shapes.cu:
// 128x128 ~ 31.5, 256x80 ~ 29, 128x80 ~ 27 TFLOP/s).  0: wide, 1: tall, 2: narrow.
inline int gemm_pick_cfg(const GemmShape& sh, int splits) {
  auto eff = [&](int bm, int bn, int ctas_per_sm, double rate) {
    const long long tm = (sh.M + bm - 1) / bm, tn = (sh.N + bn - 1) / bn;
    const double fill = ((double)sh.M * sh.N) / ((double)(tm * bm) * (double)(tn * bn));
    const long long t = tm * tn * splits, slots = 148LL * ctas_per_sm;
    const double waves = (double)t / (double)(((t + slots - 1) / slots) * slots);
    return fill * waves * rate;
  };
  const double e0 = eff(GemmWide::BM, GemmWide::BN, 1, 31.5), e1 = eff(GemmTall::BM, GemmTall::BN, 1, 29.0),
               e2 = eff(GemmNarrow::BM, GemmNarrow::BN, 2, 27.0);
  if (e0 >= e1 && e0 >= e2) return 0;
  return (e1 >= e2) ? 1 : 2;
}

template <class Epi>
inline cudaError_t launch_gemm(cudaStream_t st, GemmOperand A, GemmOperand B, GemmShape sh, Epi epi) {
  switch (gemm_pick_cfg(sh, 1)) {
    case 0: return launch_gemm_cfg<GemmWide>(st, A, B, sh, epi, 1);
    case 1: return launch_gemm_cfg<GemmTall>(st, A, B, sh, epi, 1);
    default: return launch_gemm_cfg<GemmNarrow>(st, A, B, sh, epi, 1);
  }
}

// Split-K launch; returns the number of splits actually used in *splits_out.  The epilogue must carry
// a split stride (EpiStore::split_stride).
template <class Epi>
inline cudaError_t launch_gemm_splitk(cudaStream_t st, GemmOperand A, GemmOperand B, GemmShape sh, Epi epi,
                                      int max_splits, int* splits_out) {
  const int cfg = gemm_pick_cfg(sh, 1);
  const int bm = cfg == 0 ? GemmWide::BM : (cfg == 1 ? GemmTall::BM : GemmNarrow::BM);
  const int bn = cfg == 0 ? GemmWide::BN : (cfg == 1 ? GemmTall::BN : GemmNarrow::BN);
  const int tiles = ((sh.N + bn - 1) / bn) * ((sh.M + bm - 1) / bm);
  int splits = gemm_pick_splits(tiles, sh.K, cfg == 2 ? 2 : 1, max_splits);
  int ksplit = ((sh.K + splits - 1) / splits + GM_BK - 1) / GM_BK * GM_BK;
  splits = (sh.K + ksplit - 1) / ksplit;
  if (splits_out) *splits_out = splits;
  switch (cfg) {
    case 0: return launch_gemm_cfg<GemmWide>(st, A, B, sh, epi, splits);
    case 1: return launch_gemm_cfg<GemmTall>(st, A, B, sh, epi, splits);
    default: return launch_gemm_cfg<GemmNarrow>(st, A, B, sh, epi, splits);
  }
}

}  // namespace emagls
