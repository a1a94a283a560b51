// FP64-accurate GEMM on the 5th-generation tensor cores: error-free slicing (Ozaki scheme I) of both
// operands into balanced base-256 digits (int8), int8 x int8 -> int32 `tcgen05.mma.kind::i8` products
// with the accumulators in TMEM, operands staged by TMA, FP64 recombination in the epilogue.
//
//   x(r, k) = 2^(e_r - 6) * sum_{s < T} q_s(r, k) 256^-s,   |q_0| <= 64, q_s in [-128, 127]   (slice_rows_kernel)
//   C(m, n) = sA(m) sB(n) sum_{d < T} 256^-d sum_{i + j = d} sum_k qA_i(m, k) qB_j(n, k)
//
// with sA = 2^(e - 6).  Products of slices are exact in int32 (T * 2^14 * K < 2^31, i.e. K <= 21845 for
// T = 6; the host refuses longer contractions); pairs with i + j >= T are dropped, so the result carries
// 8 T - 2 bits relative to max|a| max|b| K (T = 6: 2^-46, measured 5e-14 of |a|.|b|; the native FP64 dot
// product carries 2^-53 relative to sum |a||b|).  Base 256 uses all 8 bits of the int8 operands: the same
// 48 bits need T = 6 slices (21 slice pairs) instead of the 7 slices (28 pairs) of 7-bit digits, and the
// digits of a value are the bytes of (x + 0x808080) ^ 0x808080 -- two integer instructions per limb.
//
// Layout: one CTA = one 128 x 64 output tile at a time (persistent over tiles), T accumulators of
// 64 TMEM columns (one per diagonal i + j = d), K streamed in tiles of 64 bytes per slice through a
// 3-stage TMA -> smem ring (64-byte swizzle, K-major operands).  Warp 0: TMA producer, warp 1: MMA
// issuer (one elected thread), warps 2..17: epilogue (TMEM -> registers -> FP64, accumulators released,
// then the functor).
#pragma once
#include <type_traits>
#include <cuda.h>
#include <cuda_runtime.h>
#include <stdint.h>

namespace emagls {
namespace oz {

constexpr int TILE_M = 128, TILE_N = 64, TILE_K = 64, STAGES = 3, MAX_SLICES = 6, EPI_WARPS = 16;
// Tile width / ring depth per use: 64 x 3 stages by default; 80 x 2 stages for the backward product
// (N = 400 = 5 x 80: no padded columns, the 235 MB A operand streams through L2 5 instead of 7 times;
// 6 x 80 = 480 TMEM columns).
// EW: epilogue warps (a multiple of 4: EW / 4 per TMEM lane group, each taking every (EW / 4)-th 8-column chunk).
// 16 warps on an 80-column tile leave ten chunks to four warps per lane group (3 + 3 + 2 + 2); 20 warps take two each.
template <int NT_, int ST_, int EW_ = EPI_WARPS> struct TileCfg {
  static constexpr int NT = NT_, ST = ST_, EW = EW_, THREADS = 64 + 32 * EW_;
  static_assert(EW_ % 4 == 0 && EW_ >= 4 && 64 + 32 * EW_ <= 1024, "epilogue warps: whole lane groups");
};
using TileDefault = TileCfg<TILE_N, STAGES>;
using TileWide = TileCfg<80, 2>;
constexpr int A_SLICE_BYTES = TILE_M * TILE_K;   // 8 KB

// ------------------------------------------------------------------------------------- PTX wrappers
__device__ __forceinline__ uint32_t smem_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }

__device__ __forceinline__ void mbar_init(uint64_t* bar, uint32_t count) {
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count) : "memory");
}
__device__ __forceinline__ void mbar_expect_tx(uint64_t* bar, uint32_t bytes) {
  asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)), "r"(bytes) : "memory");
}
__device__ __forceinline__ void mbar_arrive(uint64_t* bar) {
  asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(smem_u32(bar)) : "memory");
}
__device__ __forceinline__ bool mbar_try(uint64_t* bar, uint32_t parity) {
  uint32_t ok;
  asm volatile(
      "{\n\t.reg .pred p;\n\t"
      "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\t"
      "selp.u32 %0, 1, 0, p;\n\t}"
      : "=r"(ok)
      : "r"(smem_u32(bar)), "r"(parity)
      : "memory");
  return ok != 0;
}
// bounded wait: a protocol error becomes a trap (launch failure) instead of a hung GPU
__device__ __forceinline__ void mbar_wait(uint64_t* bar, uint32_t parity) {
  if (mbar_try(bar, parity)) return;
  const long long t0 = clock64();
  while (!mbar_try(bar, parity)) {
    if (clock64() - t0 > 4000000000LL) __trap();
  }
}
__device__ __forceinline__ void fence_barrier_init() { asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory"); }
__device__ __forceinline__ void tc_fence_before() { asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void tc_fence_after() { asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory"); }

__device__ __forceinline__ void tma_load_3d(void* dst, const CUtensorMap* tm, uint64_t* bar, int c0, int c1, int c2) {
  asm volatile(
      "cp.async.bulk.tensor.3d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4, %5}], [%2];"
      ::"r"(smem_u32(dst)), "l"(reinterpret_cast<uint64_t>(tm)), "r"(smem_u32(bar)), "r"(c0), "r"(c1), "r"(c2)
      : "memory");
}
__device__ __forceinline__ void tma_prefetch_desc(const CUtensorMap* tm) {
  asm volatile("prefetch.tensormap [%0];" ::"l"(reinterpret_cast<uint64_t>(tm)) : "memory");
}

__device__ __forceinline__ void tmem_alloc(uint32_t* dst_smem, uint32_t ncols) {  // whole warp
  asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(dst_smem)), "r"(ncols)
               : "memory");
  asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
}
__device__ __forceinline__ void tmem_dealloc(uint32_t taddr, uint32_t ncols) {    // whole warp
  asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(taddr), "r"(ncols) : "memory");
}
// D[tmem] (+)= A[smem] * B[smem]^T, int8 x int8 -> int32
__device__ __forceinline__ void umma_i8(uint32_t tmem_d, uint64_t adesc, uint64_t bdesc, uint32_t idesc, uint32_t accumulate) {
  asm volatile(
      "{\n\t.reg .pred p;\n\t"
      "setp.ne.b32 p, %4, 0;\n\t"
      "tcgen05.mma.cta_group::1.kind::i8 [%0], %1, %2, %3, p;\n\t}"
      ::"r"(tmem_d), "l"(adesc), "l"(bdesc), "r"(idesc), "r"(accumulate)
      : "memory");
}
// arrive on an mbarrier once every previously issued tcgen05.mma of this thread has completed
__device__ __forceinline__ void umma_commit(uint64_t* bar) {
  asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(smem_u32(bar)) : "memory");
}
// 32 lanes x 8 consecutive 32-bit columns: thread i of the warp receives lane (base lane + i)
__device__ __forceinline__ void tmem_ld8(uint32_t taddr, int32_t (&v)[8]) {
  asm volatile("tcgen05.ld.sync.aligned.32x32b.x8.b32 {%0, %1, %2, %3, %4, %5, %6, %7}, [%8];"
               : "=r"(v[0]), "=r"(v[1]), "=r"(v[2]), "=r"(v[3]), "=r"(v[4]), "=r"(v[5]), "=r"(v[6]), "=r"(v[7])
               : "r"(taddr)
               : "memory");
}
__device__ __forceinline__ void tmem_ld_wait() { asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory"); }

// K-major operand tile, rows of 64 bytes, 64-byte swizzle (cute::UMMA::SmemDescriptor, canonical
// layout Swizzle<2,4,3> o ((8,n),2):((4,SBO),1) in 16-byte units): start address >> 4, LBO = 1
// (unused for swizzled K-major), SBO = 8 rows * 64 B = 512 B, version 1 (Blackwell), layout 4.
__device__ __forceinline__ uint64_t smem_desc_sw64(uint32_t saddr) {
  uint64_t d = 0;
  d |= (uint64_t)((saddr >> 4) & 0x3fffu);
  d |= (uint64_t)1 << 16;
  d |= (uint64_t)(512 >> 4) << 32;
  d |= (uint64_t)1 << 46;
  d |= (uint64_t)4 << 61;
  return d;
}
// cute::UMMA::InstrDescriptor: c_format S32 (2) @4, a/b format INT8 (1) @7/@10, K-major both,
// n_dim = N >> 3 @17, m_dim = M >> 4 @24
__device__ __forceinline__ uint32_t instr_desc_i8(int m, int n) {
  return (2u << 4) | (1u << 7) | (1u << 10) | ((uint32_t)(n >> 3) << 17) | ((uint32_t)(m >> 4) << 24);
}

// ------------------------------------------------------------------------------------- conversions without the XU pipe
// I2F / F2I on FP64 values run on the conversion (XU) pipe, 16 lanes per clock and SM; the epilogues below need
// eight to twelve of them per output value, so they use the classic mantissa tricks on the FP64 / integer pipes:
//   int32 -> double : the word (a ^ 0x80000000) placed in the low mantissa of 2^52 is 2^52 + 2^31 + a exactly
//   double -> int32 : x + 1.5 * 2^52 holds rn(x) (ties to even, |x| < 2^31) in its low word
constexpr double RN_MAGIC = 6755399441055744.0;   // 1.5 * 2^52
__device__ __forceinline__ double i2d_exact(int a) {
  return __hiloint2double(0x43300000, a ^ (int)0x80000000) - 4503601774854144.0;   // 2^52 + 2^31
}
// Exact integer value of one output element from its T diagonal accumulators, rounded once to FP64:
//   v = rn(sum_d acc_d 256^(T-1-d)) = rn(H 256^(T-3) + L),  H = digits 0..2, L = digits 3..T-1
// (|acc_d| < 2^31: |H|, |L| < 2^48, both exact in FP64; v itself may exceed 2^53 and is rounded once)
template <int T>
__device__ __forceinline__ double combine_diagonals(const int32_t (&a)[MAX_SLICES][8], int q) {
  double H = i2d_exact(a[0][q]);
#pragma unroll
  for (int d = 1; d < 3; ++d)
    if (d < T) H = fma(H, 256.0, i2d_exact(a[d][q]));
  if (T <= 3) return H;
  double L = i2d_exact(a[3][q]);
#pragma unroll
  for (int d = 4; d < MAX_SLICES; ++d)
    if (d < T) L = fma(L, 256.0, i2d_exact(a[d][q]));
  return fma(H, (double)(1 << (8 * (T - 3))), L);
}
// The same integer, exact, in 64-bit integer arithmetic while |v| < 2^63, which the int32 range of the accumulators does
// not imply: the host checks drain_i64_fits (Kpad <= 2016 for T = 6), longer contractions would wrap silently.
// Multiply-adds with 64-bit accumulators (IMAD.WIDE)
// instead of 11 FP64 instructions per element -- the drain is the one phase of the epilogue that cannot overlap with
// MMAs, and FP64 is the slowest pipe it could use.  For functors that declare `int64_values`.
template <int T>
__device__ __forceinline__ long long combine_diagonals_i64(const int32_t (&a)[MAX_SLICES][8], int q) {
  long long H = (long long)a[0][q];
#pragma unroll
  for (int d = 1; d < 3; ++d)
    if (d < T) H = H * 256 + (long long)a[d][q];
  if (T <= 3) return H;
  long long L = (long long)a[3][q];
#pragma unroll
  for (int d = 4; d < MAX_SLICES; ++d)
    if (d < T) L = L * 256 + (long long)a[d][q];
  return H * (long long)(1 << (8 * (T - 3))) + L;
}
// weight of the integer above: C = sA sB 256^-(T-1) v
template <int T> __device__ __forceinline__ double diagonal_weight() { return 1.0 / (double)(1ull << (8 * (T - 1))); }

// Balanced base-256 digits (see slice_digits) of ah = a * 256^(T-4), |a| <= 64, as two words: byte j of zl is
// digit T-1-j (j < 3), byte j of zh is digit T-4-j (j < T-3).  Same results as slice_digits, no F2I / I2F.
template <int T>
__device__ __forceinline__ void slice_words(double ah, uint32_t& zl, uint32_t& zh) {
  static_assert(T >= 4 && T <= 6, "hi limb: 1..3 digits, lo limb: 3 digits");
  constexpr int nh = T - 3;
  constexpr int bias_hi = (nh == 3) ? 0x808080 : (nh == 2 ? 0x8080 : 0x80);
  const double th = ah + RN_MAGIC;
  int hi = __double2loint(th);                                         // rn(ah), |hi| <= 2^22
  const double tl = fma(ah - (th - RN_MAGIC), 16777216.0, RN_MAGIC);   // the remainder is exact, |.| <= 1/2
  const int yl = __double2loint(tl) + 0x808080;                        // in (0, 2^25)
  hi += yl >> 24;                                                      // carry (0 or 1)
  zl = (uint32_t)(yl ^ 0x808080);
  zh = (uint32_t)((hi + bias_hi) ^ bias_hi);                           // |hi| <= 2^22 + 1: no carry out
}

// ------------------------------------------------------------------------------------- slicing
// Balanced base-256 digits of a (|a| <= 64): a = sum_{s < T} q_s 256^-s + r, |r| <= 256^-(T-1) / 2,
// |q_0| <= 64, q_s in [-128, 127].  Two int32 limbs (hi: digits 0..T-4, lo: the last three) are rounded
// out of the FP64 value; the balanced digits of a limb x are the bytes of (x + 0x808080) ^ 0x808080
// (adding 128 to every byte propagates the carries, the xor subtracts it again as a signed byte), and
// the carry out of the low limb (its top digit rounding up) moves into the high limb.
template <int T, class Store>
__device__ __forceinline__ void slice_digits(double a, Store&& store) {
  static_assert(T >= 4 && T <= 6, "hi limb: 1..3 digits, lo limb: 3 digits");
  constexpr int nh = T - 3;
  constexpr int bias_hi = (nh == 3) ? 0x808080 : (nh == 2 ? 0x8080 : 0x80);
  const double ah = a * (double)(1 << (8 * (nh - 1)));
  int hi = __double2int_rn(ah);
  const int lo = __double2int_rn((ah - (double)hi) * 16777216.0);     // |lo| <= 2^23
  const int yl = lo + 0x808080;                                       // in (0, 2^25)
  hi += yl >> 24;                                                     // carry (0 or 1)
  const int zl = yl ^ 0x808080;
  store(T - 1, (int)(signed char)(zl));
  store(T - 2, (int)(signed char)(zl >> 8));
  store(T - 3, (int)(signed char)(zl >> 16));
  const int zh = (hi + bias_hi) ^ bias_hi;                            // |hi| <= 2^22 + 1: no carry out
#pragma unroll
  for (int j = 0; j < nh; ++j) store(nh - 1 - j, (int)(signed char)(zh >> (8 * j)));
}

// One warp per row r: x(r, k) = src[r * rs + k * cs], k < K.  out[s][r][Kpad] (int8), scale[r] = 2^(e-6)
// with 2^e > max_k |x|.  Columns K..Kpad-1 are written as zero.
template <int T>
__global__ void slice_rows_kernel(const double* __restrict__ src, long long rs, long long cs, int R, int K, int Kpad,
                                  int8_t* __restrict__ out, double* __restrict__ scale) {
  const int lane = threadIdx.x & 31;
  const int r = blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
  if (r >= R) return;
  const double* x = src + (long long)r * rs;
  double mx = 0.0;
  for (int k = lane; k < K; k += 32) mx = fmax(mx, fabs(x[(long long)k * cs]));
#pragma unroll
  for (int m = 16; m > 0; m >>= 1) mx = fmax(mx, __shfl_xor_sync(0xffffffffu, mx, m));
  int e = 0;
  if (mx > 0.0 && mx < 1e300) frexp(mx, &e);   // mx = f 2^e, f in [0.5, 1)
  if (lane == 0) scale[r] = scalbn(1.0, e - 6);
  const double up = scalbn(1.0, 6 - e);
  for (int k = lane; k < Kpad; k += 32) {
    const double v = (k < K) ? x[(long long)k * cs] * up : 0.0;
    int8_t* o = out + (long long)r * Kpad + k;
    slice_digits<T>(v, [&](int s, int q) { o[(long long)s * R * Kpad] = (int8_t)q; });
  }
}

// ------------------------------------------------------------------------------------- GEMM
struct GemmArgs {
  int M, N, Kpad;           // C is M x N; Kpad multiple of 32 (bytes per slice row of both operands)
  const double* sA;         // [M] row scales of A
  const double* sB;         // [N] row scales of B
  int dbg;                  // microbenchmark switches: 1 = skip the epilogue work, 2 = skip the MMAs, 4 = drain only (raw functors)
  int n_fastest;            // tile order: consecutive tiles share the A rows (1) or the B rows (0)
  int tile_n;               // Cfg::NT of the launched instance (tile_origin)
};

// Persistent tile index -> (m0, n0).  Consecutive tiles run concurrently on neighbouring SMs, so the
// operand indexed by the slow dimension is fetched from DRAM once and re-read from L2 by its
// neighbours: the large operand must be the one shared (backward product: A = 274 MB of digits).
__device__ __forceinline__ void tile_origin(const GemmArgs& g, int tile, int m_tiles, int n_tiles, int& m0, int& n0) {
  if (g.n_fastest) { n0 = (tile % n_tiles) * g.tile_n; m0 = (tile / n_tiles) * TILE_M; }
  else { m0 = (tile % m_tiles) * TILE_M; n0 = (tile / m_tiles) * g.tile_n; }
}

__device__ __forceinline__ bool elect_one() {
  uint32_t pred;
  asm volatile("{\n\t.reg .pred p;\n\telect.sync _|p, 0xffffffff;\n\tselp.u32 %0, 1, 0, p;\n\t}" : "=r"(pred));
  return pred != 0;
}

// Epilogue functor: operator()(m, n0, v[8], M, N) receives 8 consecutive columns n0..n0+7 of row m
// (already scaled, FP64).  Called only for m < M; columns >= N hold zeros and must be skipped.  A functor that
// declares `static constexpr bool all_lanes = true` is entered by every lane of the warp (also m >= M) and
// guards its own stores, so that it may use warp shuffles.
// A functor that declares `static constexpr bool raw = true` works on the unscaled integers (combine_diagonals):
//   begin_tile(m, n, M, N) -> TileState   loads that do not depend on the accumulators, issued before the wait
//   apply(state, m, n0, v[8], M, N)       called for m < M
// (the forward product only needs the direction of y, so the operand scales cancel).
template <class E, class = void> struct epi_raw { static constexpr bool value = false; };
template <class E> struct epi_raw<E, decltype((void)E::raw)> { static constexpr bool value = E::raw; };
template <class E, class = void> struct epi_i64 { static constexpr bool value = false; };
template <class E> struct epi_i64<E, decltype((void)E::int64_values)> { static constexpr bool value = E::int64_values; };
template <class E, class = void> struct epi_all_lanes { static constexpr bool value = false; };
template <class E> struct epi_all_lanes<E, decltype((void)E::all_lanes)> { static constexpr bool value = E::all_lanes; };

// Bytes 0..2 of four words, one word per byte position: r0 = [a0 b0 c0 d0], r1 = [a1 b1 c1 d1], r2 = [a2 b2 c2 d2]
// (the digit words of four values -> one word per digit plane).
__device__ __forceinline__ void transpose4x3(uint32_t a, uint32_t b, uint32_t c, uint32_t d, uint32_t& r0, uint32_t& r1,
                                             uint32_t& r2) {
  const uint32_t ab_lo = __byte_perm(a, b, 0x5140), cd_lo = __byte_perm(c, d, 0x5140);   // [a0 b0 a1 b1]
  const uint32_t ab_hi = __byte_perm(a, b, 0x7362), cd_hi = __byte_perm(c, d, 0x7362);   // [a2 b2 a3 b3]
  r0 = __byte_perm(ab_lo, cd_lo, 0x5410);   // [a0 b0 c0 d0]
  r1 = __byte_perm(ab_lo, cd_lo, 0x7632);   // [a1 b1 c1 d1]
  r2 = __byte_perm(ab_hi, cd_hi, 0x5410);   // [a2 b2 c2 d2]
}
struct EpiStoreF64 {
  double* C; long long ldc;
  __device__ __forceinline__ void operator()(int m, int n0, const double (&v)[8], int M, int N) const {
    double* p = C + (long long)m * ldc + n0;
    if (n0 + 8 <= N && (reinterpret_cast<uintptr_t>(p) & 15) == 0) {   // odd ldc: rows alternate in alignment
#pragma unroll
      for (int q = 0; q < 8; q += 2) *reinterpret_cast<double2*>(p + q) = make_double2(v[q], v[q + 1]);
    } else {
      for (int q = 0; q < 8 && n0 + q < N; ++q) p[q] = v[q];
    }
  }
};

template <int T, class Epi, class Cfg = TileDefault>
__global__ void __launch_bounds__(Cfg::THREADS, 1)
ozaki_gemm_kernel(const __grid_constant__ CUtensorMap tmA, const __grid_constant__ CUtensorMap tmB, GemmArgs g, Epi epi) {
  extern __shared__ uint8_t oz_smem_raw[];
  // 1024-byte aligned carve-up: [stage][A slices | B slices]
  uint8_t* base = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(oz_smem_raw) + 1023) & ~(uintptr_t)1023);
  constexpr int NT = Cfg::NT, ST = Cfg::ST, EPI_WARPS = Cfg::EW, B_SLICE_BYTES = NT * TILE_K;
  constexpr int stage_bytes = T * (A_SLICE_BYTES + B_SLICE_BYTES);
  __shared__ __align__(8) uint64_t full_bar[ST], empty_bar[ST], tmem_full_bar, tmem_empty_bar;
  __shared__ uint32_t tmem_base_s;

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int m_tiles = (g.M + TILE_M - 1) / TILE_M, n_tiles = (g.N + NT - 1) / NT;
  const int num_tiles = m_tiles * n_tiles, tile0 = (int)blockIdx.x, tile_step = (int)gridDim.x;
  const int ksteps_total = g.Kpad / 32;
  const int num_kt = (g.Kpad + TILE_K - 1) / TILE_K;
  constexpr uint32_t tmem_cols = (T * NT <= 256) ? 256u : 512u;

  if (warp == 0 && lane == 0) {
    tma_prefetch_desc(&tmA);
    tma_prefetch_desc(&tmB);
    for (int s = 0; s < ST; ++s) { mbar_init(&full_bar[s], 1); mbar_init(&empty_bar[s], 1); }
    mbar_init(&tmem_full_bar, 1);
    mbar_init(&tmem_empty_bar, EPI_WARPS);   // one arrival per epilogue warp
    fence_barrier_init();
  }
  if (warp == 1) tmem_alloc(&tmem_base_s, tmem_cols);
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = tmem_base_s;

  if (warp == 0) {
    // ================================================================= TMA producer
    if (lane == 0) {
      int stage = 0; uint32_t phase = 0;
      for (int tile = tile0; tile < num_tiles; tile += tile_step) {
        int m0, n0;
        tile_origin(g, tile, m_tiles, n_tiles, m0, n0);
        for (int kt = 0; kt < num_kt; ++kt) {
          mbar_wait(&empty_bar[stage], phase ^ 1);
          uint8_t* sa = base + (size_t)stage * stage_bytes;
          uint8_t* sb = sa + (size_t)T * A_SLICE_BYTES;
          mbar_expect_tx(&full_bar[stage], (uint32_t)stage_bytes);
          tma_load_3d(sa, &tmA, &full_bar[stage], kt * TILE_K, m0, 0);
          tma_load_3d(sb, &tmB, &full_bar[stage], kt * TILE_K, n0, 0);
          if (++stage == ST) { stage = 0; phase ^= 1; }
        }
      }
    }
  } else if (warp == 1) {
    // ================================================================= MMA issuer
    // The whole warp walks the pipeline (uniform control flow); one elected lane issues.  The
    // T (T + 1) / 2 slice pairs of a k-step are straight-line code: every descriptor is the stage's
    // base descriptor plus a compile-time constant, so issue cost stays below the 32 cycles one
    // 128 x 64 x 32 MMA occupies the tensor pipe.
    int stage = 0; uint32_t phase = 0, acc_phase = 0;
    const bool leader = elect_one();
    for (int tile = tile0; tile < num_tiles; tile += tile_step) {
      int m0, n0;
      tile_origin(g, tile, m_tiles, n_tiles, m0, n0);
      const int n_mma = min(NT, ((g.N - n0) + 15) & ~15);
      const uint32_t idesc = instr_desc_i8(TILE_M, n_mma);
      mbar_wait(&tmem_empty_bar, acc_phase ^ 1);   // epilogue has drained the accumulators
      tc_fence_after();
      for (int kt = 0; kt < num_kt; ++kt) {
        mbar_wait(&full_bar[stage], phase);
        tc_fence_after();
        if (leader) {
          const uint32_t sa = smem_u32(base + (size_t)stage * stage_bytes);
          const uint64_t adesc0 = smem_desc_sw64(sa);
          const uint64_t bdesc0 = smem_desc_sw64(sa + (uint32_t)T * A_SLICE_BYTES);
          const int nks = min(TILE_K / 32, ksteps_total - kt * (TILE_K / 32));
          if (!(g.dbg & 2)) {
#pragma unroll
            for (int ks = 0; ks < TILE_K / 32; ++ks) {
              if (ks < nks) {
#pragma unroll
                for (int d = 0; d < T; ++d) {
#pragma unroll
                  for (int i = 0; i <= d; ++i) {
                    const uint64_t ad = adesc0 + (uint64_t)((i * A_SLICE_BYTES + ks * 32) >> 4);
                    const uint64_t bd = bdesc0 + (uint64_t)(((d - i) * B_SLICE_BYTES + ks * 32) >> 4);
                    const uint32_t accum = (ks > 0 || i > 0) ? 1u : (uint32_t)(kt > 0);
                    umma_i8(tmem_base + (uint32_t)d * NT, ad, bd, idesc, accum);
                  }
                }
              }
            }
          }
          umma_commit(&empty_bar[stage]);       // smem slot reusable once these MMAs retire
          if (kt == num_kt - 1) umma_commit(&tmem_full_bar);   // accumulators complete
        }
        __syncwarp();
        if (++stage == ST) { stage = 0; phase ^= 1; }
      }
      acc_phase ^= 1;
    }
  } else {
    // ================================================================= epilogue (warps 2..)
    const int lg = warp & 3;                          // TMEM lane group this warp may access
    const int chunk0 = ((warp - 2) >> 2) * 8;         // first 8-column chunk of this warp
    constexpr int chunk_step = 8 * (EPI_WARPS / 4);
    constexpr int CH_PER_WARP = (NT + chunk_step - 1) / chunk_step;
    uint32_t acc_phase = 0;
    for (int tile = tile0; tile < num_tiles; tile += tile_step) {
      int m0, n0;
      tile_origin(g, tile, m_tiles, n_tiles, m0, n0);
      const int n_mma = min(NT, ((g.N - n0) + 15) & ~15);
      const int m = m0 + lg * 32 + lane;
      const int n_lim = (g.dbg & 1) ? 0 : n_mma;
      // Phase 1 (drain): this warp's chunks go TMEM -> registers -> FP64 (exact integers, one rounding); the
      // accumulators are then handed back, so the MMA warp starts the next tile while phase 2 (the functor:
      // phase continuation, slicing, global stores) runs from registers.
      using Val = typename std::conditional<epi_raw<Epi>::value && epi_i64<Epi>::value, long long, double>::type;
      Val v[CH_PER_WARP][8];
      auto drain = [&]() {
#pragma unroll
        for (int ci = 0; ci < CH_PER_WARP; ++ci) {
          const int c0 = chunk0 + ci * chunk_step;
          if (c0 < n_lim) {
            int32_t a[MAX_SLICES][8];
#pragma unroll
            for (int d = 0; d < MAX_SLICES; ++d)
              if (d < T) tmem_ld8(tmem_base + ((uint32_t)(lg * 32) << 16) + (uint32_t)(d * NT + c0), a[d]);
            tmem_ld_wait();
#pragma unroll
            for (int q = 0; q < 8; ++q) {
              if constexpr (std::is_same<Val, long long>::value) v[ci][q] = combine_diagonals_i64<T>(a, q);
              else v[ci][q] = combine_diagonals<T>(a, q);
            }
          }
        }
        tc_fence_before();
        __syncwarp();
        if (lane == 0) mbar_arrive(&tmem_empty_bar);
      };
      if constexpr (epi_raw<Epi>::value) {
        auto ts = epi.begin_tile(m < g.M ? m : g.M - 1, n0 + chunk0, g.M, g.N);
        mbar_wait(&tmem_full_bar, acc_phase);
        tc_fence_after();
        drain();
        if (g.dbg & 4) { acc_phase ^= 1; continue; }
#pragma unroll
        for (int ci = 0; ci < CH_PER_WARP; ++ci) {
          const int c0 = chunk0 + ci * chunk_step;
          if (c0 < n_lim && (epi_all_lanes<Epi>::value || m < g.M)) epi.apply(ts, m, n0 + c0, v[ci], g.M, g.N);   // all_lanes: warp-uniform entry
        }
      } else {
        mbar_wait(&tmem_full_bar, acc_phase);
        tc_fence_after();
        const double sa = (m < g.M) ? g.sA[m] * diagonal_weight<T>() : 0.0;
        drain();
#pragma unroll
        for (int ci = 0; ci < CH_PER_WARP; ++ci) {
          const int c0 = chunk0 + ci * chunk_step;
          if (c0 < n_lim) {
#pragma unroll
            for (int q = 0; q < 8; ++q) {
              const int n = n0 + c0 + q;
              v[ci][q] *= sa * ((n < g.N) ? g.sB[n] : 0.0);
            }
          }
        }
#pragma unroll
        for (int ci = 0; ci < CH_PER_WARP; ++ci) {
          const int c0 = chunk0 + ci * chunk_step;
          if constexpr (epi_all_lanes<Epi>::value) {
            // functors that exchange data between lanes are entered by the whole warp (c0 and n_lim are warp-uniform)
            if (c0 < n_lim) epi(m, n0 + c0, v[ci], g.M, g.N);
          } else {
            if (c0 < n_lim && m < g.M) epi(m, n0 + c0, v[ci], g.M, g.N);
          }
        }
      }
      acc_phase ^= 1;
    }
  }
  tc_fence_before();
  __syncthreads();
  if (warp == 1) {
    tc_fence_after();
    tmem_dealloc(tmem_base, tmem_cols);
  }
}

// ------------------------------------------------------------------------------------- host side
typedef CUresult (*EncodeTiledFn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*,
                                  const cuuint64_t*, const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave,
                                  CUtensorMapSwizzle, CUtensorMapL2promotion, CUtensorMapFloatOOBfill);

inline EncodeTiledFn encode_tiled_fn() {
  static EncodeTiledFn fn = nullptr;
  if (!fn) {
    void* p = nullptr;
    cudaDriverEntryPointQueryResult qres;
    if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &p, cudaEnableDefault, &qres) != cudaSuccess ||
        qres != cudaDriverEntryPointSuccess)
      return nullptr;
    fn = reinterpret_cast<EncodeTiledFn>(p);
  }
  return fn;
}

// Sliced operand [T][rows][Kpad] int8 -> 3-D tensor map, box {TILE_K, box_rows, T}, 64-byte swizzle,
// out-of-range rows / columns read as zero.
inline bool make_operand_map(CUtensorMap* tm, const int8_t* ptr, int rows, int Kpad, int T, int box_rows) {
  EncodeTiledFn fn = encode_tiled_fn();
  if (!fn) return false;
  cuuint64_t dims[3] = {(cuuint64_t)Kpad, (cuuint64_t)rows, (cuuint64_t)T};
  cuuint64_t strides[2] = {(cuuint64_t)Kpad, (cuuint64_t)Kpad * (cuuint64_t)rows};
  cuuint32_t box[3] = {(cuuint32_t)TILE_K, (cuuint32_t)box_rows, (cuuint32_t)T};
  cuuint32_t estr[3] = {1, 1, 1};
  CUresult r = fn(tm, CU_TENSOR_MAP_DATA_TYPE_UINT8, 3, const_cast<int8_t*>(ptr), dims, strides, box, estr,
                  CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_64B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
                  CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  return r == CUDA_SUCCESS;
}

// int32 accumulators: a diagonal holds at most T pairs of products bounded by 2^14 each
inline bool contraction_fits(int Kpad, int T) { return (long long)T * 16384LL * Kpad < (1LL << 31); }
// 64-bit drain (combine_diagonals_i64): |v| <= Kpad sum_{i+j<T} max|q_i| max|q_j| 256^(T-1-i-j) < 2^63 with |q_0| <= 64,
// |q_s| <= 128 (T = 6: 1.0157 Kpad 2^52, so Kpad <= 2016; T = 4: always, given contraction_fits)
inline bool drain_i64_fits(int Kpad, int T) {
  long long per_k = 0;
  for (int d = 0; d < T; ++d)
    for (int i = 0; i <= d; ++i) per_k += (long long)(i ? 128 : 64) * (d - i ? 128 : 64) << (8 * (T - 1 - d));
  return Kpad <= 0x7FFFFFFFFFFFFFFFLL / per_k;
}

template <class Cfg>
inline size_t gemm_smem_bytes(int T) { return (size_t)Cfg::ST * T * (A_SLICE_BYTES + Cfg::NT * TILE_K) + 1024; }

template <int T, class Epi, class Cfg = TileDefault>
cudaError_t launch_ozaki_gemm_t(cudaStream_t st, const CUtensorMap& tmA, const CUtensorMap& tmB, GemmArgs g,
                                Epi epi, int num_sms) {
  static_assert(T * Cfg::NT <= 512 && Cfg::NT % 16 == 0, "TMEM holds 512 columns; UMMA N is a multiple of 16");
  const size_t smem = gemm_smem_bytes<Cfg>(T);
  cudaError_t e = cudaFuncSetAttribute(ozaki_gemm_kernel<T, Epi, Cfg>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
  if (e != cudaSuccess) return e;
  g.tile_n = Cfg::NT;
  const int tiles = ((g.M + TILE_M - 1) / TILE_M) * ((g.N + Cfg::NT - 1) / Cfg::NT);
  ozaki_gemm_kernel<T, Epi, Cfg><<<tiles < num_sms ? tiles : num_sms, Cfg::THREADS, smem, st>>>(tmA, tmB, g, epi);
  return cudaGetLastError();
}

// C = A * B^T from sliced operands Aq [T][M][Kpad], Bq [T][N][Kpad]
template <class Epi, class Cfg = TileDefault>
cudaError_t launch_ozaki_gemm(cudaStream_t st, const int8_t* Aq, const double* sA, const int8_t* Bq, const double* sB,
                              int M, int N, int Kpad, int T, Epi epi, int num_sms, int dbg = 0) {
  if (Kpad % 32 != 0 || !contraction_fits(Kpad, T)) return cudaErrorInvalidValue;
  CUtensorMap tmA, tmB;
  if (!make_operand_map(&tmA, Aq, M, Kpad, T, TILE_M) || !make_operand_map(&tmB, Bq, N, Kpad, T, Cfg::NT))
    return cudaErrorInvalidValue;
  const int m_tiles = (M + TILE_M - 1) / TILE_M, n_tiles = (N + Cfg::NT - 1) / Cfg::NT;
  GemmArgs g{M, N, Kpad, sA, sB, dbg, n_tiles < m_tiles ? 1 : 0, Cfg::NT};
  switch (T) {
    case 4: return launch_ozaki_gemm_t<4, Epi, Cfg>(st, tmA, tmB, g, epi, num_sms);
    case 6: return launch_ozaki_gemm_t<6, Epi, Cfg>(st, tmA, tmB, g, epi, num_sms);
    default: return cudaErrorInvalidValue;
  }
}

}  // namespace oz
}  // namespace emagls
