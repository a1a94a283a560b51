// Head-tracked render of a real SH-domain signal by sound-field rotation (contract in include/emagls_cuda.h and
// DESIGN.md "Head-tracked render of SH signals"): every sample is rotated by the blend of the SH rotation matrices of
// its tracker frame and the previous one, x'[n] = in[n] @ ((1 - g) Q_a + g Q_c), and the rotated signal goes through
// the static render (render.cu) with one filter pair.  Long signals are processed in time chunks with a (len - 1)-sample
// input halo, so that the rotated workspace stays within the same budget as the bank render's.
#include <algorithm>
#include <cstdint>
#include <vector>
#include "render.h"
#include "shrot.cuh"

namespace emagls {
namespace {

constexpr int SHT_MAX_ORDER = 7;   // (order + 1)^2 <= 64 channels, as emagls_rotate_sh
constexpr int SHT_T = 128;         // threads per CTA of the rotation kernel
constexpr int SHT_S = 4;           // samples per thread (strided by 32: every load and store is a 256-byte row)

}  // namespace

// Q[j][band_offset(l) + r (2l+1) + c] = getSHrotMtx(rot[f], order, 'real')[l^2 + r][l^2 + c] for frame f = f_base + j
// (blockIdx.x), and same[j] = 1 when rot[f] is bitwise equal to rot[f - 1].  rot[k] holds frame rot_base + k.
// One CTA per frame: the band recursion of shrot.cuh builds the full matrix in shared memory, of which only the
// diagonal blocks are stored.  Listener blockIdx.y reads rot + y rot_ls and writes Q + y nfr_ls blk, same + y nfr_ls.
__global__ void frame_rotations_kernel(const double* __restrict__ rot, long long rot_ls, long long rot_base,
                                       long long f_base, int order, double* __restrict__ Q, int* __restrict__ same,
                                       long long nfr_ls) {
  extern __shared__ double fr_Rr[];
  __shared__ Rot1 R1;
  __shared__ int rotate;
  const int nsh = (order + 1) * (order + 1), blk = band_offset(order + 1);
  const long long j = blockIdx.x, f = f_base + j;
  rot += blockIdx.y * rot_ls;
  Q += blockIdx.y * nfr_ls * blk;
  same += blockIdx.y * nfr_ls;
  const double* E = rot + (f - rot_base) * 9;
  if (threadIdx.x == 0) {
    double M[3][3];
    for (int e = 0; e < 9; ++e) M[e / 3][e % 3] = E[e];
    rot1_from_matrix(M, R1);
    rotate = 1;
    int eq = f > rot_base;
    for (int e = 0; eq && e < 9; ++e) eq = __double_as_longlong(E[e]) == __double_as_longlong(E[e - 9]);
    same[j] = eq;
  }
  sh_rot_real_bands(R1, &rotate, order, fr_Rr, threadIdx.x, blockDim.x);
  double* q = Q + j * blk;
  for (int l = 0; l <= order; ++l) {
    const int w = 2 * l + 1, o = band_offset(l), d = l * l;
    for (int e = threadIdx.x; e < w * w; e += blockDim.x) q[o + e] = fr_Rr[(d + e / w) * nsh + d + e % w];
  }
}

// One band (W = 2l + 1 channels from c0) of S samples that share the frame pair (qc, qa): y = x @ Q_c, and
// (1 - g) (x @ Q_a) + g y where the sample blends.  x is read column by column from `in` (row src[s]) and the result
// written to `out` (row dst[s]); the matrix entries are warp-uniform loads whenever the warp's samples share a frame.
template <int W, int S>
__device__ __forceinline__ void rotate_band(const double* __restrict__ in, long long ld_in, double* __restrict__ out,
                                            long long ld_out, int c0, const double* __restrict__ qc,
                                            const double* __restrict__ qa, const long long (&src)[S],
                                            const long long (&dst)[S], const bool (&ok)[S], const double (&g)[S],
                                            const bool (&blend)[S], bool any_blend) {
  double x[S][W];
#pragma unroll
  for (int k = 0; k < W; ++k)
#pragma unroll
    for (int s = 0; s < S; ++s) x[s][k] = ok[s] ? in[(long long)(c0 + k) * ld_in + src[s]] : 0.0;
#pragma unroll 1
  for (int j = 0; j < W; ++j) {
    double yc[S], ya[S];
#pragma unroll
    for (int s = 0; s < S; ++s) { yc[s] = 0.0; ya[s] = 0.0; }
#pragma unroll
    for (int k = 0; k < W; ++k) {
      const double q = __ldg(qc + k * W + j);
#pragma unroll
      for (int s = 0; s < S; ++s) yc[s] = fma(x[s][k], q, yc[s]);
    }
    if (any_blend) {
#pragma unroll
      for (int k = 0; k < W; ++k) {
        const double q = __ldg(qa + k * W + j);
#pragma unroll
        for (int s = 0; s < S; ++s) ya[s] = fma(x[s][k], q, ya[s]);
      }
    }
#pragma unroll
    for (int s = 0; s < S; ++s)
      if (ok[s]) out[(long long)(c0 + j) * ld_out + dst[s]] = blend[s] ? fma(g[s], yc[s], (1.0 - g[s]) * ya[s]) : yc[s];
  }
}

template <int S>
__device__ __forceinline__ void rotate_samples(const double* __restrict__ in, long long ld_in, double* __restrict__ out,
                                               long long ld_out, int order, const double* __restrict__ qc,
                                               const double* __restrict__ qa, const long long (&src)[S],
                                               const long long (&dst)[S], const bool (&ok)[S], const double (&g)[S],
                                               const bool (&blend)[S]) {
  bool any_blend = false;
#pragma unroll
  for (int s = 0; s < S; ++s) any_blend |= ok[s] && blend[s];
#define SHT_BAND(L)                                                                                                   \
  if (order >= L)                                                                                                     \
    rotate_band<2 * L + 1, S>(in, ld_in, out, ld_out, L * L, qc + band_offset(L), qa + band_offset(L), src, dst, ok, \
                              g, blend, any_blend);
  SHT_BAND(0) SHT_BAND(1) SHT_BAND(2) SHT_BAND(3) SHT_BAND(4) SHT_BAND(5) SHT_BAND(6) SHT_BAND(7)
#undef SHT_BAND
}

// out[ch][q] = (in[n, :] @ M(n))[ch] for the m samples n = h0 + q of a chunk (column-major, leading dimensions
// ld_in = the signal's length and m).  t = first_sample + n, f = t / hop, i = t - f hop, c = f, a = max(f - 1, 0),
// g = (i + 0.5) / fade for i < fade; M = Q_c exactly when a == c, when rot[a] and rot[c] are bitwise equal or when
// i >= fade.  Q and same hold frames f_base ... (frame_rotations_kernel).  Each warp covers 32 S consecutive samples,
// lane + 32 s for thread s; a thread whose samples share a frame applies each loaded matrix entry to all of them, the
// others (a frame boundary inside the warp's span, or hops shorter than that span) take them one at a time.
// Listener blockIdx.y rotates the same input with Q + y nfr_ls blk, same + y nfr_ls into out + y out_ls.
__global__ void __launch_bounds__(SHT_T, 1)
sh_track_rotate_kernel(const double* __restrict__ in, long long ld_in, long long h0, long long m, int order,
                       const double* __restrict__ Q, const int* __restrict__ same, long long nfr_ls, long long f_base,
                       long long first_sample, int hop, int fade, double* __restrict__ out, long long out_ls) {
  const int blk = band_offset(order + 1);
  Q += blockIdx.y * nfr_ls * blk;
  same += blockIdx.y * nfr_ls;
  out += blockIdx.y * out_ls;
  const long long warp = ((long long)blockIdx.x * SHT_T + threadIdx.x) / 32;
  const int lane = threadIdx.x & 31;
  long long src[SHT_S], dst[SHT_S], fr[SHT_S];
  bool ok[SHT_S], blend[SHT_S];
  double g[SHT_S];
  bool uniform = true;
#pragma unroll
  for (int s = 0; s < SHT_S; ++s) {
    const long long q = warp * 32 * SHT_S + 32 * s + lane;
    ok[s] = q < m;
    dst[s] = ok[s] ? q : 0;
    src[s] = h0 + dst[s];
    const long long t = first_sample + src[s], f = t / hop;
    const int i = (int)(t - f * hop);
    fr[s] = f;
    blend[s] = f > 0 && i < fade && !same[f - f_base];
    g[s] = blend[s] ? ((double)i + 0.5) / (double)fade : 1.0;
    uniform &= !ok[s] || f == fr[0];
  }
  if (!ok[0]) return;
  if (uniform) {
    const double* qc = Q + (fr[0] - f_base) * blk;
    rotate_samples<SHT_S>(in, ld_in, out, m, order, qc, fr[0] > 0 ? qc - blk : qc, src, dst, ok, g, blend);
    return;
  }
#pragma unroll 1
  for (int s = 0; s < SHT_S; ++s) {
    // sample s in registers (a selection unrolled over the compile-time indices keeps the arrays out of local memory)
    long long src1[1] = {0}, dst1[1] = {0}, f = 0;
    bool ok1[1] = {false}, blend1[1] = {false};
    double g1[1] = {1.0};
#pragma unroll
    for (int u = 0; u < SHT_S; ++u)
      if (u == s) { src1[0] = src[u]; dst1[0] = dst[u]; f = fr[u]; ok1[0] = ok[u]; blend1[0] = blend[u]; g1[0] = g[u]; }
    if (!ok1[0]) continue;
    const double* qc = Q + (f - f_base) * blk;
    rotate_samples<1>(in, ld_in, out, m, order, qc, f > 0 ? qc - blk : qc, src1, dst1, ok1, g1, blend1);
  }
}

void launch_frame_rotations(emagls_ctx* h, int nl, const double* rot, long long rot_ls, long long rot_base,
                            long long f_base, long long nfr, int order, double* Q, int* same, long long nfr_ls) {
  const int C = (order + 1) * (order + 1);
  frame_rotations_kernel<<<dim3((unsigned)nfr, (unsigned)nl), 128, (size_t)C * C * sizeof(double), h->stream>>>(
      rot, rot_ls, rot_base, f_base, order, Q, same, nfr_ls);
  EM_CUDA(cudaGetLastError());
}

void launch_sh_track_rotate(emagls_ctx* h, int nl, const double* in, long long ld_in, long long h0, long long m,
                            int order, const double* Q, const int* same, long long nfr_ls, long long f_base,
                            long long first_sample, int hop, int fade, double* out, long long out_ls) {
  const long long warps = (m + 32 * SHT_S - 1) / (32 * SHT_S);
  sh_track_rotate_kernel<<<dim3((unsigned)((warps * 32 + SHT_T - 1) / SHT_T), (unsigned)nl), SHT_T, 0, h->stream>>>(
      in, ld_in, h0, m, order, Q, same, nfr_ls, f_base, first_sample, hop, fade, out, out_ls);
  EM_CUDA(cudaGetLastError());
}

namespace {

void check_sh_tracked_args(const double* in, long long num_samples, int order, const double* wL, const double* wR,
                           int len, const double* rotations, long long num_frames, int hop, int fade,
                           long long first_sample, int compensate_delay, const double* out) {
  EM_REQUIRE(in && wL && wR && rotations && out, "null argument");
  EM_REQUIRE(order >= 0 && order <= SHT_MAX_ORDER, "order must lie in [0, 7]");
  EM_REQUIRE(num_samples > 0 && len > 0, "empty input");
  EM_REQUIRE(hop >= 1, "hop must be >= 1");
  EM_REQUIRE(fade >= 0 && fade <= hop, "fade must lie in [0, hop]");
  EM_REQUIRE(first_sample >= 0, "first_sample must be >= 0");
  EM_REQUIRE(num_frames >= (first_sample + num_samples - 1) / hop + 1, "track shorter than the signal");
  EM_REQUIRE(!compensate_delay || len % 2 == 0, "compensateDelay needs an even filter length");
  EM_REQUIRE(num_samples - (compensate_delay ? (len / 2 - 1) : 0) > 0, "signal shorter than the compensated delay");
}

// rot[k] is frame rot_base + k (device memory); every frame the signal uses must be there
void binaural_decode_sh_tracked_dev(emagls_ctx* h, const double* in, long long num_samples, int order,
                                    const double* wL, const double* wR, int len, const double* rot, long long rot_base,
                                    int hop, int fade, long long first_sample, int compensate_delay, double* out) {
  cudaStream_t st = h->stream;
  const int C = (order + 1) * (order + 1), blk = band_offset(order + 1);
  const long long skip = compensate_delay ? (len / 2 - 1) : 0;
  const long long out_rows = num_samples - skip;

  // Chunks of output samples [c_lo, c_hi) whose rotated input [h0, c_hi), h0 = c_lo - (len - 1) rounded down to an
  // even sample, and frame matrices fit the workspace budget (min(40 % of free memory, 16 GB), or EMAGLS_TRACK_WS_MB,
  // as the bank render).  Chunk boundaries are even, so every chunk but an odd-length last one keeps the static
  // render's fused route.
  double budget;
  {
    size_t free_b = 0, total_b = 0;
    EM_CUDA(cudaMemGetInfo(&free_b, &total_b));
    budget = std::min(0.4 * (double)free_b, 16.0 * 1073741824.0);
    const int ws_mb = env_int("EMAGLS_TRACK_WS_MB", 0);
    if (ws_mb > 0) budget = (double)ws_mb * 1048576.0;
  }
  const double per_sample = 8.0 * C + 8.0 * (blk + 1) / hop;
  const long long halo = len;          // >= len - 1 after rounding h0 down to even
  const double fixed = (double)halo * per_sample + 3.0 * 8.0 * (blk + 1);
  long long payload = (long long)std::max(0.0, (budget - fixed) / per_sample);
  payload = std::max<long long>(payload & ~1LL, 2 * (long long)len + 2);
  const bool single = payload >= num_samples - skip;

  struct Chunk { long long c_lo, c_hi, h0, f_base, nfr; };
  std::vector<Chunk> chunks;
  long long nfr_max = 0, m_max = 0;
  for (long long c_lo = skip; c_lo < num_samples;) {
    const long long c_hi = single ? num_samples : std::min((c_lo + payload) & ~1LL, num_samples);
    const long long h0 = single ? 0 : std::max<long long>(0, (c_lo - (len - 1)) & ~1LL);
    const long long f_base = std::max<long long>((first_sample + h0) / hop - 1, 0);
    const long long nfr = (first_sample + c_hi - 1) / hop - f_base + 1;
    chunks.push_back({c_lo, c_hi, h0, f_base, nfr});
    nfr_max = std::max(nfr_max, nfr);
    m_max = std::max(m_max, c_hi - h0);
    c_lo = c_hi;
  }
  EM_REQUIRE(nfr_max < 2147483647LL, "too many tracker frames in one chunk");

  Arena ar(st);
  double* ws = ar.get<double>((size_t)m_max * C);
  double* Q = ar.get<double>((size_t)nfr_max * blk);
  int* same = ar.get<int>((size_t)nfr_max);
  for (const Chunk& k : chunks) {
    const long long m = k.c_hi - k.h0;
    {
      ProfSpan ps(h, EM_PROF_RENDER_STAGE);
      frame_rotations_kernel<<<(unsigned)k.nfr, 128, (size_t)C * C * sizeof(double), st>>>(rot, 0, rot_base,
                                                                                          k.f_base, order, Q, same, 0);
      EM_CUDA(cudaGetLastError());
      const long long warps = (m + 32 * SHT_S - 1) / (32 * SHT_S);
      sh_track_rotate_kernel<<<(unsigned)((warps * 32 + SHT_T - 1) / SHT_T), SHT_T, 0, st>>>(
          in, num_samples, k.h0, m, order, Q, same, 0, k.f_base, first_sample, hop, fade, ws, 0);
      EM_CUDA(cudaGetLastError());
    }
    h->launches += 2;
    // output rows c_lo - skip .. c_hi - skip - 1 of both ears, straight into `out`
    binaural_decode_rows(h, ws, m, C, wL, wR, len, k.c_lo - k.h0, out_rows, out + (k.c_lo - skip));
  }
  // stream-ordered: the arena's cudaFreeAsync calls queue behind the work above
}

}  // namespace
}  // namespace emagls

using namespace emagls;

extern "C" {

int emagls_binaural_decode_sh_tracked_dev(emagls_handle h, const double* in, long long num_samples, int order,
                                          const double* wL, const double* wR, int len, const double* rotations,
                                          long long num_frames, int hop, int fade, long long first_sample,
                                          int compensate_delay, double* out) {
  return guarded(h, [&] {
    check_sh_tracked_args(in, num_samples, order, wL, wR, len, rotations, num_frames, hop, fade, first_sample,
                          compensate_delay, out);
    binaural_decode_sh_tracked_dev(h, in, num_samples, order, wL, wR, len, rotations, 0, hop, fade, first_sample,
                                   compensate_delay, out);
  });
}

int emagls_binaural_decode_sh_tracked(emagls_handle h, const double* in, long long num_samples, int order,
                                      const double* wL, const double* wR, int len, const double* rotations,
                                      long long num_frames, int hop, int fade, long long first_sample,
                                      int compensate_delay, double* out) {
  return guarded(h, [&] {
    check_sh_tracked_args(in, num_samples, order, wL, wR, len, rotations, num_frames, hop, fade, first_sample,
                          compensate_delay, out);
    const long long C = (order + 1) * (order + 1);
    const long long out_rows = num_samples - (compensate_delay ? (len / 2 - 1) : 0);
    // the frames the signal uses: from the one before its first frame (the first fade) to its last
    const long long f_lo = std::max<long long>(first_sample / hop - 1, 0);
    const long long f_hi = (first_sample + num_samples - 1) / hop;
    cudaStream_t st = h->stream;
    Arena ar(st);
    double* d_in = ar.upload(in, (size_t)(num_samples * C));
    double* d_wL = ar.upload(wL, (size_t)len * C);
    double* d_wR = ar.upload(wR, (size_t)len * C);
    double* d_rot = ar.upload(rotations + f_lo * 9, (size_t)(f_hi - f_lo + 1) * 9);
    double* d_out = ar.get<double>((size_t)out_rows * 2);
    binaural_decode_sh_tracked_dev(h, d_in, num_samples, order, d_wL, d_wR, len, d_rot, f_lo, hop, fade, first_sample,
                                   compensate_delay, d_out);
    EM_CUDA(cudaMemcpyAsync(out, d_out, (size_t)out_rows * 2 * sizeof(double), cudaMemcpyDeviceToHost, st));
    EM_CUDA(cudaStreamSynchronize(st));
  });
}

}  // extern "C"
