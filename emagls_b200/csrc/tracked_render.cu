// Head-tracked binaural render: binauralDecode with a filter bank [len x ch x P] whose page is picked per tracker
// frame, crossfading linearly between the pages of consecutive frames (contract in include/emagls_cuda.h and
// DESIGN.md "Head-tracked render").  Partitioned overlap-save as in render.cu; every block of L outputs runs the
// multiply-accumulate and the inverse transform once per distinct page its samples need (a (block, page) "pair"), and
// the combine kernel mixes the pairs' time signals with the crossfade weights.
#include <algorithm>
#include <climits>
#include <cstdint>
#include <cstdlib>
#include <vector>
#include "render.h"

namespace emagls {
namespace {

// wp[u][ear][ch][N] = page pages[u] of the bank, zero-padded to N (pages u >= nu: zeros, the padding of the last batch)
__global__ void gather_pad_filters_kernel(const double* __restrict__ wL, const double* __restrict__ wR, int len,
                                          int num_ch, const int* __restrict__ pages, int nu, int ub, int N,
                                          double* __restrict__ wp) {
  const long long idx = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (idx >= (long long)ub * 2 * num_ch * N) return;
  const int t = (int)(idx % N);
  const long long r = idx / N;
  const int ch = (int)(r % num_ch), ear = (int)((r / num_ch) & 1), u = (int)(r / (2 * num_ch));
  const double* w = ear ? wR : wL;
  wp[idx] = (u < nu && t < len) ? w[((long long)pages[u] * num_ch + ch) * len + t] : 0.0;
}

// Y[pair][ear][f] = sum_ch X[ch][b][f] * Hw[u(pair)][ear][ch][f] for the pairs of block b (blockIdx.y) of this chunk.
// One thread per (f, block) keeps the accumulators of G pairs in registers, so every channel-spectrum value is read
// once per group of G pairs; a block with more pairs takes several passes.  The channel loop is unrolled by CU, so
// CU * (2 G + 1) independent 16-byte loads are in flight per thread.  The pair count is uniform over a CTA (one block
// per grid row), so the predicates on q < np do not diverge.
template <int G, int CU>
__global__ void __launch_bounds__(128)
tracked_mac_kernel(const cplx* __restrict__ X, const cplx* __restrict__ Hw, const int* __restrict__ blk_off,
                   const int* __restrict__ pair_u, int num_ch, int nbc, int F, cplx* __restrict__ Y) {
  const int f = blockIdx.x * blockDim.x + threadIdx.x;
  const int b = blockIdx.y;
  if (f >= F) return;
  const int p_base = blk_off[0], p0 = blk_off[b], p1 = blk_off[b + 1];
  const long long xs = (long long)nbc * F;           // channel stride of X
  const long long hs = 2LL * num_ch * F;             // page stride of Hw
  const long long es = (long long)num_ch * F;        // ear stride of Hw
  const cplx* x = X + (long long)b * F + f;
  for (int g0 = p0; g0 < p1; g0 += G) {
    const int np = min(G, p1 - g0);
    const cplx* hp[G];
    cplx yl[G], yr[G];
#pragma unroll
    for (int q = 0; q < G; ++q) {
      hp[q] = Hw + (long long)pair_u[min(g0 + q, p1 - 1)] * hs + f;
      yl[q] = mk(0.0, 0.0); yr[q] = mk(0.0, 0.0);
    }
    int ch = 0;
    for (; ch + CU <= num_ch; ch += CU) {
      cplx xv[CU], a[CU][G], c[CU][G];
#pragma unroll
      for (int u = 0; u < CU; ++u) {
        xv[u] = x[(long long)(ch + u) * xs];
#pragma unroll
        for (int q = 0; q < G; ++q)
          if (q < np) {
            a[u][q] = hp[q][(long long)(ch + u) * F];
            c[u][q] = hp[q][es + (long long)(ch + u) * F];
          }
      }
#pragma unroll
      for (int u = 0; u < CU; ++u)
#pragma unroll
        for (int q = 0; q < G; ++q)
          if (q < np) { cfma(yl[q], xv[u], a[u][q]); cfma(yr[q], xv[u], c[u][q]); }
    }
    for (; ch < num_ch; ++ch) {
      const cplx xv = x[(long long)ch * xs];
#pragma unroll
      for (int q = 0; q < G; ++q)
        if (q < np) {
          cfma(yl[q], xv, hp[q][(long long)ch * F]);
          cfma(yr[q], xv, hp[q][es + (long long)ch * F]);
        }
    }
#pragma unroll
    for (int q = 0; q < G; ++q)
      if (q < np) {
        const long long o = (long long)(g0 + q - p_base) * 2 * F + f;
        Y[o] = yl[q];
        Y[o + F] = yr[q];
      }
  }
}

// out[ear][n - skip] = sum over the pairs of n's block of weight(page) * yseg[pair][ear][ov + i] / N for input sample
// n = (b0 + b) L + i; weight(page) = (page == c ? g : 0) + (page == a ? 1 - g : 0) with the crossfade of the contract
// (g = 1 when a == c, so the weight is exactly 1 there).  trk holds track[f_base ..].
__global__ void tracked_combine_kernel(const double* __restrict__ yseg, const int* __restrict__ blk_off,
                                       const int* __restrict__ pair_page, const int* __restrict__ trk, long long f_base,
                                       int nbk, int N, int L, int ov, long long b0, long long first_sample, int hop,
                                       int fade, long long num_samples, long long skip, long long out_rows,
                                       double* __restrict__ out) {
  const long long idx = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (idx >= (long long)nbk * L) return;
  const int b = (int)(idx / L), i = (int)(idx % L);
  const long long n = (b0 + b) * L + i;
  if (n >= num_samples || n < skip) return;
  const long long t = first_sample + n, f = t / hop;
  const int ii = (int)(t - f * hop);
  const int c = trk[f - f_base], a = trk[(f > 0 ? f - 1 : 0) - f_base];
  const double g = (a != c && ii < fade) ? ((double)ii + 0.5) / (double)fade : 1.0;
  const int p_base = blk_off[0], p0 = blk_off[b], p1 = blk_off[b + 1];
  double yl = 0.0, yr = 0.0;
  for (int p = p0; p < p1; ++p) {
    const int pg = pair_page[p];
    const double w = (pg == c ? g : 0.0) + (pg == a ? 1.0 - g : 0.0);
    if (w == 0.0) continue;
    const double* y = yseg + (long long)(p - p_base) * 2 * N + ov + i;
    yl = fma(w, y[0], yl);
    yr = fma(w, y[N], yr);
  }
  const double inv_n = 1.0 / (double)N;
  out[n - skip] = yl * inv_n;
  out[out_rows + n - skip] = yr * inv_n;
}

// (block, page) pairs of a geometry, in block order: blk_off[b] .. blk_off[b + 1] are the pairs of block b, page[] their
// bank pages.  Block b covers input samples [b L, (b + 1) L); it needs track[f] for every frame f it intersects and
// track[f - 1] where it intersects frame f's fade region.  Entries are checked against num_pages here, so every
// page the render reads is validated on the host.
struct PairTable {
  long long nblk = 0;
  std::vector<int> blk_off, page;
};

PairTable build_pairs(const int32_t* track, int num_pages, long long num_samples, long long first_sample, int hop,
                      int fade, int L) {
  PairTable pt;
  pt.nblk = (num_samples + L - 1) / L;
  pt.blk_off.reserve(pt.nblk + 1);
  std::vector<long long> mark(num_pages, -1);
  for (long long b = 0; b < pt.nblk; ++b) {
    pt.blk_off.push_back((int)pt.page.size());
    const long long t_lo = first_sample + b * L, t_hi = first_sample + std::min<long long>((b + 1) * L, num_samples) - 1;
    auto add = [&](int p) {
      EM_REQUIRE(p >= 0 && p < num_pages, "track entry outside [0, num_pages)");
      if (mark[p] != b) { mark[p] = b; pt.page.push_back(p); }
    };
    for (long long f = t_lo / hop; f <= t_hi / hop; ++f) {
      add(track[f]);
      if (f > 0 && f * hop + fade - 1 >= t_lo && fade > 0) add(track[f - 1]);
    }
    EM_REQUIRE(pt.page.size() < (size_t)INT_MAX, "track needs too many (block, page) pairs");
  }
  pt.blk_off.push_back((int)pt.page.size());
  return pt;
}

// HBM bytes of the cuFFT route for one geometry: the channel spectra of every block, and per pair the filter spectra of
// the multiply-accumulate (2 ch F complex), the two ear spectra (written, read by the inverse transform) and the two
// time signals (written by the inverse transform, read by the combine)
double modelled_bytes(const PairTable& pt, int num_ch, int N) {
  const double F = N / 2 + 1;
  return (double)pt.nblk * num_ch * F * 16 + (double)pt.page.size() * (2.0 * num_ch * F * 16 + 4 * F * 16 + 4.0 * N * 8);
}

int pow2_at_least(long long v) {
  int p = 1;
  while (p < v) p <<= 1;
  return p;
}

// The argument checks of the contract that need no table (the page range is checked by build_pairs)
void check_tracked_args(const double* in, long long num_samples, int num_ch, const double* wL, const double* wR, int len,
                        int num_pages, const int32_t* track, long long num_frames, int hop, int fade,
                        long long first_sample, int compensate_delay, const double* out) {
  EM_REQUIRE(in && wL && wR && track && out, "null argument");
  EM_REQUIRE(num_samples > 0 && num_ch > 0 && len > 0 && num_pages > 0, "empty input");
  EM_REQUIRE(hop >= 1, "hop must be >= 1");
  EM_REQUIRE(fade >= 0 && fade <= hop, "fade must lie in [0, hop]");
  EM_REQUIRE(first_sample >= 0, "first_sample must be >= 0");
  EM_REQUIRE(num_frames >= (first_sample + num_samples - 1) / hop + 1, "track shorter than the signal");
  EM_REQUIRE(!compensate_delay || len % 2 == 0, "compensateDelay needs an even filter length");
  EM_REQUIRE(num_samples - (compensate_delay ? (len / 2 - 1) : 0) > 0, "signal shorter than the compensated delay");
}

}  // namespace

void binaural_decode_tracked_dev(emagls_ctx* h, const double* in, long long num_samples, int num_ch, const double* wL,
                                 const double* wR, int len, int num_pages, const int32_t* track, long long num_frames,
                                 int hop, int fade, long long first_sample, int compensate_delay, double* out) {
  check_tracked_args(in, num_samples, num_ch, wL, wR, len, num_pages, track, num_frames, hop, fade, first_sample,
                     compensate_delay, out);
  const long long skip = compensate_delay ? (len / 2 - 1) : 0;
  const long long out_rows = num_samples - skip;
  cudaStream_t st = h->stream;
  const int ov = (len + 1) & ~1;
  int Nmin = 16;
  while (Nmin < 2 * len) Nmin <<= 1;

  // Geometry: every block runs one multiply-accumulate and one inverse transform per pair, so the FFT size is the
  // candidate (Nmin, 2 Nmin, 4 Nmin; no block much longer than the signal) with the fewest modelled HBM bytes for this
  // track (DESIGN.md "Head-tracked render").  EMAGLS_TRACK_FFT=n picks the size as EMAGLS_RENDER_FFT does.
  int N = Nmin;
  PairTable pt = build_pairs(track, num_pages, num_samples, first_sample, hop, fade, N - ov);
  if (const int want = env_int("EMAGLS_TRACK_FFT", 0); want > 0) {
    while (N < want && (long long)(N - ov) < num_samples) N <<= 1;
    if (N != Nmin) pt = build_pairs(track, num_pages, num_samples, first_sample, hop, fade, N - ov);
  } else {
    double best = modelled_bytes(pt, num_ch, N);
    for (int Nc = 2 * Nmin; Nc <= 4 * Nmin && (long long)(Nc / 2 - ov) < num_samples; Nc <<= 1) {
      PairTable pc = build_pairs(track, num_pages, num_samples, first_sample, hop, fade, Nc - ov);
      const double bytes = modelled_bytes(pc, num_ch, Nc);
      if (bytes < best) { best = bytes; N = Nc; pt = std::move(pc); }
    }
  }
  const int L = N - ov, F = N / 2 + 1;
  const long long nblk = pt.nblk;
  const int nex = ForwardStage::extra_blocks(ov, L);

  // Chunks of cb blocks whose channel spectra, pair spectra and time signals and referenced-page spectra fit the
  // workspace budget (min(40 % of free memory, 16 GB), or EMAGLS_TRACK_WS_MB)
  double budget;
  {
    size_t free_b = 0, total_b = 0;
    EM_CUDA(cudaMemGetInfo(&free_b, &total_b));
    budget = std::min(0.4 * (double)free_b, 16.0 * 1073741824.0);
    const int ws_mb = env_int("EMAGLS_TRACK_WS_MB", 0);
    if (ws_mb > 0) budget = (double)ws_mb * 1048576.0;
  }
  std::vector<long long> umark(num_pages, -1);
  auto chunk_pages = [&](long long b0, long long nbk, long long tag, std::vector<int>* pages) {
    long long nu = 0;
    for (int p = pt.blk_off[b0]; p < pt.blk_off[b0 + nbk]; ++p)
      if (umark[pt.page[p]] != tag) {
        umark[pt.page[p]] = tag;
        ++nu;
        if (pages) pages->push_back(pt.page[p]);
      }
    return nu;
  };
  long long cb = std::min<long long>(nblk, 65535);
  long long tag = 0;
  for (;;) {
    double worst = 0.0;
    for (long long b0 = 0; b0 < nblk; b0 += cb) {
      const long long nbk = std::min(cb, nblk - b0);
      const double np = pt.blk_off[b0 + nbk] - pt.blk_off[b0];
      const double nu = (double)chunk_pages(b0, nbk, tag++, nullptr);
      worst = std::max(worst, (double)num_ch * (nbk + nex) * ((double)F * 16 + (double)L * 8) +
                                  np * (2.0 * F * 16 + 2.0 * N * 8) + nu * 2.0 * num_ch * F * 16);
    }
    if (worst <= budget || cb == 1) break;
    cb = (cb + 1) / 2;
  }
  const long long nchunks = (nblk + cb - 1) / cb;

  // Host tables, one upload: blk_off [nblk + 1], pair_u [pairs] (index into the chunk's page list), pair_page [pairs],
  // the chunks' page lists, and the track frames the signal uses
  const long long npairs = (long long)pt.page.size();
  std::vector<int> cpages;
  std::vector<long long> cp_off{0};
  std::vector<int> pair_u(npairs);
  long long umax = 0, pmax = 0;
  std::vector<int> uidx(num_pages, 0);
  for (long long k = 0; k < nchunks; ++k) {
    const long long b0 = k * cb, nbk = std::min(cb, nblk - b0);
    const size_t first = cpages.size();
    chunk_pages(b0, nbk, tag++, &cpages);
    for (size_t j = first; j < cpages.size(); ++j) uidx[cpages[j]] = (int)(j - first);
    for (int p = pt.blk_off[b0]; p < pt.blk_off[b0 + nbk]; ++p) pair_u[p] = uidx[pt.page[p]];
    cp_off.push_back((long long)cpages.size());
    umax = std::max<long long>(umax, (long long)(cpages.size() - first));
    pmax = std::max<long long>(pmax, pt.blk_off[b0 + nbk] - pt.blk_off[b0]);
  }
  const long long f_base = std::max<long long>(first_sample / hop - 1, 0);
  const long long f_last = (first_sample + num_samples - 1) / hop;
  std::vector<int> tab;
  tab.reserve((size_t)(nblk + 1 + 2 * npairs + cpages.size() + (f_last - f_base + 1)));
  tab.insert(tab.end(), pt.blk_off.begin(), pt.blk_off.end());
  tab.insert(tab.end(), pair_u.begin(), pair_u.end());
  tab.insert(tab.end(), pt.page.begin(), pt.page.end());
  tab.insert(tab.end(), cpages.begin(), cpages.end());
  tab.insert(tab.end(), track + f_base, track + f_last + 1);

  Arena ar(st);
  const int* d_tab = ar.upload(tab.data(), tab.size());
  const int* d_blk_off = d_tab;
  const int* d_pair_u = d_blk_off + nblk + 1;
  const int* d_pair_page = d_pair_u + npairs;
  const int* d_cpages = d_pair_page + npairs;
  const int* d_trk = d_cpages + cpages.size();

  // cuFFT batches: ub pages of filters, pb pairs of inverse transforms (powers of two, so that tracks with similar
  // statistics share the cached plans; the last batch of a chunk is padded)
  const int ub = std::min(pow2_at_least(umax), 64), pb = std::min(pow2_at_least(pmax), 4096);
  const long long ucap = (umax + ub - 1) / ub * ub, pcap = (pmax + pb - 1) / pb * pb;
  const int nbc = (int)cb + nex;
  auto& rp = h->tracked_plans;
  ensure_plans(h, rp, N, L, num_ch, nbc, 2 * num_ch * ub, 2 * pb);
  ForwardStage fwd(h, rp, ar, in, num_samples, num_ch, N, L, ov, nbc);
  double* wp = ar.get<double>((size_t)ub * 2 * num_ch * N);
  cplx* Hw = ar.get<cplx>((size_t)ucap * 2 * num_ch * F);
  cplx* X = ar.get<cplx>((size_t)num_ch * nbc * F);
  cplx* Y = ar.get<cplx>((size_t)pcap * 2 * F);
  double* yseg = ar.get<double>((size_t)pcap * 2 * N);
  constexpr int G = 4, CU = 2;
  for (long long k = 0; k < nchunks; ++k) {
    const long long b0 = k * cb, nbk = std::min(cb, nblk - b0);
    const long long nu = cp_off[k + 1] - cp_off[k];
    const long long np = pt.blk_off[b0 + nbk] - pt.blk_off[b0];
    // filter spectra Hw[u][ear][ch][F] of the pages this chunk references
    for (long long u0 = 0; u0 < nu; u0 += ub) {
      {
        ProfSpan ps(h, EM_PROF_RENDER_STAGE);
        const long long total = (long long)ub * 2 * num_ch * N;
        gather_pad_filters_kernel<<<(unsigned)((total + 255) / 256), 256, 0, st>>>(
            wL, wR, len, num_ch, d_cpages + cp_off[k] + u0, (int)std::min<long long>(ub, nu - u0), ub, N, wp);
        EM_CUDA(cudaGetLastError());
      }
      {
        ProfSpan ps(h, EM_PROF_RENDER_FFT);
        EM_FFT(cufftExecD2Z(rp.filt, wp, reinterpret_cast<cufftDoubleComplex*>(Hw + u0 * 2 * num_ch * F)));
      }
      h->launches += 1;
    }
    fwd.run(b0, nbk, X);
    {
      ProfSpan ps(h, EM_PROF_RENDER_MAC);
      dim3 grid((unsigned)((F + 127) / 128), (unsigned)nbk);
      tracked_mac_kernel<G, CU><<<grid, 128, 0, st>>>(X, Hw, d_blk_off + b0, d_pair_u, num_ch, nbc, F, Y);
      EM_CUDA(cudaGetLastError());
    }
    for (long long q0 = 0; q0 < np; q0 += pb) {
      ProfSpan ps(h, EM_PROF_RENDER_FFT);
      EM_FFT(cufftExecZ2D(rp.inv, reinterpret_cast<cufftDoubleComplex*>(Y + q0 * 2 * F), yseg + q0 * 2 * N));
    }
    {
      ProfSpan ps(h, EM_PROF_RENDER_STAGE);
      const long long total = nbk * L;
      tracked_combine_kernel<<<(unsigned)((total + 255) / 256), 256, 0, st>>>(
          yseg, d_blk_off + b0, d_pair_page, d_trk, f_base, (int)nbk, N, L, ov, b0, first_sample, hop, fade,
          num_samples, skip, out_rows, out);
      EM_CUDA(cudaGetLastError());
    }
    h->launches += 2;
  }
  // stream-ordered: the arena's cudaFreeAsync calls queue behind the work above
}

}  // namespace emagls

using namespace emagls;

extern "C" {

int emagls_binaural_decode_tracked_dev(emagls_handle h, const double* in, long long num_samples, int num_ch,
                                       const double* wL, const double* wR, int len, int num_pages,
                                       const int32_t* track, long long num_frames, int hop, int fade,
                                       long long first_sample, int compensate_delay, double* out) {
  return guarded(h, [&] {
    binaural_decode_tracked_dev(h, in, num_samples, num_ch, wL, wR, len, num_pages, track, num_frames, hop, fade,
                                first_sample, compensate_delay, out);
  });
}

int emagls_binaural_decode_tracked(emagls_handle h, const double* in, long long num_samples, int num_ch,
                                   const double* wL, const double* wR, int len, int num_pages, const int32_t* track,
                                   long long num_frames, int hop, int fade, long long first_sample,
                                   int compensate_delay, double* out) {
  return guarded(h, [&] {
    check_tracked_args(in, num_samples, num_ch, wL, wR, len, num_pages, track, num_frames, hop, fade, first_sample,
                       compensate_delay, out);
    const long long out_rows = num_samples - (compensate_delay ? (len / 2 - 1) : 0);
    cudaStream_t st = h->stream;
    Arena ar(st);
    double* d_in = ar.upload(in, (size_t)num_samples * num_ch);
    double* d_wL = ar.upload(wL, (size_t)len * num_ch * num_pages);
    double* d_wR = ar.upload(wR, (size_t)len * num_ch * num_pages);
    double* d_out = ar.get<double>((size_t)out_rows * 2);
    binaural_decode_tracked_dev(h, d_in, num_samples, num_ch, d_wL, d_wR, len, num_pages, track, num_frames, hop, fade,
                                first_sample, compensate_delay, d_out);
    EM_CUDA(cudaMemcpyAsync(out, d_out, (size_t)out_rows * 2 * sizeof(double), cudaMemcpyDeviceToHost, st));
    EM_CUDA(cudaStreamSynchronize(st));
  });
}

}  // extern "C"
