// Render sessions (contract in include/emagls_cuda.h, DESIGN.md "Render sessions"): the static, bank and SH
// head-tracked renders streamed block by block.  Uniformly partitioned overlap-save with a frequency-domain delay line
// (FDL): FFT size N = 2 B for blocks of B samples, P = ceil(len / B) partitions of B taps.  The spectra of every page and
// partition, H[page][ear][ch][q][F], are built once at creation; every block transforms [previous block | block] of all
// channels into FDL slot k mod P, and per distinct page it needs (a "pair" as in tracked_render.cu)
//     Y[pair][ear][f] = sum_q sum_ch X[slot(k - q)][ch][f] H[page][ear][ch][q][f],
// whose inverse transforms (second half, 1/N) are mixed with the crossfade weights of the tracked render.  SH sessions
// rotate the block first (the rotation stage of sh_tracked_render.cu) and render the rotated block with one page.
// Everything a block needs is allocated at creation: the per-call path allocates nothing, builds no plan and reads no
// device property; its host work is O(frames + pages in the call).
#include <algorithm>
#include <array>
#include <cstdint>
#include <cstring>
#include <deque>
#include <memory>
#include <vector>
#include "render.h"

enum EmStreamKind { EM_STREAM_STATIC = 0, EM_STREAM_BANK = 1, EM_STREAM_SH = 2 };

struct emagls_stream_ctx {
  emagls_ctx* h = nullptr;
  int kind = EM_STREAM_STATIC;
  int num_ch = 0, len = 0, num_pages = 1, order = 0, B = 0, hop = 1, fade = 0;
  int N = 0, F = 0, P = 0;
  int cb = 1;                 // blocks per chunk: capacity of the staging buffers and of one table upload
  int pmax = 1, pcap = 1;     // distinct pages one block can need; pmax rounded up to a power of two
  long long nfr_blk = 0;      // frames one block's rotation stage covers (previous frame included)
  long long nfr_chunk = 0;    // tracker entries one chunk's table holds
  long long T = 0;            // samples processed
  // tracker entries from frame trk_base / rot_base on (the previous frame and the look-ahead)
  std::deque<int32_t> trk;
  long long trk_base = 0;
  std::deque<std::array<double, 9>> rot;
  long long rot_base = 0;
  // device memory (from the handle's pool)
  std::vector<void*> dev;
  emagls::cplx* H = nullptr;  // [pages][2][ch][P][F]
  emagls::cplx* X = nullptr;  // FDL ring [P][ch][F]
  double* seg = nullptr;      // [ch][N]: previous block | this block
  double* prev = nullptr;     // [ch][B]
  emagls::cplx* Y = nullptr;  // [pcap][2][F]
  double* yseg = nullptr;     // [pcap][2][N]
  int* d_tab = nullptr;       // block offsets, pages, track frames of one chunk
  int* d_zero = nullptr;      // page 0 (static and SH sessions)
  double* d_rot = nullptr;    // rotation matrices of one chunk (SH)
  double* Q = nullptr;        // frame rotations of one block (SH)
  int* same = nullptr;
  double* rbuf = nullptr;     // rotated block [ch][B] (SH)
  double* d_in = nullptr;     // host variant: one chunk of input [ch][cb B] and output [2][cb B]
  double* d_out = nullptr;
  // pinned host staging
  double* h_in = nullptr;
  double* h_out = nullptr;
  int* h_tab = nullptr;
  double* h_rot = nullptr;
  size_t tab_cap = 0;
  cudaEvent_t tab_ev = nullptr;  // the last table upload: the pinned table is rewritten only after it has run
  cufftHandle fwd = 0;
  std::vector<cufftHandle> inv;  // inv[j]: 2 * 2^j inverse transforms; all per-block plans share one work area
  // host scratch of a chunk (sized at creation): block offsets into the page list, a block's candidate pages
  std::vector<int> blk_off, cand;
};

namespace emagls {
namespace {

constexpr int ST_MIN_BLOCK = 16, ST_MAX_BLOCK = 8192, ST_MAX_ORDER = 7;
constexpr long long ST_CHUNK_SAMPLES = 16384;   // samples per chunk of the staging buffers

// wp[u][ear][ch][q][N] = taps [q B, (q + 1) B) of page u0 + u, zero-padded to N (pages past nu: zeros)
__global__ void stream_pad_partitions_kernel(const double* __restrict__ wL, const double* __restrict__ wR, int len,
                                             int num_ch, int P, int B, int N, long long u0, int nu, int ub,
                                             double* __restrict__ wp) {
  const long long idx = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (idx >= (long long)ub * 2 * num_ch * P * N) return;
  const int t = (int)(idx % N);
  long long r = idx / N;
  const int q = (int)(r % P);
  r /= P;
  const int ch = (int)(r % num_ch);
  r /= num_ch;
  const int ear = (int)(r & 1), u = (int)(r >> 1);
  const long long tap = (long long)q * B + t;
  const double* w = ear ? wR : wL;
  wp[idx] = (u < nu && t < B && tap < len) ? w[((u0 + u) * num_ch + ch) * len + tap] : 0.0;
}

// seg[ch] = prev[ch] | in[ch][0 .. B), prev[ch] = in[ch][0 .. B)
__global__ void stream_stage_kernel(const double* __restrict__ in, long long ld_in, int num_ch, int B,
                                    double* __restrict__ prev, double* __restrict__ seg) {
  const int idx = blockIdx.x * blockDim.x + threadIdx.x;
  if (idx >= num_ch * B) return;
  const int ch = idx / B, i = idx - ch * B;
  const double x = in[(long long)ch * ld_in + i];
  double* s = seg + (long long)ch * 2 * B;
  s[i] = prev[idx];
  s[B + i] = x;
  prev[idx] = x;
}

// Y[p][ear][f] = sum_q sum_ch X[(slot - q) mod P][ch][f] * H[pages[p]][ear][ch][q][f] for the np pages of one block.
// One thread per (f, group of G pages, blockIdx.y) keeps the G pairs' accumulators in registers, so every FDL value is
// read once per page group; the channel loop is unrolled by two, so 2 (2 G + 1) independent 16-byte loads are in
// flight per thread.  Slots and the page count are uniform over the grid, so no predicate diverges.
template <int G>
__global__ void __launch_bounds__(128)
stream_mac_kernel(const cplx* __restrict__ X, const cplx* __restrict__ H, const int* __restrict__ pages, int np,
                  int num_ch, int P, int F, int slot, cplx* __restrict__ Y) {
  const int f = blockIdx.x * blockDim.x + threadIdx.x;
  if (f >= F) return;
  const int g0 = blockIdx.y * G, n = min(G, np - g0);
  const long long cs = (long long)P * F;          // channel stride of H
  const long long es = (long long)num_ch * cs;    // ear stride of H
  const cplx* hp[G];
  cplx yl[G], yr[G];
#pragma unroll
  for (int q = 0; q < G; ++q) {
    hp[q] = H + (long long)pages[g0 + min(q, n - 1)] * 2 * es + f;
    yl[q] = mk(0.0, 0.0); yr[q] = mk(0.0, 0.0);
  }
  for (int d = 0; d < P; ++d) {
    const int sl = slot - d < 0 ? slot - d + P : slot - d;
    const cplx* x = X + (long long)sl * num_ch * F + f;
    const long long ho = (long long)d * F;
    int ch = 0;
    for (; ch + 2 <= num_ch; ch += 2) {
      cplx xv[2], a[2][G], c[2][G];
#pragma unroll
      for (int u = 0; u < 2; ++u) {
        xv[u] = x[(long long)(ch + u) * F];
#pragma unroll
        for (int q = 0; q < G; ++q)
          if (q < n) {
            a[u][q] = hp[q][(long long)(ch + u) * cs + ho];
            c[u][q] = hp[q][es + (long long)(ch + u) * cs + ho];
          }
      }
#pragma unroll
      for (int u = 0; u < 2; ++u)
#pragma unroll
        for (int q = 0; q < G; ++q)
          if (q < n) { cfma(yl[q], xv[u], a[u][q]); cfma(yr[q], xv[u], c[u][q]); }
    }
    for (; ch < num_ch; ++ch) {
      const cplx xv = x[(long long)ch * F];
#pragma unroll
      for (int q = 0; q < G; ++q)
        if (q < n) {
          cfma(yl[q], xv, hp[q][(long long)ch * cs + ho]);
          cfma(yr[q], xv, hp[q][es + (long long)ch * cs + ho]);
        }
    }
  }
#pragma unroll
  for (int q = 0; q < G; ++q)
    if (q < n) {
      const long long o = (long long)(g0 + q) * 2 * F + f;
      Y[o] = yl[q];
      Y[o + F] = yr[q];
    }
}

// out[ear * ld_out + i] = sum_p weight(pages[p]) * yseg[p][ear][B + i] / N for sample t = t0 + i of one block, with the
// weights of tracked_combine_kernel: weight(page) = (page == c ? g : 0) + (page == a ? 1 - g : 0), g = 1 when a == c.
// trk holds track[f_base ..]; without a track every sample takes page pages[0] with weight 1.
__global__ void stream_combine_kernel(const double* __restrict__ yseg, const int* __restrict__ pages, int np,
                                      const int* __restrict__ trk, long long f_base, long long t0, int B, int hop,
                                      int fade, long long ld_out, double* __restrict__ out) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= B) return;
  const int N = 2 * B;
  int c = pages[0], a = c;
  double g = 1.0;
  if (trk) {
    const long long t = t0 + i, f = t / hop;
    const int ii = (int)(t - f * hop);
    c = trk[f - f_base];
    a = trk[(f > 0 ? f - 1 : 0) - f_base];
    g = (a != c && ii < fade) ? ((double)ii + 0.5) / (double)fade : 1.0;
  }
  double yl = 0.0, yr = 0.0;
  for (int p = 0; p < np; ++p) {
    const int pg = pages[p];
    const double w = (pg == c ? g : 0.0) + (pg == a ? 1.0 - g : 0.0);
    if (w == 0.0) continue;
    const double* y = yseg + (long long)p * 2 * N + B + i;
    yl = fma(w, y[0], yl);
    yr = fma(w, y[N], yr);
  }
  const double inv_n = 1.0 / (double)N;
  out[i] = yl * inv_n;
  out[ld_out + i] = yr * inv_n;
}

int pow2_at_least(long long v) {
  int p = 1;
  while (p < v) p <<= 1;
  return p;
}

template <class T>
T* pool_get(emagls_stream_ctx* s, size_t n) {
  void* p = nullptr;
  emagls_ctx* h = s->h;
  const size_t bytes = std::max<size_t>(n, 1) * sizeof(T);
  cudaError_t e = h->pool ? cudaMallocFromPoolAsync(&p, bytes, h->pool, h->stream) : cudaMallocAsync(&p, bytes, h->stream);
  if (e != cudaSuccess) {
    cudaGetLastError();
    throw Fail{EMAGLS_ERR_CUDA, "render session: cudaMallocAsync(" + std::to_string(bytes) + " B): " +
                                    cudaGetErrorString(e)};
  }
  s->dev.push_back(p);
  return static_cast<T*>(p);
}

template <class T>
T* pinned_get(size_t n) {
  void* p = nullptr;
  EM_CUDA(cudaMallocHost(&p, std::max<size_t>(n, 1) * sizeof(T)));
  return static_cast<T*>(p);
}

void free_session(emagls_stream_ctx* s) {
  emagls_ctx* h = s->h;
  cudaStreamSynchronize(h->stream);
  if (s->fwd) cufftDestroy(s->fwd);
  for (cufftHandle p : s->inv) cufftDestroy(p);
  for (void* p : s->dev) cudaFreeAsync(p, h->stream);
  for (void* p : {(void*)s->h_in, (void*)s->h_out, (void*)s->h_tab, (void*)s->h_rot})
    if (p) cudaFreeHost(p);
  if (s->tab_ev) cudaEventDestroy(s->tab_ev);
  cudaStreamSynchronize(h->stream);
  cudaGetLastError();
  delete s;
}

struct SessionDeleter {
  void operator()(emagls_stream_ctx* s) const { free_session(s); }
};

// Geometry, buffers, plans and the filter spectra of a new session (the caller has checked the arguments)
emagls_stream_ctx* create_session(emagls_ctx* h, int kind, const double* wL, const double* wR, int len, int num_ch,
                                  int num_pages, int order, int block, int hop, int fade) {
  std::unique_ptr<emagls_stream_ctx, SessionDeleter> s(new emagls_stream_ctx());
  s->h = h;
  s->kind = kind;
  s->num_ch = num_ch; s->len = len; s->num_pages = num_pages; s->order = order;
  s->B = block; s->hop = hop; s->fade = fade;
  const int B = block, N = 2 * block, F = block + 1, P = (len + block - 1) / block;
  s->N = N; s->F = F; s->P = P;
  s->cb = (int)std::max<long long>(1, ST_CHUNK_SAMPLES / B);
  // a block intersects at most (B - 1) / hop + 2 frames and may need the frame before its first one
  const long long fr_blk = (B - 1) / hop + 2;
  s->pmax = kind == EM_STREAM_BANK ? (int)std::min<long long>(num_pages, fr_blk + 1) : 1;
  s->pcap = pow2_at_least(s->pmax);
  s->nfr_blk = fr_blk + 1;
  s->nfr_chunk = ((long long)s->cb * B - 1) / hop + 3;
  cudaStream_t st = h->stream;

  s->H = pool_get<cplx>(s.get(), (size_t)num_pages * 2 * num_ch * P * F);
  s->X = pool_get<cplx>(s.get(), (size_t)P * num_ch * F);
  s->seg = pool_get<double>(s.get(), (size_t)num_ch * N);
  s->prev = pool_get<double>(s.get(), (size_t)num_ch * B);
  s->Y = pool_get<cplx>(s.get(), (size_t)s->pcap * 2 * F);
  s->yseg = pool_get<double>(s.get(), (size_t)s->pcap * 2 * N);
  s->d_zero = pool_get<int>(s.get(), 1);
  s->d_in = pool_get<double>(s.get(), (size_t)num_ch * s->cb * B);
  s->d_out = pool_get<double>(s.get(), (size_t)2 * s->cb * B);
  s->tab_cap = kind == EM_STREAM_BANK ? (size_t)(s->cb + 1) + (size_t)s->cb * s->pmax + (size_t)s->nfr_chunk : 1;
  s->d_tab = pool_get<int>(s.get(), s->tab_cap);
  if (kind == EM_STREAM_SH) {
    const int blk = band_offset(order + 1);
    s->d_rot = pool_get<double>(s.get(), (size_t)s->nfr_chunk * 9);
    s->Q = pool_get<double>(s.get(), (size_t)s->nfr_blk * blk);
    s->same = pool_get<int>(s.get(), (size_t)s->nfr_blk);
    s->rbuf = pool_get<double>(s.get(), (size_t)num_ch * B);
    s->h_rot = pinned_get<double>((size_t)s->nfr_chunk * 9);
  }
  s->h_in = pinned_get<double>((size_t)num_ch * s->cb * B);
  s->h_out = pinned_get<double>((size_t)2 * s->cb * B);
  s->h_tab = pinned_get<int>(s->tab_cap);
  EM_CUDA(cudaEventCreateWithFlags(&s->tab_ev, cudaEventDisableTiming));
  EM_CUDA(cudaMemsetAsync(s->X, 0, (size_t)P * num_ch * F * sizeof(cplx), st));
  EM_CUDA(cudaMemsetAsync(s->seg, 0, (size_t)num_ch * N * sizeof(double), st));
  EM_CUDA(cudaMemsetAsync(s->prev, 0, (size_t)num_ch * B * sizeof(double), st));
  EM_CUDA(cudaMemsetAsync(s->Y, 0, (size_t)s->pcap * 2 * F * sizeof(cplx), st));
  EM_CUDA(cudaMemsetAsync(s->d_zero, 0, sizeof(int), st));

  s->blk_off.resize((size_t)s->cb + 1);
  s->cand.reserve((size_t)2 * fr_blk + 2);

  // plans of the per-block path: the forward transform of all channels, and inverse transforms of 2 pairs, 4 pairs, ...
  // up to pcap pairs (a block with np pages runs the smallest that holds them; the transforms of the pairs past np
  // read stale spectra and are never combined).  They run one after the other on the handle's stream, so they share
  // one work area, the largest any of them needs, from the handle's pool.
  int n[1] = {N};
  size_t ws_max = 0;
  auto make_plan = [&](cufftType type, int idist, int odist, int batch) {
    cufftHandle p = 0;
    EM_FFT(cufftCreate(&p));
    EM_FFT(cufftSetAutoAllocation(p, 0));
    size_t ws = 0;
    const cufftResult r = cufftMakePlanMany(p, 1, n, nullptr, 1, idist, nullptr, 1, odist, type, batch, &ws);
    if (r != CUFFT_SUCCESS) {
      cufftDestroy(p);
      EM_FFT(r);
    }
    EM_FFT(cufftSetStream(p, st));
    ws_max = std::max(ws_max, ws);
    return p;
  };
  s->fwd = make_plan(CUFFT_D2Z, N, F, num_ch);
  for (int b = 1; b <= s->pcap; b <<= 1) s->inv.push_back(make_plan(CUFFT_Z2D, F, N, 2 * b));
  {
    void* ws = pool_get<char>(s.get(), ws_max);
    EM_FFT(cufftSetWorkArea(s->fwd, ws));
    for (cufftHandle p : s->inv) EM_FFT(cufftSetWorkArea(p, ws));
  }

  // filter spectra: pages in batches whose padded partitions stay within 256 MB
  {
    Arena ar(st);
    const size_t wn = (size_t)len * num_ch * num_pages;
    const double* d_wL = ar.upload(wL, wn);
    const double* d_wR = ar.upload(wR, wn);
    const double per_page = 2.0 * num_ch * P * N * sizeof(double);
    const int ub = (int)std::max(1.0, std::min((double)num_pages, 268435456.0 / per_page));
    double* wp = ar.get<double>((size_t)ub * 2 * num_ch * P * N);
    // full batches of ub pages, and a plan of exactly the remaining pages for the last one, so that no transform
    // writes past the nu pages that H holds there
    struct PlanGuard {
      cufftHandle full = 0, tail = 0;
      ~PlanGuard() { if (full) cufftDestroy(full); if (tail) cufftDestroy(tail); }
    } plans;
    EM_FFT(cufftPlanMany(&plans.full, 1, n, nullptr, 1, N, nullptr, 1, F, CUFFT_D2Z, ub * 2 * num_ch * P));
    EM_FFT(cufftSetStream(plans.full, st));
    if (const int rest = num_pages % ub; rest != 0) {
      EM_FFT(cufftPlanMany(&plans.tail, 1, n, nullptr, 1, N, nullptr, 1, F, CUFFT_D2Z, rest * 2 * num_ch * P));
      EM_FFT(cufftSetStream(plans.tail, st));
    }
    for (long long u0 = 0; u0 < num_pages; u0 += ub) {
      const int nu = (int)std::min<long long>(ub, num_pages - u0);
      const cufftHandle pw = nu == ub ? plans.full : plans.tail;
      {
        ProfSpan ps(h, EM_PROF_RENDER_STAGE);
        const long long total = (long long)ub * 2 * num_ch * P * N;
        stream_pad_partitions_kernel<<<(unsigned)((total + 255) / 256), 256, 0, st>>>(d_wL, d_wR, len, num_ch, P, B, N,
                                                                                      u0, nu, ub, wp);
        EM_CUDA(cudaGetLastError());
      }
      {
        ProfSpan ps(h, EM_PROF_RENDER_FFT);
        EM_FFT(cufftExecD2Z(pw, wp, reinterpret_cast<cufftDoubleComplex*>(s->H + u0 * 2 * num_ch * P * F)));
      }
      h->launches += 2;
    }
    EM_CUDA(cudaStreamSynchronize(st));   // the plan is destroyed and the arena freed behind the work
  }
  EM_CUDA(cudaStreamSynchronize(st));
  return s.release();
}

// The checks of a process call; nothing of the session changes before they pass
void check_process(const emagls_stream_ctx* s, const double* in, long long num_samples, const int32_t* track,
                   const double* rotations, long long num_new, const double* out) {
  EM_REQUIRE(in && out, "null argument");
  EM_REQUIRE(num_samples > 0 && num_samples % s->B == 0, "num_samples must be a positive multiple of the block");
  EM_REQUIRE(num_new >= 0, "num_new_frames must be >= 0");
  const long long f_need = (s->T + num_samples - 1) / s->hop;
  if (s->kind == EM_STREAM_STATIC) {
    EM_REQUIRE(!track && !rotations && num_new == 0, "a static session takes no tracker entries");
    return;
  }
  if (s->kind == EM_STREAM_BANK) {
    EM_REQUIRE(!rotations, "a bank session takes a track of pages, not rotations");
    EM_REQUIRE(track || num_new == 0, "null track");
    for (long long j = 0; j < num_new; ++j)
      EM_REQUIRE(track[j] >= 0 && track[j] < s->num_pages, "track entry outside [0, num_pages)");
    EM_REQUIRE(s->trk_base + (long long)s->trk.size() + num_new > f_need, "track does not cover the call");
  } else {
    EM_REQUIRE(!track, "an SH session takes rotations, not a track of pages");
    EM_REQUIRE(rotations || num_new == 0, "null rotations");
    EM_REQUIRE(s->rot_base + (long long)s->rot.size() + num_new > f_need, "rotations do not cover the call");
  }
}

void append_entries(emagls_stream_ctx* s, const int32_t* track, const double* rotations, long long num_new) {
  if (s->kind == EM_STREAM_BANK) {
    s->trk.insert(s->trk.end(), track, track + num_new);
  } else if (s->kind == EM_STREAM_SH) {
    for (long long j = 0; j < num_new; ++j) {
      std::array<double, 9> r;
      std::memcpy(r.data(), rotations + 9 * j, sizeof(r));
      s->rot.push_back(r);
    }
  }
}

// Drop the entries no later block needs: blocks from sample T on use frame T / hop - 1 at the earliest
void trim_entries(emagls_stream_ctx* s) {
  const long long keep = std::max<long long>(s->T / s->hop - 1, 0);
  while (s->trk_base < keep && !s->trk.empty()) { s->trk.pop_front(); ++s->trk_base; }
  while (s->rot_base < keep && !s->rot.empty()) { s->rot.pop_front(); ++s->rot_base; }
}

// Blocks [T, T + nb B) of the stream: in[ch * ld_in + i] (i < nb B) -> out[ear * ld_out + i]
void run_chunk(emagls_stream_ctx* s, const double* in, long long ld_in, int nb, double* out, long long ld_out) {
  emagls_ctx* h = s->h;
  cudaStream_t st = h->stream;
  const int B = s->B, F = s->F, P = s->P, num_ch = s->num_ch;
  const long long t_first = s->T, t_last = s->T + (long long)nb * B - 1;
  const long long f_first = std::max<long long>(t_first / s->hop - 1, 0), f_last = t_last / s->hop;

  // per block: its distinct pages (sorted: the combine sums them in a fixed order whatever the call split), by the
  // rule of build_pairs in tracked_render.cu; one upload of the chunk's table
  std::vector<int>& blk_off = s->blk_off;
  std::fill(blk_off.begin(), blk_off.begin() + nb + 1, 0);
  if (s->kind == EM_STREAM_BANK || s->kind == EM_STREAM_SH) {
    EM_CUDA(cudaEventSynchronize(s->tab_ev));
  }
  if (s->kind == EM_STREAM_BANK) {
    int* tab = s->h_tab;
    int* pg = tab + (nb + 1);
    int np_total = 0;
    std::vector<int>& cand = s->cand;
    for (int b = 0; b < nb; ++b) {
      tab[b] = np_total;
      blk_off[b] = np_total;
      const long long t_lo = t_first + (long long)b * B, t_hi = t_lo + B - 1;
      cand.clear();
      for (long long f = t_lo / s->hop; f <= t_hi / s->hop; ++f) {
        cand.push_back(s->trk[f - s->trk_base]);
        if (f > 0 && s->fade > 0 && f * s->hop + s->fade - 1 >= t_lo) cand.push_back(s->trk[f - 1 - s->trk_base]);
      }
      std::sort(cand.begin(), cand.end());
      cand.erase(std::unique(cand.begin(), cand.end()), cand.end());
      for (int p : cand) pg[np_total++] = p;
    }
    tab[nb] = np_total;
    blk_off[nb] = np_total;
    int* tk = pg + np_total;
    for (long long f = f_first; f <= f_last; ++f) tk[f - f_first] = s->trk[f - s->trk_base];
    const size_t n_tab = (size_t)(nb + 1) + np_total + (size_t)(f_last - f_first + 1);
    EM_CUDA(cudaMemcpyAsync(s->d_tab, tab, n_tab * sizeof(int), cudaMemcpyHostToDevice, st));
    EM_CUDA(cudaEventRecord(s->tab_ev, st));
  } else if (s->kind == EM_STREAM_SH) {
    for (long long f = f_first; f <= f_last; ++f)
      std::memcpy(s->h_rot + 9 * (f - f_first), s->rot[f - s->rot_base].data(), 9 * sizeof(double));
    EM_CUDA(cudaMemcpyAsync(s->d_rot, s->h_rot, (size_t)(f_last - f_first + 1) * 9 * sizeof(double),
                            cudaMemcpyHostToDevice, st));
    EM_CUDA(cudaEventRecord(s->tab_ev, st));
  }
  const int* d_pages = s->d_tab + (nb + 1);
  const int* d_trk = d_pages + blk_off[nb];

  for (int b = 0; b < nb; ++b) {
    const long long k = s->T / B, t_lo = s->T;
    const int slot = (int)(k % P);
    const double* src = in + (long long)b * B;
    long long ld = ld_in;
    if (s->kind == EM_STREAM_SH) {
      ProfSpan ps(h, EM_PROF_RENDER_STAGE);
      const long long fb = std::max<long long>(t_lo / s->hop - 1, 0), fh = (t_lo + B - 1) / s->hop;
      launch_frame_rotations(h, s->d_rot, f_first, fb, fh - fb + 1, s->order, s->Q, s->same);
      launch_sh_track_rotate(h, in, ld_in, (long long)b * B, B, s->order, s->Q, s->same, fb, t_first, s->hop, s->fade,
                             s->rbuf);
      h->launches += 2;
      src = s->rbuf;
      ld = B;
    }
    {
      ProfSpan ps(h, EM_PROF_RENDER_STAGE);
      stream_stage_kernel<<<(num_ch * B + 255) / 256, 256, 0, st>>>(src, ld, num_ch, B, s->prev, s->seg);
      EM_CUDA(cudaGetLastError());
    }
    {
      ProfSpan ps(h, EM_PROF_RENDER_FFT);
      EM_FFT(cufftExecD2Z(s->fwd, s->seg, reinterpret_cast<cufftDoubleComplex*>(s->X + (long long)slot * num_ch * F)));
    }
    const bool bank = s->kind == EM_STREAM_BANK;
    const int np = bank ? blk_off[b + 1] - blk_off[b] : 1;
    const int* pages = bank ? d_pages + blk_off[b] : s->d_zero;
    constexpr int G = 4;
    {
      ProfSpan ps(h, EM_PROF_RENDER_MAC);
      dim3 grid((unsigned)((F + 127) / 128), (unsigned)((np + G - 1) / G));
      stream_mac_kernel<G><<<grid, 128, 0, st>>>(s->X, s->H, pages, np, num_ch, P, F, slot, s->Y);
      EM_CUDA(cudaGetLastError());
    }
    {
      ProfSpan ps(h, EM_PROF_RENDER_FFT);
      int j = 0;
      while ((1 << j) < np) ++j;
      EM_FFT(cufftExecZ2D(s->inv[j], reinterpret_cast<cufftDoubleComplex*>(s->Y), s->yseg));
    }
    {
      ProfSpan ps(h, EM_PROF_RENDER_STAGE);
      stream_combine_kernel<<<(B + 127) / 128, 128, 0, st>>>(s->yseg, pages, np, bank ? d_trk : nullptr, f_first,
                                                             t_lo, B, s->hop, s->fade, ld_out, out + (long long)b * B);
      EM_CUDA(cudaGetLastError());
    }
    h->launches += 5;
    s->T += B;
  }
}

void process(emagls_stream_ctx* s, const double* in, long long num_samples, const int32_t* track,
             const double* rotations, long long num_new, double* out, bool dev) {
  check_process(s, in, num_samples, track, rotations, num_new, out);
  append_entries(s, track, rotations, num_new);
  emagls_ctx* h = s->h;
  cudaStream_t st = h->stream;
  const long long cs = (long long)s->cb * s->B;
  for (long long c0 = 0; c0 < num_samples; c0 += cs) {
    const long long cn = std::min(cs, num_samples - c0);
    const int nb = (int)(cn / s->B);
    if (dev) {
      run_chunk(s, in + c0, num_samples, nb, out + c0, num_samples);
    } else {
      for (int ch = 0; ch < s->num_ch; ++ch)
        std::memcpy(s->h_in + (long long)ch * cn, in + (long long)ch * num_samples + c0, (size_t)cn * sizeof(double));
      EM_CUDA(cudaMemcpyAsync(s->d_in, s->h_in, (size_t)s->num_ch * cn * sizeof(double), cudaMemcpyHostToDevice, st));
      run_chunk(s, s->d_in, cn, nb, s->d_out, cn);
      EM_CUDA(cudaMemcpyAsync(s->h_out, s->d_out, (size_t)2 * cn * sizeof(double), cudaMemcpyDeviceToHost, st));
      EM_CUDA(cudaStreamSynchronize(st));
      for (int ear = 0; ear < 2; ++ear)
        std::memcpy(out + (long long)ear * num_samples + c0, s->h_out + (long long)ear * cn, (size_t)cn * sizeof(double));
    }
    trim_entries(s);
  }
}

void check_create(const double* wL, const double* wR, int len, int num_ch, int num_pages, int block, int hop, int fade,
                  const emagls_render_stream* out) {
  EM_REQUIRE(wL && wR && out, "null argument");
  EM_REQUIRE(len > 0 && num_ch > 0 && num_pages > 0, "empty filters");
  EM_REQUIRE(block >= ST_MIN_BLOCK && block <= ST_MAX_BLOCK, "block must lie in [16, 8192]");
  EM_REQUIRE(hop >= 1, "hop must be >= 1");
  EM_REQUIRE(fade >= 0 && fade <= hop, "fade must lie in [0, hop]");
}

void open_session(emagls_ctx* h, emagls_stream_ctx* s, emagls_render_stream* out) {
  h->render_streams.push_back(s);
  *out = s;
}

}  // namespace

void destroy_render_streams(emagls_ctx* h) {
  for (emagls_stream_ctx* s : h->render_streams) free_session(s);
  h->render_streams.clear();
}

}  // namespace emagls

using namespace emagls;

extern "C" {

int emagls_render_stream_create(emagls_handle h, const double* wL, const double* wR, int len, int num_ch,
                                int num_pages, int block, int hop, int fade, emagls_render_stream* out) {
  if (out) *out = nullptr;
  return guarded(h, [&] {
    check_create(wL, wR, len, num_ch, num_pages, block, hop, fade, out);
    const int kind = num_pages == 1 ? EM_STREAM_STATIC : EM_STREAM_BANK;
    open_session(h, create_session(h, kind, wL, wR, len, num_ch, num_pages, 0, block, hop, fade), out);
  });
}

int emagls_render_stream_create_sh(emagls_handle h, const double* wL, const double* wR, int len, int order,
                                   int block, int hop, int fade, emagls_render_stream* out) {
  if (out) *out = nullptr;
  return guarded(h, [&] {
    EM_REQUIRE(order >= 0 && order <= ST_MAX_ORDER, "order must lie in [0, 7]");
    const int C = (order + 1) * (order + 1);
    check_create(wL, wR, len, C, 1, block, hop, fade, out);
    open_session(h, create_session(h, EM_STREAM_SH, wL, wR, len, C, 1, order, block, hop, fade), out);
  });
}

int emagls_render_stream_process(emagls_render_stream s, const double* in, long long num_samples,
                                 const int32_t* track, const double* rotations, long long num_new_frames,
                                 double* out) {
  if (!s) return EMAGLS_ERR_INVALID;
  return guarded(s->h, [&] { process(s, in, num_samples, track, rotations, num_new_frames, out, false); });
}

int emagls_render_stream_process_dev(emagls_render_stream s, const double* in, long long num_samples,
                                     const int32_t* track, const double* rotations, long long num_new_frames,
                                     double* out) {
  if (!s) return EMAGLS_ERR_INVALID;
  return guarded(s->h, [&] { process(s, in, num_samples, track, rotations, num_new_frames, out, true); });
}

int emagls_render_stream_destroy(emagls_render_stream s) {
  if (!s) return EMAGLS_ERR_INVALID;
  emagls_ctx* h = s->h;
  return guarded(h, [&] {
    auto& v = h->render_streams;
    auto it = std::find(v.begin(), v.end(), s);
    EM_REQUIRE(it != v.end(), "not an open render session of this handle");
    v.erase(it);
    free_session(s);
  });
}

}  // extern "C"
