// Render sessions (contract in include/emagls_cuda.h, DESIGN.md "Render sessions"): the static, bank and SH
// head-tracked renders streamed block by block, for L listeners (seats) who hear one shared input stream with their own
// tracker entries.  Uniformly partitioned overlap-save with a frequency-domain delay line (FDL): FFT size N = 2 B for
// blocks of B samples, P = ceil(len / B) partitions of B taps.  The spectra of every page and partition,
// H[page][ear][ch][q][F], are built once at creation; every block transforms [previous block | block] of all channels
// into FDL slot k mod P, and per distinct page it needs (a "pair" as in tracked_render.cu)
//     Y[pair][ear][f] = sum_q sum_ch X[slot(k - q)][ch][f] H[page][ear][ch][q][f],
// whose inverse transforms (second half, 1/N) are mixed per listener with the crossfade weights of the tracked render.
// A bank session's listeners share the stage, the FDL and the pairs: a block renders the union of the pages its
// listeners need, once.  SH sessions rotate the block per listener first (the rotation stage of sh_tracked_render.cu),
// keep an FDL per listener and render each rotated block with the one page.  Either way a block takes the same number
// of launches whatever L.  Everything a block needs is allocated at creation: the per-call path allocates nothing,
// builds no plan and reads no device property; its host work is O(L frames + pages in the call).
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
  int nl = 1;                 // listeners (seats); they share the input stream
  int xch = 0;                // channels of the FDL: num_ch (static, bank) or nl num_ch (SH: one FDL per listener)
  int N = 0, F = 0, P = 0;
  int cb = 1;                 // blocks per chunk: capacity of the staging buffers and of one table upload
  int pmax = 1;               // distinct pages one listener's block can need
  int pcap = 1;               // pairs Y and yseg hold: pow2(min(num_pages, nl pmax)) (bank), nl (SH), 1 (static)
  long long fr_blk = 0;       // frames one block's samples fall in
  long long nfr_blk = 0;      // frames one block's rotation stage covers (previous frame included)
  long long nfr_chunk = 0;    // tracker entries per listener one chunk's table holds
  long long T = 0;            // samples processed
  // tracker entries from frame trk_base / rot_base on (the previous frame and the look-ahead), nl per frame:
  // trk[(f - trk_base) nl + l] is listener l's page of frame f
  std::deque<int32_t> trk;
  long long trk_base = 0;
  std::deque<std::array<double, 9>> rot;
  long long rot_base = 0;
  // device memory (from the handle's pool)
  std::vector<void*> dev;
  emagls::cplx* H = nullptr;  // [pages][2][ch][P][F]
  emagls::cplx* X = nullptr;  // FDL ring [P][xch][F]
  double* seg = nullptr;      // [xch][N]: previous block | this block
  double* prev = nullptr;     // [xch][B]
  emagls::cplx* Y = nullptr;  // [pcap][2][F]
  double* yseg = nullptr;     // [pcap][2][N]
  int* d_tab = nullptr;       // bank: the combine's pair slots and the union pages of one chunk
  int* d_zero = nullptr;      // page 0 (static and SH sessions)
  double* d_rot = nullptr;    // rotation matrices of one chunk [nl][frames][9] (SH)
  double* Q = nullptr;        // frame rotations of one block [nl][nfr_blk][band_offset(order + 1)] (SH)
  int* same = nullptr;        // [nl][nfr_blk]
  double* rbuf = nullptr;     // rotated block [nl][ch][B] (SH)
  double* d_in = nullptr;     // host variant: one chunk of input [ch][cb B] and output [nl][2][cb B]
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
  // host scratch of a chunk (sized at creation): block offsets into the union pages and the slot table, a block's
  // union, and the union slot of every page (-1: not in the block's union)
  std::vector<int> blk_off, cmb_off, uni, mark;
};

namespace emagls {
namespace {

constexpr int ST_MIN_BLOCK = 16, ST_MAX_BLOCK = 8192, ST_MAX_ORDER = 7, ST_MAX_LISTENERS = 4096;
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

// seg[ch] = prev[ch] | in[ch][0 .. B), prev[ch] = in[ch][0 .. B).  num_ch B reaches 2^31 with many SH listeners.
__global__ void stream_stage_kernel(const double* __restrict__ in, long long ld_in, int num_ch, int B,
                                    double* __restrict__ prev, double* __restrict__ seg) {
  const long long idx = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (idx >= (long long)num_ch * B) return;
  const long long ch = idx / B, i = idx - ch * B;
  const double x = in[ch * ld_in + i];
  double* s = seg + ch * 2 * B;
  s[i] = prev[idx];
  s[B + i] = x;
  prev[idx] = x;
}

// Y[p][ear][f] = sum_q sum_ch X[(slot - q) mod P][ch][f] * H[pages[p]][ear][ch][q][f] for the np pages of one block.
// One thread per (f, group of G pages, blockIdx.y) keeps the G pairs' accumulators in registers, so every FDL value is
// read once per page group; the channel loop is unrolled by two, so 2 (2 G + 1) independent 16-byte loads are in
// flight per thread.  Slots and the page count are uniform over the grid, so no predicate diverges.  blockIdx.z
// selects a listener's FDL (SH sessions): X + z num_ch F within each slot of xs values, and Y + z np 2 F.
template <int G>
__global__ void __launch_bounds__(128)
stream_mac_kernel(const cplx* __restrict__ X, long long xs, const cplx* __restrict__ H, const int* __restrict__ pages,
                  int np, int num_ch, int P, int F, int slot, cplx* __restrict__ Y) {
  const int f = blockIdx.x * blockDim.x + threadIdx.x;
  if (f >= F) return;
  const long long xz = (long long)blockIdx.z * num_ch * F;   // this listener's FDL within a slot
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
    const cplx* x = X + xz + sl * xs + f;
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
      const long long o = ((long long)blockIdx.z * np + g0 + q) * 2 * F + f;
      Y[o] = yl[q];
      Y[o + F] = yr[q];
    }
}

// out[(2 l + ear) ld_out + i] = sum over pages of weight(page) yseg[slot(page)][ear][B + i] / N for sample t = t0 + i of
// one block and listener l = blockIdx.y, with the weights of tracked_combine_kernel: c = track[f], a = track[max(f-1, 0)],
// weight(page) = (page == c ? g : 0) + (page == a ? 1 - g : 0), g = 1 when a == c.  slots[(l nfb + f - fb0) 2 + {0, 1}]
// are the union slots of a and c (the union is in ascending page order, so the two pages are added in that order, as
// the one-listener sum over the block's sorted pages; -1 marks an a outside the union, whose weight is 0 then).
// Without slots (static and SH sessions) listener l takes pair l with weight 1.
__global__ void stream_combine_kernel(const double* __restrict__ yseg, const int* __restrict__ slots, long long fb0,
                                      int nfb, long long t0, int B, int hop, int fade, long long ld_out,
                                      double* __restrict__ out) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= B) return;
  const int l = blockIdx.y, N = 2 * B;
  int sa = l, sc = l;
  double g = 1.0;
  if (slots) {
    const long long t = t0 + i, f = t / hop;
    const int ii = (int)(t - f * hop);
    const int* e = slots + ((long long)l * nfb + (f - fb0)) * 2;
    sa = e[0];
    sc = e[1];
    g = (sa != sc && ii < fade) ? ((double)ii + 0.5) / (double)fade : 1.0;
  }
  // (page, weight) in ascending page order; a == c takes g + (1 - g) = 1
  int p0 = sc, p1 = -1;
  double w0 = 1.0, w1 = 0.0;
  if (sa != sc) {
    if (sa < sc) { p0 = sa; w0 = 1.0 - g; p1 = sc; w1 = g; }
    else         { p0 = sc; w0 = g;       p1 = sa; w1 = 1.0 - g; }
  }
  double yl = 0.0, yr = 0.0;
  if (w0 != 0.0) {
    const double* y = yseg + (long long)p0 * 2 * N + B + i;
    yl = fma(w0, y[0], yl);
    yr = fma(w0, y[N], yr);
  }
  if (w1 != 0.0) {
    const double* y = yseg + (long long)p1 * 2 * N + B + i;
    yl = fma(w1, y[0], yl);
    yr = fma(w1, y[N], yr);
  }
  const double inv_n = 1.0 / (double)N;
  double* o = out + 2 * l * ld_out + i;
  o[0] = yl * inv_n;
  o[ld_out] = yr * inv_n;
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
                                  int num_pages, int order, int nl, int block, int hop, int fade) {
  std::unique_ptr<emagls_stream_ctx, SessionDeleter> s(new emagls_stream_ctx());
  s->h = h;
  s->kind = kind;
  s->num_ch = num_ch; s->len = len; s->num_pages = num_pages; s->order = order; s->nl = nl;
  s->B = block; s->hop = hop; s->fade = fade;
  const int B = block, N = 2 * block, F = block + 1, P = (len + block - 1) / block;
  s->N = N; s->F = F; s->P = P;
  // the staging buffers hold about ST_CHUNK_SAMPLES samples of every listener's output
  s->cb = (int)std::max<long long>(1, ST_CHUNK_SAMPLES / ((long long)B * nl));
  // a block intersects at most (B - 1) / hop + 2 frames and may need the frame before its first one
  const long long fr_blk = (B - 1) / hop + 2;
  s->fr_blk = fr_blk;
  s->pmax = kind == EM_STREAM_BANK ? (int)std::min<long long>(num_pages, fr_blk + 1) : 1;
  s->pcap = kind == EM_STREAM_BANK ? pow2_at_least(std::min<long long>(num_pages, (long long)nl * s->pmax))
                                   : kind == EM_STREAM_SH ? nl : 1;
  s->xch = kind == EM_STREAM_SH ? nl * num_ch : num_ch;
  s->nfr_blk = fr_blk + 1;
  s->nfr_chunk = ((long long)s->cb * B - 1) / hop + 3;
  const long long xch = s->xch;
  cudaStream_t st = h->stream;

  s->H = pool_get<cplx>(s.get(), (size_t)num_pages * 2 * num_ch * P * F);
  s->X = pool_get<cplx>(s.get(), (size_t)P * xch * F);
  s->seg = pool_get<double>(s.get(), (size_t)xch * N);
  s->prev = pool_get<double>(s.get(), (size_t)xch * B);
  s->Y = pool_get<cplx>(s.get(), (size_t)s->pcap * 2 * F);
  s->yseg = pool_get<double>(s.get(), (size_t)s->pcap * 2 * N);
  s->d_zero = pool_get<int>(s.get(), 1);
  s->d_in = pool_get<double>(s.get(), (size_t)num_ch * s->cb * B);
  s->d_out = pool_get<double>(s.get(), (size_t)2 * nl * s->cb * B);
  // bank table of one chunk: per block, 2 pair slots per listener and frame, and the union of pages
  s->tab_cap = kind == EM_STREAM_BANK
                   ? (size_t)s->cb * ((size_t)2 * nl * fr_blk + (size_t)std::min<long long>(num_pages, (long long)nl * s->pmax))
                   : 1;
  s->d_tab = pool_get<int>(s.get(), s->tab_cap);
  if (kind == EM_STREAM_SH) {
    const int blk = band_offset(order + 1);
    s->d_rot = pool_get<double>(s.get(), (size_t)nl * s->nfr_chunk * 9);
    s->Q = pool_get<double>(s.get(), (size_t)nl * s->nfr_blk * blk);
    s->same = pool_get<int>(s.get(), (size_t)nl * s->nfr_blk);
    s->rbuf = pool_get<double>(s.get(), (size_t)xch * B);
    s->h_rot = pinned_get<double>((size_t)nl * s->nfr_chunk * 9);
  }
  s->h_in = pinned_get<double>((size_t)num_ch * s->cb * B);
  s->h_out = pinned_get<double>((size_t)2 * nl * s->cb * B);
  s->h_tab = pinned_get<int>(s->tab_cap);
  EM_CUDA(cudaEventCreateWithFlags(&s->tab_ev, cudaEventDisableTiming));
  EM_CUDA(cudaMemsetAsync(s->X, 0, (size_t)P * xch * F * sizeof(cplx), st));
  EM_CUDA(cudaMemsetAsync(s->seg, 0, (size_t)xch * N * sizeof(double), st));
  EM_CUDA(cudaMemsetAsync(s->prev, 0, (size_t)xch * B * sizeof(double), st));
  EM_CUDA(cudaMemsetAsync(s->Y, 0, (size_t)s->pcap * 2 * F * sizeof(cplx), st));
  EM_CUDA(cudaMemsetAsync(s->d_zero, 0, sizeof(int), st));

  s->blk_off.resize((size_t)s->cb + 1);
  s->cmb_off.resize((size_t)s->cb + 1);
  if (kind == EM_STREAM_BANK) {
    s->uni.reserve((size_t)std::min<long long>(num_pages, (long long)nl * s->pmax));
    s->mark.assign((size_t)num_pages, -1);
  }

  // plans of the per-block path: the forward transform of all FDL channels, and inverse transforms of the pairs.  A
  // bank session has plans of 2 pairs, 4 pairs, ... up to pcap pairs (a block with np pages runs the smallest that
  // holds them; the transforms of the pairs past np read stale spectra and are never combined); the others one plan
  // of exactly pcap pairs.  They run one after the other on the handle's stream, so they share one work area, the
  // largest any of them needs, from the handle's pool.
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
  s->fwd = make_plan(CUFFT_D2Z, N, F, xch);
  if (kind == EM_STREAM_BANK) {
    for (int b = 1; b <= s->pcap; b <<= 1) s->inv.push_back(make_plan(CUFFT_Z2D, F, N, 2 * b));
  } else {
    s->inv.push_back(make_plan(CUFFT_Z2D, F, N, 2 * s->pcap));
  }
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
    for (long long j = 0; j < num_new * s->nl; ++j)
      EM_REQUIRE(track[j] >= 0 && track[j] < s->num_pages, "track entry outside [0, num_pages)");
    EM_REQUIRE(s->trk_base + (long long)s->trk.size() / s->nl + num_new > f_need, "track does not cover the call");
  } else {
    EM_REQUIRE(!track, "an SH session takes rotations, not a track of pages");
    EM_REQUIRE(rotations || num_new == 0, "null rotations");
    EM_REQUIRE(s->rot_base + (long long)s->rot.size() / s->nl + num_new > f_need, "rotations do not cover the call");
  }
}

// Entries arrive per listener ([num_new x nl], column-major) and are kept per frame (nl consecutive entries)
void append_entries(emagls_stream_ctx* s, const int32_t* track, const double* rotations, long long num_new) {
  const int L = s->nl;
  for (long long j = 0; j < num_new; ++j)
    for (int l = 0; l < L; ++l) {
      if (s->kind == EM_STREAM_BANK) {
        s->trk.push_back(track[(long long)l * num_new + j]);
      } else if (s->kind == EM_STREAM_SH) {
        std::array<double, 9> r;
        std::memcpy(r.data(), rotations + 9 * ((long long)l * num_new + j), sizeof(r));
        s->rot.push_back(r);
      }
    }
}

// Drop the entries no later block needs: blocks from sample T on use frame T / hop - 1 at the earliest
void trim_entries(emagls_stream_ctx* s) {
  const long long keep = std::max<long long>(s->T / s->hop - 1, 0);
  const size_t L = (size_t)s->nl;
  while (s->trk_base < keep && !s->trk.empty()) { s->trk.erase(s->trk.begin(), s->trk.begin() + L); ++s->trk_base; }
  while (s->rot_base < keep && !s->rot.empty()) { s->rot.erase(s->rot.begin(), s->rot.begin() + L); ++s->rot_base; }
}

// Blocks [T, T + nb B) of the stream: in[ch * ld_in + i] (i < nb B) -> out[(2 l + ear) * ld_out + i]
void run_chunk(emagls_stream_ctx* s, const double* in, long long ld_in, int nb, double* out, long long ld_out) {
  emagls_ctx* h = s->h;
  cudaStream_t st = h->stream;
  const int B = s->B, F = s->F, P = s->P, num_ch = s->num_ch, L = s->nl, hop = s->hop;
  const long long t_first = s->T, t_last = s->T + (long long)nb * B - 1;
  const long long f_first = std::max<long long>(t_first / hop - 1, 0), f_last = t_last / hop;
  const long long nfr_c = f_last - f_first + 1;

  // bank: per block, the union of the pages its listeners need, by the rule of build_pairs in tracked_render.cu, in
  // ascending page order (so the combine adds a listener's pages in the order of a one-listener session, whatever the
  // other listeners or the call split), and per listener and frame of the block the union slots of pages a and c;
  // one upload of the chunk's table
  std::vector<int>& blk_off = s->blk_off;
  std::vector<int>& cmb_off = s->cmb_off;
  std::fill(blk_off.begin(), blk_off.begin() + nb + 1, 0);
  if (s->kind == EM_STREAM_BANK || s->kind == EM_STREAM_SH) {
    EM_CUDA(cudaEventSynchronize(s->tab_ev));
  }
  auto blk_frames = [&](int b, long long& f0, int& nfb) {
    const long long t_lo = t_first + (long long)b * B;
    f0 = t_lo / hop;
    nfb = (int)((t_lo + B - 1) / hop - f0 + 1);
  };
  if (s->kind == EM_STREAM_BANK) {
    const auto page = [&](long long f, int l) { return s->trk[(size_t)((f - s->trk_base) * L + l)]; };
    std::vector<int>& uni = s->uni;
    std::vector<int>& mark = s->mark;
    const auto add = [&](int p) {
      if (mark[p] < 0) { mark[p] = 0; uni.push_back(p); }
    };
    int* tab = s->h_tab;
    int n_cmb = 0;
    for (int b = 0; b < nb; ++b) {
      long long f0;
      int nfb;
      blk_frames(b, f0, nfb);
      cmb_off[b] = n_cmb;
      n_cmb += 2 * L * nfb;
    }
    cmb_off[nb] = n_cmb;
    int* pg = tab + n_cmb;
    int np_total = 0;
    for (int b = 0; b < nb; ++b) {
      const long long t_lo = t_first + (long long)b * B;
      long long f0;
      int nfb;
      blk_frames(b, f0, nfb);
      blk_off[b] = np_total;
      uni.clear();
      for (int l = 0; l < L; ++l)
        for (long long f = f0; f < f0 + nfb; ++f) {
          add(page(f, l));
          if (f > 0 && s->fade > 0 && f * hop + s->fade - 1 >= t_lo) add(page(f - 1, l));
        }
      std::sort(uni.begin(), uni.end());
      for (int k = 0; k < (int)uni.size(); ++k) {
        mark[uni[k]] = k;
        pg[np_total++] = uni[k];
      }
      int* e = tab + cmb_off[b];
      for (int l = 0; l < L; ++l)
        for (long long f = f0; f < f0 + nfb; ++f, e += 2) {
          const int c = page(f, l);
          e[0] = mark[f > 0 ? page(f - 1, l) : c];
          e[1] = mark[c];
        }
      for (int p : uni) mark[p] = -1;
    }
    blk_off[nb] = np_total;
    EM_CUDA(cudaMemcpyAsync(s->d_tab, tab, (size_t)(n_cmb + np_total) * sizeof(int), cudaMemcpyHostToDevice, st));
    EM_CUDA(cudaEventRecord(s->tab_ev, st));
  } else if (s->kind == EM_STREAM_SH) {
    for (int l = 0; l < L; ++l)
      for (long long f = f_first; f <= f_last; ++f)
        std::memcpy(s->h_rot + 9 * (l * nfr_c + f - f_first), s->rot[(size_t)((f - s->rot_base) * L + l)].data(),
                    9 * sizeof(double));
    EM_CUDA(cudaMemcpyAsync(s->d_rot, s->h_rot, (size_t)L * nfr_c * 9 * sizeof(double), cudaMemcpyHostToDevice, st));
    EM_CUDA(cudaEventRecord(s->tab_ev, st));
  }

  for (int b = 0; b < nb; ++b) {
    const long long k = s->T / B, t_lo = s->T;
    const int slot = (int)(k % P);
    const double* src = in + (long long)b * B;
    long long ld = ld_in;
    if (s->kind == EM_STREAM_SH) {
      ProfSpan ps(h, EM_PROF_RENDER_STAGE);
      const long long fb = std::max<long long>(t_lo / hop - 1, 0), fh = (t_lo + B - 1) / hop;
      launch_frame_rotations(h, L, s->d_rot, nfr_c * 9, f_first, fb, fh - fb + 1, s->order, s->Q, s->same, s->nfr_blk);
      launch_sh_track_rotate(h, L, in, ld_in, (long long)b * B, B, s->order, s->Q, s->same, s->nfr_blk, fb, t_first,
                             hop, s->fade, s->rbuf, (long long)num_ch * B);
      h->launches += 2;
      src = s->rbuf;
      ld = B;
    }
    const long long xs = (long long)s->xch * F;   // slot stride of the FDL
    {
      ProfSpan ps(h, EM_PROF_RENDER_STAGE);
      const long long n = (long long)s->xch * B;
      stream_stage_kernel<<<(unsigned)((n + 255) / 256), 256, 0, st>>>(src, ld, s->xch, B, s->prev, s->seg);
      EM_CUDA(cudaGetLastError());
    }
    {
      ProfSpan ps(h, EM_PROF_RENDER_FFT);
      EM_FFT(cufftExecD2Z(s->fwd, s->seg, reinterpret_cast<cufftDoubleComplex*>(s->X + slot * xs)));
    }
    const bool bank = s->kind == EM_STREAM_BANK;
    const int np = bank ? blk_off[b + 1] - blk_off[b] : 1;
    const int* pages = bank ? s->d_tab + cmb_off[nb] + blk_off[b] : s->d_zero;
    constexpr int G = 4;
    {
      ProfSpan ps(h, EM_PROF_RENDER_MAC);
      dim3 grid((unsigned)((F + 127) / 128), (unsigned)((np + G - 1) / G), bank ? 1u : (unsigned)s->pcap);
      stream_mac_kernel<G><<<grid, 128, 0, st>>>(s->X, xs, s->H, pages, np, num_ch, P, F, slot, s->Y);
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
      long long f0 = 0;
      int nfb = 0;
      blk_frames(b, f0, nfb);
      stream_combine_kernel<<<dim3((unsigned)((B + 127) / 128), (unsigned)L), 128, 0, st>>>(
          s->yseg, bank ? s->d_tab + cmb_off[b] : nullptr, f0, nfb, t_lo, B, hop, s->fade, ld_out,
          out + (long long)b * B);
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
  const int no = 2 * s->nl;   // output rows: (listener, ear)
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
      EM_CUDA(cudaMemcpyAsync(s->h_out, s->d_out, (size_t)no * cn * sizeof(double), cudaMemcpyDeviceToHost, st));
      EM_CUDA(cudaStreamSynchronize(st));
      for (int r = 0; r < no; ++r)
        std::memcpy(out + (long long)r * num_samples + c0, s->h_out + (long long)r * cn, (size_t)cn * sizeof(double));
    }
    trim_entries(s);
  }
}

void check_create(const double* wL, const double* wR, int len, int num_ch, int num_pages, int num_listeners, int block,
                  int hop, int fade, const emagls_render_stream* out) {
  EM_REQUIRE(wL && wR && out, "null argument");
  EM_REQUIRE(len > 0 && num_ch > 0 && num_pages > 0, "empty filters");
  EM_REQUIRE(num_listeners >= 1 && num_listeners <= ST_MAX_LISTENERS, "num_listeners must lie in [1, 4096]");
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

int emagls_render_stream_create_listeners(emagls_handle h, const double* wL, const double* wR, int len, int num_ch,
                                          int num_pages, int num_listeners, int block, int hop, int fade,
                                          emagls_render_stream* out) {
  if (out) *out = nullptr;
  return guarded(h, [&] {
    check_create(wL, wR, len, num_ch, num_pages, num_listeners, block, hop, fade, out);
    EM_REQUIRE(num_listeners == 1 || num_pages > 1, "a static session (num_pages == 1) serves one listener");
    const int kind = num_pages == 1 ? EM_STREAM_STATIC : EM_STREAM_BANK;
    open_session(h, create_session(h, kind, wL, wR, len, num_ch, num_pages, 0, num_listeners, block, hop, fade), out);
  });
}

int emagls_render_stream_create(emagls_handle h, const double* wL, const double* wR, int len, int num_ch,
                                int num_pages, int block, int hop, int fade, emagls_render_stream* out) {
  return emagls_render_stream_create_listeners(h, wL, wR, len, num_ch, num_pages, 1, block, hop, fade, out);
}

int emagls_render_stream_create_sh_listeners(emagls_handle h, const double* wL, const double* wR, int len, int order,
                                             int num_listeners, int block, int hop, int fade,
                                             emagls_render_stream* out) {
  if (out) *out = nullptr;
  return guarded(h, [&] {
    EM_REQUIRE(order >= 0 && order <= ST_MAX_ORDER, "order must lie in [0, 7]");
    const int C = (order + 1) * (order + 1);
    check_create(wL, wR, len, C, 1, num_listeners, block, hop, fade, out);
    // the per-block forward transform (one cuFFT plan of 32-bit sizes) takes every listener's rotated block
    EM_REQUIRE((long long)num_listeners * C * 2 * block <= 2147483647LL,
               "num_listeners (order + 1)^2 2 block must stay below 2^31");
    open_session(h, create_session(h, EM_STREAM_SH, wL, wR, len, C, 1, order, num_listeners, block, hop, fade), out);
  });
}

int emagls_render_stream_create_sh(emagls_handle h, const double* wL, const double* wR, int len, int order,
                                   int block, int hop, int fade, emagls_render_stream* out) {
  return emagls_render_stream_create_sh_listeners(h, wL, wR, len, order, 1, block, hop, fade, out);
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
