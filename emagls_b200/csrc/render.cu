// binauralDecode (dependencies/binauralDecode.m:33-64): out(:,ear) = sum_ch fftfilt(w_ear(:,ch), in(:,ch)),
// i.e. the first num_samples samples of the multichannel linear convolution, as a partitioned
// overlap-save convolution.  cuFFT performs the D2Z / Z2D transforms only; the per-bin
// multiply-accumulate over channels (the HBM-bound part) is the hand-written kernel below.
#include <algorithm>
#include <cstdint>
#include <cstdlib>
#include <vector>
#include "render.h"

namespace emagls {

int env_int(const char* name, int dflt) {
  const char* e = getenv(name);
  return e ? atoi(e) : dflt;
}

void drop_plans(emagls_ctx::RenderPlans& rp) {
  if (rp.fwd) cufftDestroy(rp.fwd);
  if (rp.inv) cufftDestroy(rp.inv);
  if (rp.filt) cufftDestroy(rp.filt);
  if (rp.edge) cufftDestroy(rp.edge);
  for (auto& d : rp.direct) cufftDestroy(d.second);
  rp = emagls_ctx::RenderPlans{};
}

void ensure_plans(emagls_ctx* h, emagls_ctx::RenderPlans& rp, int N, int L, int num_ch, int nbc, int filt_batch,
                  int inv_batch) {
  if (rp.N == N && rp.L == L && rp.num_ch == num_ch && rp.nbc == nbc && rp.filt_batch == filt_batch &&
      rp.inv_batch == inv_batch && rp.fwd && rp.inv && rp.filt)
    return;
  drop_plans(rp);
  const int F = N / 2 + 1;
  int n[1] = {N};
  cufftHandle pf = 0, pi = 0, pw = 0;
  EM_FFT(cufftPlanMany(&pw, 1, n, nullptr, 1, N, nullptr, 1, F, CUFFT_D2Z, filt_batch));
  // overlapping input batches: block j of channel ch starts at (ch * nbc + j) * L
  int inembed[1] = {N}, onembed[1] = {F};
  EM_FFT(cufftPlanMany(&pf, 1, n, inembed, 1, L, onembed, 1, F, CUFFT_D2Z, num_ch * nbc));
  EM_FFT(cufftPlanMany(&pi, 1, n, nullptr, 1, F, nullptr, 1, N, CUFFT_Z2D, inv_batch));
  // boundary block e of every channel: in xe[ch][e][N], out X[ch][b][F]
  cufftHandle pe = 0;
  int e_in[1] = {N};
  EM_FFT(cufftPlanMany(&pe, 1, n, e_in, 1, MAX_EDGE * N, onembed, 1, nbc * F, CUFFT_D2Z, num_ch));
  EM_FFT(cufftSetStream(pw, h->stream));
  EM_FFT(cufftSetStream(pf, h->stream));
  EM_FFT(cufftSetStream(pi, h->stream));
  EM_FFT(cufftSetStream(pe, h->stream));
  rp.N = N; rp.L = L; rp.num_ch = num_ch; rp.nbc = nbc; rp.filt_batch = filt_batch; rp.inv_batch = inv_batch;
  rp.fwd = pf; rp.inv = pi; rp.filt = pw; rp.edge = pe;
}

namespace {

// interior blocks of one channel straight from the caller's signal: `batch` overlapping transforms at
// distance L (cuFFT plans have a fixed batch: one plan per distinct count, normally one or two)
cufftHandle direct_plan(emagls_ctx* h, emagls_ctx::RenderPlans& rp, int N, int L, int batch) {
  for (auto& d : rp.direct)
    if (d.first == batch) return d.second;
  const int F = N / 2 + 1;
  int n[1] = {N}, inembed[1] = {N}, onembed[1] = {F};
  cufftHandle p = 0;
  EM_FFT(cufftPlanMany(&p, 1, n, inembed, 1, L, onembed, 1, F, CUFFT_D2Z, batch));
  EM_FFT(cufftSetStream(p, h->stream));
  if (rp.direct.size() >= 4) { cufftDestroy(rp.direct.front().second); rp.direct.erase(rp.direct.begin()); }
  rp.direct.emplace_back(batch, p);
  return p;
}

// Segment buffer of one chunk of blocks: xp[ch][i] = in[ch][s_first + i] (zero outside the signal),
// i in [0, seg_len).  Block j of a channel is the N samples starting at xp[ch][j * L].
__global__ void stage_input_kernel(const double* __restrict__ in, long long num_samples, int num_ch,
                                   long long s_first, long long seg_len, long long ch_stride,
                                   double* __restrict__ xp) {
  long long idx = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  long long total = seg_len * num_ch;
  if (idx >= total) return;
  int ch = (int)(idx / seg_len);
  long long i = idx % seg_len;
  long long n = s_first + i;
  xp[(long long)ch * ch_stride + i] = (n >= 0 && n < num_samples) ? in[(long long)ch * num_samples + n] : 0.0;
}

__global__ void pad_filters_kernel(const double* __restrict__ wL, const double* __restrict__ wR, int len,
                                   int num_ch, int N, double* __restrict__ wp) {
  int idx = blockIdx.x * blockDim.x + threadIdx.x;
  if (idx >= 2 * num_ch * N) return;
  int t = idx % N, ch = (idx / N) % num_ch, ear = idx / (N * num_ch);
  const double* w = ear ? wR : wL;
  wp[idx] = (t < len) ? w[(long long)ch * len + t] : 0.0;
}

// Y[ear][b][f] = sum_ch X[ch][b][f] * Hw[ear][ch][f].  One thread per (f, BT consecutive blocks):
// each pair of filter-spectrum values (L2-resident) is used for BT blocks, and the channel loop is
// unrolled by CU so CU * (BT + 2) independent 16-byte loads are in flight per thread.
template <int BT, int CU>
__global__ void __launch_bounds__(128)
spectral_mac_kernel(const cplx* __restrict__ X, const cplx* __restrict__ Hw, int num_ch, int nbc,
                    int nb, int F, cplx* __restrict__ Y) {
  const int f = blockIdx.x * blockDim.x + threadIdx.x;
  const int b0 = blockIdx.y * BT;
  if (f >= F) return;
  const long long xs = (long long)nbc * F;  // channel stride of X
  const cplx* x = X + (long long)b0 * F + f;
  const cplx* hl = Hw + f;
  const cplx* hr = Hw + (long long)num_ch * F + f;
  cplx yl[BT], yr[BT];
#pragma unroll
  for (int t = 0; t < BT; ++t) { yl[t] = mk(0.0, 0.0); yr[t] = mk(0.0, 0.0); }
  // blocks past nb inside the same channel segment still exist (nbc > nb), so full tiles never
  // read out of range; the stores are guarded
  const int bt = min(BT, nbc - b0);
  int ch = 0;
  if (bt == BT) {
    for (; ch + CU <= num_ch; ch += CU) {
      cplx xv[CU][BT], a[CU], c[CU];
#pragma unroll
      for (int u = 0; u < CU; ++u) {
        a[u] = hl[(long long)(ch + u) * F];
        c[u] = hr[(long long)(ch + u) * F];
#pragma unroll
        for (int t = 0; t < BT; ++t) xv[u][t] = x[(long long)(ch + u) * xs + (long long)t * F];
      }
#pragma unroll
      for (int u = 0; u < CU; ++u)
#pragma unroll
        for (int t = 0; t < BT; ++t) { cfma(yl[t], xv[u][t], a[u]); cfma(yr[t], xv[u][t], c[u]); }
    }
  }
  for (; ch < num_ch; ++ch) {
    const cplx a = hl[(long long)ch * F], c = hr[(long long)ch * F];
#pragma unroll
    for (int t = 0; t < BT; ++t)
      if (t < bt) {
        const cplx xv = x[(long long)ch * xs + (long long)t * F];
        cfma(yl[t], xv, a); cfma(yr[t], xv, c);
      }
  }
#pragma unroll
  for (int t = 0; t < BT; ++t)
    if (b0 + t < nb) {
      Y[(long long)(b0 + t) * F + f] = yl[t];
      Y[((long long)nb + b0 + t) * F + f] = yr[t];
    }
}

// out[ear][row] = yseg[ear][b][ov + i] / N for full-signal sample n = s0 + b*L + i, row = n - skip
__global__ void unstage_output_kernel(const double* __restrict__ yseg, int nb, int N, int L, int ov, long long s0,
                                      long long num_samples, long long skip, long long out_rows,
                                      double* __restrict__ out) {
  long long idx = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  long long total = (long long)2 * nb * L;
  if (idx >= total) return;
  int i = (int)(idx % L);
  int b = (int)((idx / L) % nb);
  int ear = (int)(idx / ((long long)L * nb));
  long long n = s0 + (long long)b * L + i;
  if (n >= num_samples || n < skip) return;
  out[(long long)ear * out_rows + (n - skip)] = yseg[((long long)ear * nb + b) * N + ov + i] * (1.0 / (double)N);
}

// ---------------------------------------------------------------------------------------------
// Fused overlap-save block: one CTA per block of L output frames.  For every channel the N-point real
// FFT (as an N/2-point complex Stockham FFT, radix 4 with a leading radix-2 stage when log2(N/2) is odd,
// ping-pong in shared memory), the multiply-accumulate with both ears' filter spectra into two
// accumulators in shared memory, then the two inverse transforms and the store of the valid L frames.
// The channel spectra never reach HBM: the kernel reads the input once (plus the N/L overlap) and the
// L2-resident filter spectra, and writes the two output channels.
//   rfft:  X[k] = (Z[k] + conj(Z[M-k])) / 2 - (i/2) W_N^k (Z[k] - conj(Z[M-k])),  z[n] = x[2n] + i x[2n+1]
//   irfft: Zy[k] = (Y[k] + conj(Y[M-k])) + i conj(W_N^k) (Y[k] - conj(Y[M-k])),  y[2n] + i y[2n+1] = IFFT_M(Zy) / N
// WM[q] = exp(-2 pi i q / M) (q < M/2), WN[k] = exp(-2 pi i k / N) (k <= M), M = N / 2.
// ---------------------------------------------------------------------------------------------
__global__ void render_twiddle_kernel(int M, cplx* __restrict__ WM, cplx* __restrict__ WN) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i < M / 2) { double s_, c_; sincospi(-2.0 * (double)i / (double)M, &s_, &c_); WM[i] = mk(c_, s_); }
  if (i <= M) { double s_, c_; sincospi(-(double)i / (double)M, &s_, &c_); WN[i] = mk(c_, s_); }
}

// Stockham FFT of length M on ping-pong buffers, NB independent transforms side by side (buffer pair q at
// src + q * stride, dst + q * stride; the twiddles are shared); returns the offset-0 buffer holding the results
template <bool INV, int NB>
__device__ __forceinline__ cplx* stockham_fft(cplx* src, cplx* dst, long long stride, int M, int logM,
                                              const cplx* __restrict__ WM, int tid, int nt) {
  int p = 1;
  if (logM & 1) {
    for (int j = tid; j < M / 2; j += nt) {
#pragma unroll
      for (int q = 0; q < NB; ++q) {
        const cplx u0 = src[q * stride + j], u1 = src[q * stride + j + M / 2];
        dst[q * stride + 2 * j] = cadd(u0, u1); dst[q * stride + 2 * j + 1] = csub(u0, u1);
      }
    }
    __syncthreads();
    cplx* t_ = src; src = dst; dst = t_;
    p = 2;
  }
  const int T = M / 4;
  while (p < M) {
    const int tw = M / (4 * p);
    for (int t = tid; t < T; t += nt) {
      const int k = t & (p - 1);
      cplx w1 = WM[k * tw], w2 = WM[2 * k * tw];
      if (INV) { w1.y = -w1.y; w2.y = -w2.y; }
      const cplx w3 = cmul(w1, w2);
      const int j = ((t - k) << 2) + k;
#pragma unroll
      for (int q = 0; q < NB; ++q) {
        const cplx* sq = src + q * stride;
        cplx* dq = dst + q * stride;
        const cplx u0 = sq[t], u1 = cmul(sq[t + T], w1), u2 = cmul(sq[t + 2 * T], w2), u3 = cmul(sq[t + 3 * T], w3);
        const cplx v0 = cadd(u0, u2), v1 = csub(u0, u2), v2 = cadd(u1, u3);
        cplx v3 = csub(u1, u3);
        v3 = INV ? mk(-v3.y, v3.x) : mk(v3.y, -v3.x);          // * (+i) inverse, * (-i) forward
        dq[j] = cadd(v0, v2); dq[j + p] = cadd(v1, v3); dq[j + 2 * p] = csub(v0, v2); dq[j + 3 * p] = csub(v1, v3);
      }
    }
    __syncthreads();
    cplx* t_ = src; src = dst; dst = t_;
    p <<= 2;
  }
  return src;
}

// input block of one channel -> buffer (pairs x[2n], x[2n+1] as one complex value), asynchronously with zero fill
// outside the signal (both samples of a pair are inside or outside: the block origin and num_samples are even)
__device__ __forceinline__ void fused_load_async(cplx* buf, const double* __restrict__ x, long long s_first,
                                                 long long num_samples, int M, int tid, int nt) {
  for (int n = tid; n < M; n += nt) {
    const long long i0 = s_first + 2LL * n;
    const bool in_range = (i0 >= 0 && i0 < num_samples);
    cp_async16(buf + n, x + (in_range ? i0 : 0), in_range);
  }
}

// Two channels per pass (NB = 2): buffers [A0 | A1 | B0 | B1 | accL | accR].
__global__ void __launch_bounds__(512, 1)
fused_render_kernel(const double* __restrict__ in, long long num_samples, int num_ch, const cplx* __restrict__ Hw,
                    const cplx* __restrict__ WM, const cplx* __restrict__ WN, int N, int logM, int L, int ov,
                    long long skip, long long out_rows, double* __restrict__ out) {
  extern __shared__ __align__(16) unsigned char fr_raw[];
  const int M = N / 2, F = M + 1, tid = threadIdx.x, nt = blockDim.x;
  cplx* A = reinterpret_cast<cplx*>(fr_raw);        // A0, A1
  cplx* Bf = A + 2 * M;                             // B0, B1
  cplx* accL = Bf + 2 * M;
  cplx* accR = accL + F;
  const long long b = blockIdx.x;
  const long long s_first = b * (long long)L - ov;          // even: L and ov are even
  for (int k = tid; k < F; k += nt) { accL[k] = mk(0.0, 0.0); accR[k] = mk(0.0, 0.0); }
  // ping-pong roles: the transform of the pair in `cur` uses `oth` as scratch and leaves the spectra in one of
  // the two; the other one is free while the spectra are unpacked and accumulated, so the next pair of channels
  // is prefetched into it (cp.async) and becomes `cur` of the next iteration
  cplx* cur = A;
  cplx* oth = Bf;
  fused_load_async(cur, in, s_first, num_samples, M, tid, nt);
  if (num_ch > 1) fused_load_async(cur + M, in + num_samples, s_first, num_samples, M, tid, nt);
  cp_async_commit();
  for (int ch = 0; ch < num_ch; ch += 2) {
    const int nb2 = (ch + 1 < num_ch) ? 2 : 1;
    cp_async_wait<0>();
    __syncthreads();
    const cplx* Z = (nb2 == 2) ? stockham_fft<false, 2>(cur, oth, M, M, logM, WM, tid, nt)
                               : stockham_fft<false, 1>(cur, oth, M, M, logM, WM, tid, nt);
    cplx* freeb = (Z == cur) ? oth : cur;
    if (ch + 2 < num_ch) {
      fused_load_async(freeb, in + (long long)(ch + 2) * num_samples, s_first, num_samples, M, tid, nt);
      if (ch + 3 < num_ch) fused_load_async(freeb + M, in + (long long)(ch + 3) * num_samples, s_first, num_samples, M, tid, nt);
      cp_async_commit();
    }
    for (int q = 0; q < nb2; ++q) {
      const cplx* Zq = Z + (long long)q * M;
      const cplx* hl = Hw + (long long)(ch + q) * F;
      const cplx* hr = Hw + ((long long)num_ch + ch + q) * F;
      for (int k = tid; k < F; k += nt) {
        const cplx zk = Zq[k & (M - 1)], zm = cconj(Zq[(M - k) & (M - 1)]);
        const cplx sm_ = cadd(zk, zm), df = cmul(WN[k], csub(zk, zm));
        const cplx X = mk(0.5 * (sm_.x + df.y), 0.5 * (sm_.y - df.x));     // sm/2 - (i/2) df
        cfma(accL[k], X, hl[k]);
        cfma(accR[k], X, hr[k]);
      }
    }
    oth = (freeb == cur) ? oth : cur;
    cur = freeb;
    // the barrier at the top of the next iteration orders the reads of Z before the next transform's writes
  }
  __syncthreads();
  // both ears side by side
  const double inv_n = 1.0 / (double)N;
  for (int k = tid; k < M; k += nt) {
#pragma unroll
    for (int ear = 0; ear < 2; ++ear) {
      const cplx* acc = ear ? accR : accL;
      const cplx yk = acc[k], ym = cconj(acc[M - k]);
      const cplx sm_ = cadd(yk, ym), df = cmul(cconj(WN[k]), csub(yk, ym));
      A[ear * M + k] = mk(sm_.x - df.y, sm_.y + df.x);               // sm + i df
    }
  }
  __syncthreads();
  const cplx* zy = stockham_fft<true, 2>(A, Bf, M, M, logM, WM, tid, nt);
  for (int n = tid; n < M; n += nt) {
    const int i = 2 * n;
    if (i < ov) continue;
    const long long s0 = b * (long long)L + (i - ov);
#pragma unroll
    for (int ear = 0; ear < 2; ++ear) {
      const cplx v = zy[ear * M + n];
      if (s0 < num_samples && s0 >= skip) out[(long long)ear * out_rows + (s0 - skip)] = v.x * inv_n;
      if (s0 + 1 < num_samples && s0 + 1 >= skip) out[(long long)ear * out_rows + (s0 + 1 - skip)] = v.y * inv_n;
    }
  }
}

// ---------------------------------------------------------------------------------------------
// fused_render16_kernel (N = 4096, EMAGLS_RENDER_FUSED=2): the same overlap-save block per CTA with
// register-resident radix-16 / radix-8 Stockham passes (2048 = 16 x 16 x 8).  Four channels at a time, one
// radix-16 butterfly per thread and pass: the first pass reads its sixteen 16-byte sample pairs straight from
// global memory (coalesced over the butterfly index; they are issued before the previous group's spectra are
// accumulated, so the loads fly during that phase), the other two passes run in place in shared memory
// (read - barrier - write - barrier) on buffers padded by one element per sixteen (the stride-16 writes of the
// first pass would otherwise hit one bank).  Six barriers per FOUR transforms instead of six per two, sixteen
// independent loads per thread instead of four.
// ---------------------------------------------------------------------------------------------
constexpr int FR_M = 2048, FR_T = 512, FR_LD = FR_M + FR_M / 16;   // complex points, threads, padded buffer length
__device__ __forceinline__ int fr_pad(int i) { return i + (i >> 4); }

// Twiddles of the two in-place passes in the order the lanes read them (consecutive lanes -> consecutive entries):
// P2[ji][k] = exp(-2 pi i k 2^ji / 256) (stride-16 pass, k < 16, ji < 4) at ji * 16 + k, then
// P3[ji][tt] = exp(-2 pi i tt 2^ji / 2048) (last pass, tt < 256, ji < 3) at 64 + ji * 256 + tt.
constexpr int FR_TW = 4 * 16 + 3 * 256;
#ifndef EMAGLS_FR_TW_SMEM
#define EMAGLS_FR_TW_SMEM 0     // 1: the kernel copies the table into shared memory (A/B: slower, it shrinks the L1)
#endif
__global__ void render_twiddle_full_kernel(cplx* __restrict__ TW) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= FR_TW) return;
  const int j = (i < 64) ? ((i & 15) * 8) << (i >> 4) : ((i - 64) & 255) << ((i - 64) >> 8);
  double s_, c_;
  sincospi(-2.0 * (double)j / (double)FR_M, &s_, &c_);
  TW[i] = mk(c_, s_);
}

template <bool INV>
__device__ __forceinline__ void fr_dft4(cplx& a0, cplx& a1, cplx& a2, cplx& a3) {
  const cplx s02 = cadd(a0, a2), d02 = csub(a0, a2), s13 = cadd(a1, a3), d13 = csub(a1, a3);
  const cplx jd = INV ? mk(-d13.y, d13.x) : mk(d13.y, -d13.x);      // (+i) d13 inverse, (-i) d13 forward
  a0 = cadd(s02, s13); a1 = cadd(d02, jd); a2 = csub(s02, s13); a3 = csub(d02, jd);
}
// multiply by W16^e (forward) or its conjugate (inverse), e a compile-time exponent
template <bool INV, int E>
__device__ __forceinline__ cplx fr_w16(cplx a) {
  constexpr double c1 = 0.92387953251128673848, s1 = 0.38268343236508977173, r2 = 0.70710678118654752440;
  constexpr int e = E & 15;
  if (e == 0) return a;
  if (e == 4) return INV ? mk(-a.y, a.x) : mk(a.y, -a.x);                         // -i / +i
  if (e == 8) return mk(-a.x, -a.y);
  double c = 1.0, sn = 0.0;                                                        // W16^e = c - i sn (forward)
  if (e == 1) { c = c1; sn = s1; } else if (e == 2) { c = r2; sn = r2; } else if (e == 3) { c = s1; sn = c1; }
  else if (e == 6) { c = -r2; sn = r2; } else if (e == 9) { c = -c1; sn = -s1; }
  const double si = INV ? sn : -sn;                                                // imaginary part of the factor
  return mk(fma(a.x, c, -a.y * si), fma(a.x, si, a.y * c));
}
// in: v[4 n1 + n2] = x[4 n1 + n2]; out: X[m1 + 4 m2] at v[4 m1 + m2]
template <bool INV>
__device__ __forceinline__ void fr_dft16(cplx (&v)[16]) {
#pragma unroll
  for (int n2 = 0; n2 < 4; ++n2) fr_dft4<INV>(v[n2], v[4 + n2], v[8 + n2], v[12 + n2]);
  v[5] = fr_w16<INV, 1>(v[5]);   v[6] = fr_w16<INV, 2>(v[6]);   v[7] = fr_w16<INV, 3>(v[7]);
  v[9] = fr_w16<INV, 2>(v[9]);   v[10] = fr_w16<INV, 4>(v[10]); v[11] = fr_w16<INV, 6>(v[11]);
  v[13] = fr_w16<INV, 3>(v[13]); v[14] = fr_w16<INV, 6>(v[14]); v[15] = fr_w16<INV, 9>(v[15]);
#pragma unroll
  for (int m1 = 0; m1 < 4; ++m1) fr_dft4<INV>(v[4 * m1], v[4 * m1 + 1], v[4 * m1 + 2], v[4 * m1 + 3]);
}
// in: v[n]; out: X[m] at o[m]
template <bool INV>
__device__ __forceinline__ void fr_dft8(cplx (&v)[8], cplx (&o)[8]) {
  fr_dft4<INV>(v[0], v[2], v[4], v[6]);     // y[m1][0] at v[2 m1]
  fr_dft4<INV>(v[1], v[3], v[5], v[7]);     // y[m1][1] at v[2 m1 + 1]
  const cplx t0 = v[1], t1 = fr_w16<INV, 2>(v[3]), t2 = fr_w16<INV, 4>(v[5]), t3 = fr_w16<INV, 6>(v[7]);
  o[0] = cadd(v[0], t0); o[4] = csub(v[0], t0);
  o[1] = cadd(v[2], t1); o[5] = csub(v[2], t1);
  o[2] = cadd(v[4], t2); o[6] = csub(v[4], t2);
  o[3] = cadd(v[6], t3); o[7] = csub(v[6], t3);
}
template <bool INV> __device__ __forceinline__ cplx fr_tw(const cplx* tab, int idx) {
  const cplx w = tab[idx];
  return INV ? mk(w.x, -w.y) : w;
}
// X[q'] of fr_dft16 sits at v[4 (q' & 3) + (q' >> 2)]
#define FR_OUT16(v, qp) (v)[4 * ((qp) & 3) + ((qp) >> 2)]

// radix-16 pass with stride p (1 or 16) in place on the padded buffer Z; every thread of the CTA calls it (barriers)
template <bool INV>
__device__ __forceinline__ void fr_pass16(cplx* Z, int t, int p, bool active, const cplx* TW) {
  cplx v[16];
  const int k = t & (p - 1), a = t / p;
  if (active) {
#pragma unroll
    for (int q = 0; q < 16; ++q) v[q] = Z[fr_pad(t + 128 * q)];
    if (p > 1) {
      // twiddle w^q, w = exp(-+2 pi i k / (16 p)); only p = 16 has twiddles
      const cplx w1 = fr_tw<INV>(TW, k), w2 = fr_tw<INV>(TW, 16 + k), w4 = fr_tw<INV>(TW, 32 + k), w8 = fr_tw<INV>(TW, 48 + k);
      const cplx w3 = cmul(w1, w2), w5 = cmul(w4, w1), w6 = cmul(w4, w2), w7 = cmul(w4, w3);
      v[1] = cmul(v[1], w1); v[2] = cmul(v[2], w2); v[3] = cmul(v[3], w3); v[4] = cmul(v[4], w4);
      v[5] = cmul(v[5], w5); v[6] = cmul(v[6], w6); v[7] = cmul(v[7], w7); v[8] = cmul(v[8], w8);
      v[9] = cmul(v[9], cmul(w8, w1)); v[10] = cmul(v[10], cmul(w8, w2)); v[11] = cmul(v[11], cmul(w8, w3));
      v[12] = cmul(v[12], cmul(w8, w4)); v[13] = cmul(v[13], cmul(w8, w5)); v[14] = cmul(v[14], cmul(w8, w6));
      v[15] = cmul(v[15], cmul(w8, w7));
    }
    fr_dft16<INV>(v);
  }
  __syncthreads();
  if (active) {
    const int base = a * p * 16 + k;
#pragma unroll
    for (int qp = 0; qp < 16; ++qp) Z[fr_pad(base + qp * p)] = FR_OUT16(v, qp);
  }
  __syncthreads();
}
// last pass (radix 8, stride 256): butterflies t and t + 128 of the transform
template <bool INV>
__device__ __forceinline__ void fr_pass8(cplx* Z, int t, bool active, const cplx* TW) {
  cplx o[2][8];
  if (active) {
#pragma unroll
    for (int u = 0; u < 2; ++u) {
      const int tt = t + 128 * u;
      cplx v[8];
#pragma unroll
      for (int q = 0; q < 8; ++q) v[q] = Z[fr_pad(tt + 256 * q)];
      const cplx w1 = fr_tw<INV>(TW, 64 + tt), w2 = fr_tw<INV>(TW, 64 + 256 + tt), w4 = fr_tw<INV>(TW, 64 + 512 + tt);
      const cplx w3 = cmul(w1, w2);
      v[1] = cmul(v[1], w1); v[2] = cmul(v[2], w2); v[3] = cmul(v[3], w3); v[4] = cmul(v[4], w4);
      v[5] = cmul(v[5], cmul(w4, w1)); v[6] = cmul(v[6], cmul(w4, w2)); v[7] = cmul(v[7], cmul(w4, w3));
      fr_dft8<INV>(v, o[u]);
    }
  }
  __syncthreads();
  if (active) {
#pragma unroll
    for (int u = 0; u < 2; ++u)
#pragma unroll
      for (int qp = 0; qp < 8; ++qp) Z[fr_pad(t + 128 * u + 256 * qp)] = o[u][qp];
  }
  __syncthreads();
}

// first forward pass of channel `ch` from global memory: pairs (x[2n], x[2n+1]) at n = t + 128 q, zero outside the signal
__device__ __forceinline__ void fr_load_first(cplx (&v)[16], const double* __restrict__ in, long long num_samples, int ch,
                                              bool valid, long long s_first, int t) {
  const double* x = in + (long long)ch * num_samples;
#pragma unroll
  for (int q = 0; q < 16; ++q) {
    const long long i0 = s_first + 2LL * (t + 128 * q);
    if (valid && i0 >= 0 && i0 < num_samples) {
      const double2 d = *reinterpret_cast<const double2*>(x + i0);
      v[q] = mk(d.x, d.y);
    } else {
      v[q] = mk(0.0, 0.0);
    }
  }
}

__device__ __forceinline__ void fr_prefetch_first(const double* __restrict__ in, long long num_samples, int ch, bool valid,
                                                  long long s_first, int t) {
  if (!valid || (t & 7) != 0) return;          // one prefetch per 128-byte line (eight 16-byte pairs)
  const double* x = in + (long long)ch * num_samples;
#pragma unroll
  for (int q = 0; q < 16; ++q) {
    const long long i0 = s_first + 2LL * (t + 128 * q);
    if (i0 >= 0 && i0 < num_samples) asm volatile("prefetch.global.L2 [%0];" ::"l"(x + i0));
  }
}

// bin k of the spectra of channels cg .. cg + nc - 1 (packed transforms in Zb) into the two ears' accumulators; the
// filter spectra of all CU channels are requested before anything is computed (CU = 4: full group, CU = 1: tail)
template <int CU>
__device__ __forceinline__ void fr_accumulate(const cplx* Zb, cplx* accL, cplx* accR, const cplx* __restrict__ Hw,
                                              const cplx* __restrict__ WN, int num_ch, int cg, int k, int nc) {
  constexpr int M = FR_M, F = FR_M + 1;
  const cplx wn = WN[k];
  cplx aL = accL[k], aR = accR[k];
  const int ik = fr_pad(k & (M - 1)), im = fr_pad((M - k) & (M - 1));
  for (int c0 = 0; c0 < nc; c0 += CU) {
    cplx hl[CU], hr[CU];
#pragma unroll
    for (int u = 0; u < CU; ++u) {
      const int c = min(c0 + u, nc - 1);           // a channel past the end: loaded again, not used
      hl[u] = Hw[(long long)(cg + c) * F + k];
      hr[u] = Hw[((long long)num_ch + cg + c) * F + k];
    }
#pragma unroll
    for (int u = 0; u < CU; ++u) {
      if (c0 + u >= nc) break;
      const cplx zk = Zb[(c0 + u) * FR_LD + ik], zm = cconj(Zb[(c0 + u) * FR_LD + im]);
      const cplx sm_ = cadd(zk, zm), df = cmul(wn, csub(zk, zm));
      const cplx X = mk(0.5 * (sm_.x + df.y), 0.5 * (sm_.y - df.x));     // sm/2 - (i/2) df
      cfma(aL, X, hl[u]);
      cfma(aR, X, hr[u]);
    }
  }
  accL[k] = aL; accR[k] = aR;
}

// PRE = 1: the next group's samples are loaded into registers before the accumulation (they fly during it);
// PRE = 0: they are only pulled into L2 there and loaded afterwards (more registers for the filter spectra in flight)
template <int PRE>
__global__ void __launch_bounds__(FR_T, 1)
fused_render16_kernel(const double* __restrict__ in, long long num_samples, int num_ch, const cplx* __restrict__ Hw,
                      const cplx* __restrict__ TWg, const cplx* __restrict__ WN, int L, int ov, long long skip,
                      long long out_rows, double* __restrict__ out) {
  extern __shared__ __align__(16) unsigned char fr16_raw[];
  constexpr int M = FR_M, F = FR_M + 1, N = 2 * FR_M;
  cplx* Zb = reinterpret_cast<cplx*>(fr16_raw);        // [4][FR_LD]
  cplx* accL = Zb + 4 * FR_LD;                         // [F]
  cplx* accR = accL + F;
#if EMAGLS_FR_TW_SMEM
  cplx* TW = accR + F;                                 // [FR_TW]
#else
  const cplx* TW = TWg;
#endif
  const int tid = threadIdx.x, g4 = tid >> 7, t = tid & 127;
  cplx* Z = Zb + g4 * FR_LD;
  const long long b = blockIdx.x;
  const long long s_first = b * (long long)L - ov;     // even: L and ov are even
  cplx v[16];
  fr_load_first(v, in, num_samples, g4, g4 < num_ch, s_first, t);
  for (int k = tid; k < F; k += FR_T) { accL[k] = mk(0.0, 0.0); accR[k] = mk(0.0, 0.0); }
#if EMAGLS_FR_TW_SMEM
  for (int i = tid; i < FR_TW; i += FR_T) TW[i] = TWg[i];
#endif
  for (int cg = 0; cg < num_ch; cg += 4) {
    // ---- pass 1 (stride 1, no twiddles) from the registers loaded ahead
    fr_dft16<false>(v);
    __syncthreads();                                   // the previous group's spectra have been accumulated
    {
      const int base = 16 * t;
#pragma unroll
      for (int qp = 0; qp < 16; ++qp) Z[fr_pad(base + qp)] = FR_OUT16(v, qp);
    }
    __syncthreads();
    fr_pass16<false>(Z, t, 16, true, TW);
    fr_pass8<false>(Z, t, true, TW);
    // ---- this group's spectra are unpacked and accumulated while the next group's samples are on their way
    const bool more = cg + 4 < num_ch;
    const int nc = min(4, num_ch - cg);
    if (PRE) {
      if (more) fr_load_first(v, in, num_samples, cg + 4 + g4, cg + 4 + g4 < num_ch, s_first, t);
      for (int j = 0; j < 5; ++j) {
        const int k = tid + FR_T * j;
        if (k > M) break;                              // bin M (Nyquist) belongs to thread 0
        const cplx wn = WN[k];
        cplx aL = accL[k], aR = accR[k];
        const int ik = fr_pad(k & (M - 1)), im = fr_pad((M - k) & (M - 1));
        for (int c = 0; c < nc; ++c) {
          const cplx zk = Zb[c * FR_LD + ik], zm = cconj(Zb[c * FR_LD + im]);
          const cplx sm_ = cadd(zk, zm), df = cmul(wn, csub(zk, zm));
          const cplx X = mk(0.5 * (sm_.x + df.y), 0.5 * (sm_.y - df.x));     // sm/2 - (i/2) df
          cfma(aL, X, Hw[(long long)(cg + c) * F + k]);
          cfma(aR, X, Hw[((long long)num_ch + cg + c) * F + k]);
        }
        accL[k] = aL; accR[k] = aR;
      }
    } else {
      if (more) fr_prefetch_first(in, num_samples, cg + 4 + g4, cg + 4 + g4 < num_ch, s_first, t);
#pragma unroll
      for (int j = 0; j < 4; ++j) fr_accumulate<4>(Zb, accL, accR, Hw, WN, num_ch, cg, tid + FR_T * j, nc);
      if (tid == 0) fr_accumulate<4>(Zb, accL, accR, Hw, WN, num_ch, cg, M, nc);
      if (more) fr_load_first(v, in, num_samples, cg + 4 + g4, cg + 4 + g4 < num_ch, s_first, t);
    }
  }
  __syncthreads();
  // ---- both ears: Hermitian spectrum -> packed half-length sequence, inverse transform (transforms 0 and 1)
  for (int k = tid; k < M; k += FR_T) {
#pragma unroll
    for (int ear = 0; ear < 2; ++ear) {
      const cplx* acc = ear ? accR : accL;
      const cplx yk = acc[k], ym = cconj(acc[M - k]);
      const cplx sm_ = cadd(yk, ym), df = cmul(cconj(WN[k]), csub(yk, ym));
      Zb[ear * FR_LD + fr_pad(k)] = mk(sm_.x - df.y, sm_.y + df.x);               // sm + i df
    }
  }
  __syncthreads();
  const bool act = g4 < 2;
  fr_pass16<true>(Z, t, 1, act, TW);
  fr_pass16<true>(Z, t, 16, act, TW);
  fr_pass8<true>(Z, t, act, TW);
  const double inv_n = 1.0 / (double)N;
  for (int n = tid; n < M; n += FR_T) {
    const int i = 2 * n;
    if (i < ov) continue;
    const long long s0 = b * (long long)L + (i - ov);
#pragma unroll
    for (int ear = 0; ear < 2; ++ear) {
      const cplx y = Zb[ear * FR_LD + fr_pad(n)];
      if (s0 < num_samples && s0 >= skip) out[(long long)ear * out_rows + (s0 - skip)] = y.x * inv_n;
      if (s0 + 1 < num_samples && s0 + 1 >= skip) out[(long long)ear * out_rows + (s0 + 1 - skip)] = y.y * inv_n;
    }
  }
}

}  // namespace

ForwardStage::ForwardStage(emagls_ctx* h_, emagls_ctx::RenderPlans& rp_, Arena& ar, const double* in_,
                           long long num_samples_, int num_ch_, int N_, int L_, int ov_, int nbc_)
    : h(h_), rp(rp_), in(in_), num_samples(num_samples_), num_ch(num_ch_), N(N_), L(L_), ov(ov_), nbc(nbc_) {
  seg_len = (long long)nbc * L;
  direct = env_int("EMAGLS_RENDER_DIRECT", 1) != 0 && (num_samples % 2 == 0) &&
           (reinterpret_cast<uintptr_t>(in) % 16 == 0);
  b_int_lo = extra_blocks(ov, L);                                                          // input starts at >= 0
  b_int_hi = (num_samples - N + ov >= 0) ? (num_samples - N + ov) / L : -1;                // ends inside
  // the last nex blocks of the last channel read up to N samples past the staged segments
  xp = direct ? ar.get<double>((size_t)MAX_EDGE * N * num_ch) : ar.get<double>((size_t)seg_len * num_ch + N);
  if (!direct) EM_CUDA(cudaMemsetAsync(xp + seg_len * num_ch, 0, (size_t)N * sizeof(double), h->stream));
}

void ForwardStage::run(long long b0, long long nbk, cplx* X) {
  cudaStream_t st = h->stream;
  const int F = N / 2 + 1;
  if (direct) {
    const long long lo = std::max(b0, b_int_lo), hi = std::min(b0 + nbk - 1, b_int_hi);
    if (hi >= lo) {
      ProfSpan ps(h, EM_PROF_RENDER_FFT);
      cufftHandle pd = direct_plan(h, rp, N, L, (int)(hi - lo + 1));
      for (int ch = 0; ch < num_ch; ++ch)
        EM_FFT(cufftExecD2Z(pd, const_cast<double*>(in) + (long long)ch * num_samples + lo * L - ov,
                            reinterpret_cast<cufftDoubleComplex*>(X + ((long long)ch * nbc + (lo - b0)) * F)));
    }
    // boundary blocks of this chunk, MAX_EDGE at a time
    long long eb[MAX_EDGE];
    int ne = 0;
    auto flush = [&]() {
      for (int e = 0; e < ne; ++e) {
        ProfSpan ps(h, EM_PROF_RENDER_STAGE);
        long long total = (long long)N * num_ch;
        stage_input_kernel<<<(unsigned)((total + 255) / 256), 256, 0, st>>>(in, num_samples, num_ch, eb[e] * L - ov, N,
                                                                          (long long)MAX_EDGE * N, xp + (long long)e * N);
        EM_CUDA(cudaGetLastError());
      }
      for (int e = 0; e < ne; ++e) {
        ProfSpan ps(h, EM_PROF_RENDER_FFT);
        EM_FFT(cufftExecD2Z(rp.edge, xp + (long long)e * N, reinterpret_cast<cufftDoubleComplex*>(X + (eb[e] - b0) * F)));
      }
      h->launches += ne;
      ne = 0;
    };
    for (long long b = b0; b < b0 + nbk; ++b) {
      if (b >= lo && b <= hi) { b = hi; continue; }
      eb[ne++] = b;
      if (ne == MAX_EDGE) flush();
    }
    flush();
  } else {
    {
      ProfSpan ps(h, EM_PROF_RENDER_STAGE);
      long long total = seg_len * num_ch;
      stage_input_kernel<<<(unsigned)((total + 255) / 256), 256, 0, st>>>(in, num_samples, num_ch, b0 * L - ov, seg_len,
                                                                        seg_len, xp);
      EM_CUDA(cudaGetLastError());
    }
    {
      ProfSpan ps(h, EM_PROF_RENDER_FFT);
      EM_FFT(cufftExecD2Z(rp.fwd, xp, reinterpret_cast<cufftDoubleComplex*>(X)));
    }
    h->launches += 1;
  }
}

// Overlap-save geometry: FFT size N (power of two), overlap ov >= len - 1 (even), hop L = N - ov.
// Block b takes the N input samples starting at b*L - ov and yields output samples [b*L, (b+1)*L).
// Large N amortises the overlap (N = 8 len: 12.5 % redundant input, 0.57 spectrum bins per output
// frame instead of 1.0 at N = 2 len); the chunk (blocks per cuFFT batch) is sized so that the
// staged input, its spectra and the ear spectra of one chunk stay L2-resident between the kernels.
void binaural_decode_dev(emagls_ctx* h, const double* in, long long num_samples, int num_ch,
                         const double* wL, const double* wR, int len, int compensate_delay, double* out) {
  EM_REQUIRE(in && wL && wR && out, "null argument");
  EM_REQUIRE(num_samples > 0 && num_ch > 0 && len > 0, "empty input");
  EM_REQUIRE(!compensate_delay || len % 2 == 0, "compensateDelay needs an even filter length");
  cudaStream_t st = h->stream;
  Arena ar(st);
  const int ov = (len + 1) & ~1;
  int Nmin = 16;
  while (Nmin < 2 * len) Nmin <<= 1;
  int N = Nmin;
  {
    int want = env_int("EMAGLS_RENDER_FFT", 0);
    if (want <= 0) want = 8 * Nmin / 2;                       // default N = 8 len (next power of two)
    // no point in blocks much longer than the signal
    while (N < want && (long long)(N - ov) < num_samples) N <<= 1;
  }
  const int L = N - ov, F = N / 2 + 1;
  const long long skip = compensate_delay ? (len / 2 - 1) : 0;  // out(del:end,:), binauralDecode.m:55-56
  const long long out_rows = num_samples - skip;
  EM_REQUIRE(out_rows > 0, "signal shorter than the compensated delay");
  const long long nblk_total = (num_samples + L - 1) / L;
  const int nex = ForwardStage::extra_blocks(ov, L);  // extra hops per channel: the overlapping batch has a uniform distance L
  // blocks per chunk: as many as a memory budget allows (measured on B200: launch-bound below a few
  // hundred blocks; one chunk for a 10-minute signal is fastest, the intermediates do not need to stay
  // in L2).  EMAGLS_RENDER_CHUNK / EMAGLS_RENDER_WS_MB override.
  int chunk_max;
  if (const char* e = getenv("EMAGLS_RENDER_CHUNK")) {
    chunk_max = std::max(1, atoi(e));
  } else {
    size_t free_b = 0, total_b = 0;
    EM_CUDA(cudaMemGetInfo(&free_b, &total_b));
    double budget = std::min(0.4 * (double)free_b, 16.0 * 1073741824.0);
    const int ws_mb = env_int("EMAGLS_RENDER_WS_MB", 0);
    if (ws_mb > 0) budget = (double)ws_mb * 1048576.0;
    const double per_block = (double)num_ch * ((double)L * 8 + (double)F * 16) + 2.0 * F * 16 + 2.0 * N * 8;
    chunk_max = (int)std::max(1.0, std::min(65535.0 * 4, budget / per_block));
  }
  const int chunk = (int)std::min<long long>({nblk_total, (long long)chunk_max, 65535LL * 4});
  const int nbc = chunk + nex;
  auto& rp = h->render_plans;
  ensure_plans(h, rp, N, L, num_ch, nbc, 2 * num_ch, 2 * chunk);

  // filter spectra Hw[ear][ch][F]
  cplx* Hw = ar.get<cplx>((size_t)2 * num_ch * F);
  {
    double* wp = ar.get<double>((size_t)2 * num_ch * N);
    int total = 2 * num_ch * N;
    pad_filters_kernel<<<(total + 255) / 256, 256, 0, st>>>(wL, wR, len, num_ch, N, wp);
    EM_CUDA(cudaGetLastError());
    EM_FFT(cufftExecD2Z(rp.filt, wp, reinterpret_cast<cufftDoubleComplex*>(Hw)));
    h->launches += 1;
  }

  // Fused route (EMAGLS_RENDER_FUSED=1; off by default): one kernel per call, the channel spectra stay in shared
  // memory.  Needs the FFT and both accumulators in one CTA's shared memory (N <= 4096) and 16-byte aligned
  // channels.  Measured on B200 (10 minutes, 32 channels, 512 taps; tools/gpu_render_ab.py,
  // profiles/r01_v25_render_ab.txt): identical output to 8e-16, but 11.8 ms against 9.6 ms for the cuFFT route
  // below (15.3 ms before two channels shared a pass and the next pair was prefetched with cp.async) -- the radix-4
  // shared-memory FFT makes six barrier-separated passes per channel pair with one 512-thread CTA per SM; it needs
  // register-resident radix-8/16 passes before it can win.
  // Default route for N = 4096 (filters of 257 .. 512 taps): the register-resident fused kernel (radix 16 x 16 x 8),
  // 6.7 ms against 9.7 ms for the cuFFT route on 10 minutes x 32 channels (profiles/r02_v27_render_reps.txt).
  // EMAGLS_RENDER_FUSED=0 selects the cuFFT route, =1 the shared-memory radix-4 kernel of round 1, =3 the variant of
  // the default that only pulls the next group's samples into L2 during the accumulation (8.9 ms).
  const int fused_mode = env_int("EMAGLS_RENDER_FUSED", 2);
  if ((fused_mode == 2 || fused_mode == 3) && N == 2 * FR_M && (num_samples % 2 == 0) && (ov % 2 == 0) &&
      (reinterpret_cast<uintptr_t>(in) % 16 == 0)) {
    cplx* TW = ar.get<cplx>((size_t)FR_TW);
    cplx* WMu = ar.get<cplx>((size_t)FR_M / 2 + 1);
    cplx* WN = ar.get<cplx>((size_t)FR_M + 1);
    render_twiddle_full_kernel<<<(FR_TW + 255) / 256, 256, 0, st>>>(TW);
    render_twiddle_kernel<<<(FR_M + 1 + 255) / 256, 256, 0, st>>>(FR_M, WMu, WN);
    EM_CUDA(cudaGetLastError());
    const size_t smem = ((size_t)4 * FR_LD + 2 * (FR_M + 1) + (EMAGLS_FR_TW_SMEM ? FR_TW : 0)) * sizeof(cplx);
    static bool attr_set = false;
    if (!attr_set) {
      EM_CUDA(cudaFuncSetAttribute(fused_render16_kernel<0>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
      EM_CUDA(cudaFuncSetAttribute(fused_render16_kernel<1>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
      attr_set = true;
    }
    {
      ProfSpan ps(h, EM_PROF_RENDER_MAC);
      if (fused_mode == 2)
        fused_render16_kernel<1><<<(unsigned)nblk_total, FR_T, smem, st>>>(in, num_samples, num_ch, Hw, TW, WN, L, ov, skip,
                                                                         out_rows, out);
      else
        fused_render16_kernel<0><<<(unsigned)nblk_total, FR_T, smem, st>>>(in, num_samples, num_ch, Hw, TW, WN, L, ov, skip,
                                                                         out_rows, out);
      EM_CUDA(cudaGetLastError());
    }
    h->launches += 3;
    return;
  }
  if (fused_mode == 1 && N <= 4096 && N >= 8 && (num_samples % 2 == 0) && (ov % 2 == 0) &&
      (reinterpret_cast<uintptr_t>(in) % 16 == 0)) {
    const int M2 = N / 2;
    int logM = 0;
    while ((1 << logM) < M2) ++logM;
    cplx* WM = ar.get<cplx>((size_t)M2 / 2 + 1);
    cplx* WN = ar.get<cplx>((size_t)M2 + 1);
    render_twiddle_kernel<<<(M2 + 1 + 255) / 256, 256, 0, st>>>(M2, WM, WN);
    EM_CUDA(cudaGetLastError());
    const size_t smem = ((size_t)4 * M2 + 2 * (M2 + 1)) * sizeof(cplx);   // two channels side by side
    static size_t set_to = 0;
    if (smem > 48 * 1024 && smem > set_to) {
      EM_CUDA(cudaFuncSetAttribute(fused_render_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
      set_to = smem;
    }
    {
      ProfSpan ps(h, EM_PROF_RENDER_MAC);
      fused_render_kernel<<<(unsigned)nblk_total, 512, smem, st>>>(in, num_samples, num_ch, Hw, WM, WN, N, logM, L, ov, skip,
                                                                  out_rows, out);
      EM_CUDA(cudaGetLastError());
    }
    h->launches += 2;
    return;
  }

  ForwardStage fwd(h, rp, ar, in, num_samples, num_ch, N, L, ov, nbc);
  cplx* X = ar.get<cplx>((size_t)num_ch * nbc * F);
  cplx* Y = ar.get<cplx>((size_t)2 * chunk * F);
  double* yseg = ar.get<double>((size_t)2 * chunk * N);
  constexpr int BT = 4, CU = 4;
  for (long long b0 = 0; b0 < nblk_total; b0 += chunk) {
    const long long s0 = b0 * L;
    fwd.run(b0, std::min<long long>(chunk, nblk_total - b0), X);
    {
      ProfSpan ps(h, EM_PROF_RENDER_MAC);
      // Y is laid out [ear][chunk][F] for the fixed-size inverse plan (a partial last chunk
      // computes a few unused blocks)
      dim3 grid((unsigned)((F + 127) / 128), (unsigned)((chunk + BT - 1) / BT));
      spectral_mac_kernel<BT, CU><<<grid, 128, 0, st>>>(X, Hw, num_ch, nbc, chunk, F, Y);
      EM_CUDA(cudaGetLastError());
    }
    {
      ProfSpan ps(h, EM_PROF_RENDER_FFT);
      EM_FFT(cufftExecZ2D(rp.inv, reinterpret_cast<cufftDoubleComplex*>(Y), yseg));
    }
    {
      ProfSpan ps(h, EM_PROF_RENDER_STAGE);
      long long total = (long long)2 * chunk * L;
      unstage_output_kernel<<<(unsigned)((total + 255) / 256), 256, 0, st>>>(yseg, chunk, N, L, ov, s0, num_samples, skip,
                                                                           out_rows, out);
      EM_CUDA(cudaGetLastError());
    }
    h->launches += 2;
  }
  // stream-ordered: the arena's cudaFreeAsync calls queue behind the work above
}

void destroy_render_plans(emagls_ctx* h) {
  drop_plans(h->render_plans);
  drop_plans(h->tracked_plans);
}

}  // namespace emagls

using namespace emagls;

extern "C" {

int emagls_binaural_decode_dev(emagls_handle h, const double* in, long long num_samples, int num_ch,
                               const double* wL, const double* wR, int len, int compensate_delay,
                               double* out) {
  return guarded(h, [&] { binaural_decode_dev(h, in, num_samples, num_ch, wL, wR, len, compensate_delay, out); });
}

int emagls_binaural_decode(emagls_handle h, const double* in, long long num_samples, int num_ch,
                           const double* wL, const double* wR, int len, int compensate_delay, double* out) {
  return guarded(h, [&] {
    EM_REQUIRE(in && wL && wR && out && num_samples > 0 && num_ch > 0 && len > 0, "bad argument");
    cudaStream_t st = h->stream;
    Arena ar(st);
    const long long skip = compensate_delay ? (len / 2 - 1) : 0;
    const long long out_rows = num_samples - skip;
    EM_REQUIRE(out_rows > 0, "signal shorter than the compensated delay");
    double* d_in = ar.upload(in, (size_t)num_samples * num_ch);
    double* d_wL = ar.upload(wL, (size_t)len * num_ch);
    double* d_wR = ar.upload(wR, (size_t)len * num_ch);
    double* d_out = ar.get<double>((size_t)out_rows * 2);
    binaural_decode_dev(h, d_in, num_samples, num_ch, d_wL, d_wR, len, compensate_delay, d_out);
    EM_CUDA(cudaMemcpyAsync(out, d_out, (size_t)out_rows * 2 * sizeof(double), cudaMemcpyDeviceToHost, st));
    EM_CUDA(cudaStreamSynchronize(st));
  });
}

}  // extern "C"
