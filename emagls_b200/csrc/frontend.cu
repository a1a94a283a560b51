// The callers either side of the design path / render (SURVEY.md section 8-f):
//   getRadialFilter / applyRadialFilter  (dependencies/getRadialFilter.m:1-71, applyRadialFilter.m:1-33)
//   SH / CH encoding of the raw recording (verifyEMagLs.m:235-236, testEMagLs.m:98-105)
//   rotation of an SH-domain signal        (dependencies/binauralDecode.m:26-30 -> rotateHOA_N3D)
//   getMagLsSphericalHeadFilter, getMagLsArrayDiffuseFilter (lib/*.m)
// All signal-rate work is HBM bound: one pass over the recording per operator, coalesced along the
// sample index (MATLAB's column-major layout makes the sample index the contiguous one).
#include <cufft.h>
#include <algorithm>
#include <cmath>
#include <cstdlib>
#include <vector>
#include "engine.h"
#include "shrot.cuh"
#include "special.cuh"

namespace emagls {
namespace {

#define EM_FFT(expr)                                                                              \
  do {                                                                                            \
    cufftResult _r = (expr);                                                                      \
    if (_r != CUFFT_SUCCESS)                                                                      \
      throw ::emagls::Fail{EMAGLS_ERR_CUDA, std::string(#expr) + ": cufft error " + std::to_string((int)_r)}; \
  } while (0)

// getFadeWindow(irLen, relFadeLen) (dependencies/getFadeWindow.m:9-16)
__device__ inline double fade_window_rel(int tp, int len, double rel) {
  const int nf = (int)floor(rel * (double)len + 0.5);
  if (nf <= 0) return 1.0;
  const double den = (double)(2 * nf - 1);
  if (tp < nf) return 0.5 * (1.0 - cos(2.0 * 3.141592653589793 * (double)tp / den));
  if (tp >= len - nf) {
    const int q = tp - (len - nf) + nf;
    return 0.5 * (1.0 - cos(2.0 * 3.141592653589793 * (double)q / den));
  }
  return 1.0;
}

// ------------------------------------------------------------------------------------------
// getRadialFilter.m:42-70.  out[k*(N+1)+n]; kind: 1 tikhonov, 2 softlimit, 3 full.
// ------------------------------------------------------------------------------------------
__global__ void radial_filter_kernel(int N, const double* __restrict__ kr, int K, int array_type, int kind,
                                     double regul, double gain_lin, int nan_to_zero, cplx* __restrict__ out) {
  const int k = blockIdx.x * blockDim.x + threadIdx.x;
  if (k >= K) return;
  cplx b[MAX_SH_ORDER + 2];
  modal_coeffs(N, kr[k], array_type, b);
  for (int n = 0; n <= N; ++n) {
    const cplx bn = b[n];
    const double a2 = cabs2(bn);
    cplx r;
    if (kind == 1) {
      const double inv = 1.0 / (a2 + regul);                 // conj(b) ./ (conj(b).*b + regulConst)
      r = mk(bn.x * inv, -bn.y * inv);
    } else if (kind == 2) {
      const double a = sqrt(a2);                             // 2g/pi * |b| ./ b .* atan(pi ./ (2 g |b|))
      const double s = 2.0 * gain_lin / 3.141592653589793 * atan(3.141592653589793 / (2.0 * gain_lin * a));
      const cplx u = cdiv(mk(a, 0.0), bn);
      r = mk(u.x * s, u.y * s);
    } else {
      r = cdiv(mk(1.0, 0.0), bn);                            // 1 ./ b
    }
    if (k == K - 1) r = mk(sqrt(cabs2(r)), 0.0);             // radFilts(end,:) = abs(radFilts(end,:))
    if (nan_to_zero && (isnan(r.x) || isnan(r.y))) r = mk(0.0, 0.0);   // applyRadialFilter.m:10
    out[(long long)k * (N + 1) + n] = r;
  }
}

// ------------------------------------------------------------------------------------------
// Positive-frequency spectrum -> taps (conjugate extension, ifft, applySubsampleDelay, crop, fade):
//   out[t + len*ch] = fade(t)/nfft * sum_k c_k Re( W[ch][k] ramp_k exp(+2 pi i k (t+lo)/nfft) )
// with ramp_k = exp(-2 pi i omega_k delay) (real part at Nyquist, applySubsampleDelay.m:10-13) and
// c_k = 1 for DC/Nyquist, 2 otherwise.  The delay is circular, as in the reference.
// ------------------------------------------------------------------------------------------
__global__ void spectrum_ir_kernel(const cplx* __restrict__ W, long long w_ch_stride, long long w_k_stride,
                                   int nch, int K, int nfft, int len, int lo, double delay, double rel_fade,
                                   double* __restrict__ out) {
  const int t = blockIdx.x * blockDim.x + threadIdx.x, ch = blockIdx.y;
  if (t >= len || ch >= nch) return;
  const cplx* w = W + (long long)ch * w_ch_stride;
  double acc = 0.0;
  for (int k = 0; k < K; ++k) {
    const double omega = (double)k * (0.5 / (double)(K - 1));
    double rs, rc;
    sincos(-2.0 * 3.141592653589793 * omega * delay, &rs, &rc);
    if (k == K - 1) rs = 0.0;
    const long long r = ((long long)k * (t + lo)) % nfft;
    double es, ec;
    sincospi(2.0 * (double)r / (double)nfft, &es, &ec);
    const double pr = rc * ec - rs * es, pi_ = rc * es + rs * ec;
    const cplx v = w[(long long)k * w_k_stride];
    const double ck = (k == 0 || k == K - 1) ? 1.0 : 2.0;
    // Re(v * p); DC and Nyquist of a conjugate-symmetric spectrum contribute their real parts only
    const double term = (k == 0 || k == K - 1) ? v.x * pr : (v.x * pr - v.y * pi_);
    acc = fma(ck, term, acc);
  }
  out[(long long)ch * len + t] = acc * fade_window_rel(t, len, rel_fade) / (double)nfft;
}

// ------------------------------------------------------------------------------------------
// per-channel FIR (fftfilt of every column with its own filter), overlap-save
// ------------------------------------------------------------------------------------------
// xp[j][i] = in[ch][b*L - ov + i] (zero outside [0, n)); global block gb = c0 + j, ch = gb / nb, b = gb % nb
__global__ void fir_stage_kernel(const double* __restrict__ in, long long n, int nb, int N, int L, int ov,
                                 long long c0, long long cnt, double* __restrict__ xp) {
  const long long idx = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (idx >= cnt * N) return;
  const long long j = idx / N;
  const int i = (int)(idx % N);
  const long long gb = c0 + j;
  const long long ch = gb / nb, b = gb % nb;
  const long long s = b * L - ov + i;
  xp[idx] = (s >= 0 && s < n) ? in[ch * n + s] : 0.0;
}

__global__ void fir_pad_kernel(const double* __restrict__ filt, int flen, int nf, int N, double* __restrict__ wp) {
  const int idx = blockIdx.x * blockDim.x + threadIdx.x;
  if (idx >= nf * N) return;
  const int t = idx % N, f = idx / N;
  wp[idx] = t < flen ? filt[(long long)f * flen + t] : 0.0;
}

// X[j][f] *= Hf[map[ch(j)]][f]
__global__ void fir_mul_kernel(cplx* __restrict__ X, const cplx* __restrict__ Hf, const int* __restrict__ map,
                               int nb, int F, long long c0, long long cnt) {
  const long long idx = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (idx >= cnt * F) return;
  const long long j = idx / F;
  const int f = (int)(idx % F);
  const int ch = (int)((c0 + j) / nb);
  X[idx] = cmul(X[idx], Hf[(long long)map[ch] * F + f]);
}

__global__ void fir_unstage_kernel(const double* __restrict__ y, int nb, int N, int L, int ov, long long c0,
                                   long long cnt, long long n_total, long long skip, long long out_rows,
                                   double* __restrict__ out) {
  const long long idx = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (idx >= cnt * L) return;
  const long long j = idx / L;
  const int i = (int)(idx % L);
  const long long gb = c0 + j;
  const long long ch = gb / nb, b = gb % nb;
  const long long s = b * L + i;
  if (s >= n_total || s < skip) return;
  out[ch * out_rows + (s - skip)] = y[j * N + ov + i] * (1.0 / (double)N);
}

cufftHandle fir_plan(emagls_ctx* h, int N, int batch, int inverse) {
  for (auto& p : h->fir_plans)
    if (p.N == N && p.batch == batch && p.inverse == inverse) return p.plan;
  int n[1] = {N};
  cufftHandle pl = 0;
  EM_FFT(cufftPlanMany(&pl, 1, n, nullptr, 1, 0, nullptr, 1, 0, inverse ? CUFFT_Z2D : CUFFT_D2Z, batch));
  EM_FFT(cufftSetStream(pl, h->stream));
  if (h->fir_plans.size() >= 8) { cufftDestroy(h->fir_plans.front().plan); h->fir_plans.erase(h->fir_plans.begin()); }
  h->fir_plans.push_back({N, batch, inverse, pl});
  return pl;
}

// out[(s - skip) + out_rows*ch] = sum_t filt[t + flen*map[ch]] * in[(s - t) + n*ch], s in [skip, n_total)
void fir_channels_dev(emagls_ctx* h, Arena& ar, const double* in, long long n, int C, const double* filt, int flen,
                      int nf, const int* map_host, long long n_total, long long skip, double* out) {
  cudaStream_t st = h->stream;
  const long long out_rows = n_total - skip;
  const int ov = flen & ~1;                                // even, >= flen - 1
  int N = 16;
  while (N < 2 * flen) N <<= 1;
  const int want = 4 * N;                                  // 8 x the filter length amortises the overlap
  while (N < want && (long long)(N - ov) < n_total) N <<= 1;
  const int L = N - ov, F = N / 2 + 1;
  const long long nb = (n_total + L - 1) / L, TB = nb * C;
  EM_REQUIRE(nb < (1LL << 31), "signal too long");
  size_t free_b = 0, total_b = 0;
  EM_CUDA(cudaMemGetInfo(&free_b, &total_b));
  double budget = std::min(0.3 * (double)free_b, 8.0 * 1073741824.0);
  if (const char* e = getenv("EMAGLS_FIR_WS_MB")) budget = std::max(1.0, atof(e)) * 1048576.0;   // tests: force chunking
  const double per_block = (double)N * 8 + (double)F * 16;
  const long long Bc = std::max<long long>(1, std::min<long long>(TB, (long long)(budget / per_block)));
  int* map = ar.upload(map_host, C);
  cplx* Hf = ar.get<cplx>((size_t)nf * F);
  {
    double* wp = ar.get<double>((size_t)nf * N);
    fir_pad_kernel<<<(nf * N + 255) / 256, 256, 0, st>>>(filt, flen, nf, N, wp);
    EM_CUDA(cudaGetLastError());
    EM_FFT(cufftExecD2Z(fir_plan(h, N, nf, 0), wp, reinterpret_cast<cufftDoubleComplex*>(Hf)));
    h->launches += 1;
  }
  double* xp = ar.get<double>((size_t)Bc * N);
  cplx* X = ar.get<cplx>((size_t)Bc * F);
  for (long long c0 = 0; c0 < TB; c0 += Bc) {
    const long long cnt = std::min(Bc, TB - c0);
    {
      ProfSpan ps(h, EM_PROF_RENDER_STAGE);
      const long long tot = cnt * N;
      fir_stage_kernel<<<(unsigned)((tot + 255) / 256), 256, 0, st>>>(in, n, (int)nb, N, L, ov, c0, cnt, xp);
      EM_CUDA(cudaGetLastError());
    }
    {
      ProfSpan ps(h, EM_PROF_RENDER_FFT);
      EM_FFT(cufftExecD2Z(fir_plan(h, N, (int)cnt, 0), xp, reinterpret_cast<cufftDoubleComplex*>(X)));
    }
    {
      ProfSpan ps(h, EM_PROF_RENDER_MAC);
      const long long tot = cnt * F;
      fir_mul_kernel<<<(unsigned)((tot + 255) / 256), 256, 0, st>>>(X, Hf, map, (int)nb, F, c0, cnt);
      EM_CUDA(cudaGetLastError());
    }
    {
      ProfSpan ps(h, EM_PROF_RENDER_FFT);
      EM_FFT(cufftExecZ2D(fir_plan(h, N, (int)cnt, 1), reinterpret_cast<cufftDoubleComplex*>(X), xp));
    }
    {
      ProfSpan ps(h, EM_PROF_RENDER_STAGE);
      const long long tot = cnt * L;
      fir_unstage_kernel<<<(unsigned)((tot + 255) / 256), 256, 0, st>>>(xp, (int)nb, N, L, ov, c0, cnt, n_total, skip,
                                                                       out_rows, out);
      EM_CUDA(cudaGetLastError());
    }
    h->launches += 3;
  }
}

// ------------------------------------------------------------------------------------------
// channel mixing: out[s + n*co] (element stride es, offset off) = sum_ci in[s + n*ci] * P[ci][co].
// One thread per (sample, group of OG output channels); P in shared memory; loads and stores are
// coalesced along the sample index.  HBM bound: (Cin + Cout) * 8 B per sample.
// ------------------------------------------------------------------------------------------
template <int OG>
__global__ void __launch_bounds__(1024)
channel_mix_kernel(const double* __restrict__ in, long long n, int Cin, const double* __restrict__ P, int Cout,
                   double* __restrict__ out, int es, int off) {
  extern __shared__ double mix_P[];   // [Cin][CoutPad], CoutPad = groups * OG
  const int groups = blockDim.y, CoutPad = groups * OG;
  const int tid = threadIdx.y * blockDim.x + threadIdx.x, nt = blockDim.x * blockDim.y;
  for (int i = tid; i < Cin * CoutPad; i += nt) {
    const int ci = i / CoutPad, co = i % CoutPad;
    mix_P[i] = co < Cout ? P[(long long)ci * Cout + co] : 0.0;
  }
  __syncthreads();
  const long long s = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (s >= n) return;
  const int g = threadIdx.y;
  double acc[OG];
#pragma unroll
  for (int j = 0; j < OG; ++j) acc[j] = 0.0;
  for (int ci = 0; ci < Cin; ++ci) {
    const double x = in[(long long)ci * n + s];
    const double* p = mix_P + ci * CoutPad + g * OG;
#pragma unroll
    for (int j = 0; j < OG; ++j) acc[j] = fma(x, p[j], acc[j]);
  }
#pragma unroll
  for (int j = 0; j < OG; ++j) {
    const int co = g * OG + j;
    if (co < Cout) out[((long long)co * n + s) * es + off] = acc[j];
  }
}

void channel_mix_dev(emagls_ctx* h, const double* in, long long n, int Cin, const double* P, int Cout, double* out,
                     int es, int off) {
  constexpr int OG = 8;
  const int groups = (Cout + OG - 1) / OG;
  EM_REQUIRE(groups <= 8 && Cin <= 64, "more than 64 channels are not supported");
  dim3 block(128, groups);
  const size_t smem = (size_t)Cin * groups * OG * sizeof(double);
  channel_mix_kernel<OG><<<(unsigned)((n + 127) / 128), block, smem, h->stream>>>(in, n, Cin, P, Cout, out, es, off);
  EM_CUDA(cudaGetLastError());
  h->launches += 1;
}

// pinv(E) for E = Y.' from the solver's output Lt [ear][pair][Mc]:  P[m][c] = part(Lt[(m&1)*npair + m/2][c])
__global__ void extract_enc_kernel(const cplx* __restrict__ Lt, int npair, int M, int Mc, int imag,
                                   double* __restrict__ P) {
  const int idx = blockIdx.x * blockDim.x + threadIdx.x;
  if (idx >= M * Mc) return;
  const int m = idx / Mc, c = idx % Mc;
  const cplx v = Lt[((long long)(m & 1) * npair + m / 2) * Mc + c];
  P[idx] = imag ? v.y : v.x;
}

// P[ci][co] = Rshd[co][ci] for Rshd = getSHrotMtx(E, N, 'real'); one CTA
__global__ void sh_rot_matrix_kernel(int order, Rot1 R1in, double* __restrict__ P) {
  extern __shared__ double rot_Rr[];
  __shared__ Rot1 R1;
  __shared__ int rotate;
  const int nsh = (order + 1) * (order + 1);
  if (threadIdx.x == 0) { R1 = R1in; rotate = 1; }
  sh_rot_real_bands(R1, &rotate, order, rot_Rr, threadIdx.x, blockDim.x);
  __syncthreads();
  for (int e = threadIdx.x; e < nsh * nsh; e += blockDim.x) {
    const int ci = e / nsh, co = e % nsh;
    P[e] = rot_Rr[co * nsh + ci];
  }
}

// ------------------------------------------------------------------------------------------
// diffuse-field responses of getMagLsSphericalHeadFilter.m:42-49 / getMagLsArrayDiffuseFilter.m:63-75
//   df(x) = rms(abs(x), 2) * sqrt(size(x, 2)) / (4 pi) = sqrt(sum |x|^2) / (4 pi)
// Gn [simN+1][nsh] complex: Gn[n][c] = sum_{s in order n} (Y_hi^H Y_lo)[s][c] in the caller's basis
// (the sum over a whole order is not invariant under the real/complex change of basis, so the result
// depends on shDefinition, as in the reference); nullptr: spherical-head filter only.
// ------------------------------------------------------------------------------------------
__global__ void diffuse_filter_kernel(int simN, int order, const double* __restrict__ kr, int K, int array_type,
                                      const cplx* __restrict__ Gn, int nsh, double* __restrict__ hi_df,
                                      double* __restrict__ lo_df, double* __restrict__ alias_df) {
  const int k = blockIdx.x * blockDim.x + threadIdx.x;
  if (k >= K) return;
  cplx b[MAX_SH_ORDER + 2];
  modal_coeffs(simN, kr[k], array_type, b);
  double hi = 0.0, lo = 0.0;
  for (int n = 0; n <= simN; ++n) {
    const double a2 = cabs2(b[n]) * (double)(2 * n + 1);
    hi += a2;
    if (n <= order) lo += a2;
  }
  const double FOURPI = 12.566370614359172;
  hi_df[k] = sqrt(hi) / FOURPI;
  lo_df[k] = sqrt(lo) / FOURPI;
  if (Gn) {
    double acc = 0.0;
    for (int c = 0; c < nsh; ++c) {
      cplx v = mk(0.0, 0.0);
      for (int n = 0; n <= simN; ++n) cfma(v, b[n], Gn[n * nsh + c]);
      acc += cabs2(v);
    }
    alias_df[k] = sqrt(acc) / FOURPI;
  }
}

// Gn[n][c] = sum_{s in order n} sum_m conj(Yhi[s][m]) * Ylo[c][m]   ([S][M], [nsh][M]; real or complex basis)
__global__ void diffuse_gn_kernel(const double* __restrict__ Yhi, const double* __restrict__ Ylo, int simN, int nsh,
                                  int M, int complex_basis, cplx* __restrict__ Gn) {
  const int idx = blockIdx.x * blockDim.x + threadIdx.x;
  if (idx >= (simN + 1) * nsh) return;
  const int n = idx / nsh, c = idx % nsh;
  cplx acc = mk(0.0, 0.0);
  for (int s = n * n; s < (n + 1) * (n + 1); ++s)
    for (int m = 0; m < M; ++m) {
      if (complex_basis) {
        cfmac(acc, reinterpret_cast<const cplx*>(Yhi)[(long long)s * M + m],
              reinterpret_cast<const cplx*>(Ylo)[(long long)c * M + m]);
      } else {
        acc.x = fma(Yhi[(long long)s * M + m], Ylo[(long long)c * M + m], acc.x);
      }
    }
  Gn[idx] = acc;
}

// W[k] = 1 / (hi/lo) [* hi / (alias / alias[0])]
__global__ void diffuse_combine_kernel(const double* __restrict__ hi, const double* __restrict__ lo,
                                       const double* __restrict__ alias, int K, cplx* __restrict__ W) {
  const int k = blockIdx.x * blockDim.x + threadIdx.x;
  if (k >= K) return;
  double w = 1.0 / (hi[k] / lo[k]);                         // W_Shf
  if (alias) w *= hi[k] / (alias[k] / alias[0]);            // .* W_Alias
  W[k] = mk(w, 0.0);
}

__global__ void symmetric_spectrum_kernel(const cplx* __restrict__ W, int K, int nfft, double* __restrict__ out) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= nfft) return;
  out[i] = W[i < K ? i : nfft - i].x;
}

int radial_kind_checked(const emagls_radial_params* rp) {
  EM_REQUIRE(rp, "null argument");
  if (rp->kind < EMAGLS_RADIAL_NONE || rp->kind > EMAGLS_RADIAL_FULL)
    throw Fail{EMAGLS_ERR_INVALID, "Unkown radialFilter parameter"};   // getRadialFilter.m:65
  EM_REQUIRE(rp->array_type == EMAGLS_ARRAY_RIGID || rp->array_type == EMAGLS_ARRAY_OPEN, "Wrong array type");
  return rp->kind;
}

}  // namespace

// radFilts [K][(N+1)] on the device (row index k); 'none' -> ones
void radial_filter_dev(emagls_ctx* h, Arena& ar, const emagls_config& cfg, const emagls_radial_params& rp, int order,
                       double fs, double radius, int nfft, int nan_to_zero, cplx* out) {
  EM_REQUIRE(order >= 0 && order <= MAX_SH_ORDER, "order out of range");
  EM_REQUIRE(nfft > 0 && nfft % 2 == 0, "nfft must be even");
  const int K = nfft / 2 + 1;
  std::vector<double> kr = kr_table(cfg, fs, radius, K);
  if (rp.kind == EMAGLS_RADIAL_NONE) {
    std::vector<cplx> ones((size_t)K * (order + 1), mk(1.0, 0.0));
    EM_CUDA(cudaMemcpyAsync(out, ones.data(), ones.size() * sizeof(cplx), cudaMemcpyHostToDevice, h->stream));
    EM_CUDA(cudaStreamSynchronize(h->stream));
    return;
  }
  const double g = std::pow(10.0, rp.noise_gain_db / 20.0);
  radial_filter_kernel<<<(K + 63) / 64, 64, 0, h->stream>>>(order, ar.upload(kr.data(), K), K, rp.array_type, rp.kind,
                                                          rp.regul_const, g, nan_to_zero, out);
  EM_CUDA(cudaGetLastError());
  h->launches += 1;
}

long long radial_out_rows(long long num_samples, int nfft) { return std::max<long long>(num_samples, nfft) - nfft / 2; }

// applyRadialFilter.m:9-31 with device pointers; out [(max(n, nfft) - nfft/2) x (order+1)^2]
void apply_radial_filter_dev(emagls_ctx* h, const emagls_config& cfg, const emagls_radial_params& rp, const double* in,
                             long long n, int order, double fs, double radius, int nfft, double* out) {
  EM_REQUIRE(in && out && n > 0, "empty input");
  cudaStream_t st = h->stream;
  Arena ar(st);
  const int K = nfft / 2 + 1, L1 = order + 1, nsh = L1 * L1;
  cplx* rad = ar.get<cplx>((size_t)K * L1);
  radial_filter_dev(h, ar, cfg, rp, order, fs, radius, nfft, 1, rad);
  double* ir = ar.get<double>((size_t)nfft * L1);
  {
    dim3 grid((nfft + 127) / 128, L1);
    spectrum_ir_kernel<<<grid, 128, 0, st>>>(rad, 1, L1, L1, K, nfft, nfft, 0, (double)(nfft / 2), 0.05, ir);
    EM_CUDA(cudaGetLastError());
    h->launches += 1;
  }
  std::vector<int> map(nsh);
  for (int n2 = 0; n2 <= order; ++n2)
    for (int c = n2 * n2; c < (n2 + 1) * (n2 + 1); ++c) map[c] = n2;   // sh_repToOrder
  const long long n_total = std::max<long long>(n, nfft);              // applyRadialFilter.m:24-27
  fir_channels_dev(h, ar, in, n, nsh, ir, nfft, L1, map.data(), n_total, nfft / 2, out);
}

// verifyEMagLs.m:235-236: out [n x Mc] = in [n x M] * pinv(Y.'), Y = getSH(order, mics) (kind 0) or
// getCH(order, mic_azi) (kind 1).  Complex basis: out interleaved complex.
void encode_dev(emagls_ctx* h, const emagls_config& cfg, int kind, const double* in, long long n, int M,
                const double* mic_azi, const double* mic_zen, int order, double* out) {
  EM_REQUIRE(in && out && mic_azi && (mic_zen || kind == 1) && n > 0 && M > 0, "empty input");
  EM_REQUIRE(order >= 0 && order <= MAX_SH_ORDER, "order out of range");
  cudaStream_t st = h->stream;
  Arena ar(st);
  const int Mc = kind == 0 ? (order + 1) * (order + 1) : 2 * order + 1;
  const int cb = cfg.basis == EMAGLS_BASIS_COMPLEX ? 1 : 0;
  EM_REQUIRE(Mc <= 64 && M <= 64, "more than 64 channels are not supported");
  EM_REQUIRE(M >= Mc, "fewer microphones than harmonics");
  cplx* At = ar.get<cplx>((size_t)M * Mc);
  if (kind == 0) {
    double* Y = ar.get<double>((size_t)M * Mc * 2);
    EM_CUDA(launch_sh_angles(st, order, mic_azi, mic_zen, M, cb, Y));
    EM_CUDA(launch_sh_rows(st, Y, M, Mc, cb, At));
    h->launches += 2;
  } else {
    EM_CUDA(launch_ch_rows(st, order, mic_azi, M, cb, At));
    h->launches += 1;
  }
  cplx* Lt = unclipped_pinv_dev(h, ar, At, M, Mc);
  double* P = ar.get<double>((size_t)M * Mc);
  for (int part = 0; part <= cb; ++part) {
    extract_enc_kernel<<<(M * Mc + 255) / 256, 256, 0, st>>>(Lt, (M + 1) / 2, M, Mc, part, P);
    EM_CUDA(cudaGetLastError());
    h->launches += 1;
    channel_mix_dev(h, in, n, M, P, Mc, out, cb ? 2 : 1, part);
  }
}

// rotateHOA_N3D(in, yaw, pitch, roll) (called at binauralDecode.m:29; body restated in oracle/frontend_oracle.py)
void rotate_sh_dev(emagls_ctx* h, const double* in, long long n, int order, double yaw, double pitch, double roll,
                   double* out) {
  EM_REQUIRE(in && out && n > 0, "empty input");
  EM_REQUIRE(order >= 0 && (order + 1) * (order + 1) <= 64, "more than 64 channels are not supported");
  cudaStream_t st = h->stream;
  Arena ar(st);
  const int nsh = (order + 1) * (order + 1);
  // euler2rotationMatrix(-yaw, -pitch, roll, 'zyx') = Rx(roll) * Ry(-pitch) * Rz(-yaw)  (euler2rotationMatrix.m:19-50)
  const double a = -yaw, b = -pitch, g = roll;
  const double Rz[3][3] = {{std::cos(a), std::sin(a), 0}, {-std::sin(a), std::cos(a), 0}, {0, 0, 1}};
  const double Ry[3][3] = {{std::cos(b), 0, -std::sin(b)}, {0, 1, 0}, {std::sin(b), 0, std::cos(b)}};
  const double Rx[3][3] = {{1, 0, 0}, {0, std::cos(g), std::sin(g)}, {0, -std::sin(g), std::cos(g)}};
  double T[3][3], E[3][3];
  for (int i = 0; i < 3; ++i)
    for (int j = 0; j < 3; ++j) { double v = 0; for (int q = 0; q < 3; ++q) v += Ry[i][q] * Rz[q][j]; T[i][j] = v; }
  for (int i = 0; i < 3; ++i)
    for (int j = 0; j < 3; ++j) { double v = 0; for (int q = 0; q < 3; ++q) v += Rx[i][q] * T[q][j]; E[i][j] = v; }
  Rot1 R1;
  R1.r[0][0] = E[1][1]; R1.r[0][1] = E[1][2]; R1.r[0][2] = E[1][0];
  R1.r[1][0] = E[2][1]; R1.r[1][1] = E[2][2]; R1.r[1][2] = E[2][0];
  R1.r[2][0] = E[0][1]; R1.r[2][1] = E[0][2]; R1.r[2][2] = E[0][0];
  double* P = ar.get<double>((size_t)nsh * nsh);
  sh_rot_matrix_kernel<<<1, 256, (size_t)nsh * nsh * sizeof(double), st>>>(order, R1, P);
  EM_CUDA(cudaGetLastError());
  h->launches += 1;
  channel_mix_dev(h, in, n, nsh, P, nsh, out, 1, 0);
}

// getMagLsSphericalHeadFilter (mics == nullptr) / getMagLsArrayDiffuseFilter; w [len], Wfull [nfft] or nullptr
void diffuse_filter_dev(emagls_ctx* h, const emagls_config& cfg, double radius, const double* mic_azi,
                        const double* mic_zen, int M, int order, double fs, int len, double* w, double* Wfull) {
  EM_REQUIRE(w && len > 0, "empty input");
  cudaStream_t st = h->stream;
  Arena ar(st);
  const BinGrid bg = bin_grid(cfg, len, fs, 0);
  EM_REQUIRE(bg.nfft % 2 == 0, "nfft must be even");
  const int nfft = bg.nfft, K = bg.K;
  const int simN = (int)std::ceil(fs * M_PI * radius / cfg.speed_of_sound);   // no max(order, .) here (:38)
  EM_REQUIRE(simN <= MAX_SH_ORDER && order <= MAX_SH_ORDER, "simulation order too high");
  EM_REQUIRE(order <= simN, "order above the simulation order (reference indexes out of range here)");
  const int nsh = (order + 1) * (order + 1), S = (simN + 1) * (simN + 1);
  std::vector<double> kr = kr_table(cfg, fs, radius, K);
  double* hi = ar.get<double>(K);
  double* lo = ar.get<double>(K);
  double* alias = nullptr;
  cplx* Gn = nullptr;
  const int cb = cfg.basis == EMAGLS_BASIS_COMPLEX ? 1 : 0;
  if (mic_azi) {
    EM_REQUIRE(mic_zen && M > 0, "null argument");
    double* Yhi = ar.get<double>((size_t)S * M * 2);
    double* Ylo = ar.get<double>((size_t)nsh * M * 2);
    EM_CUDA(launch_sh_angles(st, simN, mic_azi, mic_zen, M, cb, Yhi));
    EM_CUDA(launch_sh_angles(st, order, mic_azi, mic_zen, M, cb, Ylo));
    Gn = ar.get<cplx>((size_t)(simN + 1) * nsh);
    diffuse_gn_kernel<<<((simN + 1) * nsh + 127) / 128, 128, 0, st>>>(Yhi, Ylo, simN, nsh, M, cb, Gn);
    EM_CUDA(cudaGetLastError());
    alias = ar.get<double>(K);
    h->launches += 3;
  }
  diffuse_filter_kernel<<<(K + 63) / 64, 64, 0, st>>>(simN, order, ar.upload(kr.data(), K), K, EMAGLS_ARRAY_RIGID, Gn,
                                                      nsh, hi, lo, alias);
  cplx* W = ar.get<cplx>(K);
  diffuse_combine_kernel<<<(K + 127) / 128, 128, 0, st>>>(hi, lo, alias, K, W);
  spectrum_ir_kernel<<<dim3((len + 127) / 128, 1), 128, 0, st>>>(W, 0, 1, 1, K, nfft, len, nfft / 2 - len / 2,
                                                                 (double)(nfft / 2), 0.15, w);
  EM_CUDA(cudaGetLastError());
  h->launches += 3;
  if (Wfull) {
    symmetric_spectrum_kernel<<<(nfft + 127) / 128, 128, 0, st>>>(W, K, nfft, Wfull);
    EM_CUDA(cudaGetLastError());
    h->launches += 1;
  }
}

void destroy_fir_plans(emagls_ctx* h) {
  for (auto& p : h->fir_plans) cufftDestroy(p.plan);
  h->fir_plans.clear();
}

}  // namespace emagls

using namespace emagls;

extern "C" {

void emagls_radial_params_default(emagls_radial_params* rp) {
  if (!rp) return;
  rp->kind = EMAGLS_RADIAL_TIKHONOV;      // getRadialFilter.m:9-11
  rp->regul_const = 1e-2;                 // :48-50
  rp->noise_gain_db = 20.0;               // getSMAIRMatrix.m:61-63
  rp->array_type = EMAGLS_ARRAY_RIGID;
}

int emagls_radial_filter(emagls_handle h, const emagls_config* cfg, const emagls_radial_params* rp, int order,
                         double fs, double sma_radius, int nfft, double* out) {
  return guarded(h, [&] {
    EM_REQUIRE(cfg && out, "null argument");
    radial_kind_checked(rp);
    Arena ar(h->stream);
    const size_t n = (size_t)(nfft / 2 + 1) * (order + 1);
    cplx* d = ar.get<cplx>(n);
    radial_filter_dev(h, ar, *cfg, *rp, order, fs, sma_radius, nfft, 0, d);
    // device layout [k][n] -> column-major [K x (order+1)]
    std::vector<cplx> tmp(n);
    EM_CUDA(cudaMemcpyAsync(tmp.data(), d, n * sizeof(cplx), cudaMemcpyDeviceToHost, h->stream));
    EM_CUDA(cudaStreamSynchronize(h->stream));
    const int K = nfft / 2 + 1, L1 = order + 1;
    for (int k = 0; k < K; ++k)
      for (int q = 0; q < L1; ++q) {
        out[2 * ((size_t)q * K + k)] = tmp[(size_t)k * L1 + q].x;
        out[2 * ((size_t)q * K + k) + 1] = tmp[(size_t)k * L1 + q].y;
      }
  });
}

long long emagls_apply_radial_filter_rows(long long num_samples, int nfft) { return radial_out_rows(num_samples, nfft); }

int emagls_apply_radial_filter_dev(emagls_handle h, const emagls_config* cfg, const emagls_radial_params* rp,
                                   const double* in, long long num_samples, int order, double fs, double sma_radius,
                                   int nfft, double* out) {
  return guarded(h, [&] {
    EM_REQUIRE(cfg, "null argument");
    radial_kind_checked(rp);
    apply_radial_filter_dev(h, *cfg, *rp, in, num_samples, order, fs, sma_radius, nfft, out);
  });
}

int emagls_apply_radial_filter(emagls_handle h, const emagls_config* cfg, const emagls_radial_params* rp,
                               const double* in, long long num_samples, int order, double fs, double sma_radius,
                               int nfft, double* out) {
  return guarded(h, [&] {
    EM_REQUIRE(cfg && in && out && num_samples > 0, "null argument");
    radial_kind_checked(rp);
    EM_REQUIRE(order >= 0 && order <= MAX_SH_ORDER && nfft > 0 && nfft % 2 == 0, "bad argument");
    cudaStream_t st = h->stream;
    Arena ar(st);
    const size_t nsh = (size_t)(order + 1) * (order + 1);
    const long long rows = radial_out_rows(num_samples, nfft);
    double* d_in = ar.upload(in, (size_t)num_samples * nsh);
    double* d_out = ar.get<double>((size_t)rows * nsh);
    apply_radial_filter_dev(h, *cfg, *rp, d_in, num_samples, order, fs, sma_radius, nfft, d_out);
    EM_CUDA(cudaMemcpyAsync(out, d_out, (size_t)rows * nsh * sizeof(double), cudaMemcpyDeviceToHost, st));
    EM_CUDA(cudaStreamSynchronize(st));
  });
}

static int encode_host(emagls_handle h, const emagls_config* cfg, int kind, const double* in, long long n, int M,
                       const double* mic_azi, const double* mic_zen, int order, double* out) {
  return guarded(h, [&] {
    EM_REQUIRE(cfg && in && out && mic_azi && n > 0 && M > 0 && order >= 0, "null argument");
    cudaStream_t st = h->stream;
    Arena ar(st);
    const size_t Mc = kind == 0 ? (size_t)(order + 1) * (order + 1) : (size_t)2 * order + 1;
    const size_t on = (size_t)n * Mc * (cfg->basis == EMAGLS_BASIS_COMPLEX ? 2 : 1);
    double* d_out = ar.get<double>(on);
    encode_dev(h, *cfg, kind, ar.upload(in, (size_t)n * M), n, M, ar.upload(mic_azi, M),
               mic_zen ? ar.upload(mic_zen, M) : nullptr, order, d_out);
    EM_CUDA(cudaMemcpyAsync(out, d_out, on * sizeof(double), cudaMemcpyDeviceToHost, st));
    EM_CUDA(cudaStreamSynchronize(st));
  });
}

int emagls_sh_encode(emagls_handle h, const emagls_config* cfg, const double* in, long long num_samples, int num_mics,
                     const double* mic_azi, const double* mic_zen, int order, double* out) {
  if (!mic_zen) return EMAGLS_ERR_INVALID;
  return encode_host(h, cfg, 0, in, num_samples, num_mics, mic_azi, mic_zen, order, out);
}
int emagls_sh_encode_dev(emagls_handle h, const emagls_config* cfg, const double* in, long long num_samples,
                         int num_mics, const double* mic_azi, const double* mic_zen, int order, double* out) {
  return guarded(h, [&] {
    EM_REQUIRE(cfg && mic_zen, "null argument");
    encode_dev(h, *cfg, 0, in, num_samples, num_mics, mic_azi, mic_zen, order, out);
  });
}
int emagls_ch_encode(emagls_handle h, const emagls_config* cfg, const double* in, long long num_samples, int num_mics,
                     const double* mic_azi, int order, double* out) {
  return encode_host(h, cfg, 1, in, num_samples, num_mics, mic_azi, nullptr, order, out);
}

int emagls_rotate_sh_dev(emagls_handle h, const double* in, long long num_samples, int order, double yaw_rad,
                         double pitch_rad, double roll_rad, double* out) {
  return guarded(h, [&] { rotate_sh_dev(h, in, num_samples, order, yaw_rad, pitch_rad, roll_rad, out); });
}
int emagls_rotate_sh(emagls_handle h, const double* in, long long num_samples, int order, double yaw_rad,
                     double pitch_rad, double roll_rad, double* out) {
  return guarded(h, [&] {
    EM_REQUIRE(in && out && num_samples > 0 && order >= 0, "null argument");
    cudaStream_t st = h->stream;
    Arena ar(st);
    const size_t n = (size_t)num_samples * (order + 1) * (order + 1);
    double* d_out = ar.get<double>(n);
    rotate_sh_dev(h, ar.upload(in, n), num_samples, order, yaw_rad, pitch_rad, roll_rad, d_out);
    EM_CUDA(cudaMemcpyAsync(out, d_out, n * sizeof(double), cudaMemcpyDeviceToHost, st));
    EM_CUDA(cudaStreamSynchronize(st));
  });
}

int emagls_spherical_head_filter(emagls_handle h, const emagls_config* cfg, double mic_radius, int order, double fs,
                                 int len, double* w, double* W_full) {
  return guarded(h, [&] {
    EM_REQUIRE(cfg && w && len > 0, "null argument");
    cudaStream_t st = h->stream;
    Arena ar(st);
    const int nfft = bin_grid(*cfg, len, fs, 0).nfft;
    double* d_w = ar.get<double>(len);
    double* d_W = W_full ? ar.get<double>(nfft) : nullptr;
    diffuse_filter_dev(h, *cfg, mic_radius, nullptr, nullptr, 0, order, fs, len, d_w, d_W);
    EM_CUDA(cudaMemcpyAsync(w, d_w, (size_t)len * sizeof(double), cudaMemcpyDeviceToHost, st));
    if (W_full) EM_CUDA(cudaMemcpyAsync(W_full, d_W, (size_t)nfft * sizeof(double), cudaMemcpyDeviceToHost, st));
    EM_CUDA(cudaStreamSynchronize(st));
  });
}

int emagls_array_diffuse_filter(emagls_handle h, const emagls_config* cfg, double mic_radius, const double* mic_azi,
                                const double* mic_zen, int num_mics, int order, double fs, int len, double* w) {
  return guarded(h, [&] {
    EM_REQUIRE(cfg && w && mic_azi && mic_zen && num_mics > 0 && len > 0, "null argument");
    cudaStream_t st = h->stream;
    Arena ar(st);
    double* d_w = ar.get<double>(len);
    diffuse_filter_dev(h, *cfg, mic_radius, ar.upload(mic_azi, num_mics), ar.upload(mic_zen, num_mics), num_mics,
                       order, fs, len, d_w, nullptr);
    EM_CUDA(cudaMemcpyAsync(w, d_w, (size_t)len * sizeof(double), cudaMemcpyDeviceToHost, st));
    EM_CUDA(cudaStreamSynchronize(st));
  });
}

}  // extern "C"
