// Host orchestration of the model-based eMagLS design path (getEMagLs2Filters / getEMagLsFilters).
//
// Reference flow being reproduced (lib/getEMagLs2Filters.m:44-135), restructured for a batch of
// P = num_sets * num_orient problems.  With A_k = pwGrid_k.' = Y_h diag(b_k) Y_o^T (Y_o = real SH at
// the microphones seen from head orientation o, times pinv(Y_lo) for SH-domain output):
//   once per grid       : Y_h = getSH(simN, grid) = Q R (Householder), Gh = Y_h^T Y_h
//   once per array      : b_n(kr_k) for all bins                              (getSMAIRMatrix.m:107)
//   once per HRTF set   : group delays, H = fft(h) .* ramp, |H|, H*Q and H*Y_h for the LS bins
//   once per orientation: Y_o, E_o = R-blocks * Y_o^T (TSQR route), F_o = Y_o Gh-blocks Y_o^T (Gram route)
//   per bin k           : Gram route (no singular value clipped, decided by a rigorous certificate for
//                         cond(A_k^H A_k)):  G_k = sum conj(b_n) b_n' F_nn' (DMMA GEMM), inversion,
//                             W_k = ((t Y_h) .* conj(b_k)) Y_o^T G_k^-T
//                         TSQR route (clipping possible):  C = R diag(b_k) Y_o^T -> TSQR -> Jacobi ->
//                             W_k = (t Q) conj(Q_C) Pb
//                         with t = H_k (LS bins) or |H_k| .* exp(i angle(Y_h (b_k .* (Y_o^T W_{k-1}))))
//   tail                : DC fix, ifft, sub-sample shift, crop, fade folded into one GEMM per ear
#include <algorithm>
#include <cmath>
#include <cstdio>
#include <cstdlib>
#include <optional>
#include <string>
#include <vector>
#include "engine.h"
#include "gemm.cuh"
#include "special.cuh"

namespace emagls {

namespace {

struct EpiRamp {  // H = fft(h) .* exp_omega  (applySubsampleDelay.m:10-17), columns (2k, 2k+1) = (re, im)
  double* C; long long ldc; const cplx* ramp;
  __device__ __forceinline__ void operator()(int m, int n, double re, double im, int M, int N, int) const {
    if (m >= M || n >= N) return;
    cplx r = ramp[n >> 1];
    double* q = C + (long long)m * ldc + n;
    *reinterpret_cast<double2*>(q) = make_double2(re * r.x - im * r.y, re * r.y + im * r.x);
  }
};

// rows [(pair*2 + ear)*2 + c][D]: target t = pair*2 + ear is the unit vector e_t
__global__ void unit_rows_kernel(double* rows, int npair, int D) {
  long long idx = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (idx >= (long long)npair * 4 * D) return;
  const int d = (int)(idx % D), row = (int)(idx / D);
  rows[idx] = ((row & 1) == 0 && (row >> 1) == d) ? 1.0 : 0.0;
}

__global__ void sh_to_rows_kernel(const double* __restrict__ Y, int M, int S, int complex_basis,
                                  cplx* __restrict__ rows) {
  int idx = blockIdx.x * blockDim.x + threadIdx.x;
  if (idx >= M * S) return;
  int m = idx / S, s = idx % S;
  rows[idx] = complex_basis ? reinterpret_cast<const cplx*>(Y)[(long long)s * M + m] : mk(Y[(long long)s * M + m], 0.0);
}

__global__ void real_to_cplx_kernel(const double* in, long long n, cplx* out) {
  long long idx = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (idx < n) out[idx] = mk(in[idx], 0.0);
}

// At[m][c] = getCH(N, mic_azi, 'real')(m, c): [1, sqrt2 sin(q azi), sqrt2 cos(q azi)] ordered
// [0, -1, +1, -2, +2, ...] (dependencies/getCH.m:17-28)
__global__ void ch_rows_kernel(int N, const double* __restrict__ azi, int M, cplx* __restrict__ At) {
  int idx = blockIdx.x * blockDim.x + threadIdx.x;
  const int nch = 2 * N + 1;
  if (idx >= M * nch) return;
  const int m = idx / nch, c = idx % nch;
  double v = 1.0;
  if (c > 0) {
    const int q = (c + 1) / 2;
    double sn, cs;
    sincos((double)q * azi[m], &sn, &cs);
    v = 1.4142135623730951 * ((c & 1) ? sn : cs);
  }
  At[idx] = mk(v, 0.0);
}

__global__ void fill_kernel(double* p, int n, double v) {
  int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i < n) p[i] = v;
}

// L[c][m] = Re(W[(m&1)*npair + m/2][c])
__global__ void extract_pinv_kernel(const cplx* W, int npair, int Mc, int M, double* L) {
  int idx = blockIdx.x * blockDim.x + threadIdx.x;
  if (idx >= Mc * M) return;
  int c = idx / M, m = idx % M;
  L[idx] = W[((long long)(m & 1) * npair + m / 2) * Mc + c].x;
}

}  // namespace

cudaError_t launch_fill(cudaStream_t st, double* p, int n, double v) {
  fill_kernel<<<(n + 127) / 128, 128, 0, st>>>(p, n, v);
  return cudaGetLastError();
}
cudaError_t launch_sh_rows(cudaStream_t st, const double* Y, int M, int S, int complex_basis, cplx* rows) {
  sh_to_rows_kernel<<<(M * S + 255) / 256, 256, 0, st>>>(Y, M, S, complex_basis, rows);
  return cudaGetLastError();
}

BinGrid bin_grid(const emagls_config& cfg, int len, double fs, int T) {
  EM_REQUIRE(len >= T, "len too short");  // lib/getEMagLs2Filters.m:42
  EM_REQUIRE(len % 2 == 0, "len must be even");
  const int nfft = std::min(cfg.nfft_max_len, 2 * len);
  EM_REQUIRE(nfft / 2 >= len / 2, "len exceeds NFFT_MAX_LEN (reference indexes out of range here)");
  const int K = nfft / 2 + 1;
  return {nfft, K, (fs / 2.0) / (double)(K - 1)};
}
int BinGrid::kls1(double f_cut) const {
  const int k_cut = (int)std::ceil(f_cut / df);  // 1-based MATLAB index
  return std::min(std::max(k_cut - 1, 1), K);
}

int sim_order(const emagls_config& cfg, int order, double fs, double radius) {
  return std::max(order, (int)std::ceil(fs * M_PI * radius / cfg.speed_of_sound));
}

std::vector<double> kr_table(const emagls_config& cfg, double fs, double radius, int K) {
  std::vector<double> kr(K);
  const double df = (fs / 2.0) / (double)(K - 1);
  for (int k = 0; k < K; ++k) kr[k] = 2.0 * M_PI * ((double)k * df) / cfg.speed_of_sound * radius;
  return kr;
}

double median_of(std::vector<double> v) {
  size_t n = v.size();
  std::sort(v.begin(), v.end());
  return (n & 1) ? v[n / 2] : 0.5 * (v[n / 2 - 1] + v[n / 2]);
}

DesignShape design_shape(const emagls_config& cfg, Variant v, int M, int order, int len, int K, size_t P) {
  DesignShape s;
  s.nch = (v == Variant::EMAGLS2) ? M : (v == Variant::EMAGLS_SH ? (order + 1) * (order + 1) : 2 * order + 1);
  s.cplx = v != Variant::EMAGLS2 && cfg.basis == EMAGLS_BASIS_COMPLEX;
  s.filter_elems = (size_t)len * s.nch * P * (s.cplx ? 2 : 1);
  s.spectra_elems = (size_t)2 * K * s.nch * P * 2;
  return s;
}

// ---- complex SH / CH basis (shDefinition = 'complex', lib/getEMagLsFilters.m:117-120) -----------
// pwGrid_complex = conj(T) pwGrid_real with the unitary real->complex map Y_c = Y_r T^T
// (getSH.m:25-49, getCH.m:17-28), so every bin but DC obeys W_c = W_r T^T; the DC fix
// W(1,:) = real(W(2,:)) acts on the complex-basis coefficients (lib/getEMagLsFilters.m:110-111) and
// getShFreqDomainConjugate / getChFreqDomainConjugate make the remaining spectrum the image of a
// real-basis Hermitian one.  Hence
//   w_c = tail(W_r with DC := 0) T^T + fade/nfft * real(W_r(2,:) T^T)       (designers with a DC fix)
//   w_c = tail(W_r) T^T                                                     (MagLS / LS: no DC fix)
// T rows, SH (ACN, Condon-Shortley): m = 0: e_0; m > 0: (-1)^m (e_m + i e_-m)/sqrt2; m < 0: (e_|m| - i e_-|m|)/sqrt2.
// T rows, CH ([0,-1,+1,-2,+2,..]):   the same without the (-1)^m.
template <class V>
__device__ __forceinline__ cplx to_complex_basis(V ap_, V am_, int m, int kind);
template <>
__device__ __forceinline__ cplx to_complex_basis<double>(double ap, double am, int m, int kind) {
  const double r = 0.7071067811865476;
  if (m == 0) return mk(ap, 0.0);
  if (m > 0) { const double s = (kind == 0 && (m & 1)) ? -r : r; return mk(s * ap, s * am); }
  return mk(r * ap, -r * am);
}
template <>
__device__ __forceinline__ cplx to_complex_basis<cplx>(cplx ap, cplx am, int m, int kind) {
  const double r = 0.7071067811865476;
  if (m == 0) return ap;
  if (m > 0) { const double s = (kind == 0 && (m & 1)) ? -r : r; return mk(s * (ap.x - am.y), s * (ap.y + am.x)); }
  return mk(r * (ap.x + am.y), r * (ap.y - am.x));
}
// channel j -> m and the channel indices of (+|m|, -|m|)
__device__ __forceinline__ void basis_pair(int j, int kind, int& m, int& jp, int& jm) {
  if (kind == 0) {
    int n = (int)sqrt((double)j);
    while ((n + 1) * (n + 1) <= j) ++n;
    while (n * n > j) --n;
    m = j - n * n - n;
    const int am = m < 0 ? -m : m;
    jp = n * n + n + am; jm = n * n + n - am;
  } else {
    const int am = (j + 1) / 2;
    m = (j == 0) ? 0 : ((j & 1) ? -am : am);
    jp = 2 * am; jm = (am == 0) ? 0 : 2 * am - 1;
  }
}

// out (interleaved complex) [len x nch x P]; wr [len x nch x P] real-basis filters; optional DC term
// from this ear's real-basis spectra Wsp_e [P][nch][K]
__global__ void basis_change_filters_kernel(const double* __restrict__ wr, int kind, int nch, int len,
                                            long long P, const cplx* __restrict__ Wsp_e, int K, int nfft,
                                            cplx* __restrict__ out) {
  long long idx = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (idx >= P * nch * len) return;
  const int t = (int)(idx % len);
  const int j = (int)((idx / len) % nch);
  const long long p = idx / ((long long)len * nch);
  int m, jp, jm;
  basis_pair(j, kind, m, jp, jm);
  const long long ip = p * nch + jp, im = p * nch + jm;
  cplx v = to_complex_basis<double>(wr[ip * len + t], wr[im * len + t], m, kind);
  if (Wsp_e) {
    const cplx dc = to_complex_basis<cplx>(Wsp_e[ip * K + 1], Wsp_e[im * K + 1], m, kind);
    v.x += fade_window(t, len) / (double)nfft * dc.x;
  }
  out[idx] = v;
}

// in place: spectra rows [EP][nch][K] -> complex basis; dc_quirk: DC := real(bin 1) in the new basis
__global__ void basis_change_spectra_kernel(cplx* __restrict__ Wsp, int kind, int nch, int K, long long EP,
                                            int dc_quirk) {
  long long idx = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (idx >= EP * nch * K) return;
  const int k = (int)(idx % K);
  const int j = (int)((idx / K) % nch);
  const long long ep = idx / ((long long)K * nch);
  int m, jp, jm;
  basis_pair(j, kind, m, jp, jm);
  if (m < 0 || (dc_quirk && k == 0)) return;  // the thread of +m converts both rows (and bin 1 writes DC)
  cplx* rp = Wsp + (ep * nch + jp) * K;
  cplx* rm = Wsp + (ep * nch + jm) * K;
  const cplx ap = rp[k], am = rm[k];
  const cplx cp = to_complex_basis<cplx>(ap, am, m, kind), cm = to_complex_basis<cplx>(ap, am, -m, kind);
  rp[k] = cp;
  if (m > 0) rm[k] = cm;
  if (dc_quirk && k == 1) {
    rp[0] = mk(cp.x, 0.0);
    if (m > 0) rm[0] = mk(cm.x, 0.0);
  }
}

cudaError_t launch_basis_change_filters(cudaStream_t st, const double* wr, int kind, int nch, int len,
                                        long long P, const cplx* Wsp_e, int K, int nfft, cplx* out) {
  long long n = P * nch * len;
  basis_change_filters_kernel<<<(unsigned)((n + 255) / 256), 256, 0, st>>>(wr, kind, nch, len, P, Wsp_e, K, nfft, out);
  return cudaGetLastError();
}
cudaError_t launch_basis_change_spectra(cudaStream_t st, cplx* Wsp, int kind, int nch, int K, long long EP,
                                        int dc_quirk) {
  long long n = EP * nch * K;
  basis_change_spectra_kernel<<<(unsigned)((n + 255) / 256), 256, 0, st>>>(Wsp, kind, nch, K, EP, dc_quirk);
  return cudaGetLastError();
}

// median(grpdelay(sum(h,2), 1, f, fs)) per (set, ear)  (lib/getEMagLs2Filters.m:72-75)
std::vector<double> group_delays(emagls_ctx* h, Arena& ar, const double* hL, const double* hR, int T, int D,
                                 int K, double fs, int num_sets) {
  cudaStream_t st = h->stream;
  std::vector<double> grpD((size_t)num_sets * 2);
  const int nchunk = 32;
  double* partial = ar.get<double>((size_t)nchunk * T);
  double* hsum = ar.get<double>((size_t)num_sets * 2 * T);
  double* gd = ar.get<double>((size_t)num_sets * 2 * K);
  for (int s = 0; s < num_sets; ++s)
    for (int e = 0; e < 2; ++e) {
      const double* hp = (e == 0 ? hL : hR) + (size_t)s * T * D;
      EM_CUDA(launch_colsum(st, hp, T, D, partial, nchunk, hsum + ((size_t)s * 2 + e) * T));
      EM_CUDA(launch_grpdelay(st, hsum + ((size_t)s * 2 + e) * T, T, K, fs, gd + ((size_t)s * 2 + e) * K));
      h->launches += 3;
    }
  std::vector<double> gdh((size_t)num_sets * 2 * K);
  EM_CUDA(cudaMemcpyAsync(gdh.data(), gd, gdh.size() * sizeof(double), cudaMemcpyDeviceToHost, st));
  EM_CUDA(cudaStreamSynchronize(st));
  for (int i = 0; i < num_sets * 2; ++i)
    grpD[i] = median_of(std::vector<double>(gdh.begin() + (size_t)i * K, gdh.begin() + (size_t)(i + 1) * K));
  return grpD;
}

// Hd [D][2K] (interleaved complex rows) = fft(zero-padded h) .* exp(+i 2 pi omega delay_removed), the
// Nyquist factor real (applySubsampleDelay.m:10-17 with delay = -delay_removed; an integer
// delay_removed equals circshift(h, -delay_removed), lib/getEMagLsFiltersFromAtf.m:48-49).
void hrir_spectrum(emagls_ctx* h, Arena& ar, const double* hp, int T, int D, int K, const double* tw,
                   double delay_removed, double* Hd) {
  cudaStream_t st = h->stream;
  std::vector<cplx> ramp((size_t)K);
  for (int k = 0; k < K; ++k) {
    double omega = (double)k * (0.5 / (double)(K - 1));
    double ang = 2.0 * M_PI * omega * delay_removed;
    cplx r = mk(std::cos(ang), std::sin(ang));
    if (k == K - 1) r.y = 0.0;
    ramp[k] = r;
  }
  cplx* d_ramp = ar.upload(ramp.data(), ramp.size());
  GemmOperand A{hp, T, 1}, B{tw, T, 1};  // (pageable H2D copies are staged before upload() returns)
  EpiRamp epi{Hd, 2LL * K, d_ramp};
  EM_CUDA(launch_gemm(st, A, B, GemmShape{D, 2 * K, T}, epi));
  h->launches += 1;
}

// targets * Y_reg_inv for one steering matrix held as rows At [D][Mc] (lib/getEMagLs2Filters.m:87-94).
// rows: [(pair*2 + ear)*2 + {re,im}][D];  W: [ear][pair][Mc].
void regularized_apply_dev(emagls_ctx* h, Arena& ar, const cplx* At, int D, int Mc, const double* rows,
                           int npair, double regul, cplx* W) {
  cudaStream_t st = h->stream;
  const BlockPlan bp = make_block_plan(D, Mc);
  OperatorSet ops{};
  ops.v_stride = (long long)Mc * D; ops.tau_stride = (long long)bp.nblk * bp.MC;
  ops.pb_stride = (long long)Mc * Mc;
  ops.V = ar.get<cplx>(ops.v_stride); ops.tau = ar.get<cplx>(ops.tau_stride);
  ops.Pb = ar.get<cplx>(ops.pb_stride);
  ops.info = ar.get<int>(1);
  RowSource src{};
  src.At = At; src.at_bin_stride = 0; src.at_prob_stride = 0;
  EM_CUDA(launch_factor(st, bp, src, ops, 1, 0, 1, regul, 1));
  // every pair of targets shares the one operator set: chain_bwd indexes operators by j % oc and
  // solutions by global(j), so oc = 1 addresses the pairs through the set index
  ProbMap pm1{1, 0, 1};
  EM_CUDA(launch_chain_bwd(st, bp, ops, 0, 1, rows, 0, 0, 0, 1, 0, pm1, W, (long long)npair * Mc, 1, 0, 0, npair));
  h->launches += 2;
}

cplx* unclipped_pinv_dev(emagls_ctx* h, Arena& ar, const cplx* At, int M, int Mc) {
  const int npair = (M + 1) / 2;
  double* rows = ar.get<double>((size_t)npair * 4 * M);
  const long long n = (long long)npair * 4 * M;
  unit_rows_kernel<<<(unsigned)((n + 255) / 256), 256, 0, h->stream>>>(rows, npair, M);
  EM_CUDA(cudaGetLastError());
  h->launches += 1;
  cplx* Lt = ar.get<cplx>((size_t)2 * npair * Mc);
  regularized_apply_dev(h, ar, At, M, Mc, rows, npair, 0.0, Lt);
  return Lt;
}

void design_factored(emagls_ctx* h, const emagls_config& cfg, const DesignArgs& a) {
  cudaStream_t st = h->stream;
  // ---------------- reference arithmetic on the scalar parameters (lib/getEMagLs2Filters.m:42-48)
  EM_REQUIRE(a.T > 0 && a.D > 0 && a.M > 0 && a.len > 0, "empty input");
  EM_REQUIRE(a.num_sets >= 1 && a.num_orient >= 1, "empty batch");
  EM_REQUIRE(a.rotations != nullptr || a.num_orient == 1 || a.Y_mic != nullptr, "num_orient > 1 needs rotations");
  EM_REQUIRE((a.Y_hrir == nullptr) == (a.Y_mic == nullptr), "custom bases: Y_hrir and Y_mic must be given together");
  const BinGrid bg = bin_grid(cfg, a.len, a.fs, a.T);
  EM_REQUIRE(bg.nfft % 2 == 0, "nfft must be even");  // getSMAIRMatrix.m:89
  const int nfft = bg.nfft, K = bg.K;
  const int simN = sim_order(cfg, a.order, a.fs, a.mic_radius);
  EM_REQUIRE(simN <= MAX_SH_ORDER, "simulation order too high");
  const int S = (simN + 1) * (simN + 1);
  const int P = a.num_sets * a.num_orient;
  const DesignShape shape = design_shape(cfg, a.variant, a.M, a.order, a.len, K, P);
  const int Mc = shape.nch;
  EM_REQUIRE(Mc <= 64 && a.M <= 64, "more than 64 channels are not supported");
  if (a.variant != Variant::EMAGLS2) EM_REQUIRE(a.M >= Mc, "fewer microphones than output channels");
  if (a.D < S)
    throw Fail{EMAGLS_ERR_UNSUPPORTED, "HRIR grid has fewer directions than simulation harmonics"};
  EM_REQUIRE(S >= Mc, "fewer simulation harmonics than channels");
  const int D = a.D, T = a.T;
  // complex SH-domain output: solved in the real basis, converted at the tail (see above)
  const bool cplx_out = shape.cplx;
  const int basis_kind = (a.variant == Variant::EMA_CH) ? 1 : 0;
  const int dc_fix = cplx_out ? 0 : 1;
  // bins (0-based): LS 1 .. kls1-1, MagLS kls1 .. K-1
  const int kls1 = bg.kls1(std::max(cfg.f_cut_min, 500.0 * a.order));
  const int nLS = kls1 - 1;

  Arena ar(st);
  std::optional<ProfSpan> setup_span(std::in_place, h, EM_PROF_SETUP);
  // ---------------- grid: Y_h = Q R, Gh = Y_h^T Y_h
  double* Yh = ar.get<double>((size_t)S * D);
  double* Q = ar.get<double>((size_t)S * D);
  double* R = ar.get<double>((size_t)S * S);
  double* Gh = ar.get<double>((size_t)S * S);
  int* d_qrflag = ar.get<int>(1);
  // the single-CTA Cholesky kernel gives one column to a thread (S <= 1024); larger bases keep the Householder route
  bool chol_qr = S <= 1024 && getenv("EMAGLS_QR_HOUSEHOLDER") == nullptr;
  {
    if (a.Y_hrir)
      EM_CUDA(cudaMemcpyAsync(Yh, a.Y_hrir, (size_t)S * D * sizeof(double), cudaMemcpyDeviceToDevice, st));
    else
      EM_CUDA(launch_sh_angles(st, simN, a.grid_azi, a.grid_zen, D, 0, Yh));
    GemmOperand A0{Yh, D, 1}, B0{Yh, D, 1};
    EM_CUDA(launch_gemm(st, A0, B0, GemmShape{S, S, D}, EpiStore{Gh, S, 1.0}));
    h->launches += 2;
    EM_CUDA(cudaMemsetAsync(d_qrflag, 0, sizeof(int), st));
    if (chol_qr) {
      // CholeskyQR2 (setup_kernels.cu): nine launches; the flag is read after the group-delay synchronisation below
      double* R1 = ar.get<double>((size_t)S * S);
      double* R2 = ar.get<double>((size_t)S * S);
      double* Ri = ar.get<double>((size_t)S * S);
      double* Q1 = ar.get<double>((size_t)S * D);
      EM_CUDA(cudaMemcpyAsync(R1, Gh, (size_t)S * S * sizeof(double), cudaMemcpyDeviceToDevice, st));
      EM_CUDA(launch_chol_upper(st, R1, S, d_qrflag));
      EM_CUDA(launch_tri_inverse(st, R1, S, Ri));
      // Q1[i][d] = sum_j Rinv[j][i] Y_h[j][d]
      EM_CUDA(launch_gemm(st, GemmOperand{Ri, S, 0}, GemmOperand{Yh, D, 0}, GemmShape{S, D, S}, EpiStore{Q1, D, 1.0}));
      EM_CUDA(launch_gemm(st, GemmOperand{Q1, D, 1}, GemmOperand{Q1, D, 1}, GemmShape{S, S, D}, EpiStore{R2, S, 1.0}));
      EM_CUDA(launch_chol_upper(st, R2, S, d_qrflag));
      EM_CUDA(launch_tri_inverse(st, R2, S, Ri));
      EM_CUDA(launch_gemm(st, GemmOperand{Ri, S, 0}, GemmOperand{Q1, D, 0}, GemmShape{S, D, S}, EpiStore{Q, D, 1.0}));
      EM_CUDA(launch_tri_mul(st, R2, R1, S, R));
      h->launches += 9;
    }
  }
  auto householder_qr = [&]() {
    double* work = ar.get<double>((size_t)S * D + 2 * S);
    double* Ytmp = ar.get<double>((size_t)S * D);
    EM_CUDA(cudaMemcpyAsync(Ytmp, Yh, (size_t)S * D * sizeof(double), cudaMemcpyDeviceToDevice, st));
    EM_CUDA(launch_householder_qr(st, Ytmp, D, S, Q, R, work, &h->launches));  // destroys its input
  };
  if (!chol_qr) householder_qr();
  // ---------------- array: b_n table (minus sign, Nyquist real: getSMAIRMatrix.m:107,115-117)
  const std::vector<double> kr = kr_table(cfg, a.fs, a.mic_radius, K);
  double* d_kr = ar.upload(kr.data(), K);
  cplx* bn = ar.get<cplx>((size_t)K * (simN + 1));
  EM_CUDA(launch_modal(st, simN, d_kr, K, cfg.array_type, -1.0, 1, bn, simN + 1, 1));
  const int nqs = (simN + 1) * (simN + 2) / 2, nqa = std::max(1, simN * (simN + 1) / 2);
  double* bre = ar.get<double>((size_t)K * nqs);
  double* bim = ar.get<double>((size_t)K * nqa);
  EM_CUDA(launch_gram_beta(st, bn, simN, K, bre, bim));
  h->launches += 2;

  // ---------------- orientations: Y_o = getSH at the rotated microphones (times pinv(Y_lo))
  std::vector<int> rowoff(S), roword(S);
  long long Etot = 0;
  {
    int i = 0;
    for (int n = 0; n <= simN; ++n)
      for (int m = -n; m <= n; ++m, ++i) {
        roword[i] = n;
        rowoff[i] = (int)Etot;
        Etot += (long long)(simN + 1 - n) * Mc;
      }
  }
  int* d_rowoff = ar.upload(rowoff.data(), S);
  int* d_roword = ar.upload(roword.data(), S);
  double* Yo = nullptr;  // [num_orient][Mc][S]
  {
    double* Ym = ar.get<double>((size_t)a.num_orient * a.M * S);
    const double* mic_zen = a.mic_zen;
    if (!mic_zen) {  // equatorial array (lib/getEMagLsFiltersEMAinCH.m:57)
      double* z = ar.get<double>(a.M);
      EM_CUDA(launch_fill(st, z, a.M, 1.5707963267948966));
      mic_zen = z;
      h->launches += 1;
    }
    if (a.Y_mic)
      EM_CUDA(cudaMemcpyAsync(Ym, a.Y_mic, (size_t)a.num_orient * a.M * S * sizeof(double), cudaMemcpyDeviceToDevice, st));
    else
      EM_CUDA(launch_sh_mics(st, simN, a.mic_azi, mic_zen, a.M, a.rotations, a.num_orient, Ym));
    h->launches += 1;
    Yo = Ym;
    if (a.variant != Variant::EMAGLS2) {
      // L = pinv(Y_Hi(:, 1:(order+1)^2)) at the microphones as given (getSMAIRMatrix.m:102) or
      // pinv(getCH(order, micAzi)) (lib/getEMagLsFiltersEMAinCH.m:71), obtained from the same
      // factorisation kernel with the clip disabled.
      cplx* At = ar.get<cplx>((size_t)a.M * Mc);
      if (a.variant == Variant::EMAGLS_SH) {
        double* Ym0 = ar.get<double>((size_t)a.M * S);
        if (a.Y_mic)   // custom basis: Y_lo = the leading (order+1)^2 columns of the first orientation's matrix
          EM_CUDA(cudaMemcpyAsync(Ym0, a.Y_mic, (size_t)a.M * S * sizeof(double), cudaMemcpyDeviceToDevice, st));
        else
          EM_CUDA(launch_sh_mics(st, simN, a.mic_azi, mic_zen, a.M, nullptr, 1, Ym0));
        double* tmp = ar.get<double>((size_t)a.M * Mc);
        EM_CUDA(cudaMemcpy2DAsync(tmp, (size_t)Mc * sizeof(double), Ym0, (size_t)S * sizeof(double),
                                  (size_t)Mc * sizeof(double), a.M, cudaMemcpyDeviceToDevice, st));
        long long n = (long long)a.M * Mc;
        real_to_cplx_kernel<<<(unsigned)((n + 255) / 256), 256, 0, st>>>(tmp, n, At);
        h->launches += 2;
      } else {
        ch_rows_kernel<<<(a.M * Mc + 127) / 128, 128, 0, st>>>(a.order, a.mic_azi, a.M, At);
        h->launches += 1;
      }
      cplx* Wp = unclipped_pinv_dev(h, ar, At, a.M, Mc);
      double* L = ar.get<double>((size_t)Mc * a.M);
      extract_pinv_kernel<<<(Mc * a.M + 255) / 256, 256, 0, st>>>(Wp, (a.M + 1) / 2, Mc, a.M, L);
      double* Yeff = ar.get<double>((size_t)a.num_orient * Mc * S);
      EM_CUDA(launch_left_mul(st, L, Mc, a.M, Ym, a.num_orient, S, Yeff));
      EM_CUDA(cudaGetLastError());
      h->launches += 2;
      Yo = Yeff;
    }
  }

  // ---------------- HRTF sets: group delay, H, |H|, H*Q, H*Y_h
  const std::vector<double> grpD = group_delays(h, ar, a.hL, a.hR, T, D, K, a.fs, a.num_sets);
  if (chol_qr) {   // the stream is idle after the group-delay readback: the flag costs one 4-byte copy
    int qrflag = 0;
    EM_CUDA(cudaMemcpy(&qrflag, d_qrflag, sizeof(int), cudaMemcpyDeviceToHost));
    if (qrflag) householder_qr();   // badly conditioned direction grid: Householder route
  }
  // EXTENSION (default off): diffuse-field covariance constraint, see gram_kernels.cu
  const bool wdc = cfg.diffuseness_const != 0;
  EM_REQUIRE(!wdc || (cfg.basis == EMAGLS_BASIS_REAL && Mc <= 32),
             "the diffuseness constraint is implemented for the real SH basis and up to 32 channels");
  double* Rt = wdc ? ar.get<double>((size_t)a.num_sets * K * 4) : nullptr;           // target covariance [set][K][4]
  double* absH = ar.get<double>((size_t)a.num_sets * 2 * K * D);                     // [set][ear][K][D]
  const size_t ls_elems = (size_t)a.num_sets * 2 * std::max(nLS, 1) * 2 * S;         // [set][ear][kls][c][S]
  double* Tls = ar.get<double>(ls_elems);   // H * Q
  double* Zls = ar.get<double>(ls_elems);   // H * Y_h
  {
    double* tw = ar.get<double>((size_t)2 * K * T);
    EM_CUDA(launch_dft_twiddle(st, K, T, nfft, tw));
    h->launches += 1;
    double* Hd0 = ar.get<double>((size_t)D * 2 * K);
    double* Hd1 = wdc ? ar.get<double>((size_t)D * 2 * K) : Hd0;   // the constraint needs both ears' spectra at once
    for (int s = 0; s < a.num_sets; ++s)
      for (int e = 0; e < 2; ++e) {
        double* Hd = e == 0 ? Hd0 : Hd1;
        const double* hp = (e == 0 ? a.hL : a.hR) + (size_t)s * T * D;
        hrir_spectrum(h, ar, hp, T, D, K, tw, grpD[(size_t)s * 2 + e], Hd);
        EM_CUDA(launch_abs_transpose(st, Hd, D, K, absH + ((size_t)s * 2 + e) * K * D));
        h->launches += 1;
        if (nLS > 0) {
          GemmOperand A2{Hd + 2, 2LL * K, 0}, B2{Q, D, 1}, B3{Yh, D, 1};
          const size_t off = ((size_t)s * 2 + e) * nLS * 2 * S;
          EM_CUDA(launch_gemm(st, A2, B2, GemmShape{2 * nLS, S, D}, EpiStore{Tls + off, S, 1.0}));
          EM_CUDA(launch_gemm(st, A2, B3, GemmShape{2 * nLS, S, D}, EpiStore{Zls + off, S, 1.0}));
          h->launches += 2;
        }
        if (wdc && e == 1) {
          EM_CUDA(launch_target_cov(st, Hd0, Hd1, D, K, Rt + (size_t)s * K * 4));
          h->launches += 1;
        }
      }
  }
  // ---------------- int8 tensor-core route for the two direction-grid contractions (ozaki.cuh)
  int oz_T = (cfg.precision == EMAGLS_PRECISION_FP32) ? 4 : 6;   // balanced base-256 digits: 48 (32) bits
  if (const char* e = getenv("EMAGLS_OZAKI_SLICES")) oz_T = atoi(e);
  bool use_oz = true;
  if (const char* e = getenv("EMAGLS_GEMM")) use_oz = std::string(e) != "dmma";
  // six digits: the FP64 forward functor, the reference of the integer one (launch_oz_fwd)
  const char* oz_fwd = getenv("EMAGLS_OZ_FWD");
  const int oz_fwd_raw = oz_fwd && std::string(oz_fwd) == "raw";
  // Jacobi warm starts where min |r_ii| > warm_grading max |r_ii|.  1e-8 by measurement: the errors of bins 1-15
  // against exact arithmetic are the same 1e-14 with 1e-4, 1e-6 and 1e-9 (tests/test_gpu_arbitration.py,
  // profiles/r02_v51_*), the mean sweep count falls from 6.65 to 6.4 (bins 3-18 start warm: 9.2 -> 7.0-8.4 sweeps)
  const char* wg = getenv("EMAGLS_JACOBI_WARM_GRADING");
  const double warm_grading = wg ? atof(wg) : 1e-8;
  const int KpS = oz_pad32(S), KpD = oz_pad32(D);
  // longer contractions than the int32 accumulators hold exactly go through the DMMA GEMM instead
  if ((oz_T != 4 && oz_T != 6) || K - kls1 <= 0 || !oz_contraction_fits(KpD, oz_T) || !oz_contraction_fits(KpS, oz_T))
    use_oz = false;
  int8_t *YhA_q = nullptr, *YhB_q = nullptr, *QB_q = nullptr;
  double *sYhA = nullptr, *sYhB = nullptr, *sQB = nullptr, *upH = nullptr, *scH = nullptr;
  if (use_oz) {
    YhA_q = ar.get<int8_t>((size_t)oz_T * D * KpS); sYhA = ar.get<double>(D);
    YhB_q = ar.get<int8_t>((size_t)oz_T * S * KpD); sYhB = ar.get<double>(S);
    QB_q = ar.get<int8_t>((size_t)oz_T * S * KpD);  sQB = ar.get<double>(S);
    upH = ar.get<double>((size_t)a.num_sets * 2 * K); scH = ar.get<double>((size_t)a.num_sets * 2 * K);
    EM_CUDA(launch_slice_rows(st, Yh, 1, D, D, S, KpS, oz_T, YhA_q, sYhA));   // rows = directions
    EM_CUDA(launch_slice_rows(st, Yh, D, 1, S, D, KpD, oz_T, YhB_q, sYhB));   // rows = harmonics
    EM_CUDA(launch_slice_rows(st, Q, D, 1, S, D, KpD, oz_T, QB_q, sQB));
    EM_CUDA(launch_row_scale(st, absH, (long long)a.num_sets * 2 * K, D, upH, scH));
    h->launches += 4;
  }
  setup_span.reset();

  // ---------------- memory plan: orientation chunks of OC, Gram bin groups of NB, TSQR slots of G
  const int ne = Mc * (Mc + 1) / 2, ne_ld = (ne + 1) & ~1;
  // Mc <= 32: register-resident TSQR / Jacobi / reflector kernels of tsqr_kernels.cu ("sep" block plan);
  // Mc > 32 uses the shared-memory kernel of solver_kernels.cu.
  const bool sep = Mc <= 32;
  const BlockPlan bp = sep ? make_block_plan_sep(S, Mc) : make_block_plan(S, Mc);
  const int NB = std::min(128, K - 1);
  int g_slots = sep ? 16 : 4;  // bins factorised per launch; the Jacobi kernel warm-starts along them
  if (const char* e = getenv("EMAGLS_FACTOR_SLOTS")) g_slots = std::max(1, atoi(e));
  const int G = std::min(g_slots, K - 1);
  const long long v_stride = sep ? 32LL * S : (long long)Mc * S, tau_stride = (long long)bp.nblk * bp.MC,
                  pb_stride = (long long)Mc * Mc;
  const size_t per_orient =
      (size_t)Etot * 8 + (size_t)(nqs + nqa) * ne_ld * 8 + (size_t)2 * NB * ne_ld * 8 + (size_t)NB * pb_stride * 16 + (size_t)NB * 8 +
      (size_t)G * (v_stride + tau_stride + pb_stride + (sep ? 1024 : 0)) * 16 +
      (size_t)a.num_sets * ((size_t)(1 + 6) * 4 * S * 8 + (size_t)4 * D * 8);
  size_t free_b = 0, total_b = 0;
  EM_CUDA(cudaMemGetInfo(&free_b, &total_b));
  // memory still cached in the stream-ordered pool is reusable: plan against the larger figure
  {
    cudaMemPool_t pool = h->pool;
    unsigned long long reserved = 0, used = 0;
    if ((pool || cudaDeviceGetDefaultMemPool(&pool, h->device) == cudaSuccess) &&
        cudaMemPoolGetAttribute(pool, cudaMemPoolAttrReservedMemCurrent, &reserved) == cudaSuccess &&
        cudaMemPoolGetAttribute(pool, cudaMemPoolAttrUsedMemCurrent, &used) == cudaSuccess && reserved > used)
      free_b += (size_t)(reserved - used);
  }
  const size_t wsp_bytes = a.spectra ? 0 : (size_t)2 * P * Mc * K * sizeof(cplx);
  EM_REQUIRE(free_b > wsp_bytes + (size_t)(1u << 28), "not enough device memory for the solution array");
  long long oc_fit = (long long)((double)(free_b - wsp_bytes) * 0.7 / (double)per_orient);
  if (const char* e = getenv("EMAGLS_ORIENT_CHUNK")) oc_fit = std::max(1, atoi(e));
  EM_REQUIRE(oc_fit >= 1, "not enough device memory for one orientation");
  const int OC = (int)std::min<long long>({(long long)a.num_orient, oc_fit, 8192LL});
  const int PJ = a.num_sets * OC;

  cplx* Wsp = a.spectra ? reinterpret_cast<cplx*>(a.spectra) : ar.get<cplx>((size_t)2 * P * Mc * K);
  const long long w_ear = (long long)P * Mc * K;
  EM_CUDA(cudaMemsetAsync(Wsp, 0, (size_t)2 * P * Mc * K * sizeof(cplx), st));
  double* E = ar.get<double>((size_t)OC * Etot);
  double* Fs = ar.get<double>((size_t)nqs * OC * ne_ld);
  double* Fa = ar.get<double>((size_t)nqa * OC * ne_ld);
  double* Gre = ar.get<double>((size_t)NB * OC * ne_ld);
  double* Gim = ar.get<double>((size_t)NB * OC * ne_ld);
  cplx* PbG = ar.get<cplx>((size_t)NB * OC * pb_stride);
  double* sigG = ar.get<double>((size_t)NB * OC);   // shift of the condition certificate per matrix (gram_kernels.cu)
  int* d_fail = ar.get<int>(NB + 1);
  OperatorSet ops{};
  ops.v_stride = v_stride; ops.tau_stride = tau_stride; ops.pb_stride = pb_stride;
  ops.V = ar.get<cplx>((size_t)OC * G * v_stride);
  ops.tau = ar.get<cplx>((size_t)OC * G * tau_stride);
  ops.Pb = ar.get<cplx>((size_t)OC * G * pb_stride);
  ops.info = ar.get<int>((size_t)OC * G);
  ops.stats = h->d_stats;
  cplx* Rbuf = sep ? ar.get<cplx>((size_t)OC * G * 1024) : nullptr;   // R_C of every (orientation, slot)
  auto chain_bwd = [&](int slot, int slot_n, const double* rhs, long long set_stride, long long ear_stride, int shared,
                       int nsplit, long long split_stride, const ProbMap& pm, int kb, int pj) {
    return sep ? launch_chain_bwd_sep(st, bp, ops, slot, slot_n, rhs, set_stride, ear_stride, shared, nsplit, split_stride,
                                      pm, Wsp, w_ear, K, kb, dc_fix, pj, bn + (size_t)kb * (simN + 1), simN, d_roword)
               : launch_chain_bwd(st, bp, ops, slot, slot_n, rhs, set_stride, ear_stride, shared, nsplit, split_stride, pm,
                                  Wsp, w_ear, K, kb, dc_fix, pj);
  };
  double* Cv = ar.get<double>((size_t)4 * PJ * S);
  double* Tt = use_oz ? nullptr : ar.get<double>((size_t)D * 4 * PJ);
  int8_t* Cv_q = use_oz ? ar.get<int8_t>((size_t)oz_T * 4 * PJ * KpS) : nullptr;
  int8_t* Tt_q = use_oz ? ar.get<int8_t>((size_t)oz_T * 4 * PJ * KpD) : nullptr;
  double* sCv = use_oz ? ar.get<double>((size_t)4 * PJ) : nullptr;
  double* sTt = use_oz ? ar.get<double>((size_t)4 * PJ) : nullptr;
  constexpr int MAX_SPLITS = 6;
  double* tq = ar.get<double>((size_t)MAX_SPLITS * 4 * PJ * S);   // split-K partials of t * Y_h
  // Gram route admissible iff cond_2(G) <= 1/c^2 (no singular value below c*s_max); the certificate of
  // launch_gram_chol proves cond_2(G) < thr with its own rounding margin, and normal equations are never
  // used beyond cond(G) = 1e4 (relative error floor about 2e-12 there).
  double gram_thr = (cfg.svd_regul > 0.0) ? std::min(1e4, 1.0 / (cfg.svd_regul * cfg.svd_regul)) : 1e4;
  if (getenv("EMAGLS_NO_GRAM")) gram_thr = -1.0;
  const bool debug = getenv("EMAGLS_DEBUG_INFO") != nullptr;
  std::vector<int> fail_h(NB + 1);

  // G_k of the bins gb0 .. gb0 + nb - 1 for every orientation of the chunk (packed lower triangles in Gre / Gim)
  auto assemble_gram = [&](int gb0, int nb, int oc) {
    const int ncol = oc * ne_ld;
    GemmOperand A1{bre + (size_t)gb0 * nqs, nqs, 1}, B1{Fs, (long long)ncol, 0};
    EM_CUDA(launch_gemm(st, A1, B1, GemmShape{nb, ncol, nqs}, EpiStore{Gre, (long long)ncol, 1.0}));
    if (simN > 0) {
      GemmOperand A2{bim + (size_t)gb0 * nqa, nqa, 1}, B2{Fa, (long long)ncol, 0};
      EM_CUDA(launch_gemm(st, A2, B2, GemmShape{nb, ncol, simN * (simN + 1) / 2}, EpiStore{Gim, (long long)ncol, 1.0}));
    } else {
      EM_CUDA(cudaMemsetAsync(Gim, 0, (size_t)nb * ncol * sizeof(double), st));
    }
    h->launches += 2;
  };

  for (int o0 = 0; o0 < a.num_orient; o0 += OC) {
    const int oc = std::min(OC, a.num_orient - o0);
    const int pj = a.num_sets * oc;
    const ProbMap pm{oc, o0, a.num_orient};
    bool cv_ready = false;                                      // digits of u_kb already produced by a fused tail
    const double* Yc = Yo + (size_t)o0 * Mc * S;
    {
      ProfSpan ps(h, EM_PROF_SETUP);
      for (int b0 = 0; b0 < oc; b0 += 32768) {
        int nb = std::min(32768, oc - b0);
        EM_CUDA(launch_build_E(st, R, S, simN, Yc + (size_t)b0 * Mc * S, Mc, nb, d_rowoff, d_roword, Etot,
                               E + (size_t)b0 * Etot));
        h->launches += 1;
      }
    }
    if (gram_thr > 0.0 || wdc) {
      ProfSpan ps(h, EM_PROF_GRAM);
      // build_F addresses (q*P + o) with P = oc: one launch per <= 32768 orientations is not possible
      // with that layout, so the grid's y dimension limits a chunk to 65535 orientations (OC <= 8192).
      EM_CUDA(launch_build_F(st, Gh, S, simN, Yc, Mc, oc, ne_ld, Fs, Fa));
      h->launches += 1;
    }
    // the padding columns D..KpD-1 of the t digits must read as zero (their position depends on pj)
    if (use_oz) EM_CUDA(cudaMemsetAsync(Tt_q, 0, (size_t)oz_T * 4 * pj * KpD, st));
    RowSource src{};
    src.E = E; src.Etot = Etot; src.rowoff = d_rowoff; src.roword = d_roword; src.bn = bn; src.N = simN;

    for (int gb0 = 1; gb0 < K; gb0 += NB) {
      const int nb = std::min(NB, K - gb0);
      std::fill(fail_h.begin(), fail_h.end(), 1);
      if (gram_thr > 0.0) {
        ProfSpan ps(h, EM_PROF_GRAM);
        EM_CUDA(cudaMemsetAsync(d_fail, 0, (size_t)(NB + 1) * sizeof(int), st));
        assemble_gram(gb0, nb, oc);
        EM_CUDA(launch_gram_chol(st, Gre, Gim, Mc, oc, ne_ld, nb, gram_thr, PbG, sigG, d_fail));
        h->launches += 2;
        EM_CUDA(cudaMemcpyAsync(fail_h.data(), d_fail, (size_t)(nb + 1) * sizeof(int), cudaMemcpyDeviceToHost, st));
        EM_CUDA(cudaStreamSynchronize(st));
      }
      if (debug) {
        int ng = 0;
        for (int i = 0; i < nb; ++i) ng += (fail_h[1 + i] == 0);
        fprintf(stderr, "orient chunk %d: bins %d..%d: %d Gram bins, %d TSQR bins\n", o0, gb0, gb0 + nb - 1, ng, nb - ng);
      }
      int slot_base = -1, slot_n = 0;  // bins [slot_base, slot_base + slot_n) hold valid TSQR operators
      if (gb0 == 1) cv_ready = false;
      for (int kb = gb0; kb < gb0 + nb; ++kb) {
        const bool gram = fail_h[1 + kb - gb0] == 0;
        if (gram) h->stat_gram += oc;
        const cplx* bk = bn + (size_t)kb * (simN + 1);
        if (!gram && !(kb >= slot_base && kb < slot_base + slot_n)) {
          int Gn = 0;
          while (Gn < G && kb + Gn < gb0 + nb && fail_h[1 + kb + Gn - gb0] != 0) ++Gn;
          // bins refused by the Gram route skip the fast-path test (it cannot succeed there)
          const int try_fast = gram_thr > 0.0 ? 0 : 1;
          h->stat_tsqr += (long long)oc * Gn;   // factorisations are per orientation, shared by the HRTF sets
          if (sep) {
            {
              ProfSpan ps(h, EM_PROF_FACTOR);
              EM_CUDA(launch_tsqr_sep(st, bp, src, ops, Rbuf, oc, kb, Gn));
            }
            {
              ProfSpan ps(h, EM_PROF_JACOBI);
              EM_CUDA(launch_svdclip(st, Mc, Rbuf, ops, oc, Gn, cfg.svd_regul, try_fast, warm_grading));
            }
            h->launches += 2;
          } else {
            ProfSpan ps(h, EM_PROF_FACTOR);
            EM_CUDA(launch_factor(st, bp, src, ops, oc, kb, Gn, cfg.svd_regul, try_fast));
            h->launches += 1;
          }
          slot_base = kb; slot_n = Gn;
          if (debug) {
            std::vector<int> info((size_t)oc * Gn);
            EM_CUDA(cudaMemcpyAsync(info.data(), ops.info, info.size() * sizeof(int), cudaMemcpyDeviceToHost, st));
            EM_CUDA(cudaStreamSynchronize(st));
            for (int slot = 0; slot < Gn; ++slot) {
              int nfast = 0, smax = 0; long long ssum = 0;
              for (int p = 0; p < oc; ++p) { int v = info[(size_t)p * Gn + slot]; nfast += (v == 0); smax = std::max(smax, v); ssum += v; }
              fprintf(stderr, "bin %d: fast %d/%d, sweeps max %d mean %.2f\n", kb + slot, nfast, oc, smax, (double)ssum / oc);
            }
          }
        }
        const int slot = kb - slot_base;
        const cplx* pbg = PbG + (size_t)(kb - gb0) * oc * pb_stride;
        if (kb < kls1) {
          ProfSpan ps(h, EM_PROF_CHAIN_BWD);
          const size_t off = (size_t)(kb - 1) * 2 * S;
          if (gram)
            EM_CUDA(launch_bwd_small(st, Yc, Mc, S, d_roword, bk, pbg, pm, pj, Zls + off, (long long)2 * nLS * 2 * S,
                                     (long long)nLS * 2 * S, 1, 1, 0, Wsp, w_ear, K, kb, dc_fix, nullptr, nullptr, nullptr, 0, 0, simN));
          else
            EM_CUDA(chain_bwd(slot, slot_n, Tls + off, (long long)2 * nLS * 2 * S, (long long)nLS * 2 * S, 1, 1, 0, pm, kb, pj));
          h->launches += 1;
        } else {
          if (!cv_ready) {   // else: the digits of u_kb were written by the fused tail of the previous Gram bin
            ProfSpan ps(h, EM_PROF_CHAIN_FWD);
            EM_CUDA(launch_fwd_small(st, Yc, Mc, S, d_roword, bk, pm, pj, Wsp, w_ear, K, kb - 1, Cv));
            if (use_oz) EM_CUDA(launch_slice_rows(st, Cv, S, 1, 4 * pj, S, KpS, oz_T, Cv_q, sCv));
            h->launches += use_oz ? 2 : 1;
          }
          cv_ready = false;
          int nsplit = 1;
          const long long split_stride = 4LL * pj * S;
          if (use_oz) {
            {
              ProfSpan ps(h, EM_PROF_GEMM_FWD);   // exactly one launch: the int8 tensor-core GEMM
              OzFwdArgs fa{YhA_q, sYhA, D, KpS, Cv_q, sCv, 4 * pj, oz_T, Tt_q, KpD, sTt,
                           absH + (size_t)kb * D, 2LL * K * D, (long long)K * D, upH + kb, scH + kb, K, oc,
                           kb == K - 1 ? 1 : 0, oz_fwd_raw};
              EM_CUDA(launch_oz_fwd(st, fa));
            }
            {
              ProfSpan ps(h, EM_PROF_GEMM_BWD);
              EM_CUDA(launch_oz_bwd(st, Tt_q, sTt, 4 * pj, gram ? YhB_q : QB_q, gram ? sYhB : sQB, S, KpD, oz_T, tq));
            }
          } else {
            {
              ProfSpan ps(h, EM_PROF_GEMM_FWD);
              GemmOperand A3{Yh, D, 0}, B3{Cv, S, 1};
              EpiPhase ep{Tt, 4LL * pj, absH + (size_t)kb * D, 2LL * K * D, (long long)K * D, oc, kb == K - 1 ? 1 : 0};
              EM_CUDA(launch_gemm(st, A3, B3, GemmShape{D, 4 * pj, S}, ep));
            }
            {
              ProfSpan ps(h, EM_PROF_GEMM_BWD);
              GemmOperand A4{Tt, 4LL * pj, 0}, B4{gram ? Yh : Q, D, 1};
              EM_CUDA(launch_gemm_splitk(st, A4, B4, GemmShape{4 * pj, S, D}, EpiStore{tq, S, 1.0, split_stride}, MAX_SPLITS,
                                         &nsplit));
            }
          }
          {
            ProfSpan ps(h, EM_PROF_CHAIN_BWD);
            if (gram) {
              const bool fuse = use_oz && kb + 1 < K;
              EM_CUDA(launch_bwd_small(st, Yc, Mc, S, d_roword, bk, pbg, pm, pj, tq, 0, 0, 0, nsplit, split_stride, Wsp,
                                       w_ear, K, kb, dc_fix, fuse ? bn + (size_t)(kb + 1) * (simN + 1) : nullptr, Cv_q, sCv,
                                       KpS, oz_T, simN));
              cv_ready = fuse;
            } else
              EM_CUDA(chain_bwd(slot, slot_n, tq, 0, 0, 0, nsplit, split_stride, pm, kb, pj));
          }
          h->launches += 3;   // forward GEMM, backward GEMM, backward small / chain kernel
        }
      }
    }
    if (wdc) {
      // after the recursion (the phase continuation runs on the unconstrained solutions, as in the removed reference
      // code) and before the tail; the DC bin is set again from the constrained bin 1
      ProfSpan ps(h, EM_PROF_GRAM);
      for (int gb0 = 1; gb0 < K; gb0 += NB) {
        const int nb = std::min(NB, K - gb0);
        assemble_gram(gb0, nb, oc);
        EM_CUDA(launch_diffuseness_apply(st, Gre, Gim, Mc, oc, ne_ld, nb, gb0, D, Rt, pm, pj, Wsp, w_ear, K, dc_fix ? 1 : 0, 1));
        h->launches += 1;
      }
    }
  }

  // ---------------- tail: one GEMM per (set, ear)
  {
    ProfSpan ps(h, EM_PROF_TAIL);
    double* twT = ar.get<double>((size_t)a.len * 2 * K);
    double* wtmp = cplx_out ? ar.get<double>((size_t)a.num_orient * Mc * a.len) : nullptr;
    for (int s = 0; s < a.num_sets; ++s)
      for (int e = 0; e < 2; ++e) {
        double delay = (double)(nfft / 2) + (e == 1 ? (grpD[(size_t)s * 2 + 1] - grpD[(size_t)s * 2]) : 0.0);
        EM_CUDA(launch_tail_twiddle(st, K, nfft, a.len, delay, twT));
        const cplx* Wse_c = Wsp + ((size_t)e * P + (size_t)s * a.num_orient) * Mc * K;
        const double* Wse = reinterpret_cast<const double*>(Wse_c);
        GemmOperand A5{Wse, 2LL * K, 1}, B5{twT, 2LL * K, 1};
        const size_t out_off = (size_t)s * a.num_orient * Mc * a.len;
        double* out = cplx_out ? wtmp : (e == 0 ? a.wL : a.wR) + out_off;
        EpiStore es{out, a.len, 1.0};
        EM_CUDA(launch_gemm(st, A5, B5, GemmShape{a.num_orient * Mc, a.len, 2 * K}, es));
        h->launches += 2;
        if (cplx_out) {
          cplx* outc = reinterpret_cast<cplx*>(e == 0 ? a.wL : a.wR) + out_off;
          EM_CUDA(launch_basis_change_filters(st, wtmp, basis_kind, Mc, a.len, a.num_orient, Wse_c, K, nfft, outc));
          h->launches += 1;
        }
      }
    if (cplx_out && a.spectra) {
      EM_CUDA(launch_basis_change_spectra(st, Wsp, basis_kind, Mc, K, 2LL * P, 1));
      h->launches += 1;
    }
  }
}

}  // namespace emagls
