// One-time (per grid / per HRTF set / per orientation) kernels of the design path.
#include "kernels.h"
#include "special.cuh"

namespace emagls {

// ---------------------------------------------------------------------------------------------
// getSH on a list of directions (dependencies/Spherical-Harmonic-Transform/getSH.m:17-89)
// ---------------------------------------------------------------------------------------------
__global__ void sh_angles_kernel(int N, const double* __restrict__ azi, const double* __restrict__ zen,
                                 int D, int complex_basis, double* __restrict__ out) {
  int d = blockIdx.x * blockDim.x + threadIdx.x;
  if (d >= D) return;
  double cm[MAX_SH_ORDER + 1], sm[MAX_SH_ORDER + 1];
  const double a = azi[d];
  for (int m = 0; m <= N; ++m) sincos((double)m * a, &sm[m], &cm[m]);  // cos(m*azi) as in getSH.m:67-68
  const double x = cos(zen[d]);
  if (complex_basis) complex_sh_dir(N, x, cm, sm, reinterpret_cast<cplx*>(out) + d, D);
  else real_sh_dir(N, x, cm, sm, out + d, D);
}

cudaError_t launch_sh_angles(cudaStream_t st, int N, const double* azi, const double* zen, int D,
                             int complex_basis, double* out) {
  sh_angles_kernel<<<(D + 63) / 64, 64, 0, st>>>(N, azi, zen, D, complex_basis, out);
  return cudaGetLastError();
}

// Real SH at the microphone positions seen from a rotated head: direction R_o^T u_m.
__global__ void sh_mics_kernel(int N, const double* __restrict__ mic_azi, const double* __restrict__ mic_zen,
                               int M, const double* __restrict__ rot, int B, double* __restrict__ out) {
  int idx = blockIdx.x * blockDim.x + threadIdx.x;
  if (idx >= B * M) return;
  int o = idx / M, m = idx % M;
  const int S = (N + 1) * (N + 1);
  double cm[MAX_SH_ORDER + 1], sm[MAX_SH_ORDER + 1];
  double a = mic_azi[m], x;
  if (rot == nullptr) {
    x = cos(mic_zen[m]);
  } else {
    double sz, cz, sa, ca;
    sincos(mic_zen[m], &sz, &cz);
    sincos(a, &sa, &ca);
    const double u[3] = {sz * ca, sz * sa, cz};
    const double* R = rot + (long long)o * 9;
    // v = R^T u
    double v0 = R[0] * u[0] + R[3] * u[1] + R[6] * u[2];
    double v1 = R[1] * u[0] + R[4] * u[1] + R[7] * u[2];
    double v2 = R[2] * u[0] + R[5] * u[1] + R[8] * u[2];
    double nrm = sqrt(v0 * v0 + v1 * v1 + v2 * v2);
    x = v2 / nrm;
    a = atan2(v1, v0);
  }
  for (int q = 0; q <= N; ++q) sincos((double)q * a, &sm[q], &cm[q]);
  real_sh_dir(N, x, cm, sm, out + (long long)idx * S, 1);
}

cudaError_t launch_sh_mics(cudaStream_t st, int N, const double* mic_azi, const double* mic_zen,
                           int M, const double* rot, int B, double* out) {
  int total = B * M;
  sh_mics_kernel<<<(total + 63) / 64, 64, 0, st>>>(N, mic_azi, mic_zen, M, rot, B, out);
  return cudaGetLastError();
}

__global__ void left_mul_kernel(const double* __restrict__ L, int Mc, int M, const double* __restrict__ Y,
                                int B, int S, double* __restrict__ out) {
  long long idx = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  long long total = (long long)B * Mc * S;
  if (idx >= total) return;
  int s = (int)(idx % S);
  int c = (int)((idx / S) % Mc);
  int o = (int)(idx / ((long long)S * Mc));
  const double* y = Y + (long long)o * M * S + s;
  double acc = 0.0;
  for (int m = 0; m < M; ++m) acc = fma(L[c * M + m], y[(long long)m * S], acc);
  out[idx] = acc;
}

cudaError_t launch_left_mul(cudaStream_t st, const double* L, int Mc, int M, const double* Y,
                            int B, int S, double* out) {
  long long total = (long long)B * Mc * S;
  left_mul_kernel<<<(unsigned)((total + 255) / 256), 256, 0, st>>>(L, Mc, M, Y, B, S, out);
  return cudaGetLastError();
}

// ---------------------------------------------------------------------------------------------
// modal coefficients (sphModalCoeffs.m:25-59), bnAll = -sphModalCoeffs(...) (getSMAIRMatrix.m:107)
// ---------------------------------------------------------------------------------------------
__global__ void modal_kernel(int N, const double* __restrict__ kr, int nk, int array_type, double sign,
                             int nyquist_real, cplx* __restrict__ out, long long stride_k,
                             long long stride_n) {
  int k = blockIdx.x * blockDim.x + threadIdx.x;
  if (k >= nk) return;
  cplx b[MAX_SH_ORDER + 2];
  modal_coeffs(N, kr[k], array_type, b);
  for (int n = 0; n <= N; ++n) {
    cplx v = mk(sign * b[n].x, sign * b[n].y);
    if (nyquist_real && k == nk - 1) v.y = 0.0;
    out[(long long)k * stride_k + (long long)n * stride_n] = v;
  }
}

cudaError_t launch_modal(cudaStream_t st, int N, const double* kr, int nk, int array_type,
                         double sign, int nyquist_real, cplx* out, long long stride_k,
                         long long stride_n) {
  modal_kernel<<<(nk + 63) / 64, 64, 0, st>>>(N, kr, nk, array_type, sign, nyquist_real, out, stride_k, stride_n);
  return cudaGetLastError();
}

// ---------------------------------------------------------------------------------------------
// Householder QR of the real D x S matrix of HRIR-grid harmonics (one-time per grid)
// ---------------------------------------------------------------------------------------------
constexpr int HQ_THREADS = 256, HQ_COLS = 8;

__device__ __forceinline__ double warp_sum_d(double v) {
#pragma unroll
  for (int m = 16; m > 0; m >>= 1) v += __shfl_xor_sync(0xffffffffu, v, m);
  return v;
}

// step j of the factorisation: every CTA rebuilds reflector j from column j (read-only in this
// launch), CTA 0 records it, and each warp updates one trailing column.
__global__ void hh_factor_step(double* __restrict__ A, int D, int S, int j, double* __restrict__ Vst,
                               double* __restrict__ tau, double* __restrict__ rdiag) {
  extern __shared__ double vsh[];  // D doubles + 8
  double* red = vsh + D;
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const double* colj = A + (long long)j * D;
  double xn = 0.0;
  for (int i = j + 1 + tid; i < D; i += HQ_THREADS) { double v = colj[i]; vsh[i] = v; xn = fma(v, v, xn); }
  xn = warp_sum_d(xn);
  if (lane == 0) red[warp] = xn;
  __syncthreads();
  xn = 0.0;
  for (int w = 0; w < HQ_THREADS / 32; ++w) xn += red[w];
  const double alpha = colj[j];
  double beta, t, scale;
  if (xn == 0.0) { beta = alpha; t = 0.0; scale = 0.0; }
  else {
    beta = -copysign(sqrt(alpha * alpha + xn), alpha);
    t = (beta - alpha) / beta;
    scale = 1.0 / (alpha - beta);
  }
  for (int i = j + 1 + tid; i < D; i += HQ_THREADS) vsh[i] *= scale;
  if (tid == 0) vsh[j] = 1.0;
  __syncthreads();
  if (blockIdx.x == 0) {
    for (int i = tid; i < D; i += HQ_THREADS) Vst[(long long)j * D + i] = (i >= j) ? vsh[i] : 0.0;
    if (tid == 0) { tau[j] = t; rdiag[j] = beta; }
  }
  if (t == 0.0) return;
  const int c = j + 1 + blockIdx.x * HQ_COLS + warp;
  if (c >= S) return;
  double* a = A + (long long)c * D;
  double w = 0.0;
  for (int i = j + lane; i < D; i += 32) w = fma(vsh[i], a[i], w);
  w = warp_sum_d(w) * t;
  for (int i = j + lane; i < D; i += 32) a[i] = fma(-w, vsh[i], a[i]);
}

// backward accumulation of the thin Q: Q = H_0 ... H_{S-1} [I; 0], step j touches columns >= j
__global__ void hh_formq_step(double* __restrict__ Q, int D, int S, int j, const double* __restrict__ Vst,
                              const double* __restrict__ tau) {
  extern __shared__ double vsh[];
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const double t = tau[j];
  if (t == 0.0) return;
  for (int i = j + tid; i < D; i += HQ_THREADS) vsh[i] = Vst[(long long)j * D + i];
  __syncthreads();
  const int c = j + blockIdx.x * HQ_COLS + warp;
  if (c >= S) return;
  double* q = Q + (long long)c * D;
  double w = 0.0;
  for (int i = j + lane; i < D; i += 32) w = fma(vsh[i], q[i], w);
  w = warp_sum_d(w) * t;
  for (int i = j + lane; i < D; i += 32) q[i] = fma(-w, vsh[i], q[i]);
}

__global__ void hh_init_q(double* __restrict__ Q, int D, int S) {
  long long idx = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (idx >= (long long)D * S) return;
  int c = (int)(idx / D), i = (int)(idx % D);
  Q[idx] = (i == c) ? 1.0 : 0.0;
}

__global__ void hh_extract_r(const double* __restrict__ A, int D, int S, const double* __restrict__ rdiag,
                             double* __restrict__ R) {
  int idx = blockIdx.x * blockDim.x + threadIdx.x;
  if (idx >= S * S) return;
  int i = idx / S, jc = idx % S;
  double v = 0.0;
  if (i < jc) v = A[(long long)jc * D + i];
  else if (i == jc) v = rdiag[i];
  R[idx] = v;
}

cudaError_t launch_householder_qr(cudaStream_t st, double* A, int D, int S, double* Q, double* R,
                                  double* work, long long* launches) {
  double* Vst = work;
  double* tau = work + (long long)D * S;
  double* rdiag = tau + S;
  size_t smem = (size_t)(D + 8) * sizeof(double);
  cudaError_t e = allow_dynamic_smem(hh_factor_step, smem);
  if (e == cudaSuccess) e = allow_dynamic_smem(hh_formq_step, smem);
  if (e != cudaSuccess) return e;
  long long n = 0;
  for (int j = 0; j < S; ++j) {
    int trailing = S - 1 - j;
    int grid = (trailing + HQ_COLS - 1) / HQ_COLS;
    if (grid < 1) grid = 1;
    hh_factor_step<<<grid, HQ_THREADS, smem, st>>>(A, D, S, j, Vst, tau, rdiag);
    ++n;
  }
  hh_extract_r<<<(S * S + 255) / 256, 256, 0, st>>>(A, D, S, rdiag, R);
  hh_init_q<<<(unsigned)(((long long)D * S + 255) / 256), 256, 0, st>>>(Q, D, S);
  n += 2;
  for (int j = S - 1; j >= 0; --j) {
    int cols = S - j;
    int grid = (cols + HQ_COLS - 1) / HQ_COLS;
    hh_formq_step<<<grid, HQ_THREADS, smem, st>>>(Q, D, S, j, Vst, tau);
    ++n;
  }
  if (launches) *launches += n;
  return cudaGetLastError();
}

// ---------------------------------------------------------------------------------------------
// CholeskyQR2 of the HRIR-grid basis matrix (nine launches instead of 2 S + 2 one-column Householder steps):
//   G = Y^T Y,  R1 = chol(G),  Q1 = Y R1^-1,   G2 = Q1^T Q1,  R2 = chol(G2),  Q = Q1 R2^-1,  R = R2 R1.
// One pass leaves ||Q^T Q - I|| ~ eps cond(Y)^2, the second restores eps for cond(Y) up to ~1e7 (the 2702-point
// grid at order 19 has cond 1.5).  A non-positive pivot or a diagonal ratio beyond 1e6 raises *flag and the
// caller falls back to the Householder route.
// ---------------------------------------------------------------------------------------------
// in place: upper triangle of the symmetric G [S][S] (row-major) -> R with G = R^T R; strictly lower part zeroed.
// Single CTA (S <= 1024 threads' worth of columns), left-looking by panels of 16 rows: thread i owns column i and
// accumulates the 16 panel rows at once (one coalesced global load of R[k][i] feeds 16 FMAs against the panel's
// columns of row k, staged in shared memory), then the panel is factorised row by row in shared memory.
constexpr int CH_PB = 16;
__global__ void __launch_bounds__(1024)
chol_upper_kernel(double* __restrict__ G, int S, int* __restrict__ flag) {
  extern __shared__ double ch_sm[];
  double* rk = ch_sm;                       // [2][CH_PB]: R[k][j0 .. j0+15] of the row being applied (double buffered)
  double* pan = ch_sm + 2 * CH_PB;          // [CH_PB][S]: the panel rows
  __shared__ double dmin_s, dmax_s, piv_s;
  const int tid = threadIdx.x, nt = blockDim.x;
  if (tid == 0) { dmin_s = 1e300; dmax_s = 0.0; }
  for (int j0 = 0; j0 < S; j0 += CH_PB) {
    const int pb = min(CH_PB, S - j0);
    const int i = j0 + tid;                 // this thread's column (columns < j0 are finished)
    // ---- A_panel = G[j0 + r][i] - sum_{k < j0} R[k][j0 + r] R[k][i]
    double acc[CH_PB];
#pragma unroll
    for (int r = 0; r < CH_PB; ++r) acc[r] = (i < S && r < pb && i >= j0 + r) ? G[(long long)(j0 + r) * S + i] : 0.0;
    for (int k = 0; k < j0; ++k) {
      double* rkb = rk + (k & 1) * CH_PB;
      if (tid < pb) rkb[tid] = G[(long long)k * S + j0 + tid];
      __syncthreads();
      if (i < S) {
        const double v = G[(long long)k * S + i];
#pragma unroll
        for (int r = 0; r < CH_PB; ++r) acc[r] = fma(-rkb[r], v, acc[r]);
      }
    }
    __syncthreads();
    if (i < S) {
#pragma unroll
      for (int r = 0; r < CH_PB; ++r) pan[(size_t)r * S + i] = acc[r];
    }
    __syncthreads();
    // ---- factorise the panel in shared memory: row r from the panel rows q < r
    for (int r = 0; r < pb; ++r) {
      const int j = j0 + r;
      double t = 0.0;
      if (i < S && i >= j) {
        t = pan[(size_t)r * S + i];
        for (int q = 0; q < r; ++q) t = fma(-pan[(size_t)q * S + j], pan[(size_t)q * S + i], t);
      }
      if (i == j) {                         // the pivot
        double d = t;
        if (!(d > 0.0)) { atomicExch(flag, 1); d = 1.0; }
        d = sqrt(d);
        piv_s = d;
        dmin_s = fmin(dmin_s, d); dmax_s = fmax(dmax_s, d);
      }
      __syncthreads();
      const double rjj = piv_s;
      if (i < S && i >= j) pan[(size_t)r * S + i] = (i == j) ? rjj : t / rjj;
      __syncthreads();
    }
    // ---- write the finished rows back (zeros left of the diagonal)
    for (int idx = tid; idx < pb * S; idx += nt) {
      const int r = idx / S, c = idx - r * S;
      G[(long long)(j0 + r) * S + c] = (c >= j0 + r) ? pan[(size_t)r * S + c] : 0.0;
    }
    __syncthreads();
  }
  if (tid == 0 && !(dmin_s > 1e-6 * dmax_s)) atomicExch(flag, 1);
}

// Rinv [S][S] row-major upper: column m by back substitution, one warp per column; the column under
// construction stays in shared memory, the lanes split the inner products.
constexpr int TI_WARPS = 4;
__global__ void __launch_bounds__(TI_WARPS * 32)
tri_inverse_kernel(const double* __restrict__ R, int S, double* __restrict__ Rinv) {
  extern __shared__ double ti_x[];          // [TI_WARPS][S]
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const int m = blockIdx.x * TI_WARPS + warp;
  if (m >= S) return;
  double* x = ti_x + (size_t)warp * S;
  for (int i = m; i >= 0; --i) {
    const double* Ri = R + (long long)i * S;
    double a = 0.0;
    for (int j = i + 1 + lane; j <= m; j += 32) a = fma(Ri[j], x[j], a);
    a = warp_sum_d(a);
    const double v = (((i == m) ? 1.0 : 0.0) - a) / Ri[i];
    if (lane == 0) x[i] = v;
    __syncwarp();
  }
  for (int i = lane; i < S; i += 32) Rinv[(long long)i * S + m] = (i <= m) ? x[i] : 0.0;
}

// R = R2 * R1 (both upper, row-major)
__global__ void tri_mul_kernel(const double* __restrict__ R2, const double* __restrict__ R1, int S, double* __restrict__ R) {
  const int idx = blockIdx.x * blockDim.x + threadIdx.x;
  if (idx >= S * S) return;
  const int i = idx / S, j = idx % S;
  double a = 0.0;
  for (int k = i; k <= j; ++k) a = fma(R2[(long long)i * S + k], R1[(long long)k * S + j], a);
  R[idx] = a;
}

cudaError_t launch_chol_upper(cudaStream_t st, double* G, int S, int* flag) {
  if (S > 1024) return cudaErrorInvalidValue;
  const size_t smem = (size_t)(2 * CH_PB + (size_t)CH_PB * S) * sizeof(double);
  if (smem > 200 * 1024) return cudaErrorInvalidValue;
  const cudaError_t e = allow_dynamic_smem(chol_upper_kernel, smem);
  if (e != cudaSuccess) return e;
  chol_upper_kernel<<<1, 1024, smem, st>>>(G, S, flag);
  return cudaGetLastError();
}
cudaError_t launch_tri_inverse(cudaStream_t st, const double* R, int S, double* Rinv) {
  const size_t smem = (size_t)TI_WARPS * S * sizeof(double);
  const cudaError_t e = allow_dynamic_smem(tri_inverse_kernel, smem);
  if (e != cudaSuccess) return e;
  tri_inverse_kernel<<<(S + TI_WARPS - 1) / TI_WARPS, TI_WARPS * 32, smem, st>>>(R, S, Rinv);
  return cudaGetLastError();
}
cudaError_t launch_tri_mul(cudaStream_t st, const double* R2, const double* R1, int S, double* R) {
  tri_mul_kernel<<<(S * S + 255) / 256, 256, 0, st>>>(R2, R1, S, R);
  return cudaGetLastError();
}

// ---------------------------------------------------------------------------------------------
// E rows:  E[o][rowoff[i] + (n-ord(i))*Mc + c] = sum_{j in block n, j >= i} R[i][j] Ym[o][c][j]
// ---------------------------------------------------------------------------------------------
// One CTA per (order block n, orientation o): the block's columns of Ym[o] are staged in shared memory
// ([Mc][2n+1], odd pitch: conflict free), one warp per row i < (n+1)^2 with the lanes over the channels c,
// so the R entries are warp-uniform loads and the stores are contiguous.
__global__ void __launch_bounds__(256)
build_E_kernel(const double* __restrict__ R, int S, int N, const double* __restrict__ Ym,
               int Mc, int B, const int* __restrict__ rowoff, const int* __restrict__ roword,
               long long Etot, double* __restrict__ E) {
  extern __shared__ double be_y[];
  const int n = blockIdx.x, o = blockIdx.y, w = 2 * n + 1, s0 = n * n;
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5, nw = blockDim.x >> 5;
  const double* Yo = Ym + (long long)o * Mc * S;
  for (int idx = tid; idx < Mc * w; idx += blockDim.x) be_y[idx] = Yo[(long long)(idx / w) * S + s0 + idx % w];
  __syncthreads();
  const int nrows = min(S, (n + 1) * (n + 1));
  double* Eo = E + (long long)o * Etot;
  for (int i = warp; i < nrows; i += nw) {
    const int ord = roword[i];
    const int j0 = max(s0, i), j1 = s0 + w;   // R is upper triangular
    const double* Ri = R + (long long)i * S;
    double* e = Eo + rowoff[i] + (long long)(n - ord) * Mc;
    for (int c = lane; c < Mc; c += 32) {
      const double* y = be_y + c * w - s0;
      double acc = 0.0;
      for (int j = j0; j < j1; ++j) acc = fma(Ri[j], y[j], acc);
      e[c] = acc;
    }
  }
}

cudaError_t launch_build_E(cudaStream_t st, const double* R, int S, int N, const double* Ym,
                           int Mc, int B, const int* rowoff, const int* roword, long long Etot,
                           double* E) {
  dim3 grid(N + 1, B);
  const size_t smem = (size_t)Mc * (2 * N + 1) * sizeof(double);
  if (smem > 48 * 1024) return cudaErrorInvalidValue;
  build_E_kernel<<<grid, 256, smem, st>>>(R, S, N, Ym, Mc, B, rowoff, roword, Etot, E);
  return cudaGetLastError();
}

// ---------------------------------------------------------------------------------------------
// HRIR preparation (lib/getEMagLs2Filters.m:72-81)
// ---------------------------------------------------------------------------------------------
// sum(h, 2): h is [T x D] column-major.  Two deterministic passes.
__global__ void colsum_partial(const double* __restrict__ h, int T, int D, int nchunk, double* __restrict__ partial) {
  int t = blockIdx.x * blockDim.x + threadIdx.x;
  int ch = blockIdx.y;
  if (t >= T) return;
  int per = (D + nchunk - 1) / nchunk;
  int d0 = ch * per, d1 = min(D, d0 + per);
  double acc = 0.0;
  for (int d = d0; d < d1; ++d) acc += h[(long long)d * T + t];
  partial[(long long)ch * T + t] = acc;
}
__global__ void colsum_final(const double* __restrict__ partial, int T, int nchunk, double* __restrict__ out) {
  int t = blockIdx.x * blockDim.x + threadIdx.x;
  if (t >= T) return;
  double acc = 0.0;
  for (int c = 0; c < nchunk; ++c) acc += partial[(long long)c * T + t];
  out[t] = acc;
}
cudaError_t launch_colsum(cudaStream_t st, const double* h, int T, int D, double* partial,
                          int nchunk, double* out) {
  dim3 grid((T + 127) / 128, nchunk);
  colsum_partial<<<grid, 128, 0, st>>>(h, T, D, nchunk, partial);
  colsum_final<<<(T + 127) / 128, 128, 0, st>>>(partial, T, nchunk, out);
  return cudaGetLastError();
}

// grpdelay(b, 1, f, fs) at the K bin frequencies: Re(sum n b_n z^-n / sum b_n z^-n), |den| < 10 eps -> 0
__global__ void grpdelay_kernel(const double* __restrict__ s, int T, int K, double fs, double* __restrict__ gd) {
  int k = blockIdx.x * blockDim.x + threadIdx.x;
  if (k >= K) return;
  const double f = (double)k * ((fs / 2.0) / (double)(K - 1));
  const double w = 2.0 * 3.141592653589793 * f / fs;
  double nr = 0.0, ni = 0.0, dr = 0.0, di = 0.0;
  for (int n = 0; n < T; ++n) {
    double sn, cs;
    sincos(w * (double)n, &sn, &cs);
    double b = s[n];
    dr = fma(b, cs, dr); di = fma(-b, sn, di);
    double bn = b * (double)n;
    nr = fma(bn, cs, nr); ni = fma(-bn, sn, ni);
  }
  double ad = sqrt(dr * dr + di * di);
  double out = 0.0;
  if (!(ad < 10.0 * 2.220446049250313e-16)) {
    out = (nr * dr + ni * di) / (dr * dr + di * di);  // Re(num/den)
  }
  gd[k] = out;
}
cudaError_t launch_grpdelay(cudaStream_t st, const double* s, int T, int K, double fs, double* gd) {
  grpdelay_kernel<<<(K + 63) / 64, 64, 0, st>>>(s, T, K, fs, gd);
  return cudaGetLastError();
}

__global__ void dft_twiddle_kernel(int K, int T, int nfft, double* __restrict__ tw) {
  long long idx = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (idx >= (long long)K * T) return;
  int k = (int)(idx / T), t = (int)(idx % T);
  long long r = ((long long)k * t) % nfft;
  double sn, cs;
  sincospi(-2.0 * (double)r / (double)nfft, &sn, &cs);
  tw[(long long)(2 * k) * T + t] = cs;
  tw[(long long)(2 * k + 1) * T + t] = sn;
}
cudaError_t launch_dft_twiddle(cudaStream_t st, int K, int T, int nfft, double* tw) {
  long long total = (long long)K * T;
  dft_twiddle_kernel<<<(unsigned)((total + 255) / 256), 256, 0, st>>>(K, T, nfft, tw);
  return cudaGetLastError();
}

__global__ void abs_transpose_kernel(const double* __restrict__ Hd, int D, int K, double* __restrict__ absH) {
  __shared__ double tile[32][33];
  int k0 = blockIdx.x * 32, d0 = blockIdx.y * 32;
  int tx = threadIdx.x, ty = threadIdx.y;  // 32 x 8
  for (int r = ty; r < 32; r += 8) {
    int d = d0 + r, k = k0 + tx;
    double v = 0.0;
    if (d < D && k < K) {
      const double* p = Hd + (long long)d * (2 * K) + 2 * k;
      v = sqrt(fma(p[0], p[0], p[1] * p[1]));
    }
    tile[r][tx] = v;
  }
  __syncthreads();
  for (int r = ty; r < 32; r += 8) {
    int k = k0 + r, d = d0 + tx;
    if (k < K && d < D) absH[(long long)k * D + d] = tile[tx][r];
  }
}
cudaError_t launch_abs_transpose(cudaStream_t st, const double* Hd, int D, int K, double* absH) {
  dim3 grid((K + 31) / 32, (D + 31) / 32), block(32, 8);
  abs_transpose_kernel<<<grid, block, 0, st>>>(Hd, D, K, absH);
  return cudaGetLastError();
}

// Tail (lib/getEMagLs2Filters.m:113-135) as one real matrix per ear:
//   w[t'] = fade[t'] / nfft * sum_k c_k Re( W_k * ramp_k * exp(+2 pi i k (t'+lo)/nfft) )
// ramp_k = exp(-2 pi i (k/nfft) delay), real part at Nyquist (applySubsampleDelay.m:10-13),
// c_k = 1 for DC/Nyquist, 2 otherwise; fade = getFadeWindow(len) (getFadeWindow.m:9-16).
__global__ void tail_twiddle_kernel(int K, int nfft, int len, double delay, double* __restrict__ tw) {
  long long idx = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (idx >= (long long)len * K) return;
  int tp = (int)(idx / K), k = (int)(idx % K);
  const int lo = nfft / 2 - len / 2;
  const double win = fade_window(tp, len);
  const double g = win / (double)nfft;
  // ramp
  const double omega = (double)k * (0.5 / (double)(K - 1));
  double rs, rc;
  sincos(-2.0 * 3.141592653589793 * omega * delay, &rs, &rc);
  if (k == K - 1) rs = 0.0;
  // exp(+2 pi i k (t'+lo) / nfft)
  long long r = ((long long)k * (tp + lo)) % nfft;
  double es, ec;
  sincospi(2.0 * (double)r / (double)nfft, &es, &ec);
  double pr = rc * ec - rs * es, pi_ = rc * es + rs * ec;
  double ck = (k == 0 || k == K - 1) ? 1.0 : 2.0;
  double* row = tw + (long long)tp * (2 * K);
  row[2 * k] = g * ck * pr;
  row[2 * k + 1] = (k == 0 || k == K - 1) ? 0.0 : -g * ck * pi_;
}
cudaError_t launch_tail_twiddle(cudaStream_t st, int K, int nfft, int len, double delay, double* tw) {
  long long total = (long long)len * K;
  tail_twiddle_kernel<<<(unsigned)((total + 255) / 256), 256, 0, st>>>(K, nfft, len, delay, tw);
  return cudaGetLastError();
}

}  // namespace emagls
