// Steering rows of getEMagLsFiltersEMAinSH (lib/getEMagLsFiltersEMAinSH.m:60-103), per HRIR direction d:
//   emaIrDir(k, :, d)    = smairMat(:,:,k) * Y_hor_conj(:, d)          equatorial plane-wave response (:68-69)
//   emaIrDir_sh(k, :, d) = emaIrDir(k, :, d) * pinv(YCh.') * J.'       CH decomposition + SH expansion (:81-83)
//   emaIrDir_sh(k, :, d) = emaIrDir_sh(k, :, d) * getSHrotMtx(euler2rotationMatrix(-azi, zen - pi/2, azi, 'zyz'))
// Because smairMat(:,:,k) = Ym diag(b_n(k)) the k-dependence factors out:
//   pwGrid_k(h, d) = sum_n b_n(k) Cn[d][n][h],   Cn[d][n][:] = (sum_{s in n} Ym[:, s] Yhor[s, d])^T dec Rot_d.
// One CTA per direction builds Rot_d (Ivanic-Ruedenberg band recursion,
// dependencies/Spherical-Harmonic-Transform/getSHrotMtx.m:59-121), Cn in shared memory and writes
// the rows At[k-1][d][h] of every bin.
#include "kernels.h"
#include "shrot.cuh"

namespace emagls {

namespace {

// element (row m, column m') of complex2realSHMtx (complex2realSHMtx.m:25-47) within one band
__device__ __forceinline__ cplx c2r_W(int mr, int mc) {
  const double r = 0.7071067811865476;
  if (mr == 0) return mk(mc == 0 ? 1.0 : 0.0, 0.0);
  if (mc != mr && mc != -mr) return mk(0.0, 0.0);
  const int am = mr < 0 ? -mr : mr;
  const double sg = (am & 1) ? -1.0 : 1.0;
  if (mr < 0) return (mc == mr) ? mk(0.0, r) : mk(0.0, -r * sg);
  return (mc == mr) ? mk(r * sg, 0.0) : mk(r, 0.0);
}

}  // namespace

// dec [M][nsh] complex (row-major), Ym [M][S], Yhor [S][D], bn [K][simN+1], At [(K-1)][D][nsh]
__global__ void __launch_bounds__(256)
ema_sh_rows_kernel(int order, int simN, int M, int D, int K, int complex_basis,
                   const double* __restrict__ azi, const double* __restrict__ zen,
                   const cplx* __restrict__ dec, const double* __restrict__ Ym,
                   const double* __restrict__ Yhor, const cplx* __restrict__ bn, cplx* __restrict__ At) {
  extern __shared__ __align__(16) unsigned char es_raw[];
  const int nsh = (order + 1) * (order + 1), S = (simN + 1) * (simN + 1), L1 = simN + 1;
  const int d = blockIdx.x, tid = threadIdx.x, nt = blockDim.x;
  double* Rr = reinterpret_cast<double*>(es_raw);            // [nsh][nsh] real rotation (block diagonal)
  cplx* Rc = reinterpret_cast<cplx*>(Rr + ((nsh * nsh + 1) & ~1));  // [nsh][nsh] rotation in the output basis
  cplx* Bd = Rc + nsh * nsh;                                 // [M][nsh]
  double* Pn = reinterpret_cast<double*>(Bd + M * nsh);      // [M][L1]
  cplx* Cn = reinterpret_cast<cplx*>(Pn + ((M * L1 + 1) & ~1));  // [L1][nsh]
  __shared__ Rot1 R1;
  __shared__ int rotate;

  const double az = azi[d], ze = zen[d];
  if (tid == 0) {
    rotate = (ze != 1.5707963267948966) ? 1 : 0;   // hrirGridZenRad(d) ~= pi/2  (:87)
    // euler2rotationMatrix(-azi, zen - pi/2, azi, 'zyz') = Rz(gamma) Ry(beta) Rz(alpha) with
    // Rz(t) = [c s 0; -s c 0; 0 0 1], Ry(t) = [c 0 -s; 0 1 0; s 0 c]  (euler2rotationMatrix.m:19-50)
    double sa, ca, sb, cb, sg, cg;
    sincos(-az, &sa, &ca); sincos(ze - 1.5707963267948966, &sb, &cb); sincos(az, &sg, &cg);
    const double A[3][3] = {{ca, sa, 0}, {-sa, ca, 0}, {0, 0, 1}};
    const double B[3][3] = {{cb, 0, -sb}, {0, 1, 0}, {sb, 0, cb}};
    const double G[3][3] = {{cg, sg, 0}, {-sg, cg, 0}, {0, 0, 1}};
    double BA[3][3], E[3][3];
    for (int i = 0; i < 3; ++i)
      for (int j = 0; j < 3; ++j) { double v = 0; for (int q = 0; q < 3; ++q) v += B[i][q] * A[q][j]; BA[i][j] = v; }
    for (int i = 0; i < 3; ++i)
      for (int j = 0; j < 3; ++j) { double v = 0; for (int q = 0; q < 3; ++q) v += G[i][q] * BA[q][j]; E[i][j] = v; }
    rot1_from_matrix(E, R1);
  }
  sh_rot_real_bands(R1, &rotate, order, Rr, tid, nt);
  // rotation in the output basis: real as is, complex = W.' R conj(W)  (getSHrotMtx.m:115-118)
  for (int e = tid; e < nsh * nsh; e += nt) {
    const int a = e / nsh, b = e % nsh;
    cplx val = mk(Rr[e], 0.0);
    if (complex_basis) {
      int na = (int)sqrt((double)a); while ((na + 1) * (na + 1) <= a) ++na; while (na * na > a) --na;
      int nb = (int)sqrt((double)b); while ((nb + 1) * (nb + 1) <= b) ++nb; while (nb * nb > b) --nb;
      val = mk(0.0, 0.0);
      if (na == nb) {
        const int ma = a - na * na - na, mb = b - nb * nb - nb, base = na * na + na;
        for (int si = 0; si < 2; ++si) {
          const int mi = si ? -ma : ma;
          if (si && ma == 0) break;
          const cplx wia = c2r_W(mi, ma);
          for (int sj = 0; sj < 2; ++sj) {
            const int mj = sj ? -mb : mb;
            if (sj && mb == 0) break;
            const cplx wjb = c2r_W(mj, mb);
            const double r = Rr[(base + mi) * nsh + base + mj];
            const cplx t = cmulc(wia, wjb);   // W[i][a] * conj(W[j][b])
            val.x = fma(t.x, r, val.x); val.y = fma(t.y, r, val.y);
          }
        }
      }
    }
    Rc[e] = val;
  }
  __syncthreads();
  // Bd[m][h] = sum_h' dec[m][h'] Rot[h'][h]
  for (int e = tid; e < M * nsh; e += nt) {
    const int m = e / nsh, hh = e % nsh;
    cplx acc = mk(0.0, 0.0);
    for (int q = 0; q < nsh; ++q) cfma(acc, dec[m * nsh + q], Rc[q * nsh + hh]);
    Bd[e] = acc;
  }
  // Pn[m][n] = sum_{s in order n} Ym[m][s] Yhor[s][d]
  for (int e = tid; e < M * L1; e += nt) {
    const int m = e / L1, n = e % L1;
    double acc = 0.0;
    for (int s = n * n; s < (n + 1) * (n + 1); ++s) acc = fma(Ym[(long long)m * S + s], Yhor[(long long)s * D + d], acc);
    Pn[e] = acc;
  }
  __syncthreads();
  for (int e = tid; e < L1 * nsh; e += nt) {
    const int n = e / nsh, hh = e % nsh;
    cplx acc = mk(0.0, 0.0);
    for (int m = 0; m < M; ++m) { const double p = Pn[m * L1 + n]; const cplx b = Bd[m * nsh + hh]; acc.x = fma(p, b.x, acc.x); acc.y = fma(p, b.y, acc.y); }
    Cn[e] = acc;
  }
  __syncthreads();
  for (int e = tid; e < (K - 1) * nsh; e += nt) {
    const int k = 1 + e / nsh, hh = e % nsh;
    const cplx* b = bn + (long long)k * L1;
    cplx acc = mk(0.0, 0.0);
    for (int n = 0; n < L1; ++n) cfma(acc, b[n], Cn[n * nsh + hh]);
    At[((long long)(k - 1) * D + d) * nsh + hh] = acc;
  }
}

cudaError_t launch_ema_sh_rows(cudaStream_t st, int order, int simN, int M, int D, int K, int complex_basis,
                               const double* azi, const double* zen, const cplx* dec, const double* Ym,
                               const double* Yhor, const cplx* bn, cplx* At) {
  const int nsh = (order + 1) * (order + 1), L1 = simN + 1;
  size_t smem = (size_t)((nsh * nsh + 1) & ~1) * 8 + (size_t)nsh * nsh * 16 + (size_t)M * nsh * 16 +
                (size_t)((M * L1 + 1) & ~1) * 8 + (size_t)L1 * nsh * 16;
  if (smem > 200 * 1024) return cudaErrorInvalidValue;
  const cudaError_t e = allow_dynamic_smem(ema_sh_rows_kernel, smem);
  if (e != cudaSuccess) return e;
  ema_sh_rows_kernel<<<D, 256, smem, st>>>(order, simN, M, D, K, complex_basis, azi, zen, dec, Ym, Yhor, bn, At);
  return cudaGetLastError();
}

// getCH(N, azi, basis) rows (dependencies/getCH.m:17-28): At[m][c], c ordered [0,-1,+1,-2,+2,..]
__global__ void ch_rows_any_kernel(int N, const double* __restrict__ azi, int M, int complex_basis,
                                   cplx* __restrict__ At) {
  int idx = blockIdx.x * blockDim.x + threadIdx.x;
  const int nch = 2 * N + 1;
  if (idx >= M * nch) return;
  const int m = idx / nch, c = idx % nch;
  cplx v = mk(1.0, 0.0);
  if (c > 0) {
    const int q = (c + 1) / 2;
    double sn, cs;
    sincos((double)q * azi[m], &sn, &cs);
    if (complex_basis) v = (c & 1) ? mk(cs, -sn) : mk(cs, sn);          // exp(-i q azi), exp(+i q azi)
    else v = mk(1.4142135623730951 * ((c & 1) ? sn : cs), 0.0);          // sqrt2 sin, sqrt2 cos
  }
  At[idx] = v;
}
cudaError_t launch_ch_rows(cudaStream_t st, int N, const double* azi, int M, int complex_basis, cplx* At) {
  const int n = M * (2 * N + 1);
  ch_rows_any_kernel<<<(n + 127) / 128, 128, 0, st>>>(N, azi, M, complex_basis, At);
  return cudaGetLastError();
}

// dec[m][acn] = pinvT[m][ch(mm)] * Nnm[acn]   (lib/getEMagLsFiltersEMAinSH.m:79-83 with
// getChToShExpansionMatrix.m:11-18 and getNnm.m:13-30 at zenith pi/2).  Ysh0: real SH of order N at
// (azi 0, zen pi/2), pinvT: [(m&1)*npair + m/2][nch] as produced by regularized_apply_dev.
__global__ void ema_dec_kernel(int N, int M, int npair, int complex_basis, const double* __restrict__ Ysh0,
                               const cplx* __restrict__ pinvT, cplx* __restrict__ dec) {
  int idx = blockIdx.x * blockDim.x + threadIdx.x;
  const int nsh = (N + 1) * (N + 1), nch = 2 * N + 1;
  if (idx >= M * nsh) return;
  const int m = idx / nsh, acn = idx % nsh;
  int n = (int)sqrt((double)acn); while ((n + 1) * (n + 1) <= acn) ++n; while (n * n > acn) --n;
  const int mm = acn - n * n - n, am = mm < 0 ? -mm : mm;
  // N_n|m| P_n^|m|(cos(pi/2)) without Condon-Shortley phase = Y_real(n, +|m|)(azi = 0) / (sqrt2 or 1)
  double nlm = Ysh0[n * n + n + am];
  if (am > 0) nlm *= 0.7071067811865476;
  double nnm = nlm;                                   // 'real' (getNnm.m:26-28): (-1)^m cancels the CS phase
  if (complex_basis && mm > 0 && (mm & 1)) nnm = -nlm;  // 'complex', m >= 0 keeps the CS phase (getNnm.m:17-24)
  const int ch = 2 * am - (mm < 0 ? 1 : 0);
  const cplx p = pinvT[((long long)(m & 1) * npair + m / 2) * nch + ch];
  dec[idx] = mk(p.x * nnm, p.y * nnm);
}
cudaError_t launch_ema_dec(cudaStream_t st, int N, int M, int npair, int complex_basis, const double* Ysh0,
                           const cplx* pinvT, cplx* dec) {
  const int n = M * (N + 1) * (N + 1);
  ema_dec_kernel<<<(n + 127) / 128, 128, 0, st>>>(N, M, npair, complex_basis, Ysh0, pinvT, dec);
  return cudaGetLastError();
}

// complex-basis tail (getShFreqDomainConjugate.m:12-27 / getChFreqDomainConjugate.m:11-23 + ifft):
// with U = W(k, j) and V = sgn * conj(W(k, j')) (j' the -m partner; V = U at DC and Nyquist) the
// time-domain filter is Re-tail(X1) + i Re-tail(X2), X1 = ((Ur+Vr) + i(Ui-Vi))/2, X2 = ((Ui+Vi) - i(Ur-Vr))/2.
__global__ void complex_tail_prep_kernel(const cplx* __restrict__ W, int kind, int nch, int K, long long P,
                                         cplx* __restrict__ X1, cplx* __restrict__ X2) {
  long long idx = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (idx >= P * nch * K) return;
  const int k = (int)(idx % K);
  const int j = (int)((idx / K) % nch);
  const long long p = idx / ((long long)K * nch);
  int m, jp;
  if (kind == 0) {
    int n = (int)sqrt((double)j); while ((n + 1) * (n + 1) <= j) ++n; while (n * n > j) --n;
    m = j - n * n - n;
    jp = n * n + n - m;
  } else {
    const int am = (j + 1) / 2;
    m = (j == 0) ? 0 : ((j & 1) ? -am : am);
    jp = (j == 0) ? 0 : ((j & 1) ? j + 1 : j - 1);
  }
  const cplx U = W[idx];
  cplx V = U;
  if (k != 0 && k != K - 1) {
    const cplx q = W[(p * nch + jp) * K + k];
    const double sg = (kind == 0 && (m & 1)) ? -1.0 : 1.0;
    V = mk(sg * q.x, -sg * q.y);
  }
  X1[idx] = mk(0.5 * (U.x + V.x), 0.5 * (U.y - V.y));
  X2[idx] = mk(0.5 * (U.y + V.y), -0.5 * (U.x - V.x));
}
cudaError_t launch_complex_tail_prep(cudaStream_t st, const cplx* W, int kind, int nch, int K, long long P,
                                     cplx* X1, cplx* X2) {
  long long n = P * nch * K;
  complex_tail_prep_kernel<<<(unsigned)((n + 255) / 256), 256, 0, st>>>(W, kind, nch, K, P, X1, X2);
  return cudaGetLastError();
}

__global__ void interleave_kernel(const double* __restrict__ re, const double* __restrict__ im, long long n,
                                  cplx* __restrict__ out) {
  long long idx = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (idx < n) out[idx] = mk(re[idx], im[idx]);
}
cudaError_t launch_interleave(cudaStream_t st, const double* re, const double* im, long long n, cplx* out) {
  interleave_kernel<<<(unsigned)((n + 255) / 256), 256, 0, st>>>(re, im, n, out);
  return cudaGetLastError();
}

}  // namespace emagls
