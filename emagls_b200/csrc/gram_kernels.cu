// Gram route of the eMagLS hot loop for the bins where no singular value can be clipped.
//
// Reference step (lib/getEMagLs2Filters.m:86-89): Y_reg_inv = conj(U) diag(1/max(s, c s_max)) V.'.
// With A = pwGrid.' = Y_h diag(b_k) Ym^T and G = A^H A, the clip is inactive iff
// cond_2(G) <= 1/c^2; then Y_reg_inv = pinv(A).' = conj(A) G^-T exactly, i.e.
//     W_k = ((t Y_h) .* conj(b_k)) Ym^T G^-T.
// G is assembled on the FP64 tensor cores from k-independent per-orientation blocks,
//     G_k = sum_{n,n'} conj(b_n) b_n' F_nn',   F_nn' = Ym_n (Y_h^T Y_h)_{nn'} Ym_n'^T,
// folded by the symmetries F_n'n = F_nn'^T into a symmetric (Fs) and an antisymmetric (Fa) part:
//     Re G = sum_{n<=n'} Re(conj(b_n) b_n') Fs_nn',    Im G = sum_{n<n'} Im(conj(b_n) b_n') Fa_nn'
// (one real GEMM each, [bins x pairs] x [pairs x (orientation, packed lower triangle)]).
// A warp-per-matrix inversion then yields X = G^-1 and the bound cond_2(G) <= ||G||_F ||X||_F; where that
// bound alone cannot decide cond_2(G) <= tau, a Cholesky of the shifted matrix sigma I - G does
// (gram_certify_kernel).  Bins with a refused matrix go through the TSQR + Jacobi kernels.
#include "kernels.h"
#include "ozaki.cuh"
#include "reflect.cuh"

namespace emagls {

// ---------------------------------------------------------------------------------------------
// F blocks.  grid (pairs n<=n', orientation), pair index q = n'(n'+1)/2 + n.
// Fs[(q*P + o)*ne + e], Fa[(qa*P + o)*ne + e] with qa = n'(n'-1)/2 + n (n < n'),
// e = m(m+1)/2 + m' (m >= m').
// ---------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(256)
build_F_kernel(const double* __restrict__ Gh, int S, const double* __restrict__ Y, int Mc, int P,
               int ne_ld, double* __restrict__ Fs, double* __restrict__ Fa) {
  extern __shared__ double fsm[];
  const int q = blockIdx.x, o = blockIdx.y, tid = threadIdx.x;
  int np = (int)((sqrt(8.0 * q + 1.0) - 1.0) * 0.5);
  while ((np + 1) * (np + 2) / 2 <= q) ++np;
  while (np * (np + 1) / 2 > q) --np;
  const int n = q - np * (np + 1) / 2;
  const int wn = 2 * n + 1, wnp = 2 * np + 1, s0 = n * n, sp0 = np * np;
  double* Yn = fsm;                 // [Mc][wn]
  double* Ynp = Yn + Mc * wn;       // [Mc][wnp]
  double* Z = Ynp + Mc * wnp;       // [wn][Mc]
  double* Fm = Z + wn * Mc;         // [Mc][Mc+1]
  const double* Yo = Y + (long long)o * Mc * S;
  for (int idx = tid; idx < Mc * wn; idx += blockDim.x) Yn[idx] = Yo[(long long)(idx / wn) * S + s0 + idx % wn];
  for (int idx = tid; idx < Mc * wnp; idx += blockDim.x) Ynp[idx] = Yo[(long long)(idx / wnp) * S + sp0 + idx % wnp];
  __syncthreads();
  for (int idx = tid; idx < wn * Mc; idx += blockDim.x) {
    const int s = idx / Mc, mp = idx % Mc;
    const double* g = Gh + (long long)(s0 + s) * S + sp0;
    const double* y = Ynp + mp * wnp;
    double acc = 0.0;
    for (int t = 0; t < wnp; ++t) acc = fma(g[t], y[t], acc);
    Z[idx] = acc;
  }
  __syncthreads();
  for (int idx = tid; idx < Mc * Mc; idx += blockDim.x) {
    const int m = idx / Mc, mp = idx % Mc;
    const double* y = Yn + m * wn;
    double acc = 0.0;
    for (int s = 0; s < wn; ++s) acc = fma(y[s], Z[s * Mc + mp], acc);
    Fm[m * (Mc + 1) + mp] = acc;
  }
  __syncthreads();
  const int ne = Mc * (Mc + 1) / 2;
  double* fs = Fs + ((long long)q * P + o) * ne_ld;
  double* fa = (n < np) ? Fa + ((long long)(np * (np - 1) / 2 + n) * P + o) * ne_ld : nullptr;
  if (tid == 0 && ne_ld > ne) { fs[ne] = 0.0; if (fa) fa[ne] = 0.0; }  // alignment pad column
  for (int e = tid; e < ne; e += blockDim.x) {
    int m = (int)((sqrt(8.0 * e + 1.0) - 1.0) * 0.5);
    while ((m + 1) * (m + 2) / 2 <= e) ++m;
    while (m * (m + 1) / 2 > e) --m;
    const int mp = e - m * (m + 1) / 2;
    const double a = Fm[m * (Mc + 1) + mp], b = Fm[mp * (Mc + 1) + m];
    if (n == np) fs[e] = 0.5 * (a + b);
    else { fs[e] = a + b; fa[e] = a - b; }
  }
}

cudaError_t launch_build_F(cudaStream_t st, const double* Gh, int S, int N, const double* Y, int Mc,
                           int P, int ne_ld, double* Fs, double* Fa) {
  const int wmax = 2 * N + 1;
  size_t smem = ((size_t)2 * Mc * wmax + (size_t)wmax * Mc + (size_t)Mc * (Mc + 1)) * sizeof(double);
  const cudaError_t e = allow_dynamic_smem(build_F_kernel, smem);
  if (e != cudaSuccess) return e;
  dim3 grid((N + 1) * (N + 2) / 2, P);
  build_F_kernel<<<grid, 256, smem, st>>>(Gh, S, Y, Mc, P, ne_ld, Fs, Fa);
  return cudaGetLastError();
}

// beta tables: bre[k][q] = Re(conj(b_n) b_n') (n <= n'), bim[k][qa] = Im(conj(b_n) b_n') (n < n')
__global__ void gram_beta_kernel(const cplx* __restrict__ bn, int N, int K, double* __restrict__ bre,
                                 double* __restrict__ bim) {
  const int nqs = (N + 1) * (N + 2) / 2, nqa = N * (N + 1) / 2;
  long long idx = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (idx >= (long long)K * nqs) return;
  const int k = (int)(idx / nqs), q = (int)(idx % nqs);
  int np = (int)((sqrt(8.0 * q + 1.0) - 1.0) * 0.5);
  while ((np + 1) * (np + 2) / 2 <= q) ++np;
  while (np * (np + 1) / 2 > q) --np;
  const int n = q - np * (np + 1) / 2;
  const cplx a = bn[(long long)k * (N + 1) + n], b = bn[(long long)k * (N + 1) + np];
  bre[(long long)k * nqs + q] = fma(a.x, b.x, a.y * b.y);
  if (n < np) bim[(long long)k * nqa + np * (np - 1) / 2 + n] = fma(a.x, b.y, -a.y * b.x);
}

cudaError_t launch_gram_beta(cudaStream_t st, const cplx* bn, int N, int K, double* bre, double* bim) {
  long long total = (long long)K * ((N + 1) * (N + 2) / 2);
  gram_beta_kernel<<<(unsigned)((total + 255) / 256), 256, 0, st>>>(bn, N, K, bre, bim);
  return cudaGetLastError();
}

// ---------------------------------------------------------------------------------------------
// Warp-per-matrix inverse and route decision.  Matrix id = bin * P + o.
// Output Pb[id][i][m] = Ginv[m][i] (so that W = v * Pb), fail[1 + bin] += 1 when the route is refused,
// sig[id] > 0 for a matrix the Frobenius bound leaves undecided (see gram_classify).
// ---------------------------------------------------------------------------------------------
constexpr int GC_WPC = 4;
// Relative margin of the shifted-Cholesky certificate.  It covers the error of the computed inverse
// (about cond M u < 1e-10 at cond <= 1e4), the backward error of the Cholesky of sigma I - G (about
// gamma_{M+1} M sigma < 1e-13 sigma) and the rounding of the assembled G.
constexpr double GRAM_CERT_DELTA = 1e-6;

__device__ __forceinline__ void gram_refuse(long long id, int P, int* fail) {
  atomicAdd(fail, 1);
  atomicAdd(fail + 1 + (int)(id / P), 1);
}

// Route decision from condF = ||G||_F ||X||_F, X the computed inverse (one lane per matrix).  ||X||_F >= ||G^-1||_2
// and ||G||_F >= lambda_max, so condF <= thr proves cond_2(G) <= thr; each factor exceeds its 2-norm by at most
// sqrt(Mc), so condF > Mc thr proves cond_2(G) > thr.  In between the matrix is a candidate: sig[id] =
// thr (1 - delta) / ||X||_F <= thr lambda_min, and gram_certify_kernel accepts it iff sigma I - G is positive definite.
__device__ __forceinline__ void gram_classify(double fro2, double froi2, double thr, int Mc, long long id, int P,
                                              double* sig, int* fail) {
  const double xf = sqrt(froi2), condF = sqrt(fro2) * xf;
  double s = 0.0;
  if (condF <= thr) {
  } else if (condF <= Mc * thr) {
    s = thr * (1.0 - GRAM_CERT_DELTA) / xf;
  } else {
    gram_refuse(id, P, fail);
  }
  sig[id] = s;
}

// Packed lower triangle (entry e = m(m+1)/2 + m', m >= m') into the rows of L (leading dimension LD);
// returns this lane's share of ||G||_F^2.
__device__ __forceinline__ double gram_load_lower(cplx* L, int LD, const double* gr, const double* gi, int Mc, int lane) {
  const int ne = Mc * (Mc + 1) / 2;
  double fro = 0.0;
  for (int e = lane; e < ne; e += 32) {
    int m = (int)((sqrt(8.0 * e + 1.0) - 1.0) * 0.5);
    while ((m + 1) * (m + 2) / 2 <= e) ++m;
    while (m * (m + 1) / 2 > e) --m;
    const int mp = e - m * (m + 1) / 2;
    const double re = gr[e], im = (m == mp) ? 0.0 : gi[e];
    L[m * LD + mp] = mk(re, im);
    fro += (m == mp) ? re * re : 2.0 * fma(re, re, im * im);
  }
  return fro;
}

// Right-looking Cholesky of the lower triangle of L in place, lane = row; dinv[j] = 1 / L[j][j].
// Returns false at the first pivot that is not positive and finite.
__device__ __forceinline__ bool chol_lower(cplx* L, int LD, double* dinv, int Mc, int lane) {
  for (int j = 0; j < Mc; ++j) {
    const double d = L[j * LD + j].x;
    if (!(d > 0.0) || !(d < 1e300)) return false;   // warp-uniform
    const double ljj = sqrt(d), inv = 1.0 / ljj;
    __syncwarp();
    for (int r = lane; r < Mc; r += 32) {
      if (r > j) { cplx v = L[r * LD + j]; L[r * LD + j] = mk(v.x * inv, v.y * inv); }
      else if (r == j) { L[j * LD + j] = mk(ljj, 0.0); dinv[j] = inv; }
    }
    __syncwarp();
    for (int r = lane; r < Mc; r += 32) {
      if (r > j) {
        const cplx lrj = L[r * LD + j];
        for (int c = j + 1; c <= r; ++c) {
          const cplx lcj = L[c * LD + j];
          cplx a = L[r * LD + c];
          // a -= lrj * conj(lcj)
          a.x = fma(-lrj.x, lcj.x, a.x); a.x = fma(-lrj.y, lcj.y, a.x);
          a.y = fma(-lrj.y, lcj.x, a.y); a.y = fma(lrj.x, lcj.y, a.y);
          L[r * LD + c] = a;
        }
      }
    }
    __syncwarp();
  }
  return true;
}

// shared memory of one warp of gram_chol_kernel / gram_certify_kernel: L [Mc][Mc + 1] and dinv [Mc]
__host__ __device__ inline size_t chol_warp_elems(int Mc) { return (size_t)Mc * (Mc + 1) + (Mc + 1) / 2; }

__global__ void __launch_bounds__(GC_WPC * 32)
gram_chol_kernel(const double* __restrict__ Gre, const double* __restrict__ Gim, int Mc, int P, int ne_ld,
                 long long nmat, double thr, cplx* __restrict__ Pb, double* __restrict__ sig, int* __restrict__ fail) {
  extern __shared__ __align__(16) unsigned char gsm_raw[];
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const long long id = (long long)blockIdx.x * (blockDim.x >> 5) + warp;   // blockDim.x / 32 matrices per CTA
  if (id >= nmat) return;
  const int LD = Mc + 1;
  cplx* L = reinterpret_cast<cplx*>(gsm_raw) + (size_t)warp * chol_warp_elems(Mc);
  double* dinv = reinterpret_cast<double*>(L + (size_t)Mc * LD);  // 1 / L[j][j]

  double fro = gram_load_lower(L, LD, Gre + id * ne_ld, Gim + id * ne_ld, Mc, lane);
#pragma unroll
  for (int s = 16; s > 0; s >>= 1) fro += __shfl_xor_sync(0xffffffffu, fro, s);
  __syncwarp();
  if (!chol_lower(L, LD, dinv, Mc, lane)) {
    if (lane == 0) { sig[id] = 0.0; gram_refuse(id, P, fail); }
    return;
  }
  // Li = L^-1 (lower), stored transposed in the strict upper triangle: Li[r][c] -> L[c*LD + r]
  // lane = column c;  Li[r][c] = -(sum_{l=c}^{r-1} L[r][l] Li[l][c]) / L[r][r],  Li[c][c] = dinv[c]
  for (int r = 1; r < Mc; ++r) {
    for (int c0 = 0; c0 < r; c0 += 32) {
      const int c = c0 + lane;
      cplx sum = mk(0.0, 0.0);
      if (c < r) {
        for (int l = c; l < r; ++l) {
          const cplx lrl = L[r * LD + l];
          const cplx lic = (l == c) ? mk(dinv[c], 0.0) : L[c * LD + l];
          cfma(sum, lrl, lic);
        }
        const double di = -dinv[r];
        L[c * LD + r] = mk(sum.x * di, sum.y * di);
      }
    }
    __syncwarp();
  }
  // Ginv[m][i] = sum_{l >= max(m,i)} conj(Li[l][m]) Li[l][i];  lane = i, loop over m
  double froi = 0.0;
  cplx* out = Pb + id * (long long)Mc * Mc;
  for (int m = 0; m < Mc; ++m) {
    for (int i = lane; i < Mc; i += 32) {
      cplx g = mk(0.0, 0.0);
      const int l0 = (m > i) ? m : i;
      for (int l = l0; l < Mc; ++l) {
        const cplx a = (l == m) ? mk(dinv[m], 0.0) : L[m * LD + l];   // Li[l][m]
        const cplx b = (l == i) ? mk(dinv[i], 0.0) : L[i * LD + l];   // Li[l][i]
        cfmac(g, a, b);
      }
      froi += cabs2(g);
      out[(long long)m * Mc + i] = mk(g.x, -g.y);   // Pb[m][i] = Ginv[i][m] = conj(Ginv[m][i])
    }
  }
#pragma unroll
  for (int s = 16; s > 0; s >>= 1) froi += __shfl_xor_sync(0xffffffffu, froi, s);
  if (lane == 0) gram_classify(fro, froi, thr, Mc, id, P, sig, fail);
}

// ---------------------------------------------------------------------------------------------
// Register-resident variant for Mc <= 32: lane i of a warp holds row i of the (padded 32 x 32)
// Hermitian matrix and the warp inverts it in place by sweeps,
//   sweep(k): d = A_kk;  A_kk <- -1/d;  A_ik <- A_ik / d;  A_ij <- A_ij - A_ik conj(A_jk) / d   (i, j != k),
// after which A = -G^-1.  The pivots are the Cholesky pivots (Schur-complement diagonals), so the
// positive-definiteness test is the same; every step is a full rank-1 update with no triangular load
// imbalance, no square root and one reciprocal; only the pivot column (512 B per warp) goes through
// shared memory and is read back as broadcasts.  The k loop is fully unrolled so that the row stays in
// registers.  Same outputs and route decision as gram_chol_kernel.
// ---------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(GC_WPC * 32, 3)
gram_sweep_kernel(const double* __restrict__ Gre, const double* __restrict__ Gim, int Mc, int P, int ne_ld,
                  long long nmat, double thr, cplx* __restrict__ Pb, double* __restrict__ sig, int* __restrict__ fail) {
  __shared__ cplx colbuf[GC_WPC][32];
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const long long id = (long long)blockIdx.x * GC_WPC + warp;
  if (id >= nmat) return;
  const double* gr = Gre + id * ne_ld;
  const double* gi = Gim + id * ne_ld;
  cplx* col = colbuf[warp];
  cplx a[32];
  double fro = 0.0;
#pragma unroll
  for (int j = 0; j < 32; ++j) {
    if (lane < Mc && j < Mc) {
      const int hi = max(lane, j), lo = min(lane, j);
      const int e = hi * (hi + 1) / 2 + lo;
      const double re = gr[e];
      double im = (hi == lo) ? 0.0 : gi[e];       // packed entry (hi, lo); row lane, column j
      if (j > lane) im = -im;                      // upper triangle: conj
      a[j] = mk(re, im);
      fro += fma(re, re, im * im);
    } else {
      a[j] = mk((j == lane) ? 1.0 : 0.0, 0.0);     // identity padding: inert under the sweeps
    }
  }
#pragma unroll
  for (int s = 16; s > 0; s >>= 1) fro += __shfl_xor_sync(0xffffffffu, fro, s);
  bool ok = true;
#pragma unroll
  for (int k = 0; k < 32; ++k) {
    if (ok && k < Mc) {                            // uniform across the warp
      col[lane] = a[k];
      __syncwarp();
      const double d = col[k].x;
      if (!(d > 0.0) || !(d < 1e300)) {
        ok = false;
      } else {
        const double inv = __drcp_rn(d);
        // One update for every lane: rows i != k take a_ij -= f_i conj(A_jk) with f_i = a_ik / d; the pivot row itself
        // becomes a_kj / d = conj(A_jk) / d (Hermitian), i.e. the same update from a zeroed row with f_k = -1/d,
        // and the pivot column ends as f for all of them (no divergent second path).
        cplx f = mk(a[k].x * inv, a[k].y * inv);
        if (lane == k) {
          f = mk(-inv, 0.0);
#pragma unroll
          for (int j = 0; j < 32; ++j) a[j] = mk(0.0, 0.0);
        }
#pragma unroll
        for (int j = 0; j < 32; ++j) {
          if (j == k) continue;
          const cplx cj = col[j];                  // broadcast
          // a_ij -= f * conj(A_jk)
          a[j].x = fma(-f.x, cj.x, a[j].x); a[j].x = fma(-f.y, cj.y, a[j].x);
          a[j].y = fma(-f.y, cj.x, a[j].y); a[j].y = fma(f.x, cj.y, a[j].y);
        }
        a[k] = f;
      }
      __syncwarp();
    }
  }
  if (!ok) {
    if (lane == 0) { sig[id] = 0.0; gram_refuse(id, P, fail); }
    return;
  }
  // Ginv = -A;  Pb[m][i] = Ginv[i][m]  (W = v * Pb): lane i writes column i, coalesced over the lanes
  double froi = 0.0;
  cplx* out = Pb + id * (long long)Mc * Mc;
#pragma unroll
  for (int m = 0; m < 32; ++m) {
    if (lane < Mc && m < Mc) {
      out[(long long)m * Mc + lane] = mk(-a[m].x, -a[m].y);
      froi += cabs2(a[m]);
    }
  }
#pragma unroll
  for (int s = 16; s > 0; s >>= 1) froi += __shfl_xor_sync(0xffffffffu, froi, s);
  if (lane == 0) gram_classify(fro, froi, thr, Mc, id, P, sig, fail);
}

// ---------------------------------------------------------------------------------------------
// Certificate for the candidates of the inversion kernels (Mc <= 64).  sigma = sig[id] <= thr lambda_min(G), so a
// Cholesky of sigma I - G with every pivot positive proves lambda_max(G) < sigma, i.e. cond_2(G) < thr; the first
// pivot that is not positive refuses the matrix.  lambda_max >= max_i G_ii refuses without factoring when a diagonal
// entry reaches sigma.  Candidates are a few per cent of the matrices and sit in a few neighbouring bins (contiguous
// ids), so with W warps in the grid warp w reads the 32 ids w + W l (l = lane) per round, which spreads them over all
// warps, and factors the candidates among them one after the other, skipping those of a bin that is refused already.
// ---------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(GC_WPC * 32)
gram_certify_kernel(const double* __restrict__ Gre, const double* __restrict__ Gim, int Mc, int P, int ne_ld,
                    long long nmat, const double* __restrict__ sig, int* fail) {
  extern __shared__ __align__(16) unsigned char gsm_raw[];
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const int LD = Mc + 1;
  cplx* L = reinterpret_cast<cplx*>(gsm_raw) + (size_t)warp * chol_warp_elems(Mc);
  double* dinv = reinterpret_cast<double*>(L + (size_t)Mc * LD);
  const long long nw = (long long)gridDim.x * (blockDim.x >> 5);
  for (long long base = (long long)blockIdx.x * (blockDim.x >> 5) + warp; base < nmat; base += 32 * nw) {
    const long long mine = base + nw * lane;
    const double s_lane = (mine < nmat) ? sig[mine] : 0.0;
    unsigned cand = __ballot_sync(0xffffffffu, s_lane > 0.0);
    while (cand) {
      const int l = __ffs(cand) - 1;
      cand &= cand - 1;
      const long long id = base + nw * l;
      const double s = __shfl_sync(0xffffffffu, s_lane, l);
      int refused = 0;
      if (lane == 0) refused = *reinterpret_cast<volatile const int*>(fail + 1 + id / P);
      if (__shfl_sync(0xffffffffu, refused, 0) != 0) continue;
      const double* gr = Gre + id * ne_ld;
      double dmax = 0.0;
      for (int m = lane; m < Mc; m += 32) dmax = fmax(dmax, gr[m * (m + 1) / 2 + m]);
#pragma unroll
      for (int sh = 16; sh > 0; sh >>= 1) dmax = fmax(dmax, __shfl_xor_sync(0xffffffffu, dmax, sh));
      bool ok = dmax < s;
      if (ok) {
        gram_load_lower(L, LD, gr, Gim + id * ne_ld, Mc, lane);
        __syncwarp();
        for (int r = lane; r < Mc; r += 32)   // sigma I - G
          for (int c = 0; c <= r; ++c) {
            const cplx g = L[r * LD + c];
            L[r * LD + c] = mk((c == r ? s : 0.0) - g.x, -g.y);
          }
        __syncwarp();
        ok = chol_lower(L, LD, dinv, Mc, lane);
        __syncwarp();                          // L is reloaded for the next candidate
      }
      if (!ok && lane == 0) gram_refuse(id, P, fail);
    }
  }
}

cudaError_t launch_gram_chol(cudaStream_t st, const double* Gre, const double* Gim, int Mc, int P,
                             int ne_ld, int nbins, double thr, cplx* Pb, double* sig, int* fail) {
  if (Mc > 64) return cudaErrorInvalidValue;
  const long long nmat = (long long)nbins * P;
  const size_t per_warp = chol_warp_elems(Mc) * sizeof(cplx);
  // as many warps (matrices) per CTA as the 227 KB of shared memory hold (4 up to Mc = 59, 3 from Mc = 60)
  int wpc = GC_WPC;
  while (wpc > 1 && per_warp * wpc > 227 * 1024) --wpc;
  const size_t smem = per_warp * wpc;
  if (Mc <= 32) {
    gram_sweep_kernel<<<(unsigned)((nmat + GC_WPC - 1) / GC_WPC), GC_WPC * 32, 0, st>>>(Gre, Gim, Mc, P, ne_ld, nmat, thr,
                                                                                    Pb, sig, fail);
  } else {
    const cudaError_t e = allow_dynamic_smem(gram_chol_kernel, smem);
    if (e != cudaSuccess) return e;
    gram_chol_kernel<<<(unsigned)((nmat + wpc - 1) / wpc), wpc * 32, smem, st>>>(Gre, Gim, Mc, P, ne_ld, nmat, thr,
                                                                                      Pb, sig, fail);
  }
  cudaError_t e = cudaGetLastError();
  if (e != cudaSuccess) return e;
  // certificate: one resident wave of CTAs (228 KB of shared memory per SM, 1 KB of it reserved per CTA)
  e = allow_dynamic_smem(gram_certify_kernel, smem);
  if (e != cudaSuccess) return e;
  const long long chunks = (nmat + 31) / 32;
  const long long resident = (long long)sm_count() * std::max<size_t>(1, (228 * 1024) / (smem + 1024));
  const unsigned ncta = (unsigned)std::min((chunks + wpc - 1) / wpc, resident);
  gram_certify_kernel<<<ncta, wpc * 32, smem, st>>>(Gre, Gim, Mc, P, ne_ld, nmat, sig, fail);
  return cudaGetLastError();
}

// ---------------------------------------------------------------------------------------------
// EXTENSION (config.diffuseness_const, default off): diffuse-field covariance constraint.  The reference removed
// this step before the surveyed commit (CHANGELOG.md:10-18; outputs resources/*_wDC.mat remain), so it follows the
// published formulation the CHANGELOG names (Zaunschirm, Schoerkhuber, Hoeldrich 2018) as restated in
// oracle.diffuseness_matrix: per bin, with the target covariance R = H H^H / D of the HRTF set and the covariance
// Rhat = (W pw)(W pw)^H / D = W (pw pw^H) W^H / D of the rendered plane-wave responses,
//     W <- A W,   A = X^H Q Xh^-H,   R = X^H X, Rhat = Xh^H Xh (Cholesky),   Q^H = polar factor of Xh X^H.
// pw pw^H = conj(G_k) is the Gram matrix the Gram route assembles anyway.
// ---------------------------------------------------------------------------------------------
// R[k] = {sum |HL|^2, sum |HR|^2, Re sum HL conj(HR), Im ...} / D from the two ears' spectra Hd [D][2K]
__global__ void __launch_bounds__(256)
target_cov_kernel(const double* __restrict__ HdL, const double* __restrict__ HdR, int D, int K, double* __restrict__ out) {
  const int k = blockIdx.x, tid = threadIdx.x;
  double a = 0.0, b = 0.0, cr = 0.0, ci = 0.0;
  for (int d = tid; d < D; d += blockDim.x) {
    const double2 l = *reinterpret_cast<const double2*>(HdL + ((long long)d * K + k) * 2);
    const double2 r = *reinterpret_cast<const double2*>(HdR + ((long long)d * K + k) * 2);
    a = fma(l.x, l.x, fma(l.y, l.y, a));
    b = fma(r.x, r.x, fma(r.y, r.y, b));
    cr += l.x * r.x + l.y * r.y;          // l conj(r)
    ci += l.y * r.x - l.x * r.y;
  }
  __shared__ double red[4][8];
  a = wsum(a); b = wsum(b); cr = wsum(cr); ci = wsum(ci);
  if ((tid & 31) == 0) { red[0][tid >> 5] = a; red[1][tid >> 5] = b; red[2][tid >> 5] = cr; red[3][tid >> 5] = ci; }
  __syncthreads();
  if (tid < 4) {
    double s = 0.0;
    for (int w = 0; w < 8; ++w) s += red[tid][w];
    out[(long long)k * 4 + tid] = s / (double)D;
  }
}

cudaError_t launch_target_cov(cudaStream_t st, const double* HdL, const double* HdR, int D, int K, double* out) {
  target_cov_kernel<<<K, 256, 0, st>>>(HdL, HdR, D, K, out);
  return cudaGetLastError();
}

// 2 x 2 mixing matrix (row-major a[0..3]); false when a covariance is not positive definite
__device__ bool diffuseness_mix(double r11, double r22, cplx r12, double h11r, double h22r, cplx h12r, cplx (&a)[4]) {
  // Cholesky factors (upper): R = X^H X, Rhat = Xh^H Xh
  if (!(r11 > 0.0) || !(h11r > 0.0)) return false;
  const double x11 = sqrt(r11), g11 = sqrt(h11r);
  const cplx x12 = mk(r12.x / x11, r12.y / x11), g12 = mk(h12r.x / g11, h12r.y / g11);
  const double x22s = r22 - cabs2(x12), g22s = h22r - cabs2(g12);
  if (!(x22s > 0.0) || !(g22s > 0.0) || !(x22s < 1e300) || !(g22s < 1e300)) return false;
  const double x22 = sqrt(x22s), g22 = sqrt(g22s);
  // B = Xh X^H
  const cplx b00 = cadd(mk(g11 * x11, 0.0), cmulc(g12, x12));   // g11 x11 + g12 conj(x12)   (cmulc(a, b) = a conj(b))
  const cplx b01 = mk(g12.x * x22, g12.y * x22);
  const cplx b10 = mk(g22 * x12.x, -g22 * x12.y);
  const cplx b11 = mk(g22 * x22, 0.0);
  // P = B^H B, polar factor Pm = c B (P + s I)^-1 with s = |det B|, c = sqrt(tr P + 2 s)
  const double p00 = cabs2(b00) + cabs2(b10), p11 = cabs2(b01) + cabs2(b11);
  const cplx p01 = cadd(cmulc(b01, b00), cmulc(b11, b10));      // conj(b00) b01 + conj(b10) b11
  const cplx det = csub(cmul(b00, b11), cmul(b01, b10));
  const double sdet = sqrt(cabs2(det));
  const double c = sqrt(p00 + p11 + 2.0 * sdet);
  const double m00 = p00 + sdet, m11 = p11 + sdet;
  const double dm = m00 * m11 - cabs2(p01);
  if (!(dm > 0.0)) return false;
  const double f = c / dm;
  // inv(M) = [[m11, -p01], [-conj(p01), m00]] / dm
  const cplx i00 = mk(m11 * f, 0.0), i01 = mk(-p01.x * f, -p01.y * f), i10 = mk(-p01.x * f, p01.y * f), i11 = mk(m00 * f, 0.0);
  const cplx q00 = cadd(cmul(b00, i00), cmul(b01, i10)), q01 = cadd(cmul(b00, i01), cmul(b01, i11));
  const cplx q10 = cadd(cmul(b10, i00), cmul(b11, i10)), q11 = cadd(cmul(b10, i01), cmul(b11, i11));
  // T = X^H Pm^H:  X^H = [[x11, 0], [conj(x12), x22]],  Pm^H = [[conj q00, conj q10], [conj q01, conj q11]]
  const cplx t00 = mk(x11 * q00.x, -x11 * q00.y), t01 = mk(x11 * q10.x, -x11 * q10.y);
  const cplx t10 = cadd(cmulc(cconj(x12), q00), mk(x22 * q01.x, -x22 * q01.y));   // conj(x12) conj(q00) + x22 conj(q01)
  const cplx t11 = cadd(cmulc(cconj(x12), q10), mk(x22 * q11.x, -x22 * q11.y));
  // A = T Xh^-H,  Xh^-H = [[1/g11, 0], [-conj(g12)/(g11 g22), 1/g22]]
  const double ig11 = 1.0 / g11, ig22 = 1.0 / g22;
  const cplx l10 = mk(-g12.x * ig11 * ig22, g12.y * ig11 * ig22);
  a[0] = cadd(mk(t00.x * ig11, t00.y * ig11), cmul(t01, l10));
  a[1] = mk(t01.x * ig22, t01.y * ig22);
  a[2] = cadd(mk(t10.x * ig11, t10.y * ig11), cmul(t11, l10));
  a[3] = mk(t11.x * ig22, t11.y * ig22);
  return true;
}

// one warp per (bin of the group, chunk-local problem): lane m holds W_l(m), W_r(m)
__global__ void __launch_bounds__(128)
diffuseness_apply_kernel(const double* __restrict__ Gre, const double* __restrict__ Gim, int Mc, int oc, int ne_ld, int nb,
                         int gb0, int D, const double* __restrict__ Rt, ProbMap pm, int pj, cplx* __restrict__ Wsp,
                         long long w_ear_stride, int K, int dc_fix, int nyquist_real) {
  const int lane = threadIdx.x & 31;
  const long long id = (long long)blockIdx.x * 4 + (threadIdx.x >> 5);
  if (id >= (long long)nb * pj) return;
  const int b = (int)(id / pj), j = (int)(id - (long long)b * pj);
  const int k = gb0 + b, ol = j % oc, set = j / oc;
  const long long p = pm.global(j);
  const double* gr = Gre + ((long long)b * oc + ol) * ne_ld;
  const double* gi = Gim + ((long long)b * oc + ol) * ne_ld;
  cplx* w0p = Wsp + (p * Mc + lane) * K + k;
  cplx* w1p = w0p + w_ear_stride;
  const bool act = lane < Mc;
  const cplx w0 = act ? *w0p : mk(0.0, 0.0), w1 = act ? *w1p : mk(0.0, 0.0);
  // t_b(m) = sum_m' conj(G(m, m')) conj(W_b(m'))  (pw pw^H = conj(G)); packed entry (hi, lo) holds G(hi, lo)
  cplx t0 = mk(0.0, 0.0), t1 = mk(0.0, 0.0);
  for (int mp = 0; mp < Mc; ++mp) {
    cplx v0, v1;
    v0.x = __shfl_sync(0xffffffffu, w0.x, mp); v0.y = __shfl_sync(0xffffffffu, w0.y, mp);
    v1.x = __shfl_sync(0xffffffffu, w1.x, mp); v1.y = __shfl_sync(0xffffffffu, w1.y, mp);
    if (act) {
      const int hi = max(lane, mp), lo = min(lane, mp);
      const int e = hi * (hi + 1) / 2 + lo;
      double im = (hi == lo) ? 0.0 : gi[e];
      if (mp > lane) im = -im;                       // G(lane, mp), upper triangle: conj of the stored entry
      const cplx gc = mk(gr[e], -im);                // conj(G(lane, mp))
      cfma(t0, gc, cconj(v0));
      cfma(t1, gc, cconj(v1));
    }
  }
  // Rhat_ab = sum_m W_a(m) t_b(m) / D
  const cplx h00 = wsumc(cmul(w0, t0)), h01 = wsumc(cmul(w0, t1)), h11 = wsumc(cmul(w1, t1));
  const double* rt = Rt + ((long long)set * K + k) * 4;
  cplx r12 = mk(rt[2], rt[3]), g12 = mk(h01.x / D, h01.y / D);
  if (nyquist_real && k == K - 1) { r12.y = 0.0; g12.y = 0.0; }
  cplx a[4];
  if (!diffuseness_mix(rt[0], rt[1], r12, h00.x / D, h11.x / D, g12, a)) return;   // warp-uniform
  if (act) {
    const cplx n0 = cadd(cmul(a[0], w0), cmul(a[1], w1)), n1 = cadd(cmul(a[2], w0), cmul(a[3], w1));
    *w0p = n0; *w1p = n1;
    if (dc_fix && k == 1) { w0p[-1] = mk(n0.x, 0.0); w1p[-1] = mk(n1.x, 0.0); }   // lib/getEMagLs2Filters.m:109-110
  }
}

cudaError_t launch_diffuseness_apply(cudaStream_t st, const double* Gre, const double* Gim, int Mc, int oc, int ne_ld, int nb,
                                     int gb0, int D, const double* Rt, ProbMap pm, int pj, cplx* Wsp, long long w_ear_stride,
                                     int K, int dc_fix, int nyquist_real) {
  if (Mc > 32) return cudaErrorInvalidValue;
  const long long n = (long long)nb * pj;
  diffuseness_apply_kernel<<<(unsigned)((n + 3) / 4), 128, 0, st>>>(Gre, Gim, Mc, oc, ne_ld, nb, gb0, D, Rt, pm, pj, Wsp,
                                                                    w_ear_stride, K, dc_fix, nyquist_real);
  return cudaGetLastError();
}

// ---------------------------------------------------------------------------------------------
// forward: u = b_k .* (Y_o^T w_{k-1})  ->  Cv rows (j*2+ear)*2 + {re, im}, S doubles each.
// One CTA per chunk-local problem j (set = j / oc, orientation o0 + j % oc), both ears.
// ---------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(128)
fwd_small_kernel(const double* __restrict__ Y, int Mc, int S, const int* __restrict__ roword,
                 const cplx* __restrict__ bk, ProbMap pm, const cplx* __restrict__ Wsp,
                 long long w_ear_stride, int K, int kprev, double* __restrict__ Cv) {
  __shared__ cplx w_s[2][64];
  const int j = blockIdx.x, tid = threadIdx.x;
  const int ol = j % pm.oc;
  const long long p = pm.global(j);
  for (int idx = tid; idx < 2 * Mc; idx += blockDim.x) {
    const int e = idx / Mc, m = idx % Mc;
    w_s[e][m] = Wsp[(long long)e * w_ear_stride + (p * Mc + m) * K + kprev];
  }
  __syncthreads();
  const double* Yo = Y + (long long)ol * Mc * S;
  double* c0 = Cv + ((long long)(j * 2 + 0) * 2) * S;
  double* c1 = Cv + ((long long)(j * 2 + 1) * 2) * S;
  for (int s = tid; s < S; s += blockDim.x) {
    double a0r = 0.0, a0i = 0.0, a1r = 0.0, a1i = 0.0;
#pragma unroll 8
    for (int m = 0; m < Mc; ++m) {
      const double y = Yo[(long long)m * S + s];
      a0r = fma(y, w_s[0][m].x, a0r); a0i = fma(y, w_s[0][m].y, a0i);
      a1r = fma(y, w_s[1][m].x, a1r); a1i = fma(y, w_s[1][m].y, a1i);
    }
    const cplx b = bk[roword[s]];
    c0[s] = fma(b.x, a0r, -b.y * a0i); c0[S + s] = fma(b.x, a0i, b.y * a0r);
    c1[s] = fma(b.x, a1r, -b.y * a1i); c1[S + s] = fma(b.x, a1i, b.y * a1r);
  }
}

cudaError_t launch_fwd_small(cudaStream_t st, const double* Y, int Mc, int S, const int* roword,
                             const cplx* bk, ProbMap pm, int num_prob, const cplx* Wsp,
                             long long w_ear_stride, int K, int kprev, double* Cv) {
  if (Mc > 64) return cudaErrorInvalidValue;
  fwd_small_kernel<<<num_prob, 128, 0, st>>>(Y, Mc, S, roword, bk, pm, Wsp, w_ear_stride, K, kprev, Cv);
  return cudaGetLastError();
}

// ---------------------------------------------------------------------------------------------
// backward (Gram bins): v = Y_o (conj(b_k) .* z),  W_k = v * Pb.   z rows like Cv, or shared per
// (set, ear) for the LS bins (z_shared != 0: z + set*z_set_stride + ear*z_ear_stride, [re | im]).
// ---------------------------------------------------------------------------------------------
// Fused tail (T > 0): the forward contraction of the NEXT bin, u = b_{k+1} .* (Y_o^T W_k) (fwd_small_kernel),
// and its slicing into int8 digits (slice_rows_kernel), computed while Y_o is still L2-hot and W_k is in
// shared memory: the per-orientation harmonics (102 KB) are fetched from HBM once per bin instead of
// twice, and the FP64 vector u never exists in HBM.  Same arithmetic, in the same order, as the two
// separate kernels.
struct FwdFuse {
  const cplx* bk_next;     // b_n(k+1) [N+1]; nullptr: no fused tail
  int8_t* Cv_q; double* sCv; int KpS; long long rows;   // digits [T][rows][KpS], rows = 4 * num_prob
};

template <int T>
__global__ void __launch_bounds__(256)
bwd_small_kernel(const double* __restrict__ Y, int Mc, int S, const int* __restrict__ roword,
                 const cplx* __restrict__ bk, const cplx* __restrict__ Pb, ProbMap pm,
                 const double* __restrict__ z, long long z_set_stride, long long z_ear_stride,
                 int z_shared, int nsplit, long long split_stride, cplx* __restrict__ Wsp, long long w_ear_stride, int K, int k, int dc_fix,
                 FwdFuse ff) {
  extern __shared__ __align__(16) unsigned char bsm_raw[];
  cplx* zb = reinterpret_cast<cplx*>(bsm_raw);   // [2][S]
  cplx* v = zb + 2 * (size_t)S;                  // [2][Mc]
  cplx* wk = v + 2 * Mc;                         // [2][Mc]: W_k for the fused tail
  const int j = blockIdx.x, tid = threadIdx.x, lane = tid & 31, warp = tid >> 5, nw = blockDim.x >> 5;
  const int ol = j % pm.oc;
  const long long p = pm.global(j);
  const double* Yg = Y + (long long)ol * Mc * S;
  const double* z0 = z_shared ? z + (long long)(j / pm.oc) * z_set_stride : z + ((long long)(j * 2) * 2) * S;
  const double* z1 = z0 + (z_shared ? z_ear_stride : 2LL * S);
  for (int s = tid; s < S; s += blockDim.x) {
    const cplx b = bk[roword[s]];
    double r0 = z0[s], i0 = z0[S + s], r1 = z1[s], i1 = z1[S + s];
    for (int q = 1; q < nsplit; ++q) {   // split-K partials of the backward GEMM, fixed order
      const long long o = (long long)q * split_stride;
      r0 += z0[o + s]; i0 += z0[o + S + s]; r1 += z1[o + s]; i1 += z1[o + S + s];
    }
    // conj(b) * z
    zb[s] = mk(fma(b.x, r0, b.y * i0), fma(b.x, i0, -b.y * r0));
    zb[S + s] = mk(fma(b.x, r1, b.y * i1), fma(b.x, i1, -b.y * r1));
  }
  __syncthreads();
  for (int i = warp; i < Mc; i += nw) {
    const double* y = Yg + (long long)i * S;
    double a0r = 0.0, a0i = 0.0, a1r = 0.0, a1i = 0.0;
#pragma unroll 4
    for (int s = lane; s < S; s += 32) {
      const double yv = y[s];
      const cplx q0 = zb[s], q1 = zb[S + s];
      a0r = fma(yv, q0.x, a0r); a0i = fma(yv, q0.y, a0i);
      a1r = fma(yv, q1.x, a1r); a1i = fma(yv, q1.y, a1i);
    }
#pragma unroll
    for (int sh = 16; sh > 0; sh >>= 1) {
      a0r += __shfl_xor_sync(0xffffffffu, a0r, sh); a0i += __shfl_xor_sync(0xffffffffu, a0i, sh);
      a1r += __shfl_xor_sync(0xffffffffu, a1r, sh); a1i += __shfl_xor_sync(0xffffffffu, a1i, sh);
    }
    if (lane == 0) { v[i] = mk(a0r, a0i); v[Mc + i] = mk(a1r, a1i); }
  }
  __syncthreads();
  const cplx* pb = Pb + (long long)ol * Mc * Mc;
  for (int idx = tid; idx < 2 * Mc; idx += blockDim.x) {
    const int e = idx / Mc, m = idx % Mc;
    cplx acc = mk(0.0, 0.0);
#pragma unroll 8
    for (int i = 0; i < Mc; ++i) cfma(acc, v[e * Mc + i], pb[i * Mc + m]);
    cplx* wp = Wsp + (long long)e * w_ear_stride + (p * Mc + m) * K + k;
    *wp = acc;
    if (dc_fix && k == 1) wp[-1] = mk(acc.x, 0.0);  // W(1,:) = real(W(2,:)), lib/getEMagLs2Filters.m:109-110
    if (T > 0) wk[idx] = acc;
  }
  if constexpr (T > 0) {
    __shared__ double red[4][8];
    __shared__ double up_s[4];
    __syncthreads();
    double* cv = reinterpret_cast<double*>(zb);   // [4][S]: rows e*2 + {re, im} (zb is no longer needed)
    double mx[4] = {0.0, 0.0, 0.0, 0.0};
    for (int s2 = tid; s2 < S; s2 += blockDim.x) {
      double a0r = 0.0, a0i = 0.0, a1r = 0.0, a1i = 0.0;
#pragma unroll 8
      for (int m = 0; m < Mc; ++m) {
        const double y = Yg[(long long)m * S + s2];
        a0r = fma(y, wk[m].x, a0r); a0i = fma(y, wk[m].y, a0i);
        a1r = fma(y, wk[Mc + m].x, a1r); a1i = fma(y, wk[Mc + m].y, a1i);
      }
      const cplx b = ff.bk_next[roword[s2]];
      const double c0 = fma(b.x, a0r, -b.y * a0i), c1 = fma(b.x, a0i, b.y * a0r);
      const double c2 = fma(b.x, a1r, -b.y * a1i), c3 = fma(b.x, a1i, b.y * a1r);
      cv[s2] = c0; cv[S + s2] = c1; cv[2 * S + s2] = c2; cv[3 * S + s2] = c3;
      mx[0] = fmax(mx[0], fabs(c0)); mx[1] = fmax(mx[1], fabs(c1));
      mx[2] = fmax(mx[2], fabs(c2)); mx[3] = fmax(mx[3], fabs(c3));
    }
#pragma unroll
    for (int r = 0; r < 4; ++r) {
#pragma unroll
      for (int sh = 16; sh > 0; sh >>= 1) mx[r] = fmax(mx[r], __shfl_xor_sync(0xffffffffu, mx[r], sh));
      if (lane == 0) red[r][warp] = mx[r];
    }
    __syncthreads();
    if (tid < 4) {
      double m4 = 0.0;
      for (int w = 0; w < nw; ++w) m4 = fmax(m4, red[tid][w]);
      int e = 0;
      if (m4 > 0.0 && m4 < 1e300) frexp(m4, &e);           // slice_rows_kernel: 2^e > max |x|
      ff.sCv[(long long)j * 4 + tid] = scalbn(1.0, e - 6);
      up_s[tid] = scalbn(1.0, 6 - e);
    }
    __syncthreads();
    for (int idx = tid; idx < 4 * ff.KpS; idx += blockDim.x) {
      const int r = idx / ff.KpS, s2 = idx - r * ff.KpS;
      const double x = (s2 < S) ? cv[r * S + s2] * up_s[r] : 0.0;
      int8_t* o = ff.Cv_q + ((long long)j * 4 + r) * ff.KpS + s2;
      oz::slice_digits<T>(x, [&](int t, int q) { o[(long long)t * ff.rows * ff.KpS] = (int8_t)q; });
    }
  }
}

// ---------------------------------------------------------------------------------------------
// bwd_fused_kernel: the same step (and the same fused tail) for Mc <= 32, S <= 512, organised around ONE pass
// over Y_o.  The matrix (102 KB for em32) arrives in shared memory by a single bulk copy (cp.async.bulk +
// mbarrier) while the right-hand sides are prepared; two CTAs per SM, so one computes while the other loads.
// Lane = harmonic s in both contractions (consecutive lanes read consecutive doubles of a row of Y_o: no bank
// conflicts), the right-hand sides and the results of the tail stay in registers:
//   v = Y_o zb      : per lane 8 rows x 4 components of partial sums over its harmonics, then a warp
//                     reduce-scatter (31 shuffle-adds per 32 values: lane l ends with value l), warps summed through
//                     shared memory
//   W = v Pb        : thread = (m, eight rows i), partial sums through shared memory
//   u = Y_o^T W     : W broadcast from shared memory, one accumulator set per harmonic of the lane
// 10 k warp instructions per problem instead of 27 k, Y_o read from HBM / L2 once.
// ---------------------------------------------------------------------------------------------
constexpr int BF_WARPS = 8;      // v = Y_o zb: warp = (chunk set w & 3: chunks (w & 3) + 4 c, rows 16 (w >> 2) .. + 15)
constexpr int BF_CH = 4;         // S <= 512;  tail: warp w owns the chunks w and w + 8

template <int n>
__device__ __forceinline__ void reduce_scatter_step(double (&v)[32], int lane, int off) {
  const bool upper = (lane & off) != 0;
#pragma unroll
  for (int i = 0; i < n; ++i) {
    const double keep = upper ? v[i + n] : v[i];
    const double send = upper ? v[i] : v[i + n];
    v[i] = keep + __shfl_xor_sync(0xffffffffu, send, off);
  }
}

template <int T>
__global__ void __launch_bounds__(BF_WARPS * 32, 2)
bwd_fused_kernel(const double* __restrict__ Y, int Mc, int S, const int* __restrict__ roword,
                 const cplx* __restrict__ bk, const cplx* __restrict__ Pb, ProbMap pm,
                 const double* __restrict__ z, long long z_set_stride, long long z_ear_stride,
                 int z_shared, int nsplit, long long split_stride, cplx* __restrict__ Wsp, long long w_ear_stride, int K, int k, int dc_fix,
                 FwdFuse ff, int N) {
  extern __shared__ __align__(128) unsigned char bf_raw[];
  double* Ys = reinterpret_cast<double*>(bf_raw);                    // [Mc][S]
  double* vpart = Ys + (((size_t)Mc * S + 1) & ~(size_t)1);          // [4 chunk sets][32 rows][4]: partial v, then
  cplx* wpart = reinterpret_cast<cplx*>(vpart);                      // [BF_WARPS][2][32]: partial W (same 8 KB)
  cplx* vfin = wpart + BF_WARPS * 64;                                // [2][32]
  cplx* wfin = vfin + 64;                                            // [2][32]
  cplx* bks = wfin + 64;                                             // [2][40]: b_n(k), b_n(k+1)
  double* red = reinterpret_cast<double*>(bks + 80);                 // [4][BF_WARPS] row maxima, [4] scales
  __shared__ __align__(8) uint64_t bar;
  const int j = blockIdx.x, tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const int ol = j % pm.oc;
  const long long p = pm.global(j);
  const double* Yg = Y + (long long)ol * Mc * S;
  if (tid == 0) { oz::mbar_init(&bar, 1); oz::fence_barrier_init(); }
  if (tid <= N) { bks[tid] = bk[tid]; if (T > 0) bks[40 + tid] = ff.bk_next[tid]; }
  // Pb rows of this thread (m = lane, rows 4 warp .. 4 warp + 3): issued first, consumed after the contraction
  cplx pbr[4];
  {
    const cplx* pb = Pb + (long long)ol * Mc * Mc;
#pragma unroll
    for (int ii = 0; ii < 4; ++ii) {
      const int i = 4 * warp + ii;
      pbr[ii] = (i < Mc && lane < Mc) ? pb[i * Mc + lane] : mk(0.0, 0.0);
    }
  }
  __syncthreads();
  if (tid == 0) {
    const uint32_t bytes = (uint32_t)((size_t)Mc * S * sizeof(double));
    oz::mbar_expect_tx(&bar, bytes);
    asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];"
                 ::"r"(oz::smem_u32(Ys)), "l"(Yg), "r"(bytes), "r"(oz::smem_u32(&bar)) : "memory");
  }
  // ---- conj(b_k) .* z for this lane's harmonics (both ears), while Y_o is in flight
  const double* z0 = z_shared ? z + (long long)(j / pm.oc) * z_set_stride : z + ((long long)(j * 2) * 2) * S;
  const double* z1 = z0 + (z_shared ? z_ear_stride : 2LL * S);
  const int cset = warp & 3, rhalf = warp >> 2;
  double zq[BF_CH][4];
  int sidx[BF_CH];
#pragma unroll
  for (int c = 0; c < BF_CH; ++c) {
    const int s = (cset + 4 * c) * 32 + lane;
    sidx[c] = min(s, S - 1);             // lanes past the end carry zero right-hand sides
    zq[c][0] = zq[c][1] = zq[c][2] = zq[c][3] = 0.0;
    if (s < S) {
      const cplx b = bks[roword[s]];
      double r0 = z0[s], i0 = z0[S + s], r1 = z1[s], i1 = z1[S + s];
      for (int q = 1; q < nsplit; ++q) {   // split-K partials of the backward GEMM, fixed order
        const long long o = (long long)q * split_stride;
        r0 += z0[o + s]; i0 += z0[o + S + s]; r1 += z1[o + s]; i1 += z1[o + S + s];
      }
      zq[c][0] = fma(b.x, r0, b.y * i0); zq[c][1] = fma(b.x, i0, -b.y * r0);
      zq[c][2] = fma(b.x, r1, b.y * i1); zq[c][3] = fma(b.x, i1, -b.y * r1);
    }
  }
  oz::mbar_wait(&bar, 0);
  // ---- v = Y_o zb: rows 16 rhalf + 8 g + r
#pragma unroll 1
  for (int g = 0; g < 2; ++g) {
    double acc[32];
#pragma unroll
    for (int i = 0; i < 32; ++i) acc[i] = 0.0;
    int rowoff[8];
#pragma unroll
    for (int r = 0; r < 8; ++r) rowoff[r] = min(16 * rhalf + 8 * g + r, Mc - 1) * S;   // rows >= Mc: duplicates, never used
#pragma unroll
    for (int c = 0; c < BF_CH; ++c) {
      if ((cset + 4 * c) * 32 < S) {
#pragma unroll
        for (int r = 0; r < 8; ++r) {
          const double y = Ys[rowoff[r] + sidx[c]];
          acc[4 * r + 0] = fma(y, zq[c][0], acc[4 * r + 0]); acc[4 * r + 1] = fma(y, zq[c][1], acc[4 * r + 1]);
          acc[4 * r + 2] = fma(y, zq[c][2], acc[4 * r + 2]); acc[4 * r + 3] = fma(y, zq[c][3], acc[4 * r + 3]);
        }
      }
    }
    reduce_scatter_step<16>(acc, lane, 16);
    reduce_scatter_step<8>(acc, lane, 8);
    reduce_scatter_step<4>(acc, lane, 4);
    reduce_scatter_step<2>(acc, lane, 2);
    reduce_scatter_step<1>(acc, lane, 1);
    // value (row 16 rhalf + 8 g + lane / 4, component lane % 4) of chunk set cset
    vpart[cset * 128 + (16 * rhalf + 8 * g) * 4 + lane] = acc[0];
  }
  __syncthreads();
  if (tid < 128) {
    const double sum = (vpart[tid] + vpart[128 + tid]) + (vpart[256 + tid] + vpart[384 + tid]);
    const int i = tid >> 2, q = tid & 3;                 // q: ear * 2 + {re, im}
    reinterpret_cast<double*>(vfin)[((q >> 1) * 32 + i) * 2 + (q & 1)] = sum;
  }
  __syncthreads();
  // ---- W_k = v Pb: thread (m = lane, rows 4 warp .. 4 warp + 3)
  {
    cplx a0 = mk(0.0, 0.0), a1 = mk(0.0, 0.0);
#pragma unroll
    for (int ii = 0; ii < 4; ++ii) {
      const int i = 4 * warp + ii;
      cfma(a0, vfin[i], pbr[ii]);
      cfma(a1, vfin[32 + i], pbr[ii]);
    }
    wpart[(warp * 2 + 0) * 32 + lane] = a0;
    wpart[(warp * 2 + 1) * 32 + lane] = a1;
  }
  __syncthreads();
  if (tid < 64) {
    const int e = tid >> 5, m = tid & 31;
    cplx acc = wpart[e * 32 + m];
#pragma unroll
    for (int w = 1; w < BF_WARPS; ++w) acc = cadd(acc, wpart[(w * 2 + e) * 32 + m]);
    wfin[e * 32 + m] = acc;
    if (m < Mc) {
      cplx* wp = Wsp + (long long)e * w_ear_stride + (p * Mc + m) * K + k;
      *wp = acc;
      if (dc_fix && k == 1) wp[-1] = mk(acc.x, 0.0);  // W(1,:) = real(W(2,:)), lib/getEMagLs2Filters.m:109-110
    }
  }
  if constexpr (T > 0) {
    __syncthreads();
    // ---- fused tail: u = b_{k+1} .* (Y_o^T W_k) for the harmonics of chunks warp and warp + 8, then the digits of u
    constexpr int TC = 2;
    double u[TC][4];
    int ts[TC];
#pragma unroll
    for (int c = 0; c < TC; ++c) {
      u[c][0] = u[c][1] = u[c][2] = u[c][3] = 0.0;
      ts[c] = min((warp + BF_WARPS * c) * 32 + lane, S - 1);
    }
    const bool two = (warp + BF_WARPS) * 32 < S;          // warp-uniform: second chunk exists
    if ((warp * 32) < S) {
#pragma unroll 4
      for (int m = 0; m < Mc; ++m) {
        const cplx w0 = wfin[m], w1 = wfin[32 + m];
        const int ro = m * S;
        const double y0 = Ys[ro + ts[0]];
        u[0][0] = fma(y0, w0.x, u[0][0]); u[0][1] = fma(y0, w0.y, u[0][1]);
        u[0][2] = fma(y0, w1.x, u[0][2]); u[0][3] = fma(y0, w1.y, u[0][3]);
        if (two) {
          const double y1 = Ys[ro + ts[1]];
          u[1][0] = fma(y1, w0.x, u[1][0]); u[1][1] = fma(y1, w0.y, u[1][1]);
          u[1][2] = fma(y1, w1.x, u[1][2]); u[1][3] = fma(y1, w1.y, u[1][3]);
        }
      }
    }
    double mx[4] = {0.0, 0.0, 0.0, 0.0};
#pragma unroll
    for (int c = 0; c < TC; ++c) {
      const int s = (warp + BF_WARPS * c) * 32 + lane;
      if (s < S) {
        const cplx b = bks[40 + roword[s]];
        const double c0 = fma(b.x, u[c][0], -b.y * u[c][1]), c1 = fma(b.x, u[c][1], b.y * u[c][0]);
        const double c2 = fma(b.x, u[c][2], -b.y * u[c][3]), c3 = fma(b.x, u[c][3], b.y * u[c][2]);
        u[c][0] = c0; u[c][1] = c1; u[c][2] = c2; u[c][3] = c3;
        mx[0] = fmax(mx[0], fabs(c0)); mx[1] = fmax(mx[1], fabs(c1));
        mx[2] = fmax(mx[2], fabs(c2)); mx[3] = fmax(mx[3], fabs(c3));
      } else {
        u[c][0] = u[c][1] = u[c][2] = u[c][3] = 0.0;     // padding columns of the digit rows
      }
    }
#pragma unroll
    for (int r = 0; r < 4; ++r) {
#pragma unroll
      for (int sh = 16; sh > 0; sh >>= 1) mx[r] = fmax(mx[r], __shfl_xor_sync(0xffffffffu, mx[r], sh));
      if (lane == 0) red[r * BF_WARPS + warp] = mx[r];
    }
    __syncthreads();
    if (tid < 4) {
      double m4 = red[tid * BF_WARPS];
#pragma unroll
      for (int w = 1; w < BF_WARPS; ++w) m4 = fmax(m4, red[tid * BF_WARPS + w]);
      int e = 0;
      if (m4 > 0.0 && m4 < 1e300) frexp(m4, &e);           // slice_rows_kernel: 2^e > max |x|
      ff.sCv[(long long)j * 4 + tid] = scalbn(1.0, e - 6);
      red[4 * BF_WARPS + tid] = scalbn(1.0, 6 - e + 8 * (T - 4));   // with the 256^(T-4) of oz::slice_words
    }
    __syncthreads();
    double up[4];
#pragma unroll
    for (int r = 0; r < 4; ++r) up[r] = red[4 * BF_WARPS + r];
    const long long plane = ff.rows * ff.KpS;
#pragma unroll
    for (int c = 0; c < TC; ++c) {
      const int s = (warp + BF_WARPS * c) * 32 + lane;
      if (s < ff.KpS) {
#pragma unroll
        for (int r = 0; r < 4; ++r) {
          uint32_t zl, zh;
          oz::slice_words<T>(u[c][r] * up[r], zl, zh);
          int8_t* o = ff.Cv_q + ((long long)j * 4 + r) * ff.KpS + s;
          o[(T - 1) * plane] = (int8_t)zl;
          o[(T - 2) * plane] = (int8_t)(zl >> 8);
          o[(T - 3) * plane] = (int8_t)(zl >> 16);
          o[(T - 4) * plane] = (int8_t)zh;
          if (T >= 5) o[(T - 5) * plane] = (int8_t)(zh >> 8);
          if (T >= 6) o[(T - 6) * plane] = (int8_t)(zh >> 16);
        }
      }
    }
  }
}

template <int T>
static cudaError_t launch_bwd_fused_t(cudaStream_t st, size_t smem, int num_prob, const double* Y, int Mc, int S,
                                      const int* roword, const cplx* bk, const cplx* Pb, ProbMap pm, const double* z,
                                      long long z_set_stride, long long z_ear_stride, int z_shared, int nsplit,
                                      long long split_stride, cplx* Wsp, long long w_ear_stride, int K, int k, int dc_fix,
                                      FwdFuse ff, int N) {
  const cudaError_t e = allow_dynamic_smem(bwd_fused_kernel<T>, smem);
  if (e != cudaSuccess) return e;
  bwd_fused_kernel<T><<<num_prob, BF_WARPS * 32, smem, st>>>(Y, Mc, S, roword, bk, Pb, pm, z, z_set_stride, z_ear_stride,
                                                              z_shared, nsplit, split_stride, Wsp, w_ear_stride, K, k, dc_fix, ff, N);
  return cudaGetLastError();
}

template <int T>
static cudaError_t launch_bwd_small_t(cudaStream_t st, size_t smem, int num_prob, const double* Y, int Mc, int S,
                                      const int* roword, const cplx* bk, const cplx* Pb, ProbMap pm, const double* z,
                                      long long z_set_stride, long long z_ear_stride, int z_shared, int nsplit,
                                      long long split_stride, cplx* Wsp, long long w_ear_stride, int K, int k, int dc_fix,
                                      FwdFuse ff) {
  const cudaError_t e = allow_dynamic_smem(bwd_small_kernel<T>, smem);
  if (e != cudaSuccess) return e;
  bwd_small_kernel<T><<<num_prob, 256, smem, st>>>(Y, Mc, S, roword, bk, Pb, pm, z, z_set_stride, z_ear_stride, z_shared,
                                                  nsplit, split_stride, Wsp, w_ear_stride, K, k, dc_fix, ff);
  return cudaGetLastError();
}

cudaError_t launch_bwd_small(cudaStream_t st, const double* Y, int Mc, int S, const int* roword,
                             const cplx* bk, const cplx* Pb, ProbMap pm, int num_prob, const double* z,
                             long long z_set_stride, long long z_ear_stride, int z_shared, int nsplit,
                             long long split_stride, cplx* Wsp, long long w_ear_stride, int K, int k, int dc_fix,
                             const cplx* bk_next, int8_t* Cv_q, double* sCv, int KpS, int T, int N) {
  FwdFuse ff{bk_next, Cv_q, sCv, KpS, 4LL * num_prob};
  const int Tf = bk_next ? T : 0;
#define EM_BWD_ARGS num_prob, Y, Mc, S, roword, bk, Pb, pm, z, z_set_stride, z_ear_stride, z_shared, nsplit, \
                    split_stride, Wsp, w_ear_stride, K, k, dc_fix, ff
  // bwd_fused_kernel: Y_o staged once in shared memory (two CTAs per SM must fit; the bulk copy moves multiples of
  // 16 bytes); larger problems: bwd_small_kernel, which reads Y_o twice through L2.
  const size_t fused_smem = (((size_t)Mc * S + 1) & ~(size_t)1) * sizeof(double) +
                            (size_t)(BF_WARPS * 64 + 64 + 64 + 80) * sizeof(cplx) + (4 * BF_WARPS + 4) * sizeof(double);
  if (N >= 0 && N < 40 && Mc <= 32 && S <= 128 * BF_CH && ((Mc * S) & 1) == 0 &&
      fused_smem <= 113 * 1024 && (!bk_next || KpS <= 64 * BF_WARPS)) {
    switch (Tf) {
      case 0: return launch_bwd_fused_t<0>(st, fused_smem, EM_BWD_ARGS, N);
      case 4: return launch_bwd_fused_t<4>(st, fused_smem, EM_BWD_ARGS, N);
      case 6: return launch_bwd_fused_t<6>(st, fused_smem, EM_BWD_ARGS, N);
      default: return cudaErrorInvalidValue;
    }
  }
  const size_t smem = ((size_t)2 * S + 4 * Mc) * sizeof(cplx);
  switch (Tf) {
    case 0: return launch_bwd_small_t<0>(st, smem, EM_BWD_ARGS);
    case 4: return launch_bwd_small_t<4>(st, smem, EM_BWD_ARGS);
    case 6: return launch_bwd_small_t<6>(st, smem, EM_BWD_ARGS);
    default: return cudaErrorInvalidValue;
  }
#undef EM_BWD_ARGS
}

}  // namespace emagls
