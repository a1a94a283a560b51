// Per-(problem, bin) factorisation kernel and the small chain kernels of the eMagLS hot loop.
//
// Reference step (lib/getEMagLs2Filters.m:86-89):
//     pwGrid = smairMat(:,:,k) * Y_conj;  [U,s,V] = svd(pwGrid.','econ','vector');
//     s = 1 ./ max(s, c*max(s));          Y_reg_inv = conj(U) * (s .* V.');
// Here pwGrid.' = B * C with B orthonormal (the fixed Q of the HRIR-grid SH matrix, or the
// identity for measured steering data) and C a tall [rows x Mc] complex matrix that never
// leaves the SM:  C = Q_C R_C (flat-tree Householder TSQR in shared memory),
// R_C^H J = X (one-sided Jacobi) so R_C = J diag(s) (X/s)^H, and
//     Y_reg_inv = B * conj(Q_C) * Pb,     Pb = conj(J) diag(1/(s max(s, c s_max))) X^T.
// When no singular value can be clipped (||R||_F ||R^-1||_F <= 1/c, a rigorous bound) the
// Jacobi sweeps are skipped and Pb = R_C^-T (plain least squares).
#include "kernels.h"
#include "reflect.cuh"

namespace emagls {

constexpr int FT = 256;  // threads of the factorisation kernel

BlockPlan make_block_plan(int S, int Mc) {
  BlockPlan bp;
  bp.S = S; bp.Mc = Mc; bp.sep = 0;
  bp.MC = (Mc <= 32) ? 32 : 64;
  // MC = 32: row blocks of 96 (three CTAs per SM).  Blocks of 64 (four CTAs per SM) measured on B200: the factor
  // kernel gains 2.7 % and the reflector chain, which then has 192 instead of 128 reflectors per problem, loses as much.
  bp.RB = (bp.MC == 32) ? 96 : 128;
  bp.R0 = (S < Mc + bp.RB) ? S : Mc + bp.RB;
  bp.nblk = 1 + (S - bp.R0 + bp.RB - 1) / bp.RB;
  return bp;
}

size_t factor_smem_bytes(const BlockPlan& bp) {
  return (size_t)bp.MC * (bp.MC + bp.RB + 1) * sizeof(cplx) + (size_t)(2 * bp.MC + 72) * sizeof(cplx) + 256;
}

template <int GW>
__device__ __forceinline__ cplx gsum(cplx v, unsigned mask) {
#pragma unroll
  for (int m = GW / 2; m > 0; m >>= 1) {
    v.x += __shfl_xor_sync(mask, v.x, m);
    v.y += __shfl_xor_sync(mask, v.y, m);
  }
  return v;
}
template <int GW>
__device__ __forceinline__ double gsum(double v, unsigned mask) {
#pragma unroll
  for (int m = GW / 2; m > 0; m >>= 1) v += __shfl_xor_sync(mask, v, m);
  return v;
}
__device__ __forceinline__ cplx gsum8(cplx v, unsigned mask) { return gsum<8>(v, mask); }
__device__ __forceinline__ double gsum8(double v, unsigned mask) { return gsum<8>(v, mask); }
// Householder reflector scalars for a column with pivot alpha and squared tail norm xn (LAPACK
// zlarfg conventions: beta real, H = I - tau v v^H, v = [1; sc * x]).  The tail x is left unscaled in
// shared memory; sc is applied on the fly and when the reflector is flushed.
__device__ __forceinline__ void reflector_scalars(cplx alpha, double xn, double* beta_out, cplx* tau_out,
                                                  cplx* sc_out) {
  if (xn == 0.0 && alpha.y == 0.0) {
    *beta_out = alpha.x; *tau_out = mk(0.0, 0.0); *sc_out = mk(0.0, 0.0);
    return;
  }
  const double s2 = cabs2(alpha) + xn;
  const double nrm = sqrt(s2);
  const double beta = -copysign(nrm, alpha.x);
  const double ib = 1.0 / beta;
  const cplx d = mk(alpha.x - beta, alpha.y);          // alpha - beta (no cancellation: signs agree)
  const double id2 = 1.0 / cabs2(d);
  *beta_out = beta;
  *tau_out = mk((beta - alpha.x) * ib, -alpha.y * ib);
  *sc_out = mk(d.x * id2, -d.y * id2);                 // 1 / (alpha - beta)
}

// One Householder step of qr_block with groups of GW lanes per trailing column: apply reflector j to
// the columns c > j; the group of column j+1 accumulates the tail norm of its updated column inside
// the update loop and produces the next reflector's scalars.
template <int GW>
__device__ __forceinline__ void qr_step(cplx* Wk, int LD, int Mc, bool first, int hi, int j, cplx* tau_s, cplx* sc_s) {
  const int tid = threadIdx.x, group = tid / GW, rl = tid % GW;
  const unsigned gmask = (GW == 32) ? 0xffffffffu : (((1u << GW) - 1u) << (threadIdx.x & (32 - GW) & 31));
  const int lo = first ? j + 1 : Mc;
  const cplx tau = tau_s[j], sc = sc_s[j];
  const cplx* v = Wk + (size_t)j * LD;
  const bool active = (tau.x != 0.0 || tau.y != 0.0);
  for (int c = j + 1 + group; c < Mc; c += FT / GW) {
    cplx* a = Wk + (size_t)c * LD;
    const bool next = (c == j + 1);
    const int lo_next = first ? j + 2 : Mc;    // tail of column j+1 once it becomes the pivot column
    double xn = 0.0;
    if (active) {
      cplx w = mk(0.0, 0.0);
      for (int i = lo + rl; i < hi; i += GW) cfmac(w, v[i], a[i]);
      w = gsum<GW>(w, gmask);
      w = cmulc(w, sc);                          // conj(sc) * (x^H a)  ->  (sc x)^H a
      const cplx aj = a[j];
      w = cadd(w, aj);
      const cplx f = cmul(cconj(tau), w);        // H^H = I - conj(tau) v v^H
      const cplx fs = cmul(f, sc);
      if (rl == 0) a[j] = csub(aj, f);
      for (int i = lo + rl; i < hi; i += GW) {
        cplx ai = a[i];
        cfms(ai, fs, v[i]);
        a[i] = ai;
        if (next && i >= lo_next) xn += cabs2(ai);
      }
    } else if (next) {
      for (int i = lo_next + rl; i < hi; i += GW) xn += cabs2(a[i]);
    }
    if (next) {
      xn = gsum<GW>(xn, gmask);
      __syncwarp(gmask);
      if (rl == 0) {
        double beta; cplx t2, s2;
        reflector_scalars(a[j + 1], xn, &beta, &t2, &s2);
        a[j + 1] = mk(beta, 0.0); tau_s[j + 1] = t2; sc_s[j + 1] = s2;
      }
    }
  }
}

// In-place QR of one block held in shared memory (column-major, leading dimension LD).
// first: rows [0, nrows) dense;  otherwise: upper-triangular top (Mc rows) + dense rows [Mc, Mc+nb).
// Groups of 8 lanes own one trailing column each (16 / 32 lanes once no more than 16 / 8 columns
// remain), so the per-step critical path is one fused dot/update pass, two group reductions and the
// reflector scalars.
__device__ void qr_block(cplx* Wk, int LD, int Mc, bool first, int hi, cplx* tau_s, cplx* sc_s) {
  const int tid = threadIdx.x, group = tid >> 3, rl = tid & 7;
  const unsigned gmask = 0xffu << (threadIdx.x & 24);
  if (group == 0) {
    double xn = 0.0;
    for (int i = (first ? 1 : Mc) + rl; i < hi; i += 8) xn += cabs2(Wk[i]);
    xn = gsum8(xn, gmask);
    if (rl == 0) {
      double beta; cplx tau, sc;
      reflector_scalars(Wk[0], xn, &beta, &tau, &sc);
      Wk[0] = mk(beta, 0.0); tau_s[0] = tau; sc_s[0] = sc;
    }
  }
  __syncthreads();
  for (int j = 0; j < Mc; ++j) {
    const int rem = Mc - 1 - j;
    if (rem > FT / 16) qr_step<8>(Wk, LD, Mc, first, hi, j, tau_s, sc_s);
    else if (rem > FT / 32) qr_step<16>(Wk, LD, Mc, first, hi, j, tau_s, sc_s);
    else qr_step<32>(Wk, LD, Mc, first, hi, j, tau_s, sc_s);
    __syncthreads();
  }
}

template <int MC, int RB>
__global__ void __launch_bounds__(FT, (MC == 32) ? 3 : 1)
factor_kernel(BlockPlan bp, RowSource src, OperatorSet ops, int kbase, int G, double regul, int try_fast) {
  // one element of padding per column: with LD = MC + RB the column stride is a multiple of 128 bytes and the
  // block loads / flushes below (consecutive threads -> consecutive columns) hit one bank group (ncu, round 1: 4.3-way)
  constexpr int LD = MC + RB + 1;
  extern __shared__ __align__(16) unsigned char fsm_raw[];
  cplx* Wk = reinterpret_cast<cplx*>(fsm_raw);
  cplx* tau_s = Wk + (size_t)MC * LD;
  cplx* sc_s = tau_s + MC;
  cplx* bn_s = sc_s + MC;   // up to 64 orders
  double* red = reinterpret_cast<double*>(bn_s + 72);

  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const int prob = blockIdx.x / G, slot = blockIdx.x % G, k = kbase + slot;
  const long long oidx = (long long)prob * G + slot;
  const int S = bp.S, Mc = bp.Mc;
  cplx* Vg = ops.V + oidx * ops.v_stride;
  cplx* taug = ops.tau + oidx * ops.tau_stride;

  const bool factored = (src.E != nullptr);
  if (factored) {
    for (int n = tid; n <= src.N; n += FT) bn_s[n] = src.bn[(long long)k * (src.N + 1) + n];
  }
  __syncthreads();

  // ---------------- flat-tree TSQR over row blocks
  for (int t = 0; t < bp.nblk; ++t) {
    const int r0 = (t == 0) ? 0 : bp.R0 + (t - 1) * RB;
    const int r1 = (t == 0) ? bp.R0 : min(S, r0 + RB);
    const int dst = (t == 0) ? 0 : Mc;
    const int nb = r1 - r0;
    if (factored) {
      const double* Eo = src.E + (long long)prob * src.Etot;
      for (int idx = tid; idx < nb * Mc; idx += FT) {
        int i = r0 + idx / Mc, c = idx % Mc;
        int ord = src.roword[i];
        const double* e = Eo + src.rowoff[i] + c;
        double ar = 0.0, ai = 0.0;
        for (int n = ord; n <= src.N; ++n) {
          double ev = e[(long long)(n - ord) * Mc];
          ar = fma(bn_s[n].x, ev, ar);
          ai = fma(bn_s[n].y, ev, ai);
        }
        Wk[(size_t)c * LD + dst + (i - r0)] = mk(ar, ai);
      }
    } else {
      const cplx* At = src.At + (long long)k * src.at_bin_stride + (long long)prob * src.at_prob_stride;
      for (int idx = tid; idx < nb * Mc; idx += FT) {
        int i = r0 + idx / Mc, c = idx % Mc;
        Wk[(size_t)c * LD + dst + (i - r0)] = At[(long long)i * Mc + c];
      }
    }
    __syncthreads();
    qr_block(Wk, LD, Mc, t == 0, dst + nb, tau_s, sc_s);
    // flush reflectors of this block (qr_block ends with a barrier); the tails are stored scaled
    // (v = [1; sc * x]) for the chain kernels
    for (int idx = tid; idx < nb * Mc; idx += FT) {
      int c = idx / nb, q = idx % nb;
      cplx val = Wk[(size_t)c * LD + dst + q];
      if (t != 0 || q > c) val = cmul(val, sc_s[c]);
      Vg[(long long)c * S + r0 + q] = val;
    }
    for (int c = tid; c < Mc; c += FT) taug[t * MC + c] = tau_s[c];
    __syncthreads();
  }

  // ---------------- compact R_C (upper triangular, column-major ld = MC) into region A0
  cplx* Rs = Wk;
  cplx* Xs = Wk + MC * MC;
  cplx* Js = Wk + 2 * MC * MC;
  {
    constexpr int PER = MC * MC / FT;
    cplx tmp[PER];
#pragma unroll
    for (int q = 0; q < PER; ++q) {
      int idx = tid + q * FT, c = idx / MC, r = idx % MC;
      tmp[q] = (r <= c && c < Mc) ? Wk[(size_t)c * LD + r] : mk(0.0, 0.0);
    }
    __syncthreads();
#pragma unroll
    for (int q = 0; q < PER; ++q) Rs[tid + q * FT] = tmp[q];
    __syncthreads();
  }
  // ---------------- R^-1 (upper triangular) into region A2, row by row from the bottom: if
  // ||R||_F ||R^-1||_F <= 1/c no singular value can be clipped and Pb = R^-T.  Skipped (try_fast == 0)
  // for bins the Gram route has already refused: they go straight to the Jacobi SVD.
  cplx* Ri = Js;
  bool fast = false;
  if (try_fast) {
    for (int idx = tid; idx < MC * MC; idx += FT) Ri[idx] = mk(0.0, 0.0);
    __syncthreads();
    {
      const int group = tid >> 3, rl = tid & 7;
      const unsigned gmask = 0xffu << (threadIdx.x & 24);
      for (int i = Mc - 1; i >= 0; --i) {
        const cplx rii = Rs[i * MC + i];
        for (int m = i + group; m < Mc; m += FT / 8) {
          cplx sum = mk(0.0, 0.0);
          for (int j = i + 1 + rl; j <= m; j += 8) cfma(sum, Rs[j * MC + i], Ri[m * MC + j]);
          sum = gsum8(sum, gmask);
          if (rl == 0) {
            cplx num = mk((m == i ? 1.0 : 0.0) - sum.x, -sum.y);
            Ri[m * MC + i] = cdiv(num, rii);   // Ri col-major: Ri[m*MC + i] = Rinv(i, m)
          }
        }
        __syncthreads();
      }
    }
    // Frobenius norms
    double fr = 0.0, fi = 0.0;
    for (int idx = tid; idx < MC * MC; idx += FT) { fr += cabs2(Rs[idx]); fi += cabs2(Ri[idx]); }
    fr = wsum(fr); fi = wsum(fi);
    if (lane == 0) { red[warp] = fr; red[8 + warp] = fi; }
    __syncthreads();
    if (tid == 0) {
      double a = 0.0, b = 0.0;
      for (int w = 0; w < FT / 32; ++w) { a += red[w]; b += red[8 + w]; }
      red[16] = sqrt(a) * sqrt(b);
    }
    __syncthreads();
    const double condF = red[16];
    fast = (regul > 0.0) ? (condF <= 1.0 / regul) : (condF < 1e300);  // NaN -> false
  }
  cplx* Ps = Rs;  // region A0 is reused for Pb (row-major [i][m], ld = MC)
  int sweeps = 0;
  if (fast) {
    __syncthreads();
    for (int idx = tid; idx < MC * MC; idx += FT) {
      int i = idx / MC, m = idx % MC;
      Ps[idx] = Ri[i * MC + m];  // Pb(i,m) = Rinv(m,i) = Ri[i*MC + m]
    }
    __syncthreads();
  } else {
    // ---------------- one-sided Jacobi on X = R_C^H (columns graded like the rows of R_C)
    for (int idx = tid; idx < MC * MC; idx += FT) {
      int j = idx / MC, i = idx % MC;
      cplx r = Rs[i * MC + j];  // R(j,i)
      Xs[idx] = mk(r.x, -r.y);
    }
    __syncthreads();
    for (int idx = tid; idx < MC * MC; idx += FT) Js[idx] = mk((idx / MC == idx % MC) ? 1.0 : 0.0, 0.0);
    __syncthreads();
    const int ne = (Mc + 1) & ~1;  // even number of players (index Mc is a dummy when Mc is odd)
    const double tol2 = 4.930380657631324e-32 * (double)Mc;   // (eps sqrt(Mc))^2
    // one pair per half-warp: 16 lanes x (MC/16) rows, 4-step reductions; the 2 * FT/32 half-warps
    // cover the ne/2 pairs of a round-robin round in one pass for Mc <= 32
    constexpr int RPL = MC / 16;   // rows per lane
    const int half = lane >> 4, hl = lane & 15;
    const unsigned hmask = 0xffffu << (16 * half);
    // Rotation scalars without divisions by |g| (t ph = 2 g sign(d) / (|d| + sqrt(d^2 + 4 |g|^2)),
    // d = b - a): one rsqrt-based square root, one reciprocal, one rsqrt.  A sweep whose largest
    // cosine stayed below 1e-7 leaves every pair orthogonal to ~30 * 1e-14 (quadratic convergence), two
    // orders below the 1e-12 the projector is needed to, so no trailing check sweep is run after it.
    // (Offline study on the em32 bins, row-cyclic order: the same projector to every printed digit as with
    // a 1e-9 threshold, one sweep less on most bins: 9 -> 8, 8 -> 7.)
    for (sweeps = 1; sweeps <= 40; ++sweeps) {
      int big = 0;
      for (int r = 0; r < ne - 1; ++r) {
        for (int pi = warp * 2 + half; pi < ne / 2; pi += FT / 16) {
          int p, q;
          if (pi == 0) { p = ne - 1; q = r; }
          else { p = (r + pi) % (ne - 1); q = (r - pi + (ne - 1)) % (ne - 1); }
          if (p >= Mc || q >= Mc) continue;
          if (p > q) { int t_ = p; p = q; q = t_; }
          cplx xp[RPL], xq[RPL];
          double a = 0.0, b = 0.0; cplx g = mk(0.0, 0.0);
#pragma unroll
          for (int u = 0; u < RPL; ++u) {
            int row = hl + 16 * u;
            xp[u] = Xs[p * MC + row]; xq[u] = Xs[q * MC + row];
            a += cabs2(xp[u]); b += cabs2(xq[u]);
            cfmac(g, xp[u], xq[u]);
          }
#pragma unroll
          for (int sft = 8; sft > 0; sft >>= 1) {
            a += __shfl_xor_sync(hmask, a, sft); b += __shfl_xor_sync(hmask, b, sft);
            g.x += __shfl_xor_sync(hmask, g.x, sft); g.y += __shfl_xor_sync(hmask, g.y, sft);
          }
          const double gg = cabs2(g), ab = a * b;
          if (gg > tol2 * ab && gg > 0.0) {
            if (gg > 1e-14 * ab) big = 1;
            const double d = b - a;
            const double s2 = fma(d, d, 4.0 * gg);
            const double root = s2 * rsqrt(s2);
            const double rden = __drcp_rn(fabs(d) + root);
            const double tw = copysign(2.0 * rden, d);        // t / |g|, signed
            const double cs = rsqrt(fma(tw * tw, gg, 1.0));    // 1 / sqrt(1 + t^2)
            const cplx sph = cscale(g, cs * tw);              // s * ph
            const cplx sphc = mk(sph.x, -sph.y);              // s * conj(ph)
#pragma unroll
            for (int u = 0; u < RPL; ++u) {
              int row = hl + 16 * u;
              cplx np_ = cscale(xp[u], cs); cfms(np_, sphc, xq[u]);
              cplx nq_ = cscale(xq[u], cs); cfma(nq_, sph, xp[u]);
              Xs[p * MC + row] = np_; Xs[q * MC + row] = nq_;
              cplx jp = Js[p * MC + row], jq = Js[q * MC + row];
              cplx njp = cscale(jp, cs); cfms(njp, sphc, jq);
              cplx njq = cscale(jq, cs); cfma(njq, sph, jp);
              Js[p * MC + row] = njp; Js[q * MC + row] = njq;
            }
          }
        }
        __syncthreads();
      }
      if (!__syncthreads_or(big)) break;
    }
    // singular values = column norms of X; gains 1/(s * max(s, c*smax))
    double* sv = reinterpret_cast<double*>(bn_s);  // reuse (>= 64 doubles)
    for (int j = warp; j < Mc; j += FT / 32) {
      double a = 0.0;
#pragma unroll
      for (int u = 0; u < MC / 32; ++u) a += cabs2(Xs[j * MC + lane + 32 * u]);
      a = wsum(a);
      if (lane == 0) sv[j] = sqrt(a);
    }
    __syncthreads();
    double smax = 0.0;
    for (int j = 0; j < Mc; ++j) smax = fmax(smax, sv[j]);
    __syncthreads();
    if (tid < Mc) {
      double s = sv[tid];
      sv[tid] = (s > 0.0) ? 1.0 / (s * fmax(s, regul * smax)) : 0.0;
    }
    __syncthreads();
    for (int idx = tid; idx < MC * MC; idx += FT) {
      int i = idx / MC, m = idx % MC;
      cplx acc = mk(0.0, 0.0);
      if (i < Mc && m < Mc) {
        for (int j = 0; j < Mc; ++j) {
          cplx jc = Js[j * MC + i];
          cplx xg = cscale(Xs[j * MC + m], sv[j]);
          cfmac(acc, jc, xg);  // conj(J(i,j)) * gain_j * X(m,j)
        }
      }
      Ps[idx] = acc;
    }
    __syncthreads();
  }
  {
    cplx* Pg = ops.Pb + oidx * ops.pb_stride;
    for (int idx = tid; idx < Mc * Mc; idx += FT) {
      int i = idx / Mc, m = idx % Mc;
      Pg[idx] = Ps[i * MC + m];
    }
    if (tid == 0 && ops.info) ops.info[oidx] = fast ? 0 : sweeps;
  }
}

cudaError_t launch_factor(cudaStream_t st, const BlockPlan& bp, const RowSource& src,
                          const OperatorSet& ops, int num_prob, int kbase, int G, double regul, int try_fast) {
  size_t smem = factor_smem_bytes(bp);
  cudaError_t e;
  if (bp.MC == 32) {
    e = allow_dynamic_smem(factor_kernel<32, 96>, smem);
    if (e != cudaSuccess) return e;
    factor_kernel<32, 96><<<num_prob * G, FT, smem, st>>>(bp, src, ops, kbase, G, regul, try_fast);
  } else {
    e = allow_dynamic_smem(factor_kernel<64, 128>, smem);
    if (e != cudaSuccess) return e;
    factor_kernel<64, 128><<<num_prob * G, FT, smem, st>>>(bp, src, ops, kbase, G, regul, try_fast);
  }
  return cudaGetLastError();
}

// =============================================================================================
// chain kernels: one warp per problem, both ears; x (rows x 2 ears) lives in shared memory.
// =============================================================================================
constexpr int CH_MAXW = 4;

__global__ void chain_bwd_kernel(BlockPlan bp, OperatorSet ops, int slot, int G, const double* tq,
                                 long long tq_set_stride, long long tq_ear_stride, int tq_shared,
                                 int nsplit, long long split_stride, ProbMap pm, cplx* Wsp, long long w_ear_stride,
                                 int K, int k, int dc_fix, int num_prob) {
  extern __shared__ __align__(16) unsigned char csm_raw[];
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5, wpc = blockDim.x >> 5;
  const int j = blockIdx.x * wpc + warp;
  if (j >= num_prob) return;
  const long long p = pm.global(j);
  const int S = bp.S, Mc = bp.Mc;
  cplx* x0 = reinterpret_cast<cplx*>(csm_raw) + (size_t)warp * 2 * S;
  cplx* x1 = x0 + S;
  const long long oidx = (long long)(j % pm.oc) * G + slot;
  const cplx* V = ops.V + oidx * ops.v_stride;
  const cplx* tau = ops.tau + oidx * ops.tau_stride;
  const cplx* Pb = ops.Pb + oidx * ops.pb_stride;
  const double* t0 = tq_shared ? tq + (long long)(j / pm.oc) * tq_set_stride
                               : tq + ((long long)(j * 2 + 0) * 2) * S;
  const double* t1 = t0 + (tq_shared ? tq_ear_stride : 2 * (long long)S);
  for (int i = lane; i < S; i += 32) {
    double r0 = t0[i], i0 = t0[S + i], r1 = t1[i], i1 = t1[S + i];
    for (int z = 1; z < nsplit; ++z) {   // split-K partials of the backward GEMM, fixed order
      const long long o = (long long)z * split_stride;
      r0 += t0[o + i]; i0 += t0[o + S + i]; r1 += t1[o + i]; i1 += t1[o + S + i];
    }
    x0[i] = mk(r0, i0);
    x1[i] = mk(r1, i1);
  }
  __syncwarp();
  apply_qc(bp, V, tau, x0, x1, true, lane);
  cplx* w0p = Wsp + (p * Mc) * K + k;
  cplx* w1p = w0p + w_ear_stride;
  for (int m = lane; m < Mc; m += 32) {
    cplx a0 = mk(0.0, 0.0), a1 = mk(0.0, 0.0);
    for (int i = 0; i < Mc; ++i) {
      cplx pb = Pb[i * Mc + m];
      cfma(a0, x0[i], pb);
      cfma(a1, x1[i], pb);
    }
    w0p[(long long)m * K] = a0;
    w1p[(long long)m * K] = a1;
    if (dc_fix && k == 1) {  // W(1,:) = real(W(2,:)), lib/getEMagLs2Filters.m:109-110
      w0p[(long long)m * K - 1] = mk(a0.x, 0.0);
      w1p[(long long)m * K - 1] = mk(a1.x, 0.0);
    }
  }
}

static int chain_warps(int S) {
  int w = (int)((200 * 1024) / ((size_t)2 * S * sizeof(cplx)));
  if (w < 1) w = 1;
  if (w > CH_MAXW) w = CH_MAXW;
  return w;
}

cudaError_t launch_chain_bwd(cudaStream_t st, const BlockPlan& bp, const OperatorSet& ops, int slot,
                             int G, const double* tq, long long tq_set_stride,
                             long long tq_ear_stride, int tq_shared, int nsplit, long long split_stride,
                             ProbMap pm, cplx* Wsp, long long w_ear_stride, int K, int k, int dc_fix,
                             int num_prob) {
  int w = chain_warps(bp.S);
  size_t smem = (size_t)w * 2 * bp.S * sizeof(cplx);
  const cudaError_t e = allow_dynamic_smem(chain_bwd_kernel, smem);
  if (e != cudaSuccess) return e;
  chain_bwd_kernel<<<(num_prob + w - 1) / w, w * 32, smem, st>>>(bp, ops, slot, G, tq, tq_set_stride, tq_ear_stride, tq_shared,
                                                                 nsplit, split_stride, pm, Wsp, w_ear_stride, K, k, dc_fix,
                                                                 num_prob);
  return cudaGetLastError();
}

__global__ void phase_rows_kernel(const double* Y, double* T, int num_prob, int D, const double* absH,
                                  long long abs_set_stride, long long abs_ear_stride,
                                  int orient_per_set, int nyquist) {
  long long idx = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  long long total = (long long)num_prob * 2 * D;
  if (idx >= total) return;
  int d = (int)(idx % D);
  long long pe = idx / D;
  int ear = (int)(pe & 1);
  int p = (int)(pe >> 1);
  const double* yr = Y + (pe * 2) * D;
  double re = yr[d], im = yr[D + d];
  double mag = absH[(long long)(p / orient_per_set) * abs_set_stride + (long long)ear * abs_ear_stride + d];
  double a2 = fma(re, re, im * im), tr, ti;
  if (a2 > 0.0) { double inv = mag / sqrt(a2); tr = re * inv; ti = im * inv; }
  else { tr = mag; ti = 0.0; }
  if (nyquist) ti = 0.0;
  double* tr_ = T + (pe * 2) * D;
  tr_[d] = tr; tr_[D + d] = ti;
}

cudaError_t launch_phase_rows(cudaStream_t st, const double* Y, double* T, int num_prob, int D,
                              const double* absH, long long abs_set_stride, long long abs_ear_stride,
                              int orient_per_set, int nyquist) {
  long long total = (long long)num_prob * 2 * D;
  int bs = 256;
  phase_rows_kernel<<<(unsigned)((total + bs - 1) / bs), bs, 0, st>>>(Y, T, num_prob, D, absH, abs_set_stride,
                                                                      abs_ear_stride, orient_per_set, nyquist);
  return cudaGetLastError();
}

}  // namespace emagls
