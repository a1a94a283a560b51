// Register-resident factorisation kernels for the model-based designers with Mc <= 32 channels.
//
// Reference step (lib/getEMagLs2Filters.m:86-89), as in solver_kernels.cu:
//     [U,s,V] = svd(pwGrid.','econ','vector'); s = 1 ./ max(s, c*max(s)); Y_reg_inv = conj(U) * (s .* V.');
// with pwGrid.' = Q C_k, C_k = R diag(b_k) Y_o^T [S x Mc].  The CTA-per-problem kernel of
// solver_kernels.cu keeps C_k in shared memory; every complex multiply-add then moves 40 B through a
// 128 B/clk port, which caps it at a fifth of the FP64 rate (ncu: FP64 pipe 34 %).  Here the matrix
// never sits in shared memory:
//
//   tsqr_sep_kernel   one warp per (orientation, bin).  Lane c owns column c of a 32-row block in
//                     registers; the pivot column of a Householder step is broadcast through 512 B of
//                     shared memory, every lane forms its own inner product and update without any
//                     reduction or barrier.  Flat-tree TSQR over ceil(S/32) blocks against a 32 x 32
//                     triangle R_C that lives in a separate "R space" (the stacked matrix is [R_C; block],
//                     starting from R_C = 0), so all blocks are treated alike.
//   svdclip_kernel    one CTA per orientation, bins of a group in sequence: one-sided Jacobi on
//                     X = R_C^H (cold) or X = R_C^H J_prev (warm start from the previous bin where the
//                     grading of R_C allows it), block round-robin order: a warp holds four columns of
//                     [X; J] in registers and performs the four cross rotations (six in the first round)
//                     per load/store, incrementally updated column norms (de Rijk).
//   chain_bwd_sep_kernel  applies Q_C^H to the two ears' right-hand sides from the reflector tiles and
//                     multiplies by Pb.
//
// Reflector storage ("sep" block plan): V [S][32] row-major (a block of 32 rows is one contiguous 16 KB
// tile; entry (r, c) is the tail of reflector c of block r/32, scaled so that v = [1; tail] with the 1
// at R-space row c), tau [nblk][32].
#include <algorithm>
#include "kernels.h"
#include "reflect.cuh"

namespace emagls {

BlockPlan make_block_plan_sep(int S, int Mc) {
  BlockPlan bp;
  bp.S = S; bp.Mc = Mc; bp.MC = 32; bp.RB = 32; bp.R0 = 0;
  bp.nblk = (S + 31) / 32;
  bp.sep = 1;
  return bp;
}

namespace {

constexpr int TQ_WARPS = 4;
constexpr int TQ_TRI = 528;            // packed upper triangle of a 32 x 32 matrix
constexpr int TQ_BN = 72;              // modal coefficients of one bin (orders 0..MAX_SH_ORDER)
constexpr int TQ_XBUF = 40;             // pivot column; the folded steps keep its two halves 17 entries apart
constexpr int TQ_WARP_CPLX = TQ_TRI + TQ_XBUF + TQ_BN;

__device__ __forceinline__ int tri_idx(int j, int c) { return j * 32 - ((j * (j - 1)) >> 1) + (c - j); }

// Rows of C_k = R diag(b_k) Y_o^T that belong to order n carry the factor sum_{n' >= n} |b_n'| (R is upper
// triangular).  At low frequencies the modal coefficients of the high orders fall below 2^-60 of the largest one
// (b_n ~ (kr)^n / (2n + 1)!!), i.e. far below the rounding of the rows that matter, so the 32-row blocks made of
// such rows are left out of the factorisation and of the reflector chain (bin 1 of the em32 configuration: 2 of
// 13 blocks; from bin 55 on all of them).  The count depends on the bin only, so both kernels recompute it.
__device__ __forceinline__ int significant_blocks(const cplx* bn, int N, const int* __restrict__ roword, int S, int nblk) {
  double mx = 0.0;
  for (int n = 0; n <= N; ++n) mx = fmax(mx, cabs2(bn[n]));
  const double thr = sqrt(mx) * 8.673617379884035e-19;   // 2^-60
  int ncut = N + 1;
  double tail = 0.0;
  for (int n = N; n >= 0; --n) {
    tail += sqrt(cabs2(bn[n]));
    if (tail < thr) ncut = n; else break;
  }
  int nb = 0;
  while (nb < nblk && roword[min(nb * 32, S - 1)] < ncut) ++nb;   // orders are non-decreasing along the rows
  return max(nb, 1);
}

// LAPACK zlarfg conventions, as reflector_scalars() of solver_kernels.cu: beta real, H = I - tau v v^H,
// v = [1; sc * x].
__device__ __forceinline__ void hh_scalars(cplx alpha, double xn, double* beta_out, cplx* tau_out, cplx* sc_out) {
  if (xn == 0.0 && alpha.y == 0.0) {
    *beta_out = alpha.x; *tau_out = mk(0.0, 0.0); *sc_out = mk(0.0, 0.0);
    return;
  }
  // one reciprocal square root and one reciprocal instead of a square root and two divisions:
  // nrm = s2 rsqrt(s2), 1/beta = -sign rsqrt(s2) (one Newton step each restores the last bits),
  // |alpha - beta|^2 = |alpha|^2 + s2 + 2 |Re alpha| nrm (no cancellation: the signs agree)
  const double a2 = cabs2(alpha);
  const double s2 = a2 + xn;
  double r = rsqrt(s2);
  r = fma(r * 0.5, fma(-s2 * r, r, 1.0), r);            // Newton: r <- r + r/2 (1 - s2 r^2)
  double nrm = s2 * r;
  nrm = fma(fma(-nrm, nrm, s2), 0.5 * r, nrm);           // nrm <- nrm + (s2 - nrm^2) / (2 nrm)
  const double sg = copysign(1.0, alpha.x);
  const double beta = -sg * nrm;
  const double ib = -sg * r;
  const cplx d = mk(alpha.x - beta, alpha.y);
  const double d2 = fma(2.0 * fabs(alpha.x), nrm, a2 + s2);
  const double id2 = __drcp_rn(d2);
  *beta_out = beta;
  *tau_out = mk((beta - alpha.x) * ib, -alpha.y * ib);
  *sc_out = mk(d.x * id2, -d.y * id2);
}

// E tiles: for block t (rows 32 t ..) and order n the 32 x Mc doubles E[off(r) + (n - ord(r)) Mc + c], zero where
// n < ord(r).  The four warps of a CTA factorise four bins of the SAME orientation, so a tile is fetched once
// (cp.async, three-stage ring, two tiles in flight -- also across the Householder phase of a block) and consumed
// by all of them: b[i] += b_n(bin) * tile[i][lane].
constexpr int TQ_STAGES = 3;
constexpr int TQ_TILE = 32 * 32;       // doubles per stage

__device__ __forceinline__ void tq_issue_tile(double* tile, const double* __restrict__ Eo, const int2* rowinfo, int S,
                                              int Mc, int t, int n, bool any) {
  // one commit group per call, empty when the tile stream is exhausted (any == false)
  if (any) {
    const int r0 = t * 32;
    if ((Mc & 1) == 0) {
      const int per_row = Mc >> 1;     // 16-byte chunks per row
      for (int idx = threadIdx.x; idx < 32 * per_row; idx += TQ_WARPS * 32) {
        const int i = idx / per_row, c2 = idx - i * per_row;
        const int r = min(r0 + i, S - 1);
        const int2 ri = rowinfo[r];
        const bool ok = (r0 + i < S) && (n >= ri.x);
        cp_async16(tile + i * 32 + 2 * c2, Eo + (ok ? ri.y + (n - ri.x) * Mc + 2 * c2 : 0), ok);
      }
    } else {
      for (int idx = threadIdx.x; idx < 32 * Mc; idx += TQ_WARPS * 32) {
        const int i = idx / Mc, c = idx - i * Mc;
        const int r = min(r0 + i, S - 1);
        const int2 ri = rowinfo[r];
        const bool ok = (r0 + i < S) && (n >= ri.x);
        cp_async8(tile + i * 32 + c, Eo + (ok ? ri.y + (n - ri.x) * Mc + c : 0), ok);
      }
    }
  }
  cp_async_commit();
}

__global__ void __launch_bounds__(TQ_WARPS * 32, 3)
tsqr_sep_kernel(BlockPlan bp, RowSource src, OperatorSet ops, cplx* __restrict__ Rout, int kbase, int G, int sgroups) {
  extern __shared__ __align__(16) unsigned char tq_raw[];
  const int S = bp.S, Mc = bp.Mc;
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  int2* rowinfo = reinterpret_cast<int2*>(tq_raw);                 // (order, offset into E) per row
  const int tab_bytes = ((S * (int)sizeof(int2) + 15) / 16) * 16;
  for (int i = threadIdx.x; i < S; i += blockDim.x) rowinfo[i] = make_int2(src.roword[i], src.rowoff[i]);
  double* tiles = reinterpret_cast<double*>(tq_raw + tab_bytes);
  cplx* Rt = reinterpret_cast<cplx*>(tiles + TQ_STAGES * TQ_TILE) + (size_t)warp * TQ_WARP_CPLX;
  cplx* xbuf = Rt + TQ_TRI;
  cplx* bn_s = xbuf + TQ_XBUF;
  // CTA = one orientation x four consecutive bins of the launch; a warp without a bin only helps with the tiles
  const int prob = blockIdx.x / sgroups, slot = (blockIdx.x - prob * sgroups) * TQ_WARPS + warp;
  const bool active = slot < G;
  const int k = kbase + min(slot, G - 1);
  const long long oidx = (long long)prob * G + min(slot, G - 1);
  const int N = src.N;
  for (int n = lane; n <= N; n += 32) bn_s[n] = src.bn[(long long)k * (N + 1) + n];
  for (int i = lane; i < TQ_TRI; i += 32) Rt[i] = mk(0.0, 0.0);
  __shared__ int nblk_s[TQ_WARPS];
  __syncwarp();
  const int my_nblk = significant_blocks(bn_s, N, src.roword, S, bp.nblk);   // warp-uniform
  if (lane == 0) nblk_s[warp] = active ? my_nblk : 0;
  __syncthreads();
  int cta_nblk = 0;
#pragma unroll
  for (int w = 0; w < TQ_WARPS; ++w) cta_nblk = max(cta_nblk, nblk_s[w]);
  const double* Eo = src.E + (long long)prob * src.Etot;
  const bool col_ok = lane < Mc;
  cplx* Vg = ops.V + oidx * ops.v_stride;
  cplx* taug = ops.tau + oidx * ops.tau_stride;

  // tile stream over (block, order): iterator of the next tile to issue
  int it_t = 0, it_n = rowinfo[0].x, q_issue = 0;
  auto issue_next = [&]() {
    const bool any = it_t < cta_nblk;
    tq_issue_tile(tiles + (q_issue % TQ_STAGES) * TQ_TILE, Eo, rowinfo, S, Mc, it_t, it_n, any);
    ++q_issue;
    if (any) {
      if (it_n < N) ++it_n;
      else { ++it_t; it_n = (it_t < cta_nblk) ? rowinfo[it_t * 32].x : 0; }
    }
  };
  issue_next();
  issue_next();
  int q = 0;   // tiles consumed so far
  // Mc == 32: after 16 steps the finished lanes take over the lower half of the rows of the remaining columns,
  // so that steps 16..31 cost half (the lane = column mapping otherwise idles lane c from step c on)
  const bool fold = (Mc == 32);
  const int hoff = lane < 16 ? 17 : 0;        // this lane's half of the pivot column in xbuf (folded steps)
  const int fcol = 16 + (lane & 15);          // ... and its column

  for (int t = 0; t < cta_nblk; ++t) {
    const int r0 = t * 32;
    const bool mine = active && t < my_nblk;
    cplx b[32];
#pragma unroll
    for (int i = 0; i < 32; ++i) b[i] = mk(0.0, 0.0);
    // ---- rows r0 .. r0+31 of C_k: C[r][c] = sum_{n >= ord(r)} b_n E[off(r) + (n - ord(r)) Mc + c]
    const int nlo = rowinfo[r0].x;      // orders below that of the first row contribute nothing
    for (int n = nlo; n <= N; ++n, ++q) {
      cp_async_wait<TQ_STAGES - 2>();   // tile q has landed (this thread's copies; the barrier covers the others)
      __syncthreads();                  // ... and every warp is done with the stage tile q + 2 goes into
      issue_next();
      if (mine && col_ok) {
        const double* tile = tiles + (q % TQ_STAGES) * TQ_TILE + lane;
        const cplx bnn = bn_s[n];
#pragma unroll
        for (int i = 0; i < 32; ++i) {
          const double ev = tile[i * 32];
          b[i].x = fma(bnn.x, ev, b[i].x);
          b[i].y = fma(bnn.y, ev, b[i].y);
        }
      }
    }
    if (!mine) continue;
    // ---- Householder steps on [R_C; block]: lane = column, all 32 rows
    cplx my_tau = mk(0.0, 0.0), my_sc = mk(0.0, 0.0);
    const int jsplit = fold ? 16 : Mc;
    for (int j = 0; j < jsplit; ++j) {
      if (lane == j) {
#pragma unroll
        for (int i = 0; i < 32; ++i) xbuf[i] = b[i];
      }
      __syncwarp();
      cplx w0 = mk(0.0, 0.0), w1 = mk(0.0, 0.0), w2 = mk(0.0, 0.0), w3 = mk(0.0, 0.0);
#pragma unroll
      for (int i = 0; i < 32; i += 4) {
        cfmac(w0, xbuf[i], b[i]);
        cfmac(w1, xbuf[i + 1], b[i + 1]);
        cfmac(w2, xbuf[i + 2], b[i + 2]);
        cfmac(w3, xbuf[i + 3], b[i + 3]);
      }
      const cplx w = cadd(cadd(w0, w1), cadd(w2, w3));   // lane j: ||x||^2
      const double xn = __shfl_sync(0xffffffffu, w.x, j);
      const cplx alpha = Rt[tri_idx(j, j)];
      double beta; cplx tau, sc;
      hh_scalars(alpha, xn, &beta, &tau, &sc);           // redundantly on every lane (warp-uniform values)
      __syncwarp();
      if (lane == j) { my_tau = tau; my_sc = sc; Rt[tri_idx(j, j)] = mk(beta, 0.0); }
      if (lane > j && (tau.x != 0.0 || tau.y != 0.0)) {
        const int ti = tri_idx(j, lane);
        const cplx rjc = Rt[ti];
        const cplx wc = cadd(cmulc(w, sc), rjc);         // (sc x)^H a + a_j
        const cplx f = cmul(cconj(tau), wc);             // H^H = I - conj(tau) v v^H
        const cplx fs = cmul(f, sc);
        Rt[ti] = csub(rjc, f);
#pragma unroll
        for (int i = 0; i < 32; ++i) cfms(b[i], fs, xbuf[i]);
      }
      __syncwarp();
    }
    if (!fold) {
      // ---- flush the reflector tails of this block (scaled) and its tau row
#pragma unroll
      for (int i = 0; i < 32; ++i) {
        const int r = r0 + i;
        if (r < S) Vg[(long long)r * 32 + lane] = cmul(b[i], my_sc);
      }
      taug[t * 32 + lane] = my_tau;
      continue;
    }
    // ---- fold: columns 0..15 are finished; their lanes store the tails and take rows 16..31 of columns 16..31
    if (lane < 16) {
#pragma unroll
      for (int i = 0; i < 32; ++i) {
        const int r = r0 + i;
        if (r < S) Vg[(long long)r * 32 + lane] = cmul(b[i], my_sc);
      }
      taug[t * 32 + lane] = my_tau;
    }
#pragma unroll
    for (int i = 0; i < 16; ++i) {
      const double ux = __shfl_down_sync(0xffffffffu, b[16 + i].x, 16);
      const double uy = __shfl_down_sync(0xffffffffu, b[16 + i].y, 16);
      if (lane < 16) b[i] = mk(ux, uy);
    }
    for (int j = 16; j < 32; ++j) {
      if (fcol == j) {
#pragma unroll
        for (int i = 0; i < 16; ++i) xbuf[hoff + i] = b[i];
      }
      __syncwarp();
      cplx w0 = mk(0.0, 0.0), w1 = mk(0.0, 0.0), w2 = mk(0.0, 0.0), w3 = mk(0.0, 0.0);
#pragma unroll
      for (int i = 0; i < 16; i += 4) {
        cfmac(w0, xbuf[hoff + i], b[i]);
        cfmac(w1, xbuf[hoff + i + 1], b[i + 1]);
        cfmac(w2, xbuf[hoff + i + 2], b[i + 2]);
        cfmac(w3, xbuf[hoff + i + 3], b[i + 3]);
      }
      cplx w = cadd(cadd(w0, w1), cadd(w2, w3));
      w.x += __shfl_xor_sync(0xffffffffu, w.x, 16);      // the two halves of a column (same sum on both lanes)
      w.y += __shfl_xor_sync(0xffffffffu, w.y, 16);
      const double xn = __shfl_sync(0xffffffffu, w.x, j);
      const cplx alpha = Rt[tri_idx(j, j)];
      const bool upd = fcol > j;
      const int ti = tri_idx(j, upd ? fcol : j);
      const cplx rjc = Rt[ti];                           // read by both lanes of a column before one of them writes
      double beta; cplx tau, sc;
      hh_scalars(alpha, xn, &beta, &tau, &sc);
      __syncwarp();
      if (fcol == j) { my_tau = tau; my_sc = sc; if (lane >= 16) Rt[ti] = mk(beta, 0.0); }
      if (upd && (tau.x != 0.0 || tau.y != 0.0)) {
        const cplx wc = cadd(cmulc(w, sc), rjc);
        const cplx f = cmul(cconj(tau), wc);
        const cplx fs = cmul(f, sc);
        if (lane >= 16) Rt[ti] = csub(rjc, f);
#pragma unroll
        for (int i = 0; i < 16; ++i) cfms(b[i], fs, xbuf[hoff + i]);
      }
      __syncwarp();
    }
    {
      const int rh = r0 + (lane < 16 ? 16 : 0);
#pragma unroll
      for (int i = 0; i < 16; ++i) {
        const int r = rh + i;
        if (r < S) Vg[(long long)r * 32 + fcol] = cmul(b[i], my_sc);
      }
      if (lane >= 16) taug[t * 32 + lane] = my_tau;
    }
  }
  if (!active) return;
  // ---- R_C, full 32 x 32 row-major with zeros below the diagonal
  cplx* Rg = Rout + oidx * 1024;
  for (int j = 0; j < 32; ++j) Rg[j * 32 + lane] = (lane >= j && j < Mc && lane < Mc) ? Rt[tri_idx(j, lane)] : mk(0.0, 0.0);
}

// =============================================================================================
// svdclip_kernel: Pb = conj(J) diag(1/(s max(s, c s_max))) X^T from R_C = J diag(s) (X/s)^H
//
// One CTA of 4 warps per orientation, the bins of a launch in sequence.  X and J (32 x 32 complex each,
// column-major) live in shared memory.  Order: round-robin over 16 blocks of two columns; a half-warp
// takes one block pair per round, holds its four columns of [X; J] in registers (lane = rows hl and
// hl + 16 of X and of J) and performs the four cross rotations (plus the two inner ones in round 0) before
// the columns go back, so a rotation moves 1 KB instead of 4 KB through the shared-memory port.  The two
// independent rotations of a phase are reduced together (the halves of the 16-lane group end up with one
// inner product each) and their parameters are computed once per 8-lane group, then exchanged.
// =============================================================================================
constexpr int SV_T = 128, SV_CTAS = 4;   // threads, CTAs per SM (128 registers per thread)

struct RotParam { double cs, sx, sy, na, nb; int rot; };

// rotation parameters for the pair with inner product g and squared norms (a, b); de Rijk norm update
__device__ __forceinline__ RotParam rot_param(cplx g, double a, double b, double tol2, int& big) {
  RotParam p;
  p.cs = 1.0; p.sx = 0.0; p.sy = 0.0; p.na = a; p.nb = b; p.rot = 0;
  const double gg = cabs2(g), ab = a * b;
  if (gg > tol2 * ab && gg > 0.0) {
    if (gg > 1e-14 * ab) big = 1;
    const double d = b - a;
    const double s2 = fma(d, d, 4.0 * gg);
    const double root = s2 * rsqrt(s2);
    const double rden = __drcp_rn(fabs(d) + root);
    const double tw = copysign(2.0 * rden, d);         // t / |g|, signed
    const double cs = rsqrt(fma(tw * tw, gg, 1.0));    // 1 / sqrt(1 + t^2)
    const double f = cs * tw;
    p.cs = cs; p.sx = g.x * f; p.sy = g.y * f;         // s * ph
    p.na = fma(-tw, gg, a); p.nb = fma(tw, gg, b);
    p.rot = 1;
  }
  return p;
}

__device__ __forceinline__ void rot_apply(const RotParam& p, cplx (&xp)[2], cplx (&xq)[2], cplx (&jp)[2], cplx (&jq)[2]) {
  const cplx sph = mk(p.sx, p.sy), sphc = mk(p.sx, -p.sy);
#pragma unroll
  for (int u = 0; u < 2; ++u) {
    cplx np_ = cscale(xp[u], p.cs); cfms(np_, sphc, xq[u]);
    cplx nq_ = cscale(xq[u], p.cs); cfma(nq_, sph, xp[u]);
    xp[u] = np_; xq[u] = nq_;
    cplx njp = cscale(jp[u], p.cs); cfms(njp, sphc, jq[u]);
    cplx njq = cscale(jq[u], p.cs); cfma(njq, sph, jp[u]);
    jp[u] = njp; jq[u] = njq;
  }
}

// one phase of a half-warp: the independent pairs (a, b) and (c, d)
__device__ __forceinline__ void rot_phase(cplx (&xa)[2], cplx (&xb)[2], cplx (&ja)[2], cplx (&jb)[2], double& na, double& nb,
                                          cplx (&xc)[2], cplx (&xd)[2], cplx (&jc)[2], cplx (&jd)[2], double& nc, double& nd,
                                          bool hi8, double tol2, int& big) {
  cplx g1 = mk(0.0, 0.0), g2 = mk(0.0, 0.0);
#pragma unroll
  for (int u = 0; u < 2; ++u) { cfmac(g1, xa[u], xb[u]); cfmac(g2, xc[u], xd[u]); }
  __syncwarp();
  // lanes 0-7 of the 16-lane group collect g1, lanes 8-15 collect g2
  cplx keep = hi8 ? g2 : g1;
  const cplx send = hi8 ? g1 : g2;
  keep.x += __shfl_xor_sync(0xffffffffu, send.x, 8);
  keep.y += __shfl_xor_sync(0xffffffffu, send.y, 8);
#pragma unroll
  for (int m = 4; m > 0; m >>= 1) {
    keep.x += __shfl_xor_sync(0xffffffffu, keep.x, m);
    keep.y += __shfl_xor_sync(0xffffffffu, keep.y, m);
  }
  const RotParam mine = rot_param(keep, hi8 ? nc : na, hi8 ? nd : nb, tol2, big);
  RotParam oth;
  oth.cs = __shfl_xor_sync(0xffffffffu, mine.cs, 8);
  oth.sx = __shfl_xor_sync(0xffffffffu, mine.sx, 8);
  oth.sy = __shfl_xor_sync(0xffffffffu, mine.sy, 8);
  oth.na = __shfl_xor_sync(0xffffffffu, mine.na, 8);
  oth.nb = __shfl_xor_sync(0xffffffffu, mine.nb, 8);
  oth.rot = __shfl_xor_sync(0xffffffffu, mine.rot, 8);
  const RotParam p1 = hi8 ? oth : mine, p2 = hi8 ? mine : oth;
  if (p1.rot) { rot_apply(p1, xa, xb, ja, jb); na = p1.na; nb = p1.nb; }
  if (p2.rot) { rot_apply(p2, xc, xd, jc, jd); nc = p2.na; nd = p2.nb; }
}

__global__ void __launch_bounds__(SV_T, SV_CTAS)
svdclip_kernel(int Mc, const cplx* __restrict__ Rin, OperatorSet ops, int G, double regul, int try_fast, int split_from,
               int pieces, double warm_grading) {
  extern __shared__ __align__(16) unsigned char sv_raw[];
  cplx* Xs = reinterpret_cast<cplx*>(sv_raw);           // column-major: X(i, c) = Xs[c*32 + i]
  cplx* Js = Xs + 1024;                                 // column-major
  double* nrm = reinterpret_cast<double*>(Js + 1024);   // [32]
  double* sv = nrm + 32;                                // [32]
  double* red = sv + 32;                                // [20]
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const int hw = tid >> 4, hl = tid & 15;
  const bool hi8 = (hl & 8) != 0;
  // CTAs below split_from take all G bins of one orientation; the orientations from split_from on (the remainder of
  // the last full round of CTAs) are cut into `pieces` bin ranges each, so the last round is short (launch_svdclip)
  int prob = blockIdx.x, slot_lo = 0, slot_hi = G;
  if (prob >= split_from) {
    const int r = prob - split_from, piece = r % pieces;
    prob = split_from + r / pieces;
    slot_lo = (int)((long long)piece * G / pieces);
    slot_hi = (int)((long long)(piece + 1) * G / pieces);
  }
  bool have_j = false;                      // Js holds the converged J of the previous bin

  for (int slot = slot_lo; slot < slot_hi; ++slot) {
    const long long oidx = (long long)prob * G + slot;
    const cplx* Rg = Rin + oidx * 1024;     // R_C row-major: R(j, i) = Rg[j*32 + i]
    cplx* Pg = ops.Pb + oidx * ops.pb_stride;
    bool fast = false;
    int sweeps = 0;
    if (try_fast) {
      // R into Xs (row-major), R^-1 (upper triangular, row-major) into Js, row by row from the bottom; if
      // ||R||_F ||R^-1||_F <= 1/c no singular value can be clipped and Pb = R^-T.
      cplx* Rs = Xs;
      cplx* Ri = Js;
      for (int idx = tid; idx < 1024; idx += SV_T) { Rs[idx] = Rg[idx]; Ri[idx] = mk(0.0, 0.0); }
      __syncthreads();
      const int group = tid >> 3, rl = tid & 7;
      for (int i = Mc - 1; i >= 0; --i) {
        const cplx rii = Rs[i * 32 + i];
        // Rinv(i, m) = (delta_im - sum_{j=i+1..m} R(i, j) Rinv(j, m)) / R(i, i), one group of 8 lanes per m
        for (int m0 = 0; m0 < 32; m0 += SV_T / 8) {
          const int m = m0 + group;
          const bool act = (m >= i && m < Mc);
          cplx sum = mk(0.0, 0.0);
          if (act)
            for (int j = i + 1 + rl; j <= m; j += 8) cfma(sum, Rs[i * 32 + j], Ri[j * 32 + m]);
          sum = group_sum<8>(sum);                // every lane of the warp takes part
          if (act && rl == 0) Ri[i * 32 + m] = cdiv(mk((m == i ? 1.0 : 0.0) - sum.x, -sum.y), rii);
        }
        __syncthreads();
      }
      double fr = 0.0, fi = 0.0;
      for (int idx = tid; idx < 1024; idx += SV_T) { fr += cabs2(Rs[idx]); fi += cabs2(Ri[idx]); }
      fr = wsum(fr); fi = wsum(fi);
      if (lane == 0) { red[warp] = fr; red[8 + warp] = fi; }
      __syncthreads();
      if (tid == 0) {
        double a = 0.0, b = 0.0;
        for (int w = 0; w < SV_T / 32; ++w) { a += red[w]; b += red[8 + w]; }
        red[16] = sqrt(a) * sqrt(b);
      }
      __syncthreads();
      const double condF = red[16];
      fast = (regul > 0.0) ? (condF <= 1.0 / regul) : (condF < 1e300);   // NaN -> false
      if (fast) {
        for (int idx = tid; idx < Mc * Mc; idx += SV_T) {
          const int i = idx / Mc, m = idx - i * Mc;
          Pg[idx] = Ri[m * 32 + i];               // Pb(i, m) = Rinv(m, i)
        }
      }
      have_j = false;                             // Js was used as scratch: the next Jacobi start is cold
      __syncthreads();
    }
    if (!fast) {
      // ---- starting matrix: warm (X = R^H J_prev) where the diagonal of R_C is graded by less than 1 / warm_grading
      // (the product costs eps * grading of relative accuracy in the small columns), else cold (X = R^H, J = I)
      bool use_warm = false;
      if (have_j) {
        if (tid < 32) {
          const double d = (tid < Mc) ? fabs(Rg[tid * 32 + tid].x) : 0.0;
          double dmax = d, dmin = (tid < Mc) ? d : 1e300;
#pragma unroll
          for (int m = 16; m > 0; m >>= 1) {
            dmax = fmax(dmax, __shfl_xor_sync(0xffffffffu, dmax, m));
            dmin = fmin(dmin, __shfl_xor_sync(0xffffffffu, dmin, m));
          }
          if (tid == 0) red[17] = (dmin > warm_grading * dmax) ? 1.0 : 0.0;
        }
        __syncthreads();
        use_warm = red[17] != 0.0;
      }
      if (use_warm) {
        // X(i, c) = sum_{j <= i} conj(R(j, i)) J(j, c)
        for (int idx = tid; idx < 1024; idx += SV_T) {
          const int c = idx >> 5, i = idx & 31;
          cplx acc = mk(0.0, 0.0);
          for (int j = 0; j <= i; ++j) cfmac(acc, Rg[j * 32 + i], Js[c * 32 + j]);
          Xs[idx] = acc;
        }
      } else {
        for (int idx = tid; idx < 1024; idx += SV_T) {
          const int c = idx >> 5, i = idx & 31;
          const cplx r = Rg[idx];               // R(c, i)
          Xs[idx] = mk(r.x, -r.y);
          Js[idx] = mk(c == i ? 1.0 : 0.0, 0.0);
        }
      }
      __syncthreads();
      const double tol2 = 4.930380657631324e-32 * (double)Mc;   // (eps sqrt(Mc))^2
      for (sweeps = 1; sweeps <= 40; ++sweeps) {
        int big = 0;
        // refresh the squared column norms once per sweep
        for (int c = warp; c < 32; c += SV_T / 32) {
          const double a_ = wsum(cabs2(Xs[c * 32 + lane]));
          if (lane == 0) nrm[c] = a_;
        }
        __syncthreads();
        for (int r = 0; r < 15; ++r) {
          int A, B;
          if (hw == 0) { A = 15; B = r; }
          else { A = (r + hw) % 15; B = (r - hw + 15) % 15; }
          if (A > B) { const int t_ = A; A = B; B = t_; }
          const int c0 = 2 * A, c1 = 2 * A + 1, c2 = 2 * B, c3 = 2 * B + 1;
          cplx x0[2], x1[2], x2[2], x3[2], j0[2], j1[2], j2[2], j3[2];
#pragma unroll
          for (int u = 0; u < 2; ++u) {
            const int row = hl + 16 * u;
            x0[u] = Xs[c0 * 32 + row]; x1[u] = Xs[c1 * 32 + row]; x2[u] = Xs[c2 * 32 + row]; x3[u] = Xs[c3 * 32 + row];
            j0[u] = Js[c0 * 32 + row]; j1[u] = Js[c1 * 32 + row]; j2[u] = Js[c2 * 32 + row]; j3[u] = Js[c3 * 32 + row];
          }
          double n0 = nrm[c0], n1 = nrm[c1], n2 = nrm[c2], n3 = nrm[c3];
          if (r == 0)   // pairs inside the two blocks: once per sweep
            rot_phase(x0, x1, j0, j1, n0, n1, x2, x3, j2, j3, n2, n3, hi8, tol2, big);
          rot_phase(x0, x2, j0, j2, n0, n2, x1, x3, j1, j3, n1, n3, hi8, tol2, big);
          rot_phase(x0, x3, j0, j3, n0, n3, x1, x2, j1, j2, n1, n2, hi8, tol2, big);
#pragma unroll
          for (int u = 0; u < 2; ++u) {
            const int row = hl + 16 * u;
            Xs[c0 * 32 + row] = x0[u]; Xs[c1 * 32 + row] = x1[u]; Xs[c2 * 32 + row] = x2[u]; Xs[c3 * 32 + row] = x3[u];
            Js[c0 * 32 + row] = j0[u]; Js[c1 * 32 + row] = j1[u]; Js[c2 * 32 + row] = j2[u]; Js[c3 * 32 + row] = j3[u];
          }
          if (hl == 0) { nrm[c0] = n0; nrm[c1] = n1; nrm[c2] = n2; nrm[c3] = n3; }
          __syncthreads();
        }
        if (!__syncthreads_or(big)) break;
      }
      // singular values = column norms of X; gains 1/(s * max(s, c*smax))
      for (int c = warp; c < 32; c += SV_T / 32) {
        const double a_ = wsum(cabs2(Xs[c * 32 + lane]));
        if (lane == 0) sv[c] = sqrt(a_);
      }
      __syncthreads();
      double smax = 0.0;
      for (int c = 0; c < Mc; ++c) smax = fmax(smax, sv[c]);
      __syncthreads();
      if (tid < 32) {
        const double s = sv[tid];
        sv[tid] = (tid < Mc && s > 0.0) ? 1.0 / (s * fmax(s, regul * smax)) : 0.0;
      }
      __syncthreads();
      // Pb(i, m) = sum_c conj(J(i, c)) gain_c X(m, c)
      for (int idx = tid; idx < Mc * Mc; idx += SV_T) {
        const int i = idx / Mc, m = idx - i * Mc;
        cplx acc = mk(0.0, 0.0);
        for (int c = 0; c < Mc; ++c) cfmac(acc, Js[c * 32 + i], cscale(Xs[c * 32 + m], sv[c]));
        Pg[idx] = acc;
      }
      have_j = true;
    }
    if (tid == 0) {
      if (ops.info) ops.info[oidx] = fast ? 0 : sweeps;
      if (ops.stats && !fast) { atomicAdd(ops.stats, (unsigned long long)sweeps); atomicAdd(ops.stats + 1, 1ull); }
    }
    __syncthreads();
  }
}

// =============================================================================================
// chain_bwd_sep_kernel: W_k = ((Q_C^H tq)[R space]) * Pb for both ears; one warp per problem.
// Lane l holds row l of the current 32-row block of both right-hand sides and, in registers, row l of
// the block's reflector tile (2 x 16 complex, each half fetched while the other is applied); entry c of
// the R-space part of the right-hand sides lives in lane c.  No shared memory.
// =============================================================================================
constexpr int CS_WARPS = 4;

__device__ __forceinline__ void load_half(const cplx* __restrict__ row, bool ok, cplx (&v)[16]) {
#pragma unroll
  for (int jj = 0; jj < 16; ++jj) {
    if (ok) {
      const double2 d = __ldg(reinterpret_cast<const double2*>(row + jj));
      v[jj] = mk(d.x, d.y);
    } else {
      v[jj] = mk(0.0, 0.0);
    }
  }
}

// reflectors j0 .. j0+15 of one block (Q_C^H: in order, conj(tau))
// tau_blk: the 32 scalars of this block (read with a warp-uniform address: one load instead of four shuffles)
__device__ __forceinline__ void apply_half(const cplx (&v)[16], int j0, const cplx* __restrict__ tau_blk, cplx& xb0,
                                           cplx& xb1, cplx& xr0, cplx& xr1, int lane) {
#pragma unroll
  for (int jj = 0; jj < 16; ++jj) {
    const int j = j0 + jj;
    const double2 tj = __ldg(reinterpret_cast<const double2*>(tau_blk + j));
    const cplx ta = mk(tj.x, -tj.y);
    cplx w0 = cmulc(xb0, v[jj]), w1 = cmulc(xb1, v[jj]);   // x * conj(v)
    if (lane == j) { w0 = cadd(w0, xr0); w1 = cadd(w1, xr1); }
    wsum2c(w0, w1, lane);
    const cplx f0 = cmul(ta, w0), f1 = cmul(ta, w1);
    if (lane == j) { xr0 = csub(xr0, f0); xr1 = csub(xr1, f1); }
    cfms(xb0, f0, v[jj]); cfms(xb1, f1, v[jj]);
  }
}

__device__ __forceinline__ void load_rhs(const double* __restrict__ t0, const double* __restrict__ t1, int S, int r,
                                         int nsplit, long long split_stride, cplx& x0, cplx& x1) {
  if (r < S) {
    double r0 = t0[r], i0 = t0[S + r], r1 = t1[r], i1 = t1[S + r];
    for (int z = 1; z < nsplit; ++z) {   // split-K partials of the backward GEMM, fixed order
      const long long o = (long long)z * split_stride;
      r0 += t0[o + r]; i0 += t0[o + S + r]; r1 += t1[o + r]; i1 += t1[o + S + r];
    }
    x0 = mk(r0, i0); x1 = mk(r1, i1);
  } else {
    x0 = mk(0.0, 0.0); x1 = mk(0.0, 0.0);
  }
}

__global__ void __launch_bounds__(CS_WARPS * 32, 3)
chain_bwd_sep_kernel(BlockPlan bp, OperatorSet ops, int slot, int G, const double* __restrict__ tq,
                     long long tq_set_stride, long long tq_ear_stride, int tq_shared, int nsplit,
                     long long split_stride, ProbMap pm, cplx* __restrict__ Wsp, long long w_ear_stride, int K, int k,
                     int dc_fix, int num_prob, const cplx* __restrict__ bn_k, int N, const int* __restrict__ roword) {
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const int j = blockIdx.x * CS_WARPS + warp;
  if (j >= num_prob) return;
  const int nblk = significant_blocks(bn_k, N, roword, bp.S, bp.nblk);   // the blocks tsqr_sep_kernel factorised
  const long long p = pm.global(j);
  const int S = bp.S, Mc = bp.Mc;
  const long long oidx = (long long)(j % pm.oc) * G + slot;
  const cplx* V = ops.V + oidx * ops.v_stride;
  const cplx* tau = ops.tau + oidx * ops.tau_stride;
  const cplx* Pb = ops.Pb + oidx * ops.pb_stride;
  const double* t0 = tq_shared ? tq + (long long)(j / pm.oc) * tq_set_stride : tq + ((long long)(j * 2 + 0) * 2) * S;
  const double* t1 = t0 + (tq_shared ? tq_ear_stride : 2 * (long long)S);

  cplx xr0 = mk(0.0, 0.0), xr1 = mk(0.0, 0.0);   // R-space entry `lane` of the two right-hand sides
  cplx va[16], vb[16];
  cplx xb0, xb1;
  load_half(V + (long long)lane * 32, lane < S, va);
  load_rhs(t0, t1, S, lane, nsplit, split_stride, xb0, xb1);
  for (int t = 0; t < nblk; ++t) {
    const int r = t * 32 + lane;
    load_half(V + (long long)r * 32 + 16, r < S, vb);
    const cplx* tau_blk = tau + t * 32;
    apply_half(va, 0, tau_blk, xb0, xb1, xr0, xr1, lane);
    cplx nx0 = mk(0.0, 0.0), nx1 = mk(0.0, 0.0);
    if (t + 1 < nblk) {
      load_half(V + (long long)(r + 32) * 32, r + 32 < S, va);
      load_rhs(t0, t1, S, r + 32, nsplit, split_stride, nx0, nx1);
    }
    apply_half(vb, 16, tau_blk, xb0, xb1, xr0, xr1, lane);
    xb0 = nx0; xb1 = nx1;
  }
  // W(m) = sum_i z(i) Pb(i, m)
  cplx a0 = mk(0.0, 0.0), a1 = mk(0.0, 0.0);
  for (int i = 0; i < Mc; ++i) {
    cplx z0, z1;
    z0.x = __shfl_sync(0xffffffffu, xr0.x, i); z0.y = __shfl_sync(0xffffffffu, xr0.y, i);
    z1.x = __shfl_sync(0xffffffffu, xr1.x, i); z1.y = __shfl_sync(0xffffffffu, xr1.y, i);
    if (lane < Mc) {
      const cplx pb = Pb[i * Mc + lane];
      cfma(a0, z0, pb);
      cfma(a1, z1, pb);
    }
  }
  if (lane < Mc) {
    cplx* w0p = Wsp + (p * Mc + lane) * K + k;
    cplx* w1p = w0p + w_ear_stride;
    *w0p = a0;
    *w1p = a1;
    if (dc_fix && k == 1) {  // W(1,:) = real(W(2,:)), lib/getEMagLs2Filters.m:109-110
      w0p[-1] = mk(a0.x, 0.0);
      w1p[-1] = mk(a1.x, 0.0);
    }
  }
}

}  // namespace

size_t tsqr_sep_smem_bytes(const BlockPlan& bp) {
  return (size_t)(((bp.S * (int)sizeof(int2) + 15) / 16) * 16) + (size_t)TQ_STAGES * TQ_TILE * sizeof(double) +
         (size_t)TQ_WARPS * TQ_WARP_CPLX * sizeof(cplx);
}

cudaError_t launch_tsqr_sep(cudaStream_t st, const BlockPlan& bp, const RowSource& src, const OperatorSet& ops,
                            cplx* Rout, int num_prob, int kbase, int G) {
  if (!bp.sep || bp.Mc > 32 || src.E == nullptr || src.N + 1 > TQ_BN) return cudaErrorInvalidValue;
  const size_t smem = tsqr_sep_smem_bytes(bp);
  const cudaError_t e = allow_dynamic_smem(tsqr_sep_kernel, smem);
  if (e != cudaSuccess) return e;
  const int sgroups = (G + TQ_WARPS - 1) / TQ_WARPS;
  tsqr_sep_kernel<<<num_prob * sgroups, TQ_WARPS * 32, smem, st>>>(bp, src, ops, Rout, kbase, G, sgroups);
  return cudaGetLastError();
}

cudaError_t launch_svdclip(cudaStream_t st, int Mc, const cplx* Rin, const OperatorSet& ops, int num_prob, int G,
                           double regul, int try_fast, double warm_grading) {
  if (Mc > 32) return cudaErrorInvalidValue;
  const size_t smem = (size_t)2 * 1024 * sizeof(cplx) + (size_t)(32 + 32 + 20) * sizeof(double);
  // Tail of the grid: CTAs take about equally long, so with `resident` CTAs in flight a launch lasts
  // ceil(num_prob / resident) rounds and the last round may be almost empty (3600 orientations on 592 places: 6.08
  // -> 7 rounds).  The orientations of that remainder are cut into bin ranges, as many as fit into one round, so
  // the last round lasts 1 / pieces of a full one (plus one cold Jacobi start per piece).
  const int resident = SV_CTAS * sm_count();
  int split_from = num_prob, pieces = 1;
  const int rem = num_prob % resident;
  if (num_prob > resident && rem > 0 && G > 1) {
    pieces = std::min(G, resident / rem);
    if (pieces > 1) split_from = num_prob - rem; else pieces = 1;
  }
  const int grid = split_from + (num_prob - split_from) * pieces;
  svdclip_kernel<<<grid, SV_T, smem, st>>>(Mc, Rin, ops, G, regul, try_fast, split_from, pieces, warm_grading);
  return cudaGetLastError();
}

cudaError_t launch_chain_bwd_sep(cudaStream_t st, const BlockPlan& bp, const OperatorSet& ops, int slot, int G,
                                 const double* tq, long long tq_set_stride, long long tq_ear_stride, int tq_shared,
                                 int nsplit, long long split_stride, ProbMap pm, cplx* Wsp, long long w_ear_stride,
                                 int K, int k, int dc_fix, int num_prob, const cplx* bn_k, int N, const int* roword) {
  if (!bp.sep) return cudaErrorInvalidValue;
  chain_bwd_sep_kernel<<<(num_prob + CS_WARPS - 1) / CS_WARPS, CS_WARPS * 32, 0, st>>>(
      bp, ops, slot, G, tq, tq_set_stride, tq_ear_stride, tq_shared, nsplit, split_stride, pm, Wsp, w_ear_stride, K, k,
      dc_fix, num_prob, bn_k, N, roword);
  return cudaGetLastError();
}

}  // namespace emagls
