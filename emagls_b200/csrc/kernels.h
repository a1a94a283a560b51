// Host-callable launchers of the hand-written kernels (one translation unit per group).
#pragma once
#include <cuda_runtime.h>
#include "common.cuh"

namespace emagls {

// ---------------------------------------------------------------- setup_kernels.cu
// getSH on a direction list given as angles.  out: [(N+1)^2][D] (D contiguous) real or complex.
cudaError_t launch_sh_angles(cudaStream_t st, int N, const double* azi, const double* zen, int D,
                             int complex_basis, double* out);
// getSH('real') at rotated microphone positions: for orientation o and mic m the direction is
// R_o^T * u_m.  out: [B][M][S] (S contiguous).  rot == nullptr -> identity, B = 1 and the
// angles are used exactly as given (bit-compatible with launch_sh_angles).
cudaError_t launch_sh_mics(cudaStream_t st, int N, const double* mic_azi, const double* mic_zen,
                           int M, const double* rot, int B, double* out);
// out[o][c][s] = sum_m L[c][m] * Y[o][m][s]   (L row-major [Mc][M])
cudaError_t launch_left_mul(cudaStream_t st, const double* L, int Mc, int M, const double* Y,
                            int B, int S, double* out);
// b_n table: out[k*(N+1)+n] = sign * b_n(kr_k); nyquist_real: take real part of the last row.
cudaError_t launch_modal(cudaStream_t st, int N, const double* kr, int nk, int array_type,
                         double sign, int nyquist_real, cplx* out, long long stride_k,
                         long long stride_n);
// Householder QR of the column-major real matrix A [S cols][D rows]: after the call
// Q [S][D] holds the thin orthonormal factor and R [S][S] (row-major, upper) the triangle.
// work: D*S doubles (reflectors) + 2*S doubles.
cudaError_t launch_householder_qr(cudaStream_t st, double* A, int D, int S, double* Q, double* R,
                                  double* work, long long* launches);
// CholeskyQR2 building blocks (setup_kernels.cu): in-place upper Cholesky factor of a symmetric [S][S] matrix
// (*flag set on a non-positive pivot or a diagonal ratio beyond 1e6), upper-triangular inverse, product of two
// upper-triangular matrices (all row-major).
cudaError_t launch_chol_upper(cudaStream_t st, double* G, int S, int* flag);
cudaError_t launch_tri_inverse(cudaStream_t st, const double* R, int S, double* Rinv);
cudaError_t launch_tri_mul(cudaStream_t st, const double* R2, const double* R1, int S, double* R);
// E rows for the factored steering model:  E[o][rowoff[i] + (n-ord(i))*Mc + c] =
//   sum_{j in order-n block} R[i][j] * Ym[o][c][j]
cudaError_t launch_build_E(cudaStream_t st, const double* R, int S, int N, const double* Ym,
                           int Mc, int B, const int* rowoff, const int* roword, long long Etot,
                           double* E);
// HRIR preparation
cudaError_t launch_colsum(cudaStream_t st, const double* h, int T, int D, double* partial,
                          int nchunk, double* out);
cudaError_t launch_grpdelay(cudaStream_t st, const double* s, int T, int K, double fs, double* gd);
// DFT twiddles [2K][T]: row (k,c) holds Re/Im of exp(-2 pi i k t / nfft)
cudaError_t launch_dft_twiddle(cudaStream_t st, int K, int T, int nfft, double* tw);
// absH[k][d] = | Hd[d][(k,*)] |
cudaError_t launch_abs_transpose(cudaStream_t st, const double* Hd, int D, int K, double* absH);
// tail twiddles [len][2K] for one ear: ifft + sub-sample delay + crop + fade folded into one matrix
cudaError_t launch_tail_twiddle(cudaStream_t st, int K, int nfft, int len, double delay, double* tw);

// Chunk-local problem index j -> (set = j / oc, orientation o0 + j % oc); global problem index
// p = set * num_orient + orientation addresses the solution array Wsp.
struct ProbMap {
  int oc, o0, num_orient;
  __host__ __device__ __forceinline__ long long global(int j) const {
    return (long long)(j / oc) * num_orient + o0 + (j % oc);
  }
};

// ---------------------------------------------------------------- solver_kernels.cu
struct RowSource {
  // factored model: C[i][c] = sum_{n >= ord(i)} bn[k][n] * E[o][rowoff[i] + (n-ord(i))*Mc + c]
  const double* E; long long Etot; const int* rowoff; const int* roword; const cplx* bn; int N;
  // generic: rows read from At[(bin)][i][c] (interleaved complex, c contiguous);
  // bin_shared != 0 -> the same matrix for every problem of a bin
  const cplx* At; long long at_bin_stride; long long at_prob_stride;
};
struct OperatorSet {       // per-(problem, bin-slot) outputs of the factorisation kernel
  cplx* V;    long long v_stride;    // [Mc][S] column-major (ld = S)
  cplx* tau;  long long tau_stride;  // [nblk][MC]
  cplx* Pb;   long long pb_stride;   // [Mc][Mc] row-major: W = g * Pb
  int* info;                         // [problem*G + slot]: jacobi sweeps (0 = fast path)
  unsigned long long* stats;         // optional device counters: [0] += sweeps, [1] += 1 per Jacobi problem
};
// sep == 0: rows [0, R0) form the first (dense) block and the triangle R_C lives in rows [0, Mc) of the vector
// space (solver_kernels.cu).  sep == 1: 32-row blocks against a triangle in a separate R space (tsqr_kernels.cu).
struct BlockPlan { int S, Mc, MC, RB, R0, nblk, sep; };
BlockPlan make_block_plan(int S, int Mc);
size_t factor_smem_bytes(const BlockPlan& bp);
cudaError_t launch_factor(cudaStream_t st, const BlockPlan& bp, const RowSource& src,
                          const OperatorSet& ops, int num_prob, int kbase, int G, double regul, int try_fast);
// backward: W[k] = (Q_C^H tq) * Pb; tq rows (j*2+e)*2+c (sum of nsplit split-K partials), or shared per
// set when tq_shared != 0
cudaError_t launch_chain_bwd(cudaStream_t st, const BlockPlan& bp, const OperatorSet& ops, int slot,
                             int G, const double* tq, long long tq_set_stride,
                             long long tq_ear_stride, int tq_shared, int nsplit, long long split_stride,
                             ProbMap pm, cplx* Wsp, long long w_ear_stride, int K, int k, int dc_fix,
                             int num_prob);
// ---------------------------------------------------------------- tsqr_kernels.cu (Mc <= 32, factored model)
// Register-resident TSQR (warp per (problem, bin)), Jacobi SVD-clip (CTA per problem, the G bins of a launch in
// sequence with warm starts) and reflector application for the "sep" block plan.  V [S][32], tau [nblk][32],
// R [problem*G + slot][32][32] row-major.
BlockPlan make_block_plan_sep(int S, int Mc);
cudaError_t launch_tsqr_sep(cudaStream_t st, const BlockPlan& bp, const RowSource& src, const OperatorSet& ops,
                            cplx* Rout, int num_prob, int kbase, int G);
cudaError_t launch_svdclip(cudaStream_t st, int Mc, const cplx* Rin, const OperatorSet& ops, int num_prob, int G,
                           double regul, int try_fast, double warm_grading);
cudaError_t launch_chain_bwd_sep(cudaStream_t st, const BlockPlan& bp, const OperatorSet& ops, int slot, int G,
                                 const double* tq, long long tq_set_stride, long long tq_ear_stride, int tq_shared,
                                 int nsplit, long long split_stride, ProbMap pm, cplx* Wsp, long long w_ear_stride,
                                 int K, int k, int dc_fix, int num_prob, const cplx* bn_k, int N, const int* roword);
// generic-path phase step on rows: t = absH * y/|y|
cudaError_t launch_phase_rows(cudaStream_t st, const double* Y, double* T, int num_prob, int D,
                              const double* absH, long long abs_set_stride, long long abs_ear_stride,
                              int orient_per_set, int nyquist);

// ---------------------------------------------------------------- ema_kernels.cu
cudaError_t launch_ema_sh_rows(cudaStream_t st, int order, int simN, int M, int D, int K, int complex_basis,
                               const double* azi, const double* zen, const cplx* dec, const double* Ym,
                               const double* Yhor, const cplx* bn, cplx* At);
cudaError_t launch_ch_rows(cudaStream_t st, int N, const double* azi, int M, int complex_basis, cplx* At);
cudaError_t launch_ema_dec(cudaStream_t st, int N, int M, int npair, int complex_basis, const double* Ysh0,
                           const cplx* pinvT, cplx* dec);
cudaError_t launch_complex_tail_prep(cudaStream_t st, const cplx* W, int kind, int nch, int K, long long P,
                                     cplx* X1, cplx* X2);
cudaError_t launch_interleave(cudaStream_t st, const double* re, const double* im, long long n, cplx* out);

// ---------------------------------------------------------------- gram_kernels.cu
// F blocks of the Gram route: Fs [(nqs*P) x ne], Fa [(nqa*P) x ne] (see gram_kernels.cu)
cudaError_t launch_build_F(cudaStream_t st, const double* Gh, int S, int N, const double* Y, int Mc,
                           int P, int ne_ld, double* Fs, double* Fa);
cudaError_t launch_gram_beta(cudaStream_t st, const cplx* bn, int N, int K, double* bre, double* bim);
// Inverse and condition certificate (cond_2 < thr) of nbins*P packed Hermitian matrices (Mc <= 64), two launches;
// fail[0] counts refused matrices, fail[1 + bin] those of one bin (zero: the bin may take the Gram route);
// sig: one double per matrix of scratch.
cudaError_t launch_gram_chol(cudaStream_t st, const double* Gre, const double* Gim, int Mc, int P,
                             int ne_ld, int nbins, double thr, cplx* Pb, double* sig, int* fail);
// forward of every bin: Cv rows (j*2+ear)*2+{re,im} = b_k .* (Y_o^T W_{k-1})
// EXTENSION: diffuse-field covariance constraint (gram_kernels.cu)
cudaError_t launch_target_cov(cudaStream_t st, const double* HdL, const double* HdR, int D, int K, double* out);
cudaError_t launch_diffuseness_apply(cudaStream_t st, const double* Gre, const double* Gim, int Mc, int oc, int ne_ld, int nb,
                                     int gb0, int D, const double* Rt, ProbMap pm, int pj, cplx* Wsp, long long w_ear_stride,
                                     int K, int dc_fix, int nyquist_real);
cudaError_t launch_fwd_small(cudaStream_t st, const double* Y, int Mc, int S, const int* roword,
                             const cplx* bk, ProbMap pm, int num_prob, const cplx* Wsp,
                             long long w_ear_stride, int K, int kprev, double* Cv);
// backward of a Gram bin: W_k = (Y_o (conj(b_k) .* z)) * Pb
cudaError_t launch_bwd_small(cudaStream_t st, const double* Y, int Mc, int S, const int* roword,
                             const cplx* bk, const cplx* Pb, ProbMap pm, int num_prob, const double* z,
                             long long z_set_stride, long long z_ear_stride, int z_shared, int nsplit,
                             long long split_stride, cplx* Wsp, long long w_ear_stride, int K, int k, int dc_fix,
                             // fused forward of the next bin + slicing (bk_next != nullptr): see gram_kernels.cu
                             const cplx* bk_next = nullptr, int8_t* Cv_q = nullptr, double* sCv = nullptr,
                             int KpS = 0, int T = 0, int N = -1);

// ---------------------------------------------------------------- ozaki_kernels.cu
// FP64-accurate GEMMs on the int8 tensor cores (tcgen05 + TMEM + TMA); see ozaki.cuh.
int oz_pad32(int k);
// int32 accumulation of T slice pairs of 2^14 over Kpad terms must stay below 2^31 (Kpad <= 21845 at T = 6)
bool oz_contraction_fits(int Kpad, int T);
// x(r, k) = src[r*rs + k*cs] -> balanced base-256 digits out[T][R][Kpad] (int8) and scale[r] = 2^(e_r - 6)
cudaError_t launch_slice_rows(cudaStream_t st, const double* src, long long rs, long long cs, int R, int K, int Kpad,
                              int T, int8_t* out, double* scale);
// per row of x [rows][D]: up = 2^(6-e), sc = 2^(e-6) with 2^e > max |x(row, :)|
cudaError_t launch_row_scale(cudaStream_t st, const double* x, long long rows, int D, double* up, double* sc);
struct OzFwdArgs {
  const int8_t* YhA_q; const double* sYhA; int D, KpS;   // [T][D][KpS]: rows = directions, K = harmonics
  const int8_t* Cv_q; const double* sCv; int rows;       // [T][rows][KpS]: rows = (problem, ear, re/im)
  int T;
  int8_t* Tt_q; int KpD; double* sT;                     // out: digits of t [T][rows][KpD], scales [rows]
  const double* absH; long long abs_set_stride, abs_ear_stride;
  const double* up; const double* sc; int scale_stride;  // this bin's |H| scales, indexed (set*2+ear)*scale_stride
  int orient_per_set, nyquist;
  int raw;   // six digits: the FP64 functor instead of the integer one (EMAGLS_OZ_FWD=raw)
  int dbg;   // GemmArgs::dbg (tools/microbench/oz_fwd_bench.cu)
};
cudaError_t launch_oz_fwd(cudaStream_t st, const OzFwdArgs& a);
// tq [rows][S] = t^T B with B_q [T][S][KpD] (rows = harmonics, K = directions)
cudaError_t launch_oz_bwd(cudaStream_t st, const int8_t* Tt_q, const double* sT, int rows, const int8_t* B_q,
                          const double* sB, int S, int KpD, int T, double* tq);

}  // namespace emagls
