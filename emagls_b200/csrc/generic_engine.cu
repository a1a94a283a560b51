// Designers whose per-bin steering matrix is data rather than the factored sphere model:
//   getMagLsFilters / getLsFilters  (lib/getMagLsFilters.m:44-98, lib/getLsFilters.m:27-34)
//       pwGrid = Y_conj for every bin, plain pinv (clip disabled), DC is an LS bin, no DC fix
//   getEMagLsFiltersFromAtf         (lib/getEMagLsFiltersFromAtf.m:36-151)
//       pwGrid_k = fft(atfIrs)(k,:,:) after nearest-neighbour grid matching, integer shifts
//   getEMagLsFiltersEMAinSH         (lib/getEMagLsFiltersEMAinSH.m:60-178)
//       pwGrid_k(:,d) = (equatorial array response -> CH -> SH expansion) rotated per direction
// All share the loop of lib/getEMagLs2Filters.m:85-106.  Device formulation: per bin the rows
// A_k = pwGrid_k.' [D x Mc] are factorised by the TSQR + Jacobi kernel (solver_kernels.cu), the thin
// Q_C is formed explicitly (backward stable: reflectors applied to unit vectors), and one
// persistent CTA per (problem, ear) walks the sequential bin chain
//     t = H_k                                   (LS bins)
//     t = |H_k| .* exp(i angle(A_k W_{k-1}))      (MagLS bins; real part at Nyquist)
//     W_k = (t conj(Q_C,k)) Pb_k
// keeping t and W in shared memory: the chain is latency bound, so it is one launch, not 4 per bin.
#include <algorithm>
#include <cmath>
#include <cstdio>
#include <cstdlib>
#include <optional>
#include <vector>
#include "engine.h"
#include "gemm.cuh"
#include "reflect.cuh"
#include "special.cuh"

namespace emagls {

namespace {

// ------------------------------------------------------------------------------------------
// explicit thin Q_C:  QcT[slot][c][d] = (Q_C e_c)[d].  One warp per pair of columns.
// ------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(32)
form_q_kernel(BlockPlan bp, OperatorSet ops, cplx* __restrict__ QcT) {
  extern __shared__ __align__(16) unsigned char fq_raw[];
  const int lane = threadIdx.x, slot = blockIdx.y, c0 = blockIdx.x * 2;
  const int S = bp.S, Mc = bp.Mc;
  cplx* x0 = reinterpret_cast<cplx*>(fq_raw);
  cplx* x1 = x0 + S;
  for (int i = lane; i < S; i += 32) {
    x0[i] = mk(i == c0 ? 1.0 : 0.0, 0.0);
    x1[i] = mk(i == c0 + 1 ? 1.0 : 0.0, 0.0);
  }
  __syncwarp();
  apply_qc(bp, ops.V + (long long)slot * ops.v_stride, ops.tau + (long long)slot * ops.tau_stride, x0, x1, false, lane);
  __syncwarp();
  cplx* q0 = QcT + ((long long)slot * Mc + c0) * S;
  for (int i = lane; i < S; i += 32) q0[i] = x0[i];
  if (c0 + 1 < Mc)
    for (int i = lane; i < S; i += 32) q0[S + i] = x1[i];
}

// ------------------------------------------------------------------------------------------
// the sequential chain; grid = num_prob * 2 (ear fastest), any multiple of 32 threads
// ------------------------------------------------------------------------------------------
struct ChainArgs {
  const cplx* At; long long at_slot_stride;     // rows [slot][D][Mc]; stride 0: one operator for all bins
  const cplx* QcT; const cplx* Pb;              // [slot][Mc][D], [slot][Mc][Mc] (same slot stride rule)
  const cplx* H; long long h_prob_stride, h_ear_stride;  // targets [prob][ear][K][Dh]
  cplx* W; long long w_ear_stride, w_prob_stride;         // solutions [ear][prob][Mc][K]
  int D, Mc, K, first_bin, kls1, dc_fix, nyquist_real;
  int Dh;                                                 // row length of H (= D unless columns are gathered)
  const int* gidx; long long gidx_prob_stride;            // optional: target column of direction d is gidx[prob][d]
};

__global__ void __launch_bounds__(1024)
generic_chain_kernel(ChainArgs a) {
  extern __shared__ __align__(16) unsigned char gc_raw[];
  cplx* t = reinterpret_cast<cplx*>(gc_raw);   // [D]
  cplx* w = t + a.D;                           // [Mc]
  cplx* x = w + a.Mc;                          // [Mc]
  const int tid = threadIdx.x, nt = blockDim.x, lane = tid & 31, warp = tid >> 5, nw = nt >> 5;
  const int ear = blockIdx.x & 1, prob = blockIdx.x >> 1;
  const int D = a.D, Mc = a.Mc, K = a.K;
  for (int m = tid; m < Mc; m += nt) w[m] = mk(0.0, 0.0);
  __syncthreads();
  const cplx* Hp = a.H + (long long)prob * a.h_prob_stride + (long long)ear * a.h_ear_stride;
  cplx* Wp = a.W + (long long)ear * a.w_ear_stride + (long long)prob * a.w_prob_stride;
  for (int k = a.first_bin; k < K; ++k) {
    const long long slot = a.at_slot_stride ? (long long)(k - a.first_bin) : 0;
    const cplx* Hk = Hp + (long long)k * a.Dh;
    const int* gi = a.gidx ? a.gidx + (long long)prob * a.gidx_prob_stride : nullptr;
    if (k >= a.kls1) {  // with no LS bin before it the recursion starts from W = 0, i.e. phi = angle(0) = 0
      const cplx* Ak = a.At + slot * (long long)D * Mc;
      const bool nyq = a.nyquist_real && (k == K - 1);
      for (int d = tid; d < D; d += nt) {
        const cplx* row = Ak + (long long)d * Mc;
        cplx y = mk(0.0, 0.0);
        for (int c = 0; c < Mc; ++c) cfma(y, row[c], w[c]);
        const cplx hv = Hk[gi ? gi[d] : d];
        const double mag = sqrt(cabs2(hv));
        const double a2 = cabs2(y);
        cplx tv;
        if (a2 > 0.0) { const double inv = mag / sqrt(a2); tv = mk(y.x * inv, y.y * inv); }
        else tv = mk(mag, 0.0);   // angle(0) = 0
        if (nyq) tv.y = 0.0;
        t[d] = tv;
      }
    } else {
      for (int d = tid; d < D; d += nt) t[d] = Hk[gi ? gi[d] : d];
    }
    __syncthreads();
    const cplx* Qk = a.QcT + slot * (long long)Mc * D;
    for (int c = warp; c < Mc; c += nw) {
      const cplx* q = Qk + (long long)c * D;
      cplx acc = mk(0.0, 0.0);
      for (int d = lane; d < D; d += 32) cfmac(acc, q[d], t[d]);   // conj(q) * t
#pragma unroll
      for (int sh = 16; sh > 0; sh >>= 1) {
        acc.x += __shfl_xor_sync(0xffffffffu, acc.x, sh);
        acc.y += __shfl_xor_sync(0xffffffffu, acc.y, sh);
      }
      if (lane == 0) x[c] = acc;
    }
    __syncthreads();
    const cplx* Pk = a.Pb + slot * (long long)Mc * Mc;
    for (int m = tid; m < Mc; m += nt) {
      cplx acc = mk(0.0, 0.0);
      for (int c = 0; c < Mc; ++c) cfma(acc, x[c], Pk[c * Mc + m]);
      w[m] = acc;
      Wp[(long long)m * K + k] = acc;
      if (a.dc_fix && k == 1) Wp[(long long)m * K] = mk(acc.x, 0.0);  // lib/getEMagLs2Filters.m:109-110
    }
    __syncthreads();
  }
}

// Hc[k][d] = (Hd[d][2k], Hd[d][2k+1])
__global__ void spectrum_rows_kernel(const double* __restrict__ Hd, int D, int K, cplx* __restrict__ Hc) {
  __shared__ cplx tile[32][33];
  const int k0 = blockIdx.x * 32, d0 = blockIdx.y * 32, tx = threadIdx.x, ty = threadIdx.y;  // 32 x 8
  for (int r = ty; r < 32; r += 8) {
    const int d = d0 + r, k = k0 + tx;
    if (d < D && k < K) tile[r][tx] = mk(Hd[(long long)d * 2 * K + 2 * k], Hd[(long long)d * 2 * K + 2 * k + 1]);
  }
  __syncthreads();
  for (int r = ty; r < 32; r += 8) {
    const int k = k0 + r, d = d0 + tx;
    if (k < K && d < D) Hc[(long long)k * D + d] = tile[tx][r];
  }
}

// time-domain rows as complex targets: Hc[t][d] = h[t + T*d]   (getLsFilters: wLs = h * pinv(Y_conj))
__global__ void time_rows_kernel(const double* __restrict__ h, int T, int D, cplx* __restrict__ Hc) {
  long long idx = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (idx >= (long long)T * D) return;
  const int d = (int)(idx % D), t = (int)(idx / D);
  Hc[idx] = mk(h[(long long)d * T + t], 0.0);
}

// rows of conj(Y) as steering data: At[d][c] = Y[c][d]  (Y real, [S][D] with S >= Mc)
__global__ void sh_rows_kernel(const double* __restrict__ Y, int D, int Mc, cplx* __restrict__ At) {
  long long idx = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (idx >= (long long)D * Mc) return;
  const int c = (int)(idx % Mc), d = (int)(idx / Mc);
  At[idx] = mk(Y[(long long)c * D + d], 0.0);
}

// unit vectors as MATLAB's sph2cart(azi, pi/2 - zen, 1); grid is [n x 2] column-major (azi | zen)
__global__ void grid_cart_kernel(const double* __restrict__ grid, int n, double* __restrict__ xyz) {
  int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  const double azi = grid[i], elev = 1.5707963267948966 - grid[n + i];
  double se, ce, sa, ca;
  sincos(elev, &se, &ce);
  sincos(azi, &sa, &ca);
  xyz[3 * i] = ce * ca; xyz[3 * i + 1] = ce * sa; xyz[3 * i + 2] = se;
}

// nearest neighbour of every direction of the smaller grid in the larger one
// (lib/getEMagLsFiltersFromAtf.m:80-84: first minimum of the Euclidean distance)
// Batched over head orientations (blockIdx.y): the HRIR-grid direction u points to R u.  rot_small != 0: the
// smaller grid is the HRIR grid (x <- R x); else the larger one is, which is matched by x <- R^T x.
__global__ void nn_match_kernel(const double* __restrict__ small_xyz, int ns, const double* __restrict__ large_xyz,
                                int nl, const double* __restrict__ rot, int rot_small, int* __restrict__ idx,
                                double* __restrict__ dev_deg) {
  int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= ns) return;
  double x = small_xyz[3 * i], y = small_xyz[3 * i + 1], z = small_xyz[3 * i + 2];
  if (rot) {
    const double* R = rot + 9 * blockIdx.y;
    double rx, ry, rz;
    if (rot_small) { rx = R[0] * x + R[1] * y + R[2] * z; ry = R[3] * x + R[4] * y + R[5] * z; rz = R[6] * x + R[7] * y + R[8] * z; }
    else { rx = R[0] * x + R[3] * y + R[6] * z; ry = R[1] * x + R[4] * y + R[7] * z; rz = R[2] * x + R[5] * y + R[8] * z; }
    x = rx; y = ry; z = rz;
  }
  idx += (long long)blockIdx.y * ns;
  dev_deg += (long long)blockIdx.y * ns;
  double best = 1e300; int bi = 0;
  for (int j = 0; j < nl; ++j) {
    const double dx = large_xyz[3 * j] - x, dy = large_xyz[3 * j + 1] - y, dz = large_xyz[3 * j + 2] - z;
    const double dist = sqrt(dx * dx + dy * dy + dz * dz);
    if (dist < best) { best = dist; bi = j; }
  }
  idx[i] = bi;
  double dot = x * large_xyz[3 * bi] + y * large_xyz[3 * bi + 1] + z * large_xyz[3 * bi + 2];
  dot = fmin(1.0, fmax(-1.0, dot));
  dev_deg[i] = acos(dot) * 57.29577951308232;
}

// At[k-1][i][m] = atfs(k, m, src(i)) for k = 1..K-1, from Ad [(m + M*da)][2K]
__global__ void gather_atf_kernel(const double* __restrict__ Ad, int M, int K, int Dn, const int* __restrict__ src,
                                  cplx* __restrict__ At) {
  long long id = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (id >= (long long)(K - 1) * Dn * M) return;
  const int m = (int)(id % M), i = (int)((id / M) % Dn), k = 1 + (int)(id / ((long long)M * Dn));
  const int da = src ? src[i] : i;
  const double* p = Ad + ((long long)m + (long long)M * da) * 2 * K + 2 * k;
  At[id] = mk(p[0], p[1]);
}

// Hout[k][i] = Hin[k][src[i]]
__global__ void gather_cols_kernel(const cplx* __restrict__ Hin, int K, int Din, int Dn, const int* __restrict__ src,
                                   cplx* __restrict__ Hout) {
  long long id = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (id >= (long long)K * Dn) return;
  const int i = (int)(id % Dn), k = (int)(id / Dn);
  Hout[id] = Hin[(long long)k * Din + src[i]];
}

}  // namespace

// ------------------------------------------------------------------------------------------
// shared driver: factorise every operator, form Q_C, run the chain
// ------------------------------------------------------------------------------------------
struct GenericProblem {
  const cplx* At; int num_ops;  // rows [num_ops][D][Mc]; num_ops == 1: one operator for all bins
  int D, Mc, K;
  int first_bin, kls1, dc_fix, nyquist_real;
  double regul;
  const cplx* H; long long h_prob_stride, h_ear_stride;   // [prob][ear][K][D]
  int num_prob;
  cplx* W;  // [ear][prob][Mc][K]
  long long w_ear_stride = 0;                             // 0: num_prob * Mc * K
  int Dh = 0; const int* gidx = nullptr; long long gidx_prob_stride = 0;   // see ChainArgs
};

static void run_generic(emagls_ctx* h, Arena& ar, const GenericProblem& g) {
  cudaStream_t st = h->stream;
  EM_REQUIRE(g.D >= g.Mc, "fewer directions than channels");
  EM_REQUIRE(g.Mc <= 64, "more than 64 channels are not supported");
  const BlockPlan bp = make_block_plan(g.D, g.Mc);
  OperatorSet ops{};
  ops.v_stride = (long long)g.Mc * g.D; ops.tau_stride = (long long)bp.nblk * bp.MC;
  ops.pb_stride = (long long)g.Mc * g.Mc;
  ops.V = ar.get<cplx>((size_t)g.num_ops * ops.v_stride);
  ops.tau = ar.get<cplx>((size_t)g.num_ops * ops.tau_stride);
  ops.Pb = ar.get<cplx>((size_t)g.num_ops * ops.pb_stride);
  ops.info = ar.get<int>(g.num_ops);
  cplx* QcT = ar.get<cplx>((size_t)g.num_ops * g.Mc * g.D);
  {
    ProfSpan ps(h, EM_PROF_FACTOR);
    RowSource src{};
    src.At = g.At; src.at_bin_stride = (long long)g.D * g.Mc; src.at_prob_stride = 0;
    // one "problem", num_ops bin slots: operator index = slot
    EM_CUDA(launch_factor(st, bp, src, ops, 1, 0, g.num_ops, g.regul, 1));
    const size_t smem = (size_t)2 * g.D * sizeof(cplx);
    EM_CUDA(allow_dynamic_smem(form_q_kernel, smem));
    dim3 grid((g.Mc + 1) / 2, g.num_ops);
    form_q_kernel<<<grid, 32, smem, st>>>(bp, ops, QcT);
    EM_CUDA(cudaGetLastError());
    h->launches += 2;
  }
  {
    ProfSpan ps(h, EM_PROF_CHAIN_BWD);
    ChainArgs c;
    c.At = g.At; c.at_slot_stride = g.num_ops > 1 ? 1 : 0;
    c.QcT = QcT; c.Pb = ops.Pb;
    c.H = g.H; c.h_prob_stride = g.h_prob_stride; c.h_ear_stride = g.h_ear_stride;
    c.W = g.W; c.w_ear_stride = g.w_ear_stride ? g.w_ear_stride : (long long)g.num_prob * g.Mc * g.K;
    c.w_prob_stride = (long long)g.Mc * g.K;
    c.Dh = g.Dh ? g.Dh : g.D; c.gidx = g.gidx; c.gidx_prob_stride = g.gidx_prob_stride;
    c.D = g.D; c.Mc = g.Mc; c.K = g.K; c.first_bin = g.first_bin; c.kls1 = g.kls1; c.dc_fix = g.dc_fix;
    c.nyquist_real = g.nyquist_real;
    const size_t smem = ((size_t)g.D + 2 * g.Mc) * sizeof(cplx);
    EM_CUDA(allow_dynamic_smem(generic_chain_kernel, smem));
    generic_chain_kernel<<<g.num_prob * 2, 1024, smem, st>>>(c);
    EM_CUDA(cudaGetLastError());
    h->launches += 1;
  }
}

// Hc [set][ear][K][D]: HRIR spectra as complex rows (hrir_spectrum), (set, ear) advanced by delays[set * 2 + ear]
static cplx* hrir_spectra_rows(emagls_ctx* h, Arena& ar, const double* hL, const double* hR, int T, int D, int K,
                               int nfft, int num_sets, const std::vector<double>& delays) {
  cudaStream_t st = h->stream;
  cplx* Hc = ar.get<cplx>((size_t)num_sets * 2 * K * D);
  double* tw = ar.get<double>((size_t)2 * K * T);
  EM_CUDA(launch_dft_twiddle(st, K, T, nfft, tw));
  double* Hd = ar.get<double>((size_t)D * 2 * K);
  for (int s = 0; s < num_sets; ++s)
    for (int e = 0; e < 2; ++e) {
      hrir_spectrum(h, ar, (e ? hR : hL) + (size_t)s * T * D, T, D, K, tw, delays[(size_t)s * 2 + e], Hd);
      dim3 grid((K + 31) / 32, (D + 31) / 32), block(32, 8);
      spectrum_rows_kernel<<<grid, block, 0, st>>>(Hd, D, K, Hc + ((size_t)s * 2 + e) * K * D);
      EM_CUDA(cudaGetLastError());
      h->launches += 1;
    }
  h->launches += 1;
  return Hc;
}

// tail of the SH-domain designers without the sphere model: real tail GEMM (+ basis change)
static void tail_real(emagls_ctx* h, Arena& ar, const cplx* Wsp, int P, int Mc, int K, int nfft, int len,
                      double delayL, double delayR, double* wL, double* wR) {
  cudaStream_t st = h->stream;
  ProfSpan ps(h, EM_PROF_TAIL);
  double* twT = ar.get<double>((size_t)len * 2 * K);
  for (int e = 0; e < 2; ++e) {
    EM_CUDA(launch_tail_twiddle(st, K, nfft, len, e ? delayR : delayL, twT));
    const double* We = reinterpret_cast<const double*>(Wsp + (size_t)e * P * Mc * K);
    GemmOperand A{We, 2LL * K, 1}, B{twT, 2LL * K, 1};
    EM_CUDA(launch_gemm(st, A, B, GemmShape{P * Mc, len, 2 * K}, EpiStore{e ? wR : wL, len, 1.0}));
    h->launches += 2;
  }
}

// ------------------------------------------------------------------------------------------
// getMagLsFilters / getLsFilters
// ------------------------------------------------------------------------------------------
void design_magls(emagls_ctx* h, const emagls_config& cfg, const double* hL, const double* hR, int T, int D,
                  const double* grid_azi, const double* grid_zen, int order, double fs, int len, bool ls_only,
                  double* wL, double* wR, double* spectra, int harmonics_kind, int num_sets) {
  // harmonics_kind 0: spherical harmonics (getMagLsFilters / getLsFilters); 1: circular harmonics of the
  // azimuth only (lib/getMagLsFilters2D.m:44-45), channels ordered [0,-1,+1,...]
  cudaStream_t st = h->stream;
  EM_REQUIRE(T > 0 && D > 0 && num_sets >= 1, "empty input");
  EM_REQUIRE(num_sets == 1 || !ls_only, "getLsFilters takes one HRTF set");
  EM_REQUIRE(order >= 0 && order <= MAX_SH_ORDER, "order out of range");
  const int Mc = harmonics_kind == 1 ? 2 * order + 1 : (order + 1) * (order + 1);
  EM_REQUIRE(Mc <= 64, "more than 64 channels are not supported");
  EM_REQUIRE(D >= Mc, "fewer directions than harmonics");
  const bool cplx_out = cfg.basis == EMAGLS_BASIS_COMPLEX;
  Arena ar(st);
  std::optional<ProfSpan> setup_span(std::in_place, h, EM_PROF_SETUP);
  // Y_conj.' rows in the real basis; a complex basis is a unitary change of the output (engine.cu)
  cplx* At = ar.get<cplx>((size_t)D * Mc);
  if (harmonics_kind == 1) {
    EM_CUDA(launch_ch_rows(st, order, grid_azi, D, 0, At));
    h->launches += 1;
  } else {
    double* Y = ar.get<double>((size_t)Mc * D);
    EM_CUDA(launch_sh_angles(st, order, grid_azi, grid_zen, D, 0, Y));
    long long n = (long long)D * Mc;
    sh_rows_kernel<<<(unsigned)((n + 255) / 256), 256, 0, st>>>(Y, D, Mc, At);
    EM_CUDA(cudaGetLastError());
    h->launches += 2;
  }
  GenericProblem g{};
  g.At = At; g.num_ops = 1; g.D = D; g.Mc = Mc; g.regul = 0.0; g.num_prob = 1;
  if (ls_only) {
    // wLs = h * pinv(Y_conj): every time sample is an "LS bin" (lib/getLsFilters.m:30-34)
    cplx* Hc = ar.get<cplx>((size_t)2 * T * D);
    for (int e = 0; e < 2; ++e) {
      long long n = (long long)T * D;
      time_rows_kernel<<<(unsigned)((n + 255) / 256), 256, 0, st>>>(e ? hR : hL, T, D, Hc + (size_t)e * T * D);
      EM_CUDA(cudaGetLastError());
    }
    h->launches += 2;
    setup_span.reset();
    cplx* W = ar.get<cplx>((size_t)2 * Mc * T);
    g.K = T; g.first_bin = 0; g.kls1 = T; g.dc_fix = 0; g.nyquist_real = 0;
    g.H = Hc; g.h_prob_stride = 0; g.h_ear_stride = (long long)T * D; g.W = W;
    run_generic(h, ar, g);
    // W [ear][Mc][T] is the column-major [T x Mc] filter; its imaginary parts are exactly zero
    double* tmp = cplx_out ? ar.get<double>((size_t)Mc * T) : nullptr;
    for (int e = 0; e < 2; ++e) {
      double* out = e ? wR : wL;
      const cplx* We = W + (size_t)e * Mc * T;
      EM_CUDA(cudaMemcpy2DAsync(cplx_out ? tmp : out, sizeof(double), We, sizeof(cplx), sizeof(double),
                                (size_t)Mc * T, cudaMemcpyDeviceToDevice, st));
      if (cplx_out) {
        EM_CUDA(launch_basis_change_filters(st, tmp, harmonics_kind, Mc, T, 1, nullptr, 0, 1, reinterpret_cast<cplx*>(out)));
        h->launches += 1;
      }
    }
    return;
  }
  const BinGrid bg = bin_grid(cfg, len, fs, T);   // lib/getMagLsFilters.m:38
  const int nfft = bg.nfft, K = bg.K;
  const int kls1 = bg.kls1(std::max(cfg.f_cut_min, 500.0 * order));
  // HRTF-set batch (extension, not in the reference API): the one pinv(Y) operator serves every set, the sets are
  // independent problems of the chain kernel (lib/getMagLsFilters.m:48,64-72)
  const int NS = num_sets;
  const std::vector<double> grpD = group_delays(h, ar, hL, hR, T, D, K, fs, NS);
  cplx* Hc = hrir_spectra_rows(h, ar, hL, hR, T, D, K, nfft, NS, grpD);
  setup_span.reset();
  cplx* Wsp = spectra ? reinterpret_cast<cplx*>(spectra) : ar.get<cplx>((size_t)2 * NS * Mc * K);
  g.K = K; g.first_bin = 0; g.kls1 = kls1; g.dc_fix = 0; g.nyquist_real = 1;   // lib/getMagLsFilters.m:64-72
  g.num_prob = NS;
  g.H = Hc; g.h_prob_stride = 2LL * K * D; g.h_ear_stride = (long long)K * D; g.W = Wsp;
  run_generic(h, ar, g);
  // tail per set: the right ear's shift restores that set's inter-aural group-delay difference
  double* tmp = cplx_out ? ar.get<double>((size_t)2 * Mc * len) : nullptr;
  cplx* Wset = ar.get<cplx>((size_t)2 * Mc * K);
  for (int s_ = 0; s_ < NS; ++s_) {
    const double dl = (double)(nfft / 2), dr = dl + (grpD[(size_t)s_ * 2 + 1] - grpD[(size_t)s_ * 2]);
    const cplx* Ws = Wsp;
    if (NS > 1) {   // gather this set's two ear blocks [ear][set][Mc][K] -> [ear][Mc][K]
      for (int e = 0; e < 2; ++e)
        EM_CUDA(cudaMemcpyAsync(Wset + (size_t)e * Mc * K, Wsp + ((size_t)e * NS + s_) * Mc * K,
                                (size_t)Mc * K * sizeof(cplx), cudaMemcpyDeviceToDevice, st));
      Ws = Wset;
    }
    const size_t esz = (size_t)Mc * len * (cplx_out ? 2 : 1);
    double* oL = wL + (size_t)s_ * esz;
    double* oR = wR + (size_t)s_ * esz;
    if (!cplx_out) {
      tail_real(h, ar, Ws, 1, Mc, K, nfft, len, dl, dr, oL, oR);
    } else {
      tail_real(h, ar, Ws, 1, Mc, K, nfft, len, dl, dr, tmp, tmp + (size_t)Mc * len);
      EM_CUDA(launch_basis_change_filters(st, tmp, harmonics_kind, Mc, len, 1, nullptr, 0, 1, reinterpret_cast<cplx*>(oL)));
      EM_CUDA(launch_basis_change_filters(st, tmp + (size_t)Mc * len, harmonics_kind, Mc, len, 1, nullptr, 0, 1,
                                          reinterpret_cast<cplx*>(oR)));
      h->launches += 2;
    }
  }
  if (cplx_out && spectra) {
    EM_CUDA(launch_basis_change_spectra(st, Wsp, harmonics_kind, Mc, K, 2LL * NS, 0));
    h->launches += 1;
  }
}

// ------------------------------------------------------------------------------------------
// getEMagLsFiltersFromAtf (all pointers on the device)
// ------------------------------------------------------------------------------------------
static double matlab_round(double x) { return (x < 0.0) ? -std::floor(-x + 0.5) : std::floor(x + 0.5); }

void design_from_atf(emagls_ctx* h, const emagls_config& cfg, const double* hL, const double* hR, int T, int D,
                     const double* hrir_grid, const double* atf_irs, int Ta, int M, int Da, const double* atf_grid,
                     double fs, int len, double f_trans, int num_orient, const double* rotations, double* wL,
                     double* wR, double* spectra, double* mean_dev_deg) {
  // Batch extension (not in the reference API): orientation b sees HRIR-grid direction u at R_b u, i.e. page b of
  // the outputs equals one reference call with hrirGridAziZenRad rotated by R_b.  When the ATF grid is the smaller
  // one (BASELINE config 3: 1625 < 2702) pwGrid is the whole ATF set for every orientation
  // (lib/getEMagLsFiltersFromAtf.m:72-75): the per-bin factorisations are shared by the batch and only the
  // nearest-neighbour-selected HRTF columns (:82-95) differ, which the chain kernel gathers on the fly.
  cudaStream_t st = h->stream;
  EM_REQUIRE(T > 0 && D > 0 && Ta > 0 && M > 0 && Da > 0 && len > 0, "empty input");
  const BinGrid bg = bin_grid(cfg, len, fs, T);
  EM_REQUIRE(bg.nfft % 2 == 0, "nfft must be even");
  EM_REQUIRE(M <= 64, "more than 64 channels are not supported");
  EM_REQUIRE(num_orient >= 1 && (rotations != nullptr || num_orient == 1), "num_orient > 1 needs rotations");
  const int B = num_orient;
  const int nfft = bg.nfft, K = bg.K;
  const int kls1 = bg.kls1(f_trans);                        // lib/getEMagLsFiltersFromAtf.m:38
  const bool hrtf_smaller = D <= Da;                        // min() picks the first on a tie (:62)
  const int Dn = std::min(D, Da);
  EM_REQUIRE(Dn >= M, "fewer directions than microphones");
  Arena ar(st);
  std::optional<ProfSpan> setup_span(std::in_place, h, EM_PROF_SETUP);
  // ---- grid matching (:56-96), all orientations at once
  double* hx = ar.get<double>((size_t)3 * D);
  double* ax = ar.get<double>((size_t)3 * Da);
  grid_cart_kernel<<<(D + 127) / 128, 128, 0, st>>>(hrir_grid, D, hx);
  grid_cart_kernel<<<(Da + 127) / 128, 128, 0, st>>>(atf_grid, Da, ax);
  int* d_idx = ar.get<int>((size_t)B * Dn);
  double* d_dev = ar.get<double>((size_t)B * Dn);
  {
    dim3 grid((Dn + 63) / 64, B);
    nn_match_kernel<<<grid, 64, 0, st>>>(hrtf_smaller ? hx : ax, Dn, hrtf_smaller ? ax : hx, hrtf_smaller ? Da : D,
                                         rotations, hrtf_smaller ? 1 : 0, d_idx, d_dev);
  }
  EM_CUDA(cudaGetLastError());
  h->launches += 3;
  // ---- HRIRs: integer group-delay removal (:42-49), spectra
  const std::vector<double> grpD = group_delays(h, ar, hL, hR, T, D, K, fs, 1);
  cplx* Hfull = hrir_spectra_rows(h, ar, hL, hR, T, D, K, nfft, 1, {matlab_round(grpD[0]), matlab_round(grpD[1])});
  // ---- ATF spectra (:54)
  const int Tu = std::min(Ta, nfft);   // fft(x, nfft) truncates longer responses
  double* Ad = ar.get<double>((size_t)M * Da * 2 * K);
  {
    double* tw = ar.get<double>((size_t)2 * K * Tu);
    EM_CUDA(launch_dft_twiddle(st, K, Tu, nfft, tw));
    GemmOperand A{atf_irs, Ta, 1}, Bm{tw, Tu, 1};
    EM_CUDA(launch_gemm(st, A, Bm, GemmShape{M * Da, 2 * K, Tu}, EpiStore{Ad, 2LL * K, 1.0}));
    h->launches += 2;
  }
  if (mean_dev_deg) {
    std::vector<double> dev((size_t)B * Dn);
    EM_CUDA(cudaMemcpyAsync(dev.data(), d_dev, dev.size() * sizeof(double), cudaMemcpyDeviceToHost, st));
    EM_CUDA(cudaStreamSynchronize(st));
    for (int b = 0; b < B; ++b) {
      double acc = 0.0;
      for (int i = 0; i < Dn; ++i) acc += dev[(size_t)b * Dn + i];
      mean_dev_deg[b] = acc / (double)Dn;
    }
  }
  setup_span.reset();
  cplx* Wsp = spectra ? reinterpret_cast<cplx*>(spectra) : ar.get<cplx>((size_t)2 * B * M * K);
  EM_CUDA(cudaMemsetAsync(Wsp, 0, (size_t)2 * B * M * K * sizeof(cplx), st));
  GenericProblem g{};
  g.num_ops = K - 1; g.D = Dn; g.Mc = M; g.K = K; g.first_bin = 1; g.kls1 = kls1; g.dc_fix = 1;
  g.nyquist_real = 1; g.regul = cfg.svd_regul;
  g.H = Hfull; g.h_prob_stride = 0; g.h_ear_stride = (long long)K * D; g.Dh = D;
  g.w_ear_stride = (long long)B * M * K;
  const long long natf = (long long)(K - 1) * Dn * M;
  if (!hrtf_smaller) {
    // ATF grid smaller: one set of operators for the whole batch, HRTF columns gathered per orientation
    cplx* At = ar.get<cplx>((size_t)natf);
    gather_atf_kernel<<<(unsigned)((natf + 255) / 256), 256, 0, st>>>(Ad, M, K, Dn, nullptr, At);
    EM_CUDA(cudaGetLastError());
    h->launches += 1;
    g.At = At; g.num_prob = B; g.W = Wsp; g.gidx = d_idx; g.gidx_prob_stride = Dn;
    run_generic(h, ar, g);
  } else {
    // HRTF grid smaller: the matched ATF columns, hence the operators, differ per orientation
    for (int b = 0; b < B; ++b) {
      Arena ar_b(st);
      cplx* At = ar_b.get<cplx>((size_t)natf);
      gather_atf_kernel<<<(unsigned)((natf + 255) / 256), 256, 0, st>>>(Ad, M, K, Dn, d_idx + (size_t)b * Dn, At);
      EM_CUDA(cudaGetLastError());
      h->launches += 1;
      g.At = At; g.num_prob = 1; g.W = Wsp + (size_t)b * M * K; g.gidx = nullptr;
      run_generic(h, ar_b, g);
    }
  }
  // integer shift by nfft/2, no restoration of the inter-aural delay difference (:136-138)
  tail_real(h, ar, Wsp, B, M, K, nfft, len, (double)(nfft / 2), (double)(nfft / 2), wL, wR);
}

// ------------------------------------------------------------------------------------------
// getEMagLsFiltersEMAinSH (all pointers on the device)
// ------------------------------------------------------------------------------------------
void design_ema_sh(emagls_ctx* h, const emagls_config& cfg, const double* hL, const double* hR, int T, int D,
                   const double* grid_azi, const double* grid_zen, double mic_radius, const double* mic_azi, int M,
                   int order, double fs, int len, double* wL, double* wR, double* spectra) {
  cudaStream_t st = h->stream;
  EM_REQUIRE(T > 0 && D > 0 && M > 0 && len > 0, "empty input");
  const BinGrid bg = bin_grid(cfg, len, fs, T);
  EM_REQUIRE(bg.nfft % 2 == 0, "nfft must be even");
  const int nfft = bg.nfft, K = bg.K;
  const int kls1 = bg.kls1(std::max(cfg.f_cut_min, 500.0 * order));
  const int simN = sim_order(cfg, order, fs, mic_radius);
  EM_REQUIRE(simN <= MAX_SH_ORDER, "simulation order too high");
  const int S = (simN + 1) * (simN + 1), nsh = (order + 1) * (order + 1), nch = 2 * order + 1;
  EM_REQUIRE(nsh <= 64, "more than 64 channels are not supported");
  EM_REQUIRE(M >= nch, "fewer microphones than circular harmonics");
  EM_REQUIRE(D >= nsh, "fewer directions than harmonics");
  const bool cplx_out = cfg.basis == EMAGLS_BASIS_COMPLEX;
  Arena ar(st);
  std::optional<ProfSpan> setup_span(std::in_place, h, EM_PROF_SETUP);
  // ---- array model pieces
  const std::vector<double> kr = kr_table(cfg, fs, mic_radius, K);
  cplx* bn = ar.get<cplx>((size_t)K * (simN + 1));
  EM_CUDA(launch_modal(st, simN, ar.upload(kr.data(), K), K, cfg.array_type, -1.0, 1, bn, simN + 1, 1));
  const int nmax = std::max(std::max(M, D), 1);
  double* halfpi = ar.get<double>(nmax);
  EM_CUDA(launch_fill(st, halfpi, nmax, 1.5707963267948966));
  double* Ym = ar.get<double>((size_t)M * S);
  EM_CUDA(launch_sh_mics(st, simN, mic_azi, halfpi, M, nullptr, 1, Ym));
  double* Yhor = ar.get<double>((size_t)S * D);
  EM_CUDA(launch_sh_angles(st, simN, grid_azi, halfpi, D, 0, Yhor));        // directions mapped to the equator (:68)
  double* Ysh0 = ar.get<double>(nsh);
  {
    double* zero = ar.get<double>(1);
    EM_CUDA(cudaMemsetAsync(zero, 0, sizeof(double), st));
    EM_CUDA(launch_sh_angles(st, order, zero, halfpi, 1, 0, Ysh0));
  }
  // pinv(YCh.') through the factorisation kernel with the clip disabled
  cplx* Ach = ar.get<cplx>((size_t)M * nch);
  EM_CUDA(launch_ch_rows(st, order, mic_azi, M, cplx_out ? 1 : 0, Ach));
  cplx* pinvT = unclipped_pinv_dev(h, ar, Ach, M, nch);
  cplx* dec = ar.get<cplx>((size_t)M * nsh);
  EM_CUDA(launch_ema_dec(st, order, M, (M + 1) / 2, cplx_out ? 1 : 0, Ysh0, pinvT, dec));
  cplx* At = ar.get<cplx>((size_t)(K - 1) * D * nsh);
  EM_CUDA(launch_ema_sh_rows(st, order, simN, M, D, K, cplx_out ? 1 : 0, grid_azi, grid_zen, dec, Ym, Yhor, bn, At));
  h->launches += 8;
  // ---- HRIRs
  const std::vector<double> grpD = group_delays(h, ar, hL, hR, T, D, K, fs, 1);
  cplx* Hc = hrir_spectra_rows(h, ar, hL, hR, T, D, K, nfft, 1, grpD);
  setup_span.reset();
  cplx* Wsp = spectra ? reinterpret_cast<cplx*>(spectra) : ar.get<cplx>((size_t)2 * nsh * K);
  EM_CUDA(cudaMemsetAsync(Wsp, 0, (size_t)2 * nsh * K * sizeof(cplx), st));
  GenericProblem g{};
  g.At = At; g.num_ops = K - 1; g.D = D; g.Mc = nsh; g.K = K; g.first_bin = 1; g.kls1 = kls1; g.dc_fix = 1;
  g.nyquist_real = 1; g.regul = cfg.svd_regul; g.num_prob = 1;
  g.H = Hc; g.h_prob_stride = 0; g.h_ear_stride = (long long)K * D; g.W = Wsp;
  run_generic(h, ar, g);
  const double dl = (double)(nfft / 2), dr = dl + (grpD[1] - grpD[0]);
  if (!cplx_out) {
    tail_real(h, ar, Wsp, 1, nsh, K, nfft, len, dl, dr, wL, wR);
  } else {
    // computed literally in the complex basis: the reference's complex EMA-SH path is not a unitary
    // image of its real one, so the general complex tail is used
    cplx* X = ar.get<cplx>((size_t)4 * nsh * K);          // [X1 (2 ears) | X2 (2 ears)]
    EM_CUDA(launch_complex_tail_prep(st, Wsp, 0, nsh, K, 2, X, X + (size_t)2 * nsh * K));
    double* re = ar.get<double>((size_t)2 * nsh * len);
    double* im = ar.get<double>((size_t)2 * nsh * len);
    tail_real(h, ar, X, 1, nsh, K, nfft, len, dl, dr, re, re + (size_t)nsh * len);
    tail_real(h, ar, X + (size_t)2 * nsh * K, 1, nsh, K, nfft, len, dl, dr, im, im + (size_t)nsh * len);
    EM_CUDA(launch_interleave(st, re, im, (long long)nsh * len, reinterpret_cast<cplx*>(wL)));
    EM_CUDA(launch_interleave(st, re + (size_t)nsh * len, im + (size_t)nsh * len, (long long)nsh * len,
                              reinterpret_cast<cplx*>(wR)));
    h->launches += 3;
  }
}

}  // namespace emagls
