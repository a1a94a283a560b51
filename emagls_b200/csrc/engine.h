// Host-side engine state shared by the C-ABI translation units.
#pragma once
#include <cuda_runtime.h>
#include <string>
#include <utility>
#include <vector>
#include "../../include/emagls_cuda.h"
#include "kernels.h"

// kernel classes for the built-in event profiler (emagls_profile_*)
enum EmProfClass {
  EM_PROF_SETUP = 0,      // grid QR, SH, b_n, E rows, HRIR preparation
  EM_PROF_FACTOR,         // per-(orientation, bin) TSQR + clipped inverse
  EM_PROF_CHAIN_FWD,      // Q_C * R_C * W_prev
  EM_PROF_GEMM_FWD,       // y = c Q^T + phase epilogue
  EM_PROF_GEMM_BWD,       // t Q
  EM_PROF_CHAIN_BWD,      // (Q_C^H tq) Pb
  EM_PROF_TAIL,           // ifft/shift/crop/fade GEMM
  EM_PROF_RENDER_MAC,     // spectral multiply-accumulate of the render
  EM_PROF_RENDER_FFT,     // cuFFT transforms of the render
  EM_PROF_RENDER_STAGE,   // staging copies of the render
  EM_PROF_GRAM,           // Gram route: F blocks, DMMA assembly of G_k, warp-per-matrix Cholesky
  EM_PROF_JACOBI,         // clipped inverse of R_C (one-sided Jacobi), register-resident path
  EM_PROF_NUM
};

struct emagls_ctx {
  int device = 0;
  cudaStream_t stream = nullptr;
  cudaMemPool_t pool = nullptr;   // private stream-ordered pool of this handle (scratch stays cached between calls)
  std::string err;
  long long launches = 0;
  // work statistics of the design path (emagls_stats_read): (problem, bin) pairs on the TSQR + Jacobi route and
  // on the Gram route; the Jacobi kernel adds {sweeps, problems} to the device counters d_stats[0..1]
  long long stat_tsqr = 0, stat_gram = 0;
  unsigned long long* d_stats = nullptr;
  // profiler
  bool profile = false;
  std::vector<cudaEvent_t> ev_pool;
  size_t ev_used = 0;
  struct Span { int cls; cudaEvent_t a, b; };
  std::vector<Span> spans;
  double prof_ms[EM_PROF_NUM] = {0};
  long long prof_n[EM_PROF_NUM] = {0};
  // render: cuFFT plans are expensive to build (milliseconds), so they live with the handle
  struct RenderPlans {
    int N = 0, L = 0, num_ch = 0, nbc = 0, filt_batch = 0, inv_batch = 0;
    int fwd = 0, inv = 0, filt = 0;   // cufftHandle values (0 = not created)
    int edge = 0;                     // one boundary block of every channel (zero-padded staging)
    std::vector<std::pair<int, int>> direct;  // (batch, plan): interior blocks read straight from the input
  } render_plans;
  RenderPlans tracked_plans;          // head-tracked render (tracked_render.cu), kept apart from the static render's
  // per-channel FIR of the front end (frontend.cu): cuFFT plans keyed by (size, batch, direction)
  struct FirPlan { int N, batch, inverse, plan; };
  std::vector<FirPlan> fir_plans;
};

namespace emagls {

struct Fail {
  int code; std::string msg;
};

#define EM_CUDA(expr)                                                                          \
  do {                                                                                         \
    cudaError_t _e = (expr);                                                                   \
    if (_e != cudaSuccess)                                                                     \
      throw ::emagls::Fail{EMAGLS_ERR_CUDA, std::string(#expr) + ": " + cudaGetErrorString(_e)}; \
  } while (0)

#define EM_REQUIRE(cond, msg)                                                   \
  do {                                                                          \
    if (!(cond)) throw ::emagls::Fail{EMAGLS_ERR_INVALID, std::string(msg)};    \
  } while (0)

// Handles register their private memory pool under their stream, so that every Arena built on that stream draws
// from it (api.cu); a stream without an entry uses the device's default pool.
void register_stream_pool(cudaStream_t st, cudaMemPool_t pool);
void unregister_stream_pool(cudaStream_t st);
cudaMemPool_t pool_of_stream(cudaStream_t st);

// Stream-ordered scratch arena: everything allocated through it is released when it dies.
class Arena {
 public:
  explicit Arena(cudaStream_t st) : st_(st), pool_(pool_of_stream(st)) {}
  ~Arena() {
    for (void* p : ptrs_) cudaFreeAsync(p, st_);
  }
  template <class T>
  T* get(size_t n) {
    void* p = nullptr;
    if (n == 0) n = 1;
    cudaError_t e = pool_ ? cudaMallocFromPoolAsync(&p, n * sizeof(T), pool_, st_) : cudaMallocAsync(&p, n * sizeof(T), st_);
    if (e != cudaSuccess)
      throw Fail{EMAGLS_ERR_CUDA, std::string("cudaMallocAsync(") + std::to_string(n * sizeof(T)) + " B): " +
                                      cudaGetErrorString(e)};
    ptrs_.push_back(p);
    return static_cast<T*>(p);
  }
  template <class T>
  T* upload(const T* host, size_t n) {
    T* d = get<T>(n);
    cudaError_t e = cudaMemcpyAsync(d, host, n * sizeof(T), cudaMemcpyHostToDevice, st_);
    if (e != cudaSuccess) throw Fail{EMAGLS_ERR_CUDA, std::string("H2D: ") + cudaGetErrorString(e)};
    return d;
  }

 private:
  cudaStream_t st_;
  cudaMemPool_t pool_;
  std::vector<void*> ptrs_;
};

template <class F>
int guarded(emagls_ctx* h, F&& f) {
  if (!h) return EMAGLS_ERR_INVALID;
  try {
    cudaError_t e = cudaSetDevice(h->device);
    if (e != cudaSuccess) throw Fail{EMAGLS_ERR_CUDA, std::string("cudaSetDevice: ") + cudaGetErrorString(e)};
    f();
    return EMAGLS_OK;
  } catch (const Fail& x) {
    h->err = x.msg;
    cudaGetLastError();
    return x.code;
  } catch (const std::exception& x) {
    h->err = x.what();
    return EMAGLS_ERR_INVALID;
  }
}

// RAII span: records a CUDA-event pair around the launches issued while it is alive.
class ProfSpan {
 public:
  ProfSpan(emagls_ctx* h, int cls) : h_(h), cls_(cls) {
    if (!h_->profile) return;
    a_ = next();
    cudaEventRecord(a_, h_->stream);
  }
  ~ProfSpan() {
    if (!h_->profile) return;
    cudaEvent_t b = next();
    cudaEventRecord(b, h_->stream);
    h_->spans.push_back({cls_, a_, b});
  }

 private:
  cudaEvent_t next() {
    if (h_->ev_used == h_->ev_pool.size()) {
      cudaEvent_t e;
      cudaEventCreate(&e);
      h_->ev_pool.push_back(e);
    }
    return h_->ev_pool[h_->ev_used++];
  }
  emagls_ctx* h_;
  int cls_;
  cudaEvent_t a_ = nullptr;
};

// ---- design engine (engine.cu) ---------------------------------------------------------------
enum class Variant { EMAGLS2, EMAGLS_SH, EMA_CH };

struct DesignArgs {
  Variant variant;
  const double *hL, *hR;  // device [T x D x sets]
  int T, D;
  const double *grid_azi, *grid_zen;  // device [D]
  double mic_radius;
  const double *mic_azi, *mic_zen;  // device [M]; mic_zen == nullptr: equatorial array (zenith pi/2)
  int M, order;
  double fs;
  int len, num_sets, num_orient;
  const double* rotations;  // device [B x 9] or nullptr
  double *wL, *wR;          // device [len x Mc x P]
  double* spectra;          // device or nullptr: complex [K x Mc x P x 2]
  // host-evaluated bases of a custom shFunction (SURVEY.md H8), device pointers or nullptr:
  // Y_hrir [S][D] (= MATLAB [D x S] column-major) replaces getSH(simN, grid); Y_mic [num_orient][M][S]
  // replaces getSH(simN, rotated microphones).  grid_* / mic_* / rotations are then not read.
  const double* Y_hrir = nullptr;
  const double* Y_mic = nullptr;
};
void design_factored(emagls_ctx* h, const emagls_config& cfg, const DesignArgs& a);
void destroy_render_plans(emagls_ctx* h);  // render.cu (static and head-tracked render)
void destroy_fir_plans(emagls_ctx* h);     // frontend.cu
// radFilts [K][(order+1)] (row index k) on the device (getRadialFilter.m:42-70)
void radial_filter_dev(emagls_ctx* h, Arena& ar, const emagls_config& cfg, const emagls_radial_params& rp, int order,
                       double fs, double radius, int nfft, int nan_to_zero, cplx* out);
// real-basis -> complex-basis outputs (kind 0: SH in ACN order, 1: CH ordered [0,-1,+1,...]); see engine.cu
cudaError_t launch_basis_change_filters(cudaStream_t st, const double* wr, int kind, int nch, int len,
                                        long long P, const cplx* Wsp_e, int K, int nfft, cplx* out);
cudaError_t launch_basis_change_spectra(cudaStream_t st, cplx* Wsp, int kind, int nch, int K, long long EP,
                                        int dc_quirk);
void design_magls(emagls_ctx* h, const emagls_config& cfg, const double* hL, const double* hR, int T, int D,
                  const double* grid_azi, const double* grid_zen, int order, double fs, int len, bool ls_only,
                  double* wL, double* wR, double* spectra, int harmonics_kind = 0, int num_sets = 1);
void design_from_atf(emagls_ctx* h, const emagls_config& cfg, const double* hL, const double* hR, int T, int D,
                     const double* hrir_grid, const double* atf_irs, int Ta, int M, int Da, const double* atf_grid,
                     double fs, int len, double f_trans, int num_orient, const double* rotations, double* wL,
                     double* wR, double* spectra, double* mean_dev_deg);
void design_ema_sh(emagls_ctx* h, const emagls_config& cfg, const double* hL, const double* hR, int T, int D,
                   const double* grid_azi, const double* grid_zen, double mic_radius, const double* mic_azi, int M,
                   int order, double fs, int len, double* wL, double* wR, double* spectra);
std::vector<double> group_delays(emagls_ctx* h, Arena& ar, const double* hL, const double* hR, int T, int D,
                                 int K, double fs, int num_sets);
void hrir_spectrum(emagls_ctx* h, Arena& ar, const double* hp, int T, int D, int K, const double* tw,
                   double delay_removed, double* Hd);
// targets * Y_reg_inv for one steering matrix given as rows At [D][Mc]; rows [(pair*2+ear)*2+{re,im}][D],
// W [ear][pair][Mc]
void regularized_apply_dev(emagls_ctx* h, Arena& ar, const cplx* At, int D, int Mc, const double* rows,
                           int npair, double regul, cplx* W);

}  // namespace emagls
