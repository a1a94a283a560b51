// C ABI of libemagls_cuda (see include/emagls_cuda.h).
#include <algorithm>
#include <cmath>
#include <cstring>
#include <map>
#include <mutex>
#include <vector>
#include "engine.h"
#include "special.cuh"

using namespace emagls;

namespace emagls {
namespace {
std::mutex g_pool_mu;
std::map<cudaStream_t, cudaMemPool_t> g_pools;
}  // namespace
void register_stream_pool(cudaStream_t st, cudaMemPool_t pool) { std::lock_guard<std::mutex> l(g_pool_mu); g_pools[st] = pool; }
void unregister_stream_pool(cudaStream_t st) { std::lock_guard<std::mutex> l(g_pool_mu); g_pools.erase(st); }
cudaMemPool_t pool_of_stream(cudaStream_t st) {
  std::lock_guard<std::mutex> l(g_pool_mu);
  auto it = g_pools.find(st);
  return it == g_pools.end() ? nullptr : it->second;
}
}  // namespace emagls

extern "C" {

int emagls_create(int device, emagls_handle* out) {
  if (!out) return EMAGLS_ERR_INVALID;
  *out = nullptr;
  int n = 0;
  if (cudaGetDeviceCount(&n) != cudaSuccess || device < 0 || device >= n) return EMAGLS_ERR_CUDA;
  if (cudaSetDevice(device) != cudaSuccess) return EMAGLS_ERR_CUDA;
  emagls_ctx* h = new emagls_ctx();
  h->device = device;
  if (cudaStreamCreateWithFlags(&h->stream, cudaStreamNonBlocking) != cudaSuccess) {
    delete h;
    return EMAGLS_ERR_CUDA;
  }
  // A private stream-ordered pool keeps freed scratch cached between calls without touching the device's default
  // pool (which other users of the process share); it is destroyed, and its memory returned, with the handle.
  {
    cudaMemPoolProps props{};
    props.allocType = cudaMemAllocationTypePinned;
    props.handleTypes = cudaMemHandleTypeNone;
    props.location.type = cudaMemLocationTypeDevice;
    props.location.id = device;
    if (cudaMemPoolCreate(&h->pool, &props) == cudaSuccess) {
      unsigned long long thr = ~0ull;
      cudaMemPoolSetAttribute(h->pool, cudaMemPoolAttrReleaseThreshold, &thr);
      register_stream_pool(h->stream, h->pool);
    } else {
      h->pool = nullptr;   // fall back to the default pool with its default release threshold
      cudaGetLastError();
    }
  }
  if (cudaMalloc(&h->d_stats, 4 * sizeof(unsigned long long)) != cudaSuccess ||
      cudaMemset(h->d_stats, 0, 4 * sizeof(unsigned long long)) != cudaSuccess) {
    unregister_stream_pool(h->stream);
    cudaStreamDestroy(h->stream);
    if (h->pool) cudaMemPoolDestroy(h->pool);
    delete h;
    return EMAGLS_ERR_CUDA;
  }
  *out = h;
  return EMAGLS_OK;
}

int emagls_stats_read(emagls_handle h, long long* out, int reset) {
  if (!h || !out) return EMAGLS_ERR_INVALID;
  return guarded(h, [&] {
    unsigned long long d[4] = {0, 0, 0, 0};
    EM_CUDA(cudaStreamSynchronize(h->stream));
    EM_CUDA(cudaMemcpy(d, h->d_stats, sizeof(d), cudaMemcpyDeviceToHost));
    out[0] = h->stat_tsqr; out[1] = h->stat_gram; out[2] = (long long)d[1]; out[3] = (long long)d[0];
    if (reset) {
      h->stat_tsqr = h->stat_gram = 0;
      EM_CUDA(cudaMemset(h->d_stats, 0, sizeof(d)));
    }
  });
}

int emagls_destroy(emagls_handle h) {
  if (!h) return EMAGLS_ERR_INVALID;
  cudaSetDevice(h->device);
  cudaStreamSynchronize(h->stream);
  for (cudaEvent_t e : h->ev_pool) cudaEventDestroy(e);
  emagls::destroy_render_streams(h);
  emagls::destroy_render_plans(h);
  emagls::destroy_fir_plans(h);
  unregister_stream_pool(h->stream);
  cudaStreamDestroy(h->stream);
  if (h->pool) cudaMemPoolDestroy(h->pool);
  cudaFree(h->d_stats);
  delete h;
  return EMAGLS_OK;
}

const char* emagls_last_error(emagls_handle h) { return h ? h->err.c_str() : "null handle"; }

void emagls_config_default(emagls_config* cfg) {
  if (!cfg) return;
  std::memset(cfg, 0, sizeof(*cfg));
  cfg->nfft_max_len = 2048;    // lib/getEMagLs2Filters.m:35
  cfg->f_cut_min = 1e3;        // :36
  cfg->svd_regul = 0.01;       // :39
  cfg->speed_of_sound = 343.0; // getSMAIRMatrix.m:86
  cfg->array_type = EMAGLS_ARRAY_RIGID;
  cfg->basis = EMAGLS_BASIS_REAL;
}

long long emagls_launch_count(emagls_handle h) { return h ? h->launches : 0; }

int emagls_profile_enable(emagls_handle h, int on) {
  if (!h) return EMAGLS_ERR_INVALID;
  h->profile = on != 0;
  return EMAGLS_OK;
}

static void profile_collect(emagls_ctx* h) {
  if (h->spans.empty()) return;
  cudaSetDevice(h->device);
  cudaStreamSynchronize(h->stream);
  for (auto& s : h->spans) {
    float ms = 0.f;
    if (cudaEventElapsedTime(&ms, s.a, s.b) == cudaSuccess) {
      h->prof_ms[s.cls] += ms;
      h->prof_n[s.cls] += 1;
    }
  }
  h->spans.clear();
  h->ev_used = 0;
}

int emagls_profile_read(emagls_handle h, double* ms, long long* counts, int reset) {
  if (!h || !ms || !counts) return EMAGLS_ERR_INVALID;
  profile_collect(h);
  for (int i = 0; i < EM_PROF_NUM; ++i) { ms[i] = h->prof_ms[i]; counts[i] = h->prof_n[i]; }
  if (reset)
    for (int i = 0; i < EM_PROF_NUM; ++i) { h->prof_ms[i] = 0; h->prof_n[i] = 0; }
  return EM_PROF_NUM;
}
void* emagls_stream(emagls_handle h) { return h ? (void*)h->stream : nullptr; }

// ------------------------------------------------------------------------------------------
static void fill_args(DesignArgs& a, Variant v, const double* hL, const double* hR, int T, int D,
                      const double* ga, const double* gz, double r, const double* ma, const double* mz,
                      int M, int order, double fs, int len, int ns, int no, const double* rot,
                      double* wL, double* wR, double* sp) {
  a.variant = v; a.hL = hL; a.hR = hR; a.T = T; a.D = D; a.grid_azi = ga; a.grid_zen = gz;
  a.mic_radius = r; a.mic_azi = ma; a.mic_zen = mz; a.M = M; a.order = order; a.fs = fs; a.len = len;
  a.num_sets = ns; a.num_orient = no; a.rotations = rot; a.wL = wL; a.wR = wR; a.spectra = sp;
}

// Device outputs of a design called with host memory: both ears' filters and, when asked for, the spectra.
struct DeviceOutputs {
  DesignShape s;
  double *wL, *wR, *sp;
  DeviceOutputs(Arena& ar, const DesignShape& shape, bool spectra)
      : s(shape), wL(ar.get<double>(s.filter_elems)), wR(ar.get<double>(s.filter_elems)),
        sp(spectra ? ar.get<double>(s.spectra_elems) : nullptr) {}
  // copies the outputs to the host and waits for them
  void download(cudaStream_t st, double* hwL, double* hwR, double* hsp) const {
    EM_CUDA(cudaMemcpyAsync(hwL, wL, s.filter_elems * sizeof(double), cudaMemcpyDeviceToHost, st));
    EM_CUDA(cudaMemcpyAsync(hwR, wR, s.filter_elems * sizeof(double), cudaMemcpyDeviceToHost, st));
    if (hsp) EM_CUDA(cudaMemcpyAsync(hsp, sp, s.spectra_elems * sizeof(double), cudaMemcpyDeviceToHost, st));
    EM_CUDA(cudaStreamSynchronize(st));
  }
};

static int design_host(emagls_handle h, const emagls_config* cfg, Variant v, const double* hL,
                       const double* hR, int T, int D, const double* ga, const double* gz, double r,
                       const double* ma, const double* mz, int M, int order, double fs, int len,
                       int ns, int no, const double* rot, double* wL, double* wR, double* sp) {
  return guarded(h, [&] {
    EM_REQUIRE(cfg && hL && hR && ga && gz && ma && (mz || v == Variant::EMA_CH) && wL && wR, "null argument");
    EM_REQUIRE(T > 0 && D > 0 && M > 0 && ns > 0 && no > 0 && len > 0, "empty input");
    cudaStream_t st = h->stream;
    Arena ar(st);
    const DesignShape shape = design_shape(*cfg, v, M, order, len, bin_grid(*cfg, len, fs, T).K, (size_t)ns * no);
    DeviceOutputs out(ar, shape, sp != nullptr);
    DesignArgs a;
    fill_args(a, v, ar.upload(hL, (size_t)T * D * ns), ar.upload(hR, (size_t)T * D * ns), T, D,
              ar.upload(ga, D), ar.upload(gz, D), r, ar.upload(ma, M), mz ? ar.upload(mz, M) : nullptr, M, order, fs, len,
              ns, no, rot ? ar.upload(rot, (size_t)no * 9) : nullptr, out.wL, out.wR, out.sp);
    design_factored(h, *cfg, a);
    out.download(st, wL, wR, sp);
  });
}

int emagls_design_emagls2(emagls_handle h, const emagls_config* cfg, const double* hL, const double* hR,
                          int num_samples, int num_dirs, const double* grid_azi, const double* grid_zen,
                          double mic_radius, const double* mic_azi, const double* mic_zen, int num_mics,
                          int order, double fs, int len, int num_sets, int num_orient,
                          const double* rotations, double* wL, double* wR, double* spectra) {
  return design_host(h, cfg, Variant::EMAGLS2, hL, hR, num_samples, num_dirs, grid_azi, grid_zen, mic_radius,
                     mic_azi, mic_zen, num_mics, order, fs, len, num_sets, num_orient, rotations, wL, wR, spectra);
}

int emagls_design_emagls2_dev(emagls_handle h, const emagls_config* cfg, const double* hL, const double* hR,
                              int num_samples, int num_dirs, const double* grid_azi, const double* grid_zen,
                              double mic_radius, const double* mic_azi, const double* mic_zen, int num_mics,
                              int order, double fs, int len, int num_sets, int num_orient,
                              const double* rotations, double* wL, double* wR, double* spectra) {
  return guarded(h, [&] {
    EM_REQUIRE(cfg && hL && hR && grid_azi && grid_zen && mic_azi && mic_zen && wL && wR, "null argument");
    DesignArgs a;
    fill_args(a, Variant::EMAGLS2, hL, hR, num_samples, num_dirs, grid_azi, grid_zen, mic_radius, mic_azi,
              mic_zen, num_mics, order, fs, len, num_sets, num_orient, rotations, wL, wR, spectra);
    design_factored(h, *cfg, a);
  });
}

// Custom shFunction (SURVEY.md H8): the host evaluates the handle, the bases come down as matrices.
int emagls_design_sma_basis(emagls_handle h, const emagls_config* cfg, int sh_domain, const double* hL, const double* hR,
                            int num_samples, int num_dirs, const double* Y_hrir, int num_harmonics, double mic_radius,
                            const double* Y_mic, int num_mics, int order, double fs, int len, int num_sets,
                            int num_orient, double* wL, double* wR, double* spectra) {
  return guarded(h, [&] {
    EM_REQUIRE(cfg && hL && hR && Y_hrir && Y_mic && wL && wR, "null argument");
    const int T = num_samples, D = num_dirs, M = num_mics, S = num_harmonics, ns = num_sets, no = num_orient;
    EM_REQUIRE(T > 0 && D > 0 && M > 0 && ns > 0 && no > 0 && len > 0 && S > 0, "empty input");
    const int simN = sim_order(*cfg, order, fs, mic_radius);
    EM_REQUIRE(S == (simN + 1) * (simN + 1),
               "custom bases must be evaluated at the simulation order max(order, ceil(fs pi r / c)) (getSMAIRMatrix.m:95)");
    EM_REQUIRE(cfg->basis == EMAGLS_BASIS_REAL || sh_domain == 0, "complex SH-domain output needs the default getSH");
    const Variant v = sh_domain ? Variant::EMAGLS_SH : Variant::EMAGLS2;
    cudaStream_t st = h->stream;
    Arena ar(st);
    const DesignShape shape = design_shape(*cfg, v, M, order, len, bin_grid(*cfg, len, fs, T).K, (size_t)ns * no);
    DeviceOutputs out(ar, shape, spectra != nullptr);
    // MATLAB [M x S] column-major per orientation -> [orientation][M][S] (S contiguous)
    std::vector<double> ymt((size_t)no * M * S);
    for (int o = 0; o < no; ++o)
      for (int m = 0; m < M; ++m)
        for (int s_ = 0; s_ < S; ++s_) ymt[((size_t)o * M + m) * S + s_] = Y_mic[((size_t)o * S + s_) * M + m];
    DesignArgs a;
    fill_args(a, v, ar.upload(hL, (size_t)T * D * ns), ar.upload(hR, (size_t)T * D * ns), T, D, nullptr, nullptr,
              mic_radius, nullptr, nullptr, M, order, fs, len, ns, no, nullptr, out.wL, out.wR, out.sp);
    a.Y_hrir = ar.upload(Y_hrir, (size_t)S * D);
    a.Y_mic = ar.upload(ymt.data(), ymt.size());
    EM_CUDA(cudaStreamSynchronize(st));   // ymt is a temporary
    design_factored(h, *cfg, a);
    out.download(st, wL, wR, spectra);
  });
}

int emagls_design_emagls(emagls_handle h, const emagls_config* cfg, const double* hL, const double* hR,
                         int num_samples, int num_dirs, const double* grid_azi, const double* grid_zen,
                         double mic_radius, const double* mic_azi, const double* mic_zen, int num_mics,
                         int order, double fs, int len, int num_sets, int num_orient,
                         const double* rotations, double* wL, double* wR, double* spectra) {
  return design_host(h, cfg, Variant::EMAGLS_SH, hL, hR, num_samples, num_dirs, grid_azi, grid_zen, mic_radius,
                     mic_azi, mic_zen, num_mics, order, fs, len, num_sets, num_orient, rotations, wL, wR, spectra);
}


static int magls_host(emagls_handle h, const emagls_config* cfg, const double* hL, const double* hR,
                      int num_samples, int num_dirs, const double* grid_azi, const double* grid_zen, int order,
                      double fs, int len, int num_sets, double* wL, double* wR, double* spectra) {
  return guarded(h, [&] {
    EM_REQUIRE(cfg && hL && hR && grid_azi && grid_zen && wL && wR, "null argument");
    EM_REQUIRE(num_samples > 0 && num_dirs > 0 && len > 0 && order >= 0 && num_sets > 0, "empty input");
    cudaStream_t st = h->stream;
    Arena ar(st);
    const int T = num_samples, D = num_dirs, NS = num_sets;
    const DesignShape shape = design_shape(*cfg, Variant::EMAGLS_SH, 0, order, len, bin_grid(*cfg, len, fs, T).K, NS);
    DeviceOutputs out(ar, shape, spectra != nullptr);
    design_magls(h, *cfg, ar.upload(hL, (size_t)T * D * NS), ar.upload(hR, (size_t)T * D * NS), T, D,
                 ar.upload(grid_azi, D), ar.upload(grid_zen, D), order, fs, len, false, out.wL, out.wR, out.sp, 0, NS);
    out.download(st, wL, wR, spectra);
  });
}
int emagls_design_magls(emagls_handle h, const emagls_config* cfg, const double* hL, const double* hR,
                        int num_samples, int num_dirs, const double* grid_azi, const double* grid_zen, int order,
                        double fs, int len, double* wL, double* wR, double* spectra) {
  return magls_host(h, cfg, hL, hR, num_samples, num_dirs, grid_azi, grid_zen, order, fs, len, 1, wL, wR, spectra);
}
int emagls_design_magls_batch(emagls_handle h, const emagls_config* cfg, const double* hL, const double* hR,
                              int num_samples, int num_dirs, const double* grid_azi, const double* grid_zen, int order,
                              double fs, int len, int num_sets, double* wL, double* wR, double* spectra) {
  return magls_host(h, cfg, hL, hR, num_samples, num_dirs, grid_azi, grid_zen, order, fs, len, num_sets, wL, wR, spectra);
}

int emagls_design_ls(emagls_handle h, const emagls_config* cfg, const double* hL, const double* hR,
                     int num_samples, int num_dirs, const double* grid_azi, const double* grid_zen, int order,
                     double* wL, double* wR) {
  return guarded(h, [&] {
    EM_REQUIRE(cfg && hL && hR && grid_azi && grid_zen && wL && wR, "null argument");
    EM_REQUIRE(num_samples > 0 && num_dirs > 0 && order >= 0, "empty input");
    cudaStream_t st = h->stream;
    Arena ar(st);
    const int T = num_samples, D = num_dirs;
    DeviceOutputs out(ar, design_shape(*cfg, Variant::EMAGLS_SH, 0, order, T, 0, 1), false);   // T taps, no spectra
    design_magls(h, *cfg, ar.upload(hL, (size_t)T * D), ar.upload(hR, (size_t)T * D), T, D, ar.upload(grid_azi, D),
                 ar.upload(grid_zen, D), order, 0.0, 0, true, out.wL, out.wR, nullptr);
    out.download(st, wL, wR, nullptr);
  });
}
static int from_atf_host(emagls_handle h, const emagls_config* cfg, const double* hL, const double* hR,
                         int num_samples, int num_dirs, const double* hrir_grid, const double* atf_irs,
                         int atf_samples, int num_mics, int atf_dirs, const double* atf_grid, double fs,
                         int filter_len, double f_trans, int num_orient, const double* rotations, double* wL,
                         double* wR, double* spectra, double* mean_grid_dev_deg) {
  return guarded(h, [&] {
    EM_REQUIRE(cfg && hL && hR && hrir_grid && atf_irs && atf_grid && wL && wR, "null argument");
    EM_REQUIRE(num_samples > 0 && num_dirs > 0 && atf_samples > 0 && num_mics > 0 && atf_dirs > 0 && filter_len > 0 &&
                   num_orient > 0, "empty input");
    cudaStream_t st = h->stream;
    Arena ar(st);
    const int T = num_samples, D = num_dirs, M = num_mics, B = num_orient;
    // one real channel per microphone, as the EMAGLS2 variant
    const DesignShape shape = design_shape(*cfg, Variant::EMAGLS2, M, 0, filter_len, bin_grid(*cfg, filter_len, fs, T).K, B);
    DeviceOutputs out(ar, shape, spectra != nullptr);
    design_from_atf(h, *cfg, ar.upload(hL, (size_t)T * D), ar.upload(hR, (size_t)T * D), T, D,
                    ar.upload(hrir_grid, (size_t)2 * D), ar.upload(atf_irs, (size_t)atf_samples * M * atf_dirs),
                    atf_samples, M, atf_dirs, ar.upload(atf_grid, (size_t)2 * atf_dirs), fs, filter_len, f_trans, B,
                    rotations ? ar.upload(rotations, (size_t)B * 9) : nullptr, out.wL, out.wR, out.sp, mean_grid_dev_deg);
    out.download(st, wL, wR, spectra);
  });
}
int emagls_design_from_atf(emagls_handle h, const emagls_config* cfg, const double* hL, const double* hR,
                           int num_samples, int num_dirs, const double* hrir_grid, const double* atf_irs,
                           int atf_samples, int num_mics, int atf_dirs, const double* atf_grid, double fs,
                           int filter_len, double f_trans, double* wL, double* wR, double* spectra,
                           double* mean_grid_dev_deg) {
  return from_atf_host(h, cfg, hL, hR, num_samples, num_dirs, hrir_grid, atf_irs, atf_samples, num_mics, atf_dirs,
                       atf_grid, fs, filter_len, f_trans, 1, nullptr, wL, wR, spectra, mean_grid_dev_deg);
}
int emagls_design_from_atf_batch(emagls_handle h, const emagls_config* cfg, const double* hL, const double* hR,
                                 int num_samples, int num_dirs, const double* hrir_grid, const double* atf_irs,
                                 int atf_samples, int num_mics, int atf_dirs, const double* atf_grid, double fs,
                                 int filter_len, double f_trans, int num_orient, const double* rotations, double* wL,
                                 double* wR, double* spectra, double* mean_grid_dev_deg) {
  return from_atf_host(h, cfg, hL, hR, num_samples, num_dirs, hrir_grid, atf_irs, atf_samples, num_mics, atf_dirs,
                       atf_grid, fs, filter_len, f_trans, num_orient, rotations, wL, wR, spectra, mean_grid_dev_deg);
}
int emagls_design_from_atf_batch_dev(emagls_handle h, const emagls_config* cfg, const double* hL, const double* hR,
                                     int num_samples, int num_dirs, const double* hrir_grid, const double* atf_irs,
                                     int atf_samples, int num_mics, int atf_dirs, const double* atf_grid, double fs,
                                     int filter_len, double f_trans, int num_orient, const double* rotations,
                                     double* wL, double* wR, double* spectra) {
  return guarded(h, [&] {
    EM_REQUIRE(cfg && hL && hR && hrir_grid && atf_irs && atf_grid && wL && wR, "null argument");
    design_from_atf(h, *cfg, hL, hR, num_samples, num_dirs, hrir_grid, atf_irs, atf_samples, num_mics, atf_dirs,
                    atf_grid, fs, filter_len, f_trans, num_orient, rotations, wL, wR, spectra, nullptr);
  });
}
int emagls_design_ema_ch(emagls_handle h, const emagls_config* cfg, const double* hL, const double* hR,
                         int num_samples, int num_dirs, const double* grid_azi, const double* grid_zen,
                         double mic_radius, const double* mic_azi, int num_mics, int order, double fs, int len,
                         double* wL, double* wR, double* spectra) {
  return design_host(h, cfg, Variant::EMA_CH, hL, hR, num_samples, num_dirs, grid_azi, grid_zen, mic_radius,
                     mic_azi, nullptr, num_mics, order, fs, len, 1, 1, nullptr, wL, wR, spectra);
}
int emagls_design_ema_ch_batch(emagls_handle h, const emagls_config* cfg, const double* hL, const double* hR,
                               int num_samples, int num_dirs, const double* grid_azi, const double* grid_zen,
                               double mic_radius, const double* mic_azi, int num_mics, int order, double fs, int len,
                               int num_sets, int num_orient, const double* rotations, double* wL, double* wR,
                               double* spectra) {
  return design_host(h, cfg, Variant::EMA_CH, hL, hR, num_samples, num_dirs, grid_azi, grid_zen, mic_radius,
                     mic_azi, nullptr, num_mics, order, fs, len, num_sets, num_orient, rotations, wL, wR, spectra);
}
int emagls_design_ema_sh(emagls_handle h, const emagls_config* cfg, const double* hL, const double* hR,
                         int num_samples, int num_dirs, const double* grid_azi, const double* grid_zen,
                         double mic_radius, const double* mic_azi, int num_mics, int order, double fs, int len,
                         double* wL, double* wR, double* spectra) {
  return guarded(h, [&] {
    EM_REQUIRE(cfg && hL && hR && grid_azi && grid_zen && mic_azi && wL && wR, "null argument");
    EM_REQUIRE(num_samples > 0 && num_dirs > 0 && num_mics > 0 && len > 0 && order >= 0, "empty input");
    cudaStream_t st = h->stream;
    Arena ar(st);
    const int T = num_samples, D = num_dirs;
    const DesignShape shape = design_shape(*cfg, Variant::EMAGLS_SH, 0, order, len, bin_grid(*cfg, len, fs, T).K, 1);
    DeviceOutputs out(ar, shape, spectra != nullptr);
    design_ema_sh(h, *cfg, ar.upload(hL, (size_t)T * D), ar.upload(hR, (size_t)T * D), T, D, ar.upload(grid_azi, D),
                  ar.upload(grid_zen, D), mic_radius, ar.upload(mic_azi, num_mics), num_mics, order, fs, len,
                  out.wL, out.wR, out.sp);
    out.download(st, wL, wR, spectra);
  });
}

// ------------------------------------------------------------------------------------------
// getSMAIRMatrix (dependencies/getSMAIRMatrix.m:86-127) for radialFilter = 'none'
// ------------------------------------------------------------------------------------------
// out[(k*S + s)*rows + r] = Yrows[r][s] * bn[k][ord(s)]   (getSMAIRMatrix.m:112-122)
__global__ void smair_kernel(const cplx* __restrict__ Yrows, const cplx* __restrict__ bn, int rows, int S,
                             int N, int K, cplx* __restrict__ out) {
  long long idx = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (idx >= (long long)K * S * rows) return;
  int r = (int)(idx % rows);
  int s = (int)((idx / rows) % S);
  int k = (int)(idx / ((long long)rows * S));
  int ord = (int)sqrt((double)s);
  while ((ord + 1) * (ord + 1) <= s) ++ord;
  while (ord * ord > s) --ord;
  out[idx] = cmul(Yrows[(long long)r * S + s], bn[(long long)k * (N + 1) + ord]);
}

// Yout[c][s] = sum_m Lt[(m&1)*npair + m/2][c] * Ymic[m][s]   (pinv(Y_lo) * Y_Hi, getSMAIRMatrix.m:102,119-121)
__global__ void smair_project_kernel(const cplx* __restrict__ Lt, int npair, int nsh, int M, int S,
                                     const cplx* __restrict__ Ymic, cplx* __restrict__ Yout) {
  int idx = blockIdx.x * blockDim.x + threadIdx.x;
  if (idx >= nsh * S) return;
  int c = idx / S, s = idx % S;
  cplx acc = mk(0.0, 0.0);
  for (int m = 0; m < M; ++m) cfma(acc, Lt[((long long)(m & 1) * npair + m / 2) * nsh + c], Ymic[(long long)m * S + s]);
  Yout[idx] = acc;
}

// smairMat(r, :, k) *= rad(k, ord(r)), and once more by real(rad) at the Nyquist bin
// (getSMAIRMatrix.m:131-138: the k == numPosFreqs branch multiplies the already filtered page again)
__global__ void smair_radial_kernel(cplx* __restrict__ out, const cplx* __restrict__ rad, int rows, int S, int K,
                                    int L1) {
  long long idx = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (idx >= (long long)K * S * rows) return;
  const int r = (int)(idx % rows);
  const int k = (int)(idx / ((long long)rows * S));
  int ord = (int)sqrt((double)r);
  while ((ord + 1) * (ord + 1) <= r) ++ord;
  while (ord * ord > r) --ord;
  const cplx f = rad[(long long)k * L1 + ord];
  cplx v = cmul(f, out[idx]);
  if (k == K - 1) v = mk(f.x * v.x, f.x * v.y);
  out[idx] = v;
}

static int smair_impl(emagls_handle h, const emagls_config* cfg, const emagls_radial_params* rp, const double* mic_azi,
                      const double* mic_zen, int num_mics, int order, double fs, double sma_radius,
                      int nfft, int return_raw_mic_sigs, double* out, int* sim_order_out) {
  return guarded(h, [&] {
    EM_REQUIRE(cfg && mic_azi && mic_zen && num_mics > 0, "null argument");
    EM_REQUIRE(nfft > 0 && nfft % 2 == 0, "nfft must be even");  // getSMAIRMatrix.m:89
    const int simN = sim_order(*cfg, order, fs, sma_radius);
    if (sim_order_out) *sim_order_out = simN;
    if (!out) return;
    EM_REQUIRE(simN <= MAX_SH_ORDER, "simulation order too high");
    cudaStream_t st = h->stream;
    Arena ar(st);
    const int S = (simN + 1) * (simN + 1), K = nfft / 2 + 1, M = num_mics;
    const int nsh = (order + 1) * (order + 1);
    const int cb = cfg->basis == EMAGLS_BASIS_COMPLEX ? 1 : 0;
    const std::vector<double> kr = kr_table(*cfg, fs, sma_radius, K);
    cplx* bn = ar.get<cplx>((size_t)K * (simN + 1));
    EM_CUDA(launch_modal(st, simN, ar.upload(kr.data(), K), K, cfg->array_type, -1.0, 1, bn, simN + 1, 1));
    // Y_Hi = shFunction(simulationOrder, mics, shDefinition) as rows [M][S]
    double* Y = ar.get<double>((size_t)M * S * (cb ? 2 : 1));
    EM_CUDA(launch_sh_angles(st, simN, ar.upload(mic_azi, M), ar.upload(mic_zen, M), M, cb, Y));
    cplx* Ymic = ar.get<cplx>((size_t)M * S);
    EM_CUDA(launch_sh_rows(st, Y, M, S, cb, Ymic));
    h->launches += 3;
    const cplx* Yrows = Ymic;
    int rows = M;
    if (!return_raw_mic_sigs) {
      EM_REQUIRE(M >= nsh && nsh <= 64 && M <= 4096, "fewer microphones than SH channels (or more than 64 channels)");
      // pinv(Y_Hi(:, 1:(order+1)^2)) through the factorisation kernel with the clip disabled
      cplx* Alo = ar.get<cplx>((size_t)M * nsh);
      EM_CUDA(cudaMemcpy2DAsync(Alo, (size_t)nsh * sizeof(cplx), Ymic, (size_t)S * sizeof(cplx),
                                (size_t)nsh * sizeof(cplx), M, cudaMemcpyDeviceToDevice, st));
      cplx* Lt = unclipped_pinv_dev(h, ar, Alo, M, nsh);
      cplx* Yout = ar.get<cplx>((size_t)nsh * S);
      smair_project_kernel<<<(nsh * S + 255) / 256, 256, 0, st>>>(Lt, (M + 1) / 2, nsh, M, S, Ymic, Yout);
      EM_CUDA(cudaGetLastError());
      h->launches += 1;
      Yrows = Yout;
      rows = nsh;
    }
    cplx* d_out = ar.get<cplx>((size_t)K * S * rows);
    long long total = (long long)K * S * rows;
    smair_kernel<<<(unsigned)((total + 255) / 256), 256, 0, st>>>(Yrows, bn, rows, S, simN, K, d_out);
    EM_CUDA(cudaGetLastError());
    h->launches += 1;
    if (rp && rp->kind != EMAGLS_RADIAL_NONE && !return_raw_mic_sigs) {
      cplx* rad = ar.get<cplx>((size_t)K * (order + 1));
      radial_filter_dev(h, ar, *cfg, *rp, order, fs, sma_radius, nfft, 0, rad);
      smair_radial_kernel<<<(unsigned)((total + 255) / 256), 256, 0, st>>>(d_out, rad, rows, S, K, order + 1);
      EM_CUDA(cudaGetLastError());
      h->launches += 1;
    }
    EM_CUDA(cudaMemcpyAsync(out, d_out, (size_t)total * sizeof(cplx), cudaMemcpyDeviceToHost, st));
    EM_CUDA(cudaStreamSynchronize(st));
  });
}

int emagls_smair_matrix(emagls_handle h, const emagls_config* cfg, const double* mic_azi,
                        const double* mic_zen, int num_mics, int order, double fs, double sma_radius,
                        int nfft, int return_raw_mic_sigs, double* out, int* sim_order_out) {
  return smair_impl(h, cfg, nullptr, mic_azi, mic_zen, num_mics, order, fs, sma_radius, nfft, return_raw_mic_sigs,
                    out, sim_order_out);
}

int emagls_smair_matrix_radial(emagls_handle h, const emagls_config* cfg, const emagls_radial_params* rp,
                               const double* mic_azi, const double* mic_zen, int num_mics, int order, double fs,
                               double sma_radius, int nfft, double* out, int* sim_order_out) {
  if (!h) return EMAGLS_ERR_INVALID;
  if (!rp || rp->kind < EMAGLS_RADIAL_NONE || rp->kind > EMAGLS_RADIAL_FULL) {
    h->err = "Unkown radialFilter parameter";   // getRadialFilter.m:65
    return EMAGLS_ERR_INVALID;
  }
  return smair_impl(h, cfg, rp, mic_azi, mic_zen, num_mics, order, fs, sma_radius, nfft, 0, out, sim_order_out);
}

int emagls_design_magls_2d(emagls_handle h, const emagls_config* cfg, const double* hL, const double* hR,
                           int num_samples, int num_dirs, const double* grid_azi, int order, double fs, int len,
                           double* wL, double* wR, double* spectra) {
  return guarded(h, [&] {
    EM_REQUIRE(cfg && hL && hR && grid_azi && wL && wR, "null argument");
    EM_REQUIRE(num_samples > 0 && num_dirs > 0 && len > 0 && order >= 0, "empty input");
    cudaStream_t st = h->stream;
    Arena ar(st);
    const int T = num_samples, D = num_dirs;
    const DesignShape shape = design_shape(*cfg, Variant::EMA_CH, 0, order, len, bin_grid(*cfg, len, fs, T).K, 1);
    DeviceOutputs out(ar, shape, spectra != nullptr);
    design_magls(h, *cfg, ar.upload(hL, (size_t)T * D), ar.upload(hR, (size_t)T * D), T, D, ar.upload(grid_azi, D),
                 nullptr, order, fs, len, false, out.wL, out.wR, out.sp, 1);
    out.download(st, wL, wR, spectra);
  });
}

// ------------------------------------------------------------------------------------------
// building blocks for parity tests
// ------------------------------------------------------------------------------------------
int emagls_get_sh(emagls_handle h, int order, const double* azi, const double* zen, int num_dirs, int basis,
                  double* out) {
  return guarded(h, [&] {
    EM_REQUIRE(azi && zen && out && num_dirs > 0, "null argument");
    EM_REQUIRE(order >= 0 && order <= MAX_SH_ORDER, "order out of range");
    cudaStream_t st = h->stream;
    Arena ar(st);
    const size_t S = (size_t)(order + 1) * (order + 1);
    const size_t n = S * num_dirs * (basis == EMAGLS_BASIS_COMPLEX ? 2 : 1);
    double* d_out = ar.get<double>(n);
    EM_CUDA(launch_sh_angles(st, order, ar.upload(azi, num_dirs), ar.upload(zen, num_dirs), num_dirs,
                             basis == EMAGLS_BASIS_COMPLEX, d_out));
    h->launches += 1;
    EM_CUDA(cudaMemcpyAsync(out, d_out, n * sizeof(double), cudaMemcpyDeviceToHost, st));
    EM_CUDA(cudaStreamSynchronize(st));
  });
}

int emagls_group_delay(emagls_handle h, const double* hrir, int taps, int num_dirs, int num_freqs, double fs,
                       double* gd, double* median_out) {
  return guarded(h, [&] {
    EM_REQUIRE(hrir && taps > 0 && num_dirs > 0 && num_freqs > 1 && fs > 0.0, "invalid argument");
    cudaStream_t st = h->stream;
    Arena ar(st);
    const int nchunk = 32;
    const double* d_h = ar.upload(hrir, (size_t)taps * num_dirs);
    double* partial = ar.get<double>((size_t)nchunk * taps);
    double* hsum = ar.get<double>((size_t)taps);
    double* d_gd = ar.get<double>((size_t)num_freqs);
    EM_CUDA(launch_colsum(st, d_h, taps, num_dirs, partial, nchunk, hsum));
    EM_CUDA(launch_grpdelay(st, hsum, taps, num_freqs, fs, d_gd));
    h->launches += 3;
    std::vector<double> g((size_t)num_freqs);
    EM_CUDA(cudaMemcpyAsync(g.data(), d_gd, g.size() * sizeof(double), cudaMemcpyDeviceToHost, st));
    EM_CUDA(cudaStreamSynchronize(st));
    if (gd) std::copy(g.begin(), g.end(), gd);
    if (median_out) *median_out = median_of(g);
  });
}

int emagls_sph_modal_coeffs(emagls_handle h, int order, const double* kr, int num_kr, int array_type,
                            double* out) {
  return guarded(h, [&] {
    EM_REQUIRE(kr && out && num_kr > 0, "null argument");
    EM_REQUIRE(order >= 0 && order <= MAX_SH_ORDER, "order out of range");
    cudaStream_t st = h->stream;
    Arena ar(st);
    cplx* d_out = ar.get<cplx>((size_t)num_kr * (order + 1));
    // column-major [num_kr x (order+1)]
    EM_CUDA(launch_modal(st, order, ar.upload(kr, num_kr), num_kr, array_type, 1.0, 0, d_out, 1, num_kr));
    h->launches += 1;
    EM_CUDA(cudaMemcpyAsync(out, d_out, (size_t)num_kr * (order + 1) * sizeof(cplx), cudaMemcpyDeviceToHost, st));
    EM_CUDA(cudaStreamSynchronize(st));
  });
}

int emagls_regularized_apply(emagls_handle h, const double* pw, int num_ch, int num_dirs,
                             const double* targets, int num_t, double svd_regul, double* out) {
  return guarded(h, [&] {
    EM_REQUIRE(pw && targets && out, "null argument");
    EM_REQUIRE(num_ch > 0 && num_ch <= 64 && num_dirs >= num_ch && num_t > 0, "bad shape");
    cudaStream_t st = h->stream;
    Arena ar(st);
    const int Mc = num_ch, D = num_dirs;
    // pw is [Mc x D] column-major == rows of pwGrid.' with the channel index contiguous
    cplx* At = reinterpret_cast<cplx*>(ar.upload(pw, (size_t)2 * Mc * D));
    // targets [num_t x D] complex column-major -> pairs of rows (re | im) of length D
    const int npair = (num_t + 1) / 2;
    std::vector<double> rows((size_t)npair * 4 * D, 0.0);
    for (int t = 0; t < num_t; ++t)
      for (int d = 0; d < D; ++d) {
        size_t base = ((size_t)(t / 2) * 2 + (t & 1)) * 2 * D;
        rows[base + d] = targets[2 * ((size_t)d * num_t + t)];
        rows[base + D + d] = targets[2 * ((size_t)d * num_t + t) + 1];
      }
    double* d_rows = ar.upload(rows.data(), rows.size());
    cplx* W = ar.get<cplx>((size_t)2 * npair * Mc);  // [ear][pair][Mc]
    regularized_apply_dev(h, ar, At, D, Mc, d_rows, npair, svd_regul, W);
    std::vector<cplx> Wh((size_t)2 * npair * Mc);
    EM_CUDA(cudaMemcpyAsync(Wh.data(), W, Wh.size() * sizeof(cplx), cudaMemcpyDeviceToHost, st));
    EM_CUDA(cudaStreamSynchronize(st));
    for (int t = 0; t < num_t; ++t)
      for (int m = 0; m < Mc; ++m) {
        cplx v = Wh[((size_t)(t & 1) * npair + t / 2) * Mc + m];
        out[2 * ((size_t)m * num_t + t)] = v.x;
        out[2 * ((size_t)m * num_t + t) + 1] = v.y;
      }
  });
}

}  // extern "C"
