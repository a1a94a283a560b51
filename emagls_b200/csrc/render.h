// Overlap-save machinery shared by the static render (render.cu) and the head-tracked render (tracked_render.cu):
// cuFFT plan caches and the forward transforms of the input blocks.
#pragma once
#include <cufft.h>
#include <string>
#include "engine.h"

namespace emagls {

#define EM_FFT(expr)                                                                              \
  do {                                                                                            \
    cufftResult _r = (expr);                                                                      \
    if (_r != CUFFT_SUCCESS)                                                                      \
      throw ::emagls::Fail{EMAGLS_ERR_CUDA, std::string(#expr) + ": cufft error " + std::to_string((int)_r)}; \
  } while (0)

constexpr int MAX_EDGE = 8;  // staged boundary blocks per chunk (head + tail)

int env_int(const char* name, int dflt);

// (Re)build the plans of one render geometry in `rp` (cached between calls): forward transforms of nbc blocks of every
// channel, `filt_batch` zero-padded filters and `inv_batch` inverse transforms.
void ensure_plans(emagls_ctx* h, emagls_ctx::RenderPlans& rp, int N, int L, int num_ch, int nbc, int filt_batch,
                  int inv_batch);
void drop_plans(emagls_ctx::RenderPlans& rp);

// Forward transforms of the overlap-save blocks of a multichannel signal into X[ch][nbc][F].  Block b takes the N
// input samples starting at b*L - ov.  Direct route (default when every channel of the signal is 16-byte aligned):
// interior blocks are transformed in place from `in`, one cuFFT call per channel, and only the blocks that overlap the
// ends of the signal are staged zero-padded.  Staged route: the whole chunk is copied into a segment buffer first (one
// cuFFT call per chunk).  ensure_plans must have been called on `rp` with this nbc.
struct ForwardStage {
  ForwardStage(emagls_ctx* h, emagls_ctx::RenderPlans& rp, Arena& ar, const double* in, long long num_samples,
               int num_ch, int N, int L, int ov, int nbc);
  // blocks [b0, b0 + nbk) -> X[ch][b - b0][F] (nbk <= nbc - nex)
  void run(long long b0, long long nbk, cplx* X);
  static int extra_blocks(int ov, int L) { return (ov + L - 1) / L; }

  emagls_ctx* h;
  emagls_ctx::RenderPlans& rp;
  const double* in;
  long long num_samples;
  int num_ch, N, L, ov, nbc;
  long long seg_len;
  bool direct;
  long long b_int_lo, b_int_hi;  // blocks that lie inside the signal
  double* xp;                    // staging buffer
};

}  // namespace emagls
