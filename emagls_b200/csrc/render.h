// Overlap-save machinery shared by the static render (render.cu) and the head-tracked render (tracked_render.cu):
// cuFFT plan caches and the forward transforms of the input blocks; the SH rotation stage shared by the SH
// head-tracked render and the render sessions.
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

// The static render (binauralDecode) with the first `skip` output samples dropped: out[ear * out_rows + n - skip] for
// n in [skip, num_samples).  The public entry points pass skip = 0 or len/2 - 1 (compensateDelay) and
// out_rows = num_samples - skip; the SH head-tracked render writes one time chunk into a longer output with it.
void binaural_decode_rows(emagls_ctx* h, const double* in, long long num_samples, int num_ch, const double* wL,
                          const double* wR, int len, long long skip, long long out_rows, double* out);

// ---- sound-field rotation of the SH head-tracked render (sh_tracked_render.cu), shared with the render sessions
// (stream_render.cu)

// doubles of the block-diagonal part of a rotation matrix: sum_{l <= order} (2l + 1)^2, and the offset of band l
__host__ __device__ constexpr int band_offset(int l) { return l * (4 * l * l - 1) / 3; }

// Q[j][band_offset(l) + r (2l+1) + c] = getSHrotMtx(rot[f], order, 'real')[l^2 + r][l^2 + c] for frame f = f_base + j,
// and same[j] = 1 when rot[f] is bitwise equal to rot[f - 1] (rot[k] holds frame rot_base + k).  Listener y
// (blockIdx.y; the whole-signal render launches one with zero strides) reads rot + y rot_ls and writes
// Q + y nfr_ls band_offset(order + 1) and same + y nfr_ls.
__global__ void frame_rotations_kernel(const double* __restrict__ rot, long long rot_ls, long long rot_base,
                                       long long f_base, int order, double* __restrict__ Q, int* __restrict__ same,
                                       long long nfr_ls);
// out[ch][q] = (in[h0 + q, :] @ M)[ch] for q < m with the blended frame matrices of the contract; in has leading
// dimension ld_in and in[0] sits at first_sample on the track's time axis; Q and same hold frames f_base ...
// Listener y (blockIdx.y) rotates the shared input with its own Q and same (strides as above) into out + y out_ls.
__global__ void sh_track_rotate_kernel(const double* __restrict__ in, long long ld_in, long long h0, long long m,
                                       int order, const double* __restrict__ Q, const int* __restrict__ same,
                                       long long nfr_ls, long long f_base, long long first_sample, int hop, int fade,
                                       double* __restrict__ out, long long out_ls);
// the two kernels above for nl listeners x nfr frames / m samples on h->stream (launch counting and profiling are the
// caller's)
void launch_frame_rotations(emagls_ctx* h, int nl, const double* rot, long long rot_ls, long long rot_base,
                            long long f_base, long long nfr, int order, double* Q, int* same, long long nfr_ls);
void launch_sh_track_rotate(emagls_ctx* h, int nl, const double* in, long long ld_in, long long h0, long long m,
                            int order, const double* Q, const int* same, long long nfr_ls, long long f_base,
                            long long first_sample, int hop, int fade, double* out, long long out_ls);

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
