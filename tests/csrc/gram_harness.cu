// Test harness of the Gram route's kernels (emagls_b200/csrc/gram_kernels.cu) for tests/test_gpu_gram_kernels.py.
// Including the translation units gives access to the file-static launchers of the backward step (launch_bwd_fused_t,
// launch_bwd_small_t), so each backward kernel runs directly for every digit count, as well as through
// launch_bwd_small's own choice.  ozaki_kernels.cu supplies launch_slice_rows, the unfused reference of the fused tail.
// The extern "C" entry points take host arrays (ctypes): they allocate, copy in, launch, synchronise, copy out and free,
// and return the first cudaError_t.  Every output buffer is pre-filled with a sentinel (every byte 0xFF for FP64 and
// int32, a given byte for digits) and followed by a guard region of `guard` elements, which is copied back too.
#include "../../emagls_b200/csrc/gram_kernels.cu"
#include "../../emagls_b200/csrc/ozaki_kernels.cu"

using namespace emagls;

namespace {

struct DevBuf {
  void* p = nullptr;
  ~DevBuf() { if (p) cudaFree(p); }
};

cudaError_t upload(DevBuf& b, const void* host, size_t bytes) {
  cudaError_t e = cudaMalloc(&b.p, bytes ? bytes : 1);
  if (e == cudaSuccess && bytes) e = cudaMemcpy(b.p, host, bytes, cudaMemcpyHostToDevice);
  return e;
}
cudaError_t output(DevBuf& b, size_t bytes, int fill) {
  cudaError_t e = cudaMalloc(&b.p, bytes ? bytes : 1);
  if (e == cudaSuccess) e = cudaMemset(b.p, fill, bytes);
  return e;
}
cudaError_t download(void* host, const DevBuf& b, size_t bytes) {
  return cudaMemcpy(host, b.p, bytes, cudaMemcpyDeviceToHost);
}
// the launch error if there is one, else the first error of synchronising and copying back
template <class F>
int finish(cudaError_t launch, F&& copy_back) {
  cudaError_t e = cudaDeviceSynchronize();
  if (e == cudaSuccess) e = copy_back();
  return (int)(launch != cudaSuccess ? launch : e);
}

}  // namespace

extern "C" int gh_sm_count() { return sm_count(); }

// launch_gram_chol on nbins * P packed matrices Gre, Gim [nmat][ne_ld] (host arrays).  Outputs: Pb [nmat][Mc][Mc]
// complex + guard (copied back when Pb != nullptr), sig [nmat] + guard, fail [1 + nbins] + guard; fail starts at zero.
extern "C" int gh_gram_chol(const double* Gre, const double* Gim, int Mc, int P, int ne_ld, int nbins, double thr,
                            double* Pb, double* sig, int* fail, long long guard) {
  DevBuf gr, gi, pb, sg, fl;
  const long long nmat = (long long)nbins * P;
  const size_t npb = (size_t)nmat * Mc * Mc + guard, nsig = (size_t)nmat + guard, nfail = (size_t)1 + nbins + guard;
  cudaError_t e = upload(gr, Gre, (size_t)nmat * ne_ld * 8);
  if (e == cudaSuccess) e = upload(gi, Gim, (size_t)nmat * ne_ld * 8);
  if (e == cudaSuccess) e = output(pb, npb * 16, 0xFF);
  if (e == cudaSuccess) e = output(sg, nsig * 8, 0xFF);
  if (e == cudaSuccess) e = output(fl, nfail * 4, 0xFF);
  if (e == cudaSuccess) e = cudaMemset(fl.p, 0, (size_t)(1 + nbins) * 4);
  if (e != cudaSuccess) return (int)e;
  const cudaError_t l = launch_gram_chol(0, (const double*)gr.p, (const double*)gi.p, Mc, P, ne_ld, nbins, thr,
                                         (cplx*)pb.p, (double*)sg.p, (int*)fl.p);
  return finish(l, [&] {
    cudaError_t r = Pb ? download(Pb, pb, npb * 16) : cudaSuccess;
    if (r == cudaSuccess) r = download(sig, sg, nsig * 8);
    return r == cudaSuccess ? download(fail, fl, nfail * 4) : r;
  });
}

// The same launch on device buffers the caller owns (the production-size launches, whose packed matrices are tiled on
// the device): Gre, Gim [nmat][ne_ld], Pb [nmat][Mc][Mc] scratch, sig [nmat], fail [1 + nbins] (zeroed here).
extern "C" int gh_gram_chol_device(const double* Gre, const double* Gim, int Mc, int P, int ne_ld, int nbins,
                                   double thr, void* Pb, double* sig, int* fail) {
  cudaError_t e = cudaMemset(fail, 0, (size_t)(1 + nbins) * 4);
  if (e != cudaSuccess) return (int)e;
  const cudaError_t l = launch_gram_chol(0, Gre, Gim, Mc, P, ne_ld, nbins, thr, (cplx*)Pb, sig, fail);
  return finish(l, [] { return cudaSuccess; });
}

namespace {

// launch_bwd_small's shared memory of bwd_fused_kernel, and the conditions under which it picks that kernel; forcing
// it elsewhere is refused
size_t fused_smem_bytes(int Mc, int S) {
  return (((size_t)Mc * S + 1) & ~(size_t)1) * sizeof(double) + (size_t)(BF_WARPS * 64 + 64 + 64 + 80) * sizeof(cplx) +
         (4 * BF_WARPS + 4) * sizeof(double);
}
bool fused_fits(int Mc, int S, int N, int KpS, bool tail) {
  return N >= 0 && N < 40 && Mc <= 32 && S <= 128 * BF_CH && ((Mc * S) & 1) == 0 &&
         fused_smem_bytes(Mc, S) <= 113 * 1024 && (!tail || KpS <= 64 * BF_WARPS);
}

}  // namespace

// Backward step of a Gram bin, W_k = (Y_o (conj(b_k) .* z)) Pb, with the fused forward of bin k + 1 when T > 0.
// mode 0: launch_bwd_small (its own choice of kernel), 1: bwd_fused_kernel<T>, 2: bwd_small_kernel<T>.
// Y [oc][Mc][S], Pb [oc][Mc][Mc] complex, bk / bk_next [N + 1] complex, z [nz]; Wsp [nW] complex is copied in (the
// caller's sentinels) and back.  T > 0: Cv_q [T][4 num_prob][KpS] + guard bytes (filled with `fill`), sCv
// [4 num_prob] + guard.
extern "C" int gh_bwd(int mode, int T, const double* Y, int Mc, int S, const int* roword, int N, const double* bk,
                      const double* Pb, int oc, int o0, int num_orient, int num_prob, const double* z, long long nz,
                      long long z_set_stride, long long z_ear_stride, int z_shared, int nsplit, long long split_stride,
                      double* Wsp, long long nW, long long w_ear_stride, int K, int k, int dc_fix,
                      const double* bk_next, int KpS, int8_t* Cv_q, double* sCv, long long guard, int fill) {
  if (mode == 1 && !fused_fits(Mc, S, N, KpS, T > 0)) return (int)cudaErrorInvalidValue;
  if (T != 0 && T != 4 && T != 6) return (int)cudaErrorInvalidValue;
  DevBuf y, ro, b, bn, pb, zz, w, q, sc;
  const long long rows = 4LL * num_prob;
  const size_t nq = (size_t)T * rows * KpS + guard, ns = (size_t)rows + guard;
  cudaError_t e = upload(y, Y, (size_t)oc * Mc * S * 8);
  if (e == cudaSuccess) e = upload(ro, roword, (size_t)S * 4);
  if (e == cudaSuccess) e = upload(b, bk, (size_t)(N + 1) * 16);
  if (e == cudaSuccess) e = upload(bn, bk_next, (size_t)(N + 1) * 16);
  if (e == cudaSuccess) e = upload(pb, Pb, (size_t)oc * Mc * Mc * 16);
  if (e == cudaSuccess) e = upload(zz, z, (size_t)nz * 8);
  if (e == cudaSuccess) e = upload(w, Wsp, (size_t)nW * 16);
  if (e == cudaSuccess) e = output(q, nq, fill);
  if (e == cudaSuccess) e = output(sc, ns * 8, 0xFF);
  if (e != cudaSuccess) return (int)e;
  const ProbMap pm{oc, o0, num_orient};
  const double* Yd = (const double*)y.p;
  const int* rod = (const int*)ro.p;
  const cplx *bkd = (const cplx*)b.p, *pbd = (const cplx*)pb.p;
  const double* zd = (const double*)zz.p;
  cplx* wd = (cplx*)w.p;
  const FwdFuse ff{T > 0 ? (const cplx*)bn.p : nullptr, (int8_t*)q.p, (double*)sc.p, KpS, rows};
  const size_t fused_smem = fused_smem_bytes(Mc, S);
  const size_t small_smem = ((size_t)2 * S + 4 * Mc) * sizeof(cplx);
#define GH_BWD_ARGS num_prob, Yd, Mc, S, rod, bkd, pbd, pm, zd, z_set_stride, z_ear_stride, z_shared, nsplit, \
                    split_stride, wd, w_ear_stride, K, k, dc_fix, ff
  cudaError_t l = cudaErrorInvalidValue;
  if (mode == 0) {
    l = launch_bwd_small(0, Yd, Mc, S, rod, bkd, pbd, pm, num_prob, zd, z_set_stride, z_ear_stride, z_shared, nsplit,
                         split_stride, wd, w_ear_stride, K, k, dc_fix, ff.bk_next, ff.Cv_q, ff.sCv, KpS, T, N);
  } else if (mode == 1) {
    switch (T) {
      case 0: l = launch_bwd_fused_t<0>(0, fused_smem, GH_BWD_ARGS, N); break;
      case 4: l = launch_bwd_fused_t<4>(0, fused_smem, GH_BWD_ARGS, N); break;
      case 6: l = launch_bwd_fused_t<6>(0, fused_smem, GH_BWD_ARGS, N); break;
    }
  } else if (mode == 2) {
    switch (T) {
      case 0: l = launch_bwd_small_t<0>(0, small_smem, GH_BWD_ARGS); break;
      case 4: l = launch_bwd_small_t<4>(0, small_smem, GH_BWD_ARGS); break;
      case 6: l = launch_bwd_small_t<6>(0, small_smem, GH_BWD_ARGS); break;
    }
  }
#undef GH_BWD_ARGS
  return finish(l, [&] {
    cudaError_t r = download(Wsp, w, (size_t)nW * 16);
    if (r == cudaSuccess && T > 0) r = download(Cv_q, q, nq);
    return (r == cudaSuccess && T > 0) ? download(sCv, sc, ns * 8) : r;
  });
}

// The unfused forward of bin kprev + 1: launch_fwd_small (u = b .* (Y_o^T W_kprev) into Cv [4 num_prob][S] + guard),
// then, when T > 0, launch_slice_rows of Cv into Cv_q [T][4 num_prob][KpS] + guard bytes and sCv [4 num_prob] + guard.
extern "C" int gh_fwd_slice(const double* Y, int Mc, int S, const int* roword, int N, const double* bk, int oc, int o0,
                            int num_orient, int num_prob, const double* Wsp, long long nW, long long w_ear_stride, int K,
                            int kprev, int T, int KpS, double* Cv, int8_t* Cv_q, double* sCv, long long guard, int fill) {
  DevBuf y, ro, b, w, cv, q, sc;
  const long long rows = 4LL * num_prob;
  const size_t ncv = (size_t)rows * S + guard, nq = (size_t)T * rows * KpS + guard, ns = (size_t)rows + guard;
  cudaError_t e = upload(y, Y, (size_t)oc * Mc * S * 8);
  if (e == cudaSuccess) e = upload(ro, roword, (size_t)S * 4);
  if (e == cudaSuccess) e = upload(b, bk, (size_t)(N + 1) * 16);
  if (e == cudaSuccess) e = upload(w, Wsp, (size_t)nW * 16);
  if (e == cudaSuccess) e = output(cv, ncv * 8, 0xFF);
  if (e == cudaSuccess) e = output(q, nq, fill);
  if (e == cudaSuccess) e = output(sc, ns * 8, 0xFF);
  if (e != cudaSuccess) return (int)e;
  const ProbMap pm{oc, o0, num_orient};
  cudaError_t l = launch_fwd_small(0, (const double*)y.p, Mc, S, (const int*)ro.p, (const cplx*)b.p, pm, num_prob,
                                   (const cplx*)w.p, w_ear_stride, K, kprev, (double*)cv.p);
  if (l == cudaSuccess && T > 0)
    l = launch_slice_rows(0, (const double*)cv.p, S, 1, (int)rows, S, KpS, T, (int8_t*)q.p, (double*)sc.p);
  return finish(l, [&] {
    cudaError_t r = download(Cv, cv, ncv * 8);
    if (r == cudaSuccess && T > 0) r = download(Cv_q, q, nq);
    return (r == cudaSuccess && T > 0) ? download(sCv, sc, ns * 8) : r;
  });
}
