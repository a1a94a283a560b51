// Test harness of the int8 tensor-core GEMM (emagls_b200/csrc/ozaki.cuh, ozaki_kernels.cu) for tests/test_gpu_ozaki.py.
// Including the translation unit gives access to every kernel instance the library can launch (the file-static
// oz_fwd_t included), so each one is run directly, bypassing the cost rules, as well as through the library's launch
// functions.  The extern "C" entry points take host arrays (ctypes): they allocate, copy in, launch, synchronise, copy
// out and free, and return the first cudaError_t.  Every output buffer is pre-filled with a sentinel (NaN for FP64, a
// given byte for digits) and followed by a guard region of `guard` elements, which is copied back too.
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

extern "C" int oh_sm_count() { return sm_count(); }
extern "C" int oh_contraction_fits(int Kpad, int T) { return oz::contraction_fits(Kpad, T); }
extern "C" int oh_drain_i64_fits(int Kpad, int T) { return oz::drain_i64_fits(Kpad, T); }

// launch_slice_rows: x(r, k) = src[r rs + k cs] (n_src doubles); out [T][R][Kpad] + guard bytes, scale [R] + guard
extern "C" int oh_slice_rows(const double* src, long long n_src, long long rs, long long cs, int R, int K, int Kpad, int T,
                             int Tbuf, int8_t* out, double* scale, long long guard, int fill) {
  DevBuf s, o, sc;
  const size_t nq = (size_t)Tbuf * R * Kpad + guard, ns = (size_t)R + guard;
  cudaError_t e = upload(s, src, (size_t)n_src * 8);
  if (e == cudaSuccess) e = output(o, nq, fill);
  if (e == cudaSuccess) e = output(sc, ns * 8, 0xFF);
  if (e != cudaSuccess) return (int)e;
  const cudaError_t l = launch_slice_rows(0, (const double*)s.p, rs, cs, R, K, Kpad, T, (int8_t*)o.p, (double*)sc.p);
  return finish(l, [&] {
    cudaError_t r = download(out, o, nq);
    return r == cudaSuccess ? download(scale, sc, ns * 8) : r;
  });
}

// launch_row_scale: x [rows][D]; up, sc [rows] + guard
extern "C" int oh_row_scale(const double* x, long long rows, int D, double* up, double* sc, long long guard) {
  DevBuf xb, ub, sb;
  const size_t n = (size_t)rows + guard;
  cudaError_t e = upload(xb, x, (size_t)rows * D * 8);
  if (e == cudaSuccess) e = output(ub, n * 8, 0xFF);
  if (e == cudaSuccess) e = output(sb, n * 8, 0xFF);
  if (e != cudaSuccess) return (int)e;
  const cudaError_t l = launch_row_scale(0, (const double*)xb.p, rows, D, (double*)ub.p, (double*)sb.p);
  return finish(l, [&] {
    cudaError_t r = download(up, ub, n * 8);
    return r == cudaSuccess ? download(sc, sb, n * 8) : r;
  });
}

// Backward product tq [rows][S] = t^T B, FP64 out (EpiStoreF64).  inst 0: 128 x 64 tiles, 1: 128 x 80, 2: 128 x 48,
// 3: launch_oz_bwd (its cost rule picks one of the three).  Operands: Tq [Tbuf][rows][Kpad], Bq [Tbuf][S][Kpad].
extern "C" int oh_bwd(int inst, const int8_t* Tq, const double* sT, int rows, const int8_t* Bq, const double* sB, int S,
                      int Kpad, int T, int Tbuf, double* tq, long long guard) {
  DevBuf a, sa, b, sb, c;
  const size_t nc = (size_t)rows * S + guard;
  cudaError_t e = upload(a, Tq, (size_t)Tbuf * rows * Kpad);
  if (e == cudaSuccess) e = upload(sa, sT, (size_t)rows * 8);
  if (e == cudaSuccess) e = upload(b, Bq, (size_t)Tbuf * S * Kpad);
  if (e == cudaSuccess) e = upload(sb, sB, (size_t)S * 8);
  if (e == cudaSuccess) e = output(c, nc * 8, 0xFF);
  if (e != cudaSuccess) return (int)e;
  const int8_t* A = (const int8_t*)a.p;
  const int8_t* B = (const int8_t*)b.p;
  const double *SA = (const double*)sa.p, *SB = (const double*)sb.p;
  const oz::EpiStoreF64 epi{(double*)c.p, (long long)S};
  cudaError_t l = cudaErrorInvalidValue;
  switch (inst) {
    case 0: l = oz::launch_ozaki_gemm(0, A, SA, B, SB, rows, S, Kpad, T, epi, sm_count()); break;
    case 1: l = oz::launch_ozaki_gemm<oz::EpiStoreF64, oz::TileWide>(0, A, SA, B, SB, rows, S, Kpad, T, epi, sm_count()); break;
    case 2: l = oz::launch_ozaki_gemm<oz::EpiStoreF64, oz::TileCfg<48, 3>>(0, A, SA, B, SB, rows, S, Kpad, T, epi, sm_count()); break;
    case 3: l = launch_oz_bwd(0, A, SA, rows, B, SB, S, Kpad, T, (double*)c.p); break;
  }
  return finish(l, [&] { return download(tq, c, nc * 8); });
}

// Forward product with the phase-continuation epilogue.  inst 0: EpiPhaseSliceRaw<4>, 1: EpiPhaseSliceRaw<6>,
// 2: EpiPhaseSliceFix<6> on 128 x 64 tiles, 3: EpiPhaseSliceFix<6> on 128 x 80 tiles with 20 epilogue warps,
// 4: launch_oz_fwd.  Operands Yq [Tbuf][D][KpS], Cq [Tbuf][rows][KpS]; out Tq [Tbuf][rows][KpD] + guard bytes (filled
// with `fill`), sT [rows] + guard; absH (n_abs doubles) and up, sc (n_scale doubles each) start at this bin.
extern "C" int oh_fwd(int inst, const int8_t* Yq, const double* sY, int D, int KpS, const int8_t* Cq, const double* sC,
                      int rows, int T, int Tbuf, int8_t* Tq, int KpD, double* sT, const double* absH, long long n_abs,
                      long long abs_set_stride, long long abs_ear_stride, const double* up, const double* sc,
                      long long n_scale, int scale_stride, int orient_per_set, int nyquist, long long guard, int fill) {
  DevBuf y, sy, c, scv, t, st, ab, ub, sb;
  const size_t nt = (size_t)Tbuf * rows * KpD + guard, ns = (size_t)rows + guard;
  cudaError_t e = upload(y, Yq, (size_t)Tbuf * D * KpS);
  if (e == cudaSuccess) e = upload(sy, sY, (size_t)D * 8);
  if (e == cudaSuccess) e = upload(c, Cq, (size_t)Tbuf * rows * KpS);
  if (e == cudaSuccess) e = upload(scv, sC, (size_t)rows * 8);
  if (e == cudaSuccess) e = upload(ab, absH, (size_t)n_abs * 8);
  if (e == cudaSuccess) e = upload(ub, up, (size_t)n_scale * 8);
  if (e == cudaSuccess) e = upload(sb, sc, (size_t)n_scale * 8);
  if (e == cudaSuccess) e = output(t, nt, fill);
  if (e == cudaSuccess) e = output(st, ns * 8, 0xFF);
  if (e != cudaSuccess) return (int)e;
  const OzFwdArgs a{(const int8_t*)y.p, (const double*)sy.p, D, KpS, (const int8_t*)c.p, (const double*)scv.p, rows, T,
                    (int8_t*)t.p, KpD, (double*)st.p, (const double*)ab.p, abs_set_stride, abs_ear_stride,
                    (const double*)ub.p, (const double*)sb.p, scale_stride, orient_per_set, nyquist};
  cudaError_t l = cudaErrorInvalidValue;
  const bool fits = oz::contraction_fits(KpS, T);   // the check launch_oz_fwd makes before choosing an instance
  switch (inst) {
    case 0: if (T == 4 && fits) l = oz_fwd_t<4, EpiPhaseSliceRaw<4>>(0, a); break;
    case 1: if (T == 6 && fits) l = oz_fwd_t<6, EpiPhaseSliceRaw<6>>(0, a); break;
    case 2: if (T == 6 && fits) l = oz_fwd_t<6, EpiPhaseSliceFix<6>>(0, a); break;
    case 3: if (T == 6 && fits) l = oz_fwd_t<6, EpiPhaseSliceFix<6>, oz::TileCfg<80, 2, 20>>(0, a); break;
    case 4: l = launch_oz_fwd(0, a); break;
  }
  return finish(l, [&] {
    cudaError_t r = download(Tq, t, nt);
    return r == cudaSuccess ? download(sT, st, ns * 8) : r;
  });
}
