/* Head-tracked render (NOT in the reference API): binauralDecode with a filter bank whose page a head tracker picks
 * per frame, crossfading linearly between the pages of consecutive frames.
 *
 * out = binauralDecodeTracked(in, wL, wR, track, hop, fade, compensateDelay)
 *   in            [numSamples x numCh], real
 *   wL, wR        [len x numCh x numPages], real (the bank getEMagLs2FiltersBatch returns)
 *   track         page of every frame (1-based, MATLAB numbering); frame f covers samples (f-1)*hop+1 .. f*hop
 *   hop           samples per tracker frame
 *   fade          optional, default hop: crossfade length at the start of every frame (0: hard switch)
 *   compensateDelay  optional, default false: as in binauralDecode
 * Binds emagls_binaural_decode_tracked() (include/emagls_cuda.h, contract there).
 * Build where MATLAB exists:  mex -R2018a -I../include binauralDecodeTracked.c -L../emagls_b200/lib -lemagls_cuda
 */
#include <stdlib.h>
#include "emagls_mex_common.h"

void mexFunction(int nlhs, mxArray* plhs[], int nrhs, const mxArray* prhs[]) {
  (void)nlhs;
  if (nrhs < 5) mexErrMsgIdAndTxt("eMagLS:nargin", "binauralDecodeTracked needs at least 5 arguments");
  if (mxIsComplex(prhs[0]) || mxIsComplex(prhs[1]) || mxIsComplex(prhs[2]) || mxIsComplex(prhs[3]))
    mexErrMsgIdAndTxt("eMagLS:complex", "binauralDecodeTracked takes real signals, banks and tracks");
  const long long n = (long long)mxGetM(prhs[0]);
  const int ch = (int)mxGetN(prhs[0]);
  const mwSize* wd = mxGetDimensions(prhs[1]);
  const int len = (int)wd[0];
  const int pages = mxGetNumberOfDimensions(prhs[1]) > 2 ? (int)wd[2] : 1;
  if ((int)wd[1] != ch || mxGetNumberOfElements(prhs[2]) != mxGetNumberOfElements(prhs[1]))
    mexErrMsgIdAndTxt("eMagLS:size", "size mismatch between input channels and the filter bank");
  const int hop = (int)mxGetScalar(prhs[4]);
  const int fade = (nrhs > 5 && !mxIsEmpty(prhs[5])) ? (int)mxGetScalar(prhs[5]) : hop;
  const int comp = (nrhs > 6) && mxIsLogicalScalarTrue(prhs[6]);
  /* 1-based MATLAB page numbers -> 0-based int32 */
  const long long nf = (long long)mxGetNumberOfElements(prhs[3]);
  const double* tr = mxGetDoubles(prhs[3]);
  int32_t* track = (int32_t*)malloc((size_t)(nf > 0 ? nf : 1) * sizeof(int32_t));
  long long f;
  for (f = 0; f < nf; ++f) {
    const double v = tr[f];
    if (!(v >= 1.0 && v <= (double)pages) || v != (double)(long long)v) {
      free(track);
      mexErrMsgIdAndTxt("eMagLS:track", "track(%lld) must be an integer page number in 1..%d", f + 1, pages);
    }
    track[f] = (int32_t)(v - 1.0);
  }
  const long long rows = comp ? n - len / 2 + 1 : n;
  plhs[0] = mxCreateDoubleMatrix((mwSize)(rows > 0 ? rows : 0), 2, mxREAL);
  const int rc = emagls_binaural_decode_tracked(emx_handle(), mxGetDoubles(prhs[0]), n, ch, mxGetDoubles(prhs[1]),
                                                mxGetDoubles(prhs[2]), len, pages, track, nf, hop, fade, 0, comp,
                                                mxGetDoubles(plhs[0]));
  free(track);
  emx_check(rc);
}
