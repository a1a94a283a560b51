/* Head-tracked render of a real SH signal (NOT in the reference API): the sound field is rotated against the head
 * orientation of every tracker frame, then rendered with one static filter pair.
 *
 * out = binauralDecodeShTracked(in, wL, wR, rotations, hop, fade, compensateDelay)
 *   in            [numSamples x (order+1)^2], real SH signal (real basis, ACN order)
 *   wL, wR        [len x (order+1)^2], real (e.g. getEMagLsFilters, getLsFilters)
 *   rotations     [3 x 3 x numFrames]: head orientation of frame f (f-1)*hop+1 .. f*hop, the designers' convention
 *                 (the world direction of head-frame direction u is rotations(:,:,f) * u)
 *   hop           samples per tracker frame
 *   fade          optional, default hop: length of the blend of consecutive frames' rotations (0: hard switch)
 *   compensateDelay  optional, default false: as in binauralDecode
 * Binds emagls_binaural_decode_sh_tracked() (include/emagls_cuda.h, contract there).
 * Build where MATLAB exists:  mex -R2018a -I../include binauralDecodeShTracked.c -L../emagls_b200/lib -lemagls_cuda
 */
#include <stdlib.h>
#include "emagls_mex_common.h"

void mexFunction(int nlhs, mxArray* plhs[], int nrhs, const mxArray* prhs[]) {
  (void)nlhs;
  if (nrhs < 5) mexErrMsgIdAndTxt("eMagLS:nargin", "binauralDecodeShTracked needs at least 5 arguments");
  if (mxIsComplex(prhs[0]) || mxIsComplex(prhs[1]) || mxIsComplex(prhs[2]) || mxIsComplex(prhs[3]))
    mexErrMsgIdAndTxt("eMagLS:complex", "binauralDecodeShTracked takes real-basis SH signals and filters");
  const long long n = (long long)mxGetM(prhs[0]);
  const int ch = (int)mxGetN(prhs[0]);
  int order = 0;
  while ((order + 1) * (order + 1) < ch) ++order;
  if ((order + 1) * (order + 1) != ch) mexErrMsgIdAndTxt("eMagLS:size", "in must have (order+1)^2 columns");
  const int len = (int)mxGetM(prhs[1]);
  if ((int)mxGetN(prhs[1]) != ch || mxGetM(prhs[2]) != mxGetM(prhs[1]) || mxGetN(prhs[2]) != mxGetN(prhs[1]))
    mexErrMsgIdAndTxt("eMagLS:size", "size mismatch between input channels and decoding filters");
  const mwSize* rd = mxGetDimensions(prhs[3]);
  if (rd[0] != 3 || rd[1] != 3) mexErrMsgIdAndTxt("eMagLS:rotations", "rotations must be [3 x 3 x numFrames]");
  const long long nf = mxGetNumberOfDimensions(prhs[3]) > 2 ? (long long)rd[2] : 1;
  const int hop = (int)mxGetScalar(prhs[4]);
  const int fade = (nrhs > 5 && !mxIsEmpty(prhs[5])) ? (int)mxGetScalar(prhs[5]) : hop;
  const int comp = (nrhs > 6) && mxIsLogicalScalarTrue(prhs[6]);
  /* column-major 3x3 pages -> row-major [numFrames x 9] */
  const double* rm = mxGetDoubles(prhs[3]);
  double* rot = (double*)malloc((size_t)(nf > 0 ? nf : 1) * 9 * sizeof(double));
  long long f;
  int i, j;
  for (f = 0; f < nf; ++f)
    for (i = 0; i < 3; ++i)
      for (j = 0; j < 3; ++j) rot[f * 9 + i * 3 + j] = rm[f * 9 + j * 3 + i];
  const long long rows = comp ? n - len / 2 + 1 : n;
  plhs[0] = mxCreateDoubleMatrix((mwSize)(rows > 0 ? rows : 0), 2, mxREAL);
  const int rc = emagls_binaural_decode_sh_tracked(emx_handle(), mxGetDoubles(prhs[0]), n, order,
                                                   mxGetDoubles(prhs[1]), mxGetDoubles(prhs[2]), len, rot, nf, hop,
                                                   fade, 0, comp, mxGetDoubles(plhs[0]));
  free(rot);
  emx_check(rc);
}
