/* MEX drop-in for lib/getMagLsFilters2D.m:1, binding emagls_design_magls_2d().
 * [wMlsL, wMlsR] = getMagLsFilters2D(hLHor, hRHor, horHrirGridAziRad, order, fs, len, chDefinition)
 * Build: mex -R2018a -I../include getMagLsFilters2D.c -L../emagls_b200/lib -lemagls_cuda   (needs MATLAB) */
#include "emagls_mex_common.h"

void mexFunction(int nlhs, mxArray* plhs[], int nrhs, const mxArray* prhs[]) {
  if (nrhs < 6) mexErrMsgIdAndTxt("eMagLS:nargin", "getMagLsFilters2D needs at least 6 arguments");
  emagls_config cfg; emagls_config_default(&cfg);
  cfg.basis = emx_basis(nrhs, prhs, 6);
  const int T = (int)mxGetM(prhs[0]), D = (int)mxGetN(prhs[0]);
  const int order = (int)mxGetScalar(prhs[3]), len = (int)mxGetScalar(prhs[5]), nch = 2 * order + 1;
  mxArray* wL = emx_out(len, nch, cfg.basis); mxArray* wR = emx_out(len, nch, cfg.basis);
  emx_check(emagls_design_magls_2d(emx_handle(), &cfg, mxGetDoubles(prhs[0]), mxGetDoubles(prhs[1]), T, D,
                                   mxGetDoubles(prhs[2]), order, mxGetScalar(prhs[4]), len, emx_ptr(wL), emx_ptr(wR),
                                   NULL));   /* 'len too short' on len < size(hLHor,1) */
  emx_return2(nlhs, plhs, wL, wR);
}
