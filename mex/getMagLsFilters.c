/* MEX drop-in for lib/getMagLsFilters.m:1-2, binding emagls_design_magls().
 * [wMlsL, wMlsR] = getMagLsFilters(hL, hR, hrirGridAziRad, hrirGridZenRad, order, fs, len, shDefinition, shFunction)
 * Build: mex -R2018a -I../include getMagLsFilters.c -L../emagls_b200/lib -lemagls_cuda   (needs MATLAB) */
#include "emagls_mex_common.h"

void mexFunction(int nlhs, mxArray* plhs[], int nrhs, const mxArray* prhs[]) {
  if (nrhs < 7) mexErrMsgIdAndTxt("eMagLS:nargin", "getMagLsFilters needs at least 7 arguments");
  emx_require_default_handle(nrhs, prhs, 8, "getSH");
  emagls_config cfg; emagls_config_default(&cfg);
  cfg.basis = emx_basis(nrhs, prhs, 7);
  const int T = (int)mxGetM(prhs[0]), D = (int)mxGetN(prhs[0]);
  const int order = (int)mxGetScalar(prhs[4]), len = (int)mxGetScalar(prhs[6]), nsh = (order + 1) * (order + 1);
  mxArray* wL = emx_out(len, nsh, cfg.basis); mxArray* wR = emx_out(len, nsh, cfg.basis);
  emx_check(emagls_design_magls(emx_handle(), &cfg, mxGetDoubles(prhs[0]), mxGetDoubles(prhs[1]), T, D,
                                mxGetDoubles(prhs[2]), mxGetDoubles(prhs[3]), order, mxGetScalar(prhs[5]), len,
                                emx_ptr(wL), emx_ptr(wR), NULL));   /* 'len too short' on len < size(hL,1) */
  emx_return2(nlhs, plhs, wL, wR);
}
