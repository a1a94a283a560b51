/* Render sessions (NOT in the reference API): the static, bank and SH head-tracked renders streamed block by block,
 * with the tracker entries supplied as the audio arrives.
 *
 * id  = binauralDecodeStream('create', wL, wR, block)                     static render, wL, wR [len x ch]
 * id  = binauralDecodeStream('create', wL, wR, block, hop, fade, L)       bank render, wL, wR [len x ch x pages]
 * id  = binauralDecodeStream('createSh', wL, wR, block, hop, fade, L)     SH render, wL, wR [len x (order+1)^2]
 * out = binauralDecodeStream('process', id, in, entries)
 *         in       [n x ch], n a multiple of block; out [n x 2 x L]
 *         entries  optional: the next tracker entries, appended before the call renders; bank sessions take page
 *                  numbers (1-based) [k x L], SH sessions rotations [3 x 3 x k x L] (the designers' convention)
 *         After the append the entries must cover every frame the call's samples fall in.
 * L (optional, default 1) is the number of listeners who hear the same input, each with their own entries.
 * binauralDecodeStream('destroy', id)
 * fade is optional (default hop).  The concatenated outputs of a session equal binauralDecode, binauralDecodeTracked
 * or binauralDecodeShTracked of the concatenated input (without compensateDelay: drop the first len/2 - 1 samples).
 * Sessions live in a table of this MEX file and are freed at mexAtExit (clear binauralDecodeStream).
 * Binds emagls_render_stream_*() (include/emagls_cuda.h, contract there).
 * Build where MATLAB exists:  mex -R2018a -I../include binauralDecodeStream.c -L../emagls_b200/lib -lemagls_cuda
 */
#include <stdlib.h>
#include "emagls_mex_common.h"

#define EMX_MAX_STREAMS 64

static emagls_render_stream g_streams[EMX_MAX_STREAMS];
static int g_kind[EMX_MAX_STREAMS];     /* 0 static, 1 bank, 2 SH */
static int g_ch[EMX_MAX_STREAMS];
static int g_nl[EMX_MAX_STREAMS];       /* listeners */

static void stream_at_exit(void) {
  int i;
  for (i = 0; i < EMX_MAX_STREAMS; ++i)
    if (g_streams[i]) { emagls_render_stream_destroy(g_streams[i]); g_streams[i] = NULL; }
  emx_at_exit();
}

static int stream_slot(const mxArray* a) {
  const int id = (int)mxGetScalar(a);
  if (id < 1 || id > EMX_MAX_STREAMS || !g_streams[id - 1])
    mexErrMsgIdAndTxt("eMagLS:stream", "not an open render session");
  return id - 1;
}

static mxArray* scalar(double v) {
  mxArray* a = mxCreateDoubleMatrix(1, 1, mxREAL);
  mxGetDoubles(a)[0] = v;
  return a;
}

void mexFunction(int nlhs, mxArray* plhs[], int nrhs, const mxArray* prhs[]) {
  char cmd[16] = "";
  (void)nlhs;
  if (nrhs < 1 || mxGetString(prhs[0], cmd, sizeof cmd) != 0)
    mexErrMsgIdAndTxt("eMagLS:nargin", "binauralDecodeStream needs a command");
  emagls_handle h = emx_handle();
  mexAtExit(stream_at_exit);
  if (strcmp(cmd, "create") == 0 || strcmp(cmd, "createSh") == 0) {
    const int sh = cmd[6] == 'S';
    if (nrhs < 4 + sh) mexErrMsgIdAndTxt("eMagLS:nargin", "binauralDecodeStream: too few arguments to create");
    if (mxIsComplex(prhs[1]) || mxIsComplex(prhs[2])) mexErrMsgIdAndTxt("eMagLS:complex", "filters must be real");
    const mwSize nd = mxGetNumberOfDimensions(prhs[1]);
    const mwSize* d = mxGetDimensions(prhs[1]);
    const mwSize* d2 = mxGetDimensions(prhs[2]);
    if (nd != mxGetNumberOfDimensions(prhs[2]) || d[0] != d2[0] || d[1] != d2[1] || (nd > 2 && d[2] != d2[2]))
      mexErrMsgIdAndTxt("eMagLS:size", "wL and wR differ in size");
    const int len = (int)d[0], ch = (int)d[1], pages = nd > 2 ? (int)d[2] : 1;
    const int block = (int)mxGetScalar(prhs[3]);
    const int hop = nrhs > 4 && !mxIsEmpty(prhs[4]) ? (int)mxGetScalar(prhs[4]) : 1;
    const int fade = nrhs > 5 && !mxIsEmpty(prhs[5]) ? (int)mxGetScalar(prhs[5]) : (nrhs > 4 ? hop : 0);
    const int nl = nrhs > 6 && !mxIsEmpty(prhs[6]) ? (int)mxGetScalar(prhs[6]) : 1;
    int slot = 0;
    while (slot < EMX_MAX_STREAMS && g_streams[slot]) ++slot;
    if (slot == EMX_MAX_STREAMS) mexErrMsgIdAndTxt("eMagLS:stream", "too many open render sessions");
    int rc;
    if (sh) {
      int order = 0;
      while ((order + 1) * (order + 1) < ch) ++order;
      if ((order + 1) * (order + 1) != ch || pages != 1)
        mexErrMsgIdAndTxt("eMagLS:size", "createSh takes wL, wR [len x (order+1)^2]");
      rc = emagls_render_stream_create_sh_listeners(h, mxGetDoubles(prhs[1]), mxGetDoubles(prhs[2]), len, order, nl,
                                                    block, hop, fade, &g_streams[slot]);
    } else {
      rc = emagls_render_stream_create_listeners(h, mxGetDoubles(prhs[1]), mxGetDoubles(prhs[2]), len, ch, pages, nl,
                                                 block, hop, fade, &g_streams[slot]);
    }
    emx_check(rc);
    g_kind[slot] = sh ? 2 : (pages > 1 ? 1 : 0);
    g_ch[slot] = ch;
    g_nl[slot] = nl;
    plhs[0] = scalar(slot + 1);
    return;
  }
  if (strcmp(cmd, "destroy") == 0) {
    if (nrhs < 2) mexErrMsgIdAndTxt("eMagLS:nargin", "binauralDecodeStream('destroy', id)");
    const int slot = stream_slot(prhs[1]);
    const int rc = emagls_render_stream_destroy(g_streams[slot]);
    g_streams[slot] = NULL;
    emx_check(rc);
    return;
  }
  if (strcmp(cmd, "process") != 0) mexErrMsgIdAndTxt("eMagLS:command", "unknown command");
  if (nrhs < 3) mexErrMsgIdAndTxt("eMagLS:nargin", "binauralDecodeStream('process', id, in[, entries])");
  const int slot = stream_slot(prhs[1]);
  if (mxIsComplex(prhs[2])) mexErrMsgIdAndTxt("eMagLS:complex", "in must be real");
  if ((int)mxGetN(prhs[2]) != g_ch[slot])
    mexErrMsgIdAndTxt("eMagLS:size", "size mismatch between input channels and the session's filters");
  const long long n = (long long)mxGetM(prhs[2]);
  const int has = nrhs > 3 && !mxIsEmpty(prhs[3]);
  const int nl = g_nl[slot];
  int32_t* trk = NULL;
  double* rot = NULL;
  long long k = 0, f;
  if (has && g_kind[slot] == 1) {
    const double* e = mxGetDoubles(prhs[3]);
    const long long ne = (long long)mxGetNumberOfElements(prhs[3]);
    if (nl > 1 && (long long)mxGetN(prhs[3]) != nl)
      mexErrMsgIdAndTxt("eMagLS:track", "the track must be [k x L]");
    k = ne / nl;
    trk = (int32_t*)malloc((size_t)ne * sizeof(int32_t));   /* [k x L] column-major: the C layout */
    for (f = 0; f < ne; ++f) trk[f] = (int32_t)e[f] - 1;
  } else if (has && g_kind[slot] == 2) {
    const mwSize nd = mxGetNumberOfDimensions(prhs[3]);
    const mwSize* rd = mxGetDimensions(prhs[3]);
    if (rd[0] != 3 || rd[1] != 3 || (nl > 1 && (nd != 4 || (int)rd[3] != nl)))
      mexErrMsgIdAndTxt("eMagLS:rotations", "rotations must be [3 x 3 x k x L]");
    k = nd > 2 ? (long long)rd[2] : 1;
    const double* rm = mxGetDoubles(prhs[3]);
    int i, j;
    rot = (double*)malloc((size_t)k * nl * 9 * sizeof(double));
    for (f = 0; f < k * nl; ++f)     /* column-major 3x3 pages -> row-major rows of 9, listener-major as in C */
      for (i = 0; i < 3; ++i)
        for (j = 0; j < 3; ++j) rot[f * 9 + i * 3 + j] = rm[f * 9 + j * 3 + i];
  } else if (has) {
    mexErrMsgIdAndTxt("eMagLS:stream", "a static session takes no tracker entries");
  }
  {
    const mwSize od[3] = {(mwSize)n, 2, (mwSize)nl};
    plhs[0] = mxCreateNumericArray(3, od, mxDOUBLE_CLASS, mxREAL);
  }
  const int rc = emagls_render_stream_process(g_streams[slot], mxGetDoubles(prhs[2]), n, trk, rot, k,
                                              mxGetDoubles(plhs[0]));
  free(trk);
  free(rot);
  emx_check(rc);
}
