"""ctypes wrapper of tests/csrc/gram_harness.cu, the direct test entry to the Gram route's kernels (TEST INFRASTRUCTURE
ONLY).  `compile_harness` builds it for sm_100a into a directory the caller owns; the calls take and return NumPy arrays
(or, for `gram_chol_device`, torch CUDA tensors).  Every output array is returned whole: its sentinel-filled guard
region of `guard` elements follows the data."""
from __future__ import annotations

import ctypes as C
import os
import subprocess

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
SRC = os.path.join(ROOT, "tests", "csrc", "gram_harness.cu")


def compile_harness(out_dir: str) -> str:
    from emagls_b200 import build as b
    so = os.path.join(out_dir, "gram_harness.so")
    # -Bsymbolic: the harness calls its own copies of the library's functions.  The library is loaded RTLD_GLOBAL, so
    # without it, once the library is loaded in the same process, its definitions would take over some of the harness's
    # calls: kernels compiled into the harness would then reach the library's CUDA runtime, which does not know them.
    subprocess.run([b._nvcc(), *b.ARCH, "-O3", "-std=c++17", "-Xcompiler", "-fPIC", "-shared", "-Xlinker", "-Bsymbolic",
                    "-o", so, SRC], check=True, capture_output=True, text=True)
    return so


def _p(a):
    return None if a is None else a.ctypes.data_as(C.c_void_p)


def _c(a):
    """complex128 array as contiguous interleaved doubles"""
    return np.ascontiguousarray(np.asarray(a, np.complex128)).view(np.float64)


class Harness:
    def __init__(self, so: str):
        self.lib = lib = C.CDLL(so)
        ll, i, d, vp = C.c_longlong, C.c_int, C.c_double, C.c_void_p
        for name, args in (("gh_sm_count", []),
                           ("gh_gram_chol", [vp, vp, i, i, i, i, d, vp, vp, vp, ll]),
                           ("gh_gram_chol_device", [vp, vp, i, i, i, i, d, vp, vp, vp]),
                           ("gh_bwd", [i, i, vp, i, i, vp, i, vp, vp, i, i, i, i, vp, ll, ll, ll, i, i, ll, vp, ll, ll,
                                       i, i, i, vp, i, vp, vp, ll, i]),
                           ("gh_fwd_slice", [vp, i, i, vp, i, vp, i, i, i, i, vp, ll, ll, i, i, i, i, vp, vp, vp, ll,
                                             i])):
            f = getattr(lib, name)
            f.argtypes, f.restype = args, i

    def sm_count(self) -> int:
        return self.lib.gh_sm_count()

    def gram_chol(self, Gre, Gim, Mc, P, thr, copy_pb=True, guard=64):
        """launch_gram_chol on Gre, Gim [nbins * P, ne_ld] -> (err, Pb [nmat * Mc * Mc + guard] complex or None,
        sig [nmat + guard], fail [1 + nbins + guard])"""
        Gre, Gim = np.ascontiguousarray(Gre, np.float64), np.ascontiguousarray(Gim, np.float64)
        nmat, ne_ld = Gre.shape
        assert Gim.shape == Gre.shape and nmat % P == 0
        nbins = nmat // P
        Pb = np.empty(nmat * Mc * Mc + guard, np.complex128) if copy_pb else None
        sig = np.empty(nmat + guard)
        fail = np.empty(1 + nbins + guard, np.int32)
        err = self.lib.gh_gram_chol(_p(Gre), _p(Gim), Mc, P, ne_ld, nbins, thr, _p(Pb), _p(sig), _p(fail), guard)
        return err, Pb, sig, fail

    def gram_chol_device(self, Gre, Gim, Mc, P, thr, Pb, sig, fail):
        """launch_gram_chol on torch CUDA tensors Gre, Gim [nmat, ne_ld] (float64), Pb scratch (nmat * Mc * Mc
        complex128), sig [nmat] (float64), fail [1 + nbins] (int32) -> err"""
        nmat, ne_ld = Gre.shape
        assert Gre.is_contiguous() and Gim.is_contiguous() and nmat % P == 0
        return self.lib.gh_gram_chol_device(Gre.data_ptr(), Gim.data_ptr(), Mc, P, ne_ld, nmat // P, thr,
                                            Pb.data_ptr(), sig.data_ptr(), fail.data_ptr())

    def bwd(self, mode, T, c, Wsp, guard=256, fill=0x5A):
        """Backward step of the case `c` (see tests/test_gpu_gram_kernels.py: bwd_case) through `mode`
        (0: launch_bwd_small, 1: bwd_fused_kernel<T>, 2: bwd_small_kernel<T>), T in {0, 4, 6} -> (err, Wsp (complex,
        a copy of the given one updated), Cv_q [T * rows * KpS + guard] int8, sCv [rows + guard]); no digits and scales
        (None) at T = 0"""
        W = _c(Wsp).copy()
        rows = 4 * c["num_prob"]
        q = np.empty(T * rows * c["KpS"] + guard, np.int8)
        sc = np.empty(rows + guard)
        Y, bk, Pb, z, bkn = (np.ascontiguousarray(c["Y"], np.float64), _c(c["bk"]), _c(c["Pb"]),
                             np.ascontiguousarray(c["z"], np.float64), _c(c["bk_next"]))
        ro = np.ascontiguousarray(c["roword"], np.int32)
        err = self.lib.gh_bwd(mode, T, _p(Y), c["Mc"], c["S"], _p(ro), c["N"], _p(bk), _p(Pb), c["oc"], c["o0"],
                              c["num_orient"], c["num_prob"], _p(z), z.size, c["z_set_stride"], c["z_ear_stride"],
                              c["z_shared"], c["nsplit"], c["split_stride"], _p(W), W.size // 2, c["w_ear_stride"],
                              c["K"], c["k"], c["dc_fix"], _p(bkn), c["KpS"], _p(q), _p(sc), guard, fill)
        return (err, W.view(np.complex128), q, sc) if T else (err, W.view(np.complex128), None, None)

    def fwd_slice(self, T, c, Wsp, kprev, guard=256, fill=0x5A):
        """launch_fwd_small (b = c["bk_next"], W_kprev from Wsp), then launch_slice_rows -> (err, Cv [rows * S + guard],
        Cv_q [T * rows * KpS + guard] int8, sCv [rows + guard])"""
        W = _c(Wsp)
        rows, S = 4 * c["num_prob"], c["S"]
        cv = np.empty(rows * S + guard)
        q = np.empty(T * rows * c["KpS"] + guard, np.int8)
        sc = np.empty(rows + guard)
        Y, bkn = np.ascontiguousarray(c["Y"], np.float64), _c(c["bk_next"])
        ro = np.ascontiguousarray(c["roword"], np.int32)
        err = self.lib.gh_fwd_slice(_p(Y), c["Mc"], S, _p(ro), c["N"], _p(bkn), c["oc"], c["o0"], c["num_orient"],
                                    c["num_prob"], _p(W), W.size // 2, c["w_ear_stride"], c["K"], kprev, T, c["KpS"],
                                    _p(cv), _p(q), _p(sc), guard, fill)
        return err, cv, q, sc
