"""ctypes wrapper of tests/csrc/ozaki_harness.cu, the direct test entry to every int8 tensor-core GEMM instance
(TEST INFRASTRUCTURE ONLY).  `compile_harness` builds it for sm_100a into a directory the caller owns; the calls take
and return NumPy arrays.  Every output array is returned whole: its sentinel-filled guard region of `guard` elements
follows the data."""
from __future__ import annotations

import ctypes as C
import os
import subprocess

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
SRC = os.path.join(ROOT, "tests", "csrc", "ozaki_harness.cu")

BWD_WIDTH = {0: 64, 1: 80, 2: 48}          # oh_bwd instance -> tile width; 3 = launch_oz_bwd
FWD_NAMES = {0: "raw4", 1: "raw6", 2: "fix6", 3: "fix6_nt80_w20", 4: "launch_oz_fwd"}


def compile_harness(out_dir: str) -> str:
    from emagls_b200 import build as b
    so = os.path.join(out_dir, "ozaki_harness.so")
    # -Bsymbolic: the harness calls its own copies of the library's functions.  The library is loaded RTLD_GLOBAL, so
    # without it, once the library is loaded in the same process, its definitions would take over some of the harness's
    # calls: kernels compiled into the harness would then reach the library's CUDA runtime, which does not know them.
    subprocess.run([b._nvcc(), *b.ARCH, "-O3", "-std=c++17", "-Xcompiler", "-fPIC", "-shared", "-Xlinker", "-Bsymbolic",
                    "-o", so, SRC], check=True, capture_output=True, text=True)
    return so


def _p(a):
    return a.ctypes.data_as(C.c_void_p)


class Harness:
    def __init__(self, so: str):
        self.lib = lib = C.CDLL(so)
        ll, i, vp = C.c_longlong, C.c_int, C.c_void_p
        for name, args in (("oh_sm_count", []), ("oh_contraction_fits", [i, i]), ("oh_drain_i64_fits", [i, i]),
                           ("oh_slice_rows", [vp, ll, ll, ll, i, i, i, i, i, vp, vp, ll, i]),
                           ("oh_row_scale", [vp, ll, i, vp, vp, ll]),
                           ("oh_bwd", [i, vp, vp, i, vp, vp, i, i, i, i, vp, ll]),
                           ("oh_fwd", [i, vp, vp, i, i, vp, vp, i, i, i, vp, i, vp, vp, ll, ll, ll, vp, vp, ll, i, i, i,
                                       ll, i])):
            f = getattr(lib, name)
            f.argtypes, f.restype = args, i

    def sm_count(self) -> int:
        return self.lib.oh_sm_count()

    def contraction_fits(self, Kpad: int, T: int) -> bool:
        return bool(self.lib.oh_contraction_fits(Kpad, T))

    def drain_i64_fits(self, Kpad: int, T: int) -> bool:
        return bool(self.lib.oh_drain_i64_fits(Kpad, T))

    def slice_rows(self, src, rs, cs, R, K, Kpad, T, Tbuf=None, guard=64, fill=0x5A):
        """launch_slice_rows -> (err, digits [Tbuf * R * Kpad + guard] int8, scales [R + guard])"""
        Tbuf = T if Tbuf is None else Tbuf
        src = np.ascontiguousarray(src, np.float64)
        out = np.empty(Tbuf * R * Kpad + guard, np.int8)
        sc = np.empty(R + guard, np.float64)
        err = self.lib.oh_slice_rows(_p(src), src.size, rs, cs, R, K, Kpad, T, Tbuf, _p(out), _p(sc), guard, fill)
        return err, out, sc

    def row_scale(self, x, guard=64):
        """launch_row_scale on the rows of x -> (err, up [rows + guard], sc [rows + guard])"""
        x = np.ascontiguousarray(x, np.float64)
        rows, D = x.shape
        up, sc = np.empty(rows + guard), np.empty(rows + guard)
        err = self.lib.oh_row_scale(_p(x), rows, D, _p(up), _p(sc), guard)
        return err, up, sc

    def bwd(self, inst, qA, sA, qB, sB, T, guard=64):
        """C = A B^T through backward instance `inst` -> (err, C [M * N + guard])"""
        qA, qB = np.ascontiguousarray(qA, np.int8), np.ascontiguousarray(qB, np.int8)
        sA, sB = np.ascontiguousarray(sA, np.float64), np.ascontiguousarray(sB, np.float64)
        Tbuf, M, Kpad = qA.shape
        N = qB.shape[1]
        out = np.empty(M * N + guard)
        err = self.lib.oh_bwd(inst, _p(qA), _p(sA), M, _p(qB), _p(sB), N, Kpad, T, Tbuf, _p(out), guard)
        return err, out

    def fwd(self, inst, c, T, nyquist, fill, guard=256):
        """forward product of the case `c` (see tests/test_gpu_ozaki.py: fwd_case) through instance `inst`
        -> (err, digits [Tbuf * rows * KpD + guard] int8, sT [rows + guard])"""
        qY, qC = np.ascontiguousarray(c["qY"], np.int8), np.ascontiguousarray(c["qC"], np.int8)
        Tbuf, D, KpS = qY.shape
        rows, KpD = qC.shape[1], c["KpD"]
        absH, up, sc = c["absH_bin"], c["up_bin"], c["sc_bin"]
        out = np.empty(Tbuf * rows * KpD + guard, np.int8)
        sT = np.empty(rows + guard)
        err = self.lib.oh_fwd(inst, _p(qY), _p(c["sY"]), D, KpS, _p(qC), _p(c["sC"]), rows, T, Tbuf, _p(out), KpD,
                              _p(sT), _p(absH), absH.size, c["abs_set_stride"], c["abs_ear_stride"], _p(up), _p(sc),
                              up.size, c["scale_stride"], c["orient_per_set"], int(nyquist), guard, fill)
        return err, out, sT
