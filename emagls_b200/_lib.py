"""ctypes binding of libemagls_cuda.so (the C ABI declared in include/emagls_cuda.h).

There is no CPU fallback: if the shared library is missing or a CUDA device is absent the
product path raises.
"""
from __future__ import annotations

import ctypes as C
import os

_HERE = os.path.dirname(os.path.abspath(__file__))
# EMAGLS_LIB_PATH: A/B runs of alternative builds of the same library (tools/); never a fallback
LIB_PATH = os.environ.get("EMAGLS_LIB_PATH") or os.path.join(_HERE, "lib", "libemagls_cuda.so")

c_dp = C.c_void_p  # double* / const double*


class Config(C.Structure):
    """struct emagls_config (include/emagls_cuda.h)."""
    _fields_ = [("nfft_max_len", C.c_int), ("f_cut_min", C.c_double), ("svd_regul", C.c_double),
                ("speed_of_sound", C.c_double), ("array_type", C.c_int), ("basis", C.c_int),
                ("precision", C.c_int), ("diffuseness_const", C.c_int), ("reserved", C.c_int * 4)]


class RadialParams(C.Structure):
    """struct emagls_radial_params (include/emagls_cuda.h)."""
    _fields_ = [("kind", C.c_int), ("regul_const", C.c_double), ("noise_gain_db", C.c_double),
                ("array_type", C.c_int)]


_DESIGN_ARGS = [C.c_void_p, C.POINTER(Config), c_dp, c_dp, C.c_int, C.c_int, c_dp, c_dp, C.c_double, c_dp, c_dp,
                C.c_int, C.c_int, C.c_double, C.c_int, C.c_int, C.c_int, c_dp, c_dp, c_dp, c_dp]

SIGNATURES = {
    "emagls_create": (C.c_int, [C.c_int, C.POINTER(C.c_void_p)]),
    "emagls_destroy": (C.c_int, [C.c_void_p]),
    "emagls_last_error": (C.c_char_p, [C.c_void_p]),
    "emagls_config_default": (None, [C.POINTER(Config)]),
    "emagls_launch_count": (C.c_longlong, [C.c_void_p]),
    "emagls_stream": (C.c_void_p, [C.c_void_p]),
    "emagls_stats_read": (C.c_int, [C.c_void_p, C.POINTER(C.c_longlong), C.c_int]),
    "emagls_profile_enable": (C.c_int, [C.c_void_p, C.c_int]),
    "emagls_profile_read": (C.c_int, [C.c_void_p, C.POINTER(C.c_double), C.POINTER(C.c_longlong), C.c_int]),
    "emagls_design_emagls2": (C.c_int, _DESIGN_ARGS),
    "emagls_design_emagls2_dev": (C.c_int, _DESIGN_ARGS),
    "emagls_design_emagls": (C.c_int, _DESIGN_ARGS),
    "emagls_design_sma_basis": (C.c_int, [C.c_void_p, C.POINTER(Config), C.c_int, c_dp, c_dp, C.c_int, C.c_int, c_dp,
                                          C.c_int, C.c_double, c_dp, C.c_int, C.c_int, C.c_double, C.c_int, C.c_int,
                                          C.c_int, c_dp, c_dp, c_dp]),
    "emagls_design_magls": (C.c_int, [C.c_void_p, C.POINTER(Config), c_dp, c_dp, C.c_int, C.c_int, c_dp, c_dp,
                                      C.c_int, C.c_double, C.c_int, c_dp, c_dp, c_dp]),
    "emagls_design_magls_batch": (C.c_int, [C.c_void_p, C.POINTER(Config), c_dp, c_dp, C.c_int, C.c_int, c_dp, c_dp,
                                            C.c_int, C.c_double, C.c_int, C.c_int, c_dp, c_dp, c_dp]),
    "emagls_design_ls": (C.c_int, [C.c_void_p, C.POINTER(Config), c_dp, c_dp, C.c_int, C.c_int, c_dp, c_dp,
                                   C.c_int, c_dp, c_dp]),
    "emagls_design_from_atf": (C.c_int, [C.c_void_p, C.POINTER(Config), c_dp, c_dp, C.c_int, C.c_int, c_dp, c_dp,
                                         C.c_int, C.c_int, C.c_int, c_dp, C.c_double, C.c_int, C.c_double,
                                         c_dp, c_dp, c_dp, c_dp]),
    "emagls_design_from_atf_batch": (C.c_int, [C.c_void_p, C.POINTER(Config), c_dp, c_dp, C.c_int, C.c_int, c_dp, c_dp,
                                               C.c_int, C.c_int, C.c_int, c_dp, C.c_double, C.c_int, C.c_double,
                                               C.c_int, c_dp, c_dp, c_dp, c_dp, c_dp]),
    "emagls_design_from_atf_batch_dev": (C.c_int, [C.c_void_p, C.POINTER(Config), c_dp, c_dp, C.c_int, C.c_int, c_dp,
                                                   c_dp, C.c_int, C.c_int, C.c_int, c_dp, C.c_double, C.c_int,
                                                   C.c_double, C.c_int, c_dp, c_dp, c_dp, c_dp]),
    "emagls_design_ema_ch": (C.c_int, [C.c_void_p, C.POINTER(Config), c_dp, c_dp, C.c_int, C.c_int, c_dp, c_dp,
                                       C.c_double, c_dp, C.c_int, C.c_int, C.c_double, C.c_int, c_dp, c_dp, c_dp]),
    "emagls_design_ema_ch_batch": (C.c_int, [C.c_void_p, C.POINTER(Config), c_dp, c_dp, C.c_int, C.c_int, c_dp, c_dp,
                                             C.c_double, c_dp, C.c_int, C.c_int, C.c_double, C.c_int, C.c_int, C.c_int,
                                             c_dp, c_dp, c_dp, c_dp]),
    "emagls_design_ema_sh": (C.c_int, [C.c_void_p, C.POINTER(Config), c_dp, c_dp, C.c_int, C.c_int, c_dp, c_dp,
                                       C.c_double, c_dp, C.c_int, C.c_int, C.c_double, C.c_int, c_dp, c_dp, c_dp]),
    "emagls_smair_matrix": (C.c_int, [C.c_void_p, C.POINTER(Config), c_dp, c_dp, C.c_int, C.c_int, C.c_double,
                                      C.c_double, C.c_int, C.c_int, c_dp, C.POINTER(C.c_int)]),
    "emagls_binaural_decode": (C.c_int, [C.c_void_p, c_dp, C.c_longlong, C.c_int, c_dp, c_dp, C.c_int, C.c_int, c_dp]),
    "emagls_binaural_decode_dev": (C.c_int, [C.c_void_p, c_dp, C.c_longlong, C.c_int, c_dp, c_dp, C.c_int, C.c_int,
                                             c_dp]),
    "emagls_binaural_decode_tracked": (C.c_int, [C.c_void_p, c_dp, C.c_longlong, C.c_int, c_dp, c_dp, C.c_int, C.c_int,
                                                 C.c_void_p, C.c_longlong, C.c_int, C.c_int, C.c_longlong, C.c_int,
                                                 c_dp]),
    "emagls_binaural_decode_tracked_dev": (C.c_int, [C.c_void_p, c_dp, C.c_longlong, C.c_int, c_dp, c_dp, C.c_int,
                                                     C.c_int, C.c_void_p, C.c_longlong, C.c_int, C.c_int, C.c_longlong,
                                                     C.c_int, c_dp]),
    "emagls_binaural_decode_sh_tracked": (C.c_int, [C.c_void_p, c_dp, C.c_longlong, C.c_int, c_dp, c_dp, C.c_int, c_dp,
                                                    C.c_longlong, C.c_int, C.c_int, C.c_longlong, C.c_int, c_dp]),
    "emagls_binaural_decode_sh_tracked_dev": (C.c_int, [C.c_void_p, c_dp, C.c_longlong, C.c_int, c_dp, c_dp, C.c_int,
                                                        c_dp, C.c_longlong, C.c_int, C.c_int, C.c_longlong, C.c_int,
                                                        c_dp]),
    "emagls_render_stream_create": (C.c_int, [C.c_void_p, c_dp, c_dp, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int,
                                              C.c_int, C.POINTER(C.c_void_p)]),
    "emagls_render_stream_create_sh": (C.c_int, [C.c_void_p, c_dp, c_dp, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int,
                                                 C.POINTER(C.c_void_p)]),
    "emagls_render_stream_create_listeners": (C.c_int, [C.c_void_p, c_dp, c_dp, C.c_int, C.c_int, C.c_int, C.c_int,
                                                        C.c_int, C.c_int, C.c_int, C.POINTER(C.c_void_p)]),
    "emagls_render_stream_create_sh_listeners": (C.c_int, [C.c_void_p, c_dp, c_dp, C.c_int, C.c_int, C.c_int, C.c_int,
                                                           C.c_int, C.c_int, C.POINTER(C.c_void_p)]),
    "emagls_render_stream_process": (C.c_int, [C.c_void_p, c_dp, C.c_longlong, C.c_void_p, c_dp, C.c_longlong, c_dp]),
    "emagls_render_stream_process_dev": (C.c_int, [C.c_void_p, c_dp, C.c_longlong, C.c_void_p, c_dp, C.c_longlong,
                                                   c_dp]),
    "emagls_render_stream_destroy": (C.c_int, [C.c_void_p]),
    "emagls_get_sh": (C.c_int, [C.c_void_p, C.c_int, c_dp, c_dp, C.c_int, C.c_int, c_dp]),
    "emagls_group_delay": (C.c_int, [C.c_void_p, c_dp, C.c_int, C.c_int, C.c_int, C.c_double, c_dp, c_dp]),
    "emagls_sph_modal_coeffs": (C.c_int, [C.c_void_p, C.c_int, c_dp, C.c_int, C.c_int, c_dp]),
    "emagls_regularized_apply": (C.c_int, [C.c_void_p, c_dp, C.c_int, C.c_int, c_dp, C.c_int, C.c_double, c_dp]),
    # ---- SURVEY.md section 8(f) rows (frontend.cu)
    "emagls_radial_params_default": (None, [C.POINTER(RadialParams)]),
    "emagls_radial_filter": (C.c_int, [C.c_void_p, C.POINTER(Config), C.POINTER(RadialParams), C.c_int, C.c_double,
                                       C.c_double, C.c_int, c_dp]),
    "emagls_apply_radial_filter_rows": (C.c_longlong, [C.c_longlong, C.c_int]),
    "emagls_apply_radial_filter": (C.c_int, [C.c_void_p, C.POINTER(Config), C.POINTER(RadialParams), c_dp,
                                             C.c_longlong, C.c_int, C.c_double, C.c_double, C.c_int, c_dp]),
    "emagls_apply_radial_filter_dev": (C.c_int, [C.c_void_p, C.POINTER(Config), C.POINTER(RadialParams), c_dp,
                                                 C.c_longlong, C.c_int, C.c_double, C.c_double, C.c_int, c_dp]),
    "emagls_smair_matrix_radial": (C.c_int, [C.c_void_p, C.POINTER(Config), C.POINTER(RadialParams), c_dp, c_dp,
                                             C.c_int, C.c_int, C.c_double, C.c_double, C.c_int, c_dp,
                                             C.POINTER(C.c_int)]),
    "emagls_sh_encode": (C.c_int, [C.c_void_p, C.POINTER(Config), c_dp, C.c_longlong, C.c_int, c_dp, c_dp, C.c_int,
                                   c_dp]),
    "emagls_sh_encode_dev": (C.c_int, [C.c_void_p, C.POINTER(Config), c_dp, C.c_longlong, C.c_int, c_dp, c_dp,
                                       C.c_int, c_dp]),
    "emagls_ch_encode": (C.c_int, [C.c_void_p, C.POINTER(Config), c_dp, C.c_longlong, C.c_int, c_dp, C.c_int, c_dp]),
    "emagls_rotate_sh": (C.c_int, [C.c_void_p, c_dp, C.c_longlong, C.c_int, C.c_double, C.c_double, C.c_double,
                                   c_dp]),
    "emagls_rotate_sh_dev": (C.c_int, [C.c_void_p, c_dp, C.c_longlong, C.c_int, C.c_double, C.c_double, C.c_double,
                                       c_dp]),
    "emagls_design_magls_2d": (C.c_int, [C.c_void_p, C.POINTER(Config), c_dp, c_dp, C.c_int, C.c_int, c_dp, C.c_int,
                                         C.c_double, C.c_int, c_dp, c_dp, c_dp]),
    "emagls_spherical_head_filter": (C.c_int, [C.c_void_p, C.POINTER(Config), C.c_double, C.c_int, C.c_double,
                                               C.c_int, c_dp, c_dp]),
    "emagls_array_diffuse_filter": (C.c_int, [C.c_void_p, C.POINTER(Config), C.c_double, c_dp, c_dp, C.c_int,
                                              C.c_int, C.c_double, C.c_int, c_dp]),
}

_lib = None


def load():
    """Load libemagls_cuda.so and attach prototypes; raises if it has not been built."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise RuntimeError(
            f"{LIB_PATH} is missing: build it with `python -m emagls_b200.build` "
            "(there is no CPU fallback for the eMagLS hot path)")
    lib = C.CDLL(LIB_PATH, mode=C.RTLD_GLOBAL)
    for name, (res, args) in SIGNATURES.items():
        fn = getattr(lib, name)  # AttributeError if the symbol is not exported
        fn.restype = res
        fn.argtypes = args
    _lib = lib
    return lib


class EmaglsError(RuntimeError):
    def __init__(self, code, msg):
        super().__init__(f"libemagls_cuda error {code}: {msg}")
        self.code = code
        self.msg = msg


class Handle:
    """RAII wrapper of emagls_handle (one per GPU / rank)."""

    def __init__(self, device: int = 0):
        self.lib = load()
        self._h = C.c_void_p()
        rc = self.lib.emagls_create(int(device), C.byref(self._h))
        if rc != 0 or not self._h:
            raise EmaglsError(rc, f"emagls_create(device={device}) failed: no usable CUDA device "
                                  "(the eMagLS hot path has no CPU fallback)")
        self.device = device

    def close(self):
        if getattr(self, "_h", None):
            self.lib.emagls_destroy(self._h)
            self._h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    @property
    def ptr(self):
        return self._h

    def check(self, rc: int):
        if rc != 0:
            msg = self.lib.emagls_last_error(self._h)
            raise EmaglsError(rc, msg.decode() if msg else "?")

    def default_config(self) -> Config:
        cfg = Config()
        self.lib.emagls_config_default(C.byref(cfg))
        return cfg

    PROF_CLASSES = ("setup", "factor", "chain_fwd", "gemm_fwd", "gemm_bwd", "chain_bwd", "tail",
                    "render_mac", "render_fft", "render_stage", "gram", "jacobi")

    def profile(self, on: bool = True):
        self.check(self.lib.emagls_profile_enable(self._h, 1 if on else 0))

    def profile_read(self, reset: bool = True) -> dict:
        n = len(self.PROF_CLASSES)
        ms = (C.c_double * n)()
        cnt = (C.c_longlong * n)()
        got = self.lib.emagls_profile_read(self._h, ms, cnt, 1 if reset else 0)
        if got != n:
            raise EmaglsError(got, "emagls_profile_read")
        return {k: dict(ms=ms[i], n=int(cnt[i])) for i, k in enumerate(self.PROF_CLASSES)}

    def stats_read(self, reset: bool = True) -> dict:
        out = (C.c_longlong * 4)()
        self.check(self.lib.emagls_stats_read(self._h, out, 1 if reset else 0))
        return dict(tsqr_problem_bins=int(out[0]), gram_problem_bins=int(out[1]), jacobi_problems=int(out[2]),
                    jacobi_sweeps=int(out[3]))

    @property
    def launches(self) -> int:
        return int(self.lib.emagls_launch_count(self._h))

    @property
    def stream(self) -> int:
        return int(self.lib.emagls_stream(self._h) or 0)


_default_handles = {}


def default_handle(device: int = 0) -> Handle:
    if device not in _default_handles:
        _default_handles[device] = Handle(device)
    return _default_handles[device]
