"""Host-side mirror of the reference's MATLAB interface for the eMagLS hot path.

Same function names, positional argument order, argument meaning and error behaviour as the
reference (lib/get*Filters*.m, dependencies/getSMAIRMatrix.m, dependencies/binauralDecode.m);
every call goes through the C ABI of libemagls_cuda (include/emagls_cuda.h).  Arrays follow the
MATLAB conventions: impulse responses ``[samples, dirs]`` (optionally ``[samples, dirs, sets]``),
filters ``[taps, channels]`` (batched: ``[taps, channels, batch]``), grids in radians.

Deviations from the reference interface, all explicit:
* ``shFunction`` / ``chFunction`` handles other than the default ``getSH`` / ``getCH`` are not
  accepted (a CUDA library cannot call back into host code; SURVEY.md H8).
* keyword-only batch extensions: ``rotations`` ([B,3,3], world direction of grid direction u is
  R u), ``handle``, ``config``, ``return_spectra``.
"""
from __future__ import annotations

import ctypes as C

import numpy as np

from . import _lib
from ._lib import Config, EmaglsError, Handle, RadialParams, default_handle  # noqa: F401

__all__ = ["getEMagLs2Filters", "getEMagLsFilters", "getMagLsFilters", "getLsFilters",
           "getEMagLsFiltersFromAtf", "getEMagLsFiltersEMAinCH", "getEMagLsFiltersEMAinSH",
           "getSMAIRMatrix", "binauralDecode", "binauralDecodeTracked", "getSH", "sphModalCoeffs", "regularizedApply", "grpdelay",
           "getRadialFilter", "applyRadialFilter", "encodeSH", "encodeCH", "rotateSH", "getMagLsFilters2D",
           "getMagLsSphericalHeadFilter", "getMagLsArrayDiffuseFilter", "Handle", "EmaglsError"]


def _f(x):
    x = np.asarray(x)
    if np.iscomplexobj(x):
        # never drop an imaginary part silently (numpy's cast only warns); callers that accept complex data
        # split it explicitly (binauralDecode)
        raise ValueError("complex input where the reference interface expects real data")
    return np.asfortranarray(x, dtype=np.float64)


def _p(a):
    return a.ctypes.data_as(C.c_void_p) if a is not None else None


def _vec(x):
    return np.ascontiguousarray(np.asarray(x, dtype=np.float64).ravel())


def _basis(shDefinition):
    if shDefinition is None or shDefinition == "real":
        return 0
    if shDefinition == "complex":
        return 1
    raise ValueError("shDefinition must be 'real' or 'complex'")


def _check_sh_function(shFunction):
    if shFunction is not None and shFunction is not getSH:
        raise NotImplementedError("only the default shFunction (@getSH) is evaluated on the device")


def _is_custom(shFunction):
    return shFunction is not None and shFunction is not getSH


def _rotated_angles(azi, zen, R):
    """Angles of R^T u for the unit vectors u(azi, zen): microphone positions seen from head orientation R."""
    u = np.stack([np.sin(zen) * np.cos(azi), np.sin(zen) * np.sin(azi), np.cos(zen)], 1)
    v = u @ np.asarray(R, dtype=np.float64).reshape(3, 3)          # rows: (R^T u)^T = u^T R
    return np.arctan2(v[:, 1], v[:, 0]), np.arccos(np.clip(v[:, 2], -1.0, 1.0))


def _design_sma_custom(fn_name, h, cfg, shFunction, shDefinition, hL, hR, T, D, sets, az, ze, micRadius, maz, mze,
                       order, fs, length, rot, B, Mc, return_spectra):
    """Custom shFunction handle (lib/getEMagLs2Filters.m:32): evaluated here on the host, the two basis matrices
    go down through emagls_design_sma_basis (SURVEY.md H8)."""
    if _basis(shDefinition) != 0:
        raise NotImplementedError("custom shFunction handles are supported for shDefinition = 'real'")
    simN = max(int(order), int(np.ceil(float(fs) * np.pi * float(micRadius) / cfg.speed_of_sound)))
    S = (simN + 1) ** 2
    Yh = np.asfortranarray(np.asarray(shFunction(simN, np.stack([az, ze], 1), "real"), dtype=np.float64))
    if Yh.shape != (D, S):
        raise ValueError("shFunction must return [directions, (order+1)^2]")
    Ym = np.zeros((maz.size, S, B), order="F")
    for o in range(B):
        a_o, z_o = (maz, mze) if rot is None else _rotated_angles(maz, mze, rot[o])
        Ym[:, :, o] = np.asarray(shFunction(simN, np.stack([a_o, z_o], 1), "real"), dtype=np.float64)
    P = sets * B
    K = min(cfg.nfft_max_len, 2 * length) // 2 + 1
    wL = np.zeros((length, Mc, P), order="F")
    wR = np.zeros((length, Mc, P), order="F")
    sp = np.zeros((K, Mc, P, 2), dtype=np.complex128, order="F") if return_spectra else None
    h.check(h.lib.emagls_design_sma_basis(h.ptr, C.byref(cfg), 0 if fn_name == "emagls_design_emagls2" else 1, _p(hL),
                                          _p(hR), T, D, _p(Yh), S, float(micRadius), _p(Ym), maz.size, int(order),
                                          float(fs), length, sets, B, _p(wL), _p(wR), _p(sp)))
    return wL, wR, sp


def _config(handle, config, shDefinition, applyDiffusenessConst=False):
    # a private copy: the caller's Config is never written to
    cfg = Config.from_buffer_copy(config) if config is not None else handle.default_config()
    cfg.basis = _basis(shDefinition)
    if applyDiffusenessConst:
        if cfg.basis != 0:   # as the reference did (CHANGELOG.md:18)
            raise NotImplementedError('the diffuseness constraint is not implemented for "complex" SH conventions')
        cfg.diffuseness_const = 1
    return cfg


def _prep_hrirs(hL, hR):
    hL, hR = _f(hL), _f(hR)
    if hL.shape != hR.shape:
        raise ValueError("hL and hR must have the same size")
    if hL.ndim == 2:
        sets = 1
    elif hL.ndim == 3:
        sets = hL.shape[2]
    else:
        raise ValueError("hL/hR must be [samples, dirs] or [samples, dirs, sets]")
    return hL, hR, hL.shape[0], hL.shape[1], sets


def _design_sma(fn_name, channels_of, hL, hR, hrirGridAziRad, hrirGridZenRad, micRadius, micGridAziRad,
                micGridZenRad, order, fs, length, shDefinition, shFunction, rotations, handle, config,
                return_spectra, out=None, applyDiffusenessConst=False):
    h = handle or default_handle()
    cfg = _config(h, config, shDefinition, applyDiffusenessConst)
    hL, hR, T, D, sets = _prep_hrirs(hL, hR)
    az, ze = _vec(hrirGridAziRad), _vec(hrirGridZenRad)
    maz, mze = _vec(micGridAziRad), _vec(micGridZenRad)
    if az.size != D or ze.size != D:
        raise ValueError("HRIR grid size does not match hL")
    if maz.size != mze.size:
        raise ValueError("microphone grid sizes differ")
    if rotations is None:
        rot, B = None, 1
    else:
        rot = np.ascontiguousarray(np.asarray(rotations, dtype=np.float64).reshape(-1, 9))
        B = rot.shape[0]
    M = maz.size
    Mc = channels_of(M, int(order))
    length = int(length)
    P = sets * B
    nfft = min(cfg.nfft_max_len, 2 * length)
    K = nfft // 2 + 1
    cplx_out = cfg.basis == 1 and fn_name != "emagls_design_emagls2"
    odt = np.complex128 if cplx_out else np.float64
    if _is_custom(shFunction):
        if out is not None:
            raise ValueError("out buffers are not supported together with a custom shFunction")
        wL, wR, sp = _design_sma_custom(fn_name, h, cfg, shFunction, shDefinition, hL, hR, T, D, sets, az, ze, micRadius,
                                        maz, mze, order, fs, length, None if rot is None else rot.reshape(-1, 3, 3), B,
                                        Mc, return_spectra)
        if P == 1 and rotations is None and sets == 1:
            wL, wR = wL[:, :, 0], wR[:, :, 0]
            if sp is not None:
                sp = sp[:, :, 0, :]
        return (wL, wR, sp) if return_spectra else (wL, wR)
    if out is not None:  # caller-provided (e.g. pinned) Fortran-ordered [len, Mc, P] buffers
        wL, wR = out
        for w in (wL, wR):
            if w.shape != (length, Mc, P) or w.dtype != odt or not w.flags.f_contiguous:
                raise ValueError("out buffers must be Fortran-ordered [len, channels, batch]")
    else:
        wL = np.zeros((length, Mc, P), dtype=odt, order="F")
        wR = np.zeros((length, Mc, P), dtype=odt, order="F")
    sp = np.zeros((K, Mc, P, 2), dtype=np.complex128, order="F") if return_spectra else None
    rc = getattr(h.lib, fn_name)(h.ptr, C.byref(cfg), _p(hL), _p(hR), T, D, _p(az), _p(ze), float(micRadius),
                                 _p(maz), _p(mze), M, int(order), float(fs), length, sets, B, _p(rot),
                                 _p(wL), _p(wR), _p(sp))
    h.check(rc)
    if P == 1 and rotations is None and sets == 1 and out is None:
        wL, wR = wL[:, :, 0], wR[:, :, 0]
        if sp is not None:
            sp = sp[:, :, 0, :]
    return (wL, wR, sp) if return_spectra else (wL, wR)


def getEMagLs2Filters(hL, hR, hrirGridAziRad, hrirGridZenRad, micRadius, micGridAziRad, micGridZenRad,
                      order, fs, len, shDefinition="real", shFunction=None, *, rotations=None,
                      handle=None, config=None, return_spectra=False, out=None, applyDiffusenessConst=False):
    """[wMlsL, wMlsR] = getEMagLs2Filters(...)  -- lib/getEMagLs2Filters.m:1-2.

    Returns filters ``[len, numMics]`` (``[len, numMics, batch]`` when batched).  With
    ``return_spectra`` also the positive-frequency solutions ``[K, numMics, (batch,) 2]``.
    ``applyDiffusenessConst`` (extension, default off): the diffuse-field covariance constraint of earlier
    reference versions (CHANGELOG.md:10-18), see include/emagls_cuda.h ``diffuseness_const``.
    """
    return _design_sma("emagls_design_emagls2", lambda M, N: M, hL, hR, hrirGridAziRad, hrirGridZenRad,
                       micRadius, micGridAziRad, micGridZenRad, order, fs, len, shDefinition, shFunction,
                       rotations, handle, config, return_spectra, out, applyDiffusenessConst)


def getEMagLsFilters(hL, hR, hrirGridAziRad, hrirGridZenRad, micRadius, micGridAziRad, micGridZenRad,
                     order, fs, len, shDefinition="real", shFunction=None, *, rotations=None,
                     handle=None, config=None, return_spectra=False, applyDiffusenessConst=False):
    """[wMlsL, wMlsR] = getEMagLsFilters(...)  -- lib/getEMagLsFilters.m:1-2 ([len, (order+1)^2])."""
    return _design_sma("emagls_design_emagls", lambda M, N: (N + 1) ** 2, hL, hR, hrirGridAziRad,
                       hrirGridZenRad, micRadius, micGridAziRad, micGridZenRad, order, fs, len, shDefinition,
                       shFunction, rotations, handle, config, return_spectra, None, applyDiffusenessConst)


def getMagLsFilters(hL, hR, hrirGridAziRad, hrirGridZenRad, order, fs, len, shDefinition="real",
                    shFunction=None, *, handle=None, config=None, return_spectra=False):
    """[wMlsL, wMlsR] = getMagLsFilters(...)  -- lib/getMagLsFilters.m:1-2."""
    _check_sh_function(shFunction)
    h = handle or default_handle()
    cfg = _config(h, config, shDefinition)
    hL, hR, T, D, sets = _prep_hrirs(hL, hR)
    az, ze = _vec(hrirGridAziRad), _vec(hrirGridZenRad)
    H = (int(order) + 1) ** 2
    nfft = min(cfg.nfft_max_len, 2 * int(len))
    K = nfft // 2 + 1
    odt = np.complex128 if cfg.basis == 1 else np.float64
    batched = hL.ndim == 3          # [samples, dirs, sets]: keyword-free batch extension over HRTF sets
    wL = np.zeros((int(len), H, sets), dtype=odt, order="F")
    wR = np.zeros((int(len), H, sets), dtype=odt, order="F")
    sp = np.zeros((K, H, sets, 2), dtype=np.complex128, order="F") if return_spectra else None
    h.check(h.lib.emagls_design_magls_batch(h.ptr, C.byref(cfg), _p(hL), _p(hR), T, D, _p(az), _p(ze), int(order),
                                            float(fs), int(len), sets, _p(wL), _p(wR), _p(sp)))
    if not batched:
        wL, wR = wL[:, :, 0], wR[:, :, 0]
        if sp is not None:
            sp = sp[:, :, 0, :]
    return (wL, wR, sp) if return_spectra else (wL, wR)


def getLsFilters(hL, hR, hrirGridAziRad, hrirGridZenRad, order, shDefinition="real", shFunction=None, *,
                 handle=None, config=None):
    """[wLsL, wLsR] = getLsFilters(...)  -- lib/getLsFilters.m:1-2 ([numSamples, (order+1)^2])."""
    _check_sh_function(shFunction)
    h = handle or default_handle()
    cfg = _config(h, config, shDefinition)
    hL, hR, T, D, sets = _prep_hrirs(hL, hR)
    az, ze = _vec(hrirGridAziRad), _vec(hrirGridZenRad)
    H = (int(order) + 1) ** 2
    odt = np.complex128 if cfg.basis == 1 else np.float64
    wL = np.zeros((T, H), dtype=odt, order="F")
    wR = np.zeros((T, H), dtype=odt, order="F")
    h.check(h.lib.emagls_design_ls(h.ptr, C.byref(cfg), _p(hL), _p(hR), T, D, _p(az), _p(ze), int(order),
                                   _p(wL), _p(wR)))
    return wL, wR


def getEMagLsFiltersFromAtf(hL, hR, hrirGridAziZenRad, atfIrs, atfGridAziZenRad, fs, filterLen, fTrans, *,
                            rotations=None, handle=None, config=None, return_spectra=False, return_info=False):
    """[wMlsL, wMlsR] = getEMagLsFiltersFromAtf(...)  -- lib/getEMagLsFiltersFromAtf.m:1.

    ``rotations`` ([B,3,3], keyword-only batch extension): page b of the ``[filterLen, numMics, B]`` outputs equals
    one reference call with ``hrirGridAziZenRad`` rotated by ``rotations[b]``."""
    h = handle or default_handle()
    cfg = _config(h, config, "real")
    hL, hR, T, D, sets = _prep_hrirs(hL, hR)
    if sets != 1:
        raise ValueError("getEMagLsFiltersFromAtf takes one HRTF set")
    hg = _f(np.asarray(hrirGridAziZenRad, dtype=np.float64).reshape(-1, 2))
    atf = _f(atfIrs)
    ag = _f(np.asarray(atfGridAziZenRad, dtype=np.float64).reshape(-1, 2))
    Ta, M, Da = atf.shape
    nfft = min(cfg.nfft_max_len, 2 * int(filterLen))
    K = nfft // 2 + 1
    if rotations is None:
        rot, B = None, 1
    else:
        rot = np.ascontiguousarray(np.asarray(rotations, dtype=np.float64).reshape(-1, 9))
        B = rot.shape[0]
    wL = np.zeros((int(filterLen), M, B), order="F")
    wR = np.zeros((int(filterLen), M, B), order="F")
    sp = np.zeros((K, M, B, 2), dtype=np.complex128, order="F") if return_spectra else None
    dev = np.zeros(B)
    h.check(h.lib.emagls_design_from_atf_batch(h.ptr, C.byref(cfg), _p(hL), _p(hR), T, D, _p(hg), _p(atf), Ta, M, Da,
                                               _p(ag), float(fs), int(filterLen), float(fTrans), B, _p(rot), _p(wL),
                                               _p(wR), _p(sp), _p(dev)))
    # the reference prints this line (lib/getEMagLsFiltersFromAtf.m:96)
    for v in dev[: min(B, 3)]:
        print(f"Matching HRTF and ATF grids, average grid deviation: {v:.5g} deg")
    if rotations is None:
        wL, wR = wL[:, :, 0], wR[:, :, 0]
        if sp is not None:
            sp = sp[:, :, 0, :]
    out = (wL, wR)
    if return_spectra:
        out += (sp,)
    if return_info:
        out += (dict(meanGridDevDeg=float(dev[0]) if rotations is None else dev),)
    return out


def _design_ema(fn_name, channels, hL, hR, hrirGridAziRad, hrirGridZenRad, micRadius, micGridAziRad, order,
                fs, length, shDefinition, shFunction, chFunction, handle, config, return_spectra, rotations=None):
    _check_sh_function(shFunction)
    if chFunction is not None:
        raise NotImplementedError("only the default chFunction (@getCH) is evaluated on the device")
    h = handle or default_handle()
    cfg = _config(h, config, shDefinition)
    hL, hR, T, D, sets = _prep_hrirs(hL, hR)
    batched = fn_name == "emagls_design_ema_ch" and (sets != 1 or rotations is not None)
    if sets != 1 and not batched:
        raise ValueError("getEMagLsFiltersEMAinSH takes one HRTF set")
    az, ze, maz = _vec(hrirGridAziRad), _vec(hrirGridZenRad), _vec(micGridAziRad)
    Mc = channels(int(order))
    nfft = min(cfg.nfft_max_len, 2 * int(length))
    K = nfft // 2 + 1
    odt = np.complex128 if cfg.basis == 1 else np.float64
    if batched:
        rot = None if rotations is None else np.ascontiguousarray(np.asarray(rotations, dtype=np.float64).reshape(-1, 9))
        B = 1 if rot is None else rot.shape[0]
        P = sets * B
        wL = np.zeros((int(length), Mc, P), dtype=odt, order="F")
        wR = np.zeros((int(length), Mc, P), dtype=odt, order="F")
        sp = np.zeros((K, Mc, P, 2), dtype=np.complex128, order="F") if return_spectra else None
        h.check(h.lib.emagls_design_ema_ch_batch(h.ptr, C.byref(cfg), _p(hL), _p(hR), T, D, _p(az), _p(ze),
                                                 float(micRadius), _p(maz), maz.size, int(order), float(fs),
                                                 int(length), sets, B, _p(rot), _p(wL), _p(wR), _p(sp)))
        return (wL, wR, sp) if return_spectra else (wL, wR)
    wL = np.zeros((int(length), Mc), dtype=odt, order="F")
    wR = np.zeros((int(length), Mc), dtype=odt, order="F")
    sp = np.zeros((K, Mc, 2), dtype=np.complex128, order="F") if return_spectra else None
    h.check(getattr(h.lib, fn_name)(h.ptr, C.byref(cfg), _p(hL), _p(hR), T, D, _p(az), _p(ze), float(micRadius),
                                    _p(maz), maz.size, int(order), float(fs), int(length), _p(wL), _p(wR),
                                    _p(sp)))
    return (wL, wR, sp) if return_spectra else (wL, wR)


def getEMagLsFiltersEMAinCH(hL, hR, hrirGridAziRad, hrirGridZenRad, micRadius, micGridAziRad, order, fs, len,
                            shDefinition="real", shFunction=None, chFunction=None, *, rotations=None, handle=None,
                            config=None, return_spectra=False):
    """lib/getEMagLsFiltersEMAinCH.m:1-2 -> filters [len, 2*order+1].

    Keyword-only batch extension: ``rotations`` [B,3,3] and / or ``hL, hR`` [samples, dirs, sets] give
    ``[len, 2*order+1, sets*B]`` (page b = one reference call with the HRIR grid rotated by ``rotations[b]``)."""
    return _design_ema("emagls_design_ema_ch", lambda N: 2 * N + 1, hL, hR, hrirGridAziRad, hrirGridZenRad,
                       micRadius, micGridAziRad, order, fs, len, shDefinition, shFunction, chFunction, handle,
                       config, return_spectra, rotations)


def getEMagLsFiltersEMAinSH(hL, hR, hrirGridAziRad, hrirGridZenRad, micRadius, micGridAziRad, order, fs, len,
                            shDefinition="real", shFunction=None, chFunction=None, *, handle=None, config=None,
                            return_spectra=False):
    """lib/getEMagLsFiltersEMAinSH.m:1-2 -> filters [len, (order+1)^2]."""
    return _design_ema("emagls_design_ema_sh", lambda N: (N + 1) ** 2, hL, hR, hrirGridAziRad, hrirGridZenRad,
                       micRadius, micGridAziRad, order, fs, len, shDefinition, shFunction, chFunction, handle,
                       config, return_spectra)


def getSMAIRMatrix(params: dict, *, handle=None):
    """[smairMat, params] = getSMAIRMatrix(params)  -- dependencies/getSMAIRMatrix.m:1.

    ``params`` is a dict with the reference's field names; defaults follow getSMAIRMatrix.m:30-84.
    Returns ``(smairMat [rows, S, K] complex, params_with_defaults)``.
    """
    p = dict(params)
    if "smaDesignAziZenRad" not in p:
        raise ValueError("default mic layout needs des.3.32.7.txt, which the reference does not ship")
    p.setdefault("order", 4)
    p.setdefault("fs", 48000)
    p.setdefault("smaRadius", 0.042)
    p.setdefault("arrayType", "rigid")
    p.setdefault("radialFilter", "regul")
    p.setdefault("sourceDist", 2)
    p.setdefault("dirCoeff", 0)
    p.setdefault("waveModel", "planeWave")
    p.setdefault("noiseGainDb", 20)
    p.setdefault("zStyleMaxRe", 1)
    p.setdefault("sourcePosCart", np.array([p["sourceDist"], 0.0, 0.0]))
    p.setdefault("oversamplingFactor", 4)
    p.setdefault("irLen", 2048)
    p.setdefault("returnRawMicSigs", False)
    p.setdefault("shDefinition", "real")
    p["sourceDist"] = float(np.linalg.norm(p["sourcePosCart"]))
    _check_sh_function(p.get("shFunction"))
    radial = str(p["radialFilter"]).lower() != "none" and not p["returnRawMicSigs"]
    if p["arrayType"] not in ("rigid", "open"):
        raise ValueError("Wrong array type")
    h = handle or default_handle()
    cfg = _config(h, None, p["shDefinition"])
    cfg.array_type = 0 if p["arrayType"] == "rigid" else 1
    nfft = int(p["oversamplingFactor"] * p["irLen"])
    assert nfft % 2 == 0
    mics = np.asarray(p["smaDesignAziZenRad"], dtype=np.float64).reshape(-1, 2)
    maz, mze = _vec(mics[:, 0]), _vec(mics[:, 1])
    simN = C.c_int(0)
    raw = 1 if p["returnRawMicSigs"] else 0
    h.check(h.lib.emagls_smair_matrix(h.ptr, C.byref(cfg), _p(maz), _p(mze), maz.size, int(p["order"]),
                                      float(p["fs"]), float(p["smaRadius"]), nfft, raw, None, C.byref(simN)))
    S = (simN.value + 1) ** 2
    rows = maz.size if raw else (int(p["order"]) + 1) ** 2
    K = nfft // 2 + 1
    out = np.zeros((rows, S, K), dtype=np.complex128, order="F")
    if radial:   # getSMAIRMatrix.m:129-139
        rp = _radial_params(h, p)
        h.check(h.lib.emagls_smair_matrix_radial(h.ptr, C.byref(cfg), C.byref(rp), _p(maz), _p(mze), maz.size,
                                                 int(p["order"]), float(p["fs"]), float(p["smaRadius"]), nfft,
                                                 _p(out), C.byref(simN)))
        return out, p
    h.check(h.lib.emagls_smair_matrix(h.ptr, C.byref(cfg), _p(maz), _p(mze), maz.size, int(p["order"]),
                                      float(p["fs"]), float(p["smaRadius"]), nfft, raw, _p(out), C.byref(simN)))
    return out, p


def binauralDecode(inp, inFs, decodingFilterLeft, decodingFilterRight, decodingFilterFs, compensateDelay=False,
                   signal=None, signalFs=None, horRotAngleRad=None, *, handle=None):
    """binauralOut = binauralDecode(in, inFs, decL, decR, decFs[, compensateDelay, ...])
    -- dependencies/binauralDecode.m:1-2."""
    if decodingFilterFs != inFs or (signal is not None and signalFs is not None and signalFs != inFs):
        raise NotImplementedError("binauralDecode: resampling is outside the device path")
    if signal is not None:
        raise NotImplementedError("mono-signal convolution (binauralDecode.m:45-48) is outside the device path")
    h = handle or default_handle()
    if horRotAngleRad is not None and horRotAngleRad != 0:
        # binauralDecode.m:26-30: in = rotateHOA_N3D(in, rad2deg(horRotAngleRad), 0, 0)  (emagls_rotate_sh)
        inp = rotateSH(inp, float(horRotAngleRad), handle=h)
    x, wL, wR = np.asarray(inp), np.asarray(decodingFilterLeft), np.asarray(decodingFilterRight)
    if x.ndim != 2 or wL.shape != wR.shape or wL.ndim != 2 or wL.shape[1] != x.shape[1]:
        raise ValueError("size mismatch between input channels and decoding filters")
    n, ch = x.shape
    ln = wL.shape[0]
    rows = n - (ln // 2 - 1) if compensateDelay else n

    def dec(xr, wl, wr):
        out = np.zeros((rows, 2), order="F")
        h.check(h.lib.emagls_binaural_decode(h.ptr, _p(_f(xr)), n, ch, _p(_f(wl)), _p(_f(wr)), ln,
                                             1 if compensateDelay else 0, _p(out)))
        return out
    if not (np.iscomplexobj(x) or np.iscomplexobj(wL) or np.iscomplexobj(wR)):
        return dec(x, wL, wR)
    # complex-basis signals and filters (shDefinition = 'complex'): the reference keeps real(sum_ch x * w)
    # (binauralDecode.m:59-64) = sum_ch (Re x * Re w - Im x * Im w): two real renders on the device
    out = dec(x.real, wL.real, wR.real)
    xi, wli, wri = np.imag(x), np.imag(wL), np.imag(wR)
    if np.any(xi) and (np.any(wli) or np.any(wri)):
        out -= dec(xi, wli, wri)
    return out


def binauralDecodeTracked(inp, wL, wR, track, hop, fade=None, compensateDelay=False, *, firstSample=0, handle=None):
    """Head-tracked binauralDecode (not in the reference API; emagls_binaural_decode_tracked): ``inp`` [samples, ch]
    rendered with page ``track[f]`` (0-based) of the bank ``wL``, ``wR`` [len, ch, pages] (a [len, ch] filter pair is
    one page) for the samples [f hop, (f + 1) hop) of the track's time axis, crossfading linearly from the previous
    frame's page over the first ``fade`` samples of every frame (default ``hop``; 0 switches hard).  ``firstSample`` is
    the position of inp[0] on the track's time axis.  Complex signals or banks (complex-basis designers) are rendered as
    real(sum_ch x * w), like binauralDecode: two real tracked renders (the crossfade weights are real)."""
    h = handle or default_handle()
    x, wL, wR = np.asarray(inp), np.asarray(wL), np.asarray(wR)
    if wL.ndim == 2:
        wL, wR = wL[:, :, None], wR[:, :, None]
    if x.ndim != 2 or wL.shape != wR.shape or wL.ndim != 3 or wL.shape[1] != x.shape[1]:
        raise ValueError("size mismatch between input channels and the filter bank")
    trk = np.ascontiguousarray(np.asarray(track).ravel())
    if not np.issubdtype(trk.dtype, np.integer) or (trk.size and (trk.min() < -2**31 or trk.max() >= 2**31)):
        raise ValueError("track must hold integer page numbers")
    trk = trk.astype(np.int32)
    n, ch = x.shape
    ln, _, pages = wL.shape
    hop = int(hop)
    fade = hop if fade is None else int(fade)
    rows = n - (ln // 2 - 1) if compensateDelay else n

    def dec(xr, wl, wr):
        out = np.zeros((rows, 2), order="F")
        h.check(h.lib.emagls_binaural_decode_tracked(h.ptr, _p(_f(xr)), n, ch, _p(_f(wl)), _p(_f(wr)), ln, pages,
                                                     _p(trk), trk.size, hop, fade, int(firstSample),
                                                     1 if compensateDelay else 0, _p(out)))
        return out
    if not (np.iscomplexobj(x) or np.iscomplexobj(wL) or np.iscomplexobj(wR)):
        return dec(x, wL, wR)
    out = dec(x.real, wL.real, wR.real)
    xi, wli, wri = np.imag(x), np.imag(wL), np.imag(wR)
    if np.any(xi) and (np.any(wli) or np.any(wri)):
        out -= dec(xi, wli, wri)
    return out


# ---- callers either side of the hot path (SURVEY.md section 8(f)) --------------------------------
_RADIAL_KINDS = {"none": 0, "tikhonov": 1, "softlimit": 2, "full": 3}


def _radial_params(h, p) -> RadialParams:
    rp = RadialParams()
    h.lib.emagls_radial_params_default(C.byref(rp))
    kind = str(p.get("radialFilter", "tikhonov")).lower()
    if kind not in _RADIAL_KINDS:
        raise ValueError(f'Unkown radialFilter parameter "{p.get("radialFilter")}".')   # getRadialFilter.m:65
    if str(p.get("waveModel", "planeWave")).lower() == "pointsource" and kind != "none":
        raise NotImplementedError('WaveModel parameter "pointSource" not yet implemented.')   # :37-40
    at = p.get("arrayType", "rigid")
    if at not in ("rigid", "open"):
        raise ValueError("Wrong array type")
    rp.kind = _RADIAL_KINDS[kind]
    rp.regul_const = float(p.get("regulConst", 1e-2))
    if kind == "softlimit":
        rp.noise_gain_db = float(p["noiseGainDb"])
    rp.array_type = 0 if at == "rigid" else 1
    return rp


def getRadialFilter(params: dict, *, handle=None):
    """radFilts = getRadialFilter(params) -- dependencies/getRadialFilter.m:1 ([nfft/2+1, order+1])."""
    h = handle or default_handle()
    p = dict(params)
    nfft = int(p.get("oversamplingFactor", 2) * p.get("irLen", 256))
    rp = _radial_params(h, p)
    N = int(p["order"])
    out = np.zeros((nfft // 2 + 1, N + 1), dtype=np.complex128, order="F")
    cfg = h.default_config()
    h.check(h.lib.emagls_radial_filter(h.ptr, C.byref(cfg), C.byref(rp), N, float(p["fs"]), float(p["smaRadius"]),
                                       nfft, _p(out)))
    return out.real.copy() if rp.kind == 0 else out


def applyRadialFilter(inSig, params: dict, *, handle=None):
    """sigFiltered = applyRadialFilter(inSig, params) -- dependencies/applyRadialFilter.m:1."""
    h = handle or default_handle()
    p = dict(params)
    rp = _radial_params(h, p)
    N = int(p["order"])
    nfft = int(p["nfft"])
    if nfft != int(p.get("oversamplingFactor", 2) * p.get("irLen", 256)):
        raise ValueError("params.nfft must equal oversamplingFactor * irLen (the reference would fail in "
                         "applySubsampleDelay otherwise)")
    x = _f(inSig)
    if x.ndim != 2 or x.shape[1] != (N + 1) ** 2:
        raise ValueError("inSig must be [samples, (order+1)^2]")
    rows = int(h.lib.emagls_apply_radial_filter_rows(x.shape[0], nfft))
    out = np.zeros((rows, x.shape[1]), order="F")
    cfg = h.default_config()
    h.check(h.lib.emagls_apply_radial_filter(h.ptr, C.byref(cfg), C.byref(rp), _p(x), x.shape[0], N, float(p["fs"]),
                                             float(p["smaRadius"]), nfft, _p(out)))
    return out


def encodeSH(sig, micGridAziRad, micGridZenRad, order, shDefinition="real", shFunction=None, *, handle=None):
    """shRecording = sig * pinv(getSH(order, [azi zen], shDefinition).')  -- verifyEMagLs.m:235-236."""
    _check_sh_function(shFunction)
    h = handle or default_handle()
    cfg = _config(h, None, shDefinition)
    x = _f(sig)
    maz, mze = _vec(micGridAziRad), _vec(micGridZenRad)
    if x.ndim != 2 or x.shape[1] != maz.size or mze.size != maz.size:
        raise ValueError("sig must be [samples, mics]")
    out = np.zeros((x.shape[0], (int(order) + 1) ** 2), dtype=np.complex128 if cfg.basis else np.float64, order="F")
    h.check(h.lib.emagls_sh_encode(h.ptr, C.byref(cfg), _p(x), x.shape[0], maz.size, _p(maz), _p(mze), int(order),
                                   _p(out)))
    return out


def encodeCH(sig, micGridAziRad, order, chDefinition="real", *, handle=None):
    """chSig = sig * pinv(getCH(order, azi, chDefinition).')  -- testEMagLs.m:99-102."""
    h = handle or default_handle()
    cfg = _config(h, None, chDefinition)
    x = _f(sig)
    maz = _vec(micGridAziRad)
    if x.ndim != 2 or x.shape[1] != maz.size:
        raise ValueError("sig must be [samples, mics]")
    out = np.zeros((x.shape[0], 2 * int(order) + 1), dtype=np.complex128 if cfg.basis else np.float64, order="F")
    h.check(h.lib.emagls_ch_encode(h.ptr, C.byref(cfg), _p(x), x.shape[0], maz.size, _p(maz), int(order), _p(out)))
    return out


def rotateSH(sig, yawRad, pitchRad=0.0, rollRad=0.0, *, handle=None):
    """rotateHOA_N3D(sig, yaw, pitch, roll) as called at dependencies/binauralDecode.m:26-30 (radians)."""
    h = handle or default_handle()
    if np.iscomplexobj(sig):
        raise NotImplementedError("rotateSH: rotateHOA_N3D (binauralDecode.m:29) takes real N3D signals")
    x = _f(sig)
    N = int(round(np.sqrt(x.shape[1]))) - 1
    if x.ndim != 2 or (N + 1) ** 2 != x.shape[1]:
        raise ValueError("sig must be [samples, (order+1)^2]")
    out = np.zeros_like(x, order="F")
    h.check(h.lib.emagls_rotate_sh(h.ptr, _p(x), x.shape[0], N, float(yawRad), float(pitchRad), float(rollRad),
                                   _p(out)))
    return out


def getMagLsFilters2D(hLHor, hRHor, horHrirGridAziRad, order, fs, len, chDefinition="real", *, handle=None,
                      config=None, return_spectra=False):
    """[wMlsL, wMlsR] = getMagLsFilters2D(...)  -- lib/getMagLsFilters2D.m:1."""
    h = handle or default_handle()
    cfg = _config(h, config, chDefinition)
    hL, hR, T, D, sets = _prep_hrirs(hLHor, hRHor)
    if sets != 1:
        raise ValueError("getMagLsFilters2D is not batched")
    az = _vec(horHrirGridAziRad)
    if az.size != D:
        raise ValueError("HRIR grid size does not match hLHor")
    H = 2 * int(order) + 1
    K = min(cfg.nfft_max_len, 2 * int(len)) // 2 + 1
    odt = np.complex128 if cfg.basis == 1 else np.float64
    wL = np.zeros((int(len), H), dtype=odt, order="F")
    wR = np.zeros((int(len), H), dtype=odt, order="F")
    sp = np.zeros((K, H, 2), dtype=np.complex128, order="F") if return_spectra else None
    h.check(h.lib.emagls_design_magls_2d(h.ptr, C.byref(cfg), _p(hL), _p(hR), T, D, _p(az), int(order), float(fs),
                                         int(len), _p(wL), _p(wR), _p(sp)))
    return (wL, wR, sp) if return_spectra else (wL, wR)


def getMagLsSphericalHeadFilter(micRadius, order, fs, len, *, handle=None, config=None):
    """[wShf, W_Shf] = getMagLsSphericalHeadFilter(micRadius, order, fs, len)
    -- lib/getMagLsSphericalHeadFilter.m:1."""
    h = handle or default_handle()
    cfg = config if config is not None else h.default_config()
    nfft = min(cfg.nfft_max_len, 2 * int(len))
    w = np.zeros(int(len))
    W = np.zeros(nfft)
    h.check(h.lib.emagls_spherical_head_filter(h.ptr, C.byref(cfg), float(micRadius), int(order), float(fs),
                                               int(len), _p(w), _p(W)))
    return w, W


def getMagLsArrayDiffuseFilter(micRadius, micGridAziRad, micGridZenRad, order, fs, len, shDefinition="real",
                               shFunction=None, *, handle=None, config=None):
    """wAdf = getMagLsArrayDiffuseFilter(...)  -- lib/getMagLsArrayDiffuseFilter.m:1."""
    _check_sh_function(shFunction)
    h = handle or default_handle()
    cfg = _config(h, config, shDefinition)
    maz, mze = _vec(micGridAziRad), _vec(micGridZenRad)
    w = np.zeros(int(len))
    h.check(h.lib.emagls_array_diffuse_filter(h.ptr, C.byref(cfg), float(micRadius), _p(maz), _p(mze), maz.size,
                                              int(order), float(fs), int(len), _p(w)))
    return w


# ---- building blocks (each mirrors one reference function) -------------------------------------
def getSH(N, dirs, basisType="real", *, handle=None):
    """Y_N = getSH(N, [azi zen], basisType) -- dependencies/Spherical-Harmonic-Transform/getSH.m:1."""
    h = handle or default_handle()
    dirs = np.asarray(dirs, dtype=np.float64).reshape(-1, 2)
    az, ze = _vec(dirs[:, 0]), _vec(dirs[:, 1])
    S = (int(N) + 1) ** 2
    b = _basis(basisType)
    out = np.zeros((az.size, S), dtype=np.complex128 if b else np.float64, order="F")
    h.check(h.lib.emagls_get_sh(h.ptr, int(N), _p(az), _p(ze), az.size, b, _p(out)))
    return out


def sphModalCoeffs(N, kr, arrayType="rigid", dirCoeff=0.0, *, handle=None):
    """b_N = sphModalCoeffs(N, kr, arrayType) -- dependencies/Array-Response-Simulator/sphModalCoeffs.m:1."""
    if arrayType not in ("rigid", "open"):
        raise ValueError("Wrong array type")
    h = handle or default_handle()
    kr = _vec(kr)
    out = np.zeros((kr.size, int(N) + 1), dtype=np.complex128, order="F")
    h.check(h.lib.emagls_sph_modal_coeffs(h.ptr, int(N), _p(kr), kr.size, 0 if arrayType == "rigid" else 1,
                                          _p(out)))
    return out


def grpdelay(h_sum_or_set, f, fs, *, handle=None):
    """``grpdelay(sum(h, 2), 1, f, fs)`` and its median as the designers use it (lib/getEMagLs2Filters.m:72-75).

    ``h_sum_or_set``: [taps] or [taps x dirs] (summed over the directions on the device); ``f`` must be
    ``linspace(0, fs/2, numPosFreqs)`` as in the reference.  Returns (gd [numPosFreqs], median)."""
    hnd = handle or default_handle()
    x = np.asarray(h_sum_or_set, dtype=np.float64)
    if x.ndim == 1:
        x = x[:, None]
    x = np.asfortranarray(x)
    f = _vec(f)
    if f.size < 2 or not np.allclose(f, np.linspace(0.0, fs / 2.0, f.size)):
        raise ValueError("f must be linspace(0, fs/2, numPosFreqs)")
    gd = np.zeros(f.size)
    med = np.zeros(1)
    hnd.check(hnd.lib.emagls_group_delay(hnd.ptr, _p(x), x.shape[0], x.shape[1], f.size, float(fs), _p(gd), _p(med)))
    return gd, float(med[0])


def regularizedApply(pwGrid, targets, svd_regul=0.01, *, handle=None):
    """targets * Y_reg_inv with Y_reg_inv from lib/getEMagLs2Filters.m:87-89 (one bin)."""
    h = handle or default_handle()
    pw = np.asfortranarray(np.asarray(pwGrid, dtype=np.complex128))
    t = np.asfortranarray(np.atleast_2d(np.asarray(targets, dtype=np.complex128)))
    Mc, D = pw.shape
    out = np.zeros((t.shape[0], Mc), dtype=np.complex128, order="F")
    h.check(h.lib.emagls_regularized_apply(h.ptr, _p(pw), Mc, D, _p(t), t.shape[0], float(svd_regul), _p(out)))
    return out
