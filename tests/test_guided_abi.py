"""vppb200_sgm_band_guided refuses bad operands before any CUDA call (runs without a device: the host buffers below are never
dereferenced)."""
import ctypes

import pytest

GUIDED_OOD = (3700, 3700, 0.0, 3856)        # inside the Hamming sweep domain, outside the guided one (Cmax = 240)


def _band_args(L, prm, hints, valid):
    buf = (ctypes.c_uint8 * 64)()
    one = ctypes.cast(buf, ctypes.c_void_p)
    H, W, C, D = 16, 32, 3, 16
    bws = L.vppb200_banded_workspace_bytes(H, W, C, D)
    p = None if prm is None else ctypes.byref(prm)
    h = one if hints else None
    v = one if valid else None
    return (one, one, one, one, one, H, W, C, D, 0, H, 31, None, None, one, one, one, one, ctypes.c_size_t(bws), None, p, h, v)


def _params(p):
    from vppstereo_b200 import _lib
    return _lib.VppSgmParams(int(p[0]), int(p[1]), float(p[2]), int(p[3]))


@pytest.mark.parametrize("hints,valid", [(True, False), (False, True)])
@pytest.mark.parametrize("prm", [None, (7, 17, 0.25, 50)])
def test_band_guided_refuses_half_given_hints(prm, hints, valid):
    from vppstereo_b200 import _lib
    L = _lib.lib()
    args = _band_args(L, None if prm is None else _params(prm), hints, valid)
    assert L.vppb200_sgm_band_guided(*args) == _lib.ERR_ARG


def test_band_guided_refuses_params_outside_guided_domain():
    from vppstereo_b200 import _lib
    L = _lib.lib()
    prm = _params(GUIDED_OOD)
    assert L.vppb200_sgm_params_fast(ctypes.byref(prm), 0) == 1 and L.vppb200_sgm_params_fast(ctypes.byref(prm), 1) == 0
    assert L.vppb200_sgm_band_guided(*_band_args(L, prm, True, True)) == _lib.ERR_ARG
    # a parameter set refused by every entry point is refused with hints too
    assert L.vppb200_sgm_band_guided(*_band_args(L, _params((30, 10, 0.5, 20)), True, True)) == _lib.ERR_ARG
    assert L.vppb200_sgm_band_guided(*_band_args(L, _params((-1, 17, 0.5, 35)), False, False)) == _lib.ERR_ARG
