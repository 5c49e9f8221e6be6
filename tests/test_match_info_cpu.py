"""The per-pixel match info of compute_rsgm (opt-in, include/vppstereo_b200.h), without a device: the restatement
(match_info_reference.py, the GPU tests' target) against the oracle's compute_rsgm and against the definition's own invariants, and
the argument validation of vppb200_compute_rsgm_info."""
import ctypes

import numpy as np
import pytest

import match_info_reference as mi
from conftest import ROOT

FRAMES = [((37, 70), 8, 3, True), ((46, 150), 64, 1, False), ((40, 261), 192, 3, True), ((60, 140), 64, 3, True)]


@pytest.mark.parametrize("shape,D,channels,sub", FRAMES)
def test_reference_vs_oracle(orc, shape, D, channels, sub):
    from vppstereo_b200 import synth
    p = synth.make_pair(500 + D, shape=shape, hints="random", channels=channels)
    got = mi.match_info(orc, p["left"], p["left"], p["right"], dmax=D, subpixel=sub)
    want = orc.compute_rsgm(p["left"], p["left"], p["right"], dmax=D, subpixel=sub)
    np.testing.assert_array_equal(got["disp"].view(np.uint32), want.view(np.uint32))
    st = got["state"]
    assert st.dtype == np.uint8 and st.shape == shape and st.max() <= mi.SPECKLE
    # codes 2..5 are exactly the pixels the background fill writes
    np.testing.assert_array_equal(st >= mi.NO_MATCH, got["prefill"] == 0)
    assert (got["cost"] <= got["rival"]).all()
    assert got["cost"].dtype == np.uint16 and got["rival"].dtype == np.uint16


def test_state_precedence():
    """the first rule that applies wins, in the order 2, 3, 4, 5, 1, 0"""
    m = np.array([-10, -10, -10, -10, -10, 3, 3], np.float32)
    c = np.array([0, 2.5, 0.5, 4, 5, 3, 3], np.float32)
    mask = np.array([0, 128, 0, 255, 255, 255, 0], np.uint8)
    u8 = np.where(mask == 128, np.float32(0), c).astype(np.uint8)
    s = np.array([0, 0, 0, 0, 5, 0, 3], np.uint8)
    np.testing.assert_array_equal(mi.state_map(m, c, mask, u8, s), [2, 3, 4, 5, 1, 5, 0])


def test_left_costs_definition():
    """cost / rival against a per-pixel scan, including end <= 2 (no rival: 65535) and genuine 65535 costs"""
    rng = np.random.default_rng(3)
    for S in (rng.integers(0, 65536, (2, 20, 16), dtype=np.uint16), rng.integers(0, 3, (2, 20, 24), dtype=np.uint16),
              np.full((1, 5, 8), 65535, np.uint16)):
        cost, rival = mi.left_costs(S)
        D = S.shape[-1]
        for y in range(S.shape[0]):
            for x in range(S.shape[1]):
                c = [int(v) for v in S[y, x, :min(D - 1, x) + 1]]
                b = int(np.argmin(c))
                rv = [v for d, v in enumerate(c) if abs(d - b) >= 2]
                assert cost[y, x] == c[b] and rival[y, x] == (min(rv) if rv else 65535), (y, x)


def test_costs_do_not_depend_on_uniqueness(orc):
    from vppstereo_b200 import synth
    p = synth.make_pair(31, shape=(40, 120), hints="random")
    a = mi.match_info(orc, p["left"], p["left"], p["right"], dmax=64)
    b = mi.match_info(orc, p["left"], p["left"], p["right"], dmax=64, u=0.8)
    np.testing.assert_array_equal(a["cost"], b["cost"])
    np.testing.assert_array_equal(a["rival"], b["rival"])
    np.testing.assert_array_equal(b["state"] >= mi.NO_MATCH, b["prefill"] == 0)
    # the test rejects pixels of the raw map: here some of them end up without a match
    assert (b["state"] == mi.NO_MATCH).sum() > (a["state"] == mi.NO_MATCH).sum()


# ---------------------------------------------------------------- validation before any device work
def test_info_entry_point_validation():
    """the host buffers below are never dereferenced: every status comes before any CUDA call"""
    from vppstereo_b200 import _lib
    L = _lib.lib()
    buf = (ctypes.c_uint8 * 64)()
    one = ctypes.cast(buf, ctypes.c_void_p)
    H, W, C, D = 16, 32, 3, 16
    plain = L.vppb200_rsgm_workspace_bytes_sets(H, W, C, D, 1, 2)
    info = L.vppb200_rsgm_info_workspace_bytes(H, W, C, D, 1, 2)
    assert info > plain > 0
    assert L.vppb200_rsgm_info_workspace_bytes(H, W, C, D, 1, 1) < info
    for bad in ((H, W, C, 12, 1, 1), (H, W, 2, D, 1, 1), (H, W, C, D, 0, 1), (H, W, C, D, 1, 5), (0, W, C, D, 1, 1)):
        assert L.vppb200_rsgm_info_workspace_bytes(*bad) == 0, bad

    def call(ws_bytes, state=one, cost=one, rival=one, u=1.0):
        return L.vppb200_compute_rsgm_info(one, one, one, None, None, one, H, W, C, D, 1, None, one, ws_bytes, 1, None, 7, 2, 0, None,
                                           None, u, state, cost, rival)
    for missing in ({"state": None}, {"cost": None}, {"rival": None}):
        assert call(info, **missing) == _lib.ERR_ARG, missing
    assert call(plain) == _lib.ERR_WORKSPACE                       # the plain layout is too small for the info
    assert call(info, u=0.0) == _lib.ERR_UNIQUENESS


def test_state_constants():
    """header, binding and the restatement agree on the codes"""
    import os
    import re
    from vppstereo_b200 import _lib, rsgm
    text = open(os.path.join(ROOT, "include", "vppstereo_b200.h")).read()
    defs = {k: int(v) for k, v in re.findall(r"#define VPPB200_STATE_(\w+) (\d+)", text)}
    assert defs == {k: getattr(_lib, "STATE_" + k) for k in defs} and len(defs) == 6
    assert (rsgm.STATE_MATCHED, rsgm.STATE_INTERPOLATED, rsgm.STATE_NO_MATCH, rsgm.STATE_LR_REJECTED, rsgm.STATE_BELOW_ONE,
            rsgm.STATE_SPECKLE) == (mi.MATCHED, mi.INTERPOLATED, mi.NO_MATCH, mi.LR_REJECTED, mi.BELOW_ONE, mi.SPECKLE)
