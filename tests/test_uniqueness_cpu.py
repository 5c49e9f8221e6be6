"""The uniqueness ratio of the winner-takes-all (opt-in, include/vppstereo_b200.h), without a device: the vectorised reference
(uniq_reference.py, the GPU tests' target) against a per-pixel brute force of the definition, the right conveyor's online update
(descending k) against the definition, and the argument validation of the entry points and front-ends."""
import ctypes
import math

import numpy as np
import pytest

import uniq_reference as ref


def brute(c, u):
    """the definition on one candidate list c[0..end] -> float disparity (-10 = rejected)"""
    c = [int(v) for v in c]
    b = int(np.argmin(c))
    rivals = [v for d, v in enumerate(c) if abs(d - b) >= 2]
    f = int(np.float32(1024.0) * np.float32(u))
    if not rivals or 1024 * c[b] <= f * min(rivals):
        return float(b)
    return -10.0


def brute_left(S, u):
    H, W, D = S.shape
    out = np.empty((H, W), np.float32)
    for y in range(H):
        for x in range(W):
            out[y, x] = brute(S[y, x, :min(D - 1, x) + 1], u)
    return out


def brute_right(S, u):
    H, W, D = S.shape
    out = np.empty((H, W), np.float32)
    for y in range(H):
        for x in range(W):
            end = min(D - 1, W - 1 - x)
            out[y, x] = brute([S[y, x + k, k] for k in range(end + 1)], u)
    return out


def online(c, u):
    """the conveyor's rule (common.cuh: uniq_absorb): candidates arrive in descending k; 0xFFFF is only min's identity"""
    best, far, rest, last = 0xFFFFFFFF, 0xFFFF, 0xFFFF, 0xFFFF
    for k in range(len(c) - 1, -1, -1):
        key = (int(c[k]) << 16) | k
        if key < best:
            far, best = rest, key
        elif (best & 0xFFFF) >= k + 2:
            far = min(far, int(c[k]))
        rest, last = min(rest, last), int(c[k])
    end, b = len(c) - 1, best & 0xFFFF
    rival = end >= 3 or (end == 2 and b != 1)
    f = int(np.float32(1024.0) * np.float32(u))
    return float(b) if not rival or 1024 * (best >> 16) <= f * far else -10.0


UNIQ = [0.5, 0.8, 0.95, 0.999, 1.0, 1023 / 1024, 1e-4]


def constructed_lists():
    """ties at the minimum, c2 only at b +- 1, the rival at b +- 2, flat curves, end = 0, 1, 2, u16 extremes"""
    L = [[5], [0], [65535], [3, 3], [4, 2], [65535, 65535], [1, 0, 1], [0, 1, 2], [2, 1, 0], [5, 5, 5], [0, 65535, 0],
         [65535, 0, 65535], [7, 3, 3, 7], [3, 4, 3, 9, 9], [10, 9, 10, 11, 20], [9, 10, 11, 10, 9], [1] * 40,
         [65535] * 40, [0] * 40, [65534, 65535, 65535, 65535], [100, 99, 100, 101, 104]]
    rng = np.random.default_rng(0)
    for n in (4, 7, 64, 192, 256):
        c = rng.integers(50, 60, n)
        b = int(rng.integers(0, n))
        c[b] = 40
        for off in (-1, 1):
            if 0 <= b + off < n:
                c[b + off] = 40                  # ties / neighbours at the minimum: not rivals
        for off in (-2, 2):
            if 0 <= b + off < n:
                L.append(np.where(np.arange(n) == b + off, 41, c).tolist())   # a near rival at b +- 2
        L.append(c.tolist())
    return L


@pytest.mark.parametrize("u", UNIQ)
def test_online_update_equals_definition(u):
    rng = np.random.default_rng(int(u * 1e6))
    lists = constructed_lists() + [rng.integers(0, hi, n).tolist() for n in (1, 2, 3, 5, 33, 256) for hi in (3, 40, 65536)]
    for c in lists:
        assert online(c, u) == brute(c, u), (c[:12], u)


def test_factor_edges():
    """f = 0 (u < 1/1024): only a zero best cost with a rival passes; f = 1023; f = 1024 (u = 1) passes everything"""
    assert brute([0, 5, 0, 7], 1e-4) == 0.0 and brute([1, 5, 9, 7], 1e-4) == -10.0
    assert brute([1024, 2000, 1024 + 1, 5000], 1023 / 1024) == -10.0        # 1024 * 1024 > 1023 * 1025
    assert brute([1023, 2000, 1024, 5000], 1023 / 1024) == 0.0              # 1024 * 1023 <= 1023 * 1024
    for c in constructed_lists():
        assert brute(c, 1.0) == float(np.argmin(c))
    assert brute([65535, 0, 65535, 65535, 65535], 0.5) == 1.0                # rival 65535 exists and is far above
    assert brute([65535, 65535, 65535, 65535], 0.999) == -10.0               # a genuine 65535 rival is still a rival
    assert brute([65535, 65535, 65535], 0.999) == -10.0                      # end = 2, b = 0: d = 2 is a rival
    assert brute([65535, 65535], 0.5) == 0.0                                 # end = 1: no rival


def _volumes():
    rng = np.random.default_rng(7)
    out = [rng.integers(0, 65536, (3, 32, 8), dtype=np.uint16), rng.integers(0, 6, (2, 48, 72), dtype=np.uint16),
           rng.integers(100, 140, (2, 64, 200), dtype=np.uint16)]
    sat = rng.integers(65530, 65536, (2, 32, 16), dtype=np.uint16)
    sat[sat > 65533] = 65535
    flat = np.full((1, 16, 24), 9, np.uint16)
    out += [sat, flat]
    return out


@pytest.mark.parametrize("u", [0.5, 0.8, 0.95, 0.999, 1.0, 1023 / 1024, 1e-4])
def test_reference_equals_brute_force(u):
    for S in _volumes():
        for fast, slow in ((ref.wta_left, brute_left), (ref.wta_right, brute_right)):
            np.testing.assert_array_equal(fast(S, u), slow(S, u), err_msg=f"{fast.__name__} u={u} shape={S.shape}")


def test_reference_u1_equals_plain_wta(orc):
    """u = 1 is the oracle's plain first arg-min (orc_wta_left / orc_wta_right)"""
    for S in _volumes():
        H, W, D = S.shape
        for fast, wta in ((ref.wta_left, orc.matchWTA_SSE), (ref.wta_right, orc.matchWTARight_SSE)):
            plain = np.zeros((H, W), np.float32)
            wta(S, plain, W, H, D, 0.5)
            np.testing.assert_array_equal(fast(S, 1.0), plain)


# ---------------------------------------------------------------- validation before any device work
BAD = [0.0, -0.5, 1.0001, float("nan"), float("inf")]


@pytest.mark.parametrize("u", BAD)
def test_entry_points_refuse_bad_uniqueness(u):
    """the host buffers below are never dereferenced: the status comes before any CUDA call"""
    from vppstereo_b200 import _lib
    L = _lib.lib()
    buf = (ctypes.c_uint8 * 64)()
    one = ctypes.cast(buf, ctypes.c_void_p)
    for fn in (L.vppb200_match_wta_uniq, L.vppb200_match_wta_right_uniq):
        assert fn(one, one, 32, 8, 16, u, 1, None) == _lib.ERR_UNIQUENESS
    H, W, C, D = 16, 32, 3, 16
    ws = L.vppb200_rsgm_workspace_bytes(H, W, C, D, 1)
    assert L.vppb200_compute_rsgm_uniq(one, one, one, None, None, one, H, W, C, D, 1, None, one, ws, 1, None, 7, 1, 0, None, None,
                                       u) == _lib.ERR_UNIQUENESS
    bws = L.vppb200_banded_workspace_bytes(H, W, C, D)
    assert L.vppb200_sgm_band_uniq(one, one, one, one, one, H, W, C, D, 0, H, 31, None, None, one, one, one, one, bws, None, None,
                                   None, None, u) == _lib.ERR_UNIQUENESS


@pytest.mark.parametrize("u", BAD + ["x", None])
def test_front_ends_raise_before_device_work(u):
    from vppstereo_b200 import _lib, pyrSGM, rsgm
    img = np.zeros((16, 32, 3), np.uint8)
    with pytest.raises(TypeError, match="Uniqueness must be inside"):
        rsgm.compute_rsgm(img, img, img, dmax=16, uniqueness=u, honor_uniqueness=True)
    with pytest.raises(TypeError, match="Uniqueness must be inside"):
        rsgm.compute_rsgm_stages(img, img, img, dmax=16, uniqueness=u, honor_uniqueness=True)
    S = np.zeros((8, 32, 16), np.uint16)
    for op in (pyrSGM.matchWTA_SSE, pyrSGM.matchWTARight_SSE):
        with pytest.raises(TypeError, match="Uniqueness must be inside"):
            op(S, np.zeros((8, 32), np.float32), 32, 8, 16, u, honor_uniqueness=True)
    with pytest.raises(TypeError, match="Uniqueness must be inside"):
        _lib.uniqueness(u)


def test_uniqueness_accepts_the_range():
    from vppstereo_b200 import _lib
    assert _lib.uniqueness(1) == 1.0 and _lib.uniqueness(0.95) == 0.95 and not math.isnan(_lib.uniqueness(1e-30))
