"""The per-pixel match info of compute_rsgm (opt-in, include/vppstereo_b200.h) as a NumPy restatement of its definition on the
oracle's operators: the stages of test_gpu_uniqueness.oracle_rsgm, kept apart where the definition names them, and the candidate
scan of uniq_reference.py.  Test infrastructure for test_match_info_cpu.py and test_gpu_match_info.py.

  m = left map after WTA (uniqueness test for u < 1), sub-pixel step and median3x3 (padded);  c = max(linear_interpolate(m), 0);
  crop;  mask = left_right_check(c, c_right);  u8 = uint8(c with mask == 128 set to 0);  s = filter_speckles(u8)
  state: the first rule that applies of  2: c == 0,  3: mask == 128,  4: u8 == 0,  5: s == 0,  1: m <= 0,  0: otherwise
  cost = S[b], rival = min{S[d] : d <= end, |d - b| >= 2} (65535: none), b = first arg-min over d <= end = min(D-1, x) (padded x)
"""
import numpy as np

import uniq_reference as ref

MATCHED, INTERPOLATED, NO_MATCH, LR_REJECTED, BELOW_ONE, SPECKLE = 0, 1, 2, 3, 4, 5


def _pads(H, W):
    pad_h, pad_w = (((H // 16) + 1) * 16 - H) % 16, (((W // 16) + 1) * 16 - W) % 16
    return pad_h // 2, pad_h - pad_h // 2, pad_w // 2, pad_w - pad_w // 2


def left_costs(S):
    """S uint16 [..., W, D] -> (cost, rival) uint16 [..., W] of the left view's candidates (uniq_reference's scan)"""
    S = np.asarray(S).astype(np.int64)
    W, D = S.shape[-2], S.shape[-1]
    x, d = np.arange(W)[:, None], np.arange(D)[None, :]
    c = np.where(d <= np.minimum(D - 1, x), S, ref._OUT)
    b = np.argmin(c, axis=-1)
    cost = np.take_along_axis(c, b[..., None], axis=-1)[..., 0]
    rival = np.where((np.abs(d - b[..., None]) >= 2) & (c < ref._OUT), c, ref._OUT).min(axis=-1)
    return cost.astype(np.uint16), np.where(rival == ref._OUT, 65535, rival).astype(np.uint16)


def state_map(m, c, mask, u8, s):
    """the table of the definition on the cropped stage maps"""
    st = np.full(c.shape, MATCHED, np.uint8)
    for code, hit in ((INTERPOLATED, m <= 0), (SPECKLE, s == 0), (BELOW_ONE, u8 == 0), (LR_REJECTED, mask == 128), (NO_MATCH, c == 0)):
        st[hit] = code                                             # lowest precedence first: later rules overwrite
    return st


def match_info(orc, left, left_vpp, right_vpp, hints=None, validhints=None, dmax=192, subpixel=True, params=(7, 17, 0.25, 50),
               u=1.0):
    """one frame -> dict(disp, prefill, state, cost, rival); disp is compute_rsgm's output, prefill the same before the background
    fill (rsgm.py:289-292)"""
    left, left_vpp, right_vpp = (np.ascontiguousarray(a, np.uint8) for a in (left, left_vpp, right_vpp))
    H, W = left.shape[:2]
    D = int(dmax)
    pt, pb, pl, pr = _pads(H, W)
    lp, lvp, rvp = (orc.pad_reflect(a, pt, pb, pl, pr) for a in (left, left_vpp, right_vpp))
    Hp, Wp = lp.shape[:2]
    gray = (lambda a: orc.rgb2gray(a)) if lvp.ndim == 3 and lvp.shape[2] == 3 else (lambda a: np.ascontiguousarray(a.reshape(Hp, Wp)))
    cl = np.zeros((Hp, Wp), np.uint32); cr = np.zeros((Hp, Wp), np.uint32)
    orc.census5x5_SSE(gray(lvp), cl, Wp, Hp); orc.census5x5_SSE(gray(rvp), cr, Wp, Hp)
    dsi = np.zeros((Hp, Wp, D), np.uint16)
    orc.costMeasureCensus5x5_xyd_SSE(cl, cr, dsi, Wp, Hp, D)
    if hints is not None:
        hp = np.zeros((Hp, Wp), np.float32); vp = np.zeros((Hp, Wp), np.float32)
        hp[pt:pt + H, pl:pl + W] = hints; vp[pt:pt + H, pl:pl + W] = validhints
        dsi = orc.guided_dsi(dsi, hp, vp)
    S = np.zeros_like(dsi)
    orc.aggregate_SSE(lp, dsi, S, Wp, Hp, D, *params, honor_params=True)
    crop = lambda a: np.ascontiguousarray(a[pt:pt + H, pl:pl + W])
    med, maps = [], []
    for wta, sub in ((ref.wta_left, True), (ref.wta_right, False)):
        d = np.ascontiguousarray(wta(S, u))
        if sub:
            orc.subPixelRefine(S, d, Wp, Hp, D, 0)
        f = np.zeros((Hp, Wp), np.float32)
        orc.median3x3_SSE(d, f, Wp, Hp)
        med.append(f.copy())
        orc.linear_interpolate(f, 15, 3.0)
        f[f < 0] = 0
        maps.append(crop(f))
    fl, fr = maps
    mask = orc.left_right_check(fl, fr, 1.0)
    u8 = np.where(mask == 128, np.float32(0), fl).astype(np.uint8)
    s = orc.filter_speckles_u8(u8, 0, 200, 10)
    out = s.astype(np.float32)
    if subpixel:
        out = np.where(out != 0, fl, out).astype(np.float32)
    out = np.ascontiguousarray(out)
    prefill = out.copy()
    orc.interpolate_background(out)
    cost, rival = (crop(a) for a in left_costs(S))
    return dict(disp=out, prefill=prefill, state=state_map(crop(med[0]), fl, mask, u8, s), cost=cost, rival=rival)
