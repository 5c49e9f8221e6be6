"""Drop-in for models/rsgm/rsgm.py: `compute_rsgm` with the reference's signature, running entirely on the device.

    from vppstereo_b200.rsgm import compute_rsgm          # instead of  from models.rsgm.rsgm import compute_rsgm

numpy in -> numpy out (test.py:210-225 keeps working unchanged); CUDA tensors in -> CUDA tensor out with no host
round-trip.  A leading batch dimension [N,H,W(,C)] is accepted and processed as one launch sequence.
"""
import numpy as np

from . import _lib

__all__ = ["compute_rsgm", "compute_rsgm_stages", "STATE_MATCHED", "STATE_INTERPOLATED", "STATE_NO_MATCH", "STATE_LR_REJECTED",
           "STATE_BELOW_ONE", "STATE_SPECKLE"]

# per-pixel match state of return_info=True (include/vppstereo_b200.h; the first rule that applies, in the order 2, 3, 4, 5, 1, 0):
STATE_MATCHED = _lib.STATE_MATCHED            # 0: a measured disparity (positive WTA winner, kept by every check)
STATE_INTERPOLATED = _lib.STATE_INTERPOLATED  # 1: kept by every check, but its value came from the gap interpolation
STATE_NO_MATCH = _lib.STATE_NO_MATCH          # 2: no positive match, even after the gap interpolation
STATE_LR_REJECTED = _lib.STATE_LR_REJECTED    # 3: failed the left-right check
STATE_BELOW_ONE = _lib.STATE_BELOW_ONE        # 4: 0 < disparity < 1, truncated to 0 by the uint8 map
STATE_SPECKLE = _lib.STATE_SPECKLE            # 5: removed by the speckle filter
# codes 2..5 are the pixels whose output value comes from the background fill


def _prep(left, left_vpp, right_vpp, hints, validhints, dmax):
    if dmax % 8 != 0:
        raise Exception(f"Invalid dmax ({dmax}): dmax % 8 != 0")            # models/rsgm/rsgm.py:31-32
    if dmax > 256:
        raise Exception(f"Invalid dmax ({dmax}): dmax > 256")               # models/rsgm/rsgm.py:34-35
    torch = _lib.require_cuda()
    was_numpy = not _lib.is_tensor(left_vpp)
    imgs = []
    for a in (left, left_vpp, right_vpp):
        t = _lib.as_device(a, torch.uint8)
        imgs.append(t)
    lv = imgs[1]
    # shapes: [H,W], [H,W,C], [N,H,W,C]; a 3-dim array whose last dim is 1 or 3 is a single HWC frame (rsgm.py:10-15)
    def norm(t):
        if t.dim() == 2:
            return t[None, :, :, None]
        if t.dim() == 3:
            return t[None] if t.shape[-1] in (1, 3) else t[..., None]
        if t.dim() == 4:
            return t
        raise ValueError("images must be [H,W], [H,W,C] or [N,H,W,C]")
    batched = lv.dim() == 4 or (lv.dim() == 3 and lv.shape[-1] not in (1, 3))
    imgs = [norm(t).contiguous() for t in imgs]
    N, H, W, C = imgs[1].shape
    if imgs[2].shape != imgs[1].shape:
        raise ValueError("left_vpp / right_vpp shape mismatch")
    if imgs[0].shape[:3] != (N, H, W):
        raise ValueError("left / left_vpp shape mismatch")
    if imgs[0].shape[3] != C:
        # the guide is only ever read as a byte stream; bring it to the matching images' channel count as cv2 would not
        raise ValueError("left and left_vpp must have the same number of channels")
    if C not in (1, 3):
        raise ValueError("images must have 1 or 3 channels")
    h = v = None
    if hints is not None and validhints is not None:
        h = _lib.as_device(hints, torch.float32).reshape(N, H, W).contiguous()
        v = _lib.as_device(validhints, torch.float32).reshape(N, H, W).contiguous()
    return torch, was_numpy, batched, imgs, h, v, (N, H, W, C)


def _params(honor_params, p1, p2min, alpha, gamma):
    """the validated parameters (ValueError before any device work), or None = the reference's effective ones"""
    return _lib.sgm_params(p1, p2min, alpha, gamma) if honor_params else None


def _compute(what, imgs, h, v, out, D, subpixel, rcp_lut, prm, taps, uniq, info=None):
    """vppb200_compute_rsgm_uniq, all three phases, on the images' device and its current stream; taps: None or an RsgmTaps;
    uniq: the validated uniqueness ratio, 1.0 = none; info: None, or the (state, cost, rival) tensors [N,H,W] that
    vppb200_compute_rsgm_info fills"""
    N, H, W, C = imgs[1].shape
    dev = imgs[1].device
    L = _lib.lib()
    nbytes = L.vppb200_rsgm_workspace_bytes(H, W, C, D, N) if info is None else L.vppb200_rsgm_info_workspace_bytes(H, W, C, D, N, 1)
    ws = _lib.workspace(nbytes, dev, "rsgm")
    lut = None
    if rcp_lut is not None:
        lut = rcp_lut if _lib.is_tensor(rcp_lut) else _lib.np_to_dev(rcp_lut, np.float32)
    args = (_lib.ptr(imgs[0]), _lib.ptr(imgs[1]), _lib.ptr(imgs[2]), _lib.ptr(h), _lib.ptr(v), _lib.ptr(out), H, W, C, D,
            1 if subpixel else 0, _lib.ptr(lut), _lib.ptr(ws), ws.numel(), N, _lib.stream_ptr(dev), 7, 1, 0, taps, prm, uniq)
    with _lib.torch_mod().cuda.device(dev):
        if info is None:
            _lib.call("vppb200_compute_rsgm_uniq", *args, what=what)
        else:
            _lib.call("vppb200_compute_rsgm_info", *args, *(_lib.ptr(t) for t in info), what=what)


def _info_tensors(torch, N, H, W, dev):
    """(state uint8, cost, rival uint16 as int16 storage) [N,H,W] on dev"""
    return (torch.empty((N, H, W), dtype=torch.uint8, device=dev), torch.empty((N, H, W), dtype=_lib.u16_dtype(), device=dev),
            torch.empty((N, H, W), dtype=_lib.u16_dtype(), device=dev))


def _uniq(honor_uniqueness, uniqueness, what):
    """the validated uniqueness ratio (TypeError before any device work), or 1.0 = the reference's plain first arg-min"""
    return _lib.uniqueness(uniqueness, what) if honor_uniqueness else 1.0


def compute_rsgm(left, left_vpp, right_vpp, hints=None, validhints=None, dmax=192, p1=11, p2min=17, alpha=0.5, gamma=35,
                 uniqueness=0.95, subpixel=True, rcp_lut=None, honor_params=False, honor_uniqueness=False, return_info=False):
    """compute_rsgm(...) -> float32 [H,W] disparity  (models/rsgm/rsgm.py:250-294).

    p1, p2min, alpha, gamma and uniqueness are accepted for signature compatibility and have no effect by default, exactly as in
    the reference (RSGM/pyrSGM.cpp:519 vs :557-560; StereoBMHelper.cpp:717,:745).  `honor_params=True` (extra) makes p1, p2min,
    alpha and gamma take effect (the keyword of pyrSGM.aggregate_SSE; ValueError for values outside 0..65535 or a negative or
    non-finite alpha).  Parameters outside the sweeps' domain (include/vppstereo_b200.h) are computed exactly but by slower
    per-path kernels.  `honor_uniqueness=True` (extra, independent of honor_params) makes uniqueness take effect in both WTA views:
    a pixel whose best cost is not within uniqueness of its best rival's is invalid (-10 before the tail; TypeError unless
    0 < uniqueness <= 1).  `rcp_lut` (extra, optional) overrides the host-CPU RCPSS table used by the sub-pixel step (for golden
    vectors recorded on another CPU).

    `return_info=True` (extra) returns (disp, info) with how each left pixel's value was produced, shaped like disp:
    info["state"] uint8 (STATE_* of this module: a measured match, an interpolated gap, or which check sent the pixel to the
    background fill), info["cost"] / info["rival"] uint16 (the aggregated cost of the winning disparity and the least cost of a
    disparity at least 2 away from it, 65535 if none: the quantities behind the uniqueness ratio, reported whether or not it is
    honoured).  numpy in -> numpy maps, CUDA tensors in -> CUDA tensors (uint16 travels as _lib.u16_dtype() storage).  disp is
    bit for bit what the call returns without it."""
    prm = _params(honor_params, p1, p2min, alpha, gamma)
    uq = _uniq(honor_uniqueness, uniqueness, "compute_rsgm")
    torch, was_numpy, batched, imgs, h, v, (N, H, W, C) = _prep(left, left_vpp, right_vpp, hints, validhints, int(dmax))
    out = torch.empty((N, H, W), dtype=torch.float32, device=imgs[1].device)
    info = _info_tensors(torch, N, H, W, imgs[1].device) if return_info else None
    _compute("compute_rsgm", imgs, h, v, out, int(dmax), subpixel, rcp_lut, prm, None, uq, info)
    res = out if batched else out[0]
    res = res.cpu().numpy() if was_numpy else res
    if not return_info:
        return res
    maps = {}
    for k, t, np_dtype in zip(("state", "cost", "rival"), info, (np.uint8, np.uint16, np.uint16)):
        t = t if batched else t[0]
        maps[k] = _lib.dev_to_np(t, np_dtype) if was_numpy else t
    return res, maps


def compute_rsgm_stages(left, left_vpp, right_vpp, hints=None, validhints=None, dmax=192, subpixel=True, rcp_lut=None, p1=11,
                        p2min=17, alpha=0.5, gamma=35, honor_params=False, uniqueness=0.95, honor_uniqueness=False, return_info=False):
    """Same pipeline, also returning the stage taps used by the parity tests: dict with padded `census_l/r` (uint32),
    `dsi_agg` (uint16 [Hp,Wp,D]), `disp_l/r` (float32 [Hp,Wp] after median + interpolation + clip) and `out`.
    p1 .. honor_uniqueness as in compute_rsgm; return_info=True adds compute_rsgm's `state`, `cost` and `rival` maps (numpy)."""
    prm = _params(honor_params, p1, p2min, alpha, gamma)
    uq = _uniq(honor_uniqueness, uniqueness, "compute_rsgm_stages")
    torch, was_numpy, batched, imgs, h, v, (N, H, W, C) = _prep(left, left_vpp, right_vpp, hints, validhints, int(dmax))
    dev = imgs[1].device
    D = int(dmax)
    pad_h, pad_w = (((H // 16) + 1) * 16 - H) % 16, (((W // 16) + 1) * 16 - W) % 16
    Hp, Wp = H + pad_h, W + pad_w
    out = torch.empty((N, H, W), dtype=torch.float32, device=dev)
    cl = torch.empty((N, Hp, Wp), dtype=torch.int32, device=dev)
    cr = torch.empty_like(cl)
    S = torch.empty((N, Hp, Wp, D), dtype=torch.int16, device=dev)
    dl = torch.empty((N, Hp, Wp), dtype=torch.float32, device=dev)
    dr = torch.empty_like(dl)
    taps = _lib.RsgmTaps(cl.data_ptr(), cr.data_ptr(), S.data_ptr(), dl.data_ptr(), dr.data_ptr())
    info = _info_tensors(torch, N, H, W, dev) if return_info else None
    _compute("compute_rsgm_stages", imgs, h, v, out, D, subpixel, rcp_lut, prm, taps, uq, info)
    torch.cuda.synchronize(dev)
    res = dict(census_l=_lib.dev_to_np(cl, np.uint32), census_r=_lib.dev_to_np(cr, np.uint32),
               dsi_agg=_lib.dev_to_np(S, np.uint16), disp_l=dl.cpu().numpy(), disp_r=dr.cpu().numpy(),
               out=out.cpu().numpy())
    if return_info:
        res.update((k, _lib.dev_to_np(t, dt)) for k, t, dt in zip(("state", "cost", "rival"), info, (np.uint8, np.uint16, np.uint16)))
    return res
