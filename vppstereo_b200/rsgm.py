"""Drop-in for models/rsgm/rsgm.py: `compute_rsgm` with the reference's signature, running entirely on the device.

    from vppstereo_b200.rsgm import compute_rsgm          # instead of  from models.rsgm.rsgm import compute_rsgm

numpy in -> numpy out (test.py:210-225 keeps working unchanged); CUDA tensors in -> CUDA tensor out with no host
round-trip.  A leading batch dimension [N,H,W(,C)] is accepted and processed as one launch sequence.
"""
import numpy as np

from . import _lib

__all__ = ["compute_rsgm", "compute_rsgm_stages"]


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
    """ctypes pointer to the validated parameters (ValueError before any device work), or None = the reference's effective ones"""
    return _lib.C.byref(_lib.sgm_params(p1, p2min, alpha, gamma)) if honor_params else None


def compute_rsgm(left, left_vpp, right_vpp, hints=None, validhints=None, dmax=192, p1=11, p2min=17, alpha=0.5, gamma=35,
                 uniqueness=0.95, subpixel=True, rcp_lut=None, honor_params=False):
    """compute_rsgm(...) -> float32 [H,W] disparity  (models/rsgm/rsgm.py:250-294).

    p1, p2min, alpha, gamma and uniqueness are accepted for signature compatibility and have no effect, exactly as in
    the reference (RSGM/pyrSGM.cpp:519 vs :557-560; StereoBMHelper.cpp:717,:745).  `honor_params=True` (extra) makes p1, p2min,
    alpha and gamma take effect (the keyword of pyrSGM.aggregate_SSE; ValueError for values outside 0..65535 or a negative or
    non-finite alpha).  Parameters outside the sweeps' domain (include/vppstereo_b200.h) are computed exactly but by slower
    per-path kernels.  `rcp_lut` (extra, optional) overrides the host-CPU RCPSS table used by the sub-pixel step (for golden
    vectors recorded on another CPU)."""
    prm = _params(honor_params, p1, p2min, alpha, gamma)
    torch, was_numpy, batched, imgs, h, v, (N, H, W, C) = _prep(left, left_vpp, right_vpp, hints, validhints, int(dmax))
    L = _lib.lib()
    dev = imgs[1].device
    out = torch.empty((N, H, W), dtype=torch.float32, device=dev)
    need = L.vppb200_rsgm_workspace_bytes(H, W, C, int(dmax), N)
    ws = _lib.workspace(need, dev, "rsgm")
    lut = None
    if rcp_lut is not None:
        lut = rcp_lut if _lib.is_tensor(rcp_lut) else _lib.np_to_dev(rcp_lut, np.float32)
    with torch.cuda.device(dev):
        rc = L.vppb200_compute_rsgm_ex(_lib.ptr(imgs[0]), _lib.ptr(imgs[1]), _lib.ptr(imgs[2]), _lib.ptr(h), _lib.ptr(v),
                                       _lib.ptr(out), H, W, C, int(dmax), 1 if subpixel else 0, _lib.ptr(lut), _lib.ptr(ws),
                                       _lib.C.c_size_t(ws.numel()), N, _lib.stream_ptr(dev), 7, 1, 0, None, prm)
    _lib.check(rc, "compute_rsgm")
    res = out if batched else out[0]
    return res.cpu().numpy() if was_numpy else res


def compute_rsgm_stages(left, left_vpp, right_vpp, hints=None, validhints=None, dmax=192, subpixel=True, rcp_lut=None, p1=11,
                        p2min=17, alpha=0.5, gamma=35, honor_params=False):
    """Same pipeline, also returning the stage taps used by the parity tests: dict with padded `census_l/r` (uint32),
    `dsi_agg` (uint16 [Hp,Wp,D]), `disp_l/r` (float32 [Hp,Wp] after median + interpolation + clip) and `out`.
    p1 .. honor_params as in compute_rsgm."""
    prm = _params(honor_params, p1, p2min, alpha, gamma)
    torch, was_numpy, batched, imgs, h, v, (N, H, W, C) = _prep(left, left_vpp, right_vpp, hints, validhints, int(dmax))
    L = _lib.lib()
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
    need = L.vppb200_rsgm_workspace_bytes(H, W, C, D, N)
    ws = _lib.workspace(need, dev, "rsgm")
    lut = None
    if rcp_lut is not None:
        lut = rcp_lut if _lib.is_tensor(rcp_lut) else _lib.np_to_dev(rcp_lut, np.float32)
    with torch.cuda.device(dev):
        rc = L.vppb200_compute_rsgm_ex(_lib.ptr(imgs[0]), _lib.ptr(imgs[1]), _lib.ptr(imgs[2]), _lib.ptr(h), _lib.ptr(v),
                                       _lib.ptr(out), H, W, C, D, 1 if subpixel else 0, _lib.ptr(lut), _lib.ptr(ws),
                                       _lib.C.c_size_t(ws.numel()), N, _lib.stream_ptr(dev), 7, 1, 0, _lib.C.byref(taps), prm)
    _lib.check(rc, "compute_rsgm_stages")
    torch.cuda.synchronize(dev)
    return dict(census_l=_lib.dev_to_np(cl, np.uint32), census_r=_lib.dev_to_np(cr, np.uint32),
                dsi_agg=_lib.dev_to_np(S, np.uint16), disp_l=dl.cpu().numpy(), disp_r=dr.cpu().numpy(),
                out=out.cpu().numpy())
