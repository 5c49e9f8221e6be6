"""Drop-in for vpp_standalone.py: `vpp(left, right, gt, ...) -> (lc, rc)` with the reference's signature and numba
arithmetic (everything float64, round half to even; vpp_standalone.py:14-369), running on the device.

    from vppstereo_b200.vpp_standalone import vpp        # instead of  from vpp_standalone import vpp   (test.py:16)

numpy in -> numpy copies out (inputs untouched, vpp_standalone.py:397); CUDA tensors in -> CUDA tensors out.  The
reference's numba generator is never seeded by test.py (SURVEY.md 8c.5), so its random pattern is not reproducible;
here the pattern comes from `pattern=` (extra keyword, uint8 stream in draw order) or from a torch generator.
`vpp_to_network` adds the device hand-off of test.py:179-197 (uint8 HWC -> float32 CHW / 255, replicate pad).
"""
import functools
import math

import numpy as np

from . import _lib
from . import vpp_core_opt as _core

__all__ = ["vpp", "vpp_to_network", "network_to_vpp", "sample_hints"]


def vpp(left, right, gt, wsize=3, wsizeAgg_x=64, wsizeAgg_y=3, left2right=True, blending=0.4, use_distance_patch=False,
        use_bilateral_patch=False, distance_gamma=0.3, bilateral_o_xy=2, bilateral_o_i=1, bilateral_th=.001,
        uniform_color=False, method="rnd", c_occ=0.00, g_occ=None, discard_occ=False, interpolate=True, pattern=None,
        seed=None):
    assert method in ["rnd", "maxDistance"]                                  # vpp_standalone.py:400
    torch = _lib.require_cuda()
    host = not _lib.is_tensor(left)
    lc = _lib.as_device(left, torch.uint8).clone()
    rc = _lib.as_device(right, torch.uint8).clone()
    g = _lib.as_device(gt, torch.float32)                                    # gt.astype(np.float32) (:398)
    direction = 1 if left2right else 0
    batched = g.dim() == 3
    if lc.dim() == g.dim():                                                  # gray: add the channel axis (:403-404)
        lc, rc = lc.unsqueeze(-1), rc.unsqueeze(-1)
    lc, rc = lc.contiguous(), rc.contiguous()
    H, W = g.shape[-2:]
    Cn = lc.shape[-1]
    if True:   # frames without points are left untouched by the scan itself (vpp_standalone.py:407-408): no host sync needed
        if g_occ is None:
            occ = torch.zeros(g.shape, dtype=torch.uint8, device=g.device)   # np.zeros_like(gt) (:424-425)
        else:
            occ = (_lib.as_device(g_occ, torch.float32) != 0).to(torch.uint8)
        adaptive = None
        if use_distance_patch or use_bilateral_patch:
            adaptive = _adaptive_operands(lc, g, wsize, bool(use_distance_patch), bool(use_bilateral_patch), distance_gamma,
                                          bilateral_o_xy, bilateral_o_i, bilateral_th)
        if method == "maxDistance":
            _core._scan("max_dist", lc, rc, g, W, H, Cn, uniform_color, wsize, (wsizeAgg_x, wsizeAgg_y), direction,
                        blending, c_occ, occ, discard_occ, interpolate, None, 1, want_counts=False, adaptive=adaptive)
        else:
            # no pattern given: counter-based generation inside the splat kernel (the reference's numba RNG is unseeded)
            rng_seed = None
            if pattern is None:
                rng_seed = int(seed) if seed is not None else int.from_bytes(__import__("os").urandom(8), "little")
                rng_seed |= 1 << 63                  # a given seed of 0 must still select the device generator
            _core._scan("rnd", lc, rc, g, W, H, Cn, uniform_color, wsize, None, direction, blending, c_occ, occ,
                        discard_occ, interpolate, pattern, 1, device_rng_seed=rng_seed, want_counts=False, adaptive=adaptive)
    if host:
        return lc.cpu().numpy(), rc.cpu().numpy()
    return lc, rc


# ---- adaptive patches (TPAMI extension; vpp_standalone.py:6-11, :371-394, :410-422) ----------------------------------
@functools.lru_cache(maxsize=16)
def _bilateral_weights(n, o_xy, o_i):
    """exp(-((yw^2+xw^2)/(2 o_xy^2) + di^2/(2 o_i^2))) for every patch offset and absolute intensity difference, evaluated
    with the host's libm on Python numbers of the caller's types -- the very expression and function numba evaluates
    (vpp_standalone.py:387), so the device kernel only compares tabulated float64 weights."""
    out = np.empty(((2 * n + 1) ** 2, 256), np.float64)
    for yw in range(-n, n + 1):
        for xw in range(-n, n + 1):
            row = out[(yw + n) * (2 * n + 1) + (xw + n)]
            for di in range(256):
                row[di] = math.exp(-(((yw) ** 2 + (xw) ** 2) / (2 * (o_xy ** 2)) + ((di) ** 2) / (2 * (o_i ** 2))))
    return out


def _patch_size(d, dmin, dmax, patch_size, gamma):
    """wsize of _get_patch_size_based_on_distance (vpp_standalone.py:6-9) in numba's typing: float32 ratio, float64 pow
    (libm, as Python's **), round half to even."""
    ratio = np.float32(np.float32(d) - dmin) / np.float32(dmax - dmin)
    return round((float(ratio) ** (1 / gamma)) * (patch_size - 1) + 1)


def _patch_thresholds(dmin, dmax, patch_size, gamma):
    """The patch size is a non-decreasing step function of the (float32) disparity: return, for k = 2..patch_size, the smallest
    float32 d in [dmin, dmax] whose size is >= k (inf if none), found by bisection on the float32 bit patterns with the exact
    host evaluation above.  The device then needs no pow(): size = 1 + #{k : d >= thr_k}."""
    dmin, dmax = np.float32(dmin), np.float32(dmax)
    if dmin == dmax:
        raise ZeroDivisionError("division by zero")          # numba's python error model on (d_max - d_min) == 0 (:7)
    lo_bits, hi_bits = int(dmin.view(np.int32)), int(dmax.view(np.int32))
    f32 = lambda b: np.array(b, np.int32).view(np.float32)[()]
    thr = np.full(patch_size - 1, np.inf, np.float32)
    for k in range(2, patch_size + 1):
        if _patch_size(dmax, dmin, dmax, patch_size, gamma) < k:
            break
        lo, hi = lo_bits, hi_bits                            # invariant: size(hi) >= k
        if _patch_size(dmin, dmin, dmax, patch_size, gamma) >= k:
            hi = lo
        while lo < hi:
            mid = (lo + hi) // 2
            if _patch_size(f32(mid), dmin, dmax, patch_size, gamma) >= k:
                hi = mid
            else:
                lo = mid + 1
        thr[k - 2] = f32(hi)
    return thr


@functools.lru_cache(maxsize=16)
def _ratio_steps(patch_size, gamma):
    """R_k for k = 2..patch_size: the smallest float32 ratio in [0, 1] whose patch size is >= k (vpp_standalone.py:6-9), float32
    [patch_size-1].  With dmin = 0 and dmax = 1 the ratio of _patch_size is d itself, so these are _patch_thresholds(0, 1): the
    only evaluation of pow(), with the host's libm.  vppb200_distance_patch_thresholds turns them into each frame's disparity
    thresholds on the device.  (Read-only: the array is shared by every caller.)"""
    steps = _patch_thresholds(np.float32(0.0), np.float32(1.0), int(patch_size), gamma)
    steps.setflags(write=False)
    return steps


def distance_patch_thresholds(g, patch_size, ratio_steps, thr_out, status_out, stream):
    """Queue vppb200_distance_patch_thresholds on `stream` (a raw stream handle): g float32 [N,H,W] CUDA, ratio_steps the device
    copy of _ratio_steps(patch_size, gamma), thr_out float32 [N, patch_size-1] (None when patch_size == 1), status_out int32 [N]
    (set to 1 for a frame whose hints all have one value)."""
    N, H, W = g.shape
    _lib.call("vppb200_distance_patch_thresholds", _lib.ptr(g), W, H, _lib.ptr(ratio_steps), int(patch_size), _lib.ptr(thr_out),
              _lib.ptr(status_out), N, stream, what="distance_patch_thresholds")


def bilateral_filling(g, left, n_patch, weights, th, gray_out, filled_out, stream):
    """Queue the bilateral filling of the hints g float32 [N,H,W] (vpp_standalone.py:371-394) with the gray context of the
    un-projected left image uint8 [N,H,W,C] (:414-417) on `stream`: gray_out uint8 [N,H,W], filled_out float32 [N,H,W];
    weights = the device copy of _bilateral_weights(n_patch, o_xy, o_i)."""
    N, H, W = g.shape
    _lib.call("vppb200_bgr2gray", _lib.ptr(left), _lib.ptr(gray_out), W, H, int(left.shape[-1]), N, stream, what="bgr2gray")
    _lib.call("vppb200_bilateral_filling", _lib.ptr(g), _lib.ptr(gray_out), _lib.ptr(filled_out), W, H, int(n_patch),
              _lib.ptr(weights), float(th), N, stream, what="bilateral_filling")


def _adaptive_operands(lc, g, wsize, use_distance, use_bilateral, gamma, o_xy, o_i, th):
    """(filled_g or None, thresholds or None) as device tensors for the adaptive scans."""
    torch = _lib.torch_mod()
    batched = g.dim() == 3
    gg = (g if batched else g[None]).contiguous()
    N, H, W = gg.shape
    n = (int(wsize) - 1) // 2
    filled = thr = None
    with torch.cuda.device(g.device):
        st = _lib.stream_ptr(g.device)
        if use_distance:
            steps = torch.from_numpy(_ratio_steps(int(wsize), gamma).copy()).to(g.device)
            thr = torch.empty((N, max(int(wsize) - 1, 0)), dtype=torch.float32, device=g.device) if int(wsize) > 1 else None
            status = torch.zeros(N, dtype=torch.int32, device=g.device)
            distance_patch_thresholds(gg, int(wsize), steps, thr, status, st)
            bad = np.flatnonzero(status.cpu().numpy())
            if bad.size:      # numba's python error model on (d_max - d_min) == 0 (:7), before any scan work
                raise ZeroDivisionError(f"division by zero (frame {int(bad[0])}: every hint has the same disparity)")
        if use_bilateral:
            ll = (lc if batched else lc[None]).contiguous()
            wt = torch.from_numpy(_bilateral_weights(n, o_xy, o_i)).to(g.device)
            gray = torch.empty((N, H, W), dtype=torch.uint8, device=g.device)
            filled = torch.empty_like(gg)
            bilateral_filling(gg, ll, n, wt, th, gray, filled, st)
    return filled, thr


def vpp_to_network(img_u8, pad_to=32):
    """uint8 [H,W,C] / [N,H,W,C] CUDA tensor -> float32 [N,C,H+pad,W+pad] = float32(u8/255.) with the symmetric
    replicate padding of test.py:187-197 (pad_to=None: no padding).  Returns (tensor, (left,right,top,bottom))."""
    torch = _lib.require_cuda()
    t = _lib.as_device(img_u8, torch.uint8)
    if t.dim() == 3:
        t = t[None]
    t = t.contiguous()
    N, H, W, Cn = t.shape
    pad_h = pad_w = 0
    if pad_to:
        pad_h = (((H // pad_to) + 1) * pad_to - H) % pad_to
        pad_w = (((W // pad_to) + 1) * pad_to - W) % pad_to
    pl, pr, pt, pb = pad_w // 2, pad_w - pad_w // 2, pad_h // 2, pad_h - pad_h // 2
    out = torch.empty((N, Cn, H + pad_h, W + pad_w), dtype=torch.float32, device=t.device)
    with torch.cuda.device(t.device):
        _lib.call("vppb200_u8hwc_to_f32chw", _lib.ptr(t), _lib.ptr(out), H, W, Cn, pt, pb, pl, pr, N, _lib.stream_ptr(t.device),
                  what="vpp_to_network")
    return out, (pl, pr, pt, pb)


def network_to_vpp(img_f32):
    """float32 [C,H,W] / [N,C,H,W] CUDA tensor in [0,1] (the loader's normalised image) -> uint8 [H,W,C] / [N,H,W,C] =
    (255*im.permute(1,2,0)).astype(np.uint8) of test.py:158-159,:210-212, on the device."""
    torch = _lib.require_cuda()
    t = _lib.as_device(img_f32, torch.float32)
    single = t.dim() == 3
    if single:
        t = t[None]
    t = t.contiguous()
    N, Cn, H, W = t.shape
    out = torch.empty((N, H, W, Cn), dtype=torch.uint8, device=t.device)
    with torch.cuda.device(t.device):
        _lib.call("vppb200_f32chw_to_u8hwc", _lib.ptr(t), _lib.ptr(out), H, W, Cn, N, _lib.stream_ptr(t.device),
                  what="network_to_vpp")
    return out[0] if single else out


def sample_hints(hints, validhints, probability=0.20, generator=None):
    """losses.py:5-10 on whatever device the tensors live on (torch ops only: plumbing, no kernel of ours)."""
    torch = _lib.torch_mod()
    rnd = torch.rand(validhints.shape, dtype=torch.float32, device=validhints.device, generator=generator)
    new_validhints = (validhints * (rnd < probability)).float()
    new_hints = hints * new_validhints
    new_hints[new_validhints == 0] = 0
    return new_hints, new_validhints
