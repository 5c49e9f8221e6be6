"""Drop-in for the reference's Cython module `vpp_core_opt` (vpp_core/vpp_core_opt.pyx): same callables and positional
signatures, `l` and `r` mutated in place, number of hints returned.  Arithmetic mode = Cython (c as float32).

The reference draws its random pattern from libc `rand()` while scanning.  `init_rand(seed)` here seeds a restatement
of glibc's generator (C-ABI vppb200_glibc_srand / _rand_fill), so after `init_rand(s)` the scans consume exactly the
stream the reference consumes after its `init_rand(s)`; a pre-drawn `pattern=` (uint8) may be passed instead.

numpy arrays (host) or CUDA tensors (device, no host round-trip) are accepted; a leading batch dimension is allowed
on l, r, g, g_occ for CUDA tensors (patterns are then concatenated frame by frame).
"""
import ctypes as C
import time

import numpy as np

from . import _lib

__all__ = ["get_seed", "init_rand", "virtual_projection_scan_rnd", "virtual_projection_scan_max_dist", "gt_reshape",
           "draws_per_frame", "draw_pattern", "device_pattern"]

_state = None


def get_seed():
    """Wall-clock seed (vpp_core_opt.pyx:23-28)."""
    return time.time()


def init_rand(_seed=0):
    """srand((int)_seed) on the library-private glibc-compatible generator (vpp_core_opt.pyx:33-35)."""
    global _state
    _state = (C.c_uint32 * 34)()
    seed = int(_seed) & 0xFFFFFFFF                # <int> cast of the Python number, then srand(unsigned)
    _lib.call("vppb200_glibc_srand", _state, seed, what="init_rand")


def draw_pattern(n):
    """Next n values of rand() % 256 from the generator seeded by init_rand (default seed 1, as libc)."""
    if _state is None:
        init_rand(1)
    out = np.empty(int(n), np.uint8)
    _lib.call("vppb200_glibc_rand_fill", _state, out.ctypes.data, int(n), what="draw_pattern")
    return out


def device_pattern(rng_seed, frame, n):
    """The first n values of the on-device pattern stream of `frame` (index inside the batch of one call) for `rng_seed`:
    host restatement of csrc/vpp.cu::counter_pattern, the generator the scans use when no pattern is passed
    (vppb200_vpp_scan_rnd with pattern = NULL).  Pure integer arithmetic; lets a caller (and the parity tests) replay on the
    host exactly what the device drew."""
    M32 = np.uint64(0xFFFFFFFF)
    k = np.uint64(int(rng_seed) & (2**64 - 1)) ^ np.uint64((int(frame) * 0x9E3779B97F4A7C15) & (2**64 - 1))
    key = np.uint32(int(k & M32) ^ ((int(k >> np.uint64(32)) * 0x85EBCA6B) & 0xFFFFFFFF))
    idx = np.arange(int(n), dtype=np.uint64)
    h = ((idx * np.uint64(0x9E3779B1)) & M32) ^ np.uint64(key)
    h ^= h >> np.uint64(16); h = (h * np.uint64(0x85EBCA6B)) & M32
    h ^= h >> np.uint64(13); h = (h * np.uint64(0xC2B2AE35)) & M32
    h ^= h >> np.uint64(16)
    return (h >> np.uint64(24)).astype(np.uint8)


def draws_per_frame(g, wsize, channels, uniform_color):
    """Pattern draws one scan of frame(s) g consumes (SURVEY.md A.1.6): per hint C * (#in-image patch pixels), or C."""
    if _lib.is_tensor(g):
        torch = _lib.torch_mod()
        gg = g.reshape((-1,) + tuple(g.shape[-2:]))
        H, W = gg.shape[-2:]
        n = (int(wsize) - 1) // 2
        hit = gg > 0
        if uniform_color:
            return (hit.sum(dim=(1, 2)) * channels).cpu().numpy().astype(np.int64)
        ys = torch.arange(H, device=g.device)
        xs = torch.arange(W, device=g.device)
        ny = (torch.clamp(ys + n, max=H - 1) - torch.clamp(ys - n, min=0) + 1).to(torch.int64)
        nx = (torch.clamp(xs + n, max=W - 1) - torch.clamp(xs - n, min=0) + 1).to(torch.int64)
        w = ny[:, None] * nx[None, :]
        return ((hit * w).sum(dim=(1, 2)) * channels).cpu().numpy().astype(np.int64)
    gg = np.asarray(g).reshape((-1,) + np.asarray(g).shape[-2:])
    H, W = gg.shape[-2:]
    n = (int(wsize) - 1) // 2
    hit = gg > 0
    if uniform_color:
        return hit.sum(axis=(1, 2)).astype(np.int64) * channels
    ys, xs = np.arange(H), np.arange(W)
    ny = np.minimum(ys + n, H - 1) - np.maximum(ys - n, 0) + 1
    nx = np.minimum(xs + n, W - 1) - np.maximum(xs - n, 0) + 1
    return (hit * (ny[:, None] * nx[None, :])).sum(axis=(1, 2)).astype(np.int64) * channels


def _check_views(l, r, g, g_occ, width, height, channels):
    for name, a, nd in (("l", l, 3), ("r", r, 3), ("g", g, 2), ("g_occ", g_occ, 2)):
        dims = a.dim() if _lib.is_tensor(a) else np.ndim(a)
        if dims not in (nd, nd + 1):
            raise ValueError(f"Buffer has wrong number of dimensions (expected {nd}, got {dims})")   # Cython memoryview error
    if not _lib.is_tensor(l):
        if l.dtype != np.uint8 or r.dtype != np.uint8:
            raise ValueError("Buffer dtype mismatch, expected 'uint8_t'")
        if np.asarray(g).dtype != np.float32:
            raise ValueError("Buffer dtype mismatch, expected 'float'")
        if np.asarray(g_occ).dtype != np.uint8:
            raise ValueError("Buffer dtype mismatch, expected 'uint8_t'")


def _scan(kind, l, r, g, width, height, channels, uniform_color, wsize, wagg, direction, c, c_occ, g_occ,
          discard_occluded, interpolate, pattern, arith, device_rng_seed=None, want_counts=True, adaptive=None, rows=None):
    width, height, channels, wsize, direction = int(width), int(height), int(channels), int(wsize), int(direction)
    _check_views(l, r, g, g_occ, width, height, channels)
    torch = _lib.require_cuda()
    host = not _lib.is_tensor(l)
    lt = _lib.as_device(l, torch.uint8)
    rt = _lib.as_device(r, torch.uint8)
    gt = _lib.as_device(g, torch.float32)
    ot = _lib.as_device(g_occ, torch.uint8)
    if host or lt.data_ptr() != l.data_ptr() or rt.data_ptr() != r.data_ptr():
        if not host:
            raise ValueError("l and r must be contiguous CUDA uint8 tensors (they are updated in place)")
    n = lt.numel() // (width * height * channels)
    if n < 1 or n * width * height * channels != lt.numel() or rt.numel() != lt.numel() or gt.numel() != n * width * height:
        raise ValueError("operand sizes do not match width/height/channels")
    L = _lib.lib()
    dev = lt.device
    if kind == "rnd":
        ws = _lib.workspace(L.vppb200_vpp_workspace_bytes(height, width, channels, n), dev, "vpp")
    else:
        ws = _lib.workspace(L.vppb200_vpp_max_dist_workspace_bytes(height, width, channels, wsize, int(wagg[1]), n), dev, "vpp")
    counts = torch.empty(n, dtype=torch.int32, device=dev)
    # Cython receives c, c_occ as C float; numba as Python floats
    cc, co = float(c), float(c_occ)
    filled, thr = adaptive if adaptive is not None else (None, None)
    adaptive_on = filled is not None or thr is not None
    n_thr = int(thr.shape[-1]) if thr is not None else 0
    what = "virtual_projection_scan_" + kind
    with torch.cuda.device(dev):
        # operands of the five scan entry points: the image / blend operands and the trailing five are the same for all of them
        img = (_lib.ptr(lt), _lib.ptr(rt), _lib.ptr(gt), width, height, channels, int(bool(uniform_color)), wsize)
        blend = (cc, co, _lib.ptr(ot), int(bool(discard_occluded)), int(bool(interpolate)), int(arith))
        tail = (_lib.ptr(counts), _lib.ptr(ws), ws.numel(), n, _lib.stream_ptr(dev))
        if kind == "rnd":
            pt = ot_off = None
            if device_rng_seed is None:
                if adaptive_on and n > 1:
                    raise ValueError("an explicit pattern with adaptive patches is supported for single frames only "
                                     "(the draws per frame depend on the kept patch pixels); use the device generator")
                # (adaptive patches consume at most the full-patch count: a longer pattern is fine)
                per = draws_per_frame(gt.reshape(n, height, width), wsize, channels, bool(uniform_color))
                offs = np.zeros(n + 1, np.int64)
                offs[1:] = np.cumsum(per)
                if pattern is None:
                    pattern = draw_pattern(int(offs[-1]))
                pt = _lib.as_device(pattern, torch.uint8).reshape(-1)
                if pt.numel() < offs[-1]:
                    raise ValueError(f"pattern too short: need {int(offs[-1])} draws, got {pt.numel()}")
                if pt.numel() == 0:
                    pt = torch.zeros(1, dtype=torch.uint8, device=dev)
                ot_off = torch.from_numpy(offs).to(dev)
            rnd = img + (direction,) + blend + (_lib.ptr(pt), _lib.ptr(ot_off), int(device_rng_seed or 0) & (2**64 - 1))
            if rows is not None:
                if adaptive_on:
                    raise ValueError("row bands are implemented for the fixed-patch rnd scan")
                _lib.call("vppb200_vpp_scan_rnd_rows", *rnd, int(rows[0]), int(rows[1]), *tail, what=what)
            elif adaptive_on:
                _lib.call("vppb200_vpp_scan_rnd_adaptive", *rnd, _lib.ptr(filled), _lib.ptr(thr), n_thr, *tail, what=what)
            else:
                _lib.call("vppb200_vpp_scan_rnd", *rnd, *tail, what=what)
        else:
            md = img + (int(wagg[0]), int(wagg[1]), direction) + blend
            if adaptive_on:
                _lib.call("vppb200_vpp_scan_max_dist_adaptive", *md, _lib.ptr(filled), _lib.ptr(thr), n_thr, *tail, what=what)
            elif rows is not None:
                raise ValueError("maxDistance does not split into independent row bands (SURVEY.md 8e): its windows read the current "
                                 "images")
            else:
                _lib.call("vppb200_vpp_scan_max_dist", *md, *tail, what=what)
    if host:
        np.copyto(l, lt.cpu().numpy().reshape(l.shape))
        np.copyto(r, rt.cpu().numpy().reshape(r.shape))
    if not want_counts:
        return counts                      # device tensor: no host synchronisation
    cnt = counts.cpu().numpy()
    return int(cnt[0]) if n == 1 else cnt


def virtual_projection_scan_rnd(l, r, g, width, height, channels, uniform_color, wsize, direction, c, c_occ, g_occ,
                                discard_occluded, interpolate, pattern=None, arith=0):
    """vpp_core_opt.pyx:53-131.  `pattern` (extra): pre-drawn uint8 stream; default = the init_rand generator."""
    return _scan("rnd", l, r, g, width, height, channels, uniform_color, wsize, None, direction, c, c_occ, g_occ,
                 discard_occluded, interpolate, pattern, arith)


def virtual_projection_scan_max_dist(l, r, g, width, height, channels, uniform_color, wsize, wsize_agg_x, wsize_agg_y,
                                     direction, c, c_occ, g_occ, discard_occluded, interpolate, arith=0):
    """vpp_core_opt.pyx:133-341."""
    return _scan("max_dist", l, r, g, width, height, channels, uniform_color, wsize, (wsize_agg_x, wsize_agg_y), direction, c,
                 c_occ, g_occ, discard_occluded, interpolate, None, arith)


def gt_reshape(_gt):
    """gt_reshape(gt f32[H,W]) -> f32[N,4] rows (x, y, d, 1) in raster order (vpp_core_opt.pyx:352-371)."""
    torch = _lib.require_cuda()
    host = not _lib.is_tensor(_gt)
    gt = _lib.as_device(_gt, torch.float32)
    if gt.dim() != 2:
        raise ValueError("Buffer has wrong number of dimensions (expected 2, got %d)" % gt.dim())
    H, W = gt.shape
    dev = gt.device
    out = torch.zeros((W * H, 4), dtype=torch.float32, device=dev)
    cnt = torch.zeros(1, dtype=torch.int32, device=dev)
    ws = _lib.workspace(_lib.lib().vppb200_vpp_workspace_bytes(H, W, 1, 1), dev, "vpp")
    with torch.cuda.device(dev):
        _lib.call("vppb200_gt_reshape", _lib.ptr(gt), W, H, _lib.ptr(out), _lib.ptr(cnt), _lib.ptr(ws), ws.numel(),
                  _lib.stream_ptr(dev), what="gt_reshape")
    res = out[: int(cnt.item())]
    return res.cpu().numpy() if host else res
