"""Drop-in for the reference's `pyrSGM` extension module (RSGM/pyrSGM.cpp:761-774), RSGM/ =
thirdparty/stereo-vision/reconstruction/base/rSGM/.  Same seven callables, same positional signatures, same in-place
output convention, same TypeError conditions; the work runs in sm_100a kernels behind include/vppstereo_b200.h.

Operands may be numpy arrays (copied to the device and back, so `models/rsgm/rsgm.py` works unchanged with
`import vppstereo_b200.pyrSGM as pyrSGM`) or CUDA tensors (updated in place on the device, no host round-trip;
uint16/uint32 volumes are carried as int16/int32 storage).  A leading batch dimension is accepted on every operand.
"""
import numpy as np

from . import _lib

__all__ = ["census5x5_SSE", "median3x3_SSE", "costMeasureCensus5x5_xyd_SSE", "matchWTA_SSE", "matchWTARight_SSE",
           "aggregate_SSE", "subPixelRefine"]


def _on_operand_device(fn):
    """Run an operator with the device of its first CUDA-tensor operand as the current device (numpy operands: the current
    device): outputs and staging buffers are allocated there, the launch goes to THAT device's current stream, and the library's
    per-device state (reciprocal table, side streams) is the right one -- also when the caller's current device is another GPU."""
    import functools

    @functools.wraps(fn)
    def wrapper(*args, **kwargs):
        dev = next((a.device for a in args if _lib.is_tensor(a) and a.is_cuda), None)
        if dev is None:
            return fn(*args, **kwargs)
        others = [a.device for a in args if _lib.is_tensor(a) and a.is_cuda and a.device != dev]
        if others:
            raise ValueError(f"operands live on different devices ({dev} and {others[0]})")
        with _lib.torch_mod().cuda.device(dev):
            return fn(*args, **kwargs)
    return wrapper


def _frames(numel, per_frame):
    n = numel // per_frame
    if n < 1 or n * per_frame != numel:
        raise ValueError("operand size does not match width/height/dispCount")
    return n


def _writeback(dst, t, np_dtype):
    if isinstance(dst, np.ndarray):
        if not dst.flags.writeable:
            raise ValueError("output array is read-only")
        np.copyto(dst, _lib.dev_to_np(t, np_dtype).reshape(dst.shape))


def _out_operand(dst, np_dtype, copy_in):
    """Output operand: device tensor to write (+ whether to copy back). numpy outputs are staged on the device."""
    if _lib.is_tensor(dst):
        t, _ = _lib.operand(dst, np_dtype, None)
        if t.data_ptr() != dst.data_ptr():
            raise ValueError("output tensor must be contiguous")
        return t
    if not isinstance(dst, np.ndarray):
        raise TypeError("expected a numpy array or a CUDA tensor")
    if dst.dtype != np.dtype(np_dtype):
        raise TypeError(f"output must be {np.dtype(np_dtype)}")
    if copy_in:
        return _lib.np_to_dev(dst, np_dtype)
    torch = _lib.require_cuda()
    signed = {2: torch.int16, 4: torch.int32}
    dt = torch.float32 if np.dtype(np_dtype) == np.float32 else signed[np.dtype(np_dtype).itemsize]
    return torch.empty(dst.size, dtype=dt, device="cuda")


@_on_operand_device
def census5x5_SSE(src, dst, width, height):
    """census5x5_SSE(src u8[H,W], dst u32[H,W], W, H)  RSGM/pyrSGM.cpp:14-95 -> FastFilters.cpp:181-442"""
    width, height = int(width), int(height)
    if width % 16 != 0:
        raise TypeError(f"Width must be a multiple of 16 ({width}x{height})")
    s, _ = _lib.operand(src, np.uint8, None)
    n = _frames(s.numel(), width * height)
    d = _out_operand(dst, np.uint32, False)
    _lib.call("vppb200_census5x5", _lib.ptr(s), _lib.ptr(d), width, height, n, _lib.stream_ptr(), what="census5x5_SSE")
    _writeback(dst, d, np.uint32)


@_on_operand_device
def median3x3_SSE(src, dst, width, height):
    """median3x3_SSE(src f32, dst f32, W, H)  RSGM/pyrSGM.cpp:97-178 -> FastFilters.cpp:701-757"""
    width, height = int(width), int(height)
    if width % 16 != 0:
        raise TypeError(f"Width must be a multiple of 16 ({width}x{height})")
    s, _ = _lib.operand(src, np.float32, None)
    n = _frames(s.numel(), width * height)
    d = _out_operand(dst, np.float32, False)
    _lib.call("vppb200_median3x3", _lib.ptr(s), _lib.ptr(d), width, height, n, _lib.stream_ptr(), what="median3x3_SSE")
    _writeback(dst, d, np.float32)


@_on_operand_device
def costMeasureCensus5x5_xyd_SSE(leftCensus, rightCensus, dsi, width, height, dispCount, numThreads):
    """costMeasureCensus5x5_xyd_SSE(cl, cr, dsi u16[H,W,D], W, H, D, nthreads)  RSGM/pyrSGM.cpp:180-294"""
    width, height, dispCount, numThreads = int(width), int(height), int(dispCount), int(numThreads)
    if width % 16 != 0:
        raise TypeError(f"Width must be a multiple of 16 ({width}x{height})")
    if dispCount % 8 != 0 or dispCount > 256:
        raise TypeError(f"Disparity range must be a multiple of 8 and not greater than 256 ({dispCount})")
    if numThreads not in (1, 2, 4):
        raise TypeError(f"NumThreads must be 1,2,4 ({numThreads})")
    cl, _ = _lib.operand(leftCensus, np.uint32, None)
    cr, _ = _lib.operand(rightCensus, np.uint32, None)
    n = _frames(cl.numel(), width * height)
    d = _out_operand(dsi, np.uint16, False)
    _lib.call("vppb200_cost_census5x5_xyd", _lib.ptr(cl), _lib.ptr(cr), _lib.ptr(d), width, height, dispCount, numThreads, n,
              _lib.stream_ptr(), what="costMeasureCensus5x5_xyd_SSE")
    _writeback(dsi, d, np.uint16)


@_on_operand_device
def aggregate_SSE(img, dsi, dsiAgg, width, height, dispCount, P1, P2min, Alpha, Gamma, honor_params=False):
    """aggregate_SSE(img u8, dsi, dsiAgg, W, H, D, P1, P2min, Alpha, Gamma)  RSGM/pyrSGM.cpp:504-637.
    As upstream, P1/P2min/Alpha/Gamma are parsed and then ignored (effective 7/17/0.25/50, pyrSGM.cpp:519 vs :557-560)
    unless the extra keyword honor_params=True is given.  Only the first W*H bytes of `img` are read (pyrSGM.cpp:586-588)."""
    width, height, dispCount = int(width), int(height), int(dispCount)
    if width % 16 != 0:
        raise TypeError(f"Width must be a multiple of 16 ({width}x{height})")
    if dispCount % 8 != 0 or dispCount > 256:
        raise TypeError(f"Disparity range must be a multiple of 8 and not greater than 256 ({dispCount})")
    P1, P2min, Alpha, Gamma = int(P1), int(P2min), float(Alpha), int(Gamma)     # "HHfH" parse (pyrSGM.cpp:541)
    for v in (P1, P2min, Gamma):
        if not 0 <= v <= 65535:
            raise OverflowError("unsigned short integer out of range")
    s, _ = _lib.operand(dsi, np.uint16, None)
    n = _frames(s.numel(), width * height * dispCount)
    if _lib.is_tensor(img):
        g = img.contiguous().view(-1)
    else:
        g = _lib.np_to_dev(np.ascontiguousarray(img, np.uint8).reshape(-1), np.uint8)
    per = g.numel() // n
    if per < width * height:
        raise ValueError("guide image smaller than width*height")
    if per != width * height:                      # colour buffer: keep the first W*H bytes of each frame
        g = g.view(n, per)[:, : width * height].contiguous()
    d = _out_operand(dsiAgg, np.uint16, False)
    _lib.call("vppb200_aggregate", _lib.ptr(g), _lib.ptr(s), _lib.ptr(d), width, height, dispCount, P1, P2min, Alpha, Gamma,
              int(bool(honor_params)), n, _lib.stream_ptr(), what="aggregate_SSE")
    _writeback(dsiAgg, d, np.uint16)


def _wta(sym, name, dsiAgg, dispImg, width, height, dispCount, uniqueness, honor_uniqueness):
    if honor_uniqueness:
        uniqueness = _lib.uniqueness(uniqueness, name)           # finite, 0 < u <= 1 (NaN included)
        sym += "_uniq"
    width, height, dispCount, uniqueness = int(width), int(height), int(dispCount), float(uniqueness)
    if width % 16 != 0:
        raise TypeError(f"Width must be a multiple of 16 ({width}x{height})")
    if dispCount % 8 != 0 or dispCount > 256:
        raise TypeError(f"Disparity range must be a multiple of 8 and not greater than 256 ({dispCount})")
    if uniqueness > 1.0 or uniqueness <= 0.0:
        raise TypeError(f"Uniqueness must be inside ]0,1] ({uniqueness})")
    s, _ = _lib.operand(dsiAgg, np.uint16, None)
    n = _frames(s.numel(), width * height * dispCount)
    d = _out_operand(dispImg, np.float32, False)
    _lib.call(sym, _lib.ptr(s), _lib.ptr(d), width, height, dispCount, uniqueness, n, _lib.stream_ptr(), what=name)
    _writeback(dispImg, d, np.float32)


@_on_operand_device
def matchWTA_SSE(dsiAgg, dispImg, width, height, dispCount, uniqueness, honor_uniqueness=False):
    """matchWTA_SSE(dsiAgg u16, disp f32[H,W], W, H, D, uniqueness)  RSGM/pyrSGM.cpp:296-397.
    As upstream, uniqueness is validated and then has no effect unless the extra keyword honor_uniqueness=True is given: then a
    pixel whose best cost is not below uniqueness times its best rival's (include/vppstereo_b200.h) gets -10."""
    _wta("vppb200_match_wta", "matchWTA_SSE", dsiAgg, dispImg, width, height, dispCount, uniqueness, honor_uniqueness)


@_on_operand_device
def matchWTARight_SSE(dsiAgg, dispImg, width, height, dispCount, uniqueness, honor_uniqueness=False):
    """matchWTARight_SSE(dsiAgg u16, disp f32[H,W], W, H, D, uniqueness)  RSGM/pyrSGM.cpp:399-502; honor_uniqueness as in
    matchWTA_SSE."""
    _wta("vppb200_match_wta_right", "matchWTARight_SSE", dsiAgg, dispImg, width, height, dispCount, uniqueness, honor_uniqueness)


@_on_operand_device
def subPixelRefine(dsi, dispImg, width, height, dispCount, method, rcp_lut=None):
    """subPixelRefine(dsi u16, disp f32 (read and written), W, H, D, method)  RSGM/pyrSGM.cpp:639-741.
    rcp_lut (extra, optional): 65536-entry RCPSS table recorded on another CPU (golden vectors); default = this host's."""
    width, height, dispCount, method = int(width), int(height), int(dispCount), int(method)
    if width % 16 != 0:
        raise TypeError(f"Width must be a multiple of 16 ({width}x{height})")
    if dispCount % 8 != 0 or dispCount > 256:
        raise TypeError(f"Disparity range must be a multiple of 8 and not greater than 256 ({dispCount})")
    if method not in (0, 1):
        raise TypeError(f"method must be inside {{0,1}} ({method})")
    s, _ = _lib.operand(dsi, np.uint16, None)
    n = _frames(s.numel(), width * height * dispCount)
    d = _out_operand(dispImg, np.float32, True)
    lut = _lib.np_to_dev(rcp_lut, np.float32) if rcp_lut is not None and not _lib.is_tensor(rcp_lut) else rcp_lut
    _lib.call("vppb200_subpixel_refine", _lib.ptr(s), _lib.ptr(d), width, height, dispCount, method, _lib.ptr(lut), n,
              _lib.stream_ptr(), what="subPixelRefine")
    _writeback(dispImg, d, np.float32)
