"""ctypes binding of the C-ABI library (include/vppstereo_b200.h) plus the torch plumbing around it.

PyTorch is used for device memory, streams and torch.distributed only.  There is NO CPU implementation: importing a
front-end module works anywhere (so argument validation can be tested), but any compute call raises unless the CUDA
library is built and a CUDA device is present.
"""
import ctypes as C
import os

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(HERE, "libvppstereo_b200.so")

OK = 0
ERR_WIDTH, ERR_DISP, ERR_THREADS, ERR_UNIQUENESS, ERR_METHOD, ERR_WORKSPACE, ERR_ARG, ERR_CUDA = -1, -2, -3, -4, -5, -6, -7, -100
# codes of the per-pixel match state (include/vppstereo_b200.h: VPPB200_STATE_*)
STATE_MATCHED, STATE_INTERPOLATED, STATE_NO_MATCH, STATE_LR_REJECTED, STATE_BELOW_ONE, STATE_SPECKLE = 0, 1, 2, 3, 4, 5

_lib = None


class RsgmTaps(C.Structure):
    _fields_ = [("census_l", C.c_void_p), ("census_r", C.c_void_p), ("dsi_agg", C.c_void_p),
                ("disp_l", C.c_void_p), ("disp_r", C.c_void_p)]


class VppSgmParams(C.Structure):
    """vppb200_sgm_params: the SGM penalties a caller asks compute_rsgm to honour"""
    _fields_ = [("p1", C.c_int), ("p2min", C.c_int), ("alpha", C.c_float), ("gamma", C.c_int)]


# The prototype of every function include/vppstereo_b200.h declares, in the header's order: name -> (restype, argtypes).
# tests/test_abi_prototypes.py checks it against the header under this rule:
#   int, float, double, size_t, int64_t, uint64_t, uint32_t -> their ctypes types; a const char * return -> c_char_p;
#   const vppb200_sgm_params * -> POINTER(VppSgmParams), const vppb200_rsgm_taps * -> POINTER(RsgmTaps) (pass the struct or
#   None: ctypes takes the reference); every other pointer -> c_void_p (device and host buffers are opaque addresses: an int,
#   None, a c_void_p, a ctypes array or a byref(...)).
# ctypes then converts every argument as C expects it (a Python float becomes a C float where the header says float) and
# refuses a value of the wrong kind (a float for an int) with ctypes.ArgumentError.
_i, _f, _d, _sz, _i64, _u64, _u32, _p = C.c_int, C.c_float, C.c_double, C.c_size_t, C.c_int64, C.c_uint64, C.c_uint32, C.c_void_p
_taps, _prm = C.POINTER(RsgmTaps), C.POINTER(VppSgmParams)
PROTOTYPES = {
    # library
    "vppb200_version": (C.c_char_p, ()),
    "vppb200_last_cuda_error": (C.c_char_p, ()),
    "vppb200_async_error": (_i, ()),
    "vppb200_launch_count": (_u64, ()),
    "vppb200_rcp_lut_host": (_i, (_p,)),
    "vppb200_glibc_srand": (_i, (_p, _u32)),
    "vppb200_glibc_rand_fill": (_i, (_p, _p, _i64)),
    "vppb200_stage_timing": (_i, (_i,)),
    "vppb200_stage_times": (_i, (_p, _p)),
    "vppb200_set_tuning": (_i, (_i, _i)),
    # pyrSGM operators
    "vppb200_census5x5": (_i, (_p, _p, _i, _i, _i, _p)),
    "vppb200_cost_census5x5_xyd": (_i, (_p, _p, _p, _i, _i, _i, _i, _i, _p)),
    "vppb200_aggregate": (_i, (_p, _p, _p, _i, _i, _i, _i, _i, _f, _i, _i, _i, _p)),
    "vppb200_match_wta": (_i, (_p, _p, _i, _i, _i, _f, _i, _p)),
    "vppb200_match_wta_right": (_i, (_p, _p, _i, _i, _i, _f, _i, _p)),
    "vppb200_subpixel_refine": (_i, (_p, _p, _i, _i, _i, _i, _p, _i, _p)),
    "vppb200_median3x3": (_i, (_p, _p, _i, _i, _i, _p)),
    # compute_rsgm
    "vppb200_rsgm_workspace_bytes": (_sz, (_i, _i, _i, _i, _i)),
    "vppb200_compute_rsgm": (_i, (_p, _p, _p, _p, _p, _p, _i, _i, _i, _i, _i, _p, _p, _sz, _i, _p)),
    "vppb200_rsgm_workspace_bytes_sets": (_sz, (_i, _i, _i, _i, _i, _i)),
    "vppb200_compute_rsgm_phases": (_i, (_p, _p, _p, _p, _p, _p, _i, _i, _i, _i, _i, _p, _p, _sz, _i, _p, _i, _i, _i)),
    "vppb200_compute_rsgm_tapped": (_i, (_p, _p, _p, _p, _p, _p, _i, _i, _i, _i, _i, _p, _p, _sz, _i, _p, _taps)),
    # honoured SGM parameters
    "vppb200_compute_rsgm_ex": (_i, (_p, _p, _p, _p, _p, _p, _i, _i, _i, _i, _i, _p, _p, _sz, _i, _p, _i, _i, _i, _taps, _prm)),
    "vppb200_sgm_params_fast": (_i, (_prm, _i)),
    # uniqueness ratio
    "vppb200_match_wta_uniq": (_i, (_p, _p, _i, _i, _i, _f, _i, _p)),
    "vppb200_match_wta_right_uniq": (_i, (_p, _p, _i, _i, _i, _f, _i, _p)),
    "vppb200_compute_rsgm_uniq": (_i, (_p, _p, _p, _p, _p, _p, _i, _i, _i, _i, _i, _p, _p, _sz, _i, _p, _i, _i, _i, _taps, _prm, _f)),
    # per-pixel match info
    "vppb200_rsgm_info_workspace_bytes": (_sz, (_i, _i, _i, _i, _i, _i)),
    "vppb200_compute_rsgm_info": (_i, (_p, _p, _p, _p, _p, _p, _i, _i, _i, _i, _i, _p, _p, _sz, _i, _p, _i, _i, _i, _taps, _prm, _f,
                                       _p, _p, _p)),
    # row bands
    "vppb200_banded_workspace_bytes": (_sz, (_i, _i, _i, _i)),
    "vppb200_banded_dims": (_i, (_i, _i, _i, _i, _p, _p, _p, _p)),
    "vppb200_rsgm_front_census": (_i, (_p, _p, _p, _p, _p, _p, _i, _i, _i, _i, _p, _sz, _p)),
    "vppb200_sgm_band": (_i, (_p, _p, _p, _p, _p, _i, _i, _i, _i, _i, _i, _i, _p, _p, _p, _p, _p, _p, _sz, _p)),
    "vppb200_sgm_band_ex": (_i, (_p, _p, _p, _p, _p, _i, _i, _i, _i, _i, _i, _i, _p, _p, _p, _p, _p, _p, _sz, _p, _prm)),
    "vppb200_sgm_band_guided": (_i, (_p, _p, _p, _p, _p, _i, _i, _i, _i, _i, _i, _i, _p, _p, _p, _p, _p, _p, _sz, _p, _prm, _p, _p)),
    "vppb200_sgm_band_uniq": (_i, (_p, _p, _p, _p, _p, _i, _i, _i, _i, _i, _i, _i, _p, _p, _p, _p, _p, _p, _sz, _p, _prm, _p, _p, _f)),
    "vppb200_rsgm_tail": (_i, (_p, _p, _p, _i, _i, _i, _i, _i, _p, _sz, _p)),
    # vpp_core_opt operators
    "vppb200_vpp_workspace_bytes": (_sz, (_i, _i, _i, _i)),
    "vppb200_vpp_scan_rnd": (_i, (_p, _p, _p, _i, _i, _i, _i, _i, _i, _d, _d, _p, _i, _i, _i, _p, _p, _u64, _p, _p, _sz, _i, _p)),
    "vppb200_vpp_scan_rnd_rows": (_i, (_p, _p, _p, _i, _i, _i, _i, _i, _i, _d, _d, _p, _i, _i, _i, _p, _p, _u64, _i, _i, _p, _p, _sz, _i, _p)),
    "vppb200_vpp_max_dist_workspace_bytes": (_sz, (_i, _i, _i, _i, _i, _i)),
    "vppb200_vpp_scan_max_dist": (_i, (_p, _p, _p, _i, _i, _i, _i, _i, _i, _i, _i, _d, _d, _p, _i, _i, _i, _p, _p, _sz, _i, _p)),
    "vppb200_bilateral_filling": (_i, (_p, _p, _p, _i, _i, _i, _p, _d, _i, _p)),
    "vppb200_vpp_scan_rnd_adaptive": (_i, (_p, _p, _p, _i, _i, _i, _i, _i, _i, _d, _d, _p, _i, _i, _i, _p, _p, _u64, _p, _p, _i, _p, _p, _sz, _i, _p)),
    "vppb200_vpp_scan_max_dist_adaptive": (_i, (_p, _p, _p, _i, _i, _i, _i, _i, _i, _i, _i, _d, _d, _p, _i, _i, _i, _p, _p, _i, _p, _p, _sz, _i, _p)),
    "vppb200_bgr2gray": (_i, (_p, _p, _i, _i, _i, _i, _p)),
    "vppb200_distance_patch_thresholds": (_i, (_p, _i, _i, _p, _i, _p, _p, _i, _p)),
    "vppb200_gt_reshape": (_i, (_p, _i, _i, _p, _p, _p, _sz, _p)),
    # occlusion mask
    "vppb200_occlusion_workspace_bytes": (_sz, (_i, _i, _i)),
    "vppb200_occlusion_heuristic": (_i, (_p, _p, _p, _i, _i, _i, _i, _d, _d, _d, _d, _p, _sz, _i, _p)),
    # hand-off to the networks
    "vppb200_u8hwc_to_f32chw": (_i, (_p, _p, _i, _i, _i, _i, _i, _i, _i, _i, _p)),
    "vppb200_f32chw_to_u8hwc": (_i, (_p, _p, _i, _i, _i, _i, _p)),
}
SYMBOLS = tuple(PROTOTYPES)


def sgm_params(p1, p2min, alpha, gamma):
    """(p1, p2min, alpha, gamma) -> VppSgmParams, validated on the host (no device needed): ValueError unless
    0 <= p1, p2min, gamma <= 65535 are integers and alpha is finite and >= 0 (include/vppstereo_b200.h)."""
    vals = {}
    for name, v in (("p1", p1), ("p2min", p2min), ("gamma", gamma)):
        try:
            iv = int(v)
        except (TypeError, ValueError, OverflowError):
            raise ValueError(f"{name} must be an integer in [0, 65535], got {v!r}") from None
        if iv != v or not 0 <= iv <= 65535:
            raise ValueError(f"{name} must be an integer in [0, 65535], got {v!r}")
        vals[name] = iv
    try:
        a = float(alpha)
    except (TypeError, ValueError):
        raise ValueError(f"alpha must be a finite number >= 0, got {alpha!r}") from None
    if not (np.isfinite(a) and a >= 0.0) or not np.isfinite(np.float32(a)):
        raise ValueError(f"alpha must be a finite number >= 0, got {alpha!r}")
    prm = VppSgmParams(vals["p1"], vals["p2min"], a, vals["gamma"])
    if lib().vppb200_sgm_params_fast(prm, 0) < 0:                    # the library's own validation (same rules)
        raise ValueError(f"invalid SGM parameters {(p1, p2min, alpha, gamma)}")
    return prm


def uniqueness(u, what="uniqueness"):
    """The uniqueness ratio of an opt-in WTA test as float, validated on the host: TypeError (the reference's message) unless it is
    a finite number with 0 < u <= 1 (include/vppstereo_b200.h)."""
    try:
        f = float(u)
    except (TypeError, ValueError):
        raise TypeError(f"Uniqueness must be inside ]0,1] ({u!r}, {what})") from None
    if not (0.0 < f <= 1.0) or not (0.0 < float(np.float32(f)) <= 1.0):
        raise TypeError(f"Uniqueness must be inside ]0,1] ({u!r}, {what})")
    return f


def sgm_params_fast(prm, guided=False):
    """True if the four sweeps compute these parameters (otherwise compute_rsgm falls back to the per-path kernels)."""
    return lib().vppb200_sgm_params_fast(prm, int(bool(guided))) == 1


def lib():
    """Load libvppstereo_b200.so (built by `python -m vppstereo_b200.build`); fail loudly if it is missing."""
    global _lib
    if _lib is None:
        if not os.path.exists(LIB_PATH):
            raise RuntimeError(f"{LIB_PATH} not built: run `python -m vppstereo_b200.build` (there is no CPU fallback)")
        _lib = bind(C.CDLL(LIB_PATH))
    return _lib


def bind(cdll):
    """Give every PROTOTYPES entry that `cdll` exports its restype and argtypes (also for another build of the library)."""
    for name, (restype, argtypes) in PROTOTYPES.items():
        if hasattr(cdll, name):
            fn = getattr(cdll, name)
            fn.restype, fn.argtypes = restype, argtypes
    return cdll


def call(name, *args, what=None):
    """Call the status-returning entry point `name` and raise through check() (message tagged `what`, default `name`) unless
    it returns VPPB200_OK.  A wrong number of arguments raises TypeError before anything reaches C: ctypes itself only refuses
    too few."""
    fn = getattr(lib(), name)
    if len(args) != len(fn.argtypes):
        raise TypeError(f"{name} takes {len(fn.argtypes)} arguments ({len(args)} given)")
    check(fn(*args), name if what is None else what)


TUNE_SGM_MAX_STRIP, TUNE_SGM_SWEEP, TUNE_SGM_CLUSTERS, TUNE_VPP_ROWS, TUNE_SGM_BYTE_SUMS, TUNE_VPP_MD_WAVE, TUNE_SGM_FUSE_COST, TUNE_RCP_HOST, TUNE_SGM_V_RED = 0, 1, 2, 3, 4, 5, 6, 7, 8
TUNE_SGM_V_SPLIT, TUNE_CENSUS_FUSED = 9, 10


_tuning = {}


def set_tuning(key, value):
    """Process-wide tuning / test hook (include/vppstereo_b200.h: vppb200_set_tuning)."""
    call("vppb200_set_tuning", int(key), int(value), what="set_tuning")
    _tuning[int(key)] = int(value)


def get_tuning(key, default=0):
    """The value last set through set_tuning in this process (`default` = the library's initial value)."""
    return _tuning.get(int(key), default)


def check_async(device=None):
    """Raise if a cooperative sweep on `device` reported a timed-out hand-off since the last check (synchronises the device)."""
    torch = torch_mod()
    with torch.cuda.device(device if device is not None else torch.cuda.current_device()):
        call("vppb200_async_error", what="async_error")


def launch_count():
    return int(lib().vppb200_launch_count())


def check(rc, what=""):
    """Status -> the exception class the reference raises for the same condition (RSGM/pyrSGM.cpp raises TypeError)."""
    if rc == OK:
        return
    msgs = {
        ERR_WIDTH: "Width must be a multiple of 16",
        ERR_DISP: "Disparity range must be a multiple of 8 and not greater than 256",
        ERR_THREADS: "NumThreads must be 1,2,4",
        ERR_UNIQUENESS: "Uniqueness must be inside ]0,1]",
        ERR_METHOD: "method must be inside {0,1}",
    }
    if rc in msgs:
        raise TypeError(f"{msgs[rc]} ({what})")
    if rc == ERR_WORKSPACE:
        raise RuntimeError(f"{what}: workspace missing or too small")
    if rc == ERR_ARG:
        raise ValueError(f"{what}: invalid argument")
    if rc == ERR_CUDA:
        raise RuntimeError(f"{what}: CUDA failure: {lib().vppb200_last_cuda_error().decode()}")
    raise RuntimeError(f"{what}: status {rc}")


def torch_mod():
    import torch
    return torch


def require_cuda():
    torch = torch_mod()
    if not torch.cuda.is_available():
        raise RuntimeError("vppstereo_b200 needs a CUDA device (sm_100a); there is no CPU fallback")
    lib()
    return torch


def is_tensor(x):
    return type(x).__module__.startswith("torch")


def as_device(x, dtype, device=None):
    """numpy array or torch tensor -> contiguous CUDA tensor of `dtype` (torch dtype)."""
    torch = require_cuda()
    if is_tensor(x):
        t = x
        if not t.is_cuda:
            t = t.cuda(device) if device is not None else t.cuda()
        if t.dtype != dtype:
            t = t.to(dtype)
        return t.contiguous()
    a = np.ascontiguousarray(x)
    t = torch.from_numpy(a)
    t = t.cuda(device) if device is not None else t.cuda()
    if t.dtype != dtype:
        t = t.to(dtype)
    return t


def ptr(t):
    return C.c_void_p(t.data_ptr()) if t is not None else None


def stream_ptr(device=None):
    """the current stream of `device` (default: of the current device) as the void* the C-ABI takes"""
    torch = torch_mod()
    return C.c_void_p(torch.cuda.current_stream(device).cuda_stream)


def device_of(*tensors):
    """the CUDA device of the first tensor operand: front-ends launch on ITS current stream, with it as the current device
    (the library's per-device state -- reciprocal table, side streams, sweep plan -- follows the current device)"""
    for t in tensors:
        if t is not None and is_tensor(t) and t.is_cuda:
            return t.device
    torch = torch_mod()
    return torch.device("cuda", torch.cuda.current_device())


_ws_cache = {}


def workspace(nbytes, device, tag="ws"):
    """Cached scratch buffer for the drop-in front-ends (grown on demand, never shrunk); the C-ABI never allocates on the data
    path.  One buffer per (tag, device, CURRENT STREAM): the kernels of a call run on the caller's current stream, so calls made
    under different `torch.cuda.stream(...)` contexts (or from threads with their own streams) never share scratch memory, and
    calls on one stream are ordered by the stream.  A buffer that is replaced by a larger one is handed back to the allocator
    with `record_stream`, i.e. only reused once the work queued on that stream has finished."""
    torch = torch_mod()
    dev = torch.device(device)
    index = dev.index if dev.index is not None else torch.cuda.current_device()
    stream = torch.cuda.current_stream(index)
    key = (tag, index, int(stream.cuda_stream))
    buf = _ws_cache.get(key)
    if buf is None or buf.numel() < nbytes:
        if buf is not None:
            buf.record_stream(stream)
        _ws_cache.pop(key, None)
        with torch.cuda.device(index), torch.cuda.stream(stream):
            buf = torch.empty(int(nbytes), dtype=torch.uint8, device=torch.device("cuda", index))
        _ws_cache[key] = buf
    return buf


def free_workspaces():
    """Drop every cached scratch buffer (synchronises first: kernels on private streams may still be using them)."""
    if _ws_cache:
        torch_mod().cuda.synchronize()
    _ws_cache.clear()


# torch has no uint16/uint32 arithmetic, but storage of those widths is all we need: views over int16/int32
def u16_dtype():
    return torch_mod().int16


def u32_dtype():
    return torch_mod().int32


_SIGNED_VIEW = {np.dtype(np.uint16): np.int16, np.dtype(np.uint32): np.int32}


def np_to_dev(a, np_dtype, device=None):
    """numpy array -> contiguous CUDA tensor with the same bytes (uint16/uint32 travel as int16/int32 storage)."""
    torch = require_cuda()
    a = np.ascontiguousarray(a, dtype=np_dtype)
    v = a.view(_SIGNED_VIEW[a.dtype]) if a.dtype in _SIGNED_VIEW else a
    t = torch.from_numpy(v)
    return t.cuda(device) if device is not None else t.cuda()


def dev_to_np(t, np_dtype):
    a = t.detach().cpu().numpy()
    np_dtype = np.dtype(np_dtype)
    return a.view(np_dtype) if a.dtype != np_dtype else a


def operand(x, np_dtype, torch_dtype):
    """(device tensor, was_numpy) for an input operand given as numpy array or CUDA tensor."""
    if is_tensor(x):
        torch = require_cuda()
        if not x.is_cuda:
            raise TypeError("torch operands must live on a CUDA device")
        if x.element_size() != np.dtype(np_dtype).itemsize:
            raise TypeError(f"expected {np.dtype(np_dtype).itemsize}-byte elements, got {x.dtype}")
        return x.contiguous(), False
    if not isinstance(x, np.ndarray):
        raise TypeError("expected a numpy array or a CUDA tensor")
    return np_to_dev(x, np_dtype), True
