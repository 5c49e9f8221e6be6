"""The whole hot path as one object: VPP (numba arithmetic as test.py uses it) followed by compute_rsgm on a batch of frames,
with the images staying on the device between the two (test.py:154-225 without the host round-trips).

    pipe = VppRsgmPipeline(H, W, batch=64, dmax=192)
    disp = pipe.run_device(left_u8, right_u8, hints_f32)        # CUDA tensors in, CUDA float32 [N,H,W] out
    disp = pipe.run_host(left_pinned, right_pinned, hints_pinned)  # host tensors in, pinned host float32 out

    pipe = VppRsgmPipeline(H, W, guided=True)                   # guided matching (rsgm.py:115-127) on the same hints:
    disp = pipe.run_device(left_u8, right_u8, hints_f32, validhints=valid_f32)    # compute_rsgm(left, lv, rv, hints, validhints)

The projection covers test.py's options with vpp()'s keyword names (default: rnd pattern, fixed patch, no occlusion mask):

    pipe = VppRsgmPipeline(H, W, maskocc=True)                           # the paper's default: --maskocc
    pipe = VppRsgmPipeline(H, W, maskocc=True, method="maxDistance")     # --colormethod maxDistance
    pipe = VppRsgmPipeline(H, W, maskocc=True, wsize=7, use_bilateral_patch=True, use_distance_patch=True)   # the journal's

maskocc: g_occ = occlusion_heuristic(hints)[1] with the reference's default parameters (test.py:154), computed per call on the
device; the adaptive patches' operands (bilateral filling, distance-based patch thresholds) are computed on the device too, so
no option adds a host round trip to run_device.

    pipe = VppRsgmPipeline(H, W, match_info=True)               # + how every left pixel was produced (rsgm.compute_rsgm's info)
    disp, info = pipe.run_device(left_u8, right_u8, hints_f32)  # info = {"state": uint8, "cost", "rival": uint16 storage} [N,H,W]

Three phases of neighbouring batches run concurrently on three internal streams (software pipeline across calls):
  front(k+1) = [occlusion mask, adaptive-patch operands] + VPP + pad/gray/census/cost volume
  main(k) = 8-path SGM sweeps + WTA   |   tail(k-1) = median ... fills
with two buffer sets for everything that crosses a phase boundary; the SGM sweeps alone keep the critical stream busy
and the small, latency-bound front and tail kernels fill the idle issue slots beside them.

run_host is the end-to-end path: host->device copies of the three inputs and the device->host copy of the disparities
are part of the call.  submit_host / collect is the same path for streams of batches: the copies of batch k+1 and of
batch k-1 ride their own CUDA streams while batch k computes (two staging sets, events between the streams).
"""
import numpy as np

from . import _lib
from . import vpp_core_opt as _core
from . import vpp_standalone as _vs


class VppRsgmPipeline:
    guided = False                                    # set per object by __init__(guided=...)
    _stage_marks = None   # bench-only hook (tools/bench_pipeline_modes.py): a list to which the front phase appends
                          # (step name, timing CUDA event) after each of its steps; None (the default) records nothing

    def __init__(self, H, W, channels=3, batch=64, dmax=192, wsize=3, blending=0.4, c_occ=0.0, left2right=True,
                 interpolate=True, subpixel=True, device=None, seed=1234, sgm_params=None, guided=False, uniqueness=None,
                 method="rnd", wsizeAgg_x=64, wsizeAgg_y=3, discard_occ=False, uniform_color=False, use_distance_patch=False,
                 distance_gamma=0.3, use_bilateral_patch=False, bilateral_o_xy=2, bilateral_o_i=1, bilateral_th=.001,
                 maskocc=False, match_info=False):
        # sgm_params: (p1, p2min, alpha, gamma) honoured by the matcher; None = the reference's effective values (7, 17, 0.25, 50)
        # guided: the matcher is compute_rsgm(left, lv, rv, hints, validhints) -- every entry point then takes `validhints`
        # (float32 [N,H,W], placed like `hints`).  Parameters outside the guided sweep domain run on the per-path kernels.
        # uniqueness: the WTA's uniqueness ratio, compute_rsgm(..., uniqueness=u, honor_uniqueness=True); None = off
        # method ... bilateral_th: vpp()'s keywords of the same names (vpp_standalone.py:396), numba arithmetic
        # maskocc: g_occ = occlusion_heuristic(hints)[1] (test.py:154, --maskocc); without it the mask is all zero and c_occ
        # has no effect
        # use_distance_patch: a batch with a frame whose hints all have one value has no reference output (the reference raises
        # ZeroDivisionError); that frame is projected with patch size 1 and check() / run_host() / collect() raise
        # ZeroDivisionError for it (see _raise_degenerate)
        # match_info: every entry point also returns the per-pixel match info of compute_rsgm(..., return_info=True) (state uint8,
        # cost / rival uint16 as _lib.u16_dtype() storage, [N,H,W]); run_device / run_device_serial then take `info_out`
        if method not in ("rnd", "maxDistance"):
            raise ValueError(f"method: expected 'rnd' or 'maxDistance', got {method!r}")
        for name, v in (("wsize", wsize), ("wsizeAgg_x", wsizeAgg_x), ("wsizeAgg_y", wsizeAgg_y)):
            if int(v) != v or int(v) < 1:
                raise ValueError(f"{name}: expected a window size >= 1, got {v!r}")
        self.method = method
        self.wsize_agg = (int(wsizeAgg_x), int(wsizeAgg_y))
        self.discard_occ, self.uniform_color, self.maskocc = bool(discard_occ), bool(uniform_color), bool(maskocc)
        self.use_distance_patch, self.use_bilateral_patch = bool(use_distance_patch), bool(use_bilateral_patch)
        self.distance_gamma = distance_gamma
        self.bilateral = (bilateral_o_xy, bilateral_o_i, float(bilateral_th))
        self.sgm_params = None if sgm_params is None else _lib.sgm_params(*sgm_params)
        self.uniqueness = 1.0 if uniqueness is None else _lib.uniqueness(uniqueness, "VppRsgmPipeline")
        self.guided = bool(guided)
        self.match_info = bool(match_info)
        torch = _lib.require_cuda()
        self.torch = torch
        self.H, self.W, self.C, self.N, self.D = int(H), int(W), int(channels), int(batch), int(dmax)
        self.wsize, self.blending, self.c_occ = int(wsize), float(blending), float(c_occ)
        self.direction = 1 if left2right else 0
        self.interpolate, self.subpixel = bool(interpolate), bool(subpixel)
        self.device = torch.device("cuda", torch.cuda.current_device()) if device is None else torch.device(device)
        if self.device.type != "cuda":
            raise ValueError("VppRsgmPipeline needs a CUDA device")
        if self.device.index is None:
            self.device = torch.device("cuda", torch.cuda.current_device())
        self.seed = int(seed)
        self.step = 0                                 # pattern-seed counter
        self.calls = 0                                # buffer-set parity
        L = _lib.lib()
        with torch.cuda.device(self.device):
            ws_bytes = (L.vppb200_rsgm_info_workspace_bytes if self.match_info else L.vppb200_rsgm_workspace_bytes_sets)
            self.ws_rsgm = torch.empty(ws_bytes(self.H, self.W, self.C, self.D, self.N, 2), dtype=torch.uint8, device=self.device)
            ws_vpp = L.vppb200_vpp_workspace_bytes(self.H, self.W, self.C, self.N)
            if self.method == "maxDistance":     # + the row wavefront's dependency table
                ws_vpp = max(ws_vpp, L.vppb200_vpp_max_dist_workspace_bytes(self.H, self.W, self.C, self.wsize, self.wsize_agg[1],
                                                                            self.N))
            self.ws_vpp = torch.empty(ws_vpp, dtype=torch.uint8, device=self.device)
            self.occ = torch.zeros((self.N, self.H, self.W), dtype=torch.uint8, device=self.device)
            # buffers of the optional front-phase steps: produced and consumed inside one front phase, and front phases are
            # ordered on one stream, so a single copy of each serves both buffer sets
            self.ws_occ = self.gray = self.filled = self.bl_weights = self.ratio_steps = self.thr = None
            self.status = self.status_host = None
            if self.maskocc:
                self.ws_occ = torch.empty(L.vppb200_occlusion_workspace_bytes(self.H, self.W, self.N), dtype=torch.uint8,
                                          device=self.device)
            if self.use_bilateral_patch:
                self.gray = torch.empty((self.N, self.H, self.W), dtype=torch.uint8, device=self.device)
                self.filled = torch.empty((self.N, self.H, self.W), dtype=torch.float32, device=self.device)
                wt = _vs._bilateral_weights((self.wsize - 1) // 2, self.bilateral[0], self.bilateral[1])
                self.bl_weights = torch.from_numpy(wt).to(self.device)
            if self.use_distance_patch:
                self.ratio_steps = torch.from_numpy(_vs._ratio_steps(self.wsize, distance_gamma).copy()).to(self.device)
                if self.wsize > 1:
                    self.thr = torch.empty((self.N, self.wsize - 1), dtype=torch.float32, device=self.device)
                # degenerate-frame status words (see _raise_degenerate): one per way of calling, so that each is read only
                # by the call that owns it -- run_device / run_device_serial (reported by check()), run_host; submit_host
                # gives every staging set its own
                self.status = torch.zeros(self.N, dtype=torch.int32, device=self.device)
                self.status_host = torch.zeros(self.N, dtype=torch.int32, device=self.device)
            self.lv = torch.empty((self.N, self.H, self.W, self.C), dtype=torch.uint8, device=self.device)
            self.rv = torch.empty_like(self.lv)
            # two projected-image sets + VPP stream: see run_device
            self.lv2, self.rv2 = [self.lv, torch.empty_like(self.lv)], [self.rv, torch.empty_like(self.lv)]
            self.vpp_stream = torch.cuda.Stream(self.device)      # front phase: VPP + pad/gray/census/cost volume
            # the sweeps are the critical path: their CTAs are scheduled ahead of the front / tail kernels that fill in beside them
            self.main_stream = torch.cuda.Stream(self.device, priority=-1)       # SGM sweeps + WTA
            self.tail_stream = torch.cuda.Stream(self.device)     # median ... background fill
            self.front_done = [torch.cuda.Event(), torch.cuda.Event()]
            self.main_done = [None, None]
            self.tail_done = [None, None]
            self.last_n = None                        # batch size of the latest run_device call
            self.disp = torch.empty((self.N, self.H, self.W), dtype=torch.float32, device=self.device)
            # staging for run_host
            self.d_left = torch.empty_like(self.lv)
            self.d_right = torch.empty_like(self.lv)
            self.d_hints = torch.empty((self.N, self.H, self.W), dtype=torch.float32, device=self.device)
            self.d_valid = torch.empty_like(self.d_hints) if self.guided else None
            self.h_disp = torch.empty((self.N, self.H, self.W), dtype=torch.float32).pin_memory()
            self.info = self._info_buffers(self.device) if self.match_info else None       # run_device's default info_out
            self.h_info = self._info_buffers("cpu") if self.match_info else None           # run_host's pinned copies
            self._stream_sets = None                  # created by the first submit_host
            self.host_depth = 3                       # staging sets of the streaming host API
            # the zero-filled occlusion mask / status and the tables above were queued on the constructing stream, while the
            # first call's front phase runs on this object's own streams (which do not wait for it when inputs_ready=True):
            # finish them here
            torch.cuda.current_stream(self.device).synchronize()

    def close(self):
        """Wait for everything queued on the pipeline's own streams.  The buffers belong to this object while the kernels that
        use them run on private streams the caching allocator does not track: they must not be released (and handed to another
        tensor) before that work has finished.  Called by __del__; call it yourself before dropping a pipeline with batches
        still in flight."""
        try:
            for s in (self.vpp_stream, self.main_stream, self.tail_stream):
                s.synchronize()
            _lib.check_async(self.device)
            if self._stream_sets is not None:
                self._stream_sets["h2d"].synchronize(); self._stream_sets["d2h"].synchronize()
        except RuntimeError:
            raise
        except Exception:
            pass

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def check(self):
        """Wait for the device and raise if a sweep reported a timed-out hand-off between its CTAs (vppb200_async_error), or
        ZeroDivisionError for a degenerate frame (use_distance_patch, see _raise_degenerate) of a run_device /
        run_device_serial call since the last check()."""
        _lib.check_async(self.device)
        if self.status is None:
            return
        torch = self.torch
        with torch.cuda.device(self.device):
            self.vpp_stream.synchronize()
            bad = self.status.cpu().numpy()
            if bad.any():
                with torch.cuda.stream(self.vpp_stream):      # ordered before every later front phase (serial ones wait for it)
                    self.status.zero_()
                self._raise_degenerate(bad, "a run_device / run_device_serial call since the last check()")

    @staticmethod
    def _raise_degenerate(status, which):
        """use_distance_patch: the reference divides by (dmax - dmin) (vpp_standalone.py:7) and raises ZeroDivisionError for a
        frame whose hints all have one value.  run_device does not synchronise, so the thresholds kernel only records such a
        frame in a device status word of the call (the frame is projected with patch size 1: defined and deterministic, but
        not a reference output, since the reference has none).  The calls that synchronise anyway raise for it: run_host()
        and collect() for their own batch, check() for the run_device / run_device_serial calls since the previous check();
        each status is cleared once read, so the pipeline stays usable for the next batch."""
        f = int(np.flatnonzero(status)[0])
        raise ZeroDivisionError(f"division by zero: every hint of frame {f} of {which} has the same disparity "
                                "(use_distance_patch); that batch's output is not the reference's")

    _INFO = (("state", "uint8"), ("cost", "int16"), ("rival", "int16"))       # info maps and their torch storage (uint16 as int16)

    def _info_buffers(self, device):
        torch = self.torch
        return {k: (torch.empty((self.N, self.H, self.W), dtype=getattr(torch, dt), device=device) if device != "cpu" else
                    torch.empty((self.N, self.H, self.W), dtype=getattr(torch, dt)).pin_memory()) for k, dt in self._INFO}

    @staticmethod
    def _info_slice(info, N):
        return {k: t[:N] for k, t in info.items()}

    def workspace_bytes(self):
        return self.ws_rsgm.numel() + self.ws_vpp.numel() + (self.ws_occ.numel() if self.ws_occ is not None else 0)

    def _check(self, left, right, hints, out=None, host=False, validhints=None, info_out=None):
        """Operand validation shared by every entry point: the kernels receive raw pointers, so a wrong dtype, shape, device
        or a non-contiguous view would be read as garbage or out of bounds.  Returns the batch size."""
        torch = self.torch
        if info_out is not None and not self.match_info:
            raise ValueError("info_out: given to a pipeline without match info (construct it with match_info=True)")
        if info_out is not None and (not isinstance(info_out, dict) or set(info_out) != {k for k, _ in self._INFO}):
            raise TypeError(f"info_out: expected a dict with the keys {[k for k, _ in self._INFO]}")
        if self.guided and validhints is None:
            raise ValueError("validhints: required by a guided pipeline (guided=True)")
        if not self.guided and validhints is not None:
            raise ValueError("validhints: given to an unguided pipeline (construct it with guided=True)")
        ops = (("left", left), ("right", right), ("hints", hints)) + ((("validhints", validhints),) if self.guided else ())
        for name, t in ops:
            if not isinstance(t, torch.Tensor):
                raise TypeError(f"{name}: expected a torch tensor, got {type(t).__name__}")
        if left.dim() != 4 or tuple(left.shape[1:]) != (self.H, self.W, self.C):
            raise ValueError(f"left: expected [N,{self.H},{self.W},{self.C}], got {tuple(left.shape)}")
        N = int(left.shape[0])
        if not 1 <= N <= self.N:
            raise ValueError(f"batch of {N} frames does not fit this pipeline (batch={self.N})")
        want = (("left", left, torch.uint8, (N, self.H, self.W, self.C)), ("right", right, torch.uint8, (N, self.H, self.W, self.C)),
                ("hints", hints, torch.float32, (N, self.H, self.W)))
        if self.guided:
            want += (("validhints", validhints, torch.float32, (N, self.H, self.W)),)
        if out is not None:
            if not isinstance(out, torch.Tensor):
                raise TypeError("out: expected a torch tensor")
            want += (("out", out, torch.float32, (N, self.H, self.W)),)
        if info_out is not None:
            for k, dt in self._INFO:
                if not isinstance(info_out[k], torch.Tensor):
                    raise TypeError(f"info_out[{k!r}]: expected a torch tensor")
                want += ((f"info_out[{k!r}]", info_out[k], getattr(torch, dt), (N, self.H, self.W)),)
        for name, t, dt, shape in want:
            if t.dtype != dt:
                raise TypeError(f"{name}: expected {dt}, got {t.dtype}")
            if tuple(t.shape) != shape:
                raise ValueError(f"{name}: expected shape {shape}, got {tuple(t.shape)}")
            if not t.is_contiguous():
                raise ValueError(f"{name}: must be contiguous")
            on_host = host and name != "out"
            if on_host:
                if t.is_cuda:
                    raise ValueError(f"{name}: expected a host tensor (use run_device for CUDA tensors)")
            elif not t.is_cuda or t.device != self.device:
                raise ValueError(f"{name}: expected a CUDA tensor on {self.device}, got {t.device}")
        return N

    def _next_seed(self, step):
        """Pattern seed of one call: a function of the pipeline's seed and the call counter (or of an explicit `step`)."""
        if step is None:
            self.step += 1
            step = self.step
        return (self.seed * 0x9E3779B97F4A7C15 + int(step)) & (2**64 - 1)

    def pattern_seed(self, step):
        """The rng_seed the VPP kernels receive on call number `step` (1-based) -- with vpp_core_opt.device_pattern this
        replays the projected pattern of any frame on the host."""
        return (self.seed * 0x9E3779B97F4A7C15 + int(step)) & (2**64 - 1)

    def _vpp(self, left, lv, rv, hints, seed, N, stream, status):
        # VPP of the projected-image pair lv / rv in place (vpp_standalone.py:396-432), numba arithmetic; `left` = the
        # un-projected left image, `status` = the call's degenerate-frame status words (use_distance_patch).  Every step is queued on `stream`, in the reference's order: occlusion mask, adaptive-patch
        # operands, scan (rnd: pattern drawn on the device from `seed`).
        s = stream.cuda_stream
        self._mark("copy", stream)
        if self.maskocc:                              # occlusion_heuristic(hints)[1] straight into the mask the scan reads
            _lib.call("vppb200_occlusion_heuristic", _lib.ptr(hints), None, _lib.ptr(self.occ), self.W, self.H, 9, 7, 2.0, 0.4375,
                      1.0, 0.1, _lib.ptr(self.ws_occ), self.ws_occ.numel(), N, s, what="occlusion_heuristic")
        self._mark("occlusion", stream)
        filled = thr = None
        if self.use_bilateral_patch:
            filled = self.filled[:N]
            _vs.bilateral_filling(hints, left, (self.wsize - 1) // 2, self.bl_weights, self.bilateral[2], self.gray[:N], filled, s)
        if self.use_distance_patch:
            thr = self.thr[:N] if self.thr is not None else None
            _vs.distance_patch_thresholds(hints, self.wsize, self.ratio_steps, thr, status, s)
        self._mark("patch_operands", stream)
        img = (_lib.ptr(lv), _lib.ptr(rv), _lib.ptr(hints), self.W, self.H, self.C, int(self.uniform_color), self.wsize)
        blend = (self.blending, self.c_occ, _lib.ptr(self.occ), int(self.discard_occ), int(self.interpolate), 1)
        tail = (None, _lib.ptr(self.ws_vpp), self.ws_vpp.numel(), N, s)
        adaptive = () if filled is None and thr is None else (_lib.ptr(filled), _lib.ptr(thr), 0 if thr is None else self.wsize - 1)
        if self.method == "maxDistance":
            md = img + self.wsize_agg + (self.direction,) + blend
            _lib.call("vppb200_vpp_scan_max_dist_adaptive" if adaptive else "vppb200_vpp_scan_max_dist", *md, *adaptive, *tail,
                      what="vpp_scan_max_dist")
        else:
            rnd = img + (self.direction,) + blend + (None, None, seed)
            _lib.call("vppb200_vpp_scan_rnd_adaptive" if adaptive else "vppb200_vpp_scan_rnd", *rnd, *adaptive, *tail,
                      what="vpp_scan_rnd")
        self._mark("scan", stream)

    def _mark(self, name, stream):
        if self._stage_marks is not None:
            ev = self.torch.cuda.Event(enable_timing=True)
            ev.record(stream)
            self._stage_marks.append((name, ev))

    def _phase(self, phases, b, left, lv, rv, out, N, stream, hints, validhints, info=None):
        # hints / validhints go to every phase of a guided batch (their nullness selects the sweeps' state); FRONT reads them;
        # info (match_info): the same three maps in every phase of a batch (MAIN fills set b's cost maps, TAIL writes them)
        h, v = (_lib.ptr(hints), _lib.ptr(validhints)) if self.guided else (None, None)
        args = (_lib.ptr(left), _lib.ptr(lv), _lib.ptr(rv), h, v, _lib.ptr(out), self.H, self.W, self.C, self.D,
                1 if self.subpixel else 0, None, _lib.ptr(self.ws_rsgm), self.ws_rsgm.numel(), N, stream.cuda_stream, phases, 2, b,
                None, self.sgm_params, self.uniqueness)
        if self.match_info:
            _lib.call("vppb200_compute_rsgm_info", *args, *(_lib.ptr(info[k]) for k, _ in self._INFO), what="compute_rsgm_phases")
        else:
            _lib.call("vppb200_compute_rsgm_uniq", *args, what="compute_rsgm_phases")

    def run_device(self, left, right, hints, out=None, inputs_ready=None, step=None, validhints=None, info_out=None):
        """VPP (in copies) + compute_rsgm; all operands CUDA tensors [N,H,W,C] uint8 / [N,H,W] float32.
        `validhints` (guided pipelines only, required there): compute_rsgm(left, lv, rv, hints, validhints).
        match_info pipelines return (out, info): info = `info_out` (a dict like the pipeline's own, see __init__) or the
        pipeline's own buffers, valid in current-stream order like `out` (and like the default `out`, overwritten by the
        next call); `info_out` to a pipeline without match_info: ValueError.

        The work is queued on the pipeline's three streams (front / main / tail, see the module docstring) and the caller's
        current stream is made to wait for the result, so `out` is valid in current-stream order like the output of any
        kernel launch, while the phases of the NEXT call can already run beside this one's.
        `inputs_ready`: None = the inputs were produced on the current stream (the front phase waits for everything queued
        on it so far, which includes the previous result: no overlap between calls); True = the inputs are complete; a
        torch.cuda.Event = wait for that event.  The inputs must stay untouched until the front phase has read them
        (`self.front_done[k & 1]` of call k).
        `step`: explicit call number for the pattern seed (default: the pipeline's own counter, 1, 2, ...)."""
        torch = self.torch
        N = self._check(left, right, hints, out, validhints=validhints, info_out=info_out)
        with torch.cuda.device(self.device):
            info = self._info_out(info_out, N)
            out = self._run_device(left, right, hints, validhints, out, inputs_ready, step, N, self.status, info)
            return (out, info) if self.match_info else out

    def _info_out(self, info_out, N):
        if not self.match_info:
            return None
        return self._info_slice(self.info, N) if info_out is None else info_out

    def _run_device(self, left, right, hints, validhints, out, inputs_ready, step, N, status, info=None):
        torch = self.torch
        out = self.disp[:N] if out is None else out
        caller = torch.cuda.current_stream(self.device)
        front, main, tail = self.vpp_stream, self.main_stream, self.tail_stream
        b = self.calls & 1
        self.calls += 1
        lv, rv = self.lv2[b][:N], self.rv2[b][:N]
        seed = self._next_seed(step)
        # ---- front: VPP into projected-image set b, then the matcher's front phase into buffer set b
        if inputs_ready is None:
            front.wait_stream(caller)
        elif inputs_ready is not True:
            front.wait_event(inputs_ready)
        if self.main_done[b] is not None:
            front.wait_event(self.main_done[b])          # set b (guide, cost volume) was last read by the sweeps two calls ago
        if N != self.last_n:
            # the matcher's workspace is laid out for the call's batch size: the buffers of a call with another N overlap both
            # sets of the calls before it, so it starts when they have finished (no overlap across a change of N)
            for ev in self.main_done + self.tail_done:
                if ev is not None:
                    front.wait_event(ev)
        self.last_n = N
        with torch.cuda.stream(front):
            lv.copy_(left); rv.copy_(right)              # vpp() returns copies (vpp_standalone.py:397)
            self._vpp(left, lv, rv, hints, seed, N, front, status)
            self._phase(1, b, left, lv, rv, out, N, front, hints, validhints, info)
            self.front_done[b].record(front)
        # ---- main: the four SGM sweeps + WTA (the critical stream)
        main.wait_event(self.front_done[b])
        if self.tail_done[b] is not None:
            main.wait_event(self.tail_done[b])           # raw disparities of set b were last read by the tail two calls ago
        with torch.cuda.stream(main):
            self._phase(2, b, left, lv, rv, out, N, main, hints, validhints, info)
            ev = torch.cuda.Event(); ev.record(main)
            self.main_done[b] = ev
        # ---- tail: everything after WTA; `out` may still be read by work the caller queued before this call
        tail.wait_stream(caller)
        tail.wait_event(self.main_done[b])
        with torch.cuda.stream(tail):
            self._phase(4, b, left, lv, rv, out, N, tail, hints, validhints, info)
            ev = torch.cuda.Event(); ev.record(tail)
            self.tail_done[b] = ev
        caller.wait_event(ev)
        self.lv, self.rv = self.lv2[b], self.rv2[b]     # the projected pair of the latest call
        return out

    def run_device_serial(self, left, right, hints, out=None, step=None, validhints=None, info_out=None):
        """The same computation, everything in order on the current stream (no overlap between calls, no internal streams
        except the right-image branches): what bench.py times stage by stage.  match_info / info_out as in run_device."""
        torch = self.torch
        N = self._check(left, right, hints, out, validhints=validhints, info_out=info_out)
        with torch.cuda.device(self.device):
            info = self._info_out(info_out, N)
            out = self._run_device_serial(left, right, hints, validhints, out, step, N, info)
            return (out, info) if self.match_info else out

    def _run_device_serial(self, left, right, hints, validhints, out, step, N, info=None):
        torch = self.torch
        out = self.disp[:N] if out is None else out
        st = torch.cuda.current_stream(self.device)
        for s in (self.vpp_stream, self.main_stream, self.tail_stream):
            st.wait_stream(s)
        b = self.calls & 1
        self.calls += 1
        lv, rv = self.lv2[b][:N], self.rv2[b][:N]
        seed = self._next_seed(step)
        lv.copy_(left); rv.copy_(right)
        self._vpp(left, lv, rv, hints, seed, N, st, self.status)
        self._phase(7, b, left, lv, rv, out, N, st, hints, validhints, info)
        for s in (self.vpp_stream, self.main_stream, self.tail_stream):
            s.wait_stream(st)
        self.lv, self.rv = self.lv2[b], self.rv2[b]
        return out

    def run_host(self, left, right, hints, validhints=None):
        """Host tensors (ideally pinned) in, pinned host float32 [N,H,W] out; the copies are part of the call.  match_info
        pipelines return (disp, info) with info on pinned host memory too (valid until the next run_host)."""
        torch = self.torch
        N = self._check(left, right, hints, host=True, validhints=validhints)
        with torch.cuda.device(self.device):
            self.d_left[:N].copy_(left, non_blocking=True)
            self.d_right[:N].copy_(right, non_blocking=True)
            self.d_hints[:N].copy_(hints, non_blocking=True)
            dv = None
            if self.guided:
                dv = self.d_valid[:N]
                dv.copy_(validhints, non_blocking=True)
            if self.status_host is not None:
                self.status_host.zero_()          # current stream: the front phase below waits for it (inputs_ready=None)
            info = self._info_out(None, N)
            out = self._run_device(self.d_left[:N], self.d_right[:N], self.d_hints[:N], dv, None, None, None, N, self.status_host, info)
            self.h_disp[:N].copy_(out, non_blocking=True)
            if info is not None:
                for k, t in info.items():
                    self.h_info[k][:N].copy_(t, non_blocking=True)
            torch.cuda.current_stream(self.device).synchronize()
            if self.status_host is not None:
                bad = self.status_host[:N].cpu().numpy()     # the current stream is idle: this reads this call's words
                if bad.any():
                    self._raise_degenerate(bad, "this run_host batch")
        if self.match_info:
            return self.h_disp[:N], self._info_slice(self.h_info, N)
        return self.h_disp[:N]

    # ---- streaming front-end: overlapped host<->device copies ---------------------------------------------------
    def _streaming(self):
        torch = self.torch
        if self._stream_sets is None:
            with torch.cuda.device(self.device):
                sets = []
                for _ in range(self.host_depth):
                    sets.append(dict(left=torch.empty_like(self.lv), right=torch.empty_like(self.lv),
                                     hints=torch.empty_like(self.d_hints), disp=torch.empty_like(self.disp),
                                     valid=torch.empty_like(self.d_hints) if self.guided else None,
                                     h_disp=torch.empty((self.N, self.H, self.W), dtype=torch.float32).pin_memory(),
                                     status=torch.empty_like(self.status) if self.status is not None else None,
                                     h_status=torch.zeros(self.N, dtype=torch.int32).pin_memory(),
                                     info=self._info_buffers(self.device) if self.match_info else None,
                                     h_info=self._info_buffers("cpu") if self.match_info else None,
                                     copied_in=torch.cuda.Event(), computed=torch.cuda.Event(), copied_out=torch.cuda.Event(),
                                     busy=False))
                self._stream_sets = dict(sets=sets, h2d=torch.cuda.Stream(self.device), d2h=torch.cuda.Stream(self.device), turn=0)
        return self._stream_sets

    def submit_host(self, left, right, hints, on_computed=None, validhints=None):
        """Queue one batch of host tensors (pinned for real overlap); returns a ticket for collect().  At most `host_depth`
        (3) batches are in flight: submitting one more first requires collecting the oldest.  Keeping two batches queued
        behind the running one lets the next batch's inputs arrive, and its front phase start, while the current sweeps run.
        `on_computed(disp)`: called with the batch's device result right after it has been queued (current stream = the stream
        it becomes valid on), e.g. to hand it to dist.PeerGather.push beside the device->host copy."""
        torch = self.torch
        ss = self._streaming()
        slot = ss["turn"] % self.host_depth
        st = ss["sets"][slot]
        if st["busy"]:
            raise RuntimeError(f"submit_host: collect() the batch submitted {self.host_depth} calls ago first")
        N = self._check(left, right, hints, host=True, validhints=validhints)
        compute = torch.cuda.current_stream(self.device)
        with torch.cuda.device(self.device):
            with torch.cuda.stream(ss["h2d"]):
                # the staging set was last read by the compute of two submits ago, which collect() has waited for
                st["left"][:N].copy_(left, non_blocking=True)
                st["right"][:N].copy_(right, non_blocking=True)
                st["hints"][:N].copy_(hints, non_blocking=True)
                if self.guided:
                    st["valid"][:N].copy_(validhints, non_blocking=True)
                if st["status"] is not None:
                    st["status"].zero_()                 # this batch's own status words (read back with its disparities)
                st["copied_in"].record(ss["h2d"])
            compute.wait_event(st["copied_in"])
            info = self._info_slice(st["info"], N) if self.match_info else None
            self._run_device(st["left"][:N], st["right"][:N], st["hints"][:N], st["valid"][:N] if self.guided else None,
                             st["disp"][:N], st["copied_in"], None, N, st["status"], info)
            st["computed"].record(compute)
            if on_computed is not None:
                on_computed(st["disp"][:N])
            with torch.cuda.stream(ss["d2h"]):
                ss["d2h"].wait_event(st["computed"])
                st["h_disp"][:N].copy_(st["disp"][:N], non_blocking=True)
                if info is not None:
                    for k, t in info.items():
                        st["h_info"][k][:N].copy_(t, non_blocking=True)
                if st["status"] is not None:
                    st["h_status"][:N].copy_(st["status"][:N], non_blocking=True)
                st["copied_out"].record(ss["d2h"])
        st["busy"], st["n"] = True, N
        ss["turn"] += 1
        return slot

    def collect(self, ticket):
        """Wait for a submitted batch; returns its pinned host float32 [N,H,W] disparities (valid until that staging set is
        reused by the `host_depth`-th submit_host after it was submitted); match_info pipelines: (disp, info), info pinned too.  use_distance_patch: ZeroDivisionError if this
        batch has a frame whose hints all have one value (see _raise_degenerate); the batches around it are unaffected."""
        st = self._streaming()["sets"][ticket]
        if not st["busy"]:
            raise RuntimeError("collect: nothing in flight for this ticket")
        st["copied_out"].synchronize()
        st["busy"] = False
        if st["status"] is not None and st["h_status"][:st["n"]].any():
            self._raise_degenerate(st["h_status"][:st["n"]].numpy(), f"the batch of ticket {ticket}")
        if self.match_info:
            return st["h_disp"][:st["n"]], self._info_slice(st["h_info"], st["n"])
        return st["h_disp"][:st["n"]]
