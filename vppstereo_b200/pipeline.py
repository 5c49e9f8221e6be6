"""The whole hot path as one object: VPP (rnd pattern, numba arithmetic as test.py uses it) followed by compute_rsgm on a
batch of frames, with the images staying on the device between the two (test.py:158-225 without the host round-trips).

    pipe = VppRsgmPipeline(H, W, batch=64, dmax=192)
    disp = pipe.run_device(left_u8, right_u8, hints_f32)        # CUDA tensors in, CUDA float32 [N,H,W] out
    disp = pipe.run_host(left_pinned, right_pinned, hints_pinned)  # host tensors in, pinned host float32 out

Three phases of neighbouring batches run concurrently on three internal streams (software pipeline across calls):
  front(k+1) = VPP + pad/gray/census/cost volume   |   main(k) = 8-path SGM sweeps + WTA   |   tail(k-1) = median ... fills
with two buffer sets for everything that crosses a phase boundary; the SGM sweeps alone keep the critical stream busy
and the small, latency-bound front and tail kernels fill the idle issue slots beside them.

run_host is the end-to-end path: host->device copies of the three inputs and the device->host copy of the disparities
are part of the call.  submit_host / collect is the same path for streams of batches: the copies of batch k+1 and of
batch k-1 ride their own CUDA streams while batch k computes (two staging sets, events between the streams).
"""
import ctypes as C

from . import _lib
from . import vpp_core_opt as _core


class VppRsgmPipeline:
    def __init__(self, H, W, channels=3, batch=64, dmax=192, wsize=3, blending=0.4, c_occ=0.0, left2right=True,
                 interpolate=True, subpixel=True, device=None, seed=1234, sgm_params=None):
        # sgm_params: (p1, p2min, alpha, gamma) honoured by the matcher; None = the reference's effective values (7, 17, 0.25, 50)
        self.sgm_params = None if sgm_params is None else _lib.sgm_params(*sgm_params)
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
        self.lib = L
        with torch.cuda.device(self.device):
            self.ws_rsgm = torch.empty(L.vppb200_rsgm_workspace_bytes_sets(self.H, self.W, self.C, self.D, self.N, 2),
                                       dtype=torch.uint8, device=self.device)
            self.ws_vpp = torch.empty(L.vppb200_vpp_workspace_bytes(self.H, self.W, self.C, self.N), dtype=torch.uint8,
                                      device=self.device)
            self.occ = torch.zeros((self.N, self.H, self.W), dtype=torch.uint8, device=self.device)
            self.lv = torch.empty((self.N, self.H, self.W, self.C), dtype=torch.uint8, device=self.device)
            self.rv = torch.empty_like(self.lv)
            # two projected-image sets + VPP stream: see run_device
            self.lv2, self.rv2 = [self.lv, torch.empty_like(self.lv)], [self.rv, torch.empty_like(self.lv)]
            self.vpp_stream = torch.cuda.Stream(self.device)      # front phase: VPP + pad/gray/census/cost volume
            # the sweeps are the critical path: their CTAs are scheduled ahead of the front / tail kernels that fill in beside them
            prio = int(__import__("os").environ.get("VPPB200_MAIN_PRIORITY", "-1"))
            self.main_stream = torch.cuda.Stream(self.device, priority=prio)     # SGM sweeps + WTA
            self.tail_stream = torch.cuda.Stream(self.device)     # median ... background fill
            self.front_done = [torch.cuda.Event(), torch.cuda.Event()]
            self.main_done = [None, None]
            self.tail_done = [None, None]
            self.disp = torch.empty((self.N, self.H, self.W), dtype=torch.float32, device=self.device)
            # staging for run_host
            self.d_left = torch.empty_like(self.lv)
            self.d_right = torch.empty_like(self.lv)
            self.d_hints = torch.empty((self.N, self.H, self.W), dtype=torch.float32, device=self.device)
            self.h_disp = torch.empty((self.N, self.H, self.W), dtype=torch.float32).pin_memory()
            self._stream_sets = None                  # created by the first submit_host
            self.host_depth = 3                       # staging sets of the streaming host API
            # the zero-filled occlusion mask above was queued on the constructing stream, while the first call's front phase
            # runs on this object's own streams (which do not wait for it when inputs_ready=True): finish it here
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
        """Wait for the device and raise if a sweep reported a timed-out hand-off between its CTAs (vppb200_async_error)."""
        _lib.check_async(self.device)

    def workspace_bytes(self):
        return self.ws_rsgm.numel() + self.ws_vpp.numel()

    def _check(self, left, right, hints, out=None, host=False):
        """Operand validation shared by every entry point: the kernels receive raw pointers, so a wrong dtype, shape, device
        or a non-contiguous view would be read as garbage or out of bounds.  Returns the batch size."""
        torch = self.torch
        for name, t in (("left", left), ("right", right), ("hints", hints)):
            if not isinstance(t, torch.Tensor):
                raise TypeError(f"{name}: expected a torch tensor, got {type(t).__name__}")
        if left.dim() != 4 or tuple(left.shape[1:]) != (self.H, self.W, self.C):
            raise ValueError(f"left: expected [N,{self.H},{self.W},{self.C}], got {tuple(left.shape)}")
        N = int(left.shape[0])
        if not 1 <= N <= self.N:
            raise ValueError(f"batch of {N} frames does not fit this pipeline (batch={self.N})")
        want = (("left", left, torch.uint8, (N, self.H, self.W, self.C)), ("right", right, torch.uint8, (N, self.H, self.W, self.C)),
                ("hints", hints, torch.float32, (N, self.H, self.W)))
        if out is not None:
            if not isinstance(out, torch.Tensor):
                raise TypeError("out: expected a torch tensor")
            want += (("out", out, torch.float32, (N, self.H, self.W)),)
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

    def _phase(self, phases, b, left, lv, rv, out, N, stream):
        L = self.lib
        prm = None if self.sgm_params is None else C.byref(self.sgm_params)
        rc = L.vppb200_compute_rsgm_ex(_lib.ptr(left), _lib.ptr(lv), _lib.ptr(rv), None, None, _lib.ptr(out), self.H, self.W,
                                       self.C, self.D, 1 if self.subpixel else 0, None, _lib.ptr(self.ws_rsgm),
                                       C.c_size_t(self.ws_rsgm.numel()), N, C.c_void_p(stream.cuda_stream), phases, 2, b, None, prm)
        _lib.check(rc, "compute_rsgm_phases")

    def run_device(self, left, right, hints, out=None, inputs_ready=None, step=None):
        """VPP (in copies) + compute_rsgm; all operands CUDA tensors [N,H,W,C] uint8 / [N,H,W] float32.

        The work is queued on the pipeline's three streams (front / main / tail, see the module docstring) and the caller's
        current stream is made to wait for the result, so `out` is valid in current-stream order like the output of any
        kernel launch, while the phases of the NEXT call can already run beside this one's.
        `inputs_ready`: None = the inputs were produced on the current stream (the front phase waits for everything queued
        on it so far, which includes the previous result: no overlap between calls); True = the inputs are complete; a
        torch.cuda.Event = wait for that event.  The inputs must stay untouched until the front phase has read them
        (`self.front_done[k & 1]` of call k).
        `step`: explicit call number for the pattern seed (default: the pipeline's own counter, 1, 2, ...)."""
        torch = self.torch
        N = self._check(left, right, hints, out)
        with torch.cuda.device(self.device):
            return self._run_device(left, right, hints, out, inputs_ready, step, N)

    def _run_device(self, left, right, hints, out, inputs_ready, step, N):
        torch, L = self.torch, self.lib
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
        with torch.cuda.stream(front):
            lv.copy_(left); rv.copy_(right)              # vpp() returns copies (vpp_standalone.py:397)
            rc = L.vppb200_vpp_scan_rnd(_lib.ptr(lv), _lib.ptr(rv), _lib.ptr(hints), self.W, self.H, self.C, 0, self.wsize,
                                        self.direction, C.c_double(self.blending), C.c_double(self.c_occ), _lib.ptr(self.occ),
                                        0, int(self.interpolate), 1, None, None, C.c_uint64(seed), None, _lib.ptr(self.ws_vpp),
                                        C.c_size_t(self.ws_vpp.numel()), N, C.c_void_p(front.cuda_stream))
            _lib.check(rc, "vpp_scan_rnd")
            self._phase(1, b, left, lv, rv, out, N, front)
            self.front_done[b].record(front)
        # ---- main: the four SGM sweeps + WTA (the critical stream)
        main.wait_event(self.front_done[b])
        if self.tail_done[b] is not None:
            main.wait_event(self.tail_done[b])           # raw disparities of set b were last read by the tail two calls ago
        with torch.cuda.stream(main):
            self._phase(2, b, left, lv, rv, out, N, main)
            ev = torch.cuda.Event(); ev.record(main)
            self.main_done[b] = ev
        # ---- tail: everything after WTA; `out` may still be read by work the caller queued before this call
        tail.wait_stream(caller)
        tail.wait_event(self.main_done[b])
        with torch.cuda.stream(tail):
            self._phase(4, b, left, lv, rv, out, N, tail)
            ev = torch.cuda.Event(); ev.record(tail)
            self.tail_done[b] = ev
        caller.wait_event(ev)
        self.lv, self.rv = self.lv2[b], self.rv2[b]     # the projected pair of the latest call
        return out

    def run_device_serial(self, left, right, hints, out=None, step=None):
        """The same computation, everything in order on the current stream (no overlap between calls, no internal streams
        except the right-image branches): what bench.py times stage by stage."""
        torch = self.torch
        N = self._check(left, right, hints, out)
        with torch.cuda.device(self.device):
            return self._run_device_serial(left, right, hints, out, step, N)

    def _run_device_serial(self, left, right, hints, out, step, N):
        torch, L = self.torch, self.lib
        out = self.disp[:N] if out is None else out
        st = torch.cuda.current_stream(self.device)
        for s in (self.vpp_stream, self.main_stream, self.tail_stream):
            st.wait_stream(s)
        b = self.calls & 1
        self.calls += 1
        lv, rv = self.lv2[b][:N], self.rv2[b][:N]
        seed = self._next_seed(step)
        lv.copy_(left); rv.copy_(right)
        rc = L.vppb200_vpp_scan_rnd(_lib.ptr(lv), _lib.ptr(rv), _lib.ptr(hints), self.W, self.H, self.C, 0, self.wsize,
                                    self.direction, C.c_double(self.blending), C.c_double(self.c_occ), _lib.ptr(self.occ),
                                    0, int(self.interpolate), 1, None, None, C.c_uint64(seed), None, _lib.ptr(self.ws_vpp),
                                    C.c_size_t(self.ws_vpp.numel()), N, C.c_void_p(st.cuda_stream))
        _lib.check(rc, "vpp_scan_rnd")
        self._phase(7, b, left, lv, rv, out, N, st)
        for s in (self.vpp_stream, self.main_stream, self.tail_stream):
            s.wait_stream(st)
        self.lv, self.rv = self.lv2[b], self.rv2[b]
        return out

    def run_host(self, left, right, hints):
        """Host tensors (ideally pinned) in, pinned host float32 [N,H,W] out; the copies are part of the call."""
        torch = self.torch
        N = self._check(left, right, hints, host=True)
        with torch.cuda.device(self.device):
            self.d_left[:N].copy_(left, non_blocking=True)
            self.d_right[:N].copy_(right, non_blocking=True)
            self.d_hints[:N].copy_(hints, non_blocking=True)
            out = self.run_device(self.d_left[:N], self.d_right[:N], self.d_hints[:N])
            self.h_disp[:N].copy_(out, non_blocking=True)
            torch.cuda.current_stream(self.device).synchronize()
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
                                     h_disp=torch.empty((self.N, self.H, self.W), dtype=torch.float32).pin_memory(),
                                     copied_in=torch.cuda.Event(), computed=torch.cuda.Event(), copied_out=torch.cuda.Event(),
                                     busy=False))
                self._stream_sets = dict(sets=sets, h2d=torch.cuda.Stream(self.device), d2h=torch.cuda.Stream(self.device), turn=0)
        return self._stream_sets

    def submit_host(self, left, right, hints, on_computed=None):
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
        N = self._check(left, right, hints, host=True)
        compute = torch.cuda.current_stream(self.device)
        with torch.cuda.device(self.device):
            with torch.cuda.stream(ss["h2d"]):
                # the staging set was last read by the compute of two submits ago, which collect() has waited for
                st["left"][:N].copy_(left, non_blocking=True)
                st["right"][:N].copy_(right, non_blocking=True)
                st["hints"][:N].copy_(hints, non_blocking=True)
                st["copied_in"].record(ss["h2d"])
            compute.wait_event(st["copied_in"])
            self.run_device(st["left"][:N], st["right"][:N], st["hints"][:N], out=st["disp"][:N], inputs_ready=st["copied_in"])
            st["computed"].record(compute)
            if on_computed is not None:
                on_computed(st["disp"][:N])
            with torch.cuda.stream(ss["d2h"]):
                ss["d2h"].wait_event(st["computed"])
                st["h_disp"][:N].copy_(st["disp"][:N], non_blocking=True)
                st["copied_out"].record(ss["d2h"])
        st["busy"], st["n"] = True, N
        ss["turn"] += 1
        return slot

    def collect(self, ticket):
        """Wait for a submitted batch; returns its pinned host float32 [N,H,W] disparities (valid until that staging set is
        reused by the `host_depth`-th submit_host after it was submitted)."""
        st = self._streaming()["sets"][ticket]
        if not st["busy"]:
            raise RuntimeError("collect: nothing in flight for this ticket")
        st["copied_out"].synchronize()
        st["busy"] = False
        return st["h_disp"][:st["n"]]
