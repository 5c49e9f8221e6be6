"""compute_rsgm of an OVERSIZED frame with the aggregation split into row bands (SURVEY.md 8e rows 2 and 5).

The 8-path aggregation is what makes a frame big: at Middlebury size the Hamming volume and the aggregated volume are 1.1 + 2.2 GB
per frame.  Census, cost volume, the horizontal sweeps and WTA are row local; the three vertical / diagonal paths of each pass chain
through all rows.  The reference's own answer, `StripedStereoSGM` (RSGM/StereoSGM.h:116-133), restarts those paths a few rows above
each strip and is approximate.  Here the split is EXACT: a band's v-sweep continues from the row state (the three paths'
L(x, d) and their minima for one image row, 3.4 MB at Middlebury width) that the neighbouring band's sweep exported, so the bands
form a pipeline -- pass 0 flows down the bands, pass 1 flows back up -- and the result equals the unsplit compute_rsgm bit for bit.

    BandedRsgm(H, W, ...).compute(left, left_vpp, right_vpp)            one GPU, bands one after the other (a frame whose volumes
                                                                        do not fit beside other work; also the parity reference)
    BandedRsgmDist(H, W, ...).compute(left, left_vpp, right_vpp)        one band per rank (one process per GPU): the row state and
                                                                        the raw disparity bands travel over NVLink through
                                                                        peer-mapped buffers (dist.PeerGather: copy engines + stream
                                                                        wait-value flags, no collective kernel)

Where a STREAM of frames has to go fast, shard by frame instead (dist.run_sharded / bench.py): frames are independent, a band
pipeline cannot beat that -- its sweeps do the same work plus the hand-off -- and the chain of rows of one frame is serial either
way (DESIGN.md 6 has the measurements).
"""
import ctypes as C

from . import _lib
from .dist import shard_range

PH_COST, PH_H_FWD, PH_V_DOWN, PH_V_UP, PH_H_BWD = 1, 2, 4, 8, 16


class BandedRsgm:
    def __init__(self, H, W, channels=3, dmax=192, n_bands=2, subpixel=True, device=None, sgm_params=None, uniqueness=None):
        # sgm_params: (p1, p2min, alpha, gamma) honoured by the sweeps; None = the reference's effective values.  Bands exist on the
        # sweeps only, so parameters outside their domain (include/vppstereo_b200.h) are refused here.
        # uniqueness: the WTA's uniqueness ratio (compute_rsgm(..., honor_uniqueness=True)); None = off
        self.uniqueness = 1.0 if uniqueness is None else _lib.uniqueness(uniqueness, "BandedRsgm")
        self.sgm_params = None
        if sgm_params is not None:
            prm = _lib.sgm_params(*sgm_params)
            if not _lib.sgm_params_fast(prm, guided=False):
                raise ValueError(f"SGM parameters {tuple(sgm_params)} are outside the sweep domain (no banded path for them)")
            self.sgm_params = prm
        torch = _lib.require_cuda()
        self.torch = torch
        self.H, self.W, self.C, self.D = int(H), int(W), int(channels), int(dmax)
        if self.D % 8 != 0:
            raise Exception(f"Invalid dmax ({dmax}): dmax % 8 != 0")            # models/rsgm/rsgm.py:31-32
        if self.D > 256:
            raise Exception(f"Invalid dmax ({dmax}): dmax > 256")               # models/rsgm/rsgm.py:34-35
        self.subpixel = bool(subpixel)
        self.device = torch.device("cuda", torch.cuda.current_device()) if device is None else torch.device(device)
        L = _lib.lib()
        hp, wp, sw, vb = C.c_int(0), C.c_int(0), C.c_int64(0), C.c_int64(0)
        _lib.call("vppb200_banded_dims", self.H, self.W, self.C, self.D, C.byref(hp), C.byref(wp), C.byref(sw), C.byref(vb),
                  what="banded_dims")
        self.Hp, self.Wp, self.state_words, self.vol_row_bytes = hp.value, wp.value, sw.value, vb.value
        self.bands = self._split(int(n_bands))
        with torch.cuda.device(self.device):
            self.ws = torch.empty(L.vppb200_banded_workspace_bytes(self.H, self.W, self.C, self.D), dtype=torch.uint8, device=self.device)
            self.guide = torch.empty(self.Hp * self.Wp, dtype=torch.uint8, device=self.device)
            self.cl = torch.empty((self.Hp, self.Wp), dtype=torch.int32, device=self.device)
            self.cr = torch.empty_like(self.cl)
            self.dl = torch.empty((self.Hp, self.Wp), dtype=torch.float32, device=self.device)
            self.dr = torch.empty_like(self.dl)

    def _split(self, n):
        """row bands of the PADDED frame, at least 3 rows each"""
        n = max(1, min(n, self.Hp // 3))
        out = []
        for r in range(n):
            lo, hi = shard_range(self.Hp, r, n)
            out.append((lo, hi - lo))
        return out

    def band_buffers(self, rows):
        """(cost, S) layout-T volumes of a band of `rows` rows"""
        torch = self.torch
        with torch.cuda.device(self.device):
            return (torch.empty(rows * self.vol_row_bytes, dtype=torch.uint8, device=self.device),
                    torch.empty(rows * self.vol_row_bytes, dtype=torch.int16, device=self.device))

    def state_buffer(self):
        with self.torch.cuda.device(self.device):
            return self.torch.empty(self.state_words, dtype=self.torch.int32, device=self.device)

    def _images(self, left, left_vpp, right_vpp):
        torch = self.torch
        out = []
        for t in (left, left_vpp, right_vpp):
            t = _lib.as_device(t, torch.uint8, self.device)
            if t.dim() == 2:
                t = t[..., None]
            if tuple(t.shape) != (self.H, self.W, self.C):
                raise ValueError(f"expected one frame of shape {(self.H, self.W, self.C)}, got {tuple(t.shape)}")
            out.append(t.contiguous())
        return out

    def front(self, left, left_vpp, right_vpp):
        """pad + gray + census of the whole frame (rsgm.py:254-262, :8-28)"""
        l, lv, rv = self._images(left, left_vpp, right_vpp)
        with self.torch.cuda.device(self.device):
            _lib.call("vppb200_rsgm_front_census", _lib.ptr(l), _lib.ptr(lv), _lib.ptr(rv), _lib.ptr(self.guide), _lib.ptr(self.cl),
                      _lib.ptr(self.cr), self.H, self.W, self.C, self.D, _lib.ptr(self.ws), self.ws.numel(),
                      _lib.stream_ptr(self.device), what="rsgm_front_census")

    def run_band(self, band, phases, cost, S, state_in=None, state_out=None, stream=None, hints=None, validhints=None):
        """phases of one band (vppb200_sgm_band_guided); hints / validhints: float32 [H,W] CUDA tensors of the whole frame or both
        None, the same nullness for every phase of every band of a frame"""
        row0, rows = band
        torch = self.torch
        dl = self.dl[row0:row0 + rows]
        dr = self.dr[row0:row0 + rows]
        with torch.cuda.device(self.device):
            st = _lib.stream_ptr(self.device) if stream is None else stream.cuda_stream
            _lib.call("vppb200_sgm_band_uniq", _lib.ptr(self.guide), _lib.ptr(self.cl), _lib.ptr(self.cr), _lib.ptr(cost),
                      _lib.ptr(S), self.H, self.W, self.C, self.D, row0, rows, int(phases), _lib.ptr(state_in), _lib.ptr(state_out),
                      _lib.ptr(dl), _lib.ptr(dr), None, _lib.ptr(self.ws), self.ws.numel(), st, self.sgm_params, _lib.ptr(hints),
                      _lib.ptr(validhints), self.uniqueness, what="sgm_band")

    def _hints(self, hints, validhints):
        """guided matching operands (rsgm.py:115-127) as compute_rsgm takes them -> (hints, validhints) float32 [H,W] CUDA tensors,
        or (None, None).  Refused with ValueError before any device work: one operand without the other, and parameters outside the
        guided sweep domain (there is no per-path band path)."""
        if (hints is None) != (validhints is None):
            raise ValueError("hints and validhints must be given together")
        if hints is None:
            return None, None
        if self.sgm_params is not None and not _lib.sgm_params_fast(self.sgm_params, guided=True):
            p = self.sgm_params
            raise ValueError(f"SGM parameters {(p.p1, p.p2min, p.alpha, p.gamma)} are outside the guided sweep domain (no banded path "
                             "for them)")
        out = []
        for name, a in (("hints", hints), ("validhints", validhints)):
            t = _lib.as_device(a, self.torch.float32, self.device)
            if t.numel() != self.H * self.W:
                raise ValueError(f"{name}: expected one frame of shape {(self.H, self.W)}, got {tuple(t.shape)}")
            out.append(t.reshape(self.H, self.W).contiguous())
        return tuple(out)

    def tail(self, out=None):
        """median .. background fill on the raw maps of the whole frame (rsgm.py:273-292)"""
        torch = self.torch
        with torch.cuda.device(self.device):
            out = torch.empty((self.H, self.W), dtype=torch.float32, device=self.device) if out is None else out
            _lib.call("vppb200_rsgm_tail", _lib.ptr(self.dl), _lib.ptr(self.dr), _lib.ptr(out), self.H, self.W, self.C, self.D,
                      1 if self.subpixel else 0, _lib.ptr(self.ws), self.ws.numel(), _lib.stream_ptr(self.device), what="rsgm_tail")
        return out

    def compute(self, left, left_vpp, right_vpp, hints=None, validhints=None):
        """compute_rsgm(left, left_vpp, right_vpp, hints, validhints) -> float32 [H,W]: all bands on this GPU, one after the other.
        numpy in -> numpy out, CUDA tensors in -> CUDA tensor out.  hints / validhints: guided matching, float32 [H,W], both or
        neither (ValueError otherwise)."""
        h, v = self._hints(hints, validhints)
        host = not _lib.is_tensor(left_vpp)
        self.front(left, left_vpp, right_vpp)
        bufs = [self.band_buffers(rows) for _, rows in self.bands]
        states = [self.state_buffer() for _ in self.bands]
        nb = len(self.bands)
        for k, band in enumerate(self.bands):                          # pass 0 flows down the bands
            self.run_band(band, PH_COST | PH_H_FWD | PH_V_DOWN, *bufs[k], state_in=states[k - 1] if k > 0 else None,
                          state_out=states[k] if k + 1 < nb else None, hints=h, validhints=v)
        ups = [self.state_buffer() for _ in self.bands]
        for k in reversed(range(nb)):                                  # pass 1 flows back up, then the band's last sweep + WTA
            self.run_band(self.bands[k], PH_V_UP | PH_H_BWD, *bufs[k], state_in=ups[k + 1] if k + 1 < nb else None,
                          state_out=ups[k] if k > 0 else None, hints=h, validhints=v)
        out = self.tail()
        return out.cpu().numpy() if host else out


class BandedRsgmDist(BandedRsgm):
    """One band per rank of the process group (one process per GPU).  Every rank calls compute() with the same frame; the row state
    travels rank r -> r+1 (pass 0) and r -> r-1 (pass 1), the raw disparity bands go to every rank, every rank runs the (cheap,
    whole-frame) tail and returns the full disparity map.  Transfers: dist.PeerGather (peer-mapped buffers, DMA, flag words)."""

    def __init__(self, H, W, channels=3, dmax=192, subpixel=True, device=None, group=None, sgm_params=None, uniqueness=None):
        import torch.distributed as dist
        from .dist import PeerGather
        self.group = group
        self.world = dist.get_world_size(group) if dist.is_initialized() else 1
        self.rank = dist.get_rank(group) if dist.is_initialized() else 0
        super().__init__(H, W, channels, dmax, n_bands=self.world, subpixel=subpixel, device=device, sgm_params=sgm_params,
                         uniqueness=uniqueness)
        if len(self.bands) != self.world:
            raise ValueError("frame too small for one band per rank")
        torch = self.torch
        self.band = self.bands[self.rank]
        self.cost, self.S = self.band_buffers(self.band[1])
        rows_max = max(r for _, r in self.bands)
        # mailboxes: [slot = message kind][source rank]: 0 = row state of pass 0 (from rank-1), 1 = row state of pass 1 (from rank+1)
        self.state_box = PeerGather((self.state_words,), torch.int32, self.device, group=group, depth=2)
        self.disp_box = PeerGather((2, rows_max, self.Wp), torch.float32, self.device, group=group, depth=2)
        self.frame = 0

    def compute(self, left, left_vpp, right_vpp, hints=None, validhints=None):
        """as BandedRsgm.compute (hints / validhints: the whole frame on every rank)"""
        h, v = self._hints(hints, validhints)
        torch = self.torch
        host = not _lib.is_tensor(left_vpp)
        r, nb, f = self.rank, self.world, self.frame
        self.frame += 1
        sb, db = self.state_box, self.disp_box
        self.front(left, left_vpp, right_vpp)
        self.run_band(self.band, PH_COST | PH_H_FWD, self.cost, self.S, hints=h, validhints=v)
        # ---- pass 0: wait for the band above, sweep down, hand the row state to the band below
        state_in = None
        if r > 0:
            sb.wait_from(2 * f, r - 1)
            state_in = sb.bufs[0, r - 1]
        out_state = self.state_buffer() if r + 1 < nb else None
        self.run_band(self.band, PH_V_DOWN, self.cost, self.S, state_in=state_in, state_out=out_state, hints=h, validhints=v)
        if r > 0:
            sb.release_to(2 * f, r - 1)
        if r + 1 < nb:
            sb.send(2 * f, out_state, r + 1)
        # ---- pass 1: wait for the band below, sweep up, hand the row state to the band above; then the last sweep + WTA
        state_in = None
        if r + 1 < nb:
            sb.wait_from(2 * f + 1, r + 1)
            state_in = sb.bufs[1, r + 1]
        out_state = self.state_buffer() if r > 0 else None
        self.run_band(self.band, PH_V_UP | PH_H_BWD, self.cost, self.S, state_in=state_in, state_out=out_state, hints=h,
                      validhints=v)
        if r + 1 < nb:
            sb.release_to(2 * f + 1, r + 1)
        if r > 0:
            sb.send(2 * f + 1, out_state, r - 1)
        # ---- raw disparities of every band to every rank, then the whole-frame tail everywhere
        row0, rows = self.band
        mine = torch.zeros(db.shape, dtype=torch.float32, device=self.device)
        mine[0, :rows] = self.dl[row0:row0 + rows]
        mine[1, :rows] = self.dr[row0:row0 + rows]
        db.push(f, mine)
        full = db.wait(f)
        for q, (q0, qn) in enumerate(self.bands):
            if q != r:
                self.dl[q0:q0 + qn] = full[q, 0, :qn]
                self.dr[q0:q0 + qn] = full[q, 1, :qn]
        db.release(f)
        out = self.tail()
        return out.cpu().numpy() if host else out

    def close(self):
        self.state_box.close()
        self.disp_box.close()
