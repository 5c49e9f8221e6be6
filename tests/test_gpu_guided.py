"""Guided matching (models/rsgm/rsgm.py:115-127, `compute_rsgm(..., hints, validhints)`) on every path that runs it:
the cost kernel with the modulation fused in (compute_rsgm), the row bands (BandedRsgm / BandedRsgmDist) and the batched pipeline
(VppRsgmPipeline(guided=True)).  All bit-exact: compute_rsgm against the oracle, the others against compute_rsgm."""
import os
import subprocess
import sys

import numpy as np
import pytest

from conftest import ROOT, assert_same

pytestmark = pytest.mark.gpu

GUIDED_OOD = (3700, 3700, 0.0, 3856)        # inside the Hamming sweep domain, outside the guided one


def _pads(H, W):
    pad_h, pad_w = (((H // 16) + 1) * 16 - H) % 16, (((W // 16) + 1) * 16 - W) % 16
    return pad_h // 2, pad_h - pad_h // 2, pad_w // 2, pad_w - pad_w // 2


def dense_hints(seed, H, W, D, density=0.3):
    """hints at ~30 % of the pixels (every row, the first and last two included), non-integer, some beyond D; validhints that
    differ from hints > 0 both ways (0 on some hinted pixels, 1 on some pixels without a hint)"""
    rng = np.random.default_rng(seed)
    mask = rng.random((H, W)) < density
    h = np.where(mask, rng.uniform(0.25, 1.25 * D + 4, (H, W)), 0).astype(np.float32)
    valid = (h > 0).astype(np.float32)
    valid[mask & (rng.random((H, W)) < 0.15)] = 0.0
    valid[~mask & (rng.random((H, W)) < 0.05)] = 1.0
    return h, valid


def _frames(seed, shape, D, n, channels):
    from vppstereo_b200 import synth
    out = []
    for f in range(n):
        p = synth.make_pair(seed + f, shape=shape, hints="random", channels=channels)
        p["hints"], p["valid"] = dense_hints(seed + 100 + f, shape[0], shape[1], D)
        out.append(p)
    return out


# (shape, D, channels, sub-pixel, frames): paddings non-zero on both sides, and pad_top <= 1 so that constant-12 rows of the padded
# frame lie inside the user frame (46: pad 1 + 1; 47: 0 + 1; 45: 1 + 2)
CASES = [((37, 70), 8, 3, True, 1), ((46, 150), 64, 1, False, 2), ((47, 261), 192, 3, True, 3), ((45, 300), 256, 3, False, 1),
         ((61, 99), 64, 3, True, 2), ((46, 90), 256, 1, True, 1)]


@pytest.mark.parametrize("shape,D,channels,sub,n", CASES)
def test_guided_compute_rsgm_vs_oracle(orc, shape, D, channels, sub, n):
    from vppstereo_b200 import rsgm
    fr = _frames(500 + D + n, shape, D, n, channels)
    left = np.stack([p["left"] for p in fr]); right = np.stack([p["right"] for p in fr])
    hints = np.stack([p["hints"] for p in fr]); valid = np.stack([p["valid"] for p in fr])
    got = rsgm.compute_rsgm(left if n > 1 else left[0], left if n > 1 else left[0], right if n > 1 else right[0],
                            hints=hints if n > 1 else hints[0], validhints=valid if n > 1 else valid[0], dmax=D, subpixel=sub)
    got = got if n > 1 else got[None]
    for f, p in enumerate(fr):
        want = orc.compute_rsgm(p["left"], p["left"], p["right"], hints=p["hints"], validhints=p["valid"], dmax=D, subpixel=sub)
        assert_same(got[f], want, f"guided compute_rsgm {shape} D={D} C={channels} sub={sub} frame {f}/{n}")
        # the gate is validhints, not hints > 0: the case has hinted pixels with valid = 0 and unhinted ones with valid = 1
        assert ((p["valid"] > 0) & (p["hints"] == 0)).any() and ((p["valid"] == 0) & (p["hints"] > 0)).any()
        assert (p["hints"][[0, 1, -2, -1]] > 0).any(axis=1).all() and (p["hints"] > D).any() and (p["hints"] % 1 != 0).any()


@pytest.mark.parametrize("shape,D", [((46, 150), 64), ((47, 100), 192)])
def test_guided_aggregated_volume_vs_oracle(orc, shape, D):
    """the dsi_agg tap: the oracle's guided cost volume (orc.guided_dsi) aggregated by the oracle"""
    from vppstereo_b200 import rsgm
    p = _frames(77 + D, shape, D, 1, 3)[0]
    st = rsgm.compute_rsgm_stages(p["left"], p["left"], p["right"], hints=p["hints"], validhints=p["valid"], dmax=D)
    H, W = shape
    pt, pb, pl, pr = _pads(H, W)
    cl, cr = st["census_l"][0], st["census_r"][0]
    Hp, Wp = cl.shape
    dsi = np.zeros((Hp, Wp, D), np.uint16)
    orc.costMeasureCensus5x5_xyd_SSE(cl, cr, dsi, Wp, Hp, D)
    hp = np.zeros((Hp, Wp), np.float32); vp = np.zeros((Hp, Wp), np.float32)
    hp[pt:pt + H, pl:pl + W] = p["hints"]; vp[pt:pt + H, pl:pl + W] = p["valid"]
    dsi = orc.guided_dsi(dsi, hp, vp)
    S = np.zeros_like(dsi)
    orc.aggregate_SSE(orc.pad_reflect(p["left"], pt, pb, pl, pr), dsi, S, Wp, Hp, D)
    assert_same(st["dsi_agg"][0], S, f"guided aggregated volume {shape} D={D}")


def _kernel_names(fn):
    import torch
    from torch.profiler import ProfilerActivity, profile
    torch.cuda.synchronize()
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        fn()
        torch.cuda.synchronize()
    return {e.name for e in prof.events() if e.device_type == torch.autograd.DeviceType.CUDA}


def test_guided_modulation_is_fused_into_the_cost_kernel():
    from vppstereo_b200 import rsgm
    p = _frames(9, (40, 96), 32, 1, 3)[0]
    run = lambda: rsgm.compute_rsgm(p["left"], p["left"], p["right"], hints=p["hints"], validhints=p["valid"], dmax=32)
    run()
    names = _kernel_names(run)
    assert any("cost_tile_kernel" in n for n in names), sorted(names)
    assert any("sgm_v2_kernel" in n for n in names), sorted(names)
    assert not any("guided_tile_kernel" in n or "guided_u8_kernel" in n for n in names), sorted(names)
    assert sum("cost_tile_kernel" in n for n in names) == 1, sorted(names)


# ---------------------------------------------------------------- row bands
BAND_CASES = [((40, 120), 64, 2), ((61, 200), 192, 3), ((90, 330), 48, 5), ((33, 70), 32, 1), ((128, 700), 96, 4), ((50, 100), 8, 7)]


@pytest.mark.parametrize("shape,D,nb", BAND_CASES)
def test_guided_bands_on_one_gpu_equal_unsplit(orc, shape, D, nb):
    from vppstereo_b200 import rsgm
    from vppstereo_b200.banded import BandedRsgm
    p = _frames(700 + D + nb, shape, D, 1, 3)[0]
    g = dict(hints=p["hints"], validhints=p["valid"])
    want = rsgm.compute_rsgm(p["left"], p["left"], p["right"], dmax=D, **g)
    assert_same(want, orc.compute_rsgm(p["left"], p["left"], p["right"], dmax=D, **g), "unsplit vs oracle")
    b = BandedRsgm(shape[0], shape[1], 3, dmax=D, n_bands=nb)
    got = b.compute(p["left"], p["left"], p["right"], **g)
    assert_same(got, want, f"{nb} guided bands {shape} D={D}")
    got2 = b.compute(p["left"], p["left"], p["right"], **g)           # buffers reused
    assert_same(got2, want, "second call")
    plain = b.compute(p["left"], p["left"], p["right"])                 # the same object unguided
    assert_same(plain, rsgm.compute_rsgm(p["left"], p["left"], p["right"], dmax=D), "unguided call on the same object")


def test_guided_bands_narrow_strips_and_gray():
    from vppstereo_b200 import _lib, rsgm
    from vppstereo_b200.banded import BandedRsgm
    p = _frames(31, (70, 400), 64, 1, 1)[0]
    g = dict(hints=p["hints"], validhints=p["valid"])
    for strip in (0, 64):
        _lib.set_tuning(_lib.TUNE_SGM_MAX_STRIP, strip)
        try:
            want = rsgm.compute_rsgm(p["left"], p["left"], p["right"], dmax=64, subpixel=False, **g)
            got = BandedRsgm(70, 400, 1, dmax=64, n_bands=3, subpixel=False).compute(p["left"], p["left"], p["right"], **g)
            assert_same(got, want, f"strip {strip}")
        finally:
            _lib.set_tuning(_lib.TUNE_SGM_MAX_STRIP, 0)


@pytest.mark.parametrize("nb", [1, 3])
def test_guided_bands_honour_params(nb):
    import torch
    from vppstereo_b200 import rsgm
    from vppstereo_b200.banded import BandedRsgm
    prm = (3, 30, 0.3, 80)
    p = _frames(710 + nb, (61, 200), 64, 1, 3)[0]
    l, r = torch.from_numpy(p["left"]).cuda(), torch.from_numpy(p["right"]).cuda()
    h, v = torch.from_numpy(p["hints"]).cuda(), torch.from_numpy(p["valid"]).cuda()
    want = rsgm.compute_rsgm(l, l, r, hints=h, validhints=v, dmax=64, p1=prm[0], p2min=prm[1], alpha=prm[2], gamma=prm[3],
                             honor_params=True)
    got = BandedRsgm(61, 200, 3, dmax=64, n_bands=nb, sgm_params=prm).compute(l, l, r, hints=h, validhints=v)
    assert torch.is_tensor(got) and got.is_cuda
    assert_same(got.cpu().numpy(), want.cpu().numpy(), f"{nb} guided bands, honoured parameters")


def test_guided_bands_argument_errors():
    from vppstereo_b200.banded import BandedRsgm
    p = _frames(5, (40, 120), 32, 1, 3)[0]
    b = BandedRsgm(40, 120, 3, dmax=32, n_bands=2, sgm_params=GUIDED_OOD)     # fine for Hamming costs
    with pytest.raises(ValueError, match="guided"):
        b.compute(p["left"], p["left"], p["right"], hints=p["hints"], validhints=p["valid"])
    b = BandedRsgm(40, 120, 3, dmax=32, n_bands=2)
    with pytest.raises(ValueError):
        b.compute(p["left"], p["left"], p["right"], hints=p["hints"])
    with pytest.raises(ValueError):
        b.compute(p["left"], p["left"], p["right"], validhints=p["valid"])
    with pytest.raises(ValueError):
        b.compute(p["left"], p["left"], p["right"], hints=p["hints"][:20], validhints=p["valid"][:20])


def test_guided_one_band_per_rank_two_gpus(tmp_path):
    import torch
    if torch.cuda.device_count() < 2:
        pytest.skip("needs two GPUs")
    port = 29800 + os.getpid() % 90
    cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node", "2", "--master-addr", "127.0.0.1",
           "--master-port", str(port), os.path.join(ROOT, "tests", "mgpu_banded_guided_worker.py"), str(tmp_path)]
    r = subprocess.run(cmd, capture_output=True, text=True, timeout=900, cwd=ROOT)
    assert r.returncode == 0, r.stdout[-2000:] + r.stderr[-4000:]
    for rank in range(2):
        text = open(tmp_path / f"rank{rank}.txt").read()
        assert text.startswith("OK"), text


# ---------------------------------------------------------------- batched pipeline
PH, PW, PD, PB = 60, 140, 64, 3


@pytest.fixture(scope="module")
def pipe_batches():
    """six batches of PB frames with LiDAR hints and their validhints, the last one partial (N = 2), resident on the device"""
    import torch
    from vppstereo_b200 import synth
    out = []
    for b in range(6):
        n = PB if b < 5 else 2
        fr = [synth.make_pair(80 + PB * b + f, shape=(PH, PW), hints="lidar") for f in range(n)]
        hints = np.stack([q["hints"] for q in fr])
        valid = (hints > 0).astype(np.float32)
        valid[:, ::7, ::5] = 1.0                                      # gates that differ from hints > 0
        valid[:, 1::9, :] = 0.0
        out.append(tuple(torch.from_numpy(np.ascontiguousarray(a)).cuda()
                         for a in (np.stack([q["left"] for q in fr]), np.stack([q["right"] for q in fr]), hints, valid)))
    torch.cuda.synchronize()
    return out


def _run_overlapped(pipe, batches):
    """consecutive run_device calls without a host synchronisation in between (inputs resident: the phases of neighbouring
    calls overlap, except across the change to the partial batch); the outputs, captured in current-stream order"""
    import torch
    res = [pipe.run_device(l, r, h, inputs_ready=True, validhints=v).clone() for l, r, h, v in batches]
    torch.cuda.synchronize()
    pipe.check()
    return res


def _run_serial(pipe, batches):
    """run_device_serial call by call: the outputs and the projected pairs"""
    import torch
    res = []
    for l, r, h, v in batches:
        N = l.shape[0]
        out = pipe.run_device_serial(l, r, h, validhints=v).clone()
        res.append((out, pipe.lv[:N].clone(), pipe.rv[:N].clone()))
        torch.cuda.synchronize()
    return res


def test_guided_pipeline_run_device(pipe_batches):
    """overlapped run_device and in-order run_device_serial (same seed, same call order) both equal guided compute_rsgm of the
    projected pair, call by call, both buffer sets and a partial batch included"""
    from vppstereo_b200 import rsgm
    from vppstereo_b200.pipeline import VppRsgmPipeline
    mk = lambda: VppRsgmPipeline(PH, PW, 3, batch=PB, dmax=PD, seed=3, guided=True)
    serial, pipe = mk(), mk()
    ser = _run_serial(serial, pipe_batches)
    outs = _run_overlapped(pipe, pipe_batches)
    for k, ((l, r, h, v), (sout, lv, rv), out) in enumerate(zip(pipe_batches, ser, outs)):
        want = rsgm.compute_rsgm(l, lv, rv, hints=h, validhints=v, dmax=PD)
        assert_same(sout.cpu().numpy(), want.cpu().numpy(), f"run_device_serial call {k + 1} (N={l.shape[0]})")
        assert_same(out.cpu().numpy(), want.cpu().numpy(), f"run_device call {k + 1} (N={l.shape[0]})")
    serial.close(); pipe.close()


def test_guided_pipeline_vs_oracle(orc, pipe_batches):
    """one batch through the projection and the guided matcher of the oracle, with the pattern the device drew"""
    import torch
    from vppstereo_b200 import vpp_core_opt
    from vppstereo_b200.pipeline import VppRsgmPipeline
    pipe = VppRsgmPipeline(PH, PW, 3, batch=PB, dmax=PD, seed=11, guided=True)
    l, r, h, v = pipe_batches[1]
    out = pipe.run_device(l, r, h, validhints=v).clone()
    torch.cuda.synchronize()
    ln, rn, hn, vn = (t.cpu().numpy() for t in (l, r, h, v))
    for f in range(l.shape[0]):
        pattern = vpp_core_opt.device_pattern(pipe.pattern_seed(1), f, orc.stream_length(hn[f], 3, 3, False))
        lw, rw = orc.vpp(ln[f], rn[f], hn[f], stream=pattern, mode=1)
        assert_same(pipe.lv[f].cpu().numpy(), lw, f"frame {f}: projected left")
        want = orc.compute_rsgm(ln[f], lw, rw, hints=hn[f], validhints=vn[f], dmax=PD)
        assert_same(out[f].cpu().numpy(), want, f"frame {f}: disparities")
    pipe.close()


def test_guided_pipeline_host_entry_points(pipe_batches):
    """run_host and submit_host / collect compute what run_device computes (same seed, same call order)"""
    from vppstereo_b200.pipeline import VppRsgmPipeline
    batches = pipe_batches[:4] + pipe_batches[5:] + pipe_batches[4:5]
    mk = lambda: VppRsgmPipeline(PH, PW, 3, batch=PB, dmax=PD, seed=5, guided=True)
    ref = mk()
    want = [o.cpu().numpy() for o in _run_overlapped(ref, batches)]
    ref.close()
    host_b = [tuple(t.cpu().pin_memory() for t in b) for b in batches]
    hp = mk()
    for k, (l, r, h, v) in enumerate(host_b):
        assert_same(hp.run_host(l, r, h, validhints=v).numpy(), want[k], f"run_host call {k + 1}")
    hp.close()
    sp = mk()
    tickets, got = [], []
    for l, r, h, v in host_b:
        if len(tickets) == sp.host_depth:
            got.append(sp.collect(tickets.pop(0)).numpy().copy())
        tickets.append(sp.submit_host(l, r, h, validhints=v))
    while tickets:
        got.append(sp.collect(tickets.pop(0)).numpy().copy())
    for k, g in enumerate(got):
        assert_same(g, want[k], f"submit_host call {k + 1}")
    sp.close()


@pytest.mark.parametrize("prm", [(3, 30, 0.3, 80), GUIDED_OOD, (30, 10, 0.5, 20)])
def test_guided_pipeline_sgm_params(pipe_batches, prm):
    """honoured parameters inside the guided sweep domain (sweeps) and outside it (per-path kernels, through the same phases)"""
    from vppstereo_b200 import _lib, rsgm
    from vppstereo_b200.pipeline import VppRsgmPipeline
    fast = _lib.sgm_params_fast(_lib.sgm_params(*prm), guided=True)
    assert fast == (prm == (3, 30, 0.3, 80))
    pipe = VppRsgmPipeline(PH, PW, 3, batch=PB, dmax=PD, seed=3, guided=True, sgm_params=prm)
    serial = VppRsgmPipeline(PH, PW, 3, batch=PB, dmax=PD, seed=3, guided=True, sgm_params=prm)
    outs = _run_overlapped(pipe, pipe_batches[:3])
    for k, ((l, r, h, v), out, (sout, lv, rv)) in enumerate(zip(pipe_batches[:3], outs, _run_serial(serial, pipe_batches[:3]))):
        assert_same(out.cpu().numpy(), sout.cpu().numpy(), f"{prm} call {k + 1}: run_device vs run_device_serial")
        want = rsgm.compute_rsgm(l, lv, rv, hints=h, validhints=v, dmax=PD, p1=prm[0], p2min=prm[1], alpha=prm[2], gamma=prm[3],
                                 honor_params=True)
        assert_same(out.cpu().numpy(), want.cpu().numpy(), f"{prm} call {k + 1}")
    pipe.close(); serial.close()


def test_guided_pipeline_argument_errors(pipe_batches):
    import torch
    from vppstereo_b200.pipeline import VppRsgmPipeline
    l, r, h, v = pipe_batches[0]
    g = VppRsgmPipeline(PH, PW, 3, batch=PB, dmax=PD, guided=True)
    u = VppRsgmPipeline(PH, PW, 3, batch=PB, dmax=PD)
    assert g.d_valid is not None and u.d_valid is None
    calls0 = g.calls
    with pytest.raises(ValueError, match="validhints"):
        g.run_device(l, r, h)
    with pytest.raises(ValueError, match="validhints"):
        g.run_device_serial(l, r, h)
    with pytest.raises(ValueError, match="validhints"):
        g.run_host(l.cpu(), r.cpu(), h.cpu())
    with pytest.raises(ValueError, match="validhints"):
        g.submit_host(l.cpu(), r.cpu(), h.cpu())
    with pytest.raises(ValueError, match="validhints"):
        u.run_device(l, r, h, validhints=v)
    with pytest.raises(ValueError, match="validhints"):
        u.run_host(l.cpu(), r.cpu(), h.cpu(), validhints=v.cpu())
    with pytest.raises(TypeError, match="validhints"):
        g.run_device(l, r, h, validhints=v.double())
    with pytest.raises(ValueError, match="validhints"):
        g.run_device(l, r, h, validhints=v[:2])
    with pytest.raises(ValueError, match="validhints"):
        g.run_device(l, r, h, validhints=v.cpu())
    assert g.calls == calls0, "a refused call must not advance the pipeline"
    torch.cuda.synchronize()
    g.close(); u.close()
