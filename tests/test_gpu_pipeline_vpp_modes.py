"""VppRsgmPipeline with the projection options of test.py (vpp()'s keywords): the occlusion mask (--maskocc), the maxDistance
pattern and the adaptive patches, plus the device-side distance-patch thresholds (vppb200_distance_patch_thresholds) that
let the pipeline -- and vpp() -- compute the patch sizes without a host round trip.  Bar: bit-exact against the host
reference of the thresholds (vpp_standalone._patch_thresholds) and against the CPU oracle, per frame."""
import numpy as np
import pytest

from conftest import assert_same

H, W, DMAX = 60, 140, 64


@pytest.fixture(scope="module")
def mods():
    import torch
    assert torch.cuda.is_available()
    from vppstereo_b200 import _lib, synth, vpp_core_opt, vpp_standalone
    _lib.lib()
    return synth, vpp_core_opt, vpp_standalone


# ---- the R_k table (host, no device) ------------------------------------------------------------------------------------
@pytest.mark.parametrize("wsize", [1, 3, 5, 7, 9])
@pytest.mark.parametrize("gamma", [0.1, 0.3, 1, 2])
def test_ratio_steps_table(wsize, gamma):
    """R_k = the smallest float32 ratio in [0, 1] whose patch size (vpp_standalone.py:6-9 restated: float64 pow of the float32
    ratio, round half to even) is >= k: size(R_k) >= k and size(the float32 just below R_k) < k."""
    from vppstereo_b200 import vpp_standalone as vs
    size = lambda r: round((float(np.float32(r)) ** (1 / gamma)) * (wsize - 1) + 1)
    steps = vs._ratio_steps(wsize, gamma)
    assert steps.dtype == np.float32 and steps.shape == (wsize - 1,)
    for k in range(2, wsize + 1):
        r = steps[k - 2]
        assert 0 < r <= 1, (k, r)
        assert size(r) >= k, (k, r)
        assert size(np.nextafter(r, np.float32(0))) < k, (k, r)
        assert vs._patch_size(r, np.float32(0), np.float32(1), wsize, gamma) == size(r)


def test_bad_keywords():
    """Unknown method / bad window: ValueError from the constructor, before anything is allocated (no device needed)."""
    from vppstereo_b200.pipeline import VppRsgmPipeline
    with pytest.raises(ValueError, match="method"):
        VppRsgmPipeline(H, W, batch=2, dmax=DMAX, method="bogus")
    for kw in (dict(wsize=0), dict(wsizeAgg_x=0), dict(wsizeAgg_y=-1), dict(wsize=2.5)):
        with pytest.raises(ValueError):
            VppRsgmPipeline(H, W, batch=2, dmax=DMAX, **kw)


# ---- vppb200_distance_patch_thresholds against _patch_thresholds ------------------------------------------------------
def _frame_with_range(rng, dmin, dmax, h, w):
    """hints at 30 % of the pixels, values in [dmin, dmax], both ends present"""
    g = np.zeros((h, w), np.float32)
    idx = rng.choice(h * w, size=max(2, (h * w * 3) // 10), replace=False)
    v = rng.uniform(dmin, dmax, idx.size).astype(np.float32)
    v = np.clip(v, dmin, dmax)
    v[0], v[-1] = dmin, dmax
    g.reshape(-1)[idx] = v
    return g


RANGES = [(1.5, 190.25), (0.5, 3.0), (10.0, 10.5), (2.0, 64.0), (1.0, 200.0),             # test_patch_threshold_tabulation's
          (4.0, float(np.nextafter(np.float32(4.0), np.float32(9)))),                        # one ulp
          (100.0, float(np.float32(100.0) + np.float32(3 * 2 ** -17))), (0.5, 0.5000305)]    # a few ulps / a tiny span


@pytest.mark.gpu
@pytest.mark.parametrize("wsize", [1, 3, 5, 7, 9])
@pytest.mark.parametrize("gamma", [0.1, 0.3, 1, 2])
def test_thresholds_kernel_vs_host(mods, wsize, gamma):
    """Per frame, bit for bit: the thresholds of a batch that mixes frames of many (dmin, dmax) ranges, a frame without hints
    (+inf, status clear) and a frame whose hints all have one value (+inf, status set).  Odd frame size: the frames start at
    every 16-byte alignment, so the kernel's vector loads see every head / tail split."""
    import torch
    _, _, vs = mods
    rng = np.random.default_rng(wsize * 100 + int(gamma * 10))
    h, w = 17, 37
    ranges = RANGES + [tuple(sorted(rng.uniform(0.5, 250.0, 2).astype(np.float32).tolist())) for _ in range(6)]
    frames = [_frame_with_range(rng, np.float32(lo), np.float32(hi), h, w) for lo, hi in ranges]
    empty = len(frames); frames.append(np.zeros((h, w), np.float32))
    degen = len(frames); frames.append(np.where(rng.random((h, w)) < 0.2, np.float32(7.25), np.float32(0)).astype(np.float32))
    g = torch.from_numpy(np.stack(frames)).cuda()
    n = g.shape[0]
    steps = torch.from_numpy(vs._ratio_steps(wsize, gamma).copy()).cuda()
    thr = torch.full((n, wsize - 1), -1.0, dtype=torch.float32, device="cuda") if wsize > 1 else None
    status = torch.zeros(n, dtype=torch.int32, device="cuda")
    vs.distance_patch_thresholds(g, wsize, steps, thr, status, torch.cuda.current_stream().cuda_stream)
    st = status.cpu().numpy()
    assert st.tolist() == [0] * degen + [1], st
    if wsize == 1:
        return
    got = thr.cpu().numpy()
    for f in range(len(ranges)):
        pos = frames[f][frames[f] > 0]
        want = vs._patch_thresholds(pos.min(), pos.max(), wsize, gamma)
        assert_same(got[f], want, f"frame {f} range {ranges[f]}")
    assert np.isinf(got[empty]).all() and np.isinf(got[degen]).all()


@pytest.mark.gpu
def test_thresholds_kernel_full_frames(mods):
    """K-size frames (1242x375, the reduction's vector loop runs many rounds) with lidar-like hints."""
    import torch
    synth, _, vs = mods
    frames = [synth.make_pair(f, shape="K", hints="lidar", foreground=2)["hints"] for f in range(3)]
    g = torch.from_numpy(np.stack(frames)).cuda()
    steps = torch.from_numpy(vs._ratio_steps(7, 0.3).copy()).cuda()
    thr = torch.empty((3, 6), dtype=torch.float32, device="cuda")
    status = torch.zeros(3, dtype=torch.int32, device="cuda")
    vs.distance_patch_thresholds(g, 7, steps, thr, status, torch.cuda.current_stream().cuda_stream)
    assert not status.cpu().numpy().any()
    for f, fr in enumerate(frames):
        pos = fr[fr > 0]
        assert_same(thr[f].cpu().numpy(), vs._patch_thresholds(pos.min(), pos.max(), 7, 0.3), f"K frame {f}")


# ---- the pipeline against the oracle --------------------------------------------------------------------------------
def _batch(mods, C, f0, hints="random", n=2):
    synth = mods[0]
    frames = [synth.make_pair(f0 + i, shape=(H, W), hints=hints, channels=3, density=0.05, foreground=3) for i in range(n)]
    left = np.stack([p["left"][..., :C] for p in frames])
    right = np.stack([p["right"][..., :C] for p in frames])
    g = np.stack([(p["hints"] * np.float32(0.4)).astype(np.float32) for p in frames])
    return left, right, g


def _cuda(*arrays):
    import torch
    return tuple(torch.from_numpy(np.ascontiguousarray(a)).cuda() for a in arrays)


def _vpp_kw(kw):
    return {k: v for k, v in kw.items() if k != "maskocc"}


def _oracle(orc, mods, kw, left, right, g, seed):
    """per frame: (lw, rw, disparity) of test.py's chain on the oracle: occlusion mask, vpp (the device pattern of `seed` for
    rnd), compute_rsgm"""
    vco = mods[1]
    C = left.shape[-1]
    wsize, uniform = kw.get("wsize", 3), kw.get("uniform_color", False)
    out = []
    for i in range(left.shape[0]):
        mask = orc.occlusion_heuristic(g[i])[1] if kw.get("maskocc") else None
        li, ri = (left[i], right[i]) if C == 3 else (left[i][..., 0], right[i][..., 0])
        stream = None
        if kw.get("method", "rnd") == "rnd":
            stream = vco.device_pattern(seed, i, orc.stream_length(g[i], wsize, C, uniform))
        lw, rw = orc.vpp(li, ri, g[i], g_occ=mask, mode=1, stream=stream, **_vpp_kw(kw))
        out.append((lw.reshape(H, W, C), rw.reshape(H, W, C), orc.compute_rsgm(li, lw, rw, dmax=DMAX)))
    return out


CONFIGS = [
    dict(maskocc=True, c_occ=0.1),                                                           # the paper's default
    dict(maskocc=True, c_occ=0.1, method="maxDistance"),
    dict(maskocc=True, c_occ=0.1, wsize=7, use_bilateral_patch=True, use_distance_patch=True, bilateral_o_i=3),   # journal
    dict(maskocc=True, c_occ=0.1, wsize=7, use_bilateral_patch=True, use_distance_patch=True, method="maxDistance"),
    dict(wsize=5, use_bilateral_patch=True, bilateral_o_i=3),
    dict(maskocc=True, c_occ=0.2, wsize=5, use_distance_patch=True, discard_occ=True, left2right=False),
    dict(wsize=5, use_distance_patch=True, distance_gamma=1.0, uniform_color=True, method="maxDistance", wsizeAgg_x=16,
         wsizeAgg_y=5, left2right=False),
    dict(maskocc=True, c_occ=0.1, uniform_color=True),
    dict(maskocc=True, c_occ=0.1, wsize=5, use_bilateral_patch=True, discard_occ=True, method="maxDistance"),
    dict(maskocc=True, c_occ=0.1, discard_occ=True, left2right=False, method="maxDistance"),
]


@pytest.mark.gpu
@pytest.mark.parametrize("C", [3, 1])
@pytest.mark.parametrize("cfg", range(len(CONFIGS)))
def test_pipeline_modes_vs_oracle(mods, orc, cfg, C):
    """run_device of a 2-frame batch: the projected pair and the disparities equal the oracle's chain frame by frame."""
    import torch
    from vppstereo_b200.pipeline import VppRsgmPipeline
    kw = CONFIGS[cfg]
    left, right, g = _batch(mods, C, 10 * cfg + C, hints="lidar" if cfg % 2 else "random")
    if kw.get("maskocc"):
        masks = [orc.occlusion_heuristic(g[i])[1] for i in range(2)]
        assert any((m[g[i] > 0] == 1).any() for i, m in enumerate(masks)), "no hint is masked as occluded"
    pipe = VppRsgmPipeline(H, W, C, batch=2, dmax=DMAX, seed=5 + cfg, **kw)
    L, R, G = _cuda(left, right, g)
    pipe.run_device(L, R, G)                                   # call 1: a different pattern seed, buffers dirtied
    disp = pipe.run_device(L, R, G).clone()                    # call 2
    torch.cuda.synchronize()
    pipe.check()
    want = _oracle(orc, mods, kw, left, right, g, pipe.pattern_seed(2))
    for i, (lw, rw, d) in enumerate(want):
        assert_same(pipe.lv[i].cpu().numpy(), lw, f"cfg {cfg} C={C} frame {i}: left image")
        assert_same(pipe.rv[i].cpu().numpy(), rw, f"cfg {cfg} C={C} frame {i}: right image")
        assert_same(disp[i].cpu().numpy(), d, f"cfg {cfg} C={C} frame {i}: disparity")
    assert (pipe.lv.cpu().numpy() != left).any()
    pipe.close()


@pytest.mark.gpu
@pytest.mark.parametrize("kw", [CONFIGS[1], CONFIGS[2]], ids=["maskocc-maxDistance", "maskocc-bilateral-distance-rnd"])
def test_pipeline_modes_overlapped_match_serial(mods, orc, kw):
    """Five back-to-back run_device(inputs_ready=True) calls (the front phase -- mask, adaptive operands, scan -- of call k+1
    beside the sweeps of call k) return what run_device_serial returns, and the last one what the oracle computes."""
    import torch
    from vppstereo_b200.pipeline import VppRsgmPipeline
    batches = [_batch(mods, 3, 200 + 2 * b, hints="lidar" if b % 2 else "random") for b in range(5)]
    dev = [_cuda(*b) for b in batches]
    serial = VppRsgmPipeline(H, W, 3, batch=2, dmax=DMAX, seed=9, **kw)
    want = [serial.run_device_serial(*b).clone() for b in dev]
    pipe = VppRsgmPipeline(H, W, 3, batch=2, dmax=DMAX, seed=9, **kw)
    outs = [torch.empty((2, H, W), dtype=torch.float32, device="cuda") for _ in dev]
    for b, o in zip(dev, outs):
        pipe.run_device(*b, out=o, inputs_ready=True)
    torch.cuda.synchronize()
    pipe.check()
    for k in range(5):
        assert_same(outs[k].cpu().numpy(), want[k].cpu().numpy(), f"overlapped call {k}")
    ref = _oracle(orc, mods, kw, *batches[-1], pipe.pattern_seed(5))
    for i in range(2):
        assert_same(outs[-1][i].cpu().numpy(), ref[i][2], f"last call vs oracle, frame {i}")
    serial.close(); pipe.close()


@pytest.mark.gpu
def test_pipeline_modes_streaming_host_matches_run_host(mods):
    """submit_host / collect (copies and phases of neighbouring batches overlapped) against run_host, maskocc + maxDistance +
    adaptive patches."""
    import torch
    from vppstereo_b200.pipeline import VppRsgmPipeline
    kw = CONFIGS[3]
    batches = [tuple(torch.from_numpy(a).pin_memory() for a in _batch(mods, 3, 300 + 2 * b)) for b in range(5)]
    a = VppRsgmPipeline(H, W, 3, batch=2, dmax=DMAX, seed=3, **kw)
    want = [a.run_host(*b).clone() for b in batches]
    p = VppRsgmPipeline(H, W, 3, batch=2, dmax=DMAX, seed=3, **kw)
    got, tickets = [], []
    for b in batches:
        if len(tickets) == p.host_depth:
            got.append(p.collect(tickets.pop(0)).clone())
        tickets.append(p.submit_host(*b))
    got += [p.collect(t).clone() for t in tickets]
    for k in range(5):
        assert_same(got[k].numpy(), want[k].numpy(), f"streamed batch {k}")
    a.close(); p.close()


@pytest.mark.gpu
def test_pipeline_distance_patch_degenerate_frame(mods, orc):
    """use_distance_patch with a frame whose hints all have one value (the reference raises ZeroDivisionError): run_host
    raises it, and the next batch on the same pipeline is the oracle's (the status was cleared).  run_device does not raise
    (it does not synchronise); check() does, once."""
    import torch
    from vppstereo_b200.pipeline import VppRsgmPipeline
    kw = dict(maskocc=True, c_occ=0.1, wsize=5, use_distance_patch=True)
    left, right, g = _batch(mods, 3, 400)
    bad = g.copy()
    bad[1] = np.where(bad[1] > 0, np.float32(12.5), np.float32(0))
    pipe = VppRsgmPipeline(H, W, 3, batch=2, dmax=DMAX, seed=11, **kw)
    host = lambda *a: tuple(torch.from_numpy(x).pin_memory() for x in a)
    with pytest.raises(ZeroDivisionError, match="frame 1"):
        pipe.run_host(*host(left, right, bad))
    got = pipe.run_host(*host(left, right, g)).clone()          # call 2
    want = _oracle(orc, mods, kw, left, right, g, pipe.pattern_seed(2))
    for i in range(2):
        assert_same(got[i].numpy(), want[i][2], f"batch after the degenerate one, frame {i}")
    pipe.run_device(*_cuda(left, right, bad))                  # call 3: recorded for check(), not for run_host
    got = pipe.run_host(*host(left, right, g)).clone()          # call 4
    want = _oracle(orc, mods, kw, left, right, g, pipe.pattern_seed(4))
    for i in range(2):
        assert_same(got[i].numpy(), want[i][2], f"run_host beside an unchecked degenerate run_device, frame {i}")
    with pytest.raises(ZeroDivisionError, match="frame 1 of a run_device"):
        pipe.check()
    pipe.check()
    pipe.close()


@pytest.mark.gpu
def test_pipeline_distance_patch_degenerate_frame_streamed(mods):
    """submit_host / collect with three batches in flight and a degenerate frame in batch 2: only collect() of batch 2
    raises ZeroDivisionError; every other batch returns what run_host returns for it (each batch has its own status)."""
    import torch
    from vppstereo_b200.pipeline import VppRsgmPipeline
    kw = dict(maskocc=True, c_occ=0.1, wsize=5, use_distance_patch=True, use_bilateral_patch=True, bilateral_o_i=3)
    batches = [list(_batch(mods, 3, 500 + 2 * b)) for b in range(6)]
    batches[2][2][0] = np.where(batches[2][2][0] > 0, np.float32(9.75), np.float32(0))
    batches = [tuple(torch.from_numpy(np.ascontiguousarray(a)).pin_memory() for a in b) for b in batches]
    a = VppRsgmPipeline(H, W, 3, batch=2, dmax=DMAX, seed=13, **kw)
    want = []
    for k, b in enumerate(batches):
        if k == 2:
            with pytest.raises(ZeroDivisionError, match="frame 0"):
                a.run_host(*b)
            want.append(None)
        else:
            want.append(a.run_host(*b).clone())
    p = VppRsgmPipeline(H, W, 3, batch=2, dmax=DMAX, seed=13, **kw)
    results, tickets = {}, []

    def take(k, t):
        if k == 2:
            with pytest.raises(ZeroDivisionError, match="frame 0"):
                p.collect(t)
        else:
            results[k] = p.collect(t).clone()

    for k, b in enumerate(batches):
        if len(tickets) == p.host_depth:         # batches k-3 .. k-1 in flight: collect(k-3) after k-1's front was queued
            take(*tickets.pop(0))
        tickets.append((k, p.submit_host(*b)))
    for k, t in tickets:
        take(k, t)
    assert sorted(results) == [0, 1, 3, 4, 5]
    for k, got in results.items():
        assert_same(got.numpy(), want[k].numpy(), f"streamed batch {k}")
    p.check()                                    # nothing left over for check()
    a.close(); p.close()
