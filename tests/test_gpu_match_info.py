"""The per-pixel match info of compute_rsgm (opt-in, include/vppstereo_b200.h) on every path that produces it, bit for bit against
the restatement of its definition (match_info_reference.py): the fused backward sweep + WTA (sgm_h_kernel MODE 4), the per-row WTA on
the materialised volume (wta_rows_info_kernel: test tap, parameters outside the sweep domain, VPPB200_TUNE_SGM_SWEEP = 0), the info
variants of the tail kernels and the batched pipeline.  Turning the info on must not change a disparity."""
import numpy as np
import pytest

from conftest import assert_same
import match_info_reference as mi

pytestmark = pytest.mark.gpu

IN_DOMAIN, OUT_OF_DOMAIN = (11, 17, 0.5, 35), (30, 10, 0.5, 20)
# the shapes of test_gpu_uniqueness.py: D covers FULLK (64, 192, 256) and not (8, 72, 200); narrow widths give end < D-1 over many columns
CASES = [((37, 70), 8, 3, True, 1), ((46, 150), 64, 1, False, 2), ((33, 100), 72, 3, True, 3), ((40, 261), 192, 3, True, 1),
         ((30, 230), 200, 1, True, 2), ((29, 300), 256, 3, False, 1)]
KEYS = ("state", "cost", "rival")


@pytest.fixture(scope="module")
def mods():
    import torch
    assert torch.cuda.is_available()
    from vppstereo_b200 import _lib, rsgm, synth
    _lib.lib()
    _lib.set_tuning(_lib.TUNE_RCP_HOST, 1)            # the oracle's sub-pixel reciprocal is this host's RCPSS
    return rsgm, synth, _lib


@pytest.fixture
def tuning(mods):
    _lib = mods[2]
    yield lambda key, value: _lib.set_tuning(key, value)
    _lib.set_tuning(_lib.TUNE_SGM_SWEEP, 1)


def _kw(u=None, prm=None):
    kw = {} if u is None else dict(uniqueness=u, honor_uniqueness=True)
    if prm is not None:
        kw.update(p1=prm[0], p2min=prm[1], alpha=prm[2], gamma=prm[3], honor_params=True)
    return kw


def _frames(synth, seed, shape, channels, n, hints="random"):
    fr = [synth.make_pair(seed + f, shape=shape, hints=hints, channels=channels) for f in range(n)]
    return fr, np.stack([p["left"] for p in fr]), np.stack([p["right"] for p in fr])


def _same_info(got, want, what, f=None):
    for k in KEYS:
        assert_same(got[k] if f is None else got[k][f], want[k], f"{what} {k}")


@pytest.mark.parametrize("u", [None, 0.8])
@pytest.mark.parametrize("shape,D,channels,sub,n", CASES)
def test_compute_rsgm_info_vs_reference(mods, orc, shape, D, channels, sub, n, u):
    rsgm, synth = mods[0], mods[1]
    fr, left, right = _frames(synth, 900 + D, shape, channels, n)
    kw = dict(dmax=D, subpixel=sub, **_kw(u))
    disp, info = rsgm.compute_rsgm(left, left, right, return_info=True, **kw)          # fused sweep (MODE 4)
    assert_same(disp, rsgm.compute_rsgm(left, left, right, **kw), "disp with vs without the info")
    assert info["state"].dtype == np.uint8 and info["cost"].dtype == np.uint16 and info["state"].shape == disp.shape
    st = rsgm.compute_rsgm_stages(left, left, right, return_info=True, **kw)          # volume tap: wta_rows_info_kernel
    assert_same(st["out"], disp, "stages out")
    for f, p in enumerate(fr):
        want = mi.match_info(orc, p["left"], p["left"], p["right"], dmax=D, subpixel=sub, u=1.0 if u is None else u)
        assert_same(disp[f], want["disp"], f"disp {shape} D={D} u={u} frame {f}")
        _same_info(info, want, f"{shape} D={D} u={u} frame {f}", f)
        _same_info(st, want, f"stages {shape} D={D} u={u} frame {f}", f)


@pytest.mark.parametrize("guided", [False, True])
@pytest.mark.parametrize("prm", [None, IN_DOMAIN, OUT_OF_DOMAIN])
@pytest.mark.parametrize("u", [None, 0.8])
def test_params_and_guided(mods, orc, prm, guided, u):
    rsgm, synth = mods[0], mods[1]
    p = synth.make_pair(77, shape=(45, 130), hints="random")
    g = dict(hints=p["hints"], validhints=(p["hints"] > 0).astype(np.float32)) if guided else {}
    kw = dict(dmax=64, **g, **_kw(u, prm))
    disp, info = rsgm.compute_rsgm(p["left"], p["left"], p["right"], return_info=True, **kw)
    assert_same(disp, rsgm.compute_rsgm(p["left"], p["left"], p["right"], **kw), "disp with vs without the info")
    want = mi.match_info(orc, p["left"], p["left"], p["right"], dmax=64, params=prm or (7, 17, 0.25, 50), u=1.0 if u is None else u,
                         **g)
    assert_same(disp, want["disp"], f"disp params {prm} guided={guided} u={u}")
    _same_info(info, want, f"params {prm} guided={guided} u={u}")


def test_paths_agree_and_costs_ignore_uniqueness(mods, tuning):
    """fused sweep, volume tap and the per-path kernels (TUNE_SGM_SWEEP = 0) give the same info; cost / rival do not depend on
    whether the uniqueness test is honoured"""
    import torch
    rsgm, synth, _lib = mods
    _, left, right = _frames(synth, 300, (30, 200), 3, 2, hints="lidar")
    L, R = (torch.from_numpy(a).cuda() for a in (left, right))
    runs = {}
    for u in (None, 0.9):
        d, info = rsgm.compute_rsgm(L, L, R, dmax=64, return_info=True, **_kw(u))          # CUDA tensors in -> CUDA tensors out
        assert info["state"].is_cuda and info["cost"].dtype == _lib.u16_dtype() and info["rival"].shape == (2, 30, 200)
        runs[(u, "sweep")] = (d.cpu().numpy(), {k: _lib.dev_to_np(t, np.uint8 if k == "state" else np.uint16) for k, t in info.items()})
        st = rsgm.compute_rsgm_stages(left, left, right, dmax=64, return_info=True, **_kw(u))
        runs[(u, "taps")] = (st["out"], st)
        tuning(_lib.TUNE_SGM_SWEEP, 0)
        runs[(u, "per-path")] = rsgm.compute_rsgm(left, left, right, dmax=64, return_info=True, **_kw(u))
        tuning(_lib.TUNE_SGM_SWEEP, 1)
    for u in (None, 0.9):
        for path in ("taps", "per-path"):
            assert_same(runs[(u, path)][0], runs[(u, "sweep")][0], f"disp {path} u={u}")
            _same_info(runs[(u, path)][1], runs[(u, "sweep")][1], f"{path} vs sweep u={u}")
    for k in ("cost", "rival"):
        assert_same(runs[(0.9, "sweep")][1][k], runs[(None, "sweep")][1][k], f"{k}: uniqueness on vs off")
    assert not np.array_equal(runs[(0.9, "sweep")][1]["state"], runs[(None, "sweep")][1]["state"])


def _kernel_names(fn):
    import torch
    from torch.profiler import ProfilerActivity, profile
    torch.cuda.synchronize()
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        fn()
        torch.cuda.synchronize()
    return [e.name for e in prof.events() if e.device_type == torch.autograd.DeviceType.CUDA]


def test_profiler_kernels(mods):
    """the default call launches none of the info variants; the info call at the bench shape launches as many kernels, with the
    fused backward sweep in MODE 4 and the three left-view tail kernels in their info variants"""
    import torch
    from vppstereo_b200 import synth
    rsgm = mods[0]
    p = synth.make_pair(5, shape=(375, 1242), hints="lidar")
    L, R = (torch.from_numpy(p[k]).cuda() for k in ("left", "right"))
    run = lambda **kw: rsgm.compute_rsgm(L, L, R, dmax=192, **kw)
    run(); run(return_info=True)                                     # warm-up
    dflt = _kernel_names(run)
    info = _kernel_names(lambda: run(return_info=True))
    assert not any("info" in n or "sgm_h_kernel<3, 4," in n for n in dflt), sorted(set(dflt))
    assert any("sgm_h_kernel<3, 2, -1" in n for n in dflt), sorted(set(dflt))
    assert len(info) == len(dflt), (sorted(set(info)), sorted(set(dflt)))
    assert any("sgm_h_kernel<3, 4, -1" in n for n in info) and not any("sgm_h_kernel<3, 2, -1" in n for n in info), sorted(set(info))
    for k in ("interp_clip_info_kernel", "speckle_rows_info_kernel", "speckle_apply_info_kernel"):
        assert sum(k in n for n in info) == 1, (k, sorted(set(info)))
    strip = lambda names: sorted(n for n in names if "sgm_h_kernel" not in n and "interp_clip" not in n and "speckle_rows" not in n
                                 and "speckle_apply" not in n)
    assert strip(info) == strip(dflt)


def _to_np(info):
    from vppstereo_b200 import _lib
    return {k: _lib.dev_to_np(t, np.uint8 if k == "state" else np.uint16) for k, t in info.items()}


@pytest.mark.parametrize("opts", [{}, dict(maskocc=True), dict(maskocc=True, method="maxDistance")], ids=["rnd", "maskocc", "maxDistance"])
def test_pipeline_info(mods, opts):
    """every way of calling a match_info pipeline gives, call by call, compute_rsgm(return_info=True) of its projected pair"""
    import torch
    from vppstereo_b200.pipeline import VppRsgmPipeline
    rsgm, synth = mods[0], mods[1]
    frames = [synth.make_pair(80 + f, shape=(60, 140), hints="lidar") for f in range(5)]
    batches = [tuple(torch.from_numpy(np.stack([q[k] for q in frames[b:b + 2]])).cuda() for k in ("left", "right", "hints"))
               for b in (0, 2)]
    batches.append(tuple(torch.from_numpy(frames[4][k][None]).cuda() for k in ("left", "right", "hints")))   # partial batch
    for mode in ("device", "serial", "host", "stream"):
        pipe = VppRsgmPipeline(60, 140, 3, batch=2, dmax=64, seed=3, match_info=True, **opts)
        outs = []
        for k, b in enumerate(batches + batches[:1]):
            if mode == "device":
                out, info = pipe.run_device(*b)
            elif mode == "serial":
                out, info = pipe.run_device_serial(*b)
            elif mode == "host":
                out, info = pipe.run_host(*(t.cpu().pin_memory() for t in b))
            else:
                ticket = pipe.submit_host(*(t.cpu().pin_memory() for t in b))
                torch.cuda.synchronize()                             # the projected pair below is read before the next submit
            if mode == "stream":
                outs.append([None, None, b[0], pipe.lv[:b[0].shape[0]].clone(), pipe.rv[:b[0].shape[0]].clone(), ticket])
                if k % 2 == 1 or k == len(batches):
                    for o in outs:
                        if o[0] is None:
                            d, i = pipe.collect(o[5])
                            o[0], o[1] = d.clone(), _to_np({kk: t.clone() for kk, t in i.items()})   # (pinned, reused)
                continue
            outs.append([out.clone(), _to_np({kk: t.clone() for kk, t in info.items()}), b[0], pipe.lv[:b[0].shape[0]].clone(),
                         pipe.rv[:b[0].shape[0]].clone()])
        torch.cuda.synchronize()
        for k, (out, info, left, lv, rv, *_) in enumerate(outs):
            d, want = rsgm.compute_rsgm(left, lv, rv, dmax=64, return_info=True)
            assert_same(out.cpu().numpy(), d.cpu().numpy(), f"pipeline {mode} call {k}")
            _same_info(info, _to_np(want), f"pipeline {mode} call {k}")
        pipe.close()


def test_pipeline_default_unchanged_and_info_out(mods):
    """without match_info the entry points return what they always returned; info_out is validated like `out`, refused by a
    pipeline without match_info, and filled when given"""
    import torch
    from vppstereo_b200 import _lib
    from vppstereo_b200.pipeline import VppRsgmPipeline
    synth = mods[1]
    p = synth.make_pair(11, shape=(60, 140), hints="lidar")
    L, R, G = (torch.from_numpy(p[k][None]).cuda() for k in ("left", "right", "hints"))
    plain = VppRsgmPipeline(60, 140, 3, batch=2, dmax=64, seed=5)
    pipe = VppRsgmPipeline(60, 140, 3, batch=2, dmax=64, seed=5, match_info=True)
    want = plain.run_device(L, R, G, step=1)
    assert isinstance(want, torch.Tensor)
    good = {"state": torch.empty((1, 60, 140), dtype=torch.uint8, device="cuda"),
            "cost": torch.empty((1, 60, 140), dtype=_lib.u16_dtype(), device="cuda"),
            "rival": torch.empty((1, 60, 140), dtype=_lib.u16_dtype(), device="cuda")}
    with pytest.raises(ValueError, match="info_out"):
        plain.run_device(L, R, G, info_out=good)
    with pytest.raises(ValueError, match="info_out"):
        plain.run_device_serial(L, R, G, info_out=good)
    bad = [(TypeError, dict(good, cost=good["cost"].to(torch.int32))), (TypeError, dict(good, state=good["cost"])),
           (ValueError, dict(good, rival=good["rival"][:, :, :100])), (ValueError, dict(good, state=good["state"].cpu())),
           (ValueError, dict(good, cost=torch.empty((1, 140, 60), dtype=_lib.u16_dtype(), device="cuda").transpose(1, 2))),
           (TypeError, {"state": good["state"]})]
    for exc, io in bad:
        with pytest.raises(exc):
            pipe.run_device(L, R, G, info_out=io)
    out, info = pipe.run_device(L, R, G, step=1, info_out=good)
    assert info is good
    torch.cuda.synchronize()
    assert_same(out.cpu().numpy(), want.cpu().numpy(), "match_info pipeline vs plain")
    out2, info2 = pipe.run_device_serial(L, R, G, step=1)
    torch.cuda.synchronize()
    assert_same(out2.cpu().numpy(), want.cpu().numpy(), "serial")
    _same_info(_to_np(info2), _to_np(good), "own buffers vs info_out")
    pipe.close(); plain.close()
