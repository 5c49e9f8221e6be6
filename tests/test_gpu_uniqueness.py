"""The uniqueness ratio of the winner-takes-all (opt-in, include/vppstereo_b200.h) on every path that runs it, bit for bit: the
fused backward sweep + WTA (sgm_h_kernel MODE 3), the per-row WTA on the materialised volume (wta_rows_uniq_kernel: test tap,
parameters outside the sweep domain, VPPB200_TUNE_SGM_SWEEP = 0, the pyrSGM operators), the row bands and the batched pipeline."""
import numpy as np
import pytest

from conftest import assert_same
import uniq_reference as ref

pytestmark = pytest.mark.gpu

U = [0.5, 0.8, 0.95, 0.999]


def _pads(H, W):
    pad_h, pad_w = (((H // 16) + 1) * 16 - H) % 16, (((W // 16) + 1) * 16 - W) % 16
    return pad_h // 2, pad_h - pad_h // 2, pad_w // 2, pad_w - pad_w // 2


def oracle_rsgm(orc, left, left_vpp, right_vpp, hints=None, validhints=None, dmax=192, subpixel=True, params=(7, 17, 0.25, 50),
                u=1.0):
    """orc_compute_rsgm step by step on the oracle's operators with honoured SGM parameters, WTA by the uniqueness test's
    reference (uniq_reference.py; u = 1 is the plain first arg-min)"""
    left, left_vpp, right_vpp = (np.ascontiguousarray(a, np.uint8) for a in (left, left_vpp, right_vpp))
    H, W = left.shape[:2]
    D = int(dmax)
    pt, pb, pl, pr = _pads(H, W)
    lp, lvp, rvp = (orc.pad_reflect(a, pt, pb, pl, pr) for a in (left, left_vpp, right_vpp))
    Hp, Wp = lp.shape[:2]
    gray = (lambda a: orc.rgb2gray(a)) if lvp.ndim == 3 and lvp.shape[2] == 3 else (lambda a: np.ascontiguousarray(a.reshape(Hp, Wp)))
    cl = np.zeros((Hp, Wp), np.uint32); cr = np.zeros((Hp, Wp), np.uint32)
    orc.census5x5_SSE(gray(lvp), cl, Wp, Hp); orc.census5x5_SSE(gray(rvp), cr, Wp, Hp)
    dsi = np.zeros((Hp, Wp, D), np.uint16)
    orc.costMeasureCensus5x5_xyd_SSE(cl, cr, dsi, Wp, Hp, D)
    if hints is not None:
        hp = np.zeros((Hp, Wp), np.float32); vp = np.zeros((Hp, Wp), np.float32)
        hp[pt:pt + H, pl:pl + W] = hints; vp[pt:pt + H, pl:pl + W] = validhints
        dsi = orc.guided_dsi(dsi, hp, vp)
    S = np.zeros_like(dsi)
    orc.aggregate_SSE(lp, dsi, S, Wp, Hp, D, *params, honor_params=True)
    maps, raw = [], []
    for wta, sub in ((ref.wta_left, True), (ref.wta_right, False)):
        d = np.ascontiguousarray(wta(S, u))
        if sub:
            orc.subPixelRefine(S, d, Wp, Hp, D, 0)
        f = np.zeros((Hp, Wp), np.float32)
        orc.median3x3_SSE(d, f, Wp, Hp)
        orc.linear_interpolate(f, 15, 3.0)
        f[f < 0] = 0
        raw.append(f.copy())
        maps.append(np.ascontiguousarray(f[pt:pt + H, pl:pl + W]))
    fl, fr = maps
    mask = orc.left_right_check(fl, fr, 1.0)
    u8 = np.where(mask == 128, np.float32(0), fl).astype(np.uint8)
    u8 = orc.filter_speckles_u8(u8, 0, 200, 10)
    out = u8.astype(np.float32)
    if subpixel:
        out = np.where(out != 0, fl, out).astype(np.float32)
    out = np.ascontiguousarray(out)
    orc.interpolate_background(out)
    return out, raw[0], raw[1]


@pytest.fixture(scope="module")
def mods():
    import torch
    assert torch.cuda.is_available()
    from vppstereo_b200 import _lib, pyrSGM, rsgm, synth
    _lib.lib()
    _lib.set_tuning(_lib.TUNE_RCP_HOST, 1)            # the oracle's sub-pixel reciprocal is this host's RCPSS
    return rsgm, synth, _lib, pyrSGM


@pytest.fixture
def tuning(mods):
    _lib = mods[2]
    yield lambda key, value: _lib.set_tuning(key, value)
    _lib.set_tuning(_lib.TUNE_SGM_MAX_STRIP, 0)
    _lib.set_tuning(_lib.TUNE_SGM_SWEEP, 1)


def _uq(u, prm=None):
    kw = dict(uniqueness=u, honor_uniqueness=True)
    if prm is not None:
        kw.update(p1=prm[0], p2min=prm[1], alpha=prm[2], gamma=prm[3], honor_params=True)
    return kw


IN_DOMAIN, OUT_OF_DOMAIN = (11, 17, 0.5, 35), (30, 10, 0.5, 20)
# (shape, D, channels, sub-pixel, frames): D covers FULLK (64, 192, 256) and not (8, 72, 200); narrow widths give end < D-1 over
# many columns
CASES = [((37, 70), 8, 3, True, 1), ((46, 150), 64, 1, False, 2), ((33, 100), 72, 3, True, 3), ((40, 261), 192, 3, True, 1),
         ((30, 230), 200, 1, True, 2), ((29, 300), 256, 3, False, 1)]


@pytest.mark.parametrize("u", U)
@pytest.mark.parametrize("shape,D,channels,sub,n", CASES)
def test_compute_rsgm_uniq_vs_oracle(mods, orc, shape, D, channels, sub, n, u):
    rsgm, synth = mods[0], mods[1]
    fr = [synth.make_pair(900 + D + f, shape=shape, hints="random", channels=channels) for f in range(n)]
    left = np.stack([p["left"] for p in fr]); right = np.stack([p["right"] for p in fr])
    st = rsgm.compute_rsgm_stages(left, left, right, dmax=D, subpixel=sub, **_uq(u))       # xyd path (the volume tap)
    got = rsgm.compute_rsgm(left, left, right, dmax=D, subpixel=sub, **_uq(u))             # fused sweep
    for f, p in enumerate(fr):
        want, dl, dr = oracle_rsgm(orc, p["left"], p["left"], p["right"], dmax=D, subpixel=sub, u=u)
        assert_same(st["disp_l"][f], dl, f"disp_l {shape} D={D} u={u} frame {f}")
        assert_same(st["disp_r"][f], dr, f"disp_r {shape} D={D} u={u} frame {f}")
        assert_same(st["out"][f], want, f"stages out {shape} D={D} u={u} frame {f}")
        assert_same(got[f], want, f"compute_rsgm {shape} D={D} u={u} frame {f}")


@pytest.mark.parametrize("shape,D,channels,sub,n", CASES)
def test_u1_equals_default(mods, shape, D, channels, sub, n):
    rsgm, synth = mods[0], mods[1]
    fr = [synth.make_pair(40 + D + f, shape=shape, hints="random", channels=channels) for f in range(n)]
    left = np.stack([p["left"] for p in fr]); right = np.stack([p["right"] for p in fr])
    assert_same(rsgm.compute_rsgm(left, left, right, dmax=D, subpixel=sub, **_uq(1.0)),
                rsgm.compute_rsgm(left, left, right, dmax=D, subpixel=sub), "u = 1 vs default")
    a = rsgm.compute_rsgm_stages(left, left, right, dmax=D, subpixel=sub, **_uq(1.0))
    b = rsgm.compute_rsgm_stages(left, left, right, dmax=D, subpixel=sub)
    for k in ("disp_l", "disp_r", "out"):
        assert_same(a[k], b[k], f"u = 1 vs default {k}")


@pytest.mark.parametrize("u", [0.8, 0.95])
@pytest.mark.parametrize("prm", [IN_DOMAIN, OUT_OF_DOMAIN])
def test_honoured_params_and_guided(mods, orc, prm, u):
    rsgm, synth = mods[0], mods[1]
    p = synth.make_pair(77, shape=(45, 130), hints="random")
    v = (p["hints"] > 0).astype(np.float32)
    want, _, _ = oracle_rsgm(orc, p["left"], p["left"], p["right"], dmax=64, params=prm, u=u)
    assert_same(rsgm.compute_rsgm(p["left"], p["left"], p["right"], dmax=64, **_uq(u, prm)), want, f"params {prm} u={u}")
    want, _, _ = oracle_rsgm(orc, p["left"], p["left"], p["right"], hints=p["hints"], validhints=v, dmax=64, params=prm, u=u)
    got = rsgm.compute_rsgm(p["left"], p["left"], p["right"], hints=p["hints"], validhints=v, dmax=64, **_uq(u, prm))
    assert_same(got, want, f"guided params {prm} u={u}")


@pytest.mark.parametrize("sweep,strip", [(0, 0), (1, 32), (1, 64)])
def test_tuning_paths(mods, orc, tuning, sweep, strip):
    rsgm, synth, _lib = mods[0], mods[1], mods[2]
    tuning(_lib.TUNE_SGM_SWEEP, sweep)
    tuning(_lib.TUNE_SGM_MAX_STRIP, strip)
    fr = [synth.make_pair(300 + f, shape=(30, 200), hints="random") for f in range(2)]
    left = np.stack([q["left"] for q in fr]); right = np.stack([q["right"] for q in fr])
    got = rsgm.compute_rsgm(left, left, right, dmax=64, **_uq(0.9))
    for f, q in enumerate(fr):
        want, _, _ = oracle_rsgm(orc, q["left"], q["left"], q["right"], dmax=64, u=0.9)
        assert_same(got[f], want, f"sweep={sweep} strip={strip} frame {f}")


def _adversarial(rng, H, W, D):
    S = rng.integers(0, 65536, (H, W, D), dtype=np.uint16)
    S[0] = 65535                                                     # saturated rows: genuine 65535 rivals
    S[1] = rng.integers(65533, 65536, (W, D))
    S[2] = 7                                                         # flat
    S[3] = rng.integers(0, 3, (W, D))                                # ties everywhere
    return S


@pytest.mark.parametrize("D", [8, 64, 72, 192, 256])
@pytest.mark.parametrize("u", U + [1e-4])
def test_pyrsgm_operators_vs_reference(mods, D, u):
    pyrSGM = mods[3]
    rng = np.random.default_rng(D)
    H, W = 6, 96
    for S in (_adversarial(rng, H, W, D), rng.integers(100, 110, (H, W, D), dtype=np.uint16)):
        for op, want_fn in ((pyrSGM.matchWTA_SSE, ref.wta_left), (pyrSGM.matchWTARight_SSE, ref.wta_right)):
            got = np.zeros((H, W), np.float32)
            op(S, got, W, H, D, u, honor_uniqueness=True)
            assert_same(got, want_fn(S, u), f"{op.__name__} D={D} u={u}")
            plain = np.zeros((H, W), np.float32)
            op(S, plain, W, H, D, u)
            op(S, got, W, H, D, 1.0, honor_uniqueness=True)
            assert_same(got, plain, f"{op.__name__} u = 1 vs plain")


@pytest.mark.parametrize("nb", [1, 2, 3, 7])
def test_banded_uniq(mods, nb):
    from vppstereo_b200.banded import BandedRsgm
    rsgm, synth = mods[0], mods[1]
    p = synth.make_pair(710 + nb, shape=(61, 200), hints="random")
    for u in (0.8, 1.0):
        want = rsgm.compute_rsgm(p["left"], p["left"], p["right"], dmax=64, **_uq(u))
        got = BandedRsgm(61, 200, 3, dmax=64, n_bands=nb, uniqueness=u).compute(p["left"], p["left"], p["right"])
        assert_same(got, want, f"{nb} bands u={u}")
    with pytest.raises(TypeError):
        BandedRsgm(61, 200, 3, dmax=64, n_bands=nb, uniqueness=0.0)


def test_pipeline_uniq(mods):
    import torch
    from vppstereo_b200.pipeline import VppRsgmPipeline
    rsgm, synth = mods[0], mods[1]
    frames = [synth.make_pair(80 + f, shape=(60, 140), hints="lidar") for f in range(5)]
    batches = [tuple(torch.from_numpy(np.stack([q[k] for q in frames[b:b + 2]])).cuda() for k in ("left", "right", "hints"))
               for b in (0, 2)]
    batches.append(tuple(torch.from_numpy(frames[4][k][None]).cuda() for k in ("left", "right", "hints")))   # partial batch
    for mode in ("device", "serial", "host"):
        pipe = VppRsgmPipeline(60, 140, 3, batch=2, dmax=64, seed=3, uniqueness=0.85)
        outs = []
        for b in batches + batches[:1]:
            if mode == "device":
                out = pipe.run_device(*b)
            elif mode == "serial":
                out = pipe.run_device_serial(*b)
            else:
                out = pipe.run_host(*(t.cpu().pin_memory() for t in b))
            outs.append((out.clone(), b[0], pipe.lv[:b[0].shape[0]].clone(), pipe.rv[:b[0].shape[0]].clone()))
        torch.cuda.synchronize()
        for k, (out, left, lv, rv) in enumerate(outs):
            want = rsgm.compute_rsgm(left, lv, rv, dmax=64, **_uq(0.85))
            assert_same(out.cpu().numpy(), want.cpu().numpy(), f"pipeline {mode} call {k}")
        pipe.close()
    with pytest.raises(TypeError):
        VppRsgmPipeline(60, 140, 3, batch=2, dmax=64, uniqueness=float("nan"))


def _kernel_names(fn):
    import torch
    from torch.profiler import ProfilerActivity, profile
    torch.cuda.synchronize()
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        fn()
        torch.cuda.synchronize()
    return [e.name for e in prof.events() if e.device_type == torch.autograd.DeviceType.CUDA]


def test_profiler_kernels(mods):
    """default and u = 1 launch the same kernels and none of the opt-in variants; an opt-in call at the bench shape launches as
    many kernels, with the fused backward sweep replaced by its MODE 3 instantiation"""
    import torch
    from vppstereo_b200 import synth
    rsgm = mods[0]
    p = synth.make_pair(5, shape=(375, 1242), hints="lidar")
    L, R = (torch.from_numpy(p[k]).cuda() for k in ("left", "right"))
    run = lambda **kw: rsgm.compute_rsgm(L, L, R, dmax=192, **kw)
    run(); run(**_uq(0.9))                                           # warm-up
    dflt = _kernel_names(run)
    one = _kernel_names(lambda: run(**_uq(1.0)))
    opt = _kernel_names(lambda: run(**_uq(0.9)))
    assert sorted(dflt) == sorted(one)
    assert not any("uniq" in n or "sgm_h_kernel<3, 3," in n for n in dflt), sorted(set(dflt))
    assert len(opt) == len(dflt), (sorted(set(opt)), sorted(set(dflt)))
    assert any("sgm_h_kernel<3, 3, -1" in n for n in opt) and not any("sgm_h_kernel<3, 2, -1" in n for n in opt), sorted(set(opt))
