"""Honoured SGM parameters (compute_rsgm(honor_params=True), VppRsgmPipeline / BandedRsgm(sgm_params=...), the C ABI's
vppb200_compute_rsgm_ex / vppb200_sgm_band_ex): bit-exact against the oracle's StereoSGM recursion with the parameters as
arguments, on the four sweeps inside their parameter domain and on the saturating per-path kernels outside it.

The parity target is `oracle_rsgm` below: the oracle's compute_rsgm pipeline (oracle/rsgm_oracle.c, orc_compute_rsgm) restated
from the oracle's own operators, with aggregate_SSE(honor_params=True) as the aggregation step; a CPU test pins it to
orc.compute_rsgm at the reference's effective parameters.  The CPU-only cases carry no gpu mark."""
import ctypes

import numpy as np
import pytest

from conftest import assert_same

# (p1, p2min, alpha, gamma) inside the sweep domain
IN_DOMAIN = [
    (11, 17, 0.5, 35),          # rsgm.py's own defaults
    (3, 30, 0.3, 80),           # non-dyadic alpha: the float product and its truncation matter
    (5, 20, 1.0 / 3.0, 60),
    (17, 17, 0.5, 40),          # P1 = P2min
    (10, 10, 0.5, 265),         # P2max - P1 = 255
    (0, 0, 0.0, 0),
    (7, 17, 0.25, 50),          # the reference's effective values, honoured
]
# outside it: the per-path kernels
OUT_OF_DOMAIN = [
    (30, 10, 0.5, 20),          # P2min < P1
    (10, 20, 0.5, 266),         # gamma - P1 = 256
    (7, 17, 0.25, 40000),       # lines entering through the border start at C + P2: S saturates
]
BAD = [(-1, 17, 0.5, 35), (7, 17, 0.5, 65536), (7, 17, -0.5, 35), (7, 17, float("nan"), 35), (7, 70000, 0.5, 35),
       (7, 17, float("inf"), 35)]


def _pads(H, W):
    pad_h, pad_w = (((H // 16) + 1) * 16 - H) % 16, (((W // 16) + 1) * 16 - W) % 16
    return pad_h // 2, pad_h - pad_h // 2, pad_w // 2, pad_w - pad_w // 2


def oracle_rsgm(orc, left, left_vpp, right_vpp, hints=None, validhints=None, dmax=192, subpixel=True, params=(7, 17, 0.25, 50)):
    """orc_compute_rsgm (models/rsgm/rsgm.py:250-294) step by step on the oracle's operators, with the SGM parameters taking
    effect: pad (BORDER_REFLECT) -> gray -> census -> cost volume (+ guided) -> aggregate_SSE(honor_params=True) -> WTA left +
    sub-pixel / WTA right -> median + interpolation + clip -> crop -> LR check -> speckles -> sub-pixel restore -> background fill"""
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
    if hints is not None and validhints is not None:
        hp = np.zeros((Hp, Wp), np.float32); vp = np.zeros((Hp, Wp), np.float32)
        hp[pt:pt + H, pl:pl + W] = hints; vp[pt:pt + H, pl:pl + W] = validhints
        dsi = orc.guided_dsi(dsi, hp, vp)
    S = np.zeros_like(dsi)
    orc.aggregate_SSE(lp, dsi, S, Wp, Hp, D, *params, honor_params=True)      # guide: the first Wp*Hp bytes of the padded left
    maps = []
    for wta, sub in ((orc.matchWTA_SSE, True), (orc.matchWTARight_SSE, False)):
        d = np.zeros((Hp, Wp), np.float32)
        wta(S, d, Wp, Hp, D)
        if sub:
            orc.subPixelRefine(S, d, Wp, Hp, D, 0)
        f = np.zeros((Hp, Wp), np.float32)
        orc.median3x3_SSE(d, f, Wp, Hp)
        orc.linear_interpolate(f, 15, 3.0)
        f[f < 0] = 0
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
    return out


def _oracle_agg(orc, left, st, D, prm, hints=None, valid=None):
    """the oracle's aggregated volume of one frame from the stage taps' census images: cost volume (+ guided modulation) and
    StereoSGM with the parameters as arguments, guided by the first Wp*Hp bytes of the padded `left` (RSGM/pyrSGM.cpp:586-588)"""
    H, W = left.shape[:2]
    pt, pb, pl, pr = _pads(H, W)
    cl, cr = st["census_l"][0], st["census_r"][0]
    Hp, Wp = cl.shape
    dsi = np.zeros((Hp, Wp, D), np.uint16)
    orc.costMeasureCensus5x5_xyd_SSE(cl, cr, dsi, Wp, Hp, D)
    if hints is not None:
        hp = np.zeros((Hp, Wp), np.float32); vp = np.zeros((Hp, Wp), np.float32)
        hp[pt:pt + H, pl:pl + W] = hints; vp[pt:pt + H, pl:pl + W] = valid
        dsi = orc.guided_dsi(dsi, hp, vp)
    lp = orc.pad_reflect(left, pt, pb, pl, pr)
    S = np.zeros_like(dsi)
    orc.aggregate_SSE(lp, dsi, S, Wp, Hp, D, *prm, honor_params=True)
    return S


# ---------------------------------------------------------------- CPU: validation before any device work
def _abi_args(L, bad):
    """otherwise valid arguments of vppb200_compute_rsgm_ex / vppb200_sgm_band_ex on host buffers (never dereferenced: the
    parameters are refused first)"""
    buf = (ctypes.c_uint8 * 64)()
    one = ctypes.cast(buf, ctypes.c_void_p)
    H, W, C, D = 16, 32, 3, 16
    ws = L.vppb200_rsgm_workspace_bytes(H, W, C, D, 1)
    prm = ctypes.byref(_params_struct(bad))
    rsgm = (one, one, one, None, None, one, H, W, C, D, 1, one, one, ctypes.c_size_t(ws), 1, None, 7, 1, 0, None, prm)
    bws = L.vppb200_banded_workspace_bytes(H, W, C, D)
    band = (one, one, one, one, one, H, W, C, D, 0, H, 31, None, None, one, one, one, one, ctypes.c_size_t(bws), None, prm)
    return rsgm, band


def _params_struct(p):
    from vppstereo_b200 import _lib
    return _lib.VppSgmParams(int(p[0]), int(p[1]), float(p[2]), int(p[3]))


@pytest.mark.parametrize("bad", BAD[:5])
def test_ex_entry_points_refuse_bad_params(bad):
    from vppstereo_b200 import _lib
    L = _lib.lib()
    rsgm_args, band_args = _abi_args(L, bad)
    assert L.vppb200_compute_rsgm_ex(*rsgm_args) == _lib.ERR_ARG
    assert L.vppb200_sgm_band_ex(*band_args) == _lib.ERR_ARG
    assert L.vppb200_sgm_params_fast(ctypes.byref(_params_struct(bad)), 0) == _lib.ERR_ARG


def test_sweep_domain_classification():
    """vppb200_sgm_params_fast: the domain of the sweeps (include/vppstereo_b200.h) at its edges"""
    from vppstereo_b200 import _lib
    L = _lib.lib()
    fast = lambda p, guided=0: L.vppb200_sgm_params_fast(ctypes.byref(_params_struct(p)), guided)
    assert L.vppb200_sgm_params_fast(None, 0) == 1 and L.vppb200_sgm_params_fast(None, 1) == 1
    for p in IN_DOMAIN:
        assert fast(p) == 1 and fast(p, 1) == 1, p
    for p in OUT_OF_DOMAIN:
        assert fast(p) == 0, p
    assert fast((3900, 3900, 0.0, 4071)) == 1 and fast((3900, 3900, 0.0, 4072)) == 0     # Cmax + P2max <= 4095, Hamming
    assert fast((3700, 3700, 0.0, 3855), 1) == 1 and fast((3700, 3700, 0.0, 3856), 1) == 0   # guided costs (<= 240)
    assert fast((0, 300, 5.0, 0)) == 0                  # P2max = P2min counts too


@pytest.mark.parametrize("bad", BAD)
def test_front_ends_raise_value_error(bad):
    """the Python front-ends validate before they touch the device (this test runs without one)"""
    from vppstereo_b200 import rsgm
    from vppstereo_b200.banded import BandedRsgm
    from vppstereo_b200.pipeline import VppRsgmPipeline
    img = np.zeros((16, 32, 3), np.uint8)
    p1, p2min, alpha, gamma = bad
    with pytest.raises(ValueError):
        rsgm.compute_rsgm(img, img, img, dmax=16, p1=p1, p2min=p2min, alpha=alpha, gamma=gamma, honor_params=True)
    with pytest.raises(ValueError):
        rsgm.compute_rsgm_stages(img, img, img, dmax=16, p1=p1, p2min=p2min, alpha=alpha, gamma=gamma, honor_params=True)
    with pytest.raises(ValueError):
        VppRsgmPipeline(16, 32, 3, batch=1, dmax=16, sgm_params=bad)
    with pytest.raises(ValueError):
        BandedRsgm(16, 32, 3, dmax=16, sgm_params=bad)


@pytest.mark.parametrize("prm", OUT_OF_DOMAIN)
def test_banded_refuses_out_of_domain(prm):
    from vppstereo_b200.banded import BandedRsgm
    with pytest.raises(ValueError):
        BandedRsgm(16, 32, 3, dmax=16, sgm_params=prm)


@pytest.mark.parametrize("shape,D,channels,sub,guided", [((37, 70), 32, 3, True, False), ((48, 64), 64, 1, True, True),
                                                         ((21, 50), 16, 3, False, True)])
def test_oracle_restatement_matches_oracle(orc, shape, D, channels, sub, guided):
    """oracle_rsgm at the reference's effective parameters is orc.compute_rsgm bit for bit (no device needed)"""
    from vppstereo_b200 import synth
    p = synth.make_pair(shape[0] + D, shape=shape, hints="random", channels=channels)
    kw = dict(hints=p["hints"], validhints=(p["hints"] > 0).astype(np.float32)) if guided else {}
    want = orc.compute_rsgm(p["left"], p["left"], p["right"], dmax=D, subpixel=sub, **kw)
    assert_same(oracle_rsgm(orc, p["left"], p["left"], p["right"], dmax=D, subpixel=sub, **kw), want, "restated oracle pipeline")


# ---------------------------------------------------------------- GPU
@pytest.fixture(scope="module")
def mods():
    import torch
    assert torch.cuda.is_available()
    from vppstereo_b200 import rsgm, synth, _lib
    _lib.lib()
    return rsgm, synth, _lib


@pytest.fixture
def tuning(mods):
    _lib = mods[2]
    yield lambda key, value: _lib.set_tuning(key, value)
    _lib.set_tuning(_lib.TUNE_SGM_MAX_STRIP, 0)
    _lib.set_tuning(_lib.TUNE_SGM_SWEEP, 1)


def _honoured(prm):
    return dict(p1=prm[0], p2min=prm[1], alpha=prm[2], gamma=prm[3], honor_params=True)


SHAPES = [((37, 70), 32, 3, True), ((48, 64), 64, 1, True), ((50, 121), 96, 3, False), ((33, 200), 192, 3, True)]


@pytest.mark.gpu
@pytest.mark.parametrize("prm", IN_DOMAIN)
@pytest.mark.parametrize("shape,D,channels,sub", SHAPES)
def test_compute_rsgm_params_vs_oracle(mods, orc, prm, shape, D, channels, sub):
    rsgm, synth = mods[0], mods[1]
    p = synth.make_pair(shape[0] + D, shape=shape, hints="random", channels=channels)
    want = oracle_rsgm(orc, p["left"], p["left"], p["right"], dmax=D, subpixel=sub, params=prm)
    got = rsgm.compute_rsgm(p["left"], p["left"], p["right"], dmax=D, subpixel=sub, **_honoured(prm))
    assert_same(got, want, f"compute_rsgm {prm} {shape} D={D} C={channels}")
    if prm == (7, 17, 0.25, 50):
        assert_same(got, rsgm.compute_rsgm(p["left"], p["left"], p["right"], dmax=D, subpixel=sub), "honoured defaults vs default call")


@pytest.mark.gpu
@pytest.mark.parametrize("sweep", [1, 0])
@pytest.mark.parametrize("prm", [(11, 17, 0.5, 35), (3, 30, 0.3, 80), (10, 10, 0.5, 265)])
def test_aggregated_volume_vs_oracle(mods, orc, tuning, prm, sweep):
    """the dsi_agg stage tap against the oracle's aggregate_SSE(honor_params=True) on the same census volume, with the sweeps and
    with the sweeps turned off (the per-path kernel)"""
    rsgm, synth, _lib = mods
    tuning(_lib.TUNE_SGM_SWEEP, sweep)
    p = synth.make_pair(17, shape=(45, 100), hints="random")
    st = rsgm.compute_rsgm_stages(p["left"], p["left"], p["right"], dmax=48, **_honoured(prm))
    assert_same(st["dsi_agg"][0], _oracle_agg(orc, p["left"], st, 48, prm), f"aggregated volume {prm} sweep={sweep}")


@pytest.mark.gpu
@pytest.mark.parametrize("prm", OUT_OF_DOMAIN)
def test_fallback_outside_domain_vs_oracle(mods, orc, prm):
    rsgm, synth = mods[0], mods[1]
    shape, D = (96, 192), 32
    p = synth.make_pair(3, shape=shape, hints="random", channels=1)
    st = rsgm.compute_rsgm_stages(p["left"], p["left"], p["right"], dmax=D, **_honoured(prm))
    want_S = _oracle_agg(orc, p["left"], st, D, prm)
    assert_same(st["dsi_agg"][0], want_S, f"aggregated volume {prm}")
    if prm[3] == 40000:
        assert (want_S == 65535).any(), "the case is meant to saturate S"
    want = oracle_rsgm(orc, p["left"], p["left"], p["right"], dmax=D, params=prm)
    assert_same(st["out"][0], want, f"compute_rsgm_stages {prm}")
    got = rsgm.compute_rsgm(p["left"], p["left"], p["right"], dmax=D, **_honoured(prm))
    assert_same(got, want, f"compute_rsgm {prm}")
    # guided costs (hints): the same fallback on the modulated volume
    v = (p["hints"] > 0).astype(np.float32)
    want = oracle_rsgm(orc, p["left"], p["left"], p["right"], hints=p["hints"], validhints=v, dmax=D, params=prm)
    got = rsgm.compute_rsgm(p["left"], p["left"], p["right"], hints=p["hints"], validhints=v, dmax=D, **_honoured(prm))
    assert_same(got, want, f"guided compute_rsgm {prm}")


def _kernel_names(fn):
    import torch
    from torch.profiler import ProfilerActivity, profile
    torch.cuda.synchronize()
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        fn()
        torch.cuda.synchronize()
    return {e.name for e in prof.events() if e.device_type == torch.autograd.DeviceType.CUDA}


@pytest.mark.gpu
def test_sweeps_run_for_in_domain_params(mods, tuning):
    """a silent fallback would pass every exactness test: the kernels that run are checked too"""
    rsgm, synth, _lib = mods
    p = synth.make_pair(9, shape=(40, 96), hints="random")
    run = lambda prm: rsgm.compute_rsgm(p["left"], p["left"], p["right"], dmax=32, **_honoured(prm))
    run((11, 17, 0.5, 35)); run((30, 10, 0.5, 20))                      # warm-up (module load, workspace)
    names = _kernel_names(lambda: run((11, 17, 0.5, 35)))
    assert any("sgm_v2_kernel" in n for n in names) and any("sgm_h_kernel" in n for n in names), sorted(names)
    assert not any("sgm_path_" in n for n in names), sorted(names)
    names = _kernel_names(lambda: run((30, 10, 0.5, 20)))
    assert any("sgm_path_generic_kernel" in n for n in names), sorted(names)
    assert not any("sgm_v2_kernel" in n or "sgm_h_kernel" in n for n in names), sorted(names)
    # in-domain parameters without the sweeps: the same per-path kernel as outside the domain
    tuning(_lib.TUNE_SGM_SWEEP, 0)
    names = _kernel_names(lambda: run((11, 17, 0.5, 35)))
    assert any("sgm_path_generic_kernel" in n for n in names), sorted(names)
    assert not any("sgm_path_fast" in n for n in names), sorted(names)


@pytest.mark.gpu
@pytest.mark.parametrize("strip", [32, 64, 96, 0])
def test_strips_and_guided(mods, orc, tuning, strip):
    """forced narrow strips (halo hand-off between CTAs; at 96 columns the team's last CTA holds a single column group) and
    guided costs (normalised state)"""
    rsgm, synth, _lib = mods
    tuning(_lib.TUNE_SGM_MAX_STRIP, strip)
    prm = (3, 30, 0.3, 80)
    frames = [synth.make_pair(300 + f, shape=(30, 200), hints="random") for f in range(2)]
    left = np.stack([q["left"] for q in frames]); right = np.stack([q["right"] for q in frames])
    hints = np.stack([q["hints"] for q in frames]); valid = (hints > 0).astype(np.float32)
    got = rsgm.compute_rsgm(left, left, right, dmax=64, **_honoured(prm))
    got_g = rsgm.compute_rsgm(left, left, right, hints=hints, validhints=valid, dmax=64, **_honoured(prm))
    for f, q in enumerate(frames):
        want = oracle_rsgm(orc, q["left"], q["left"], q["right"], dmax=64, params=prm)
        assert_same(got[f], want, f"strip={strip} frame {f}")
        want = oracle_rsgm(orc, q["left"], q["left"], q["right"], hints=q["hints"], validhints=valid[f], dmax=64, params=prm)
        assert_same(got_g[f], want, f"guided strip={strip} frame {f}")


@pytest.mark.gpu
def test_unnormalised_state_rule_follows_p2(mods, orc):
    """24 * H + 128 would keep the v-sweep state un-normalised at H = 2720; with P2max = 250 the rule switches to normalised"""
    rsgm, synth = mods[0], mods[1]
    prm = (7, 17, 0.25, 250)
    p = synth.make_pair(1, shape=(2720, 64), hints="random", channels=1)
    st = rsgm.compute_rsgm_stages(p["left"], p["left"], p["right"], dmax=16, **_honoured(prm))
    assert_same(st["dsi_agg"][0], _oracle_agg(orc, p["left"], st, 16, prm), "aggregated volume H=2720")
    want = oracle_rsgm(orc, p["left"], p["left"], p["right"], dmax=16, params=prm)
    assert_same(st["out"][0], want, "compute_rsgm H=2720")


@pytest.mark.gpu
def test_pipeline_sgm_params(mods):
    """VppRsgmPipeline(sgm_params=...): run_device (overlapped phases) and run_device_serial equal compute_rsgm(honor_params=True)
    on the pipeline's projected pair"""
    import torch
    from vppstereo_b200.pipeline import VppRsgmPipeline
    rsgm, synth = mods[0], mods[1]
    prm = (11, 17, 0.5, 35)
    frames = [synth.make_pair(80 + f, shape=(60, 140), hints="lidar") for f in range(6)]
    batches = [tuple(torch.from_numpy(np.stack([q[k] for q in frames[2 * b:2 * b + 2]])).cuda() for k in ("left", "right", "hints"))
               for b in range(3)]
    for serial in (False, True):
        pipe = VppRsgmPipeline(60, 140, 3, batch=2, dmax=64, seed=3, sgm_params=prm)
        for b in batches:
            out = (pipe.run_device_serial(*b) if serial else pipe.run_device(*b)).clone()
            torch.cuda.synchronize()
            want = rsgm.compute_rsgm(b[0], pipe.lv, pipe.rv, dmax=64, **_honoured(prm))
            assert_same(out.cpu().numpy(), want.cpu().numpy(), f"pipeline serial={serial}")
        dflt = VppRsgmPipeline(60, 140, 3, batch=2, dmax=64, seed=3)
        d = dflt.run_device_serial(*batches[0]).clone()
        assert_same(d.cpu().numpy(), rsgm.compute_rsgm(batches[0][0], dflt.lv, dflt.rv, dmax=64).cpu().numpy(), "default pipeline")
        pipe.close(); dflt.close()


@pytest.mark.gpu
@pytest.mark.parametrize("nb", [1, 2, 3])
def test_banded_sgm_params(mods, nb):
    from vppstereo_b200.banded import BandedRsgm
    rsgm, synth = mods[0], mods[1]
    prm = (3, 30, 0.3, 80)
    p = synth.make_pair(710 + nb, shape=(61, 200), hints="random")
    want = rsgm.compute_rsgm(p["left"], p["left"], p["right"], dmax=64, **_honoured(prm))
    got = BandedRsgm(61, 200, 3, dmax=64, n_bands=nb, sgm_params=prm).compute(p["left"], p["left"], p["right"])
    assert_same(got, want, f"{nb} bands, honoured parameters")
