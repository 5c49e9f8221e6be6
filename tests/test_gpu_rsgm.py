"""GPU parity tests of the rSGM hot path: CUDA kernels (through the C-ABI, via the reference-shaped Python front-ends)
against the CPU oracle on seeded inputs, against the committed golden vectors produced by the unmodified reference,
and -- at the benchmark's full size -- through size-independent properties.  Bar: bit-exact (integer / index work;
float32 disparities compared on their bit patterns)."""
import hashlib

import numpy as np
import pytest

from conftest import assert_same, golden_rsgm_names, load_golden_rsgm

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def mods():
    import torch
    assert torch.cuda.is_available()
    from vppstereo_b200 import pyrSGM, rsgm, synth, _lib
    _lib.lib()
    return pyrSGM, rsgm, synth, _lib


def _gray(rng, H, W):
    # smooth-ish texture with plateaus so that census ties and equal costs occur
    a = rng.integers(0, 256, (H // 4 + 2, W // 4 + 2)).astype(np.float32)
    a = np.kron(a, np.ones((4, 4), np.float32))[:H, :W]
    a += rng.integers(-6, 7, (H, W))
    return np.clip(a, 0, 255).astype(np.uint8)


SHAPES = [(8, 16), (24, 48), (40, 64), (37 + 11, 16 * 7), (64, 256), (100, 320)]


@pytest.mark.parametrize("H,W", SHAPES)
def test_census(mods, orc, H, W):
    pyrSGM = mods[0]
    rng = np.random.default_rng(H * 1000 + W)
    src = _gray(rng, H, W)
    want = np.zeros((H, W), np.uint32); orc.census5x5_SSE(src, want, W, H)
    got = np.full((H, W), 0xDEADBEEF, np.uint32); pyrSGM.census5x5_SSE(src, got, W, H)
    assert_same(got, want, f"census {H}x{W}")


@pytest.mark.parametrize("H,W,D", [(8, 16, 8), (24, 48, 16), (40, 64, 64), (30, 80, 72), (20, 272, 256), (16, 208, 192)])
def test_cost_volume(mods, orc, H, W, D):
    pyrSGM = mods[0]
    rng = np.random.default_rng(D)
    cl = rng.integers(0, 1 << 24, (H, W), dtype=np.uint32); cr = rng.integers(0, 1 << 24, (H, W), dtype=np.uint32)
    want = np.zeros((H, W, D), np.uint16); orc.costMeasureCensus5x5_xyd_SSE(cl, cr, want, W, H, D, 1)
    got = np.zeros((H, W, D), np.uint16); pyrSGM.costMeasureCensus5x5_xyd_SSE(cl, cr, got, W, H, D, 1)
    assert_same(got, want, "cost volume")


def _census_dsi(orc, rng, H, W, D):
    l, r = _gray(rng, H, W), _gray(rng, H, W)
    cl = np.zeros((H, W), np.uint32); cr = np.zeros((H, W), np.uint32)
    orc.census5x5_SSE(l, cl, W, H); orc.census5x5_SSE(r, cr, W, H)
    dsi = np.zeros((H, W, D), np.uint16); orc.costMeasureCensus5x5_xyd_SSE(cl, cr, dsi, W, H, D, 1)
    return l, dsi


@pytest.mark.parametrize("H,W,D", [(8, 16, 8), (12, 32, 16), (24, 48, 64), (21, 64, 72), (16, 80, 128), (12, 96, 192), (10, 48, 256)])
def test_aggregate_census_costs(mods, orc, H, W, D):
    """aggregate_SSE drop-in (generic saturating kernel) on census costs, gray and colour guide, args ignored."""
    pyrSGM = mods[0]
    rng = np.random.default_rng(7 * D + H)
    img, dsi = _census_dsi(orc, rng, H, W, D)
    want = np.zeros_like(dsi); orc.aggregate_SSE(img, dsi, want, W, H, D)
    got = np.zeros_like(dsi); pyrSGM.aggregate_SSE(img, dsi, got, W, H, D, 11, 17, 0.5, 35)   # rsgm.py:61 arguments: ignored
    assert_same(got, want, "aggregate (gray guide)")
    colour = rng.integers(0, 256, (H, W, 3), dtype=np.uint8)
    want = np.zeros_like(dsi); orc.aggregate_SSE(colour, dsi, want, W, H, D)
    got = np.zeros_like(dsi); pyrSGM.aggregate_SSE(colour, dsi, got, W, H, D, 11, 17, 0.5, 35)
    assert_same(got, want, "aggregate (colour guide: first W*H bytes)")


@pytest.mark.parametrize("scale", [1, 300, 9000])
def test_aggregate_saturation_and_params(mods, orc, scale):
    """arbitrary uint16 costs (saturation at 65535, uint16 wrap on pass 1's first row) and honoured parameters"""
    pyrSGM = mods[0]
    H, W, D = 9, 32, 24
    rng = np.random.default_rng(scale)
    img = rng.integers(0, 256, (H, W), dtype=np.uint8)
    dsi = (rng.integers(0, 8, (H, W, D)) * scale).astype(np.uint16)
    dsi[0, :4, :] = 255                       # the first-line 255 -> 12 rule (StereoSGM_SSE.hpp:120)
    want = np.zeros_like(dsi); orc.aggregate_SSE(img, dsi, want, W, H, D)
    got = np.zeros_like(dsi); pyrSGM.aggregate_SSE(img, dsi, got, W, H, D, 7, 17, 0.25, 50)
    assert_same(got, want, f"aggregate scale {scale}")
    want = np.zeros_like(dsi); orc.aggregate_SSE(img, dsi, want, W, H, D, 20, 24, 0.5, 70, honor_params=True)
    got = np.zeros_like(dsi); pyrSGM.aggregate_SSE(img, dsi, got, W, H, D, 20, 24, 0.5, 70, honor_params=True)
    assert_same(got, want, f"aggregate honoured params, scale {scale}")


@pytest.mark.parametrize("H,W,D", [(8, 16, 8), (10, 48, 16), (12, 64, 64), (9, 96, 72), (8, 224, 192), (8, 272, 256)])
def test_wta_subpixel_median(mods, orc, H, W, D):
    pyrSGM = mods[0]
    rng = np.random.default_rng(3 * D + W)
    S = rng.integers(0, 40, (H, W, D)).astype(np.uint16)        # many ties -> first arg-min matters
    S[rng.random((H, W, D)) < 0.02] = 0
    for name, f_ref, f_new in (("left", orc.matchWTA_SSE, pyrSGM.matchWTA_SSE), ("right", orc.matchWTARight_SSE, pyrSGM.matchWTARight_SSE)):
        want = np.zeros((H, W), np.float32); f_ref(S, want, W, H, D, 0.95)
        got = np.full((H, W), -1, np.float32); f_new(S, got, W, H, D, 0.95)
        assert_same(got, want, f"WTA {name}")
    wl = np.zeros((H, W), np.float32); orc.matchWTA_SSE(S, wl, W, H, D, 0.95)
    for method in (0, 1):
        want = wl.copy(); orc.subPixelRefine(S, want, W, H, D, method)
        got = wl.copy(); pyrSGM.subPixelRefine(S, got, W, H, D, method)
        assert_same(got, want, f"subPixelRefine method {method}")
    src = want
    want = np.zeros((H, W), np.float32); orc.median3x3_SSE(src, want, W, H)
    got = np.zeros((H, W), np.float32); pyrSGM.median3x3_SSE(src, got, W, H)
    assert_same(got, want, "median3x3")


def test_operator_errors(mods):
    pyrSGM = mods[0]
    a8 = np.zeros((8, 24), np.uint8); a32 = np.zeros((8, 24), np.uint32)
    with pytest.raises(TypeError):
        pyrSGM.census5x5_SSE(a8, a32, 24, 8)                      # width % 16
    ok32 = np.zeros((8, 32), np.uint32)
    with pytest.raises(TypeError):
        pyrSGM.costMeasureCensus5x5_xyd_SSE(ok32, ok32, np.zeros((8, 32, 12), np.uint16), 32, 8, 12, 1)   # D % 8
    with pytest.raises(TypeError):
        pyrSGM.costMeasureCensus5x5_xyd_SSE(ok32, ok32, np.zeros((8, 32, 8), np.uint16), 32, 8, 8, 3)     # threads
    with pytest.raises(TypeError):
        pyrSGM.matchWTA_SSE(np.zeros((8, 32, 8), np.uint16), np.zeros((8, 32), np.float32), 32, 8, 8, 1.5)
    with pytest.raises(TypeError):
        pyrSGM.subPixelRefine(np.zeros((8, 32, 8), np.uint16), np.zeros((8, 32), np.float32), 32, 8, 8, 2)


@pytest.mark.parametrize("name", golden_rsgm_names())
def test_golden_stages(mods, golden_lut, name):
    """every stage against the reference's recorded outputs (tests/golden/make_golden.py)"""
    pyrSGM, rsgm = mods[0], mods[1]
    g = load_golden_rsgm(name)
    D = int(g["D"])
    kw = {}
    if "hints" in g:
        kw = dict(hints=g["hints"], validhints=g["validhints"])
    st = rsgm.compute_rsgm_stages(g["left"], g["left_vpp"], g["right_vpp"], dmax=D, subpixel=True, rcp_lut=golden_lut, **kw)
    assert_same(st["census_l"][0], g["census_l"], "census L")
    assert_same(st["census_r"][0], g["census_r"], "census R")
    agg = st["dsi_agg"][0]
    Hp, Wp = g["census_l"].shape
    assert_same(agg[Hp // 2], g["agg_row"], "aggregated volume, middle row")
    assert hashlib.sha256(np.ascontiguousarray(agg).tobytes()).hexdigest() == str(g["agg_sha"]), "aggregated volume sha256"
    assert_same(st["disp_l"][0], g["disp_l"], "left disparity after median/interp/clip")
    assert_same(st["disp_r"][0], g["disp_r"], "right disparity after median/interp/clip")
    assert_same(st["out"][0], g["out_sub"], "compute_rsgm(subpixel=True)")
    out_int = rsgm.compute_rsgm(g["left"], g["left_vpp"], g["right_vpp"], dmax=D, subpixel=False, rcp_lut=golden_lut, **kw)
    assert_same(out_int, g["out_int"], "compute_rsgm(subpixel=False)")
    # stand-alone operators on the recorded aggregated volume
    got = np.zeros((Hp, Wp), np.float32); pyrSGM.matchWTA_SSE(agg, got, Wp, Hp, D, 0.95)
    assert_same(got, g["wta_l"], "matchWTA_SSE")
    sp = got.copy(); pyrSGM.subPixelRefine(agg, sp, Wp, Hp, D, 0, rcp_lut=golden_lut)
    assert_same(sp, g["subpix0"], "subPixelRefine(0)")
    sp1 = got.copy(); pyrSGM.subPixelRefine(agg, sp1, Wp, Hp, D, 1)
    assert_same(sp1, g["subpix1"], "subPixelRefine(1)")
    got = np.zeros((Hp, Wp), np.float32); pyrSGM.matchWTARight_SSE(agg, got, Wp, Hp, D, 0.95)
    assert_same(got, g["wta_r"], "matchWTARight_SSE")
    got = np.zeros((Hp, Wp), np.float32); pyrSGM.median3x3_SSE(g["subpix0"], got, Wp, Hp)
    assert_same(got, g["median"], "median3x3_SSE")


@pytest.mark.parametrize("shape,D,channels,sub", [((37, 70), 32, 3, True), ((48, 64), 64, 1, True), ((50, 121), 96, 3, False),
                                                  ((33, 200), 192, 3, True), ((20, 40), 8, 1, True)])
def test_compute_rsgm_vs_oracle(mods, orc, shape, D, channels, sub):
    rsgm, synth = mods[1], mods[2]
    p = synth.make_pair(shape[0] + D, shape=shape, hints="random", channels=channels)
    want = orc.compute_rsgm(p["left"], p["left"], p["right"], dmax=D, subpixel=sub)
    got = rsgm.compute_rsgm(p["left"], p["left"], p["right"], dmax=D, subpixel=sub)
    assert_same(got, want, f"compute_rsgm {shape} D={D} C={channels}")


@pytest.fixture
def tuning(mods):
    _lib = mods[3]
    yield lambda key, value: _lib.set_tuning(key, value)
    _lib.set_tuning(_lib.TUNE_SGM_MAX_STRIP, 0)
    _lib.set_tuning(_lib.TUNE_SGM_SWEEP, 1)


@pytest.mark.parametrize("strip", [32, 64, 100])
@pytest.mark.parametrize("shape,D,channels", [((37, 70), 32, 3), ((40, 120), 64, 1), ((33, 200), 192, 3), ((30, 100), 72, 3),
                                              ((24, 90), 256, 1), ((20, 150), 8, 1), ((26, 330), 16, 3)])
def test_sweep_cluster_strips(mods, orc, tuning, strip, shape, D, channels):
    """the cluster sweep with forced narrow strips (multi-CTA clusters, DSMEM halo exchange of the diagonal paths,
    ring wrap-around) against the oracle, stage tap of the aggregated volume included"""
    rsgm, synth, _lib = mods[1], mods[2], mods[3]
    tuning(_lib.TUNE_SGM_MAX_STRIP, strip)
    frames = [synth.make_pair(shape[0] + D + f, shape=shape, hints="random", channels=channels) for f in range(3)]
    left = np.stack([p["left"] for p in frames]); right = np.stack([p["right"] for p in frames])
    st = rsgm.compute_rsgm_stages(left, left, right, dmax=D)
    for f, p in enumerate(frames):
        want = orc.compute_rsgm(p["left"], p["left"], p["right"], dmax=D)
        assert_same(st["out"][f], want, f"sweep strip={strip} {shape} D={D} frame {f}")
    # the production path (last sweep fused with WTA, the final S never written)
    fused16 = rsgm.compute_rsgm(left, left, right, dmax=D)
    assert_same(fused16, st["out"], f"fused sweep, strip={strip}")
    # the aggregated volume itself, against the stand-alone operator (generic per-path kernel) on the same inputs
    tuning(_lib.TUNE_SGM_SWEEP, 0)
    st0 = rsgm.compute_rsgm_stages(left, left, right, dmax=D)
    assert_same(st["dsi_agg"], st0["dsi_agg"], f"aggregated volume, sweep strip={strip} vs per-path kernels")
    assert_same(st["out"], st0["out"], "sweep vs per-path kernels, final disparity")


def _kernels(fn):
    """names of the kernels fn() launches, one entry per launch"""
    import torch
    from torch.profiler import ProfilerActivity, profile
    torch.cuda.synchronize()
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        fn()
        torch.cuda.synchronize()
    return [e.name for e in prof.events() if e.device_type == torch.autograd.DeviceType.CUDA]


@pytest.mark.parametrize("shape,channels", [((37, 70), 3), ((5, 17), 1), ((64, 333), 3), ((23, 1242), 3), ((130, 64), 1)])
def test_census_fused_front(mods, orc, shape, channels):
    """pad + gray + census as one kernel per image (bulk-copied source window, gray band in shared memory) against the two-kernel
    front and the oracle; frames 1.. of a batch start at addresses that are not 16-byte aligned.  The two-kernel front is what
    runs when the batch itself does not start on a 16-byte boundary: the same batch from such a source is the reference."""
    import torch
    rsgm, synth = mods[1], mods[2]
    D = 32 if shape[1] >= 64 else 8
    frames = [synth.make_pair(900 + f, shape=shape, hints="random", channels=channels) for f in range(3)]
    left = np.stack([p["left"] for p in frames]); right = np.stack([p["right"] for p in frames])

    def misaligned(a):                              # the same bytes on the device, starting one byte past an aligned address
        buf = torch.empty(a.size + 1, dtype=torch.uint8, device="cuda")
        buf[1:].copy_(torch.from_numpy(a).reshape(-1))
        view = buf[1:].view(a.shape)
        assert view.data_ptr() % 16 == 1
        return view
    left_m, right_m = misaligned(left), misaligned(right)
    got = rsgm.compute_rsgm(left, left, right, dmax=D)
    two = rsgm.compute_rsgm(left_m, left_m, right_m, dmax=D).cpu().numpy()
    assert_same(got, two, f"fused front vs pad_gray + census {shape} C={channels}")
    names = _kernels(lambda: rsgm.compute_rsgm(left, left, right, dmax=D))
    assert any("census_fused_kernel" in n for n in names) and not any("census5x5_kernel" in n for n in names), sorted(names)
    names = _kernels(lambda: rsgm.compute_rsgm(left_m, left_m, right_m, dmax=D))
    assert any("census5x5_kernel" in n for n in names) and not any("census_fused_kernel" in n for n in names), sorted(names)
    for f in (0, 2):
        want = orc.compute_rsgm(frames[f]["left"], frames[f]["left"], frames[f]["right"], dmax=D)
        assert_same(got[f], want, f"fused front {shape} C={channels} frame {f}")


def test_sweep_split_launches(mods, orc):
    """a batch that does not fill its last round of teams is swept in two launches with different strip widths (plan_v_split):
    same result as the same frames swept one per call (a single frame never splits), and as the oracle on the frames either
    side of the split.  On 148 SMs these 80 frames go as 37 frames on 2-group strips + 43 frames on 3-group strips."""
    rsgm, synth = mods[1], mods[2]
    shape, D, n = (24, 200), 16, 80
    frames = [synth.make_pair(500 + f, shape=shape, hints="random", channels=1) for f in range(n)]
    left = np.stack([p["left"] for p in frames]); right = np.stack([p["right"] for p in frames])
    got = rsgm.compute_rsgm(left, left, right, dmax=D)
    single = np.stack([rsgm.compute_rsgm(left[f], left[f], right[f], dmax=D) for f in range(n)])
    assert_same(got, single, "split sweep vs one frame per call")
    # two v-sweeps per plan: four launches when the batch splits, two for one frame
    count = lambda fn: sum(1 for e in _kernels(fn) if "sgm_v2_kernel" in e)
    assert count(lambda: rsgm.compute_rsgm(left, left, right, dmax=D)) == 4
    assert count(lambda: rsgm.compute_rsgm(left[0], left[0], right[0], dmax=D)) == 2
    for f in (0, 36, 37, 79):
        want = orc.compute_rsgm(frames[f]["left"], frames[f]["left"], frames[f]["right"], dmax=D)
        assert_same(got[f], want, f"split sweep frame {f}")


def test_compute_rsgm_random_shapes(mods, orc):
    """Seeded random sweep over frame shapes (any H >= 5, W >= 17: padded to multiples of 16, often not of 32), disparity ranges
    (multiples of 8 up to 256), gray / colour, guided or not, sub-pixel on / off, batches of 1-3: bit-exact against the oracle."""
    rsgm, synth = mods[1], mods[2]
    rng = np.random.default_rng(4242)
    for case in range(48):
        H, W = int(rng.integers(5, 80)), int(rng.integers(17, 300))
        D = int(rng.integers(1, 33)) * 8
        ch = int(rng.choice([1, 3])); sub = bool(rng.integers(2)); guided = rng.integers(4) == 0; nb = int(rng.integers(1, 4))
        frames = [synth.make_pair(int(rng.integers(10000)), shape=(H, W), hints="random", channels=ch, density=0.1) for _ in range(nb)]
        left = np.stack([p["left"] for p in frames]); right = np.stack([p["right"] for p in frames])
        hints = np.stack([p["hints"] for p in frames]) if guided else None
        valid = (hints > 0).astype(np.float32) if guided else None
        got = rsgm.compute_rsgm(left, left, right, hints=hints, validhints=valid, dmax=D, subpixel=sub)
        for f, p in enumerate(frames):
            want = orc.compute_rsgm(p["left"], p["left"], p["right"], hints=None if not guided else p["hints"],
                                    validhints=None if not guided else (p["hints"] > 0).astype(np.float32), dmax=D, subpixel=sub)
            assert_same(got[f], want, f"case {case}: {H}x{W} D={D} C={ch} sub={sub} guided={guided} frame {f}/{nb}")


def test_compute_rsgm_guided_and_batch(mods, orc):
    rsgm, synth = mods[1], mods[2]
    frames = [synth.make_pair(f, shape=(45, 100), hints="random") for f in range(3)]
    want = [orc.compute_rsgm(p["left"], p["left"], p["right"], hints=p["hints"], validhints=(p["hints"] > 0).astype(np.float32),
                             dmax=64) for p in frames]
    left = np.stack([p["left"] for p in frames]); right = np.stack([p["right"] for p in frames])
    hints = np.stack([p["hints"] for p in frames])
    got = rsgm.compute_rsgm(left, left, right, hints=hints, validhints=(hints > 0).astype(np.float32), dmax=64)
    assert got.shape == (3, 45, 100)
    for f in range(3):
        assert_same(got[f], want[f], f"guided batch frame {f}")


def test_compute_rsgm_device_tensors(mods, orc):
    """CUDA tensors in -> CUDA tensor out, no host round-trip, same numbers"""
    import torch
    rsgm, synth = mods[1], mods[2]
    p = synth.make_pair(5, shape=(40, 90), hints="random")
    want = orc.compute_rsgm(p["left"], p["left"], p["right"], dmax=48)
    l, r = torch.from_numpy(p["left"]).cuda(), torch.from_numpy(p["right"]).cuda()
    got = rsgm.compute_rsgm(l, l, r, dmax=48)
    assert got.is_cuda and got.dtype == torch.float32
    assert_same(got.cpu().numpy(), want, "device-tensor compute_rsgm")


def test_kitti_shape_properties(mods, orc):
    """BASELINE config 2 shape (1242x375, D=192): one frame against the oracle, then batch properties:
    a frame's result does not depend on its batch neighbours, and the run is deterministic."""
    rsgm, synth = mods[1], mods[2]
    frames = [synth.make_pair(f, shape="K", hints="lidar") for f in range(4)]
    want0 = orc.compute_rsgm(frames[0]["left"], frames[0]["left"], frames[0]["right"], dmax=192)
    left = np.stack([p["left"] for p in frames]); right = np.stack([p["right"] for p in frames])
    got = rsgm.compute_rsgm(left, left, right, dmax=192)
    assert_same(got[0], want0, "K-shape frame 0 vs oracle")
    again = rsgm.compute_rsgm(left[::-1].copy(), left[::-1].copy(), right[::-1].copy(), dmax=192)
    assert_same(again[::-1], got, "batch order independence / determinism")
    # sanity: away from the left band where x < d the matcher recovers the synthetic ground truth
    gt = frames[0]["gt"]
    xs = np.arange(gt.shape[1])[None, :]
    sel = (xs > gt + 16) & (got[0] > 0)
    assert np.median(np.abs(got[0] - gt)[sel]) < 4.0    # the synthetic right view is warped with d(u), not d(x)


def test_middlebury_shape_vs_oracle(mods, orc):
    """Full-resolution Middlebury shape (2880x1988 -> padded 2880x2000, D=192; SURVEY.md 8 sizes 'M'): VPP-projected pair
    through compute_rsgm on device tensors, bit-exact against the oracle.  The frame spans an 18-CTA team in the sweeps."""
    import torch
    from vppstereo_b200 import vpp_standalone
    rsgm, synth = mods[1], mods[2]
    p = synth.make_pair(2, shape="M", hints="random")
    pattern = np.random.default_rng(2).integers(0, 256, orc.stream_length(p["hints"], 3, 3, 0), dtype=np.uint8)
    L, R, G = (torch.from_numpy(p[k]).cuda() for k in ("left", "right", "hints"))
    lv, rv = vpp_standalone.vpp(L, R, G, pattern=pattern)
    got = rsgm.compute_rsgm(L, lv, rv, dmax=192)
    lw, rw = orc.vpp(p["left"], p["right"], p["hints"], stream=pattern, mode=1)
    assert_same(lv.cpu().numpy(), lw, "VPP left"); assert_same(rv.cpu().numpy(), rw, "VPP right")
    want = orc.compute_rsgm(p["left"], lw, rw, dmax=192)
    assert_same(got.cpu().numpy(), want, "M-shape compute_rsgm")


def test_pipeline_streaming_matches_synchronous(mods):
    """VppRsgmPipeline.submit_host/collect (copies overlapped on their own streams, up to host_depth = 3 batches in flight)
    returns what the synchronous run_host returns for the same batches and pattern seeds."""
    import torch
    from vppstereo_b200.pipeline import VppRsgmPipeline
    synth = mods[2]
    frames = [synth.make_pair(40 + f, shape=(60, 140), hints="lidar") for f in range(10)]
    batches = []
    for b in range(5):
        fr = frames[2 * b:2 * b + 2]
        batches.append(tuple(torch.from_numpy(np.stack([p[k] for p in fr])).pin_memory() for k in ("left", "right", "hints")))
    sync_pipe = VppRsgmPipeline(60, 140, 3, batch=2, dmax=64, seed=5)
    want = [sync_pipe.run_host(*b).clone().numpy() for b in batches]
    pipe = VppRsgmPipeline(60, 140, 3, batch=2, dmax=64, seed=5)
    got, pending = [], []
    for b in batches:
        pending.append(pipe.submit_host(*b))
        if len(pending) == pipe.host_depth:
            got.append(pipe.collect(pending.pop(0)).clone().numpy())
    with pytest.raises(RuntimeError):
        pipe.collect(pending[0] - 1 if pending[0] > 0 else pipe.host_depth - 1)       # already collected
    while pending:
        got.append(pipe.collect(pending.pop(0)).clone().numpy())
    for k in range(5):
        assert_same(got[k], want[k], f"streamed batch {k}")
    with pytest.raises(RuntimeError):
        pipe.collect(0)
    tickets = [pipe.submit_host(*batches[0]) for _ in range(pipe.host_depth)]
    with pytest.raises(RuntimeError):
        pipe.submit_host(*batches[0])                  # a fourth batch needs a collect first
    for tk in tickets:                                 # nothing stays in flight when the pipeline is dropped
        assert pipe.collect(tk).shape == (2, 60, 140)
    pipe.close()


def test_pipeline_phases_overlapped_match_serial_and_oracle(mods, orc):
    """run_device queues front / main / tail of consecutive calls on three streams with two buffer sets; every call must
    return what the in-order run_device_serial returns, and (pattern passed through the device generator, so VPP is checked
    separately) compute_rsgm of the projected pair must equal the oracle's."""
    import torch
    from vppstereo_b200.pipeline import VppRsgmPipeline
    synth = mods[2]
    frames = [synth.make_pair(70 + f, shape=(72, 160), hints="lidar") for f in range(10)]
    batches = []
    for b in range(5):
        fr = frames[2 * b:2 * b + 2]
        batches.append(tuple(torch.from_numpy(np.stack([p[k] for p in fr])).cuda() for k in ("left", "right", "hints")))
    serial = VppRsgmPipeline(72, 160, 3, batch=2, dmax=64, seed=9)
    want, proj = [], []
    for b in batches:
        want.append(serial.run_device_serial(*b).clone())
        proj.append((serial.lv.clone(), serial.rv.clone()))
    # (dirty the allocator's free blocks first: the pipeline's zero-initialised occlusion mask must be complete before its own
    # streams run the first front phase -- regression test for a constructor / first-call ordering bug)
    junk = torch.full((96 << 20,), 255, dtype=torch.uint8, device="cuda"); torch.cuda.synchronize(); del junk
    pipe = VppRsgmPipeline(72, 160, 3, batch=2, dmax=64, seed=9)
    outs = [torch.empty((2, 72, 160), dtype=torch.float32, device="cuda") for _ in batches]
    for b, o in zip(batches, outs):                    # back to back: phases of neighbouring calls overlap
        pipe.run_device(*b, out=o, inputs_ready=True)
    torch.cuda.synchronize()
    for k in range(5):
        assert_same(outs[k].cpu().numpy(), want[k].cpu().numpy(), f"overlapped call {k}")
    # default output buffer + in-order semantics on the caller's stream
    got = [pipe.run_device(*b).clone() for b in batches[:3]]
    torch.cuda.synchronize()
    pipe2 = VppRsgmPipeline(72, 160, 3, batch=2, dmax=64, seed=9)
    for k in range(5):
        pipe2.run_device_serial(*batches[k])
    for k in range(3):
        w = pipe2.run_device_serial(*batches[k]).clone()
        assert_same(got[k].cpu().numpy(), w.cpu().numpy(), f"in-order call {k}")
    # the matcher half against the oracle on the projected pair of the last serial call
    lv, rv = proj[-1]
    for i in range(2):
        ref = orc.compute_rsgm(batches[-1][0][i].cpu().numpy(), lv[i].cpu().numpy(), rv[i].cpu().numpy(), dmax=64)
        assert_same(want[-1][i].cpu().numpy(), ref, f"serial call vs oracle, frame {i}")
