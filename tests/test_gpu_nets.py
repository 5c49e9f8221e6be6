"""BASELINE configs[3]: the projected pair goes to RAFT-Stereo / PSMNet as DEVICE tensors (test.py:179-231).  The networks are the
reference's own classes (byte-compiled under oracle/_ref/refmodels, random weights: no checkpoints offline); they are consumers of
the path, not part of it.  Checked: (a) the device hand-off (vpp on CUDA tensors -> vpp_to_network) gives the networks exactly the
tensors the reference flow builds on the host (numpy /255., permute, .cuda(), replicate pad), so with identical weights the
network outputs agree to float tolerance; (b) the sweeps' cooperative grid survives a network (a convolutional stack defined
here, so that this check runs everywhere) running beside it on another stream; (c) sample_hints equals losses.py:5-10 under the
same CUDA generator state (SURVEY 8 f-4)."""
import os

import numpy as np
import pytest

from conftest import ROOT, assert_same

pytestmark = pytest.mark.gpu

HAVE_NETS = os.path.isdir(os.path.join(ROOT, "oracle", "_ref", "refmodels"))


@pytest.fixture(scope="module")
def nets():
    import torch
    if not HAVE_NETS:
        pytest.skip("oracle/_ref/refmodels not built (python oracle/build_ref.py where /root/reference exists)")
    from oracle import ref
    RAFT, PSM = ref.load_nets()
    torch.manual_seed(7)
    raft = RAFT(None).cuda().eval()
    psm = PSM(192).cuda().eval()
    return raft, psm


def _reference_feed(img_u8_hwc, ht, wt):
    """test.py:179-197: torch.from_numpy(x/255.).permute(2,0,1).unsqueeze(0).float() -> .cuda() -> F.pad(replicate) to /32"""
    import torch
    import torch.nn.functional as F
    t = torch.from_numpy(img_u8_hwc / 255.).permute(2, 0, 1).unsqueeze(0).float().cuda()
    pad_ht = (((ht // 32) + 1) * 32 - ht) % 32
    pad_wd = (((wt // 32) + 1) * 32 - wt) % 32
    _pad = [pad_wd // 2, pad_wd - pad_wd // 2, pad_ht // 2, pad_ht - pad_ht // 2]
    return F.pad(t, _pad, mode="replicate"), _pad


def _handoff_inputs(orc, shape):
    """The three network inputs of one frame, built both ways: (device flow, reference flow) as (im2, im2_vpp, im3_vpp) tuples."""
    import torch
    from vppstereo_b200 import synth, vpp_standalone, vpp_core_opt
    H, W = shape
    p = synth.make_pair(11, shape=shape, hints="lidar")
    n = int(vpp_core_opt.draws_per_frame(p["hints"], 3, 3, False).sum())
    pattern = np.random.default_rng(3).integers(0, 256, n, dtype=np.uint8)
    # reference flow: host VPP (the oracle in numba arithmetic = vpp_standalone.vpp), numpy images -> tensors -> GPU
    lw, rw = orc.vpp(p["left"], p["right"], p["hints"], stream=pattern, mode=1)
    ref2, _pad = _reference_feed(lw, H, W)
    ref3, _ = _reference_feed(rw, H, W)
    ref0, _ = _reference_feed(p["left"], H, W)
    # device flow: nothing leaves the GPU between the projection and the network
    L, R, G = (torch.from_numpy(p[k]).cuda() for k in ("left", "right", "hints"))
    lv, rv = vpp_standalone.vpp(L, R, G, pattern=pattern)
    dev2, pad = vpp_standalone.vpp_to_network(lv)
    dev3, _ = vpp_standalone.vpp_to_network(rv)
    dev0, _ = vpp_standalone.vpp_to_network(L)
    assert list(pad) == _pad
    for a, b, what in ((dev2, ref2, "im2_vpp"), (dev3, ref3, "im3_vpp"), (dev0, ref0, "im2")):
        assert_same(a.cpu().numpy(), b.cpu().numpy(), f"network input {what}")
    return (dev0, dev2, dev3), (ref0, ref2, ref3)


@pytest.mark.parametrize("shape", [(256, 330), (375, 1242)])
def test_network_inputs_device_handoff_equal_reference_feed(orc, shape):
    """(a) without the networks: the padding and the three tensors handed to them are bit-identical between the two flows."""
    _handoff_inputs(orc, shape)


@pytest.mark.parametrize("shape", [(256, 330), (375, 1242)])      # (PSMNet's 64x64 pooling branch needs >= 256 rows)
def test_nets_device_handoff_vs_reference_flow(nets, orc, shape):
    import torch
    raft, psm = nets
    H, W = shape
    (dev0, dev2, dev3), (ref0, ref2, ref3) = _handoff_inputs(orc, shape)
    with torch.no_grad():
        iters = 8 if H > 300 else 12
        _, d_dev = raft(dev0, dev2, dev3, test_mode=True, iters=iters)
        _, d_ref = raft(ref0, ref2, ref3, test_mode=True, iters=iters)
        assert torch.isfinite(d_dev).all()
        assert torch.allclose(d_dev, d_ref, rtol=1e-4, atol=1e-3), float((d_dev - d_ref).abs().max())
        if H <= 300:                                  # PSMNet's 3-D cost volume at K size is a bench matter, not a parity one
            o_dev = psm(im2=dev2, im3=dev3)[0]
            o_ref = psm(im2=ref2, im3=ref3)[0]
            assert torch.isfinite(o_dev).all()
            assert torch.allclose(o_dev, o_ref, rtol=1e-4, atol=1e-3), float((o_dev - o_ref).abs().max())


def _side_network():
    """A convolutional network (random weights) to run on another stream: it needs nothing outside this repository."""
    import torch
    torch.manual_seed(7)
    layers, ch = [], 3
    for c in (64, 128, 128, 256, 256, 128):
        layers += [torch.nn.Conv2d(ch, c, 3, padding=1), torch.nn.BatchNorm2d(c), torch.nn.ReLU()]
        ch = c
    return torch.nn.Sequential(*layers).cuda().eval()


def test_sweeps_beside_a_running_network(orc):
    """The v-sweep is a cooperative grid whose CTAs wait for each other; a network running on another stream takes SMs, registers
    and shared memory at the same time.  The result must stay bit-exact and no hand-off may time out (vppb200_async_error)."""
    import torch
    from vppstereo_b200 import synth, _lib
    from vppstereo_b200.pipeline import VppRsgmPipeline
    net = _side_network()
    B, H, W, D = 8, 120, 420, 64
    fr = [synth.make_pair(300 + i, shape=(H, W), hints="lidar") for i in range(B)]
    L, R, G = (torch.from_numpy(np.stack([f[k] for f in fr])).cuda() for k in ("left", "right", "hints"))
    pipe = VppRsgmPipeline(H, W, 3, batch=B, dmax=D, seed=3)
    want = pipe.run_device_serial(L, R, G, step=1).clone()
    torch.cuda.synchronize()
    x = torch.rand(2, 3, 256, 512, device="cuda")
    side = torch.cuda.Stream()
    outs = []
    with torch.no_grad():
        for rep in range(6):
            with torch.cuda.stream(side):
                for _ in range(2):
                    net(x)
            outs.append(pipe.run_device(L, R, G, out=torch.empty_like(want), inputs_ready=True, step=1))
    torch.cuda.synchronize()
    pipe.check()                                      # raises if a hand-off wait timed out
    for k, o in enumerate(outs):
        assert_same(o.cpu().numpy(), want.cpu().numpy(), f"call {k} beside the network")
    # against the oracle too (frame 0)
    from vppstereo_b200 import vpp_core_opt
    pat = vpp_core_opt.device_pattern(pipe.pattern_seed(1), 0, orc.stream_length(fr[0]["hints"], 3, 3, False))
    lw, rw = orc.vpp(fr[0]["left"], fr[0]["right"], fr[0]["hints"], stream=pat, mode=1)
    assert_same(want[0].cpu().numpy(), orc.compute_rsgm(fr[0]["left"], lw, rw, dmax=D), "frame 0 vs oracle")
    pipe.close()


def test_sample_hints_equals_reference():
    """losses.py:5-10: same CUDA generator state => the same random mask, the same sampled hints"""
    import torch
    if not os.path.exists(os.path.join(ROOT, "oracle", "_ref", "losses_ref.pycode")):
        pytest.skip("oracle/_ref/losses_ref.pycode not built")
    from oracle import ref
    from vppstereo_b200 import vpp_standalone
    losses = ref.load_losses()
    g = torch.Generator(device="cuda").manual_seed(5)
    hints = torch.rand(2, 1, 375, 1242, device="cuda", generator=g) * 190
    valid = (torch.rand(2, 1, 375, 1242, device="cuda", generator=g) < 0.3).float()
    for prob in (0.2, 0.05, 1.0):
        torch.manual_seed(1234)
        want_h, want_v = losses.sample_hints(hints.clone(), valid.clone(), prob)
        torch.manual_seed(1234)
        got_h, got_v = vpp_standalone.sample_hints(hints.clone(), valid.clone(), prob)
        assert_same(got_v.cpu().numpy(), want_v.cpu().numpy(), f"validhints p={prob}")
        assert_same(got_h.cpu().numpy(), want_h.cpu().numpy(), f"hints p={prob}")
