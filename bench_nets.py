"""bench.py --workload nets: BASELINE configs[3] -- "VPP output fed as device tensors to RAFT-Stereo and PSMNet (random-init) at
1242x375, end-to-end pairs/s".

Per frame (test.py runs batch 1, test.py:158-231): hints + pair -> virtual pattern projection -> network -> disparity on the host.
  device flow (this repo):  pinned host frame -> H2D -> vpp() on CUDA tensors -> vpp_to_network (uint8 HWC -> float32 CHW / 255, replicate
                            pad to /32, one kernel) -> network -> D2H of the disparity.  Nothing returns to the host in between.
  reference flow:           the reference's own vpp() (numba, one host core: oracle/_ref/vpp_standalone_ref) -> numpy / 255. ->
                            torch -> .cuda() -> F.pad -> the same network -> D2H  (test.py:158-197 as written).
The networks are the reference's own classes with random weights (consumers, not part of the rebuilt path); RAFT-Stereo runs the
32 iterations of test.py:226, PSMNet maxdisp 192.  One JSON line; `value` = device flow through RAFT-Stereo with the frame already
in HBM, `e2e` = the same from pinned host memory; the other three combinations and both reference-flow figures are in `config`.
--impl reference prints the reference flow as its own line."""
import json
import os
import sys
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
H, W, C, D = 375, 1242, 3, 192
METRIC = "VPP -> RAFT-Stereo / PSMNet end-to-end pairs/s @1242x375, 5% hints (device tensors, random-init nets)"


def _nets(dev):
    import torch
    from oracle import ref                         # the reference's network classes: the consumer side, test infrastructure
    RAFT, PSM = ref.load_nets()
    torch.manual_seed(0)
    return {"raft-stereo": RAFT(None).to(dev).eval(), "psmnet": PSM(D).to(dev).eval()}


def _forward(name, net, im0, im2, im3):
    if name == "raft-stereo":
        return -net(im0, im2, im3, test_mode=True, iters=32)[1].squeeze(1)       # test.py:226-236
    return net(im2=im2, im3=im3)[0]


def main(args, reference=False):
    import numpy as np
    import torch
    import torch.nn.functional as F
    from vppstereo_b200 import synth, vpp_standalone
    import bench
    torch.cuda.set_device(0)
    dev = torch.device("cuda", 0)
    steps = args.steps if args.steps is not None else 30
    frames = [synth.make_pair(f, shape="K", hints="lidar") for f in range(4)]
    pinned = [tuple(torch.from_numpy(p[k]).pin_memory() for k in ("left", "right", "hints")) for p in frames]
    resident = [tuple(t.to(dev) for t in fr) for fr in pinned]
    nets = _nets(dev)
    out_h = torch.empty((1, H, W), dtype=torch.float32).pin_memory()

    def crop(d, pad):
        ht, wd = d.shape[-2:]
        return d[..., pad[2]:ht - pad[3], pad[0]:wd - pad[1]]

    def device_flow(name, k, from_host):
        l, r, g = pinned[k % 4] if from_host else resident[k % 4]
        if from_host:
            l, r, g = l.to(dev, non_blocking=True), r.to(dev, non_blocking=True), g.to(dev, non_blocking=True)
        lv, rv = vpp_standalone.vpp(l, r, g, wsize=3, blending=0.4, method="rnd", seed=k)
        im2, pad = vpp_standalone.vpp_to_network(lv)
        im3, _ = vpp_standalone.vpp_to_network(rv)
        im0, _ = vpp_standalone.vpp_to_network(l)
        d = crop(_forward(name, nets[name], im0, im2, im3), pad)
        if from_host:
            out_h.copy_(d.reshape(1, H, W), non_blocking=True)
        return d

    refns = None

    def reference_flow(name, k):
        l, r, g = (frames[k % 4][key] for key in ("left", "right", "hints"))
        lb, rb = refns.vpp_standalone.vpp(l, r, g, blending=0.4, wsize=3, method="rnd")           # host, numba (test.py:158)
        im2 = torch.from_numpy(lb / 255.).permute(2, 0, 1).unsqueeze(0).float().cuda()             # test.py:179-184
        im3 = torch.from_numpy(rb / 255.).permute(2, 0, 1).unsqueeze(0).float().cuda()
        im0 = torch.from_numpy(l / 255.).permute(2, 0, 1).unsqueeze(0).float().cuda()
        pad_ht, pad_wd = (((H // 32) + 1) * 32 - H) % 32, (((W // 32) + 1) * 32 - W) % 32
        pad = [pad_wd // 2, pad_wd - pad_wd // 2, pad_ht // 2, pad_ht - pad_ht // 2]
        im0, im2, im3 = (F.pad(t, pad, mode="replicate") for t in (im0, im2, im3))
        return crop(_forward(name, nets[name], im0, im2, im3), pad).cpu()

    def timed(fn, n):
        torch.cuda.synchronize(dev)
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        t0 = time.perf_counter()
        e0.record()
        for k in range(n):
            fn(k)
        e1.record()
        torch.cuda.synchronize(dev)
        return max(e0.elapsed_time(e1) * 1e-3, 0.0), time.perf_counter() - t0

    res = {}
    with torch.no_grad():
        if reference:
            from oracle import ref
            refns = ref.load()
            for name in nets:
                reference_flow(name, 0)
                _, wall = timed(lambda k: reference_flow(name, k), max(steps // 2, 3))
                res[name] = max(steps // 2, 3) / wall
            line = {"impl": "reference", "metric": METRIC, "value": res["raft-stereo"], "unit": "pairs/s", "n_gpus": 1, "steps": max(steps // 2, 3),
                    "warmup": 1, "ms_per_step": 1e3 / res["raft-stereo"], "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
                    "dtype": "f32", "data": "synthetic",
                    "config": {"workload": "configs[3]: reference flow (numba vpp on one host core, host round trip) -> the same random-init networks on the GPU",
                               "pairs_per_s": res},
                    "cpu_baseline": {"value": res["raft-stereo"], "unit": "pairs/s", "cores": 1, "kind": "reference",
                                     "sample": "numba vpp() of the reference on one host core per frame + network on the GPU"},
                    "e2e": {"value": res["raft-stereo"], "unit": "pairs/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
            print(json.dumps(line), flush=True)
            return
        launches0 = __import__("vppstereo_b200._lib", fromlist=["x"]).launch_count()
        for name in nets:
            for from_host in (False, True):
                for k in range(3):
                    device_flow(name, k, from_host)
                dev_s, wall = timed(lambda k: device_flow(name, k, from_host), steps)
                res[(name, from_host)] = (steps / dev_s, steps / wall)
        # the projection + hand-off alone (what this repo contributes to the flow), per frame
        def vpp_only(k):
            l, r, g = resident[k % 4]
            lv, rv = vpp_standalone.vpp(l, r, g, wsize=3, blending=0.4, method="rnd", seed=k)
            vpp_standalone.vpp_to_network(lv); vpp_standalone.vpp_to_network(rv); vpp_standalone.vpp_to_network(l)
        vpp_only(0)
        vpp_s, _ = timed(vpp_only, 50)
        launches = __import__("vppstereo_b200._lib", fromlist=["x"]).launch_count() - launches0
        ref_res = None
        try:
            from oracle import ref
            refns = ref.load()
            ref_res = {}
            for name in nets:
                reference_flow(name, 0)
                n = 5
                _, wall = timed(lambda k: reference_flow(name, k), n)
                ref_res[name] = n / wall
        except Exception as e:
            ref_res = {"unavailable": repr(e)}
    v, e = res[("raft-stereo", False)][0], res[("raft-stereo", True)][1]
    peak, peak_src = bench.measured_peak()
    vpp_bytes = 4 * H * W * C + 4 * H * W + H * W + 3 * 4 * 3 * 384 * 1248 + 3 * H * W * C
    line = {
        "metric": METRIC, "value": v, "unit": "pairs/s", "n_gpus": 1, "steps": steps, "warmup": 3, "ms_per_step": 1e3 / v,
        "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": {"workload": "configs[3]: K-shape pair + LiDAR-like 5% hints -> VPP rnd 3x3 (device) -> vpp_to_network -> RAFT-Stereo (32 iterations) / PSMNet (maxdisp 192), "
                               "batch 1 per step as test.py, random-init reference networks",
                   "pairs_per_s": {"raft-stereo": {"device_flow_resident": res[("raft-stereo", False)][0], "device_flow_from_host": res[("raft-stereo", True)][1]},
                                   "psmnet": {"device_flow_resident": res[("psmnet", False)][0], "device_flow_from_host": res[("psmnet", True)][1]}},
                   "reference_flow_pairs_per_s": ref_res,
                   "vpp_and_handoff_ms_per_frame": 1e3 * vpp_s / 50,
                   "note": "the networks dominate (they are the reference's, unmodified); the projection + hand-off this repo contributes is vpp_and_handoff_ms_per_frame"},
        "roofline": {"bound": "hbm", "kernel": "vpp rnd + u8hwc_to_f32chw hand-off (batch 1; latency bound at this size)",
                     "achieved": vpp_bytes / (vpp_s / 50) / 1e9, "peak": peak, "unit": "GB/s", "frac": vpp_bytes / (vpp_s / 50) / 1e9 / peak,
                     "traffic": None, "peak_source": peak_src},
        "cpu_baseline": None if not isinstance(ref_res, dict) or "unavailable" in ref_res else
        {"value": ref_res["raft-stereo"], "unit": "pairs/s", "cores": 1, "kind": "reference",
         "sample": "5 frames: the reference's numba vpp() on one host core + host round trip + the same network on the GPU"},
        "e2e": {"value": e, "unit": "pairs/s", "h2d_bytes_per_step": 2 * H * W * C + 4 * H * W, "d2h_bytes_per_step": 4 * H * W},
        "gpu_launches": int(launches),
    }
    print(json.dumps(line), flush=True)


if __name__ == "__main__":
    sys.path.insert(0, ROOT)
    import argparse
    ap = argparse.ArgumentParser()
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--impl", default="b200")
    a = ap.parse_args()
    main(a, reference=a.impl == "reference")
