"""What the projection options of VppRsgmPipeline cost, in one process; prints one JSON line.

    python tools/bench_pipeline_modes.py [--steps 20] [--warmup 3] [--serial-calls 3]

Workload: 64 synthetic KITTI-size pairs (1242x375, 3 channels, D = 192, LiDAR-like 5 % hints with 3 foreground boxes from
synth) per step, inputs resident in HBM.  Configurations:
  default            VppRsgmPipeline's defaults (rnd, fixed 3x3 patch, no mask): the kernels bench.py times
  maskocc_rnd        maskocc=True (test.py --maskocc, the paper's default)
  maskocc_maxdist    maskocc=True, method="maxDistance", wsizeAgg 64x3
  journal            maskocc=True, wsize=7, use_bilateral_patch=True, use_distance_patch=True (rnd)
For each: ms per step of back-to-back run_device(inputs_ready=True) (rounds in the order A B C D D C B A, CUDA events around
each round), the run_device_serial stage split (copies, occlusion, bilateral + thresholds, scan, matcher; CUDA events
between the front-phase steps, mean over --serial-calls calls) and the library's kernel launches per call.  The same
configurations composed from the single-call front-ends (filter.occlusion_heuristic -> vpp_standalone.vpp -> rsgm.compute_rsgm,
as bench_m.py composes them) are timed per step the same way.  Checked before timing: the pipeline's maskocc_maxdist batch
equals the composed chain bit for bit.  The device name and power limit are read in the same process.  Writes nothing.
"""
import argparse
import json
import os
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.dont_write_bytecode = True

CONFIGS = {
    "default": {},
    "maskocc_rnd": dict(maskocc=True),
    "maskocc_maxdist": dict(maskocc=True, method="maxDistance", wsizeAgg_x=64, wsizeAgg_y=3),
    "journal": dict(maskocc=True, wsize=7, use_bilateral_patch=True, use_distance_patch=True),
}


def gpu_info(index):
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader", "-i", str(index)],
                             capture_output=True, text=True, timeout=20).stdout.strip()
        return out.splitlines()[0] if out else None
    except Exception:
        return None


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--serial-calls", type=int, default=3)
    args = ap.parse_args()
    import numpy as np
    import torch
    from vppstereo_b200 import _lib, filter as vfilter, rsgm, synth, vpp_standalone
    from vppstereo_b200.pipeline import VppRsgmPipeline
    if not torch.cuda.is_available():
        raise SystemExit("bench_pipeline_modes.py needs a CUDA device")
    dev = torch.device("cuda", 0)
    torch.cuda.set_device(dev)
    t_start = time.time()
    res = {"device": torch.cuda.get_device_name(dev), "nvidia_smi (name, power limit, max SM clock)": gpu_info(0)}
    B, (H, W), C, D = 64, synth.SHAPES["K"], 3, 192
    frames = synth.make_batch(B, shape="K", hints="lidar", channels=C, foreground=3)
    left, right, hints = (torch.from_numpy(frames[k]).to(dev) for k in ("left", "right", "hints"))
    torch.cuda.synchronize(dev)
    res["workload"] = f"K {W}x{H}x{C} D={D}, {B} pairs/step, lidar-like 5% hints + 3 foreground boxes, inputs resident"
    res["configs"] = CONFIGS
    pipes = {name: VppRsgmPipeline(H, W, C, batch=B, dmax=D, device=dev, **kw) for name, kw in CONFIGS.items()}

    def composed(kw, seed):
        vkw = {k: v for k, v in kw.items() if k != "maskocc"}
        mask = vfilter.occlusion_heuristic(hints)[1] if kw.get("maskocc") else None
        lv, rv = vpp_standalone.vpp(left, right, hints, g_occ=mask, seed=seed, **vkw)
        return rsgm.compute_rsgm(left, lv, rv, dmax=D)

    # check: the pipeline == the composed front-ends (maxDistance: no pattern seed involved)
    got = pipes["maskocc_maxdist"].run_device_serial(left, right, hints).clone()
    want = composed(CONFIGS["maskocc_maxdist"], None)
    torch.cuda.synchronize(dev)
    assert torch.equal(got.view(torch.int32), want.view(torch.int32)), "maskocc_maxdist: pipeline != composed front-ends"
    res["checked"] = "maskocc_maxdist pipeline == occlusion_heuristic -> vpp -> compute_rsgm, bit for bit"
    del got, want

    def timed(fn):
        for _ in range(args.warmup):
            fn()
        torch.cuda.synchronize(dev)
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(args.steps):
            fn()
        e1.record()
        torch.cuda.synchronize(dev)
        return e0.elapsed_time(e1) / args.steps

    names = list(CONFIGS)
    order = names + names[::-1]
    pipe_ms = {n: [] for n in names}
    for n in order:
        p = pipes[n]
        pipe_ms[n].append(round(timed(lambda: p.run_device(left, right, hints, inputs_ready=True)), 3))
        p.check()
    comp_ms = {n: [] for n in names}
    for n in order:
        comp_ms[n].append(round(timed(lambda: composed(CONFIGS[n], 12345)), 3))

    split, launches = {}, {}
    for n in names:
        p = pipes[n]
        p.run_device_serial(left, right, hints)
        torch.cuda.synchronize(dev)
        l0 = _lib.launch_count()
        p.run_device(left, right, hints)
        torch.cuda.synchronize(dev)
        launches[n] = _lib.launch_count() - l0
        acc = {}
        for _ in range(args.serial_calls):
            p._stage_marks = []
            st = torch.cuda.current_stream(dev)
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record(st)
            p.run_device_serial(left, right, hints)
            e1.record(st)
            torch.cuda.synchronize(dev)
            marks = [("start", e0)] + p._stage_marks + [("matcher", e1)]
            p._stage_marks = None
            for (_, a), (name, b) in zip(marks, marks[1:]):
                acc[name] = acc.get(name, 0.0) + a.elapsed_time(b) / args.serial_calls
        split[n] = {k: round(v, 3) for k, v in acc.items()}
        p.check()
    for p in pipes.values():
        p.close()
    res["run_device_ms_per_step"] = {"order": " ".join(order), "steps_per_round": args.steps, **pipe_ms}
    res["composed_front_ends_ms_per_step"] = {"order": " ".join(order), "steps_per_round": args.steps, **comp_ms}
    res["composed_vs_pipeline"] = {n: round(float(np.mean(comp_ms[n]) / np.mean(pipe_ms[n])), 3) for n in names}
    res["run_device_serial_stage_ms"] = split
    res["stage_names"] = ("copy = input copies into the projected-image buffers; occlusion = occlusion_heuristic; "
                          "patch_operands = bgr2gray + bilateral filling + distance thresholds; scan = the VPP scan; "
                          "matcher = compute_rsgm (front + sweeps + tail)")
    res["launches_per_run_device"] = launches
    res["wall_s"] = round(time.time() - t_start, 1)
    print(json.dumps(res))


if __name__ == "__main__":
    main()
