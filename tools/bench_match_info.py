"""Cost of the opt-in per-pixel match info at bench.py's workload, alternated with the default in one process.

    python tools/bench_match_info.py [--steps 20] [--rounds 3] [--warmup 3]

Workload as bench.py's default: 64 synthetic KITTI-size pairs (1242x375, 3 channels, D = 192) per step through
VppRsgmPipeline.run_device with the inputs resident in HBM.  Two pipelines on the same inputs, alternated round by round:
  default  match_info=False: the kernels of bench.py (fused backward sweep sgm_h_kernel MODE 2)
  info     match_info=True: sgm_h_kernel MODE 4 + the info variants of the left-view tail kernels, writing state / cost / rival
Per round: the pipeline step (device events over --steps overlapped steps) and the per-stage times of one compute_rsgm call on the
first 16 pairs without and with return_info (vppb200_stage_times; the info's sweep is booked on SGM_H_BWD, its tail kernels on
MEDIAN_INTERP and TAIL).  The JSON line reports every round, the medians, the
spread of the default rounds, and the extra bytes the info moves per step as computed from the shapes (13 B per padded pixel: the
sweep writes cost + rival, the crop reads them and writes them cropped, and the state map).  The device name and power limit are
read in the same process.  Needs a CUDA device; writes nothing.
"""
import argparse
import ctypes
import json
import os
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.dont_write_bytecode = True


def power_limit_w(index):
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=power.limit", "--format=csv,noheader,nounits", "-i", str(index)],
                             capture_output=True, text=True, timeout=10).stdout.strip()
        return float(out.splitlines()[0])
    except Exception:
        return None


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--rounds", type=int, default=3)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--batch", type=int, default=64)
    args = ap.parse_args()
    import numpy as np
    import torch
    from vppstereo_b200 import _lib, rsgm, synth
    from vppstereo_b200.pipeline import VppRsgmPipeline
    if not torch.cuda.is_available():
        raise SystemExit("bench_match_info.py needs a CUDA device")
    dev = torch.device("cuda", 0)
    torch.cuda.set_device(dev)
    B, (H, W), C, D = args.batch, synth.SHAPES["K"], 3, 192
    frames = synth.make_batch(B, shape="K", hints="lidar", channels=C)
    left, right, hints = (torch.from_numpy(frames[k]).to(dev) for k in ("left", "right", "hints"))
    pipes = {"default": VppRsgmPipeline(H, W, C, batch=B, dmax=D, device=dev),
             "info": VppRsgmPipeline(H, W, C, batch=B, dmax=D, device=dev, match_info=True)}

    def step_ms(cfg):
        pipe = pipes[cfg]
        for _ in range(args.warmup):
            pipe.run_device(left, right, hints, inputs_ready=True)
        torch.cuda.synchronize(dev)
        ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        ev0.record()
        for _ in range(args.steps):
            pipe.run_device(left, right, hints, inputs_ready=True)
        ev1.record()
        torch.cuda.synchronize(dev)
        _lib.check_async(dev)
        return ev0.elapsed_time(ev1) / args.steps

    L = _lib.lib()
    stages = ["pad_gray", "census", "cost", "sgm_h_fwd", "sgm_v_down", "sgm_v_up", "sgm_h_bwd", "wta", "median_interp", "tail"]

    def stage_ms(cfg):
        n = min(16, B)
        run = lambda: rsgm.compute_rsgm(left[:n], left[:n], right[:n], dmax=D, return_info=cfg == "info")
        run()
        torch.cuda.synchronize(dev)
        L.vppb200_stage_timing(1)
        for _ in range(3):
            run()
        ms = (ctypes.c_float * len(stages))()
        calls = ctypes.c_int(0)
        _lib.call("vppb200_stage_times", ms, ctypes.byref(calls))
        L.vppb200_stage_timing(0)
        return [ms[i] / max(calls.value, 1) for i in range(len(stages))]

    Hp, Wp = H + (((H // 16) + 1) * 16 - H) % 16, W + (((W // 16) + 1) * 16 - W) % 16
    t0 = time.time()
    res = {"workload": f"K {W}x{H}x{C} D={D}, {B} pairs/step, VppRsgmPipeline.run_device, inputs resident",
           "device": torch.cuda.get_device_name(dev), "power_limit_w": power_limit_w(0), "steps_per_round": args.steps,
           "rounds": args.rounds, "info_bytes_per_step_from_shapes": 13 * B * Hp * Wp}
    step = {"default": [], "info": []}
    st = {"default": [], "info": []}
    for _ in range(args.rounds):
        for cfg in ("default", "info"):
            step[cfg].append(step_ms(cfg))
            st[cfg].append(stage_ms(cfg))
    for cfg in ("default", "info"):
        res[cfg] = {"step_ms_rounds": [round(m, 3) for m in step[cfg]], "step_ms_median": round(float(np.median(step[cfg])), 3),
                    "stage_ms_16_pairs_median": {k: round(float(np.median([r[i] for r in st[cfg]])), 3) for i, k in enumerate(stages)}}
    res["default_spread_ms"] = round(max(step["default"]) - min(step["default"]), 3)
    res["info_minus_default_ms"] = round(res["info"]["step_ms_median"] - res["default"]["step_ms_median"], 3)
    res["info_vs_default_step"] = round(res["info"]["step_ms_median"] / res["default"]["step_ms_median"], 4)
    res["wall_s"] = round(time.time() - t0, 1)
    for p in pipes.values():
        p.close()
    print(json.dumps(res))


if __name__ == "__main__":
    main()
