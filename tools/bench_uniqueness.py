"""Cost of the opt-in uniqueness test at bench.py's workload, alternated with the default in one process.

    python tools/bench_uniqueness.py [--steps 20] [--rounds 3] [--warmup 3] [--uniqueness 0.95]

Workload as bench.py's default: 64 synthetic KITTI-size pairs (1242x375, 3 channels, D = 192) per step through
VppRsgmPipeline.run_device with the inputs resident in HBM.  One pipeline object runs both configurations (the uniqueness ratio is
swapped between rounds, the buffers stay the same):
  default  uniqueness off: the fused backward sweep + WTA of bench.py (sgm_h_kernel MODE 2)
  uniq     uniqueness = --uniqueness: the same pipeline with sgm_h_kernel MODE 3
Per round: the pipeline step (device events over --steps overlapped steps) and the SGM_H_BWD stage of one compute_rsgm call on the
first 16 pairs (vppb200_stage_times).  The JSON line reports every round and the medians; "default_within_spread" says whether
every default round lies inside [min, max] of the default rounds of a second pass made after the uniq rounds.  The device name and
power limit are read in the same process.  Needs a CUDA device; writes nothing.
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
    ap.add_argument("--uniqueness", type=float, default=0.95)
    args = ap.parse_args()
    import numpy as np
    import torch
    from vppstereo_b200 import _lib, rsgm, synth
    from vppstereo_b200.pipeline import VppRsgmPipeline
    if not torch.cuda.is_available():
        raise SystemExit("bench_uniqueness.py needs a CUDA device")
    dev = torch.device("cuda", 0)
    torch.cuda.set_device(dev)
    B, (H, W), C, D = args.batch, synth.SHAPES["K"], 3, 192
    frames = synth.make_batch(B, shape="K", hints="lidar", channels=C)
    left, right, hints = (torch.from_numpy(frames[k]).to(dev) for k in ("left", "right", "hints"))
    pipe = VppRsgmPipeline(H, W, C, batch=B, dmax=D, device=dev)
    U = {"default": 1.0, "uniq": _lib.uniqueness(args.uniqueness)}
    L = _lib.lib()
    nst = 10

    def step_ms(cfg):
        pipe.uniqueness = U[cfg]
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

    def h_bwd_ms(cfg):
        kw = {} if cfg == "default" else dict(uniqueness=U[cfg], honor_uniqueness=True)
        n = min(16, B)
        rsgm.compute_rsgm(left[:n], left[:n], right[:n], dmax=D, **kw)
        torch.cuda.synchronize(dev)
        L.vppb200_stage_timing(1)
        for _ in range(3):
            rsgm.compute_rsgm(left[:n], left[:n], right[:n], dmax=D, **kw)
        ms = (ctypes.c_float * nst)()
        calls = ctypes.c_int(0)
        _lib.call("vppb200_stage_times", ms, ctypes.byref(calls))
        L.vppb200_stage_timing(0)
        return ms[6] / max(calls.value, 1)

    t0 = time.time()
    res = {"workload": f"K {W}x{H}x{C} D={D}, {B} pairs/step, VppRsgmPipeline.run_device, inputs resident",
           "device": torch.cuda.get_device_name(dev), "power_limit_w": power_limit_w(0), "uniqueness": U["uniq"],
           "steps_per_round": args.steps, "rounds": args.rounds}
    step = {"default": [], "uniq": [], "default_after": []}
    hb = {"default": [], "uniq": []}
    for _ in range(args.rounds):
        for cfg in ("default", "uniq"):
            step[cfg].append(step_ms(cfg))
            hb[cfg].append(h_bwd_ms(cfg))
    for _ in range(args.rounds):
        step["default_after"].append(step_ms("default"))
    for cfg in ("default", "uniq"):
        res[cfg] = {"step_ms_rounds": [round(m, 3) for m in step[cfg]], "step_ms_median": round(float(np.median(step[cfg])), 3),
                    "sgm_h_bwd_ms_16_pairs_rounds": [round(m, 3) for m in hb[cfg]],
                    "sgm_h_bwd_ms_16_pairs_median": round(float(np.median(hb[cfg])), 3)}
    res["default_after_ms_rounds"] = [round(m, 3) for m in step["default_after"]]
    allv = step["default"] + step["default_after"]
    res["default_spread_ms"] = round(max(allv) - min(allv), 3)
    res["uniq_vs_default_step"] = round(res["uniq"]["step_ms_median"] / res["default"]["step_ms_median"], 4)
    res["uniq_vs_default_h_bwd"] = round(res["uniq"]["sgm_h_bwd_ms_16_pairs_median"] / res["default"]["sgm_h_bwd_ms_16_pairs_median"], 4)
    res["wall_s"] = round(time.time() - t0, 1)
    pipe.close()
    print(json.dumps(res))


if __name__ == "__main__":
    main()
