"""Step time of the K-shape workload with the default and with honoured SGM parameters, alternated in one process.

    python tools/bench_sgm_params.py [--steps 20] [--rounds 3] [--warmup 3] [--ood-steps 2]

Workload as bench.py's default: 64 synthetic KITTI-size pairs (1242x375, 3 channels, D = 192) per step through
VppRsgmPipeline.run_device with the inputs resident in HBM.  One pipeline object runs every configuration (its matcher
parameters are swapped between runs, the buffers stay the same):
  default   the reference's effective parameters (7, 17, 0.25, 50), i.e. what bench.py measures
  honoured  rsgm.py's defaults (11, 17, 0.5, 35), inside the sweep domain: the same four sweeps
  ood       (30, 10, 0.5, 20), outside the domain (P2min < P1): the saturating per-path kernels, timed once (--ood-steps)
default and honoured alternate for --rounds rounds of --steps steps each; the JSON line reports the median round.  The device
name and power limit are read in the same process.  Needs a CUDA device; writes nothing.
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

CONFIGS = {"default": None, "honoured": (11, 17, 0.5, 35), "ood": (30, 10, 0.5, 20)}


def power_limit_w(index):
    try:
        import pynvml
        pynvml.nvmlInit()
        return pynvml.nvmlDeviceGetPowerManagementLimit(pynvml.nvmlDeviceGetHandleByIndex(index)) / 1000.0
    except Exception:
        pass
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
    ap.add_argument("--ood-steps", type=int, default=2)
    ap.add_argument("--batch", type=int, default=64)
    args = ap.parse_args()
    import numpy as np
    import torch
    from vppstereo_b200 import _lib, synth
    from vppstereo_b200.pipeline import VppRsgmPipeline
    if not torch.cuda.is_available():
        raise SystemExit("bench_sgm_params.py needs a CUDA device")
    dev = torch.device("cuda", 0)
    torch.cuda.set_device(dev)
    B, (H, W), C, D = args.batch, synth.SHAPES["K"], 3, 192
    frames = synth.make_batch(B, shape="K", hints="lidar", channels=C)
    left, right, hints = (torch.from_numpy(frames[k]).to(dev) for k in ("left", "right", "hints"))
    pipe = VppRsgmPipeline(H, W, C, batch=B, dmax=D, device=dev)
    params = {k: (None if v is None else _lib.sgm_params(*v)) for k, v in CONFIGS.items()}
    assert _lib.sgm_params_fast(params["honoured"]) and not _lib.sgm_params_fast(params["ood"])

    def run(cfg, steps, warmup):
        pipe.sgm_params = params[cfg]
        for _ in range(warmup):
            pipe.run_device(left, right, hints, inputs_ready=True)
        torch.cuda.synchronize(dev)
        ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        ev0.record()
        for _ in range(steps):
            pipe.run_device(left, right, hints, inputs_ready=True)
        ev1.record()
        torch.cuda.synchronize(dev)
        _lib.check_async(dev)
        return ev0.elapsed_time(ev1) / steps

    t0 = time.time()
    rounds = {"default": [], "honoured": []}
    for _ in range(args.rounds):
        for cfg in ("default", "honoured"):
            rounds[cfg].append(run(cfg, args.steps, args.warmup))
    ood = run("ood", args.ood_steps, 1) if args.ood_steps > 0 else None
    res = {"workload": f"K {W}x{H}x{C} D={D}, {B} pairs/step, VppRsgmPipeline.run_device, inputs resident",
           "device": torch.cuda.get_device_name(dev), "power_limit_w": power_limit_w(0),
           "steps_per_round": args.steps, "rounds": args.rounds}
    for cfg, ms in rounds.items():
        med = float(np.median(ms))
        res[cfg] = {"params": CONFIGS[cfg] or (7, 17, 0.25, 50), "ms_per_step_median": round(med, 3),
                    "ms_per_step_rounds": [round(m, 3) for m in ms], "pairs_per_s": round(B * 1000.0 / med, 1)}
    res["honoured_vs_default"] = round(res["honoured"]["ms_per_step_median"] / res["default"]["ms_per_step_median"], 4)
    if ood is not None:
        res["ood"] = {"params": CONFIGS["ood"], "ms_per_step": round(ood, 3), "steps": args.ood_steps,
                      "pairs_per_s": round(B * 1000.0 / ood, 1)}
    res["wall_s"] = round(time.time() - t0, 1)
    pipe.close()
    print(json.dumps(res))


if __name__ == "__main__":
    main()
