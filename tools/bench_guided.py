"""What guided matching costs on the hot paths, in one process; prints one JSON line.

    python tools/bench_guided.py [--steps 200] [--warmup 10] [--cost-calls 20] [--m-reps 3] [--parent-lib PATH]

(a) pipeline   64 synthetic KITTI-size pairs (1242x375, 3 channels, D = 192, LiDAR-like hints from synth) per step through
               VppRsgmPipeline.run_device with the inputs resident in HBM: unguided vs guided=True (validhints = hints > 0).
               Rounds of --steps steps in the order A B B A; ms per step from CUDA events around each round.
(b) cost       the COST stage (pad/census excluded) of guided batch-64 compute_rsgm on one projected batch, read with
               vppb200_stage_timing.  With --parent-lib (the same library built from another revision) both libraries run
               alternately in this process (order N P P N), and their disparities are compared bit for bit.
(c) banded     one guided Middlebury-size frame (2880x1988, D = 192): BandedRsgm with 2 bands vs unsplit compute_rsgm on one GPU,
               alternated; seconds per frame with a device synchronise around each call.
Checked before timing: the guided batch of (a) equals guided compute_rsgm of the same projected pair, and (c) banded == unsplit.
The device name and power limit are read in the same process.  Needs a CUDA device; writes nothing.
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


def gpu_info(index):
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader", "-i", str(index)],
                             capture_output=True, text=True, timeout=20).stdout.strip()
        return out.splitlines()[0] if out else None
    except Exception:
        return None


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--steps", type=int, default=200)
    ap.add_argument("--warmup", type=int, default=10)
    ap.add_argument("--cost-calls", type=int, default=20)
    ap.add_argument("--m-reps", type=int, default=3)
    ap.add_argument("--parent-lib", default=None, help="libvppstereo_b200.so of the revision to compare the COST stage with")
    ap.add_argument("--skip", default="", help="comma-separated parts to leave out (a, b, c)")
    args = ap.parse_args()
    skip = set(filter(None, args.skip.split(",")))
    import numpy as np
    import torch
    from vppstereo_b200 import _lib, rsgm, synth
    from vppstereo_b200.banded import BandedRsgm
    from vppstereo_b200.pipeline import VppRsgmPipeline
    if not torch.cuda.is_available():
        raise SystemExit("bench_guided.py needs a CUDA device")
    dev = torch.device("cuda", 0)
    torch.cuda.set_device(dev)
    t_start = time.time()
    res = {"device": torch.cuda.get_device_name(dev), "nvidia_smi": gpu_info(0)}
    B, (H, W), C, D = 64, synth.SHAPES["K"], 3, 192
    frames = synth.make_batch(B, shape="K", hints="lidar", channels=C)
    left, right, hints = (torch.from_numpy(frames[k]).to(dev) for k in ("left", "right", "hints"))
    valid = (hints > 0).float()
    torch.cuda.synchronize(dev)

    # ---- (a) pipeline, unguided vs guided
    if "a" not in skip:
        pipes = {"unguided": VppRsgmPipeline(H, W, C, batch=B, dmax=D, device=dev),
                 "guided": VppRsgmPipeline(H, W, C, batch=B, dmax=D, device=dev, guided=True)}
        kw = {"unguided": {}, "guided": {"validhints": valid}}
        g = pipes["guided"]
        out = g.run_device(left, right, hints, validhints=valid).clone()
        want = rsgm.compute_rsgm(left, g.lv, g.rv, hints=hints, validhints=valid, dmax=D)
        torch.cuda.synchronize(dev)
        assert torch.equal(out.view(torch.int32), want.view(torch.int32)), "guided pipeline != guided compute_rsgm"
        plain = rsgm.compute_rsgm(left, g.lv, g.rv, dmax=D)
        res["guided_changes_pixels"] = int((plain.view(torch.int32) != want.view(torch.int32)).sum())

        def run(name):
            p = pipes[name]
            for _ in range(args.warmup):
                p.run_device(left, right, hints, inputs_ready=True, **kw[name])
            torch.cuda.synchronize(dev)
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            for _ in range(args.steps):
                p.run_device(left, right, hints, inputs_ready=True, **kw[name])
            e1.record()
            torch.cuda.synchronize(dev)
            p.check()
            return e0.elapsed_time(e1) / args.steps

        rounds = {"unguided": [], "guided": []}
        for name in ("unguided", "guided", "guided", "unguided"):
            rounds[name].append(run(name))
        res["pipeline"] = {"workload": f"K {W}x{H}x{C} D={D}, {B} pairs/step, run_device, inputs resident", "steps_per_round": args.steps,
                           "order": "A B B A", **{k: [round(v, 3) for v in ms] for k, ms in rounds.items()}}
        res["pipeline"]["guided_vs_unguided"] = round(float(np.mean(rounds["guided"]) / np.mean(rounds["unguided"])), 4)
        lv, rv = g.lv.clone(), g.rv.clone()
        for p in pipes.values():
            p.close()
        del pipes, g
    else:
        lv, rv = left.clone(), right.clone()
    torch.cuda.empty_cache()

    # ---- (b) COST stage of guided compute_rsgm, this library vs --parent-lib
    if "b" not in skip:
        libs = {"this": _lib.lib()}
        if args.parent_lib:
            libs["parent"] = _lib.bind(ctypes.CDLL(os.path.abspath(args.parent_lib)))
        need = max(L.vppb200_rsgm_workspace_bytes(H, W, C, D, B) for L in libs.values())
        ws = torch.empty(need, dtype=torch.uint8, device=dev)
        outs = {k: torch.empty((B, H, W), dtype=torch.float32, device=dev) for k in libs}
        st = ctypes.c_void_p(torch.cuda.current_stream(dev).cuda_stream)
        P = _lib.ptr

        def call(name):
            rc = libs[name].vppb200_compute_rsgm(P(left), P(lv), P(rv), P(hints), P(valid), P(outs[name]), H, W, C, D, 1, None, P(ws),
                                                 ctypes.c_size_t(ws.numel()), B, st)
            assert rc == 0, f"{name}: compute_rsgm status {rc}"

        def cost_ms(name):
            L = libs[name]
            call(name)                                     # warm
            torch.cuda.synchronize(dev)
            L.vppb200_stage_timing(1)
            for _ in range(args.cost_calls):
                call(name)
            ms = (ctypes.c_float * 10)()
            calls = ctypes.c_int(0)
            L.vppb200_stage_times(ms, ctypes.byref(calls))
            L.vppb200_stage_timing(0)
            return ms[2] / max(calls.value, 1), sum(ms) / max(calls.value, 1)

        order = ["this", "parent", "parent", "this"] if "parent" in libs else ["this", "this"]
        cost = {k: [] for k in libs}
        total = {k: [] for k in libs}
        for name in order:
            c, t = cost_ms(name)
            cost[name].append(round(c, 4)); total[name].append(round(t, 3))
        torch.cuda.synchronize(dev)
        want = rsgm.compute_rsgm(left, lv, rv, hints=hints, validhints=valid, dmax=D)
        torch.cuda.synchronize(dev)
        assert torch.equal(outs["this"].view(torch.int32), want.view(torch.int32)), "raw call != compute_rsgm"
        res["cost_stage"] = {"workload": f"guided compute_rsgm, {B} K frames, D={D}", "calls_per_round": args.cost_calls,
                             "order": " ".join(order), "cost_ms": cost, "all_stages_ms": total}
        if "parent" in libs:
            res["cost_stage"]["parent_equal"] = bool(torch.equal(outs["parent"].view(torch.int32), outs["this"].view(torch.int32)))
        else:
            res["cost_stage"]["parent"] = "not measured"
        del ws, outs
        torch.cuda.empty_cache()

    # ---- (c) one guided M frame: 2 bands vs unsplit
    if "c" not in skip:
        Hm, Wm = synth.SHAPES["M"]
        Dm = 192
        p = synth.make_pair(0, shape="M", hints="lidar")
        l, r = torch.from_numpy(p["left"]).to(dev), torch.from_numpy(p["right"]).to(dev)
        h = torch.from_numpy(p["hints"]).to(dev)
        v = (h > 0).float()
        band = BandedRsgm(Hm, Wm, 3, dmax=Dm, n_bands=2, device=dev)
        unsplit = lambda: rsgm.compute_rsgm(l, l, r, hints=h, validhints=v, dmax=Dm)
        banded = lambda: band.compute(l, l, r, hints=h, validhints=v)
        a, b = unsplit(), banded()
        torch.cuda.synchronize(dev)
        assert torch.equal(a.view(torch.int32), b.view(torch.int32)), "guided M frame: 2 bands != unsplit"
        del a, b
        times = {"unsplit": [], "bands2": []}
        fns = {"unsplit": unsplit, "bands2": banded}
        for name in ("unsplit", "bands2", "bands2", "unsplit") * max(1, args.m_reps // 2):
            torch.cuda.synchronize(dev)
            t0 = time.perf_counter()
            fns[name]()
            torch.cuda.synchronize(dev)
            times[name].append(round(time.perf_counter() - t0, 4))
        res["banded_m"] = {"workload": f"one guided M frame {Wm}x{Hm}x3 D={Dm}, one GPU", "s_per_frame": times}
    res["wall_s"] = round(time.time() - t_start, 1)
    print(json.dumps(res))


if __name__ == "__main__":
    main()
