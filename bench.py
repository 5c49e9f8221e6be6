#!/usr/bin/env python
"""Benchmark of the VPP + rSGM hot path (BASELINE.json: "VPP pairs/s & rSGM fps @1242x375, 5% hints, D=192; % of HBM peak").

    python bench.py [--gpus N] [--steps K] [--warmup W] [--batch B] [--impl reference] [--dump-outputs DIR]

One step = one pass of the hot path (VPP random-pattern projection, then compute_rsgm: census, Hamming cost volume,
8-path SGM, WTA + sub-pixel, LR check, speckle filter, fills) over one batch of synthetic KITTI-shape pairs
(configs[1]: 1242x375, LiDAR-like 5 % hints, D=192, batch 64 per GPU).  Prints ONE JSON line (rank 0).
  value      whole-job pairs/s with the inputs resident in HBM
  e2e        the same through the host-buffer API (pinned H2D of inputs + D2H of disparities inside the timed region)
  roofline   the dominant kernel, sgm_v2_kernel (one vertical+diagonal sweep = 3 of the 8 SGM paths, 2 sweeps per step):
             its compulsory bytes per sweep of the batch (cost volume read + S read-modify-write = 5*W*H*D per frame, DESIGN.md 4) /
             its average launch duration measured live with CUDA events on the launching stream, against
             MEASURED_PEAKS.json hbm_gbs; the whole aggregation against SURVEY.md 8d's 4*W*H*D + W*H is reported beside it
  cpu_baseline  the reference's own CPU code (oracle/_ref) on the host cores, bounded sample, rank 0 at N=1
--impl reference: times that CPU path instead, same metric/config, all host cores.
--dump-outputs DIR: writes what the last timed step computed as float32 .npy files (see dump_outputs); the inputs and the
pattern seeds depend on the arguments only, so two builds run with the same arguments can be compared output for output.
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
# The path keeps ~10 CUDA streams busy (three pipeline phases, two side branches, H2D / D2H, the peer gather's copy, credit and
# consumer streams); with the default of 8 hardware connections two of them share a queue and a stream that is parked in a
# wait (peer flag, event) holds up the one behind it.  Must be set before the CUDA context exists.
os.environ.setdefault("CUDA_DEVICE_MAX_CONNECTIONS", "32")

METRIC = "VPP pairs/s & rSGM fps @1242x375, 5% hints, D=192; % of HBM peak"
H, W, C, D = 375, 1242, 3, 192
HP, WP = 384, 1248
ALG_BYTES_AGG = 4 * WP * HP * D + WP * HP            # SURVEY.md 8(d): aggregate, per frame (368.5 MB)
ALG_BYTES_VSWEEP = 5 * WP * HP * D + WP * HP         # one v-sweep launch, per frame: uint8 costs in, uint16 S in and out (460 MB)
ALG_BYTES_VPP = 4 * H * W * C + 4 * H * W + H * W    # + C * in-image patch pixels of the hints (added at run time)
STAGES = ["pad_gray", "census", "cost_volume", "sgm_h_fwd", "sgm_v_down", "sgm_v_up", "sgm_h_bwd_wta", "wta_unfused", "median_interp",
          "tail"]


def measured_peak():
    try:
        with open(os.path.join(ROOT, "MEASURED_PEAKS.json")) as f:
            return float(json.load(f)["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
    except Exception:
        return 6650.0, "fallback (B200_PROFILING.md)"


class ClockSampler(threading.Thread):
    """SM clock / throttle reasons sampled DURING the timed region (B200_PROFILING.md recipe).  NVML in-process every
    10 ms (a timed region of a few hundred ms still gets tens of samples); nvidia-smi polling if NVML is unavailable."""
    Q = "clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown," \
        "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap"
    NAMES = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]

    def __init__(self, index):
        super().__init__(daemon=True)
        self.index, self.samples, self.stop_flag, self.source = index, [], False, "nvml"
        self.nv = self.handle = None
        try:
            import pynvml
            pynvml.nvmlInit()
            vis = os.environ.get("CUDA_VISIBLE_DEVICES", "")
            phys = index
            if vis:
                ent = vis.split(",")[index].strip()
                phys = int(ent) if ent.isdigit() else index
            self.nv, self.handle = pynvml, pynvml.nvmlDeviceGetHandleByIndex(phys)
            self.max_mhz = pynvml.nvmlDeviceGetMaxClockInfo(self.handle, pynvml.NVML_CLOCK_SM)
            self._sample_nvml()                         # fail here, not in the thread
            self.samples.clear()
        except Exception:
            self.nv, self.source = None, "nvidia-smi"

    def _sample_nvml(self):
        nv = self.nv
        mhz = nv.nvmlDeviceGetClockInfo(self.handle, nv.NVML_CLOCK_SM)
        try:
            bits = nv.nvmlDeviceGetCurrentClocksEventReasons(self.handle)
        except Exception:
            bits = nv.nvmlDeviceGetCurrentClocksThrottleReasons(self.handle)
        flags = [bool(bits & 0x8), bool(bits & 0x40), bool(bits & 0x20), bool(bits & 0x4)]   # hw, hw_thermal, sw_thermal, sw_power_cap
        self.samples.append((int(mhz), int(self.max_mhz), flags))

    def _sample_smi(self):
        out = subprocess.run(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits", "-i", str(self.index)],
                             capture_output=True, text=True, timeout=5).stdout.strip()
        s = [x.strip() for x in out.split(",")]
        if len(s) >= 6 and s[0].isdigit():
            self.samples.append((int(s[0]), int(s[1]) if s[1].isdigit() else 0, [x.lower().startswith("active") for x in s[2:6]]))

    def run(self):
        while not self.stop_flag:
            try:
                self._sample_nvml() if self.nv else self._sample_smi()
            except Exception:
                pass
            time.sleep(0.01 if self.nv else 0.2)

    def summary(self):
        self.stop_flag = True
        if not self.samples:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["unsampled"]}
        sm = sorted(s[0] for s in self.samples)
        reasons = [n for i, n in enumerate(self.NAMES) if any(s[2][i] for s in self.samples)]
        return {"sm_mhz": sm[len(sm) // 2], "sm_max_mhz": max(s[1] for s in self.samples), "reasons": reasons,
                "samples": len(self.samples), "source": self.source}


# ---------------------------------------------------------------------------------------- CPU reference arm
def _cpu_frame(f, kind, shape, dmax):
    """VPP + compute_rsgm of one synthetic frame on one core with the reference's own code (oracle/_ref), or with the
    oracle port when the compiled reference is absent."""
    import numpy as np
    from vppstereo_b200 import synth
    p = synth.make_pair(f, shape=shape, hints="lidar")
    t0 = time.perf_counter()
    if kind == "reference":
        from oracle import ref
        r = ref.load()
        l, rr = p["left"].copy(), p["right"].copy()
        Hh, Ww = p["hints"].shape
        r.vpp_core_opt.init_rand(1 + f)
        r.vpp_core_opt.virtual_projection_scan_rnd(l, rr, p["hints"], Ww, Hh, 3, False, 3, 1, 0.4, 0.0,
                                                   np.zeros((Hh, Ww), np.uint8), False, True)
        out = r.rsgm.compute_rsgm(p["left"], l, rr, dmax=dmax)
    else:
        from oracle import oracle as orc
        n = orc.stream_length(p["hints"], 3, 3, False)
        l, rr = orc.vpp(p["left"], p["right"], p["hints"], stream=np.zeros(n, np.uint8), mode=0)
        out = orc.compute_rsgm(p["left"], l, rr, dmax=dmax)
    return time.perf_counter() - t0, float(out.mean())


def cpu_worker_main(kind):
    """Worker process of the CPU arm: line protocol on stdin/stdout (pipes only: the GPU box has no /dev/shm semaphores).
    'run <f0> <n>' -> runs n K-shape frames, answers '<seconds> <mean>'; 'quit' ends."""
    os.environ["OMP_NUM_THREADS"] = "1"
    _cpu_frame(0, kind, (48, 96), 32)                 # warm-up: numba JIT of the reference's tail functions (not timed)
    print("ready", flush=True)
    for line in sys.stdin:
        parts = line.split()
        if not parts or parts[0] == "quit":
            break
        f0, n = int(parts[1]), int(parts[2])
        t0 = time.perf_counter()
        m = 0.0
        for i in range(n):
            m += _cpu_frame(f0 + i, kind, "K", D)[1]
        print(f"{time.perf_counter() - t0:.6f} {m / max(n, 1):.6f}", flush=True)


class CpuBaseline:
    """All host cores, one single-threaded worker process per core (the reference is single-threaded per frame:
    models/rsgm/rsgm.py:44 passes numThreads=1), frame-parallel."""

    def __init__(self, cores=None):
        from oracle import ref
        self.kind = "reference" if ref.available() else "port"
        if self.kind == "port":
            from oracle import oracle as orc
            orc.build()
        self.cores = cores or min(len(os.sched_getaffinity(0)), 64)
        env = dict(os.environ, OMP_NUM_THREADS="1", CUDA_VISIBLE_DEVICES="")
        self.procs = [subprocess.Popen([sys.executable, os.path.abspath(__file__), "--cpu-worker", self.kind], stdin=subprocess.PIPE,
                                       stdout=subprocess.PIPE, text=True, env=env, cwd=ROOT) for _ in range(self.cores)]
        for p in self.procs:
            line = p.stdout.readline()
            if line.strip() != "ready":
                raise RuntimeError(f"cpu worker failed to start: {line!r}")

    def step(self, f0, frames=None):
        """one bounded sample: `frames` K-shape frames spread over the workers; returns (frames, seconds, per-frame seconds)"""
        frames = frames or self.cores
        per = [frames // self.cores + (1 if w < frames % self.cores else 0) for w in range(self.cores)]
        t0 = time.perf_counter()
        off = 0
        for p, n in zip(self.procs, per):
            p.stdin.write(f"run {f0 + off} {n}\n"); p.stdin.flush()
            off += n
        lat = []
        for p, n in zip(self.procs, per):
            secs = float(p.stdout.readline().split()[0])
            if n:
                lat.append(secs / n)
        dt = time.perf_counter() - t0
        return frames, dt, sum(lat) / max(len(lat), 1)

    def close(self):
        for p in self.procs:
            try:
                p.stdin.write("quit\n"); p.stdin.flush()
                p.wait(timeout=30)
            except Exception:
                p.kill()

    def describe(self, frames_per_step, steps):
        what = "compiled reference (Cython vpp_core_opt + SSE pyrSGM + rsgm.py glue from oracle/_ref)" if self.kind == "reference" \
            else "C oracle port (oracle/*.c)"
        return f"{what}; {steps} step(s) x {frames_per_step} K-shape frames (1242x375, D=192), frame-parallel over {self.cores} single-threaded worker processes"


def run_reference_arm(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    cb = CpuBaseline()
    for w in range(min(args.warmup, 1)):               # workers are already JIT-warm; one untimed sample is enough
        cb.step(10_000 + w * cb.cores)
    tot_f, tot_t, lat = 0, 0.0, []
    for k in range(args.steps):
        f, dt, per = cb.step(k * cb.cores)
        tot_f += f; tot_t += dt; lat.append(per)
    cb.close()
    v = tot_f / tot_t
    line = {"impl": "reference", "metric": METRIC, "value": v, "unit": "pairs/s", "n_gpus": args.gpus, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": 1e3 * tot_t / max(args.steps, 1), "higher_is_better": True, "scaling": "weak",
            "vs_baseline": None, "dtype": "u16", "data": "synthetic",
            "config": {"workload": "configs[1]: KITTI-shape 1242x375x3 pairs, LiDAR-like 5% hints, VPP rnd 3x3 + rSGM D=192",
                       "frames_per_step": cb.cores, "single_frame_latency_s": sum(lat) / len(lat)},
            "cpu_baseline": {"value": v, "unit": "pairs/s", "cores": cb.cores, "kind": cb.kind,
                             "sample": cb.describe(cb.cores, args.steps)},
            "e2e": {"value": v, "unit": "pairs/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
            "gpu_launches": 0}
    print(json.dumps(line), flush=True)


# ---------------------------------------------------------------------------------------- parity probe
PROBE_STEP = 1 << 20          # call number (pattern seed) of the probe batch: fixed, whatever was timed before it
PROBE_FRAMES = (0, 63)
BENCH_CHECK = os.path.join(ROOT, "tests", "golden", "bench_check.json")


def bench_inputs(rank, B):
    """The benchmark's synthetic batch of one rank: 8 distinct K-shape frames tiled to B (generation is host work, not part of
    the path).  Returns numpy arrays left, right [B,H,W,3] uint8 and hints [B,H,W] float32."""
    import numpy as np
    from vppstereo_b200 import synth
    uniq = min(B, 8)
    frames = [synth.make_pair(rank * 1000 + f, shape="K", hints="lidar") for f in range(uniq)]
    idx = [i % uniq for i in range(B)]
    return (np.stack([frames[i]["left"] for i in idx]), np.stack([frames[i]["right"] for i in idx]),
            np.stack([frames[i]["hints"] for i in idx]))


def probe_digest(lv, rv, disp):
    """sha256 over the projected pair (uint8) and the disparity bit patterns (float32) of one frame"""
    import hashlib
    import numpy as np
    h = hashlib.sha256()
    for a in (lv, rv, disp):
        h.update(np.ascontiguousarray(a).tobytes())
    return h.hexdigest()


def parity_probe(batch=64, pipe=None, tensors=None):
    """One extra batch of rank 0's benchmark inputs through the very pipeline object and code path that was timed
    (VppRsgmPipeline.run_device: device-generated pattern, three streams, the planner's v-sweep shape for this batch), with a
    fixed pattern seed; sha256 of the projected pair and of the disparity bits of frames 0 and batch-1.  bench.py asserts them
    against tests/golden/bench_check.json, which tests/golden/make_bench_check.py derives with the CPU oracle."""
    import torch
    from vppstereo_b200 import _lib
    from vppstereo_b200.pipeline import VppRsgmPipeline
    dev = torch.device("cuda", torch.cuda.current_device())
    if tensors is None:
        tensors = tuple(torch.from_numpy(a).to(dev) for a in bench_inputs(0, batch))
    own = pipe is None
    if own:
        pipe = VppRsgmPipeline(H, W, C, batch=batch, dmax=D, device=dev)
    was = _lib.get_tuning(_lib.TUNE_RCP_HOST, 0)
    _lib.set_tuning(_lib.TUNE_RCP_HOST, 0)           # the committed hashes are for the library's default (fixed) RCPSS table
    try:
        out = pipe.run_device(*tensors, inputs_ready=True, step=PROBE_STEP)
        torch.cuda.synchronize(dev)
        frames = [f if f < batch else batch - 1 for f in PROBE_FRAMES]
        digests = [probe_digest(pipe.lv[f].cpu().numpy(), pipe.rv[f].cpu().numpy(), out[f].cpu().numpy()) for f in frames]
    finally:
        _lib.set_tuning(_lib.TUNE_RCP_HOST, was)
        if own:
            pipe.close()
    return {"frames": frames, "step": PROBE_STEP, "sha256": digests}


def assert_parity_probe(probe, batch):
    """Compare with the committed oracle-derived digests; a mismatch is fatal (no JSON line is printed)."""
    if batch != 64:
        probe["expected"] = None
        probe["ok"] = None            # the committed digests are for the configured batch of 64
        return probe
    with open(BENCH_CHECK) as f:
        want = json.load(f)
    probe["expected"] = want["sha256"]
    probe["ok"] = probe["sha256"] == want["sha256"]
    if not probe["ok"]:
        raise SystemExit(f"bench.py: PARITY PROBE FAILED: disparities of the timed path differ from the oracle-derived digests "
                         f"in {BENCH_CHECK}: got {probe['sha256']}, want {want['sha256']}")
    return probe


# ---------------------------------------------------------------------------------------- GPU arm
def ncu_traffic():
    """dram read + write bytes of one v-sweep launch from the committed ncu capture of this build (tools/ncu_traffic.py writes
    profiles/vsweep_traffic.json from the .ncu-rep); None when the file is missing"""
    try:
        with open(os.path.join(ROOT, "profiles", "vsweep_traffic.json")) as f:
            d = json.load(f)
        return float(d["dram_bytes_read"]) + float(d["dram_bytes_write"]), d.get("source")
    except Exception:
        return None, None


DUMP_FRAMES = 16              # disparity maps written by --dump-outputs: a fixed, seeded choice of frames of the batch
DUMP_PAIRS = 2                # ... and the projected pairs of the first two of them


def dump_outputs(outdir, disp, lv, rv):
    """Writes what one step of the pipeline computed, as float32: disparity.npy [16,H,W] (the disparities run_device returns, for
    16 frames chosen with a fixed seed: the whole batch is 119 MB), left_vpp.npy / right_vpp.npy [2,H,W,C] (the projected pair
    of the first two of those frames, uint8 values) and disparity_frames.npy (the batch indices of the 16 frames).  52 MB."""
    import numpy as np
    import torch
    frames = np.sort(np.random.default_rng(0).choice(disp.shape[0], min(DUMP_FRAMES, disp.shape[0]), replace=False))
    idx = torch.from_numpy(frames).to(disp.device)
    os.makedirs(outdir, exist_ok=True)
    arrays = {"disparity": disp.index_select(0, idx), "left_vpp": lv.index_select(0, idx[:DUMP_PAIRS]),
              "right_vpp": rv.index_select(0, idx[:DUMP_PAIRS])}
    for name, t in arrays.items():
        np.save(os.path.join(outdir, name + ".npy"), t.float().cpu().numpy())
    np.save(os.path.join(outdir, "disparity_frames.npy"), frames.astype(np.float32))


def time_steps(step, n, sync_all, torch):
    """n calls of step() between two CUDA events on the current stream, barrier + synchronize on both sides -> ms"""
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    sync_all()
    ev0.record()
    for k in range(n):
        step(k)
    ev1.record()
    sync_all()
    return ev0.elapsed_time(ev1)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=None,
                    help="timed steps, exactly (default: 200 for --workload K, 3 for M, 30 for nets)")
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--batch", type=int, default=64, help="frames per GPU per step (configs[1]: 64)")
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--workload", default="K", choices=["K", "M", "nets"],
                    help="K = configs[1] (default, the metric's configuration); M = configs[2] (Middlebury frame, maxDistance + occlusion "
                         "mask, row bands across the GPUs); nets = configs[3] (VPP -> RAFT-Stereo / PSMNet as device tensors)")
    ap.add_argument("--sustained-steps", type=int, default=0,
                    help="steps of an additional measurement reported beside the --steps one, e.g. 200 for >= 5 s (0 = off)")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--cpu-frames", type=int, default=0, help="frames in the cpu_baseline sample (default: one per core)")
    ap.add_argument("--dump-outputs", default=None, metavar="DIR",
                    help="write what the last timed step computed (rank 0's batch) to DIR/*.npy, float32, 52 MB")
    ap.add_argument("--cpu-worker", default=None, help=argparse.SUPPRESS)
    args = ap.parse_args()
    if args.steps is not None and args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and (args.workload != "K" or args.impl != "b200"):
        ap.error("--dump-outputs is implemented for --workload K --impl b200 only")
    if args.steps is None and args.workload == "K":
        args.steps = 200
    if args.cpu_worker:
        return cpu_worker_main(args.cpu_worker)
    if args.impl == "reference" and args.workload == "nets":
        import bench_nets
        return bench_nets.main(args, reference=True)
    if args.impl == "reference" and args.workload == "M":
        import bench_m
        return bench_m.main(args, reference=True)
    if args.impl == "reference":
        return run_reference_arm(args)
    if args.workload == "M":
        import bench_m
        return bench_m.main(args)
    if args.workload == "nets":
        import bench_nets
        return bench_nets.main(args)

    import ctypes
    import numpy as np
    import torch
    import torch.distributed as dist
    from vppstereo_b200 import _lib
    from vppstereo_b200.dist import PeerGather
    from vppstereo_b200.pipeline import VppRsgmPipeline

    rank = int(os.environ.get("RANK", "0")); world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    numa_cpus = None
    if os.environ.get("VPPB200_NUMA_BIND", "1") != "0":
        from vppstereo_b200.dist import bind_to_gpu_numa
        numa_cpus = bind_to_gpu_numa(local_rank)      # before the pinned staging buffers are allocated
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
    B = args.batch
    warmup = max(args.warmup, 3)

    # synthetic inputs: a few distinct frames tiled to the batch (generation is host work, not part of the path)
    left_h, right_h, hints_h = (torch.from_numpy(a).pin_memory() for a in bench_inputs(rank, B))
    left, right, hints = left_h.to(dev), right_h.to(dev), hints_h.to(dev)
    n_hints = float((hints_h > 0).sum()) / B
    pipe = VppRsgmPipeline(H, W, C, batch=B, dmax=D, device=dev)
    L = _lib.lib()
    for key, env in ((_lib.TUNE_SGM_BYTE_SUMS, "VPPB200_BYTE_SUMS"), (_lib.TUNE_SGM_CLUSTERS, "VPPB200_TEAMS"),
                     (_lib.TUNE_SGM_MAX_STRIP, "VPPB200_MAX_STRIP"), (_lib.TUNE_SGM_V_RED, "VPPB200_V_RED")):   # A/B experiments only
        if env in os.environ:
            _lib.set_tuning(key, int(os.environ[env]))

    # ---- the path's only exchange: every rank's disparities to every rank, once per step, on the copy engines
    # (dist.PeerGather: peer-mapped buffers, DMA over NVLink, stream memory operations; nothing on the SMs or on the compute
    # streams).  A consumer stream takes each gathered step and releases its buffer.
    pg = PeerGather((B, H, W), torch.float32, dev, depth=2) if world > 1 else None
    consumer = torch.cuda.Stream(dev) if world > 1 else None
    gstep = [0]
    if os.environ.get("VPPB200_CENSUS_FUSED", "1") == "0":    # experiment: pad_gray + census as two kernels
        _lib.set_tuning(_lib.TUNE_CENSUS_FUSED, 0)
    if os.environ.get("VPPB200_V_SPLIT", "1") == "0":         # experiment: single-plan v-sweeps
        _lib.set_tuning(_lib.TUNE_SGM_V_SPLIT, 0)
    gmode = os.environ.get("VPPB200_GATHER", "p2p")           # experiments: none | nccl | p2p (default)
    if pg is not None and gmode == "nccl":
        pg.available, pg.why = False, "forced by VPPB200_GATHER=nccl"

    def gather(out):
        if gmode == "none":
            return
        k = gstep[0]
        gstep[0] += 1
        pg.push(k, out)
        with torch.cuda.stream(consumer):
            pg.wait(k)
            pg.release(k)

    def step_device(_k=0):
        out = pipe.run_device(left, right, hints, inputs_ready=True)     # the inputs are resident in HBM (definition of `value`)
        if world > 1:
            gather(out)
        return out

    def sync_all():
        torch.cuda.synchronize(dev)
        if world > 1:
            dist.barrier()
            torch.cuda.synchronize(dev)

    for _ in range(warmup):
        step_device()
    sync_all()

    # ---- timed region 1: device-resident inputs, exactly --steps steps
    sampler = ClockSampler(local_rank); sampler.start()
    launches0 = _lib.launch_count()
    ms_total = time_steps(step_device, args.steps, sync_all, torch)
    launches = _lib.launch_count() - launches0
    if args.dump_outputs and rank == 0:
        # run_device returns pipe.disp; pipe.lv / pipe.rv hold the projected pair of the latest call (the steps below overwrite them)
        dump_outputs(args.dump_outputs, pipe.disp, pipe.lv, pipe.rv)
    # the same, sustained over >= 5 s (power and clocks settle): reported beside the --steps figure
    sus_n = args.sustained_steps if args.sustained_steps > args.steps else 0
    ms_sus = time_steps(step_device, sus_n, sync_all, torch) if sus_n else None
    clocks = sampler.summary()

    # ---- per-stage / per-kernel launch durations: a few more steps WITHOUT the cross-step overlap (VPP of step k+1 otherwise
    # shares the SMs with the sweeps of step k and stretches them), CUDA events at the stage boundaries of the stream
    L.vppb200_stage_timing(1)
    for k in range(5):
        pipe.run_device_serial(left, right, hints)
    sync_all()
    st_ms = (ctypes.c_float * len(STAGES))(); calls = ctypes.c_int(0)
    L.vppb200_stage_times(st_ms, ctypes.byref(calls))
    L.vppb200_stage_timing(0)
    stage_ms = {s: st_ms[i] / max(calls.value, 1) for i, s in enumerate(STAGES)}
    rsgm_ms = sum(stage_ms.values())

    # ---- VPP alone (same stream, CUDA events) for its own roofline line
    lv, rv = pipe.lv, pipe.rv

    def vpp_only(_k=0):
        lv.copy_(left); rv.copy_(right)
        rc = L.vppb200_vpp_scan_rnd(_lib.ptr(lv), _lib.ptr(rv), _lib.ptr(hints), W, H, C, 0, 3, 1, ctypes.c_double(0.4), ctypes.c_double(0.0),
                                    _lib.ptr(pipe.occ), 0, 1, 1, None, None, ctypes.c_uint64(7), None, _lib.ptr(pipe.ws_vpp),
                                    ctypes.c_size_t(pipe.ws_vpp.numel()), B, _lib.stream_ptr(dev))
        _lib.check(rc, "vpp")
    vpp_only(); torch.cuda.synchronize(dev)
    vpp_ms = time_steps(vpp_only, 10, lambda: torch.cuda.synchronize(dev), torch) / 10

    # ---- timed region 2: end to end through the host-buffer API
    # (submit_host / collect: every step copies its inputs from pinned host memory and its disparities back to the host; the
    #  copies of neighbouring steps overlap this step's kernels on separate streams, up to three batches in flight; at N > 1
    #  the same per-step gather as above rides along: exactly n batches are submitted, gathered and collected in the region)
    hook = gather if world > 1 else None

    def e2e_run(n):
        ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        sync_all()
        ev0.record()
        pending, res = [], None
        for k in range(n):
            pending.append(pipe.submit_host(left_h, right_h, hints_h, on_computed=hook))
            if len(pending) == pipe.host_depth:
                res = pipe.collect(pending.pop(0))
        while pending:
            res = pipe.collect(pending.pop(0))
        ev1.record()
        sync_all()
        return ev0.elapsed_time(ev1), res
    e2e_run(3)
    e2e_ms, res = e2e_run(args.steps)
    e2e_sus_ms = e2e_run(sus_n)[0] if sus_n else None
    check_val = float(res[0].mean())

    # ---- single-frame latency (test.py runs batch 1): host frame in -> host disparity out, one frame at a time
    lat_ms = None
    if rank == 0:
        p1 = VppRsgmPipeline(H, W, C, batch=1, dmax=D, device=dev)
        l1, r1, g1 = left_h[:1].clone().pin_memory(), right_h[:1].clone().pin_memory(), hints_h[:1].clone().pin_memory()
        for _ in range(3):
            p1.run_host(l1, r1, g1)
        ts = []
        for _ in range(20):
            t0 = time.perf_counter(); p1.run_host(l1, r1, g1); ts.append((time.perf_counter() - t0) * 1e3)
        lat_ms = sorted(ts)[len(ts) // 2]
        p1.close()

    # ---- parity probe: the timed pipeline object on rank 0's inputs with a fixed pattern seed, against oracle-derived digests
    probe = None
    if rank == 0:
        probe = assert_parity_probe(parity_probe(B, pipe=pipe, tensors=(left, right, hints)), B)

    # max over ranks
    vals = [ms_total, e2e_ms, ms_sus or 0.0, e2e_sus_ms or 0.0]
    t = torch.tensor(vals, dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    ms_total, e2e_ms, ms_sus_m, e2e_sus_m = (float(x) for x in t)

    cpu_baseline = None
    if rank == 0 and world == 1 and not args.no_cpu_baseline:
        try:
            cb = CpuBaseline()
            f, dt, per = cb.step(0, frames=args.cpu_frames or cb.cores)
            cb.close()
            cpu_baseline = {"value": f / dt, "unit": "pairs/s", "cores": cb.cores, "kind": cb.kind,
                            "sample": cb.describe(f, 1), "single_frame_latency_s": per}
        except Exception as e:      # the baseline is reported, never required for the GPU number
            cpu_baseline = {"value": None, "unit": "pairs/s", "cores": 0, "kind": "unavailable", "sample": repr(e)}

    if rank == 0:
        peak, peak_src = measured_peak()
        frames_total = world * B * args.steps
        v_s = 0.5 * (stage_ms["sgm_v_down"] + stage_ms["sgm_v_up"]) * 1e-3          # average launch of the dominant kernel (+ its P2 table kernel)
        achieved = ALG_BYTES_VSWEEP * B / v_s / 1e9
        agg_s = sum(stage_ms[k] for k in ("sgm_h_fwd", "sgm_v_down", "sgm_v_up", "sgm_h_bwd_wta")) * 1e-3
        agg_achieved = ALG_BYTES_AGG * B / agg_s / 1e9
        vpp_bytes = (ALG_BYTES_VPP + C * 9 * n_hints) * B
        traffic, traffic_src = ncu_traffic()
        gbs = lambda nbytes, ms: nbytes / (ms * 1e-3) / 1e9

        def roof(nbytes, ms, what):
            return {"what": what, "achieved": gbs(nbytes, ms), "peak": peak, "unit": "GB/s", "frac": gbs(nbytes, ms) / peak, "ms": ms,
                    "algorithmic_bytes": nbytes}
        line = {
            "metric": METRIC, "value": frames_total / (ms_total * 1e-3), "unit": "pairs/s", "n_gpus": world, "steps": args.steps,
            "warmup": warmup, "ms_per_step": ms_total / args.steps, "higher_is_better": True, "scaling": "weak",
            "vs_baseline": None, "dtype": "u16", "data": "synthetic",
            "config": {"workload": "configs[1]: KITTI-shape 1242x375x3 pairs, LiDAR-like 5% hints, VPP rnd 3x3 blending 0.4 + rSGM D=192, batch 64 per GPU",
                       "batch_per_gpu": B, "frames_per_step": world * B, "l2": "inputs per step (298 MB) and cost volumes (17.7 GB) exceed the 126 MB L2",
                       "collective": (f"per step, every rank's disparities to every rank ({B * H * W * 4 * (world - 1)} B out per rank): "
                                      f"{'copy engines over peer-mapped memory (dist.PeerGather), off the SMs and off the compute streams' if pg.available else 'NCCL all_gather (peer mapping unavailable: ' + pg.why + ')'}; "
                                      "inside both timed regions; configs[4]'s 1024-frame sequence = 16/N such steps per rank") if world > 1 else "none",
                       "host_affinity": f"GPU-local NUMA cores ({len(numa_cpus)})" if numa_cpus else "unchanged",
                       "overlap": "three-phase software pipeline across steps on three streams: front(k+1) = VPP + pad/gray/census/cost volume, main(k) = SGM sweeps + WTA, tail(k-1) = median..fills; two buffer sets; right-image branches on side streams",
                       "stage_ms_per_step_serial": {k: round(v, 3) for k, v in stage_ms.items()}, "vpp_ms_per_step": round(vpp_ms, 3),
                       "rsgm_fps": B / (rsgm_ms * 1e-3), "vpp_pairs_per_s": B / (vpp_ms * 1e-3), "check_mean_disp": check_val,
                       "latency_batch1_ms": lat_ms,
                       "latency_note": "one K-shape frame, pinned host in -> host out through VppRsgmPipeline(batch=1).run_host, median of 20; the reference needs cpu_baseline.single_frame_latency_s per frame on one core"},
            "sustained": None if not sus_n else {"steps": sus_n, "value": world * B * sus_n / (ms_sus_m * 1e-3), "ms_per_step": ms_sus_m / sus_n,
                                                 "e2e_value": world * B * sus_n / (e2e_sus_m * 1e-3), "seconds": ms_sus_m * 1e-3,
                                                 "what": "the same two timed regions run for --sustained-steps steps (>= 5 s each)"},
            "roofline": {"bound": "hbm", "kernel": "sgm_v2_kernel (v-sweep: paths r1+r2+r3 of one pass over the batch; 2 sweeps per step, each 36 frames x 8 CTAs + 28 frames x 10 CTAs = two cooperative launches timed together)",
                         "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak,
                         "traffic": traffic if B == 64 else None, "traffic_source": traffic_src, "peak_source": peak_src,
                         "algorithmic_bytes_per_launch": ALG_BYTES_VSWEEP * B, "launch_ms": v_s * 1e3},
            # the other kernels of the step against the same peak, each on SURVEY.md 8(d)'s bytes for its row
            "roofline_aggregate_8_paths": roof(ALG_BYTES_AGG * B, agg_s * 1e3, "h_fwd + v_down + v_up + h_bwd(+WTA) vs SURVEY 8d aggregate bytes (4WHD+WH)"),
            "roofline_vpp": roof(vpp_bytes, vpp_ms, "VPP rnd: images in/out + hints + mask + pattern draws (SURVEY 8d)"),
            "roofline_census": roof(2 * (H * W * C + 4 * WP * HP) * B, stage_ms["census"],
                                    "pad + RGB2GRAY + census 5x5 of both images in one kernel each (TMA-staged row bands): the uint8 image in, 4 bytes out per padded pixel"),
            "roofline_cost_volume": roof((8 * WP * HP + WP * HP * D) * B, stage_ms["cost_volume"], "Hamming volume: two census images in, uint8 volume out"),
            "roofline_h_fwd": roof(3 * WP * HP * D * B, stage_ms["sgm_h_fwd"], "h-sweep fwd: uint8 costs in, uint16 S out"),
            "roofline_h_bwd_wta": roof((3 * WP * HP * D + 8 * WP * HP) * B, stage_ms["sgm_h_bwd_wta"], "h-sweep bwd + WTA: costs + S in, two disparity maps out"),
            "e2e": {"value": frames_total / (e2e_ms * 1e-3), "unit": "pairs/s",
                    "h2d_bytes_per_step": int(left_h.numel() + right_h.numel() + hints_h.numel() * 4),
                    "d2h_bytes_per_step": int(B * H * W * 4)},
            "gpu_launches": int(launches),
            "parity_probe": probe,
            "clocks": clocks,
            "cpu_baseline": cpu_baseline,
        }
        print(json.dumps(line), flush=True)
    if world > 1:
        pg.close()
        dist.destroy_process_group()


if __name__ == "__main__":
    sys.dont_write_bytecode = True        # the benchmark writes nothing into the tree it runs from (which may be read-only)
    main()
