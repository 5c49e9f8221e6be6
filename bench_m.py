"""bench.py --workload M: BASELINE configs[2] -- "Middlebury full-res 2880x1988, histogram-based pattern with occlusion handling".

Per frame (test.py:154-176 with --maskocc --colormethod maxDistance, then rsgm): 5 % random hints ->
filter.occlusion_heuristic (occlusion mask) -> vpp(method="maxDistance", wsizeAgg 64x3, g_occ=mask) -> compute_rsgm(D=192), all on
CUDA tensors through the reference-shaped front-ends (no host hop between the stages).

How an oversized frame spreads over the GPUs of a box (SURVEY.md 8e, DESIGN.md 6):
  * a STREAM of frames shards by frame: every rank runs whole frames (an M frame needs ~8 GB of workspace, 180 GB hold a batch) --
    this is what `value` measures at N GPUs (weak scaling, batch of `--batch` frames per rank and step), no collective but the
    gather of the disparities (dist.PeerGather);
  * one frame's rnd projection, census and cost volume split exactly by row bands (dist.vpp_rnd_banded, dist.band_with_halo;
    tests/test_gpu_bands.py) -- measured here as `bands` at N > 1 for the single-frame case;
  * maxDistance does not split by rows (its windows read the current images); its colour channels are independent, but a
    one-channel scan takes as long as the three-channel one (`max_dist_channels`: the scan is bound by the depth of the hint
    dependency chain, the channels already run side by side on one GPU), so sharding it 3 ways buys nothing: replicas win;
  * the SGM sweeps of one frame chain through all rows; see DESIGN.md 6 for the band pipeline.
One JSON line (rank 0)."""
import json
import os
import sys
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
H, W, C, D = 1988, 2880, 3, 192
HP, WP = 2000, 2880
METRIC = "Middlebury-shape 2880x1988 pairs/s: occlusion mask + VPP maxDistance 64x3 + rSGM D=192, 5% hints"


def _cpu_frame(f):
    """the reference's own code on one core: occlusion_heuristic + Cython maxDistance scan + compute_rsgm of one M frame"""
    import numpy as np
    from oracle import ref
    from vppstereo_b200 import synth
    r = ref.load()
    p = synth.make_pair(f, shape="M", hints="random")
    t0 = time.perf_counter()
    occ = r.filter.occlusion_heuristic(p["hints"])[1]
    t1 = time.perf_counter()
    l, rr = p["left"].copy(), p["right"].copy()
    r.vpp_core_opt.virtual_projection_scan_max_dist(l, rr, p["hints"], W, H, 3, False, 3, 64, 3, 1, 0.4, 0.0,
                                                    (occ != 0).astype(np.uint8), False, True)
    t2 = time.perf_counter()
    r.rsgm.compute_rsgm(p["left"], l, rr, dmax=D)
    t3 = time.perf_counter()
    return {"occlusion_s": t1 - t0, "vpp_max_dist_s": t2 - t1, "rsgm_s": t3 - t2, "total_s": t3 - t0}


def main(args, reference=False):
    if getattr(args, "cpu_m_worker", False) or reference:
        # the reference arm: one frame per host core, frame-parallel (each worker is this script with --cpu-m-worker)
        import subprocess
        rank = int(os.environ.get("RANK", "0"))
        if rank != 0:
            return
        cores = min(len(os.sched_getaffinity(0)), 16)
        env = dict(os.environ, OMP_NUM_THREADS="1", CUDA_VISIBLE_DEVICES="", NUMBA_NUM_THREADS="1")
        t0 = time.perf_counter()
        procs = [subprocess.Popen([sys.executable, os.path.abspath(__file__), "--cpu-frame", str(100 + i)], stdout=subprocess.PIPE, text=True,
                                  env=env, cwd=ROOT) for i in range(cores)]
        outs = [json.loads(p.communicate()[0].strip().splitlines()[-1]) for p in procs]
        wall = time.perf_counter() - t0
        v = cores / wall
        line = {"impl": "reference", "metric": METRIC, "value": v, "unit": "pairs/s", "n_gpus": args.gpus, "steps": 1, "warmup": 0,
                "ms_per_step": 1e3 * wall, "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "u16", "data": "synthetic",
                "config": {"workload": "configs[2]: M-shape frames, reference code (numba occlusion_heuristic, Cython scan_max_dist, SSE rSGM), one frame per core",
                           "per_frame_seconds_mean": {k: sum(o[k] for o in outs) / len(outs) for k in outs[0]}},
                "cpu_baseline": {"value": v, "unit": "pairs/s", "cores": cores, "kind": "reference", "sample": f"{cores} M frames, one per single-threaded worker"},
                "e2e": {"value": v, "unit": "pairs/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
        print(json.dumps(line), flush=True)
        return

    import numpy as np
    import torch
    import torch.distributed as dist
    import bench
    from vppstereo_b200 import _lib, filter as vfilter, rsgm, synth, vpp_standalone
    from vppstereo_b200 import dist as vd
    rank = int(os.environ.get("RANK", "0")); world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
    # frames per rank and step.  The projection is bound by the depth of its hint dependency chain (~0.27 s for one frame and
    # 0.30 s for twelve; 24 / 48 / 72 frames: 0.39 / 0.58 / 0.77 s: the resident row warps saturate at ~8 ms per added frame), so
    # a step projects all B frames in one call; the matcher then runs in chunks of CHUNK frames
    # (8 M frames = 8 teams of 18 SMs in the v-sweeps, ~8.5 GB of workspace each)
    B = args.batch if args.batch != 64 else 48
    CHUNK = 8
    steps = args.steps if args.steps is not None else 3
    uniq = [synth.make_pair(rank * 100 + f, shape="M", hints="random") for f in range(2)]
    idx = [i % 2 for i in range(B)]
    host = tuple(torch.from_numpy(np.stack([uniq[i][k] for i in idx])).pin_memory() for k in ("left", "right", "hints"))
    left, right, hints = (t.to(dev) for t in host)
    out_h = torch.empty((B, H, W), dtype=torch.float32).pin_memory()
    pg = vd.PeerGather((B, H, W), torch.float32, dev, depth=2) if world > 1 else None
    kstep = [0]
    ev = {k: [torch.cuda.Event(enable_timing=True) for _ in range(2)] for k in ("occ", "vpp", "rsgm")}

    def one_step(l, r, g, timed=False):
        if timed: ev["occ"][0].record()
        mask = vfilter.occlusion_heuristic(g)[1]                                       # test.py:154
        if timed: ev["occ"][1].record(); ev["vpp"][0].record()
        lv, rv = vpp_standalone.vpp(l, r, g, wsize=3, wsizeAgg_x=64, wsizeAgg_y=3, blending=0.4, method="maxDistance", g_occ=mask)
        if timed: ev["vpp"][1].record(); ev["rsgm"][0].record()
        n = l.shape[0]
        d = torch.empty((n, H, W), dtype=torch.float32, device=dev) if n > CHUNK else None
        for a in range(0, n, CHUNK):
            part = rsgm.compute_rsgm(l[a:a + CHUNK], lv[a:a + CHUNK], rv[a:a + CHUNK], dmax=D)
            if d is None:
                d = part
            else:
                d[a:a + CHUNK].copy_(part)
        if timed: ev["rsgm"][1].record()
        if pg is not None:
            k = kstep[0]; kstep[0] += 1
            pg.push(k, d); pg.wait(k); pg.release(k)
        return d

    def sync_all():
        torch.cuda.synchronize(dev)
        if world > 1:
            dist.barrier(); torch.cuda.synchronize(dev)

    one_step(left, right, hints); one_step(left, right, hints)
    sync_all()
    launches0 = _lib.launch_count()
    ms = bench.time_steps(lambda k: one_step(left, right, hints), steps, sync_all, torch)
    launches = _lib.launch_count() - launches0
    # end to end: pinned host frames in, host disparities out, every step
    def e2e_step(k):
        l, r, g = (t.to(dev, non_blocking=True) for t in host)
        out_h.copy_(one_step(l, r, g), non_blocking=True)
    e2e_step(0)
    e2e_ms = bench.time_steps(e2e_step, steps, sync_all, torch)
    # stage split of one batch and the single-frame latency
    one_step(left, right, hints, timed=True); torch.cuda.synchronize(dev)
    stage_ms = {k: ev[k][0].elapsed_time(ev[k][1]) for k in ev}
    l1, r1, g1 = left[:1].contiguous(), right[:1].contiguous(), hints[:1].contiguous()
    B_save, pg_save = B, pg
    pg = None
    one_step(l1, r1, g1)
    one_step(l1, r1, g1, timed=True); torch.cuda.synchronize(dev)
    lat_ms = {k: ev[k][0].elapsed_time(ev[k][1]) for k in ev}
    # maxDistance: one colour channel alone vs all three (is a 3-way channel split worth anything?)
    gray_l, gray_r = l1[..., :1].contiguous(), r1[..., :1].contiguous()
    def md(lc, rc):
        torch.cuda.synchronize(dev); t0 = time.perf_counter()
        vpp_standalone.vpp(lc, rc, g1, wsize=3, wsizeAgg_x=64, wsizeAgg_y=3, blending=0.4, method="maxDistance")
        torch.cuda.synchronize(dev); return (time.perf_counter() - t0) * 1e3
    md(gray_l, gray_r); md(l1, r1)
    md_ms = {"one_channel_ms": md(gray_l, gray_r), "three_channels_ms": md(l1, r1)}
    # single oversized frame, row bands of the stages that split exactly (N > 1): rnd projection across the ranks
    bands = None
    if world > 1:
        pat_seed = 5
        vd.vpp_rnd_banded(l1[0], r1[0], g1[0], seed=pat_seed)
        sync_all(); t0 = time.perf_counter()
        vd.vpp_rnd_banded(l1[0], r1[0], g1[0], seed=pat_seed)
        sync_all(); t_b = (time.perf_counter() - t0) * 1e3
        sync_all(); t0 = time.perf_counter()
        vpp_standalone.vpp(l1[0], r1[0], g1[0], seed=pat_seed)
        sync_all(); t_1 = (time.perf_counter() - t0) * 1e3
        bands = {"vpp_rnd_one_frame_banded_ms": t_b, "vpp_rnd_one_frame_single_gpu_ms": t_1,
                 "note": "exact (tests/test_gpu_bands.py); the gather of the bands costs more than the 5 % hint projection saves at this size"}
    # one frame's aggregation split into one row band per rank (vppstereo_b200.banded: exact, the row state of the vertical sweeps
    # travels over NVLink): latency of a single frame, and frames per second when consecutive frames are in flight on alternating
    # streams -- against the unsplit compute_rsgm of one frame at a time on one GPU
    banded = None
    if world > 1:
        from vppstereo_b200.banded import BandedRsgmDist
        pb = synth.make_pair(7, shape="M", hints="random")             # the SAME frame on every rank (the batch above is per rank)
        l1, r1, g1 = (torch.from_numpy(pb[k_])[None].to(dev) for k_ in ("left", "right", "hints"))
        lv1, rv1 = vpp_standalone.vpp(l1[0], r1[0], g1[0], wsize=3, wsizeAgg_x=64, wsizeAgg_y=3, blending=0.4, method="maxDistance")
        lanes = [BandedRsgmDist(H, W, C, dmax=D, device=dev) for _ in range(3)]
        streams = [torch.cuda.Stream(dev) for _ in lanes]
        ref = rsgm.compute_rsgm(l1[0], lv1, rv1, dmax=D)
        got = lanes[0].compute(l1[0], lv1, rv1)
        same = bool((got.view(torch.int32) == ref.view(torch.int32)).all())
        def t_loop(fn, n):
            sync_all(); t0 = time.perf_counter()
            for k in range(n):
                fn(k)
            sync_all(); return (time.perf_counter() - t0) * 1e3 / n
        def banded_sync(k):
            lanes[0].compute(l1[0], lv1, rv1); torch.cuda.synchronize(dev)
        def banded_pipe(k):
            with torch.cuda.stream(streams[k % 3]):
                lanes[k % 3].compute(l1[0], lv1, rv1)
        def unsplit_sync(k):
            rsgm.compute_rsgm(l1[0], lv1, rv1, dmax=D); torch.cuda.synchronize(dev)
        def unsplit_stream(k):
            rsgm.compute_rsgm(l1[0], lv1, rv1, dmax=D)
        banded_sync(0); banded_pipe(0); banded_pipe(1); banded_pipe(2); unsplit_sync(0)
        banded = {"bit_exact_vs_unsplit": same, "bands": lanes[0].bands,
                  "volume_bytes_per_gpu": int(lanes[0].band[1] * lanes[0].vol_row_bytes * 3), "volume_bytes_unsplit": int(lanes[0].Hp * lanes[0].vol_row_bytes * 3),
                  "row_state_bytes": int(lanes[0].state_words * 4),
                  "latency_ms_banded": t_loop(banded_sync, 10), "latency_ms_unsplit_one_gpu": t_loop(unsplit_sync, 10),
                  "ms_per_frame_banded_3_in_flight": t_loop(banded_pipe, 30), "ms_per_frame_unsplit_one_gpu_stream": t_loop(unsplit_stream, 30),
                  "note": "compute_rsgm only (the projection is per frame, not banded); frames of a stream shard by frame instead (`value`)"}
        for b_ in lanes:
            b_.close()
    pg = pg_save
    t = torch.tensor([ms, e2e_ms], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    ms, e2e_ms = float(t[0]), float(t[1])

    cpu_baseline = None
    if rank == 0 and world == 1 and not args.no_cpu_baseline:
        try:
            import subprocess
            env = dict(os.environ, OMP_NUM_THREADS="1", CUDA_VISIBLE_DEVICES="", NUMBA_NUM_THREADS="1")
            o = subprocess.run([sys.executable, os.path.abspath(__file__), "--cpu-frame", "100"], capture_output=True, text=True, env=env, cwd=ROOT,
                               timeout=900)
            per = json.loads(o.stdout.strip().splitlines()[-1])
            cpu_baseline = {"value": 1.0 / per["total_s"], "unit": "pairs/s", "cores": 1, "kind": "reference",
                            "sample": "one M frame on one core: numba occlusion_heuristic + Cython scan_max_dist + SSE rSGM (oracle/_ref)", "per_frame_seconds": per}
        except Exception as e:
            cpu_baseline = {"value": None, "unit": "pairs/s", "cores": 0, "kind": "unavailable", "sample": repr(e)}

    if rank == 0:
        peak, peak_src = bench.measured_peak()
        frames = world * B * steps
        alg_rsgm = (2 * 2 * WP * HP * D + 4 * WP * HP * 4) * B           # SURVEY 8d "fused" row scaled to M: S written and read once per pass
        alg_vpp = (4 * H * W * C + 4 * H * W + H * W) * B
        line = {
            "metric": METRIC, "value": frames / (ms * 1e-3), "unit": "pairs/s", "n_gpus": world, "steps": steps, "warmup": 2,
            "ms_per_step": ms / steps, "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "u16", "data": "synthetic",
            "config": {"workload": f"configs[2]: Middlebury-shape 2880x1988x3 pairs, 5% random hints, occlusion_heuristic mask + VPP maxDistance 64x3 blending 0.4 + rSGM D=192, batch {B} per GPU, frames sharded over the GPUs",
                       "batch_per_gpu": B, "frames_per_step": world * B,
                       "stage_ms_per_batch": {k: round(v, 2) for k, v in stage_ms.items()},
                       "single_frame_latency_ms": {k: round(v, 2) for k, v in lat_ms.items()},
                       "max_dist_channels": md_ms, "bands": bands, "banded_rsgm": banded,
                       "collective": "none" if world == 1 else f"per step, copy-engine gather of the disparities (PeerGather available={pg.available})"},
            "roofline": {"bound": "hbm", "kernel": "compute_rsgm at M (the projection is bound by the hint dependency chain, not by bandwidth: DESIGN.md 4)",
                         "achieved": alg_rsgm / (stage_ms["rsgm"] * 1e-3) / 1e9, "peak": peak, "unit": "GB/s",
                         "frac": alg_rsgm / (stage_ms["rsgm"] * 1e-3) / 1e9 / peak, "traffic": None, "peak_source": peak_src,
                         "algorithmic_bytes": alg_rsgm},
            "roofline_vpp_max_dist": {"achieved": alg_vpp / (stage_ms["vpp"] * 1e-3) / 1e9, "peak": peak, "unit": "GB/s",
                                      "frac": alg_vpp / (stage_ms["vpp"] * 1e-3) / 1e9 / peak, "algorithmic_bytes": alg_vpp},
            "e2e": {"value": frames / (e2e_ms * 1e-3), "unit": "pairs/s", "h2d_bytes_per_step": int(B * (2 * H * W * C + 4 * H * W)),
                    "d2h_bytes_per_step": int(B * H * W * 4)},
            "gpu_launches": int(launches), "cpu_baseline": cpu_baseline,
        }
        print(json.dumps(line), flush=True)
    if world > 1:
        pg.close()
        dist.destroy_process_group()


if __name__ == "__main__":
    sys.path.insert(0, ROOT)
    if len(sys.argv) >= 3 and sys.argv[1] == "--cpu-frame":
        print(json.dumps(_cpu_frame(int(sys.argv[2]))), flush=True)
