"""Worker of tests/test_gpu_guided.py::test_guided_one_band_per_rank_two_gpus: guided matching with one band per rank; the banded
result on every rank == the unsplit guided compute_rsgm on that rank's own GPU, for several frames in a row (mailboxes reused)."""
import os
import sys

import numpy as np
import torch
import torch.distributed as dist

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)


def main():
    outdir = sys.argv[1]
    rank, local = int(os.environ["RANK"]), int(os.environ["LOCAL_RANK"])
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    dist.init_process_group("nccl", device_id=dev)
    from vppstereo_b200 import rsgm, synth
    from vppstereo_b200.banded import BandedRsgmDist
    msgs = []
    for shape, D in (((96, 330), 64), ((300, 700), 192)):
        b = BandedRsgmDist(shape[0], shape[1], 3, dmax=D, device=dev)
        for f in range(4):
            p = synth.make_pair(60 + f, shape=shape, hints="random", density=0.3)
            valid = (p["hints"] > 0).astype(np.float32)
            valid[::5, ::3] = 1.0
            l, r = torch.from_numpy(p["left"]).to(dev), torch.from_numpy(p["right"]).to(dev)
            h, v = torch.from_numpy(p["hints"]).to(dev), torch.from_numpy(valid).to(dev)
            got = b.compute(l, l, r, hints=h, validhints=v)
            want = rsgm.compute_rsgm(l, l, r, hints=h, validhints=v, dmax=D)
            torch.cuda.synchronize(dev)
            a, w = got.cpu().numpy().view(np.uint32), want.cpu().numpy().view(np.uint32)
            if not np.array_equal(a, w):
                msgs.append(f"{shape} D={D} frame {f}: {(a != w).sum()} of {a.size} values differ")
        dist.barrier()
        b.close()
    with open(os.path.join(outdir, f"rank{rank}.txt"), "w") as fh:
        fh.write(("FAIL\n" if msgs else "OK\n") + "\n".join(msgs) + "\n")
    dist.destroy_process_group()


if __name__ == "__main__":
    main()
