"""df_allreduce_fwd (one-shot, peer memory) against torch.distributed.all_reduce (NCCL), graph-timed, one process per GPU:

    python -m torch.distributed.run --nproc_per_node N tools/bench_allreduce.py [--iters 50] [--out FILE]

Sizes: the SDXL 1024^2 activations of the three levels (320 / 640 / 1280 channels at 128^2 / 64^2 / 32^2 latents, one CFG
branch: 10.5 / 5.2 / 2.6 MB) and the 3840^2 level-0 activation (480^2 x 320: 147 MB).  Each size is all-reduced `iters` times
inside one CUDA graph; the best of 5 replays is reported as us per call and as algorithm bandwidth (bytes / time).  GB/s of
NVLink traffic per rank is (n-1) x that for the one-shot kernel.  Needs one GPU per rank: ranks sharing a GPU would measure
time slicing."""
import argparse
import json
import os
import sys

import torch
from torch import distributed as dist

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))

SIZES = (("sdxl1024_l0", 128 * 128, 320), ("sdxl1024_l1", 64 * 64, 640), ("sdxl1024_l2", 32 * 32, 1280),
         ("sdxl3840_l0", 480 * 480, 320))


def _time(fn, iters):
    g = torch.cuda.CUDAGraph()
    with torch.cuda.graph(g):
        for _ in range(iters):
            fn()
    g.replay()
    torch.cuda.synchronize()
    best = float("inf")
    for _ in range(5):
        dist.barrier()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        g.replay()
        e1.record()
        e1.synchronize()
        best = min(best, e0.elapsed_time(e1) * 1e3 / iters)
    return best


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--iters", type=int, default=50)
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    from distrifuser_b200.utils import DistriConfig, PatchParallelismCommManager
    cfg = DistriConfig(do_classifier_free_guidance=False, parallelism="tensor", use_cuda_graph=False)
    n = cfg.n_device_per_batch
    if torch.cuda.device_count() < n:
        raise SystemExit(f"{n} ranks on {torch.cuda.device_count()} GPUs: not measured (needs one GPU per rank)")
    cm = PatchParallelismCommManager(cfg)
    cm.register_allreduce(max(r * c * 2 for _, r, c in SIZES))   # one site: every call is the next in sequence
    cm.register_output(1, 4, 8, 8)
    cm.create_buffer()
    rows = []
    for name, r, c in SIZES:
        x = torch.randn(r, c, device=cfg.device).half()
        out = torch.empty_like(x)
        nccl = x.clone()

        def ours():
            cm.step_begin(0)
            cm.all_reduce(0, x, out)
        us_ours = _time(ours, a.iters)
        us_nccl = _time(lambda: dist.all_reduce(nccl), a.iters)
        nbytes = r * c * 2
        rows.append(dict(size=name, bytes=nbytes, n=n, one_shot_us=us_ours, one_shot_GBps=nbytes / us_ours / 1e3,
                         nccl_us=us_nccl, nccl_GBps=nbytes / us_nccl / 1e3))
    if cfg.rank == 0:
        gpu = torch.cuda.get_device_name()
        import subprocess
        power = subprocess.run(["nvidia-smi", "--query-gpu=power.limit", "--format=csv,noheader", "-i", "0"],
                               capture_output=True, text=True).stdout.strip()
        res = dict(gpu=gpu, power_limit=power, iters=a.iters, results=rows)
        print(json.dumps(res))
        if a.out:
            with open(a.out, "w") as f:
                json.dump(res, f, indent=1)
    dist.barrier()
    cm.close()
    dist.destroy_process_group()


if __name__ == "__main__":
    main()
