"""SDXL ms/image with parallelism="tensor" and "patch" in the same call, alternating, same GPUs and CFG layout:

    python -m torch.distributed.run --nproc_per_node N tools/bench_tp.py [--size 1024] [--steps 50] [--reps 2]
                                                                      [--no-split] [--out FILE]

Random-weight SDXL UNet, synthetic latent pipeline, CUDA graphs (the configuration of bench.py).  Also reports the summed
df_allreduce_fwd kernel time of one tensor-parallel UNet call (CUDA events from the _lib.PROFILE hooks, eager call), the
arena bytes of both modes, and the GPU name and power limit read in the same run.  Needs one GPU per rank."""
import argparse
import json
import os
import subprocess
import sys
import time

import torch
from torch import distributed as dist

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--size", type=int, default=1024)
    ap.add_argument("--steps", type=int, default=50)
    ap.add_argument("--reps", type=int, default=2)
    ap.add_argument("--no-split", action="store_true")
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    from distrifuser_b200 import _lib
    from distrifuser_b200.pipelines import DistriSDXLPipeline
    from distrifuser_b200.utils import DistriConfig
    pipes = {}
    for par in ("tensor", "patch"):
        cfg = DistriConfig(height=a.size, width=a.size, split_batch=not a.no_split, parallelism=par)
        if torch.cuda.device_count() < cfg.world_size:
            raise SystemExit(f"{cfg.world_size} ranks on {torch.cuda.device_count()} GPUs: not measured")
        pipes[par] = DistriSDXLPipeline.from_synthetic(cfg)
    times = {p: [] for p in pipes}
    for _ in range(a.reps):
        for par, pipe in pipes.items():
            dist.barrier()
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            pipe(prompt="", num_inference_steps=a.steps, generator=torch.Generator().manual_seed(0))
            torch.cuda.synchronize()
            times[par].append((time.perf_counter() - t0) * 1e3)
    # all-reduce kernel time of one eager tensor-parallel UNet call
    unet, si = pipes["tensor"].pipeline.unet, pipes["tensor"].static_inputs
    _lib.PROFILE = []
    with torch.no_grad():
        unet.set_counter(0)
        unet(**si, return_dict=False, record=True)
    torch.cuda.synchronize()
    ar = [e for e in _lib.PROFILE if e["kind"] == "allreduce"]
    ar_ms = sum(e["start"].elapsed_time(e["end"]) for e in ar)
    _lib.PROFILE = None
    if dist.get_rank() == 0:
        power = subprocess.run(["nvidia-smi", "--query-gpu=power.limit", "--format=csv,noheader", "-i", "0"],
                               capture_output=True, text=True).stdout.strip()
        res = dict(gpu=torch.cuda.get_device_name(), power_limit=power, world=dist.get_world_size(), size=a.size,
                   steps=a.steps, split_batch=not a.no_split, ms_per_image={p: min(t) for p, t in times.items()},
                   all_ms=times, allreduce_sites=len(ar), allreduce_ms_per_step=ar_ms,
                   arena_bytes={p: pipes[p].comm_manager._arena_bytes for p in pipes})
        print(json.dumps(res))
        if a.out:
            with open(a.out, "w") as f:
                json.dump(res, f, indent=1)
    dist.barrier()
    for p in pipes.values():
        p.comm_manager.close()
    dist.destroy_process_group()


if __name__ == "__main__":
    main()
