"""TEST INFRASTRUCTURE (oracle).  Generates tests/golden/*.pt by EXECUTING THE UNMODIFIED REFERENCE
(/root/reference/distrifuser/modules/pp/*.py, models/distri_sdxl_unet_pp.py, utils.py:112-199) on CPU under
gloo, through the diffusers stub.  Runs only in the build container (the reference tree does not exist on
the GPU box); the vectors it writes are committed.

    python -m oracle.make_golden [--only chain|unet] [--case NAME]
"""
import argparse
import os
import sys
import time

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "oracle", "diffusers_stub"))

from oracle import harness, workloads  # noqa: E402

GOLDEN = os.path.join(ROOT, "tests", "golden")
MAX_VALUE_BYTES = 800_000          # keeps every fixture under 1 MB


def _sampled(outs, seed=0):
    """outs[rank][step] = tuple of tensors.  When the values exceed MAX_VALUE_BYTES, keeps the same fixed, seeded sample of
    flat positions of every tensor of a given size (every rank, step and stage stays covered) and records the full shapes;
    tests/test_oracle_vs_golden.py compares the oracle at those positions."""
    flat = [t for per_rank in outs for per_step in per_rank for t in per_step]
    if sum(4 * t.numel() for t in flat) <= MAX_VALUE_BYTES:
        return {"outs": outs}
    keep = MAX_VALUE_BYTES // (4 * len(flat))
    g = torch.Generator().manual_seed(seed)
    index = {n: torch.randperm(n, generator=g)[:keep].sort().values for n in sorted({t.numel() for t in flat})}
    pick = lambda t: t.reshape(-1)[index[t.numel()]].clone()
    return {"outs": [[tuple(pick(t) for t in per_step) for per_step in per_rank] for per_rank in outs],
            "shapes": [[tuple(tuple(t.shape) for t in per_step) for per_step in per_rank] for per_rank in outs],
            "index": index}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--only", choices=["chain", "unet"], default=None)
    ap.add_argument("--case", default=None)
    a = ap.parse_args()
    os.makedirs(GOLDEN, exist_ok=True)
    if a.only in (None, "chain"):
        for case in workloads.CHAIN_CASES:
            if a.case and case.name != a.case:
                continue
            t0 = time.time()
            outs = harness.run_chain(case, impl="reference")
            torch.save({"case": case.__dict__, **_sampled(outs), "source": "reference modules, gloo, fp32"},
                       os.path.join(GOLDEN, f"{case.name}.pt"))
            print(f"{case.name}: {time.time() - t0:.1f}s", flush=True)
    if a.only in (None, "unet"):
        for case in workloads.UNET_CASES:
            if a.case and case.name != a.case:
                continue
            t0 = time.time()
            outs = harness.run_unet(case, impl="reference")
            torch.save({"case": case.__dict__, "outs": [o.clone() for o in outs],
                        "source": "reference DistriUNetPP @ /root/reference over oracle/diffusers_stub, gloo, fp32"},
                       os.path.join(GOLDEN, f"unet_{case.name}.pt"))
            print(f"unet_{case.name}: {time.time() - t0:.1f}s  std={outs[-1].std():.4f}", flush=True)


if __name__ == "__main__":
    main()
