"""TEST INFRASTRUCTURE (oracle) -- the tensor-parallel reference arm: runs the UNMODIFIED reference DistriUNetTP
(/root/reference/distrifuser/models/distri_sdxl_unet_tp.py, modules/tp/*.py) on CPU under gloo over the diffusers stub, on
the seeded tiny UNets of oracle/workloads.py, and writes tests/golden/unet_tp_*.pt:

    python -m oracle.tp_reference [--case NAME]

Runs only where the reference tree exists; the vectors it writes are committed.  Tensor parallelism equals the unsharded
model up to summation order, so no oracle restatement is needed: the world-1 oracle (oracle/pp_modules.py) restates it.

Two adapters, both applied to module instances before the reference wraps them (the stub files stay as they are):
  * the reference's tensor-parallel modules read attributes of diffusers 0.24.0 that the stub does not define --
    ResnetBlock2D.upsample / downsample (None), time_embedding_norm ("default"), skip_time_act (False)
    (modules/tp/resnet.py:22,102-173); Attention.group_norm / norm_cross (None) (modules/tp/attention.py:103-109);
    GEGLU.gelu (F.gelu) (modules/tp/feed_forward.py:66).  They are set to diffusers' defaults, which is what the stub computes.
  * the reference block calls self.conv_shortcut when diffusers' USE_PEFT_BACKEND flag is set (modules/tp/resnet.py:195),
    an attribute it never defines; it is pointed at the wrapped block's own conv_shortcut, which the non-PEFT branch calls.
"""
from __future__ import annotations

import argparse
import dataclasses
import os
import sys
import tempfile
import time

import torch
from torch import distributed as dist
from torch import multiprocessing as mp
from torch.nn import functional as F

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
for _p in (ROOT, os.path.join(ROOT, "oracle", "diffusers_stub")):
    if _p not in sys.path:
        sys.path.insert(0, _p)

from oracle import harness, workloads  # noqa: E402

GOLDEN = os.path.join(ROOT, "tests", "golden")


@dataclasses.dataclass(frozen=True)
class TPCase(workloads.UNetCase):
    """A tensor-parallel UNet case (DistriConfig(parallelism="tensor")); every step is synchronous."""
    parallelism: str = "tensor"


# No CFG-split cases: the reference's CFG-split tensor-parallel path cannot run (distri_sdxl_unet_tp.py:160 calls the
# attribute split_group).  Each CFG half of a split run computes the same function as the no-split case with the same n.
TP_CASES = (
    TPCase("tp_sdxl_w2_nosplit", world_size=2, split_batch=False),
    TPCase("tp_sdxl_w4_nosplit", world_size=4, split_batch=False),       # level 0 has 1 head: three members own none
    TPCase("tp_sd15_w2_nosplit", family="tiny_sd15", world_size=2, split_batch=False),
    TPCase("tp_sd15_w4_nosplit", family="tiny_sd15", world_size=4, split_batch=False),   # 2 heads: two members own none
)


def _diffusers_defaults(unet):
    from diffusers.models.attention import GEGLU
    from diffusers.models.attention_processor import Attention
    from diffusers.models.resnet import ResnetBlock2D
    for m in unet.modules():
        if isinstance(m, ResnetBlock2D):
            m.upsample = m.downsample = None
            m.time_embedding_norm = "default"
            m.skip_time_act = False
        elif isinstance(m, Attention):
            m.group_norm = m.norm_cross = None
        elif isinstance(m, GEGLU):
            m.gelu = F.gelu


def _worker(rank, case, port, outdir):
    harness._paths("reference")
    from distrifuser.models.distri_sdxl_unet_tp import DistriUNetTP
    from distrifuser.modules.tp.resnet import DistriResnetBlock2DTP
    harness._init(rank, case.world_size, port)
    cfg = workloads.DuckConfig(case.world_size, rank, height=8 * case.latent, width=8 * case.latent,
                               do_classifier_free_guidance=case.cfg, split_batch=case.split_batch,
                               warmup_steps=case.warmup_steps, comm_checkpoint=case.comm_checkpoint, mode=case.mode)
    cfg.parallelism = "tensor"
    ucfg = workloads.unet_config(case.family)
    unet = workloads.make_unet(case.family, case.weight_seed)
    _diffusers_defaults(unet)
    model = DistriUNetTP(unet, cfg)
    for m in model.modules():
        if isinstance(m, DistriResnetBlock2DTP):
            m.conv_shortcut = m.module.conv_shortcut
    outs = []
    with torch.no_grad():
        model.set_counter(0)
        model(**workloads.unet_inputs(case, 0, ucfg), return_dict=False, record=True)   # pipelines.py:144-145
        model.set_counter(0)                                                         # pipelines.py:57
        for t in range(case.steps):
            outs.append(model(**workloads.unet_inputs(case, t, ucfg), return_dict=False)[0].clone())
    torch.save(outs, os.path.join(outdir, f"rank{rank}.pt"))
    dist.barrier()
    dist.destroy_process_group()


def run_tp_reference(case):
    """-> outs[step] = eps [B,4,S,S] of the reference DistriUNetTP (asserted identical on every rank)."""
    assert case.world_size > 1
    with tempfile.TemporaryDirectory() as d:
        mp.spawn(_worker, args=(case, harness.free_port(), d), nprocs=case.world_size, join=True)
        per_rank = [torch.load(os.path.join(d, f"rank{r}.pt")) for r in range(case.world_size)]
    for r in range(1, case.world_size):
        for a, b in zip(per_rank[0], per_rank[r]):
            assert torch.equal(a, b), "the reference's output must be identical on all ranks"
    return per_rank[0]


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--case", default=None)
    a = ap.parse_args()
    os.makedirs(GOLDEN, exist_ok=True)
    for case in TP_CASES:
        if a.case and case.name != a.case:
            continue
        t0 = time.time()
        outs = run_tp_reference(case)
        torch.save({"case": case.__dict__, "outs": [o.clone() for o in outs],
                    "source": "reference DistriUNetTP @ /root/reference over oracle/diffusers_stub, gloo, fp32"},
                   os.path.join(GOLDEN, f"unet_{case.name}.pt"))
        print(f"unet_{case.name}: {time.time() - t0:.1f}s  std={outs[-1].std():.4f}", flush=True)


if __name__ == "__main__":
    main()
