"""world_size-2/4 host logic of the product on CPU (gloo): DistriConfig group / rank math under a real process group
and the arena layout computed by PatchParallelismCommManager -- every rank must derive the identical layout, because
peers address each other's slots by offset (no GPU needed: only the pure-host parts run here)."""
import os
import tempfile

import pytest
import torch
from torch import distributed as dist
from torch import multiprocessing as mp

from oracle.harness import free_port


def _worker(rank, world, port, cfg_on, split, outdir):
    dist.init_process_group("gloo", rank=rank, world_size=world, init_method=f"tcp://127.0.0.1:{port}")
    from distrifuser_b200.utils import DistriConfig, PatchParallelismCommManager
    cfg = DistriConfig(height=512, width=512, do_classifier_free_guidance=cfg_on, split_batch=split, use_cuda_graph=False)
    assert cfg.world_size == world and cfg.rank == rank and cfg.device.type == "cpu"
    n = cfg.n_device_per_batch
    assert n == (world // 2 if (cfg_on and split) else world)                       # utils.py:68-75
    grp = cfg.patch_group_ranks()
    assert len(grp) == n and grp[cfg.split_idx()] == rank
    if cfg_on and split:
        assert cfg.batch_group is not None and cfg.split_group is not None          # utils.py:84-96
        t = torch.tensor([float(rank)])
        dist.all_reduce(t, group=cfg.batch_group)
        assert t.item() == float(sum(grp))
    cm = PatchParallelismCommManager(cfg)
    b = 1 if (cfg_on and split) else 2
    i0 = cm.register_tensor([2, b, 32, 1, 1, 1], torch.float32, layer_type="gn")
    i1 = cm.register_tensor([2, b, 320, 1, 64], torch.float16, layer_type="conv2d")
    i2 = cm.register_tensor((b, 4096 // n, 1280), torch.float16, layer_type="attn")
    assert (i0, i1, i2) == (0, 1, 2) and cm.numel_dict["attn"] == b * (4096 // n) * 1280  # utils.py:130-149
    cm.register_output(2, 4, 64, 64)
    total, bank = cm._layout()
    layout = dict(total=total, bank=bank, off=list(cm.tensor_off), out=cm.output_off, slots=list(cm.slot_bytes))
    for k in range(len(cm.tensor_off)):
        assert cm.tensor_off[k] % 256 == 0
        if k:
            assert cm.tensor_off[k] >= cm.tensor_off[k - 1] + n * cm.slot_bytes[k - 1]    # slots never overlap
    assert total == cm.tensor_off[0] + 3 * bank and cm.output_off + 2 * 4 * 64 * 64 * 2 <= cm.tensor_off[0] + bank
    gathered = [None] * world
    dist.all_gather_object(gathered, (cfg.batch_idx(), layout))
    same_branch = [lay for bi, lay in gathered if bi == cfg.batch_idx()]
    assert all(lay == layout for lay in same_branch), "ranks of one patch group disagree on the arena layout"
    torch.save(layout, os.path.join(outdir, f"r{rank}.pt"))
    dist.barrier()
    dist.destroy_process_group()


@pytest.mark.parametrize("world,cfg_on,split", [(2, True, True), (2, True, False), (4, True, True), (4, False, True)])
def test_config_and_arena_layout_multirank(world, cfg_on, split, monkeypatch):
    monkeypatch.setenv("CUDA_VISIBLE_DEVICES", "")      # the spawned ranks take the host path on GPU machines too
    with tempfile.TemporaryDirectory() as d:
        mp.spawn(_worker, args=(world, free_port(), cfg_on, split, d), nprocs=world, join=True)
        assert len(os.listdir(d)) == world


def test_unsupported_parallelism_is_loud():
    from distrifuser_b200.utils import DistriConfig
    with pytest.raises(NotImplementedError):
        DistriConfig(parallelism="tensor")


def test_cpu_tensor_is_rejected_by_the_wrappers():
    """The product path has no CPU fallback: the wrappers refuse non-CUDA / non-fp16 activations."""
    from torch import nn
    from distrifuser_b200.modules.pp.groupnorm import DistriGroupNorm
    from distrifuser_b200.utils import DistriConfig
    cfg = DistriConfig(height=64, width=64)
    gn = DistriGroupNorm(nn.GroupNorm(2, 8), cfg)
    with pytest.raises(RuntimeError, match="no CPU"):
        gn(torch.randn(1, 8, 4, 4))
