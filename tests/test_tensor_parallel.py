"""Tensor parallelism (DistriConfig(parallelism="tensor")): the fused all-reduce kernel, the host arena layout of its slot
ring, and the tensor-parallel UNet / pipeline against goldens produced by the unmodified reference DistriUNetTP
(python -m oracle.tp_reference).  Tensor parallelism is exact: its goldens equal the unsharded model up to summation order,
so the GPU tests hold the product to the same bar as tests/test_unet_gpu.py."""
import dataclasses
import os
import tempfile

import pytest
import torch
from torch import distributed as dist
from torch import multiprocessing as mp

from oracle import harness, workloads
from oracle.harness import free_port
from oracle.tp_reference import TP_CASES, TPCase

TP = {c.name: c for c in TP_CASES}


def _gold(golden_dir, name):
    p = os.path.join(golden_dir, f"unet_{name}.pt")
    assert os.path.exists(p), f"missing golden fixture unet_{name}.pt"
    return torch.load(p)


# ------------------------------------------------------------------------------------------------------------- CPU
@pytest.mark.parametrize("name", ["tp_sdxl_w2_nosplit", "tp_sdxl_w4_nosplit"])
def test_sdxl_tp_golden_equals_unsharded(name, golden_dir):
    gold = _gold(golden_dir, name)
    assert gold["case"] == TP[name].__dict__
    w1 = _gold(golden_dir, "sdxl_w1")["outs"]
    for a, b in zip(gold["outs"], w1):
        assert (a - b).abs().max().item() < 1e-5


@pytest.mark.parametrize("name", ["tp_sd15_w2_nosplit", "tp_sd15_w4_nosplit"])
def test_sd15_tp_golden_equals_world1_oracle(name, golden_dir):
    gold = _gold(golden_dir, name)
    case = TP[name]
    w1 = workloads.UNetCase("sd15_w1", family=case.family, world_size=1, split_batch=False)
    for a, b in zip(gold["outs"], harness.run_unet(w1, impl="oracle")):
        assert (a - b).abs().max().item() < 1e-5


def _reference_head_split(heads, n, r):
    """modules/tp/attention.py:15-29, restated."""
    sliced = heads // n
    rem = heads % n
    if r < rem:
        sliced += 1
    if sliced == 0:
        return None
    start = r * sliced if r < rem else rem * (sliced + 1) + (r - rem) * sliced
    return start, sliced


@pytest.mark.parametrize("n", [2, 4, 8])
def test_head_split_matches_reference(n):
    from distrifuser_b200.modules.tp.attention import head_split
    for heads in range(1, 21):
        covered = []
        for r in range(n):
            start, count = head_split(heads, n, r)
            ref = _reference_head_split(heads, n, r)
            assert (ref is None and count == 0) or ref == (start, count)
            covered += range(start, start + count)
        assert covered == list(range(heads))


def _layout_worker(rank, world, port, outdir):
    dist.init_process_group("gloo", rank=rank, world_size=world, init_method=f"tcp://127.0.0.1:{port}")
    from distrifuser_b200.utils import DistriConfig, PatchParallelismCommManager
    cfg = DistriConfig(height=256, width=256, do_classifier_free_guidance=False, parallelism="tensor", use_cuda_graph=False)
    assert cfg.device.type == "cpu" and cfg.n_device_per_batch == world
    layouts = []
    for nsites in (1, 7, 232):
        cm = PatchParallelismCommManager(cfg)
        for k in range(nsites):
            cm.register_allreduce(1000 + (k * 7919) % 4000 if k else 5000)     # the largest site is 5000 bytes
        cm.register_output(2, 4, 32, 32)
        total, _ = cm._layout()
        layouts.append((total, cm.ar_ring_off, cm.ar_slot_bytes, cm._flags_ar_off))
        assert cm.ar_slot_bytes == 5120 and total == cm.ar_ring_off + 2 * world * 5120
    assert len(set(layouts)) == 1, "the arena must not grow with the number of all-reduce sites"
    gathered = [None] * world
    dist.all_gather_object(gathered, layouts[0])
    assert all(g == layouts[0] for g in gathered), "ranks disagree on the all-reduce ring layout"
    torch.save(layouts[0], os.path.join(outdir, f"r{rank}.pt"))
    dist.barrier()
    dist.destroy_process_group()


@pytest.mark.parametrize("world", [2, 4])
def test_tp_arena_layout_multirank(world, monkeypatch):
    monkeypatch.setenv("CUDA_VISIBLE_DEVICES", "")
    with tempfile.TemporaryDirectory() as d:
        mp.spawn(_layout_worker, args=(world, free_port(), d), nprocs=world, join=True)
        assert len(os.listdir(d)) == world


def test_sdxl_tp_arena_bytes_from_shapes():
    """The ring holds 2 x n slots of the largest all-reduce: at 1024^2 the 640-channel up-sampler conv at 128^2 latents
    (21.0 MB per CFG branch), at 3840^2 the same conv at 480^2 (294.9 MB)."""
    from distrifuser_b200.compat.unet_2d_condition import SDXL
    from distrifuser_b200.models.distri_sdxl_unet_tp import allreduce_max_bytes, tp_arena_bytes
    for side, lat in ((1024, 128), (3840, 480)):
        assert allreduce_max_bytes(SDXL, side, side, 1) == lat * lat * 640 * 2
        out_img = (2 * 4 * lat * lat * 2 + 1023) // 1024 * 1024
        for n in (2, 4, 8):
            for world, b in ((n, 2), (2 * n, 1)):
                if world > 8:
                    continue
                ring = 2 * n * (b * lat * lat * 640 * 2)
                assert tp_arena_bytes(SDXL, side, side, n, world) == 1024 + 3 * out_img + ring


def test_tensor_parallel_needs_two_devices_and_naive_patch_raises():
    from distrifuser_b200.utils import DistriConfig
    with pytest.raises(NotImplementedError, match="parallelism=\"patch\""):
        DistriConfig(parallelism="tensor")
    with pytest.raises(NotImplementedError):
        DistriConfig(parallelism="naive_patch")


# ------------------------------------------------------------------------------------------------------------- GPU
def _check(name, outs, golden_dir):
    gold = _gold(golden_dir, name)["outs"]
    for r, per_rank in enumerate(outs):
        assert all(torch.equal(a, b) for a, b in zip(per_rank, outs[0])), f"rank {r} differs from rank 0"
        for t, (a, b) in enumerate(zip(per_rank, gold)):
            assert a.shape == b.shape
            err = (a - b).abs()
            psnr = 10 * torch.log10(b.abs().max() ** 2 / max((err ** 2).mean().item(), 1e-20)).item()
            assert err.mean().item() < 4e-3 and err.max().item() < 4e-2 and psnr > 45, \
                f"{name} rank{r} step{t}: mean {err.mean():.2e} max {err.max():.2e} psnr {psnr:.1f} dB"


@pytest.mark.gpu
@pytest.mark.parametrize("world", [2, 4])
def test_allreduce_kernel(world):
    """Bit-exact against an fp32 sum rounded once, identical on every rank; C = 4, members that contribute nothing, and 200
    replays of a captured graph after 3 eager calls (ring reuse, sequence numbers from the device clock)."""
    from mp_tp import run_allreduce
    res = run_allreduce(world)
    for r in range(world):
        for call, (got, want) in enumerate(zip(res[r]["got"], res[r]["want"])):
            for k, (g, w) in enumerate(zip(got, want)):
                assert torch.equal(g, w), f"rank {r} call {call} site {k}: max err {(g.float() - w.float()).abs().max()}"
                assert torch.equal(g, res[0]["got"][call][k])


@pytest.mark.gpu
@pytest.mark.parametrize("use_graph", [False, True], ids=["eager", "graph"])
@pytest.mark.parametrize("name", ["tp_sdxl_w2_nosplit", "tp_sdxl_w4_nosplit", "tp_sd15_w2_nosplit", "tp_sd15_w4_nosplit"])
def test_tp_unet(name, use_graph, golden_dir):
    from mp_tp import run_tp_unet
    _check(name, run_tp_unet(TP[name], use_graph=use_graph), golden_dir)


@pytest.mark.gpu
@pytest.mark.parametrize("use_graph", [False, True], ids=["eager", "graph"])
def test_tp_unet_cfg_split(use_graph, golden_dir):
    """world 4 = CFG split x tensor-parallel groups of 2; each CFG half computes what the no-split n = 2 case computes."""
    from mp_tp import run_tp_unet
    case = dataclasses.replace(TP["tp_sdxl_w2_nosplit"], world_size=4, split_batch=True)
    _check("tp_sdxl_w2_nosplit", run_tp_unet(case, use_graph=use_graph), golden_dir)


@pytest.mark.gpu
@pytest.mark.multigpu(8)
def test_tp_unet_eight_gpus(golden_dir):
    from mp_tp import run_tp_unet
    case = dataclasses.replace(TP["tp_sdxl_w4_nosplit"], world_size=8, split_batch=True)
    _check("tp_sdxl_w4_nosplit", run_tp_unet(case), golden_dir)


@pytest.mark.gpu
def test_tp_pipeline_trajectory():
    """Public API: DistriSDXLPipeline.from_synthetic(DistriConfig(parallelism="tensor")) at n = 2; two images with the same
    seed are bit-identical and an 8-step trajectory stays within 35 dB PSNR of the fp32 oracle trajectory."""
    from mp_tp import run_tp_trajectory
    case = TPCase("tp_traj", world_size=2, split_batch=False)
    outs = run_tp_trajectory(case)
    want = harness.run_trajectory(workloads.UNetCase("traj_w1", world_size=1))
    for first, second in outs:
        assert torch.equal(first, second), "second image with the same seed differs from the first"
        assert torch.equal(first, outs[0][0])
        mse = ((first - want) ** 2).mean().item()
        psnr = 10 * torch.log10(want.abs().max() ** 2 / max(mse, 1e-20)).item()
        assert psnr > 35, f"trajectory PSNR {psnr:.1f} dB"


@pytest.mark.gpu
def test_tp_full_size_sdxl_unet_step_vs_oracle():
    """The full SDXL UNet at 512^2, n = 2, one CFG step, against the world-1 fp32 oracle (bar of
    test_full_size_sdxl_unet_step_vs_oracle)."""
    from mp_tp import run_tp_unet
    case = TPCase("tp_sdxl_full_512", family="sdxl", world_size=2, split_batch=False, latent=64, steps=1)
    outs = run_tp_unet(case)
    want = harness.run_unet(workloads.UNetCase("sdxl_full_512", family="sdxl", world_size=1, latent=64, steps=1),
                            impl="oracle")[0]
    assert torch.equal(outs[0][0], outs[1][0])
    got = outs[0][0]
    assert got.shape == want.shape == (2, 4, 64, 64) and torch.isfinite(got).all()
    err = (got - want).abs()
    std = want.std().item()
    psnr = 10 * torch.log10(want.abs().max() ** 2 / max((err ** 2).mean().item(), 1e-20)).item()
    assert err.mean().item() < 1.2e-2 * std and err.max().item() < 0.12 * std and psnr > 45, \
        f"mean {err.mean():.2e} max {err.max():.2e} std {std:.3f} psnr {psnr:.1f} dB"
