"""Multi-rank drivers of the tensor-parallel product path (test infrastructure): the fused all-reduce kernel on its own,
and the UNet / pipeline with DistriConfig(parallelism="tensor").  One process per rank, gloo only for rendezvous; with
fewer GPUs than ranks the ranks share cuda:0 through CUDA IPC (as in mp_product.py)."""
from __future__ import annotations

import os
import sys
import tempfile

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
for p in (ROOT, os.path.join(ROOT, "oracle", "diffusers_stub"), os.path.join(ROOT, "tests")):
    if p not in sys.path:
        sys.path.insert(0, p)


def _init(rank, world, port):
    from torch import distributed as dist
    if torch.cuda.device_count() < world:
        os.environ["DISTRIFUSER_B200_SHARE_GPU"] = "1"
    os.environ["LOCAL_RANK"] = str(rank)
    dist.init_process_group("gloo", rank=rank, world_size=world, init_method=f"tcp://127.0.0.1:{port}")


def _finish(comm_manager):
    from torch import distributed as dist
    torch.cuda.synchronize()
    dist.barrier()
    if comm_manager is not None:
        comm_manager.close()
    dist.destroy_process_group()


def _spawn(fn, world, *args):
    from oracle.harness import free_port
    from torch import multiprocessing as mp
    with tempfile.TemporaryDirectory() as d:
        mp.spawn(fn, args=(world, free_port(), d, *args), nprocs=world, join=True)
        return [torch.load(os.path.join(d, f"rank{r}.pt")) for r in range(world)]


# ------------------------------------------------------------------------------------------------ all-reduce kernel
def _partials(seed, n, shape):
    g = torch.Generator().manual_seed(seed)
    return [torch.randn(*shape, generator=g).half() for _ in range(n)]


def expected_allreduce(parts, bias, residual, contrib):
    """fp32 sum of the contributing partials in member order, + bias, + residual, rounded to fp16 once."""
    acc = torch.zeros(parts[0].shape, dtype=torch.float32)
    for s, p in enumerate(parts):
        if contrib >> s & 1:
            acc += p.float()
    if bias is not None:
        acc += bias.float()
    if residual is not None:
        acc += residual.float()
    return acc.half()


# (rows, C, with bias, with residual, member that contributes nothing or -1)
AR_SITES = ((64, 4, True, False, -1), (1000, 320, True, True, -1), (96, 64, True, False, 1), (8, 1280, False, True, 0))


def _allreduce_worker(rank, world, port, outdir, graph_calls):
    _init(rank, world, port)
    from distrifuser_b200.utils import DistriConfig, PatchParallelismCommManager
    cfg = DistriConfig(height=64, width=64, do_classifier_free_guidance=False, parallelism="tensor", use_cuda_graph=False)
    dev = cfg.device
    cm = PatchParallelismCommManager(cfg)
    sites = [cm.register_allreduce(rows * C * 2) for rows, C, *_ in AR_SITES]
    cm.register_output(1, 4, 8, 8)
    cm.create_buffer()

    def inputs(call):
        out = []
        for k, (rows, C, has_b, has_r, idle) in enumerate(AR_SITES):
            parts = _partials(1000 * call + k, world, (rows, C))
            g = torch.Generator().manual_seed(77 + k)
            bias = torch.randn(C, generator=g).half() if has_b else None
            res = torch.randn(rows, C, generator=g).half() if has_r else None
            contrib = ((1 << world) - 1) & ~(1 << idle if idle >= 0 else 0)
            out.append((parts, bias, res, contrib))
        return out

    static = [(torch.empty(rows, C, dtype=torch.float16, device=dev), torch.empty(rows, C, dtype=torch.float16, device=dev))
              for rows, C, *_ in AR_SITES]
    biases = [None if b is None else b.to(dev) for _, b, _, _ in inputs(0)]
    ress = [None if r is None else r.to(dev) for _, _, r, _ in inputs(0)]

    def one_call():
        cm.step_begin(0)
        for k, (rows, C, _, _, idle) in enumerate(AR_SITES):
            part, out = static[k]
            contrib = ((1 << world) - 1) & ~(1 << idle if idle >= 0 else 0)
            cm.all_reduce(sites[k], None if rank == idle else part, out, bias=biases[k], residual=ress[k], contrib_mask=contrib)

    results, wants = [], []
    calls = 3 + graph_calls
    graph = None
    for call in range(calls):
        inp = inputs(call)
        for k in range(len(AR_SITES)):
            static[k][0].copy_(inp[k][0][rank].to(dev))
        if call < 3:
            one_call()                                      # eager
        else:
            if graph is None:
                torch.cuda.synchronize()
                graph = torch.cuda.CUDAGraph()
                with torch.cuda.graph(graph):
                    one_call()
            graph.replay()                                  # seq numbers come from the device clock
        results.append([o.clone() for _, o in static])
        wants.append([expected_allreduce(*inp[k]) for k in range(len(AR_SITES))])
    torch.cuda.synchronize()
    got = [[o.cpu() for o in per] for per in results]
    torch.save({"got": got, "want": wants}, os.path.join(outdir, f"rank{rank}.pt"))
    _finish(cm)


def run_allreduce(world, graph_calls=200):
    """-> per rank {"got": [call][site] outputs, "want": [call][site] expected}."""
    return _spawn(_allreduce_worker, world, graph_calls)


# ------------------------------------------------------------------------------------------------ UNet / pipeline
def _config(case, use_graph):
    from distrifuser_b200.utils import DistriConfig
    return DistriConfig(height=8 * case.latent, width=8 * case.latent, do_classifier_free_guidance=case.cfg,
                        split_batch=case.split_batch, warmup_steps=case.warmup_steps, mode=case.mode,
                        use_cuda_graph=use_graph, parallelism="tensor")


def _pipeline(case, cfg):
    from oracle import workloads as W
    from distrifuser_b200.compat.unet_2d_condition import UNet2DConditionModel
    from distrifuser_b200.pipelines import DistriSDPipeline, DistriSDXLPipeline
    ucfg = W.unet_config(case.family)
    unet = UNet2DConditionModel(**ucfg)
    unet.load_state_dict(W.make_unet(case.family, case.weight_seed).state_dict(), strict=True)
    cls = DistriSDXLPipeline if ucfg.get("addition_embed_type") == "text_time" else DistriSDPipeline
    return cls.from_synthetic(cfg, unet=unet), ucfg


def _unet_worker(rank, world, port, outdir, case, use_graph):
    _init(rank, world, port)
    from oracle import workloads as W
    from distrifuser_b200.models.distri_sdxl_unet_tp import allreduce_max_bytes
    cfg = _config(case, use_graph)
    pipe, ucfg = _pipeline(case, cfg)
    model = pipe.pipeline.unet
    cm = pipe.comm_manager
    b = 1 if (case.cfg and case.split_batch) else case.batch
    assert max(cm.ar_bytes) == allreduce_max_bytes(ucfg, cfg.height, cfg.width, b)
    outs = []
    with torch.no_grad():
        model.set_counter(0)
        for t in range(case.steps):
            inp = W.unet_inputs(case, t, ucfg)
            dev = lambda x: x.to(cfg.device, torch.float16) if x.is_floating_point() else x.to(cfg.device)
            kw = dict(sample=dev(inp["sample"]), timestep=inp["timestep"].to(cfg.device).float(),
                      encoder_hidden_states=dev(inp["encoder_hidden_states"]))
            if inp["added_cond_kwargs"] is not None:
                kw["added_cond_kwargs"] = {k: dev(v) for k, v in inp["added_cond_kwargs"].items()}
            outs.append(model(**kw, return_dict=False)[0].float().cpu().clone())
    torch.save(outs, os.path.join(outdir, f"rank{rank}.pt"))
    _finish(cm)


def run_tp_unet(case, use_graph=False):
    """-> outs[rank][step] = eps of the whole batch (every rank holds it)."""
    return _spawn(_unet_worker, case.world_size, case, use_graph)


def _traj_worker(rank, world, port, outdir, case, num_steps, guidance):
    _init(rank, world, port)
    cfg = _config(case, True)
    pipe, _ = _pipeline(case, cfg)
    lats = []
    for _ in range(2):                                  # the same seed twice: nothing may leak from one image into the next
        g = torch.Generator().manual_seed(case.input_seed)
        lats.append(pipe(prompt="a photo", num_inference_steps=num_steps, guidance_scale=guidance, generator=g).images)
    torch.cuda.synchronize()
    torch.save([lat.float().cpu() for lat in lats], os.path.join(outdir, f"rank{rank}.pt"))
    _finish(pipe.comm_manager)


def run_tp_trajectory(case, num_steps=8, guidance=5.0):
    """-> per rank [first image latents, second image latents] of the public pipeline API."""
    return _spawn(_traj_worker, case.world_size, case, num_steps, guidance)
