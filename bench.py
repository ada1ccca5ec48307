#!/usr/bin/env python
"""bench.py -- SDXL 50-step latency (ms/image) of the B200-native patch-parallel UNet path.

    python bench.py --gpus 1 --steps 5 --warmup 3                       # ours, one GPU
    python bench.py ... --dump-outputs DIR                              # also write the last timed image's latents
    python -m torch.distributed.run --nproc-per-node N ... bench.py --gpus N ...
    python bench.py --impl reference ...                                # the reference's CPU path (oracle port), host cores
    python bench.py --impl reference-gpu ...                            # extra: the UNMODIFIED reference on the same GPUs
                                                                        # (needs it installed under baseline/_ref: DESIGN.md 6)

A "step" of our arm is one full image: 50 denoising steps (CFG pair per step) of the SDXL UNet at --resolution (default
1024x1024 = BASELINE.json configs[1]'s workload; strong scaling: the same image at every N), Euler scheduler, 4 warm-up
synchronous steps (DistriConfig defaults), synthetic inputs, random-init weights (no network for checkpoints).
`value` times the loop with inputs resident in HBM; `e2e` times DistriSDXLPipeline.__call__ with pinned-host prompt
embeddings / latents copied in and the final latents copied out inside the timed region.  Extra blocks of the same JSON
line: `roofline` (tcgen05 attention kernel at the step's shapes), `exposed_comm` (synchronous / asynchronous step split),
`hires` (the north-star 3840x3840 image at the same N), `cpu_baseline` (N=1).
"""
from __future__ import annotations

import argparse
import json
import os
import statistics
import subprocess
import sys
import tempfile
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
for p in (ROOT,):
    if p not in sys.path:
        sys.path.insert(0, p)

STEPS_PER_IMAGE = 50
print_json = print
METRIC = "SDXL 50-step latency (ms/image)"          # BASELINE.json's metric; --model sd15 (configs[4]) reports the same quantity for SD1.5


def metric_name(model: str) -> str:
    return METRIC if model == "sdxl" else METRIC.replace("SDXL", "SD1.5")


def parse():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference", "reference-gpu"])
    ap.add_argument("--resolution", type=int, default=1024)
    ap.add_argument("--model", default="sdxl", choices=["sdxl", "sd15"])
    ap.add_argument("--mode", default="corrected_async_gn")
    ap.add_argument("--no-split-batch", action="store_true")
    ap.add_argument("--no-cuda-graph", action="store_true")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-exposed-comm", action="store_true")
    ap.add_argument("--no-roofline", action="store_true")
    ap.add_argument("--no-hires", action="store_true", help="skip the 3840x3840 block")
    ap.add_argument("--hires-resolution", type=int, default=3840)
    ap.add_argument("--cpu-budget-s", type=float, default=200.0, help="wall budget of the CPU reference arm")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write the latents the last timed image returned to DIR/images.npy (float32), to compare two builds")
    a = ap.parse_args()
    if a.steps < 1:
        ap.error("--steps must be at least 1")
    if a.dump_outputs is not None:
        if a.impl != "ours":
            ap.error("--dump-outputs applies to --impl ours")
        try:                                                    # fail before the timed run, not after it
            os.makedirs(a.dump_outputs, exist_ok=True)
        except OSError as e:
            ap.error(f"--dump-outputs: {e}")
        if not os.access(a.dump_outputs, os.W_OK):
            ap.error(f"--dump-outputs: {a.dump_outputs} is not writable")
    return a


# ------------------------------------------------------------------------------------------------ clocks
class ClockSampler:
    """nvidia-smi clocks line of /opt/skills/guides/B200_PROFILING.md, sampled DURING the timed region."""
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index: int):
        self.index, self.proc, self.path = index, None, None

    def start(self):
        try:
            self.path = tempfile.mktemp(suffix=".csv")
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits", "-lms", "200",
                                          "-i", str(self.index)], stdout=open(self.path, "w"), stderr=subprocess.DEVNULL)
        except Exception:
            self.proc = None

    def stop(self) -> dict:
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        try:
            self.proc.wait(timeout=5)
        except Exception:
            self.proc.kill()
        sm, mx, reasons = [], None, set()
        for line in open(self.path):
            f = [x.strip() for x in line.split(",")]
            if len(f) < 9:
                continue
            try:
                sm.append(float(f[1])); mx = float(f[2])
            except ValueError:
                continue
            for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), f[5:9]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        os.unlink(self.path)
        return {"sm_mhz": statistics.median(sm) if sm else None, "sm_max_mhz": mx, "reasons": sorted(reasons), "samples": len(sm)}


def load_peaks() -> dict:
    try:
        return json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
    except Exception:
        return {}


# ------------------------------------------------------------------------------------------------ reference arm / cpu baseline
def usable_cpus() -> int:
    """CPUs this process may really use: the smaller of os.cpu_count(), the affinity mask and the cgroup CPU quota."""
    n = os.cpu_count() or 1
    try:
        n = min(n, len(os.sched_getaffinity(0)))
    except Exception:
        pass
    try:
        quota, period = open("/sys/fs/cgroup/cpu.max").read().split()[:2]
        if quota != "max":
            n = min(n, max(1, int(int(quota) / int(period))))
    except Exception:
        pass
    return max(1, n)


def pick_cpu_threads(torch) -> int:
    """Thread count for the CPU reference legs: the fastest of {usable CPUs, 1/2, 1/4} on a 1536^3 fp32 matmul probe (a shared
    128-thread host ran the full-UNet step 25x slower with all threads than round 1's 64-thread hosts; oversubscribed OpenMP teams
    spin on every one of the ~2 000 ops of a step)."""
    n = usable_cpus()
    a = torch.randn(1536, 1536)
    best, best_t = n, None
    for cand in sorted({n, max(1, n // 2), max(1, n // 4)}, reverse=True):
        torch.set_num_threads(cand)
        a @ a
        dt = float("inf")
        for _ in range(4):
            t0 = time.perf_counter()
            a @ a
            dt = min(dt, time.perf_counter() - t0)
        if best_t is None or dt < 0.9 * best_t:
            best, best_t = cand, dt
    return best


FLOPS_STEP = {512: 3.18e12, 1024: 13.52e12, 2048: 71.82e12, 3840: 464.92e12}   # SDXL, per CFG-pair denoise step (SURVEY Appendix B)


def cpu_reference_samples(model: str, resolution: int, want_timed: int, want_warm: int, budget_s: float, sample_resolution=None):
    """Times the oracle port of the reference's CPU path (fp32, world_size 1: the stock UNet forward exactly as
    DistriUNetPP.forward runs it when nothing is wrapped, distri_sdxl_unet_pp.py:118-133) on ALL host cores, at the benched
    resolution.  One SAMPLE = one denoise step of ONE classifier-free-guidance branch (batch 1) of the full-size UNet; the
    reference's single-device step runs the two branches as one batch-2 forward (twice the work on a CPU), so
    ms/image = sample x 2 branches x 50 steps.  Samples are REAL forwards at the benched size (no FLOP-ratio scaling);
    as many of the requested warm-up / timed samples as fit the wall budget are run, and the count that ran is reported."""
    sys.path.insert(0, os.path.join(ROOT, "oracle", "diffusers_stub"))
    import torch
    from oracle import pp_modules, workloads
    t_begin = time.perf_counter()
    threads = int(os.environ.get("DF_CPU_THREADS", "0")) or pick_cpu_threads(torch)
    torch.set_num_threads(threads)                      # torchrun exports OMP_NUM_THREADS=1: do not inherit it silently
    family = "sdxl" if model == "sdxl" else "sd15"
    target_resolution = resolution
    scale, scale_note = 1.0, ""
    if sample_resolution is not None and sample_resolution != resolution:
        # bounded sample for the in-arm `cpu_baseline` key: the reference's own CPU-runnable case (BASELINE.json configs[0], 512^2),
        # scaled to the benched image by the per-step FLOP ratio of SURVEY Appendix B
        if model == "sdxl" and resolution in FLOPS_STEP and sample_resolution in FLOPS_STEP:
            scale = FLOPS_STEP[resolution] / FLOPS_STEP[sample_resolution]
        else:
            scale = (resolution / sample_resolution) ** 2
        scale_note = f"; sampled at {sample_resolution}x{sample_resolution} and scaled x{scale:.2f} (per-step FLOP ratio to {resolution}x{resolution})"
        resolution = sample_resolution
    latent = resolution // 8
    unet = workloads.make_unet(family, 0)
    cfg = workloads.DuckConfig(1, 0, height=resolution, width=resolution, do_classifier_free_guidance=False)
    wrapped = pp_modules.OracleUNetPP(unet, cfg)
    case = workloads.UNetCase("cpu", family=family, world_size=1, latent=latent, cfg=False)
    inp = workloads.unet_inputs(case, 0, workloads.unet_config(family))
    build_s = time.perf_counter() - t_begin
    times, warm_done, warm_t = [], 0, 0.0

    def one():
        t0 = time.perf_counter()
        wrapped(**inp)
        return time.perf_counter() - t0

    with torch.no_grad():
        first = one()
        if first > 20.0 or first > 0.25 * budget_s:
            times.append(first)                     # a sample this long is its own warm-up (allocation effects << 1 %): count it
        else:
            warm_done, warm_t = 1, first
            for i in range(1, max(1, want_warm)):   # more warm-up samples only while they fit 40 % of the budget
                if (time.perf_counter() - t_begin) + warm_t > 0.4 * budget_s:
                    break
                warm_t = one()
                warm_done += 1
        while len(times) < max(1, want_timed):      # at least one timed sample; more only while the next one fits the budget
            if times and (time.perf_counter() - t_begin) + times[-1] > budget_s:
                break
            times.append(one())
    sample_s = sum(times) / len(times)
    ms_image = sample_s * 2 * STEPS_PER_IMAGE * 1e3 * scale
    sample = (f"{len(times)} timed + {warm_done} warm-up samples; one sample = one denoise step of one CFG branch (batch 1, fp32) of "
              f"the full {family} UNet at {resolution}x{resolution} on {threads} host threads: {sample_s:.2f} s/sample "
              f"(min {min(times):.2f}, max {max(times):.2f}); ms/image = sample x 2 branches x {STEPS_PER_IMAGE} steps; "
              f"model build {build_s:.0f} s outside the timed region{scale_note}")
    return dict(ms_image=ms_image, threads=threads, sample=sample, sample_s=sample_s, timed=len(times), warm=warm_done)


def run_reference(a):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    r = cpu_reference_samples(a.model, a.resolution, max(1, a.steps), max(1, a.warmup), a.cpu_budget_s)
    ms_image = r["ms_image"]
    line = {"metric": metric_name(a.model), "value": ms_image, "unit": "ms/image", "n_gpus": a.gpus, "steps": r["timed"], "warmup": r["warm"],
            "steps_requested": a.steps, "warmup_requested": a.warmup,
            "ms_per_step": r["sample_s"] * 1e3, "ms_per_step_is": "one bounded sample (see cpu_baseline.sample), not one image",
            "higher_is_better": False, "scaling": "strong", "vs_baseline": None, "dtype": "f32",
            "data": "synthetic", "impl": "reference",
            "config": {"workload": f"{a.model.upper()} UNet {a.resolution}x{a.resolution}, 50-step Euler, CFG batch 2, reference CPU path "
                                   f"(oracle port, world_size 1), bounded sample of the same workload",
                       "inputs_larger_than_l2": True},
            "cpu_baseline": {"value": ms_image, "unit": "ms/image", "cores": r["threads"], "kind": "port", "sample": r["sample"]},
            "e2e": {"value": ms_image, "unit": "ms/image", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
            "gpu_launches": 0}
    print_json(json.dumps(line))


# ------------------------------------------------------------------------------------------------ the unmodified reference on the GPU(s)
def run_reference_gpu(a):
    """SURVEY 8(d)(ii) "same-box GPU baseline": the UNMODIFIED reference package (baseline/_ref, installed with
    `pip install --no-deps --target`) -- its DistriConfig, PatchParallelismCommManager (NCCL all_gather), pp modules,
    DistriUNetPP and DistriSDXLPipeline.prepare()/CUDA graphs -- on the same synthetic fp16 workload.  diffusers is absent, so
    the UNet it wraps is the diffusers-0.24 restatement of oracle/diffusers_stub (torch SDPA / cuDNN / eager GroupNorm) and
    the denoising loop is the same latent-space stand-in our arm uses.  Reported as an extra arm; never the `reference` slot."""
    ref_dir = os.path.join(ROOT, "baseline", "_ref")
    if not os.path.isdir(os.path.join(ref_dir, "distrifuser")):
        print_json(json.dumps({"impl": "reference-gpu", "unavailable": "baseline/_ref/distrifuser is not installed (a clean checkout does "
                                                                        "not have it: pip install --no-deps --target baseline/_ref <a distrifuser "
                                                                        "source tree>)"}))
        return
    sys.path.insert(0, os.path.join(ROOT, "oracle", "diffusers_stub"))
    sys.path.insert(0, ref_dir)
    import torch
    from torch import distributed as dist
    from distrifuser.pipelines import DistriSDXLPipeline as RefPipeline          # the reference, unmodified
    from distrifuser.utils import DistriConfig as RefConfig
    from oracle import workloads
    from distrifuser_b200.compat.pipeline import SyntheticLatentPipeline        # diffusers' loop stand-in (shared by both arms)
    R = a.resolution
    if "RANK" in os.environ:
        torch.cuda.set_device(int(os.environ.get("LOCAL_RANK", "0")))
    cfg = RefConfig(height=R, width=R, mode=a.mode, split_batch=not a.no_split_batch, use_cuda_graph=not a.no_cuda_graph)
    dev = cfg.device
    unet = workloads.make_unet("sdxl", 0, dtype=torch.float16).to(dev)
    from distrifuser.models.distri_sdxl_unet_pp import DistriUNetPP as RefUNetPP
    unet = RefUNetPP(unet, cfg)
    pipe = RefPipeline(SyntheticLatentPipeline(unet, None, sdxl=True, device=dev, dtype=torch.float16), cfg)
    pipe.set_progress_bar_config(disable=True)
    g = torch.Generator().manual_seed(1234)
    ucfg = workloads.unet_config("sdxl")
    embeds = torch.randn(2, 77, ucfg["cross_attention_dim"], generator=g).half().to(dev)
    pooled = torch.randn(2, ucfg["projection_class_embeddings_input_dim"] - 6 * ucfg["addition_time_embed_dim"], generator=g).half().to(dev)
    lat = torch.randn(1, 4, R // 8, R // 8, generator=g).to(dev)
    world = cfg.world_size

    def image():
        return pipe(prompt_embeds=embeds, pooled_prompt_embeds=pooled, latents=lat, num_inference_steps=STEPS_PER_IMAGE,
                    guidance_scale=5.0, output_type="latent")

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    for _ in range(max(1, a.warmup)):
        image()
    barrier()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(a.steps):
        image()
    e1.record()
    barrier()
    ms = torch.tensor([e0.elapsed_time(e1)], device=dev)
    if world > 1:
        dist.all_reduce(ms, op=dist.ReduceOp.MAX)
    ms_image = ms.item() / a.steps
    if cfg.rank == 0:
        line = {"metric": metric_name(a.model), "value": ms_image, "unit": "ms/image", "n_gpus": world, "steps": a.steps, "warmup": max(1, a.warmup),
                "ms_per_step": ms_image, "ms_per_denoise_step": ms_image / STEPS_PER_IMAGE, "higher_is_better": False,
                "scaling": "strong", "vs_baseline": None, "dtype": "f16", "data": "synthetic", "impl": "reference-gpu",
                "config": {"workload": f"SDXL UNet {R}x{R}, 50-step Euler, CFG batch 2, random-init weights; UNMODIFIED reference "
                                       f"(baseline/_ref) over the diffusers-0.24 stub UNet, NCCL, torch SDPA / cuDNN",
                           "mode": cfg.mode, "cuda_graph": cfg.use_cuda_graph, "n_device_per_batch": cfg.n_device_per_batch}}
        print_json(json.dumps(line))
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()


# ------------------------------------------------------------------------------------------------ ours
def build_pipe(a, resolution):
    import torch
    from distrifuser_b200.pipelines import DistriSDPipeline, DistriSDXLPipeline
    from distrifuser_b200.utils import DistriConfig
    cfg = DistriConfig(height=resolution, width=resolution, mode=a.mode, split_batch=not a.no_split_batch,
                       use_cuda_graph=not a.no_cuda_graph)
    cls = DistriSDXLPipeline if a.model == "sdxl" else DistriSDPipeline
    pipe = cls.from_synthetic(cfg, seed=0)
    pipe.set_progress_bar_config(disable=True)
    return cfg, pipe


def make_inputs(a, pipe, dev, R):
    import torch
    ucfg = pipe.pipeline.unet.config
    g = torch.Generator().manual_seed(1234)                                   # scripts/run_sdxl.py:32
    embeds_h = torch.randn(2, 77, ucfg.cross_attention_dim, generator=g).half().pin_memory()
    pooled_h = None
    if a.model == "sdxl":
        pooled_h = torch.randn(2, ucfg.projection_class_embeddings_input_dim - 6 * ucfg.addition_time_embed_dim, generator=g).half().pin_memory()
    lat_h = torch.randn(1, 4, R // 8, R // 8, generator=g).pin_memory()
    out_h = torch.empty(1, 4, R // 8, R // 8).pin_memory()
    return dict(embeds_h=embeds_h, pooled_h=pooled_h, lat_h=lat_h, out_h=out_h, embeds_d=embeds_h.to(dev), lat_d=lat_h.to(dev),
                pooled_d=pooled_h.to(dev) if pooled_h is not None else None)


def attention_roofline(a, pipe, cfg, image, ms_image, dev, world, R):
    """Dominant-kernel roofline (fmha_fwd_kernel, self-attention launches).
      (1) one instrumented eager image records the shape of every attention / GroupNorm launch of the model;
      (2) every distinct self-attention shape is then timed with CUDA events as a CUDA graph of `count` back-to-back launches
          on ROTATING buffers (total footprint > L2), i.e. the kernel's average launch duration at exactly the step's shapes
          without the host-launch gaps that eager in-model events pick up for 30-us kernels.
    The kernel is timed ALONE (a graph of attention launches only), so the BURST tensor peak of MEASURED_PEAKS.json is the
    denominator; the fraction of the sustained figure is printed beside it."""
    import ctypes as C
    import torch
    from distrifuser_b200 import _lib
    saved = cfg.use_cuda_graph
    try:
        cfg.use_cuda_graph = False
        _lib.PROFILE = []
        image(False)
        torch.cuda.synchronize()
        prof, _lib.PROFILE = _lib.PROFILE, None
    finally:
        cfg.use_cuda_graph = saved
        _lib.PROFILE = None
    gn = [p for p in prof if p["kind"] == "gn"]
    gn_ms = sum(p["start"].elapsed_time(p["end"]) for p in gn)
    gn_b = sum(p["bytes"] for p in gn)
    gn_shapes = {}
    for p in gn:
        gn_shapes[p["shape"]] = gn_shapes.get(p["shape"], 0) + 1
    gn_shapes = {k: v // STEPS_PER_IMAGE for k, v in gn_shapes.items()}
    per_step = {}
    for p in prof:
        if p["kind"] == "self":
            per_step[p["shape"]] = per_step.get(p["shape"], 0) + 1
    per_step = {k: v // STEPS_PER_IMAGE for k, v in per_step.items()}          # launches of that shape per denoise step
    L = _lib.lib()
    seg = (C.c_int32 * 8)(*range(8))
    total_ms_step, total_fl_step, detail = 0.0, 0.0, []
    traffic_db = {}
    try:
        traffic_db = json.load(open(os.path.join(ROOT, "profiles", "ncu_traffic.json")))
    except Exception:
        pass
    traffic_sum, traffic_n = 0.0, 0
    for (bb, lq_, lkv_, heads_, d_), count in per_step.items():
        Cq = heads_ * d_
        nbuf = count
        while nbuf > 4 and nbuf * (2 * bb * lq_ * Cq + bb * lkv_ * 2 * Cq) * 2 > 8e9:    # 3840^2 shapes: bound the footprint
            nbuf //= 2
        qs = [torch.randn(bb, lq_, Cq, device=dev, dtype=torch.float16) for _ in range(nbuf)]
        kvs = [torch.randn(bb, lkv_, 2 * Cq, device=dev, dtype=torch.float16) for _ in range(nbuf)]
        outs = [torch.empty_like(q_) for q_ in qs]
        side = torch.cuda.Stream(device=dev)

        from distrifuser_b200.modules.pp.attn import _shared_workspace
        ws_bytes = L.df_attn_workspace_bytes(bb, lq_, lkv_, 1, heads_, d_)          # same scratch (balanced-tail schedule) as in the model
        ws_ptr = _shared_workspace(dev, ws_bytes).data_ptr() if ws_bytes else None

        def launch_all():
            st = torch.cuda.current_stream().cuda_stream
            for i in range(count):
                q_, kv_, o_ = qs[i % nbuf], kvs[i % nbuf], outs[i % nbuf]
                _lib.check(L.df_attn_fwd(_lib.null_comm(), q_.data_ptr(), kv_.data_ptr(), o_.data_ptr(), None, bb, lq_, lkv_,
                                         heads_, d_, q_.stride(1), kv_.stride(1), o_.stride(1), 1, 0, seg, 0, 0, 0.0, ws_ptr,
                                         ws_bytes, st), "df_attn_fwd")
        with torch.cuda.stream(side):
            launch_all()
        torch.cuda.synchronize()
        g = torch.cuda.CUDAGraph()
        with torch.cuda.graph(g):
            launch_all()
        for _ in range(2):
            g.replay()
        reps = 5 if lq_ * lkv_ < 1e8 else 2
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        torch.cuda.synchronize()
        e0.record()
        for _ in range(reps):
            g.replay()
        e1.record()
        torch.cuda.synchronize()
        ms_launch = e0.elapsed_time(e1) / reps / count
        fl = 4.0 * bb * lq_ * lkv_ * Cq
        total_ms_step += ms_launch * count
        total_fl_step += fl * count
        key = f"fmha_fwd_kernel b{bb} lq{lq_} lkv{lkv_} h{heads_} d{d_}"
        tr = traffic_db.get(key, {}).get("dram_bytes")
        if tr is not None:
            traffic_sum += tr * count
            traffic_n += count
        detail.append({"shape": {"b": bb, "lq": lq_, "lkv": lkv_, "heads": heads_, "d": d_}, "launches_per_step": count,
                       "avg_launch_ms": ms_launch, "tflops": fl / ms_launch / 1e9,
                       "algorithmic_bytes": 2.0 * (2 * bb * lq_ * Cq + bb * lkv_ * 2 * Cq), "ncu_dram_bytes": tr,
                       "footprint_mb": nbuf * (2 * bb * lq_ * Cq + bb * lkv_ * 2 * Cq) * 2 / 1e6})
        del qs, kvs, outs, g
    peaks = load_peaks()
    burst = peaks.get("bf16_tflops", 1590.0)
    sustained = peaks.get("bf16_tflops_sustained", 1400.0)
    ach = total_fl_step / (total_ms_step * 1e-3) / 1e12 if total_ms_step > 0 else 0.0
    n_launch = sum(per_step.values())
    roof = {"kernel": "fmha_fwd_kernel (self-attention launches of one denoise step)", "bound": "tensor", "achieved": ach,
            "peak": burst, "unit": "TFLOP/s", "frac": ach / burst,
            "frac_of_sustained": ach / sustained, "peak_sustained": sustained,
            # average per launch over the step's launches, from the ncu --set full captures summarised in profiles/ncu_traffic.json
            # (dram__bytes_read.sum + dram__bytes_write.sum of ONE launch of each shape); null when a shape has no capture
            "traffic": (traffic_sum / traffic_n) if traffic_n == n_launch and n_launch else None,
            "traffic_source": "profiles/ncu_traffic.json" if traffic_n == n_launch and n_launch else None,
            "peak_source": ("MEASURED_PEAKS.json bf16_tflops (burst: the kernel is timed alone), of measured" if peaks
                            else "fallback 1.59 PFLOP/s burst (B200_PROFILING.md), of fallback"),
            "launches_per_step": n_launch, "avg_launch_ms": total_ms_step / max(n_launch, 1),
            "ms_per_step": total_ms_step, "share_of_step": total_ms_step / (ms_image / STEPS_PER_IMAGE),
            "method": "CUDA events around a CUDA graph of the step's launches of each shape, rotating buffers (> L2)",
            "shapes": detail,
            "groupnorm": groupnorm_roofline(gn_shapes, dev, peaks, gn_b, gn_ms, len(gn))}
    return roof


def groupnorm_roofline(gn_shapes, dev, peaks, eager_bytes, eager_ms, eager_launches):
    """GroupNorm(+SiLU) launches of one denoise step, timed like the attention launches: one CUDA graph holding every launch of
    the step (each on its own buffers, > L2 in total), CUDA events around 5 replays.  Algorithmic bytes: one read and one write of
    the activation (SURVEY 8d: 2 * N * 2 B)."""
    import torch
    from distrifuser_b200 import _lib
    L = _lib.lib()
    items = []
    for (bb, cc, hh, ww), count in gn_shapes.items():
        for _ in range(count):
            x = torch.randn(bb, cc, hh, ww, device=dev, dtype=torch.float16).contiguous(memory_format=torch.channels_last)
            items.append((x, torch.empty_like(x), torch.ones(cc, device=dev, dtype=torch.float16), torch.zeros(cc, device=dev, dtype=torch.float16),
                          torch.zeros(L.df_groupnorm_scratch_bytes(bb, 32, hh, ww, cc), dtype=torch.uint8, device=dev), (bb, cc, hh, ww)))
    if not items:
        return None

    def launch_all():
        st = torch.cuda.current_stream().cuda_stream
        for x, y, g_, b_, scr, (bb, cc, hh, ww) in items:
            _lib.check(L.df_groupnorm_fwd(_lib.null_comm(), x.data_ptr(), None, 0, y.data_ptr(), g_.data_ptr(), b_.data_ptr(), bb, hh, ww, cc, 32,
                                          1e-5, 0, 0, 0, 1, 0, 0, 0, 1, scr.data_ptr(), st), "df_groupnorm_fwd")
    side = torch.cuda.Stream(device=dev)
    with torch.cuda.stream(side):
        launch_all()
    torch.cuda.synchronize()
    g = torch.cuda.CUDAGraph()
    with torch.cuda.graph(g):
        launch_all()
    for _ in range(2):
        g.replay()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    torch.cuda.synchronize()
    e0.record()
    for _ in range(5):
        g.replay()
    e1.record()
    torch.cuda.synchronize()
    ms_step = e0.elapsed_time(e1) / 5
    nbytes = sum(4.0 * it[0].numel() for it in items)
    peak = peaks.get("hbm_gbs", 6650.0)
    ach = nbytes / (ms_step * 1e-3) / 1e9
    return {"bound": "hbm", "achieved": ach, "peak": peak, "unit": "GB/s", "frac": ach / peak, "launches_per_step": len(items),
            "ms_per_step": ms_step, "algorithmic_bytes_per_step": nbytes,
            "method": "CUDA events around a CUDA graph of the step's GroupNorm launches (local statistics), separate buffers (> L2)",
            "eager_in_model": {"achieved": eager_bytes / (eager_ms * 1e-3) / 1e9 if eager_ms > 0 else 0.0, "launches": eager_launches,
                               "ms_per_image": eager_ms, "note": "CUDA events around eager launches: includes host launch gaps"}}


def step_times(pipe, cfg, reps=8):
    """ms of ONE UNet call of each kind through the captured graphs (or eager when graphs are off): synchronous (counter 0)
    and steady-state asynchronous (counter warmup+2), max over ranks.  Every rank replays the same sequence, so the peers'
    flags always arrive."""
    import torch
    from torch import distributed as dist
    unet = pipe.pipeline.unet
    si = pipe.static_inputs
    out = {}
    for name, counter in (("sync", 0), ("async", cfg.warmup_steps + 2)):
        def call():
            unet.set_counter(counter)
            unet(si["sample"], si["timestep"], si["encoder_hidden_states"], added_cond_kwargs=si.get("added_cond_kwargs"),
                 return_dict=False)
        unet.set_counter(0)
        for c in range(cfg.warmup_steps + 3):             # bring the epoch clock into the state this kind of step expects
            unet(si["sample"], si["timestep"], si["encoder_hidden_states"], added_cond_kwargs=si.get("added_cond_kwargs"),
                 return_dict=False)
        for _ in range(2):
            call()
        if cfg.world_size > 1:
            dist.barrier()
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(reps):
            call()
        e1.record()
        torch.cuda.synchronize()
        ms = torch.tensor([e0.elapsed_time(e1) / reps], device=cfg.device)
        if cfg.world_size > 1:
            dist.all_reduce(ms, op=dist.ReduceOp.MAX)
        out[name] = ms.item()
    return out


DUMP_MAX_BYTES = 64 << 20


def dump_outputs(out_dir: str, arrays: dict):
    """Writes each tensor as out_dir/<name>.npy in float32.  The bench inputs and weights come from fixed seeds, so two
    builds run with the same arguments can be compared output for output."""
    import numpy as np
    host = {name: t.detach().float().cpu().numpy() for name, t in arrays.items()}
    total = sum(x.nbytes for x in host.values())
    if total > DUMP_MAX_BYTES:
        raise ValueError(f"--dump-outputs: {total} bytes of outputs exceed the {DUMP_MAX_BYTES}-byte limit")
    for name, x in host.items():
        np.save(os.path.join(out_dir, f"{name}.npy"), x)


def run_ours(a):
    import torch
    from torch import distributed as dist
    from distrifuser_b200 import _lib
    _lib.lib()
    assert torch.cuda.is_available(), "bench.py (ours) needs a GPU"
    R = a.resolution
    cfg, pipe = build_pipe(a, R)
    rank, world = cfg.rank, cfg.world_size
    assert world == a.gpus, f"--gpus {a.gpus} but WORLD_SIZE is {world} (launch with torch.distributed.run)"
    dev = cfg.device
    io = make_inputs(a, pipe, dev, R)

    def make_image(pipe_, io_):
        def image(host: bool):
            kw = dict(num_inference_steps=STEPS_PER_IMAGE, guidance_scale=5.0, output_type="latent")
            if host:
                r = pipe_(prompt_embeds=io_["embeds_h"], pooled_prompt_embeds=io_["pooled_h"], latents=io_["lat_h"], **kw)
                io_["out_h"].copy_(r.images, non_blocking=True)
            else:
                r = pipe_(prompt_embeds=io_["embeds_d"], pooled_prompt_embeds=io_["pooled_d"], latents=io_["lat_d"], **kw)
            io_["images"] = r.images                        # a fresh tensor per image: later images do not overwrite it
            return r
        return image
    image = make_image(pipe, io)

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def timed(fn, host: bool, k: int):
        barrier()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(k):
            fn(host)
        e1.record()
        barrier()
        ms = torch.tensor([e0.elapsed_time(e1)], device=dev)
        if world > 1:
            dist.all_reduce(ms, op=dist.ReduceOp.MAX)
        return ms.item()

    warm = max(a.warmup, 3)
    for _ in range(warm):
        image(False)
    sampler = ClockSampler(dev.index or 0)
    if rank == 0:
        sampler.start()
    n0 = _lib.LAUNCHES["total"]
    total_ms = timed(image, False, a.steps)
    launches = _lib.LAUNCHES["total"] - n0
    timed_images = io["images"]                             # what the last timed image returned (written by --dump-outputs)
    e2e_ms = timed(image, True, a.steps)
    clocks = sampler.stop() if rank == 0 else None
    ms_image = total_ms / a.steps
    ms_image_e2e = e2e_ms / a.steps

    # ---- exposed communication (SURVEY 8d): same kernels with every publication / peer wait removed after warm-up
    #      (mode "no_sync" = compute-only lower bound); whole image and split by step kind
    exposed = None
    if world > 1 and cfg.n_device_per_batch > 1 and not a.no_exposed_comm and a.mode != "no_sync":
        st_mode = step_times(pipe, cfg)
        pipe.set_mode("no_sync")
        for _ in range(2):
            image(False)
        nosync_ms = timed(image, False, max(2, min(a.steps, 5))) / max(2, min(a.steps, 5))
        st_nosync = step_times(pipe, cfg)
        pipe.set_mode(a.mode)
        image(False)
        base = st_nosync["async"]                   # a step of pure compute (no publication, no peer wait, local GroupNorm)
        n_sync, n_async = cfg.warmup_steps + 1, STEPS_PER_IMAGE - cfg.warmup_steps - 1
        ex_sync, ex_async = st_mode["sync"] - base, st_mode["async"] - base
        exposed = {"ms_image_no_sync": nosync_ms, "exposed_comm_pct": 100.0 * (ms_image - nosync_ms) / ms_image,
                   "definition": "(t(mode) - t(no_sync)) / t(mode) over the whole 50-step image; no_sync keeps the 5 synchronous warm-up steps",
                   "sync_step_ms": st_mode["sync"], "async_step_ms": st_mode["async"], "compute_only_step_ms": base,
                   "exposed_ms_per_sync_step": ex_sync, "exposed_ms_per_async_step": ex_async,
                   "exposed_pct_sync_step": 100.0 * ex_sync / st_mode["sync"], "exposed_pct_async_step": 100.0 * ex_async / st_mode["async"],
                   "exposed_pct_image_from_steps": 100.0 * (n_sync * ex_sync + n_async * ex_async) / (n_sync * st_mode["sync"] + n_async * st_mode["async"]),
                   "steps": {"sync": n_sync, "async": n_async},
                   "method": "CUDA events around 8 replays of the captured graph of each step kind, max over ranks; compute-only = the "
                             "steady-state step of mode no_sync (same kernels, no publication / peer waits, local GroupNorm statistics)"}

    roof = None
    if not a.no_roofline:
        roof = attention_roofline(a, pipe, cfg, image, ms_image, dev, world, R)

    # ---- hires: the north-star configuration (3840x3840) at the same N, one timed image after prepare()'s warm-up calls
    hires = None
    if not a.no_hires and a.hires_resolution != R and a.model == "sdxl":
        try:
            if getattr(pipe, "comm_manager", None) is not None:
                barrier()
                pipe.comm_manager.close()
            del pipe, image
            import gc
            gc.collect()
            torch.cuda.empty_cache()
            HR = a.hires_resolution
            t0 = time.perf_counter()
            cfg_h, pipe_h = build_pipe(a, HR)
            io_h = make_inputs(a, pipe_h, dev, HR)
            image_h = make_image(pipe_h, io_h)
            n_img = 1 if world == 1 else 2
            if world > 1:
                image_h(False)                       # one un-timed image: the first NVLink stores of every slot
            hms = timed(image_h, False, n_img) / n_img
            hires = {"resolution": HR, "ms_per_image": hms, "ms_per_denoise_step": hms / STEPS_PER_IMAGE, "images_timed": n_img,
                     "parallelism": f"cfg{2 if (world > 1 and cfg_h.split_batch) else 1} x patch{cfg_h.n_device_per_batch}",
                     "setup_s": None, "workload": f"SDXL UNet {HR}x{HR}, 50-step Euler, CFG batch 2 (BASELINE.json configs[3] image size)"}
            if world > 1 and cfg_h.n_device_per_batch > 1 and not a.no_exposed_comm:
                st_h = step_times(pipe_h, cfg_h, reps=3)
                pipe_h.set_mode("no_sync")
                st_hn = step_times(pipe_h, cfg_h, reps=3)
                base = st_hn["async"]
                n_sync, n_async = cfg_h.warmup_steps + 1, STEPS_PER_IMAGE - cfg_h.warmup_steps - 1
                hires["exposed_comm"] = {
                    "sync_step_ms": st_h["sync"], "async_step_ms": st_h["async"], "compute_only_step_ms": base,
                    "exposed_pct_sync_step": 100.0 * (st_h["sync"] - base) / st_h["sync"],
                    "exposed_pct_async_step": 100.0 * (st_h["async"] - base) / st_h["async"],
                    "exposed_pct_image_from_steps": 100.0 * (n_sync * (st_h["sync"] - base) + n_async * (st_h["async"] - base)) /
                                                    (n_sync * st_h["sync"] + n_async * st_h["async"])}
            hires["setup_s"] = time.perf_counter() - t0 - hms * n_img / 1e3
            if getattr(pipe_h, "comm_manager", None) is not None:
                barrier()
                pipe_h.comm_manager.close()
        except Exception as e:                         # the headline line must survive a hires failure (e.g. out of memory)
            hires = {"resolution": a.hires_resolution, "error": f"{type(e).__name__}: {e}"[:300]}

    cpu = None
    if rank == 0 and world == 1 and not a.no_cpu_baseline:        # reported at N=1 only (rank 0's host cores)
        # a REAL sample at the benched size (5-26 s per 1024^2 sample with the probed thread count); only images above 1024^2 are
        # sampled at 1024^2 and scaled by the per-step FLOP ratio, to keep the default run within minutes
        r = cpu_reference_samples(a.model, R, 1, 1, 60.0, sample_resolution=1024 if R > 1024 else None)
        cpu = {"value": r["ms_image"], "unit": "ms/image", "cores": r["threads"], "kind": "port", "sample": r["sample"]}

    if rank == 0:
        n, b = cfg.n_device_per_batch, (1 if (cfg.do_classifier_free_guidance and cfg.split_batch and world > 1) else 2)
        h2d = io["embeds_h"].numel() * 2 + (io["pooled_h"].numel() * 2 if io["pooled_h"] is not None else 0) + io["lat_h"].numel() * 4
        line = {"metric": metric_name(a.model), "value": ms_image, "unit": "ms/image", "n_gpus": world, "steps": a.steps, "warmup": warm,
                "ms_per_step": ms_image, "ms_per_denoise_step": ms_image / STEPS_PER_IMAGE, "higher_is_better": False,
                "scaling": "strong", "vs_baseline": None, "dtype": "f16", "data": "synthetic",
                "config": {"workload": f"{a.model.upper()} UNet {R}x{R}, 50-step Euler, CFG batch 2, random-init weights",
                           "parallelism": f"cfg{2 if b == 1 else 1} x patch{n}", "mode": cfg.mode, "warmup_steps": cfg.warmup_steps,
                           "cuda_graph": cfg.use_cuda_graph, "l2": "working set (5.1 GB of weights per step) exceeds the 126 MB L2; no explicit flush"},
                "roofline": roof, "cpu_baseline": cpu, "exposed_comm": exposed, "hires": hires,
                "e2e": {"value": ms_image_e2e, "unit": "ms/image", "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": io["out_h"].numel() * 4},
                "gpu_launches": launches, "clocks": clocks}
        print_json(json.dumps(line))
        if a.dump_outputs is not None:                        # after the line: a failed dump does not lose the measurement
            dump_outputs(a.dump_outputs, {"images": timed_images})
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()


def main():
    a = parse()
    # exactly ONE line on stdout: libraries (e.g. "NCCL version ..." at communicator creation) write there too, so the real
    # stdout is parked and fd 1 points at stderr until the JSON line is emitted
    sys.stdout.flush()
    real_stdout = os.dup(1)
    os.dup2(2, 1)
    out = os.fdopen(real_stdout, "w")

    def emit(line: str):
        out.write(line + "\n")
        out.flush()

    global print_json
    print_json = emit
    if a.impl == "reference":
        run_reference(a)
    elif a.impl == "reference-gpu":
        run_reference_gpu(a)
    else:
        run_ours(a)


if __name__ == "__main__":
    main()
