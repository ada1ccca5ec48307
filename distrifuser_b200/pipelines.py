"""DistriSDXLPipeline / DistriSDPipeline -- same API surface as distrifuser/pipelines.py:10-299
(`from_pretrained(distri_config, **kwargs)`, `__call__`, `set_progress_bar_config`, `prepare`, attributes
`.pipeline .distri_config .static_inputs`).

`from_pretrained` uses the real diffusers pipelines when the package (and weights) are available.  This image has
neither, so `from_synthetic` builds the same object around a random-weight UNet of the SDXL / SD1.x architecture
and a latent-space pipeline stand-in (compat/pipeline.py): that is what bench.py and the parity tests drive."""
import os

import torch

from .models.distri_sdxl_unet_pp import DistriUNetPP
from .models.distri_sdxl_unet_tp import DistriUNetTP
from .utils import DistriConfig, PatchParallelismCommManager


def _wrap(unet, distri_config: DistriConfig):
    if distri_config.parallelism == "patch":                         # pipelines.py:30-37
        return DistriUNetPP(unet, distri_config)
    if distri_config.parallelism == "tensor":
        return DistriUNetTP(unet, distri_config)
    raise ValueError(f"Unknown / unsupported parallelism: {distri_config.parallelism}")


class _DistriPipelineBase:
    sdxl = True

    def __init__(self, pipeline, module_config: DistriConfig):
        self.pipeline = pipeline
        self.distri_config = module_config
        self.static_inputs = None
        self.prepare()

    def set_progress_bar_config(self, **kwargs):                     # pipelines.py:44-45
        self.pipeline.set_progress_bar_config(**kwargs)

    @torch.no_grad()
    def __call__(self, *args, **kwargs):                             # pipelines.py:47-58
        assert "height" not in kwargs, "height should not be in kwargs"
        assert "width" not in kwargs, "width should not be in kwargs"
        config = self.distri_config
        if not config.do_classifier_free_guidance:
            if "guidance_scale" not in kwargs:
                kwargs["guidance_scale"] = 1
            else:
                assert kwargs["guidance_scale"] == 1
        self.pipeline.unet.set_counter(0)
        return self.pipeline(height=config.height, width=config.width, *args, **kwargs)

    def _static_inputs(self):
        raise NotImplementedError

    @torch.no_grad()
    def prepare(self, **kwargs):                                     # pipelines.py:60-167 / 217-299
        cfg = self.distri_config
        pipeline = self.pipeline
        assert cfg.height % 8 == 0 and cfg.width % 8 == 0
        static_inputs = self._static_inputs(**kwargs)
        unet = pipeline.unet
        # cuDNN heuristics pick legacy sm80 "wo_smem" implicit-GEMM kernels for several 3x3 shapes on sm_100
        # (profiles/r1_launches_1024.md); autotuning happens in the un-captured passes below
        torch.backends.cudnn.benchmark = True
        comm_manager = None
        # the reference creates the manager only for n_device_per_batch > 1 (pipelines.py:132); the final epsilon
        # gather also goes through the arena here, so any world_size > 1 needs one
        if cfg.world_size > 1:
            comm_manager = PatchParallelismCommManager(cfg)
            unet.set_comm_manager(comm_manager)
            unet.set_counter(0)
            unet(**static_inputs, return_dict=False, record=True)    # registration pass (pipelines.py:138-139)
            comm_manager.create_buffer()                             # pipelines.py:140-141
        unet.set_counter(0)
        unet(**static_inputs, return_dict=False, record=True)        # pre-run (pipelines.py:144-145)
        self.static_inputs = static_inputs
        self.comm_manager = comm_manager
        self._capture_graphs()

    @torch.no_grad()
    def _capture_graphs(self):
        """Three graphs: synchronous step, first asynchronous step, steady state (pipelines.py:147-165); tensor parallelism
        has synchronous steps only and captures one (pipelines.py:154-155)."""
        cfg, unet, static_inputs = self.distri_config, self.pipeline.unet, self.static_inputs
        static_outputs, cuda_graphs = [], []
        unet.setup_cuda_graph(None, None, None)
        if cfg.use_cuda_graph:
            if self.comm_manager is not None:
                self.comm_manager.clear()
            torch.cuda.synchronize()
            counters = [0] if cfg.parallelism == "tensor" else [0, cfg.warmup_steps + 1, cfg.warmup_steps + 2]
            unet.static_inputs = None
            pool = None
            from . import _lib
            launches = []
            # the compute kernels are captured on a stream of priority DF_COMPUTE_PRIO (default -1 = above the publication
            # stream's 0): when a K/V projection finishes, the attention grid that follows it takes the SM slots before the
            # publication kernel of the same K/V does -- a publication CTA that got there first keeps a persistent attention
            # CTA out of its SM for the whole transfer (profiles/r2_exposed_comm_n8.txt)
            patch_peers = cfg.n_device_per_batch > 1 and cfg.parallelism == "patch"
            prio = int(os.environ.get("DF_COMPUTE_PRIO", "-1" if patch_peers else "0"))   # no publications without patch peers
            capture_stream = torch.cuda.Stream(device=cfg.device, priority=prio)
            for counter in counters:
                graph = torch.cuda.CUDAGraph()
                n0 = _lib.LAUNCHES["total"]
                with torch.cuda.graph(graph, pool=pool, stream=capture_stream):
                    unet.set_counter(counter)
                    output = unet(**static_inputs, return_dict=False, record=True)[0]
                    static_outputs.append(output)
                launches.append(_lib.LAUNCHES["total"] - n0)
                pool = graph.pool()
                cuda_graphs.append(graph)
            unet.setup_cuda_graph(static_outputs, cuda_graphs, launches)

    def set_mode(self, mode: str):
        """Switch the synchronisation mode (e.g. to "no_sync", the compute-only lower bound used for the exposed
        communication metric, SURVEY 8d) on the same arena and re-capture the graphs."""
        self.distri_config.mode = mode
        self._capture_graphs()


class DistriSDXLPipeline(_DistriPipelineBase):
    sdxl = True

    @staticmethod
    def from_pretrained(distri_config: DistriConfig, **kwargs):      # pipelines.py:19-42
        try:
            from diffusers import StableDiffusionXLPipeline, UNet2DConditionModel
        except ImportError as e:
            raise ImportError("from_pretrained needs `diffusers` and the SDXL checkpoint; neither exists in this "
                              "environment -- use DistriSDXLPipeline.from_synthetic(distri_config)") from e
        device = distri_config.device
        name = kwargs.pop("pretrained_model_name_or_path", "stabilityai/stable-diffusion-xl-base-1.0")
        torch_dtype = kwargs.pop("torch_dtype", torch.float16)
        unet = UNet2DConditionModel.from_pretrained(name, torch_dtype=torch_dtype, subfolder="unet").to(device)
        unet = _wrap(unet, distri_config)
        pipeline = StableDiffusionXLPipeline.from_pretrained(name, torch_dtype=torch_dtype, unet=unet, **kwargs).to(device)
        return DistriSDXLPipeline(pipeline, distri_config)

    @staticmethod
    def from_synthetic(distri_config: DistriConfig, unet=None, unet_config: dict | None = None, seed: int = 0,
                       scheduler=None, torch_dtype=torch.float16):
        """Random-weight SDXL UNet (torch default init under manual_seed(seed), SURVEY 8d) + latent pipeline."""
        from .compat.pipeline import SyntheticLatentPipeline
        from .compat.unet_2d_condition import SDXL, UNet2DConditionModel
        if unet is None:
            torch.manual_seed(seed)
            with torch.device(distri_config.device):
                unet = UNet2DConditionModel(**(unet_config or SDXL))
        unet = unet.to(distri_config.device, torch_dtype).eval()
        unet = _wrap(unet, distri_config)
        pipe = SyntheticLatentPipeline(unet, scheduler, sdxl=True, device=distri_config.device, dtype=torch_dtype)
        return DistriSDXLPipeline(pipe, distri_config)

    def _static_inputs(self, **kwargs):                              # pipelines.py:62-129
        cfg, pipeline = self.distri_config, self.pipeline
        device = cfg.device
        height, width = cfg.height, cfg.width
        prompt_embeds, _, pooled, _ = pipeline.encode_prompt(
            prompt="", prompt_2=None, device=device, num_images_per_prompt=1, do_classifier_free_guidance=False,
            negative_prompt=None, negative_prompt_2=None, prompt_embeds=None, negative_prompt_embeds=None,
            pooled_prompt_embeds=None, negative_pooled_prompt_embeds=None)
        batch_size = 2 if cfg.do_classifier_free_guidance else 1
        latents = pipeline.prepare_latents(batch_size, pipeline.unet.config.in_channels, height, width,
                                           prompt_embeds.dtype, device, None)
        if getattr(pipeline, "text_encoder_2", None) is None:
            proj_dim = int(pooled.shape[-1])
        else:
            proj_dim = pipeline.text_encoder_2.config.projection_dim
        add_time_ids = pipeline._get_add_time_ids((height, width), (0, 0), (height, width), dtype=prompt_embeds.dtype,
                                                  text_encoder_projection_dim=proj_dim)
        prompt_embeds = prompt_embeds.to(device).repeat(batch_size, 1, 1)
        add_text_embeds = pooled.to(device).repeat(batch_size, 1)
        add_time_ids = add_time_ids.to(device).repeat(batch_size, 1)
        t = torch.zeros([batch_size], device=device, dtype=torch.float32)
        return {"sample": latents, "timestep": t, "encoder_hidden_states": prompt_embeds,
                "added_cond_kwargs": {"text_embeds": add_text_embeds, "time_ids": add_time_ids}}


class DistriSDPipeline(_DistriPipelineBase):
    sdxl = False

    @staticmethod
    def from_pretrained(distri_config: DistriConfig, **kwargs):      # pipelines.py:178-200
        try:
            from diffusers import StableDiffusionPipeline, UNet2DConditionModel
        except ImportError as e:
            raise ImportError("from_pretrained needs `diffusers` and the SD checkpoint; neither exists in this "
                              "environment -- use DistriSDPipeline.from_synthetic(distri_config)") from e
        device = distri_config.device
        name = kwargs.pop("pretrained_model_name_or_path", "CompVis/stable-diffusion-v1-4")
        torch_dtype = kwargs.pop("torch_dtype", torch.float16)
        unet = UNet2DConditionModel.from_pretrained(name, torch_dtype=torch_dtype, subfolder="unet").to(device)
        unet = _wrap(unet, distri_config)
        pipeline = StableDiffusionPipeline.from_pretrained(name, torch_dtype=torch_dtype, unet=unet, **kwargs).to(device)
        return DistriSDPipeline(pipeline, distri_config)

    @staticmethod
    def from_synthetic(distri_config: DistriConfig, unet=None, unet_config: dict | None = None, seed: int = 0,
                       scheduler=None, torch_dtype=torch.float16):
        from .compat.pipeline import SyntheticLatentPipeline
        from .compat.unet_2d_condition import SD15, UNet2DConditionModel
        if unet is None:
            torch.manual_seed(seed)
            with torch.device(distri_config.device):
                unet = UNet2DConditionModel(**(unet_config or SD15))
        unet = unet.to(distri_config.device, torch_dtype).eval()
        unet = _wrap(unet, distri_config)
        pipe = SyntheticLatentPipeline(unet, scheduler, sdxl=False, device=distri_config.device, dtype=torch_dtype)
        return DistriSDPipeline(pipe, distri_config)

    def _static_inputs(self, **kwargs):                              # pipelines.py:219-259
        cfg, pipeline = self.distri_config, self.pipeline
        device = cfg.device
        enc = pipeline.encode_prompt("", device, num_images_per_prompt=1, do_classifier_free_guidance=False,
                                     negative_prompt=None, prompt_embeds=None, negative_prompt_embeds=None,
                                     lora_scale=None, clip_skip=kwargs.get("clip_skip", None))
        prompt_embeds = enc[0]
        batch_size = 2 if cfg.do_classifier_free_guidance else 1
        latents = pipeline.prepare_latents(batch_size, pipeline.unet.config.in_channels, cfg.height, cfg.width,
                                           prompt_embeds.dtype, device, None)
        prompt_embeds = prompt_embeds.to(device).repeat(batch_size, 1, 1)
        t = torch.zeros([batch_size], device=device, dtype=torch.float32)
        return {"sample": latents, "timestep": t, "encoder_hidden_states": prompt_embeds}
