"""DistriUNetTP -- drop-in for distrifuser/models/distri_sdxl_unet_tp.py:14-214 (tensor-parallel UNet wrapper).

Same constructor, forward signature (with `record`), counter protocol and CFG batch split as DistriUNetPP.  Inside a CFG
branch the n members of the patch group shard attention heads, feed-forward columns and ResnetBlock2D channels; the partial
results meet in df_allreduce_fwd (one fused all-reduce kernel per reference dist.all_reduce).  Every call is a synchronous
step; one CUDA graph serves every call (pipelines.py:154-155).  Every rank holds the full image of its CFG branch, and the
final epsilon still goes through df_output_gather, which is also the per-call world barrier.

Differences from the reference: the CFG-split path gathers the two branches through the arena (the reference calls the
attribute distri_config.split_group as a function, distri_sdxl_unet_tp.py:160, so its eager CFG-split path cannot run), and
n == 1 is refused by DistriConfig instead of running the unwrapped model."""
import torch
from torch import nn

from ..modules.base_module import BaseModule
from ..modules.tp.attention import DistriAttentionTP
from ..modules.tp.base import replicated_group_norm
from ..modules.tp.conv2d import DistriConv2dTP
from ..modules.tp.feed_forward import DistriFeedForwardTP
from ..modules.tp.resnet import DistriResnetBlock2DTP
from ..utils import DistriConfig
from .base_model import BaseModel
from .distri_sdxl_unet_pp import DistriUNetPP, _is_attention


def allreduce_max_bytes(unet_config: dict, height: int, width: int, batch: int) -> int:
    """Largest all-reduce payload of a UNet call (fp16): the widest activation a sharded module produces at each
    resolution -- the up-sampler conv of a level runs at the finer resolution with the coarser width."""
    boc = tuple(unet_config["block_out_channels"])
    best = 0
    for lvl, c in enumerate(boc):
        widest = max(c, boc[lvl + 1]) if lvl + 1 < len(boc) else c
        best = max(best, batch * (height // 8 >> lvl) * (width // 8 >> lvl) * widest * 2)
    return best


def tp_arena_bytes(unet_config: dict, height: int, width: int, n: int, world: int) -> int:
    """Bytes of one rank's arena for tensor parallelism over n devices per CFG branch (world / n branches): header, the
    three banks of the output image and the all-reduce ring.  Pure host arithmetic."""
    from types import SimpleNamespace
    from ..utils import PatchParallelismCommManager
    cm = PatchParallelismCommManager(SimpleNamespace(n_device_per_batch=n, world_size=world))
    batch = 1 if world > n else 2               # CFG split: one branch per patch group
    cm.register_allreduce(allreduce_max_bytes(unet_config, height, width, batch))
    cm.register_output(2, unet_config.get("out_channels", 4), height // 8, width // 8)
    return cm._layout()[0]


def _is_resnet(m: nn.Module) -> bool:
    return all(hasattr(m, a) for a in ("conv1", "conv2", "norm1", "norm2", "time_emb_proj"))


def _is_feed_forward(m: nn.Module) -> bool:
    net = getattr(m, "net", None)
    return isinstance(net, nn.ModuleList) and len(net) == 3 and hasattr(net[0], "proj") and isinstance(net[2], nn.Linear)


class DistriUNetTP(DistriUNetPP):  # for Tensor Parallelism
    def __init__(self, model: nn.Module, distri_config: DistriConfig):
        assert distri_config.parallelism == "tensor" and distri_config.n_device_per_batch > 1
        for name, module in list(model.named_modules()):             # distri_sdxl_unet_tp.py:18-37
            if isinstance(module, BaseModule):
                continue
            for subname, submodule in list(module.named_children()):
                if isinstance(submodule, BaseModule):
                    continue
                if _is_attention(submodule):
                    setattr(module, subname, DistriAttentionTP(submodule, distri_config))
                elif _is_feed_forward(submodule):
                    setattr(module, subname, DistriFeedForwardTP(submodule, distri_config))
                elif _is_resnet(submodule):
                    setattr(module, subname, DistriResnetBlock2DTP(submodule, distri_config))
                elif isinstance(submodule, nn.Conv2d) and (subname == "conv_out" or "downsamplers" in name
                                                           or "upsamplers" in name):
                    setattr(module, subname, DistriConv2dTP(submodule, distri_config))
        # the remaining GroupNorms (Transformer2DModel.norm, conv_norm_out) run replicated on the GroupNorm kernel; the
        # UNet's conv_norm_out -> SiLU pair is fused into it
        for module in list(model.modules()):
            if isinstance(module, BaseModule):
                continue
            for subname, submodule in list(module.named_children()):
                if isinstance(submodule, nn.GroupNorm):
                    gn = replicated_group_norm(submodule, distri_config)
                    gn.fuse_silu = subname == "conv_norm_out" and hasattr(module, "fused_norm_act")
                    setattr(module, subname, gn)
        if hasattr(model, "fused_norm_act"):
            model.fused_norm_act = True
        model.to(memory_format=torch.channels_last)
        BaseModel.__init__(self, model, distri_config)

    def _graph_index(self) -> int:
        return 0

    def _strip_row0(self, hs: int, h: int) -> int:
        assert hs == h                       # every member holds the whole image of its CFG branch
        return 0

    def _step_kind(self) -> int:
        return 0

