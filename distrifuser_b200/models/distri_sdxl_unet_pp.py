"""DistriUNetPP -- drop-in for distrifuser/models/distri_sdxl_unet_pp.py:15-214 (patch-parallel UNet wrapper).

Same constructor, forward signature (including the non-diffusers `record` kwarg), counter protocol, CFG batch
split and three-graph replay as the reference.  Differences, all internal:
  * the wrappers are installed for every world size (the reference leaves world_size==1 unwrapped, :18), so the
    sm_100a kernels are the only attention / GroupNorm path;
  * the final epsilon all_gather + cat (:162-169,186-193) is df_output_gather: each rank stores its strip into
    every peer's arena and waits on flags;
  * GroupNorm -> SiLU pairs of ResnetBlock2D / conv_norm_out run fused inside the GroupNorm kernel.
"""
import torch
from torch import nn

from .. import _lib
from ..modules.base_module import BaseModule, nvtx_range
from ..modules.pp.attn import DistriCrossAttentionPP, DistriSelfAttentionPP
from ..modules.pp.conv2d import DistriConv2dPP
from ..modules.pp.groupnorm import DistriGroupNorm
from ..utils import DistriConfig
from .base_model import BaseModel


def _is_attention(m: nn.Module) -> bool:
    return all(hasattr(m, a) for a in ("to_q", "to_k", "to_v", "to_out", "heads"))


def _output_cls():
    try:
        from diffusers.models.unet_2d_condition import UNet2DConditionOutput
    except Exception:
        from ..compat.unet_2d_condition import UNet2DConditionOutput
    return UNet2DConditionOutput


class DistriUNetPP(BaseModel):  # for Patch Parallelism
    def __init__(self, model: nn.Module, distri_config: DistriConfig):
        for name, module in list(model.named_modules()):             # distri_sdxl_unet_pp.py:19-40
            if isinstance(module, BaseModule):
                continue
            for subname, submodule in list(module.named_children()):
                if isinstance(submodule, nn.Conv2d):
                    k = submodule.kernel_size
                    if k == (1, 1) or k == 1:
                        continue
                    setattr(module, subname, DistriConv2dPP(submodule, distri_config, is_first_layer=subname == "conv_in"))
                elif _is_attention(submodule):
                    if subname == "attn1":
                        setattr(module, subname, DistriSelfAttentionPP(submodule, distri_config))
                    else:
                        assert subname == "attn2"
                        setattr(module, subname, DistriCrossAttentionPP(submodule, distri_config))
                elif isinstance(submodule, nn.GroupNorm):
                    setattr(module, subname, DistriGroupNorm(submodule, distri_config))
        # GroupNorm -> SiLU fusion where the block exposes the switch (compat UNet; diffusers blocks keep SiLU separate)
        for module in model.modules():
            if hasattr(module, "fused_norm_act"):
                module.fused_norm_act = True
                for nm in ("norm1", "norm2", "conv_norm_out"):
                    sub = getattr(module, nm, None)
                    if isinstance(sub, DistriGroupNorm):
                        sub.fuse_silu = True
        model.to(memory_format=torch.channels_last)
        super().__init__(model, distri_config)

    def _graph_index(self) -> int:
        cfg = self.distri_config
        if self.counter <= cfg.warmup_steps:                         # distri_sdxl_unet_pp.py:108-113
            return 0
        return 1 if self.counter == cfg.warmup_steps + 1 else 2

    def _strip_row0(self, hs: int, h: int) -> int:
        """First image row of this rank's output strip (its patch)."""
        if self.distri_config.n_device_per_batch == 1:
            assert hs == h
            return 0
        return self.distri_config.split_idx() * hs

    def _step_kind(self) -> int:
        cfg = self.distri_config
        if self.counter <= cfg.warmup_steps or cfg.mode == "full_sync":
            return 0
        return 2 if cfg.mode == "no_sync" else 1

    @nvtx_range("DistriUNetPP")
    def forward(
        self,
        sample: torch.FloatTensor,
        timestep,
        encoder_hidden_states: torch.Tensor,
        class_labels=None,
        timestep_cond=None,
        attention_mask=None,
        cross_attention_kwargs=None,
        added_cond_kwargs=None,
        down_block_additional_residuals=None,
        mid_block_additional_residual=None,
        down_intrablock_additional_residuals=None,
        encoder_attention_mask=None,
        return_dict: bool = True,
        record: bool = False,
    ):
        cfg = self.distri_config
        b, c, h, w = sample.shape
        assert (class_labels is None and timestep_cond is None and attention_mask is None
                and cross_attention_kwargs is None and down_block_additional_residuals is None
                and mid_block_additional_residual is None and down_intrablock_additional_residuals is None
                and encoder_attention_mask is None)                  # distri_sdxl_unet_pp.py:63-72
        split = cfg.world_size > 1 and cfg.do_classifier_free_guidance and cfg.split_batch
        if split:                                                    # distri_sdxl_unet_pp.py:77-87 / 134-146
            assert b == 2
            i = cfg.batch_idx()
            sample = sample[i:i + 1]
            if torch.is_tensor(timestep) and timestep.ndim > 0:
                timestep = timestep[i:i + 1]
            encoder_hidden_states = encoder_hidden_states[i:i + 1]
            if added_cond_kwargs is not None:                        # new dict: the caller's is not mutated (SURVEY D-10)
                added_cond_kwargs = {k: v[i:i + 1] for k, v in added_cond_kwargs.items()}

        if cfg.use_cuda_graph and not record and self.cuda_graphs is not None:
            si = self.static_inputs                                  # distri_sdxl_unet_pp.py:89-106
            assert si["sample"].shape == sample.shape
            si["sample"].copy_(sample)
            if torch.is_tensor(timestep):
                si["timestep"].copy_(timestep.expand(si["timestep"].shape) if timestep.ndim == 0 else timestep)
            else:
                si["timestep"].fill_(timestep)                       # no .item() host sync (SURVEY A6)
            si["encoder_hidden_states"].copy_(encoder_hidden_states)
            if added_cond_kwargs is not None:
                for k in added_cond_kwargs:
                    si["added_cond_kwargs"][k].copy_(added_cond_kwargs[k])
            graph_idx = self._graph_index()
            self.cuda_graphs[graph_idx].replay()
            if self.graph_launches is not None:
                _lib.LAUNCHES["total"] += self.graph_launches[graph_idx]
            output = self.static_outputs[graph_idx]
        else:
            cm = self.comm_manager
            live = cm is not None and cm.arena is not None
            if cm is not None and cm.arena is None and cfg.world_size > 1 and cm.output_spec is None:
                cm.register_output(b if not split else 2, c, h, w)
            if live:
                cm.step_begin(self._step_kind())
            # NHWC inside the UNet; `sample` itself stays the (sliced) view of the caller's tensor so that a captured
            # graph re-reads the static input on every replay
            sample_cl = sample.contiguous(memory_format=torch.channels_last)
            output = self.model(sample_cl, timestep, encoder_hidden_states, added_cond_kwargs=added_cond_kwargs,
                                return_dict=False)[0]
            if cfg.world_size > 1 and live:                          # distri_sdxl_unet_pp.py:162-169 / 186-193
                B = 2 if split else b
                if self.output_buffer is None:
                    self.output_buffer = torch.empty((B, c, h, w), device=output.device, dtype=output.dtype)
                strip = output.contiguous()
                bs, _, hs, _ = strip.shape
                batch0 = cfg.batch_idx() if split else 0
                row0 = self._strip_row0(hs, h)
                _lib.check(_lib.lib().df_output_gather(cm.world, strip.data_ptr(), self.output_buffer.data_ptr(), B, c, h, w,
                                                       bs, hs, batch0, row0, 0, cm.output_off,
                                                       torch.cuda.current_stream().cuda_stream), "df_output_gather")
                output = self.output_buffer
            elif cfg.world_size > 1:
                # registration pass: buffers do not exist yet, the value is never consumed
                B = 2 if split else b
                output = output.new_zeros((B, c, h, w))
            if cm is not None:
                cm.join()
            if record:
                if self.static_inputs is None:                       # distri_sdxl_unet_pp.py:194-201
                    self.static_inputs = {"sample": sample, "timestep": timestep,
                                          "encoder_hidden_states": encoder_hidden_states,
                                          "added_cond_kwargs": added_cond_kwargs}
                self.synchronize()

        if return_dict:
            output = _output_cls()(sample=output)
        else:
            output = (output,)
        self.counter += 1
        return output

    @property
    def add_embedding(self):
        return self.model.add_embedding
