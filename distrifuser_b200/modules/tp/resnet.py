"""DistriResnetBlock2DTP -- drop-in for distrifuser/modules/tp/resnet.py:10-201.

norm1 is replicated; conv1 and time_emb_proj shard the output channels, norm2 runs groups/n groups over the local channels
(GroupNorm kernel in local mode, time-embedding addend and SiLU fused), conv2 shards the input channels and runs without
bias.  df_allreduce_fwd then sums the partials and adds conv2.bias, the shortcut and the shortcut's bias in one pass
(resnet.py:177-199).  The shortcut is the wrapped block's own conv_shortcut.

The GroupNorm and GEMM kernels read channels in groups of 8.  When the local share of channels is not a multiple of 8 (e.g.
20 channels of a narrow model over 4 devices), the shard is padded with whole dummy groups whose weights are zero: their
normalised value is exactly 0 and their conv2 columns are zero, so the result does not change."""
import torch
from torch import nn
from torch.nn import functional as F

from ...utils import DistriConfig
from ..base_module import nvtx_range
from .base import TPModule, replicated_group_norm, shard_range


def _padded(t: torch.Tensor, size: int, dim: int = 0) -> torch.Tensor:
    """t zero-padded to `size` along `dim`."""
    if t.shape[dim] == size:
        return t.clone()
    shape = list(t.shape)
    shape[dim] = size - t.shape[dim]
    return torch.cat([t, t.new_zeros(shape)], dim)


class DistriResnetBlock2DTP(TPModule):
    def __init__(self, module: nn.Module, distri_config: DistriConfig):
        super().__init__(module, distri_config)
        n, r = distri_config.n_device_per_batch, distri_config.split_idx()
        assert getattr(module, "time_embedding_norm", "default") == "default" and module.output_scale_factor == 1.0
        conv1, conv2, temb, norm2 = module.conv1, module.conv2, module.time_emb_proj, module.norm2
        c0, c1 = shard_range(conv1.out_channels, n, r)
        assert norm2.num_groups % n == 0, "norm2 groups must split over the devices"
        groups = norm2.num_groups // n
        cpg = (c1 - c0) // groups
        extra = 0
        while (c1 - c0 + extra * cpg) % 8:
            extra += 1
        width = c1 - c0 + extra * cpg
        dev, dt = conv1.weight.device, conv1.weight.dtype
        with torch.no_grad():
            sc1 = nn.Conv2d(conv1.in_channels, width, conv1.kernel_size, conv1.stride, conv1.padding, bias=conv1.bias is not None,
                            device=dev, dtype=dt)
            sc1.weight.copy_(_padded(conv1.weight[c0:c1], width))
            if conv1.bias is not None:
                sc1.bias.copy_(_padded(conv1.bias[c0:c1], width))
            st = nn.Linear(temb.in_features, width, bias=temb.bias is not None, device=dev, dtype=dt)
            st.weight.copy_(_padded(temb.weight[c0:c1], width))
            if temb.bias is not None:
                st.bias.copy_(_padded(temb.bias[c0:c1], width))
            sn2 = nn.GroupNorm(groups + extra, width, norm2.eps, norm2.affine, device=dev, dtype=dt)
            if norm2.affine:
                sn2.weight.copy_(_padded(norm2.weight[c0:c1], width))
                sn2.bias.copy_(_padded(norm2.bias[c0:c1], width))
            sc2 = nn.Conv2d(width, conv2.out_channels, conv2.kernel_size, conv2.stride, conv2.padding, bias=conv2.bias is not None,
                            device=dev, dtype=dt)
            sc2.weight.copy_(_padded(conv2.weight[:, c0:c1], width, 1))
            if conv2.bias is not None:
                sc2.bias.copy_(conv2.bias)
        module.conv1, module.time_emb_proj, module.conv2 = sc1, st, sc2
        module.norm1, module.norm2 = replicated_group_norm(module.norm1, distri_config), replicated_group_norm(sn2, distri_config)
        module.norm1.fuse_silu = module.norm2.fuse_silu = True
        # the UNet's batched time-embedding GEMM (compat UNet2DConditionModel._batched_temb) reads these sharded weights and
        # folds conv1.bias into the embedding
        module.fused_norm_act = True
        self._tail = None

    def _tail_bias(self):
        """conv2.bias + conv_shortcut.bias, cached on the parameters' versions."""
        m = self.module
        b2, sc = m.conv2.bias, m.conv_shortcut
        if sc is None or sc.bias is None:
            return b2
        key = (b2._version, sc.bias._version, b2.data_ptr(), sc.bias.data_ptr())
        if self._tail is None or self._tail[0] != key:
            if torch.cuda.is_current_stream_capturing():
                raise RuntimeError("conv biases changed since the last eager call; run one eager UNet call before capture")
            with torch.no_grad():
                self._tail = (key, (b2.detach() + sc.bias.detach()).contiguous())
        return self._tail[1]

    @nvtx_range("DistriResnetBlock2DTP")
    def forward(self, input_tensor: torch.Tensor, temb: torch.Tensor, scale: float = 1.0) -> torch.Tensor:
        assert scale == 1.0
        self._require_cuda_half(input_tensor, "DistriResnetBlock2DTP")
        m = self.module
        x = input_tensor.contiguous(memory_format=torch.channels_last)
        h = m.norm1(x)                                                   # GroupNorm + SiLU, replicated
        t = getattr(m, "temb_proj", None)
        folded = t is not None and getattr(m, "temb_has_conv1_bias", False)
        h = F.conv2d(h, m.conv1.weight, None if folded else m.conv1.bias, padding=m.conv1.padding)
        if t is None:
            t = F.linear(F.silu(temb), m.time_emb_proj.weight, m.time_emb_proj.bias)
        h = m.norm2(h, addend=t)                                         # GroupNorm(h + t) + SiLU over the local groups
        partial = F.conv2d(h, m.conv2.weight, None, padding=m.conv2.padding).contiguous(memory_format=torch.channels_last)
        sc = m.conv_shortcut
        res = x if sc is None else F.conv2d(x, sc.weight, None).contiguous(memory_format=torch.channels_last)
        out = self._all_reduce(partial, torch.empty_like(partial, memory_format=torch.channels_last), bias=self._tail_bias(),
                               residual=res)
        self.counter += 1
        return out
