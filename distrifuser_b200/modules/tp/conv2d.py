"""DistriConv2dTP -- drop-in for distrifuser/modules/tp/conv2d.py:9-56 (conv_out and the down / up-sampler convolutions).

Input channels are sharded; each member convolves its channel slice in cuDNN without bias and df_allreduce_fwd sums the
partials and adds the bias (conv2d.py:52-54)."""
import torch
from torch import nn
from torch.nn import functional as F

from ...utils import DistriConfig
from ..base_module import nvtx_range
from .base import TPModule, shard_range


class DistriConv2dTP(TPModule):
    def __init__(self, module: nn.Conv2d, distri_config: DistriConfig):
        n, r = distri_config.n_device_per_batch, distri_config.split_idx()
        c0, c1 = shard_range(module.in_channels, n, r)
        sharded = nn.Conv2d(c1 - c0, module.out_channels, module.kernel_size, module.stride, module.padding,
                            module.dilation, module.groups, module.bias is not None, module.padding_mode,
                            device=module.weight.device, dtype=module.weight.dtype)
        with torch.no_grad():
            sharded.weight.copy_(module.weight[:, c0:c1])
            if module.bias is not None:
                sharded.bias.copy_(module.bias)
        super().__init__(sharded, distri_config)
        self.c0, self.c1 = c0, c1

    @nvtx_range("DistriConv2dTP")
    def forward(self, x: torch.Tensor, *args, **kwargs) -> torch.Tensor:
        self._require_cuda_half(x, "DistriConv2dTP")
        m = self.module
        xs = x[:, self.c0:self.c1].contiguous(memory_format=torch.channels_last)
        partial = F.conv2d(xs, m.weight, None, stride=m.stride, padding=m.padding, dilation=m.dilation, groups=m.groups)
        partial = partial.contiguous(memory_format=torch.channels_last)
        out = self._all_reduce(partial, torch.empty_like(partial, memory_format=torch.channels_last), bias=m.bias)
        self.counter += 1
        return out
