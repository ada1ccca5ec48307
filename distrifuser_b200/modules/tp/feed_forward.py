"""DistriFeedForwardTP -- drop-in for distrifuser/modules/tp/feed_forward.py:10-79.

The GEGLU projection is column-parallel and keeps [hidden slice ; gate slice] (feed_forward.py:26-35); it runs on the fused
tcgen05 GEMM + GEGLU epilogue when that supports the sharded shape, otherwise cuBLAS + df_geglu (the GEGLU module decides).
The second Linear is row-parallel without bias; df_allreduce_fwd sums the partials and adds the bias (feed_forward.py:77-79)."""
import torch
from torch import nn
from torch.nn import functional as F

from ...utils import DistriConfig
from ..base_module import nvtx_range
from .base import TPModule, linear_like, shard_range


class DistriFeedForwardTP(TPModule):
    def __init__(self, module: nn.Module, distri_config: DistriConfig):
        super().__init__(module, distri_config)
        n, r = distri_config.n_device_per_batch, distri_config.split_idx()
        proj, fc2 = module.net[0].proj, module.net[2]
        assert proj.out_features % (2 * n) == 0 and fc2.in_features % n == 0
        mid = fc2.in_features
        h0, h1 = shard_range(mid, n, r)
        rows = torch.cat([torch.arange(h0, h1), torch.arange(mid + h0, mid + h1)]).to(proj.weight.device)
        module.net[0].proj = linear_like(proj, proj.weight.data[rows], None if proj.bias is None else proj.bias.data[rows])
        module.net[2] = linear_like(fc2, fc2.weight.data[:, h0:h1], None if fc2.bias is None else fc2.bias.data)

    @nvtx_range("DistriFeedForwardTP")
    def forward(self, hidden_states: torch.Tensor, scale: float = 1.0) -> torch.Tensor:
        assert scale == 1.0
        self._require_cuda_half(hidden_states, "DistriFeedForwardTP")
        net = self.module.net
        h = net[1](net[0](hidden_states))
        partial = F.linear(h, net[2].weight)
        out = self._all_reduce(partial, torch.empty_like(partial), bias=net[2].bias)
        self.counter += 1
        return out
