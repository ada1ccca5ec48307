"""Shared pieces of the tensor-parallel wrappers: the all-reduce site protocol and weight slicing."""
import torch
from torch import nn

from ..base_module import BaseModule
from ..pp.groupnorm import DistriGroupNorm


def shard_range(size: int, n: int, r: int) -> tuple[int, int]:
    """[start, end) of member r's equal share of `size` (size % n == 0)."""
    assert size % n == 0, f"{size} does not split over {n} devices"
    k = size // n
    return r * k, (r + 1) * k


def linear_like(src: nn.Linear, weight: torch.Tensor, bias: torch.Tensor | None) -> nn.Linear:
    out = nn.Linear(weight.shape[1], weight.shape[0], bias=bias is not None, device=weight.device, dtype=weight.dtype)
    with torch.no_grad():
        out.weight.copy_(weight)
        if bias is not None:
            out.bias.copy_(bias)
    return out


def replicated_group_norm(module: nn.GroupNorm, distri_config) -> DistriGroupNorm:
    """The GroupNorm kernel in local mode: every member normalises its whole tensor, nothing is exchanged."""
    gn = DistriGroupNorm(module, distri_config)
    gn.replicated = True
    return gn


class TPModule(BaseModule):
    """A wrapper whose output is the sum of the patch group's partial results (one all-reduce site per call)."""

    def _all_reduce(self, partial, out, bias=None, residual=None, contrib_mask=None):
        cm = self.comm_manager
        if self._recording() and self.idx is None:
            self.idx = cm.register_allreduce(out.numel() * out.element_size())
        return cm.all_reduce(self.idx or 0, partial, out, bias=bias, residual=residual, contrib_mask=contrib_mask)
