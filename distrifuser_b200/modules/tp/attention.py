"""DistriAttentionTP -- drop-in for distrifuser/modules/tp/attention.py:10-177.

Heads are split over the patch group with the reference's remainder rule (attention.py:15-29).  Each member projects its
heads' q | k | v in one GEMM, runs df_attn_fwd over its local heads (one K/V segment), multiplies by its columns of to_out
without the bias, and df_allreduce_fwd sums the members' partials and adds the bias (attention.py:159-161)."""
import torch
from torch import nn
from torch.nn import functional as F

from ...utils import DistriConfig
from ..base_module import nvtx_range
from ..pp.attn import DistriAttentionPP
from .base import TPModule, linear_like


def head_split(heads: int, n: int, r: int) -> tuple[int, int]:
    """(first head, number of heads) of member r: the first heads % n members take one extra head."""
    sliced, rem = heads // n, heads % n
    if r < rem:
        return r * (sliced + 1), sliced + 1
    return rem * (sliced + 1) + (r - rem) * sliced, sliced


class DistriAttentionTP(TPModule, DistriAttentionPP):
    def __init__(self, module: nn.Module, distri_config: DistriConfig):
        n, r = distri_config.n_device_per_batch, distri_config.split_idx()
        heads = module.heads
        dim = module.to_q.out_features // heads
        start, count = head_split(heads, n, r)
        assert module.rescale_output_factor == 1.0
        cols = slice(start * dim, (start + count) * dim)
        sl = lambda lin: linear_like(lin, lin.weight.data[cols], None if lin.bias is None else lin.bias.data[cols])
        module.to_q, module.to_k, module.to_v = sl(module.to_q), sl(module.to_k), sl(module.to_v)
        out = module.to_out[0]
        module.to_out[0] = linear_like(out, out.weight.data[:, cols], out.bias.data if out.bias is not None else None)
        module.heads = count
        super().__init__(module, distri_config)       # DistriAttentionPP: fused to_kv of the local heads
        self.sliced_heads = count
        self.contrib_mask = sum(1 << m for m in range(n) if head_split(heads, n, m)[1] > 0)
        self._w_qkv, self._w_qkv_key = None, None

    def _qkv_weight(self):
        """[to_q ; to_kv] of the local heads as one matrix, rebuilt when either changes (version counters)."""
        wq, wkv = self.module.to_q.weight, self.to_kv.weight
        key = (wq._version, wkv._version, wq.data_ptr(), wkv.data_ptr(), wq.dtype, wq.device)
        if key != self._w_qkv_key:
            if torch.cuda.is_current_stream_capturing():
                raise RuntimeError("DistriAttentionTP: attention weights changed since the last eager call; run one eager "
                                   "UNet call before capturing CUDA graphs")
            with torch.no_grad():
                self._w_qkv = torch.cat([wq.detach(), wkv.detach()], 0).contiguous()
            self._w_qkv_key = key
        return self._w_qkv

    @nvtx_range("DistriAttentionTP")
    def forward(self, hidden_states, encoder_hidden_states=None, attention_mask=None, **kwargs):
        assert attention_mask is None
        self._require_cuda_half(hidden_states, "DistriAttentionTP")
        attn = self.module
        b, l, _ = hidden_states.shape
        to_out = attn.to_out[0]
        out = torch.empty((b, l, to_out.out_features), dtype=hidden_states.dtype, device=hidden_states.device)
        partial = None
        if self.sliced_heads > 0:
            to_q, to_kv = attn.to_q, self.to_kv
            cs = to_q.out_features
            if encoder_hidden_states is None and to_q.bias is None and to_kv.bias is None:
                qkv = F.linear(hidden_states, self._qkv_weight())      # q | k | v of the local heads in one GEMM
                q, kv = qkv[..., :cs], qkv[..., cs:]
            elif encoder_hidden_states is None:
                q, kv = to_q(hidden_states), to_kv(hidden_states)
            else:                                                     # K/V of the text recomputed every call (attention.py:117)
                q, kv = to_q(hidden_states), to_kv(encoder_hidden_states)
            o = self._attend(q, kv, kv.shape[1], 1, 0, False, kind="self" if encoder_hidden_states is None else "cross")
            partial = F.linear(o, to_out.weight)                     # row-parallel, bias after the sum (attention.py:156-161)
        residual = hidden_states.contiguous() if attn.residual_connection else None
        out = self._all_reduce(partial, out, bias=to_out.bias, residual=residual, contrib_mask=self.contrib_mask)
        out = attn.to_out[1](out)
        self.counter += 1
        return out
