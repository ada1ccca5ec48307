"""DistriGroupNorm -- drop-in for distrifuser/modules/pp/groupnorm.py:10-97.

The statistics reduction, the cross-rank exchange of (E[x], E[x^2]) and the normalise+affine pass run in
df_groupnorm_fwd (csrc/groupnorm.cu).  Statistics travel in fp32 (the reference ships them in the activation
dtype, groupnorm.py:34 / SURVEY D-5); every mode formula, the local-count Bessel factor (D-1) and the
negative-variance patch (D-3) follow the reference."""
import torch
from torch import nn

from ... import _lib
from ...utils import DistriConfig
from ..base_module import BaseModule, nvtx_range

MODE_LOCAL, MODE_SYNC, MODE_CORRECTED, MODE_STALE = 0, 1, 2, 3


class DistriGroupNorm(BaseModule):
    def __init__(self, module: nn.GroupNorm, distri_config: DistriConfig):
        assert isinstance(module, nn.GroupNorm)
        super().__init__(module, distri_config)
        self.replicated = False         # set by tensor parallelism: every rank normalises its whole tensor, nothing is exchanged
        self.fuse_silu = False          # set by the block-level fusion in DistriUNetPP
        self._scratch = None

    def _plan(self):
        """-> (kernel mode, bessel, neg_var_fallback) for this call, following groupnorm.py:29-93."""
        cfg = self.distri_config
        if cfg.n_device_per_batch == 1 or self.replicated:
            return MODE_LOCAL, 0, 0                                  # reference leaves the stock module (unwrapped)
        stat_modes = cfg.mode in ("stale_gn", "corrected_async_gn")
        neg_fb = int(cfg.mode == "corrected_async_gn")
        if stat_modes:
            if not self._bound():
                return MODE_LOCAL, 1, neg_fb                         # groupnorm.py:43-44 (registration pass)
            if self._is_sync_step():
                return MODE_SYNC, 1, neg_fb                          # groupnorm.py:45-47
            return (MODE_CORRECTED if neg_fb else MODE_STALE), 1, neg_fb   # groupnorm.py:48-56
        if self._is_sync_step() or cfg.mode in ("sync_gn", "full_sync"):
            return (MODE_SYNC if self._bound() else MODE_LOCAL), 1, 0      # groupnorm.py:74-91
        return MODE_LOCAL, 0, 0                                      # groupnorm.py:92-93 (stock nn.GroupNorm)

    @nvtx_range("DistriGroupNorm")
    def forward(self, x: torch.Tensor, addend: torch.Tensor | None = None, pad_for=None) -> torch.Tensor:
        """`addend` ([b, C], optional) is added to every pixel before the norm: GroupNorm(x + addend[:, :, None, None]).
        `pad_for` (a DistriConv2dPP that consumes this output, optional): the result is returned as the conv's PADDED input
        [b, C, h+2, w] with both halo rows in place (boundary rows shipped to the neighbours by the same kernel): feed it to
        pad_for.forward_padded()."""
        module = self.module
        cfg = self.distri_config
        assert x.ndim == 4
        self._require_cuda_half(x, "DistriGroupNorm")
        b, c, h, w = x.shape
        G = module.num_groups
        if cfg.n_device_per_batch > 1 and not self.replicated and self._recording() and self.idx is None:
            # the reference registers only in the two statistics modes (groupnorm.py:29-35); the peer-memory
            # exchange needs a slot in every mode that synchronises (sync_gn / full_sync / warm-up steps)
            self.idx = self.comm_manager.register_tensor([2, b, G, 1, 1, 1], torch.float32, layer_type="gn")
        mode, bessel, neg_fb = self._plan()
        x = x.contiguous(memory_format=torch.channels_last)
        halo = pad_for.halo_plan(x) if pad_for is not None else None
        if halo is None:
            y = torch.empty_like(x, memory_format=torch.channels_last)
        else:
            y = torch.empty((b, c, h + 2, w), dtype=x.dtype, device=x.device, memory_format=torch.channels_last)
        L = _lib.lib()
        nbytes = L.df_groupnorm_scratch_bytes(b, G, h, w, c)
        if self._scratch is None or self._scratch.numel() < nbytes:
            self._scratch = torch.zeros(nbytes, dtype=torch.uint8, device=x.device)   # carries a self-resetting ticket
        cm = self.comm_manager
        if mode != MODE_LOCAL:
            comm, off, sb, mask = cm.group, cm.tensor_off[self.idx], cm.slot_bytes[self.idx], cm.group_mask()
        else:
            comm, off, sb, mask = _lib.null_comm(), 0, 0, 1
        gamma = module.weight.data_ptr() if module.affine else None
        beta = module.bias.data_ptr() if module.affine else None
        prof = _lib.PROFILE
        if prof is not None:
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
        apitch = 0
        if addend is not None:
            addend = addend.reshape(b, c)
            if addend.stride(1) != 1 or addend.stride(0) % 8 != 0 or addend.data_ptr() % 16 != 0:
                addend = addend.contiguous()
            apitch = addend.stride(0)                 # a column slice of the batched time-embedding projection: no copy
            assert addend.dtype == x.dtype
        st = torch.cuda.current_stream().cuda_stream
        if halo is None:
            _lib.check(L.df_groupnorm_fwd(comm, x.data_ptr(), addend.data_ptr() if addend is not None else None, apitch, y.data_ptr(), gamma, beta, b, h, w, c, G, float(module.eps),
                                          mode, bessel, neg_fb, int(self.fuse_silu), self.idx or 0, off, sb, mask,
                                          self._scratch.data_ptr(), st), "df_groupnorm_fwd")
        else:
            h_idx, h_off, h_sb, up, down, push = halo
            _lib.check(L.df_groupnorm_halo_fwd(cm.group, x.data_ptr(), addend.data_ptr() if addend is not None else None, apitch, y.data_ptr(), gamma,
                                               beta, b, h, w, c, G, float(module.eps), mode, bessel, neg_fb, int(self.fuse_silu),
                                               self.idx or 0, off, sb, mask, self._scratch.data_ptr(), h_idx, h_off, h_sb, up, down,
                                               int(push), 1, st), "df_groupnorm_halo_fwd")
        if prof is not None:
            e1.record()
            prof.append(dict(kernel="groupnorm", kind="gn", flops=0.0, bytes=4.0 * x.numel(), shape=tuple(x.shape),
                             start=e0, end=e1))
        self.counter += 1
        return y
