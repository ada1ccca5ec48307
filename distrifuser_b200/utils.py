"""DistriConfig and PatchParallelismCommManager -- same names, constructor signatures and method names as the
reference (distrifuser/utils.py:23-110 and :112-199); internals are B200-native.

The reference ships activations with batched async NCCL all_gathers into one flat buffer per peer.  Here every
rank owns a *symmetric arena* mapped into all peers with CUDA IPC (NVLink 5 / NVSwitch peer memory); producers
store straight into the peers' slots and stamp release flags, consumers acquire the flags on the device.  The
epoch clock lives in device memory, so a captured CUDA graph replays unchanged step after step.
"""
from __future__ import annotations

import ctypes as C
import os

import torch
from torch import distributed as dist

from . import _lib
from ._lib import AR_RING, DfComm, NBANKS


def is_power_of_2(n: int) -> bool:
    return (n & (n - 1) == 0) and n != 0


class DistriConfig:
    """Reference: distrifuser/utils.py:23-110 (arguments, derived fields, batch_idx / split_idx)."""

    def __init__(
        self,
        height: int = 1024,
        width: int = 1024,
        do_classifier_free_guidance: bool = True,
        split_batch: bool = True,
        warmup_steps: int = 4,
        comm_checkpoint: int = 60,
        mode: str = "corrected_async_gn",
        use_cuda_graph: bool = True,
        parallelism: str = "patch",
        split_scheme: str = "row",
        verbose: bool = False,
    ):
        if dist.is_available() and dist.is_initialized():
            rank, world_size = dist.get_rank(), dist.get_world_size()
        elif "RANK" in os.environ and "WORLD_SIZE" in os.environ:
            # one process per GPU (torchrun); NCCL is the bootstrap / rendezvous plane only -- the data path is
            # peer memory (see PatchParallelismCommManager)
            backend = "nccl" if torch.cuda.is_available() else "gloo"
            dist.init_process_group(backend)
            rank, world_size = dist.get_rank(), dist.get_world_size()
        else:
            rank, world_size = 0, 1                                     # utils.py:44-47 (single GPU)
        assert is_power_of_2(world_size)                                # utils.py:49
        assert world_size <= _lib.MAX_WORLD, (
            f"distrifuser_b200 shards one image over the GPUs of ONE NVSwitch box (<= {_lib.MAX_WORLD} ranks, "
            f"DF_MAX_WORLD); got world_size={world_size}")
        assert mode in ("corrected_async_gn", "stale_gn", "sync_gn", "separate_gn", "full_sync", "no_sync")
        if parallelism not in ("patch", "tensor"):
            raise NotImplementedError(
                f"parallelism={parallelism!r}: distrifuser_b200 implements \"patch\" and \"tensor\" (naive_patch is out of scope)")

        self.world_size = world_size
        self.rank = rank
        self.height = height
        self.width = width
        self.do_classifier_free_guidance = do_classifier_free_guidance
        self.split_batch = split_batch
        self.warmup_steps = warmup_steps
        self.comm_checkpoint = comm_checkpoint       # kept for API parity; publication is per layer here
        self.mode = mode
        self.use_cuda_graph = use_cuda_graph
        self.parallelism = parallelism
        self.split_scheme = split_scheme
        self.verbose = verbose

        if do_classifier_free_guidance and split_batch:                 # utils.py:68-75
            n_device_per_batch = world_size // 2
            if n_device_per_batch == 0:
                n_device_per_batch = 1
        else:
            n_device_per_batch = world_size
        self.n_device_per_batch = n_device_per_batch
        if parallelism == "tensor" and n_device_per_batch == 1:
            # the reference falls back to the unwrapped model here; this package has no second single-device path
            raise NotImplementedError(
                "parallelism=\"tensor\" over one device per CFG branch is the unsharded model: use parallelism=\"patch\", "
                "which runs exactly that on one device")

        if torch.cuda.is_available():
            ndev = torch.cuda.device_count()
            if os.environ.get("DISTRIFUSER_B200_SHARE_GPU") == "1":
                local = 0                                               # test hook: all ranks on one device
            else:
                local = int(os.environ.get("LOCAL_RANK", rank)) % max(ndev, 1)
            device = torch.device(f"cuda:{local}")
            torch.cuda.set_device(device)                               # utils.py:80-82
        else:
            device = torch.device("cpu")                                # host-logic tests only; kernels need CUDA
        self.device = device

        batch_group = None
        split_group = None
        if do_classifier_free_guidance and split_batch and world_size >= 2:   # utils.py:84-96
            half = world_size // 2
            batch_groups = [dist.new_group(list(range(i * half, (i + 1) * half))) for i in range(2)]
            batch_group = batch_groups[self.batch_idx()]
            split_groups = [dist.new_group([i, i + half]) for i in range(half)]
            split_group = split_groups[self.split_idx()]
        self.batch_group = batch_group
        self.split_group = split_group

    def batch_idx(self, rank: int | None = None) -> int:                # utils.py:98-104
        if rank is None:
            rank = self.rank
        if self.do_classifier_free_guidance and self.split_batch:
            return 1 - int(rank < (self.world_size // 2))
        return 0

    def split_idx(self, rank: int | None = None) -> int:                # utils.py:106-109
        if rank is None:
            rank = self.rank
        return rank % self.n_device_per_batch

    # -- additions used by the B200 path
    def patch_group_ranks(self) -> list[int]:
        """World ranks of the patch group of this rank (the reference's batch_group, utils.py:87-90)."""
        n = self.n_device_per_batch
        if self.do_classifier_free_guidance and self.split_batch and self.world_size >= 2:
            base = self.batch_idx() * (self.world_size // 2)
        else:
            base = 0
        return list(range(base, base + n))


def _align(x: int, a: int) -> int:
    return (x + a - 1) // a * a


def _dense(t: torch.Tensor) -> bool:
    """[rows, C] in memory: NHWC (channels_last) for 4-D tensors, contiguous otherwise."""
    return t.is_contiguous(memory_format=torch.channels_last) if t.ndim == 4 else t.is_contiguous()


class _Holder:
    """Exposes a raw device allocation to torch through __cuda_array_interface__."""

    def __init__(self, ptr: int, nbytes: int):
        self.__cuda_array_interface__ = {"shape": (nbytes,), "typestr": "|u1", "data": (ptr, False), "version": 3}


class PatchParallelismCommManager:
    """Reference: distrifuser/utils.py:112-199.  Same method names; `comm_checkpoint` batching is replaced by
    per-layer peer stores, and `handles[idx].wait()` by device-side flag acquisition."""

    def __init__(self, distri_config: DistriConfig):
        self.distri_config = distri_config
        self.torch_dtype = None
        self.numel = 0
        self.numel_dict = {}
        self.buffer_list = None          # set by create_buffer (list of per-peer arena views, bank 0)
        self.starts, self.ends, self.shapes = [], [], []
        self.idx_queue = []
        self.handles = None
        # B200 path state
        self.slot_bytes: list[int] = []
        self.dtypes: list[torch.dtype] = []
        self.tensor_off: list[int] = []
        self.layer_types: list[str] = []
        self.output_spec = None          # (B, C, H, W) of the final epsilon, registered by DistriUNetPP
        self.output_off = 0
        self.ar_bytes: list[int] = []    # payload bytes of every registered all-reduce site (tensor parallelism), in call order
        self.ar_ring_off = 0
        self.ar_slot_bytes = 0
        self.arena = None                # torch uint8 view of this rank's arena
        self._arena_ptr = None
        self._peer_ptrs: list[int] = []
        self.group: DfComm | None = None
        self.world: DfComm | None = None
        self.clock = None
        self.comm_stream = None
        self._keepalive: list[torch.Tensor] = []
        self._forked = False
        self.epoch_host = 0              # host mirror of the device clock (debug / get_buffer_list only)

    # ------------------------------------------------------------------ registration (utils.py:130-149)
    def register_tensor(self, shape, torch_dtype: torch.dtype, layer_type: str = None, slot_bytes: int | None = None) -> int:
        assert self.arena is None, "register_tensor after create_buffer"
        if self.torch_dtype is None:
            self.torch_dtype = torch_dtype
        numel = 1
        for dim in shape:
            numel *= dim
        self.starts.append(self.numel)
        self.numel += numel
        self.ends.append(self.numel)
        self.shapes.append(tuple(shape))
        if layer_type is not None:
            self.numel_dict[layer_type] = self.numel_dict.get(layer_type, 0) + numel
        esize = torch.empty((), dtype=torch_dtype).element_size()
        self.slot_bytes.append(_align(slot_bytes if slot_bytes is not None else numel * esize, 256))
        self.dtypes.append(torch_dtype)
        self.layer_types.append(layer_type or "")
        return len(self.starts) - 1

    def register_output(self, B: int, Cc: int, H: int, W: int):
        self.output_spec = (B, Cc, H, W)

    def register_allreduce(self, nbytes: int) -> int:
        """One all-reduce site of the tensor-parallel path (called in execution order during the registration pass); returns
        its site index.  The sites share one small ring of slots sized for the largest of them, so the arena does not grow
        with their number."""
        assert self.arena is None, "register_allreduce after create_buffer"
        self.ar_bytes.append(int(nbytes))
        return len(self.ar_bytes) - 1

    # ------------------------------------------------------------------ arena layout (pure host arithmetic)
    def _layout(self):
        """Offsets of the symmetric arena: [group flags u32[nt][n] | world flags u32[world] (| all-reduce flags
        u32[DF_AR_RING][n])] then DF_NBANKS banks, each holding n source slots per registered tensor and one output image,
        then (tensor parallelism) the all-reduce ring: DF_AR_RING x n slots of the largest registered all-reduce.
        Returns (total_bytes, bank_stride)."""
        cfg = self.distri_config
        n, world = cfg.n_device_per_batch, cfg.world_size
        nt = len(self.slot_bytes)
        self._flags_group_off = 0
        self._flags_world_off = _align(4 * max(nt, 1) * n, 256)
        header = _align(self._flags_world_off + 4 * world, 1024)
        self._flags_ar_off = 0
        if self.ar_bytes:
            self._flags_ar_off = _align(self._flags_world_off + 4 * world, 256)
            header = _align(self._flags_ar_off + 4 * AR_RING * n, 1024)
        off = header
        self.tensor_off = []
        for sb in self.slot_bytes:
            self.tensor_off.append(off)
            off += n * sb
        self.output_off = off
        if self.output_spec is not None:
            B, Cc, H, W = self.output_spec
            off += _align(B * Cc * H * W * 2, 1024)
        bank_stride = _align(off - header, 1024)
        total = header + NBANKS * bank_stride
        self.ar_slot_bytes = _align(max(self.ar_bytes), 256) if self.ar_bytes else 0
        self.ar_ring_off = total
        return total + AR_RING * n * self.ar_slot_bytes, bank_stride

    # ------------------------------------------------------------------ arena creation (utils.py:151-164)
    def create_buffer(self):
        cfg = self.distri_config
        assert cfg.device.type == "cuda", "the communication arena needs a CUDA device"
        L = _lib.lib()
        n, world = cfg.n_device_per_batch, cfg.world_size
        nt = len(self.slot_bytes)
        if cfg.rank == 0 and cfg.verbose:
            print(f"Create buffer with {self.numel / 1e6:.3f}M parameters for {nt} tensors on each device.")
            for layer_type, numel in self.numel_dict.items():
                print(f"  {layer_type}: {numel / 1e6:.3f}M parameters")
        total, bank_stride = self._layout()
        # tensor_off is relative to the arena base; bank k adds k*bank_stride
        ptr = C.c_void_p()
        handle = (C.c_ubyte * _lib.IPC_HANDLE_BYTES)()
        _lib.check(L.df_symm_alloc(total, C.byref(ptr), handle), "df_symm_alloc")
        self._arena_ptr = ptr.value
        self._arena_bytes = total
        self.arena = torch.as_tensor(_Holder(ptr.value, total), device=cfg.device)
        handles = [None] * world
        if world > 1:
            dist.all_gather_object(handles, bytes(handle))
        else:
            handles = [bytes(handle)]
        self._peer_ptrs = []
        for r in range(world):
            if r == cfg.rank:
                self._peer_ptrs.append(ptr.value)
            else:
                p = C.c_void_p()
                buf = (C.c_ubyte * _lib.IPC_HANDLE_BYTES).from_buffer_copy(handles[r])
                _lib.check(L.df_symm_open(buf, C.byref(p)), f"df_symm_open(rank {r})")
                self._peer_ptrs.append(p.value)
        # local scratch: clock [4] u32, tickets [nt+1] u32
        self.clock = torch.zeros(4, dtype=torch.int32, device=cfg.device)
        self._tickets = torch.zeros(nt + 3, dtype=torch.int32, device=cfg.device)   # [nt]: world gather, [nt + 2]: all-reduce
        members = cfg.patch_group_ranks()
        g = DfComm()
        for i, r in enumerate(members):
            g.base[i] = self._peer_ptrs[r]
            g.flags[i] = self._peer_ptrs[r] + self._flags_group_off
        g.clock, g.tickets = self.clock.data_ptr(), self._tickets.data_ptr()
        g.bank_stride, g.world, g.rank = bank_stride, n, cfg.split_idx()
        # device-side flag waits trap (CUDA error instead of a hung GPU) after this long; raise it when a rank may stall for
        # a long time inside a step (cudnn.benchmark autotune in the eager pre-run, ncu / compute-sanitizer serialisation)
        timeout_ns = int(float(os.environ.get("DF_SPIN_TIMEOUT_S", "0")) * 1e9)
        g.spin_timeout_ns = timeout_ns
        w = DfComm()
        for r in range(world):
            w.base[r] = self._peer_ptrs[r]
            w.flags[r] = self._peer_ptrs[r] + self._flags_world_off
        w.clock, w.tickets = self.clock.data_ptr(), self._tickets.data_ptr() + 4 * nt   # world ticket after the group's
        w.bank_stride, w.world, w.rank = bank_stride, world, cfg.rank
        w.spin_timeout_ns = timeout_ns
        self.group, self.world, self.bank_stride = g, w, bank_stride
        # publication stream: the asynchronous K/V transfers have a whole denoise step of slack, so they must not pre-empt the
        # compute kernels' CTA scheduling (DF_COMM_PRIO=-1 restores the high priority of round 1)
        self.comm_stream = torch.cuda.Stream(device=cfg.device, priority=int(os.environ.get("DF_COMM_PRIO", "0")))
        import atexit
        import weakref
        ref = weakref.ref(self)
        atexit.register(lambda: ref() is not None and ref().close())
        self.handles = [None for _ in range(nt)]
        self.buffer_list = [self.arena for _ in range(n)]     # non-None marks "buffers created" (utils.py:160-163); views: get_buffer_list
        if world > 1:
            dist.barrier()          # every arena is mapped everywhere before the first peer store
        torch.cuda.synchronize(cfg.device)

    def get_buffer_list(self, idx: int, bank: int | None = None) -> list[torch.Tensor]:
        """Per-peer views of tensor `idx` (utils.py:166-168).  `bank` defaults to the bank of the last published
        epoch; with rotating banks these views are only meaningful for inspection, kernels address slots themselves."""
        cfg = self.distri_config
        if bank is None:
            bank = int(self.clock[0].item()) % NBANKS
        dtype = self.dtypes[idx]
        esize = torch.empty((), dtype=dtype).element_size()
        out = []
        for s in range(cfg.n_device_per_batch):
            o = bank * self.bank_stride + self.tensor_off[idx] + s * self.slot_bytes[idx]
            nb = (self.ends[idx] - self.starts[idx]) * esize
            out.append(self.arena[o:o + nb].view(dtype).view(self.shapes[idx]))
        return out

    # ------------------------------------------------------------------ step protocol
    # ALL-REDUCE RING REUSE (tensor parallelism).  Every UNet call is a synchronous step (df_step_begin kind 0), and all-reduce
    # `site` of the call with epoch e carries seq = e * nsites + site: consecutive all-reduces of a rank -- also across calls --
    # have consecutive seq and alternate between the DF_AR_RING = 2 ring slots; flags are compared wrap-safely.  A rank that
    # pushes all-reduce k+2 into slot (k % 2) of a peer has passed the wait of all-reduce k+1, i.e. seen that peer's k+1 flag;
    # the peer stamps that flag in its k+1 kernel, which by stream order starts after its all-reduce k kernel -- the last read
    # of slot (k % 2) -- completed.  So a slot is never overwritten while it is read, without any acknowledgement.  That holds
    # only if an all-reduce kernel cannot start before the previous kernel of its stream has finished: df_allreduce_fwd is
    # therefore always launched WITHOUT programmatic dependent launch, whatever DF_PDL selects for the other kernels (those
    # touch no memory before griddepcontrol.wait, i.e. before the all-reduce that precedes them has completed).  Members
    # that own no heads push nothing but still stamp and wait, so every member passes every all-reduce.
    #
    # BANK-REUSE INVARIANT.  Bank e % 3 is overwritten by the peers' stores of epoch e+3 without any "consumed"
    # acknowledgement.  That is safe only because every UNet call ends with df_output_gather, which makes each rank wait
    # for the epsilon strip of EVERY world rank: no rank can start call t+1 before all ranks finished the kernels of call
    # t, so ranks drift by < 1 call and a store of epoch e+3 can never meet a read of epoch e (reads of epoch e happen in
    # calls e and e+1 only).  A path that skips the gather (e.g. returning the local strip) must add its own per-call
    # world barrier, or stale K/V / halo rows get corrupted silently.
    def step_begin(self, kind: int):
        """kind 0 = synchronous, 1 = asynchronous, 2 = frozen (see df_step_begin)."""
        st = torch.cuda.current_stream().cuda_stream
        _lib.check(_lib.lib().df_step_begin(self.clock.data_ptr(), kind, st), "df_step_begin")
        self.epoch_host += 1

    def all_reduce(self, site: int, partial: torch.Tensor | None, out: torch.Tensor, bias: torch.Tensor | None = None,
                   residual: torch.Tensor | None = None, contrib_mask: int | None = None) -> torch.Tensor:
        """out = sum of the patch group's partials + bias (+ residual) on every member (df_allreduce_fwd).  Tensors are NHWC
        (channels_last) 4-D or [..., C] sequences, contiguous in that layout; partial None = this member owns nothing.  Before
        create_buffer (registration pass) the result is this rank's partial + bias (+ residual): shapes only."""
        cfg = self.distri_config
        C = out.shape[1] if out.ndim == 4 else out.shape[-1]
        rows = out.numel() // C
        live = self.arena is not None
        n = cfg.n_device_per_batch if live else 1
        if contrib_mask is None:
            contrib_mask = (1 << n) - 1
        if not live:
            comm, contrib_mask = _lib.null_comm(), int(partial is not None)
        else:
            comm = self.group
        for t in (partial, residual):
            assert t is None or (t.shape == out.shape and t.dtype == torch.float16 and _dense(t)), "all_reduce: layout"
        assert _dense(out) and (bias is None or (bias.is_contiguous() and bias.numel() == C))
        prof = _lib.PROFILE
        if prof is not None:
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
        _lib.check(_lib.lib().df_allreduce_fwd(
            comm, None if partial is None else partial.data_ptr(), out.data_ptr(), rows, C,
            None if bias is None else bias.data_ptr(), None if residual is None else residual.data_ptr(), contrib_mask,
            site, max(len(self.ar_bytes), 1), self.ar_ring_off, self.ar_slot_bytes, self._flags_ar_off if live else 0,
            len(self.slot_bytes) + 2, torch.cuda.current_stream().cuda_stream), "df_allreduce_fwd")
        if prof is not None:
            e1.record()
            nb = 2.0 * out.numel()
            prof.append(dict(kernel="allreduce_kernel", kind="allreduce", flops=0.0, bytes=nb * (n + 2 + (residual is not None)),
                             shape=(rows, C), start=e0, end=e1))
        return out

    def group_mask(self) -> int:
        return (1 << self.distri_config.n_device_per_batch) - 1

    def peers_mask(self) -> int:
        return self.group_mask() & ~(1 << self.distri_config.split_idx())

    def enqueue(self, idx: int, tensor: torch.Tensor, async_stream: bool = True, num_ctas: int | None = None):
        """Publish `tensor` (this rank's fresh activation of layer idx) into every peer's slot
        (utils.py:181-190: copy into the flat buffer + batched async all_gather)."""
        L = _lib.lib()
        esz = tensor.element_size()
        if tensor.is_contiguous():
            rows, row_bytes, pitch = 1, tensor.numel() * esz, tensor.numel() * esz
        else:
            # a [.., rows, cols] view with a uniform row pitch (e.g. the k|v columns of a fused q|k|v projection)
            assert tensor.stride(-1) == 1 and tensor.ndim >= 2
            cols, pitch_el = tensor.shape[-1], tensor.stride(-2)
            for dim in range(tensor.ndim - 2):
                assert tensor.stride(dim) == tensor.stride(dim + 1) * tensor.shape[dim + 1], "rows must have one pitch"
            rows, row_bytes, pitch = tensor.numel() // cols, cols * esz, pitch_el * esz
        nbytes = rows * row_bytes
        if num_ctas is None:
            # synchronous steps wait for the data right away: use the whole NVLink; asynchronous publication hides under the
            # attention that follows and should take few SM slots
            num_ctas = int(os.environ.get("DF_PUB_CTAS", "64")) if async_stream else 296
        main = torch.cuda.current_stream()
        if async_stream:
            self.comm_stream.wait_stream(main)      # fork: publication overlaps the compute that follows
            self._forked = True
            stream = self.comm_stream
            self._keepalive.append(tensor)
        else:
            stream = main
        _lib.check(L.df_slot_publish(self.group, tensor.data_ptr(), rows, row_bytes, pitch, self.tensor_off[idx],
                                     self.slot_bytes[idx], idx, self.peers_mask(), num_ctas, stream.cuda_stream),
                   "df_slot_publish")

    def wait(self, idx: int):
        _lib.check(_lib.lib().df_slot_wait(self.group, idx, self.peers_mask(),
                                           torch.cuda.current_stream().cuda_stream), "df_slot_wait")

    def communicate(self):
        """Kept for API parity (utils.py:170-179): publication happens per layer, nothing is queued."""
        self.idx_queue = []

    def join(self):
        """Re-join the communication stream (end of a UNet call; required before a graph capture ends)."""
        if self._forked:
            torch.cuda.current_stream().wait_stream(self.comm_stream)
            self._forked = False
        self._keepalive.clear()

    def clear(self):                                                    # utils.py:192-199
        self.communicate()
        self.join()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def close(self):
        """Unmaps the peers' arenas and frees this rank's (also run from __del__ and at interpreter exit)."""
        if getattr(self, "_arena_ptr", None) is None:
            return
        L = _lib.lib()
        torch.cuda.synchronize(self.distri_config.device)
        for r, p in enumerate(self._peer_ptrs):
            if r != self.distri_config.rank:
                L.df_symm_close(p)
        self.arena = None
        L.df_symm_free(self._arena_ptr)
        self._arena_ptr = None
