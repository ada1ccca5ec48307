"""ctypes binding of libdistrifuser_b200.so (C ABI: include/distrifuser_b200.h).

The product path has no CPU or PyTorch fallback: if the extension is missing this module raises."""
from __future__ import annotations

import ctypes as C
import os

HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.environ.get("DF_LIB_PATH") or os.path.join(HERE, "libdistrifuser_b200.so")   # DF_LIB_PATH: a prebuilt variant (kernel experiments)

NBANKS = 3
MAX_WORLD = 8
IPC_HANDLE_BYTES = 64
TENSORMAP_BYTES = 128
AR_RING = 2          # DF_AR_RING: depth of the all-reduce slot ring (tensor parallelism)

EXPORTS = (
    "df_last_error", "df_version", "df_device_sm_count", "df_symm_alloc", "df_symm_open", "df_symm_close",
    "df_symm_free", "df_step_begin", "df_slot_publish", "df_slot_wait", "df_groupnorm_scratch_bytes",
    "df_groupnorm_fwd", "df_groupnorm_halo_fwd", "df_halo_push", "df_halo_assemble", "df_attn_make_kvmaps", "df_attn_workspace_bytes", "df_attn_fwd",
    "df_output_gather", "df_geglu", "df_add_layernorm", "df_bias_residual_add", "df_linear_supported", "df_linear_geglu_block", "df_linear_fwd",
    "df_allreduce_fwd",
)


class DfComm(C.Structure):
    _fields_ = [("base", C.c_void_p * MAX_WORLD), ("flags", C.c_void_p * MAX_WORLD), ("clock", C.c_void_p),
                ("tickets", C.c_void_p), ("bank_stride", C.c_uint64), ("spin_timeout_ns", C.c_uint64), ("world", C.c_int32),
                ("rank", C.c_int32)]


_lib = None


def lib():
    global _lib
    if _lib is None:
        if not os.path.exists(LIB_PATH):
            raise RuntimeError(
                f"{LIB_PATH} is missing: build it with `python -m distrifuser_b200.build` "
                "(distrifuser_b200 has no fallback path; the CUDA extension is the product)")
        L = C.CDLL(LIB_PATH)
        vp, u64, i32, u32, i64, f32 = C.c_void_p, C.c_uint64, C.c_int, C.c_uint32, C.c_int64, C.c_float
        L.df_last_error.restype = C.c_char_p
        L.df_version.restype = i32
        L.df_device_sm_count.argtypes = [C.POINTER(i32)]
        L.df_symm_alloc.argtypes = [C.c_size_t, C.POINTER(vp), vp]
        L.df_symm_open.argtypes = [vp, C.POINTER(vp)]
        L.df_symm_close.argtypes = [vp]
        L.df_symm_free.argtypes = [vp]
        L.df_step_begin.argtypes = [vp, i32, vp]
        L.df_slot_publish.argtypes = [DfComm, vp, u64, u64, u64, u64, u64, i32, u32, i32, vp]
        L.df_slot_wait.argtypes = [DfComm, i32, u32, vp]
        L.df_groupnorm_scratch_bytes.argtypes = [i32, i32, i32, i32, i32]
        L.df_groupnorm_scratch_bytes.restype = C.c_size_t
        L.df_groupnorm_fwd.argtypes = [DfComm, vp, vp, i64, vp, vp, vp, i32, i32, i32, i32, i32, f32, i32, i32, i32, i32, i32,
                                       u64, u64, u32, vp, vp]
        L.df_groupnorm_halo_fwd.argtypes = [DfComm, vp, vp, i64, vp, vp, vp, i32, i32, i32, i32, i32, f32, i32, i32, i32, i32, i32,
                                            u64, u64, u32, vp, i32, u64, u64, i32, i32, i32, i32, vp]
        L.df_halo_push.argtypes = [DfComm, vp, i32, i32, i32, i32, i32, u64, u64, i32, i32, vp]
        L.df_halo_assemble.argtypes = [DfComm, vp, vp, i32, i32, i32, i32, i32, u64, u64, i32, i32, i32, vp]
        L.df_attn_make_kvmaps.argtypes = [DfComm, u64, u64, i32, i32, i32, i32, vp, vp]
        L.df_attn_workspace_bytes.argtypes = [i32, i32, i32, i32, i32, i32]
        L.df_attn_workspace_bytes.restype = C.c_size_t
        L.df_attn_fwd.argtypes = [DfComm, vp, vp, vp, vp, i32, i32, i32, i32, i32, i64, i64, i64, i32, i32,
                                  C.POINTER(C.c_int32), i32, i32, f32, vp, C.c_size_t, vp]
        L.df_geglu.argtypes = [vp, vp, i64, i32, i64, i64, vp]
        L.df_add_layernorm.argtypes = [vp, vp, vp, vp, vp, vp, i64, i32, f32, vp]
        L.df_bias_residual_add.argtypes = [vp, vp, vp, vp, i64, i32, vp]
        L.df_linear_supported.argtypes = [i64, i32, i32, i32]
        L.df_linear_geglu_block.argtypes = [i64, i32, i32]
        L.df_linear_fwd.argtypes = [DfComm, vp, vp, vp, vp, vp, i64, i32, i32, i64, i64, i64, i64, i32, i32, i32, i32, i32, u32, u64,
                                    u64, i32, vp]
        L.df_allreduce_fwd.argtypes = [DfComm, vp, vp, i64, i32, vp, vp, u32, i32, i32, u64, u64, u64, i32, vp]
        L.df_output_gather.argtypes = [DfComm, vp, vp, i32, i32, i32, i32, i32, i32, i32, i32, i32, u64, vp]
        for name in EXPORTS:
            getattr(L, name)  # AttributeError if the header and the library disagree
        _lib = L
    return _lib


# kernels launched per C-ABI call (bench.py reports the count of OUR launches inside the timed region)
KERNELS_PER_CALL = {"df_groupnorm_fwd": 1, "df_groupnorm_halo_fwd": 1, "df_attn_fwd": 1, "df_halo_push": 1, "df_halo_assemble": 1,
                    "df_slot_publish": 1, "df_slot_wait": 1, "df_step_begin": 1, "df_output_gather": 2, "df_geglu": 1, "df_add_layernorm": 1, "df_bias_residual_add": 1,
                    "df_linear_fwd": 1, "df_allreduce_fwd": 1}
LAUNCHES = {"total": 0}
PROFILE = None   # bench.py sets this to a list; kernels then bracket their launch with CUDA events on the launching stream


def check(rc: int, what: str = ""):
    LAUNCHES["total"] += KERNELS_PER_CALL.get(what, 0)
    if rc != 0:
        raise RuntimeError(f"distrifuser_b200 {what} failed ({rc}): {lib().df_last_error().decode()}")


def null_comm() -> DfComm:
    """Communicator of a single-rank run (no peers, no arena)."""
    c = DfComm()
    c.world, c.rank, c.bank_stride = 1, 0, 0
    return c
