"""ctypes binding of libthinkdiff_b200.so (C ABI declared in include/thinkdiff_b200.h).

There is no fallback: if the library has not been built (``make`` / ``__graft_entry__.build()``) importing the
product raises, and on a device that is not sm_100 every call raises ``RuntimeError`` with the library's message.
"""
from __future__ import annotations

import ctypes as C
import os

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.environ.get("THINKDIFF_B200_LIB", os.path.join(_HERE, "libthinkdiff_b200.so"))  # override: A/B builds

F32, BF16 = 0, 1
BWD_NORM_W2, BWD_GELU_W1, BWD_ALL, BWD_SMALL2_ONLY, BWD_W2_ONLY, BWD_GELU_ONLY, BWD_W1_ONLY = 1, 2, 3, 4, 8, 16, 32
FWD_LINEAR1, FWD_REST, FWD_ALL, FWD_DEFER_LOSS = 1, 2, 3, 4
STEP_CTL_SCALE_OFFSET = 20

_vp, _i32, _i64, _f32 = C.c_void_p, C.c_int32, C.c_int64, C.c_float

# name -> (restype, argtypes); mirrors include/thinkdiff_b200.h declaration by declaration
SIGNATURES = {
    "td_last_error": (C.c_char_p, []),
    "td_version": (_i32, []),
    "td_device_check": (_i32, []),
    "td_profile_enable": (_i32, [_i32]),
    "td_profile_report": (_i32, [C.c_char_p, _i32]),
    "td_profile_timeline": (_i32, [C.c_char_p, _i32]),
    "td_cu_seqlens": (_i32, [_vp, _i32, _vp, _vp]),
    "td_pack_varlen": (_i32, [_vp, _vp, _vp, _i32, _i64, _i64, _vp, _vp]),
    "td_pack_varlen_indexed": (_i32, [_vp, _vp, _vp, _i32, _i64, _i64, _vp, _vp, _vp]),
    "td_pack_varlen2": (_i32, [_vp, _vp, _vp, _vp, _i32, _i64, _i64, _vp, _vp]),
    "td_pack_padded": (_i32, [_vp, _vp, _vp, _i32, _i32, _i64, _vp, _vp, _vp]),
    "td_cast_f32_to_bf16": (_i32, [_vp, _vp, _i64, _vp]),
    "td_aligner_fwd_workspace_bytes": (_i64, [_i64, _i32, _i32]),
    "td_aligner_fwd": (_i32, [_vp, _i64, _i32, _i32, _vp, _vp, _vp, _vp, _vp, _f32, _vp, _vp, _vp, _vp, _vp, _i32, _vp, _i64, _vp]),
    "td_aligner_bwd_workspace_bytes": (_i64, [_i64, _i32, _i32]),
    "td_aligner_bwd": (_i32, [_vp, _i32, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _i64, _i32, _i32, _f32, _vp, _vp, _vp, _vp, _vp, _vp, _i64, _i32, _vp]),
    "td_aligner_mse_fwd_workspace_bytes": (_i64, [_i64, _i32, _i32]),
    "td_aligner_norm_partials_bytes": (_i64, [_i64, _i32]),
    "td_aligner_mse_fwd": (_i32, [_vp, _i64, _i32, _i32, _vp, _vp, _vp, _vp, _vp, _f32, _vp, _i32, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _i64, _i32, _vp]),
    "td_aligner_bwd_dh2": (_i32, [_vp, _vp, _vp, _vp, _vp, _vp, _i64, _i32, _i32, _f32, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _i32, _vp, _i64, _i32, _vp]),
    "td_rmsnorm_fwd": (_i32, [_vp, _vp, _f32, _i64, _i32, _vp, _i32, _vp, _vp]),
    "td_rmsnorm_bwd_workspace_bytes": (_i64, [_i64, _i32]),
    "td_rmsnorm_bwd": (_i32, [_vp, _i32, _vp, _vp, _vp, _i64, _i32, _vp, _vp, _vp, _vp, _i64, _vp]),
    "td_gemm_workspace_bytes": (_i64, []),
    "td_linear_bf16": (_i32, [_vp, _i64, _i32, _vp, _i32, _vp, _vp, _vp, _i64, _vp]),
    "td_linear_bf16_dx": (_i32, [_vp, _i64, _i32, _vp, _i32, _vp, _vp, _i64, _vp]),
    "td_lm_head_ce_workspace_bytes": (_i64, [_i64]),
    "td_lm_head_ce_fwd_bwd": (_i32, [_vp, _i64, _i32, _vp, _i32, _vp, _f32, _vp, _vp, _vp, _vp, _vp, _i64, _vp]),
    "td_t5_attention_workspace_bytes": (_i64, [_i64, _i32]),
    "td_t5_attention_fwd": (_i32, [_vp, _i64, _vp, _i64, _vp, _i64, _vp, _vp, _i32, _i32, _i32, _i32, _i32, _i64, _i32, _vp, _i32, _vp, _i64, _vp, _vp]),
    "td_t5_attention_bwd": (_i32, [_vp, _i64, _vp, _i64, _vp, _i64, _vp, _i64, _vp, _vp, _i32, _i32, _i32, _i32, _i32, _i64, _i32, _vp, _i32, _vp, _i64,
                                   _vp, _vp, _i64, _vp, _i64, _vp, _i64, _vp, _i64, _vp]),
    "td_t5_ffn_workspace_bytes": (_i64, [_i64, _i32, _i32]),
    "td_t5_ffn_fwd": (_i32, [_vp, _i64, _i32, _i32, _vp, _f32, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _i64, _vp]),
    "td_t5_ffn_bwd": (_i32, [_vp, _vp, _vp, _vp, _vp, _vp, _vp, _i64, _i32, _i32, _vp, _vp, _vp, _i64, _vp]),
    "td_gemm_bf16_f32out": (_i32, [_vp, _i64, _i32, _vp, _i64, _i32, _i64, _i32, _i64, _f32, _vp, _i32, _i32, _vp, _i64, _vp]),
    "td_adamw_step": (_i32, [_i32, _vp, _vp, _vp, _vp, _vp, C.POINTER(_i64), C.POINTER(_f32), _f32, _f32, _f32, _f32, _i64, _f32, _vp, _vp]),
    "td_step_ctl_bytes": (_i64, []),
    "td_step_ctl_init": (_i32, [_vp, _f32, _i64, _vp]),
    "td_step_ctl_update": (_i32, [_vp, _vp, _i32, _f32, _f32, _i32, _f32, _f32, _f32, _vp]),
    "td_grad_stats": (_i32, [_vp, _i64, _vp, _vp]),
    "td_peer_alloc": (_i32, [_i64, C.POINTER(_vp), C.c_char_p]),
    "td_peer_free": (_i32, [_vp]),
    "td_peer_open": (_i32, [C.c_char_p, C.POINTER(_vp)]),
    "td_peer_close": (_i32, [_vp]),
    "td_peer_signal": (_i32, [_vp, _i32, _i32, _vp]),
    "td_peer_wait": (_i32, [_vp, _i32, _i32, _f32, _vp]),
    "td_peer_post": (_i32, [_vp, _vp, _i32, _i64, _vp]),
    "td_sum_slots": (_i32, [_vp, _i64, _i32, _vp, _i64, _vp]),
    "td_adamw_slots_step": (_i32, [_vp, _vp, _i64, _i32, _vp, _vp, _vp, _i32, _i64, _f32, _f32, _f32, _f32, _f32, _i64, _f32, _vp, _vp]),
    "td_aligner_bwd_dh2_scatter": (_i32, [_vp, _vp, _vp, _vp, _vp, _vp, _i64, _i32, _i32, _f32, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _i32, _i32, _vp, _vp, _i64, _i32, _vp]),
    "td_gemm_schedule": (_i32, [_i64, _i32, _i64, _i32, _i32, _vp, _i32]),
    "td_scatter_tile_owner": (_i32, [_i32, _i32, _i32, _i32, _i32, _vp, _vp]),
    "td_gemm_tn_scatter": (_i32, [_vp, _i64, _vp, _i64, _i64, _i32, _i64, _f32, _vp, _i32, _i32, _vp, _i64, _vp]),
    "td_loss_workspace_bytes": (_i64, [_i64]),
    "td_masked_mse_fwd_bwd": (_i32, [_vp, _i32, _vp, _i32, _vp, _i64, _i32, _f32, _vp, _vp, _vp, _i64, _vp]),
    "td_masked_ce_fwd_bwd": (_i32, [_vp, _i32, _vp, _i64, _i32, _f32, _vp, _vp, _vp, _i64, _vp]),
}


class PeerFold(C.Structure):
    """``td_peer_fold`` of include/thinkdiff_b200.h: the exchange protocol's tiny launches folded into a backward call."""

    _fields_ = [("signal_flags", C.c_void_p), ("signal_slot", C.c_int32), ("small_dst", C.c_void_p), ("small_base", C.c_void_p),
                ("small_numel", C.c_int64)]


class LibraryMissing(ImportError):
    pass


_lib = None
launch_count = 0  # number of C-ABI calls that enqueue device work (bench.py reports kernel launches from here)


def lib():
    global _lib
    if _lib is None:
        if not os.path.isfile(LIB_PATH):
            raise LibraryMissing(
                f"{LIB_PATH} is not built. Run `make` (or `python -c 'import __graft_entry__ as g; g.build()'`). "
                "thinkdiff_mlre_b200 has no CPU or PyTorch fallback."
            )
        h = C.CDLL(LIB_PATH)
        for name, (res, args) in SIGNATURES.items():
            fn = getattr(h, name)  # AttributeError here = header and library out of sync
            fn.restype, fn.argtypes = res, args
        _lib = h
    return _lib


def last_error() -> str:
    return lib().td_last_error().decode("utf-8", "replace")


def check(rc: int, what: str = "") -> None:
    if rc != 0:
        raise RuntimeError(f"libthinkdiff_b200 {what} failed (rc={rc}): {last_error()}")


def ptr(t):
    """Device pointer of a torch tensor (None -> NULL)."""
    return None if t is None else C.c_void_p(t.data_ptr())


_raw_stream = None


def stream_ptr():
    """cudaStream_t of torch's current stream on the current device (fast path: one C call, no Stream object)."""
    global _raw_stream
    import torch

    if _raw_stream is None:
        _raw_stream = getattr(torch._C, "_cuda_getCurrentRawStream", False)
    if _raw_stream:
        return C.c_void_p(_raw_stream(torch.cuda.current_device()))
    return C.c_void_p(torch.cuda.current_stream().cuda_stream)


def dtype_code(t) -> int:
    import torch

    if t.dtype == torch.float32:
        return F32
    if t.dtype == torch.bfloat16:
        return BF16
    raise TypeError(f"unsupported dtype {t.dtype}: the aligner path handles float32 and bfloat16")


def profile_enable(on: bool) -> None:
    check(lib().td_profile_enable(int(on)), "td_profile_enable")


def profile_timeline() -> list:
    """[(tag, stream, start_ms, end_ms)] for every launch recorded since profile_enable(True), relative to the first one."""
    buf = C.create_string_buffer(1 << 20)
    check(lib().td_profile_timeline(buf, len(buf)), "td_profile_timeline")
    out = []
    for line in buf.value.decode().splitlines():
        tag, stream, t0, t1 = line.split(",")
        out.append((tag, stream, float(t0), float(t1)))
    return out


def profile_report() -> dict:
    """{tag: {"launches": n, "ms": total device ms, "work": total algorithmic FLOPs or bytes}} since profile_enable(True)."""
    buf = C.create_string_buffer(1 << 16)
    check(lib().td_profile_report(buf, len(buf)), "td_profile_report")
    out = {}
    for line in buf.value.decode().splitlines():
        tag, n, ms, work = line.split(",")
        out[tag] = {"launches": int(n), "ms": float(ms), "work": float(work)}
    return out
