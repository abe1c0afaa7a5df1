"""ctypes binding of the C-ABI library ``libnsd_b200.so`` (include/nsd_b200.h).

There is no fallback: if the shared library has not been built, or a call
fails, an exception is raised.  The compute path of this package is the CUDA
library and nothing else.
"""
from __future__ import annotations

import ctypes as C
import os
from typing import Optional

import torch

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "libnsd_b200.so")

F32, BF16 = 0, 1

vp, i32, i64, f32, u64, sz = C.c_void_p, C.c_int, C.c_int64, C.c_float, C.c_uint64, C.c_size_t

# name -> (restype, argtypes); mirrors include/nsd_b200.h one to one
SIGNATURES = {
    "nsd_version": (i32, []),
    "nsd_last_error": (C.c_char_p, []),
    "nsd_launch_count": (C.c_ulonglong, []),
    "nsd_device_info": (i32, [C.POINTER(i32)] * 3),
    "nsd_frontend_fwd": (i32, [vp, vp, vp, vp, vp, i32, i32, i32, i32, i32, i32, i32, vp, vp, vp, i32, vp, f32, f32, u64, vp, vp]),
    "nsd_frame_counts": (i32, [vp, i32, i32, i32, i32, vp, vp, vp]),
    "nsd_input_noise": (i32, [vp, vp, i32, i32, i32, f32, f32, u64, vp]),
    "nsd_frontend_bwd": (i32, [vp, i32, vp, vp, vp, i32, i32, i32, i32, i32, i32, vp, vp, vp, sz, vp]),
    "nsd_frontend_bwd_workspace": (sz, [i32, i32]),
    "nsd_frontend_bwd_input": (i32, [vp, i32, vp, vp, vp, vp, i32, i32, i32, i32, i32, i32, i32, vp, vp, vp]),
    "nsd_gemm_f32": (i32, [i32, i32, i32, i32, i32, vp, i32, vp, i32, vp, i32, vp, f32, vp]),
    "nsd_gemm_bf16": (i32, [i32, i32, i32, i32, i32, vp, i32, vp, i32, vp, i32, i32, vp, f32, vp]),
    "nsd_gemm_bf16_x2": (i32, [i32, i32, i32, i32, i32, vp, vp, i32, vp, vp, i32, vp, vp, i32, i32, vp]),
    "nsd_colsum": (i32, [vp, i32, i32, i32, i32, vp, vp, sz, vp]),
    "nsd_colsum_workspace": (sz, [i32]),
    "nsd_cast": (i32, [vp, i32, vp, i32, sz, vp]),
    "nsd_cast_transpose": (i32, [vp, i32, i32, i32, i32, vp, i32, vp, i32, vp]),
    "nsd_swap01_f32": (i32, [vp, vp, i32, i32, i32, vp]),
    "nsd_gru_fwd_f32": (i32, [vp, i32, vp, vp, i32, i32, i32, i32, vp, i32, vp, vp, vp, vp, vp, vp]),
    "nsd_gru_bwd_f32": (i32, [vp, i32, vp, i32, vp, vp, vp, vp, vp, i32, i32, i32, i32, vp, i32, vp, vp, vp, sz, vp]),
    "nsd_gru_bwd_workspace": (sz, [i32, i32]),
    "nsd_gru_fwd_bf16": (i32, [vp, i32, vp, vp, i32, i32, i32, i32, i32, vp, vp, i32, vp, vp, vp, vp, vp, f32, u64, vp, vp, vp, sz, vp]),
    "nsd_gru_bwd_bf16": (i32, [vp, i32, vp, i32, vp, vp, vp, vp, vp, i32, i32, i32, i32, i32, vp, vp, i32, f32, u64, vp, vp, vp, vp, sz, vp]),
    "nsd_gru_tc_workspace": (sz, [i32, i32, i32]),
    "nsd_dropout": (i32, [vp, vp, i32, sz, f32, u64, vp]),
    "nsd_ctc_loss": (i32, [vp, i64, i64, i64, i32, vp, i32, vp, vp, i32, i32, i32, i32, i32, i32, vp, vp, vp, vp, sz, vp]),
    "nsd_ctc_workspace": (sz, [i32, i32, i32, i32]),
    "nsd_log_softmax_f32": (i32, [vp, vp, i64, i32, vp]),
    "nsd_adam_step": (i32, [i32, vp, vp, vp, vp, vp, vp, f32, f32, f32, f32, f32, i32, f32, vp]),
    "nsd_set_gemm_sm_reserve": (i32, [i32]),
    "nsd_layernorm_fwd": (i32, [vp, vp, vp, f32, i32, f32, u64, vp, vp, vp, vp, i32, i32, vp]),
    "nsd_layernorm_bwd": (i32, [vp, i32, vp, vp, vp, vp, vp, i32, f32, u64, vp, vp, vp, vp, i32, i32, vp, sz, vp]),
    "nsd_layernorm_bwd_workspace": (sz, [i32, i32]),
    "nsd_act_fwd": (i32, [vp, i32, f32, u64, vp, vp, sz, vp]),
    "nsd_act_bwd": (i32, [vp, i32, vp, i32, f32, u64, vp, sz, vp]),
    "nsd_glu_fwd": (i32, [vp, vp, i32, i32, vp]),
    "nsd_glu_bwd": (i32, [vp, vp, vp, i32, i32, vp]),
    "nsd_residual": (i32, [vp, vp, f32, f32, u64, f32, u64, i64, vp, sz, vp]),
    "nsd_dwconv_fwd": (i32, [vp, vp, vp, vp, i32, i32, i32, i32, i32, i32, vp]),
    "nsd_dwconv_bwd_w": (i32, [vp, vp, vp, vp, i32, i32, i32, i32, vp, sz, vp]),
    "nsd_dwconv_bwd_w_workspace": (sz, [i32, i32, i32]),
    "nsd_strided_dwconv_fwd": (i32, [vp, vp, vp, vp, i32, i32, i32, i32, i32, vp]),
    "nsd_strided_dwconv_bwd": (i32, [vp, vp, vp, vp, vp, i32, i32, i32, i32, i32, vp, sz, vp]),
    "nsd_strided_dwconv_bwd_workspace": (sz, [i32, i32, i32]),
    "nsd_posenc_mask": (i32, [vp, vp, vp, vp, vp, i32, i32, i32, vp]),
    "nsd_set_seed_offset_ptr": (i32, [vp]),
    "nsd_cast_colsum": (i32, [vp, i32, i32, vp, i32, vp, vp, sz, vp]),
    "nsd_cast_colsum_workspace": (sz, [i32, i32]),
    "nsd_bgemm": (i32, [vp, i32, i64, i64, i64, i64, vp, i32, i64, i64, i64, i64, vp, vp, i32, i64, i64, i64, vp, i64, i32, i32, i32, i32, i32, f32, i32, vp]),
    "nsd_softmax_mask_fwd": (i32, [vp, vp, i32, vp, i32, i32, i32, i32, f32, u64, vp]),
    "nsd_softmax_mask_bwd": (i32, [vp, vp, i32, i32, i32, i32, f32, u64, vp]),
    "nsd_index_reduce": (i32, [vp, vp, i32, sz, i32, vp, vp]),
    "nsd_axpb": (i32, [vp, f32, f32, vp, sz, vp]),
    "nsd_sum_f32": (i32, [vp, sz, f32, f32, i32, vp, vp]),
    "nsd_log_softmax_bwd": (i32, [vp, vp, vp, i64, i32, vp]),
    "nsd_sqnorm_multi": (i32, [i32, vp, vp, vp, vp, sz, vp]),
    "nsd_sqnorm_workspace": (sz, [i32, vp]),
    "nsd_adamw_step": (i32, [i32, vp, vp, vp, vp, vp, vp, f32, f32, f32, f32, f32, i32, f32, vp, f32, vp, vp]),
    "nsd_stream_push_workspace": (sz, [i32, i32, i32, i32]),
    "nsd_stream_push": (i32, [vp, vp, i32, vp, vp, vp, i32, vp, i32, vp, vp, i32, i32, i32, i32, i32, i32, i32, i32, vp, vp, vp, vp, vp, vp,
                              vp, vp, vp, vp, vp, vp, sz, vp]),
    "nsd_stream_push_slots": (i32, [vp, vp, i32, vp, vp, vp, i32, vp, i32, vp, vp, vp, vp, vp, i32, i32, i32, i32, i32, i32, i32, vp, vp, vp,
                                    vp, vp, vp, vp, vp, vp, vp, vp, vp, sz, vp]),
    "nsd_multi_copy_f32": (i32, [i32, vp, vp, vp, vp]),
    "nsd_set_adam_late_wait": (i32, [i32]),
    "nsd_transpose_bf16_multi": (i32, [i32, vp, vp, i32, i32, i32, i32, vp]),
    "nsd_greedy_decode": (i32, [vp, i64, i64, i64, vp, i32, i32, i32, i32, vp, vp, vp]),
    "nsd_edit_distance": (i32, [vp, i32, vp, vp, i32, vp, i32, vp, vp, sz, vp]),
    "nsd_edit_distance_workspace": (sz, [i32, i32]),
    "nsd_ctc_beam_state_bytes": (sz, [i32, i32, i32]),
    "nsd_ctc_beam_init": (i32, [vp, sz, i32, i32, i32, vp]),
    "nsd_ctc_beam_reset": (i32, [vp, sz, i32, i32, i32, vp, vp]),
    "nsd_ctc_beam_advance": (i32, [vp, i64, i64, i64, i32, vp, i32, i32, i32, i32, vp, f32, f32, i32, i32, vp, sz, vp, vp]),
    "nsd_ctc_beam_nbest": (i32, [vp, i32, i32, i32, i32, vp, i32, vp, vp, vp, vp]),
    "nsd_ctc_word_beam_state_bytes": (sz, [i32, i32, i32]),
    "nsd_ctc_word_beam_init": (i32, [vp, sz, i32, i32, i32, i32, vp]),
    "nsd_ctc_word_beam_reset": (i32, [vp, sz, i32, i32, i32, i32, vp, vp]),
    "nsd_ctc_word_beam_advance": (i32, [vp, i64, i64, i64, i32, vp, i32, i32, i32, i32, i32, vp, i32, vp, i32, vp, vp, i32, i32, i32, f32,
                                        f32, i32, i32, vp, sz, vp, vp]),
    "nsd_ctc_word_beam_nbest": (i32, [vp, i32, i32, i32, vp, i32, vp, i32, vp, vp, i32, i32, i32, i32, f32, f32, i32, i32, vp, i32, vp,
                                      vp, i32, vp, vp, vp, vp]),
    "nsd_ctc_word_beam_live": (i32, [vp, i32, i32, i32, vp, i32, vp, vp]),
    "nsd_ctc_align_workspace": (sz, [i32, i32, i32, i32]),
    "nsd_ctc_align": (i32, [vp, i64, i64, i64, i32, vp, i32, vp, vp, i32, i32, i32, i32, i32, vp, vp, vp, vp, vp, vp, vp, sz, vp]),
}

_lib: Optional[C.CDLL] = None
launch_count = 0          # number of library calls that enqueue kernels (bench.py reports it)


class NsdError(RuntimeError):
    pass


def lib() -> C.CDLL:
    global _lib
    if _lib is None:
        if not os.path.exists(LIB_PATH):
            raise ImportError(
                f"{LIB_PATH} is missing: build it with `make` (or `python -c 'import __graft_entry__ as g; g.build()'`)."
                " neural_speech_decoder_b200 has no CPU or PyTorch fallback.")
        l = C.CDLL(LIB_PATH)
        for name, (res, args) in SIGNATURES.items():
            fn = getattr(l, name)          # AttributeError here = header / library mismatch
            fn.restype = res
            fn.argtypes = args
        _lib = l
    return _lib


def check(status: int, what: str = "") -> None:
    if status != 0:
        msg = lib().nsd_last_error().decode(errors="replace")
        raise NsdError(f"{what or 'nsd call'} failed with status {status}: {msg}")


_prof_names = False       # False: off; None: every entry point; set: the named entry points
_prof_events = []


def profile_begin(names) -> None:
    """Bracket the named entry points (None = all) with CUDA events on the current stream (bench.py)."""
    global _prof_names, _prof_events
    _prof_names, _prof_events = names, []


def profile_end():
    """-> {entry point: (calls, total ms)}; synchronises."""
    global _prof_names
    _prof_names = False
    torch.cuda.synchronize()
    out = {}
    for name, e0, e1 in _prof_events:
        n, t = out.get(name, (0, 0.0))
        out[name] = (n + 1, t + e0.elapsed_time(e1))
    _prof_events.clear()
    return out


def call(name: str, *args) -> None:
    """Invoke a status-returning entry point and raise on failure."""
    global launch_count
    launch_count += 1
    if _prof_names is not False and (_prof_names is None or name in _prof_names):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        check(getattr(lib(), name)(*args), name)
        e1.record()
        _prof_events.append((name, e0, e1))
        return
    check(getattr(lib(), name)(*args), name)


def ptr(t: Optional[torch.Tensor]):
    return None if t is None else t.data_ptr()


def stream() -> int:
    return torch.cuda.current_stream().cuda_stream


def dtype_code(dt: torch.dtype) -> int:
    if dt == torch.float32:
        return F32
    if dt == torch.bfloat16:
        return BF16
    raise NsdError(f"unsupported dtype {dt}")


def require_cuda(t: torch.Tensor, name: str) -> None:
    if not t.is_cuda:
        raise NsdError(f"{name} must be a CUDA tensor: this package has no CPU path (got device {t.device})")
