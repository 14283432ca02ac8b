"""ctypes binding of libb2h.so (C-ABI declared in include/b2h.h).

There is no CPU or PyTorch fallback: if the library is missing, or the device is not sm_100, every
entry point raises.  torch is used only for device memory and streams."""
from __future__ import annotations

import ctypes
import os
from ctypes import c_char_p, c_double, c_float, c_int, c_int64, c_void_p

import torch

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "libb2h.so")

# enums of include/b2h.h
FP32, BF16, FP32_FFMA = 0, 1, 2
LOSS_L1, LOSS_CONFL1 = 0, 1
PAD_REPEAT_FIRST, PAD_ZEROS = 0, 1
DT_F32, DT_BF16 = 0, 1
PRECISIONS = {"fp32": FP32, "bf16": BF16, "fp32-ffma": FP32_FFMA}
LOSSES = {"L1": LOSS_L1, "confL1": LOSS_CONFL1}
PAD_MODES = {"repeat_first": PAD_REPEAT_FIRST, "zeros": PAD_ZEROS}


def dtype_code(dtype):
    """The C-ABI `x_dtype` of a float32 / bfloat16 keypoint input."""
    return DT_BF16 if dtype == torch.bfloat16 else DT_F32

_SIGNATURES = {
    "b2h_last_error": (c_char_p, []),
    "b2h_version": (c_int, []),
    "b2h_device_ok": (c_int, []),
    "b2h_param_count": (c_int64, [c_int, c_int, c_int]),
    "b2h_param_offset": (c_int64, [c_int, c_int, c_int, c_int, c_int]),
    "b2h_packed_bytes": (c_int64, [c_int, c_int, c_int]),
    "b2h_gp_layout_check": (c_int64, [c_int, c_int, c_int]),
    "b2h_train_subwindows": (c_int, [c_int, c_int, c_int, c_int, c_int, c_int, c_void_p]),
    "b2h_workspace_bytes": (c_int64, [c_int, c_int, c_int, c_int, c_int, c_int]),
    "b2h_supported": (c_int, [c_int, c_int, c_int, c_int, c_int]),
    "b2h_forward_supported": (c_int, [c_int, c_int, c_int, c_int, c_int]),
    "b2h_kernel_choice": (c_int, [c_int, c_int, c_int, c_int, c_int, c_int]),
    "b2h_pack_weights": (c_int, [c_void_p, c_void_p, c_int, c_int, c_int, c_void_p]),
    "b2h_preprocess": (c_int, [c_void_p, c_void_p, c_void_p, c_int64, c_void_p, c_void_p, c_int, c_int, c_int, c_float, c_int,
                               c_int, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p,
                               c_void_p]),
    "b2h_preprocess_status": (c_int, []),
    "b2h_verify_fastdiv": (c_int, [c_float, c_void_p, c_void_p]),
    "b2h_preprocess_h5": (c_int, [c_void_p, c_int64, c_void_p, c_void_p, c_int, c_int, c_int, c_float, c_int, c_int, c_void_p,
                                  c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p]),
    "b2h_conv_forward": (c_int, [c_void_p, c_int, c_void_p, c_void_p, c_void_p, c_void_p, c_int, c_int, c_int, c_int,
                                 c_int, c_int, c_int, c_float, c_void_p]),
    "b2h_conv_forward_windows": (c_int, [c_void_p, c_int, c_int64, c_void_p, c_void_p, c_int, c_void_p, c_void_p, c_void_p, c_void_p,
                                         c_int, c_int, c_int, c_int, c_int, c_int, c_int, c_float, c_void_p]),
    "b2h_conv_forward_utterances": (c_int, [c_void_p, c_int, c_int64, c_void_p, c_int, c_void_p, c_void_p, c_void_p, c_int,
                                            c_int, c_int, c_int, c_float, c_void_p, c_int64, c_void_p]),
    "b2h_utterances_workspace_bytes": (c_int64, [c_int64, c_int, c_int, c_int, c_int, c_int]),
    "b2h_utterances_plan": (c_int, [c_int64, c_int, c_int, c_int, c_int, c_int, c_void_p]),
    "b2h_utterance_subwindows": (c_int, [c_int, c_int, c_int, c_void_p]),
    "b2h_train_forward_backward": (c_int, [c_void_p, c_int, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p,
                                           c_void_p, c_void_p, c_int, c_int, c_int, c_int, c_int, c_int, c_int, c_void_p,
                                           c_void_p, c_int64, c_void_p]),
    "b2h_train_forward_backward_windows": (c_int, [c_void_p, c_int, c_void_p, c_void_p, c_int64, c_void_p, c_void_p, c_int,
                                                   c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_int, c_int,
                                                   c_int, c_int, c_int, c_int, c_int, c_void_p, c_void_p, c_int64, c_void_p]),
    "b2h_train_forward_backward_utterances": (c_int, [c_void_p, c_int, c_void_p, c_void_p, c_int64, c_void_p, c_void_p, c_int,
                                                      c_int, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_int, c_int,
                                                      c_int, c_int, c_int, c_void_p, c_void_p, c_int64, c_void_p]),
    "b2h_train_step_utterances": (c_int, [c_void_p, c_int, c_void_p, c_void_p, c_int64, c_void_p, c_void_p, c_int, c_int,
                                          c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_int, c_int, c_int, c_int, c_int,
                                          c_double, c_double, c_double, c_double, c_int64, c_void_p, c_void_p, c_void_p,
                                          c_int64, c_void_p]),
    "b2h_train_utterances_workspace_bytes": (c_int64, [c_int, c_int, c_int, c_int, c_int, c_int]),
    "b2h_train_utterances_plan": (c_int, [c_int, c_int, c_int, c_int, c_int, c_int, c_void_p]),
    "b2h_validate_utterances": (c_int, [c_void_p, c_int, c_void_p, c_void_p, c_int64, c_void_p, c_void_p, c_int, c_int, c_void_p,
                                        c_void_p, c_void_p, c_void_p, c_int, c_int, c_int, c_int, c_int, c_void_p, c_int64,
                                        c_void_p]),
    "b2h_validate_utterances_workspace_bytes": (c_int64, [c_int, c_int, c_int, c_int, c_int, c_int]),
    "b2h_validate_utterances_plan": (c_int, [c_int, c_int, c_int, c_int, c_int, c_int, c_void_p]),
    "b2h_conv_backward": (c_int, [c_void_p, c_int, c_void_p, c_void_p, c_void_p, c_void_p, c_int, c_int, c_int, c_int,
                                  c_int, c_int, c_void_p, c_int64, c_void_p]),
    "b2h_mask_output": (c_int, [c_void_p, c_void_p, c_int, c_int, c_int, c_void_p]),
    "b2h_pose_l1": (c_int, [c_void_p, c_void_p, c_void_p, c_void_p, c_int, c_int, c_int, c_int, c_void_p, c_void_p,
                            c_void_p, c_void_p]),
    "b2h_adam_step": (c_int, [c_void_p, c_void_p, c_void_p, c_void_p, c_int64, c_double, c_double, c_double, c_double,
                              c_int64, c_void_p, c_void_p, c_float, c_void_p, c_int, c_int, c_int, c_void_p]),
    "b2h_train_step": (c_int, [c_void_p, c_int, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p,
                               c_void_p, c_int, c_int, c_int, c_int, c_int, c_int, c_int, c_double, c_double, c_double,
                               c_double, c_int64, c_void_p, c_void_p, c_void_p, c_int64, c_void_p]),
    "b2h_train_step_windows": (c_int, [c_void_p, c_int, c_void_p, c_void_p, c_int64, c_void_p, c_void_p, c_int, c_void_p,
                                       c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_int, c_int, c_int, c_int, c_int,
                                       c_int, c_int, c_double, c_double, c_double, c_double, c_int64, c_void_p, c_void_p,
                                       c_void_p, c_int64, c_void_p]),
    "b2h_train_step_dp": (c_int, [c_void_p, c_int, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p,
                                  c_void_p, c_int, c_int, c_int, c_int, c_int, c_int, c_int, c_double, c_double, c_double,
                                  c_double, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_int, c_int, c_float,
                                  c_void_p, c_int64, c_void_p]),
    "b2h_dp_exchange_floats": (c_int64, [c_int, c_int, c_int, c_int]),
    "b2h_dp_exchange_fill": (c_int64, [c_int, c_int, c_int, c_int, c_int]),
    "b2h_dp_status": (c_int, []),
    "b2h_pos_emb_concat": (c_int, [c_void_p, c_void_p, c_int, c_int, c_int, c_int, c_void_p]),
    "b2h_format_prediction": (c_int, [c_void_p, c_void_p, c_int64, c_int, c_void_p]),
    "b2h_tc_probe": (c_int, [c_void_p, c_void_p, c_void_p, c_int, c_int, c_int, c_int, c_void_p]),
    "b2h_tc_status": (c_int, []),
    "b2h_debug_timing": (None, [c_void_p]),
    "b2h_launch_count": (c_int64, []),
}

_lib = None


class B2HError(RuntimeError):
    pass


def load():
    """Loads libb2h.so (once).  Raises if it has not been built: python -c 'import __graft_entry__ as g; g.build()'."""
    global _lib
    if _lib is None:
        if not os.path.isfile(LIB_PATH):
            raise B2HError(f"{LIB_PATH} not found: the CUDA library is not built (run __graft_entry__.build()). "
                           "hand_pose_sl_b200 has no CPU / PyTorch fallback.")
        lib = ctypes.CDLL(LIB_PATH)
        for name, (res, args) in _SIGNATURES.items():
            fn = getattr(lib, name)
            fn.restype = res
            fn.argtypes = args
        _lib = lib
    return _lib


def exported_symbols():
    return sorted(_SIGNATURES)


def last_error() -> str:
    return load().b2h_last_error().decode()


def check(rc: int):
    if rc != 0:
        raise B2HError(f"libb2h error {rc}: {last_error()}")


def require_device(t: torch.Tensor, what: str):
    if not t.is_cuda:
        raise B2HError(f"{what} must be a CUDA tensor: hand_pose_sl_b200 has no CPU fallback (got device {t.device})")


_dev_checked = set()


def require_sm100(device):
    idx = device.index if device.index is not None else torch.cuda.current_device()
    if idx not in _dev_checked:
        major, _ = torch.cuda.get_device_capability(idx)
        if major != 10:
            raise B2HError(f"hand_pose_sl_b200 targets sm_100a (B200); device {idx} is sm_{major}x")
        _dev_checked.add(idx)


def ptr(t):
    return None if t is None else c_void_p(t.data_ptr())


def ptrs(args):
    """C arguments: every tensor of `args` replaced by its pointer."""
    return tuple(ptr(a) if isinstance(a, torch.Tensor) else a for a in args)


def lengths_i32(lengths, device, B):
    """`lengths` is `batch["n_frames"]`, a CPU int64 tensor in the reference (traintest.py:91)."""
    t = torch.as_tensor(lengths)
    if t.numel() != B:
        raise RuntimeError(f"lengths has {t.numel()} entries for a batch of {B}")
    return t.to(device=device, dtype=torch.int32, non_blocking=True).contiguous()


def stream_ptr(device=None):
    return c_void_p(torch.cuda.current_stream(device).cuda_stream)


def launch_count() -> int:
    return int(load().b2h_launch_count())


def query(name, *args) -> int:
    """The count or byte size C-ABI query `name` returns for `args`; a negative result is an error code: B2HError."""
    n = getattr(load(), name)(*args)
    if n < 0:
        raise B2HError(last_error())
    return int(n)


def param_count(n_in, C, pos_emb) -> int:
    return query("b2h_param_count", n_in, C, int(pos_emb))


def param_offset(n_in, C, pos_emb, layer, is_bias) -> int:
    return query("b2h_param_offset", n_in, C, int(pos_emb), layer, int(is_bias))


def packed_bytes(n_in, C, pos_emb) -> int:
    return query("b2h_packed_bytes", n_in, C, int(pos_emb))


def workspace_bytes(B, T, n_in, C, pos_emb, precision) -> int:
    return query("b2h_workspace_bytes", B, T, n_in, C, int(pos_emb), precision)
