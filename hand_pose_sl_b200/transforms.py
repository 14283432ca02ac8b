"""Drop-ins for the reference's per-item transforms (body2hand/src/steps/utils.py:180-210, 261-277) and
the data-item construction feeding them (body2hand/src/dataloaders/text_pose_dataset.py:14-68,
511-544, 587-649), executed as ONE CUDA kernel over whole clips / batches of windows (K0).

`PreprocessRightHand` is the fused equivalent of
    Compose([WristDifference(), ChestDifference(), NormalizeFixedFactor(1280), BuildRightHandItem()])
applied after load_keypoints + crop + pad + clip + to_tensor; it returns the reference's item dict
keys stacked over windows.  The individual transform classes keep the reference's names and
`item -> item` call signature for (T,·) CUDA tensors; they are thin views over the same kernel."""
from __future__ import annotations

import numpy as np
import torch

from . import _lib

BODY_HEAD_KEYPOINTS = [0, 1, 2, 3, 4, 5, 6, 7, 15, 16, 17, 18]   # text_pose_dataset.py:14


def _dev_f32(a, device):
    t = torch.as_tensor(a)
    return t.to(device=device, dtype=torch.float32, non_blocking=True).contiguous()


class PreprocessRightHand:
    """K0.  factor=1280 and dif_encoding=True are run.py's training defaults (run.py:41,90);
    infer_utterance.py defaults dif_encoding to False (infer_utterance.py:34)."""

    def __init__(self, factor=1280, dif_encoding=True, normalize=True, pad_mode="repeat_first", with_left_hand=True,
                 emit_bf16=False):
        self.factor = float(factor)
        self.dif_encoding = bool(dif_encoding)
        self.normalize = bool(normalize)
        if pad_mode not in ("repeat_first", "zeros"):
            raise ValueError("pad_mode must be 'repeat_first' (JSON datasets) or 'zeros' (H5 dataset)")
        self.pad_mode = _lib.PAD_REPEAT_FIRST if pad_mode == "repeat_first" else _lib.PAD_ZEROS
        self.with_left_hand = with_left_hand
        self.emit_bf16 = emit_bf16

    def _outputs(self, W, T, n_body, device):
        f32 = dict(dtype=torch.float32, device=device)
        out = {
            "input_kp": torch.empty((W, T, n_body, 2), **f32), "input_conf": torch.empty((W, T, n_body), **f32),
            "target_kp": torch.empty((W, T, 21, 2), **f32), "target_conf": torch.empty((W, T, 21), **f32),
            "n_frames": torch.empty((W,), dtype=torch.int64, device=device),
        }
        if self.with_left_hand:
            out["left_hand_kp"] = torch.empty((W, T, 21, 2), **f32)
            out["left_hand_conf"] = torch.empty((W, T, 21), **f32)
        return out

    @staticmethod
    def _alias(out):
        # BuildRightHandItem keeps the originals next to the aliases (utils.py:265-269)
        out["body_kp"], out["body_conf"] = out["input_kp"], out["input_conf"]
        out["right_hand_kp"], out["right_hand_conf"] = out["target_kp"], out["target_conf"]
        return out

    def __call__(self, pose25, hand_left, hand_right, win_start, T, out=None, win_end=None):
        """pose25 (F,25,3), hand_left/right (F,21,3) fp32 CUDA tensors (OpenPose [x,y,c]); win_start (W,)
        int64; `win_end` (W,) optional exclusive end of the utterance each window is cropped from; `out` = the dict returned by an earlier call with the same (W, T) to reuse its buffers; returns the stacked item dict: input_kp (W,T,12,2), input_conf (W,T,12), target_kp
        (W,T,21,2), target_conf (W,T,21), left_hand_*, n_frames (W,) int64 (device)."""
        _lib.require_device(pose25, "pose25")
        _lib.require_sm100(pose25.device)
        dev = pose25.device
        F = pose25.shape[0]
        if tuple(pose25.shape[1:]) != (25, 3) or tuple(hand_left.shape) != (F, 21, 3) or tuple(hand_right.shape) != (F, 21, 3):
            raise RuntimeError("expected pose25 (F,25,3), hand_left (F,21,3), hand_right (F,21,3)")
        pose25, hand_left, hand_right = (_dev_f32(a, dev) for a in (pose25, hand_left, hand_right))
        ws = torch.as_tensor(win_start).to(device=dev, dtype=torch.int64).contiguous()
        we = None if win_end is None else torch.as_tensor(win_end).to(device=dev, dtype=torch.int64).contiguous()
        W = ws.numel()
        if we is not None and we.numel() != W:
            raise RuntimeError("win_end must have one entry per window")
        if out is None:
            out = self._outputs(W, T, 12, dev)
            bf = torch.empty((W, T, 24), dtype=torch.bfloat16, device=dev) if self.emit_bf16 else None
        else:      # caller-owned output dict of a previous call with the same (W, T): steady-state loops, CUDA graphs
            bf = out["input_kp_bf16"].view(W, T, 24) if self.emit_bf16 else None
        lib = _lib.load()
        _lib.check(lib.b2h_preprocess(_lib.ptr(pose25), _lib.ptr(hand_left), _lib.ptr(hand_right), F, _lib.ptr(ws), _lib.ptr(we), W, T,
                                      self.pad_mode, self.factor, int(self.dif_encoding), int(self.normalize),
                                      _lib.ptr(out["input_kp"]), _lib.ptr(out["input_conf"]), _lib.ptr(out["target_kp"]),
                                      _lib.ptr(out["target_conf"]), _lib.ptr(out.get("left_hand_kp")),
                                      _lib.ptr(out.get("left_hand_conf")), _lib.ptr(out["n_frames"]), _lib.ptr(bf),
                                      _lib.stream_ptr(dev)))
        if bf is not None:
            out["input_kp_bf16"] = bf.view(W, T, 12, 2)
        return self._alias(out)

    def frame_stream(self, pose25, hand_left, hand_right, dtype=torch.bfloat16, out=None):
        """Streaming inference (BASELINE config 5): the network input of EVERY UNIQUE FRAME of a clip, once --
        (F, 12, 2) in `dtype` (bf16 feeds the tensor-core net directly; fp32 is the reference item's `input_kp`).
        Only what the net reads is written (804 B read + 48 B written per frame in bf16), no targets / confidences.
        Sliding windows over the clip are then VIEWS of this stream: `ConvModel.predict_windows(stream, starts, T)`
        applies the crop + pad rule on the fly, so 4x-overlapping windows are neither written nor re-read."""
        _lib.require_device(pose25, "pose25")
        _lib.require_sm100(pose25.device)
        dev = pose25.device
        F = pose25.shape[0]
        if tuple(pose25.shape[1:]) != (25, 3) or tuple(hand_left.shape) != (F, 21, 3) or tuple(hand_right.shape) != (F, 21, 3):
            raise RuntimeError("expected pose25 (F,25,3), hand_left (F,21,3), hand_right (F,21,3)")
        if dtype not in (torch.bfloat16, torch.float32):
            raise ValueError("dtype must be torch.bfloat16 or torch.float32")
        pose25, hand_left, hand_right = (_dev_f32(a, dev) for a in (pose25, hand_left, hand_right))
        if out is None:
            out = torch.empty((F, 12, 2), dtype=dtype, device=dev)
        if getattr(self, "_zero_start", None) is None or self._zero_start.device != dev:
            self._zero_start = torch.zeros(1, dtype=torch.int64, device=dev)
        f32 = _lib.ptr(out) if dtype == torch.float32 else None
        b16 = _lib.ptr(out) if dtype == torch.bfloat16 else None
        _lib.check(_lib.load().b2h_preprocess(_lib.ptr(pose25), _lib.ptr(hand_left), _lib.ptr(hand_right), F, _lib.ptr(self._zero_start),
                                              None, 1, F, self.pad_mode, self.factor, int(self.dif_encoding), int(self.normalize),
                                              f32, None, None, None, None, None, None, b16, _lib.stream_ptr(dev)))
        return out

    def training_stream(self, pose25, hand_left, hand_right, dtype=torch.bfloat16):
        """Training from device-resident frames: the per-frame preprocessed training data of a whole clip, from ONE K0
        launch (one window covering the clip) -- {input_kp (F, 12, 2) in `dtype`, target_kp (F, 21, 2) fp32,
        target_conf (F, 21) fp32}, 300 B per frame in bf16.  Per-frame preprocessing does not depend on the window, so
        the crops of `steps.fused_train_step_windows` / `runner.WindowTrainStepRunner` over these streams are exactly
        the windows `__call__` materialises.  (H5 rows: `from_h5_rows(rows, [0], F)` with the window axis dropped.)"""
        _lib.require_device(pose25, "pose25")
        _lib.require_sm100(pose25.device)
        dev = pose25.device
        F = pose25.shape[0]
        if tuple(pose25.shape[1:]) != (25, 3) or tuple(hand_left.shape) != (F, 21, 3) or tuple(hand_right.shape) != (F, 21, 3):
            raise RuntimeError("expected pose25 (F,25,3), hand_left (F,21,3), hand_right (F,21,3)")
        if dtype not in (torch.bfloat16, torch.float32):
            raise ValueError("dtype must be torch.bfloat16 or torch.float32")
        pose25, hand_left, hand_right = (_dev_f32(a, dev) for a in (pose25, hand_left, hand_right))
        f32 = dict(dtype=torch.float32, device=dev)
        out = {"input_kp": torch.empty((F, 12, 2), dtype=dtype, device=dev), "target_kp": torch.empty((F, 21, 2), **f32),
               "target_conf": torch.empty((F, 21), **f32)}
        x32 = _lib.ptr(out["input_kp"]) if dtype == torch.float32 else None
        x16 = _lib.ptr(out["input_kp"]) if dtype == torch.bfloat16 else None
        start = torch.zeros(1, dtype=torch.int64, device=dev)
        _lib.check(_lib.load().b2h_preprocess(_lib.ptr(pose25), _lib.ptr(hand_left), _lib.ptr(hand_right), F, _lib.ptr(start), None,
                                              1, F, self.pad_mode, self.factor, int(self.dif_encoding), int(self.normalize), x32,
                                              None, _lib.ptr(out["target_kp"]), _lib.ptr(out["target_conf"]), None, None, None,
                                              x16, _lib.stream_ptr(dev)))
        return out

    def from_h5_rows(self, rows150, win_start, T, win_end=None):
        """Packed rows of TextPoseH5Dataset.array2item (text_pose_dataset.py:587-612): (F,150) =
        [x0..x49|y0..y49|c0..c49]; body = 8 keypoints."""
        _lib.require_device(rows150, "rows150")
        _lib.require_sm100(rows150.device)
        dev = rows150.device
        if rows150.dim() != 2 or rows150.shape[1] != 150:
            raise RuntimeError("expected rows (F,150)")
        rows150 = _dev_f32(rows150, dev)
        F = rows150.shape[0]
        ws = torch.as_tensor(win_start).to(device=dev, dtype=torch.int64).contiguous()
        we = None if win_end is None else torch.as_tensor(win_end).to(device=dev, dtype=torch.int64).contiguous()
        W = ws.numel()
        out = self._outputs(W, T, 8, dev)
        lib = _lib.load()
        _lib.check(lib.b2h_preprocess_h5(_lib.ptr(rows150), F, _lib.ptr(ws), _lib.ptr(we), W, T, self.pad_mode, self.factor,
                                         int(self.dif_encoding), int(self.normalize), _lib.ptr(out["input_kp"]),
                                         _lib.ptr(out["input_conf"]), _lib.ptr(out["target_kp"]),
                                         _lib.ptr(out["target_conf"]), _lib.ptr(out.get("left_hand_kp")),
                                         _lib.ptr(out.get("left_hand_conf")), _lib.ptr(out["n_frames"]),
                                         _lib.stream_ptr(dev)))
        return self._alias(out)


# ---- host-side index math of the windowing (bit-exact integer work, no arithmetic on keypoints) ----
def select_window(n_total, n, selection_type, rng=None):
    """select_jsons (text_pose_dataset.py:52-68) as (start, stop).  `rng` is a `random.Random`-like
    object; the draw is `rng.randint(0, n_total - n)`, inclusive on both ends like the reference."""
    if n_total <= n:
        return 0, n_total
    if selection_type == "first":
        return 0, n
    if selection_type == "randomcrop":
        import random as _random
        start = (rng or _random).randint(0, n_total - n)
        return start, start + n
    raise ValueError("selection_type must be 'first' or 'randomcrop' (the reference returns None otherwise)")


def sliding_window_starts(n_frames, T=64, stride=64):
    """Streaming inference (BASELINE config 5): window i starts at i*stride; the tail window is padded by
    the dataset's pad rule."""
    return np.arange(0, max(int(n_frames), 1), int(stride), dtype=np.int64)
