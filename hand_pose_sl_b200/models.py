"""Drop-in for the reference's `models.ConvModel` (body2hand/src/models/HandPoseModels.py:17-84).

Same constructor `ConvModel(conv_channels, activation, pos_emb)`, same parameter names and shapes
(`conv{1..4}.{weight,bias}`, fp32, (Cout,Cin,5)), same `forward(inp: (B,T,K,2)) -> (B,T,21,2)`, same
default initialisation under the same `torch.manual_seed` (the four nn.Conv1d are built in the
reference's order).  Behind it: one fused CUDA launch per forward (libb2h.so via ctypes), the
parameters being views of ONE flat fp32 buffer so the optimiser and the gradient all-reduce are
single launches too.  Extra kwarg `precision` in {"fp32","bf16"} selects the FFMA kernel (1e-4 parity)
or the tcgen05 kernel (bf16 operands, fp32 accumulation in TMEM, 2e-2 parity)."""
from __future__ import annotations

import weakref

import numpy as np
import torch
import torch.nn as nn

from . import _lib

_OWNERS = weakref.WeakValueDictionary()   # id(model) -> model, looked up through Parameter._b2h_owner_id
ANY_LENGTH = object()                      # ConvModel._check_input's T of a frame stream read as sequences of any length


def owner_of(param):
    """The ConvModel whose flat buffer `param` is a view of (None if it is not one of ours)."""
    return _OWNERS.get(getattr(param, "_b2h_owner_id", None))


class LinearPositionalEmbedding(nn.Module):
    """HandPoseModels.py:66-84.  The reference concatenates a constant row t/max_len in front of the
    channels (and only works when T == max_len); here the row is generated inside the conv kernel."""

    def __init__(self, max_len=100):
        super().__init__()
        self.max_len = max_len
        self.pe = (torch.arange(max_len).float() / max_len)[None, None, :]

    def forward(self, inp, lengths=None):
        """(B, C, T) -> (B, C+1, T): the constant row t/max_len in front of the channels (HandPoseModels.py:78-84;
        `lengths` is accepted and ignored exactly like the reference).  One CUDA launch; like the reference's
        torch.cat it raises unless T == max_len."""
        _lib.require_device(inp, "LinearPositionalEmbedding input")
        if inp.dim() != 3:
            raise RuntimeError(f"LinearPositionalEmbedding expects (B, C, T), got {tuple(inp.shape)}")
        B, Cc, T = inp.shape
        if T != self.max_len:
            raise RuntimeError(f"Sizes of tensors must match except in dimension 1. Expected size {self.max_len} but got size {T}")
        x = inp.to(torch.float32).contiguous()
        out = torch.empty((B, Cc + 1, T), dtype=torch.float32, device=x.device)
        _lib.check(_lib.load().b2h_pos_emb_concat(_lib.ptr(x), _lib.ptr(out), B, Cc, T, self.max_len, _lib.stream_ptr(x.device)))
        return out


class _ConvForward(torch.autograd.Function):
    @staticmethod
    def forward(ctx, x, model, *params):
        y = model._forward_impl(x)
        ctx.model = model
        ctx.save_for_backward(x)
        return y

    @staticmethod
    def backward(ctx, grad_y):
        (x,) = ctx.saved_tensors
        model = ctx.model
        grads = model._backward_impl(x, grad_y)
        return (None, None) + tuple(grads)


class ConvModel(nn.Module):
    def __init__(self, conv_channels, activation, pos_emb, precision="fp32", n_keypoints=12, pos_emb_max_len=100,
                 pos_emb_any_length=False):
        """Reference signature `ConvModel(conv_channels, activation, pos_emb)` (HandPoseModels.py:18) + extensions:
        `precision`; `n_keypoints` (input keypoints: 12 in run.py, 8 for the H5 items); and for SURVEY 8f N4
        `pos_emb_max_len` (LinearPositionalEmbedding(max_len), 100 in the reference) / `pos_emb_any_length=True`, which
        lifts the reference's T == max_len restriction (its torch.cat fails otherwise): the kernels generate the row
        t / max_len for whatever window length they are given."""
        super().__init__()
        n_in = n_keypoints * 2
        self.pos_emb_any_length = bool(pos_emb_any_length)
        if pos_emb:
            self.pos_emb = LinearPositionalEmbedding(max_len=int(pos_emb_max_len))          # HandPoseModels.py:23
            self.conv1 = nn.Conv1d(n_in + 1, conv_channels, kernel_size=5, padding=2)      # :24
        else:
            self.pos_emb = None
            self.conv1 = nn.Conv1d(n_in, conv_channels, kernel_size=5, padding=2)          # :28
        self.conv2 = nn.Conv1d(conv_channels, conv_channels, kernel_size=5, padding=2)     # :30
        self.conv3 = nn.Conv1d(conv_channels, conv_channels, kernel_size=5, padding=2)     # :31
        self.conv4 = nn.Conv1d(conv_channels, 2 * 21, kernel_size=5, padding=2)            # :32
        if activation == "ReLU":
            self.activation = nn.ReLU()                                                     # :34-35
        else:
            raise ValueError()                                                              # :37
        if precision not in _lib.PRECISIONS:
            raise ValueError(f"precision must be one of {sorted(_lib.PRECISIONS)}")
        self.precision = precision
        self.conv_channels = int(conv_channels)
        self.n_in = n_in
        self._flat = None
        self._packed = None
        self._packed_versions = None
        self._workspace = None
        self._utt_workspace = None
        self._val_workspace = None
        self._flatten()

    # ------------------------------------------------------------------ flat parameter storage
    def _ordered_params(self):
        return [self.conv1.weight, self.conv1.bias, self.conv2.weight, self.conv2.bias,
                self.conv3.weight, self.conv3.bias, self.conv4.weight, self.conv4.bias]

    def _flatten(self):
        """Make the 8 parameters views of one contiguous fp32 buffer (state_dict order)."""
        ps = self._ordered_params()
        dev = ps[0].device
        flat = torch.empty(sum(p.numel() for p in ps), dtype=torch.float32, device=dev)
        off = 0
        with torch.no_grad():
            for p in ps:
                n = p.numel()
                flat[off:off + n].copy_(p.detach().reshape(-1).to(torch.float32))
                p.data = flat[off:off + n].view(p.shape)
                p._b2h_owner_id = id(self)
                off += n
        _OWNERS[id(self)] = self
        self._flat = flat
        self._packed = None
        self._packed_versions = None
        self._workspace = None

    def __getstate__(self):
        st = dict(self.__dict__)
        for k in ("_flat", "_packed", "_packed_versions", "_workspace", "_utt_workspace", "_val_workspace"):
            st[k] = None
        return st

    def __setstate__(self, st):
        self.__dict__.update(st)
        self._flatten()

    def _is_flat(self):
        if self._flat is None:
            return False
        base, off = self._flat.data_ptr(), 0
        for p in self._ordered_params():
            if p.data_ptr() != base + off * 4 or p.dtype != torch.float32 or not p.is_contiguous():
                return False
            off += p.numel()
        return True

    def _apply(self, fn, *args, **kwargs):
        out = super()._apply(fn, *args, **kwargs)    # .to()/.cuda()/.float(): moves every param on its own
        self._flatten()
        return out

    def flat_parameters(self):
        if not self._is_flat():
            self._flatten()
        return self._flat

    def mark_packed_stale(self):
        self._packed_versions = None

    def _geometry(self):
        # C-ABI `pos_emb`: 0 = off, 1 = on with max_len 100 (the reference), n > 1 = on with max_len n
        if self.pos_emb is None:
            return self.n_in, self.conv_channels, 0
        return self.n_in, self.conv_channels, (1 if self.pos_emb.max_len == 100 else int(self.pos_emb.max_len))

    def packed_weights(self, fresh_from_kernel=False):
        """Extension-owned operand layouts (fp32 tap-major + bf16 UMMA blocks), rebuilt lazily when any
        parameter's version counter moved (load_state_dict, a stock torch optimiser, manual edits)."""
        flat = self.flat_parameters()
        _lib.require_device(flat, "ConvModel parameters")
        n_in, C, pe = self._geometry()
        if self._packed is None or self._packed.device != flat.device:
            self._packed = torch.zeros(_lib.packed_bytes(n_in, C, pe), dtype=torch.uint8, device=flat.device)
            self._packed_versions = None
        versions = tuple(p._version for p in self._ordered_params())
        if fresh_from_kernel:
            self._packed_versions = versions
        elif self._packed_versions != versions:
            lib = _lib.load()
            _lib.check(lib.b2h_pack_weights(_lib.ptr(flat), _lib.ptr(self._packed), n_in, C, pe, _lib.stream_ptr(flat.device)))
            self._packed_versions = versions
        return self._packed

    def _cached_workspace(self, attr, query, a, b, zero=False):
        """The buffer cached in `attr`, grown on demand (zeroed if `zero`) to the size C-ABI `query`(a, b, geometry,
        precision) returns."""
        n_in, C, pe = self._geometry()
        need = _lib.query(query, int(a), int(b), n_in, C, pe, _lib.PRECISIONS[self.precision])
        buf, dev = getattr(self, attr), self._flat.device
        if buf is None or buf.numel() < need or buf.device != dev:
            buf = (torch.zeros if zero else torch.empty)(need, dtype=torch.uint8, device=dev)
            setattr(self, attr, buf)
        return buf

    def workspace(self, B, T, segments=False):
        """The training workspace for a batch of B windows of T frames, or (segments=True) for B segments of at most T
        frames (b2h_train_utterances_workspace_bytes).  One buffer, grown on demand: its header is shared by every step."""
        query = "b2h_train_utterances_workspace_bytes" if segments else "b2h_workspace_bytes"
        return self._cached_workspace("_workspace", query, B, T, zero=True)    # holds the fused kernel's grid-barrier words

    # ------------------------------------------------------------------ kernels
    def _check_input(self, x, T=None):
        """The model-level checks of every entry point, on windows x (B, T, K, 2) or, with T given, on a frame stream
        x (F, K, 2) read as windows of T frames (T = ANY_LENGTH: as sequences of any length): a CUDA tensor on an sm_100
        device and on the model's device, K * 2 = n_in channels, float32 / bfloat16, and the pos_emb window length.
        Returns (B or F, T)."""
        stream = T is not None
        _lib.require_device(x, "frame stream" if stream else "ConvModel input")
        _lib.require_sm100(x.device)
        if x.dim() != (3 if stream else 4):
            raise RuntimeError(f"ConvModel expects {'a frame stream (F, K, 2)' if stream else '(B, T, K, 2)'}, "
                               f"got {tuple(x.shape)}")
        if x.shape[-2] * x.shape[-1] != self.n_in:
            # the reference fails inside conv1 with a channel-mismatch RuntimeError (SURVEY.md §0.4)
            raise RuntimeError(f"expected input with {self.n_in} channels (K*2), got {x.shape[-2] * x.shape[-1]} channels instead")
        T = T if stream else x.shape[1]
        if self.pos_emb is not None and T != self.pos_emb.max_len and not self.pos_emb_any_length:
            # torch.cat in LinearPositionalEmbedding.forward fails unless T == max_len (HandPoseModels.py:82)
            got = " (sequences of any length need pos_emb_any_length=True)" if T is ANY_LENGTH else f", got {T}"
            raise RuntimeError(f"Sizes of tensors must match: pos_emb requires T == {self.pos_emb.max_len}{got}")
        if x.dtype not in (torch.float32, torch.bfloat16):
            raise RuntimeError(f"ConvModel input must be float32 or bfloat16, got {x.dtype}")
        if self._flat.device != x.device:
            raise RuntimeError(f"input is on {x.device} but the model is on {self._flat.device}")
        return x.shape[0], T

    def _forward_impl(self, inp, lengths=None, out_scale=1.0):
        B, T = self._check_input(inp)
        x = inp.contiguous()
        n_in, C, pe = self._geometry()
        packed = self.packed_weights()
        y = torch.empty((B, T, 21, 2), dtype=torch.float32, device=x.device)
        len32 = None if lengths is None else _lib.lengths_i32(lengths, x.device, B)
        _lib.check(_lib.load().b2h_conv_forward(_lib.ptr(x), _lib.dtype_code(x.dtype), _lib.ptr(self._flat), _lib.ptr(packed),
                                                _lib.ptr(len32), _lib.ptr(y), B, T, n_in, C, pe,
                                                _lib.PRECISIONS[self.precision], 1 if len32 is not None else 0,
                                                float(out_scale), _lib.stream_ptr(x.device)))
        return y

    def _backward_impl(self, x, grad_y):
        B, T = x.shape[0], x.shape[1]
        xc = x.contiguous()
        gy = grad_y.to(torch.float32).contiguous().view(B, T, 42)
        n_in, C, pe = self._geometry()
        packed = self.packed_weights()
        ws = self.workspace(B, T)
        grads = torch.empty_like(self._flat)
        lib = _lib.load()
        _lib.check(lib.b2h_conv_backward(_lib.ptr(xc), _lib.dtype_code(xc.dtype),
                                         _lib.ptr(gy), _lib.ptr(self._flat), _lib.ptr(packed), _lib.ptr(grads), B, T,
                                         n_in, C, pe, _lib.PRECISIONS[self.precision], _lib.ptr(ws), ws.numel(),
                                         _lib.stream_ptr(xc.device)))
        out, off = [], 0
        for p in self._ordered_params():
            out.append(grads[off:off + p.numel()].view(p.shape))
            off += p.numel()
        return out

    def forward(self, inp):
        """inp (B,T,K,2) -> (B,T,21,2)   HandPoseModels.py:40-64.  (The reference returns a permuted
        view of a (B,42,T) tensor; this returns the same values contiguous.)"""
        if not self._is_flat():
            self._flatten()
        if torch.is_grad_enabled() and inp.requires_grad:
            # the kernels compute parameter gradients only: a trainable module in front of this one would silently get none
            raise RuntimeError("ConvModel computes no input gradient: its input must not require grad "
                               "(detach it, or run the modules in front of ConvModel without autograd)")
        if torch.is_grad_enabled() and any(p.requires_grad for p in self._ordered_params()):
            return _ConvForward.apply(inp, self, *self._ordered_params())
        return self._forward_impl(inp)

    @torch.no_grad()
    def predict(self, inp, lengths=None, denormalize=None):
        """Inference helper: forward with the optional fused epilogues -- mask_output(lengths)
        (steps/utils.py:309-312) and `prediction *= 1280` (steps/traintest.py:270-271)."""
        if not self._is_flat():
            self._flatten()
        return self._forward_impl(inp, lengths=lengths, out_scale=1.0 if denormalize is None else float(denormalize))


    @torch.no_grad()
    def predict_windows(self, frames, win_start, T, win_end=None, pad_mode="repeat_first", lengths=None, denormalize=None, out=None):
        """Streaming inference over sliding windows WITHOUT materialising them: `frames` (F, K, 2) is the per-frame
        network input of a whole clip (`PreprocessRightHand.frame_stream`), window w covers frames
        [win_start[w], win_start[w] + T) cut at win_end[w] (default F) and padded by the dataset's rule
        (text_pose_dataset.py:511-518 repeat-first / :614-622 zeros).  Returns (W, T, 21, 2), identical to
        `predict` on the materialised (W, T, K, 2) windows.  Every shape `predict` runs on the tensor cores: bf16 mode with
        conv_channels <= 256 and T <= 256, conv_channels <= 48 and T <= 640 or conv_channels <= 32 and T <= 1024 (the
        last two with at most 32 input channels), fp32 mode with conv_channels <= 32 and T <= 256, at any number of
        windows; other shapes raise B2HError."""
        if not self._is_flat():
            self._flatten()
        F, T = self._check_input(frames, T)
        dev = frames.device
        x = frames.contiguous()
        ws = torch.as_tensor(win_start).to(device=dev, dtype=torch.int64).contiguous()
        we = None if win_end is None else torch.as_tensor(win_end).to(device=dev, dtype=torch.int64).contiguous()
        W = ws.numel()
        len32 = None if lengths is None else _lib.lengths_i32(lengths, dev, W)
        n_in, C, pe = self._geometry()
        y = out if out is not None else torch.empty((W, T, 21, 2), dtype=torch.float32, device=dev)
        _lib.check(_lib.load().b2h_conv_forward_windows(
            _lib.ptr(x), _lib.dtype_code(x.dtype), F, _lib.ptr(ws), _lib.ptr(we), _lib.PAD_MODES[pad_mode],
            _lib.ptr(self._flat), _lib.ptr(self.packed_weights()), _lib.ptr(len32), _lib.ptr(y), W, T, n_in, C, pe,
            _lib.PRECISIONS[self.precision], 1 if len32 is not None else 0, 1.0 if denormalize is None else float(denormalize),
            _lib.stream_ptr(dev)))
        return y

    def utterances_workspace(self, n_frames, n_utt):
        """The workspace of predict_utterances (the device-side sub-window plan), cached on the model like workspace()."""
        return self._cached_workspace("_utt_workspace", "b2h_utterances_workspace_bytes", n_frames, n_utt)

    def validate_workspace(self, n_seg, max_len):
        """The workspace of steps.validate_utterances (sub-window table, segment pairs, per-sub-window sums) for n_seg
        segments of at most max_len frames, cached on the model like utterances_workspace() and apart from the training
        workspace, so a validation pass may sit between training steps (and graphs) on the same stream."""
        return self._cached_workspace("_val_workspace", "b2h_validate_utterances_workspace_bytes", n_seg, max_len)

    @torch.no_grad()
    def predict_utterances(self, frames, offsets, denormalize=None, out=None):
        """Inference over packed utterances of any length, one prediction per frame: the reference's infer_utterance
        (steps/traintest.py:214-300) for every utterance at once.  `frames` (F, K, 2) is a frame stream
        (`PreprocessRightHand.frame_stream`), `offsets` (S + 1,) int64 non-decreasing (`PackedClips.offsets`): utterance u
        owns rows [offsets[u], offsets[u+1]).  Returns (F, 21, 2) fp32 (`out` if given): row f of utterance u is
        ConvModel.forward of frames[offsets[u]:offsets[u+1]] as one sequence at that frame (times `denormalize`, e.g. 1280);
        rows outside [offsets[0], offsets[S]) are not written (zeros when `out` is None).  Host offsets (numpy, list, CPU
        tensor) are checked here (ValueError) and uploaded; device offsets are used as given, checked by the kernels (bad ones
        write nothing and set b2h_tc_status).  Served in bf16 mode for conv_channels <= 256 and in fp32 mode for
        conv_channels <= 32 with at most 32 input channels; other shapes raise B2HError."""
        if not self._is_flat():
            self._flatten()
        F, _ = self._check_input(frames, ANY_LENGTH)
        dev = frames.device
        x = frames.contiguous()
        if isinstance(offsets, torch.Tensor) and offsets.is_cuda:
            if offsets.dtype != torch.int64 or offsets.dim() != 1 or offsets.numel() < 1 or offsets.device != dev:
                raise ValueError("device offsets must be a 1-D int64 tensor of S + 1 entries on the frames' device")
            off = offsets.contiguous()
        else:
            o = np.asarray(offsets.cpu() if isinstance(offsets, torch.Tensor) else offsets)
            if o.ndim != 1 or o.size < 1 or not np.issubdtype(o.dtype, np.integer):
                raise ValueError("offsets must be a 1-D integer array of S + 1 entries")
            if (np.diff(o) < 0).any() or o[0] < 0 or o[-1] > F:
                raise ValueError(f"offsets must be non-decreasing within [0, {F}]")
            off = torch.from_numpy(o.astype(np.int64)).to(dev)
        S = off.numel() - 1
        n_in, C, pe = self._geometry()
        y = out if out is not None else torch.zeros((F, 21, 2), dtype=torch.float32, device=dev)
        ws = self.utterances_workspace(F, S)
        _lib.check(_lib.load().b2h_conv_forward_utterances(
            _lib.ptr(x), _lib.dtype_code(x.dtype), F, _lib.ptr(off), S, _lib.ptr(self._flat), _lib.ptr(self.packed_weights()),
            _lib.ptr(y), n_in, C, pe, _lib.PRECISIONS[self.precision], 1.0 if denormalize is None else float(denormalize),
            _lib.ptr(ws), ws.numel(), _lib.stream_ptr(dev)))
        return y


def format_prediction(prediction, fmt="openpose"):
    """SURVEY 8f N2: (..., 21, 2) predictions -> (..., 63) rows in the reference's writer layouts:
    "openpose" = [x,y,1.0]*21 (array2open_pose, steps/utils.py:355-364), "h5" = [x*21 | y*21 | 0*21]
    (order_and_reshape_toh5, steps/traintest.py:302-317).  Pure data movement on the GPU (bit-exact)."""
    _lib.require_device(prediction, "prediction")
    if prediction.shape[-2:] != (21, 2) or prediction.dtype != torch.float32:
        raise RuntimeError("format_prediction expects float32 (..., 21, 2)")
    mode = {"openpose": 0, "h5": 1}[fmt]
    p = prediction.contiguous()
    rows = p.numel() // 42
    out = torch.empty(p.shape[:-2] + (63,), dtype=torch.float32, device=p.device)
    _lib.check(_lib.load().b2h_format_prediction(_lib.ptr(p), _lib.ptr(out), rows, mode, _lib.stream_ptr(p.device)))
    return out
