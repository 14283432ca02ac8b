"""Drop-ins for the hot-path pieces of the reference's `steps` package
(body2hand/src/steps/utils.py, body2hand/src/steps/traintest.py): `mask_output`, `maskedPoseL1`,
`poderatedPoseL1`, the Adam step, and the fused training iteration of traintest.py:94-123.
Every arithmetic op runs in libb2h.so; nothing here computes on the CPU or through torch ops."""
from __future__ import annotations

import torch
import torch.nn as nn

from . import _lib
from .models import ANY_LENGTH, ConvModel, owner_of


class _MaskOutput(torch.autograd.Function):
    @staticmethod
    def forward(ctx, output, len32):
        B, T = output.shape[0], output.shape[1]
        row = output[0, 0].numel() if output.dim() > 2 else 1
        lib = _lib.load()
        _lib.check(lib.b2h_mask_output(_lib.ptr(output), _lib.ptr(len32), B, T, row, _lib.stream_ptr(output.device)))
        ctx.mark_dirty(output)
        ctx.save_for_backward(len32)
        return output

    @staticmethod
    def backward(ctx, grad):
        (len32,) = ctx.saved_tensors
        g = grad.contiguous().clone()
        B, T = g.shape[0], g.shape[1]
        row = g[0, 0].numel() if g.dim() > 2 else 1
        lib = _lib.load()
        _lib.check(lib.b2h_mask_output(_lib.ptr(g), _lib.ptr(len32), B, T, row, _lib.stream_ptr(g.device)))
        return g, None


def mask_output(output, lengths):
    """steps/utils.py:309-312: `output[i, len_i:, :] = 0` in place; returns the same tensor."""
    _lib.require_device(output, "mask_output input")
    if output.dtype != torch.float32 or not output.is_contiguous():
        raise RuntimeError("mask_output expects a contiguous float32 tensor (ConvModel's output is)")
    len32 = _lib.lengths_i32(lengths, output.device, output.shape[0])
    return _MaskOutput.apply(output, len32)


class _PoseL1(torch.autograd.Function):
    @staticmethod
    def forward(ctx, prediction, target, len32, scores, kind):
        B, T = prediction.shape[0], prediction.shape[1]
        row = prediction[0, 0].numel()
        pred = prediction.contiguous()
        tgt = target.to(device=pred.device, dtype=torch.float32).contiguous()
        sc = None if scores is None else scores.to(device=pred.device, dtype=torch.float32).contiguous()
        loss = torch.empty((), dtype=torch.float32, device=pred.device)
        need_grad = prediction.requires_grad
        d_pred = torch.empty_like(pred) if need_grad else None
        scratch = torch.empty(B, dtype=torch.float32, device=pred.device)
        lib = _lib.load()
        _lib.check(lib.b2h_pose_l1(_lib.ptr(pred), _lib.ptr(tgt), _lib.ptr(sc), _lib.ptr(len32), B, T, row, kind,
                                   _lib.ptr(loss), _lib.ptr(d_pred), _lib.ptr(scratch), _lib.stream_ptr(pred.device)))
        ctx.d_pred = d_pred
        return loss

    @staticmethod
    def backward(ctx, grad_loss):
        d = ctx.d_pred
        if d is None:
            return None, None, None, None, None
        return d * grad_loss, None, None, None, None


def _criterion_checks(prediction, target):
    _lib.require_device(prediction, "criterion prediction")
    if prediction.dtype != torch.float32:
        raise RuntimeError("criterion expects float32 predictions")
    if prediction.shape != target.shape:
        raise RuntimeError(f"prediction {tuple(prediction.shape)} and target {tuple(target.shape)} differ")


class maskedPoseL1(nn.Module):
    """steps/utils.py:413-428: mean over the batch of per-sample mean |pred-target| over the first
    len_i frames."""

    def forward(self, prediction, target, lengths):
        _criterion_checks(prediction, target)
        len32 = _lib.lengths_i32(lengths, prediction.device, prediction.shape[0])
        return _PoseL1.apply(prediction, target, len32, None, _lib.LOSS_L1)


class poderatedPoseL1(nn.Module):
    """steps/utils.py:431-452: confidence-weighted, SUM over the batch of per-sample means."""

    def forward(self, prediction, target, lengths, scores):
        _criterion_checks(prediction, target)
        len32 = _lib.lengths_i32(lengths, prediction.device, prediction.shape[0])
        return _PoseL1.apply(prediction, target, len32, scores, _lib.LOSS_CONFL1)


class L12Pixels:
    """steps/utils.py:291-299 (host scalar)."""

    def __init__(self, num_joints, upsample):
        self.num_joints = num_joints
        self.upsample = upsample

    def __call__(self, mse):
        return mse / self.num_joints * self.upsample


def adjust_learning_rate(base_lr, lr_decay, optimizer, epoch):
    """steps/utils.py:301-307"""
    lr = base_lr * (0.1 ** (epoch / lr_decay))
    for param_group in optimizer.param_groups:
        param_group["lr"] = lr
    return lr


def _flat_view(gs, P):
    """The per-parameter gradients our backward returns are slices of one flat tensor: view them as it."""
    g0 = gs[0]
    base, off = g0.data_ptr(), 0
    for g in gs:
        if g.dtype != torch.float32 or not g.is_contiguous() or g.data_ptr() != base + off * 4:
            return None
        off += g.numel()
    if g0.untyped_storage().nbytes() - g0.storage_offset() * 4 < P * 4:
        return None
    return g0.as_strided((P,), (1,))


class FusedAdam(torch.optim.Optimizer):
    """torch.optim.Adam(params, lr) with torch's defaults (traintest.py:48), one CUDA launch per step
    over the model's flat parameter buffer.  state_dict() keeps torch's layout
    ({state: {i: {step, exp_avg, exp_avg_sq}}, param_groups}) so `last_optim.pth` files interchange
    with the reference (traintest.py:64-70, 147)."""

    def __init__(self, params, lr=1e-3, betas=(0.9, 0.999), eps=1e-8):
        defaults = dict(lr=lr, betas=betas, eps=eps, weight_decay=0, amsgrad=False, maximize=False, foreach=None,
                        capturable=False, differentiable=False, fused=None)
        super().__init__(params, defaults)
        self._flat_state = {}

    def _owner(self, group):
        ps = group["params"]
        model = owner_of(ps[0])
        if model is None or len(ps) != 8:
            return None
        if not model._is_flat():
            model._flatten()
        if any(a is not b for a, b in zip(ps, model._ordered_params())):
            return None
        return model

    def _group_state(self, gi, group, model):
        """flat exp_avg / exp_avg_sq for a whole-model group, exposed per parameter as views."""
        flat = model.flat_parameters()
        st = self._flat_state.get(gi)
        if st is None or st["m"].device != flat.device or st["m"].numel() != flat.numel():
            m = torch.zeros_like(flat)
            v = torch.zeros_like(flat)
            step = 0
            off = 0
            for p in group["params"]:          # adopt anything load_state_dict() put there
                ps = self.state.get(p, {})
                n = p.numel()
                if "exp_avg" in ps:
                    m[off:off + n].copy_(ps["exp_avg"].reshape(-1))
                    v[off:off + n].copy_(ps["exp_avg_sq"].reshape(-1))
                    step = int(ps["step"]) if "step" in ps else step
                off += n
            step_t = torch.tensor(float(step))      # ONE host tensor shared by the 8 per-parameter states
            # device-side step counter + learning rate, shared by every runner built on this optimiser (a captured
            # graph advances / reads them on the device); "dev_step_mirror" = the value the host believes is in step_dev
            st = {"m": m, "v": v, "step": step, "step_t": step_t,
                  "step_dev": torch.full((1,), step, dtype=torch.int64, device=flat.device), "dev_step_mirror": step,
                  "lr_dev": torch.full((1,), float(group["lr"]), dtype=torch.float64, device=flat.device),
                  "lr_mirror": float(group["lr"])}
            self._flat_state[gi] = st
            off = 0
            for p in group["params"]:
                n = p.numel()
                self.state[p] = {"step": step_t,
                                 "exp_avg": m[off:off + n].view(p.shape),
                                 "exp_avg_sq": v[off:off + n].view(p.shape)}
                off += n
        return st

    def load_state_dict(self, state_dict):
        super().load_state_dict(state_dict)
        self._flat_state = {}                  # re-adopt the loaded tensors on the next step

    @torch.no_grad()
    def step(self, closure=None, flat_grads=None, grad_scale=1.0):
        loss = closure() if closure is not None else None
        lib = _lib.load()
        for gi, group in enumerate(self.param_groups):
            b1, b2 = group["betas"]
            model = self._owner(group)
            if model is not None:
                st = self._group_state(gi, group, model)
                flat = model.flat_parameters()
                if flat_grads is None:
                    gs = [p.grad for p in group["params"]]
                    if any(g is None for g in gs):
                        continue
                    fg = _flat_view(gs, flat.numel())
                    if fg is None:
                        fg = torch.cat([g.reshape(-1).to(torch.float32) for g in gs])
                else:
                    fg = flat_grads
                st["step"] += 1
                n_in, C, pe = model._geometry()
                packed = model.packed_weights()
                _lib.check(lib.b2h_adam_step(_lib.ptr(flat), _lib.ptr(fg), _lib.ptr(st["m"]), _lib.ptr(st["v"]),
                                             flat.numel(), float(group["lr"]), b1, b2, group["eps"], st["step"],
                                             None, None, float(grad_scale), _lib.ptr(packed), n_in, C, pe,
                                             _lib.stream_ptr(flat.device)))
                model.packed_weights(fresh_from_kernel=True)
                st["step_t"].fill_(float(st["step"]))
            else:
                for p in group["params"]:
                    if p.grad is None:
                        continue
                    _lib.require_device(p, "FusedAdam parameter")
                    s = self.state[p]
                    if "exp_avg" not in s:
                        s["step"] = torch.tensor(0.0)
                        s["exp_avg"] = torch.zeros_like(p, memory_format=torch.contiguous_format)
                        s["exp_avg_sq"] = torch.zeros_like(p, memory_format=torch.contiguous_format)
                    s["step"] = s["step"] + 1
                    g = p.grad.contiguous()
                    _lib.check(lib.b2h_adam_step(_lib.ptr(p), _lib.ptr(g), _lib.ptr(s["exp_avg"]), _lib.ptr(s["exp_avg_sq"]),
                                                 p.numel(), float(group["lr"]), b1, b2, group["eps"], int(s["step"]),
                                                 None, None, float(grad_scale), None, 0, 0, 0, _lib.stream_ptr(p.device)))
                    owner = owner_of(p)
                    if owner is not None:
                        owner.mark_packed_stale()
        return loss


def _dense_inputs(model: ConvModel, batch, loss):
    """The C arguments in front of `params` of the dense training entry points (x, x_dtype, target, conf, lengths; tensors
    stay tensors), and the batch size, window length and device."""
    x = batch["input_kp"]
    B, T = model._check_input(x)
    dev = x.device
    tgt = batch["target_kp"].to(device=dev, dtype=torch.float32).contiguous()
    conf = batch["target_conf"].to(device=dev, dtype=torch.float32).contiguous() if _lib.LOSSES[loss] == _lib.LOSS_CONFL1 else None
    return (x.contiguous(), _lib.dtype_code(x.dtype), tgt, conf, _lib.lengths_i32(batch["n_frames"], dev, B)), B, T, dev


def _stream_inputs(model: ConvModel, streams, T, loss):
    """The three training streams, checked: (frames, x_dtype, target_frames, conf_frames, n_frames) and the device."""
    x = streams["input_kp"]
    F, T = model._check_input(x, T)
    dev = x.device
    tgt = streams["target_kp"].to(device=dev, dtype=torch.float32).contiguous()
    if tgt.numel() != F * 42:
        raise RuntimeError(f"target_kp stream has {tgt.numel()} values for {F} frames (expected (F, 21, 2))")
    conf = None
    if _lib.LOSSES[loss] == _lib.LOSS_CONFL1:
        conf = streams["target_conf"].to(device=dev, dtype=torch.float32).contiguous()
        if conf.numel() != F * 21:
            raise RuntimeError(f"target_conf stream has {conf.numel()} values for {F} frames (expected (F, 21))")
    return (x.contiguous(), _lib.dtype_code(x.dtype), tgt, conf, F), dev


def _view_inputs(model: ConvModel, streams, win_start, T, lengths, win_end, pad_mode, loss):
    """`_dense_inputs` of the *_windows entry points: (frames, x_dtype, target_frames, conf_frames, n_frames, win_start,
    win_end, pad_mode, lengths), and the number of windows, T and the device."""
    head, dev = _stream_inputs(model, streams, T, loss)
    ws = torch.as_tensor(win_start).to(device=dev, dtype=torch.int64).contiguous()
    W = ws.numel()
    we = None if win_end is None else torch.as_tensor(win_end).to(device=dev, dtype=torch.int64).contiguous()
    if we is not None and we.numel() != W:
        raise RuntimeError("win_end must have one entry per window")
    return (*head, ws, we, _lib.PAD_MODES[pad_mode], _lib.lengths_i32(lengths, dev, W)), W, T, dev


def _segment_inputs(model: ConvModel, streams, seg_start, seg_end, max_len, loss):
    """`_view_inputs` of the *_utterances entry points: (frames, x_dtype, target_frames, conf_frames, n_frames, seg_start,
    seg_end, n_seg, max_len), and the number of segments, max_len and the device.  max_len defaults to the longest host-side
    segment; device segments need it given."""
    head, dev = _stream_inputs(model, streams, ANY_LENGTH, loss)
    on_device = any(isinstance(t, torch.Tensor) and t.is_cuda for t in (seg_start, seg_end))
    if max_len is None:
        if on_device:
            raise ValueError("max_len is required when the segments are already on the device")
        lens = torch.as_tensor(seg_end).reshape(-1).to(torch.int64) - torch.as_tensor(seg_start).reshape(-1).to(torch.int64)
        max_len = int(lens.max()) if lens.numel() else 1
    ss = torch.as_tensor(seg_start).to(device=dev, dtype=torch.int64).contiguous()
    se = torch.as_tensor(seg_end).to(device=dev, dtype=torch.int64).contiguous()
    S = ss.numel()
    if S < 1 or se.numel() != S:
        raise RuntimeError("seg_start and seg_end must have one entry per segment (at least one)")
    return (*head, ss, se, S, int(max_len)), S, int(max_len), dev


def _train_step(entry, model, optimizer, inputs, loss, who):
    """forward + criterion + backward + reduction + Adam + re-pack through C entry point `entry`
    (b2h_train_step[_windows|_utterances]).  The segment step takes its shape in `inputs` and the Adam step from the
    device-side counter, which it advances."""
    args, W, T, dev = inputs
    segments = entry.endswith("_utterances")
    group = optimizer.param_groups[0]
    if optimizer._owner(group) is not model:
        raise RuntimeError(f"{who} needs FusedAdam(model.parameters()) over exactly this model")
    st = optimizer._group_state(0, group, model)
    if segments and st["dev_step_mirror"] != st["step"]:
        st["step_dev"].fill_(int(st["step"]))
    st["step"] += 1
    n_in, C, pe = model._geometry()
    packed = model.packed_weights()
    ws = model.workspace(W, T, segments)
    flat = model.flat_parameters()
    loss_out = torch.empty((), dtype=torch.float32, device=dev)
    b1, b2 = group["betas"]
    _lib.check(getattr(_lib.load(), entry)(
        *_lib.ptrs(args), _lib.ptr(flat), _lib.ptr(packed), _lib.ptr(st["m"]), _lib.ptr(st["v"]), _lib.ptr(loss_out),
        *(() if segments else (W, T)), n_in, C, pe, _lib.LOSSES[loss], _lib.PRECISIONS[model.precision], float(group["lr"]),
        b1, b2, group["eps"], st["step"], _lib.ptr(st["step_dev"]) if segments else None, None, _lib.ptr(ws), ws.numel(),
        _lib.stream_ptr(dev)))
    if segments:
        st["dev_step_mirror"] = st["step"]
    model.packed_weights(fresh_from_kernel=True)
    st["step_t"].fill_(float(st["step"]))
    return loss_out


def _forward_backward(entry, model, inputs, loss, want_pred):
    """forward + criterion + backward and the gradient reduction through C entry point `entry`
    (b2h_train_forward_backward[_windows|_utterances])."""
    args, W, T, dev = inputs
    segments = entry.endswith("_utterances")
    n_in, C, pe = model._geometry()
    packed = model.packed_weights()
    ws = model.workspace(W, T, segments)
    flat = model.flat_parameters()
    grads = torch.empty_like(flat)
    loss_out = torch.empty((), dtype=torch.float32, device=dev)
    pred = torch.empty((W, T, 21, 2), dtype=torch.float32, device=dev) if want_pred else None
    _lib.check(getattr(_lib.load(), entry)(
        *_lib.ptrs(args), _lib.ptr(flat), _lib.ptr(packed), _lib.ptr(grads), _lib.ptr(loss_out), _lib.ptr(pred),
        *(() if segments else (W, T)), n_in, C, pe, _lib.LOSSES[loss], _lib.PRECISIONS[model.precision], None, _lib.ptr(ws),
        ws.numel(), _lib.stream_ptr(dev)))
    return (loss_out, grads, pred) if want_pred else (loss_out, grads)


def fused_train_step(model: ConvModel, batch, optimizer: FusedAdam, loss="L1"):
    """The body of the reference's hot loop, traintest.py:94-121, as two launches:
    forward + mask_output + criterion + backward (one kernel), cross-CTA gradient reduction + Adam +
    weight re-pack (one kernel).  `batch` is the reference's batch dict (input_kp, target_kp, n_frames
    [, target_conf]) with tensors already on the model's device.  Returns the loss as a 0-dim device
    tensor (no host sync; call .item() only when you log it, cf. traintest.py:123)."""
    return _train_step("b2h_train_step", model, optimizer, _dense_inputs(model, batch, loss), loss, "fused_train_step")


def forward_backward(model: ConvModel, batch, loss="L1", want_pred=False):
    """traintest.py:94-120 without the optimiser: returns (loss 0-dim tensor, flat gradient tensor
    [, masked prediction]).  Used by the data-parallel trainer (all-reduce between this and Adam)."""
    return _forward_backward("b2h_train_forward_backward", model, _dense_inputs(model, batch, loss), loss, want_pred)


def fused_train_step_windows(model: ConvModel, streams, win_start, T, lengths, optimizer: FusedAdam, win_end=None,
                             pad_mode="repeat_first", loss="L1"):
    """`fused_train_step` on window views of device-resident frame streams: `streams` = {input_kp (F, K, 2) fp32 / bf16,
    target_kp (F, 21, 2), target_conf (F, 21) for confL1} (`PreprocessRightHand.training_stream`); window w covers frames
    [win_start[w], win_start[w] + T) cut at win_end[w] (default F) and padded by the dataset's rule, in all three streams.
    `lengths` = the windows' n_frames.  Bit-identical to `fused_train_step` on the windows K0 materialises; served where
    the tensor cores train (b2h_kernel_choice tile / wide), B2HError otherwise.  Returns the 0-dim device loss."""
    inputs = _view_inputs(model, streams, win_start, T, lengths, win_end, pad_mode, loss)
    return _train_step("b2h_train_step_windows", model, optimizer, inputs, loss, "fused_train_step_windows")


def forward_backward_windows(model: ConvModel, streams, win_start, T, lengths, win_end=None, pad_mode="repeat_first",
                             loss="L1", want_pred=False):
    """`forward_backward` on window views of frame streams (see `fused_train_step_windows`): returns (loss, flat gradients
    [, masked prediction (W, T, 21, 2)]), bit-identical to `forward_backward` on the materialised windows."""
    inputs = _view_inputs(model, streams, win_start, T, lengths, win_end, pad_mode, loss)
    return _forward_backward("b2h_train_forward_backward_windows", model, inputs, loss, want_pred)


def fused_train_step_utterances(model: ConvModel, streams, seg_start, seg_end, optimizer: FusedAdam, max_len=None, loss="L1"):
    """`fused_train_step` on SEGMENTS of device-resident frame streams, each trained as one whole sequence (utterances of
    any length): `streams` as in `fused_train_step_windows`; segment s = frames [seg_start[s], seg_end[s]) of all three
    streams, zero-padded only at its own two ends -- the reference's forward on a batch of one window of exactly L_s frames
    with lengths = [L_s].  L1 = (1/S) sum_s (per-segment mean), confL1 = sum_s (per-segment confidence-weighted mean).
    Whole utterances: `GpuPoseDataset.utterance_segments`.  `max_len` bounds every L_s (default: the longest host-side
    segment; required for device segments).  A segment outside [0, F] or not of 1..max_len frames (checked on the device)
    makes the step a no-op with a NaN loss and b2h_tc_status 81.  Served where the tile kernel trains (conv_channels <= 32,
    at most 32 input channels, bf16 or fp32 mode); B2HError otherwise.  Two launches; returns the 0-dim device loss."""
    inputs = _segment_inputs(model, streams, seg_start, seg_end, max_len, loss)
    return _train_step("b2h_train_step_utterances", model, optimizer, inputs, loss, "fused_train_step_utterances")


def forward_backward_utterances(model: ConvModel, streams, seg_start, seg_end, max_len=None, loss="L1", want_pred=False):
    """`forward_backward` on segments (see `fused_train_step_utterances`): returns (loss, flat gradients [, masked
    prediction (S, max_len, 21, 2): row t of segment s, zero for t >= L_s])."""
    inputs = _segment_inputs(model, streams, seg_start, seg_end, max_len, loss)
    return _forward_backward("b2h_train_forward_backward_utterances", model, inputs, loss, want_pred)


@torch.no_grad()
def validate_utterances(model: ConvModel, streams, seg_start, seg_end, max_len=None, loss="L1", per_segment=False):
    """validate() (traintest.py:168-211) on SEGMENTS of device-resident frame streams, each evaluated as one whole sequence:
    the loss `fused_train_step_utterances` computes for the same streams and segments (L1 = (1/S) sum_s per-segment mean,
    confL1 = sum_s per-segment confidence-weighted mean), from one forward and no backward.  Segment s is frames
    [seg_start[s], seg_end[s]) zero-padded only at its own two ends, the sequence `predict_utterances` sees at inference, so
    no pad frame reaches the last frames of a short utterance as it does in `validate_batch`'s padded crops.  Arguments as in
    `fused_train_step_utterances` (segments may overlap, repeat or leave gaps; `max_len` is required for device segments).
    Returns the 0-dim device loss, or (loss, seg_loss (S,)) with per_segment=True.  Parameters, packed weights and the
    optimiser state are only read; the workspace is `model.validate_workspace`, apart from the training one.  A segment
    outside [0, F] or not of 1..max_len frames (checked on the device) gives NaN in loss and every seg_loss entry and
    b2h_tc_status 81.  Deterministic (fixed summation order); three launches, graph capturable.  Served in bf16 mode for
    conv_channels <= 256 and in fp32 mode for conv_channels <= 32 with at most 32 input channels; B2HError otherwise.

    A validation split of whole utterances, reported in pixels as traintest.py:207 does:

        val_s, val_e = dataset.utterance_segments(val_indices)
        l1 = validate_utterances(model, dataset.training_streams(), val_s, val_e, loss="L1")
        print(L12Pixels(21, 1280)(l1.item()))
    """
    args, S, max_len, dev = _segment_inputs(model, streams, seg_start, seg_end, max_len, loss)
    n_in, C, pe = model._geometry()
    packed = model.packed_weights()
    flat = model.flat_parameters()
    ws = model.validate_workspace(S, max_len)
    loss_out = torch.empty((), dtype=torch.float32, device=dev)
    seg_loss = torch.empty(S, dtype=torch.float32, device=dev) if per_segment else None
    _lib.check(_lib.load().b2h_validate_utterances(
        *_lib.ptrs(args), _lib.ptr(flat), _lib.ptr(packed), _lib.ptr(seg_loss), _lib.ptr(loss_out), n_in, C, pe,
        _lib.LOSSES[loss], _lib.PRECISIONS[model.precision], _lib.ptr(ws), ws.numel(), _lib.stream_ptr(dev)))
    return (loss_out, seg_loss) if per_segment else loss_out


@torch.no_grad()
def validate_batch(model: ConvModel, batch, loss="L1"):
    """validate() body, traintest.py:174-207, for one batch: forward + mask_output + criterion."""
    pred = model.predict(batch["input_kp"], lengths=batch["n_frames"])
    if loss == "L1":
        return maskedPoseL1()(pred, batch["target_kp"], batch["n_frames"])
    return poderatedPoseL1()(pred, batch["target_kp"], batch["n_frames"], batch["target_conf"])
