"""Low-overhead steady-state runners: static device buffers, pre-bound C-ABI arguments, optional CUDA
graph capture.  The fused train step is ONE cooperative launch (~25 µs of GPU time at the reference's batch
sizes), so the per-call Python/torch bookkeeping of the modular API would dominate; these runners are
what a training / serving loop uses once shapes are fixed (SURVEY.md §0.7: launch latency, not the
tensor pipe or HBM, bounds every BASELINE config).

Input staging: every slot is ONE contiguous device buffer  [input_kp | target_kp | target_conf? | n_frames(int32)]
(WindowTrainStepRunner, over frame streams resident on the device: [win_start | win_end | n_frames];
UtteranceTrainStepRunner: [seg_start | seg_end])
and `host_stage(batch)` builds the same layout in pinned host memory, so a step's inputs travel with ONE
cudaMemcpyAsync (`load_staged`).  With `x_dtype=torch.bfloat16` the keypoint input is shipped as bf16 -- the bf16
kernels round it to bf16 on the way into shared memory anyway (cvt.rn == torch's CPU rounding), so the result is
bit-identical and the copy is 0.8 MB shorter at batch 256 x 64."""
from __future__ import annotations

import torch

from . import _lib
from .models import ConvModel
from .steps import FusedAdam, _dense_inputs, _segment_inputs, _view_inputs


def _align(n, a=256):
    return (n + a - 1) // a * a


def _check_x_dtype(model, x_dtype):
    if x_dtype == torch.bfloat16 and model.precision != "bf16":
        raise ValueError("bf16 inputs are only bit-identical to fp32 inputs in bf16 mode")


class _StepBuffers:
    """Static per-slot buffers shared by TrainStepRunner, WindowTrainStepRunner and parallel.DataParallelTrainer."""

    def _init_buffers(self, model: ConvModel, optimizer: FusedAdam, B: int, T: int, loss: str, n_slots: int, x_dtype):
        x_dtype = x_dtype or torch.float32
        if x_dtype not in (torch.float32, torch.bfloat16):
            raise ValueError("x_dtype must be torch.float32 or torch.bfloat16")
        _check_x_dtype(model, x_dtype)
        self.x_dtype = x_dtype
        K = model.n_in // 2
        conf = _lib.LOSSES[loss] == _lib.LOSS_CONFL1
        self._init_common(model, optimizer, B, T, loss, n_slots, (
            ("x", "input_kp", x_dtype, (B, T, K, 2)), ("target", "target_kp", torch.float32, (B, T, 21, 2)),
            ("conf", "target_conf", torch.float32, (B, T, 21) if conf else None), ("lengths", "n_frames", torch.int32, (B,))))
        self.lengths.fill_(T)

    def _init_common(self, model, optimizer, B, T, loss, n_slots, fields):
        """`fields`: (attribute, batch key, dtype, shape per slot or None) of every section of a slot.  A slot is ONE
        contiguous device buffer (every section 256-B aligned); `host_stage` builds the same layout in pinned host memory."""
        self.model, self.opt, self.B, self.T = model, optimizer, B, T
        self.loss_name = loss
        self.kind = _lib.LOSSES[loss]
        flat = model.flat_parameters()
        dev = flat.device
        _lib.require_device(flat, "model")
        _lib.require_sm100(dev)
        self.dev = dev
        group = optimizer.param_groups[0]
        if optimizer._owner(group) is not model:
            raise RuntimeError(f"{type(self).__name__} needs FusedAdam(model.parameters()) over exactly this model")
        self.state = optimizer._group_state(0, group, model)
        self.n_slots = n_slots
        self._fields = [(name, key, dtype) for name, key, dtype, shape in fields if shape is not None]
        # byte layout of one slot (every section 256-B aligned)
        self._sec = {}
        off = 0
        for name, _, dtype, shape in fields:
            nbytes = 0 if shape is None else torch.Size(shape).numel() * dtype.itemsize
            self._sec[name] = (off, nbytes)
            off = _align(off + nbytes)
        self.slot_bytes = off
        self.stage = torch.zeros((n_slots, self.slot_bytes), dtype=torch.uint8, device=dev)
        for name, _, dtype, shape in fields:
            o, n = self._sec[name]
            setattr(self, name, None if shape is None else self.stage[:, o:o + n].view(dtype).view((n_slots,) + tuple(shape)))
        self.loss = torch.zeros((n_slots,), dtype=torch.float32, device=dev)
        # Pinned, device-mapped host words: with step(..., to_host=True) the kernel stores the step's loss straight into host
        # memory (a 4-byte posted write over PCIe) -- a cudaMemcpy D2H of the loss queues behind the NEXT batch's 3.5 MB
        # H2D copy on the copy engine and serialises the input pipeline (measured: 109 -> 88 us per end-to-end step).
        self.loss_host = torch.zeros((n_slots,), dtype=torch.float32).pin_memory()
        # Adam step counter and learning rate in device memory, owned by the optimiser state and shared by every runner
        # on it: a captured graph advances the counter itself and follows adjust_learning_rate (traintest.py:83-84)
        self.step_dev = self.state["step_dev"]
        self.lr_dev = self.state["lr_dev"]
        self.ws = model.workspace(B, T)
        self.packed = model.packed_weights()
        self.lib = _lib.load()
        self.graph = None
        self._graph_steps = 0

    @property
    def host_steps(self):
        return int(self.state["step"])

    def _advance(self, n):
        self.state["step"] += n
        self.state["dev_step_mirror"] = self.state["step"]

    # ------------------------------------------------------------------ inputs
    def load(self, batch, slot=0, non_blocking=True):
        """Copy one batch dict (CPU pinned or device tensors) into slot `slot` (one copy per tensor; `load_staged` moves
        the same bytes with a single copy)."""
        for name, key, _ in self._fields:
            getattr(self, name)[slot].copy_(torch.as_tensor(batch[key]), non_blocking=non_blocking)

    def host_stage(self, batch, out=None):
        """Pack a batch dict (CPU tensors) into ONE pinned host buffer with the slot's byte layout (the collate step of a
        data loader).  Returns the uint8 tensor `load_staged` takes."""
        if out is None:
            out = torch.zeros(self.slot_bytes, dtype=torch.uint8).pin_memory()
        for name, key, dtype in self._fields:
            o, n = self._sec[name]
            out[o:o + n].view(dtype).copy_(torch.as_tensor(batch[key]).reshape(-1))
        return out

    def load_staged(self, staged, slot=0, non_blocking=True):
        """ONE host -> device copy of a `host_stage` buffer into slot `slot`."""
        self.stage[slot].copy_(staged, non_blocking=non_blocking)

    # ------------------------------------------------------------------ bookkeeping shared by step()/replay()
    def _sync_host_state(self):
        """Before enqueuing (never while capturing): follow a changed learning rate and out-of-band weight edits."""
        if torch.cuda.is_current_stream_capturing():
            return
        st = self.state
        lr = float(self.opt.param_groups[0]["lr"])
        if lr != st["lr_mirror"]:
            self.lr_dev.fill_(lr)
            st["lr_mirror"] = lr
        if st["dev_step_mirror"] != st["step"]:          # the modular optimiser path stepped in between
            self.step_dev.fill_(int(st["step"]))
            st["dev_step_mirror"] = st["step"]
        self.packed = self.model.packed_weights()        # cheap version compare; re-packs after load_state_dict etc.

    def _x_dt(self):
        return _lib.dtype_code(self.x_dtype)

    def _bind(self, entry, decode, tail=None):
        """Pre-binds the C arguments of step(): `decode(batch)` (steps._dense_inputs / _view_inputs) gives the leading
        arguments of a slot's batch dict {key: slot tensor}; `tail` the arguments after eps (default: b2h_train_step's)."""
        self._entry = entry
        self._decoded = [decode({key: getattr(self, name)[s] for name, key, _ in self._fields})[0] for s in range(self.n_slots)]
        self._inputs = [_lib.ptrs(args) for args in self._decoded]
        n_in, C, pe = self.model._geometry()
        self._shape = (self.B, self.T, n_in, C, pe, self.kind, _lib.PRECISIONS[self.model.precision])
        self._tail = tail or (0, _lib.ptr(self.step_dev), _lib.ptr(self.lr_dev), _lib.ptr(self.ws), self.ws.numel())

    def _model_args(self, loss):
        """The model and optimiser arguments shared by every training entry point, from params through eps, read fresh."""
        g = self.opt.param_groups[0]
        b1, b2 = g["betas"]
        return (_lib.ptr(self.model._flat), _lib.ptr(self.packed), _lib.ptr(self.state["m"]), _lib.ptr(self.state["v"]),
                _lib.ptr(loss), *self._shape, float(g["lr"]), b1, b2, g["eps"])

    def step(self, slot=0, to_host=False):
        """Enqueue one training step on the batch in slot `slot` on the current stream; returns the 0-dim loss tensor: on
        the device, or (to_host=True) the pinned host word the kernel writes -- valid once the stream has been synchronised."""
        self._sync_host_state()
        loss = (self.loss_host if to_host else self.loss)[slot:slot + 1]
        _lib.check(self._entry(*self._inputs[slot], *self._model_args(loss), *self._tail, _lib.stream_ptr(self.dev)))
        self._advance(1)
        return loss[0]

    def check_status(self):
        """Raise if a device-side wait gave up (grid barrier, MMA completion, data-parallel peer wait).  Synchronises."""
        tc = int(self.lib.b2h_tc_status())
        dp = int(self.lib.b2h_dp_status())
        if tc == 81 and not dp:
            raise _lib.B2HError("bad segment list (tc_status=81): a segment outside the streams or not of 1..max_len frames; "
                                "that step changed no parameter, moment or step counter and its loss is NaN")
        if tc or dp:
            raise _lib.B2HError(f"device-side wait timed out (tc_status={tc}, dp_status={dp}): "
                                + ("a data-parallel peer never delivered its gradients; parameter updates were suppressed "
                                   "from that step on" if tc == 51 or dp else "kernel protocol error"))

    def capture(self, n_steps=None):
        """Capture `n_steps` consecutive steps (slot i % n_slots) into one CUDA graph."""
        n_steps = n_steps or self.n_slots
        torch.cuda.synchronize(self.dev)
        self._sync_host_state()
        saved = (int(self.state["step"]), self.step_dev.clone(), self.model._flat.clone(), self.state["m"].clone(), self.state["v"].clone())
        s = torch.cuda.Stream(self.dev)
        s.wait_stream(torch.cuda.current_stream(self.dev))
        with torch.cuda.stream(s):
            for i in range(3):                       # warm-up outside capture (lazy module load, attributes)
                self.step(i % self.n_slots)
        torch.cuda.current_stream(self.dev).wait_stream(s)
        torch.cuda.synchronize(self.dev)
        g = torch.cuda.CUDAGraph()
        with torch.cuda.graph(g):
            for i in range(n_steps):
                self.step(i % self.n_slots)
        # undo the warm-up / capture bookkeeping: graphs only record, they do not execute
        self.state["step"] = self.state["dev_step_mirror"] = saved[0]
        self.step_dev.copy_(saved[1]); self.model._flat.copy_(saved[2])
        self.state["m"].copy_(saved[3]); self.state["v"].copy_(saved[4])
        self.model.mark_packed_stale(); self.packed = self.model.packed_weights()
        torch.cuda.synchronize(self.dev)
        self.graph, self._graph_steps = g, n_steps
        return g

    def replay(self):
        self._sync_host_state()
        self.graph.replay()
        self._advance(self._graph_steps)

    def finish(self):
        """Publish the step count to the optimiser's torch-layout state (for state_dict()) and surface any
        device-side timeout."""
        self.state["step_t"].fill_(float(self.host_steps))
        self.model.packed_weights(fresh_from_kernel=True)
        self.check_status()


class TrainStepRunner(_StepBuffers):
    """steps/traintest.py:94-121 for a fixed (B, T): `load(batch)` / `load_staged(buf)` copies a batch into the static
    buffers, `step()` enqueues forward+mask+loss+backward+reduce+Adam+repack (bf16 mode: ONE cooperative launch).
    The Adam step counter and the learning rate live on the device so a captured graph can be replayed."""

    def __init__(self, model: ConvModel, optimizer: FusedAdam, B: int, T: int, loss: str = "L1", n_slots: int = 1, x_dtype=None):
        self._init_buffers(model, optimizer, B, T, loss, n_slots, x_dtype)
        self._bind(self.lib.b2h_train_step, lambda batch: _dense_inputs(model, batch, loss))


class WindowTrainStepRunner(_StepBuffers):
    """TrainStepRunner over window views of device-resident frame streams (`PreprocessRightHand.training_stream`,
    `GpuPoseDataset.training_streams`): a slot holds only the step's crop list, ONE buffer
    [win_start int64 | win_end int64 | lengths int32] (20 B per window: 5 KB at B = 256 instead of a 3.54 MB batch),
    loaded from a dict {win_start, win_end, n_frames} (`GpuPoseDataset.crops`) by `load` / `host_stage` + `load_staged`.
    Steps, capture, replay and finish behave as TrainStepRunner's; the results are bit-identical to TrainStepRunner on the
    windows K0 materialises.  `streams` stay referenced by the runner (a captured graph reads them by address)."""

    def __init__(self, model: ConvModel, optimizer: FusedAdam, streams, B: int, T: int, loss: str = "L1", n_slots: int = 1,
                 pad_mode: str = "repeat_first"):
        _check_x_dtype(model, streams["input_kp"].dtype)
        self._init_common(model, optimizer, B, T, loss, n_slots, (
            ("win_start", "win_start", torch.int64, (B,)), ("win_end", "win_end", torch.int64, (B,)),
            ("lengths", "n_frames", torch.int32, (B,))))
        self._bind(self.lib.b2h_train_step_windows, lambda crops: _view_inputs(
            model, streams, crops["win_start"], T, crops["n_frames"], crops["win_end"], pad_mode, loss))
        self.win_end.fill_(streams["input_kp"].shape[0])
        self.lengths.fill_(T)


class UtteranceTrainStepRunner(_StepBuffers):
    """TrainStepRunner over SEGMENTS of device-resident frame streams, each trained as one whole sequence
    (`steps.fused_train_step_utterances`): a slot holds the step's segment list, ONE buffer [seg_start int64 | seg_end int64]
    of n_seg segments of at most max_len frames each, loaded from a dict {seg_start, seg_end} or the pair
    `GpuPoseDataset.utterance_segments` returns, by `load` / `host_stage` + `load_staged`.  Steps, capture, replay,
    `pipelined_steps` and finish behave as TrainStepRunner's; a bad segment list makes its step a no-op that
    `check_status` reports.  `streams` stay referenced by the runner (a captured graph reads them by address)."""

    def __init__(self, model: ConvModel, optimizer: FusedAdam, streams, n_seg: int, max_len: int, loss: str = "L1",
                 n_slots: int = 1):
        _check_x_dtype(model, streams["input_kp"].dtype)
        self._init_common(model, optimizer, n_seg, max_len, loss, n_slots, (
            ("seg_start", "seg_start", torch.int64, (n_seg,)), ("seg_end", "seg_end", torch.int64, (n_seg,))))
        self.ws = model.workspace(n_seg, max_len, segments=True)
        self._bind(self.lib.b2h_train_step_utterances, lambda segs: _segment_inputs(
            model, streams, segs["seg_start"], segs["seg_end"], max_len, loss))
        self._shape = self._shape[2:]               # (n_seg, max_len) travel with the segment list, not after the loss
        self.seg_end.fill_(1)                       # a valid list until the first load: segment s = frame 0

    @staticmethod
    def _as_dict(segs):
        return segs if isinstance(segs, dict) else {"seg_start": segs[0], "seg_end": segs[1]}

    def load(self, segs, slot=0, non_blocking=True):
        super().load(self._as_dict(segs), slot, non_blocking)

    def host_stage(self, segs, out=None):
        return super().host_stage(self._as_dict(segs), out)


def pipelined_steps(runner, batches, status_every=0, copy_streams=1):
    """Training loop with a double-buffered input pipeline (what a DataLoader with prefetch gives the reference loop,
    steps/traintest.py:87-123): while step i runs, batch i+1 travels host -> device on copy stream(s) into the other
    slot.  `runner` is a TrainStepRunner, WindowTrainStepRunner or parallel.DataParallelTrainer with n_slots >= 2; `batches` yields either
    `runner.host_stage(...)` buffers or reference-style batch dicts in pinned host memory.  A staged buffer can be moved as
    `copy_streams` contiguous pieces on as many streams: in isolation two halves in parallel reach 49 GB/s against
    42 GB/s for one 3.5 MB copy on B200, but inside this loop the extra per-step host calls cost more than the copy
    gains (150 -> 124 Mframes/s measured), so the default is one stream.  Yields the loss of EVERY step as a float, in
    order (the device -> host read of traintest.py:123); with the runners of this package the read of step i's loss happens
    after step i+1 has been enqueued (one step of lag), which keeps the GPU fed."""
    if runner.n_slots < 2:
        raise RuntimeError("pipelined_steps needs a runner with n_slots >= 2")
    dev = runner.dev if hasattr(runner, "dev") else runner.x.device     # (a runner without its own device attribute)
    main = torch.cuda.current_stream(dev)
    ncs = max(1, int(copy_streams))
    cstreams = [torch.cuda.Stream(dev) for _ in range(ncs)]
    ready = [[torch.cuda.Event() for _ in range(ncs)] for _ in range(2)]     # piece h of the batch landed in slot s
    freed = [torch.cuda.Event(), torch.cuda.Event()]                         # the step that read slot s has finished
    used = [False, False]
    it = iter(batches)

    def issue(i, batch):
        s = i & 1
        staged = isinstance(batch, torch.Tensor)
        k = ncs if staged else 1
        n = batch.numel() if staged else 0
        for h in range(k):
            cs = cstreams[h]
            if used[s]:
                cs.wait_event(freed[s])                  # do not overwrite a slot a step is still reading
            with torch.cuda.stream(cs):
                if staged:
                    lo, hi = n * h // k // 256 * 256, (n * (h + 1) // k // 256 * 256 if h + 1 < k else n)
                    runner.stage[s][lo:hi].copy_(batch[lo:hi], non_blocking=True)
                else:
                    runner.load(batch, slot=s)
                ready[s][h].record(cs)
        return k

    nxt = next(it, None)
    if nxt is None:
        return
    pieces = {0: issue(0, nxt)}
    to_host = hasattr(runner, "loss_host")
    done = [torch.cuda.Event(), torch.cuda.Event()]      # step on slot s finished: its loss word is in host memory
    pending = None                                       # (slot, loss tensor) of the previous step, not yet read
    i = 0
    while True:
        s = i & 1
        nxt = next(it, None)
        if nxt is not None:
            pieces[(i + 1) & 1] = issue(i + 1, nxt)      # travels while step i computes
        for h in range(pieces[s]):
            main.wait_event(ready[s][h])
        if to_host:
            # The kernel writes the loss into pinned host memory and step i's loss is READ after step i+1 has been
            # enqueued: a host that waits for step i before launching step i+1 leaves the GPU idle for the launch +
            # wake-up latency of every step (measured: 68 us per step for a 27 us kernel).  Every loss is still read,
            # in order, inside the loop; it is yielded one step late.
            loss = runner.step(s, to_host=True)
            freed[s].record(main)
            done[s].record(main)
            used[s] = True
            if pending is not None:
                done[pending[0]].synchronize()
                yield float(pending[1])
            pending = (s, loss)
        else:
            loss = runner.step(s)
            freed[s].record(main)
            used[s] = True
            yield float(loss.item())
        if status_every and (i + 1) % status_every == 0:
            runner.check_status()
        if nxt is None:
            break
        i += 1
    if pending is not None:
        done[pending[0]].synchronize()
        yield float(pending[1])


class ForwardRunner:
    """ConvModel.forward for a fixed (B, T) with static buffers (inference serving loop)."""

    def __init__(self, model: ConvModel, B: int, T: int, n_slots: int = 1, x_dtype=torch.float32, out_scale: float = 1.0):
        self.model, self.B, self.T = model, B, T
        flat = model.flat_parameters()
        dev = flat.device
        _lib.require_device(flat, "model")
        _lib.require_sm100(dev)
        self.dev = dev
        K = model.n_in // 2
        self.x = torch.zeros((n_slots, B, T, K, 2), dtype=x_dtype, device=dev)
        self.y = torch.zeros((n_slots, B, T, 21, 2), dtype=torch.float32, device=dev)
        self.n_slots = n_slots
        self.out_scale = float(out_scale)
        self.packed = model.packed_weights()
        self.lib = _lib.load()
        self.graph = None

    def run(self, slot=0):
        m = self.model
        if not torch.cuda.is_current_stream_capturing():
            self.packed = m.packed_weights()             # follows load_state_dict / optimiser updates (version compare)
        n_in, C, pe = m._geometry()
        _lib.check(self.lib.b2h_conv_forward(
            _lib.ptr(self.x[slot]), _lib.dtype_code(self.x.dtype), _lib.ptr(m._flat),
            _lib.ptr(self.packed), None, _lib.ptr(self.y[slot]), self.B, self.T, n_in, C, pe, _lib.PRECISIONS[m.precision], 0,
            self.out_scale, _lib.stream_ptr(self.dev)))
        return self.y[slot]

    def capture(self, n_runs=None):
        n_runs = n_runs or self.n_slots
        torch.cuda.synchronize(self.dev)
        s = torch.cuda.Stream(self.dev)
        s.wait_stream(torch.cuda.current_stream(self.dev))
        with torch.cuda.stream(s):
            self.run(0)
        torch.cuda.current_stream(self.dev).wait_stream(s)
        torch.cuda.synchronize(self.dev)
        g = torch.cuda.CUDAGraph()
        with torch.cuda.graph(g):
            for i in range(n_runs):
                self.run(i % self.n_slots)
        self.graph = g
        return g

    def replay(self):
        """Replay the captured graph; weights changed since capture (load_state_dict, training) are re-packed first
        (the packed buffer keeps its address, so the captured launches see them)."""
        self.packed = self.model.packed_weights()
        self.graph.replay()
