"""Data-parallel training (SURVEY.md §8e).  The reference is single-process; windows are independent
units (per-sample zero padding, no cross-sample op: HandPoseModels.py:55-58), so training shards by
batch with ONE gradient all-reduce per step over the flat fp32 gradient buffer (76 KB at C=30) and
inference / preprocessing shard with no collective at all.

Combine rule: maskedPoseL1 divides by the local batch size (steps/utils.py:428), so with equal
per-rank batches  global_grad = (1/W) * sum_r grad_r;  poderatedPoseL1 sums over the batch
(steps/utils.py:452), so  global_grad = sum_r grad_r."""
from __future__ import annotations

import torch
import torch.distributed as dist

from . import _lib
from .models import ConvModel
from .runner import _StepBuffers
from .steps import FusedAdam, _dense_inputs


def shard_range(n_items: int, rank: int, world: int):
    """Contiguous block partition in rank order (rank r gets items [lo, hi))."""
    per, rem = divmod(n_items, world)
    lo = rank * per + min(rank, rem)
    return lo, lo + per + (1 if rank < rem else 0)


def shard_batch(batch: dict, rank: int, world: int):
    """Rank r's slice of a reference-style batch dict (tensors indexed on dim 0, lists sliced)."""
    B = batch["input_kp"].shape[0]
    if B % world != 0:
        raise RuntimeError(f"global batch {B} is not divisible by world size {world}: the loss combine rule "
                           "(mean of per-rank means) needs equal per-rank batches")
    lo, hi = shard_range(B, rank, world)
    return {k: (v[lo:hi] if hasattr(v, "__getitem__") else v) for k, v in batch.items()}


def grad_scale_for(loss: str, world: int) -> float:
    return 1.0 / world if loss == "L1" else 1.0


def allreduce_flat(flat_grads: torch.Tensor, group=None):
    """The one collective of a training step: SUM over ranks of the flat gradient buffer, in place."""
    if dist.is_available() and dist.is_initialized() and dist.get_world_size(group) > 1:
        dist.all_reduce(flat_grads, op=dist.ReduceOp.SUM, group=group)
    return flat_grads


def combine_losses(loss: torch.Tensor, kind: str, group=None):
    """Logging only: the global loss value from per-rank losses."""
    if dist.is_available() and dist.is_initialized() and dist.get_world_size(group) > 1:
        out = loss.detach().clone()
        dist.all_reduce(out, op=dist.ReduceOp.SUM, group=group)
        return out / dist.get_world_size(group) if kind == "L1" else out
    return loss


def broadcast_parameters(model: ConvModel, src: int = 0, group=None):
    """Identical replicas: rank `src`'s flat parameter buffer to every rank."""
    if dist.is_available() and dist.is_initialized() and dist.get_world_size(group) > 1:
        flat = model.flat_parameters()
        dist.broadcast(flat, src=src, group=group)
        model.mark_packed_stale()


def _symmetric_exchange_buffer(n_floats: int, device, group, fill: int = 0):
    """Peer-mapped exchange buffer on every rank (torch symmetric memory: cuMem allocations mapped into every peer over
    NVLink, plus -- when the fabric supports it -- one multicast (NVLS) address that reaches all of them).  Returns
    (local tensor, handle, device array of peer base pointers indexed by rank, multicast address or 0)."""
    import torch.distributed._symmetric_memory as symm_mem
    world = dist.get_world_size(group)
    buf = symm_mem.empty(n_floats, dtype=torch.float32, device=device)
    buf.view(torch.int32).fill_(fill - (1 << 32) if fill >= (1 << 31) else fill)     # b2h_dp_exchange_fill: sentinel or zero
    hdl = symm_mem.rendezvous(buf, group if group is not None else dist.group.WORLD)
    ptrs = [int(p) for p in hdl.buffer_ptrs]
    if len(ptrs) != world or hdl.rank != dist.get_rank(group):
        raise RuntimeError("symmetric memory rendezvous returned an unexpected peer table")
    mc = 0
    try:
        mc = int(getattr(hdl, "multicast_ptr", 0) or 0)
    except Exception:  # noqa: BLE001
        mc = 0
    torch.cuda.synchronize(device)
    dist.barrier(group)                                   # every rank's buffer is zeroed before anyone signals
    return buf, hdl, torch.tensor(ptrs, dtype=torch.int64, device=device), mc


class DataParallelTrainer(_StepBuffers):
    """One process per GPU.  exchange="p2p" (default when symmetric memory is available): step() = ONE cooperative
    launch per rank in bf16 mode -- forward+mask+loss+backward, cross-CTA reduction, push of the reduced gradient
    words into every peer's exchange buffer over NVLink (one multimem.st per slot through the NVSwitch when a multicast
    mapping exists, `multicast=True`), sum in rank order, Adam + re-pack; no NCCL call on the step path.
    exchange="nccl": ... -> dist.all_reduce(flat grads) -> Adam kernel (baseline).
    Static buffers; the whole step can be captured in a CUDA graph either way.  A peer that never delivers is a
    device-side timeout: parameter updates stop and `finish()` / `check_status()` raise."""

    def __init__(self, model: ConvModel, optimizer: FusedAdam, B: int, T: int, loss: str = "L1", group=None,
                 n_slots: int = 1, exchange: str = "auto", x_dtype=None, multicast: bool = True):
        self.group = group
        self.world = dist.get_world_size(group) if dist.is_initialized() else 1
        broadcast_parameters(model, 0, group)
        self._init_buffers(model, optimizer, B, T, loss, n_slots, x_dtype)
        dev = self.dev
        self.grads = torch.zeros_like(model.flat_parameters())
        if exchange not in ("auto", "p2p", "nccl"):
            raise ValueError("exchange must be 'auto', 'p2p' or 'nccl'")
        self.exchange = "nccl"
        self.sym = self.sym_hdl = self.peer_ptrs = None
        self.mc_ptr = 0
        self.peers_seen = self.world
        if self.world > 1 and exchange in ("auto", "p2p"):
            try:
                n_in_, C_, pe_ = model._geometry()
                nfl = int(self.lib.b2h_dp_exchange_floats(n_in_, C_, pe_, self.world))
                fill = int(self.lib.b2h_dp_exchange_fill(T, n_in_, C_, pe_, _lib.PRECISIONS[model.precision]))
                self.sym, self.sym_hdl, self.peer_ptrs, mc = _symmetric_exchange_buffer(nfl, dev, group, fill)
                self.mc_ptr = mc if multicast else 0
                self.peers_seen = int(self.peer_ptrs.numel())
                self.epoch_dev = torch.zeros((1,), dtype=torch.int64, device=dev)
                self.rank = dist.get_rank(group)
                self.exchange = "p2p"
            except Exception as e:  # noqa: BLE001  (no peer access / symmetric memory unavailable)
                if exchange == "p2p":
                    raise
                import warnings
                warnings.warn(f"symmetric-memory gradient exchange unavailable ({type(e).__name__}: {e}); using NCCL all-reduce")
        tail = None                # exchange="nccl": step() below runs forward_backward + all-reduce + the Adam kernel
        if self.exchange == "p2p":  # b2h_train_step_dp's arguments after eps
            tail = (_lib.ptr(self.step_dev), _lib.ptr(self.epoch_dev), _lib.ptr(self.lr_dev), _lib.ptr(self.sym),
                    _lib.ptr(self.peer_ptrs), (self.mc_ptr or None), self.rank, self.world,
                    grad_scale_for(self.loss_name, self.world), _lib.ptr(self.ws), self.ws.numel())
        self._bind(self.lib.b2h_train_step_dp, lambda batch: _dense_inputs(model, batch, loss), tail)

    def step(self, slot=0, to_host=False):
        if self.exchange == "p2p":
            return super().step(slot, to_host)
        self._sync_host_state()
        m, g = self.model, self.opt.param_groups[0]
        n_in, C, pe = m._geometry()
        b1, b2 = g["betas"]
        sp = _lib.stream_ptr(self.dev)
        loss = (self.loss_host if to_host else self.loss)[slot:slot + 1]
        _lib.check(self.lib.b2h_train_forward_backward(
            *self._inputs[slot], _lib.ptr(m._flat), _lib.ptr(self.packed), _lib.ptr(self.grads), _lib.ptr(loss), None,
            *self._shape, _lib.ptr(self.step_dev), _lib.ptr(self.ws), self.ws.numel(), sp))
        allreduce_flat(self.grads, self.group)
        _lib.check(self.lib.b2h_adam_step(
            _lib.ptr(m._flat), _lib.ptr(self.grads), _lib.ptr(self.state["m"]), _lib.ptr(self.state["v"]), m._flat.numel(),
            float(g["lr"]), b1, b2, g["eps"], 0, _lib.ptr(self.step_dev), _lib.ptr(self.lr_dev),
            grad_scale_for(self.loss_name, self.world), _lib.ptr(self.packed), n_in, C, pe, sp))
        self._advance(1)
        return loss[0]

    def replica_checksum(self):
        """(sum, sum of squares) of the flat parameters in float64 -- equal on every rank iff the replicas are
        bit-identical for all practical purposes; `replicas_identical()` all-gathers and compares the raw bits."""
        flat = self.model.flat_parameters().double()
        return torch.stack([flat.sum(), (flat * flat).sum()])

    def replicas_identical(self):
        flat = self.model.flat_parameters()
        if self.world == 1:
            return True
        gathered = [torch.empty_like(flat) for _ in range(self.world)]
        dist.all_gather(gathered, flat.contiguous(), group=self.group)
        return all(torch.equal(gathered[0], t) for t in gathered[1:])
