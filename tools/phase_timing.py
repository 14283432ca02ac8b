"""Bring-up: per-phase clock64 stamps of CTA 0 of the tensor-core tile kernels (fwd B=512, train B=256), labelled.
Steady state: the stamps are switched on BEFORE the CUDA graph is captured, so every replayed step writes them and the
buffer holds the last step of a back-to-back run.  Under torchrun (world > 1) the train step is the data-parallel one."""
import os
import sys

import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import hand_pose_sl_b200 as b2h  # noqa: E402
from hand_pose_sl_b200 import _lib, synthetic  # noqa: E402
from hand_pose_sl_b200.runner import ForwardRunner, TrainStepRunner  # noqa: E402

world = int(os.environ.get("WORLD_SIZE", "1"))
rank = int(os.environ.get("RANK", "0"))
lrank = int(os.environ.get("LOCAL_RANK", "0"))
torch.cuda.set_device(lrank)
dev = torch.device("cuda", lrank)
if world > 1:
    import torch.distributed as dist
    dist.init_process_group("nccl", device_id=dev)
lib = _lib.load()
buf = torch.zeros(1024, dtype=torch.int64, device=dev)

FWD = (["start", "pre-wait", "setup", "staging", "weights"] + [f"F{l}:{p}" for l in range(3) for p in ("issued", "ready", "epilogue")]
       + ["F3:issued", "F3:ready", "F3:target", "F3:chunk0", "F3:chunk1", "F3:epilogue"])
TRAIN = (["start", "pre-wait", "setup", "staging", "weights"] + [f"F{l}:{p}" for l in range(3) for p in ("issued", "ready", "epilogue")]
         + ["F3:issued", "F3:ready", "F3:target", "F3:chunk0", "F3:chunk1", "F3:epilogue"]
         # backward, stamped by the issuing thread: "wait" = for the epilogue handshake before dgrad / wgrad_0 (the tensor
         # pipe still works off the previous wgrad), "ready" = wgrad_0 complete, "sync" = epilogue warps done
         + ["B3:issued"] + [f"B{l}:{p}" for l in (2, 1, 0) for p in ("wait", "issued")] + ["B0:ready", "B:sync"]
         + ["readout", "barrier", "gather"])
TAIL1 = ["adam", "end"]
TAILDP = ["pushed", "collected", "adam", "end"]


def marks(name):
    """per-CTA %globaltimer marks of the fused train kernel: launch skew vs barrier wait"""
    m = buf.cpu()[128:128 + 4 * 192].view(192, 4)
    m = m[m[:, 0] != 0]
    if m.numel() == 0:
        return
    t0 = int(m[:, 0].min())
    start, arrive, passed, end = [(m[:, i] - t0).tolist() for i in range(4)]
    srt = sorted(start)
    print(f"[r{rank}] {name}: {len(start)} CTAs; start spread {max(start)} ns (median {srt[len(srt) // 2]}), "
          f"arrive min/median/max {min(arrive)}/{sorted(arrive)[len(arrive) // 2]}/{max(arrive)} ns, "
          f"pass min/max {min(passed)}/{max(passed)}, end min/max {min(end)}/{max(end)}; "
          f"own work (arrive-start) min/median/max {min(a - b for a, b in zip(arrive, start))}/"
          f"{sorted(a - b for a, b in zip(arrive, start))[len(start) // 2]}/{max(a - b for a, b in zip(arrive, start))}", flush=True)


def show(name, labels):
    marks(name)
    st = [int(v) for v in buf.cpu()[:128].tolist() if v != 0]
    d = [st[i + 1] - st[i] for i in range(len(st) - 1)]
    lab = labels[1:len(st)] + ["?"] * max(0, len(st) - len(labels))
    print(f"[r{rank}] {name}: {len(st)} stamps, total {st[-1] - st[0]} cycles")
    print("   " + "  ".join(f"{a}={b}" for a, b in zip(lab, d)), flush=True)


torch.manual_seed(0)
m = b2h.ConvModel(30, "ReLU", False, precision="bf16").to(dev)
opt = b2h.FusedAdam(m.parameters(), lr=2e-4)
if world > 1:
    from hand_pose_sl_b200.parallel import DataParallelTrainer
    tr = DataParallelTrainer(m, opt, 256, 64, "L1", n_slots=8, multicast=os.environ.get("B2H_MULTICAST", "1") == "1")
    print(f"[r{rank}] exchange={tr.exchange} multicast={bool(tr.mc_ptr)}", flush=True)
else:
    tr = TrainStepRunner(m, opt, 256, 64, n_slots=8)
for s in range(8):
    tr.load(synthetic.model_batch(256, 64, seed=1234 + 100 * rank + s), slot=s, non_blocking=False)
labels = TRAIN + (TAILDP if world > 1 and tr.exchange == "p2p" else TAIL1)

for _ in range(3):
    tr.step(0)
torch.cuda.synchronize()
buf.zero_(); lib.b2h_debug_timing(_lib.ptr(buf))
tr.step(0); torch.cuda.synchronize()
show("train, single step after a sync", labels)
buf.zero_()
tr.capture(8)                      # stamps stay on: captured launches carry the buffer pointer
for rep in range(3):
    for _ in range(6):
        tr.replay()
    torch.cuda.synchronize()
    show(f"train, steady state (graph replay, rep {rep})", labels)
ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
ev0.record()
for _ in range(25):
    tr.replay()
ev1.record(); torch.cuda.synchronize()
print(f"[r{rank}] train: {ev0.elapsed_time(ev1) / 200 * 1e3:.2f} us/step (graph, stamps on)", flush=True)
lib.b2h_debug_timing(None)
tr.finish()

if world == 1:
    fr = ForwardRunner(m, 512, 64, x_dtype=torch.bfloat16)
    fr.x[0].copy_(synthetic.model_batch(512, 64, seed=99)["input_kp"])
    for _ in range(3):
        fr.run(0)
    torch.cuda.synchronize()
    buf.zero_(); lib.b2h_debug_timing(_lib.ptr(buf))
    fr.run(0); torch.cuda.synchronize()
    lib.b2h_debug_timing(None)
    show("fwd, single launch", FWD + ["end"])
if world > 1:
    dist.barrier()
    sys.stdout.flush()
    os._exit(0)
