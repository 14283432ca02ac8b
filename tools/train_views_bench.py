"""Training from device-resident frame streams vs materialised batches (DESIGN §4, §5).

1. 256 x 64, C = 30, bf16, L1, graph-replayed steps: 40 rotating resident dense batches (> L2, as bench.py) vs
   WindowTrainStepRunner crops into an 8 h stream (> L2), random starts, about half of them odd; and, for reference, the
   K0-per-step pipeline (GpuPoseDataset.batch + TrainStepRunner.load + step, eager).
2. The same comparison at C = 256 (wide kernels).
3. End to end: pipelined_steps over pinned host-staged 3.54 MB batches vs 5 KB crop buffers, median of five 400-step
   segments.
Each compared pair starts from the same weights, runs the same crops, and is asserted bit-identical after its steps.
Prints one JSON object (and writes it to --out when given) with the card's name and power limit read in the same run."""
import argparse
import json
import os
import random
import statistics
import subprocess
import sys
import time

import numpy as np
import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import hand_pose_sl_b200 as b2h  # noqa: E402
from hand_pose_sl_b200 import synthetic  # noqa: E402
from hand_pose_sl_b200.runner import TrainStepRunner, WindowTrainStepRunner, pipelined_steps  # noqa: E402

DEV = torch.device("cuda:0")
B, T, N_ROT = 256, 64, 40


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader", "-i", "0"],
                       capture_output=True, text=True).stdout.strip()
    return q or torch.cuda.get_device_name(0)


def timed_replays(runner, reps):
    ev = [torch.cuda.Event(enable_timing=True) for _ in range(2)]
    runner.replay()
    torch.cuda.synchronize()
    ev[0].record()
    for _ in range(reps):
        runner.replay()
    ev[1].record()
    torch.cuda.synchronize()
    return ev[0].elapsed_time(ev[1]) * 1e3 / (reps * runner._graph_steps)      # us per step


def make_model(C, seed=0):
    torch.manual_seed(seed)
    m = b2h.ConvModel(C, "ReLU", False, precision="bf16").to(DEV)
    return m, b2h.FusedAdam(m.parameters(), lr=1e-4)


def draw_crops(F, rng, n):
    out = []
    for _ in range(n):
        odd = rng.random(B) < 0.5                        # about half of the starts odd (8 B off a 16-B target row)
        s = (rng.integers(0, F - T, size=B) & ~1) | odd
        out.append({"win_start": torch.from_numpy(s.astype(np.int64)),
                    "win_end": torch.full((B,), F, dtype=torch.int64),
                    "n_frames": torch.from_numpy(rng.integers(T // 2, T + 1, size=B).astype(np.int64))})
    return out


def dense_of(pre, clip, c):
    mat = pre(*clip, c["win_start"].numpy(), T, win_end=c["win_end"].numpy())
    return {"input_kp": mat["input_kp_bf16"], "target_kp": mat["target_kp"], "n_frames": c["n_frames"]}


def compare_step(C, pre, clip, streams, crops, reps, ds=None):
    F = streams["input_kp"].shape[0]
    md, od = make_model(C)
    mv, ov = make_model(C)
    dense = TrainStepRunner(md, od, B, T, n_slots=N_ROT, x_dtype=torch.bfloat16)
    view = WindowTrainStepRunner(mv, ov, streams, B, T, n_slots=N_ROT)
    for k, c in enumerate(crops):
        dense.load(dense_of(pre, clip, c), slot=k)
        view.load(c, slot=k)
    dense.capture(N_ROT)
    view.capture(N_ROT)
    res = {"C": C, "B": B, "T": T, "stream_frames": F, "stream_MB": round(sum(v.numel() * v.element_size() for v in streams.values()) / 1e6, 1),
           "dense_batches_MB": round(N_ROT * dense.slot_bytes / 1e6, 1)}
    us_d, us_v = [], []
    for _ in range(3):                                   # alternate the two, three rounds
        us_d.append(timed_replays(dense, reps))
        us_v.append(timed_replays(view, reps))
    dense.finish(); view.finish()
    torch.cuda.synchronize()
    assert torch.equal(md.flat_parameters(), mv.flat_parameters()), "views and dense batches diverged"
    assert torch.equal(od._flat_state[0]["m"], ov._flat_state[0]["m"]) and torch.equal(od._flat_state[0]["v"], ov._flat_state[0]["v"])
    res["dense_us_per_step"] = [round(x, 2) for x in us_d]
    res["views_us_per_step"] = [round(x, 2) for x in us_v]
    res["bit_identical_after_steps"] = 3 * (reps + 1) * N_ROT
    if ds is not None:                                   # K0 per step: GpuPoseDataset.batch + load + step, eager
        mk, ok = make_model(C)
        r = TrainStepRunner(mk, ok, B, T, n_slots=1, x_dtype=None)
        idx = np.arange(B) % len(ds)
        for _ in range(5):
            r.load(ds.batch(idx)); r.step(0)
        torch.cuda.synchronize()
        n = 200
        t0 = time.perf_counter()
        for _ in range(n):
            r.load(ds.batch(idx)); r.step(0)
        torch.cuda.synchronize()
        res["k0_per_step_us_per_step"] = round((time.perf_counter() - t0) * 1e6 / n, 2)
        r.finish()
    return res


def e2e(C, pre, clip, streams, crops, seg, nseg):
    out = {}
    losses = {}
    for name in ("staged_batches", "crop_buffers"):
        m, o = make_model(C)
        if name == "staged_batches":
            r = TrainStepRunner(m, o, B, T, n_slots=2, x_dtype=torch.bfloat16)
            bufs = [r.host_stage({k: (v.cpu() if torch.is_tensor(v) else v) for k, v in dense_of(pre, clip, c).items()}) for c in crops]
        else:
            r = WindowTrainStepRunner(m, o, streams, B, T, n_slots=2)
            bufs = [r.host_stage(c) for c in crops]
        list(pipelined_steps(r, [bufs[i % len(bufs)] for i in range(50)]))        # warm-up
        times, seq = [], []
        for _ in range(nseg):
            feed = [bufs[i % len(bufs)] for i in range(seg)]
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            seq.extend(pipelined_steps(r, feed))
            torch.cuda.synchronize()
            times.append((time.perf_counter() - t0) * 1e6 / seg)
        r.finish()
        losses[name] = seq
        us = statistics.median(times)
        out[name] = {"us_per_step_median": round(us, 2), "segments_us": [round(x, 2) for x in times],
                     "Mframes_per_s": round(B * T / us, 1), "bytes_per_step": int(bufs[0].numel())}
    assert losses["staged_batches"] == losses["crop_buffers"], "end-to-end loss sequences differ"
    out["identical_loss_sequence_steps"] = len(losses["crop_buffers"])
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--hours", type=float, default=8.0)
    ap.add_argument("--fps", type=float, default=30.0)
    ap.add_argument("--reps", type=int, default=10)
    ap.add_argument("--seg", type=int, default=400)
    ap.add_argument("--out", help="also write the JSON object to this file")
    a = ap.parse_args()
    F = int(a.hours * 3600 * a.fps)
    pose, lh, rh = synthetic.synthetic_clip(F, seed=3)
    utt = 300                                            # the K0-per-step reference draws 64-frame crops of 300-frame clips
    off = np.arange(0, F + 1, utt, dtype=np.int64)
    n_utt = len(off) - 1
    packed = b2h.PackedClips(pose25=pose, hand_left=lh, hand_right=rh, offsets=off, n_frames_meta=np.full(n_utt, utt),
                             texts=[""] * n_utt, utt_ids=list(range(n_utt)), json_paths=[[None] * utt] * n_utt)
    ds = b2h.GpuPoseDataset(packed, T, selection="randomcrop", device=DEV, rng=random.Random(0))
    clip = (ds.pose, ds.lh, ds.rh)
    pre = b2h.PreprocessRightHand(emit_bf16=True)
    streams = pre.training_stream(*clip)
    crops = draw_crops(F, np.random.default_rng(0), N_ROT)
    res = {"card": card(), "torch": torch.__version__}
    res["c30"] = compare_step(30, pre, clip, streams, crops, a.reps, ds=ds)
    res["c256"] = compare_step(256, pre, clip, streams, crops, max(1, a.reps // 4))
    res["e2e_c30"] = e2e(30, pre, clip, streams, crops, a.seg, 5)
    res["card_after"] = card()
    s = json.dumps(res)
    print(s)
    if a.out:
        os.makedirs(os.path.dirname(a.out) or ".", exist_ok=True)
        with open(a.out, "w") as f:
            f.write(s + "\n")


if __name__ == "__main__":
    main()
