"""Training on segments (UtteranceTrainStepRunner, each segment one whole sequence) against window-view training
(WindowTrainStepRunner) on the same crops of the same seeded frame streams, bf16 mode:
  (a) 128 whole utterances of the seeded 30-600-frame mix (tools/utterances_bench.py's distribution), conv_channels 30 and
      32: the segment step (max_len 600) against window views of T = 600 frames, win_end at the utterance end, zero padding,
      lengths = the utterance lengths;
  (b) 256 random crops of at most 64 frames (GpuPoseDataset(max_frames=64, selection="randomcrop")'s draw) of the same
      mix, C = 30: the segment step (max_len 64) against window views of T = 64 (repeat-first padding, as the dataset).
Each arm starts from the same weights and is one graph-captured fused step; the arms are timed alternately with CUDA events
(median over --repeats windows of --replays replays, after warm-up).  Reports microseconds per step, real frames per
second (the frames the segments / crops hold) and the MMA rows computed per step, counted on the CPU from the plans
(b2h_train_utterances_plan + b2h_utterance_subwindows; b2h_train_subwindows for the windows), and the card's name and
power limit read in the same run.  The streams (~25k frames, a few MB) stay in L2 between steps.

    python tools/utterances_train_bench.py [--repeats 9] [--replays 50] [--out profiles/utterances_train_bench_b200.json]
"""
import argparse
import ctypes
import json
import os
import statistics
import subprocess
import sys

import numpy as np
import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import hand_pose_sl_b200 as b2h  # noqa: E402
from hand_pose_sl_b200 import _lib  # noqa: E402
from hand_pose_sl_b200.runner import UtteranceTrainStepRunner, WindowTrainStepRunner  # noqa: E402

DEV = torch.device("cuda:0")


def gpu_info():
    try:
        return subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                              capture_output=True, text=True, timeout=30).stdout.strip()
    except Exception as e:  # noqa: BLE001
        return f"unavailable ({e})"


def streams_for(lengths, seed):
    F = int(lengths.sum())
    g = torch.Generator().manual_seed(seed)
    s = {"input_kp": (torch.randn((F, 12, 2), generator=g) * 0.5).to(torch.bfloat16),
         "target_kp": torch.randn((F, 21, 2), generator=g) * 0.3, "target_conf": torch.rand((F, 21), generator=g)}
    return {k: v.to(DEV) for k, v in s.items()}


def segment_rows(m, starts, ends, max_len):
    lib = _lib.load()
    n_in, C, pe = m._geometry()
    ts = ctypes.c_int(0)
    kind = lib.b2h_train_utterances_plan(len(starts), max_len, n_in, C, pe, _lib.PRECISIONS[m.precision], ctypes.byref(ts))
    assert kind == 2, "the segment step runs on the tile kernel"
    return ts.value, sum(ts.value * lib.b2h_utterance_subwindows(int(e - s), ts.value, 0, None) for s, e in zip(starts, ends))


def window_rows(m, n_win, T):
    n_in, C, pe = m._geometry()
    n_sub = _lib.load().b2h_train_subwindows(T, n_in, C, pe, _lib.PRECISIONS[m.precision], 0, None)
    if n_sub > 1:
        return n_win * n_sub * 256
    mb = 64 if T <= 64 else 128 if T <= 128 else 256
    return n_win * mb / ((mb + 2) // (T + 2))


def make_model(C, seed):
    torch.manual_seed(seed)
    m = b2h.ConvModel(C, "ReLU", False, precision="bf16").to(DEV)
    return m, b2h.FusedAdam(m.parameters(), lr=1e-4)


def time_alternating(graphs, repeats, replays):
    """{name: graph} -> {name: (median, min, max) ms per replay}, the arms interleaved window by window."""
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    for g in graphs.values():
        for _ in range(5):
            g.replay()
    torch.cuda.synchronize()
    ms = {k: [] for k in graphs}
    for _ in range(repeats):
        for k, g in graphs.items():
            ev0.record()
            for _ in range(replays):
                g.replay()
            ev1.record()
            torch.cuda.synchronize()
            ms[k].append(ev0.elapsed_time(ev1) / replays)
    return {k: (statistics.median(v), min(v), max(v)) for k, v in ms.items()}


def compare(label, C, lengths, starts, ends, win_T, win_end, n_frames, pad_mode, max_len, streams, args):
    mu, ou = make_model(C, C)
    mw, ow = make_model(C, C)
    ru = UtteranceTrainStepRunner(mu, ou, streams, len(starts), max_len, loss="L1")
    ru.load({"seg_start": torch.from_numpy(starts), "seg_end": torch.from_numpy(ends)})
    rw = WindowTrainStepRunner(mw, ow, streams, len(starts), win_T, loss="L1", pad_mode=pad_mode)
    rw.load({"win_start": torch.from_numpy(starts), "win_end": torch.from_numpy(win_end), "n_frames": torch.from_numpy(n_frames)})
    graphs = {"segments": ru.capture(1), "window_views": rw.capture(1)}
    t = time_alternating(graphs, args.repeats, args.replays)
    ru.finish()
    rw.finish()
    frames = int((ends - starts).sum())
    Ts, rows_u = segment_rows(mu, starts, ends, max_len)
    out = []
    for arm, rows, extra in (("segments", rows_u, dict(max_len=max_len, Ts=Ts)), ("window_views", window_rows(mw, len(starts), win_T),
                                                                                  dict(T=win_T, pad_mode=pad_mode))):
        med, lo, hi = t[arm]
        r = dict(workload=label, C=C, arm=arm, n=len(starts), frames=frames, us=med * 1e3, us_min=lo * 1e3, us_max=hi * 1e3,
                 frames_per_s=frames / (med * 1e-3), mma_rows=int(rows), mma_rows_per_sequence=rows / len(starts), **extra)
        print(json.dumps(r), flush=True)
        out.append(r)
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--repeats", type=int, default=9)
    ap.add_argument("--replays", type=int, default=50)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    assert torch.cuda.is_available(), "the benchmark runs on the GPU only"
    res = {"gpu": gpu_info(), "device": torch.cuda.get_device_name(0), "results": []}
    print(res["gpu"], flush=True)
    rng = np.random.default_rng(0)
    # (a) 128 whole utterances
    L = np.clip(rng.exponential(170.0, 128) + 30, 30, 600).astype(np.int64)
    off = np.concatenate([[0], np.cumsum(L)]).astype(np.int64)
    st = streams_for(L, 1)
    for C in (30, 32):
        res["results"] += compare("128_whole_utterances", C, L, off[:-1], off[1:], 600, off[1:], L, "zeros", 600, st, args)
    # (b) 256 dataset crops of at most 64 frames
    L2 = np.clip(rng.exponential(170.0, 256) + 30, 30, 600).astype(np.int64)
    off2 = np.concatenate([[0], np.cumsum(L2)]).astype(np.int64)
    crop_start = off2[:-1] + np.array([rng.integers(0, max(int(n) - 64, 0) + 1) for n in L2], dtype=np.int64)
    crop_end = crop_start + np.minimum(L2, 64)
    st2 = streams_for(L2, 2)
    res["results"] += compare("256_crops_max_frames_64", 30, L2, crop_start, crop_end, 64, off2[1:], np.minimum(L2, 64),
                              "repeat_first", 64, st2, args)
    assert _lib.load().b2h_tc_status() == 0
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            json.dump(res, f, indent=1)
    print(json.dumps({"gpu": res["gpu"]}))


if __name__ == "__main__":
    main()
