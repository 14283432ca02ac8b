"""Inference over packed utterances (ConvModel.predict_utterances) against sliding windows over the same frame stream.

bf16 mode, conv_channels 30 and 256, two workloads on one seeded bf16 frame stream each:
  (a) a 1 h clip (108 000 frames) as ONE utterance, against predict_windows with 64-frame windows at stride 64 and 16;
  (b) ~5 000 seeded utterances of 30-600 frames (mean ~200) packed into one stream.
Every call is captured in a CUDA graph and timed with CUDA events (median of --repeats windows of --replays replays, after
warm-up).  Reports microseconds per call, unique frames per second and the MMA rows computed per unique frame (from the
plans: tile kernel 64 / 128 / 256 rows per window of up to 64 / 128 / 256 frames, wide kernel 256 rows per
floor(258 / (T + 2)) windows), and the card's name and power limit read in the same run.

    python tools/utterances_bench.py [--repeats 7] [--replays 20] [--out results.json]
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

CLIP = 108_000
WIN_T = 64


def gpu_info():
    try:
        return subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                              capture_output=True, text=True, timeout=30).stdout.strip()
    except Exception as e:  # noqa: BLE001
        return f"unavailable ({e})"


def time_graph(graph, repeats, replays):
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    for _ in range(3):
        graph.replay()
    torch.cuda.synchronize()
    ms = []
    for _ in range(repeats):
        ev0.record()
        for _ in range(replays):
            graph.replay()
        ev1.record()
        torch.cuda.synchronize()
        ms.append(ev0.elapsed_time(ev1) / replays)
    return statistics.median(ms), min(ms), max(ms)


def capture(fn):
    side = torch.cuda.Stream()
    side.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(side):
        fn()
    torch.cuda.current_stream().wait_stream(side)
    torch.cuda.synchronize()
    graph = torch.cuda.CUDAGraph()
    with torch.cuda.graph(graph):
        fn()
    return graph


def rows_per_window(kind, T):
    """MMA rows one window of T frames occupies: the tile kernel's segment rows over the windows it holds, the wide
    kernel's 256-row tile over floor(258 / (T + 2))."""
    if kind == 4:
        return 256 / (258 // (T + 2))
    mb = 64 if T <= 64 else 128 if T <= 128 else 256
    return mb / ((mb + 2) // (T + 2))


def utterance_rows(m, F, lengths):
    lib = _lib.load()
    n_in, C, pe = m._geometry()
    ts = ctypes.c_int(0)
    kind = lib.b2h_utterances_plan(F, len(lengths), n_in, C, pe, _lib.PRECISIONS[m.precision], ctypes.byref(ts))
    n_sub = sum(lib.b2h_utterance_subwindows(int(L), ts.value, 0, None) for L in lengths)
    return kind, ts.value, n_sub, n_sub * rows_per_window(kind, ts.value)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--repeats", type=int, default=7)
    ap.add_argument("--replays", type=int, default=20)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    assert torch.cuda.is_available(), "the benchmark runs on the GPU only"
    dev = torch.device("cuda:0")
    res = {"gpu": gpu_info(), "device": torch.cuda.get_device_name(0), "results": []}
    print(res["gpu"], flush=True)
    rng = np.random.default_rng(0)
    mix = np.clip(rng.exponential(170.0, 5000) + 30, 30, 600).astype(np.int64)
    workloads = {"clip_1h": np.array([CLIP], dtype=np.int64), "utterances_5000": mix}
    lib = _lib.load()
    for C in (30, 256):
        torch.manual_seed(C)
        m = b2h.ConvModel(C, "ReLU", False, precision="bf16").to(dev)
        for name, lengths in workloads.items():
            F = int(lengths.sum())
            g = torch.Generator().manual_seed(C)
            x = (torch.randn(F, 12, 2, generator=g) * 0.5).to(torch.bfloat16).to(dev)
            off = torch.from_numpy(np.concatenate([[0], np.cumsum(lengths)])).to(dev)
            y = torch.empty((F, 21, 2), device=dev)
            graph = capture(lambda: m.predict_utterances(x, off, out=y))
            med, lo, hi = time_graph(graph, args.repeats, args.replays)
            assert lib.b2h_tc_status() == 0
            kind, Ts, n_sub, rows = utterance_rows(m, F, lengths)
            r = dict(C=C, workload=name, path="predict_utterances", frames=F, utterances=len(lengths), kernel=kind, Ts=Ts,
                     sub_windows=n_sub, us=med * 1e3, us_min=lo * 1e3, us_max=hi * 1e3, frames_per_s=F / (med * 1e-3),
                     mma_rows_per_frame=rows / F)
            print(json.dumps(r), flush=True)
            res["results"].append(r)
            if name != "clip_1h":
                continue
            for stride in (64, 16):
                starts = torch.from_numpy(b2h.sliding_window_starts(F, WIN_T, stride)).to(dev)
                yw = torch.empty((starts.numel(), WIN_T, 21, 2), device=dev)
                graph = capture(lambda: m.predict_windows(x, starts, WIN_T, out=yw))
                med, lo, hi = time_graph(graph, args.repeats, args.replays)
                assert lib.b2h_tc_status() == 0
                kind = lib.b2h_kernel_choice(WIN_T, 24, C, 0, _lib.PRECISIONS["bf16"], 0)
                rows = starts.numel() * rows_per_window(kind, WIN_T)
                r = dict(C=C, workload=name, path=f"predict_windows T={WIN_T} stride={stride}", frames=F,
                         windows=starts.numel(), kernel=kind, us=med * 1e3, us_min=lo * 1e3, us_max=hi * 1e3,
                         frames_per_s=F / (med * 1e-3), mma_rows_per_frame=rows / F)
                print(json.dumps(r), flush=True)
                res["results"].append(r)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            json.dump(res, f, indent=1)


if __name__ == "__main__":
    main()
