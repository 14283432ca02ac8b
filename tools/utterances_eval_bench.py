"""Validation over whole utterances (steps.validate_utterances) against what a user could run instead.

bf16 mode, conv_channels 30 and 256, on the seeded ~5 000-utterance mix of tools/utterances_bench.py (30-600 frames, one
segment per utterance, max_len 600) over one seeded stream.  Arms, every one captured in a CUDA graph:
  validate            validate_utterances(loss="L1"): planning kernel, forward with the criterion, finishing kernel;
  predict             predict_utterances alone over the same frames (the floor: the forward without the criterion);
  predict+torch       predict_utterances, then the per-segment masked L1 in torch ops (per-frame |pred - target| means,
                      segment sums by index_add_, the mean over segments): what a user can do without the new call;
  forward_backward    (C = 30 only) forward_backward_utterances on the same segments: the training path's loss.
The arms are replayed in alternation (one window of --replays replays each, --repeats rounds) and timed with CUDA events;
the table reports the median window per arm.  The losses of all arms are printed next to each other.  The card's name and
power limit are read in the same run.

    python tools/utterances_eval_bench.py [--repeats 9] [--replays 20] [--out results.json]
"""
import argparse
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

MAX_LEN = 600


def gpu_info():
    try:
        return subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                              capture_output=True, text=True, timeout=30).stdout.strip()
    except Exception as e:  # noqa: BLE001
        return f"unavailable ({e})"


def capture(fn):
    side = torch.cuda.Stream()
    side.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(side):
        fn()
    torch.cuda.current_stream().wait_stream(side)
    torch.cuda.synchronize()
    graph = torch.cuda.CUDAGraph()
    with torch.cuda.graph(graph):
        out = fn()
    return graph, out


def time_alternating(graphs, repeats, replays):
    """Median / min / max ms per replay of each graph, the graphs taking turns window by window."""
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    for g in graphs.values():
        for _ in range(3):
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


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--repeats", type=int, default=9)
    ap.add_argument("--replays", type=int, default=20)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    assert torch.cuda.is_available(), "the benchmark runs on the GPU only"
    dev = torch.device("cuda:0")
    res = {"gpu": gpu_info(), "device": torch.cuda.get_device_name(0), "results": []}
    print(res["gpu"], flush=True)
    rng = np.random.default_rng(0)
    lengths = np.clip(rng.exponential(170.0, 5000) + 30, 30, 600).astype(np.int64)      # tools/utterances_bench.py's mix
    off_np = np.concatenate([[0], np.cumsum(lengths)]).astype(np.int64)
    F, S = int(off_np[-1]), len(lengths)
    lib = _lib.load()
    for C in (30, 256):
        torch.manual_seed(C)
        m = b2h.ConvModel(C, "ReLU", False, precision="bf16").to(dev)
        g = torch.Generator().manual_seed(C)
        streams = {"input_kp": (torch.randn(F, 12, 2, generator=g) * 0.5).to(torch.bfloat16).to(dev),
                   "target_kp": (torch.randn(F, 21, 2, generator=g) * 0.3).to(dev),
                   "target_conf": torch.rand(F, 21, generator=g).to(dev)}
        off = torch.from_numpy(off_np).to(dev)
        ss, se = off[:-1].contiguous(), off[1:].contiguous()
        seg_of_frame = torch.from_numpy(np.repeat(np.arange(S), lengths)).to(dev)
        y = torch.empty((F, 21, 2), device=dev)

        def torch_criterion():
            m.predict_utterances(streams["input_kp"], off, out=y)
            per_frame = (y - streams["target_kp"]).abs().sum(dim=(1, 2))
            seg = torch.zeros(S, device=dev).index_add_(0, seg_of_frame, per_frame) / (42.0 * (se - ss).float())
            return seg.mean()

        arms = {"validate": lambda: b2h.validate_utterances(m, streams, ss, se, max_len=MAX_LEN, loss="L1"),
                "predict": lambda: m.predict_utterances(streams["input_kp"], off, out=y),
                "predict+torch": torch_criterion}
        if C <= 32:
            arms["forward_backward"] = lambda: b2h.forward_backward_utterances(m, streams, ss, se, max_len=MAX_LEN,
                                                                               loss="L1")[0]
        graphs, outs = {}, {}
        for k, fn in arms.items():
            graphs[k], outs[k] = capture(fn)
        times = time_alternating(graphs, args.repeats, args.replays)
        assert lib.b2h_tc_status() == 0
        losses = {k: float(v) for k, v in outs.items() if k != "predict"}
        for k, (med, lo, hi) in times.items():
            r = dict(C=C, workload="utterances_5000", arm=k, frames=F, segments=S, us=med * 1e3, us_min=lo * 1e3,
                     us_max=hi * 1e3, frames_per_s=F / (med * 1e-3), loss=losses.get(k))
            print(json.dumps(r), flush=True)
            res["results"].append(r)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            json.dump(res, f, indent=1)


if __name__ == "__main__":
    main()
