"""Streaming inference on a 1 h clip for wide models and long windows: window views vs materialised windows.

For each (conv_channels, T, stride) it times two CUDA-graph-replayed pipelines over the same clip with CUDA events
(median of --repeats timed windows of --replays replays each, after warm-up):
  (a) views:        PreprocessRightHand.frame_stream (one bf16 row per unique frame) + ConvModel.predict_windows
  (b) materialised: PreprocessRightHand(emit_bf16=True) writing the (W, T) windows + ConvModel.predict on them
asserts that both produce bit-identical predictions, and prints the bytes each pipeline moves (computed from the shapes).

    python tools/stream_views_bench.py [--frames 108000] [--repeats 7] [--replays 10] [--out results.json]
"""
import argparse
import json
import os
import statistics
import subprocess
import sys

import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import hand_pose_sl_b200 as b2h  # noqa: E402
from hand_pose_sl_b200 import synthetic  # noqa: E402

SHAPES = [(128, 64, 16), (256, 64, 16), (256, 64, 64), (256, 126, 40), (30, 512, 128)]
RAW = 25 * 3 * 4 + 2 * 21 * 3 * 4        # raw OpenPose bytes of one frame (pose25 + both hands)
K0_SLOT = 12 * 2 * 4 + 12 * 4 + 21 * 2 * 4 + 21 * 4 + 12 * 2 * 2   # input_kp, input_conf, target_kp, target_conf, bf16 copy
IN_ROW = 12 * 2 * 2                      # one bf16 network-input row
OUT_ROW = 42 * 4                         # one fp32 prediction row


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
    g = torch.cuda.CUDAGraph()
    with torch.cuda.graph(g):
        fn()
    return g


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--frames", type=int, default=108000)
    ap.add_argument("--repeats", type=int, default=7)
    ap.add_argument("--replays", type=int, default=10)
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    if not torch.cuda.is_available():
        sys.exit("stream_views_bench.py needs a GPU")
    dev = torch.device("cuda:0")
    F = a.frames
    pose, lh, rh = (torch.from_numpy(x).to(dev) for x in synthetic.synthetic_clip(F, seed=7))
    stream_bytes = F * IN_ROW
    print(f"GPU: {gpu_info()}")
    print(f"clip: {F} frames; bf16 frame stream {stream_bytes / 1e6:.1f} MB (fits the 126 MB L2: the views re-read it from L2)")
    results = []
    for C, T, stride in SHAPES:
        torch.manual_seed(C)
        m = b2h.ConvModel(C, "ReLU", False, precision="bf16").to(dev)
        starts = torch.from_numpy(b2h.sliding_window_starts(F, T, stride)).to(dev)
        W = starts.numel()
        pre_v = b2h.PreprocessRightHand()
        s = torch.empty((F, 12, 2), dtype=torch.bfloat16, device=dev)
        ya = torch.empty((W, T, 21, 2), dtype=torch.float32, device=dev)

        def views():
            pre_v.frame_stream(pose, lh, rh, out=s)
            m.predict_windows(s, starts, T, denormalize=1280.0, out=ya)

        pre_m = b2h.PreprocessRightHand(with_left_hand=False, emit_bf16=True)
        mat = pre_m(pose, lh, rh, starts, T)
        yb = {}

        def materialised():
            pre_m(pose, lh, rh, starts, T, out=mat)
            yb["y"] = m.predict(mat["input_kp_bf16"], denormalize=1280.0)

        ga, gb = capture(views), capture(materialised)
        ga.replay(); gb.replay()
        torch.cuda.synchronize()
        identical = torch.equal(ya, yb["y"])
        assert identical, f"views != materialised windows for C={C} T={T} stride={stride}"
        # alternate the two pipelines so that both see the same clock / neighbour conditions
        ta, tb = [], []
        for _ in range(2):
            ta.append(time_graph(ga, a.repeats, a.replays))
            tb.append(time_graph(gb, a.repeats, a.replays))
        ms_a = statistics.median([t[0] for t in ta])
        ms_b = statistics.median([t[0] for t in tb])
        bytes_a = F * (RAW + IN_ROW) + W * T * (IN_ROW + OUT_ROW)           # K0 over unique frames; views read rows (L2)
        bytes_b = W * T * (RAW + K0_SLOT) + W * T * (IN_ROW + OUT_ROW)      # K0 per window slot; forward reads its bf16 copy
        r = {"C": C, "T": T, "stride": stride, "windows": W, "identical": identical,
             "views_ms": ms_a, "materialised_ms": ms_b, "speedup": ms_b / ms_a,
             "views_spread_ms": [min(t[1] for t in ta), max(t[2] for t in ta)],
             "materialised_spread_ms": [min(t[1] for t in tb), max(t[2] for t in tb)],
             "views_bytes": bytes_a, "materialised_bytes": bytes_b,
             "materialised_window_buffer_bytes": W * T * K0_SLOT}
        results.append(r)
        print(f"C={C:3d} T={T:4d} stride={stride:3d} W={W:6d}: views {ms_a:8.3f} ms ({bytes_a / 1e6:7.1f} MB), "
              f"materialised {ms_b:8.3f} ms ({bytes_b / 1e6:7.1f} MB), x{ms_b / ms_a:.3f}, outputs bit-identical")
        del ga, gb, mat, yb
        torch.cuda.empty_cache()
    out = {"gpu": gpu_info(), "frames": F, "stream_bytes": stream_bytes, "stream_l2_resident": stream_bytes < 126e6, "results": results}
    if a.out:
        with open(a.out, "w") as f:
            json.dump(out, f, indent=1)
    print(json.dumps(out))


if __name__ == "__main__":
    main()
