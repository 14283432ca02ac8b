"""K0 only.  `k0_prof.py F reps`: `reps` launches of the preprocessing kernel on an F-frame clip (ncu target).
`k0_prof.py time F1 F2 ...`: CUDA-graph replay timing per clip length, measured like bench.py's `preprocess` section."""
import os
import sys

import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import hand_pose_sl_b200 as b2h
from hand_pose_sl_b200 import synthetic

dev = torch.device("cuda:0")
pre = b2h.PreprocessRightHand()
starts = torch.zeros(1, dtype=torch.int64, device=dev)


def clip(F):
    pose, lh, rh = synthetic.synthetic_clip(F, seed=1234)
    return tuple(torch.from_numpy(a).to(dev) for a in (pose, lh, rh))


if sys.argv[1:2] == ["time"]:
    for F in (int(a) for a in sys.argv[2:]):
        tp, tl, tr = clip(F)
        out = pre(tp, tl, tr, starts, F)
        for _ in range(3):
            pre(tp, tl, tr, starts, F, out=out)
        torch.cuda.synchronize()
        g = torch.cuda.CUDAGraph()
        with torch.cuda.graph(g):
            for _ in range(4):
                pre(tp, tl, tr, starts, F, out=out)
        g.replay()
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(10):
            g.replay()
        e1.record()
        torch.cuda.synchronize()
        us = e0.elapsed_time(e1) / 40 * 1e3
        print(f"K0 {F} frames: {us:.2f} us/launch (graph replay), {F * 1452 / us / 1e6:.3f} TB/s")
        del tp, tl, tr, out, g
else:
    F = int(sys.argv[1]) if len(sys.argv) > 1 else 108000
    reps = int(sys.argv[2]) if len(sys.argv) > 2 else 3
    tp, tl, tr = clip(F)
    for _ in range(reps):
        pre(tp, tl, tr, starts, F)
    torch.cuda.synchronize()
print("k0_prof done")
