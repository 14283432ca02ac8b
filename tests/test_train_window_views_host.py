"""CPU tier: the C-ABI of training on window views (argument checks return their codes before any launch) and the
host-side crop list of GpuPoseDataset (the same draws and lengths as `batch()`)."""
import ctypes
import random

import numpy as np
import torch

import hand_pose_sl_b200 as b2h
from hand_pose_sl_b200 import _lib, synthetic

EINVAL, ESHAPE, EALIGN = -1, -2, -3


def _codes():
    import os
    import re
    txt = open(os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "include", "b2h.h")).read()
    return {k: int(v) for k, v in re.findall(r"#define\s+(B2H_E[A-Z]+)\s+(-?\d+)", txt)}


def test_window_training_entry_points_are_bound():
    lib = ctypes.CDLL(_lib.LIB_PATH)
    for name in ("b2h_train_forward_backward_windows", "b2h_train_step_windows"):
        assert hasattr(lib, name) and name in _lib.exported_symbols()


def _bufs():
    """host buffers that stand in for device pointers: every check below fails before anything is launched"""
    keep = [np.zeros(4096, dtype=np.float32) for _ in range(8)]
    addr = [k.ctypes.data for k in keep]
    al = [a + (-a) % 16 for a in addr]          # 16-B aligned addresses inside each buffer
    return keep, al


def _call_fb(lib, frames, tgt, conf, n_frames, ws, we, pad, al, loss_kind=_lib.LOSS_L1, C=30, T=64, prec=_lib.BF16):
    v = ctypes.c_void_p
    return lib.b2h_train_forward_backward_windows(v(frames), _lib.DT_BF16, v(tgt), v(conf), n_frames, v(ws), v(we), pad,
                                                  v(al[4]), v(al[5]), v(al[6]), v(al[7]), v(al[7] + 16), None, 2, T, 24, C, 0,
                                                  loss_kind, prec, None, v(al[6]), 1 << 30, None)


def _call_step(lib, frames, tgt, conf, n_frames, ws, we, pad, al, C=30, T=64, prec=_lib.BF16):
    v = ctypes.c_void_p
    return lib.b2h_train_step_windows(v(frames), _lib.DT_BF16, v(tgt), v(conf), n_frames, v(ws), v(we), pad, v(al[4]),
                                      v(al[5]), v(al[6]), v(al[7]), v(al[7] + 64), v(al[7] + 128), 2, T, 24, C, 0, _lib.LOSS_L1,
                                      prec, 1e-3, 0.9, 0.999, 1e-8, 1, None, None, v(al[6]), 1 << 30, None)


def test_window_training_argument_checks():
    codes = _codes()
    assert (codes["B2H_EINVAL"], codes["B2H_ESHAPE"], codes["B2H_EALIGN"]) == (EINVAL, ESHAPE, EALIGN)
    lib = _lib.load()
    keep, al = _bufs()
    x, t, c, ws = al[0], al[1], al[2], al[3]
    for call in (_call_fb, _call_step):
        assert call(lib, x, t, None, 100, 0, None, _lib.PAD_REPEAT_FIRST, al) == EINVAL        # null win_start
        assert "null" in _lib.last_error()
        assert call(lib, x, 0, None, 100, ws, None, _lib.PAD_REPEAT_FIRST, al) == EINVAL       # null target_frames
        assert call(lib, x, t, None, 100, ws, None, 7, al) == EINVAL                           # bad pad_mode
        assert "pad_mode" in _lib.last_error()
        assert call(lib, x, t, None, -1, ws, None, _lib.PAD_ZEROS, al) == ESHAPE               # n_frames < 0
        assert call(lib, x + 8, t, None, 100, ws, None, _lib.PAD_ZEROS, al) == EALIGN          # frames: 16 B
        assert call(lib, x, t + 4, None, 100, ws, None, _lib.PAD_ZEROS, al) == EALIGN          # target_frames: 8 B
        # FFMA shapes are refused with the served shapes named: fp32 C = 64, fp32-ffma, bf16 16-channel fallback
        for C, T, prec in ((64, 64, _lib.FP32), (30, 64, _lib.FP32_FFMA)):
            assert call(lib, x, t, None, 100, ws, None, _lib.PAD_ZEROS, al, C=C, T=T, prec=prec) == ESHAPE
            assert "window views are trained on the tensor cores" in _lib.last_error()
    # conf_frames: 4-B alignment (its 84-B rows sit at 4 mod 16 at odd frames); confL1 without it is EINVAL
    assert _call_fb(lib, x, t, c + 2, 100, ws, None, _lib.PAD_ZEROS, al, loss_kind=_lib.LOSS_CONFL1) == EALIGN
    assert _call_fb(lib, x, t, None, 100, ws, None, _lib.PAD_ZEROS, al, loss_kind=_lib.LOSS_CONFL1) == EINVAL
    del keep


def test_views_accept_8_byte_aligned_targets_where_dense_needs_16():
    """the dense entry point keeps its 16-B rule for target; the view entry points get past the alignment checks with an
    8-B aligned target and a 4-B aligned conf stream (they stop at the shape refusal, still before any launch)"""
    lib = _lib.load()
    keep, al = _bufs()
    x, t, c, ws = al[0], al[1], al[2], al[3]
    assert _call_fb(lib, x, t + 8, c + 4, 100, ws, None, _lib.PAD_ZEROS, al, loss_kind=_lib.LOSS_CONFL1, C=64,
                    prec=_lib.FP32) == ESHAPE
    v = ctypes.c_void_p
    rc = lib.b2h_train_forward_backward(v(x), _lib.DT_BF16, v(t + 8), None, v(al[4]), v(al[5]), v(al[6]), v(al[7]),
                                        v(al[7] + 16), None, 2, 64, 24, 30, 0, _lib.LOSS_L1, _lib.BF16, None, v(al[6]), 1 << 30,
                                        None)
    assert rc == EALIGN
    del keep


def _packed(ns):
    clips = [synthetic.synthetic_clip(n, seed=40 + n) for n in ns]
    return b2h.PackedClips(pose25=np.concatenate([c[0] for c in clips]), hand_left=np.concatenate([c[1] for c in clips]),
                           hand_right=np.concatenate([c[2] for c in clips]),
                           offsets=np.cumsum([0] + [c[0].shape[0] for c in clips]).astype(np.int64),
                           n_frames_meta=np.array([c[0].shape[0] + (i % 3) for i, c in enumerate(clips)], dtype=np.int64),
                           texts=[""] * len(ns), utt_ids=list(range(len(ns))),
                           json_paths=[[None] * c[0].shape[0] for c in clips])


class _RecordK0:
    """stands in for K0 in `batch()`: records the windows it is asked to materialise"""

    def __call__(self, pose, lh, rh, win_start, T, win_end=None):
        self.win_start, self.win_end, self.T = np.asarray(win_start), np.asarray(win_end), T
        return {}


def test_dataset_crops_match_batch_draws():
    packed = _packed((40, 97, 150, 64, 300, 81, 10))
    idx = [3, 1, 4, 1, 5, 6, 2, 0, 6, 4]
    for selection in ("randomcrop", "first"):
        for T in (32, 64, 200):
            a = b2h.GpuPoseDataset(packed, T, selection=selection, device="cpu", rng=random.Random(7))
            b = b2h.GpuPoseDataset(packed, T, selection=selection, device="cpu", rng=random.Random(7))
            rec = _RecordK0()
            b.pre = rec
            for _ in range(3):
                c = a.crops(idx)
                out = b.batch(idx)
                assert rec.T == T
                assert np.array_equal(c["win_start"].numpy(), rec.win_start)
                assert np.array_equal(c["win_end"].numpy(), rec.win_end)
                assert torch.equal(c["n_frames"], out["n_frames"])
                assert c["win_start"].dtype == c["win_end"].dtype == c["n_frames"].dtype == torch.int64
