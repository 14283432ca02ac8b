"""GPU tier: training on window views of device-resident frame streams.  Every case first pins the kernel it exists to
reach, then requires the result over views of `PreprocessRightHand.training_stream` to equal, bit for bit, the same call
on the windows K0 materialises: loss, gradients and masked prediction, five Adam steps (params, m, v, packed bytes, each
loss), the window runner (eager, graph-captured, pipelined) and the dataset's crop path."""
import numpy as np
import pytest
import torch

import hand_pose_sl_b200 as b2h
from hand_pose_sl_b200 import _lib, synthetic
from hand_pose_sl_b200.runner import TrainStepRunner, WindowTrainStepRunner, pipelined_steps

pytestmark = pytest.mark.gpu
DEV = "cuda:0"
NONE, FFMA, TILE, WIDE_TRAIN = 0, 1, 2, 5


def _tc_clean():
    torch.cuda.synchronize()
    assert _lib.load().b2h_tc_status() == 0, "tensor-core kernel hit a wait timeout"


def _model(C, prec="bf16", seed=0, **kw):
    torch.manual_seed(seed)
    return b2h.ConvModel(C, "ReLU", kw.pop("pos_emb", False), precision=prec, **kw).to(DEV)


def _choice(m, T):
    n_in, C, pe = m._geometry()
    return _lib.load().b2h_kernel_choice(T, n_in, C, pe, _lib.PRECISIONS[m.precision], 1)


def _n_sub(m, T):
    n_in, C, pe = m._geometry()
    return _lib.load().b2h_train_subwindows(T, n_in, C, pe, _lib.PRECISIONS[m.precision], 0, None)


_CLIPS = {}


def _clip(F, pad_mode="repeat_first"):
    """(clip tensors, K0, bf16 streams, fp32 streams) of a seeded synthetic clip"""
    key = (F, pad_mode)
    if key not in _CLIPS:
        t = tuple(torch.from_numpy(a).to(DEV) for a in synthetic.synthetic_clip(F, seed=5))
        pre = b2h.PreprocessRightHand(emit_bf16=True, pad_mode=pad_mode)
        _CLIPS[key] = (t, pre, pre.training_stream(*t), pre.training_stream(*t, dtype=torch.float32))
    return _CLIPS[key]


def _windows(F, T, n, seed):
    """start 0, odd starts, starts whose crop runs past the clip, win_end cuts mid-window, ragged lengths (some reaching
    into pad rows)"""
    rng = np.random.default_rng(seed)
    starts = rng.integers(0, max(F - T, 1), size=n)
    starts[0] = 0
    starts[1::4] |= 1
    starts[2::7] = F - T // 3 - rng.integers(0, 3, size=starts[2::7].size)
    ends = np.full(n, F, dtype=np.int64)
    ends[3::5] = np.minimum(starts[3::5] + rng.integers(1, T, size=starts[3::5].size), F)
    lengths = rng.integers(1, T + 1, size=n)
    lengths[::3] = T
    return starts.astype(np.int64), ends, torch.from_numpy(lengths.astype(np.int64))


def _mat(pre, t, starts, T, ends):
    return pre(*t, starts, T, win_end=ends)


def _check_fb(m, streams_list, mat, starts, T, ends, lengths, pad_mode="repeat_first"):
    for loss in ("L1", "confL1"):
        for streams in streams_list:
            xm = mat["input_kp_bf16"] if streams["input_kp"].dtype == torch.bfloat16 else mat["input_kp"]
            batch = {"input_kp": xm, "target_kp": mat["target_kp"], "target_conf": mat["target_conf"], "n_frames": lengths}
            lv, gv, pv = b2h.forward_backward_windows(m, streams, starts, T, lengths, win_end=ends, pad_mode=pad_mode,
                                                      loss=loss, want_pred=True)
            _tc_clean()
            ld, gd, pd = b2h.forward_backward(m, batch, loss=loss, want_pred=True)
            _tc_clean()
            assert torch.equal(lv, ld), (loss, float(lv), float(ld))
            assert torch.equal(gv, gd), loss
            assert torch.equal(pv, pd), loss


@pytest.mark.parametrize("prec,C,T,n", [("bf16", 30, 37, 41), ("bf16", 30, 64, 300), ("bf16", 30, 200, 23),
                                        ("fp32", 30, 64, 29), ("fp32", 30, 128, 17),
                                        ("bf16", 30, 300, 9), ("bf16", 30, 1000, 5), ("fp32", 30, 200, 11),
                                        ("bf16", 64, 64, 450), ("bf16", 80, 33, 37), ("bf16", 256, 126, 13)])
def test_forward_backward_windows_equal_materialised(prec, C, T, n):
    m = _model(C, prec)
    want = TILE if C <= 32 else WIDE_TRAIN
    assert _choice(m, T) == want
    sub = T > (128 if prec == "fp32" else 256)
    assert (_n_sub(m, T) > 1) == sub
    F = 3000
    t, pre, s16, s32 = _clip(F)
    starts, ends, lengths = _windows(F, T, n, seed=C * 1000 + T)
    _check_fb(m, (s16, s32) if prec == "bf16" else (s32,), _mat(pre, t, starts, T, ends), starts, T, ends, lengths)


def test_pos_emb_windows():
    m = _model(30, pos_emb=True)
    assert _choice(m, 100) == TILE
    F = 900
    t, pre, s16, s32 = _clip(F)
    starts, ends, lengths = _windows(F, 100, 21, seed=3)
    _check_fb(m, (s16, s32), _mat(pre, t, starts, 100, ends), starts, 100, ends, lengths)


def test_eight_keypoints_from_h5_rows_zero_padding():
    m = _model(30, n_keypoints=8)
    T, F = 64, 700
    assert _choice(m, T) == TILE
    g = torch.Generator().manual_seed(8)
    rows = (torch.rand((F, 150), generator=g) * 1000.0).to(DEV)
    pre = b2h.PreprocessRightHand(pad_mode="zeros")
    whole = pre.from_h5_rows(rows, [0], F)
    streams = {k: whole[k][0] for k in ("input_kp", "target_kp", "target_conf")}
    starts, ends, lengths = _windows(F, T, 33, seed=8)
    mat = pre.from_h5_rows(rows, starts, T, win_end=ends)
    mat["input_kp_bf16"] = None
    _check_fb(m, (streams,), mat, starts, T, ends, lengths, pad_mode="zeros")


def test_bulk_and_row_staged_windows_share_a_tile():
    """T = 64 holds two windows per tile: pair an aligned uncut window (bulk copy) with an odd start, a cut window and a
    crop past the clip end (row-by-row staging), also with a target stream whose base is only 8-B aligned."""
    m = _model(30)
    T, F = 64, 1000
    t, pre, s16, _ = _clip(F)
    starts = np.array([0, 1, 2, 3, 100, 100, 998, 4, 10, 11], dtype=np.int64)
    ends = np.array([F, F, F, F, F, 130, F, F, 40, F], dtype=np.int64)
    lengths = torch.tensor([64, 64, 50, 64, 64, 64, 64, 7, 64, 33])
    mat = _mat(pre, t, starts, T, ends)
    _check_fb(m, (s16,), mat, starts, T, ends, lengths)
    # shifted by one frame: the stream's base row is 8 B off a 16-B boundary, so the bulk-eligible windows change parity
    buf = torch.zeros(((F + 1) * 42,), dtype=torch.float32, device=DEV)
    buf[42:] = s16["target_kp"].reshape(-1)
    shifted = buf.view(F + 1, 21, 2)[1:]
    assert shifted.data_ptr() % 16 == 8
    _check_fb(m, (dict(s16, target_kp=shifted),), mat, starts, T, ends, lengths)


@pytest.mark.parametrize("C,T,fused", [(30, 64, True), (30, 64, False), (64, 64, False)])
def test_five_steps_equal_dense_steps(C, T, fused):
    F = 2000
    t, pre, s16, _ = _clip(F)
    out = []
    for views in (True, False):
        m = _model(C, seed=4)
        opt = b2h.FusedAdam(m.parameters(), lr=1e-3)
        st = opt._group_state(0, opt.param_groups[0], m)
        losses = []
        for k in range(5):
            starts, ends, lengths = _windows(F, T, 40, seed=100 + k)
            n_in, Cc, pe = m._geometry()
            lib = _lib.load()
            packed, ws, flat = m.packed_weights(), m.workspace(40, T), m.flat_parameters()
            loss = torch.zeros((), dtype=torch.float32, device=DEV)
            st["step"] += 1
            step_dev = _lib.ptr(st["step_dev"]) if fused else None
            common = (_lib.ptr(flat), _lib.ptr(packed), _lib.ptr(st["m"]), _lib.ptr(st["v"]), _lib.ptr(loss), 40, T, n_in, Cc, pe,
                      _lib.LOSS_L1, _lib.BF16, 1e-3, 0.9, 0.999, 1e-8, st["step"], step_dev, None, _lib.ptr(ws), ws.numel(),
                      _lib.stream_ptr(torch.device(DEV)))
            len32 = lengths.to(DEV, torch.int32)
            if views:
                ws_, we_ = (torch.from_numpy(a).to(DEV) for a in (starts, ends))
                _lib.check(lib.b2h_train_step_windows(_lib.ptr(s16["input_kp"]), _lib.DT_BF16, _lib.ptr(s16["target_kp"]), None,
                                                      F, _lib.ptr(ws_), _lib.ptr(we_), _lib.PAD_REPEAT_FIRST, _lib.ptr(len32),
                                                      *common))
            else:
                mat = _mat(pre, t, starts, T, ends)
                _lib.check(lib.b2h_train_step(_lib.ptr(mat["input_kp_bf16"]), _lib.DT_BF16, _lib.ptr(mat["target_kp"]), None,
                                              _lib.ptr(len32), *common))
            m.packed_weights(fresh_from_kernel=True)
            _tc_clean()
            losses.append(loss.clone())
        out.append((losses, m.flat_parameters().clone(), st["m"].clone(), st["v"].clone(), m.packed_weights().clone()))
    (lv, pv, mv, vv, kv), (ld, pd, md, vd, kd) = out
    assert all(torch.equal(a, b) for a, b in zip(lv, ld))
    assert torch.equal(pv, pd) and torch.equal(mv, md) and torch.equal(vv, vd) and torch.equal(kv, kd)


@pytest.mark.parametrize("C", [30, 64])
def test_window_runner_equals_train_step_runner(C):
    T, B, F, n_slots = 64, 48, 2500, 3
    t, pre, s16, _ = _clip(F)
    crops = []
    for k in range(6):
        starts, ends, lengths = _windows(F, T, B, seed=200 + k)
        crops.append({"win_start": torch.from_numpy(starts), "win_end": torch.from_numpy(ends), "n_frames": lengths})
    res = []
    for views in (True, False):
        m = _model(C, seed=6)
        opt = b2h.FusedAdam(m.parameters(), lr=1e-3)
        if views:
            r = WindowTrainStepRunner(m, opt, s16, B, T, n_slots=n_slots)
            batches = crops
        else:
            r = TrainStepRunner(m, opt, B, T, n_slots=n_slots, x_dtype=torch.bfloat16)
            batches = []
            for c in crops:
                mat = _mat(pre, t, c["win_start"].numpy(), T, c["win_end"].numpy())
                batches.append({"input_kp": mat["input_kp_bf16"], "target_kp": mat["target_kp"], "n_frames": c["n_frames"]})
        losses = []
        for k in range(3):                                     # eager, each slot once
            r.load(batches[k], slot=k)
            losses.append(r.step(k).clone())
        r.load_staged(r.host_stage({kk: (v.cpu() if torch.is_tensor(v) else v) for kk, v in batches[3].items()}), slot=0)
        r.load(batches[4], slot=1)
        r.load(batches[5], slot=2)
        r.capture(n_slots)                                     # graph over the rotating slots
        r.replay()
        losses.extend(r.loss.clone().unbind(0))
        r.finish()
        _tc_clean()
        # pipelined loop over host-staged buffers
        staged = [r.host_stage({kk: (v.cpu() if torch.is_tensor(v) else v) for kk, v in b.items()}) for b in batches]
        pl = list(pipelined_steps(r, staged))
        r.finish()
        res.append((losses, pl, m.flat_parameters().clone()))
    (lv, plv, pv), (ld, pld, pd) = res
    assert all(torch.equal(a, b) for a, b in zip(lv, ld))
    assert plv == pld
    assert torch.equal(pv, pd)


def test_dataset_crops_equal_batches():
    import random
    clips = [synthetic.synthetic_clip(n, seed=30 + n) for n in (40, 97, 150, 64, 300, 81)]
    packed = b2h.PackedClips(pose25=np.concatenate([c[0] for c in clips]), hand_left=np.concatenate([c[1] for c in clips]),
                             hand_right=np.concatenate([c[2] for c in clips]),
                             offsets=np.cumsum([0] + [c[0].shape[0] for c in clips]).astype(np.int64),
                             n_frames_meta=np.array([c[0].shape[0] + 3 for c in clips], dtype=np.int64),
                             texts=[""] * 6, utt_ids=list(range(6)), json_paths=[[None] * c[0].shape[0] for c in clips])
    T = 64
    res = []
    for views in (True, False):
        ds = b2h.GpuPoseDataset(packed, T, selection="randomcrop", device=DEV, rng=random.Random(11))
        m = _model(30, seed=9)
        opt = b2h.FusedAdam(m.parameters(), lr=1e-3)
        losses = []
        for k in range(4):
            idx = [(k * 5 + j) % 6 for j in range(8)]
            if views:
                c = ds.crops(idx)
                losses.append(b2h.fused_train_step_windows(m, ds.training_streams(), c["win_start"], T, c["n_frames"], opt,
                                                           win_end=c["win_end"]).clone())
            else:
                b = ds.batch(idx)
                losses.append(b2h.fused_train_step(m, b, opt).clone())
        _tc_clean()
        res.append((losses, m.flat_parameters().clone()))
    assert all(torch.equal(a, b) for a, b in zip(res[0][0], res[1][0]))
    assert torch.equal(res[0][1], res[1][1])


@pytest.mark.parametrize("prec,C,T,n_kp", [("fp32", 64, 64, 12), ("fp32-ffma", 30, 64, 12), ("bf16", 33, 260, 8)])
def test_ffma_shapes_are_refused(prec, C, T, n_kp):
    m = _model(C, prec, n_keypoints=n_kp)
    assert _choice(m, T) == FFMA
    F = 400
    s = {"input_kp": torch.zeros((F, n_kp, 2), device=DEV), "target_kp": torch.zeros((F, 21, 2), device=DEV)}
    with pytest.raises(_lib.B2HError, match="window views are trained on the tensor cores"):
        b2h.forward_backward_windows(m, s, np.array([0, 5]), T, [T, T])
    opt = b2h.FusedAdam(m.parameters(), lr=1e-3)
    with pytest.raises(_lib.B2HError, match="window views are trained on the tensor cores"):
        b2h.fused_train_step_windows(m, s, np.array([0, 5]), T, [T, T], opt)
    _tc_clean()
