"""GPU tier: streaming inference over window views for wide models (the streamed-weight kernel, conv_channels <= 256) and
long windows (the row-space kernel, T <= 1024).  `ConvModel.predict_windows` on a frame stream must return exactly
what `predict` returns on the windows K0 materialises, for every shape `predict` runs on the tensor cores."""
import numpy as np
import pytest
import torch

import b2h_oracle as oracle
import hand_pose_sl_b200 as b2h
from hand_pose_sl_b200 import _lib, synthetic

pytestmark = pytest.mark.gpu
DEV = "cuda:0"
KERNELS_WITH_VIEWS = (2, 3, 4)     # B2H_KERNEL_TC_TILE, _TC_ROWSPACE, _TC_WIDE (include/b2h.h)


def _tc_clean():
    torch.cuda.synchronize()
    assert _lib.load().b2h_tc_status() == 0, "tensor-core kernel hit a wait timeout"


def _model(C, prec="bf16", seed=0, **kw):
    m = b2h.ConvModel(C, "ReLU", kw.pop("pos_emb", False), precision=prec, **kw)
    if not kw and not m.pos_emb:
        m.load_state_dict(oracle.init_params(C, False, seed=seed))
    return m.to(DEV)


_CLIPS = {}


def _clip(F, pad_mode):
    """(device clip tensors, K0 with emit_bf16, bf16 stream, fp32 stream) of a seeded synthetic clip, cached per module."""
    key = (F, pad_mode)
    if key not in _CLIPS:
        pose, lh, rh = synthetic.synthetic_clip(F, seed=21)
        t = tuple(torch.from_numpy(a).to(DEV) for a in (pose, lh, rh))
        pre = b2h.PreprocessRightHand(emit_bf16=True, pad_mode=pad_mode)
        _CLIPS[key] = (t, pre, pre.frame_stream(*t), pre.frame_stream(*t, dtype=torch.float32), (pose, lh, rh))
    return _CLIPS[key]


def _check_views(m, F, T, starts, pad_mode, ends=None, lengths=None, denormalize=None):
    """predict_windows on the bf16 / fp32 streams == predict on K0's materialised bf16 / fp32 windows, bit for bit."""
    t, pre, s16, s32, _ = _clip(F, pad_mode)
    starts = np.asarray(starts, dtype=np.int64)
    mat = pre(*t, starts, T, win_end=ends)
    for stream, x in ((s16, mat["input_kp_bf16"]), (s32, mat["input_kp"])):
        y_view = m.predict_windows(stream, starts, T, win_end=ends, pad_mode=pad_mode, lengths=lengths, denormalize=denormalize)
        _tc_clean()
        y_mat = m.predict(x, lengths=lengths, denormalize=denormalize)
        _tc_clean()
        assert y_view.shape == (len(starts), T, 21, 2)
        assert torch.equal(y_view, y_mat)
    return y_view


@pytest.mark.parametrize("pad_mode", ["repeat_first", "zeros"])
@pytest.mark.parametrize("T,stride", [(64, 16), (64, 64), (126, 40), (200, 50), (256, 7)])
@pytest.mark.parametrize("C", [80, 128, 256])
def test_wide_views_equal_materialised_windows(C, T, stride, pad_mode):
    assert _lib.load().b2h_kernel_choice(T, 24, C, 0, _lib.PRECISIONS["bf16"], 0) == 4
    F = 1000
    _check_views(_model(C, seed=C + T), F, T, b2h.sliding_window_starts(F, T, stride), pad_mode)


@pytest.mark.parametrize("pad_mode", ["repeat_first", "zeros"])
@pytest.mark.parametrize("C,T", [(30, 257), (30, 512), (30, 1024), (48, 257), (48, 640)])
def test_rowspace_views_equal_materialised_windows(C, T, pad_mode):
    assert _lib.load().b2h_kernel_choice(T, 24, C, 0, _lib.PRECISIONS["bf16"], 0) == 3
    F = 3000
    _check_views(_model(C, seed=C + T), F, T, b2h.sliding_window_starts(F, T, T // 3), pad_mode)


@pytest.mark.parametrize("pad_mode", ["repeat_first", "zeros"])
@pytest.mark.parametrize("C,T", [(256, 64), (256, 126), (30, 300)])
def test_view_tile_and_window_edges(C, T, pad_mode):
    """Window counts that do not fill the last tile, more tiles than CTAs (the persistent loop and the weight ring wrap),
    win_end cuts inside the stream, windows that start at or past the end of the stream, and a clip shorter than a window."""
    m = _model(C, seed=3)
    F = 1100
    gh = max(258 // (T + 2), 1)
    for W in (1, gh + 1, 2 * gh + 1):
        _check_views(m, F, T, np.arange(W) * 37, pad_mode)
    if T == 64:
        starts = np.arange(500) * 2                                             # 167 tiles of 3 windows > 148 CTAs
        _check_views(m, F, T, starts, pad_mode)
    starts = b2h.sliding_window_starts(F, T, 16)
    _check_views(m, F, T, starts, pad_mode, ends=np.minimum(starts + 45, F).astype(np.int64))
    _check_views(m, F, T, np.array([F - 5, F - 1, F, F + 3, 5 * F], dtype=np.int64), pad_mode)   # partly / wholly padding
    _check_views(m, 40, T, np.array([0, 8, 39], dtype=np.int64), pad_mode)                   # clip shorter than a window


@pytest.mark.parametrize("C,T", [(128, 64), (256, 200), (30, 300)])
def test_view_epilogues(C, T):
    """mask_output(lengths) + de-normalisation through views == the same options on the materialised windows."""
    F = 1000
    starts = b2h.sliding_window_starts(F, T, 24)
    lengths = torch.from_numpy((np.arange(len(starts)) * 13) % (T + 5)).to(torch.int32)
    y = _check_views(_model(C, seed=7), F, T, starts, "repeat_first", lengths=lengths, denormalize=1280.0)
    for w in range(min(len(starts), 16)):
        assert not y[w, int(lengths[w]):].any()


def _materialise(frames, starts, T, ends=None, pad_mode="repeat_first"):
    """Test-local restatement of the window rule: crop [s, s+T) cut at min(end, F), then repeat-first or zero padding."""
    F = frames.shape[0]
    idx = np.empty((len(starts), T), dtype=np.int64)
    for w, s in enumerate(starts):
        cend = min(int(ends[w]) if ends is not None else F, F)
        f = s + np.arange(T)
        bad = (f >= cend) | (f < 0)
        f[bad] = s if (pad_mode == "repeat_first" and 0 <= s < cend) else -1
        idx[w] = f
    ix = torch.from_numpy(idx).to(frames.device)
    out = frames[ix.clamp(min=0)]
    out[ix < 0] = 0
    return out


def test_materialise_helper_matches_k0():
    F, T = 1000, 64
    starts = np.array([0, 16, 900, 960, 999, 1000, 1200], dtype=np.int64)
    ends = np.array([1000, 50, 1000, 990, 1000, 1000, 1000], dtype=np.int64)
    for pad_mode in ("repeat_first", "zeros"):
        t, pre, s16, _, _ = _clip(F, pad_mode)
        mat = pre(*t, starts, T, win_end=ends)
        assert torch.equal(_materialise(s16, starts, T, ends, pad_mode), mat["input_kp_bf16"])


@pytest.mark.parametrize("pad_mode", ["repeat_first", "zeros"])
@pytest.mark.parametrize("C,T", [(128, 64), (256, 126), (30, 300)])
@pytest.mark.parametrize("layout", ["pos_emb_any_length", "8_keypoints"])
def test_view_channel_layouts(layout, C, T, pad_mode):
    """25 input channels (pos-emb row first: the scalar staging path; zero rows keep t / max_len) and 16 input channels
    (two 16-B chunks) on a stream built directly, against a test-local materialisation of its windows."""
    torch.manual_seed(C + T)
    if layout == "pos_emb_any_length":
        m = _model(C, pos_emb=True, pos_emb_any_length=True)
        K = 12
    else:
        m = _model(C, n_keypoints=8)
        K = 8
    F = 700
    g = torch.Generator().manual_seed(T)
    frames = (torch.randn(F, K, 2, generator=g) * 0.3).to(DEV)
    starts = np.concatenate([b2h.sliding_window_starts(F, T, 33), [F + 2]]).astype(np.int64)
    ends = np.minimum(starts + T - 9, F).astype(np.int64)
    for dtype in (torch.bfloat16, torch.float32):
        fs = frames.to(dtype)
        for e in (None, ends):
            y_view = m.predict_windows(fs, starts, T, win_end=e, pad_mode=pad_mode)
            y_mat = m.predict(_materialise(fs, starts, T, e, pad_mode))
            _tc_clean()
            assert torch.equal(y_view, y_mat)


def test_wide_views_vs_oracle():
    """C=256, 64-frame windows at stride 16 through views, against the oracle pipeline (reference transforms + ConvModel)."""
    F, T, C = 1000, 64, 256
    _, _, s16, _, (pose, lh, rh) = _clip(F, "repeat_first")
    starts = b2h.sliding_window_starts(F, T, 16)
    sd = oracle.init_params(C, False, seed=5)
    m = b2h.ConvModel(C, "ReLU", False, precision="bf16")
    m.load_state_dict(sd)
    y = m.to(DEV).predict_windows(s16, starts, T, denormalize=1280)
    _tc_clean()
    want = oracle.preprocess_windows(pose, lh, rh, starts, T)
    ref = oracle.conv_model_forward(sd, torch.from_numpy(want["input_kp"])).contiguous().numpy() * np.float32(1280)
    assert oracle.rel_err(y.cpu().numpy(), ref) <= 2e-2


def test_wide_views_graph_capture():
    """frame_stream(out=) + predict_windows(out=) captured in a CUDA graph for C=256: the replay equals the eager calls,
    and after load_state_dict (packed weights refreshed outside the graph) it follows the new weights."""
    F, T, C = 1000, 64, 256
    t, pre, _, _, _ = _clip(F, "repeat_first")
    starts = torch.from_numpy(b2h.sliding_window_starts(F, T, 16)).to(DEV)
    m = _model(C, seed=1)
    stream = torch.empty((F, 12, 2), dtype=torch.bfloat16, device=DEV)
    y = torch.empty((starts.numel(), T, 21, 2), dtype=torch.float32, device=DEV)
    side = torch.cuda.Stream()
    side.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(side):                      # warm-up: lazy buffers and the packed weights exist before capture
        pre.frame_stream(*t, out=stream)
        m.predict_windows(stream, starts, T, denormalize=1280, out=y)
    torch.cuda.current_stream().wait_stream(side)
    graph = torch.cuda.CUDAGraph()
    with torch.cuda.graph(graph):
        pre.frame_stream(*t, out=stream)
        m.predict_windows(stream, starts, T, denormalize=1280, out=y)
    for seed in (1, 2):
        if seed == 2:
            m.load_state_dict(oracle.init_params(C, False, seed=seed))
            m.packed_weights()
        y.zero_()
        graph.replay()
        _tc_clean()
        eager = m.predict_windows(pre.frame_stream(*t), starts, T, denormalize=1280)
        _tc_clean()
        assert torch.equal(y, eager)
        assert torch.equal(y, _model(C, seed=seed).predict_windows(pre.frame_stream(*t), starts, T, denormalize=1280))


@pytest.mark.parametrize("prec", ["bf16", "fp32"])
@pytest.mark.parametrize("C", [30, 48, 64, 80, 256])
@pytest.mark.parametrize("T", [64, 256, 257, 1024, 1025])
def test_view_dispatch_rule(T, C, prec):
    """predict_windows serves exactly the shapes predict runs on a tensor-core kernel: it raises B2HError when
    b2h_kernel_choice is not the tile, row-space or wide kernel, and otherwise returns what predict returns."""
    choice = _lib.load().b2h_kernel_choice(T, 24, C, 0, _lib.PRECISIONS[prec], 0)
    m = _model(C, prec, seed=2)
    F = 1200
    _, pre, s16, s32, _ = _clip(F, "repeat_first")
    t = _clip(F, "repeat_first")[0]
    starts = np.array([0, 100, 1100], dtype=np.int64)
    frames = s16 if prec == "bf16" else s32
    if choice not in KERNELS_WITH_VIEWS:
        with pytest.raises(_lib.B2HError):
            m.predict_windows(frames, starts, T)
        return
    mat = pre(*t, starts, T)
    x = mat["input_kp_bf16"] if prec == "bf16" else mat["input_kp"]
    y_mat = m.predict(x)
    _tc_clean()
    assert torch.equal(m.predict_windows(frames, starts, T), y_mat)
    _tc_clean()


@pytest.mark.parametrize("B", [1, 297, 600])
@pytest.mark.parametrize("C,T", [(48, 257), (48, 400), (48, 640), (40, 641), (64, 257), (30, 1024)])
def test_rowspace_limits_hold_at_every_batch(C, T, B):
    """The row-space kernel packs more windows into a CTA as the batch grows, but never more than fit in shared memory, so
    a shape b2h_forward_supported reports runs at every batch: predict and predict_windows equal predict over chunks of at
    most 100 windows bit for bit (each row accumulates the same taps and k-steps whichever tile holds it) and the oracle
    within 2e-2.  Where not even one window fits, both raise."""
    m = _model(C, seed=C + T)
    F = 4000
    t, pre, s16, _, (pose, lh, rh) = _clip(F, "repeat_first")
    starts = (np.arange(B, dtype=np.int64) * 37) % (F - T)
    if not _lib.load().b2h_forward_supported(T, 24, C, 0, _lib.PRECISIONS["bf16"]):
        x = torch.zeros((B, T, 12, 2), dtype=torch.bfloat16, device=DEV)
        with pytest.raises(_lib.B2HError):
            m.predict(x)
        with pytest.raises(_lib.B2HError):
            m.predict_windows(s16, starts, T)
        return
    x = pre(*t, starts, T)["input_kp_bf16"]
    y = m.predict(x)
    _tc_clean()
    y_view = m.predict_windows(s16, starts, T)
    _tc_clean()
    y_chunks = torch.cat([m.predict(x[i:i + 100]) for i in range(0, B, 100)])
    _tc_clean()
    assert torch.equal(y, y_chunks) and torch.equal(y_view, y_chunks)
    sd = oracle.init_params(C, False, seed=C + T)
    want = oracle.preprocess_windows(pose, lh, rh, starts, T)
    ref = oracle.conv_model_forward(sd, torch.from_numpy(want["input_kp"])).contiguous().numpy()
    assert oracle.rel_err(y.cpu().numpy(), ref) <= 2e-2
