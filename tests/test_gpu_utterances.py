"""GPU tier: ConvModel.predict_utterances (b2h_conv_forward_utterances) -- every utterance of a packed frame stream predicted
as one sequence, like the reference's infer_utterance -- against the float64 reference per utterance, bit for bit against
window views where both run the same kernel, on a 1 h clip, under graph capture, and with bad device offsets."""
import ctypes

import numpy as np
import pytest
import torch

import conv_ref
import hand_pose_sl_b200 as b2h
from hand_pose_sl_b200 import _lib

pytestmark = pytest.mark.gpu
DEV = "cuda:0"
TOL = {"bf16": 2e-2, "fp32": 1e-4}
BAD_OFFSETS = 80          # b2h_tc_status id of the planning kernel (include/b2h.h)


def _tc_clean():
    torch.cuda.synchronize()
    assert _lib.load().b2h_tc_status() == 0, "tensor-core kernel hit a wait timeout"


def _model(n_in, C, pos, prec, seed=0):
    torch.manual_seed(seed)
    m = b2h.ConvModel(C, "ReLU", pos, precision=prec, n_keypoints=n_in // 2, pos_emb_any_length=pos)
    sd = {k: v.detach().clone() for k, v in m.state_dict().items()}
    return m.to(DEV), sd


def _plan(F, S, m):
    n_in, C, pe = m._geometry()
    ts = ctypes.c_int(0)
    kind = _lib.load().b2h_utterances_plan(F, S, n_in, C, pe, _lib.PRECISIONS[m.precision], ctypes.byref(ts))
    return kind, ts.value


def _subwindows(L, Ts):
    lib = _lib.load()
    out = (ctypes.c_int * 3)()
    res = []
    for i in range(lib.b2h_utterance_subwindows(L, Ts, 0, None)):
        lib.b2h_utterance_subwindows(L, Ts, i, out)
        res.append(tuple(out))
    return res


def _rel(a, b):
    a, b = np.asarray(a, dtype=np.float64), np.asarray(b, dtype=np.float64)
    return float(np.abs(a - b).max() / max(np.abs(b).max(), 1e-30))


def _packed_stream(m, head=37, tail=50, seed=0):
    """Utterance lengths around every cut of the plan's sub-window length, packed (shuffled) behind `head` rows and before
    `tail` rows that belong to no utterance.  Returns (frames fp32 CPU, offsets int64, Ts, family)."""
    Ts = 256
    for _ in range(3):                                        # the plan's Ts depends on the mean length, which depends on Ts
        lens = [0, 1, 2, 8, 9, 16, 17, Ts - 16, Ts - 15, Ts, Ts + 1, 2 * Ts - 32, 2 * Ts - 31, 1000, 3000]
        np.random.default_rng(seed).shuffle(lens)
        offsets = np.concatenate([[0], np.cumsum(lens)]) + head
        F = int(offsets[-1]) + tail
        kind, ts = _plan(F, len(lens), m)
        if ts == Ts:
            break
        Ts = ts
    assert ts == Ts and kind in (2, 4)
    g = torch.Generator().manual_seed(seed)
    frames = torch.randn(F, m.n_in // 2, 2, generator=g) * 0.5
    return frames, offsets.astype(np.int64), Ts, kind


GEOMETRIES = [(24, 30, False, "bf16"), (24, 30, False, "fp32"), (16, 30, False, "bf16"), (24, 30, True, "bf16"),
              (24, 48, False, "bf16"), (24, 64, False, "bf16"), (24, 128, False, "bf16"), (24, 256, False, "bf16")]


@pytest.mark.parametrize("frames_dtype", [torch.float32, torch.bfloat16])
@pytest.mark.parametrize("n_in,C,pos,prec", GEOMETRIES)
def test_utterances_against_float64_reference(n_in, C, pos, prec, frames_dtype):
    m, sd = _model(n_in, C, pos, prec, seed=C + n_in)
    frames, offsets, Ts, kind = _packed_stream(m, seed=C)
    x = frames.to(frames_dtype)
    y = torch.full((frames.shape[0], 21, 2), float("nan"), device=DEV)
    assert m.predict_utterances(x.to(DEV), offsets, out=y) is y
    _tc_clean()
    yc = y.cpu()
    inside = np.zeros(frames.shape[0], dtype=bool)
    for a, b in zip(offsets[:-1], offsets[1:]):
        inside[a:b] = True
        if b == a:
            continue
        ref = conv_ref.forward(sd, x[a:b].float().double()[None], pos=100 if pos else None)["pred"][0]
        assert _rel(yc[a:b], ref) <= TOL[prec], (b - a, Ts, kind, _rel(yc[a:b], ref))
    assert not torch.isnan(yc[torch.from_numpy(inside)]).any()
    assert torch.isnan(yc[torch.from_numpy(~inside)]).all()           # rows of no utterance are not written
    # bit-identity with window views where the views run the same kernel family at Ts: each sub-window that lies inside its
    # utterance (a view cut at the utterance end pads zeros where the sequence ends instead, so cut sub-windows differ
    # near the end by design) equals predict_windows rows [clo, chi)
    if pos or _lib.load().b2h_kernel_choice(Ts, n_in, C, 0, _lib.PRECISIONS[prec], 0) != kind:
        return
    xs = x.to(DEV)
    starts, ends, cores = [], [], []
    for a, b in zip(offsets[:-1], offsets[1:]):
        for s, clo, chi in _subwindows(int(b - a), Ts):
            if s + Ts <= b - a:
                starts.append(a + s); ends.append(b); cores.append((clo, chi))
    assert starts
    yv = m.predict_windows(xs, np.array(starts), Ts, win_end=np.array(ends), pad_mode="zeros").cpu()
    _tc_clean()
    for w, (s, (clo, chi)) in enumerate(zip(starts, cores)):
        assert torch.equal(yv[w, clo:chi], yc[s + clo:s + chi]), (w, s, clo, chi)


@pytest.mark.parametrize("C", [30, 256])
def test_one_hour_clip_as_one_utterance(C):
    """108 000 frames as ONE utterance: a local float64 oracle at ~20 places (the cuts, both ends, the interior) on the slice
    [f - 40, f + 40) compared at least 8 frames from an artificial slice edge (the receptive field is +-8), bit-identity
    with window views on sampled sub-windows, and two runs bitwise equal."""
    F = 108_000
    m, sd = _model(24, C, False, "bf16", seed=C)
    kind, Ts = _plan(F, 1, m)
    assert Ts == 256
    g = torch.Generator().manual_seed(C)
    frames = (torch.randn(F, 12, 2, generator=g) * 0.5).to(torch.bfloat16)
    xs = frames.to(DEV)
    offsets = torch.tensor([0, F], dtype=torch.int64, device=DEV)
    y = m.predict_utterances(xs, offsets)
    y2 = m.predict_utterances(xs, offsets)
    _tc_clean()
    assert torch.equal(y, y2)
    yc = y.cpu()
    cuts = _subwindows(F, Ts)
    assert len(cuts) == 482
    rng = np.random.default_rng(C)
    places = [0, 1, F - 1, F - 9] + [s + clo for s, clo, _ in cuts[1:]][::60] + list(rng.integers(0, F, 8))
    assert len(places) >= 20
    got, want = [], []
    for f in places:
        lo, hi = max(0, f - 40), min(F, f + 40)
        ref = conv_ref.forward(sd, frames[lo:hi].float().double()[None])["pred"][0]
        keep_lo = lo if lo == 0 else lo + 8
        keep_hi = hi if hi == F else hi - 8
        got.append(yc[keep_lo:keep_hi]); want.append(ref[keep_lo - lo:keep_hi - lo])
    assert _rel(torch.cat(got), torch.cat(want)) <= TOL["bf16"]
    if _lib.load().b2h_kernel_choice(Ts, 24, C, 0, _lib.PRECISIONS["bf16"], 0) == kind:
        sample = cuts[:3] + cuts[200:203] + cuts[-3:]
        yv = m.predict_windows(xs, np.array([s for s, _, _ in sample]), Ts, win_end=np.full(len(sample), F), pad_mode="zeros")
        _tc_clean()
        for w, (s, clo, chi) in enumerate(sample):
            assert torch.equal(yv[w, clo:chi].cpu(), yc[s + clo:s + chi])


@pytest.mark.parametrize("C", [30, 256])
def test_graph_capture_and_denormalize(C):
    """A captured predict_utterances replayed on new frames with the same device offsets equals the eager call, and
    denormalize=1280 is 1280 x the unscaled output."""
    m, _ = _model(24, C, False, "bf16", seed=1)
    frames, offsets, _, _ = _packed_stream(m, seed=3)
    F = frames.shape[0]
    off = torch.from_numpy(offsets).to(DEV)
    buf = frames.to(torch.bfloat16).to(DEV)
    y = torch.zeros((F, 21, 2), device=DEV)
    side = torch.cuda.Stream()
    side.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(side):                      # warm-up: workspace and packed weights exist before capture
        m.predict_utterances(buf, off, denormalize=1280, out=y)
    torch.cuda.current_stream().wait_stream(side)
    graph = torch.cuda.CUDAGraph()
    with torch.cuda.graph(graph):
        m.predict_utterances(buf, off, denormalize=1280, out=y)
    for seed in (4, 5):
        g = torch.Generator().manual_seed(seed)
        buf.copy_((torch.randn(F, 12, 2, generator=g) * 0.5).to(torch.bfloat16))
        y.zero_()
        graph.replay()
        _tc_clean()
        eager = m.predict_utterances(buf, off, denormalize=1280)
        plain = m.predict_utterances(buf, offsets)
        _tc_clean()
        assert torch.equal(y, eager)
        assert torch.equal(eager, plain * 1280)


def test_bad_device_offsets_write_nothing():
    m, _ = _model(24, 30, False, "bf16")
    F = 500
    x = torch.randn(F, 12, 2, device=DEV)
    for bad in ([0, 100, 50, 200], [0, 100, F + 1], [-1, 100], [10, 5]):
        y = torch.full((F, 21, 2), float("nan"), device=DEV)
        m.predict_utterances(x, torch.tensor(bad, dtype=torch.int64, device=DEV), out=y)
        torch.cuda.synchronize()
        assert _lib.load().b2h_tc_status() == BAD_OFFSETS, bad
        assert torch.isnan(y).all(), bad
    y = m.predict_utterances(x, torch.tensor([0, 100, 100, 500], dtype=torch.int64, device=DEV))   # valid again afterwards
    _tc_clean()
    assert not torch.isnan(y).any()


def test_host_checks_and_empty_calls():
    m, _ = _model(24, 30, False, "bf16")
    x = torch.randn(300, 12, 2, device=DEV)
    for bad in ([0, 100, 50], [0, 301], [-1, 10], [[0, 10]], [0.0, 10.0]):
        with pytest.raises(ValueError):
            m.predict_utterances(x, np.array(bad))
    y = torch.full((300, 21, 2), 7.0, device=DEV)
    m.predict_utterances(x, [5], out=y)                      # S = 0: nothing to do
    m.predict_utterances(x, [0, 0, 0], out=y)                # empty utterances write nothing
    _tc_clean()
    assert (y == 7.0).all()
    with pytest.raises(RuntimeError, match="pos_emb requires T"):
        b2h.ConvModel(30, "ReLU", True, precision="bf16").to(DEV).predict_utterances(torch.zeros(10, 12, 2, device=DEV), [0, 10])
    with pytest.raises(_lib.B2HError, match="utterances are served"):
        _model(24, 64, False, "fp32")[0].predict_utterances(x, [0, 300])
    with pytest.raises(_lib.B2HError, match="utterances are served"):
        _model(24, 30, False, "fp32-ffma")[0].predict_utterances(x, [0, 300])
