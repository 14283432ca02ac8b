"""GPU tier: validation on segments of device-resident frame streams, each segment one whole sequence
(b2h_validate_utterances / steps.validate_utterances): against the float64 reference per segment, the criterion against the
float64 criterion on predict_utterances' rows, the loss against the segment training step's, no side effects, bad device
segments, determinism and graph replay, and a 1 h segment and the 5 000-utterance mix.  Every case first pins the plan
(family and sub-window length) it exists to reach."""
import ctypes

import numpy as np
import pytest
import torch

import conv_ref
import hand_pose_sl_b200 as b2h
from hand_pose_sl_b200 import _lib
from test_gpu_gradient_paths import SPLIT_TOL, _bf16_bounds
from test_gpu_train_utterances import _model, _on_dev, _segments, _streams

pytestmark = pytest.mark.gpu
DEV = "cuda:0"
TILE, WIDE = 2, 4
BAD_SEGMENTS = 81         # b2h_tc_status id of a refused segment list (include/b2h.h)


def _tc_status():
    torch.cuda.synchronize()
    return int(_lib.load().b2h_tc_status())


def _vplan(m, S, max_len):
    n_in, C, pe = m._geometry()
    ts = ctypes.c_int(0)
    kind = _lib.load().b2h_validate_utterances_plan(S, max_len, n_in, C, pe, _lib.PRECISIONS[m.precision], ctypes.byref(ts))
    return kind, ts.value


def _fplan(m, F, S):
    n_in, C, pe = m._geometry()
    ts = ctypes.c_int(0)
    kind = _lib.load().b2h_utterances_plan(F, S, n_in, C, pe, _lib.PRECISIONS[m.precision], ctypes.byref(ts))
    return kind, ts.value


def _criterion64(pred, streams, ss, se, kind):
    """float64 per-segment criterion of rows pred[a:b] (the stream rows of each segment) and the loss rule."""
    tgt = streams["target_kp"].double().cpu()
    conf = streams["target_conf"].double().cpu()
    p = pred.double().cpu()
    out = []
    for a, b in zip(ss.tolist(), se.tolist()):
        s = torch.ones((b - a, 21, 1), dtype=torch.float64) if kind == "L1" else conf[a:b, :, None]
        out.append(float((p[a:b] * s - tgt[a:b] * s).abs().sum()) / (42.0 * (b - a)))
    return np.asarray(out)


def _combine(seg, kind):
    return float(np.mean(seg)) if kind == "L1" else float(np.sum(seg))


# ---------------------------------------------------------------------------------------------------- float64 reference
# (precision, input channels, conv_channels, pos-emb, {max_len: (family, Ts) the plan takes})
_GEOMETRIES = [
    ("bf16", 24, 30, False, {64: (TILE, 64), 300: (TILE, 128), 600: (TILE, 256)}),
    ("fp32", 24, 30, False, {64: (TILE, 64), 300: (TILE, 128), 600: (TILE, 256)}),
    ("bf16", 16, 30, False, {64: (TILE, 64), 600: (TILE, 256)}),
    ("bf16", 24, 30, True, {300: (TILE, 128)}),
    ("bf16", 24, 64, False, {300: (TILE, 128), 600: (WIDE, 256)}),
    ("bf16", 24, 128, False, {64: (WIDE, 64), 600: (WIDE, 256)}),
    ("bf16", 16, 256, True, {64: (WIDE, 64), 300: (WIDE, 256)}),
]


@pytest.mark.parametrize("prec,n_in,C,pos,plans", _GEOMETRIES, ids=[f"{g[0]}-n{g[1]}-C{g[2]}-pos{int(g[3])}" for g in _GEOMETRIES])
def test_matches_float64_reference(prec, n_in, C, pos, plans):
    """Per segment: the float64 forward of exactly L_s frames (bf16 / no rounding model) and the criterion.  Lengths 1, 2, 8,
    9 and around every cut of the plan's Ts, gaps, a duplicate and an overlapping segment; fp32 and bf16 frames; both
    losses.  A segment's loss moves no further than its weighted mean prediction error, so the bound is the prediction
    tolerance of the segment-training tests (times the segment's largest |prediction|) plus 1e-6 relative."""
    m, sd = _model(n_in, C, pos, prec, seed=C + n_in)
    pe = m.pos_emb.max_len if pos else None
    rnd = "bf16" if prec == "bf16" else "none"
    for max_len, want in plans.items():
        Ts = want[1]
        cand = [1, 2, 8, 9, Ts - 1, Ts, Ts + 1, 2 * Ts - 33, 2 * Ts - 32, 2 * Ts - 31, max_len]
        lengths = sorted({L for L in cand if 1 <= L <= max_len})
        ss, se, F = _segments(lengths, seed=max_len + C)
        assert _vplan(m, len(ss), max_len) == want
        streams = _streams(F, n_in, seed=max_len)
        for x_dtype in ((torch.float32, torch.bfloat16) if prec == "bf16" else (torch.float32,)):
            dev_streams = _on_dev(streams, x_dtype)
            x = dev_streams["input_kp"].float().cpu()
            preds = [conv_ref.forward(sd, x[a:b][None], pe, rnd)["pred"] for a, b in zip(ss.tolist(), se.tolist())]
            if rnd == "bf16":
                i = int(np.argmax(se - ss))
                ptol = _bf16_bounds(sd, x[ss[i]:se[i]][None], pe)["pred"]
            else:
                ptol = SPLIT_TOL
            for kind in ("L1", "confL1"):
                loss, seg = b2h.validate_utterances(m, dev_streams, torch.from_numpy(ss), torch.from_numpy(se),
                                                    max_len=max_len, loss=kind, per_segment=True)
                assert _tc_status() == 0
                seg = seg.cpu().double().numpy()
                for s, (a, b) in enumerate(zip(ss.tolist(), se.tolist())):
                    ref, _, _ = conv_ref.criterion(preds[s], streams["target_kp"][a:b][None], [b - a], kind,
                                                   streams["target_conf"][a:b][None])
                    ref = float(ref)
                    bound = ptol * float(preds[s].abs().max()) + 1e-6 * abs(ref)
                    assert abs(seg[s] - ref) <= bound, (prec, C, max_len, x_dtype, kind, s, b - a, seg[s], ref, bound)
                assert abs(float(loss) - _combine(seg, kind)) <= 1e-6 * abs(_combine(seg, kind))


# ---------------------------------------------------------------------------------------------------- criterion exactness
@pytest.mark.parametrize("C,max_len,lo,hi,want", [(30, 300, 30, 180, (TILE, 128)), (128, 64, 10, 64, (WIDE, 64)),
                                                  (256, 600, 257, 440, (WIDE, 256))])
def test_criterion_equals_float64_criterion_on_predictions(C, max_len, lo, hi, want):
    """Disjoint segments that tile the stream (the utterances of predict_utterances), both plans pinned to the same family
    and Ts: seg_loss against the float64 criterion applied to predict_utterances' rows within 1e-5 relative, loss against
    the float64 combination of the returned seg_loss within 1e-6."""
    m, _ = _model(24, C, False, "bf16", seed=C)
    rng = np.random.default_rng(C)
    lengths = rng.integers(lo, hi + 1, size=41).astype(np.int64)
    lengths[0] = max_len
    off = np.concatenate([[0], np.cumsum(lengths)]).astype(np.int64)
    F = int(off[-1])
    ss, se = off[:-1], off[1:]
    assert _vplan(m, len(ss), max_len) == want and _fplan(m, F, len(ss)) == want
    streams = _on_dev(_streams(F, 24, seed=C), torch.bfloat16)
    pred = m.predict_utterances(streams["input_kp"], torch.from_numpy(off).to(DEV))
    for kind in ("L1", "confL1"):
        loss, seg = b2h.validate_utterances(m, streams, torch.from_numpy(ss), torch.from_numpy(se), max_len=max_len,
                                            loss=kind, per_segment=True)
        assert _tc_status() == 0
        ref = _criterion64(pred, streams, ss, se, kind)
        seg = seg.cpu().double().numpy()
        assert np.all(np.abs(seg - ref) <= 1e-5 * np.abs(ref)), (C, kind)
        assert abs(float(loss) - _combine(seg, kind)) <= 1e-6 * abs(_combine(seg, kind)), (C, kind)


# ---------------------------------------------------------------------------------------------------- agreement with training
@pytest.mark.parametrize("prec", ["bf16", "fp32"])
def test_loss_equals_segment_training_loss(prec):
    m, _ = _model(24, 30, False, prec, seed=7)
    ss, se, F = _segments([1, 9, 40, 127, 128, 129, 250, 300], seed=7)
    streams = _on_dev(_streams(F, 24, seed=7))
    assert _vplan(m, len(ss), 300) == (TILE, 128)
    for kind in ("L1", "confL1"):
        lv = b2h.validate_utterances(m, streams, ss, se, max_len=300, loss=kind)
        lt, _ = b2h.forward_backward_utterances(m, streams, ss, se, max_len=300, loss=kind)
        assert _tc_status() == 0
        assert abs(float(lv) - float(lt)) <= 1e-5 * abs(float(lt)), (prec, kind, float(lv), float(lt))


# ---------------------------------------------------------------------------------------------------- side effects
def test_no_side_effects_and_three_launches():
    m, _ = _model(24, 30, False, "bf16", seed=4)
    opt = b2h.FusedAdam(m.parameters(), lr=1e-3)
    ss, se, F = _segments([30, 195, 600, 77], seed=4)
    streams = _on_dev(_streams(F, 24, seed=4))
    assert _vplan(m, len(ss), 600) == (TILE, 256)
    b2h.fused_train_step_utterances(m, streams, ss, se, opt, max_len=600)
    st = opt._group_state(0, opt.param_groups[0], m)
    ss_d, se_d = torch.from_numpy(ss).to(DEV), torch.from_numpy(se).to(DEV)
    b2h.validate_utterances(m, streams, ss_d, se_d, max_len=600)          # workspace allocated, plan warmed
    torch.cuda.synchronize()
    train_ws = m._workspace.clone()
    before = [m.flat_parameters().clone(), m.packed_weights().clone(), st["m"].clone(), st["v"].clone(), st["step_dev"].clone()]
    n0 = _lib.launch_count()
    loss = b2h.validate_utterances(m, streams, ss_d, se_d, max_len=600, loss="confL1")
    assert _lib.launch_count() - n0 == 3
    assert _tc_status() == 0 and torch.isfinite(loss).item()
    after = [m.flat_parameters(), m.packed_weights(), st["m"], st["v"], st["step_dev"]]
    for a, b in zip(before, after):
        assert torch.equal(a, b)
    assert torch.equal(train_ws, m._workspace)
    b2h.fused_train_step_utterances(m, streams, ss, se, opt, max_len=600)   # training goes on after it
    assert _tc_status() == 0 and int(st["step_dev"]) == 2


# ---------------------------------------------------------------------------------------------------- bad device segments
@pytest.mark.parametrize("C", [30, 256])
def test_bad_segments_give_nan(C):
    m, _ = _model(24, C, False, "bf16", seed=6)
    ss, se, F = _segments([40, 120, 64], seed=2)
    streams = _on_dev(_streams(F, 24, seed=2))
    assert _vplan(m, len(ss), 128)[0] == (TILE if C == 30 else WIDE)
    good_s, good_e = torch.from_numpy(ss).to(DEV), torch.from_numpy(se).to(DEV)
    ref_loss, ref_seg = b2h.validate_utterances(m, streams, good_s, good_e, max_len=128, per_segment=True)
    ref_loss, ref_seg = ref_loss.clone(), ref_seg.clone()
    assert _tc_status() == 0
    g0, g1 = int(ss[0]), int(ss[1])
    bads = {"end < start": (0, g0, g0 - 1), "L > max_len": (1, g1, g1 + 129), "end > F": (2, F - 10, F + 1),
            "L = 0": (0, g0, g0)}
    for name, (i, a, e) in bads.items():
        s_s, s_e = good_s.clone(), good_e.clone()
        s_s[i], s_e[i] = a, e
        loss, seg = b2h.validate_utterances(m, streams, s_s, s_e, max_len=128, per_segment=True)
        assert _tc_status() == BAD_SEGMENTS, name
        assert torch.isnan(loss).item() and bool(torch.isnan(seg).all()), name
        loss, seg = b2h.validate_utterances(m, streams, good_s, good_e, max_len=128, per_segment=True)
        assert _tc_status() == 0, name
        assert torch.equal(loss, ref_loss) and torch.equal(seg, ref_seg), name


# ---------------------------------------------------------------------------------------------------- determinism
@pytest.mark.parametrize("C,prec,max_len,want", [(30, "bf16", 600, (TILE, 256)), (30, "fp32", 64, (TILE, 64)),
                                                 (256, "bf16", 64, (WIDE, 64))])
def test_deterministic_and_graph_replay(C, prec, max_len, want):
    m, _ = _model(24, C, False, prec, seed=3)
    rng = np.random.default_rng(3)
    S, F = 200, 40000
    lens = rng.integers(1, max_len + 1, size=S)
    a = rng.integers(0, F - max_len, size=S)
    ss, se = torch.from_numpy(a.astype(np.int64)).to(DEV), torch.from_numpy((a + lens).astype(np.int64)).to(DEV)
    streams = _on_dev(_streams(F, 24, seed=3), torch.bfloat16)
    assert _vplan(m, S, max_len) == want
    l1, s1 = [t.clone() for t in b2h.validate_utterances(m, streams, ss, se, max_len=max_len, loss="confL1", per_segment=True)]
    l2, s2 = [t.clone() for t in b2h.validate_utterances(m, streams, ss, se, max_len=max_len, loss="confL1", per_segment=True)]
    assert torch.equal(l1, l2) and torch.equal(s1, s2)
    out = {}
    side = torch.cuda.Stream()
    side.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(side):
        b2h.validate_utterances(m, streams, ss, se, max_len=max_len, loss="confL1", per_segment=True)
    torch.cuda.current_stream().wait_stream(side)
    torch.cuda.synchronize()
    graph = torch.cuda.CUDAGraph()
    with torch.cuda.graph(graph):
        out["l"], out["s"] = b2h.validate_utterances(m, streams, ss, se, max_len=max_len, loss="confL1", per_segment=True)
    graph.replay()
    graph.replay()
    assert _tc_status() == 0
    assert torch.equal(out["l"], l1) and torch.equal(out["s"], s1)


# ---------------------------------------------------------------------------------------------------- scale
@pytest.mark.parametrize("C", [30, 256])
def test_one_hour_segment_and_utterance_mix(C):
    """One 108 000-frame segment, and the seeded 5 000-utterance mix of tools/utterances_bench.py, against the float64
    criterion on predict_utterances' rows of the same frames."""
    m, _ = _model(24, C, False, "bf16", seed=C)
    rng = np.random.default_rng(0)
    mix = np.clip(rng.exponential(170.0, 5000) + 30, 30, 600).astype(np.int64)
    for lengths, max_len in ((np.array([108000], dtype=np.int64), 108000), (mix, 600)):
        off = np.concatenate([[0], np.cumsum(lengths)]).astype(np.int64)
        F = int(off[-1])
        ss, se = off[:-1], off[1:]
        assert _vplan(m, len(ss), max_len) == (TILE if C == 30 else WIDE, 256)
        streams = _on_dev(_streams(F, 24, seed=C), torch.bfloat16)
        pred = m.predict_utterances(streams["input_kp"], torch.from_numpy(off).to(DEV))
        for kind in ("L1", "confL1"):
            loss, seg = b2h.validate_utterances(m, streams, torch.from_numpy(ss), torch.from_numpy(se), max_len=max_len,
                                                loss=kind, per_segment=True)
            assert _tc_status() == 0
            ref = _criterion64(pred, streams, ss, se, kind)
            seg = seg.cpu().double().numpy()
            assert np.all(np.abs(seg - ref) <= 1e-5 * np.abs(ref)), (C, len(ss), kind, float(np.abs(seg - ref).max()))
            assert abs(float(loss) - _combine(seg, kind)) <= 1e-6 * abs(_combine(seg, kind)), (C, len(ss), kind)
