"""GPU tier: training on segments of device-resident frame streams, each segment one whole sequence
(b2h_train_forward_backward_utterances / b2h_train_step_utterances): against the float64 reference per segment, against
dense training on the materialised windows, the fused step against forward_backward + FusedAdam, bad device segments,
the runner under graph capture and in pipelined_steps, and a 1 h utterance.  Every case first pins the plan it exists
to reach."""
import ctypes

import numpy as np
import pytest
import torch

import b2h_oracle as oracle
import conv_ref
import hand_pose_sl_b200 as b2h
from hand_pose_sl_b200 import _lib
from hand_pose_sl_b200.runner import UtteranceTrainStepRunner, pipelined_steps
from test_gpu_gradient_paths import BF16_CAP, SPLIT_FLIP_EPS, SPLIT_TOL, _bf16_bounds

pytestmark = pytest.mark.gpu
DEV = "cuda:0"
TILE = 2
BAD_SEGMENTS = 81         # b2h_tc_status id of a refused segment list (include/b2h.h)


def _tc_status():
    torch.cuda.synchronize()
    return int(_lib.load().b2h_tc_status())


def _model(n_in, C, pos, prec, seed=0):
    torch.manual_seed(seed)
    m = b2h.ConvModel(C, "ReLU", pos, precision=prec, n_keypoints=n_in // 2, pos_emb_any_length=pos)
    sd = {k: v.detach().clone() for k, v in m.state_dict().items()}
    return m.to(DEV), sd


def _plan(m, S, max_len):
    n_in, C, pe = m._geometry()
    ts = ctypes.c_int(0)
    kind = _lib.load().b2h_train_utterances_plan(S, max_len, n_in, C, pe, _lib.PRECISIONS[m.precision], ctypes.byref(ts))
    return kind, ts.value


def _streams(F, n_in, seed):
    g = torch.Generator().manual_seed(seed)
    return {"input_kp": torch.randn((F, n_in // 2, 2), generator=g) * 0.5,
            "target_kp": torch.randn((F, 21, 2), generator=g) * 0.3,
            "target_conf": torch.rand((F, 21), generator=g)}


def _on_dev(streams, x_dtype=torch.float32):
    d = {k: v.to(DEV) for k, v in streams.items()}
    d["input_kp"] = d["input_kp"].to(x_dtype)
    return d


def _segments(lengths, seed):
    """Segments of the given lengths laid out with gaps (rows of no segment), plus a duplicate of the longest one and one
    overlapping it; returns (seg_start, seg_end, F)."""
    rng = np.random.default_rng(seed)
    starts, pos = [], int(rng.integers(0, 9))
    for L in lengths:
        starts.append(pos)
        pos += L + int(rng.integers(0, 13))
    F = pos + 40
    i = int(np.argmax(lengths))
    starts += [starts[i], starts[i] + min(5, lengths[i] - 1)]
    lens = list(lengths) + [lengths[i], lengths[i] - min(5, lengths[i] - 1)]
    ss = np.asarray(starts, dtype=np.int64)
    return ss, ss + np.asarray(lens, dtype=np.int64), F


def _reference(sd, streams, ss, se, pos, rnd, kind, max_len, want_pred=True, pred_gpu=None):
    """float64 reference of the segment step: per segment one window of exactly L frames, combined by the loss rule.  For
    rnd == "none" (fp32 mode) also the summed ReLU-flip allowance of the gradients (conv_ref.relu_flip_allowance).
    pred_gpu (the kernel's masked prediction): the backward takes the kernel's L1-sign decisions.  |r| is not differentiable
    at 0, and a residual within the mode's precision of zero may take either sign; with loss weights 1 / (42 L S) one such
    decision in a 1-frame segment moves a gradient by percents.  The prediction itself is checked against the reference."""
    x = streams["input_kp"].float()
    S = len(ss)
    pred = torch.zeros((S, max_len, 21, 2), dtype=torch.float64) if want_pred else None
    loss, grads, allow = 0.0, {k: 0.0 for k in conv_ref.NAMES}, {k: 0.0 for k in conv_ref.NAMES}
    for s, (a, b) in enumerate(zip(ss.tolist(), se.tolist())):
        L = b - a
        f = conv_ref.forward(sd, x[a:b][None], pos, rnd)
        ls, p, d = conv_ref.criterion(f["pred"], streams["target_kp"][a:b][None], [L], kind, streams["target_conf"][a:b][None])
        if kind == "L1":
            ls, d = ls / S, d / S
        if pred_gpu is not None:
            sc = torch.ones((1, L, 21, 2), dtype=torch.float64) if kind == "L1" else \
                streams["target_conf"][a:b][None, :, :, None].double().expand(1, L, 21, 2)
            r = pred_gpu[s, :L][None].double() * sc - streams["target_kp"][a:b][None].double() * sc
            d = torch.sign(r) * sc / (42.0 * L) / (S if kind == "L1" else 1)
        up = []
        g = conv_ref.backward(sd, x[a:b][None], d, pos, rnd, fwd=f, upstream=up)
        if rnd == "none":
            al = conv_ref.relu_flip_allowance(sd, f, up, SPLIT_FLIP_EPS)
            allow = {k: allow[k] + al[k] for k in conv_ref.NAMES}
        loss += float(ls)
        grads = {k: grads[k] + g[k] for k in conv_ref.NAMES}
        if want_pred:
            pred[s, :L] = p[0]
    return loss, pred, grads, allow


def _split(m, flat):
    out, off = {}, 0
    for k, p in zip(conv_ref.NAMES, m._ordered_params()):
        out[k] = flat[off:off + p.numel()].view(p.shape).double().cpu()
        off += p.numel()
    return out


def _check_against_reference(m, sd, streams, ss, se, max_len, prec, pos, x_dtype, kind, want_pred=True):
    rnd = "bf16" if prec == "bf16" else "none"
    pe = m.pos_emb.max_len if pos else None
    dev_streams = _on_dev(streams, x_dtype)
    out = b2h.forward_backward_utterances(m, dev_streams, torch.from_numpy(ss), torch.from_numpy(se), max_len=max_len,
                                          loss=kind, want_pred=want_pred)
    loss, grads = out[0], out[1]
    assert _tc_status() == 0
    ref_streams = dict(streams, input_kp=dev_streams["input_kp"].float().cpu())
    r_loss, r_pred, r_g, allow = _reference(sd, ref_streams, ss, se, pe, rnd, kind, max_len, want_pred,
                                            out[2].cpu() if want_pred else None)
    where = (prec, x_dtype, kind, max_len)
    assert abs(float(loss) - r_loss) <= 1e-4 * abs(r_loss), (where, float(loss), r_loss)
    if want_pred:
        pred = out[2]
        if rnd == "bf16":
            i = int(np.argmax(se - ss))
            ptol = _bf16_bounds(sd, ref_streams["input_kp"][ss[i]:se[i]][None], pe)["pred"]
        else:
            ptol = SPLIT_TOL
        assert oracle.rel_err(pred.cpu().double().numpy(), r_pred.numpy()) <= ptol, where
        for s, (a, b) in enumerate(zip(ss.tolist(), se.tolist())):
            assert not pred[s, b - a:].any(), (where, s)
    for k, v in _split(m, grads).items():
        ref = r_g[k].numpy()
        if rnd == "bf16":
            assert oracle.rel_err(v.numpy(), ref) <= BF16_CAP, (where, k, oracle.rel_err(v.numpy(), ref))
        else:             # fp32 mode: 1e-4 beyond what hidden ReLU decisions within its precision of zero can move
            excess = float((np.abs(v.numpy() - ref) - np.asarray(allow[k])).max()) / float(np.abs(ref).max())
            assert excess <= SPLIT_TOL, (where, k, excess, oracle.rel_err(v.numpy(), ref))


_GEOMETRIES = [("bf16", 24, 30, False), ("fp32", 24, 30, False), ("bf16", 16, 30, False), ("bf16", 24, 30, True),
               ("bf16", 24, 32, False)]


@pytest.mark.parametrize("prec,n_in,C,pos", _GEOMETRIES)
def test_matches_float64_reference(prec, n_in, C, pos):
    """Lengths around every cut of each sub-window length the plan reaches (max_len 64 / 320 / 3000 in bf16 mode, 64 / 3000
    in fp32 mode), duplicate and overlapping segments, rows of no segment; fp32 and bf16 frames; both losses."""
    m, sd = _model(n_in, C, pos, prec, seed=C + n_in)
    bounds = {64: 64, 320: 128, 3000: 256} if prec == "bf16" else {64: 64, 3000: 128}
    for max_len, Ts in bounds.items():
        cand = [1, 2, 16, 17, Ts - 16, Ts - 15, Ts, Ts + 1, 2 * Ts - 32, 2 * Ts - 31, 3000, max_len]
        lengths = sorted({L for L in cand if L <= max_len})
        ss, se, F = _segments(lengths, seed=max_len + C)
        assert _plan(m, len(ss), max_len) == (TILE, Ts)
        streams = _streams(F, n_in, seed=max_len)
        for x_dtype in ((torch.float32, torch.bfloat16) if prec == "bf16" else (torch.float32,)):
            for kind in ("L1", "confL1"):
                _check_against_reference(m, sd, streams, ss, se, max_len, prec, pos, x_dtype, kind)


@pytest.mark.parametrize("L", [64, 200, 256, 300])
def test_equals_dense_training(L):
    """S segments of one length L against the materialised (S, L) windows with lengths = L (no pad frames: the same
    semantics).  Masked predictions bit-identical; loss and gradients equal up to the fp32 summation order."""
    m, _ = _model(24, 30, False, "bf16", seed=3)
    S = 37
    F = 4000
    streams = _on_dev(_streams(F, 24, seed=L))
    rng = np.random.default_rng(L)
    ss = rng.integers(0, F - L, size=S).astype(np.int64)
    se = ss + L
    assert _plan(m, S, L)[0] == TILE
    idx = torch.from_numpy(ss)[:, None] + torch.arange(L)[None, :]
    batch = {"input_kp": streams["input_kp"][idx.to(DEV)], "target_kp": streams["target_kp"][idx.to(DEV)],
             "target_conf": streams["target_conf"][idx.to(DEV)], "n_frames": torch.full((S,), L, dtype=torch.int64)}
    for kind in ("L1", "confL1"):
        lu, gu, pu = b2h.forward_backward_utterances(m, streams, torch.from_numpy(ss), torch.from_numpy(se), max_len=L,
                                                     loss=kind, want_pred=True)
        ld, gd, pd = b2h.forward_backward(m, batch, loss=kind, want_pred=True)
        assert _tc_status() == 0
        if L <= 256:      # one sub-window per segment, the dense kernel's geometry: the same arithmetic on every row
            assert torch.equal(pu, pd), (L, kind, float((pu - pd).abs().max()))
        else:             # the plan cuts 300 frames into three 128-frame sub-windows, the dense kernel into two of 256
            assert oracle.rel_err(pu.cpu().numpy(), pd.cpu().numpy()) <= 1e-6, (L, kind)
        assert abs(float(lu) - float(ld)) <= 1e-6 * abs(float(ld)), (L, kind, float(lu), float(ld))
        assert oracle.rel_err(gu.cpu().numpy(), gd.cpu().numpy()) <= 5e-5, (L, kind)


def _state(m, opt):
    st = opt._group_state(0, opt.param_groups[0], m)
    return (m.flat_parameters().clone(), st["m"].clone(), st["v"].clone(), st["step_dev"].clone(),
            m.packed_weights().clone())


@pytest.mark.parametrize("prec", ["bf16", "fp32"])
def test_fused_step_equals_forward_backward_plus_adam(prec):
    lr, b1 = 1e-3, 0.9
    ma, _ = _model(24, 30, False, prec, seed=5)
    mb, _ = _model(24, 30, False, prec, seed=5)
    oa, ob = b2h.FusedAdam(ma.parameters(), lr=lr), b2h.FusedAdam(mb.parameters(), lr=lr)
    ss, se, F = _segments([30, 195, 600, 77, 256, 1], seed=9)
    streams = _on_dev(_streams(F, 24, seed=9))
    assert _plan(ma, len(ss), 600) == (TILE, 256 if prec == "bf16" else 128)
    sa = oa._group_state(0, oa.param_groups[0], ma)
    for t in (1, 2, 3):
        before = int(sa["step_dev"])
        la = b2h.fused_train_step_utterances(ma, streams, ss, se, oa, max_len=600, loss="confL1")
        lb, g = b2h.forward_backward_utterances(mb, streams, ss, se, max_len=600, loss="confL1")
        ob.step(flat_grads=g)
        assert _tc_status() == 0
        sb = ob._group_state(0, ob.param_groups[0], mb)
        assert int(sa["step_dev"]) == before + 1 == t and sa["step"] == t
        assert abs(float(la) - float(lb)) <= 1e-6 * abs(float(lb))
        pa, pb = ma.flat_parameters(), mb.flat_parameters()
        rms = float(sb["m"].pow(2).mean().sqrt())
        assert float((sa["m"] - sb["m"]).abs().max()) <= 1e-5 * rms + 1e-30
        # the two paths sum the gradient partials in different orders: elements far below the rms carry relative noise
        vref = sb["v"]
        assert float(((sa["v"] - vref).abs() / (vref + float(vref.pow(2).mean().sqrt()))).max()) <= 1e-5
        p_tol = torch.finfo(torch.float32).eps * pb.abs() + 1e-4 * lr / (1.0 - b1 ** t)
        assert bool(((pa - pb).abs() <= p_tol).all()), (prec, t, float((pa - pb).abs().max()))
    # the packed weights the step scattered are fresh: a forward now equals one after a forced re-pack
    off = torch.from_numpy(np.array([0, 300, F], dtype=np.int64))
    y1 = ma.predict_utterances(streams["input_kp"], off)
    ma.mark_packed_stale()
    y2 = ma.predict_utterances(streams["input_kp"], off)
    assert torch.equal(y1, y2)


def test_bad_segments_make_the_step_a_no_op():
    m, _ = _model(24, 30, False, "bf16", seed=6)
    opt = b2h.FusedAdam(m.parameters(), lr=1e-3)
    ss, se, F = _segments([40, 120, 64], seed=2)
    streams = _on_dev(_streams(F, 24, seed=2))
    b2h.fused_train_step_utterances(m, streams, ss, se, opt, max_len=128)
    assert _tc_status() == 0
    good_s, good_e = torch.from_numpy(ss).to(DEV), torch.from_numpy(se).to(DEV)
    g0, g1 = int(ss[0]), int(ss[1])
    bads = {"L = 0": (0, g0, g0), "end < start": (0, g0, g0 - 1), "end > F": (2, F - 10, F + 1), "L > max_len": (1, g1, g1 + 129),
            "start < 0": (0, -1, 10)}
    for name, (i, a, e) in bads.items():
        s_s, s_e = good_s.clone(), good_e.clone()
        s_s[i], s_e[i] = a, e
        before = _state(m, opt)
        loss = b2h.fused_train_step_utterances(m, streams, s_s, s_e, opt, max_len=128)
        assert _tc_status() == BAD_SEGMENTS, name
        assert torch.isnan(loss).item(), name
        after = _state(m, opt)
        for a, b in zip(before, after):
            assert torch.equal(a, b), name
    runner = UtteranceTrainStepRunner(m, opt, streams, len(ss), 128)
    runner.load({"seg_start": good_s, "seg_end": good_e.clone().fill_(0)})
    runner.step()
    with pytest.raises(_lib.B2HError, match="tc_status=81"):
        runner.check_status()
    runner.load((good_s, good_e))
    runner.step()
    runner.check_status()


def _segment_lists(F, S, max_len, n, seed):
    rng = np.random.default_rng(seed)
    out = []
    for _ in range(n):
        L = rng.integers(1, max_len + 1, size=S)
        a = rng.integers(0, F - max_len, size=S)
        out.append((torch.from_numpy(a.astype(np.int64)), torch.from_numpy((a + L).astype(np.int64))))
    return out


def test_runner_graph_replay_equals_eager_steps():
    S, max_len, F = 24, 300, 5000
    streams = _on_dev(_streams(F, 24, seed=4), torch.bfloat16)
    lists = _segment_lists(F, S, max_len, 6, seed=4)
    m1, _ = _model(24, 30, False, "bf16", seed=8)
    m2, _ = _model(24, 30, False, "bf16", seed=8)
    o1, o2 = b2h.FusedAdam(m1.parameters(), lr=1e-3), b2h.FusedAdam(m2.parameters(), lr=1e-3)
    assert _plan(m1, S, max_len) == (TILE, 128)      # three 128-frame sub-windows: 384 rows, two of 256: 512
    runner = UtteranceTrainStepRunner(m1, o1, streams, S, max_len, loss="L1", n_slots=2)
    runner.load(lists[0], 0)
    runner.load(lists[1], 1)
    runner.capture(n_steps=2)
    losses = []
    for k in range(0, 6, 2):
        runner.load_staged(runner.host_stage(lists[k]), 0)
        runner.load(lists[k + 1], 1)
        runner.replay()
        torch.cuda.synchronize()
        losses += [float(runner.loss[0]), float(runner.loss[1])]
    runner.finish()
    ref = [float(b2h.fused_train_step_utterances(m2, streams, a, e, o2, max_len=max_len)) for a, e in lists]
    assert _tc_status() == 0
    assert losses == ref
    s1, s2 = o1._group_state(0, o1.param_groups[0], m1), o2._group_state(0, o2.param_groups[0], m2)
    assert torch.equal(m1.flat_parameters(), m2.flat_parameters())
    assert torch.equal(s1["m"], s2["m"]) and torch.equal(s1["v"], s2["v"])
    assert int(s1["step_dev"]) == int(s2["step_dev"]) == 6


def test_runner_pipelined_steps_equal_eager_steps():
    S, max_len, F = 16, 200, 3000
    streams = _on_dev(_streams(F, 24, seed=12))
    lists = _segment_lists(F, S, max_len, 4, seed=12)
    m1, _ = _model(24, 30, False, "fp32", seed=2)
    m2, _ = _model(24, 30, False, "fp32", seed=2)
    o1, o2 = b2h.FusedAdam(m1.parameters(), lr=1e-3), b2h.FusedAdam(m2.parameters(), lr=1e-3)
    runner = UtteranceTrainStepRunner(m1, o1, streams, S, max_len, loss="confL1", n_slots=2)
    losses = list(pipelined_steps(runner, [runner.host_stage(l) for l in lists]))
    runner.finish()
    ref = [float(b2h.fused_train_step_utterances(m2, streams, a, e, o2, max_len=max_len, loss="confL1")) for a, e in lists]
    assert losses == ref
    assert torch.equal(m1.flat_parameters(), m2.flat_parameters())


def test_one_hour_utterance():
    """One segment of 108 000 frames (1 h at 30 fps) and 255 short ones in one step, against the float64 reference."""
    m, sd = _model(24, 30, False, "bf16", seed=1)
    rng = np.random.default_rng(1)
    lengths = [108000] + [int(v) for v in rng.integers(30, 601, size=255)]
    ss, se, F = _segments(lengths, seed=1)
    ss, se = ss[:256], se[:256]
    assert _plan(m, 256, 108000) == (TILE, 256)
    # (the masked prediction would be 256 x 108 000 rows: the loss and the gradients are checked)
    _check_against_reference(m, sd, _streams(F, 24, seed=1), ss, se, 108000, "bf16", False, torch.float32, "L1",
                             want_pred=False)
