"""CPU tier: training on segments (b2h_train_forward_backward_utterances / b2h_train_step_utterances) without a GPU -- the
argument checks, the plan's sub-window length on both sides of every tie, the workspace query against the bound, and a
float64 proof that the library's cuts (b2h_utterance_subwindows), with rows at or past the segment end zero in every layer
and the criterion on the core rows weighted 1 / (42 L), reproduce the whole sequence's forward, loss and gradients."""
import ctypes

import numpy as np
import pytest

from hand_pose_sl_b200 import _lib

OK, EINVAL, ESHAPE, EALIGN, EWORKSPACE = 0, -1, -2, -3, -6
TILE, NONE = 2, 0
BF16, FP32, FFMA = _lib.PRECISIONS["bf16"], _lib.PRECISIONS["fp32"], _lib.PRECISIONS["fp32-ffma"]


def _plan(S, L, C=30, prec=BF16, n_in=24, pos_emb=0):
    ts = ctypes.c_int(-1)
    k = _lib.load().b2h_train_utterances_plan(S, L, n_in, C, pos_emb, prec, ctypes.byref(ts))
    return k, ts.value


def _count(L, Ts):
    return _lib.load().b2h_utterance_subwindows(L, Ts, 0, None)


def _subwindows(L, Ts):
    lib = _lib.load()
    n = lib.b2h_utterance_subwindows(L, Ts, 0, None)
    out = (ctypes.c_int * 3)()
    cuts = []
    for i in range(n):
        assert lib.b2h_utterance_subwindows(L, Ts, i, out) == n
        cuts.append(tuple(out))
    return cuts


# ---------------------------------------------------------------------------------------------------- argument checks
def _buf(nbytes, off=0):
    a = np.zeros(nbytes + 128, dtype=np.uint8)
    base = (-a.ctypes.data) % 64
    return a, ctypes.c_void_p(a.ctypes.data + base + off)


def _call(is_step, **over):
    keep = []

    def p(nbytes, off=0):
        a, ptr = _buf(nbytes, off)
        keep.append(a)
        return ptr

    F, S = 100, 3
    args = dict(frames=p(F * 24 * 4), x_dtype=0, target=p(F * 168), conf=p(F * 84), n_frames=F, seg_start=p(8 * S),
                seg_end=p(8 * S), n_seg=S, max_len=40, params=p(4 * 20000), packed=p(1 << 16))
    if is_step:
        args.update(m=p(4 * 20000), v=p(4 * 20000), loss=p(64), n_in=24, C=30, pos_emb=0, loss_kind=0, precision=BF16, lr=1e-3,
                    b1=0.9, b2=0.999, eps=1e-8, step=1, step_dev=p(64), lr_dev=None)
    else:
        args.update(grads=p(4 * 20000), loss=p(64), pred=p(S * 40 * 168), n_in=24, C=30, pos_emb=0, loss_kind=0,
                    precision=BF16, step_dev=None)
    args.update(ws=p(1 << 16), ws_bytes=1 << 16, stream=None)
    for k, v in over.items():
        args[k] = p(64, v[1]) if isinstance(v, tuple) and v[0] == "misaligned" else v
    lib = _lib.load()
    return (lib.b2h_train_step_utterances if is_step else lib.b2h_train_forward_backward_utterances)(*args.values())


_ARGS = [
    (dict(frames=None), EINVAL, "null pointer"),
    (dict(seg_start=None), EINVAL, "null pointer"),
    (dict(seg_end=None), EINVAL, "null pointer"),
    (dict(params=None), EINVAL, "null pointer"),
    (dict(packed=None), EINVAL, "null pointer"),
    (dict(ws=None), EINVAL, "null pointer"),
    (dict(loss=None), EINVAL, "null pointer"),
    (dict(x_dtype=5), EINVAL, "bad x_dtype 5"),
    (dict(C=100000), ESHAPE, "unsupported geometry n_in=24 C=100000"),
    (dict(n_seg=0), ESHAPE, "bad n_seg=0"),
    (dict(n_seg=-4), ESHAPE, "bad n_seg=-4"),
    (dict(max_len=0), ESHAPE, "max_len=0"),
    (dict(n_frames=-1), ESHAPE, "n_frames=-1"),
    (dict(precision=9), EINVAL, "bad precision 9"),
    (dict(target=None), EINVAL, "null target"),
    (dict(loss_kind=7), EINVAL, "bad loss_kind 7"),
    (dict(loss_kind=1, conf=None), EINVAL, "confL1 needs scores"),
    (dict(frames=("misaligned", 8)), EALIGN, "16-byte aligned"),
    (dict(target=("misaligned", 4)), EALIGN, "8-byte"),
    (dict(seg_start=("misaligned", 4)), EALIGN, "8-byte"),
    (dict(ws=("misaligned", 8)), EALIGN, "16-byte aligned"),
    (dict(C=64), ESHAPE, "segments are trained by the tile kernel"),
    (dict(C=33), ESHAPE, "segments are trained by the tile kernel"),
    (dict(n_in=48), ESHAPE, "segments are trained by the tile kernel"),
    (dict(precision=FFMA), ESHAPE, "segments are trained by the tile kernel"),
    (dict(ws_bytes=4096), EWORKSPACE, "workspace 4096 B <"),
]


@pytest.mark.parametrize("step", [False, True], ids=["forward_backward", "step"])
@pytest.mark.parametrize("over,code,fragment", _ARGS)
def test_argument_checks(step, over, code, fragment):
    """Every refusal happens on the host before anything is enqueued, so host buffers exercise all of them."""
    rc = _call(step, **over)
    assert rc == code, (over, rc, _lib.last_error())
    who = "b2h_train_step_utterances:" if step else "b2h_train_forward_backward_utterances:"
    msg = _lib.last_error()
    assert msg.startswith(who) and fragment in msg, msg


def test_step_and_forward_backward_specific_checks():
    assert _call(True, m=None) == EINVAL and "null pointer" in _lib.last_error()
    assert _call(True, step=0, step_dev=None) == EINVAL and "step must be >= 1" in _lib.last_error()
    assert _call(True, step_dev=None) == EINVAL and "null step_dev" in _lib.last_error()
    assert _call(False, grads=None) == EINVAL and "null pointer" in _lib.last_error()
    assert _call(False, pred=("misaligned", 8)) == EALIGN and "pred_out" in _lib.last_error()


# ---------------------------------------------------------------------------------------------------- the plan
def _rows(L, Ts):
    return Ts * _count(L, Ts)


@pytest.mark.parametrize("prec,menu", [(BF16, (256, 128, 64)), (FP32, (128, 64))])
def test_plan_takes_fewest_rows_ties_to_longer(prec, menu):
    """The plan's Ts for a segment of max_len frames is the menu entry with the fewest MMA rows (Ts per sub-window), ties to
    the longer Ts -- checked at every max_len up to 2000, so on both sides of every tie."""
    ties = 0
    for L in range(1, 2001):
        rows = {Ts: _rows(L, Ts) for Ts in menu}
        best = min(rows.values())
        want = max(Ts for Ts in menu if rows[Ts] == best)
        ties += sum(1 for Ts in menu if rows[Ts] == best) > 1
        assert _plan(7, L, prec=prec) == (TILE, want), (L, rows)
    assert ties >= 32
    # the tie boundaries of the bf16 menu, spelled out
    if prec == BF16:
        for L, Ts in [(64, 64), (65, 128), (128, 128), (129, 256), (256, 256), (257, 128), (320, 128), (321, 256),
                      (480, 256), (481, 128), (600, 256), (108000, 256)]:
            assert _plan(3, L) == (TILE, Ts), L
    else:
        assert _plan(3, 64, prec=FP32) == (TILE, 64) and _plan(3, 65, prec=FP32) == (TILE, 128)
        assert _plan(3, 3000, prec=FP32) == (TILE, 128)


def test_plan_refusals():
    assert _plan(4, 100, C=64) == (NONE, 0)
    assert _plan(4, 100, C=33) == (NONE, 0)
    assert _plan(4, 100, C=32) == (TILE, 128)
    assert _plan(4, 100, n_in=48) == (NONE, 0)
    assert _plan(4, 100, n_in=32) == (TILE, 128)
    assert _plan(4, 100, n_in=32, pos_emb=1) == (NONE, 0)         # 33 input rows
    assert _plan(4, 100, prec=FFMA) == (NONE, 0)
    assert _plan(0, 100) == (NONE, 0) and _plan(4, 0) == (NONE, 0)
    assert _plan(4, 100, C=100000) == (NONE, 0)


def test_workspace_query():
    lib = _lib.load()
    for S, L, prec in [(1, 1, BF16), (128, 600, BF16), (256, 64, BF16), (256, 108000, BF16), (64, 3000, FP32)]:
        k, Ts = _plan(S, L, prec=prec)
        need = lib.b2h_train_utterances_workspace_bytes(S, L, 24, 30, 0, prec)
        max_sub = S * _count(L, Ts)
        # header, >= 1 gradient + loss partial slice, the table (count + max_sub int4), prefix sums, max_sub {segment, length}
        floor = 1024 + 4 * (19032 + 1) + 16 * (1 + max_sub) + 4 * (S + 1) + 8 * max_sub
        assert need % 256 == 0 and need >= floor, (S, L, need, floor)
        # exactly: the table starts where the tile kernel's training of max_sub windows of Ts frames ends its partials (the
        # dense workspace without its trailing 256 B), the pairs at the 16-byte boundary after the prefix sums
        plan_off = lib.b2h_workspace_bytes(max_sub, Ts, 24, 30, 0, prec) - 256
        pairs = (16 * (1 + max_sub) + 4 * (S + 1) + 15) // 16 * 16
        assert need == (plan_off + pairs + 8 * max_sub + 255) // 256 * 256, (S, L, need)
        assert lib.b2h_train_utterances_workspace_bytes(S + 1, L, 24, 30, 0, prec) >= need
    assert lib.b2h_train_utterances_workspace_bytes(0, 100, 24, 30, 0, BF16) == ESHAPE and "bad n_seg=0" in _lib.last_error()
    assert lib.b2h_train_utterances_workspace_bytes(4, 0, 24, 30, 0, BF16) == ESHAPE
    assert lib.b2h_train_utterances_workspace_bytes(4, 100, 24, 64, 0, BF16) == ESHAPE
    assert "segments are trained by the tile kernel" in _lib.last_error()
    assert lib.b2h_train_utterances_workspace_bytes(4, 100, 24, 30, 0, FFMA) == ESHAPE


# ---------------------------------------------------------------------------------------------------- float64 proof
def _fwd_bwd(Ws, bs, x, valid, tgt, core, w_row):
    """The kernels' arithmetic on a batch of (sub-)windows x (n, R, cin): four convs (padding 2), ReLU on the first three,
    rows with valid == False zero after every layer; criterion sum over rows with core == True of |pred - tgt| * w_row
    (the per-row loss weight); its gradients by hand.  Returns (pred, loss, [dW_l], [db_l]) summed over the batch."""
    a = [x * valid[..., None]]
    z = []
    for l in range(4):
        n, R, _ = a[-1].shape
        p = np.zeros((n, R + 4, a[-1].shape[2]))
        p[:, 2:R + 2] = a[-1]
        zl = bs[l] + sum(p[:, k:k + R] @ Ws[l][:, :, k].T for k in range(5))
        z.append(zl)
        if l < 3:
            a.append(np.maximum(zl, 0.0) * valid[..., None])
    pred = z[3] * valid[..., None]
    r = pred - tgt
    on = (core & valid)[..., None]
    loss = float((np.abs(r) * on * w_row[..., None]).sum())
    dz = np.sign(r) * on * w_row[..., None]
    dW, db = [None] * 4, [None] * 4
    for l in (3, 2, 1, 0):
        n, R, cin = a[l].shape
        p = np.zeros((n, R + 4, cin))
        p[:, 2:R + 2] = a[l]
        dW[l] = np.stack([np.einsum("nro,nri->oi", dz, p[:, k:k + R]) for k in range(5)], axis=2)
        db[l] = dz.sum(axis=(0, 1))
        if l > 0:
            dp = np.zeros((n, R + 4, cin))
            for k in range(5):
                dp[:, k:k + R] += dz @ Ws[l][:, :, k]
            dz = dp[:, 2:R + 2] * ((z[l - 1] > 0) & valid[..., None])
    return pred, loss, dW, db


def test_subwindows_reproduce_the_whole_sequence_training():
    """For every L in 1..700 and every Ts the tile kernel trains: the library's sub-windows of a segment of L frames --
    Ts rows from the first frame, rows at or past L zero in every layer, criterion on the core rows weighted 1 / (42 L) --
    give the whole sequence's masked prediction on every core row, its loss, and (summed over the sub-windows) its weight and
    bias gradients, to 1e-12 in float64.  The weight-gradient sums run over every row of a sub-window, unmasked: context
    rows carry d(loss)/d(activation) of the core rows within the +-8-frame receptive field."""
    rng = np.random.default_rng(11)
    n_in, C, Lmax = 4, 6, 700
    Ws = [rng.standard_normal((C, n_in, 5)) * 0.5] + [rng.standard_normal((C, C, 5)) * 0.3 for _ in range(2)]
    Ws.append(rng.standard_normal((42, C, 5)) * 0.3)
    bs = [rng.standard_normal(w.shape[0]) * 0.1 for w in Ws]
    frames = rng.standard_normal((Lmax, n_in))
    target = rng.standard_normal((Lmax, 42))
    for L in range(1, Lmax + 1):
        w = 1.0 / (42 * L)
        ones = np.ones((1, L), dtype=bool)
        pw, lw, dWw, dbw = _fwd_bwd(Ws, bs, frames[None, :L], ones, target[None, :L], ones, np.full((1, L), w))
        sp, sg = np.abs(pw).max(), max(np.abs(d).max() for d in dWw + dbw)
        for Ts in (64, 128, 256):
            cuts = _subwindows(L, Ts)
            n = len(cuts)
            x = np.zeros((n, Ts, n_in))
            tg = np.zeros((n, Ts, 42))
            valid = np.zeros((n, Ts), dtype=bool)
            core = np.zeros((n, Ts), dtype=bool)
            for i, (start, clo, chi) in enumerate(cuts):
                m = min(Ts, L - start)
                x[i, :m] = frames[start:start + m]
                tg[i, :m] = target[start:start + m]
                valid[i, :m] = True
                core[i, clo:chi] = True
            p, ls, dW, db = _fwd_bwd(Ws, bs, x, valid, tg, core, np.full((n, Ts), w))
            for i, (start, clo, chi) in enumerate(cuts):
                assert np.abs(p[i, clo:chi] - pw[0, start + clo:start + chi]).max() <= 1e-12 * sp, (L, Ts, i)
            assert abs(ls - lw) <= 1e-12 * max(lw, 1e-300), (L, Ts, ls, lw)
            for l in range(4):
                assert np.abs(dW[l] - dWw[l]).max() <= 1e-12 * sg, (L, Ts, l)
                assert np.abs(db[l] - dbw[l]).max() <= 1e-12 * sg, (L, Ts, l)
