"""CPU tier: validation on segments (b2h_validate_utterances) without a GPU -- the argument checks, the plan's family and
sub-window length (the forward's family rule, the training's sizing), the forward and training plans unchanged beside it,
and the workspace query against the table, the segment pairs and the per-sub-window sums."""
import ctypes

import numpy as np
import pytest

from hand_pose_sl_b200 import _lib

OK, EINVAL, ESHAPE, EALIGN, EWORKSPACE = 0, -1, -2, -3, -6
NONE, TILE, WIDE = 0, 2, 4
BF16, FP32, FFMA = _lib.PRECISIONS["bf16"], _lib.PRECISIONS["fp32"], _lib.PRECISIONS["fp32-ffma"]
SERVED = "segments are validated by the utterance forward"


def _vplan(S, L, C=30, prec=BF16, n_in=24, pos_emb=0):
    ts = ctypes.c_int(-1)
    k = _lib.load().b2h_validate_utterances_plan(S, L, n_in, C, pos_emb, prec, ctypes.byref(ts))
    return k, ts.value


def _tplan(S, L, C=30, prec=BF16, n_in=24, pos_emb=0):
    ts = ctypes.c_int(-1)
    k = _lib.load().b2h_train_utterances_plan(S, L, n_in, C, pos_emb, prec, ctypes.byref(ts))
    return k, ts.value


def _fplan(F, S, C=30, prec=BF16, n_in=24, pos_emb=0):
    ts = ctypes.c_int(-1)
    k = _lib.load().b2h_utterances_plan(F, S, n_in, C, pos_emb, prec, ctypes.byref(ts))
    return k, ts.value


def _count(L, Ts):
    return _lib.load().b2h_utterance_subwindows(L, Ts, 0, None)


# ---------------------------------------------------------------------------------------------------- argument checks
def _call(**over):
    keep = []

    def p(nbytes, off=0):
        a = np.zeros(nbytes + 128, dtype=np.uint8)
        keep.append(a)
        return ctypes.c_void_p(a.ctypes.data + (-a.ctypes.data) % 64 + off)

    F, S = 100, 3
    args = dict(frames=p(F * 24 * 4), x_dtype=0, target=p(F * 168), conf=p(F * 84), n_frames=F, seg_start=p(8 * S),
                seg_end=p(8 * S), n_seg=S, max_len=40, params=p(4 * 20000), packed=p(1 << 16), seg_loss=p(4 * S), loss=p(64),
                n_in=24, C=30, pos_emb=0, loss_kind=0, precision=BF16, ws=p(1 << 16), ws_bytes=1 << 16, stream=None)
    for k, v in over.items():
        args[k] = p(64, v[1]) if isinstance(v, tuple) and v[0] == "misaligned" else v
    return _lib.load().b2h_validate_utterances(*args.values())


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
    (dict(C=257), ESHAPE, "unsupported geometry n_in=24 C=257"),
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
    (dict(seg_loss=("misaligned", 2)), EALIGN, "4-byte aligned"),
    (dict(loss=("misaligned", 2)), EALIGN, "4-byte aligned"),
    (dict(ws=("misaligned", 8)), EALIGN, "16-byte aligned"),
    (dict(C=33, precision=FP32), ESHAPE, SERVED),
    (dict(n_in=48, precision=FP32), ESHAPE, SERVED),
    (dict(precision=FFMA), ESHAPE, SERVED),
    (dict(ws_bytes=64), EWORKSPACE, "workspace 64 B <"),
]


@pytest.mark.parametrize("over,code,fragment", _ARGS)
def test_argument_checks(over, code, fragment):
    """Every refusal happens on the host before anything is enqueued, so host buffers exercise all of them."""
    rc = _call(**over)
    assert rc == code, (over, rc, _lib.last_error())
    msg = _lib.last_error()
    assert msg.startswith("b2h_validate_utterances:") and fragment in msg, msg


def test_refusal_names_what_is_served():
    assert _call(precision=FFMA) == ESHAPE
    msg = _lib.last_error()
    assert "bf16 mode for conv_channels <= 256" in msg and "fp32 mode for conv_channels <= 32" in msg and "fp32-ffma" in msg


def test_seg_loss_is_optional():
    """seg_loss_out is nullable: with the workspace too small the call gets as far as the workspace check (no launch)."""
    assert _call(seg_loss=None, ws_bytes=64) == EWORKSPACE


# ---------------------------------------------------------------------------------------------------- the plan
def test_plan_family():
    """Tile where the forward's tile kernel fits (bf16 C <= 64, fp32 mode C <= 32), else wide in bf16 mode up to C = 256."""
    for C in (1, 16, 30, 32, 48):
        for prec in ((BF16, FP32) if C <= 32 else (BF16,)):
            for L in (1, 64, 65, 128, 129, 256, 257, 600, 108000):
                assert _vplan(9, L, C=C, prec=prec)[0] == TILE, (C, prec, L)
    for L in (64, 100, 128):
        assert _vplan(9, L, C=64) == (TILE, 64 if L == 64 else 128)
    assert _vplan(9, 600, C=64) == (WIDE, 256)            # the 256-frame tile of C = 64 exceeds shared memory
    assert _vplan(9, 600, C=64, n_in=16) == (TILE, 256)
    for C in (65, 128, 200, 256):
        assert _vplan(9, 64, C=C) == (WIDE, 64)
        for L in (1, 100, 257, 600, 108000):
            assert _vplan(9, L, C=C)[0] == WIDE, (C, L)
    for C in (33, 48, 64, 256):
        assert _vplan(9, 100, C=C, prec=FP32) == (NONE, 0)
    assert _vplan(9, 100, prec=FFMA) == (NONE, 0)
    assert _vplan(9, 100, n_in=48) == (TILE, 128) and _vplan(9, 100, n_in=48, prec=FP32) == (NONE, 0)
    assert _vplan(9, 100, C=257) == (NONE, 0) and _vplan(0, 100) == (NONE, 0) and _vplan(9, 0) == (NONE, 0)


@pytest.mark.parametrize("C,prec", [(30, BF16), (30, FP32), (256, BF16)])
def test_plan_sub_window_length(C, prec):
    """Ts is the menu entry whose family computes the fewest MMA rows for a segment of max_len frames (tile: Ts rows per
    sub-window; wide: 256 / floor(258 / (Ts + 2))), ties to the longer Ts -- around every cut."""
    tile = C <= 32

    def rows(L, Ts):
        return (Ts if tile else 256.0 / (258 // (Ts + 2))) * _count(L, Ts)

    for L in (1, 63, 64, 65, 127, 128, 129, 255, 256, 257, 320, 321, 480, 481, 600, 2000, 108000):
        got = _vplan(11, L, C=C, prec=prec)
        r = {Ts: rows(L, Ts) for Ts in (256, 128, 64)}
        best = None
        for Ts in (256, 128, 64):
            if best is None or r[Ts] < r[best]:
                best = Ts
        assert got == (TILE if tile else WIDE, best), (L, r, got)
    if tile:
        assert [_vplan(3, L, prec=prec)[1] for L in (64, 65, 128, 129, 256, 257)] == [64, 128, 128, 256, 256, 128]


def test_forward_and_train_plans_unchanged():
    """The forward and train plan queries return their old values for the same arguments."""
    assert [_tplan(3, L) for L in (64, 65, 128, 129, 256, 257, 600, 108000)] == \
        [(TILE, 64), (TILE, 128), (TILE, 128), (TILE, 256), (TILE, 256), (TILE, 128), (TILE, 256), (TILE, 256)]
    assert _tplan(3, 3000, prec=FP32) == (TILE, 128) and _tplan(4, 100, C=64) == (NONE, 0)
    assert _tplan(4, 100, prec=FFMA) == (NONE, 0)
    assert _fplan(108000, 1) == (TILE, 256) and _fplan(108000, 1, C=256) == (WIDE, 256)
    assert _fplan(64 * 50, 50, C=256) == (WIDE, 64) and _fplan(976205, 5000) == (TILE, 256)
    assert _fplan(100, 3, prec=FFMA) == (NONE, 0) and _fplan(100, 3, C=64, prec=FP32) == (NONE, 0)


# ---------------------------------------------------------------------------------------------------- workspace
@pytest.mark.parametrize("C", [30, 256])
def test_workspace_query(C):
    """The table (count + max_sub int4), the prefix sums, max_sub {segment, length} int2 and max_sub float sums, with
    max_sub = S * n(max_len) sub-windows of the plan's Ts; S up to 5 000, max_len up to 108 000."""
    lib = _lib.load()
    for S in (1, 7, 128, 5000):
        for L in (1, 64, 257, 600, 3000, 108000):
            k, Ts = _vplan(S, L, C=C)
            max_sub = S * _count(L, Ts)
            pairs = (16 * (1 + max_sub) + 4 * (S + 1) + 15) // 16 * 16
            want = (pairs + 8 * max_sub + 4 * max_sub + 255) // 256 * 256
            assert lib.b2h_validate_utterances_workspace_bytes(S, L, 24, C, 0, BF16) == want, (S, L)
    assert lib.b2h_validate_utterances_workspace_bytes(0, 100, 24, 30, 0, BF16) == ESHAPE and "bad n_seg=0" in _lib.last_error()
    assert lib.b2h_validate_utterances_workspace_bytes(4, 0, 24, 30, 0, BF16) == ESHAPE
    assert lib.b2h_validate_utterances_workspace_bytes(4, 100, 24, 64, 0, FP32) == ESHAPE and SERVED in _lib.last_error()
    assert lib.b2h_validate_utterances_workspace_bytes(4, 100, 24, 30, 0, FFMA) == ESHAPE
    assert lib.b2h_validate_utterances_workspace_bytes(4, 100, 24, 300, 0, BF16) == ESHAPE
