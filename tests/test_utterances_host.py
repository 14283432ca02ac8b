"""CPU tier: the forward over packed utterances (b2h_conv_forward_utterances) without a GPU -- its argument checks, the
plan's choice of kernel family and sub-window length, the sub-window bound that sizes its grid and workspace, and a
float64 proof that the library's own cuts (b2h_utterance_subwindows) reproduce the whole-sequence forward in every core."""
import ctypes

import numpy as np
import pytest

from hand_pose_sl_b200 import _lib

OK, EINVAL, ESHAPE, EALIGN, EWORKSPACE = 0, -1, -2, -3, -6
TILE, WIDE, NONE = 2, 4, 0
MENU = (64, 128, 256)


def _plan(n_frames, n_utt, C, prec="bf16", n_in=24, pos_emb=0):
    ts = ctypes.c_int(-1)
    k = _lib.load().b2h_utterances_plan(n_frames, n_utt, n_in, C, pos_emb, _lib.PRECISIONS[prec], ctypes.byref(ts))
    return k, ts.value


def _subwindows(L, Ts):
    lib = _lib.load()
    n = lib.b2h_utterance_subwindows(L, Ts, 0, None)
    assert n >= 0, _lib.last_error()
    out = (ctypes.c_int * 3)()
    cuts = []
    for i in range(n):
        assert lib.b2h_utterance_subwindows(L, Ts, i, out) == n
        cuts.append(tuple(out))
    return cuts


# ---------------------------------------------------------------------------------------------------- argument checks
def _buf(nbytes, off=0):
    """A 64-byte aligned host buffer (kept alive by the returned array) and a pointer `off` bytes into it."""
    a = np.zeros(nbytes + 128, dtype=np.uint8)
    base = (-a.ctypes.data) % 64
    return a, ctypes.c_void_p(a.ctypes.data + base + off)


def _call(**over):
    keep = []

    def p(nbytes, off=0):
        a, ptr = _buf(nbytes, off)
        keep.append(a)
        return ptr

    F, S = 100, 3
    args = dict(frames=p(F * 24 * 4), x_dtype=0, n_frames=F, offsets=p(8 * (S + 1)), n_utt=S, params=p(4 * 20000),
                packed=p(1 << 16), y=p(F * 168), n_in=24, C=30, pos_emb=0, precision=_lib.PRECISIONS["bf16"], out_scale=1.0,
                ws=p(1 << 16), ws_bytes=1 << 16, stream=None)
    for k, v in over.items():
        args[k] = p(64, v[1]) if isinstance(v, tuple) and v[0] == "misaligned" else v
    return _lib.load().b2h_conv_forward_utterances(*args.values())


_ARGS = [
    (dict(frames=None), EINVAL, "null pointer"),
    (dict(offsets=None), EINVAL, "null pointer"),
    (dict(params=None), EINVAL, "null pointer"),
    (dict(packed=None), EINVAL, "null pointer"),
    (dict(y=None), EINVAL, "null pointer"),
    (dict(ws=None), EINVAL, "null pointer"),
    (dict(y=None, x_dtype=5), EINVAL, "null pointer"),
    (dict(x_dtype=5), EINVAL, "bad x_dtype 5"),
    (dict(x_dtype=5, C=100000), EINVAL, "bad x_dtype 5"),
    (dict(C=100000), ESHAPE, "unsupported geometry n_in=24 C=100000"),
    (dict(n_utt=-1), ESHAPE, "bad n_utt=-1"),
    (dict(n_frames=-1), ESHAPE, "bad n_utt=3 n_frames=-1"),
    (dict(n_utt=0, frames=("misaligned", 4)), OK, None),            # nothing to do: succeeds before the alignment test
    (dict(n_utt=0, precision=9), OK, None),
    (dict(frames=("misaligned", 8)), EALIGN, "16-byte aligned"),
    (dict(y=("misaligned", 8)), EALIGN, "16-byte aligned"),
    (dict(packed=("misaligned", 4)), EALIGN, "16-byte aligned"),
    (dict(ws=("misaligned", 8)), EALIGN, "16-byte aligned"),
    (dict(offsets=("misaligned", 4)), EALIGN, "offsets 8-byte aligned"),
    (dict(offsets=("misaligned", 8)), EWORKSPACE, None),           # 8-byte aligned offsets are fine (tiny workspace below)
    (dict(precision=9), EINVAL, "bad precision 9"),
    (dict(precision=9, ws=("misaligned", 8)), EALIGN, "16-byte aligned"),
    (dict(precision=_lib.PRECISIONS["fp32"], C=64), ESHAPE, "utterances are served in bf16 mode"),
    (dict(precision=_lib.PRECISIONS["fp32"], n_in=48), ESHAPE, "utterances are served in bf16 mode"),
    (dict(precision=_lib.PRECISIONS["fp32-ffma"]), ESHAPE, "utterances are served in bf16 mode"),
    (dict(ws_bytes=255), EWORKSPACE, "workspace 255 B <"),
    (dict(ws_bytes=0, precision=_lib.PRECISIONS["fp32-ffma"]), ESHAPE, "utterances are served"),
]


@pytest.mark.parametrize("over,code,fragment", _ARGS)
def test_argument_checks(over, code, fragment):
    """The checks run in check_common's order (null, dtype, geometry, shape, then alignment, precision, workspace), all
    on the host before anything is enqueued, so host buffers exercise every refusal."""
    if over == dict(offsets=("misaligned", 8)):
        over = dict(over, ws_bytes=16)
    rc = _call(**over)
    assert rc == code, (over, rc, _lib.last_error())
    if fragment is not None:
        msg = _lib.last_error()
        assert msg.startswith("b2h_conv_forward_utterances:") and fragment in msg, msg


def test_workspace_query():
    lib = _lib.load()
    bf16, fp32 = _lib.PRECISIONS["bf16"], _lib.PRECISIONS["fp32"]
    assert lib.b2h_utterances_workspace_bytes(1000, 0, 24, 30, 0, bf16) == 256
    assert lib.b2h_utterances_workspace_bytes(1000, 5, 24, 64, 0, fp32) == ESHAPE
    assert "utterances are served" in _lib.last_error()
    assert lib.b2h_utterances_workspace_bytes(1000, 5, 24, 30, 0, _lib.PRECISIONS["fp32-ffma"]) == ESHAPE
    assert lib.b2h_utterances_workspace_bytes(1000, 5, 24, 100000, 0, bf16) == ESHAPE
    assert lib.b2h_utterances_workspace_bytes(-1, 5, 24, 30, 0, bf16) == ESHAPE
    for F, S, C, prec in [(108000, 1, 30, bf16), (1_000_000, 5000, 256, bf16), (500, 40, 30, fp32), (0, 3, 30, bf16)]:
        k, Ts = _plan(F, S, C, "bf16" if prec == bf16 else "fp32")
        need = lib.b2h_utterances_workspace_bytes(F, S, 24, C, 0, prec)
        bound = S + F // (Ts - 32)
        assert need % 256 == 0 and need >= 16 * (1 + bound) + 4 * (S + 1), (F, S, C, need)
        # exactly: the table (count + bound int4) and the prefix sums, rounded to 256 B
        assert need == (16 * (1 + bound) + 4 * (S + 1) + 255) // 256 * 256, (F, S, C, need)


# ---------------------------------------------------------------------------------------------------- the plan
def test_plan_family_and_segment_length():
    # a 1 h clip as one utterance: 256-frame sub-windows, 482 of them, ~1.14 MMA rows per frame
    assert _plan(108000, 1, 30) == (TILE, 256)
    assert _plan(108000, 1, 30, "fp32") == (TILE, 256)
    assert _plan(108000, 1, 256) == (WIDE, 256)
    assert len(_subwindows(108000, 256)) == 482
    # ~5 000 utterances of mean 200 frames: one 256-frame sub-window each (two of 128 compute as many rows; ties go long)
    assert _plan(1_000_000, 5000, 30) == (TILE, 256)
    assert _plan(1_000_000, 5000, 256) == (WIDE, 256)
    # short utterances: 64-frame sub-windows (one 64-row segment each instead of a mostly empty 128- or 256-row tile)
    assert _plan(40 * 100, 100, 30) == (TILE, 64)
    assert _plan(40 * 100, 100, 30, "fp32") == (TILE, 64)
    assert _plan(100 * 100, 100, 30) == (TILE, 128)
    # the wide kernel packs 3 windows of 64 frames into one 256-row tile (85 rows each)
    assert _plan(40 * 100, 100, 256) == (WIDE, 64)
    # C = 64: the tile kernel holds 128-frame windows, the wide kernel serves 256
    assert _plan(100 * 100, 100, 64) == (TILE, 128)
    assert _plan(1000 * 100, 100, 64) == (WIDE, 256)
    assert _plan(1000 * 100, 100, 48) == (TILE, 256)
    # unserved: fp32 mode beyond the tile kernel, the FFMA mode, bad geometry
    assert _plan(10000, 10, 64, "fp32")[0] == NONE
    assert _plan(10000, 10, 30, "fp32", n_in=48)[0] == NONE
    assert _plan(10000, 10, 30, "fp32-ffma") == (NONE, 0)
    assert _plan(10000, 10, 100000) == (NONE, 0)


@pytest.mark.parametrize("seed", range(6))
def test_subwindow_bound(seed):
    """The grid and the workspace are sized for n_utt + n_frames // (Ts - 32) sub-windows: the exact count of seeded
    length mixes (empty, short, around the cuts, long) never exceeds it; n (Ts - 32) + 32 frames are exactly n sub-windows."""
    rng = np.random.default_rng(seed)
    S = int(rng.integers(1, 300))
    kind = seed % 3
    if kind == 0:
        L = rng.integers(0, 40, S)
    elif kind == 1:
        L = rng.integers(30, 601, S)
    else:
        L = np.concatenate([rng.integers(0, 3000, S - 1), [int(rng.integers(5000, 20000))]])
    for Ts in MENU:
        exact = sum(len(_subwindows(int(l), Ts)) for l in L)
        assert exact <= S + int(L.sum()) // (Ts - 32), (Ts, exact)
        for l in L[:50]:
            assert len(_subwindows(int(l), Ts)) <= 1 + int(l) // (Ts - 32)
    for Ts in MENU:
        L1 = 10 * (Ts - 32) + 32
        assert len(_subwindows(L1, Ts)) == 10 and len(_subwindows(L1 + 1, Ts)) == 11


def test_subwindow_query_refusals():
    lib = _lib.load()
    out = (ctypes.c_int * 3)()
    assert lib.b2h_utterance_subwindows(0, 256, 0, None) == 0
    assert lib.b2h_utterance_subwindows(-1, 256, 0, None) == ESHAPE
    assert lib.b2h_utterance_subwindows(100, 32, 0, None) == ESHAPE
    assert lib.b2h_utterance_subwindows(100, 256, 1, out) == EINVAL
    assert lib.b2h_utterance_subwindows(100, 256, 0, out) == 1 and tuple(out) == (0, 0, 100)


# ---------------------------------------------------------------------------------------------------- float64 proof
def _conv_stack(Ws, bs, x, valid):
    """The kernels' arithmetic on a batch of segments: x (n, R, cin) with zero rows around, four convs (padding 2), ReLU
    on the first three, every row with valid == False set to zero after each layer (the epilogues write zeros there)."""
    a = x * valid[..., None]
    for l in range(4):
        n, R, _ = a.shape
        p = np.zeros((n, R + 4, a.shape[2]))
        p[:, 2:R + 2] = a
        z = bs[l] + sum(p[:, k:k + R] @ Ws[l][:, :, k].T for k in range(5))
        a = (np.maximum(z, 0.0) if l < 3 else z) * valid[..., None]
    return a


def test_cores_reproduce_the_whole_sequence():
    """For every L in 1..1200 and every Ts of the menu: the library's sub-windows' cores partition [0, L), and the conv
    stack on each sub-window -- Ts rows from its first frame, rows at or past the utterance end zero in every layer, as
    the kernels run it -- equals the whole sequence's forward on its core rows to 1e-12 (float64).  The receptive field is
    +-8 frames and every interior cut has >= 16 real frames of context."""
    rng = np.random.default_rng(7)
    n_in, C, Lmax = 4, 6, 1200
    Ws = [rng.standard_normal((C, n_in, 5)) * 0.5] + [rng.standard_normal((C, C, 5)) * 0.3 for _ in range(2)]
    Ws.append(rng.standard_normal((42, C, 5)) * 0.3)
    bs = [rng.standard_normal(w.shape[0]) * 0.1 for w in Ws]
    frames = rng.standard_normal((Lmax, n_in))
    for L in range(1, Lmax + 1):
        whole = _conv_stack(Ws, bs, frames[None, :L], np.ones((1, L), dtype=bool))[0]
        scale = np.abs(whole).max()
        for Ts in MENU:
            cuts = _subwindows(L, Ts)
            covered = np.zeros(L, dtype=int)
            x = np.zeros((len(cuts), Ts, n_in))
            valid = np.zeros((len(cuts), Ts), dtype=bool)
            for w, (start, clo, chi) in enumerate(cuts):
                n = min(Ts, L - start)
                assert 0 <= start and 0 <= clo < chi <= n <= Ts
                assert clo == 0 or clo >= 16, (L, Ts, w)                 # context before an interior cut
                assert start + chi == L or n - chi >= 16, (L, Ts, w)      # ... and after it
                covered[start + clo:start + chi] += 1
                x[w, :n] = frames[start:start + n]
                valid[w, :n] = True
            assert (covered == 1).all(), (L, Ts)
            got = _conv_stack(Ws, bs, x, valid)
            for w, (start, clo, chi) in enumerate(cuts):
                err = np.abs(got[w, clo:chi] - whole[start + clo:start + chi]).max()
                assert err <= 1e-12 * scale, (L, Ts, w, err)
