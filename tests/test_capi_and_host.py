"""CPU tier: the C-ABI library loads and exports every symbol include/b2h.h declares; geometry queries;
host-side logic of the drop-in modules (no compute call happens without a GPU)."""
import ctypes
import os
import pickle
import random
import re

import numpy as np
import pytest
import torch
from hypothesis import given, settings, strategies as st

import b2h_oracle as oracle
import hand_pose_sl_b200 as b2h
from hand_pose_sl_b200 import _lib

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _header_symbols():
    txt = open(os.path.join(ROOT, "include", "b2h.h")).read()
    txt = re.sub(r"/\*.*?\*/", "", txt, flags=re.S)
    return sorted(set(re.findall(r"\b(b2h_[a-z0-9_]+)\s*\(", txt)))


def test_library_exports_every_declared_symbol():
    lib = ctypes.CDLL(_lib.LIB_PATH)
    syms = _header_symbols()
    assert len(syms) >= 20
    for s in syms:
        assert hasattr(lib, s), f"{s} declared in include/b2h.h but not exported"
    assert sorted(_lib.exported_symbols()) == syms       # the ctypes table binds exactly the header


def test_geometry_queries():
    assert _lib.param_count(24, 30, 0) == 19032          # SURVEY.md §0.2
    assert _lib.param_count(24, 256, 0) == 740650        # SURVEY.md §8a
    assert _lib.param_count(24, 30, 1) == 19032 + 30 * 5
    off = [_lib.param_offset(24, 30, 0, l, b) for l in (1, 2, 3, 4) for b in (0, 1)]
    sizes = [30 * 24 * 5, 30, 30 * 30 * 5, 30, 30 * 30 * 5, 30, 42 * 30 * 5, 42]
    assert off == list(np.cumsum([0] + sizes[:-1]))
    assert _lib.packed_bytes(24, 30, 0) > 0 and _lib.packed_bytes(24, 30, 0) % 128 == 0
    lib = _lib.load()
    assert lib.b2h_param_count(24, 100000, 0) < 0 and "unsupported geometry" in _lib.last_error()
    assert lib.b2h_supported(64, 24, 30, 0, _lib.FP32) == 1
    assert lib.b2h_supported(64, 24, 30, 0, _lib.BF16) == 1
    assert lib.b2h_supported(100000, 24, 30, 0, _lib.FP32) == 0
    # forward-only coverage is wider: bf16 inference runs conv_channels up to 256 and windows up to 1024 frames
    assert lib.b2h_forward_supported(64, 24, 256, 0, _lib.BF16) == 1
    assert lib.b2h_forward_supported(200, 24, 256, 0, _lib.BF16) == 1
    assert lib.b2h_forward_supported(200, 24, 30, 0, _lib.BF16) == 1
    assert lib.b2h_forward_supported(1000, 24, 30, 0, _lib.BF16) == 1
    assert lib.b2h_forward_supported(1000, 24, 256, 0, _lib.BF16) == 0
    assert lib.b2h_supported(64, 24, 256, 0, _lib.BF16) == 1          # wide training kernels (bf16 mode)
    assert lib.b2h_supported(64, 24, 256, 0, _lib.FP32) == 0          # fp32 mode: no training kernel at C = 256
    assert lib.b2h_forward_supported(64, 24, 256, 0, _lib.FP32) == 1


def test_gradient_partial_slot_layout_is_a_bijection():
    """The tensor-core train kernel reads its weight-gradient accumulators out as [k][ci/4][co][4] slots (coalesced
    stores); the Adam tail maps slots back to flat parameter indices.  Host-side check of that map for every geometry
    the kernel serves (incl. pos_emb's 25 input channels and C = 32 where cin == the padded reduction)."""
    lib = _lib.load()
    for n_in, C, pe in ((24, 30, 0), (24, 30, 1), (24, 32, 0), (24, 16, 0), (16, 30, 0), (24, 64, 0), (24, 256, 0), (24, 1, 0)):
        assert lib.b2h_gp_layout_check(n_in, C, pe) == 0, (n_in, C, pe)
    assert lib.b2h_workspace_bytes(256, 64, 24, 30, 0, _lib.BF16) > 1024 + 128 * 19032 * 4


def test_kernel_choice_pins_the_tensor_core_paths():
    """The dispatch of b2h_conv_forward / the train entry points goes through b2h_kernel_choice: in bf16 mode every
    BASELINE config, the reference default crop (200 frames) and the wide variant run tcgen05 kernels -- no silent
    FFMA fallback -- and fp32 mode runs the split-operand tcgen05 kernel wherever it fits."""
    lib = _lib.load()
    NONE, FFMA, TILE, ROWSPACE, WIDE, WIDE_TRAIN = 0, 1, 2, 3, 4, 5
    fwd = lambda T, C, prec, pe=0: lib.b2h_kernel_choice(T, 24, C, pe, prec, 0)
    trn = lambda T, C, prec, pe=0: lib.b2h_kernel_choice(T, 24, C, pe, prec, 1)
    for T in (1, 9, 64, 100, 126, 128, 129, 200, 256):
        assert fwd(T, 30, _lib.BF16) == TILE and trn(T, 30, _lib.BF16) == TILE, T
        # fp32 mode = the same tcgen05 tile kernel with bf16 high/low operand pairs (3 MMAs per product); its doubled
        # activation buffers fit 128-frame segments, longer windows train as overlapping 128-frame sub-windows with real
        # context frames at the cuts; FFMA is the explicit arbiter mode
        assert fwd(T, 30, _lib.FP32) == TILE and trn(T, 30, _lib.FP32) == TILE, T
        assert fwd(T, 30, _lib.FP32_FFMA) == FFMA and trn(T, 30, _lib.FP32_FFMA) == FFMA, T
    assert fwd(64, 64, _lib.FP32) == FFMA and trn(64, 64, _lib.FP32) == FFMA                # split covers C <= 32
    assert fwd(100, 30, _lib.BF16, 1) == TILE and trn(100, 30, _lib.BF16, 1) == TILE        # pos_emb: 25 input channels
    assert fwd(64, 64, _lib.BF16) == TILE and trn(64, 64, _lib.BF16) == WIDE_TRAIN          # C > 32 trains on the wide tcgen05 kernels
    assert fwd(200, 64, _lib.BF16) == ROWSPACE                                              # tile does not fit smem
    assert fwd(257, 30, _lib.BF16) == ROWSPACE and fwd(1000, 30, _lib.BF16) == ROWSPACE
    # row space beyond 256 frames: C <= 48 up to T = 640, C <= 32 up to T = 1024, at any batch; beyond that one window's
    # buffers and the weights do not fit in shared memory
    assert fwd(640, 48, _lib.BF16) == ROWSPACE and fwd(1024, 30, _lib.BF16) == ROWSPACE
    assert fwd(257, 64, _lib.BF16) == NONE and fwd(641, 48, _lib.BF16) == NONE
    assert trn(257, 30, _lib.BF16) == TILE and trn(1000, 30, _lib.BF16) == TILE and trn(300, 30, _lib.FP32) == TILE   # sub-windows
    for C in (80, 96, 128, 256):
        for T in (64, 126, 200, 256):
            assert fwd(T, C, _lib.BF16) == WIDE, (T, C)
    assert fwd(300, 256, _lib.BF16) == NONE and fwd(2000, 30, _lib.BF16) == NONE
    for C in (33, 64, 80, 128, 256):
        for T in (9, 64, 126, 200, 256):
            assert trn(T, C, _lib.BF16) == WIDE_TRAIN, (T, C)
    assert trn(300, 256, _lib.BF16) == NONE and trn(64, 256, _lib.FP32) == NONE             # fp32 mode: 396 KB of activations
    # bf16 training falls back to FFMA (unrounded fp32 operands) exactly where no tensor-core training kernel fits and FFMA's
    # shared memory does: 16 input channels, no positional row, C = 33..36, T = 257..264 (include/b2h.h, DESIGN §1)
    on_ffma = {(n_in, pe, C, T) for n_in in (16, 24) for pe in (0, 1) for C in range(30, 50) for T in range(250, 272)
               if lib.b2h_kernel_choice(T, n_in, C, pe, _lib.BF16, 1) == FFMA}
    assert on_ffma == {(16, 0, C, T) for C in range(33, 37) for T in range(257, 265)}
    assert all(lib.b2h_supported(T, 16, C, 0, _lib.BF16) == 1 for C in (33, 36) for T in (257, 264))
    assert lib.b2h_kernel_choice(257, 24, 33, 0, _lib.BF16, 1) == NONE and lib.b2h_kernel_choice(265, 16, 33, 0, _lib.BF16, 1) == NONE
    assert fwd(64, 256, _lib.FP32) == FFMA
    assert lib.b2h_kernel_choice(64, 24, 30, 0, 7, 0) == NONE                                # bad precision
    for T, C in ((64, 30), (200, 30), (64, 256), (300, 256)):
        assert lib.b2h_forward_supported(T, 24, C, 0, _lib.BF16) == int(fwd(T, C, _lib.BF16) != NONE)
    # a shape without a training kernel is refused with a message that names the limits (no launch is attempted)
    import ctypes
    buf = (ctypes.c_char * 4096)()
    ptr = ctypes.c_void_p((ctypes.addressof(buf) + 255) // 256 * 256)
    rc = lib.b2h_train_forward_backward(ptr, 0, ptr, None, ptr, ptr, ptr, ptr, ptr, None, 4, 64, 24, 256, 0, _lib.LOSS_L1, _lib.FP32,
                                        None, ptr, 1 << 20, None)
    assert rc == -2 and "no training kernel for conv_channels=256" in _lib.last_error()


# Argument names of the entry points whose checks the table below pins, in C-ABI order (include/b2h.h).
_ABI_ARGS = {
    "b2h_conv_forward": "x x_dtype params packed lengths y B T n_in C pos_emb precision apply_mask out_scale stream",
    "b2h_conv_forward_windows": "x x_dtype n_frames win_start win_end pad_mode params packed lengths y B T n_in C pos_emb "
                                "precision apply_mask out_scale stream",
    "b2h_train_forward_backward": "x x_dtype target conf lengths params packed grads loss pred B T n_in C pos_emb loss_kind "
                                  "precision step_dev ws ws_bytes stream",
    "b2h_train_forward_backward_windows": "x x_dtype target conf n_frames win_start win_end pad_mode lengths params packed "
                                          "grads loss pred B T n_in C pos_emb loss_kind precision step_dev ws ws_bytes stream",
    "b2h_conv_backward": "x x_dtype d_y params packed grads B T n_in C pos_emb precision ws ws_bytes stream",
    "b2h_train_step": "x x_dtype target conf lengths params packed m v loss B T n_in C pos_emb loss_kind precision lr b1 b2 "
                      "eps step step_dev lr_dev ws ws_bytes stream",
    "b2h_train_step_windows": "x x_dtype target conf n_frames win_start win_end pad_mode lengths params packed m v loss B T "
                              "n_in C pos_emb loss_kind precision lr b1 b2 eps step step_dev lr_dev ws ws_bytes stream",
    "b2h_train_step_dp": "x x_dtype target conf lengths params packed m v loss B T n_in C pos_emb loss_kind precision lr b1 "
                         "b2 eps step_dev epoch_dev lr_dev sym peers mc rank world grad_scale ws ws_bytes stream",
}
_FWD = ("b2h_conv_forward", "b2h_conv_forward_windows")
_VIEWS = ("b2h_conv_forward_windows", "b2h_train_forward_backward_windows", "b2h_train_step_windows")
_TRAIN = tuple(n for n in _ABI_ARGS if n not in _FWD)
_LOSS = tuple(n for n in _TRAIN if n != "b2h_conv_backward")      # the entry points that compute the criterion
_ALL = tuple(_ABI_ARGS)
OK, EINVAL, ESHAPE, EALIGN, EWORKSPACE = 0, -1, -2, -3, -6

# (entry points, overrides of the defaults, expected code, fragment of b2h_last_error()).  Every case is refused (or, for
# B == 0 in the forward, accepted) before anything is launched, so host buffers stand in for device memory.  Cases that
# are bad in two ways pin the order of the checks.
_ARG_CASES = [
    (_ALL, dict(x=None), EINVAL, "null pointer"),
    (_ALL, dict(params=None), EINVAL, "null pointer"),
    (_ALL, dict(packed=None), EINVAL, "null pointer"),
    (_FWD, dict(y=None), EINVAL, "null pointer"),
    (_TRAIN, dict(ws=None), EINVAL, "null pointer"),
    (_VIEWS, dict(win_start=None), EINVAL, "null pointer"),
    (("b2h_train_step", "b2h_train_step_windows", "b2h_train_step_dp"), dict(m=None), EINVAL, "null pointer"),
    (("b2h_train_step_dp",), dict(step_dev=None), EINVAL, "null pointer"),
    (("b2h_train_step_dp",), dict(peers=None), EINVAL, "null pointer"),
    (("b2h_train_step_dp",), dict(rank=2), EINVAL, "bad rank/world"),
    (("b2h_conv_backward",), dict(grads=None), EINVAL, "null output"),
    (("b2h_conv_backward",), dict(d_y=None), EINVAL, "null d_y"),
    (("b2h_train_forward_backward", "b2h_train_forward_backward_windows"), dict(loss=None), EINVAL, "null loss_out"),
    (("b2h_train_step", "b2h_train_step_windows"), dict(step=0), EINVAL, "step must be >= 1"),
    (_ALL, dict(x_dtype=5), EINVAL, "bad x_dtype 5"),
    (_ALL, dict(x_dtype=5, C=100000), EINVAL, "bad x_dtype 5"),
    (_VIEWS, dict(pad_mode=7), EINVAL, "bad pad_mode 7"),
    (_VIEWS, dict(pad_mode=7, x_dtype=5), EINVAL, "bad x_dtype 5"),
    (_ALL, dict(C=100000), ESHAPE, "unsupported geometry n_in=24 C=100000"),
    (_ALL, dict(n_in=0, B=-1), ESHAPE, "unsupported geometry"),
    (_ALL, dict(B=-1), ESHAPE, "bad B=-1 T=64"),
    (_ALL, dict(T=0), ESHAPE, "bad B=2 T=0"),
    (_TRAIN, dict(B=0), ESHAPE, "bad B=0 T=64"),
    (_VIEWS, dict(n_frames=-1), ESHAPE, "bad B=2 T=64"),
    (_FWD, dict(B=0, x=1), OK, None),                     # an empty forward succeeds before the alignment test
    (_FWD, dict(apply_mask=1, lengths=None), EINVAL, "apply_mask needs lengths"),
    (_LOSS, dict(target=None), EINVAL, "null target/lengths"),
    (_LOSS, dict(lengths=None), EINVAL, "null target/lengths"),
    (_LOSS, dict(loss_kind=3), EINVAL, "bad loss_kind 3"),
    (_LOSS, dict(loss_kind=1), EINVAL, "confL1 needs scores"),
    (_ALL, dict(x=8), EALIGN, "16-byte aligned"),
    (_FWD, dict(y=8), EALIGN, "16-byte aligned"),
    (_ALL, dict(packed=8), EALIGN, "16-byte aligned"),
    (tuple(n for n in _LOSS if n not in _VIEWS), dict(target=8), EALIGN, "x, target and packed must be 16-byte aligned"),
    (tuple(n for n in _TRAIN if n in _VIEWS), dict(target=4), EALIGN, "target_frames 8-byte"),
    (tuple(n for n in _TRAIN if n in _VIEWS), dict(target=8, conf=4, loss_kind=1, C=256, T=300), ESHAPE,
     "window views are trained on the tensor cores"),
    (("b2h_train_forward_backward_windows",), dict(conf=2, loss_kind=1), EALIGN, "conf_frames 4-byte"),
    (_FWD, dict(x=8, y=None), EINVAL, "null pointer"),
    (_ALL, dict(precision=7), EINVAL, "bad precision 7"),
    (_FWD, dict(precision=7, x=8), EALIGN, "16-byte aligned"),              # forward: alignment before precision
    (_TRAIN, dict(precision=7, x=8), EINVAL, "bad precision 7"),            # training: precision before alignment
    (_LOSS, dict(precision=7, loss_kind=3), EINVAL, "bad precision 7"),
    (("b2h_conv_forward",), dict(C=256, T=300), ESHAPE, "no kernel for C=256, T=300, precision=1"),
    (("b2h_conv_forward_windows",), dict(C=256, T=300), ESHAPE, "window views are served in bf16 mode"),
    (("b2h_conv_forward_windows",), dict(C=64, precision=2), ESHAPE, "materialise the windows"),
    (tuple(n for n in _TRAIN if n not in _VIEWS), dict(C=256, T=300), ESHAPE, "no training kernel for conv_channels=256, T=300"),
    (tuple(n for n in _TRAIN if n in _VIEWS), dict(C=256, T=300), ESHAPE, "window views are trained on the tensor cores"),
    (tuple(n for n in _TRAIN if n in _VIEWS), dict(C=30, precision=2), ESHAPE, "precision=2"),
    (_TRAIN, dict(ws_bytes=64), EWORKSPACE, "workspace 64 B <"),
    (_TRAIN, dict(ws=8), EALIGN, "workspace must be 16-byte aligned"),
    (_TRAIN, dict(ws=8, ws_bytes=64), EWORKSPACE, "workspace 64 B <"),
]


def _abi_call(lib, keep, name, over):
    """Calls entry point `name` with a well-formed bf16 C=30 T=64 batch of 2 (host buffers), changed by `over`.  A pointer
    override is None or a byte offset into its aligned buffer."""
    assert set(over) <= set(_ABI_ARGS[name].split()), (name, over)
    v = ctypes.c_void_p
    bufs = {}

    def buf(key, off=0):
        if key not in bufs:
            keep.append(np.zeros(1 << 16, dtype=np.uint8))
            a = keep[-1].ctypes.data
            bufs[key] = a + (-a) % 256
        return v(bufs[key] + off)

    scalars = dict(x_dtype=_lib.DT_BF16, n_frames=100, pad_mode=_lib.PAD_REPEAT_FIRST, B=2, T=64, n_in=24, C=30, pos_emb=0,
                   precision=_lib.BF16, apply_mask=0, out_scale=1.0, loss_kind=_lib.LOSS_L1, ws_bytes=1 << 30, lr=1e-3,
                   b1=0.9, b2=0.999, eps=1e-8, step=1, rank=0, world=2, grad_scale=0.5)
    nulls = ("conf", "win_end", "stream", "mc", "step_dev", "lr_dev", "pred") if name != "b2h_train_step_dp" else \
        ("conf", "win_end", "stream", "mc", "lr_dev")
    args = []
    for a in _ABI_ARGS[name].split():
        if a in scalars:
            args.append(over.get(a, scalars[a]))
        elif a in over:
            args.append(None if over[a] is None else buf(a, over[a]))
        else:
            args.append(None if a in nulls else buf(a))
    return getattr(lib, name)(*args)


def test_null_and_bad_arguments_return_error_codes():
    lib = _lib.load()
    assert lib.b2h_conv_forward(None, 0, None, None, None, None, 1, 64, 24, 30, 0, 0, 0, 1.0, None) == -1
    assert "null pointer" in _lib.last_error()
    assert lib.b2h_preprocess(None, None, None, 0, None, None, 0, 64, 0, 1280.0, 1, 1, None, None, None, None, None, None,
                              None, None, None) == -1
    assert lib.b2h_pack_weights(None, None, 24, 30, 0, None) == -1
    assert lib.b2h_adam_step(None, None, None, None, 10, 1e-3, 0.9, 0.999, 1e-8, 1, None, None, 1.0, None, 0, 0, 0, None) == -1
    # the argument checks of every forward / training entry point: code and message, case by case
    keep = []
    for names, over, code, fragment in _ARG_CASES:
        for name in names:
            rc = _abi_call(lib, keep, name, over)
            assert rc == code, (name, over, rc, _lib.last_error())
            if fragment is not None:
                msg = _lib.last_error()
                assert msg.startswith(name + ":") and fragment in msg, (name, over, msg)


def test_convmodel_is_a_drop_in_on_the_host_side():
    torch.manual_seed(0)
    m = b2h.ConvModel(30, "ReLU", False)
    sd = oracle.init_params(30, False, seed=0)           # == reference ConvModel under the same seed
    assert list(m.state_dict().keys()) == list(sd.keys())
    for k, v in m.state_dict().items():
        assert v.dtype == torch.float32 and torch.equal(v, sd[k])
    assert sum(p.numel() for p in m.parameters()) == 19032
    with pytest.raises(ValueError):
        b2h.ConvModel(30, "Tanh", False)                 # HandPoseModels.py:37
    # parameters are views of one flat buffer, and stay so through load_state_dict / deepcopy / pickle
    assert m._is_flat()
    g = {k: torch.randn_like(v) for k, v in sd.items()}
    m.load_state_dict(g)
    assert m._is_flat() and torch.equal(m.flat_parameters()[:30 * 24 * 5].view(30, 24, 5), g["conv1.weight"])
    m2 = pickle.loads(pickle.dumps(m))
    assert all(torch.equal(a, b) for a, b in zip(m.state_dict().values(), m2.state_dict().values()))
    m3 = b2h.ConvModel(30, "ReLU", True)
    assert m3.conv1.weight.shape == (30, 25, 5) and m3.pos_emb is not None
    # no CPU fallback: a CPU input is refused loudly
    with pytest.raises(RuntimeError, match="no CPU fallback"):
        m(torch.zeros(1, 64, 12, 2))


def test_state_dict_interchanges_with_reference_layout(tmp_path):
    sd = oracle.init_params(30, False, seed=3)
    path = tmp_path / "last_model.pth"
    torch.save(sd, path)                                  # what the reference writes (traintest.py:146)
    m = b2h.ConvModel(30, "ReLU", False)
    m.load_state_dict(torch.load(path))
    for k, v in m.state_dict().items():
        assert torch.equal(v, sd[k])


def test_fused_adam_state_dict_layout():
    m = b2h.ConvModel(30, "ReLU", False)
    opt = b2h.FusedAdam(m.parameters(), lr=2e-4)
    ref = torch.optim.Adam(m.parameters(), lr=2e-4)
    a, b = opt.state_dict(), ref.state_dict()
    assert a["param_groups"][0]["params"] == b["param_groups"][0]["params"]
    for k in ("lr", "betas", "eps", "weight_decay", "amsgrad"):
        assert a["param_groups"][0][k] == b["param_groups"][0][k]


@settings(max_examples=200, deadline=None)
@given(n_total=st.integers(1, 5000), n=st.integers(1, 300), sel=st.sampled_from(["first", "randomcrop"]),
       seed=st.integers(0, 2**31 - 1))
def test_select_window_matches_oracle(n_total, n, sel, seed):
    rng = random.Random(seed)
    state = rng.getstate()
    s, e = b2h.select_window(n_total, n, sel, rng)
    rng.setstate(state)
    draw = rng.randint(0, n_total - n) if (n_total > n and sel == "randomcrop") else None
    assert (s, e) == oracle.select_window(n_total, n, sel, draw)
    assert 0 <= s <= e <= n_total and e - s == min(n, n_total)


def test_select_window_requires_mode_for_long_clips():
    with pytest.raises(ValueError):
        b2h.select_window(100, 10, None)


def test_sliding_window_starts():
    assert list(b2h.sliding_window_starts(200, 64, 64)) == [0, 64, 128, 192]
    assert list(b2h.sliding_window_starts(65, 64, 16)) == [0, 16, 32, 48, 64]


def test_pipelined_steps_slot_discipline(monkeypatch):
    """runner.pipelined_steps (host logic, CUDA stream/event calls faked): batch i+1 is loaded into the other slot
    before step i is enqueued, a slot is only overwritten after the step that read it was recorded, the main stream
    waits for the landing event of the slot it steps on, and every batch produces exactly one loss."""
    import contextlib
    import torch
    from hand_pose_sl_b200 import runner as R

    log = []

    class FakeEvent:
        n = 0

        def __init__(self):
            FakeEvent.n += 1
            self.id = FakeEvent.n

        def record(self, stream=None):
            log.append(("record", self.id, getattr(stream, "name", "?")))

    class FakeStream:
        def __init__(self, dev=None, name="copy"):
            self.name = name

        def wait_event(self, ev):
            log.append(("wait", self.name, ev.id))

    main = FakeStream(name="main")
    monkeypatch.setattr(torch.cuda, "current_stream", lambda dev=None: main)
    monkeypatch.setattr(torch.cuda, "Stream", FakeStream)
    monkeypatch.setattr(torch.cuda, "Event", FakeEvent)
    monkeypatch.setattr(torch.cuda, "stream", lambda s: contextlib.nullcontext())

    class FakeRunner:
        n_slots = 2
        x = torch.zeros(1)

        def load(self, batch, slot=0):
            log.append(("load", batch, slot))

        def step(self, slot=0):
            log.append(("step", slot))
            return torch.tensor(float(slot))

    losses = list(R.pipelined_steps(FakeRunner(), range(5)))
    assert losses == [0.0, 1.0, 0.0, 1.0, 0.0]
    loads = [e for e in log if e[0] == "load"]
    steps = [e for e in log if e[0] == "step"]
    assert [(b, s) for _, b, s in loads] == [(0, 0), (1, 1), (2, 0), (3, 1), (4, 0)] and len(steps) == 5
    for i in range(4):       # load(i+1) precedes step(i)
        assert log.index(("load", i + 1, (i + 1) & 1)) < [k for k, e in enumerate(log) if e[0] == "step"][i]
    # event ids in construction order: ready[slot][piece] = 1, 2 (2 slots x 1 copy stream), freed[0], freed[1] = 3, 4
    ready = {0: 1, 1: 2}
    freed = {0: 3, 1: 4}
    for i in range(5):       # step i is preceded by main.wait(ready[slot]) and followed by record(freed[slot])
        k = [k for k, e in enumerate(log) if e[0] == "step"][i]
        assert log[k - 1] == ("wait", "main", ready[i & 1]) and log[k + 1] == ("record", freed[i & 1], "main")
    for i in range(2, 5):    # overwriting a slot waits for the step that read it
        k = log.index(("load", i, i & 1))
        assert log[k - 1] == ("wait", "copy", freed[i & 1])
        assert ("record", freed[i & 1], "main") in log[:k]
    assert list(R.pipelined_steps(FakeRunner(), [])) == []
    FakeRunner.n_slots = 1
    with pytest.raises(RuntimeError):
        list(R.pipelined_steps(FakeRunner(), range(2)))


def test_host_placement_helper_is_fail_soft():
    """hostbind.bind_host_to_gpu: pure host plumbing for the N>1 launchers -- never raises, reports what it did."""
    import os

    from hand_pose_sl_b200 import hostbind

    assert hostbind._parse_cpulist("0-3,8,10-11\n") == {0, 1, 2, 3, 8, 10, 11}
    assert hostbind._parse_cpulist("") == set()
    before = os.sched_getaffinity(0)
    info = hostbind.bind_host_to_gpu(0)          # no GPU / one NUMA node here: says why and leaves the process alone
    assert isinstance(info, dict) and "bound" in info
    if not info["bound"]:
        assert "why" in info
        assert os.sched_getaffinity(0) == before
