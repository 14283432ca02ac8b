"""GPU tier: every forward and training kernel path, in every input layout, against the float64 reference of
tests/conv_ref.py -- the forward with its mask / de-normalise epilogue, forward_backward with both criteria, and the
modular backward model(x).backward(d_y) of an arbitrary d_y.

Each case of CASES first asserts the kernel it exists to reach (b2h_kernel_choice, b2h_train_subwindows, and the plan
arithmetic of the kernels restated with the device's SM count), so a case that lands on another kernel fails.

Tolerances (relative max-norm, max|kernel - reference| / max|reference|, per tensor):
  * FFMA kernel (any precision mode) against rounding="none": fp32 accumulation order only.  The unrounded formulas in
    float32 and in float64 differ by <= 8.8e-7 on the gradients and <= 2.4e-7 on the prediction (random inputs, C = 30,
    128, 256), so FFMA_TOL = 1e-5.  In entry (c) a pre-activation within 1e-5 of its layer's maximum of zero may take the
    other ReLU decision in fp32; conv_ref.relu_flip_allowance bounds what every such flip can move, element by element,
    and that bound is added.
  * bf16 mode (tile, row-space, wide kernels) against rounding="bf16": an activation on a bf16 rounding boundary rounds
    the other way under another fp32 summation order.  The spread that causes is measured per case and per tensor by
    evaluating the same rounded formulas in float32 and in float64 on the CPU (_bf16_bounds); the bound is 4x that
    spread, at least BF16_FLOOR (one bf16 ulp, 2^-8, of a single activation's share of a sum over >= 2 frames), at most
    the 1e-2 the suite allows the bf16 gradients elsewhere.
  * fp32 mode (split bf16 high/low operands on the tile kernel) against rounding="none": the documented 1e-4; the forward
    and entry (b) with the ReLU / L1-sign flip rule of test_gpu_train._grads_close, entry (c) with the element-wise
    ReLU-flip allowance above for pre-activations within SPLIT_FLIP_EPS of zero.  A Gaussian d_y has no sign coherence:
    a gradient element is a sum of terms of both signs, so one flipped ReLU moves it by percents, which a rule written for
    the criterion's gradients cannot tell from a bug and the allowance bounds exactly.
  * criterion entry (b): the loss within 1e-4 of the reference's; gradients as test_loss_and_gradients_odd_shapes_vs_oracle
    judges them (bf16: 1e-2 against the bf16-rounded reference, which absorbs L1-sign flips; FFMA: 1e-4, 1e-3 above
    10 000 frames where fp32 noise flips the sign of a few residuals).

Batches larger than one wave of tiles (MULTI_WAVE) are checked by decomposition: with confL1 (a batch sum) and with a
given d_y the gradient is a sum over windows, so the full batch equals the sum of its sub-batches of <= 120 windows up to
fp32 summation order (DECOMP_TOL), the masked predictions are bit-identical, and one 16-window sub-batch is compared
with the reference."""
import numpy as np
import pytest
import torch

import b2h_oracle as oracle
import conv_ref
import hand_pose_sl_b200 as b2h
from hand_pose_sl_b200 import _lib, synthetic
from test_gpu_train import _grads_close

pytestmark = pytest.mark.gpu
DEV = "cuda:0"
NONE, FFMA, TILE, ROWSPACE, WIDE, WIDE_TRAIN = 0, 1, 2, 3, 4, 5
FFMA_TOL = 1e-5
FLIP_EPS = 1e-5
BF16_FLOOR = 2e-3
BF16_CAP = 1e-2
SPLIT_TOL = 1e-4
# fp32 mode carries every operand as a bf16 high + low pair: a product is off by <= ~3 * 2^-18 of itself (the dropped
# low x low term and the rounding of the low halves), and sum |w a| <= 3.2 max|z| on these cases, so a pre-activation is
# off by <= ~4e-5 of its layer's max|z| per layer, ~1e-4 with what the layers below pass on
SPLIT_FLIP_EPS = 1e-4
# Decomposition: the per-window bf16 operands are identical, only the order of the fp32 sums over rows differs (the
# split-K tile ranges, the partial-slice reduction, the final sum of the sub-batches).  A fp32 sum of n terms drifts like
# a random walk, ~u * sqrt(n) * |partial sum| with u = 2^-24; n <= 600 accumulations of 16-row MMA steps per tile range
# plus <= 40 slices gives ~1.5e-6 of the element, ~6e-6 at four standard deviations.  DECOMP_TOL = 5e-5 leaves a margin
# of 8 and is still 20x tighter than the bf16 spread at C = 256 (~9e-4); a dropped or doubled tile moves the gradient
# by percents.
DECOMP_TOL = 5e-5
DECOMP_MAX = 120


def _case(name, prec, n_kp, pos, B, T, C, entries, reason, fwd=None, train=None, plan=()):
    return pytest.param(dict(prec=prec, n_kp=n_kp, pos=pos, B=B, T=T, C=C, entries=entries, fwd=fwd, train=train,
                             plan=plan, reason=reason), id=name)


CASES = [
    # tile kernel, 8 keypoints: 16-channel staging (one 16-wide K step for conv1)
    _case("tile-bf16-8kp-B7-T64-C30", "bf16", 8, None, 7, 64, 30, "abc", "16-channel staging, two 64-row segments",
          fwd=TILE, train=TILE),
    _case("tile-fp32-8kp-B7-T64-C30", "fp32", 8, None, 7, 64, 30, "abc", "16-channel staging, split operands",
          fwd=TILE, train=TILE),
    _case("tile-bf16-8kp-B5-T37-C16", "bf16", 8, None, 5, 37, 16, "abc", "16-channel staging, C = 16, odd T",
          fwd=TILE, train=TILE),
    _case("tile-fp32-8kp-B5-T37-C16", "fp32", 8, None, 5, 37, 16, "abc", "16-channel staging, C = 16, odd T, split",
          fwd=TILE, train=TILE),
    _case("tile-bf16-8kp-pos37-B4-T129-C30", "bf16", 8, 37, 4, 129, 30, "abc", "positional row t/37 in scalar staging, NT = 2",
          fwd=TILE, train=TILE, plan=("nt2",)),
    _case("tile-fp32-8kp-pos37-B4-T129-C30", "fp32", 8, 37, 4, 129, 30, "abc", "positional row, two 128-frame sub-windows",
          fwd=TILE, train=TILE, plan=("nsub2",)),
    # tile kernel, sub-windows: mode 2 applies d_y to the core rows only
    _case("tilesub-bf16-12kp-pos100-B2-T300-C30", "bf16", 12, 100, 2, 300, 30, "abc",
          "sub-windows: given d_y on core rows only, positional row past the cut", fwd=ROWSPACE, train=TILE, plan=("nsub",)),
    _case("tilesub-bf16-12kp-pos100-B1-T1024-C16", "bf16", 12, 100, 1, 1024, 16, "abc", "five 256-frame sub-windows",
          fwd=ROWSPACE, train=TILE, plan=("nsub",)),
    _case("tilesub-fp32-12kp-B3-T200-C30", "fp32", 12, None, 3, 200, 30, "abc", "sub-windows of 128 frames (split)",
          fwd=TILE, train=TILE, plan=("nsub2",)),
    # tile forward only where the layout or C decides it
    _case("tilefwd-bf16-8kp-B3-T200-C64", "bf16", 8, None, 3, 200, 64, "a", "tile NT = 2 at C = 64, reached only with 16 channels",
          fwd=TILE, plan=("nt2",)),
    _case("tilefwd-bf16-12kp-B5-T100-C33", "bf16", 12, None, 5, 100, 33, "a", "C not a multiple of 16", fwd=TILE),
    _case("tilefwd-bf16-12kp-B4-T64-C48", "bf16", 12, None, 4, 64, 48, "a", "C = 48 on the tile forward", fwd=TILE),
    # row-space forward
    _case("rowspace-bf16-8kp-B3-T640-C48", "bf16", 8, None, 3, 640, 48, "a", "16 channels against a reference", fwd=ROWSPACE),
    _case("rowspace-bf16-12kp-pos1024-B2-T1024-C30", "bf16", 12, 1024, 2, 1024, 30, "a", "positional row t/1024",
          fwd=ROWSPACE),
    # wide forward
    _case("widefwd-bf16-8kp-B5-T64-C128", "bf16", 8, None, 5, 64, 128, "a", "16-channel vector staging", fwd=WIDE),
    _case("widefwd-bf16-12kp-pos100-B3-T126-C256", "bf16", 12, 100, 3, 126, 256, "a", "positional row at T != max_len",
          fwd=WIDE),
    # wide training
    _case("widetrain-bf16-8kp-B9-T64-C80", "bf16", 8, None, 9, 64, 80, "abc", "16-channel vector staging, C = 80",
          fwd=WIDE, train=WIDE_TRAIN),
    _case("widetrain-bf16-12kp-pos64-B6-T64-C128", "bf16", 12, 64, 6, 64, 128, "abc", "scalar staging of the positional row",
          fwd=WIDE, train=WIDE_TRAIN),
    _case("widetrain-bf16-12kp-B4-T256-C33", "bf16", 12, None, 4, 256, 33, "abc", "gh = 1 at T = 256, C = 33 padding",
          fwd=TILE, train=WIDE_TRAIN, plan=("gh1",)),
    # FFMA
    _case("ffma-fp32ffma-12kp-B600-T64-C30", "fp32-ffma", 12, None, 600, 64, 30, "abc",
          "more windows than CTAs: each CTA accumulates over its windows", fwd=FFMA, train=FFMA, plan=("ffma_multi",)),
    _case("ffma-fp32-8kp-B5-T150-C64", "fp32", 8, None, 5, 150, 64, "abc", "fp32 mode beyond the tile kernel",
          fwd=FFMA, train=FFMA),
    _case("ffma-bf16-8kp-B3-T257-C33", "bf16", 8, None, 3, 257, 33, "abc", "bf16 training that lands on FFMA",
          fwd=ROWSPACE, train=FFMA),
]

MULTI_WAVE = [
    pytest.param(dict(B=600, T=64, C=256), id="wide-B600-T64-C256"),      # 200 tiles, wgrad split 6 over 200 (uneven)
    pytest.param(dict(B=300, T=200, C=64), id="wide-B300-T200-C64"),      # 300 tiles, wgrad split 37 over 300 (uneven)
]


# ---------------------------------------------------------------------------------------------- plan arithmetic
def _sms():
    return torch.cuda.get_device_properties(0).multi_processor_count


def _pe_arg(pos):
    """The C-ABI pos_emb of ConvModel._geometry: 0 = off, 1 = max_len 100, n = max_len n."""
    return 0 if pos is None else (1 if pos == 100 else int(pos))


def _ru(x, m):
    return (x + m - 1) // m * m


def _wide_wgrad_items(n_in, C, pe):
    """wide_wgrad_items (b2h_wide_tc.cuh): work items (layer, 64/128-row co block, 64-column ci block)."""
    cin = [n_in + (1 if pe else 0), C, C, C]
    cout = [C, C, C, 42]
    n = 0
    for l in range(4):
        M = 64 if _ru(cout[l], 16) <= 64 else 128
        n += ((_ru(cout[l], 16) + M - 1) // M) * ((_ru(cin[l], 16) + 63) // 64)
    return n


def _wide_plan(B, T, n_in, C, pe):
    gh = 258 // (T + 2)
    n_tiles = (B + gh - 1) // gh
    ksplit = max(1, _sms() // _wide_wgrad_items(n_in, C, pe))
    return gh, n_tiles, min(ksplit, n_tiles)


def _ffma_train_grid(B, T, n_in, C, pe):
    """plan_ffma (b2h_conv_fp32.cu), training: <= 2 CTAs per SM by shared memory."""
    TR = _ru(T, 8) + 4
    ld0, ldc, ldg = _ru(n_in + (1 if pe else 0), 4), _ru(C, 4), _ru(max(C, 42), 4)
    smem = TR * (ld0 + 3 * ldc + 2 * ldg) * 4
    per_sm = min(2, max(1, 220 * 1024 // (smem + 1024)))
    return min(B, _sms() * per_sm)


def _assert_kernels(c):
    lib = _lib.load()
    n_in, pe, prec = 2 * c["n_kp"], _pe_arg(c["pos"]), _lib.PRECISIONS[c["prec"]]
    B, T, C = c["B"], c["T"], c["C"]
    if c["fwd"] is not None:
        assert lib.b2h_kernel_choice(T, n_in, C, pe, prec, 0) == c["fwd"], "forward lands on another kernel"
    if c["train"] is not None:
        assert lib.b2h_kernel_choice(T, n_in, C, pe, prec, 1) == c["train"], "training lands on another kernel"
    nsub = lib.b2h_train_subwindows(T, n_in, C, pe, prec, 0, None) if c["train"] == TILE else 1
    for p in c["plan"]:
        if p == "nt2":          # plan_tile: a 128 < T <= 256 segment is two 128-row MMA tiles
            assert nsub == 1 and 128 < T <= 256
        elif p == "nsub":
            assert nsub > 1, nsub
        elif p == "nsub2":
            assert nsub == 2, nsub
        elif p == "gh1":        # plan_wide: one window per tile
            assert 258 // (T + 2) == 1
        elif p == "ffma_multi":
            grid = _ffma_train_grid(B, T, n_in, C, pe)
            assert B > grid, (B, grid)
        else:
            raise AssertionError(p)


# ---------------------------------------------------------------------------------------------- helpers
def _model(sd, c):
    pos = c["pos"]
    m = b2h.ConvModel(c["C"], "ReLU", pos is not None, precision=c["prec"], n_keypoints=c["n_kp"],
                      pos_emb_max_len=pos if pos is not None else 100, pos_emb_any_length=True)
    m.load_state_dict(sd)
    return m.to(DEV)


def _setup(c, seed):
    sd = oracle.init_params(c["C"], c["pos"] is not None, seed=seed, n_in=2 * c["n_kp"])
    batch = synthetic.model_batch(c["B"], c["T"], seed=seed + 1, ragged=True, len_seed=seed + 2, n_kp=c["n_kp"])
    return sd, batch


def _d_y(B, T, seed):
    """Seeded Gaussian d(loss)/d(prediction), non-zero on every row (mode 2 applies no mask)."""
    g = torch.Generator().manual_seed(seed)
    d = torch.randn(B, T, 21, 2, generator=g) * 1e-3
    assert (d != 0).all()
    return d


def _rounding(kernel, prec):
    return "bf16" if (kernel != FFMA and prec == "bf16") else "none"


def _rel(v, ref):
    return oracle.rel_err(np.asarray(v, dtype=np.float64), np.asarray(ref, dtype=np.float64))


def _bf16_bounds(sd, x, pos, d_y=None):
    """Per-tensor bounds for the bf16 kernels: 4x the float32-vs-float64 spread of the bf16-rounded formulas (the
    prediction under "pred"), clamped to [BF16_FLOOR, BF16_CAP]."""
    f32 = conv_ref.forward(sd, x, pos, "bf16", dtype=torch.float32)
    f64 = conv_ref.forward(sd, x, pos, "bf16")
    out = {"pred": _rel(f32["pred"], f64["pred"])}
    if d_y is not None:
        g32 = conv_ref.backward(sd, x, d_y, pos, "bf16", dtype=torch.float32, fwd=f32)
        g64 = conv_ref.backward(sd, x, d_y, pos, "bf16", fwd=f64)
        out.update({k: _rel(g32[k], g64[k]) for k in conv_ref.NAMES})
    return {k: min(BF16_CAP, max(4.0 * v, BF16_FLOOR)) for k, v in out.items()}


def _grads_of(model):
    return {k: p.grad.detach().double().cpu() for k, p in zip(conv_ref.NAMES, model._ordered_params())}


def _split(model, flat):
    out, off = {}, 0
    for k, p in zip(conv_ref.NAMES, model._ordered_params()):
        out[k] = flat[off:off + p.numel()].view(p.shape).double().cpu()
        off += p.numel()
    return out


def _check_status():
    torch.cuda.synchronize()
    assert _lib.load().b2h_tc_status() == 0, "a tensor-core kernel reported a wait timeout"


# ---------------------------------------------------------------------------------------------- entries
def _entry_forward(c, m, sd, batch):
    """(a) predict() with the fused mask_output(lengths) and de-normalise (x 1280) epilogue."""
    kern, pos = c["fwd"], c["pos"]
    rnd = _rounding(kern, c["prec"])
    y = m.predict(batch["input_kp"].to(DEV), lengths=batch["n_frames"], denormalize=1280.0)
    _check_status()
    f = conv_ref.forward(sd, batch["input_kp"], pos, rnd)
    want = oracle.mask_output(f["pred"].clone(), batch["n_frames"]) * 1280.0
    err = _rel(y.cpu(), want)
    if rnd == "bf16":
        tol = _bf16_bounds(sd, batch["input_kp"], pos)["pred"]
    else:
        tol = FFMA_TOL if kern == FFMA else SPLIT_TOL
    assert err <= tol, f"forward: rel err {err:.3g} > {tol:.3g}"
    for i, ln in enumerate(batch["n_frames"]):
        assert not y[i, int(ln):].any(), "mask_output epilogue"


def _entry_criterion(c, m, sd, batch, kind):
    """(b) forward_backward: loss, masked prediction and the gradients of the criterion."""
    kern, pos, prec = c["train"], c["pos"], c["prec"]
    rnd = _rounding(kern, prec)
    db = {k: (v.to(DEV) if k != "n_frames" else v) for k, v in batch.items()}
    loss, grads, pred = b2h.forward_backward(m, db, loss=kind, want_pred=True)
    _check_status()
    f = conv_ref.forward(sd, batch["input_kp"], pos, rnd)
    r_loss, r_masked, d_pred = conv_ref.criterion(f["pred"], batch["target_kp"], batch["n_frames"], kind,
                                                  batch["target_conf"])
    r_g = conv_ref.backward(sd, batch["input_kp"], d_pred, pos, rnd, fwd=f)
    assert abs(float(loss) - float(r_loss)) <= 1e-4 * abs(float(r_loss)), (float(loss), float(r_loss))
    ptol = _bf16_bounds(sd, batch["input_kp"], pos)["pred"] if rnd == "bf16" else (FFMA_TOL if kern == FFMA else SPLIT_TOL)
    assert _rel(pred.cpu(), r_masked) <= ptol
    for k, v in _split(m, grads).items():
        ref = r_g[k].numpy()
        if rnd == "bf16":
            assert _rel(v, ref) <= 1e-2, (kind, k, _rel(v, ref))
        elif kern == FFMA:
            gtol = 1e-4 if c["B"] * c["T"] < 10000 else 1e-3
            assert _rel(v, ref) <= gtol, (kind, k, _rel(v, ref))
        else:
            assert _grads_close(v.numpy(), ref, "fp32", SPLIT_TOL), (kind, k, _rel(v, ref))


def _entry_modular_backward(c, m, sd, batch, x_dtype):
    """(c) model(x).backward(d_y): the modular path through b2h_conv_backward."""
    kern, pos, prec = c["train"], c["pos"], c["prec"]
    rnd = _rounding(kern, prec)
    x = batch["input_kp"].to(x_dtype)
    d_y = _d_y(c["B"], c["T"], seed=c["B"] * 7 + c["T"])
    for p in m.parameters():
        p.grad = None
    m(x.to(DEV)).backward(d_y.to(DEV))
    _check_status()
    got = _grads_of(m)
    x_ref = x.float()
    f = conv_ref.forward(sd, x_ref, pos, rnd)
    up = []
    r_g = conv_ref.backward(sd, x_ref, d_y.double(), pos, rnd, fwd=f, upstream=up)
    if rnd == "bf16":
        tol = _bf16_bounds(sd, x_ref, pos, d_y.double())
        for k in conv_ref.NAMES:
            err = _rel(got[k], r_g[k])
            assert err <= tol[k], f"{x_dtype} {k}: rel err {err:.3g} > {tol[k]:.3g}"
    else:
        tol, eps = (FFMA_TOL, FLIP_EPS) if kern == FFMA else (SPLIT_TOL, SPLIT_FLIP_EPS)
        allow = conv_ref.relu_flip_allowance(sd, f, up, eps)
        for k in conv_ref.NAMES:
            ref = r_g[k]
            excess = ((got[k] - ref).abs() - allow[k]).max()
            err = float(excess) / float(ref.abs().max())
            assert err <= tol, f"{x_dtype} {k}: rel err beyond the ReLU-flip allowance {err:.3g} > {tol}"


@pytest.mark.parametrize("c", CASES)
def test_kernel_path_matches_float64_reference(c):
    _assert_kernels(c)
    seed = 1000 * c["n_kp"] + 10 * c["C"] + c["T"] + c["B"]
    sd, batch = _setup(c, seed)
    m = _model(sd, c)
    if "a" in c["entries"]:
        _entry_forward(c, m, sd, batch)
    if "b" in c["entries"]:
        for kind in ("L1", "confL1"):
            _entry_criterion(c, m, sd, batch, kind)
    if "c" in c["entries"]:
        for x_dtype in (torch.float32, torch.bfloat16):
            _entry_modular_backward(c, m, sd, batch, x_dtype)


@pytest.mark.parametrize("c", MULTI_WAVE)
def test_multi_wave_wide_training_equals_its_sub_batches(c):
    """Wide training beyond one wave of tiles: persistent tile loop (a CTA owns >= 2 tiles and stages the next one
    while the current one computes) and split-K weight gradients whose tile ranges are uneven."""
    B, T, C, n_in = c["B"], c["T"], c["C"], 24
    lib = _lib.load()
    assert lib.b2h_kernel_choice(T, n_in, C, 0, _lib.BF16, 1) == WIDE_TRAIN
    gh, n_tiles, ksplit = _wide_plan(B, T, n_in, C, 0)
    assert n_tiles > _sms(), (n_tiles, _sms())                    # a CTA loops over several tiles
    per = (n_tiles + ksplit - 1) // ksplit
    assert n_tiles % ksplit != 0 and n_tiles - (ksplit - 1) * per != per, (n_tiles, ksplit)   # uneven tile ranges
    assert DECOMP_MAX % gh == 0                                   # sub-batch windows keep their place inside a tile
    case = dict(prec="bf16", n_kp=12, pos=None, B=B, T=T, C=C, train=WIDE_TRAIN)
    sd, batch = _setup(case, seed=B + T + C)
    m = _model(sd, case)
    db = {k: (v.to(DEV) if k != "n_frames" else v) for k, v in batch.items()}
    chunks = [(lo, min(B, lo + DECOMP_MAX)) for lo in range(0, B, DECOMP_MAX)]

    # (b) confL1: loss and gradient are sums over windows
    loss, grads, pred = b2h.forward_backward(m, db, loss="confL1", want_pred=True)
    _check_status()
    g_full = grads.double().cpu()
    g_sum = torch.zeros_like(g_full)
    l_sum = 0.0
    for lo, hi in chunks:
        sub = {k: v[lo:hi] for k, v in db.items()}
        l_s, g_s, p_s = b2h.forward_backward(m, sub, loss="confL1", want_pred=True)
        _check_status()
        assert torch.equal(p_s, pred[lo:hi]), f"masked prediction of windows {lo}..{hi}"
        g_sum += g_s.double().cpu()
        l_sum += float(l_s)
    assert abs(float(loss) - l_sum) <= 1e-5 * abs(l_sum)
    off = 0
    for k, p in zip(conv_ref.NAMES, m._ordered_params()):
        a, b = g_full[off:off + p.numel()], g_sum[off:off + p.numel()]
        off += p.numel()
        assert _rel(a, b) <= DECOMP_TOL, (k, _rel(a, b))

    # (c) the modular backward of a given d_y, fp32 and bf16 input
    d_y = _d_y(B, T, seed=B + T)
    for x_dtype in (torch.float32, torch.bfloat16):
        x = batch["input_kp"].to(x_dtype).to(DEV)
        dyd = d_y.to(DEV)
        for p in m.parameters():
            p.grad = None
        m(x).backward(dyd)
        _check_status()
        full = _grads_of(m)
        acc = {k: torch.zeros_like(v) for k, v in full.items()}
        for lo, hi in chunks:
            for p in m.parameters():
                p.grad = None
            m(x[lo:hi]).backward(dyd[lo:hi])
            _check_status()
            for k, v in _grads_of(m).items():
                acc[k] += v
        for k in conv_ref.NAMES:
            assert _rel(full[k], acc[k]) <= DECOMP_TOL, (x_dtype, k, _rel(full[k], acc[k]))

    # one 16-window sub-batch against the reference
    sub = {k: v[:16] for k, v in batch.items()}
    sc = dict(case, B=16, entries="bc")
    for kind in ("L1", "confL1"):
        _entry_criterion(sc, m, sd, sub, kind)
    _entry_modular_backward(sc, m, sd, sub, torch.float32)


def test_modular_forward_refuses_an_input_that_requires_grad():
    """The kernels compute no input gradient: autograd through ConvModel with an input that requires grad (a trainable
    module in front of it) raises instead of silently leaving that module without a gradient."""
    sd = oracle.init_params(30, False, seed=3)
    m = b2h.ConvModel(30, "ReLU", False, precision="bf16")
    m.load_state_dict(sd)
    m = m.to(DEV)
    x = synthetic.model_batch(2, 64, seed=4)["input_kp"].to(DEV)
    front = torch.nn.Parameter(torch.ones((), device=DEV))
    with pytest.raises(RuntimeError, match="input gradient"):
        m(x * front)
    with torch.no_grad():                                          # inference is unaffected
        y = m(x * front)
    assert y.shape == (2, 64, 21, 2)
    m(x).sum().backward()                                          # an input without grad still trains the weights
    assert m.conv1.weight.grad is not None
