"""GPU tier: one training step of every optimizer path against torch's Adam in float64 and the packed buffer against a
numpy restatement of its layout, byte for byte.

Which kernel applies Adam depends on the entry point, the precision, the batch and conv_channels: adam_gp_wide_kernel,
adam_kernel (more than 64 slices), adam_gp_tile_kernel, adam_flat_kernel (an already-reduced gradient), adam_dp_kernel,
or the fused tail of the tile train kernel (one pass or several per CTA).  The bias corrections come in three forms: host pow(), device ipow and
the tail's fp32 expm1f.  Each case pins its path (kernel choice, slice count, slot count) and then checks two
consecutive steps, each from its own snapshot:
  m within 1e-5 * rms_l, v within 1e-5 relative, p within one fp32 ulp + 1e-4 * lr / (1 - b1^t),
where rms_l is the RMS of tensor l's first gradient and the gradient is forward_backward's at the pre-step weights.
That admits the other slice-summation order of the fused tail and the three bias-correction forms (~3e-7); it does
not admit a bias correction off by 1e-4, a missed grad_scale, a stale step count or a mis-decoded slot."""
import numpy as np
import pytest
import torch

import b2h_oracle as oracle
import hand_pose_sl_b200 as b2h
from hand_pose_sl_b200 import _lib, synthetic
from optim_ref import adam_step_f64, gp_total, pack_reference, train_nparts

pytestmark = pytest.mark.gpu
DEV = "cuda:0"
N_IN = 24
FFMA, TILE, WIDE_TRAIN = 1, 2, 5
STEPS = 2


def _case(name, entry, prec, C, B, t0, T=64, pe=False, loss="L1", lr=1e-3, lr2=None, betas=(0.9, 0.999), eps=1e-8,
          path=None):
    return pytest.param(dict(entry=entry, prec=prec, C=C, B=B, T=T, pe=pe, loss=loss, t0=t0, lr=lr, lr2=lr2, betas=betas,
                             eps=eps, path=path), id=name)


CASES = [
    # fused_train_step, tile kernel, <= 64 slices: adam_gp_wide_kernel, host pow()
    _case("fused-tile-fp32-C30-B4", "fused", "fp32", 30, 4, 0, path="few"),
    _case("fused-tile-bf16-C30-B4", "fused", "bf16", 30, 4, 99999, loss="confL1", path="few"),
    _case("fused-tile-fp32-C30-B128", "fused", "fp32", 30, 128, 9, loss="confL1", path="few"),
    _case("fused-tile-bf16-C30-B128", "fused", "bf16", 30, 128, 999, path="few"),
    _case("fused-tile-fp32-C16-B6", "fused", "fp32", 16, 6, 9, path="few"),
    _case("fused-tile-bf16-C30-posemb-T100-B4", "fused", "bf16", 30, 4, 0, T=100, pe=True, path="few"),
    # fused_train_step, tile kernel, > 64 slices: adam_kernel on the slot layout, host pow()
    _case("fused-tile-fp32-C30-B130", "fused", "fp32", 30, 130, 999, path="many"),
    _case("fused-tile-bf16-C30-B130", "fused", "bf16", 30, 130, 0, loss="confL1", path="many"),
    _case("fused-tile-fp32-C30-B256", "fused", "fp32", 30, 256, 99999, path="many"),
    _case("fused-tile-bf16-C30-B256", "fused", "bf16", 30, 256, 9, path="many"),
    # fused_train_step, fp32-ffma, one slice per CTA: <= 64 slices: adam_gp_wide_kernel up to 100 000 slots,
    # adam_gp_tile_kernel above; > 64 slices: adam_kernel; host pow()
    _case("fused-ffma-C30-B8", "fused", "fp32-ffma", 30, 8, 9, loss="confL1", path="few"),
    _case("fused-ffma-C64-B4", "fused", "fp32-ffma", 64, 4, 999, path="few"),
    _case("fused-ffma-C128-B4", "fused", "fp32-ffma", 128, 4, 0, path="few-slots>1e5"),
    _case("fused-ffma-C30-B130", "fused", "fp32-ffma", 30, 130, 99999, path="many"),
    # fused_train_step, wide kernels (bf16): adam_gp_wide_kernel up to 100 000 slots, adam_gp_tile_kernel above
    _case("fused-wide-C64-B6", "fused", "bf16", 64, 6, 0, path="slots<=1e5"),
    _case("fused-wide-C80-B5-betas0.8-eps", "fused", "bf16", 80, 5, 9, betas=(0.8, 0.99), eps="rms", path="slots<=1e5"),
    _case("fused-wide-C96-B6", "fused", "bf16", 96, 6, 99999, loss="confL1", path="slots>1e5"),
    _case("fused-wide-C136-B4", "fused", "bf16", 136, 4, 999, path="slots>1e5"),
    _case("fused-wide-C256-B4", "fused", "bf16", 256, 4, 9, path="slots>1e5"),
    # TrainStepRunner, tile kernel: Adam in the fused tail (fp32 expm1f bias corrections), several passes per CTA
    _case("runner-tile-fp32-B4", "runner", "fp32", 30, 4, 0, path="multi-pass"),
    _case("runner-tile-bf16-B4", "runner", "bf16", 30, 4, 999, loss="confL1", path="multi-pass"),
    _case("runner-tile-fp32-B166", "runner", "fp32", 30, 166, 9, path="multi-pass"),
    _case("runner-tile-bf16-B166", "runner", "bf16", 30, 166, 0, path="multi-pass"),
    # ... one slot per thread
    _case("runner-tile-fp32-B168", "runner", "fp32", 30, 168, 999, loss="confL1", path="one-pass"),
    _case("runner-tile-bf16-B168", "runner", "bf16", 30, 168, 9, path="one-pass"),
    _case("runner-tile-fp32-B256", "runner", "fp32", 30, 256, 99999, path="one-pass"),
    _case("runner-tile-bf16-B256-lr-change", "runner", "bf16", 30, 256, 0, lr2=3e-4, path="one-pass"),
    _case("runner-tile-fp32-B300", "runner", "fp32", 30, 300, 9, path="one-pass-capped"),
    _case("runner-tile-bf16-B300", "runner", "bf16", 30, 300, 999, loss="confL1", path="one-pass-capped"),
    _case("runner-tile-fp32-T200-B48", "runner", "fp32", 30, 48, 9, T=200, path="one-pass"),
    # TrainStepRunner, separate Adam launch with the device-side step counter and learning rate (device ipow)
    _case("runner-wide-C96-B6-lr-change", "runner", "bf16", 96, 6, 9, lr2=2e-4, path="slots>1e5"),
    _case("runner-ffma-C64-B4", "runner", "fp32-ffma", 64, 4, 0, loss="confL1", path="few"),
    # DataParallelTrainer without a process group: reduction, then adam_flat_kernel on the reduced gradient, device ipow
    _case("dptrainer-bf16-C30-B16", "dptrainer", "bf16", 30, 16, 999, path="few"),
    # b2h_train_step_dp, world 1, grad_scale 0.5: the fused tail (tile) / reduce_* + adam_dp_kernel (three launches)
    _case("train_step_dp-tile-bf16-C30-B200", "dp", "bf16", 30, 200, 9, path="one-pass"),
    _case("train_step_dp-tile-fp32-C30-B8", "dp", "fp32", 30, 8, 99999, loss="confL1", path="multi-pass"),
    _case("train_step_dp-ffma-C64-B4", "dp", "fp32-ffma", 64, 4, 0, path="few"),
]


def _assert_path(c):
    """The case lands on the side of every dispatch threshold its name says."""
    lib = _lib.load()
    pe = 1 if c["pe"] else 0
    choice = lib.b2h_kernel_choice(c["T"], N_IN, c["C"], pe, _lib.PRECISIONS[c["prec"]], 1)
    path = c["path"]
    slots = gp_total(N_IN, c["C"], pe)
    if path.startswith("slots"):
        assert choice == WIDE_TRAIN
        assert (slots <= 100000) == (path == "slots<=1e5"), slots
        return
    assert choice == (FFMA if c["prec"] == "fp32-ffma" else TILE)
    n = train_nparts(c["B"], c["T"], N_IN, c["C"], pe, c["prec"])
    per = ((slots + n - 1) // n + 3) // 4 * 4          # fused tail: slots per CTA (one pass while <= 256 threads)
    if path.startswith("few"):
        assert n <= 64, n
        assert (slots <= 100000) == (path == "few"), slots
    elif path == "many":
        assert n > 64, n
    elif path == "multi-pass":
        assert per > 256, (n, per)
    elif path.startswith("one-pass"):
        assert per <= 256, (n, per)
        if path == "one-pass-capped":
            assert n < (c["B"] + 1) // 2, n
    else:
        raise AssertionError(path)


def _per_tensor(model):
    out, off = [], 0
    for p in model._ordered_params():
        out.append((off, off + p.numel()))
        off += p.numel()
    return out


def _moments(opt):
    """exp_avg / exp_avg_sq of the 8 parameters from the optimizer's torch-layout state, flattened in state_dict order."""
    st = opt.state_dict()["state"]
    m = torch.cat([st[i]["exp_avg"].reshape(-1) for i in range(8)]).double().cpu().numpy()
    v = torch.cat([st[i]["exp_avg_sq"].reshape(-1) for i in range(8)]).double().cpu().numpy()
    return m, v


def _seed_optimizer_state(opt, model, rms, t0, seed):
    """m0 = 0.5 rms_l N(0,1), v0 = (rms_l U(0.5, 2))^2, step t0, through the public torch-layout load_state_dict."""
    gen = torch.Generator().manual_seed(seed)
    state = {}
    for i, p in enumerate(model._ordered_params()):
        m0 = 0.5 * rms[i] * torch.randn(p.shape, generator=gen, dtype=torch.float64)
        v0 = (rms[i] * (0.5 + 1.5 * torch.rand(p.shape, generator=gen, dtype=torch.float64))) ** 2
        state[i] = {"step": torch.tensor(float(t0)), "exp_avg": m0.float(), "exp_avg_sq": v0.float()}
    opt.load_state_dict({"state": state, "param_groups": opt.state_dict()["param_groups"]})


class _DpStep:
    """b2h_train_step_dp on one rank: exchange buffer sized by b2h_dp_exchange_floats and filled per
    b2h_dp_exchange_fill, a one-entry device table of peer buffers, epoch counter from 0."""

    def __init__(self, model, opt, batch, c):
        self.lib = _lib.load()
        self.model, self.opt, self.c = model, opt, c
        n_in, C, pe = model._geometry()
        prec = _lib.PRECISIONS[c["prec"]]
        nfl = int(self.lib.b2h_dp_exchange_floats(n_in, C, pe, 1))
        fill = int(self.lib.b2h_dp_exchange_fill(c["T"], n_in, C, pe, prec))
        assert nfl > 0 and fill in (0, 0xFFFFFFFF)
        assert (fill != 0) == (c["prec"] != "fp32-ffma")       # the tile kernel's sentinel words / zeroed flags
        self.sym = torch.empty(nfl, dtype=torch.float32, device=DEV)
        self.sym.view(torch.int32).fill_(fill - (1 << 32) if fill >= (1 << 31) else fill)
        self.peers = torch.tensor([self.sym.data_ptr()], dtype=torch.int64, device=DEV)
        self.epoch = torch.zeros(1, dtype=torch.int64, device=DEV)
        self.st = opt._group_state(0, opt.param_groups[0], model)
        self.batch = batch

    def step(self):
        c, m, st, b = self.c, self.model, self.st, self.batch
        n_in, C, pe = m._geometry()
        g = self.opt.param_groups[0]
        kind = _lib.LOSSES[c["loss"]]
        x = b["input_kp"].contiguous()
        tgt = b["target_kp"].contiguous()
        conf = b["target_conf"].contiguous() if kind == _lib.LOSS_CONFL1 else None
        len32 = b["n_frames"].to(device=DEV, dtype=torch.int32)
        loss = torch.empty(1, dtype=torch.float32, device=DEV)
        ws = m.workspace(c["B"], c["T"])
        st["lr_dev"].fill_(float(g["lr"]))
        _lib.check(self.lib.b2h_train_step_dp(
            _lib.ptr(x), _lib.DT_F32, _lib.ptr(tgt), _lib.ptr(conf), _lib.ptr(len32), _lib.ptr(m.flat_parameters()),
            _lib.ptr(m.packed_weights()), _lib.ptr(st["m"]), _lib.ptr(st["v"]), _lib.ptr(loss), c["B"], c["T"], n_in, C, pe,
            kind, _lib.PRECISIONS[c["prec"]], float(g["lr"]), g["betas"][0], g["betas"][1], g["eps"], _lib.ptr(st["step_dev"]),
            _lib.ptr(self.epoch), _lib.ptr(st["lr_dev"]), _lib.ptr(self.sym), _lib.ptr(self.peers), None, 0, 1, 0.5,
            _lib.ptr(ws), ws.numel(), _lib.stream_ptr(torch.device(DEV))))
        torch.cuda.synchronize()
        assert self.lib.b2h_dp_status() == 0, "adam_dp_kernel: wait for the peer flag timed out"
        assert self.lib.b2h_tc_status() == 0


@pytest.mark.parametrize("c", CASES)
def test_optimizer_step_matches_float64_adam(c):
    from hand_pose_sl_b200 import parallel
    from hand_pose_sl_b200.runner import TrainStepRunner
    _assert_path(c)
    lib = _lib.load()
    C, B, T, pe, loss = c["C"], c["B"], c["T"], c["pe"], c["loss"]
    seed = C * 1000 + B + T
    sd = oracle.init_params(C, pe, seed=seed)
    model = b2h.ConvModel(C, "ReLU", pe, precision=c["prec"])
    model.load_state_dict(sd)
    model = model.to(DEV)
    batch = synthetic.model_batch(B, T, seed=seed + 1, ragged=True, len_seed=seed + 2)
    db = {k: (v.to(DEV) if k != "n_frames" else v) for k, v in batch.items()}
    spans = _per_tensor(model)
    n_in, Cg, peg = model._geometry()

    # rms_l of each tensor's gradient at the start conditions the seeded moments and scales the tolerances
    _, g0 = b2h.forward_backward(model, db, loss=loss)
    g0 = g0.double().cpu().numpy()
    rms = [float(np.sqrt(np.mean(g0[a:b] ** 2))) for a, b in spans]
    assert min(rms) > 0, rms
    eps = float(np.median(rms)) if c["eps"] == "rms" else c["eps"]      # eps ~ sqrt(v_hat): where eps sits matters
    opt = b2h.FusedAdam(model.parameters(), lr=c["lr"], betas=c["betas"], eps=eps)
    _seed_optimizer_state(opt, model, rms, c["t0"], seed)
    grad_scale = 1.0

    if c["entry"] == "runner":
        runner = TrainStepRunner(model, opt, B, T, loss)
        runner.load(batch, non_blocking=False)
    elif c["entry"] == "dptrainer":
        runner = parallel.DataParallelTrainer(model, opt, B, T, loss)
        assert runner.world == 1 and runner.exchange == "nccl"
        runner.load(batch, non_blocking=False)
    elif c["entry"] == "dp":
        runner = _DpStep(model, opt, db, c)
        grad_scale = 0.5

    for s in range(STEPS):
        t = c["t0"] + s + 1
        if s == 1 and c["lr2"] is not None:
            opt.param_groups[0]["lr"] = c["lr2"]
        lr = opt.param_groups[0]["lr"]
        _, gr = b2h.forward_backward(model, db, loss=loss)
        gr = gr.double().cpu().numpy()
        p0 = model.flat_parameters().double().cpu().numpy()
        m0, v0 = _moments(opt)

        if c["entry"] == "fused":
            b2h.fused_train_step(model, db, opt, loss=loss)
        elif c["entry"] in ("runner", "dptrainer"):
            runner.step(0)
            runner.finish()
        else:
            runner.step()
        torch.cuda.synchronize()
        assert lib.b2h_tc_status() == 0

        p1_32 = model.flat_parameters().cpu().numpy()
        p1 = p1_32.astype(np.float64)
        m1, v1 = _moments(opt)
        p_ref, m_ref, v_ref = adam_step_f64(p0, gr, m0, v0, t, lr, c["betas"], eps, grad_scale)
        p_tol_abs = 1e-4 * lr / (1.0 - c["betas"][0] ** t)
        ulp = np.spacing(np.abs(p_ref).astype(np.float32)).astype(np.float64)
        for l, (a, b) in enumerate(spans):
            where = f"step {s + 1} (t={t}) tensor {l}"
            dm = np.abs(m1[a:b] - m_ref[a:b]).max() / rms[l]
            assert dm <= 1e-5, f"{where}: |m - m_ref| = {dm:.3g} rms"
            dv = np.abs(v1[a:b] - v_ref[a:b]) / (v_ref[a:b] + 1e-12 * rms[l] ** 2)
            assert dv.max() <= 1e-5, f"{where}: |v - v_ref| / v_ref = {dv.max():.3g}"
            dp = np.abs(p1[a:b] - p_ref[a:b]) / (ulp[a:b] + p_tol_abs)
            assert dp.max() <= 1.0, (f"{where}: |p - p_ref| = {dp.max():.3g} x (ulp + 1e-4 lr / bc1); "
                                     f"Adam moved it by {np.abs(p_ref[a:b] - p0[a:b]).max():.3g}")
        # the re-packed operand layouts == the layout restated in numpy, byte for byte (padding included)
        packed = model._packed.cpu().numpy()
        want = pack_reference(p1_32, n_in, Cg, peg)
        assert packed.shape == want.shape
        bad = np.flatnonzero(packed != want)
        assert bad.size == 0, f"step {s + 1}: {bad.size} packed bytes differ, first at byte {bad[0]}"
        # the step counter advanced exactly once
        if c["entry"] != "dp":
            assert float(opt.state_dict()["state"][0]["step"]) == t
        if c["entry"] != "fused":
            assert int(opt._group_state(0, opt.param_groups[0], model)["step_dev"].item()) == t
