"""CPU tier: tests/conv_ref.py, the float64 reference of the GPU gradient-path tests, against torch autograd of the
reference formulas, against the oracle's bf16-operand emulation and against the golden vectors of the reference."""
import numpy as np
import pytest
import torch
import torch.nn.functional as F

import b2h_oracle as oracle
import conv_ref
from conftest import golden_sd, load_golden


def _autograd_reference(sd, x, pos):
    """The reference formulas (HandPoseModels.py:40-84, the positional row built for the actual T) in float64 with
    parameters that require grad: returns (prediction (B, T, 21, 2), parameter dict)."""
    ps = {k: v.double().clone().requires_grad_(True) for k, v in sd.items()}
    B, T = x.shape[:2]
    h = x.double().reshape(B, T, -1).permute(0, 2, 1)
    if pos is not None:
        row = (torch.arange(T).float() / pos).double()
        h = torch.cat([row[None, None, :].repeat(B, 1, 1), h], dim=1)
    for l in range(1, 5):
        h = F.conv1d(h, ps[f"conv{l}.weight"], ps[f"conv{l}.bias"], padding=2)
        if l < 4:
            h = F.relu(h)
    return h.view(B, 21, 2, T).permute(0, 3, 1, 2), ps


def _inputs(n_kp, pe, B, T, seed):
    from hand_pose_sl_b200 import synthetic    # pure CPU generator (the package imports no CUDA code at import time)
    sd = oracle.init_params(30, pe is not None, seed=seed, n_in=2 * n_kp)
    batch = synthetic.model_batch(B, T, seed=seed + 1, ragged=True, len_seed=seed + 2, n_kp=n_kp)
    return sd, batch


POS = [pytest.param(None, 64, id="nopos"), pytest.param(100, 100, id="pos100-T100"), pytest.param(37, 64, id="pos37-T64"),
       pytest.param("T", 53, id="posT-T53")]


@pytest.mark.parametrize("n_kp", [8, 12])
@pytest.mark.parametrize("pos,T", POS)
def test_backward_of_any_dy_equals_float64_autograd(n_kp, pos, T):
    pe = T if pos == "T" else pos
    sd, batch = _inputs(n_kp, pe, 3, T, seed=11 * n_kp + T)
    gen = torch.Generator().manual_seed(T)
    d_y = torch.randn(3, T, 21, 2, generator=gen, dtype=torch.float64)
    ln = batch["n_frames"]
    i = int(torch.argmin(ln))
    assert int(ln[i]) < T and (d_y[i, int(ln[i]):] != 0).any()           # non-zero beyond the sequence length too
    pred, ps = _autograd_reference(sd, batch["input_kp"], pe)
    (pred * d_y).sum().backward()
    f = conv_ref.forward(sd, batch["input_kp"], pe)
    assert torch.allclose(f["pred"], pred.detach(), rtol=0, atol=1e-12 * float(pred.detach().abs().max()))
    g = conv_ref.backward(sd, batch["input_kp"], d_y, pe)
    for k in conv_ref.NAMES:
        ref = ps[k].grad
        assert float((g[k] - ref).abs().max()) <= 1e-12 * float(ref.abs().max()), k


@pytest.mark.parametrize("kind", ["L1", "confL1"])
@pytest.mark.parametrize("n_kp,pos,T", [(12, None, 64), (8, 37, 64), (12, 100, 100)])
def test_criterion_and_backward_equal_float64_autograd(kind, n_kp, pos, T):
    """criterion() = mask_output + maskedPoseL1 / poderatedPoseL1 as the oracle writes them (literal per-sample loops),
    and backward() of its d(loss)/d(pred) = autograd through the whole chain."""
    sd, batch = _inputs(n_kp, pos, 4, T, seed=5 * T + n_kp)
    pred, ps = _autograd_reference(sd, batch["input_kp"], pos)
    masked = oracle.mask_output(pred.clone(), batch["n_frames"])
    tgt, conf = batch["target_kp"].double(), batch["target_conf"].double()
    if kind == "L1":
        loss = oracle.masked_pose_l1(masked, tgt, batch["n_frames"])
    else:
        loss = oracle.poderated_pose_l1(masked, tgt, batch["n_frames"], conf)
    loss.backward()
    f = conv_ref.forward(sd, batch["input_kp"], pos)
    c_loss, c_masked, d_pred = conv_ref.criterion(f["pred"], tgt, batch["n_frames"], kind, conf)
    assert abs(float(c_loss) - loss.item()) <= 1e-12 * abs(loss.item())
    assert torch.allclose(c_masked, masked.detach(), rtol=0, atol=1e-12 * float(masked.abs().max()))
    for i, ln in enumerate(batch["n_frames"]):
        assert not d_pred[i, int(ln):].any()
    g = conv_ref.backward(sd, batch["input_kp"], d_pred, pos)
    for k in conv_ref.NAMES:
        ref = ps[k].grad
        assert float((g[k] - ref).abs().max()) <= 1e-12 * float(ref.abs().max()), k


@pytest.mark.parametrize("kind", ["L1", "confL1"])
@pytest.mark.parametrize("name", ["convmodel_c30.npz", "convmodel_c64.npz", "convmodel_c30_t200.npz"])
def test_bf16_rounding_matches_the_oracle_emulation(name, kind):
    """rounding="bf16" evaluated in float32 performs the operations of oracle.train_grads_bf16_emulated (same rounding
    points, same torch ops): the two agree to fp32 rounding."""
    g = load_golden(name)
    sd = golden_sd(g)
    x, tgt, conf = (torch.from_numpy(g[k]) for k in ("input_kp", "target_kp", "target_conf"))
    e_loss, e_g, e_pred = oracle.train_grads_bf16_emulated(sd, x, tgt, g["lengths"], kind, conf)
    f = conv_ref.forward(sd, x, None, "bf16", dtype=torch.float32)
    loss, masked, d_pred = conv_ref.criterion(f["pred"], tgt, g["lengths"], kind, conf)
    assert abs(float(loss) - e_loss) <= 1e-6 * abs(e_loss)
    assert oracle.rel_err(masked.numpy(), e_pred.numpy()) <= 1e-6
    gr = conv_ref.backward(sd, x, d_pred, None, "bf16", dtype=torch.float32, fwd=f)
    for k in conv_ref.NAMES:
        assert oracle.rel_err(gr[k].numpy(), e_g[k].numpy()) <= 1e-5, k


@pytest.mark.parametrize("name", ["convmodel_c30.npz", "convmodel_c30_b1.npz", "convmodel_c30_posemb.npz",
                                  "convmodel_c64.npz", "convmodel_c30_t200.npz"])
def test_forward_and_gradients_match_golden(name):
    """The golden vectors were written by the unmodified reference (fp32): forward within 5e-6 and first-step
    gradients within 1e-5, the tolerances tests/test_oracle_golden.py holds the oracle to."""
    g = load_golden(name)
    sd = golden_sd(g)
    pos = 100 if bool(g["pos_emb"]) else None
    x = torch.from_numpy(g["input_kp"])
    f = conv_ref.forward(sd, x, pos)
    assert oracle.rel_err(f["pred"].numpy(), g["pred"]) < 5e-6
    for kind in ("L1", "confL1"):
        _, masked, d_pred = conv_ref.criterion(f["pred"], torch.from_numpy(g["target_kp"]), g["lengths"], kind,
                                               torch.from_numpy(g["target_conf"]))
        assert oracle.rel_err(masked.numpy(), g["pred_masked"]) < 5e-6
        gr = conv_ref.backward(sd, x, d_pred, pos, fwd=f)
        for k in conv_ref.NAMES:
            assert oracle.rel_err(gr[k].numpy(), g[f"grad_{kind}_" + k.replace(".", "_")]) < 1e-5, (kind, k)


def test_wide_forward_matches_golden():
    g = load_golden("convmodel_c256_fwd.npz")
    sd = oracle.init_params(int(g["C"]), False, seed=int(g["seed"]))
    f = conv_ref.forward(sd, torch.from_numpy(g["input_kp"]))
    assert oracle.rel_err(f["pred"].numpy(), g["pred"]) < 1e-5


def test_positional_row_follows_max_len():
    """The row is t / max_len for the actual T, as an fp32 quotient, and bf16 rounding rounds that quotient."""
    row = conv_ref.pos_row(129, 37)
    assert row.dtype == torch.float32 and float(row[37]) == 1.0 and float(row[128]) == np.float32(128) / np.float32(37)
    x = torch.zeros(1, 5, 8, 2)
    a0 = conv_ref.forward(oracle.init_params(16, True, seed=0, n_in=16), x, 37, "bf16")["a"][0]
    want = (torch.arange(5).float() / 37).to(torch.bfloat16).double()
    assert a0.shape == (1, 17, 5) and torch.equal(a0[0, 0], want) and not a0[0, 1:].any()
