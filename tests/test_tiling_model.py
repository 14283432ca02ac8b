"""CPU tier: a numpy model of the tensor-core kernels' tiling (b2h_train_tc.cuh / b2h_wide_tc.cuh) against the oracle.

The kernels pack whole windows into a row segment `[2 zero rows][window][2 zero rows][window]...`, compute every conv as
`out[row 2+m] = bias + sum_k W_k . in[row m+k]` over the WHOLE segment (tap k = +k rows of the operand's start address)
and zero the rows that are not real frames.  This model executes exactly that arithmetic in float64 with the plans'
geometry (segment rows MB, windows per segment gh = (MB+2)//(T+2), rows past a window's end invalid) and must reproduce
the reference forward: shared zero rows really isolate neighbouring windows, for every T and batch tail."""
import numpy as np
import pytest
import torch

import b2h_oracle as oracle
from hand_pose_sl_b200 import synthetic


def plan(T, wide):
    """(segment rows MB, segments per tile, windows per segment) as plan_tile / plan_wide choose them."""
    if wide:
        return 256, 1, 258 // (T + 2)
    if T <= 64:
        return 64, 2, 66 // (T + 2)
    mb = 256 if T > 128 else 128
    return mb, 1, (mb + 2) // (T + 2)


def tiled_forward(sd, x, wide):
    B, T = x.shape[:2]
    MB, nseg, gh = plan(T, wide)
    assert gh >= 1
    W = [sd[f"conv{i}.weight"].double().numpy() for i in range(1, 5)]        # (co, ci, k)
    b = [sd[f"conv{i}.bias"].double().numpy() for i in range(1, 5)]
    xin = x.reshape(B, T, -1).double().numpy()
    y = np.zeros((B, T, 42))
    wpt = nseg * gh
    for tile in range((B + wpt - 1) // wpt):
        for h in range(nseg):
            m = np.arange(MB)
            wj, t = m // (T + 2), m % (T + 2)
            gw = tile * wpt + h * gh + wj
            valid = (t < T) & (wj < gh) & (gw < B)
            buf = np.zeros((MB + 8, xin.shape[2]))                              # HR = MB + 8 rows, rows 0,1 and the tail stay zero
            buf[2 + m[valid]] = xin[gw[valid], t[valid]]
            for l in range(4):
                out = np.zeros((MB, W[l].shape[0]))
                for k in range(5):
                    out += buf[m + k] @ W[l][:, :, k].T                          # output row 2+m reads input row m+k
                out += b[l]
                if l < 3:
                    out = np.maximum(out, 0.0)
                out[~valid] = 0.0                                               # the epilogue writes zeros on non-frame rows
                buf = np.zeros((MB + 8, out.shape[1]))
                buf[2 + m] = out
            y[gw[valid], t[valid]] = out[valid]
    return y


@pytest.mark.parametrize("B,T,C,wide", [(5, 64, 30, False), (7, 21, 30, False), (3, 9, 16, False), (4, 65, 30, False),
                                        (3, 126, 30, False), (2, 128, 24, False), (3, 129, 30, False), (2, 200, 30, False),
                                        (2, 256, 30, False), (7, 64, 48, True), (5, 126, 40, True), (2, 200, 40, True),
                                        (4, 1, 30, False), (10, 31, 40, True)])
def test_tiling_reproduces_the_reference_forward(B, T, C, wide):
    sd = oracle.init_params(C, False, seed=B * 7 + T)
    x = synthetic.model_batch(B, T, seed=B * 100 + T)["input_kp"]
    ref = oracle.conv_model_forward_f64(sd, x.numpy())
    got = tiled_forward(sd, x, wide).reshape(B, T, 21, 2)
    assert oracle.rel_err(got, ref) < 1e-10


def test_windows_per_tile():
    assert plan(64, False) == (64, 2, 1) and plan(31, False) == (64, 2, 2) and plan(9, False) == (64, 2, 6)
    assert plan(126, False) == (128, 1, 1) and plan(200, False) == (256, 1, 1)
    assert plan(64, True) == (256, 1, 3) and plan(126, True) == (256, 1, 2) and plan(200, True) == (256, 1, 1)


def tiled_train(sd, x, target, lengths):
    """fwd + masked L1 + bwd in the tile formulation (b2h_train_tc.cuh): dgrad dA_{l-1}[row] = sum_k' dZ_l[row+k'-2] W_l[.,.,4-k'],
    ReLU mask on the saved activation, wgrad dW_l[k] = sum_rows dZ_l[row]^T in_l[row+k-2] over the WHOLE segment (zero rows
    included), bias gradient = dZ_l^T ones(valid rows).  float64; returns (loss, grads dict)."""
    B, T = x.shape[:2]
    MB, nseg, gh = plan(T, False)
    W = [sd[f"conv{i}.weight"].double().numpy() for i in range(1, 5)]
    b = [sd[f"conv{i}.bias"].double().numpy() for i in range(1, 5)]
    xin = x.reshape(B, T, -1).double().numpy()
    tgt = target.reshape(B, T, -1).double().numpy()
    ln = np.asarray(lengths)
    gW = [np.zeros_like(w) for w in W]
    gb = [np.zeros_like(v) for v in b]
    loss = 0.0
    wpt = nseg * gh
    HR = MB + 8
    for tile in range((B + wpt - 1) // wpt):
        for h in range(nseg):
            m = np.arange(MB)
            wj, t = m // (T + 2), m % (T + 2)
            gw = tile * wpt + h * gh + wj
            valid = (t < T) & (wj < gh) & (gw < B)
            gwc = np.where(valid, gw, 0)
            acts = [np.zeros((HR, xin.shape[2]))]
            acts[0][2 + m[valid]] = xin[gw[valid], t[valid]]
            for l in range(4):
                out = sum(acts[l][m + k] @ W[l][:, :, k].T for k in range(5)) + b[l]
                if l < 3:
                    out = np.maximum(out, 0.0)
                out[~valid] = 0.0
                buf = np.zeros((HR, out.shape[1]))
                buf[2 + m] = out
                acts.append(buf)
            pred = acts[4][2 + m]
            live = valid & (t < ln[gwc])                                   # mask_output + loss only on t < len
            d = np.where(live[:, None], pred - tgt[gwc, np.minimum(t, T - 1)], 0.0)
            n_el = (ln[gwc] * 42.0)[:, None]
            loss += np.where(live[:, None], np.abs(d) / n_el, 0.0).sum() / B
            dz = np.zeros((HR, 42))
            dz[2 + m] = np.where(live[:, None], np.sign(d) / (B * n_el), 0.0)
            ones = np.zeros(HR)
            ones[2 + m[valid]] = 1.0
            for l in range(3, -1, -1):
                rows = 2 + m
                for k in range(5):
                    gW[l][:, :, k] += dz[rows].T @ acts[l][rows + k - 2]      # K loop over the segment's rows
                gb[l] += dz[rows].T @ ones[rows]
                if l > 0:
                    da = sum(dz[m + kp] @ W[l][:, :, 4 - kp] for kp in range(5))   # dA row 2+m reads dZ rows m+k'
                    da = np.where((acts[l][2 + m] > 0.0) & valid[:, None], da, 0.0)
                    dz = np.zeros((HR, da.shape[1]))
                    dz[2 + m] = da
    grads = {}
    for i in range(4):
        grads[f"conv{i + 1}.weight"], grads[f"conv{i + 1}.bias"] = gW[i], gb[i]
    return loss, grads


@pytest.mark.parametrize("B,T,C", [(5, 64, 30), (7, 21, 16), (3, 101, 24), (2, 200, 30), (4, 9, 30)])
def test_tiling_reproduces_the_reference_train_step(B, T, C):
    sd = oracle.init_params(C, False, seed=B + T)
    batch = synthetic.model_batch(B, T, seed=3 * B + T, ragged=True, len_seed=T)
    loss, grads = tiled_train(sd, batch["input_kp"], batch["target_kp"], batch["n_frames"])
    st = oracle.TrainState(sd)
    ref_loss, ref_g = oracle.train_step(st, batch["input_kp"], batch["target_kp"], batch["n_frames"], "L1")
    assert abs(loss - ref_loss) <= 1e-6 * abs(ref_loss)
    for k, v in grads.items():
        # float64 model vs the fp32 reference: a residual within fp32 noise of zero may take the other sign (L1)
        assert oracle.rel_err(v, ref_g[k].numpy()) <= 1e-4, k        # observed <= 1e-6 on these seeds


@pytest.mark.parametrize("T,prec", [(129, "fp32"), (160, "fp32"), (200, "fp32"), (224, "fp32"), (225, "fp32"), (256, "fp32"), (300, "fp32"),
                                    (257, "bf16"), (480, "bf16"), (481, "bf16"), (1000, "bf16")])
def test_subwindow_decomposition_reproduces_the_window_gradient(T, prec):
    """fp32 mode trains 129..256-frame windows as overlapping 128-frame sub-windows (b2h_train_subwindows): each reads REAL
    context frames at its cuts and applies the criterion to its core rows only.  CPU proof, with the library's own cut
    points and the oracle's formulas in float64: the losses and ALL parameter gradients of the sub-windows sum to the
    window's (the backward is linear in d(loss)/d(pred); activations are exact up to 8 frames from a cut and dZ reaches at
    most 6 frames beyond the core, so >= 16 frames of context suffice)."""
    import ctypes
    import torch
    import torch.nn.functional as F
    from hand_pose_sl_b200 import _lib
    lib = _lib.load()
    P = _lib.PRECISIONS[prec]
    Ts = 128 if prec == "fp32" else 256
    n = lib.b2h_train_subwindows(T, 24, 30, 0, P, 0, None)
    assert n >= 2 and 2 * (Ts - 16) + (n - 2) * (Ts - 32) >= T and (n == 2 or 2 * (Ts - 16) + (n - 3) * (Ts - 32) < T)
    assert lib.b2h_train_subwindows(Ts, 24, 30, 0, P, 0, None) == 1
    subs = []
    for i in range(n):
        out = (ctypes.c_int * 4)()
        assert lib.b2h_train_subwindows(T, 24, 30, 0, P, i, out) == n
        subs.append(tuple(out))
    # the cores tile [0, T) and every interior cut has >= 16 frames of context inside its sub-window
    cores = [(s + lo, s + hi) for s, lo, hi, L in subs]
    assert cores[0][0] == 0 and cores[-1][1] == T and all(cores[i][1] == cores[i + 1][0] for i in range(n - 1))
    for i, (s, lo, hi, L) in enumerate(subs):
        assert L == Ts and 0 <= s <= T - L and (i == 0 or lo >= 16) and (i == n - 1 or hi + 16 <= L)
    torch.manual_seed(T)
    sd = {k: v.double() for k, v in oracle.init_params(30, False, seed=T).items()}
    x = torch.randn(T, 24, dtype=torch.float64) * 0.2
    tgt = torch.randn(T, 42, dtype=torch.float64) * 0.1
    length = T - 37

    def grads(xs, ts, live, n_el):            # xs (L,24): forward with zero padding at the ends, L1 over the `live` rows
        ps = {k: v.clone().requires_grad_(True) for k, v in sd.items()}
        h = xs.t()[None]
        for l in range(1, 5):
            h = F.conv1d(h, ps[f"conv{l}.weight"], ps[f"conv{l}.bias"], padding=2)
            if l < 4:
                h = F.relu(h)
        pred = h[0].t()
        loss = ((pred - ts).abs() * live[:, None]).sum() / n_el
        loss.backward()
        return loss.detach(), {k: v.grad for k, v in ps.items()}

    live_full = (torch.arange(T) < length).double()
    ref_loss, ref_g = grads(x, tgt, live_full, length * 42)
    tot_loss, tot_g = 0.0, None
    for s, lo, hi, L in subs:
        t = torch.arange(L)
        live = ((t >= lo) & (t < hi) & (s + t < length)).double()
        l_i, g_i = grads(x[s:s + L], tgt[s:s + L], live, length * 42)
        tot_loss = tot_loss + l_i
        tot_g = g_i if tot_g is None else {k: tot_g[k] + g_i[k] for k in g_i}
    assert abs(float(tot_loss) - float(ref_loss)) <= 1e-12 * abs(float(ref_loss))
    for k in ref_g:
        assert float((tot_g[k] - ref_g[k]).abs().max()) <= 1e-12 * float(ref_g[k].abs().max()), k
