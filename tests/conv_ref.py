"""Plain reference of ConvModel's forward, its backward for an arbitrary d(loss)/d(prediction), and the two criteria, for
every input layout (any number of input channels, with or without the positional row t / max_len) and the two rounding
models of the kernels.  torch in float64 (or in float32, to measure how much a summation order alone moves a result);
imports nothing from the package.

    conv_l(a)[b, o, t] = bias_l[o] + sum_{i,k} W_l[o, i, k] a[b, i, t + k - 2]      (zeros outside [0, T))
    a_0 = [pos row | x],  a_l = ReLU(conv_l(a_{l-1})) for l = 1..3,  prediction = conv_4(a_3)

`rounding` says where operands are rounded before they enter a product:
  "none": nowhere.  Models the FFMA kernel (any precision mode) and is the exact value the fp32 mode is judged against.
  "bf16": the weights, the input (the positional row included), the post-ReLU activations and every d(loss)/d(pre-
          activation) (d_y included) go to bf16; sums, biases, the criterion and the ReLU decisions stay exact.  This is
          the tile, row-space and wide kernels in bf16 mode: they stage the positional row as the fp32 quotient t / max_len
          rounded to bf16 like every other input channel (b2h_train_tc.cuh, b2h_conv_tc.cu, b2h_wide_tc.cuh staging).
"""
import torch
import torch.nn.functional as F

NAMES = ["conv1.weight", "conv1.bias", "conv2.weight", "conv2.bias", "conv3.weight", "conv3.bias", "conv4.weight",
         "conv4.bias"]
ROUNDINGS = ("none", "bf16")


def _rounder(rounding):
    if rounding == "none":
        return lambda t: t
    if rounding == "bf16":
        return lambda t: t.to(torch.bfloat16).to(t.dtype)
    raise ValueError(rounding)


def pos_row(T, max_len):
    """LinearPositionalEmbedding's row for a T-frame window: the fp32 quotient t / max_len (HandPoseModels.py:70-75,
    generated for any T)."""
    return torch.arange(T).float() / max_len


def _input(x, pos, rnd, dtype):
    """(B, T, K, 2) or (B, T, n_in) -> a_0 (B, [1 +] n_in, T), rounded."""
    x = torch.as_tensor(x)
    B, T = x.shape[:2]
    a = rnd(x.reshape(B, T, -1).to(dtype)).permute(0, 2, 1)
    if pos is not None:
        row = rnd(pos_row(T, pos).to(dtype))
        a = torch.cat([row[None, None, :].expand(B, 1, T), a], dim=1)
    return a.contiguous()


def _weights(sd, rnd, dtype):
    W = [rnd(torch.as_tensor(sd[f"conv{l}.weight"]).to(dtype)) for l in range(1, 5)]
    b = [torch.as_tensor(sd[f"conv{l}.bias"]).to(dtype) for l in range(1, 5)]
    return W, b


def forward(sd, x, pos=None, rounding="none", dtype=torch.float64):
    """Returns {"z": [z_1..z_4] pre-activations (B, C_l, T), "a": [a_0..a_3] layer inputs (a_0 = the rounded input with
    the positional row in front, a_l = the rounded post-ReLU activations), "pred": (B, T, 21, 2)}.  `pos` is None (no
    positional row) or max_len."""
    rnd = _rounder(rounding)
    W, b = _weights(sd, rnd, dtype)
    a = [_input(x, pos, rnd, dtype)]
    z = []
    for l in range(4):
        z.append(F.conv1d(a[-1], W[l], b[l], padding=2))
        if l < 3:
            a.append(rnd(F.relu(z[-1])))
    B, _, T = z[3].shape
    return {"z": z, "a": a, "pred": z[3].permute(0, 2, 1).reshape(B, T, 21, 2)}


def backward(sd, x, d_y, pos=None, rounding="none", dtype=torch.float64, fwd=None, upstream=None):
    """All eight parameter gradients (dict by state_dict name) of sum(prediction * d_y) for an arbitrary d_y (B, T, 21, 2):
    what ConvModel's backward computes below the criterion.  Every row of d_y counts (nothing is masked here).
    `upstream` (a list, optional) receives d(loss)/d(a_l) before the ReLU mask for l = 3, 2, 1 (index l - 1)."""
    rnd = _rounder(rounding)
    W, _ = _weights(sd, rnd, dtype)
    f = fwd if fwd is not None else forward(sd, x, pos, rounding, dtype)
    a, z = f["a"], f["z"]
    B, T = a[0].shape[0], a[0].shape[2]
    dz = rnd(torch.as_tensor(d_y).to(dtype).reshape(B, T, 42).permute(0, 2, 1))
    g = {}
    if upstream is not None:
        upstream[:] = [None] * 3
    for l in (3, 2, 1, 0):
        g[f"conv{l + 1}.weight"] = torch.nn.grad.conv1d_weight(a[l], W[l].shape, dz, padding=2)
        g[f"conv{l + 1}.bias"] = dz.sum(dim=(0, 2))
        if l > 0:
            up = torch.nn.grad.conv1d_input(a[l].shape, W[l], dz, padding=2)
            if upstream is not None:
                upstream[l - 1] = up
            dz = rnd(up * (z[l - 1] > 0).to(dtype))
    return {k: g[k] for k in NAMES}


def criterion(pred, target, lengths, kind, conf=None):
    """mask_output (steps/utils.py:309-312) followed by maskedPoseL1 ("L1", batch mean of per-sample means,
    :413-428) or poderatedPoseL1 ("confL1", batch sum of per-sample means of the confidence-weighted residual,
    :431-452).  Returns (loss, masked prediction, d(loss)/d(pred)) in pred's dtype; d(loss)/d(pred) is zero on the masked
    rows.  |r| has the derivative sign(r) (0 at r = 0, as torch's l1_loss)."""
    pred = torch.as_tensor(pred)
    dtype = pred.dtype
    B, T = pred.shape[:2]
    ln = torch.as_tensor(lengths, dtype=torch.int64).reshape(B)
    mask = (torch.arange(T)[None, :] < ln[:, None]).to(dtype)[:, :, None, None]
    p = pred * mask
    tg = torch.as_tensor(target).to(dtype)
    n_el = (ln.to(dtype) * 42)[:, None, None, None]
    if kind == "L1":
        s = torch.ones_like(p)
        scale = 1.0 / (B * n_el)
    elif kind == "confL1":
        s = torch.as_tensor(conf).to(dtype)[:, :, :, None].expand(B, T, 21, 2)
        scale = 1.0 / n_el
    else:
        raise ValueError(kind)
    r = p * s - tg * s
    loss = ((r.abs() * mask) * scale).sum()
    d = torch.sign(r) * s * mask * scale
    return loss, p, d


def relu_flip_allowance(sd, fwd, upstream, eps):
    """Elementwise bound (dict by name) on how far the gradients of backward(rounding="none") move when any hidden
    pre-activation within eps * max|z_m| of zero takes the other ReLU decision: such a flip adds or removes one upstream
    value at one (window, channel, frame) of dZ_m, which reaches the weight and bias gradients of layer m + 1 and, through
    the dgrad chain, the layers below.  The effects of the flips are summed in absolute value (first order: two flips
    interact only through each other's tiny activations)."""
    W, _ = _weights(sd, _rounder("none"), fwd["z"][0].dtype)
    a, z = fwd["a"], fwd["z"]
    bound = {f"conv{l + 1}.weight": torch.zeros_like(W[l]) for l in range(4)}
    bound.update({f"conv{l + 1}.bias": torch.zeros(W[l].shape[0], dtype=W[l].dtype) for l in range(4)})
    for m in range(3):
        thr = eps * float(z[m].abs().max())
        for b, c, t in (z[m].abs() <= thr).nonzero().tolist():
            dz = torch.zeros_like(z[m][b:b + 1])
            dz[0, c, t] = upstream[m][b, c, t]
            for l in range(m, -1, -1):
                bound[f"conv{l + 1}.weight"] += torch.nn.grad.conv1d_weight(a[l][b:b + 1], W[l].shape, dz, padding=2).abs()
                bound[f"conv{l + 1}.bias"] += dz.sum(dim=(0, 2)).abs()
                if l > 0:
                    dz = torch.nn.grad.conv1d_input(a[l][b:b + 1].shape, W[l], dz, padding=2) * (z[l - 1][b:b + 1] > 0).to(dz.dtype)
    return bound
