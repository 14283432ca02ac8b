"""Plain references for the optimizer step of every training path: torch's Adam element update in float64, a numpy
restatement of the packed weight buffer, and the slice count of the tile kernel read off the public workspace size.

`pack_reference` is written from the layout comments of hand_pose_sl_b200/csrc/b2h_common.cuh (struct Geo, make_geo,
umma_b_offset), not from the kernels, so that comparing a buffer the kernels packed against it checks the layout itself."""
import numpy as np
import torch

from hand_pose_sl_b200 import _lib

KW = 5          # kernel_size of every Conv1d
COUT = 42       # 2 * 21 output channels of conv4


def adam_step_f64(p, g, m, v, t, lr, betas=(0.9, 0.999), eps=1e-8, grad_scale=1.0):
    """torch.optim.Adam single-tensor step (amsgrad=False, weight_decay=0, maximize=False) of step number t (1-based)
    in float64, with the gradient scaled by grad_scale first:
        m.lerp_(g, 1-b1); v.mul_(b2).addcmul_(g, g, 1-b2)
        denom = v.sqrt() / sqrt(1-b2^t) + eps;  p.addcdiv_(m, denom, value=-lr/(1-b1^t))
    Returns (p', m', v') as float64 arrays."""
    b1, b2 = float(betas[0]), float(betas[1])
    p, g, m, v = (np.asarray(a, dtype=np.float64) for a in (p, g, m, v))
    g = g * float(grad_scale)
    m = m + (g - m) * (1.0 - b1)
    v = v * b2 + (1.0 - b2) * g * g
    step_size = float(lr) / (1.0 - b1 ** int(t))
    denom = np.sqrt(v) / np.sqrt(1.0 - b2 ** int(t)) + float(eps)
    return p - step_size * (m / denom), m, v


def _ru(x, m):
    return (x + m - 1) // m * m


def layer_shapes(n_in, C, pos_emb):
    """(cin, cout) of conv1..conv4; pos_emb adds the positional row in front of conv1's input channels."""
    cin0 = n_in + (1 if pos_emb else 0)
    return [(cin0, C), (C, C), (C, C), (C, COUT)]


def packed_layout(n_in, C, pos_emb):
    """Byte offsets of the packed buffer's sections (each 128-B aligned, in this order) and its total size:
    wf[4] fp32 forward taps, wd[4] fp32 dgrad taps (layers 2..4), tf[4] bf16 UMMA B forward, td[4] bf16 UMMA B dgrad
    (layers 2..4), tfl[4] bf16 low halves (forward), bias fp32 [4][64]."""
    shapes = layer_shapes(n_in, C, pos_emb)
    off = {"wf": [], "wd": [], "tf": [], "td": [], "tfl": []}
    b = 0
    for cin, cout in shapes:
        off["wf"].append(b); b = _ru(b + KW * cin * cout * 4, 128)
    for l, (cin, cout) in enumerate(shapes):
        off["wd"].append(b)
        if l > 0:
            b = _ru(b + KW * cin * cout * 4, 128)
    for cin, cout in shapes:
        off["tf"].append(b); b = _ru(b + KW * _ru(cin, 16) * _ru(cout, 16) * 2, 128)
    for l, (cin, cout) in enumerate(shapes):
        off["td"].append(b)
        if l > 0:
            b = _ru(b + KW * _ru(cout, 16) * _ru(cin, 16) * 2, 128)
    for cin, cout in shapes:
        off["tfl"].append(b); b = _ru(b + KW * _ru(cin, 16) * _ru(cout, 16) * 2, 128)
    off["bias"] = b
    off["total"] = b + 4 * 64 * 4
    return off


def _bf16_bits(x):
    """Round-to-nearest-even bf16 of float32 x (torch's cast), as uint16 bit patterns."""
    return torch.from_numpy(np.ascontiguousarray(x, dtype=np.float32)).to(torch.bfloat16).view(torch.int16).numpy().view(np.uint16)


def _umma_section(dense):
    """UMMA B-operand section of dense[k][kk][n] (k = tap, kk = reduction index padded to a multiple of 16, n = row
    padded to a multiple of 16): blocks q = k*(KP/16) + s, each [2 k-chunks][N rows][8 bf16], i.e. the element
    (k, kk = 16 s + 8 chunk + within, n) sits at [k][s][chunk][n][within]."""
    K, KP, N = dense.shape
    return dense.reshape(K, KP // 16, 2, 8, N).transpose(0, 1, 2, 4, 3).reshape(-1)


def pack_reference(flat_params, n_in, C, pos_emb):
    """The packed weight buffer (uint8, b2h_packed_bytes long) of the flat fp32 parameters (state_dict order: conv1.weight
    (C, cin, 5), conv1.bias, ..., conv4.bias).  Every byte no layout entry covers is zero."""
    w = np.asarray(flat_params, dtype=np.float32).reshape(-1)
    lay = packed_layout(n_in, C, pos_emb)
    buf = np.zeros(lay["total"], dtype=np.uint8)

    def f32(off, n):
        return buf[off:off + 4 * n].view(np.float32)

    def u16(off, n):
        return buf[off:off + 2 * n].view(np.uint16)

    bias = f32(lay["bias"], 4 * 64).reshape(4, 64)
    o = 0
    for l, (cin, cout) in enumerate(layer_shapes(n_in, C, pos_emb)):
        W = w[o:o + cout * cin * KW].reshape(cout, cin, KW); o += cout * cin * KW
        b = w[o:o + cout]; o += cout
        bias[l, :min(cout, 64)] = b[:64]
        # fp32 forward taps Wf[k][ci][co] = W[co][ci][k]
        f32(lay["wf"][l], KW * cin * cout)[:] = W.transpose(2, 1, 0).reshape(-1)
        # bf16 forward operand: reduction = ci (padded), rows = co (padded); high halves and low halves w - bf16(w)
        hi = _bf16_bits(W)
        lo = _bf16_bits(W - torch.from_numpy(hi.view(np.int16)).view(torch.bfloat16).float().numpy())
        KP, N = _ru(cin, 16), _ru(cout, 16)
        for key, bits in (("tf", hi), ("tfl", lo)):
            dense = np.zeros((KW, KP, N), dtype=np.uint16)
            dense[:, :cin, :cout] = bits.transpose(2, 1, 0)
            u16(lay[key][l], dense.size)[:] = _umma_section(dense)
        if l > 0:
            # fp32 dgrad taps Wd[k'][co][ci] = W[co][ci][4-k']
            f32(lay["wd"][l], KW * cin * cout)[:] = W[:, :, ::-1].transpose(2, 0, 1).reshape(-1)
            # bf16 dgrad operand: reduction = co (padded), rows = ci (padded), tap reversed
            KP, N = _ru(cout, 16), _ru(cin, 16)
            dense = np.zeros((KW, KP, N), dtype=np.uint16)
            dense[:, :cout, :cin] = hi[:, :, ::-1].transpose(2, 0, 1)
            u16(lay["td"][l], dense.size)[:] = _umma_section(dense)
    assert o == w.size, (o, w.size)
    return buf


def gp_total(n_in, C, pos_emb):
    """Slots of one gradient-partial slice: per layer [k][kp/4][cout][4] weight slots (kp = cin padded to 16) and the
    bias slots padded to a multiple of 4."""
    return sum(KW * cout * _ru(cin, 16) + _ru(cout, 4) for cin, cout in layer_shapes(n_in, C, pos_emb))


def _prec(prec):
    return _lib.PRECISIONS[prec] if isinstance(prec, str) else int(prec)


def train_nparts(B, T, n_in, C, pe, prec):
    """Gradient-partial slices (= CTAs) of the tile or the FFMA kernel's training path for this shape, from
    b2h_workspace_bytes: roundup256(1024 + 4 * nparts * (gp_total + 1)) + 256.  The rounding slack is smaller than one
    slice."""
    lib = _lib.load()
    assert lib.b2h_kernel_choice(T, n_in, C, int(pe), _prec(prec), 1) in (1, 2), "not a tile- or FFMA-kernel training shape"
    ws = _lib.workspace_bytes(B, T, n_in, C, pe, _prec(prec))
    return (ws - 256 - 1024) // (4 * (gp_total(n_in, C, pe) + 1))
