"""CPU tier: the references the optimizer-path tests compare against.  adam_step_f64 is torch.optim.Adam; the packed
buffer restated from the layout comments has the size the library allocates; the tile kernel's slice count read off
the workspace size behaves as the layout says (needs the built libb2h.so, no GPU)."""
import numpy as np
import pytest
import torch

from hand_pose_sl_b200 import _lib
from optim_ref import adam_step_f64, gp_total, pack_reference, packed_layout, tile_nparts


@pytest.mark.parametrize("t", [1, 2, 10, 1000, 100000])
@pytest.mark.parametrize("eps", [1e-8, 1e-3])
@pytest.mark.parametrize("betas", [(0.9, 0.999), (0.8, 0.99)])
def test_adam_step_f64_is_torch_adam(betas, eps, t):
    gen = torch.Generator().manual_seed(t)
    n = 4096
    p = torch.randn(n, generator=gen, dtype=torch.float64)
    g = torch.randn(n, generator=gen, dtype=torch.float64) * 1e-2
    m = torch.randn(n, generator=gen, dtype=torch.float64) * 5e-3
    v = (torch.rand(n, generator=gen, dtype=torch.float64) * 1e-2) ** 2
    lr = 3e-3
    q = p.clone().requires_grad_(True)
    opt = torch.optim.Adam([q], lr=lr, betas=betas, eps=eps)
    opt.load_state_dict({"state": {0: {"step": torch.tensor(float(t - 1)), "exp_avg": m.clone(), "exp_avg_sq": v.clone()}},
                         "param_groups": opt.state_dict()["param_groups"]})
    q.grad = g.clone()
    opt.step()
    st = opt.state[q]
    assert float(st["step"]) == t
    p1, m1, v1 = adam_step_f64(p.numpy(), g.numpy(), m.numpy(), v.numpy(), t, lr, betas, eps)
    for got, want in ((p1, q.detach()), (m1, st["exp_avg"]), (v1, st["exp_avg_sq"])):
        want = want.numpy()
        assert np.max(np.abs(got - want)) <= 1e-12 * np.max(np.abs(want))
    # grad_scale multiplies the gradient before anything else
    p2, m2, v2 = adam_step_f64(p.numpy(), 2 * g.numpy(), m.numpy(), v.numpy(), t, lr, betas, eps)
    p3, m3, v3 = adam_step_f64(p.numpy(), g.numpy(), m.numpy(), v.numpy(), t, lr, betas, eps, grad_scale=2.0)
    assert np.array_equal(p2, p3) and np.array_equal(m2, m3) and np.array_equal(v2, v3)


@pytest.mark.parametrize("pos_emb", [0, 1, 250])
def test_pack_reference_size_matches_library(pos_emb):
    for C in range(1, 257):
        P = _lib.param_count(24, C, pos_emb)
        want = _lib.packed_bytes(24, C, pos_emb)
        assert packed_layout(24, C, pos_emb)["total"] == want, C
        buf = pack_reference(np.zeros(P, dtype=np.float32), 24, C, pos_emb)
        assert buf.size == want and buf.dtype == np.uint8 and not buf.any(), C


def test_pack_reference_places_every_parameter():
    """Each parameter lands in its fp32 forward tap, its bf16 high half and low half, and (layers 2..4) its fp32 and bf16
    dgrad taps; biases only in the [4][64] section.  Distinct values make a collision or a missing entry visible."""
    n_in, C, pe = 24, 30, 1
    P = _lib.param_count(n_in, C, pe)
    w = (np.arange(P, dtype=np.float32) + 1.0) * np.float32(1.0 / 1024)
    buf = pack_reference(w, n_in, C, pe)
    lay = packed_layout(n_in, C, pe)
    f32 = buf[:lay["tf"][0]].view(np.float32)
    bias = buf[lay["bias"]:].view(np.float32).reshape(4, 64)
    weights = np.concatenate([w[_lib.param_offset(n_in, C, pe, l, 0):_lib.param_offset(n_in, C, pe, l, 1)] for l in (1, 2, 3, 4)])
    dgrad = np.concatenate([w[_lib.param_offset(n_in, C, pe, l, 0):_lib.param_offset(n_in, C, pe, l, 1)] for l in (2, 3, 4)])
    # fp32 sections: every weight once in Wf, layers 2..4 once more in Wd, nothing else
    assert np.array_equal(np.sort(f32[f32 != 0]), np.sort(np.concatenate([weights, dgrad])))
    for l in range(4):
        b0 = _lib.param_offset(n_in, C, pe, l + 1, 1)
        cout = 42 if l == 3 else C
        assert np.array_equal(bias[l, :cout], w[b0:b0 + cout]) and not bias[l, cout:].any()
    # conv2.weight[co=3, ci=7, k=1] in Wf[k][ci][co] and Wd[4-k][co][ci]
    i = _lib.param_offset(n_in, C, pe, 2, 0) + (3 * C + 7) * 5 + 1
    assert f32[lay["wf"][1] // 4 + (1 * C + 7) * C + 3] == w[i]
    assert f32[lay["wd"][1] // 4 + ((4 - 1) * C + 3) * C + 7] == w[i]
    # bf16 sections: high halves of every weight (forward + dgrad), low halves only forward
    hi = buf[lay["tf"][0]:lay["tfl"][0]].view(np.uint16)
    n_nonzero_lo = np.count_nonzero(buf[lay["tfl"][0]:lay["bias"]].view(np.uint16))
    assert np.count_nonzero(hi) == weights.size + dgrad.size
    assert 0 < n_nonzero_lo <= weights.size


def test_tile_nparts_follows_the_batch():
    """At T <= 64 the tile kernel packs two windows per CTA and runs at most one CTA per SM (148 on a B200; the library
    assumes 148 when no device is present)."""
    for B in (1, 2, 4, 127, 128, 130, 166, 168, 256, 296, 300):
        for prec in ("fp32", "bf16"):
            assert tile_nparts(B, 64, 24, 30, 0, prec) == min(148, (B + 1) // 2), (B, prec)
    assert gp_total(24, 30, 0) == 21260 and gp_total(24, 80, 0) == 93884 and gp_total(24, 96, 0) == 128012
