"""CPU tier: the oracle against the live, unmodified reference classes (skipped unless B2H_REFERENCE_ROOT names a
checkout of the original project; tests/test_oracle_golden.py checks the oracle against its stored outputs)."""
import numpy as np
import pytest
import torch

import b2h_oracle as oracle
import ref_loader
from hand_pose_sl_b200 import synthetic

pytestmark = pytest.mark.skipif(not ref_loader.available(), reason="needs B2H_REFERENCE_ROOT: a checkout of the original project")


@pytest.mark.parametrize("C,B,T,pe", [(30, 3, 64, False), (30, 2, 100, True), (48, 2, 37, False)])
def test_forward_loss_grads_live(C, B, T, pe):
    M, U, _ = ref_loader.load()
    torch.manual_seed(0)
    net = M.ConvModel(C, "ReLU", pe)
    sd = oracle.init_params(C, pe, seed=0)
    for k, v in net.state_dict().items():
        assert torch.equal(v, sd[k]), k                  # same construction order -> same init
    batch = synthetic.model_batch(B, T, seed=7, ragged=True, len_seed=11)
    x, tgt, conf, ln = batch["input_kp"], batch["target_kp"], batch["target_conf"], batch["n_frames"]
    ref = net(x)
    mine = oracle.conv_model_forward(sd, x, pe)
    assert torch.equal(ref, mine)
    ref_m = U.mask_output(ref.clone(), ln)
    assert torch.equal(ref_m, oracle.mask_output(mine.clone(), ln))
    assert float(U.maskedPoseL1()(ref_m, tgt, ln)) == float(oracle.masked_pose_l1(ref_m, tgt, ln))
    assert float(U.poderatedPoseL1()(ref_m, tgt, ln, conf)) == float(oracle.poderated_pose_l1(ref_m, tgt, ln, conf))


def test_transforms_live():
    _, U, D = ref_loader.load()
    pose, lh, rh = synthetic.synthetic_clip(40, seed=5)
    out = oracle.preprocess_windows(pose, lh, rh, np.array([0]), 40)
    r_kp, r_cf, l_kp, l_cf, b_kp, b_cf = oracle.load_keypoints_arrays(pose.reshape(40, 75), lh.reshape(40, 63), rh.reshape(40, 63))
    item = {"body_kp": torch.tensor(b_kp), "right_hand_kp": torch.tensor(r_kp), "left_hand_kp": torch.tensor(l_kp),
            "body_conf": torch.tensor(b_cf), "right_hand_conf": torch.tensor(r_cf), "left_hand_conf": torch.tensor(l_cf)}
    for t in (U.WristDifference(), U.ChestDifference(), U.NormalizeFixedFactor(1280), U.BuildRightHandItem()):
        item = t(item)
    assert np.array_equal(item["input_kp"].numpy(), out["input_kp"][0])
    assert np.array_equal(item["target_kp"].numpy(), out["target_kp"][0])
    assert np.array_equal(item["left_hand_kp"].numpy(), out["left_hand_kp"][0])


def test_writers_live():
    """array2open_pose / L12Pixels from steps/utils.py and order_and_reshape_toh5 from steps/traintest.py (taken from
    the file unmodified: the module itself needs h5py and package-relative imports)."""
    _, U, _ = ref_loader.load()
    to_h5 = ref_loader.load_function("steps/traintest.py", "order_and_reshape_toh5")
    pred = (torch.rand((5, 21, 2), generator=torch.Generator().manual_seed(3)) * 1280.0).float()
    for t in range(5):
        assert np.array_equal(np.asarray(U.array2open_pose(pred[t].numpy())), oracle.array2open_pose(pred[t].numpy()).astype(np.float64))
    assert np.array_equal(to_h5(pred), oracle.order_and_reshape_toh5(pred.numpy()))
    assert U.L12Pixels(21, 1280)(0.5) == oracle.l1_to_pixels(0.5, 21, 1280)


def test_host_scalars_live():
    """The host-side mirrors (a17): adjust_learning_rate (steps/utils.py:301-307) and L12Pixels (:291-299)."""
    import hand_pose_sl_b200 as b2h
    _, U, _ = ref_loader.load()
    w = torch.nn.Parameter(torch.zeros(3))
    for epoch in (0, 1, 7, 30):
        o_ref, o_mine = torch.optim.Adam([w], lr=1.0), torch.optim.Adam([w], lr=1.0)
        assert U.adjust_learning_rate(2e-4, 10, o_ref, epoch) == b2h.adjust_learning_rate(2e-4, 10, o_mine, epoch)
        assert o_ref.param_groups[0]["lr"] == o_mine.param_groups[0]["lr"]
    for joints in (4, 12, 21):
        assert U.L12Pixels(joints, 1280)(0.0371) == b2h.L12Pixels(joints, 1280)(0.0371)
