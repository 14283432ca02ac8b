"""Generates tests/golden/*.npz by EXECUTING THE UNMODIFIED REFERENCE (oracle/ref_loader.py) on seeded
synthetic inputs:  B2H_REFERENCE_ROOT=<checkout of the original project> python oracle/make_golden.py
tests/test_oracle_golden.py reads only the fixtures, so it runs without the reference.  TEST INFRASTRUCTURE ONLY."""
import os
import random
import sys

import numpy as np
import torch

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(HERE)
sys.path.insert(0, ROOT)
sys.path.insert(0, HERE)

import ref_loader  # noqa: E402
from hand_pose_sl_b200 import synthetic  # noqa: E402

OUT = os.path.join(ROOT, "tests", "golden")
PARAM_NAMES = ["conv1.weight", "conv1.bias", "conv2.weight", "conv2.bias",
               "conv3.weight", "conv3.bias", "conv4.weight", "conv4.bias"]


def _np(sd):
    return {k.replace(".", "_"): v.detach().numpy().copy() for k, v in sd.items()}


def golden_model(C, B, T, pos_emb, name, steps=3, lr=2e-4):
    M, U, _ = ref_loader.load()
    torch.manual_seed(0)
    net = M.ConvModel(C, "ReLU", pos_emb)
    sd0 = {k: v.detach().clone() for k, v in net.state_dict().items()}
    batch = synthetic.model_batch(B, T, seed=1234, ragged=True)
    x, tgt, conf, lengths = batch["input_kp"], batch["target_kp"], batch["target_conf"], batch["n_frames"]
    out = {"lengths": lengths.numpy(), "input_kp": x.numpy(), "target_kp": tgt.numpy(),
           "target_conf": conf.numpy(), "C": np.int64(C), "pos_emb": np.int64(pos_emb), "lr": np.float64(lr)}
    out.update({"w0_" + k: v for k, v in _np(sd0).items()})

    with torch.no_grad():
        pred = net(x)
        out["pred"] = pred.contiguous().numpy().copy()
        masked = U.mask_output(pred.clone(), lengths)
        out["pred_masked"] = masked.contiguous().numpy().copy()

    for kind in ("L1", "confL1"):
        net.load_state_dict(sd0)
        crit = U.maskedPoseL1() if kind == "L1" else U.poderatedPoseL1()
        opt = torch.optim.Adam(net.parameters(), lr=lr)            # traintest.py:48
        losses = []
        for s in range(steps):
            pred = net(x)                                          # traintest.py:94
            pred = U.mask_output(pred, lengths)                    # :111
            loss = crit(pred, tgt, lengths) if kind == "L1" else crit(pred, tgt, lengths, conf)  # :115/:117
            opt.zero_grad()
            loss.backward()
            if s == 0:
                out.update({f"grad_{kind}_" + k.replace(".", "_"): p.grad.detach().numpy().copy()
                            for k, p in net.named_parameters()})
            opt.step()
            losses.append(float(loss.item()))
        out[f"loss_{kind}"] = np.asarray(losses, dtype=np.float64)
        out.update({f"w{steps}_{kind}_" + k: v for k, v in _np(net.state_dict()).items()})
    np.savez_compressed(os.path.join(OUT, name), **out)
    print(name, {k: getattr(v, "shape", None) for k, v in out.items() if k in ("pred", "loss_L1", "loss_confL1")},
          out["loss_L1"], out["loss_confL1"])


def golden_preprocess(name="preprocess.npz", F=150, T=64):
    """Reference data path: load_keypoints (per frame dict) -> FastTextPoseDataset.pad/clip/to_tensor
    -> Compose([WristDifference, ChestDifference, NormalizeFixedFactor(1280), BuildRightHandItem])."""
    _, U, D = ref_loader.load()
    pose, lh, rh = synthetic.synthetic_clip(F, seed=1234)
    out = {"pose25": pose, "hand_left": lh, "hand_right": rh, "T": np.int64(T)}
    starts = np.array([0, 48, 96, 120, 149], dtype=np.int64)
    out["win_start"] = starts

    ds = D.FastTextPoseDataset.__new__(D.FastTextPoseDataset)
    ds.max_frames = T
    tf_dif = [U.WristDifference(), U.ChestDifference(), U.NormalizeFixedFactor(1280), U.BuildRightHandItem()]
    tf_nodif = [U.NormalizeFixedFactor(1280), U.BuildRightHandItem()]

    def frame_dict(i):
        # python floats of the fp32 values: float(np.float32) is exact, .float() returns the same fp32
        return {"people": [{"pose_keypoints_2d": [float(v) for v in pose[i].reshape(-1)],
                            "hand_left_keypoints_2d": [float(v) for v in lh[i].reshape(-1)],
                            "hand_right_keypoints_2d": [float(v) for v in rh[i].reshape(-1)]}]}

    for tag, tfs in (("dif", tf_dif), ("nodif", tf_nodif)):
        acc = {}
        for s in starts:
            frames = list(range(int(s), F))
            sel, start = D.select_jsons(frames, T, selection_type="first")          # crop [s, s+T)
            item = {"body_kp": [], "right_hand_kp": [], "left_hand_kp": [],
                    "body_conf": [], "right_hand_conf": [], "left_hand_conf": [], "json_paths": []}
            for fi in sel:
                r_kp, r_cf, l_kp, l_cf, b_kp, b_cf = D.load_keypoints(frame_dict(fi))
                item["body_kp"].append(b_kp); item["body_conf"].append(b_cf)
                item["right_hand_kp"].append(r_kp); item["right_hand_conf"].append(r_cf)
                item["left_hand_kp"].append(l_kp); item["left_hand_conf"].append(l_cf)
                item["json_paths"].append(None)
            item["n_frames"] = min(len(frames), T)                                   # :447
            item = D.FastTextPoseDataset.pad(ds, item)                               # :511-519
            item = D.FastTextPoseDataset.clip(ds, item)                              # :520-529
            item = D.FastTextPoseDataset.to_tensor(ds, item)                         # :536-544
            for t in tfs:
                item = t(item)
            for k in ("input_kp", "input_conf", "target_kp", "target_conf", "left_hand_kp", "left_hand_conf"):
                acc.setdefault(k, []).append(item[k].numpy().copy())
            acc.setdefault("n_frames", []).append(item["n_frames"])
        for k, v in acc.items():
            out[f"{tag}_{k}"] = np.stack(v) if k != "n_frames" else np.asarray(v, dtype=np.int64)

    # H5 path: array2item -> pad(zeros) -> clip -> to_tensor -> transforms   (:587-649)
    h5 = D.TextPoseH5Dataset.__new__(D.TextPoseH5Dataset)
    h5.max_frames = T
    rng = np.random.default_rng(99)
    for tag, n in (("h5short", 40), ("h5long", 90)):
        arr = rng.uniform(0, 1280, size=(n, 150)).astype(np.float32)
        arr[:, 100:] = rng.uniform(0, 1, size=(n, 50)).astype(np.float32)
        item = D.TextPoseH5Dataset.array2item(h5, arr)
        nfr = min(item["body_kp"].shape[0], T)                                      # :661-662
        item = D.TextPoseH5Dataset.pad(h5, item)
        item = D.TextPoseH5Dataset.clip(h5, item)
        item = D.TextPoseH5Dataset.to_tensor(h5, item)
        for t in tf_dif:
            item = t(item)
        out[f"{tag}_array"] = arr
        out[f"{tag}_n_frames"] = np.int64(nfr)
        for k in ("input_kp", "input_conf", "target_kp", "target_conf", "left_hand_kp", "left_hand_conf"):
            out[f"{tag}_{k}"] = item[k].numpy().copy()
    np.savez_compressed(os.path.join(OUT, name), **out)
    print(name, out["dif_input_kp"].shape, out["dif_n_frames"], out["h5short_input_kp"].shape)


def golden_windowing(name="windowing.npz"):
    """select_jsons (text_pose_dataset.py:52-68) under a seeded `random`."""
    _, _, D = ref_loader.load()
    cases = []
    random.seed(7)
    for n_total, n in [(10, 64), (64, 64), (65, 64), (200, 64), (1000, 200), (101, 100), (5000, 64)]:
        for sel in ("first", "randomcrop"):
            for _ in range(3):
                state_probe = random.getstate()
                frames, start = D.select_jsons(list(range(n_total)), n, selection_type=sel)
                # recover the draw the reference made (if any) to feed the index-math restatement
                random.setstate(state_probe)
                draw = random.randint(0, n_total - n) if (n_total > n and sel == "randomcrop") else -1
                cases.append([n_total, n, 0 if sel == "first" else 1, draw, start, frames[0], frames[-1], len(frames)])
    np.savez_compressed(os.path.join(OUT, name), cases=np.asarray(cases, dtype=np.int64))
    print(name, len(cases))


def golden_wide(C=256, B=2, T=64, name="convmodel_c256_fwd.npz"):
    """Wide variant (`--conv-channels 256`): forward only, and only the reference's OUTPUTS are stored -- the 740 650
    weights are the reference's default init right after torch.manual_seed(0), which oracle.init_params(C, seed=0)
    reproduces; per-tensor checksums pin that."""
    M, U, _ = ref_loader.load()
    torch.manual_seed(0)
    net = M.ConvModel(C, "ReLU", False)
    batch = synthetic.model_batch(B, T, seed=4321, ragged=True)
    x, lengths = batch["input_kp"], batch["n_frames"]
    out = {"lengths": lengths.numpy(), "input_kp": x.numpy(), "C": np.int64(C), "seed": np.int64(0)}
    for k, v in net.state_dict().items():
        out["sum_" + k.replace(".", "_")] = np.float64(v.double().sum().item())
        out["abssum_" + k.replace(".", "_")] = np.float64(v.double().abs().sum().item())
    with torch.no_grad():
        pred = net(x)
        out["pred"] = pred.contiguous().numpy().copy()
        out["pred_masked"] = U.mask_output(pred.clone(), lengths).contiguous().numpy().copy()
    np.savez_compressed(os.path.join(OUT, name), **out)
    print(name, out["pred"].shape, float(np.abs(out["pred"]).max()))


def golden_writers(name="writers.npz"):
    """Inference writers (SURVEY 8f N2): array2open_pose (steps/utils.py:355-364), order_and_reshape_toh5
    (steps/traintest.py:302-317), L12Pixels (steps/utils.py:291-299) executed from the reference on a seeded prediction."""
    _, U, _ = ref_loader.load()
    to_h5 = ref_loader.load_function("steps/traintest.py", "order_and_reshape_toh5")
    g = torch.Generator().manual_seed(99)
    pred = (torch.rand((7, 21, 2), generator=g) * 1280.0).float()
    out = {"pred": pred.numpy(),
           "openpose": np.asarray([U.array2open_pose(pred[t].numpy()) for t in range(pred.shape[0])], dtype=np.float64),
           "h5": np.asarray(to_h5(pred)),
           "l1": np.float64(0.0123), "l1_pixels_21": np.float64(U.L12Pixels(21, 1280)(0.0123)),
           "l1_pixels_4": np.float64(U.L12Pixels(4, 1280)(0.0123))}
    np.savez_compressed(os.path.join(OUT, name), **out)
    print(name, out["openpose"].shape, out["h5"].shape, out["h5"].dtype)


if __name__ == "__main__":
    os.makedirs(OUT, exist_ok=True)
    torch.set_num_threads(1)          # deterministic summation order in the fixtures
    golden_model(30, 4, 64, False, "convmodel_c30.npz")
    golden_model(30, 2, 100, True, "convmodel_c30_posemb.npz")
    golden_model(64, 2, 64, False, "convmodel_c64.npz", steps=2)
    golden_model(30, 1, 64, False, "convmodel_c30_b1.npz", steps=1)
    golden_model(30, 3, 200, False, "convmodel_c30_t200.npz", steps=1)
    golden_wide()
    golden_writers()
    golden_preprocess()
    golden_windowing()
