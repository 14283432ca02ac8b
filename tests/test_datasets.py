"""SURVEY §8f rows N1/N3: metadata-JSON -> packed arrays (CPU) and the GPU-resident dataset (GPU) against the
reference's own FastTextPoseDataset methods / the oracle."""
import random

import numpy as np
import pytest
import torch

import b2h_oracle as oracle
import hand_pose_sl_b200 as b2h
import ref_loader
from hand_pose_sl_b200 import synthetic


def _metadata(n_utt=5, seed=0):
    rng = np.random.default_rng(seed)
    meta = []
    for u in range(n_utt):
        n = int(rng.integers(3, 90))
        pose, lh, rh = synthetic.synthetic_clip(n, seed=seed * 100 + u)
        frames = [{"json_path": f"utt{u}/frame{i:04d}.json",
                   "json_data": {"people": [{"pose_keypoints_2d": [float(v) for v in pose[i].reshape(-1)],
                                             "hand_left_keypoints_2d": [float(v) for v in lh[i].reshape(-1)],
                                             "hand_right_keypoints_2d": [float(v) for v in rh[i].reshape(-1)],
                                             "face_keypoints_2d": [0.0] * 210}]}} for i in range(n)]
        meta.append({"utt_id": f"utt{u}", "text": f"sentence {u}", "n_frames": n, "frame_jsons": frames})
    return meta


def test_pack_metadata_round_trip():
    meta = _metadata()
    pk = b2h.pack_metadata(meta)
    assert len(pk) == 5 and pk.offsets[-1] == sum(m["n_frames"] for m in meta)
    u, i = 3, 2
    fr = meta[u]["frame_jsons"][i]["json_data"]["people"][0]
    f = int(pk.offsets[u]) + i
    assert np.array_equal(pk.pose25[f].reshape(-1), np.asarray(fr["pose_keypoints_2d"], dtype=np.float32))
    assert np.array_equal(pk.hand_right[f].reshape(-1), np.asarray(fr["hand_right_keypoints_2d"], dtype=np.float32))
    assert pk.texts[u] == "sentence 3" and pk.json_paths[u][i] == "utt3/frame0002.json"


def test_split_metadata_semantics():
    data = list(range(20))
    tr, va, te = b2h.split_metadata(data)
    assert tr == data[:14] and va == data[-3:] and te == data[14:17]       # split_metadata.py:13-30
    assert len(tr) + len(va) + len(te) == 20


@pytest.mark.gpu
@pytest.mark.parametrize("selection", ["first", "randomcrop"])
def test_gpu_dataset_matches_reference_items(selection):
    """Items of GpuPoseDataset == what the reference's load_keypoints / pad / clip / to_tensor / Compose produce
    (restated in the oracle, pinned against the reference in tests/test_oracle_golden.py) -- bit-exact."""
    T = 40
    meta = _metadata(n_utt=6, seed=3)
    pk = b2h.pack_metadata(meta)
    ds = b2h.GpuPoseDataset(pk, max_frames=T, selection=selection, rng=random.Random(11))
    chk = random.Random(11)
    for u in range(len(ds)):
        item = ds[u]
        n = meta[u]["n_frames"]
        start, stop = oracle.select_window(n, T, selection, chk.randint(0, n - T) if (n > T and selection == "randomcrop") else None)
        lo = int(pk.offsets[u])
        want = oracle.preprocess_windows(pk.pose25[lo:lo + n], pk.hand_left[lo:lo + n], pk.hand_right[lo:lo + n],
                                         np.array([start]), T)
        for k in ("input_kp", "input_conf", "target_kp", "target_conf", "left_hand_kp", "left_hand_conf", "body_kp", "right_hand_kp"):
            assert np.array_equal(item[k].cpu().numpy(), want[k if k in want else k][0]), (u, k)
        assert item["n_frames"] == min(n, T) and item["text"] == f"sentence {u}"
        assert item["json_paths"][0] == f"utt{u}/frame{start:04d}.json"
    # one launch for a whole batch == the stacked items
    ds2 = b2h.GpuPoseDataset(pk, max_frames=T, selection="first")
    b = ds2.batch([0, 2, 5])
    for j, u in enumerate([0, 2, 5]):
        it = ds2[u]
        assert torch.equal(b["input_kp"][j], it["input_kp"]) and torch.equal(b["target_kp"][j], it["target_kp"])
    assert b["n_frames"].device.type == "cpu" and b["n_frames"].dtype == torch.int64      # traintest.py:91


@pytest.mark.skipif(not ref_loader.available(), reason="needs B2H_REFERENCE_ROOT: a checkout of the original project")
def test_pack_metadata_feeds_reference_identically():
    """The packed arrays hold exactly the numbers the reference's load_keypoints reads from the same metadata."""
    _, _, D = ref_loader.load()
    meta = _metadata(n_utt=2, seed=9)
    pk = b2h.pack_metadata(meta)
    fr = meta[1]["frame_jsons"][4]["json_data"]
    r_kp, r_cf, l_kp, l_cf, b_kp, b_cf = D.load_keypoints(fr)
    f = int(pk.offsets[1]) + 4
    got = oracle.load_keypoints_arrays(pk.pose25[f:f + 1].reshape(1, 75), pk.hand_left[f:f + 1].reshape(1, 63), pk.hand_right[f:f + 1].reshape(1, 63))
    assert np.array_equal(got[4][0], np.asarray(b_kp, dtype=np.float32)) and np.array_equal(got[0][0], np.asarray(r_kp, dtype=np.float32))
    assert np.array_equal(got[5][0], np.asarray(b_cf, dtype=np.float32))
