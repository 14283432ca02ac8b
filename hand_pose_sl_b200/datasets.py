"""SURVEY.md §8f rows N1 / N3: the data formats either side of the hot path.

N3  `pack_metadata`  -- one-shot converter from the reference's metadata-JSON schema
    (How2Sign/util_scripts/build_dataset.py:56-74, merge_utt_jsons.py:38-47: a list of
    {utt_id, text, n_frames, frame_jsons: [{json_path, json_data}]}) to packed fp32 keypoint arrays, and
    `split_metadata` with the 70/15/15 semantics of split_metadata.py:13-30.
N1  `GpuPoseDataset` -- a torch Dataset that keeps the packed arrays resident on the GPU and yields the item dict of
    FastTextPoseDataset.__getitem__ (body2hand/src/dataloaders/text_pose_dataset.py:430-509: body_kp (T,12,2),
    body_conf (T,12), right_hand_kp/left_hand_kp (T,21,2), *_conf (T,21), n_frames, text, json_paths, + the
    BuildRightHandItem aliases) through ONE K0 launch -- per item, or per batch via `batch(indices)`.
The reference spends its data-loading time in per-frame Python list parsing; here parsing happens once, offline.
Host code only does bookkeeping (offsets, crop starts); every arithmetic op on keypoints runs in K0 (bit-exact)."""
from __future__ import annotations

import random as _random
from dataclasses import dataclass, field

import numpy as np
import torch
from torch.utils.data import Dataset

from .transforms import PreprocessRightHand, select_window


@dataclass
class PackedClips:
    pose25: np.ndarray            # (F, 25, 3) fp32 [x, y, c]
    hand_left: np.ndarray         # (F, 21, 3)
    hand_right: np.ndarray        # (F, 21, 3)
    offsets: np.ndarray           # (U+1,) int64: utterance u owns frames [offsets[u], offsets[u+1])
    n_frames_meta: np.ndarray     # (U,) int64: metadata["n_frames"] (text_pose_dataset.py:447 uses it, not the crop)
    texts: list = field(default_factory=list)
    utt_ids: list = field(default_factory=list)
    json_paths: list = field(default_factory=list)   # per utterance: list of per-frame paths (or None)

    def __len__(self):
        return len(self.offsets) - 1


def _frame_arrays(frame):
    """One frame of the metadata (a dict with "json_data", or the OpenPose dict itself) -> three flat fp32 rows.
    Mirrors load_keypoints' inputs: people[0].pose_keypoints_2d / hand_left_keypoints_2d / hand_right_keypoints_2d
    (text_pose_dataset.py:29-43); face keypoints are never read."""
    data = frame["json_data"] if isinstance(frame, dict) and "json_data" in frame else frame
    person = data["people"][0]
    pose = np.asarray(person["pose_keypoints_2d"], dtype=np.float64).astype(np.float32)       # .float() of the reference
    lh = np.asarray(person["hand_left_keypoints_2d"], dtype=np.float64).astype(np.float32)
    rh = np.asarray(person["hand_right_keypoints_2d"], dtype=np.float64).astype(np.float32)
    if pose.shape[0] != 75 or lh.shape[0] != 63 or rh.shape[0] != 63:
        raise ValueError("expected BODY_25 (75) and 21-point hands (63) OpenPose arrays")
    return pose, lh, rh


def pack_metadata(metadata: list) -> PackedClips:
    """N3: metadata list (build_dataset.py:56-74) -> PackedClips."""
    poses, lhs, rhs, offsets, nmeta, texts, ids, paths = [], [], [], [0], [], [], [], []
    for utt in metadata:
        plist = []
        for fr in utt["frame_jsons"]:
            p, l, r = _frame_arrays(fr)
            poses.append(p); lhs.append(l); rhs.append(r)
            plist.append(fr.get("json_path") if isinstance(fr, dict) else None)
        offsets.append(offsets[-1] + len(utt["frame_jsons"]))
        nmeta.append(int(utt.get("n_frames", len(utt["frame_jsons"]))))
        texts.append(utt.get("text", ""))
        ids.append(utt.get("utt_id"))
        paths.append(plist)
    F = offsets[-1]
    return PackedClips(
        pose25=np.asarray(poses, dtype=np.float32).reshape(F, 25, 3),
        hand_left=np.asarray(lhs, dtype=np.float32).reshape(F, 21, 3),
        hand_right=np.asarray(rhs, dtype=np.float32).reshape(F, 21, 3),
        offsets=np.asarray(offsets, dtype=np.int64), n_frames_meta=np.asarray(nmeta, dtype=np.int64),
        texts=texts, utt_ids=ids, json_paths=paths)


def split_metadata(data: list):
    """split_metadata.py:13-30: train = first 70 %, validation = last 15 %, test = the middle."""
    n = len(data)
    n_train, n_val = int(n * 0.7), int(n * 0.15)
    train = data[:n_train]
    val = data[n - n_val:] if n_val > 0 else []
    test = data[n_train:n - n_val]
    return train, val, test


class GpuPoseDataset(Dataset):
    """N1.  `selection` in {"first", "randomcrop"} (text_pose_dataset.py:52-68); `rng` = a random.Random for the crop
    draw (the reference uses the global `random`).  dif_encoding / normalize / factor = the transform chain of run.py:85-102."""

    def __init__(self, packed: PackedClips, max_frames: int, selection: str = "first", dif_encoding: bool = True,
                 normalize: bool = True, factor: float = 1280, device="cuda", rng=None):
        self.packed, self.max_frames, self.selection = packed, int(max_frames), selection
        self.device = torch.device(device)
        self.rng = rng or _random
        self.pose = torch.from_numpy(packed.pose25).to(self.device)
        self.lh = torch.from_numpy(packed.hand_left).to(self.device)
        self.rh = torch.from_numpy(packed.hand_right).to(self.device)
        self.pre = PreprocessRightHand(factor=factor, dif_encoding=dif_encoding, normalize=normalize, pad_mode="repeat_first")
        self._streams = {}

    def __len__(self):
        return len(self.packed)

    def _crop(self, idx):
        lo, hi = int(self.packed.offsets[idx]), int(self.packed.offsets[idx + 1])
        start, stop = select_window(hi - lo, self.max_frames, self.selection, self.rng)     # :52-68
        return lo + start, lo + stop, start

    def _draw(self, indices):
        """Crop draws (in index order) and sequence lengths of one batch: shared by `batch()` and `crops()`."""
        starts, ends, rel = zip(*(self._crop(int(i)) for i in indices))
        nf = [min(int(self.packed.n_frames_meta[int(i)]), self.max_frames) for i in indices]           # :447
        return starts, ends, rel, nf

    def crops(self, indices):
        """The crop list of a training step over `training_streams()`: {win_start, win_end, n_frames} as CPU int64 (B,)
        tensors -- the same `select_window` draws (one per index, in order) and the same n_frames rule as `batch()`."""
        starts, ends, _, nf = self._draw(indices)
        return {"win_start": torch.tensor(starts, dtype=torch.int64), "win_end": torch.tensor(ends, dtype=torch.int64),
                "n_frames": torch.tensor(nf, dtype=torch.int64)}

    def training_streams(self, dtype=torch.bfloat16):
        """Per-frame training data of ALL packed frames, built once per dtype and cached ({input_kp, target_kp,
        target_conf}, `PreprocessRightHand.training_stream`).  Per-frame preprocessing does not depend on the window, so the
        windows of `crops()` over these streams equal the windows `batch()` materialises with the same draws."""
        if dtype not in self._streams:
            self._streams[dtype] = self.pre.training_stream(self.pose, self.lh, self.rh, dtype=dtype)
        return self._streams[dtype]

    def batch(self, indices):
        """Stacked item dict for several utterances with ONE preprocessing launch (what DataLoader + default_collate
        produce, traintest.py:87): tensors (B,T,...) on the device, n_frames (B,) CPU int64 like the reference
        (traintest.py:91), text / json_paths / utt_id as python lists (collate_function, steps/utils.py:383-396)."""
        starts, ends, rel, nf = self._draw(indices)
        out = self.pre(self.pose, self.lh, self.rh, np.asarray(starts, dtype=np.int64), self.max_frames,
                       win_end=np.asarray(ends, dtype=np.int64))
        out["n_frames"] = torch.tensor(nf, dtype=torch.int64)
        out["text"] = [self.packed.texts[int(i)] for i in indices]
        out["utt_id"] = [self.packed.utt_ids[int(i)] for i in indices]
        out["json_paths"] = [self.packed.json_paths[int(i)][r:r + self.max_frames] for i, r in zip(indices, rel)]
        return out

    def __getitem__(self, idx):
        b = self.batch([idx])
        item = {k: (v[0] if torch.is_tensor(v) and v.dim() > 0 else v) for k, v in b.items()
                if k not in ("text", "utt_id", "json_paths", "n_frames")}
        item["n_frames"] = int(b["n_frames"][0])
        item["text"], item["utt_id"], item["json_paths"] = b["text"][0], b["utt_id"][0], b["json_paths"][0]
        return item
