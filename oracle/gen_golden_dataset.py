"""Golden vectors for the segment-index rules, produced by the UNMODIFIED reference dataset.py.

Run in the build container (needs /root/reference):  python -m oracle.gen_golden_dataset
Writes tests/golden/dataset_indices.npz: for a grid of (num_frames, num_segments, new_length) the outputs of
TSNDataSet._get_val_indices / _get_test_indices, and of _sample_indices under numpy.random.seed(SEED + case#).
Cases where the reference itself raises (a video shorter than new_length) are recorded as such.
"""
from __future__ import annotations

import os
import sys

import numpy as np
import torch

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, os.path.dirname(HERE))
from oracle import ref_shims  # noqa: E402

GOLDEN_PATH = os.path.join(os.path.dirname(HERE), "tests", "golden", "dataset_indices.npz")
SEED = 20240
FRAMES = list(range(1, 41)) + [57, 64, 100, 123, 250, 1000]
SEGMENTS = [1, 2, 3, 5, 9, 25]
NEW_LENGTH = [1, 5]


def grid():
    return [(nf, ns, nl) for nl in NEW_LENGTH for ns in SEGMENTS for nf in FRAMES]


def make_tree(root, n_videos=7, feat_dim=16, seed=3):
    """A miniature dataset in the reference's on-disk format: <root>/vK/img_00001.t7 ... one tensor per frame."""
    g = torch.Generator().manual_seed(seed)
    lines = []
    for v in range(n_videos):
        nf = int(torch.randint(2, 14, (1,), generator=g))
        d = os.path.join(root, f"v{v}")
        os.makedirs(d)
        for f in range(1, nf + 1):
            torch.save(torch.randn(feat_dim, generator=g), os.path.join(d, "img_{:05d}.t7".format(f)))
        lines.append(f"{d} {nf} {v % 3}")
    lst = os.path.join(root, "list.txt")
    with open(lst, "w") as fh:
        fh.write("\n".join(lines) + "\n")
    return lst


def reference_dataset(num_segments, new_length, tmp_list):
    ds_mod = ref_shims.load_dataset()
    return ds_mod.TSNDataSet("", tmp_list, num_dataload=1, num_segments=num_segments, new_length=new_length,
                             modality="RGB", random_shift=False, test_mode=True), ds_mod


def main():
    import tempfile
    out = {}
    with tempfile.TemporaryDirectory() as tmp:
        lst = os.path.join(tmp, "list.txt")
        with open(lst, "w") as f:
            f.write("video_0 10 0\n")
        for c, (nf, ns, nl) in enumerate(grid()):
            ds, mod = reference_dataset(ns, nl, lst)
            rec = mod.VideoRecord(["v", str(nf), "0"])
            key = f"{nf}_{ns}_{nl}"
            for name, fn in (("val", ds._get_val_indices), ("test", ds._get_test_indices), ("sample", ds._sample_indices)):
                np.random.seed(SEED + c)
                try:
                    out[f"{name}/{key}"] = np.asarray(fn(rec), dtype=np.int64)
                except Exception as e:  # noqa: BLE001  (the reference's own failure modes are part of the contract)
                    out[f"{name}/{key}"] = np.array([-1], dtype=np.int64)
                    out[f"{name}_error/{key}"] = np.array(type(e).__name__)
    os.makedirs(os.path.dirname(GOLDEN_PATH), exist_ok=True)
    np.savez_compressed(GOLDEN_PATH, seed=np.array(SEED), **out)
    print("wrote", GOLDEN_PATH, len(out), "arrays,", os.path.getsize(GOLDEN_PATH), "bytes")


if __name__ == "__main__":
    main()
