"""Input pipeline (SURVEY 8f n3): segment-index rules, the TSNDataSet drop-in, packed shards and the paired loader.
CPU only.  Golden index tables and items come from the unmodified reference (oracle/gen_golden_dataset.py,
oracle/gen_reference_checks.py)."""
import os

import numpy as np
import pytest
import torch

from oracle import dataset_oracle as dorc
from oracle import gen_golden_dataset as gg
from oracle import gen_reference_checks as grc
from ta3n_b200 import dataset as D
from tests.golden_util import ReferenceCheck

GOLDEN = np.load(gg.GOLDEN_PATH)
RULES = {"val": (D.val_segment_indices, dorc.val_indices), "test": (D.test_segment_indices, dorc.test_indices),
         "sample": (D.random_segment_indices, dorc.sample_indices)}


@pytest.mark.parametrize("rule", ["val", "test", "sample"])
def test_index_rules_match_reference_golden(rule):
    """Product rules and oracle restatement against the reference's own outputs over the whole grid, including the
    cases where the reference raises (clips shorter than new_length)."""
    product, oracle = RULES[rule]
    for c, (nf, ns, nl) in enumerate(gg.grid()):
        key = f"{nf}_{ns}_{nl}"
        want = GOLDEN[f"{rule}/{key}"]
        for fn in (product, oracle):
            np.random.seed(int(GOLDEN["seed"]) + c)
            if f"{rule}_error/{key}" in GOLDEN.files:
                with pytest.raises((IndexError, ValueError)):
                    fn(nf, ns, nl)
            else:
                got = np.asarray(fn(nf, ns, nl))
                assert got.shape == want.shape and np.array_equal(got.astype(np.int64), want), (rule, key, fn.__module__)


@pytest.mark.parametrize("mode", grc.TSN_MODES)
def test_tsn_dataset_equals_live_reference(tmp_path, mode):
    """Item for item, the frames and label the reference's TSNDataSet returned for the same tree and seeds
    (stored by oracle/gen_reference_checks.py)."""
    ref = ReferenceCheck(f"tsn/{mode}").meta
    lst = gg.make_tree(str(tmp_path))
    kw = dict(num_dataload=10, num_segments=5, new_length=1, modality="RGB",
              random_shift=(mode == "random"), test_mode=(mode == "test"))
    mine = D.TSNDataSet("", lst, **kw)
    assert ref["len"] == len(mine) == 10                       # list tiled to num_dataload (dataset.py:70-75)
    for i in range(len(mine)):
        np.random.seed(100 + i)
        xm, ym = mine[i]
        xr = torch.stack([torch.load(os.path.join(str(tmp_path), f"v{v}", "img_{:05d}.t7".format(f)))
                          for v, f in ref["frames"][i]]).reshape(ref["item_shape"])
        assert ref["labels"][i] == ym and torch.equal(xr, xm), (mode, i)


def test_packed_shard_serves_the_same_items(tmp_path):
    lst = gg.make_tree(str(tmp_path))
    shard = os.path.join(str(tmp_path), "source_T5.npy")
    shape = D.pack_list(lst, shard, num_segments=5)
    assert shape == (7, 5, 16)
    files = D.TSNDataSet("", lst, num_dataload=11, num_segments=5, random_shift=False, test_mode=True)
    packed = D.PackedTSNDataSet(shard, num_dataload=11)
    assert len(packed) == len(files) == 11
    assert [int(r) for r in packed.order] == dorc.repeat_list(7, 11)
    for i in range(11):
        xf, yf = files[i]
        xp, yp = packed[i]
        assert yf == yp and torch.equal(xf, xp)
    with pytest.raises(ValueError):
        D.pack_list(lst, shard, num_segments=5, rule="random")


def test_gather_fills_the_staging_buffer_in_batch_order(tmp_path):
    lst = gg.make_tree(str(tmp_path))
    shard = os.path.join(str(tmp_path), "g.npy")
    D.pack_list(lst, shard, num_segments=5)
    packed = D.PackedTSNDataSet(shard, num_dataload=11)
    out, lab = torch.full((6, 5, 16), -1.0), torch.full((6,), -1, dtype=torch.int64)
    idx = np.array([10, 0, 7, 3])                       # unsorted, with a repeated underlying row (10 -> row 3)
    packed.gather(idx, out, lab)
    for k, i in enumerate(idx):
        x, y = packed[int(i)]
        assert torch.equal(out[k], x) and int(lab[k]) == y
    assert torch.all(out[4:] == -1) and torch.all(lab[4:] == -1)        # a short batch leaves the tail alone
    with pytest.raises(IndexError):
        packed.gather(np.array([11]), out, lab)
    packed.gather(np.array([], dtype=np.int64), out, lab)               # empty batch: no-op
    assert torch.all(out[4:] == -1)


def test_paired_loader_covers_each_epoch_like_zip_of_random_samplers(tmp_path):
    src_root, tgt_root = os.path.join(str(tmp_path), "s"), os.path.join(str(tmp_path), "t")
    os.makedirs(src_root), os.makedirs(tgt_root)
    ls, lt = gg.make_tree(src_root, n_videos=9, seed=1), gg.make_tree(tgt_root, n_videos=5, seed=2)
    D.pack_list(ls, os.path.join(src_root, "p.npy"), 3)
    D.pack_list(lt, os.path.join(tgt_root, "p.npy"), 3)
    # main.py:145-153 tiles the shorter list so that both loaders have the same number of iterations
    source = D.PackedTSNDataSet(os.path.join(src_root, "p.npy"), num_dataload=9)
    target = D.PackedTSNDataSet(os.path.join(tgt_root, "p.npy"), num_dataload=7)
    loader = D.PairedFeatureLoader(source, target, batch_sizes=(4, 3), seed=5, pin_memory=False)
    assert len(loader) == 3
    for epoch in range(2):
        seen_s, seen_t, sizes = [], [], []
        for (xs, ys), (xt, yt) in loader:
            assert xs.shape[1:] == (3, 16) and xt.shape[1:] == (3, 16) and xs.dtype == torch.float32
            sizes.append((xs.shape[0], xt.shape[0]))
            for x, y in zip(xs, ys):          # every item is one of the dataset's rows with its own label
                hits = [i for i in range(len(source)) if torch.equal(source[i][0], x) and source[i][1] == int(y)]
                assert hits
                seen_s.append(hits[0])
            seen_t.extend(int(v) for v in yt)
            assert all(any(torch.equal(target[i][0], x) for i in range(len(target))) for x in xt)
        assert sizes == [(4, 3), (4, 3), (1, 1)]                 # last short batch, as DataLoader(drop_last=False)
        assert sorted(seen_s) == list(range(9))                    # a permutation of the source set
        assert len(seen_t) == 7


def test_loader_staging_buffers_are_not_overwritten_early(tmp_path):
    """A yielded batch must stay intact while the next one is consumed (async H2D copies read it)."""
    lst = gg.make_tree(str(tmp_path), n_videos=12, seed=7)
    shard = os.path.join(str(tmp_path), "p.npy")
    D.pack_list(lst, shard, 3)
    ds = D.PackedTSNDataSet(shard)
    loader = D.PairedFeatureLoader(ds, ds, batch_sizes=(2, 2), seed=1, pin_memory=False)
    prev = None
    for (xs, _), _ in loader:
        if prev is not None:
            view, snapshot = prev
            assert torch.equal(view, snapshot)
        prev = (xs, xs.clone())
    with pytest.raises(ValueError):
        D.PairedFeatureLoader(ds, ds, batch_sizes=(2, 2), depth=2)
