"""Generate ``tests/golden/reference_checks.npz``: what the UNMODIFIED reference computes in the checks of
``tests/test_oracle_vs_reference.py`` and in the TSNDataSet check of ``tests/test_dataset.py``, so that those
tests compare the oracle and the product against stored vectors on any machine.

Run where the reference tree is importable (oracle/ref_shims.py):  python -m oracle.gen_reference_checks

Each check stores named tensors (``record``): a tensor of at most SAMPLE entries in full, a larger one as a fixed
seeded sample of SAMPLE entries (``pick``) plus the float64 norm of the whole tensor.  Checks of exact equality
store the sha256 of the tensor's bytes.  Inputs are not stored: they regenerate from the seeds.
"""
from __future__ import annotations

import hashlib
import json
import os
import sys
import tempfile
from collections import OrderedDict

import numpy as np
import torch

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, os.path.dirname(HERE))

from oracle import gen_golden, ref_shims  # noqa: E402
from oracle import gen_golden_dataset as gg  # noqa: E402

GOLDEN_PATH = os.path.join(os.path.dirname(HERE), "tests", "golden", "reference_checks.npz")
SAMPLE = 128

# gen_golden.CASES compared output for output and gradient for gradient
OUTPUT_CASES = ["cfg1_train_masked", "t9_attnframe", "noattn_f256", "general_attn", "avgpool_transattn",
                "avgpool_noattn_f256"]
MCD_RUNS = [(False, 0.0), (True, 0.7)]
TSN_MODES = ["test", "val", "random"]


def pick(t: torch.Tensor) -> np.ndarray:
    """All entries of a small tensor; of a larger one the same SAMPLE entries every time (seeded by its size)."""
    flat = t.detach().reshape(-1).cpu()
    if flat.numel() > SAMPLE:
        idx = np.sort(np.random.default_rng(flat.numel()).choice(flat.numel(), SAMPLE, replace=False))
        flat = flat[torch.from_numpy(idx)]
    return flat.numpy().copy()


def sha(t: torch.Tensor) -> str:
    return hashlib.sha256(t.detach().contiguous().cpu().numpy().tobytes()).hexdigest()


def record(tensors) -> tuple:
    """(values, index): the picks of every tensor in one float32 array, and per name its shape, slice and norm."""
    vals, index, off = [], OrderedDict(), 0
    for name, t in tensors.items():
        v = pick(t).astype(np.float32)
        index[name] = {"shape": list(t.shape), "offset": off, "n": int(v.size),
                       "norm": float(t.detach().double().norm())}
        vals.append(v)
        off += v.size
    return np.concatenate(vals), index


def flat_outputs(outs):
    """The outputs of the 10-tuple that the checks compare, in a fixed order."""
    return [outs[0], outs[1], *outs[3], *outs[4], outs[5], outs[6], *outs[8], *outs[9]]


def case_outputs(case):
    model, outs, loss, _ = gen_golden.run_reference(gen_golden.CASES[case])
    t = OrderedDict([("loss", loss)])
    t.update((f"out/{i}", o) for i, o in enumerate(flat_outputs(outs)))
    t.update((f"grad/{n}", p.grad) for n, p in model.named_parameters() if p.grad is not None)
    return t, {"no_grad": [n for n, p in model.named_parameters() if p.grad is None]}


def state_dict_init():
    ref_models, _, _ = ref_shims.load()
    torch.manual_seed(7)
    m = ref_models.VideoModel(12, "video", "trn-m", "RGB", train_segments=5, val_segments=5, add_fc=1,
                              fc_dim=512, partial_bn=False, use_bn="none", ens_DA="none",
                              use_attn="TransAttn", share_params="Y", verbose=False)
    sd = m.state_dict()
    return OrderedDict(), {"keys": list(sd), "shapes": [list(v.shape) for v in sd.values()],
                           "sha256": [sha(v) for v in sd.values()]}


def train_loop():
    """main.py:418-583 (forward, loss, backward, clip_grad_norm_, SGD-Nesterov, DANN learning rate), three
    iterations of case cfg1_small_c5."""
    from torch.nn.utils import clip_grad_norm_
    c = gen_golden.CASES["cfg1_small_c5"]
    model, _, _, _ = gen_golden.run_reference(c)
    model.zero_grad(set_to_none=True)
    _, xs, xt, labels, _ = gen_golden.case_inputs(c)
    lr0 = 3e-2
    opt = torch.optim.SGD(model.parameters(), lr0, momentum=0.9, weight_decay=1e-4, nesterov=True)   # main.py:83
    t = OrderedDict()
    for it in range(3):
        p = it / 3.0
        for gparam in opt.param_groups:
            gparam["lr"] = lr0 / (1. + 10 * p) ** 0.75                                              # main.py:800-802
        outs = model(xs, xt, list(gen_golden.BETA), 0, is_train=True, reverse=False)
        loss = gen_golden.reference_loss(outs, labels)
        opt.zero_grad()
        loss.backward()
        t[f"loss/{it}"] = loss.detach()
        t[f"total_norm/{it}"] = clip_grad_norm_(model.parameters(), 0.05)    # small max_norm: clipping is active
        opt.step()
    t.update((f"param/{n}", p.detach()) for n, p in model.named_parameters())
    return t, {}


def weighted_losses():
    """main.py:160-167, 204-205: criterion / criterion_domain with class and domain weights on case ragged_6_3."""
    c = gen_golden.CASES["ragged_6_3"]
    _, outs, _, _ = gen_golden.run_reference(c)
    labels = gen_golden.case_inputs(c)[3]
    cw = 1.0 / torch.tensor([0.05, 0.2, 0.1, 0.05, 0.1, 0.05, 0.05, 0.1, 0.1, 0.05, 0.1, 0.05])
    dw = torch.tensor([1.0 / 300, 1.0 / 170])
    criterion = torch.nn.CrossEntropyLoss(weight=cw)                 # main.py:204
    criterion_domain = torch.nn.CrossEntropyLoss(weight=dw)          # main.py:205
    (_, out_s, _, pd_s, _, _, out_t, _, pd_t, _) = outs
    ref = criterion(out_s, labels)                                   # main.py:446
    alls = []
    for lvl in range(3):                                             # main.py:513-536
        ps, pt = pd_s[lvl].view(-1, 2), pd_t[lvl].view(-1, 2)
        dom = torch.cat((torch.zeros(ps.size(0)).long(), torch.ones(pt.size(0)).long()), 0)
        alls.append(torch.cat((ps, pt), 0))
        ref = ref + criterion_domain(alls[-1], dom)
    _, _, ref_loss = ref_shims.load()
    ref = ref + gen_golden.GAMMA * ref_loss.attentive_entropy(torch.cat((out_s, out_t), 0), alls[1])
    t = OrderedDict([("loss", ref)])
    for dom, out, pd in (("s", out_s, pd_s), ("t", out_t, pd_t)):
        t[f"out_{dom}"] = out
        t.update((f"pred_domain_{dom}/{lvl}", pd[lvl]) for lvl in range(3))
    return t, {}


def _perturbed_variant(num_class, seed, **kw):
    """A reference VideoModel moved away from its degenerate 0.001 init by seeded noise on every weight, and a
    small batch drawn from the same generator afterwards (the recipe the oracle side repeats)."""
    ref_models, _, _ = ref_shims.load()
    torch.manual_seed(seed)
    m = ref_models.VideoModel(num_class, "video", "trn-m", "RGB", train_segments=5, val_segments=5, add_fc=1,
                              fc_dim=512, dropout_i=0.0, dropout_v=0.0, partial_bn=False, use_bn="none",
                              share_params="Y", verbose=False, **kw)
    m.train()                                  # (the reference's train() override returns None)
    sd = m.state_dict()
    meta = {"keys": list(sd), "sha256": [sha(v) for v in sd.values()],
            "param_names": [n for n, _ in m.named_parameters()]}
    g = torch.Generator().manual_seed(seed + 1)
    with torch.no_grad():
        for k, v in m.named_parameters():
            if "weight" in k:
                v.add_(0.02 * torch.randn(v.shape, generator=g))
    xs, xt = torch.randn(6, 5, 2048, generator=g), torch.randn(4, 5, 2048, generator=g)
    labels = torch.randint(0, num_class, (6,), generator=g)
    return m, xs, xt, labels, meta


def mcd(reverse, mu):
    """ens_DA='MCD' (models.py:276-279, 716-720; main.py:447, 548-556): outputs and every gradient of
    CE(out_s) + CE(out_s_2) - dis_MCD(out_t, out_t_2) (loss.py:29-30)."""
    _, _, ref_loss = ref_shims.load()
    m, xs, xt, labels, meta = _perturbed_variant(7, 11, ens_DA="MCD", use_attn="TransAttn")
    outs = m(xs, xt, [0.75, 0.75, 0.5], mu, is_train=True, reverse=reverse)
    ce = torch.nn.CrossEntropyLoss()
    loss = ce(outs[1], labels) + ce(outs[2], labels) - ref_loss.dis_MCD(outs[6], outs[7])
    loss.backward()
    t = OrderedDict([("loss", loss)])
    t.update((f"out/{i}", outs[i]) for i in (1, 2, 6, 7))
    t.update((f"grad/{n}", p.grad) for n, p in m.named_parameters() if p.grad is not None)
    return t, meta


def general_attention_loss(outs, labels):
    """compose_loss plus terms that read the attention weights themselves (shared by both sides of the check)."""
    from oracle import ta3n_oracle as orc
    return orc.compose_loss(outs, labels, 0.003, use_attn="general") + 0.5 * (outs[0] ** 2).sum() + \
        0.25 * (outs[5] ** 2).sum()


def general_attention():
    """use_attn='general' (models.py:320-325 attn_layer, :359-366 softmax over the relations, :379-388
    re-weighting) with trained-like weights: outputs and every gradient."""
    m, xs, xt, labels, meta = _perturbed_variant(9, 21, ens_DA="none", use_attn="general")
    outs = m(xs, xt, [0.75, 0.6, 0.5], 0, is_train=True, reverse=False)
    loss = general_attention_loss(outs, labels)
    loss.backward()
    t = OrderedDict([("loss", loss)])
    t.update((f"out/{i}", outs[i]) for i in (0, 1, 5, 6))
    t.update((f"grad/{n}", p.grad) for n, p in m.named_parameters() if p.grad is not None)
    return t, meta


def tsn_items(mode):
    """The reference TSNDataSet over gg.make_tree: per item the (video, frame) of every row it returns (frames are
    told apart by their random contents) and its label."""
    ds_mod = ref_shims.load_dataset()
    with tempfile.TemporaryDirectory() as tmp:
        lst = gg.make_tree(tmp)
        frames = {}
        for line in open(lst):
            d, nf, _ = line.split()
            v = int(os.path.basename(d)[1:])
            for f in range(1, int(nf) + 1):
                x = torch.load(os.path.join(d, "img_{:05d}.t7".format(f)))
                frames[x.numpy().tobytes()] = (v, f)
        ds = ds_mod.TSNDataSet("", lst, num_dataload=10, num_segments=5, new_length=1, modality="RGB",
                               random_shift=(mode == "random"), test_mode=(mode == "test"))
        where, labels = [], []
        for i in range(len(ds)):
            np.random.seed(100 + i)
            x, y = ds[i]
            where.append([frames[row.numpy().tobytes()] for row in x.reshape(-1, x.shape[-1])])
            labels.append(int(y))
    return OrderedDict(), {"len": len(ds), "item_shape": list(x.shape), "frames": where, "labels": labels}


def checks():
    out = OrderedDict()
    for case in OUTPUT_CASES:
        out[f"case/{case}"] = case_outputs(case)
    out["state_dict_init"] = state_dict_init()
    out["train_loop"] = train_loop()
    out["weighted_losses"] = weighted_losses()
    for reverse, mu in MCD_RUNS:
        out[f"mcd/{reverse}_{mu}"] = mcd(reverse, mu)
    out["general_attention"] = general_attention()
    for mode in TSN_MODES:
        out[f"tsn/{mode}"] = tsn_items(mode)
    return out


def main():
    blob, meta = {}, {"sample": SAMPLE, "torch": torch.__version__, "checks": {}}
    for name, (tensors, extra) in checks().items():
        entry = dict(extra)
        if tensors:
            blob[name], entry["tensors"] = record(tensors)
        meta["checks"][name] = entry
    blob["meta_json"] = np.frombuffer(json.dumps(meta).encode(), dtype=np.uint8)
    np.savez_compressed(GOLDEN_PATH, **blob)
    print("wrote", GOLDEN_PATH, os.path.getsize(GOLDEN_PATH), "bytes")


if __name__ == "__main__":
    main()
