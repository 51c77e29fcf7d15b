"""Shared helpers: load the golden fixtures, compare tensors normwise."""
from __future__ import annotations

import json
import os

import numpy as np
import torch

from oracle.gen_reference_checks import pick

GOLDEN_PATH = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "ta3n_golden.npz")

# Tolerance of the path (north_star): 1e-3 *normwise* relative per tensor, fp32 (SURVEY §8c).
TOL_PATH = 1e-3
# fp32-vs-fp32 restatements of the same math should agree far tighter than that.
TOL_FP32 = 2e-5


def load_golden():
    z = np.load(GOLDEN_PATH)
    meta = json.loads(bytes(z["meta_json"]).decode())
    return z, meta


def rel_err(a, b) -> float:
    """||a-b||_2 / ||b||_2 with b the reference (zero reference -> absolute norm)."""
    a = torch.as_tensor(np.asarray(a) if not torch.is_tensor(a) else a).detach().double().cpu().reshape(-1)
    b = torch.as_tensor(np.asarray(b) if not torch.is_tensor(b) else b).detach().double().cpu().reshape(-1)
    assert a.shape == b.shape, (a.shape, b.shape)
    den = b.norm().item()
    num = (a - b).norm().item()
    return num / den if den > 0 else num


def abs_err(a, b) -> float:
    a = torch.as_tensor(np.asarray(a) if not torch.is_tensor(a) else a).detach().double().cpu().reshape(-1)
    b = torch.as_tensor(np.asarray(b) if not torch.is_tensor(b) else b).detach().double().cpu().reshape(-1)
    assert a.shape == b.shape, (a.shape, b.shape)
    return (a - b).norm().item()


def assert_close(a, b, tol, what="", noise=0.0):
    """||a-b|| <= tol*||b|| + 8*noise, where ``noise`` is the reference's own fp32 rounding error
    ||ref_fp32 - ref_fp64|| for this tensor (matters only for sums that cancel, e.g. the bias
    gradients of the domain heads, whose source and target halves have opposite signs)."""
    b_t = torch.as_tensor(np.asarray(b) if not torch.is_tensor(b) else b).detach().double().cpu()
    d = abs_err(a, b)
    den = b_t.norm().item()
    bound = tol * den + 8.0 * float(noise)
    assert d <= bound or (den == 0 and d == 0), \
        f"{what}: ||diff||={d:.3e} > {tol:.1e}*||ref||({den:.3e}) + 8*noise({float(noise):.3e})"
    return d / den if den > 0 else d


REFERENCE_CHECKS_PATH = os.path.join(os.path.dirname(GOLDEN_PATH), "reference_checks.npz")


class ReferenceCheck:
    """One check of ``reference_checks.npz`` (oracle/gen_reference_checks.py): what the reference computed, by
    name -- each tensor in full, or a fixed sample of its entries and the norm of the whole tensor."""

    def __init__(self, name: str):
        z = np.load(REFERENCE_CHECKS_PATH)
        self.meta = json.loads(bytes(z["meta_json"]).decode())["checks"][name]
        self.index = self.meta.get("tensors", {})
        self.values = z[name] if self.index else None

    def names(self, prefix: str):
        return [k[len(prefix):] for k in self.index if k.startswith(prefix)]

    def norm(self, key: str) -> float:
        return self.index[key]["norm"]

    def _picked(self, key):
        e = self.index[key]
        return self.values[e["offset"]:e["offset"] + e["n"]]

    def __getitem__(self, key) -> torch.Tensor:
        """The whole tensor (only for tensors stored in full)."""
        e = self.index[key]
        assert e["n"] == int(np.prod(e["shape"])), f"{key} is stored as a sample"
        return torch.from_numpy(self._picked(key).copy()).reshape(e["shape"])

    def assert_close(self, key, got, tol, what=""):
        """assert_close of the stored entries; for a sampled tensor also ||got|| against the stored norm."""
        e = self.index[key]
        assert list(got.shape) == e["shape"], (what, tuple(got.shape), e["shape"])
        err = assert_close(pick(got), self._picked(key), tol, what)
        if e["n"] < got.numel():
            got_norm = got.detach().double().norm().item()
            assert abs(got_norm - e["norm"]) <= tol * e["norm"], f"{what}: norm {got_norm:.6e} vs {e['norm']:.6e}"
        return err


def sample(t: torch.Tensor, stride: int):
    return t.detach().reshape(-1).double().cpu()[::stride]


def check_outputs_against_golden(z, case: str, outs, tol: float, stride: int):
    """outs = reference-shaped 10-tuple."""
    (attn_s, out_s, _, pd_s, feat_s, attn_t, out_t, _, pd_t, feat_t) = outs
    k = case + "/"
    worst = 0.0
    for dom, attn, out, pd, feat in (("s", attn_s, out_s, pd_s, feat_s), ("t", attn_t, out_t, pd_t, feat_t)):
        pairs = [(f"attn_{dom}", attn), (f"out_{dom}", out), (f"pred_rel_{dom}", pd[0]),
                 (f"pred_video_{dom}", pd[1]), (f"pred_frame_{dom}", pd[2]), (f"feat_video_{dom}", feat[1])]
        for name, t in pairs:
            assert tuple(t.shape) == z[k + name].shape, (name, tuple(t.shape), z[k + name].shape)
            worst = max(worst, assert_close(t, z[k + name], tol, f"{case}:{name}"))
        assert tuple(feat[0].shape) == tuple(out.shape)
        worst = max(worst, assert_close(feat[0], z[k + f"out_{dom}"], tol, f"{case}:feat0_{dom}"))
        worst = max(worst, assert_close(sample(feat[2], stride), z[k + f"feat_fc_{dom}_sample"], tol,
                                        f"{case}:feat_fc_{dom}"))
        cs = z[k + f"feat_fc_{dom}_checksum"]
        got = feat[2].detach().double().cpu()
        assert abs(got.norm().item() - cs[1]) <= tol * cs[1], f"{case}:feat_fc_{dom} norm"
    return worst


# Gradients that are zero by construction: the bias of the last attn_layer Linear shifts every logit of the softmax
# over the relations by the same amount (models.py:364), so the reference's value is pure rounding noise (~1e-8).
STRUCTURAL_ZERO_GRADS = ("attn_layer.2.bias",)


def check_grads_against_golden(z, case: str, grads: dict, used: list, tol: float, stride: int, noise_scale: float = 1.0):
    worst = 0.0
    for name in used:
        g = grads[name]
        assert g is not None, f"{case}: no grad for {name}"
        if name in STRUCTURAL_ZERO_GRADS:
            assert g.detach().double().norm().item() <= 1e-6, f"{case}: {name} must vanish"
            continue
        ref_norm = float(z[f"{case}/grad_norm/{name}"])
        # rounding-noise floor of this gradient: the reference's own |fp32 - fp64|, but never below a few
        # fp32 ulps of the O(1e-2) summands of the domain-head bias sums (their opposite-sign halves cancel
        # to ~1e-7, and ONE sample of |fp32 - fp64| can come out luckily small)
        noise = max(float(z[f"{case}/grad_noise/{name}"]), 4e-9) * noise_scale
        got_norm = g.detach().double().norm().item()
        assert abs(got_norm - ref_norm) <= tol * ref_norm + 8 * noise, \
            f"{case}: grad norm {name}: {got_norm:.6e} vs {ref_norm:.6e} (noise {noise:.2e})"
        worst = max(worst, assert_close(sample(g, stride), z[f"{case}/grad_sample/{name}"], tol * 4,
                                        f"{case}:grad_sample:{name}",
                                        noise=max(float(z[f"{case}/grad_sample_noise/{name}"]), 4e-9) * noise_scale))
    return worst
