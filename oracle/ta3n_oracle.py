"""CPU oracle for the TA3N hot path  --  TEST INFRASTRUCTURE, NOT PRODUCT CODE.

Only ``tests/``, ``__graft_entry__.smoke()`` and ``bench.py``'s CPU-baseline /
``--impl reference`` legs may import this module.  The product package
(``ta3n_b200``) never imports it and has no CPU fallback.

What it is: a functional, eager-PyTorch (CPU, fp32 or fp64) restatement of the
one code path of cmhungsteve/TA3N that this repo accelerates:

    VideoModel.forward with frame_aggregation='trn-m' (the hot path; 'avgpool', the paper's baseline aggregation,
    as an off-path variant), baseline_type='video',
    add_fc=1, use_bn='none', ens_DA='none', share_params='Y',
    use_attn in {'TransAttn','general','none'}, use_attn_frame in {'none','TransAttn'}

plus the loss composition that main.py applies right after it.  Each function
cites the reference file:line it follows (paths relative to /root/reference).

Parity pinning: the reference ships no tests or golden vectors (SURVEY.md §4),
so this oracle is pinned against what the reference itself computes, imported
unmodified through ``oracle/ref_shims.py``:
  * ``oracle/gen_reference_checks.py`` ran the reference classes to produce
    ``tests/golden/reference_checks.npz``; ``tests/test_oracle_vs_reference.py``
    compares every output and every parameter gradient of this file with it;
  * ``oracle/gen_golden.py`` ran the reference to produce ``tests/golden/*.npz``;
    ``tests/test_oracle_golden.py`` checks this oracle against those fixtures
    everywhere.

The arithmetic itself lives in PyTorch (a third-party dependency of the
reference, requirements.txt:98 pins torch==2.2.0; this image has 2.11.0); the
oracle therefore uses the same ATen CPU ops in the same order as the reference
so that its timing is a fair stand-in for "the reference's CPU path" where the
Python reference itself cannot travel (the GPU box has no /root/reference).
"""
from __future__ import annotations

import itertools
import math
from collections import OrderedDict
from dataclasses import dataclass
from typing import Dict, List, Optional, Sequence, Tuple

import torch
import torch.nn.functional as F

FEATURE_DIM = 2048     # ResNet-101 pool5 width; models.py:125-126 reads fc.in_features
NUM_BOTTLENECK = 256   # models.py:223
INIT_STD = 1e-3        # models.py:128


@dataclass(frozen=True)
class PathConfig:
    """The knobs of the hot path (constructor args of models.py:59-67 that matter here)."""
    num_class: int = 12
    num_segments: int = 5          # train_segments == val_segments for trn-m (SURVEY App. D Q3)
    fc_dim: int = 512
    dropout_i: float = 0.5
    dropout_v: float = 0.5
    use_attn: str = "TransAttn"    # or 'general' / 'none'
    use_attn_frame: str = "none"   # or 'TransAttn'
    ens_DA: str = "none"           # or 'MCD': a second video-level classifier (models.py:276-279, 716-720)
    frame_aggregation: str = "trn-m"   # or 'avgpool' (models.py:240-241, 425-433, 620-626): no relation level

    @property
    def video_dim(self) -> int:    # feat_aggregated_dim = feat_video_dim, models.py:240-250
        return self.shared_dim if self.frame_aggregation == "avgpool" else NUM_BOTTLENECK

    @property
    def shared_dim(self) -> int:   # models.py:129
        return min(self.fc_dim, FEATURE_DIM)


# ----------------------------------------------------------------------------
# static relation tables                                     TRNmodule.py:30-41
# ----------------------------------------------------------------------------
def relation_tuples(num_frames: int, subsample: int = 3) -> List[List[Tuple[int, ...]]]:
    """Frame tuples actually evaluated per scale, largest scale first.

    TRNmodule.py:34   scales = [T, T-1, ..., 2]
    TRNmodule.py:36-41 all lexicographic combinations per scale, min(3, N) kept
    TRNmodule.py:60   the first (largest) scale uses combination 0 only
    TRNmodule.py:71   evenly spaced pick: idx_k = ceil(k * N / n_sel)
    """
    chosen: List[List[Tuple[int, ...]]] = []
    for pos, scale in enumerate(range(num_frames, 1, -1)):
        combos = list(itertools.combinations(range(num_frames), scale))
        if pos == 0:
            chosen.append([combos[0]])
            continue
        n_sel = min(subsample, len(combos))
        picks = [int(math.ceil(k * len(combos) / n_sel)) for k in range(n_sel)]
        chosen.append([combos[i] for i in picks])
    return chosen


# ----------------------------------------------------------------------------
# parameters                                   models.py:119-325 (_prepare_DA)
# ----------------------------------------------------------------------------
def _std_linear(n_in: int, n_out: int) -> Tuple[torch.Tensor, torch.Tensor]:
    """nn.Linear followed by normal_(w, 0, 0.001), constant_(b, 0)   (models.py:141-143 etc.)."""
    lin = torch.nn.Linear(n_in, n_out)          # consumes RNG exactly like the reference
    torch.nn.init.normal_(lin.weight, 0, INIT_STD)
    torch.nn.init.constant_(lin.bias, 0)
    return lin.weight.detach(), lin.bias.detach()


def _default_linear(n_in: int, n_out: int) -> Tuple[torch.Tensor, torch.Tensor]:
    """nn.Linear with PyTorch's default init (TRNmodule.py:48-52, models.py:289-293)."""
    lin = torch.nn.Linear(n_in, n_out)
    return lin.weight.detach(), lin.bias.detach()


def init_params(cfg: PathConfig, seed: Optional[int] = None) -> "OrderedDict[str, torch.Tensor]":
    """Create the state_dict of the reference VideoModel for this path, in the
    reference's construction order so the same seed yields the same values.

    Order (models.py): :141 shared, :156 fc_feature_source, :161 fc_feature_domain,
    :166 fc_classifier_source, :170 fc_classifier_domain, :224 TRN (TRNmodule.py:45-54),
    :225-226 bn_trn_{S,T}, :258/:262 fc_feature_video_source{,_2}, :267 fc_feature_domain_video,
    :272 fc_classifier_video_source, :281 fc_classifier_domain_video, :286-294 relation discs.
    """
    if seed is not None:
        torch.manual_seed(seed)
    Fd, H, C, T = cfg.shared_dim, cfg.video_dim, cfg.num_class, cfg.num_segments
    trn = cfg.frame_aggregation == "trn-m"
    p: "OrderedDict[str, torch.Tensor]" = OrderedDict()

    def put(name, wb):
        p[name + ".weight"], p[name + ".bias"] = wb

    put("fc_feature_shared_source", _std_linear(FEATURE_DIM, Fd))
    put("fc_feature_source", _std_linear(Fd, Fd))               # registered, unused (App. C)
    put("fc_feature_domain", _std_linear(Fd, Fd))
    put("fc_classifier_source", _std_linear(Fd, C))             # executed, output dropped
    put("fc_classifier_domain", _std_linear(Fd, 2))
    for i, scale in enumerate(range(T, 1, -1) if trn else ()):
        put(f"TRN.fc_fusion_scales.{i}.1", _default_linear(scale * Fd, H))
    for dom in ("S", "T") if trn else ():                       # BatchNorm1d(256), unused here
        p[f"bn_trn_{dom}.weight"] = torch.ones(H)
        p[f"bn_trn_{dom}.bias"] = torch.zeros(H)
        p[f"bn_trn_{dom}.running_mean"] = torch.zeros(H)
        p[f"bn_trn_{dom}.running_var"] = torch.ones(H)
        p[f"bn_trn_{dom}.num_batches_tracked"] = torch.tensor(0, dtype=torch.long)
    put("fc_feature_video_source", _std_linear(H, H))           # unused
    put("fc_feature_video_source_2", _std_linear(H, H))         # unused
    put("fc_feature_domain_video", _std_linear(H, H))
    put("fc_classifier_video_source", _std_linear(H, C))
    if cfg.ens_DA == "MCD":                                     # models.py:276-279
        put("fc_classifier_video_source_2", _std_linear(H, C))
    put("fc_classifier_domain_video", _std_linear(H, 2))
    for i in range(T - 1) if trn else ():                       # models.py:285-294: trn-m only
        put(f"relation_domain_classifier_all.{i}.0", _default_linear(H, H))
        put(f"relation_domain_classifier_all.{i}.2", _default_linear(H, 2))
    if cfg.use_attn == "general":                               # models.py:320-325: attn_layer, PyTorch default init
        assert trn, "general attention is defined over the relation features"
        put("attn_layer.0", _default_linear(H, H))
        put("attn_layer.2", _default_linear(H, 1))
    return p


USED_PARAM_PREFIXES = (
    "fc_feature_shared_source", "fc_feature_domain.", "fc_classifier_domain.",
    "TRN.", "fc_feature_domain_video", "fc_classifier_video_source",      # (also ..._source_2 under MCD)
    "fc_classifier_domain_video", "relation_domain_classifier_all", "attn_layer",
)


def used_param_names(params: Dict[str, torch.Tensor]) -> List[str]:
    """Names of the parameters that receive gradients on this path (SURVEY App. C)."""
    return [k for k in params
            if k.startswith(USED_PARAM_PREFIXES) and params[k].dtype.is_floating_point]


# ----------------------------------------------------------------------------
# building blocks
# ----------------------------------------------------------------------------
class _FlipGrad(torch.autograd.Function):
    """Gradient reversal: identity forward, -beta * g backward (models.py:20-29)."""

    @staticmethod
    def forward(ctx, x, beta):
        ctx.beta = float(beta)
        return x.view_as(x)

    @staticmethod
    def backward(ctx, g):
        return g.neg() * ctx.beta, None


def grad_reverse(x: torch.Tensor, beta: float) -> torch.Tensor:
    return _FlipGrad.apply(x, beta)


def general_attention(p: Dict[str, torch.Tensor], feat: torch.Tensor) -> torch.Tensor:
    """get_general_attn (models.py:359-366): feat (B, n, H) -> softmax over the n segments of attn_layer(feat), (B, n)."""
    n = feat.size(1)
    hid = torch.tanh(F.linear(feat.reshape(-1, feat.size(-1)), p["attn_layer.0.weight"], p["attn_layer.0.bias"]))
    s = F.linear(hid, p["attn_layer.2.weight"], p["attn_layer.2.bias"]).view(-1, n, 1)
    return F.softmax(s, dim=1).view(-1, n)


def entropy_attention(logits: torch.Tensor) -> torch.Tensor:
    """w = 1 - H(softmax(logits)) along dim 1 (models.py:351-357)."""
    q = F.softmax(logits, dim=1)
    lq = F.log_softmax(logits, dim=1)
    return 1 - torch.sum(-q * lq, 1)


def _apply_dropout(x: torch.Tensor, p: float, train: bool, mask: Optional[torch.Tensor]) -> torch.Tensor:
    """nn.Dropout semantics (models.py:133-134).  ``mask`` (0/1 keep mask, same shape)
    overrides the RNG so that CUDA and oracle see the same drops."""
    if not train or p <= 0.0:
        return x
    if mask is None:
        return F.dropout(x, p, True)
    return x * mask.to(x.dtype) * (1.0 / (1.0 - p))


def _relu(x: torch.Tensor, gate: Optional[torch.Tensor]) -> torch.Tensor:
    """ReLU, or -- when ``gate`` (0/1, same shape) is given -- the linear map x * gate.

    Gates let a test evaluate the oracle *on a prescribed activation pattern*: a reduced-precision
    forward (tf32) flips the sign of the ~1e-4 fraction of pre-activations that sit within rounding
    error of zero; each flip changes a gradient entry by O(1), so gradients of the two networks differ
    by ~sqrt(fraction) ~ 1e-2 even though every product is accurate to ~1e-4.  With the pattern pinned,
    gradients must agree to rounding accuracy again."""
    return F.relu(x) if gate is None else x * gate.to(x.dtype)


def activation_pattern(params, xs, xt, beta, cfg: "PathConfig") -> Dict[str, torch.Tensor]:
    """The ReLU on/off pattern of a plain (dropout-free) oracle forward, in the ``gates`` format
    (M = Bs+Bt rows, source first) -- used to test the gate plumbing against itself."""
    p = params
    T, Fd, R = cfg.num_segments, cfg.shared_dim, cfg.num_segments - 1
    tuples = relation_tuples(T)
    x = torch.cat([xs, xt], 0)
    M = x.size(0)
    pre = F.linear(x.reshape(-1, x.size(-1)), p["fc_feature_shared_source.weight"], p["fc_feature_shared_source.bias"])
    feat = F.relu(pre)
    hf = F.linear(feat, p["fc_feature_domain.weight"], p["fc_feature_domain.bias"])
    g = {"shared": pre > 0, "frame_disc": hf > 0}
    if cfg.use_attn_frame != "none":
        pf = F.linear(F.relu(hf), p["fc_classifier_domain.weight"], p["fc_classifier_domain.bias"])
        feat = (entropy_attention(pf).view(-1, 1) + 1) * feat
    f3 = feat.view(M, T, Fd)
    trn, rel = [], []
    for i, rels in enumerate(tuples):
        acc = 0
        for tau in rels:
            z = F.linear(f3[:, list(tau), :].reshape(M, -1), p[f"TRN.fc_fusion_scales.{i}.1.weight"],
                         p[f"TRN.fc_fusion_scales.{i}.1.bias"])
            trn.append(z > 0)
            acc = acc + F.relu(z)
        rel.append(acc)
    g["trn"] = trn
    hr = [F.linear(rel[i], p[f"relation_domain_classifier_all.{i}.0.weight"],
                   p[f"relation_domain_classifier_all.{i}.0.bias"]) for i in range(R)]
    g["rel_disc"] = [h > 0 for h in hr]
    relf = torch.stack(rel, 1)
    if cfg.use_attn == "general":
        relf = (general_attention(p, relf).unsqueeze(-1) + 1) * relf
    elif cfg.use_attn != "none":
        pr = torch.stack([F.linear(F.relu(hr[i]), p[f"relation_domain_classifier_all.{i}.2.weight"],
                                   p[f"relation_domain_classifier_all.{i}.2.bias"]) for i in range(R)], 1)
        w = entropy_attention(pr.reshape(-1, 2)).view(M, R)
        relf = (w.unsqueeze(-1) + 1) * relf
    vid = relf.sum(1)
    g["video_disc"] = F.linear(vid, p["fc_feature_domain_video.weight"], p["fc_feature_domain_video.bias"]) > 0
    return g


def trn_multiscale(x: torch.Tensor, weights: Sequence[torch.Tensor], biases: Sequence[torch.Tensor],
                   tuples: List[List[Tuple[int, ...]]], gates: Optional[Sequence[torch.Tensor]] = None,
                   input_relu: bool = True) -> torch.Tensor:
    """RelationModuleMultiScale.forward (TRNmodule.py:58-82).

    x (N, T, F) -> (N, T-1, H);  out[:, i] = sum_r relu(W_i . concat_j relu(x[:, tau_ir[j]]) + b_i)
    ``gates`` (optional): one (N,H) 0/1 tensor per evaluated relation, see ``_relu``.
    ``input_relu=False`` drops the leading nn.ReLU (TRNmodule.py:49): inside VideoModel its input is the
    already rectified shared feature, so it is an identity -- and when the shared layer's pattern is
    pinned by a gate it must not re-decide the sign of the few units the gate kept at a tiny negative value.
    """
    per_scale = []
    q = 0
    for i, rels in enumerate(tuples):
        acc = None
        for tau in rels:
            u = x[:, list(tau), :].reshape(x.size(0), -1)             # :60-61 / :75-76
            a = _relu(F.linear(F.relu(u) if input_relu else u, weights[i], biases[i]),   # :46-54 ReLU-Linear-ReLU
                      None if gates is None else gates[q])
            q += 1
            acc = a if acc is None else acc + a                        # :79
        per_scale.append(acc.unsqueeze(1))
    return torch.cat(per_scale, 1)                                     # :81


def two_layer_disc(x: torch.Tensor, w1, b1, w2, b2, beta: float, gate: Optional[torch.Tensor] = None) -> torch.Tensor:
    """GradReverse -> Linear -> ReLU -> Linear(->2) (models.py:456-470, 477-479)."""
    h = _relu(F.linear(grad_reverse(x, beta), w1, b1), gate)
    return F.linear(h, w2, b2)


# ----------------------------------------------------------------------------
# one domain through the path                            models.py:557-704
# ----------------------------------------------------------------------------
def _forward_domain(p: Dict[str, torch.Tensor], x: torch.Tensor, beta: Sequence[float], mu: float,
                    cfg: PathConfig, train: bool, reverse: bool,
                    mask_i: Optional[torch.Tensor], mask_v: Optional[torch.Tensor],
                    gates: Optional[Dict[str, torch.Tensor]] = None):
    T, Fd, H = cfg.num_segments, cfg.shared_dim, NUM_BOTTLENECK
    R = T - 1
    batch = x.size(0)
    tuples = relation_tuples(T)
    gates = gates or {}

    flat = x.reshape(-1, x.size(-1))                                                   # :557
    feat = F.linear(flat, p["fc_feature_shared_source.weight"], p["fc_feature_shared_source.bias"])  # :565
    feat = _relu(feat, gates.get("shared"))                                            # :572
    feat = _apply_dropout(feat, cfg.dropout_i, train, mask_i)                          # :574
    feat_frames = feat.view(batch, T, Fd)                                              # :578

    pred_frame = two_layer_disc(feat, p["fc_feature_domain.weight"], p["fc_feature_domain.bias"],
                                p["fc_classifier_domain.weight"], p["fc_classifier_domain.bias"],
                                beta[2], gates.get("frame_disc"))                      # :606
    if cfg.use_attn_frame != "none":                                                   # :612-614, :368-377
        w_frame = entropy_attention(pred_frame)
        feat = (w_frame.view(-1, 1) + 1) * feat

    # fc_classifier_source (:617) is executed by the reference but its output is
    # dropped for baseline_type='video' (:437-441); it has no effect on any output.

    if cfg.frame_aggregation == "avgpool":
        return _forward_domain_avgpool(p, feat, feat_frames, pred_frame, beta, mu, cfg, train, reverse, mask_v, gates)

    rel = trn_multiscale(feat.view(batch, T, Fd),
                         [p[f"TRN.fc_fusion_scales.{i}.1.weight"] for i in range(R)],
                         [p[f"TRN.fc_fusion_scales.{i}.1.bias"] for i in range(R)],
                         tuples, gates.get("trn"), input_relu="shared" not in gates)   # :635

    pred_rel = torch.stack(
        [two_layer_disc(rel[:, i, :],
                        p[f"relation_domain_classifier_all.{i}.0.weight"],
                        p[f"relation_domain_classifier_all.{i}.0.bias"],
                        p[f"relation_domain_classifier_all.{i}.2.weight"],
                        p[f"relation_domain_classifier_all.{i}.2.bias"], beta[0],
                        None if "rel_disc" not in gates else gates["rel_disc"][i])
         for i in range(R)], 1)                                                        # :472-488 -> (B,R,2)

    if cfg.use_attn != "none":                                                         # :643-645, :379-388
        if cfg.use_attn == "general":                                                  # :382-383, :359-366
            w_rel = general_attention(p, rel)
        else:
            w_rel = entropy_attention(pred_rel.reshape(-1, 2)).view(batch, R)
        rel_att = (w_rel.unsqueeze(-1) + 1) * rel
        attn = w_rel
    else:                                                                              # :647
        rel_att = rel
        attn = rel[:, :, 0]

    feat_video = rel_att.sum(1)                                                        # :651
    vid = _apply_dropout(feat_video, cfg.dropout_v, train, mask_v)                     # :679
    if reverse:                                                                        # :682-684
        vid = grad_reverse(vid, mu)
    pred_video = F.linear(vid, p["fc_classifier_video_source.weight"],
                          p["fc_classifier_video_source.bias"])                        # :686
    pred_dom_video = two_layer_disc(vid, p["fc_feature_domain_video.weight"],
                                    p["fc_feature_domain_video.bias"],
                                    p["fc_classifier_domain_video.weight"],
                                    p["fc_classifier_domain_video.bias"], beta[1],
                                    gates.get("video_disc"))                           # :694

    pred_domain = [pred_rel, pred_dom_video, pred_frame.view(batch, T, 2)]            # reversed list, :722
    feats = [pred_video, feat_video, feat_frames]                                      # reversed list, :722
    pred_video_2 = pred_video                                                          # :713 out_2 = out
    if cfg.ens_DA == "MCD":                                                            # :716-720 (share_params == 'Y')
        pred_video_2 = F.linear(vid, p["fc_classifier_video_source_2.weight"], p["fc_classifier_video_source_2.bias"])
    return attn, pred_video, pred_video_2, pred_domain, feats


def _forward_domain_avgpool(p, feat, feat_frames, pred_frame, beta, mu, cfg: PathConfig, train: bool, reverse: bool,
                            mask_v, gates):
    """frame_aggregation='avgpool' behind the frame level (models.py:620-626, 425-433, 679-706): the frame features,
    re-weighted by the frame-level domain attention under use_attn='TransAttn' (:427-430), are averaged over the segments
    (:432); the video-level layers are shared_dim wide (:240-241, 250); there is no relation level -- the reference puts
    the video-level domain prediction into that slot of pred_domain (:703-706) and the first feature of every video into
    the attention output (:624-626)."""
    batch, T, Fd = feat_frames.size(0), cfg.num_segments, cfg.shared_dim
    if cfg.use_attn == "TransAttn":                                                     # :427-430
        feat = (entropy_attention(pred_frame).view(-1, 1) + 1) * feat
    feat_video = feat.view(batch, T, Fd).sum(1) / T                                     # :432 AvgPool2d([T, 1])
    attn = feat_video[:, 0]                                                             # :625-626
    vid = _apply_dropout(feat_video, cfg.dropout_v, train, mask_v)                      # :679
    if reverse:                                                                         # :682-684
        vid = grad_reverse(vid, mu)
    pred_video = F.linear(vid, p["fc_classifier_video_source.weight"], p["fc_classifier_video_source.bias"])   # :686
    pred_dom_video = two_layer_disc(vid, p["fc_feature_domain_video.weight"], p["fc_feature_domain_video.bias"],
                                    p["fc_classifier_domain_video.weight"], p["fc_classifier_domain_video.bias"],
                                    beta[1], gates.get("video_disc"))                   # :694
    pred_domain = [pred_dom_video, pred_dom_video, pred_frame.view(batch, T, 2)]        # :705-706 dummy relation slot
    feats = [pred_video, feat_video, feat_frames]
    pred_video_2 = pred_video
    if cfg.ens_DA == "MCD":
        pred_video_2 = F.linear(vid, p["fc_classifier_video_source_2.weight"], p["fc_classifier_video_source_2.bias"])
    return attn, pred_video, pred_video_2, pred_domain, feats


def split_gates(gates: Optional[Dict[str, torch.Tensor]], bs: int, T: int):
    """Split activation-pattern gates given for M = Bs+Bt rows (source first) into per-domain dicts.
    Keys: 'shared', 'frame_disc' (M*T,F); 'trn' (n_rel,M,H); 'rel_disc' (R,M,H); 'video_disc' (M,H)."""
    if not gates:
        return None, None
    out = ({}, {})
    for k, g in gates.items():
        if k in ("shared", "frame_disc"):
            out[0][k], out[1][k] = g[:bs * T], g[bs * T:]
        elif k in ("trn", "rel_disc"):
            out[0][k], out[1][k] = [t[:bs] for t in g], [t[bs:] for t in g]
        else:
            out[0][k], out[1][k] = g[:bs], g[bs:]
    return out


def forward(params: Dict[str, torch.Tensor], input_source: torch.Tensor, input_target: torch.Tensor,
            beta: Sequence[float], mu: float, cfg: PathConfig, train: bool = True, reverse: bool = False,
            masks: Optional[Dict[str, torch.Tensor]] = None, gates: Optional[Dict[str, torch.Tensor]] = None):
    """VideoModel.forward (models.py:545-722) -> the reference's 10-tuple.

    ``masks`` may hold keep-masks 'i_source' (Bs*T,F), 'i_target', 'v_source' (Bs,H), 'v_target'.
    ``gates`` pins the ReLU activation pattern (see ``_relu`` / ``split_gates``); default: real ReLUs.
    """
    masks = masks or {}
    gs, gt = split_gates(gates, input_source.size(0), cfg.num_segments)
    src = _forward_domain(params, input_source, beta, mu, cfg, train, reverse,
                          masks.get("i_source"), masks.get("v_source"), gs)
    tgt = _forward_domain(params, input_target, beta, mu, cfg, train, reverse,
                          masks.get("i_target"), masks.get("v_target"), gt)
    return src + tgt


# ----------------------------------------------------------------------------
# loss composition of the shipped script     main.py:446, 508-538, 559-562
# ----------------------------------------------------------------------------
def attentive_entropy(pred: torch.Tensor, pred_domain: torch.Tensor) -> torch.Tensor:
    """loss.py:15-25."""
    dq = F.softmax(pred_domain, dim=1)
    dlq = F.log_softmax(pred_domain, dim=1)
    weights = 1 + torch.sum(-dq * dlq, 1)
    q = F.softmax(pred, dim=1)
    lq = F.log_softmax(pred, dim=1)
    return torch.mean(weights * torch.sum(-q * lq, 1))


def dis_MCD(out1: torch.Tensor, out2: torch.Tensor) -> torch.Tensor:
    """loss.py:29-30: the classifier discrepancy of MCD (main.py:548-556)."""
    return torch.mean(torch.abs(F.softmax(out1, dim=1) - F.softmax(out2, dim=1)))


def compose_loss(outputs, label_source: torch.Tensor, gamma: float = 0.003,
                 place_adv: Sequence[str] = ("Y", "Y", "Y"), use_attn: str = "TransAttn",
                 class_weight: Optional[torch.Tensor] = None,
                 domain_weight: Optional[torch.Tensor] = None) -> torch.Tensor:
    """use_target='uSv', adv_DA='RevGrad', add_loss_DA='attentive_entropy'.

    main.py:160-167  weight_source_class (--weighted_class_loss) / weight_domain_loss (--weighted_class_loss_DA)
    main.py:204-205  criterion = CrossEntropyLoss(weight=weight_source_class), criterion_domain = ...(weight_domain_loss)
    main.py:446      class CE on source only
    main.py:508-538  for l in (relation, video, frame): CE(cat(pred_S, pred_T), cat(0s, 1s))
    main.py:559-562  + gamma * attentive_entropy(cat(out_S, out_T), pred_domain_all[1])
                     (only when use_attn != 'none', main.py:559)
    """
    (_, out_s, _, pd_s, _, _, out_t, _, pd_t, _) = outputs
    cw = None if class_weight is None else class_weight.to(out_s.dtype)
    dw = None if domain_weight is None else torch.as_tensor(domain_weight).to(out_s.dtype)
    loss = F.cross_entropy(out_s, label_source, weight=cw)
    stacked = []
    for lvl, flag in enumerate(place_adv):
        if flag != "Y":
            continue
        ps = pd_s[lvl].reshape(-1, 2)
        pt = pd_t[lvl].reshape(-1, 2)
        dom = torch.cat([torch.zeros(ps.size(0), dtype=torch.long),
                         torch.ones(pt.size(0), dtype=torch.long)])
        both = torch.cat([ps, pt], 0)
        stacked.append(both)
        loss = loss + F.cross_entropy(both, dom, weight=dw)
    if use_attn != "none" and len(stacked) > 1:
        loss = loss + gamma * attentive_entropy(torch.cat([out_s, out_t], 0), stacked[1])
    return loss


def train_step(params: Dict[str, torch.Tensor], xs, xt, labels, beta, cfg: PathConfig,
               gamma: float = 0.003, train: bool = True, masks=None, gates=None, class_weight=None,
               domain_weight=None):
    """forward + composed loss + backward; returns (loss, outputs, grads-by-name)."""
    names = used_param_names(params)
    leaves = {k: params[k].detach().clone().requires_grad_(True) for k in names}
    live = dict(params)
    live.update(leaves)
    outs = forward(live, xs, xt, beta, 0.0, cfg, train=train, reverse=False, masks=masks, gates=gates)
    loss = compose_loss(outs, labels, gamma, use_attn=cfg.use_attn, class_weight=class_weight,
                        domain_weight=domain_weight)
    grads = torch.autograd.grad(loss, [leaves[k] for k in names], allow_unused=True)
    return loss.detach(), outs, OrderedDict(zip(names, grads))


def synthetic_batch(batch: int, cfg: PathConfig, seed: int = 4321, dtype=torch.float32):
    """Synthetic (B,T,2048) N(0,1) features and labels arange(B) % C (SURVEY §8d)."""
    g = torch.Generator().manual_seed(seed)
    xs = torch.randn(batch, cfg.num_segments, FEATURE_DIM, generator=g).to(dtype)
    xt = torch.randn(batch, cfg.num_segments, FEATURE_DIM, generator=g).to(dtype)
    labels = torch.arange(batch) % cfg.num_class
    return xs, xt, labels


# ---- the optimizer step that follows loss.backward() (SURVEY 8f row n2) ------------------------------------
def clip_grad_norm(grads: Dict[str, torch.Tensor], max_norm: float) -> Tuple[torch.Tensor, torch.Tensor]:
    """``clip_grad_norm_(model.parameters(), args.clip_gradient)`` of main.py:578-581 restated on a dict of
    gradients (in place).  torch.nn.utils.clip_grad_norm_: total = ||(||g_i||_2)_i||_2,
    coef = clamp(max_norm / (total + 1e-6), max=1), g_i *= coef.  Returns (total_norm, coef)."""
    total = torch.linalg.vector_norm(torch.stack([torch.linalg.vector_norm(g) for g in grads.values()]))
    coef = torch.clamp(max_norm / (total + 1e-6), max=1.0)
    for g in grads.values():
        g.mul_(coef)
    return total, coef


def sgd_nesterov_step(params: Dict[str, torch.Tensor], grads: Dict[str, torch.Tensor],
                      bufs: Dict[str, torch.Tensor], lr: float, momentum: float = 0.9,
                      weight_decay: float = 1e-4) -> None:
    """``torch.optim.SGD(params, lr, momentum, weight_decay, nesterov=True).step()`` (main.py:83, 583), in
    place on ``params`` / ``bufs``.  Only parameters that received a gradient are touched (SGD skips
    ``grad is None``).  The first step of torch clones d into the buffer; a zero-initialised buffer gives the
    same value (momentum*0 + d)."""
    for k, g in grads.items():
        d = g.add(params[k], alpha=weight_decay)
        buf = bufs.setdefault(k, torch.zeros_like(d))
        buf.mul_(momentum).add_(d)
        params[k].add_(d.add(buf, alpha=momentum), alpha=-lr)


def lr_dann(lr0: float, p: float) -> float:
    """adjust_learning_rate_dann, main.py:800-802 (p = progress in [0, 1], main.py:349)."""
    return lr0 / (1.0 + 10.0 * p) ** 0.75


def beta_dann(p: float) -> float:
    """main.py:350: the value that replaces negative entries of --beta."""
    return 2.0 / (1.0 + math.exp(-10.0 * p)) - 1.0


def train_iteration(params, bufs, xs, xt, labels, beta, cfg: PathConfig, lr: float, gamma: float = 0.003,
                    momentum: float = 0.9, weight_decay: float = 1e-4, clip_gradient: Optional[float] = 20.0,
                    train: bool = True, masks=None, gates=None):
    """One full iteration of main.py:418-583: train_step, clip, SGD-Nesterov.  Updates params/bufs in place;
    returns (loss, total_norm or None)."""
    loss, _, grads = train_step(params, xs, xt, labels, beta, cfg, gamma, train=train, masks=masks, gates=gates)
    grads = OrderedDict((k, g.clone()) for k, g in grads.items() if g is not None)
    total = None
    if clip_gradient is not None:
        total, _ = clip_grad_norm(grads, clip_gradient)
    sgd_nesterov_step(params, grads, bufs, lr, momentum, weight_decay)
    return loss, total
