"""Pin the oracle against the reference: what the unmodified reference computes for fixed seeds -- outputs,
gradients, initial parameters, a training loop, loss terms -- stored in tests/golden/reference_checks.npz by
oracle/gen_reference_checks.py, which holds the reference side of every check below."""
import pytest
import torch

from oracle import gen_golden
from oracle import gen_reference_checks as grc
from oracle import ta3n_oracle as orc
from tests.golden_util import STRUCTURAL_ZERO_GRADS, TOL_FP32, ReferenceCheck


@pytest.mark.parametrize("case", grc.OUTPUT_CASES)
def test_oracle_equals_live_reference(case):
    ref = ReferenceCheck(f"case/{case}")
    c = gen_golden.CASES[case]
    cfg, xs, xt, labels, masks = gen_golden.case_inputs(c)
    params = orc.init_params(cfg, seed=gen_golden.MODEL_SEED)       # the reference's init (test_oracle_golden.py)
    loss, outs, grads = orc.train_step(params, xs, xt, labels, gen_golden.BETA, cfg, gen_golden.GAMMA,
                                       train=c["train"], masks=masks)
    ref.assert_close("loss", loss, TOL_FP32, "loss")
    flat = grc.flat_outputs(outs)
    assert len(flat) == len(ref.names("out/"))
    for i, a in enumerate(flat):
        ref.assert_close(f"out/{i}", a, TOL_FP32, f"output {i}")
    for name in ref.meta["no_grad"]:
        assert name not in grads
    for name in ref.names("grad/"):
        if name in STRUCTURAL_ZERO_GRADS:
            assert ref.norm(f"grad/{name}") < 1e-6 and float(grads[name].norm()) < 1e-6
        else:
            ref.assert_close(f"grad/{name}", grads[name], 2e-4, f"grad {name}")


def test_reference_state_dict_keys_match_oracle_init():
    ref = ReferenceCheck("state_dict_init").meta
    p = orc.init_params(orc.PathConfig(num_class=12, num_segments=5, fc_dim=512), seed=7)
    assert list(p.keys()) == ref["keys"]
    for k, shape, digest in zip(ref["keys"], ref["shapes"], ref["sha256"]):
        assert list(p[k].shape) == shape, k
        assert grc.sha(p[k]) == digest, k          # bit for bit the reference's initial value


def test_oracle_train_iteration_equals_reference_loop():
    """main.py:418-583 on the reference (model forward, loss, backward, clip_grad_norm_, SGD-Nesterov step,
    DANN learning-rate schedule) against oracle.train_iteration, three iterations."""
    ref = ReferenceCheck("train_loop")
    c = gen_golden.CASES["cfg1_small_c5"]
    cfg, xs, xt, labels, masks = gen_golden.case_inputs(c)
    params = orc.init_params(cfg, seed=gen_golden.MODEL_SEED)
    bufs = {}
    lr0 = 3e-2
    for it in range(3):
        lr = orc.lr_dann(lr0, it / 3.0)
        loss, total = orc.train_iteration(params, bufs, xs, xt, labels, gen_golden.BETA, cfg, lr, gen_golden.GAMMA,
                                          clip_gradient=0.05, train=c["train"], masks=masks)
        ref.assert_close(f"loss/{it}", loss, TOL_FP32, f"loss it{it}")
        ref.assert_close(f"total_norm/{it}", total, 1e-5, f"total_norm it{it}")
        assert float(ref[f"total_norm/{it}"]) > 0.05
    for name in ref.names("param/"):
        ref.assert_close(f"param/{name}", params[name], 1e-6, f"param {name}")


def test_weighted_losses_match_the_reference_criteria():
    """main.py:160-167, 204-205: criterion / criterion_domain with class / domain weights, on the reference's
    outputs, against oracle.compose_loss(class_weight=, domain_weight=)."""
    ref = ReferenceCheck("weighted_losses")
    labels = gen_golden.case_inputs(gen_golden.CASES["ragged_6_3"])[3]
    cw = 1.0 / torch.tensor([0.05, 0.2, 0.1, 0.05, 0.1, 0.05, 0.05, 0.1, 0.1, 0.05, 0.1, 0.05])
    dw = torch.tensor([1.0 / 300, 1.0 / 170])
    pd_s = [ref[f"pred_domain_s/{lvl}"] for lvl in range(3)]
    pd_t = [ref[f"pred_domain_t/{lvl}"] for lvl in range(3)]
    outs_ref = (None, ref["out_s"], None, pd_s, None, None, ref["out_t"], None, pd_t, None)
    got = orc.compose_loss(outs_ref, labels, gen_golden.GAMMA, class_weight=cw, domain_weight=dw)
    ref.assert_close("loss", got.detach(), 1e-6, "weighted loss")


def _perturbed_params(ref, cfg, seed):
    """The oracle side of gen_reference_checks._perturbed_variant: the reference's init (checked bit for bit), the
    same seeded noise on every weight, the batch drawn after it."""
    p_init = orc.init_params(cfg, seed=seed)
    assert list(p_init.keys()) == ref.meta["keys"]
    for k, digest in zip(ref.meta["keys"], ref.meta["sha256"]):
        assert grc.sha(p_init[k]) == digest, k
    g = torch.Generator().manual_seed(seed + 1)
    for k in ref.meta["param_names"]:               # the reference's named_parameters() order
        if "weight" in k:
            p_init[k].add_(0.02 * torch.randn(p_init[k].shape, generator=g))
    xs, xt = torch.randn(6, 5, 2048, generator=g), torch.randn(4, 5, 2048, generator=g)
    labels = torch.randint(0, cfg.num_class, (6,), generator=g)
    params = {k: v.detach().clone().requires_grad_(v.dtype.is_floating_point) for k, v in p_init.items()}
    return params, xs, xt, labels


@pytest.mark.parametrize("reverse,mu", grc.MCD_RUNS)
def test_oracle_mcd_variant_equals_live_reference(reverse, mu):
    """ens_DA='MCD' (models.py:276-279, 716-720; main.py:447, 548-556): the second video-level classifier, the
    `reverse=True` pass and the discrepancy loss dis_MCD (loss.py:29-30) -- outputs and every gradient of
       CE(out_s) + CE(out_s_2) - dis_MCD(out_t, out_t_2)  on the reference vs the oracle."""
    ref = ReferenceCheck(f"mcd/{reverse}_{mu}")
    cfg = orc.PathConfig(num_class=7, num_segments=5, fc_dim=512, dropout_i=0.0, dropout_v=0.0, ens_DA="MCD")
    params, xs, xt, labels = _perturbed_params(ref, cfg, 11)
    o = orc.forward(params, xs, xt, [0.75, 0.75, 0.5], mu, cfg, train=True, reverse=reverse)
    loss = torch.nn.functional.cross_entropy(o[1], labels) + torch.nn.functional.cross_entropy(o[2], labels) - \
        orc.dis_MCD(o[6], o[7])
    loss.backward()
    ref.assert_close("loss", loss.detach(), TOL_FP32, "MCD loss")
    for i in (1, 2, 6, 7):
        ref.assert_close(f"out/{i}", o[i].detach(), TOL_FP32, f"MCD output {i}")
    assert not torch.equal(o[1], o[2])
    for name in ref.names("grad/"):
        ref.assert_close(f"grad/{name}", params[name].grad, 2e-4, f"MCD grad {name}")


def test_oracle_general_attention_equals_live_reference():
    """use_attn='general' (models.py:320-325 attn_layer, :359-366 softmax over the relations, :379-388 re-weighting) with
    trained-like weights and a loss that also reads the attention weights themselves: outputs and every gradient."""
    ref = ReferenceCheck("general_attention")
    cfg = orc.PathConfig(num_class=9, num_segments=5, fc_dim=512, dropout_i=0.0, dropout_v=0.0, use_attn="general")
    params, xs, xt, labels = _perturbed_params(ref, cfg, 21)
    o = orc.forward(params, xs, xt, [0.75, 0.6, 0.5], 0, cfg, train=True, reverse=False)
    loss = grc.general_attention_loss(o, labels)
    loss.backward()
    ref.assert_close("loss", loss.detach(), TOL_FP32, "loss")
    for i in (0, 1, 5, 6):
        ref.assert_close(f"out/{i}", o[i].detach(), TOL_FP32, f"output {i}")
    assert float(ref["out/0"].std()) > 1e-3, "attention weights should not be uniform in this test"
    for name in ref.names("grad/"):
        if name in STRUCTURAL_ZERO_GRADS:
            assert ref.norm(f"grad/{name}") < 1e-6 and float(params[name].grad.norm()) < 1e-6
        else:
            ref.assert_close(f"grad/{name}", params[name].grad, 2e-4, f"grad {name}")
    assert ref.norm("grad/attn_layer.0.weight") > 0
