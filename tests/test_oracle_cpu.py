"""Pins oracle/restatement.py against the golden fixtures produced by the REAL reference
(oracle/make_golden.py, oracle/make_golden_generate.py, oracle/make_golden_checks.py)."""
import glob
import os

import numpy as np
import pytest
import torch

import open_musiclm_b200 as O
from oracle import restatement as R
from oracle.make_golden_checks import digest

GOLD = sorted(glob.glob(os.path.join(os.path.dirname(__file__), "golden", "tiny_*.pt")))
CHECKS = os.path.join(os.path.dirname(__file__), "golden", "reference_checks.pt")


def cfg_from_fixture(fx):
    kw = fx["kwargs"]
    common = dict(dim=kw["dim"], depth=kw["depth"], heads=kw["heads"], ff_dropout=kw["ff_dropout"],
                  grad_shrink_alpha=kw["grad_shrink_alpha"], ce_weights=fx["ce_weights"],
                  use_conv_ff=kw.get("use_conv_ff", True), rel_pos_bias_type=kw.get("relative_position_bias_type", "continuous"),
                  abs_pos=kw.get("use_absolute_position_embeddings", False))
    cb = kw.get("clap_codebook_size", 1024)
    if fx["stage"] == "semantic":
        return R.semantic_cfg(codebook=cb, n_clap_q=kw["num_clap_quantizers"], **common)
    if fx["stage"] == "coarse":
        return R.coarse_cfg(codebook=cb, n_clap_q=kw["num_clap_quantizers"], n_coarse_q=kw["num_coarse_quantizers"], **common)
    return R.fine_cfg(codebook=cb, n_clap_q=kw["num_clap_quantizers"], n_coarse_q=kw["num_coarse_quantizers"],
                      n_fine_q=kw["num_fine_quantizers"], **common)


def rel(a, b):
    return float((a.double() - b.double()).norm() / b.double().norm().clamp_min(1e-30))


@pytest.mark.parametrize("path", GOLD, ids=[os.path.basename(p) for p in GOLD])
def test_restatement_matches_reference_fixture(path):
    fx = torch.load(path, weights_only=False)
    cfg = cfg_from_fixture(fx)
    sd = {k: v.clone().requires_grad_(v.is_floating_point() and not k.endswith("beta")) for k, v in fx["state_dict"].items()}
    toks = [t.numpy() for t in fx["tokens"]]
    loss, logits, labels, ids, mask = R.loss_and_logits(cfg, sd, toks)
    # integer path: bit exact
    for a, b in zip(ids, fx["ids"]):
        assert np.array_equal(a, b.numpy())
    assert np.array_equal(mask, fx["key_mask"].numpy())
    for a, b in zip(labels, fx["labels"]):
        assert np.array_equal(a, b.numpy())
    # floating point path
    for a, b in zip(logits, fx["logits"]):
        assert a.shape == b.shape
        assert rel(a.detach(), b) < 2e-5
    assert abs(float(loss) - float(fx["loss"])) / abs(float(fx["loss"])) < 1e-5
    loss.backward()
    for k, gref in fx["grads"].items():
        g = sd[k].grad
        if gref is None:
            assert g is None or float(g.abs().max()) == 0.0, k
        elif float(gref.norm()) < 1e-6:
            # e.g. rel_pos_bias.net.3.bias: a per-head constant cancels in the softmax, gradient is rounding noise
            assert float(g.norm()) < 1e-5, k
        else:
            assert rel(g, gref) < 2e-4, (k, rel(g, gref))


def test_restatement_optimizer_steps():
    path = [p for p in GOLD if p.endswith("tiny_coarse.pt")][0]
    fx = torch.load(path, weights_only=False)
    cfg = cfg_from_fixture(fx)
    params = {k: v.clone() for k, v in fx["state_dict"].items() if not k.endswith("beta")}
    toks = [t.numpy() for t in fx["tokens"]]
    state = {}
    for it, gold in enumerate(fx["opt_steps"]):
        sd = {k: v.clone().requires_grad_(True) for k, v in params.items()}
        for k, v in fx["state_dict"].items():
            if k.endswith("beta"):
                sd[k] = v
        loss, *_ = R.loss_and_logits(cfg, sd, toks)
        loss.backward()
        grads = {k: sd[k].grad for k in params}
        assert abs(float(loss) - float(gold["loss"])) / float(gold["loss"]) < 1e-4
        norm = R.clip_and_adamw(params, grads, state, step=it, lr=3e-4, wd=1e-2, warmup_iters=10)
        assert abs(norm - float(gold["grad_norm"])) / float(gold["grad_norm"]) < 1e-4
        if gold["params"] is not None:
            for k, v in gold["params"].items():
                if fx["grads"][k] is not None and float(fx["grads"][k].norm()) < 1e-6:
                    continue    # gradient is rounding noise (softmax-invariant bias): Adam turns its sign into +-lr
                assert rel(params[k], v) < 1e-5, k


def test_forgetful_mask_matches_reference():
    """The reference's utils.generate_mask_with_prob((4, 50), 0.15) after torch.manual_seed(11) is stored in
    tests/golden/reference_checks.pt."""
    m_ref = torch.load(CHECKS, weights_only=False)["mask"]
    shape = (4, 50)
    torch.manual_seed(11)
    rand = torch.randn(shape)
    m = R.forgetful_mask(shape, 0.15, rand.numpy())
    assert np.array_equal(m, m_ref.numpy())


@pytest.mark.parametrize("stage", ["semantic", "coarse", "fine"])
def test_restatement_matches_reference_live(stage):
    """Mid-size random config against what the reference computed for it (tests/golden/reference_checks.pt): its loss
    and a fixed, seeded sample of its logits, on its own initial weights under torch.manual_seed(5) (rebuilt here with
    the bit-identical init of this package and checked against the reference's digests)."""
    fx = torch.load(CHECKS, weights_only=False)["live"][stage]
    torch.manual_seed(5)
    model = getattr(O, f"create_{stage}_transformer")(**fx["kwargs"])
    sd = {k: v.detach() for k, v in model.state_dict().items()}
    assert [(k, tuple(v.shape), str(v.dtype), digest(v)) for k, v in sd.items()] == fx["state"]
    kw = dict(dim=192, depth=2, heads=3, ce_weights=fx["ce_weights"])
    if stage == "semantic":
        cfg = R.semantic_cfg(**kw)
    elif stage == "coarse":
        cfg = R.coarse_cfg(**kw)
    else:
        cfg = R.fine_cfg(**kw)
    loss, logits, *_ = R.loss_and_logits(cfg, sd, [t.numpy() for t in fx["tokens"]])
    assert abs(float(loss) - float(fx["loss"])) / float(fx["loss"]) < 1e-5
    assert len(logits) == len(fx["logits"])
    for a, b in zip(logits, fx["logits"]):
        assert tuple(a.shape) == b["shape"]
        assert rel(a.reshape(-1)[b["index"].long()], b["value"]) < 2e-5


GEN = sorted(glob.glob(os.path.join(os.path.dirname(__file__), "golden", "gen_*.pt")))


def _cfg_of(fx):
    kw = fx["kwargs"]
    base = dict(dim=kw["dim"], depth=kw["depth"], heads=kw["heads"], codebook=kw.get("clap_codebook_size", 1024),
                n_clap_q=kw.get("num_clap_quantizers", 12))
    if fx["stage"] == "semantic":
        return R.semantic_cfg(**base)
    if fx["stage"] == "coarse":
        return R.coarse_cfg(n_coarse_q=kw["num_coarse_quantizers"], **base)
    return R.fine_cfg(n_coarse_q=kw["num_coarse_quantizers"], n_fine_q=kw["num_fine_quantizers"], **base)


@pytest.mark.parametrize("path", GEN, ids=[os.path.basename(p) for p in GEN])
def test_generate_restatement_reproduces_reference_tokens(path):
    """oracle.generate against the token sequences the REAL reference's wrapper.generate produced under the same
    Gumbel noise stream (oracle/make_golden_generate.py): bit-exact, including the eos handling and the [b, n, q] fold."""
    fx = torch.load(path, weights_only=False)
    cfg = _cfg_of(fx)
    uni = fx["uniforms"]
    out = R.generate(cfg, fx["state_dict"], [t.numpy() for t in fx["cond"]], lambda step, shape: uni[step],
                     pred_token_ids=None if fx["prefix"] is None else fx["prefix"].numpy(), max_time_steps=fx["max_time_steps"],
                     filter_thres=fx["filter_thres"], temperature=fx["temperature"],
                     include_eos_in_output=fx["include_eos_in_output"], allow_eos_in_output=fx["allow_eos_in_output"])
    assert out.shape == fx["out"].shape and torch.equal(out, fx["out"])
