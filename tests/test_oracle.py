"""CPU: the fp32 restatement (oracle/mudpt_oracle.py) against the golden vectors that
oracle/make_golden.py produced by running the REFERENCE (trainers/mudpt.py:249-251)."""
import numpy as np
import pytest
import torch

from oracle import mudpt_oracle as orc
from tests import golden_util as gu


@pytest.mark.parametrize("name", gu.TINY + ["vitb16_cfg1"])
def test_oracle_matches_reference_golden(name):
    c = gu.load(name)
    g = c["golden"]
    torch.set_num_threads(8)
    res = orc.forward_backward(c["sd"], c["image"], c["tokenized"], c["labels"])
    np.testing.assert_allclose(res["logits"].numpy(), g["logits"], rtol=0, atol=2e-4)
    np.testing.assert_allclose(res["image_features"].numpy(), g["image_features"], rtol=1e-4, atol=2e-5)
    np.testing.assert_allclose(res["text_features"].numpy(), g["text_features"], rtol=1e-4, atol=2e-5)
    np.testing.assert_allclose(float(res["loss"]), float(g["loss"]), rtol=1e-5, atol=1e-5)
    for k in orc.TRAINABLE:
        ref = torch.from_numpy(g["grad/" + k])
        m = orc.metrics(res["grads"][k], ref) if ref.numel() else {"cos": 1.0, "rel_l2": 0.0}
        if ref.numel() and float(ref.norm()) > 0:
            assert m["cos"] > 0.99999 and m["rel_l2"] < 2e-3, (k, m)


def test_golden_low_rank_storage_round_trip(tmp_path, monkeypatch):
    """golden_util.save keeps a low-rank weight gradient as two factors and loading multiplies them back; a full-rank
    gradient and every other array are stored as they are."""
    rng = np.random.default_rng(0)
    arrays = {"grad/low": (rng.standard_normal((300, 3)) @ rng.standard_normal((3, 200))).astype(np.float32),
              "grad/full": rng.standard_normal((100, 100)).astype(np.float32),
              "logits": rng.standard_normal((4, 7)).astype(np.float32), "arch": np.array("tiny")}
    monkeypatch.setattr(gu, "GOLDEN_DIR", str(tmp_path))
    gu.save(str(tmp_path / "case.npz"), arrays)
    stored = np.load(tmp_path / "case.npz").files
    assert "grad/low" not in stored and gu.LOWRANK + "grad/low/a" in stored and "grad/full" in stored
    back = gu._read("case")
    assert set(back) == set(arrays)
    low = arrays["grad/low"]
    assert back["grad/low"].dtype == np.float32 and np.abs(back["grad/low"] - low).max() <= 1e-6 * np.abs(low).max()
    for k in ("grad/full", "logits", "arch"):
        assert np.array_equal(back[k], arrays[k]), k


def test_post_eot_tokens_are_dead():
    """SURVEY.md 8c(i): tokens after EOT do not influence features or gradients (causal mask),
    so the text tower may be truncated to max(eot)+1 rows exactly."""
    c = gu.load("tiny_a")
    sd = dict(c["sd"])
    res0 = orc.forward_backward(sd, c["image"], c["tokenized"], c["labels"])
    eot = c["tokenized"].argmax(-1)
    suf = sd["mudpt_prompt_learner.token_suffix"].clone()
    n_ctx = c["n_ctx"]
    for i, e in enumerate(eot.tolist()):
        suf[i, e + 1 - (1 + n_ctx):] += 5.0 * torch.randn_like(suf[i, e + 1 - (1 + n_ctx):])
    sd["mudpt_prompt_learner.token_suffix"] = suf
    res1 = orc.forward_backward(sd, c["image"], c["tokenized"], c["labels"])
    assert torch.equal(res0["logits"], res1["logits"])
    for k in orc.TRAINABLE:
        assert torch.equal(res0["grads"][k], res1["grads"][k]), k


def test_truncated_text_tower_equals_full():
    c = gu.load("tiny_d")
    sd = c["sd"]
    prompts, shared, deep, t2v = orc.prompt_learner(sd)
    eot = c["tokenized"].argmax(-1).long()
    full = orc.text_tower(sd, prompts, eot, deep)
    L = int(eot.max()) + 1
    trunc = orc.text_tower(sd, prompts[:, :L], eot, deep)
    np.testing.assert_allclose(trunc.numpy(), full.numpy(), rtol=1e-5, atol=1e-6)


@pytest.mark.needs_reference
def test_oracle_matches_live_reference():
    """Pin the restatement against the reference run live (build container only)."""
    import torch.nn.functional as F
    from oracle import ref_shims
    model, cfg = ref_shims.build_reference_model("tiny", [f"class {i}" for i in range(6)], seed=3, n_ctx=2, depth=3)
    sd = {k: v.detach().clone() for k, v in model.state_dict().items()}
    g = torch.Generator().manual_seed(5)
    image = torch.randn(3, 3, 32, 32, generator=g)
    labels = torch.tensor([1, 5, 0])
    logits = model(image)
    loss = F.cross_entropy(logits, labels)
    loss.backward()
    res = orc.forward_backward(sd, image, model.tokenized_prompts, labels)
    np.testing.assert_allclose(res["logits"].numpy(), logits.detach().numpy(), atol=1e-4, rtol=0)
    for n, p in model.named_parameters():
        if p.requires_grad:
            m = orc.metrics(res["grads"][n], p.grad)
            assert m["cos"] > 0.99999, (n, m)


# ---------------------------------------------------------------------------------------------
# CoCoOp (BASELINE config 4): oracle/cocoop_oracle.py against the reference's trainers/cocoop.py
# ---------------------------------------------------------------------------------------------

@pytest.mark.parametrize("name", gu.COCOOP)
def test_cocoop_oracle_matches_reference_golden(name):
    from oracle import cocoop_oracle as co
    c = gu.load_cocoop(name)
    g = c["golden"]
    res = co.forward_backward(c["sd"], c["image"], c["tokenized"], c["labels"])
    np.testing.assert_allclose(res["logits"].numpy(), g["logits"], rtol=0, atol=2e-4)
    np.testing.assert_allclose(float(res["loss"]), float(g["loss"]), rtol=1e-5, atol=1e-5)
    for k in co.TRAINABLE:
        m = orc.metrics(res["grads"][k], torch.from_numpy(g["grad/" + k]))
        assert m["cos"] > 0.99999 and m["rel_l2"] < 2e-3, (k, m)


@pytest.mark.needs_reference
def test_cocoop_oracle_matches_live_reference():
    from oracle import cocoop_oracle as co, ref_shims
    from mudpt_b200 import synthetic as syn
    _, clip_model_mod, _ = ref_shims.import_reference()
    ref_cocoop = ref_shims.import_reference_cocoop()
    arch = syn.ARCHS["tiny"]
    cfg = ref_shims.make_cfg(n_ctx=3, depth=1, ctx_init="", size=arch.image_resolution, name="CoCoOp")
    torch.manual_seed(11)
    clip_model = clip_model_mod.CLIP(*arch.astuple(), None).float()
    model = ref_cocoop.CustomCLIP(cfg, ["dog", "class 7", "small red bird"], clip_model)
    sd = {k: v.detach().clone() for k, v in model.state_dict().items()}
    image = torch.randn(2, 3, 32, 32, generator=torch.Generator().manual_seed(5))
    labels = torch.tensor([2, 0])
    model.train()
    loss = model(image, labels)
    loss.backward()
    res = co.forward_backward(sd, image, model.tokenized_prompts, labels)
    np.testing.assert_allclose(float(res["loss"]), float(loss.detach()), rtol=1e-5, atol=1e-5)
    for k in co.TRAINABLE:
        p = dict(model.named_parameters())[k]
        m = orc.metrics(res["grads"][k], p.grad)
        assert m["cos"] > 0.99999, (k, m)
