"""Pin the CPU oracle against the golden vectors produced by the unmodified reference
(tests/golden/make_golden.py, tests/golden/make_golden_full.py)."""
import os
import sys

import numpy as np
import pytest
import torch

from oracle import caption_oracle as O

GOLD = os.path.join(os.path.dirname(__file__), "golden")
CASES = ["tiny_default", "tiny_cfgpy", "tiny_variants"]


def _load(name):
    g = torch.load(os.path.join(GOLD, name + ".pt"), weights_only=False)
    cfg = O.OracleConfig(**g["ctor"])
    return g, cfg


@pytest.mark.parametrize("name", CASES)
def test_state_dict_layout(name):
    g, cfg = _load(name)
    shapes = O.param_shapes(cfg)
    assert list(shapes.keys()) == g["state_dict_keys"]
    for k, v in g["state_dict"].items():
        assert tuple(v.shape) == shapes[k], k
    # sinusoid table is reproduced bit-exactly (model.py:502-514)
    assert torch.equal(O.sinusoid_table(cfg.max_length - 1, cfg.decode_input_size),
                       g["state_dict"]["decoder.position_embedding.pos_table"])


@pytest.mark.parametrize("name", CASES)
def test_loss_and_logits(name):
    g, cfg = _load(name)
    logits = O.logits_forward(g["state_dict"], cfg, g["features"], g["positions"], g["captions"])
    torch.testing.assert_close(logits, g["logits"], rtol=1e-5, atol=1e-6)
    torch.testing.assert_close(logits, g["policy_logits"], rtol=1e-5, atol=1e-6)
    loss = O.loss_from_logits(cfg, logits, g["captions"])
    torch.testing.assert_close(loss, g["loss"], rtol=1e-6, atol=1e-6)


@pytest.mark.parametrize("name", CASES)
def test_grads(name):
    g, cfg = _load(name)
    loss, grads = O.loss_and_grads(g["state_dict"], cfg, g["features"], g["positions"], g["captions"])
    assert set(grads) == set(g["grads"])
    for k in grads:
        torch.testing.assert_close(grads[k], g["grads"][k], rtol=1e-4, atol=1e-7, msg=lambda m, k=k: f"{k}: {m}")


@pytest.mark.parametrize("name", CASES)
def test_adam_two_steps(name):
    g, cfg = _load(name)
    sd = {k: v.clone() for k, v in g["state_dict"].items()}
    losses = O.train_steps(sd, cfg, [(g["features"], g["positions"], g["captions"]),
                                     (g["features2"], g["positions2"], g["captions2"])])
    np.testing.assert_allclose(losses, g["adam_losses"].numpy(), rtol=1e-5)
    for k, v in g["state_dict_after_2_steps"].items():
        torch.testing.assert_close(sd[k], v, rtol=1e-4, atol=2e-6, msg=lambda m, k=k: f"{k}: {m}")


@pytest.mark.parametrize("name", CASES)
def test_greedy(name):
    g, cfg = _load(name)
    ids, att = O.generate_caption_vector(g["state_dict"], cfg, g["features"], g["positions"])
    assert torch.equal(ids, g["greedy_ids"])
    assert ids.shape == (g["features"].shape[0], cfg.max_length + 1)
    np.testing.assert_allclose(np.stack(att, 0), g["greedy_attention"].numpy(), rtol=1e-5, atol=1e-7)


@pytest.mark.parametrize("name", CASES)
@pytest.mark.parametrize("k", [2, 3])
def test_beam(name, k):
    g, cfg = _load(name)
    ids = O.beam_search(g["state_dict"], cfg, g["features"], g["positions"], beam_size=k)
    assert torch.equal(ids, g[f"beam{k}_ids"])


@pytest.mark.parametrize("name", CASES)
def test_policy_beam(name):
    g, cfg = _load(name)
    ids = O.beam_search(g["state_dict"], cfg, g["features"], g["positions"], beam_size=3, log_domain=True)
    assert torch.equal(ids, g["policy_beam3_ids"])


def _full_case(name):
    """tests/golden/full_width.pt: outputs of the unmodified reference at the benchmarked widths; weights / inputs are
    regenerated from their seeds and must hash to what the reference was run on."""
    sys.path.insert(0, GOLD)
    try:
        import make_golden_full as G
    finally:
        sys.path.remove(GOLD)
    case = torch.load(os.path.join(GOLD, "full_width.pt"), weights_only=False)[name]
    cfg, sd, f, p, c, sha = G.regenerate(name)
    if sha != case["sha256"]:
        pytest.skip("this torch build draws a different CPU random stream than the one the golden was made with")
    return case, cfg, sd, f, p, c


@pytest.mark.parametrize("name", ["modelA", "modelB"])
def test_full_width_reference_outputs(name):
    """The oracle against the reference at the BENCHMARKED widths (model A: ctor defaults, model B: core/config.py
    defaults, vocab 10k, 36 x 2048 regions): logits, loss, greedy ids and decision gaps, beam ids."""
    case, cfg, sd, f, p, c = _full_case(name)
    B, T, V = case["batch"], cfg.max_length - 1, cfg.num_vocab
    logits = O.logits_forward(sd, cfg, f, p, c).reshape(B, T, V)
    torch.testing.assert_close(logits[:, :, :64], case["logits_slice"], rtol=1e-5, atol=2e-6)
    torch.testing.assert_close(logits.max(dim=-1).values, case["logits_row_max"], rtol=1e-5, atol=2e-6)
    assert torch.equal(logits.argmax(dim=-1), case["logits_row_argmax"])
    assert abs(float(logits.double().abs().sum()) - float(case["logits_abs_sum"])) < 1e-6 * float(case["logits_abs_sum"])
    torch.testing.assert_close(O.loss_from_logits(cfg, logits, c), case["loss"], rtol=1e-6, atol=1e-6)
    ids, _, gaps = O.generate_caption_vector(sd, cfg, f, p, return_gaps=True)
    assert torch.equal(ids, case["greedy_ids"])
    torch.testing.assert_close(gaps, case["greedy_gaps"], rtol=1e-3, atol=2e-6)
    k = 3                                               # beam 5 of model A was checked when the golden was generated
    out, trace = O.beam_search(sd, cfg, f[:2], p[:2], beam_size=k, return_trace=True)
    assert torch.equal(out, case[f"beam{k}_ids"])
    torch.testing.assert_close(trace, case[f"beam{k}_gaps"], rtol=1e-3, atol=1e-9)


@pytest.mark.parametrize("name", ["modelA", "modelB"])
def test_full_width_reference_grads(name):
    """Backward of the oracle against the reference at the benchmarked widths: Frobenius norm, sum and the leading 32
    elements of every parameter gradient."""
    case, cfg, sd, f, p, c = _full_case(name)
    _, grads = O.loss_and_grads(sd, cfg, f, p, c)
    assert set(case["grad_stats"]) <= set(grads)
    for k, (norm, total, head) in case["grad_stats"].items():
        g = grads[k]
        assert abs(float(g.double().norm()) - norm) <= 1e-5 * norm + 1e-12, k
        assert abs(float(g.double().sum()) - total) <= 1e-4 * norm + 1e-9, k
        torch.testing.assert_close(g.reshape(-1)[:32], head, rtol=1e-4, atol=1e-6 * max(norm, 1e-30) + 1e-9,
                                   msg=lambda m, k=k: f"{k}: {m}")


def test_decode_captions():
    vocab = {0: "<NULL>", 1: "<START>", 2: "<END>", 3: "<UNK>", 4: "a", 5: "dog"}
    out = O.decode_captions(np.array([[1, 4, 5, 2, 0, 0], [1, 5, 0, 4, 0, 0]]), vocab)
    assert out == ["a dog .", "dog a"]


def test_synthetic_batch_contract():
    f, p, c = O.synthetic_batch(16, 36, 64, 84, 22, 1000, seed=3)
    pad = O.region_is_pad(p)
    assert not pad[:, 0].any()                      # region 0 = whole image, never padding
    assert torch.equal(p[:, 0, :4], torch.tensor([0., 0., 1., 1.]).expand(16, 4))
    assert (f >= 0).all() and (f[pad] == 0).all()
    assert (c[:, 0] == 1).all() and ((c == 2).sum(1) == 1).all()
    n_valid = (~pad).sum(1)
    assert (n_valid >= 18).all() and (n_valid <= 36).all()
    # padding is trailing
    assert torch.equal(pad, torch.arange(36)[None, :] >= n_valid[:, None])

