"""Model-level parity on a B200 (`pytest -m gpu`): the drop-in Transformer (CUDA path through the C ABI)
against (1) the golden vectors produced by the unmodified reference and (2) the CPU oracle on seeded
synthetic inputs.  Tolerances are the north_star's: 1e-4 relative in fp32 mode, 2e-2 in bf16 mode;
greedy / beam ids identical in fp32 mode except at reported near-ties (gap < 1e-5)."""
import os

import numpy as np
import pytest
import torch

import icap_loader
from oracle import caption_oracle as O

pytestmark = pytest.mark.gpu
pkg = icap_loader.load()
GOLD = os.path.join(os.path.dirname(__file__), "golden")
DEV = torch.device("cuda:0")


def rel(a, b):
    a, b = a.double().cpu(), b.double().cpu()
    return float((a - b).abs().max() / (b.abs().max() + 1e-30))


def build(cfg_kwargs, sd, precision):
    m = pkg.Transformer(device=DEV, **cfg_kwargs)
    m.load_state_dict(sd)
    m = m.to(DEV).eval()
    m.set_precision(precision)
    return m


def load_gold(name):
    g = torch.load(os.path.join(GOLD, name + ".pt"), weights_only=False)
    return g


def ids_match_except_near_ties(ids, ref_ids, oracle_gaps, tol=1e-5, what=""):
    """Rows may diverge from the reference only at a decision whose top-k gap -- as computed by the ORACLE, [B, T] --
    is below tol; every such exempted decision is reported (north_star: "each of which is reported").  Returns the
    list of unexcused mismatches."""
    ids, ref_ids = ids.cpu(), ref_ids.cpu()
    bad = []
    for b in range(ids.shape[0]):
        neq = (ids[b] != ref_ids[b]).nonzero()
        if len(neq) == 0:
            continue
        first = int(neq[0]) - 1          # decision index that produced the first differing token
        gap = float(oracle_gaps[b, first]) if oracle_gaps is not None else None
        if gap is None or not gap < tol:
            bad.append((b, first, gap))
        else:
            print(f"near-tie{' ' + what if what else ''}: image {b}, decision {first}: oracle gap {gap:.3e} < {tol:g} "
                  f"-> ids {int(ids[b, first + 1])} (CUDA) vs {int(ref_ids[b, first + 1])} (reference)")
    return bad


def greedy_gaps(sd, kw, f, p):
    """[B, T] top-2 logit gap of every greedy decision, from the ORACLE."""
    return O.generate_caption_vector(sd, O.OracleConfig(**kw), f, p, return_gaps=True)[2]


def beam_gaps(sd, kw, f, p, k, log_domain=False):
    """[B, T] score gap between the k-th and (k+1)-th candidate of every beam step, from the ORACLE."""
    return O.beam_search(sd, O.OracleConfig(**kw), f, p, beam_size=k, log_domain=log_domain, return_trace=True)[1]


# ------------------------------------------------------------------------------------------ golden (reference outputs)
def test_golden_fp32_loss_logits_grads():
    g = load_gold("tiny_default")
    m = build(g["ctor"], g["state_dict"], "fp32")
    lg = m.logits(g["features"], g["positions"], g["captions"])
    assert rel(lg, g["logits"]) < 1e-4
    # eval(): the golden vectors were produced in eval mode (attention dropout 0.1 is hard-wired in train mode)
    loss = m(g["features"], g["positions"], g["captions"])["loss"]
    assert abs(float(loss) - float(g["loss"])) / float(g["loss"]) < 1e-5
    loss.backward()
    worst = 0.0
    for name, q in m.named_parameters():
        ref = g["grads"][name]
        err = float((q.grad.cpu() - ref).abs().max() / (ref.abs().max() + 1e-12))
        worst = max(worst, err)
        assert err < 2e-4, (name, err)
    assert float(m.decoder.word_embedding.weight.grad[0].abs().sum()) == 0.0     # padding_idx row


def test_golden_fp32_adam_two_steps_torch_optimizer_path():
    """The reference wrapper's own loop: zero_grad / forward / backward / torch.optim.Adam.step (models.py:115-126)."""
    g = load_gold("tiny_default")
    m = build(g["ctor"], g["state_dict"], "fp32")
    opt = torch.optim.Adam((p for p in m.parameters() if p.requires_grad), lr=5e-4)
    losses = []
    for f, p, c in ((g["features"], g["positions"], g["captions"]), (g["features2"], g["positions2"], g["captions2"])):
        opt.zero_grad()
        loss = m(f, p, c)["loss"]
        loss.backward()
        opt.step()
        losses.append(float(loss))
    np.testing.assert_allclose(losses, g["adam_losses"].numpy(), rtol=2e-5)
    after = g["state_dict_after_2_steps"]
    for k, v in m.state_dict().items():
        assert torch.allclose(v.cpu(), after[k], rtol=1e-3, atol=2e-5), k


def test_golden_fp32_fused_train_step():
    """Same two steps through the fused path (explicit backward + flat fused Adam)."""
    g = load_gold("tiny_default")
    m = build(g["ctor"], g["state_dict"], "fp32")
    losses = []
    for f, p, c in ((g["features"], g["positions"], g["captions"]), (g["features2"], g["positions2"], g["captions2"])):
        losses.append(float(m.train_step_fused(f, p, c, lr=5e-4, train_mode=False)))
    np.testing.assert_allclose(losses, g["adam_losses"].numpy(), rtol=2e-5)
    after = g["state_dict_after_2_steps"]
    for k, v in m.state_dict().items():
        assert torch.allclose(v.cpu(), after[k], rtol=1e-3, atol=2e-5), k


def test_golden_fp32_greedy_and_beam_ids():
    g = load_gold("tiny_default")
    m = build(g["ctor"], g["state_dict"], "fp32")
    ids, att = m.generate_caption_vector(g["features"], g["positions"])
    assert ids.shape == g["greedy_ids"].shape and ids.dtype == torch.long
    F_, P_ = g["features"], g["positions"]
    assert not ids_match_except_near_ties(ids, g["greedy_ids"], greedy_gaps(g["state_dict"], g["ctor"], F_, P_))
    assert len(att) == g["greedy_attention"].shape[0]
    if torch.equal(ids.cpu(), g["greedy_ids"]):
        np.testing.assert_allclose(np.stack(att, 0), g["greedy_attention"].numpy(), rtol=1e-3, atol=1e-6)
    for k in (2, 3):
        out = m.beam_search(g["features"], g["positions"], beam_size=k)
        assert out.shape == g[f"beam{k}_ids"].shape
        assert not ids_match_except_near_ties(out, g[f"beam{k}_ids"], beam_gaps(g["state_dict"], g["ctor"], F_, P_, k),
                                              tol=1e-6, what=f"beam-{k}")
    m.log_domain_beam = True
    out = m.beam_search(g["features"], g["positions"], beam_size=3)
    assert not ids_match_except_near_ties(out, g["policy_beam3_ids"],
                                          beam_gaps(g["state_dict"], g["ctor"], F_, P_, 3, log_domain=True), tol=1e-5)


def test_golden_bf16_within_tolerance():
    g = load_gold("tiny_default")
    m = build(g["ctor"], g["state_dict"], "bf16")
    lg = m.logits(g["features"], g["positions"], g["captions"])
    assert rel(lg, g["logits"]) < 2e-2
    loss = m(g["features"], g["positions"], g["captions"])["loss"]
    assert abs(float(loss) - float(g["loss"])) / float(g["loss"]) < 2e-2


@pytest.mark.parametrize("name", ["tiny_cfgpy", "tiny_variants"])
def test_golden_variants_fp32(name):
    """config.py-default flavour (encode_mask + split_image_objects, 8 heads of dim 4) and the
    split_position + move_first_image_feature + FocalLoss flavour, against the reference's own outputs."""
    g = load_gold(name)
    m = build(g["ctor"], g["state_dict"], "fp32")
    assert rel(m.logits(g["features"], g["positions"], g["captions"]), g["logits"]) < 1e-4
    loss = m(g["features"], g["positions"], g["captions"])["loss"]
    assert abs(float(loss.detach()) - float(g["loss"])) / float(g["loss"]) < 1e-5
    loss.backward()
    for pname, q in m.named_parameters():
        ref = g["grads"][pname]
        err = float((q.grad.cpu() - ref).norm() / (ref.norm() + 1e-12))
        assert err < 5e-4, (pname, err)
    ids, att = m.generate_caption_vector(g["features"], g["positions"])
    F_, P_ = g["features"], g["positions"]
    assert not ids_match_except_near_ties(ids, g["greedy_ids"], greedy_gaps(g["state_dict"], g["ctor"], F_, P_))
    for k in (2, 3):
        out = m.beam_search(g["features"], g["positions"], beam_size=k)
        assert not ids_match_except_near_ties(out, g[f"beam{k}_ids"], beam_gaps(g["state_dict"], g["ctor"], F_, P_, k),
                                              tol=1e-6, what=f"beam-{k}")
    # fused train steps (explicit backward + flat Adam, focal factor folded into Adam's gradient scale)
    m2 = build(g["ctor"], g["state_dict"], "fp32")
    losses = [float(m2.train_step_fused(f, p, c, lr=5e-4, train_mode=False))
              for f, p, c in ((g["features"], g["positions"], g["captions"]),
                              (g["features2"], g["positions2"], g["captions2"]))]
    np.testing.assert_allclose(losses, g["adam_losses"].numpy(), rtol=2e-5)
    for k, v in m2.state_dict().items():
        assert torch.allclose(v.cpu(), g["state_dict_after_2_steps"][k], rtol=1e-3, atol=2e-5), k


def test_config1_shapes_bf16_and_fp32_vs_oracle():
    """BASELINE configs[0]: core/config.py defaults (d256, 32 heads of dim 8, FFN 256, 2+5 blocks, encode_mask,
    split_image_objects, max_length 51), batch 8 of 36x2048 regions, greedy decode."""
    kw = dict(num_vocab=10000, max_length=51, encode_dim_positions=84, encode_dim_features=2048, output_name="x",
              dropout=0.0, encode_mask=True, split_image_objects=True, encode_input_size=256, encode_q_k_dim=256,
              encode_v_dim=256, encode_hidden_size=256, encode_num_blocks=2, encode_num_heads=32, dim_word_embedding=256,
              decode_input_size=256, decode_q_k_dim=256, decode_v_dim=256, decode_hidden_size=256, decode_num_blocks=5,
              decode_num_heads=32)
    cfg = O.OracleConfig(**kw)
    sd = O.init_state_dict(cfg, seed=0)
    f, p, c = O.synthetic_batch(8, 36, 2048, 84, 51, 10000, seed=1234)
    ref_logits = O.logits_forward(sd, cfg, f, p, c)
    m = build(kw, sd, "fp32")
    assert rel(m.logits(f, p, c), ref_logits) < 1e-4
    ref_ids, _, ref_gaps = O.generate_caption_vector(sd, cfg, f, p, return_gaps=True)
    ids, att = m.generate_caption_vector(f, p)
    assert ids.shape == (8, 52) and len(att) == 50 and att[0].shape == (8, 36)
    assert not ids_match_except_near_ties(ids, ref_ids, ref_gaps)
    mb = build(kw, sd, "bf16")
    assert rel(mb.logits(f, p, c), ref_logits) < 2e-2


@pytest.mark.parametrize("name", ["modelA", "modelB"])
def test_full_width_reference_golden(name):
    """The CUDA path against outputs of the UNMODIFIED reference at the benchmarked widths (tests/golden/full_width.pt,
    made by tests/golden/make_golden_full.py): model A = ctor defaults (BASELINE configs[1-3]), model B = core/config.py
    defaults (configs[0]); vocab 10k, 36 x 2048 regions.  fp32 mode: logits / loss within 1e-4, greedy and beam ids
    identical except at reported near-ties; bf16 mode: logits / loss within 2e-2."""
    import sys
    sys.path.insert(0, GOLD)
    try:
        import make_golden_full as G
    finally:
        sys.path.remove(GOLD)
    case = torch.load(os.path.join(GOLD, "full_width.pt"), weights_only=False)[name]
    cfg, sd, f, p, c, sha = G.regenerate(name)
    if sha != case["sha256"]:
        pytest.skip("this torch build draws a different CPU random stream than the one the golden was made with")
    kw = case["ctor"]
    for precision, tol in (("fp32", 1e-4), ("bf16", 2e-2)):
        m = build(kw, sd, precision)
        lg = m.logits(f, p, c)
        assert rel(lg[:, :, :64], case["logits_slice"]) < tol, precision
        assert rel(lg.max(dim=-1).values, case["logits_row_max"]) < tol, precision
        with torch.no_grad():
            loss = float(m(f, p, c)["loss"])
        assert abs(loss - float(case["loss"])) / float(case["loss"]) < tol, (precision, loss)
        if precision == "fp32":
            ids, att = m.generate_caption_vector(f, p)
            assert ids.shape == case["greedy_ids"].shape and len(att) == cfg.max_length - 1
            assert not ids_match_except_near_ties(ids, case["greedy_ids"], case["greedy_gaps"], what=name + " greedy")
            for k in ((3, 5) if name == "modelA" else (3,)):
                out = m.beam_search(f[:2], p[:2], beam_size=k)
                assert not ids_match_except_near_ties(out, case[f"beam{k}_ids"], case[f"beam{k}_gaps"], tol=1e-6,
                                                      what=f"{name} beam-{k}")


# ------------------------------------------------------------------------------------------ oracle, model A shapes
def model_a_cfg(**over):
    kw = dict(num_vocab=10000, max_length=22, encode_dim_positions=84, encode_dim_features=2048, output_name="x",
              dropout=0.0)
    kw.update(over)
    return kw


@pytest.mark.parametrize("precision,tol_logits,tol_loss", [("fp32", 1e-4, 1e-5), ("bf16", 2e-2, 2e-2)])
def test_model_a_vs_oracle(precision, tol_logits, tol_loss):
    kw = model_a_cfg()
    cfg = O.OracleConfig(**kw)
    sd = O.init_state_dict(cfg, seed=0)
    f, p, c = O.synthetic_batch(6, 36, 2048, 84, 22, 10000, seed=1234)
    ref_logits = O.logits_forward(sd, cfg, f, p, c)
    ref_loss, ref_grads = O.loss_and_grads(sd, cfg, f, p, c)
    m = build(kw, sd, precision)
    lg = m.logits(f, p, c)
    assert rel(lg, ref_logits) < tol_logits
    loss = m(f, p, c)["loss"]
    assert abs(float(loss) - float(ref_loss)) / float(ref_loss) < tol_loss
    loss.backward()
    assert_grads_match(m, ref_grads, precision)


def assert_grads_match(m, ref_grads, precision):
    # Gradients: Frobenius-relative error per parameter.  (A max-abs criterion is not robust here: a ReLU
    # pre-activation within rounding distance of 0 flips its mask bit and moves one row of dW1 by ~1e-3 of
    # max|dW1| -- observed, and inherent to any re-ordered fp32 summation.)  bf16 mode: activations AND
    # activation-gradients are rounded to bf16 through 12 layers; ~5% is what that gives.
    ftol, mtol = (5e-4, 5e-3) if precision == "fp32" else (0.15, 0.35)
    for name, q in m.named_parameters():
        r = ref_grads[name]
        g = q.grad.cpu()
        assert float((g - r).norm() / (r.norm() + 1e-12)) < ftol, name
        assert float((g - r).abs().max() / (r.abs().max() + 1e-12)) < mtol, name
        if float(r.norm()) > 0:
            # direction and scale separately: a wrong constant factor on a small tensor cannot hide in the Frobenius bound
            cos = float((g.double() * r.double()).sum() / (g.double().norm() * r.double().norm() + 1e-30))
            ratio = float(g.norm() / r.norm())
            assert cos > (0.999999 if precision == "fp32" else 0.985), (name, cos)
            assert abs(ratio - 1.0) < (1e-3 if precision == "fp32" else 0.06), (name, ratio)


def test_model_a_encode_mask_vs_oracle():
    kw = model_a_cfg(encode_mask=True, encode_num_blocks=2, decode_num_blocks=2)
    cfg = O.OracleConfig(**kw)
    sd = O.init_state_dict(cfg, seed=3)
    f, p, c = O.synthetic_batch(5, 36, 2048, 84, 22, 10000, seed=7)
    m = build(kw, sd, "fp32")
    assert rel(m.logits(f, p, c), O.logits_forward(sd, cfg, f, p, c)) < 1e-4


def test_model_a_decode_vs_oracle_fp32():
    kw = model_a_cfg(encode_num_blocks=2, decode_num_blocks=2, max_length=12)
    cfg = O.OracleConfig(**kw)
    sd = O.init_state_dict(cfg, seed=1)
    f, p, _ = O.synthetic_batch(6, 36, 2048, 84, 12, 10000, seed=5)
    m = build(kw, sd, "fp32")
    ref_ids, ref_att, ref_gaps = O.generate_caption_vector(sd, cfg, f, p, return_gaps=True)
    ids, att = m.generate_caption_vector(f, p)
    assert not ids_match_except_near_ties(ids, ref_ids, ref_gaps)
    if torch.equal(ids.cpu(), ref_ids):
        np.testing.assert_allclose(np.stack(att, 0), np.stack(ref_att, 0), rtol=1e-3, atol=1e-6)
        assert rel(m.last_gaps.t(), ref_gaps) < 1e-2
    for k in (3, 5):
        ref, ref_trace = O.beam_search(sd, cfg, f, p, beam_size=k, return_trace=True)
        out = m.beam_search(f, p, beam_size=k)
        assert not ids_match_except_near_ties(out, ref, ref_trace, tol=1e-6, what="beam")


def test_decode_with_generated_pad_tokens():
    """A generated token id 0 is treated as padding in later steps (SURVEY.md §8a): force it via the bias."""
    kw = model_a_cfg(encode_num_blocks=1, decode_num_blocks=2, max_length=8, num_vocab=400, encode_dim_features=64)
    cfg = O.OracleConfig(**kw)
    sd = O.init_state_dict(cfg, seed=2)
    sd["classifer.bias"][0] = 2.0           # makes <NULL> win some, not all, decisions
    f, p, _ = O.synthetic_batch(16, 9, 64, 84, 8, 400, seed=11)
    ref_ids, _, ref_gaps = O.generate_caption_vector(sd, cfg, f, p, return_gaps=True)
    assert (ref_ids[:, 1:-1] == 0).any() and (ref_ids[:, 1:-1] != 0).any()
    m = build(kw, sd, "fp32")
    ids, _ = m.generate_caption_vector(f, p)
    assert not ids_match_except_near_ties(ids, ref_ids, ref_gaps)
    ref, ref_trace = O.beam_search(sd, cfg, f, p, beam_size=3, return_trace=True)
    out = m.beam_search(f, p, beam_size=3)
    assert not ids_match_except_near_ties(out, ref, ref_trace, tol=1e-6, what="beam")


@pytest.mark.parametrize("B,R", [(1, 37), (3, 37), (2, 5)])
def test_odd_shapes_vs_oracle(B, R):
    """Real data has R = NUM_OBJECT + 1 = 37 regions (features.py:101) and the demo path runs batch 1: loss,
    logits, gradients (fp32) and decode ids against the oracle at those shapes; bf16 within tolerance."""
    kw = model_a_cfg(encode_num_blocks=2, decode_num_blocks=2, max_length=10, num_vocab=777)
    cfg = O.OracleConfig(**kw)
    sd = O.init_state_dict(cfg, seed=5)
    f, p, c = O.synthetic_batch(B, R, 2048, 84, 10, 777, seed=31 + B + R)
    ref_logits = O.logits_forward(sd, cfg, f, p, c)
    ref_loss, ref_grads = O.loss_and_grads(sd, cfg, f, p, c)
    m = build(kw, sd, "fp32")
    assert rel(m.logits(f, p, c), ref_logits) < 1e-4
    loss = m(f, p, c)["loss"]
    assert abs(float(loss) - float(ref_loss)) / float(ref_loss) < 1e-5
    loss.backward()
    for name, q in m.named_parameters():
        r = ref_grads[name]
        # tiny batches: one ReLU pre-activation within rounding distance of 0 moves a whole gradient row (see
        # test_model_a_vs_oracle), so the Frobenius bound is looser than at batch 6
        assert float((q.grad.cpu() - r).norm() / (r.norm() + 1e-12)) < 5e-3, name
    ref_ids, _, ref_gaps = O.generate_caption_vector(sd, cfg, f, p, return_gaps=True)
    ids, att = m.generate_caption_vector(f, p)
    assert att[0].shape == (B, R)
    assert not ids_match_except_near_ties(ids, ref_ids, ref_gaps)
    ref, ref_trace = O.beam_search(sd, cfg, f, p, beam_size=3, return_trace=True)
    out = m.beam_search(f, p, beam_size=3)
    assert not ids_match_except_near_ties(out, ref, ref_trace, tol=1e-6, what="beam")
    mb = build(kw, sd, "bf16")
    assert rel(mb.logits(f, p, c), ref_logits) < 2e-2
    assert mb.beam_search(f, p, beam_size=3).shape == ref.shape


def test_config5_scaled_shapes_vs_oracle():
    """BASELINE configs[4] shapes (scaled variant): d_model 1024, 16 heads, FFN 4096, 100 regions, vocab 30k (2+2
    blocks here so the CPU oracle finishes in seconds): logits fp32 / bf16, beam-5 ids in fp32, loss and every
    parameter gradient in both precisions (the vocabulary-30000 cross-entropy and bias-gradient kernels)."""
    kw = dict(num_vocab=30000, max_length=22, encode_dim_positions=84, encode_dim_features=2048, output_name="x",
              dropout=0.0, encode_input_size=1024, encode_q_k_dim=1024, encode_v_dim=1024, encode_hidden_size=4096,
              encode_num_blocks=2, encode_num_heads=16, dim_word_embedding=1024, decode_input_size=1024,
              decode_q_k_dim=1024, decode_v_dim=1024, decode_hidden_size=4096, decode_num_blocks=2, decode_num_heads=16)
    cfg = O.OracleConfig(**kw)
    sd = O.init_state_dict(cfg, seed=0)
    f, p, c = O.synthetic_batch(3, 100, 2048, 84, 22, 30000, seed=99)
    ref_logits = O.logits_forward(sd, cfg, f, p, c)
    m = build(kw, sd, "fp32")
    assert rel(m.logits(f, p, c), ref_logits) < 1e-4
    ref, ref_trace = O.beam_search(sd, cfg, f, p, beam_size=5, return_trace=True)
    out = m.beam_search(f, p, beam_size=5)
    assert out.shape == ref.shape
    assert not ids_match_except_near_ties(out, ref, ref_trace, tol=1e-6, what="beam-5")
    ref_loss, ref_grads = O.loss_and_grads(sd, cfg, f, p, c)
    loss = m(f, p, c)["loss"]
    assert abs(float(loss) - float(ref_loss)) / float(ref_loss) < 1e-5
    loss.backward()
    assert_grads_match(m, ref_grads, "fp32")
    mb = build(kw, sd, "bf16")
    assert rel(mb.logits(f, p, c), ref_logits) < 2e-2
    loss = mb(f, p, c)["loss"]
    assert abs(float(loss) - float(ref_loss)) / float(ref_loss) < 2e-2
    loss.backward()
    assert_grads_match(mb, ref_grads, "bf16")


def test_full_size_decode_properties_bf16(monkeypatch):
    """Config 3 shapes (512 images, beam 5 and greedy, model A, bf16): size-independent properties --
    ids in range, <START> first, whole-graph decode == eager decode, and image independence (decoding a slice
    of the batch alone gives the same ids as inside the full batch: the path shards by image)."""
    kw = model_a_cfg()
    torch.manual_seed(0)
    m = pkg.Transformer(device=DEV, **kw).to(DEV).eval()
    f, p, _ = O.synthetic_batch(512, 36, 2048, 84, 22, 10000, seed=4321)
    f, p = f.to(DEV), p.to(DEV)
    for k in (5, 1):
        ids = m.beam_search(f, p, beam_size=k) if k > 1 else m.generate_caption_vector(f, p)[0][:, :22]
        assert ids.shape == (512, 22) and ids.dtype == torch.long
        assert bool((ids[:, 0] == 1).all()) and int(ids.min()) >= 0 and int(ids.max()) < 10000
        monkeypatch.setenv("ICAP_DECODE_GRAPH", "0")
        eager = m.beam_search(f, p, beam_size=k) if k > 1 else m.generate_caption_vector(f, p)[0][:, :22]
        assert torch.equal(ids, eager)
        # the step start as three launches (beam reorder, embedding, LayerNorm) instead of icap_decode_embed_ln
        monkeypatch.setenv("ICAP_DECODE_FUSED_START", "0")
        unfused = m.beam_search(f, p, beam_size=k) if k > 1 else m.generate_caption_vector(f, p)[0][:, :22]
        monkeypatch.delenv("ICAP_DECODE_FUSED_START")
        monkeypatch.delenv("ICAP_DECODE_GRAPH")
        assert torch.equal(ids, unfused)
        part = m.beam_search(f[128:256], p[128:256], beam_size=k) if k > 1 else \
            m.generate_caption_vector(f[128:256], p[128:256])[0][:, :22]
        same = (part == ids[128:256]).all(dim=1).float().mean()
        assert float(same) > 0.97, float(same)       # bf16 GEMM tiles differ with M: allow rare near-tie flips


# ------------------------------------------------------------------------------------------ full-size properties
def test_full_size_train_step_properties_bf16():
    """Config 2 shapes (B=256, R=36, T=21, V=10k): loss ~ ln(V) at init, decreases under Adam, stays finite;
    graph replay == eager."""
    kw = model_a_cfg(dropout=0.2)
    torch.manual_seed(0)
    m = pkg.Transformer(device=DEV, **kw).to(DEV).train()
    f, p, c = O.synthetic_batch(256, 36, 2048, 84, 22, 10000, seed=1)
    f, p, c = f.to(DEV), p.to(DEV), c.to(DEV)
    losses = [float(m.train_step_fused(f, p, c, lr=5e-4)) for _ in range(6)]
    assert abs(losses[0] - np.log(10000)) < 0.6
    assert all(np.isfinite(losses)) and losses[-1] < losses[0]
    gs = pkg.GraphedTrainStep(m, 256, 36, 22, lr=5e-4)
    gs.load(f, p, c)
    l0 = float(gs.step())
    l1 = float(gs.step())
    assert np.isfinite(l0) and np.isfinite(l1) and l1 < losses[0]
    assert gs.launches_per_step > 100


def test_policy_network_logits_and_external_loss_gradients():
    """SURVEY.md 8(f)#1: PolicyNetwork.forward returns differentiable logits (model_RL.py:75-90).  A PyTorch
    cross-entropy on top of them must reproduce the oracle's loss and every parameter gradient (fp32 mode), and the
    log-domain beam search must match the oracle's PolicyNetwork beam."""
    kw = model_a_cfg(encode_num_blocks=2, decode_num_blocks=2, max_length=12, num_vocab=1000)
    cfg = O.OracleConfig(**kw)
    sd = O.init_state_dict(cfg, seed=4)
    f, p, c = O.synthetic_batch(5, 36, 2048, 84, 12, 1000, seed=8)
    pk = {k: v for k, v in kw.items() if k != "output_name"}
    m = pkg.PolicyNetwork(device=DEV, **pk)
    m.load_state_dict(sd)
    m = m.to(DEV).eval()
    m.set_precision("fp32")
    logits = m(f, p, c)
    assert logits.shape == (5, 11, 1000) and logits.requires_grad
    assert rel(logits.detach(), O.logits_forward(sd, cfg, f, p, c)) < 1e-4
    tgt = c[:, 1:].long().to(DEV)
    loss = torch.nn.functional.cross_entropy(logits.reshape(-1, 1000), tgt.reshape(-1), ignore_index=0)
    ref_loss, ref_grads = O.loss_and_grads(sd, cfg, f, p, c)
    assert abs(float(loss) - float(ref_loss)) / float(ref_loss) < 1e-5
    loss.backward()
    for name, q in m.named_parameters():
        r = ref_grads[name]
        assert float((q.grad.cpu() - r).norm() / (r.norm() + 1e-12)) < 5e-4, name
    seq, logp = m.sample(logits.detach())
    assert seq.shape == (5, 11) and logp.shape == (5, 11, 1000)
    # sample = log_softmax + arg-max on the CUDA path (model_RL.py:93-97), differentiable in the log-probabilities
    x = logits.detach().clone().requires_grad_(True)
    seq2, logp2 = m.sample(x)
    ref_lp = torch.log_softmax(x.detach().double(), dim=2)
    assert torch.equal(seq2.cpu(), ref_lp.argmax(2).cpu()) and seq2.dtype == torch.long
    assert rel(logp2.detach(), ref_lp) < 1e-6
    w = torch.randn_like(logp2)
    (logp2 * w).sum().backward()
    xr = x.detach().double().requires_grad_(True)
    (torch.log_softmax(xr, dim=2) * w.double()).sum().backward()
    assert rel(x.grad, xr.grad) < 1e-5
    ref, ref_trace = O.beam_search(sd, cfg, f, p, beam_size=3, log_domain=True, return_trace=True)
    out = m.beam_search(f, p, beam_size=3)
    assert not ids_match_except_near_ties(out, ref, ref_trace, tol=1e-6, what="beam")


def test_train_step_fused_auto_graph_equals_eager(monkeypatch):
    """The drop-in wrapper's train_step (core/models.py:115-126 -> train_step_fused) replays one CUDA graph per batch
    shape.  Same losses and weights as the eager launch sequence -- including when a NEW shape is captured in the
    middle of a run (the capture's warm-up steps must not leak into the weights or the Adam moments)."""
    kw = model_a_cfg(encode_num_blocks=1, decode_num_blocks=1, num_vocab=500, encode_dim_features=256)
    sd = O.init_state_dict(O.OracleConfig(**kw), seed=0)
    batches = [O.synthetic_batch(16, 12, 256, 84, 22, 500, seed=20),
               O.synthetic_batch(16, 12, 256, 84, 22, 500, seed=21),
               O.synthetic_batch(9, 12, 256, 84, 22, 500, seed=22),          # new batch size: second capture, mid-run
               O.synthetic_batch(16, 12, 256, 84, 22, 500, seed=23),          # back to the first graph
               O.synthetic_batch(9, 7, 256, 84, 22, 500, seed=24)]            # third capture (regions differ)
    out = {}
    for graph in ("0", "1"):
        monkeypatch.setenv("ICAP_TRAIN_GRAPH", graph)
        m = build(kw, sd, "fp32").train()
        losses = [float(m.train_step_fused(f, p, c, lr=5e-4, train_mode=False)) for f, p, c in batches]
        out[graph] = (losses, {n: q.detach().clone() for n, q in m.state_dict().items()}, m.optimizer_state_dict())
        assert len(m._train_graphs) == (3 if graph == "1" else 0)
    # the two trajectories of the note below differ by up to 9e-6 in the loss of step 5 (profiles/r2_fp32_bimodal_trajectory.log);
    # a leaked warm-up step (one extra Adam update at lr 5e-4) moves the next losses by ~1e-2
    for a, b in zip(out["0"][0], out["1"][0]):
        assert abs(a - b) <= 1e-4 * abs(a), (out["0"][0], out["1"][0])
    # Whole tensors in norm: Adam's first steps move every weight by ~lr * sign(g), so an element whose gradient is at
    # the rounding-noise level of the fp32 atomics (embedding scatter-add, column sums) may flip between two runs.
    # A leaked warm-up step would move EVERY element by ~lr: ~2e-2 of the norm.
    for n, q in out["0"][1].items():
        if q.is_floating_point() and q.dim() >= 2:
            assert float((q - out["1"][1][n]).norm()) <= 1e-3 * float(q.norm()), n
    assert out["0"][2]["step"] == out["1"][2]["step"] == len(batches)
    # The trajectory itself is bimodal at the 4e-3 level, eagerly AND through graphs (tools/graph_eager_repro.py): the
    # fp32 atomics of the split-K weight gradients round differently from run to run, the weights after step 1 then
    # differ by <= 6e-8, and ONE ReLU pre-activation of batch 2 sits within that distance of zero -- its mask bit flips
    # and moves every gradient by ~1e-4.  A leaked warm-up step (what this test is about) adds a whole extra gradient
    # to the moments: ~0.1-1 of their norm.
    ma, mb = out["0"][2]["exp_avg"], out["1"][2]["exp_avg"]
    assert float((ma - mb).norm()) <= 2e-2 * float(ma.norm())
    va, vb = out["0"][2]["exp_avg_sq"], out["1"][2]["exp_avg_sq"]
    assert float((va - vb).norm()) <= 2e-2 * float(va.norm())


def test_model_a_bf16_batch256_vs_oracle():
    """The BENCHMARKED configuration (BASELINE configs[1]: model A, batch 256, bf16) against the CPU oracle: logits and
    loss within the north_star's 2e-2 (dropout off on both sides: the oracle has no RNG stream to share)."""
    kw = model_a_cfg()
    cfg = O.OracleConfig(**kw)
    sd = O.init_state_dict(cfg, seed=0)
    f, p, c = O.synthetic_batch(256, 36, 2048, 84, 22, 10000, seed=1234)
    with torch.no_grad():
        ref_logits = O.logits_forward(sd, cfg, f, p, c)
        ref_loss = O.loss_from_logits(cfg, ref_logits, c)
    m = build(kw, sd, "bf16")
    lg = m.logits(f, p, c)
    assert lg.shape == ref_logits.shape
    assert rel(lg, ref_logits) < 2e-2
    loss = m(f, p, c)["loss"]
    assert abs(float(loss) - float(ref_loss)) / float(ref_loss) < 2e-2
    # fused graph step on the same batch (eval-mode arithmetic): its reported loss is the same number
    l2 = float(m.train_step_fused(f, p, c, lr=5e-4, train_mode=False))
    assert abs(l2 - float(ref_loss)) / float(ref_loss) < 2e-2


@pytest.mark.parametrize("variant", ["default", "split_image_objects", "split_position_move_first"])
@pytest.mark.parametrize("precision", ["fp32", "bf16"])
def test_dp_bucket_slices_are_final_when_fired(variant, precision):
    """Data-parallel bucket schedule against the REAL backward tape (ADVICE r1: with split_image_objects the
    image_encoder closures reported offsets below tensors that complete later).  A one-element bucket size makes every
    closure fire; each fired slice [lo, hi) of the flat gradient buffer is snapshotted exactly as DataParallel._fire
    would hand it to NCCL (after the main and the wgrad side stream) and must equal the final gradient."""
    over = dict(encode_num_blocks=2, decode_num_blocks=2, num_vocab=500, encode_dim_features=256)
    if variant == "split_image_objects":
        over.update(split_image_objects=True, encode_mask=True)
    elif variant == "split_position_move_first":
        over.update(split_position=True, move_first_image_feature=True)
    kw = model_a_cfg(**over)
    torch.manual_seed(0)
    m = pkg.Transformer(device=DEV, **kw).to(DEV).train()
    m.set_precision(precision)
    eng = m._engine()
    eng.dp_unnormalized = True
    f, p, c = O.synthetic_batch(8, 12, 256, 84, 22, 500, seed=3)
    f, p, c = f.to(DEV), p.to(DEV), c.to(DEV)
    plan = pkg.GradBuckets(eng.g32.numel(), 1)
    comm = torch.cuda.Stream(device=DEV)
    fired = []

    def fire(sl):
        if sl is None:
            return
        comm.wait_stream(torch.cuda.current_stream(DEV))
        if eng._bwd_side is not None:
            comm.wait_stream(eng._bwd_side)
        with torch.cuda.stream(comm):
            fired.append((sl, eng.g32[sl[0]:sl[1]].clone()))

    eng.bucket_hook = lambda lo: fire(plan.on_done(lo))
    eng.forward_backward(f, p, c, train_mode=False)
    eng.bucket_hook = None
    fire(plan.flush())
    torch.cuda.synchronize()
    assert len(fired) > 4 and sum(b - a for (a, b), _ in fired) == eng.g32.numel()
    names = {off: n for n, off in eng.offsets.items()}
    for (a, b), snap in fired:
        final = eng.g32[a:b]
        if not torch.equal(snap, final):
            idx = int((snap != final).nonzero()[0]) + a
            owner = max(o for o in names if o <= idx)
            raise AssertionError(f"slice [{a}, {b}) was fired before it was final: element {idx} ({names[owner]})")


def test_checkpoint_and_optimizer_resume(tmp_path):
    """state_dict round trip in the reference's format + optimizer-state resume: (2 steps, save, 1 step) ==
    (load into a fresh model, 1 step)."""
    kw = model_a_cfg(encode_num_blocks=1, decode_num_blocks=1, num_vocab=500, encode_dim_features=256)
    f, p, c = O.synthetic_batch(16, 12, 256, 84, 22, 500, seed=6)
    torch.manual_seed(0)
    a = pkg.Transformer(device=DEV, **kw).to(DEV).train()
    a.set_precision("fp32")
    for _ in range(2):
        a.train_step_fused(f, p, c, lr=5e-4, train_mode=False)
    torch.save(a.state_dict(), tmp_path / "model_2.pt")
    torch.save(a.optimizer_state_dict(), tmp_path / "opt_2.pt")
    a.train_step_fused(f, p, c, lr=5e-4, train_mode=False)
    b = pkg.Transformer(device=DEV, **kw).to(DEV).train()
    b.set_precision("fp32")
    sd = torch.load(tmp_path / "model_2.pt")
    assert list(sd.keys()) == list(O.init_state_dict(O.OracleConfig(**kw), seed=0).keys())      # reference key order
    b.load_state_dict(sd)
    b.load_optimizer_state_dict(torch.load(tmp_path / "opt_2.pt"))
    b.train_step_fused(f, p, c, lr=5e-4, train_mode=False)
    for (n1, q1), (n2, q2) in zip(a.state_dict().items(), b.state_dict().items()):
        assert n1 == n2 and torch.allclose(q1, q2, rtol=1e-5, atol=1e-6), n1


def test_missing_library_fails_loudly(monkeypatch):
    N = pkg._native
    monkeypatch.setattr(N, "_lib", None)
    monkeypatch.setattr(N, "LIB_PATH", "/nonexistent/libicap.so")
    with pytest.raises(N.IcapError):
        N.lib()


@pytest.mark.parametrize("mode", ["train_fp32", "eval_fp32", "eval_bf16", "train_bf16"])
def test_resnet_extractor_vs_torchvision(mode):
    """SURVEY.md 8f #4: the ResNet-101 region feature extractor (core/preprocess.py:26-62) on libicap -- every
    convolution one icap_gemm over an NHWC (patch) matrix, BatchNorm / ReLU / residual / pooling kernels of conv.cu --
    against torchvision's resnet101 children[:9] with the same random-init weights on the CPU.  The reference never
    calls .eval() on its extractor, so the default is batch-statistics BatchNorm ("train"); eval uses running statistics
    (non-trivial ones here).  fp32 mode: 2e-3 of the feature scale.  bf16 mode (tcgen05 GEMMs, bf16 activations through
    101 layers): 3e-2 with running statistics; with batch statistics of only 3 crops a random-init trunk is
    ill-conditioned -- torch's OWN bf16 execution of the same module differs from its fp32 one by 0.31 of the feature
    scale (cosine 0.988; calibrated on the CPU) -- so that case checks the direction (cosine > 0.97) and a loose bound."""
    import sys
    tv = pytest.importorskip("torchvision")
    pkg_dir = os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "image-caption_b200")
    sys.path.insert(0, pkg_dir)
    try:
        from core.preprocess import ResnetExtractor
        torch.manual_seed(0)
        ref = torch.nn.Sequential(*list(tv.models.resnet101(weights=None).children())[:9])
        g = torch.Generator().manual_seed(1)
        for m_ in ref.modules():                      # non-trivial affine / running statistics
            if isinstance(m_, torch.nn.BatchNorm2d):
                m_.weight.data.uniform_(0.5, 1.5, generator=g)
                m_.bias.data.uniform_(-0.2, 0.2, generator=g)
                m_.running_mean.uniform_(-0.1, 0.1, generator=g)
                m_.running_var.uniform_(0.5, 1.5, generator=g)
        ext = ResnetExtractor()
        ext.submodule.load_state_dict(ref.state_dict())
        ext.precision = "bf16" if mode.endswith("bf16") else "fp32"
        x = torch.randn(3, 3, 224, 224, generator=g)
        train = mode.startswith("train")
        ref.train(train)
        ext.train(train)
        with torch.no_grad():
            want = ref(x).flatten(1)
        got = torch.from_numpy(ext(x))
        assert got.shape == (3, 2048)
        err = float((got - want).abs().max() / want.abs().max())
        print(f"resnet101 trunk [{mode}]: max abs err / max |feature| = {err:.2e}, {ext.launches} launches")
        cos = float(torch.nn.functional.cosine_similarity(got.flatten().double(), want.flatten().double(), dim=0))
        if mode == "train_bf16":
            assert cos > 0.97 and err < 0.6, (cos, err)
        else:
            assert err < (3e-2 if mode.endswith("bf16") else 2e-3), err
        if train and mode != "train_bf16":            # running statistics were updated like nn.BatchNorm2d does
            sd_o, sd_r = ext.submodule.state_dict(), ref.state_dict()
            for k in ("1.running_mean", "1.running_var", "7.2.bn3.running_var"):
                assert torch.allclose(sd_o[k].cpu(), sd_r[k], rtol=5e-2 if mode.endswith("bf16") else 2e-3, atol=1e-3), k
            assert int(sd_o["1.num_batches_tracked"]) == 1
    finally:
        sys.path.remove(pkg_dir)
        for m_ in [k for k in sys.modules if k == "core" or k.startswith("core.")]:
            sys.modules.pop(m_)
