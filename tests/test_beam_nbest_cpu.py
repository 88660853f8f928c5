"""The beam search that stops at <END>, without a GPU: the CPU restatement (tests/beam_eos_oracle.py) on the three tiny
reference configurations keeps its own contract -- best first by length-normalised score, <NULL> after the end of a
caption, scores equal to the teacher-forced log-likelihood of the tokens -- and Transformer.beam_search_nbest rejects
bad arguments before it needs a device."""
import os

import numpy as np
import pytest
import torch

import icap_loader
from beam_eos_oracle import END, NULL, beam_search_eos, hypothesis_length, normalised, teacher_forced_logprob
from oracle import caption_oracle as O

pkg = icap_loader.load()
GOLD = os.path.join(os.path.dirname(__file__), "golden")
CASES = ["tiny_default", "tiny_cfgpy", "tiny_variants"]


def load_case(name, end_bias):
    g = torch.load(os.path.join(GOLD, name + ".pt"), weights_only=False)
    sd = {k: v.clone() for k, v in g["state_dict"].items()}
    sd["classifer.bias"][END] += end_bias           # captions of varied lengths: some hypotheses end early
    return g, sd, O.OracleConfig(**g["ctor"])


def check_nbest(ids, scores, lens, alpha, cfg, sd, f, p):
    B, n, L = ids.shape
    for b in range(B):
        norm = [normalised(scores[b, i], int(lens[b, i]), alpha) for i in range(n)]
        assert all(norm[i] >= norm[i + 1] for i in range(n - 1)), (b, norm)
        for i in range(n):
            row = ids[b, i]
            assert int(row[0]) == 1
            assert int(lens[b, i]) == hypothesis_length(row)
            stop = [j for j in range(1, L) if int(row[j]) in (END, NULL)]
            if stop:
                assert all(int(x) == NULL for x in row[stop[0] + 1:]), row
    rep = lambda x: x.repeat_interleave(n, dim=0)
    logits = O.logits_forward(sd, cfg, rep(f), rep(p), ids.reshape(B * n, L))
    ll = teacher_forced_logprob(logits, ids.reshape(B * n, L), cfg.pad_idx)
    np.testing.assert_allclose(scores.reshape(-1).double().numpy(), ll, rtol=1e-4, atol=1e-4)


@pytest.mark.parametrize("name", CASES)
@pytest.mark.parametrize("k,n,alpha,end_bias", [(3, 3, 0.0, 3.0), (4, 2, 0.6, 3.0), (5, 5, 1.0, 5.0), (2, 1, 0.6, 0.0)])
def test_oracle_nbest_contract(name, k, n, alpha, end_bias):
    g, sd, cfg = load_case(name, end_bias)
    f, p = g["features"], g["positions"]
    ids, scores, lens, trace = beam_search_eos(sd, cfg, f, p, beam_size=k, n_best=n, length_penalty=alpha,
                                               return_trace=True)
    assert ids.shape == (f.shape[0], n, cfg.max_length) and trace.shape == (f.shape[0], cfg.max_length - 1)
    assert bool((trace >= 0).all())
    check_nbest(ids, scores, lens, alpha, cfg, sd, f, p)


def test_oracle_finishes_hypotheses_and_keeps_their_score():
    """With a strong <END> bias some hypotheses end early; a finished one keeps its score to the last step."""
    g, sd, cfg = load_case("tiny_default", 6.0)
    ids, scores, lens = beam_search_eos(sd, cfg, g["features"], g["positions"], beam_size=4)
    assert int((lens < cfg.max_length - 1).sum()) > 0
    assert bool((ids == END).any())


def test_hypothesis_length_rule():
    assert hypothesis_length([1, 7, 8, 2, 0, 0]) == 3          # up to and including <END>
    assert hypothesis_length([1, 7, 0, 0, 0, 0]) == 1          # before <NULL>
    assert hypothesis_length([1, 0, 0, 0]) == 0
    assert hypothesis_length([1, 7, 8, 9]) == 3                # never finished: every position
    assert hypothesis_length([1, 2, 0]) == 1


def test_beam_search_nbest_argument_errors_without_a_gpu():
    g = torch.load(os.path.join(GOLD, "tiny_default.pt"), weights_only=False)
    m = pkg.Transformer(device=torch.device("cpu"), **g["ctor"])
    f, p = g["features"], g["positions"]
    for kw in (dict(beam_size=0), dict(beam_size=9), dict(beam_size=2.5), dict(beam_size=3, n_best=4),
               dict(beam_size=3, n_best=0), dict(length_penalty=-0.1), dict(length_penalty=float("nan")),
               dict(length_penalty=float("inf"))):
        with pytest.raises(ValueError):
            m.beam_search_nbest(f, p, **kw)
