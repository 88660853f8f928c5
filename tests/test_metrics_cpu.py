"""Caption metrics without a GPU: the fp64 reference scorer pinned to hand-derived values, ids scored like the strings
decode_captions makes of them, and the argument checks of the device entry points."""
import importlib.util
import os

import numpy as np
import pytest
import torch

import caption_metrics_oracle as M
import icap_loader

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
pkg = icap_loader.load()
N = pkg._native


def _utils():
    spec = importlib.util.spec_from_file_location("icap_core_utils", os.path.join(ROOT, "image-caption_b200", "core", "utils.py"))
    mod = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(mod)
    return mod


REFS = {0: [["a", "b"]], 1: [["c", "d"]]}


def test_hand_derived_values():
    per, corpus, _ = M.score([["a", "b"]], [0], REFS)
    assert per["CIDEr-D"][0] == pytest.approx(5.0, abs=1e-12)
    assert per["CIDEr"][0] == pytest.approx(5.0, abs=1e-12)
    assert [per[f"Bleu_{k}"][0] for k in (1, 2, 3, 4)] == pytest.approx([1.0, 1.0, 0.01, 0.001], rel=1e-6)
    assert per["ROUGE_L"][0] == pytest.approx(1.0)
    per, corpus, _ = M.score([["a", "b", "c"]], [0], REFS)
    assert per["CIDEr-D"][0] == pytest.approx(3.756471, abs=1e-6)
    assert per["CIDEr"][0] == pytest.approx(3.809008, abs=1e-6)
    assert [per[f"Bleu_{k}"][0] for k in (1, 2, 3, 4)] == pytest.approx([0.666667, 0.577350, 6.9336e-6, 4.2729e-6],
                                                                       rel=1e-4)
    assert per["ROUGE_L"][0] == pytest.approx(0.829932, abs=1e-6)
    # one candidate: the corpus values are the sentence values
    assert corpus["Bleu_2"] == pytest.approx(per["Bleu_2"][0]) and corpus["CIDEr-D"] == pytest.approx(3.756471, abs=1e-6)


def test_empty_row_scores_zero():
    rows = np.array([[1, 0, 0, 0], [0, 0, 0, 0]])
    refs = np.array([[1, 5, 6, 2], [1, 7, 2, 0]])
    per, _, counts = M.score_ids(rows, [0, 1], refs, [0, 1])
    for name, v in per.items():
        assert np.all(v == 0.0), name
    assert counts["testlen"] == 0 and counts["guess"] == [0, 0, 0, 0]
    assert M.row_tokens([1, 2, 5]) == [2] and M.row_tokens([0, 1, 2]) == [1, 2]


def test_ids_score_like_decoded_strings():
    """Random rows with <START>, <END>, <NULL> and junk after <END>: scoring the ids equals scoring the strings
    decode_captions makes of them, split on spaces."""
    utils = _utils()
    rng = np.random.default_rng(0)
    vocab = 60
    idx_to_word = {0: "<NULL>", 1: "<START>", 2: "<END>", 3: "<UNK>"}
    idx_to_word.update({i: f"w{i}" for i in range(4, vocab)})

    def rows(n, w):
        x = rng.integers(3, 12, size=(n, w))                       # a small alphabet: shared n-grams
        x[rng.random((n, w)) < 0.1] = 0
        x[:, 0] = np.where(rng.random(n) < 0.8, 1, x[:, 0])
        ends = rng.integers(1, w + 2, size=n)                      # w + 1: no <END>
        for i, e in enumerate(ends):
            if e < w:
                x[i, e] = 2
        x[rng.random((n, w)) < 0.03] = 1                           # <START> as an ordinary word elsewhere
        return x

    n_img = 9
    ref_rows, ref_imgs = rows(30, 14), rng.integers(0, n_img, size=30)
    ref_imgs[:n_img] = np.arange(n_img)
    cand_rows, cand_imgs = rows(20, 12), rng.integers(0, n_img, size=20)
    per_ids, corpus_ids, _ = M.score_ids(cand_rows, cand_imgs, ref_rows, ref_imgs)
    dec = lambda r: [s.split(" ") if s else [] for s in utils.decode_captions(r, idx_to_word)]   # noqa: E731
    refs = {}
    for words, img in zip(dec(ref_rows), ref_imgs):
        refs.setdefault(int(img), []).append(words)
    per_str, corpus_str, _ = M.score(dec(cand_rows), [int(i) for i in cand_imgs], refs)
    for k in per_ids:
        np.testing.assert_allclose(per_ids[k], per_str[k], rtol=0, atol=1e-12, err_msg=k)
    assert corpus_ids == pytest.approx(corpus_str, abs=1e-12)
    assert corpus_ids["CIDEr-D"] > 0 and corpus_ids["Bleu_1"] > 0


def test_reward_is_weighted_cider_d_plus_bleu4():
    t = np.array([[5, 6, 7, 2, 0], [8, 9, 2, 0, 0], [5, 9, 7, 6, 2]])
    s = np.array([[5, 6, 7, 2, 0], [8, 2, 0, 0, 0], [4, 4, 4, 4, 4]])
    per, _, _ = M.score_ids(s, range(3), t, range(3))
    np.testing.assert_allclose(M.reward(t, s, 0.5, 2.0), 0.5 * per["CIDEr-D"] + 2.0 * per["Bleu_4"])
    assert per["CIDEr-D"][0] > per["CIDEr-D"][1] > per["CIDEr-D"][2] == 0.0


def test_argument_checks_without_a_gpu():
    # the C entry points validate before any CUDA call
    with pytest.raises(N.IcapError, match="row width"):
        N.call("icap_caption_cook", None, 0, 4, 129, 129, None, None, None, None, None, None)
    with pytest.raises(N.IcapError, match="candidate width"):
        N.call("icap_caption_score", None, 0, 4, 200, 200, None, 1, None, 10, None, None, None, None, None, None, None,
               None, 16, None, None, 1.0, 1.0, None, None)
    with pytest.raises(N.IcapError, match="null pointer"):
        N.call("icap_caption_df", 4, None, 10, None, None, None, None, 16, None, None)
    # the Python wrappers refuse what the packing cannot represent, and CPU tensors
    from image_caption_b200.metrics import CaptionScorer, CaptionReward, MAX_VOCAB
    refs = np.ones((4, 10), dtype=np.int64)
    with pytest.raises(N.IcapError, match="vocabulary"):
        CaptionScorer(refs, np.arange(4), MAX_VOCAB + 1, "cuda:0")
    with pytest.raises(N.IcapError, match="row"):
        CaptionScorer(np.ones((4, 129), dtype=np.int64), np.arange(4), 1000, "cuda:0")
    with pytest.raises(N.IcapError, match="CUDA"):
        CaptionScorer(refs, np.arange(4), 1000, "cpu")
    with pytest.raises(N.IcapError, match="CUDA"):
        CaptionReward().on_device(torch.ones(4, 10, dtype=torch.long), torch.ones(4, 10, dtype=torch.long))
    with pytest.raises(N.IcapError):
        CaptionReward()(np.full((2, 5), MAX_VOCAB), np.ones((2, 5), dtype=np.int64))
