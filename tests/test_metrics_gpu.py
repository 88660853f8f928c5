"""Caption metrics on the GPU against the fp64 reference scorer: CaptionScorer, CaptionReward, the device reward inside
the self-critical loss, and the scores main.py train / evaluation print and write."""
import os
import pickle
import sys

import numpy as np
import pytest
import torch

import caption_metrics_oracle as M
import icap_loader

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
PKG = os.path.join(ROOT, "image-caption_b200")
pkg = icap_loader.load()
DEV = torch.device("cuda:0")
NAMES = ("CIDEr-D", "CIDEr", "ROUGE_L", "Bleu_1", "Bleu_2", "Bleu_3", "Bleu_4")


def _zipf_ids(rng, shape, vocab):
    ids = 3 + rng.zipf(1.3, size=shape) % (vocab - 3)
    hi = rng.random(shape) < 0.05                          # some ids at the top of the vocabulary
    ids[hi] = vocab - 1 - rng.integers(0, 4, size=int(hi.sum()))
    return ids


def _rows(rng, n, width, vocab):
    x = _zipf_ids(rng, (n, width), vocab)
    x[:, 0] = 1
    lens = rng.integers(0, width, size=n)
    for i, l in enumerate(lens):
        if 1 + l < width:
            x[i, 1 + l] = 2
            x[i, 2 + l:] = rng.choice([0, 0, 5], size=width - 2 - l)     # padding and junk after <END>
    kinds = rng.integers(0, 12, size=n)
    x[kinds == 0, 1:] = 0                                  # empty row
    x[kinds == 1, 1] = 2                                   # only <END>
    rep = np.flatnonzero(kinds == 2)                       # repeated n-grams
    x[rep, 1:] = np.tile([7, 8], width)[:width - 1]
    x[rng.random((n, width)) < 0.02] = 0                   # <NULL> inside the caption
    return x


def _split(seed, vocab, width, n_img=40):
    rng = np.random.default_rng(seed)
    per = rng.integers(1, 8, size=n_img)
    ref_imgs = np.repeat(np.arange(n_img), per)
    refs = _rows(rng, len(ref_imgs), width, vocab)
    dup = np.flatnonzero(per >= 2)
    starts = np.concatenate([[0], np.cumsum(per)[:-1]])
    refs[starts[dup] + 1] = refs[starts[dup]]              # duplicate references
    perm = rng.permutation(len(ref_imgs))                  # references in any order
    refs, ref_imgs = refs[perm], ref_imgs[perm]
    cand_imgs = rng.integers(0, n_img, size=3 * n_img)
    cands = _rows(rng, len(cand_imgs), width, vocab)
    copy = rng.random(len(cand_imgs)) < 0.3                # some candidates equal one of their references
    for i in np.flatnonzero(copy):
        cands[i] = refs[rng.choice(np.flatnonzero(ref_imgs == cand_imgs[i]))]
    return refs, ref_imgs, cands, cand_imgs


CASES = [(500, 12, torch.int32), (10000, 22, torch.int64), (30000, 51, torch.int32), (32768, 51, torch.int64)]


@pytest.mark.gpu
@pytest.mark.parametrize("vocab,width,dtype", CASES)
def test_scorer_matches_reference(vocab, width, dtype):
    refs, ref_imgs, cands, cand_imgs = _split(vocab + width, vocab, width)
    scorer = pkg.CaptionScorer(torch.as_tensor(refs).to(dtype), ref_imgs, vocab, DEV)
    per, corpus = scorer.score(torch.as_tensor(cands).to(dtype).to(DEV), torch.as_tensor(cand_imgs).to(DEV))
    o_per, o_corpus, o_counts = M.score_ids(cands, cand_imgs, refs, ref_imgs)
    for name in NAMES:
        tol = 1e-4 if name.startswith("CIDEr") else 1e-5
        np.testing.assert_allclose(per[name].cpu().numpy(), o_per[name], rtol=0, atol=tol, err_msg=name)
    assert scorer.last_counts == o_counts["correct"] + o_counts["guess"] + [o_counts["testlen"], o_counts["reflen"]]
    for name in o_corpus:
        assert corpus[name] == pytest.approx(o_corpus[name], abs=1e-4 if name.startswith("CIDEr") else 1e-5), name
    assert o_corpus["CIDEr-D"] > 0.1 and o_corpus["Bleu_1"] > 0.1       # the split exercises real overlap
    # every document frequency in the table, decoded from its key
    keys = scorer.table.keys.cpu().numpy().view(np.uint64)
    dfs = scorer.table.df.cpu().numpy()
    got = {}
    for k, d in zip(keys[keys != 0], dfs[keys != 0]):
        n = int(k >> np.uint64(60))
        got[tuple(int((k >> np.uint64(45 - 15 * j)) & np.uint64(0x7FFF)) for j in range(n))] = int(d)
    gts = {}
    for row, img in zip(refs, ref_imgs):
        gts.setdefault(int(img), []).append(M.row_tokens(row))
    assert got == dict(M.document_frequency(gts))
    # two calls: bitwise the same
    per2, corpus2 = scorer.score(torch.as_tensor(cands).to(dtype).to(DEV), torch.as_tensor(cand_imgs).to(DEV))
    for name in NAMES:
        assert torch.equal(per[name], per2[name]), name
    assert corpus2 == corpus


@pytest.mark.gpu
def test_reward_on_device_graph_and_host_entry():
    from image_caption_b200.transformer import _graph_capture
    rng = np.random.default_rng(5)
    B, T, vocab = 32, 22, 10000
    rw = pkg.CaptionReward(cider_weight=0.7, bleu_weight=1.3)

    def batch():
        t = _rows(rng, B, T, vocab)[:, 1:]
        s = np.where(rng.random((B, T - 1)) < 0.6, t, _zipf_ids(rng, (B, T - 1), vocab))
        return t, s

    t, s = batch()
    ref = M.reward(t, s, 0.7, 1.3)
    got = rw.on_device(torch.as_tensor(t).to(DEV), torch.as_tensor(s).to(DEV)).cpu().numpy()
    np.testing.assert_allclose(got, ref, rtol=0, atol=2e-4)
    np.testing.assert_array_equal(rw(t, s), got)
    # captured once, replayed on new inputs
    ts, ss = torch.as_tensor(t).to(DEV), torch.as_tensor(s).to(DEV)
    rw.on_device(ts, ss)
    torch.cuda.synchronize()
    g = torch.cuda.CUDAGraph()
    with _graph_capture(g):
        out = rw.on_device(ts, ss)
    for _ in range(3):
        t, s = batch()
        ts.copy_(torch.as_tensor(t))
        ss.copy_(torch.as_tensor(s))
        g.replay()
        np.testing.assert_array_equal(out.cpu().numpy(), rw(t, s))
        np.testing.assert_allclose(out.cpu().numpy(), M.reward(t, s, 0.7, 1.3), rtol=0, atol=2e-4)


@pytest.fixture
def core_modules(monkeypatch):
    monkeypatch.setenv("ICAP_MAX_LENGTH", "10")
    monkeypatch.setenv("ICAP_SYNTHETIC_VOCAB", "500")
    monkeypatch.setenv("ICAP_CAPTION_MODEL", "RL_Transformer")
    sys.path.insert(0, PKG)
    try:
        yield
    finally:
        sys.path.remove(PKG)
        for m in [k for k in sys.modules if k == "core" or k.startswith("core.")]:
            sys.modules.pop(m)


@pytest.mark.gpu
def test_self_critic_loss_with_device_reward_matches_host_reward(core_modules):
    from core.models import SelfCriticNetwork
    from core.dataset import SyntheticCaptionDataset
    ds = SyntheticCaptionDataset(4, 36, 2048, 84, 12, 500, seed=7)
    img = ds.image_idx[:8]
    f, p, c = ds.features[img], ds.positions[img], ds.captions[:8]
    torch.manual_seed(0)
    net = SelfCriticNetwork(reward_fn=pkg.CaptionReward(1, 1))
    net.model.eval()
    dev_out = net.compute_loss(f, p, c)
    net.loss.structure_criterion.reward_fn = lambda tgt, seq: M.reward(tgt, seq, 1.0, 1.0)
    host_out = net.compute_loss(f, p, c)
    assert dev_out["reward"].shape == host_out["reward"].shape == (8, 1)
    torch.testing.assert_close(dev_out["reward"], host_out["reward"], rtol=0, atol=1e-4)
    assert abs(float(dev_out["loss"]) - float(host_out["loss"])) < 1e-5


def _run(args, cwd, extra_env=None):
    import subprocess
    env = dict(os.environ, ICAP_MAX_LENGTH="10", ICAP_SYNTHETIC_VOCAB="500", ICAP_BATCH_SIZE="8", ICAP_NUM_EPOCH="1")
    env.update(extra_env or {})
    return subprocess.run([sys.executable, os.path.join(PKG, "main.py"), *args], cwd=cwd, env=env, capture_output=True,
                          text=True, timeout=900)


def _scores_file(path):
    out = {}
    for line in open(path).read().splitlines():
        if ": " in line:
            k, v = line.split(": ")
            out[k] = float(v)
    return out


@pytest.mark.gpu
def test_cli_scores_synthetic_and_train_with_cider_reward(tmp_path):
    env = {}
    r = _run(["train", "--num-images", "16", "--max-iters", "2"], tmp_path, env)
    assert r.returncode == 0, r.stderr[-3000:]
    assert "valid scores" in r.stdout and "CIDEr-D" in r.stdout
    r = _run(["evaluation", "--split", "test", "--epoch", "1", "--num-images", "16"], tmp_path, env)
    assert r.returncode == 0, r.stderr[-3000:]
    assert "16 captions in" in r.stdout and "[evaluation] scores" in r.stdout
    path = os.path.join(tmp_path, "data", "maxlen49_36obj_1wordCount", "test",
                        "maxlen49_36obj_1wordCount_256_25b_32h_split_img_obj", "test_scores.txt")
    assert set(_scores_file(path)) == {"Bleu_1", "Bleu_2", "Bleu_3", "Bleu_4", "ROUGE_L", "CIDEr", "CIDEr-D"}
    rl = dict(env, ICAP_CAPTION_MODEL="RL_Transformer")
    r = _run(["train", "--num-images", "16", "--max-iters", "3", "--reward", "cider"], tmp_path, rl)
    assert r.returncode == 0, r.stderr[-3000:]
    assert "loss" in r.stdout and "valid scores" in r.stdout


@pytest.mark.gpu
def test_cli_scores_reference_layout_match_reference_scorer(tmp_path):
    """evaluation over data/<MODEL_NAME>/test/: the written scores equal the reference scorer on the written candidate
    strings against the decoded reference captions, and the region-cache and tensor feeds score the same."""
    from test_cli import _write_split
    env = {"ICAP_OUTPUT_NAME": "ctor_defaults", "ICAP_MAX_LENGTH": "10"}
    data_root = os.path.join(tmp_path, "data", "maxlen49_36obj_1wordCount")
    for split, n, seed in (("train", 12, 1), ("valid", 5, 2), ("test", 9, 3)):
        _, _, C, idxs = _write_split(data_root, split, n, 37, 84, 12, 300, seed=seed)
    r = _run(["train", "--max-iters", "2"], tmp_path, env)
    assert r.returncode == 0, r.stderr[-3000:]
    out_dir = os.path.join(data_root, "test", "ctor_defaults")
    lines = []
    for flag in ("True", "False"):
        r = _run(["evaluation", "--split", "test", "--epoch", "1", "--beam-size", "3", "--region-cache", flag], tmp_path,
                 env)
        assert r.returncode == 0, r.stderr[-3000:]
        lines.append([ln for ln in r.stdout.splitlines() if ln.startswith("[evaluation] scores")][0].split(": ", 1)[1])
    assert lines[0] == lines[1]
    with open(os.path.join(out_dir, "test.candidate.captions.pkl"), "rb") as fh:
        cands = pickle.load(fh)
    words = {0: "<NULL>", 1: "<START>", 2: "<END>", 3: "<UNK>"}
    words.update({i: f"w{i}" for i in range(4, 300)})
    refs = {}
    for row, img in zip(C, idxs):
        toks = []
        for t, i in enumerate(row):          # decode_captions, split on spaces
            if i == 1 and t == 0:
                continue
            if i == 2:
                toks.append(".")
                break
            if i != 0:
                toks.append(words[int(i)])
        refs.setdefault(int(img), []).append(toks)
    _, o_corpus, _ = M.score([c.split(" ") if c else [] for c in cands], list(range(len(cands))), refs)
    written = _scores_file(os.path.join(out_dir, "test_scores.txt"))       # two evaluations appended: same values
    for k, v in o_corpus.items():
        assert written[k] == pytest.approx(v, abs=1e-4 if k.startswith("CIDEr") else 1e-5), k
