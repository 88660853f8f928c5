"""fp64 reference of the caption metrics the library computes on the GPU: a literal, dict-based restatement of
coco-caption's bleu_scorer.py (option='closest') and rouge.py and of pyciderevalcap's cider_scorer.py and
ciderD_scorer.py.  Tokens are any hashable values (ids or words), so the same code scores id rows and the strings
core/utils.py::decode_captions makes of them."""
import math
from collections import Counter

import numpy as np

NULL, START, END = 0, 1, 2
TINY, SMALL = 1e-15, 1e-9
BETA = 1.2
SIGMA = 6.0


def row_tokens(row):
    """ids -> tokens, read like decode_captions: skip <START> at position 0, drop <NULL>, stop after the first <END>."""
    out = []
    for t, idx in enumerate(row):
        idx = int(idx)
        if idx == START and t == 0:
            continue
        if idx == END:
            out.append(idx)
            break
        if idx != NULL:
            out.append(idx)
    return out


def precook(words, n=4):
    counts = Counter()
    for k in range(1, n + 1):
        for i in range(len(words) - k + 1):
            counts[tuple(words[i:i + k])] += 1
    return counts


def document_frequency(refs):
    """refs: {image: [token list, ...]} -> {ngram: number of images with the ngram in at least one reference}."""
    df = Counter()
    for rs in refs.values():
        for g in set(g for r in rs for g in precook(r)):
            df[g] += 1
    return df


def _bleu(correct, guess, testlen, reflen):
    out, bleu = [], 1.0
    for k in range(4):
        bleu *= (float(correct[k]) + TINY) / (float(guess[k]) + SMALL)
        out.append(bleu ** (1.0 / (k + 1)))
    ratio = (testlen + TINY) / (reflen + SMALL)
    if ratio < 1:
        out = [b * math.exp(1 - 1 / ratio) for b in out]
    return out


def _lcs(a, b):
    prev = [0] * (len(b) + 1)
    for x in a:
        cur = [0]
        for j, y in enumerate(b):
            cur.append(prev[j] + 1 if x == y else max(prev[j + 1], cur[j]))
        prev = cur
    return prev[-1]


def _vec(counts, df, ref_len):
    vec, norm, length = [{} for _ in range(4)], [0.0] * 4, 0
    for g, tf in counts.items():
        n = len(g) - 1
        vec[n][g] = float(tf) * (ref_len - math.log(max(1.0, df.get(g, 0))))
        norm[n] += vec[n][g] ** 2
        if n == 1:
            length += tf
    return vec, [math.sqrt(x) for x in norm], length


def _cider(vc, nc, lc, vr, nr, lr, clipped):
    delta = float(lc - lr)
    val = [0.0] * 4
    for n in range(4):
        for g in vc[n]:
            r = vr[n].get(g, 0.0)
            val[n] += (min(vc[n][g], r) if clipped else vc[n][g]) * r
        if nc[n] != 0 and nr[n] != 0:
            val[n] /= nc[n] * nr[n]
        if clipped:
            val[n] *= math.exp(-(delta ** 2) / (2 * SIGMA ** 2))
    return val


def score(cands, cand_imgs, refs, df=None):
    """cands: token lists; cand_imgs: image of each; refs: {image: [token list, ...]} (the df set unless `df` is given,
    with log(len(refs)) as ref_len).  -> (per-candidate dict of float64 arrays, corpus dict, corpus BLEU counts)."""
    if df is None:
        df = document_frequency(refs)
    ref_len = math.log(float(len(refs)))
    keys = ("CIDEr-D", "CIDEr", "ROUGE_L", "Bleu_1", "Bleu_2", "Bleu_3", "Bleu_4")
    per = {k: np.zeros(len(cands)) for k in keys}
    counts = {"correct": [0] * 4, "guess": [0] * 4, "testlen": 0, "reflen": 0}
    for i, (c, img) in enumerate(zip(cands, cand_imgs)):
        rs = refs.get(img, [])
        cc = precook(c)
        # BLEU
        maxref = Counter()
        for r in rs:
            for g, n in precook(r).items():
                maxref[g] = max(maxref[g], n)
        reflen = min((abs(len(r) - len(c)), len(r)) for r in rs)[1] if rs else 0
        correct, guess = [0] * 4, [max(0, len(c) - k) for k in range(4)]
        for g, n in cc.items():
            correct[len(g) - 1] += min(maxref.get(g, 0), n)
        for k in range(4):
            counts["correct"][k] += correct[k]
            counts["guess"][k] += guess[k]
        counts["testlen"] += len(c)
        counts["reflen"] += reflen
        for k, b in enumerate(_bleu(correct, guess, len(c), reflen)):
            per[f"Bleu_{k + 1}"][i] = b
        if not rs:
            continue
        # ROUGE-L
        lcs = [_lcs(r, c) for r in rs]
        p = max(l / len(c) if c else 0.0 for l in lcs)
        rec = max(l / len(r) if r else 0.0 for l, r in zip(lcs, rs))
        per["ROUGE_L"][i] = (1 + BETA ** 2) * p * rec / (rec + BETA ** 2 * p) if p != 0 and rec != 0 else 0.0
        # CIDEr / CIDEr-D
        vc, nc, lc = _vec(cc, df, ref_len)
        sd, sc = np.zeros(4), np.zeros(4)
        for r in rs:
            vr, nr, lr = _vec(precook(r), df, ref_len)
            sd += _cider(vc, nc, lc, vr, nr, lr, True)
            sc += _cider(vc, nc, lc, vr, nr, lr, False)
        per["CIDEr-D"][i] = float(np.mean(sd)) / len(rs) * 10.0
        per["CIDEr"][i] = float(np.mean(sc)) / len(rs) * 10.0
    corpus = {f"Bleu_{k + 1}": b for k, b in enumerate(
        _bleu(counts["correct"], counts["guess"], counts["testlen"], counts["reflen"]))}
    corpus["ROUGE_L"] = float(np.mean(per["ROUGE_L"])) if len(cands) else 0.0
    corpus["CIDEr"] = float(np.mean(per["CIDEr"])) if len(cands) else 0.0
    corpus["CIDEr-D"] = float(np.mean(per["CIDEr-D"])) if len(cands) else 0.0
    return per, corpus, counts


def score_ids(cand_rows, cand_imgs, ref_rows, ref_imgs):
    """The same on id rows: references grouped by their image number."""
    refs = {}
    for row, img in zip(ref_rows, ref_imgs):
        refs.setdefault(int(img), []).append(row_tokens(row))
    return score([row_tokens(r) for r in cand_rows], [int(i) for i in cand_imgs], refs)


def reward(target_rows, sample_rows, cider_weight=1.0, bleu_weight=1.0):
    """Self-critical reward: sample i scored against the single reference target i, df over the batch's targets."""
    B = len(target_rows)
    per, _, _ = score_ids(sample_rows, range(B), target_rows, range(B))
    return cider_weight * per["CIDEr-D"] + bleu_weight * per["Bleu_4"]
