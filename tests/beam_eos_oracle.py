"""CPU restatement of the beam search that stops at <END> (Transformer.beam_search_nbest, icap_beam_select_eos +
icap_beam_finalize in include/icap.h), in the style of oracle.caption_oracle.beam_search: every step re-runs the decoder
on the whole prefix of every hypothesis.  TEST INFRASTRUCTURE ONLY; the reference has no such search, so this module
sits beside the tests instead of in the reference oracle."""
import numpy as np
import torch
import torch.nn.functional as F

from oracle import caption_oracle as O

END, NULL = 2, 0


def hypothesis_length(row, end_idx=END, pad_idx=NULL):
    """Generated tokens of a token row (position 0 = <START>): up to and including the first <END>, before a first
    <NULL>, all of them if neither occurs."""
    for j in range(1, len(row)):
        if int(row[j]) == end_idx:
            return j
        if int(row[j]) == pad_idx:
            return j - 1
    return len(row) - 1


def normalised(score, length, alpha):
    return float(score) / ((5.0 + length) / 6.0) ** alpha


@torch.no_grad()
def beam_search_eos(sd, cfg, object_features, position_features, beam_size=5, n_best=None, length_penalty=0.0,
                    return_trace=False):
    """-> (ids LongTensor [B, n, max_length], scores FloatTensor [B, n] (log-probability), lengths LongTensor [B, n]),
    best first by score / ((5 + len) / 6)^length_penalty (ties: lower beam slot); with return_trace also the score gap
    between the k-th and (k+1)-th candidate of every step [B, max_length - 1] (+inf with only k candidates)."""
    k = beam_size
    n = k if n_best is None else n_best
    V, pad = cfg.num_vocab, cfg.pad_idx
    T = cfg.max_length - 1
    enc = O.encoder_forward(sd, cfg, object_features, position_features)
    B = enc.shape[0]
    region_pad = O.region_is_pad(position_features)
    cap = torch.zeros(B, k, cfg.max_length, dtype=torch.long)
    cap[:, :, 0] = 1
    prev = torch.zeros(B, k)
    trace = []
    for t in range(T):
        kin = 1 if t == 0 else k                       # step 0: every beam holds <START>, only beam 0 competes
        cand = torch.full((B, kin * V), float("-inf"))
        for r in range(kin):
            dec, _, _ = O.decoder_forward(sd, cfg, cap[:, r, :t + 1].clone(), enc, O._keypad_mask(region_pad, t + 1))
            lp = torch.log_softmax(F.linear(dec[:, t], sd["classifer.weight"], sd["classifer.bias"]), dim=1)
            cand[:, r * V:(r + 1) * V] = lp + prev[:, r:r + 1]
            if t >= 1:
                fin = (cap[:, r, t] == END) | (cap[:, r, t] == pad)
                cand[fin, r * V:(r + 1) * V] = float("-inf")
                cand[fin, r * V + pad] = prev[fin, r]
        s, idx = torch.sort(cand, dim=1, descending=True, stable=True)      # ties: lower r * V + j first
        if return_trace:
            trace.append(s[:, k - 1] - s[:, k])
        prev = s[:, :k].clone()
        parent, token = idx[:, :k] // V, idx[:, :k] % V
        cap = torch.gather(cap, 1, parent[:, :, None].expand(B, k, cfg.max_length)).clone()
        cap[:, :, t + 1] = token
    ids = torch.zeros(B, n, cfg.max_length, dtype=torch.long)
    scores = torch.zeros(B, n)
    lens = torch.zeros(B, n, dtype=torch.long)
    for b in range(B):
        ln = [hypothesis_length(cap[b, s]) for s in range(k)]
        order = sorted(range(k), key=lambda s: (-normalised(prev[b, s], ln[s], length_penalty), s))[:n]
        for i, s in enumerate(order):
            ids[b, i], scores[b, i], lens[b, i] = cap[b, s], prev[b, s], ln[s]
    if return_trace:
        return ids, scores, lens, torch.stack(trace, 1)
    return ids, scores, lens


def teacher_forced_logprob(logits, ids, pad_idx=NULL):
    """Log-likelihood of token rows under teacher-forced logits [M, T, V] (fp64): the sum of log_softmax at positions
    1.. up to and including the first <END> / <NULL> (or all T) -- the tokens a hypothesis scored while unfinished."""
    lp = torch.log_softmax(logits.double(), dim=2)
    out = []
    for m in range(ids.shape[0]):
        total = 0.0
        for j in range(1, ids.shape[1]):
            tok = int(ids[m, j])
            total += float(lp[m, j - 1, tok])
            if tok in (END, pad_idx):
                break
        out.append(total)
    return np.array(out)
