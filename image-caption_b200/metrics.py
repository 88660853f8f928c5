"""Caption scores on the GPU: BLEU-1..4, ROUGE-L, CIDEr and CIDEr-D over token ids (libicap icap_caption_*).

`CaptionScorer` scores a split's decoded captions against its references, the scores the reference computes with
pycocoevalcap at the end of every epoch and in `main.py evaluation` (main.py:136-147,183-190, core/evaluations.py:12-34;
METEOR and SPICE need Java and are not computed).  `CaptionReward` is the self-critical reward of loss.py:160-186,
`cider_weight * CIDEr-D + bleu_weight * BLEU-4` per sample, usable as `reward_fn` of the RL loss and capturable in a
CUDA graph.

Rows are read like core/utils.py::decode_captions: a <START> at position 0 is skipped, <NULL> dropped, the row ends at
the first <END>, which counts as a token (the '.' decode_captions emits).  Scoring ids therefore gives the numbers
pycocoevalcap gives on the decoded strings split on spaces (for a vocabulary without a literal '.' word).  There is no
CPU fallback: every entry point needs CUDA tensors / a CUDA device.
"""
from __future__ import annotations

import math
from typing import Dict, Tuple

import numpy as np
import torch

from . import _native as N
from ._native import IcapError

MAX_WIDTH = 128          # widest row the kernels cook (MAX_LENGTH = 49 decodes rows of 52 ids)
MAX_VOCAB = 32768        # ids are packed 15 bits each into one uint64 n-gram key
SCORE_NAMES = ("CIDEr-D", "CIDEr", "ROUGE_L", "Bleu_1", "Bleu_2", "Bleu_3", "Bleu_4")


def _stream(dev: torch.device) -> int:
    return torch.cuda.current_stream(dev).cuda_stream


def _check_rows(x: torch.Tensor, what: str) -> None:
    if not isinstance(x, torch.Tensor) or x.dim() != 2 or x.dtype not in (torch.int32, torch.int64):
        raise IcapError(f"{what}: expected a 2-D int32 / int64 tensor")
    if not 1 <= x.shape[1] <= MAX_WIDTH:
        raise IcapError(f"{what}: row width {x.shape[1]} outside [1, {MAX_WIDTH}]")
    if x.device.type != "cuda":
        raise IcapError(f"{what}: tensors must be on a CUDA device (there is no CPU fallback)")
    if x.shape[1] > 1 and x.stride(1) != 1:
        raise IcapError(f"{what}: rows must be contiguous")


class _Cooked:
    """Device buffers of a cooked row set: distinct n-gram keys / counts per row, n-gram and token counts, the tokens
    after the cut, and per-order tf-idf norms (filled by `prep`)."""

    def __init__(self, n: int, width: int, dev: torch.device):
        self.n, self.width = n, width
        self.keys = torch.empty(n, 4 * width, dtype=torch.int64, device=dev)      # uint64 bit patterns
        self.counts = torch.empty(n, 4 * width, dtype=torch.int32, device=dev)
        self.nkeys = torch.empty(n, dtype=torch.int32, device=dev)
        self.lens = torch.empty(n, dtype=torch.int32, device=dev)
        self.toks = torch.empty(n, width, dtype=torch.int32, device=dev)
        self.norms = torch.empty(n, 4, dtype=torch.float64, device=dev)

    def cook(self, rows: torch.Tensor, stream: int) -> None:
        N.call("icap_caption_cook", rows.data_ptr(), int(rows.dtype == torch.int64), self.n, self.width, rows.stride(0),
               self.keys.data_ptr(), self.counts.data_ptr(), self.nkeys.data_ptr(), self.lens.data_ptr(),
               self.toks.data_ptr(), stream)


class _Table:
    """Open-addressing hash table key -> document frequency (0 = empty slot, linear probing)."""

    def __init__(self, cap: int, dev: torch.device):
        self.cap = cap
        self.keys = torch.zeros(cap, dtype=torch.int64, device=dev)
        self.df = torch.zeros(cap, dtype=torch.int32, device=dev)

    @property
    def nbytes(self) -> int:
        return self.keys.numel() * 8 + self.df.numel() * 4

    def fill(self, n_img: int, img_off: torch.Tensor, refs: _Cooked, stream: int) -> None:
        self.keys.zero_()
        self.df.zero_()
        N.call("icap_caption_df", n_img, img_off.data_ptr(), refs.width, refs.keys.data_ptr(), refs.nkeys.data_ptr(),
               self.keys.data_ptr(), self.df.data_ptr(), self.cap, None, stream)
        N.call("icap_caption_ref_prep", refs.n, refs.width, refs.keys.data_ptr(), refs.counts.data_ptr(),
               refs.nkeys.data_ptr(), n_img, self.keys.data_ptr(), self.df.data_ptr(), self.cap, refs.norms.data_ptr(),
               stream)


def _capacity(n_keys: int) -> int:
    """Smallest power of two >= 1.5 x the keys to insert: the table can never fill up."""
    return 1 << max(4, math.ceil(math.log2(max(1, (3 * n_keys + 1) // 2))))


def _score(cand: torch.Tensor, cand_img: torch.Tensor, n_img: int, img_off: torch.Tensor, refs: _Cooked, table: _Table,
           scores, reward, cider_weight: float, bleu_weight: float, corpus, stream: int) -> None:
    ptr = lambda t: None if t is None else t.data_ptr()                                                  # noqa: E731
    N.call("icap_caption_score", cand.data_ptr(), int(cand.dtype == torch.int64), cand.shape[0], cand.shape[1],
           cand.stride(0), cand_img.data_ptr(), n_img, img_off.data_ptr(), refs.width, refs.keys.data_ptr(),
           refs.counts.data_ptr(), refs.nkeys.data_ptr(), refs.lens.data_ptr(), refs.toks.data_ptr(),
           refs.norms.data_ptr(), table.keys.data_ptr(), table.df.data_ptr(), table.cap, ptr(scores), ptr(reward),
           float(cider_weight), float(bleu_weight), ptr(corpus), stream)


def corpus_bleu(counts) -> Tuple[float, float, float, float]:
    """Corpus BLEU-1..4 (option 'closest') from the summed counts {correct[4], guess[4], testlen, reflen}."""
    c = [int(x) for x in counts]
    out, bleu = [], 1.0
    for k in range(4):
        bleu *= (c[k] + 1e-15) / (c[4 + k] + 1e-9)
        out.append(bleu ** (1.0 / (k + 1)))
    ratio = (c[8] + 1e-15) / (c[9] + 1e-9)
    if ratio < 1:
        out = [b * math.exp(1 - 1 / ratio) for b in out]
    return tuple(out)


class CaptionScorer:
    """Scores captions of one split against its references.  The document frequencies of CIDEr / CIDEr-D come from the
    reference set (ref_len = log(number of images)) and are built once, here.

    ref_tokens: [R, W] id rows (tensor or ndarray, W <= 128), ref_image_idxs: [R] image of every row; every image
    0 .. n_img-1 needs at least one reference."""

    def __init__(self, ref_tokens, ref_image_idxs, num_vocab: int, device):
        if not 0 < int(num_vocab) <= MAX_VOCAB:
            raise IcapError(f"CaptionScorer: vocabulary of {num_vocab} ids; n-gram keys hold ids below {MAX_VOCAB}")
        refs = torch.as_tensor(np.asarray(ref_tokens) if not isinstance(ref_tokens, torch.Tensor) else ref_tokens)
        img = torch.as_tensor(np.asarray(ref_image_idxs)).to(torch.int64).cpu()
        if refs.dim() != 2 or not 1 <= refs.shape[1] <= MAX_WIDTH:
            raise IcapError(f"CaptionScorer: references must be [R, W] rows with W in [1, {MAX_WIDTH}], "
                            f"got {tuple(refs.shape)}")
        if img.shape != (refs.shape[0],) or refs.shape[0] == 0 or int(img.min()) < 0:
            raise IcapError("CaptionScorer: one non-negative image number per reference row is needed")
        dev = torch.device(device)
        if dev.type != "cuda":
            raise IcapError("CaptionScorer: needs a CUDA device (there is no CPU fallback)")
        per_image = torch.bincount(img)
        if bool((per_image == 0).any()):
            raise IcapError("CaptionScorer: images without a reference caption (every image 0..n-1 needs one)")
        self.n_img = int(per_image.numel())
        self.num_vocab = int(num_vocab)
        self.device = dev
        order = torch.sort(img, stable=True).indices
        rows = refs.to(torch.int64)[order].contiguous().to(dev)
        self.img_off = torch.cat([torch.zeros(1, dtype=torch.int64), per_image.cumsum(0)]).to(dev)
        st = _stream(dev)
        self.refs = _Cooked(rows.shape[0], rows.shape[1], dev)
        self.refs.cook(rows, st)
        n_unique = torch.zeros(1, dtype=torch.int64, device=dev)
        N.call("icap_caption_df", self.n_img, self.img_off.data_ptr(), self.refs.width, self.refs.keys.data_ptr(),
               self.refs.nkeys.data_ptr(), None, None, 0, n_unique.data_ptr(), st)
        self.table = _Table(_capacity(int(n_unique.item())), dev)     # the one host read: sizes the table
        self.table.fill(self.n_img, self.img_off, self.refs, st)

    @property
    def table_bytes(self) -> int:
        return self.table.nbytes

    def score(self, cand_tokens: torch.Tensor, cand_image_idxs: torch.Tensor) -> Tuple[Dict[str, torch.Tensor], Dict[str, float]]:
        """cand_tokens [M, W] (CUDA, int32 / int64), cand_image_idxs [M] (CUDA) -> (per-caption fp32 [M] tensors
        keyed by SCORE_NAMES, corpus scores {Bleu_1..4, ROUGE_L, CIDEr, CIDEr-D}).  Corpus BLEU is computed from the
        summed integer counts (`self.last_counts`), the other corpus scores are means over the captions."""
        _check_rows(cand_tokens, "CaptionScorer.score")
        if not isinstance(cand_image_idxs, torch.Tensor) or cand_image_idxs.device != cand_tokens.device:
            raise IcapError("CaptionScorer.score: image numbers must be a tensor on the device of the captions")
        if cand_image_idxs.shape != (cand_tokens.shape[0],):
            raise IcapError("CaptionScorer.score: one image number per caption is needed")
        dev = cand_tokens.device
        M = cand_tokens.shape[0]
        img = cand_image_idxs.to(torch.int64).contiguous()
        scores = torch.zeros(M, len(SCORE_NAMES), dtype=torch.float32, device=dev)
        counts = torch.zeros(10, dtype=torch.int64, device=dev)
        _score(cand_tokens, img, self.n_img, self.img_off, self.refs, self.table, scores, None, 0.0, 0.0, counts,
               _stream(dev))
        per = {name: scores[:, i] for i, name in enumerate(SCORE_NAMES)}
        self.last_counts = counts.cpu().tolist()
        corpus = {f"Bleu_{k + 1}": b for k, b in enumerate(corpus_bleu(self.last_counts))}
        means = scores.double().mean(0).tolist() if M else [0.0] * len(SCORE_NAMES)
        corpus.update(ROUGE_L=means[2], CIDEr=means[1], **{"CIDEr-D": means[0]})
        return per, corpus


class CaptionReward:
    """Self-critical reward `cider_weight * CIDEr-D + bleu_weight * BLEU-4` of every sampled caption against its own
    target (gts = {i: [target_i]}): document frequencies over the batch's targets, ref_len = log(B).

    `on_device(target, sample)` keeps everything on the GPU (no host sync): clear the table, cook the targets, count
    document frequencies, reference norms, score -- six stream-ordered launches into buffers cached per shape, so a call
    inside a CUDA-graph capture allocates nothing.  `__call__(target, sample)` takes and returns ndarrays (the
    `reward_fn` contract of core/TRANSFORMER/loss.py)."""

    def __init__(self, cider_weight: float = 1.0, bleu_weight: float = 1.0):
        self.cider_weight = float(cider_weight)
        self.bleu_weight = float(bleu_weight)
        self._bufs = {}

    def _buffers(self, target: torch.Tensor, sample: torch.Tensor):
        key = (target.shape[0], target.shape[1], target.device)
        b = self._bufs.get(key)
        if b is None:
            B, W, dev = target.shape[0], target.shape[1], target.device
            b = {"refs": _Cooked(B, W, dev), "table": _Table(_capacity(B * 4 * W), dev),
                 "idx": torch.arange(B + 1, dtype=torch.int64, device=dev),
                 "reward": torch.zeros(B, dtype=torch.float32, device=dev)}
            self._bufs[key] = b
        return b

    def on_device(self, target: torch.Tensor, sample: torch.Tensor) -> torch.Tensor:
        """target [B, T], sample [B, T'] (CUDA int32 / int64) -> fp32 [B] reward.  The returned tensor is a cached
        buffer: the next call with the same shapes overwrites it."""
        _check_rows(target, "CaptionReward target")
        _check_rows(sample, "CaptionReward sample")
        if sample.shape[0] != target.shape[0] or sample.device != target.device:
            raise IcapError("CaptionReward: target and sample need the same batch size and device")
        B = target.shape[0]
        if B == 0:
            return torch.zeros(0, dtype=torch.float32, device=target.device)
        b = self._buffers(target, sample)
        st = _stream(target.device)
        b["refs"].cook(target, st)
        b["table"].fill(B, b["idx"], b["refs"], st)
        _score(sample, b["idx"], B, b["idx"], b["refs"], b["table"], None, b["reward"], self.cider_weight,
               self.bleu_weight, None, st)
        return b["reward"]

    def __call__(self, target, sequence) -> np.ndarray:
        target, sequence = np.asarray(target), np.asarray(sequence)
        for a in (target, sequence):
            if a.size and (int(a.max()) >= MAX_VOCAB or int(a.min()) < 0):
                raise IcapError(f"CaptionReward: ids must lie in [0, {MAX_VOCAB})")
        dev = torch.device("cuda", torch.cuda.current_device()) if torch.cuda.is_available() else None
        if dev is None:
            raise IcapError("CaptionReward: needs a CUDA device (there is no CPU fallback)")
        t = torch.as_tensor(target.astype(np.int64)).to(dev)
        s = torch.as_tensor(sequence.astype(np.int64)).to(dev)
        return self.on_device(t, s).cpu().numpy().copy()
