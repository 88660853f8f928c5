"""CPU oracle for the caption-generator hot path.  TEST INFRASTRUCTURE ONLY.

This file is a CPU restatement (functional, state_dict driven, torch-CPU fp32 /
fp64 arithmetic) of the reference algorithm in shao-chi/Image-Caption:

    core/TRANSFORMER/modules.py   (attention / FFN / blocks)
    core/TRANSFORMER/model.py     (Transformer, Encoder, Decoder, PositionalEncoding)
    core/TRANSFORMER/model_RL.py  (PolicyNetwork logits / log-softmax beam variant)
    core/TRANSFORMER/loss.py:13-28 (FocalLoss)
    core/models.py:111-126        (Adam train_step)

It is the checker for the CUDA path.  Only ``tests/``, ``__graft_entry__.smoke()``
and ``bench.py``'s cpu_baseline / ``--impl reference`` leg may import it; the
product package (``image-caption_b200/``) never does and has no CPU fallback.

Parity pin: the reference ships no tests / golden vectors (SURVEY.md §4, §8c), so
this oracle is pinned against OUTPUTS OF THE REFERENCE ITSELF: the fixtures in
``tests/golden/*.pt`` were produced by ``tests/golden/make_golden.py`` importing the
unmodified reference classes, and ``tests/test_oracle.py`` checks every function
here against them.

All hot-path arithmetic in the reference is PyTorch ATen (pinned torch==1.7.1,
requirements.txt:57); the oracle uses the same ATen CPU operators through
``torch.nn.functional`` so that fp32 rounding behaviour matches the reference's.
"""
from __future__ import annotations

import math
from dataclasses import dataclass, asdict
from typing import Dict, Iterator, List, Optional, Tuple

import numpy as np
import torch
import torch.nn.functional as F

Tensor = torch.Tensor


@dataclass
class OracleConfig:
    """Constructor arguments of the reference ``Transformer`` (model.py:10-36)."""
    num_vocab: int
    max_length: int
    encode_dim_positions: int
    encode_dim_features: int
    output_name: str = "x"
    encode_mask: bool = False
    pad_idx: int = 0
    dropout: float = 0.2
    encode_input_size: int = 512
    encode_q_k_dim: int = 512
    encode_v_dim: int = 512
    encode_hidden_size: int = 2048
    encode_num_blocks: int = 6
    encode_num_heads: int = 8
    dim_word_embedding: int = 512
    decode_input_size: int = 512
    decode_q_k_dim: int = 512
    decode_v_dim: int = 512
    decode_hidden_size: int = 2048
    decode_num_blocks: int = 6
    decode_num_heads: int = 8
    move_first_image_feature: bool = False
    split_position: bool = False
    split_image_objects: bool = False

    def ctor_kwargs(self) -> dict:
        return asdict(self)


LN_EPS = 1e-6  # modules.py:57,105 ; model.py:247,396


# --------------------------------------------------------------------------
# blocks  (modules.py)
# --------------------------------------------------------------------------
def _layer_norm(x: Tensor, sd: Dict[str, Tensor], prefix: str) -> Tensor:
    return F.layer_norm(x, (x.shape[-1],), sd[prefix + ".weight"], sd[prefix + ".bias"], LN_EPS)


def _mha(sd, prefix: str, q_in: Tensor, kv_in: Tensor, mask: Optional[Tensor], num_heads: int
         ) -> Tuple[Tensor, Tensor]:
    """MultiHeadAttention.forward, eval mode (modules.py:67-92) + SDPA (modules.py:16-27).

    mask: bool [B, Lq, Lk], True = masked out.  q is divided by sqrt(dh) BEFORE QK^T.
    """
    B, Lq, _ = q_in.shape
    Lk = kv_in.shape[1]
    wq, wk, wv = sd[prefix + ".q_linear.weight"], sd[prefix + ".k_linear.weight"], sd[prefix + ".v_linear.weight"]
    dk = wq.shape[0] // num_heads
    dv = wv.shape[0] // num_heads
    q = F.linear(q_in, wq).view(B, Lq, num_heads, dk).transpose(1, 2)
    k = F.linear(kv_in, wk).view(B, Lk, num_heads, dk).transpose(1, 2)
    v = F.linear(kv_in, wv).view(B, Lk, num_heads, dv).transpose(1, 2)
    att = torch.matmul(q / (dk ** 0.5), k.transpose(2, 3))
    if mask is not None:
        att = att.masked_fill(mask.unsqueeze(1), -np.inf)
    att = torch.softmax(att, dim=-1)
    out = torch.matmul(att, v).transpose(1, 2).contiguous().view(B, Lq, -1)
    out = F.linear(out, sd[prefix + ".joint_linear.weight"])
    out = _layer_norm(out + q_in, sd, prefix + ".layer_norm")
    return out, att


def _ffn(sd, prefix: str, x: Tensor) -> Tensor:
    """FeedForward.forward, eval mode (modules.py:110-122)."""
    h = F.relu(F.linear(x, sd[prefix + ".position_wise_1.weight"], sd[prefix + ".position_wise_1.bias"]))
    o = F.linear(h, sd[prefix + ".position_wise_2.weight"], sd[prefix + ".position_wise_2.bias"])
    return _layer_norm(o + x, sd, prefix + ".layer_norm")


def _encoder_block(sd, prefix, x, num_heads, non_pad_mask=None, attention_mask=None):
    """EncoderBlock.forward (modules.py:146-157)."""
    out, att = _mha(sd, prefix + ".multihead_attention", x, x, attention_mask, num_heads)
    out = _ffn(sd, prefix + ".feed_forward", out)
    if non_pad_mask is not None:
        out = out * non_pad_mask
    return out, att


def _decoder_block(sd, prefix, x, enc, num_heads, non_pad_mask, self_mask, ctx_mask):
    """DecoderBlock.forward (modules.py:185-206)."""
    out, self_att = _mha(sd, prefix + ".self_attention", x, x, self_mask, num_heads)
    out, ctx_att = _mha(sd, prefix + ".encode_attention", out, enc, ctx_mask, num_heads)
    out = _ffn(sd, prefix + ".feed_forward", out)
    if non_pad_mask is not None:
        out = out * non_pad_mask
    return out, self_att, ctx_att


# --------------------------------------------------------------------------
# masks (model.py:202-209, 334-358, 461-486)
# --------------------------------------------------------------------------
def region_is_pad(position_features: Tensor) -> Tensor:
    """A region is padding iff its position row is all zero (model.py:206)."""
    return torch.count_nonzero(position_features, dim=2).eq(0)  # [B, R] bool


def _keypad_mask(pad: Tensor, lq: int) -> Tensor:
    return pad.unsqueeze(1).expand(pad.shape[0], lq, pad.shape[1])


def _subsequent_mask(batch: int, length: int) -> Tensor:
    m = torch.triu(torch.ones((length, length), dtype=torch.uint8), diagonal=1)
    return m.unsqueeze(0).expand(batch, length, length)


# --------------------------------------------------------------------------
# Encoder (model.py:212-332)
# --------------------------------------------------------------------------
def encoder_forward(sd, cfg: OracleConfig, object_features: Tensor, position_features: Tensor) -> Tensor:
    H = cfg.encode_num_heads
    B, R, _ = object_features.shape
    wf = sd["encoder.feature_embedding.weight"]
    wp = sd["encoder.position_embedding.weight"]
    if cfg.split_image_objects:
        # model.py:258-292 : per region a 2-token sequence [whole image (region 0), region i]
        img_f = object_features[:, 0].unsqueeze(1).repeat(1, R, 1)
        img_p = position_features[:, 0].unsqueeze(1).repeat(1, R, 1)
        feat = torch.cat([img_f.reshape(-1, img_f.shape[2]).unsqueeze(1),
                          object_features.reshape(-1, object_features.shape[2]).unsqueeze(1)], dim=1)
        pos = torch.cat([img_p.reshape(-1, img_p.shape[2]).unsqueeze(1),
                         position_features.reshape(-1, position_features.shape[2]).unsqueeze(1)], dim=1)
        pad2 = region_is_pad(pos)
        non_pad2 = (~pad2).float().unsqueeze(-1)
        mask2 = (_keypad_mask(pad2, 2).to(torch.uint8) + _subsequent_mask(B * R, 2)).gt(0)
        emb_f = F.linear(feat, wf)
        emb_p = F.linear(pos, wp)  # NB: the reference uses position_embedding on the full row here
        out = _layer_norm(emb_f + emb_p, sd, "encoder.norm")
        out, _ = _encoder_block(sd, "encoder.image_encoder", out, H, non_pad2, mask2)
        out = out[:, 1, :].reshape(B, R, -1) + emb_p[:, 1, :].reshape(B, R, -1)
    else:
        emb_f = F.linear(object_features, wf)
        if cfg.split_position:
            out = emb_f + F.linear(position_features[:, :, :4], wp) \
                + F.linear(position_features[:, :, 4:], sd["encoder.object_embedding.weight"])
        else:
            out = emb_f + F.linear(position_features, wp)
    out = _layer_norm(out, sd, "encoder.norm")

    pad = region_is_pad(position_features)
    non_pad = (~pad).float().unsqueeze(-1)
    mask = (_keypad_mask(pad, R).to(torch.uint8) + _subsequent_mask(B, R)).gt(0)
    for i in range(cfg.encode_num_blocks):
        if cfg.encode_mask:
            out, _ = _encoder_block(sd, f"encoder.encoder.{i}", out, H, non_pad, mask)
        else:
            out, _ = _encoder_block(sd, f"encoder.encoder.{i}", out, H)
    return out


# --------------------------------------------------------------------------
# Decoder (model.py:362-459) and PositionalEncoding (model.py:489-517)
# --------------------------------------------------------------------------
def sinusoid_table(num_positions: int, dim: int) -> Tensor:
    """float64 numpy table -> FloatTensor [1, num_positions, dim] (model.py:502-514)."""
    j = np.arange(dim)
    pos = np.arange(num_positions, dtype=np.float64)[:, None]
    table = pos / np.power(10000, 2 * (j // 2) / dim)[None, :]
    table[:, 0::2] = np.sin(table[:, 0::2])
    table[:, 1::2] = np.cos(table[:, 1::2])
    return torch.tensor(table, dtype=torch.float32).unsqueeze(0)


def decoder_forward(sd, cfg: OracleConfig, caption_vector: Tensor, encode_output: Tensor,
                    context_attention_mask: Tensor) -> Tuple[Tensor, Tensor, Tensor]:
    B, T = caption_vector.shape
    H = cfg.decode_num_heads
    non_pad = caption_vector.ne(cfg.pad_idx).float().unsqueeze(-1)
    keypad = caption_vector.eq(cfg.pad_idx).unsqueeze(1).expand(B, T, T)
    self_mask = (keypad.to(torch.uint8) + _subsequent_mask(B, T)).gt(0)

    emb = F.embedding(caption_vector, sd["decoder.word_embedding.weight"], padding_idx=cfg.pad_idx)
    x = F.linear(emb, sd["decoder.word_embedding_linear.weight"])
    x = x + sd["decoder.position_embedding.pos_table"][:, :T]
    x = _layer_norm(x, sd, "decoder.norm")
    self_att = ctx_att = None
    for i in range(cfg.decode_num_blocks):
        x, self_att, ctx_att = _decoder_block(sd, f"decoder.decoder.{i}", x, encode_output, H,
                                              non_pad, self_mask, context_attention_mask)
    if cfg.move_first_image_feature:  # model.py:451-457
        first = encode_output[:, 0].unsqueeze(1)
        h = F.relu(F.linear(x + first, sd["decoder.position_wise_1.weight"], sd["decoder.position_wise_1.bias"]))
        h = F.linear(h, sd["decoder.position_wise_2.weight"], sd["decoder.position_wise_2.bias"])
        x = _layer_norm(h + x, sd, "decoder.layer_norm")
    return x, self_att, ctx_att


# --------------------------------------------------------------------------
# Transformer.forward (model.py:79-98) / PolicyNetwork.forward (model_RL.py:75-90)
# --------------------------------------------------------------------------
def logits_forward(sd, cfg: OracleConfig, object_features, position_features, target_caption) -> Tensor:
    """Teacher-forced logits [B, T, V] (== PolicyNetwork.forward)."""
    inp = target_caption[:, :-1].long()
    ctx_mask = _keypad_mask(region_is_pad(position_features), inp.shape[1])
    enc = encoder_forward(sd, cfg, object_features, position_features)
    dec, _, _ = decoder_forward(sd, cfg, inp, enc, ctx_mask)
    return F.linear(dec, sd["classifer.weight"], sd["classifer.bias"])


def loss_from_logits(cfg: OracleConfig, logits: Tensor, target_caption: Tensor) -> Tensor:
    tgt = target_caption[:, 1:].long().contiguous().view(-1)
    ce = F.cross_entropy(logits.view(-1, logits.shape[2]), tgt, ignore_index=cfg.pad_idx, reduction="mean")
    if cfg.output_name.find("FocalLoss") != -1:  # model.py:73-74 ; loss.py:20-28 (gamma = 2)
        pt = torch.exp(-ce)
        return ((1 - pt) ** 2 * ce).mean()
    return ce


def forward_loss(sd, cfg, object_features, position_features, target_caption) -> Dict[str, Tensor]:
    logits = logits_forward(sd, cfg, object_features, position_features, target_caption)
    return {"loss": loss_from_logits(cfg, logits, target_caption)}


def loss_and_grads(sd, cfg, object_features, position_features, target_caption
                   ) -> Tuple[Tensor, Dict[str, Tensor]]:
    """loss.backward() of models.py:125 : grads for every parameter (buffers excluded)."""
    names = [k for k in sd if not k.endswith("pos_table")]
    leaf = {k: (sd[k].detach().clone().requires_grad_(True) if k in names else sd[k]) for k in sd}
    loss = forward_loss(leaf, cfg, object_features, position_features, target_caption)["loss"]
    grads = torch.autograd.grad(loss, [leaf[k] for k in names], allow_unused=True)
    out = {k: (g if g is not None else torch.zeros_like(sd[k])) for k, g in zip(names, grads)}
    return loss.detach(), out


# --------------------------------------------------------------------------
# Adam (models.py:111-113,126 : torch.optim.Adam defaults, lr given)
# --------------------------------------------------------------------------
class AdamState:
    def __init__(self, sd: Dict[str, Tensor], lr: float = 5e-4, betas=(0.9, 0.999), eps: float = 1e-8):
        self.lr, self.b1, self.b2, self.eps, self.t = lr, betas[0], betas[1], eps, 0
        self.names = [k for k in sd if not k.endswith("pos_table")]
        self.m = {k: torch.zeros_like(sd[k]) for k in self.names}
        self.v = {k: torch.zeros_like(sd[k]) for k in self.names}

    def step(self, sd: Dict[str, Tensor], grads: Dict[str, Tensor]) -> None:
        """In-place update, same operation order as torch.optim.Adam (no amsgrad, wd=0)."""
        self.t += 1
        bc1 = 1 - self.b1 ** self.t
        bc2 = 1 - self.b2 ** self.t
        step_size = self.lr / bc1
        for k in self.names:
            g = grads[k]
            self.m[k].mul_(self.b1).add_(g, alpha=1 - self.b1)
            self.v[k].mul_(self.b2).addcmul_(g, g, value=1 - self.b2)
            denom = (self.v[k].sqrt() / math.sqrt(bc2)).add_(self.eps)
            sd[k].addcdiv_(self.m[k], denom, value=-step_size)


def train_steps(sd, cfg, batches, lr=5e-4) -> List[float]:
    """TRANSFORMER.train_step (models.py:115-126) repeated; eval-mode (dropout-free) arithmetic."""
    opt = AdamState(sd, lr=lr)
    losses = []
    for feats, pos, cap in batches:
        loss, grads = loss_and_grads(sd, cfg, feats, pos, cap)
        opt.step(sd, grads)
        losses.append(float(loss))
    return losses


# --------------------------------------------------------------------------
# decoding (model.py:101-200)
# --------------------------------------------------------------------------
@torch.no_grad()
def generate_caption_vector(sd, cfg, object_features, position_features, return_gaps: bool = False):
    """Greedy decode, full-prefix recompute exactly as model.py:101-132.

    Returns (LongTensor [B, max_length+1], list of max_length-1 float32 arrays [B, R]);
    with return_gaps also the top-2 logit gap of every decision [B, max_length-1].
    """
    enc = encoder_forward(sd, cfg, object_features, position_features)
    B = enc.shape[0]
    pad = region_is_pad(position_features)
    cap = torch.zeros(B, cfg.max_length + 1, dtype=torch.long)
    cap[:, 0] = 1
    attention_list, gaps = [], []
    for t in range(cfg.max_length - 1):
        inp = cap[:, :t + 1].clone()
        dec, _, att = decoder_forward(sd, cfg, inp, enc, _keypad_mask(pad, t + 1))
        attention_list.append(np.mean(att.numpy()[:, :, t], axis=1))
        logits = F.linear(dec[:, t], sd["classifer.weight"], sd["classifer.bias"])
        if return_gaps:
            top2 = torch.topk(logits, 2, dim=1).values
            gaps.append((top2[:, 0] - top2[:, 1]))
        cap[:, t + 1] = torch.argmax(torch.softmax(logits, dim=1), dim=1)
    if return_gaps:
        return cap, attention_list, torch.stack(gaps, 1)
    return cap, attention_list


@torch.no_grad()
def beam_search(sd, cfg, object_features, position_features, beam_size: int = 1,
                log_domain: bool = False, return_trace: bool = False):
    """Beam search exactly as model.py:135-200 (probability-domain additive scores, no EOS
    handling, ``topk(sorted=False)``, returns slot 0).  ``log_domain=True`` gives the
    PolicyNetwork variant (model_RL.py:72,157,182 : LogSoftmax).

    return_trace additionally returns, per step, the score gap between the k-th and
    (k+1)-th candidate (near-tie reporting)."""
    V = cfg.num_vocab
    sm = (lambda x: torch.log_softmax(x, dim=1)) if log_domain else (lambda x: torch.softmax(x, dim=1))
    enc = encoder_forward(sd, cfg, object_features, position_features)
    B = enc.shape[0]
    pad = region_is_pad(position_features)
    cap = torch.zeros(beam_size, B, cfg.max_length, dtype=torch.long)
    cap[:, :, 0] = 1
    inp = cap[0, :, :1].clone()
    dec, _, _ = decoder_forward(sd, cfg, inp, enc, _keypad_mask(pad, 1))
    out = sm(F.linear(dec[:, 0], sd["classifer.weight"], sd["classifer.bias"]))
    trace = []
    if return_trace:
        s = torch.sort(out, dim=1, descending=True).values
        trace.append(s[:, beam_size - 1] - s[:, beam_size])
    prob, idx = torch.topk(out, k=beam_size, dim=1, sorted=False)
    prob, idx = prob.transpose(0, 1), idx.transpose(0, 1)
    cap[:, :, 1] = idx
    for t in range(1, cfg.max_length - 1):
        cands = []
        for b in range(beam_size):
            inp = cap[b, :, :t + 1].clone()
            dec, _, _ = decoder_forward(sd, cfg, inp, enc, _keypad_mask(pad, t + 1))
            o = sm(F.linear(dec[:, t], sd["classifer.weight"], sd["classifer.bias"])) + prob[b].unsqueeze(1)
            cands.append(o)
        scores = torch.cat(cands, 1)
        if return_trace:
            s = torch.sort(scores, dim=1, descending=True).values
            trace.append(s[:, beam_size - 1] - s[:, beam_size])
        prob, idx = torch.topk(scores, k=beam_size, dim=1, sorted=False)
        prob, idx = prob.transpose(0, 1), idx.transpose(0, 1)
        cols = torch.stack([torch.arange(B)] * beam_size)
        cap = cap[idx // V, cols].clone()
        cap[:, :, t + 1] = idx % V
    if return_trace:
        return cap[0], torch.stack(trace, 1)
    return cap[0]


# --------------------------------------------------------------------------
# ids -> strings (core/utils.py:67-103), kept because generate_caption returns strings
# --------------------------------------------------------------------------
def decode_captions(captions: np.ndarray, index_to_word: Dict[int, str]) -> List[str]:
    captions = np.asarray(captions)
    if captions.ndim == 1:
        captions = captions[None, :]
    decoded = []
    for row in captions:
        words = []
        for t, idx in enumerate(row):
            word = index_to_word[int(idx)]
            if word == "<START>" and t == 0:
                continue
            if word == "<END>":
                words.append(".")
                break
            if word != "<NULL>":
                words.append(word)
        decoded.append(" ".join(words))
    return decoded


# --------------------------------------------------------------------------
# synthetic inputs (SURVEY.md §8d) and reference-style initialisation
# --------------------------------------------------------------------------
def synthetic_batch(batch: int, regions: int, dim_features: int, dim_positions: int, max_length: int,
                    num_vocab: int, seed: int = 1234) -> Tuple[Tensor, Tensor, Tensor]:
    """features [B,R,Df] f32 (>=0, zero on padded regions), positions [B,R,Dp] f32 (row 0 = whole
    image [0,0,1,1,0..], padded rows all-zero), captions [B,max_length] int32 = [1, w.., 2, 0..]."""
    g = torch.Generator().manual_seed(seed)
    lo = (regions + 1) // 2
    n_valid = torch.randint(lo, regions + 1, (batch,), generator=g)
    feats = torch.randn(batch, regions, dim_features, generator=g).abs_()
    pos = torch.zeros(batch, regions, dim_positions)
    xy = torch.rand(batch, regions, 4, generator=g)
    x = torch.sort(xy[:, :, 0:2], dim=2).values
    y = torch.sort(xy[:, :, 2:4], dim=2).values
    pos[:, :, 0], pos[:, :, 2] = x[:, :, 0], x[:, :, 1]
    pos[:, :, 1], pos[:, :, 3] = y[:, :, 0], y[:, :, 1]
    if dim_positions > 4:
        cls = torch.randint(4, dim_positions, (batch, regions), generator=g)
        conf = torch.rand(batch, regions, generator=g) * 0.99 + 0.01
        pos.scatter_(2, cls.unsqueeze(-1), conf.unsqueeze(-1))
    pos[:, 0] = 0
    pos[:, 0, 2] = 1
    pos[:, 0, 3] = 1
    valid = (torch.arange(regions)[None, :] < n_valid[:, None])
    feats *= valid.unsqueeze(-1)
    pos *= valid.unsqueeze(-1)
    cap = torch.zeros(batch, max_length, dtype=torch.int32)
    cap[:, 0] = 1
    n_words = torch.randint(min(5, max_length - 2), max_length - 1, (batch,), generator=g)
    words = torch.randint(4, num_vocab, (batch, max_length), generator=g, dtype=torch.int32)
    for b in range(batch):
        n = int(n_words[b])
        cap[b, 1:1 + n] = words[b, :n]
        cap[b, 1 + n] = 2
    return feats, pos, cap


def _walk(prefix: str, children) -> Iterator[Tuple[str, Tuple[int, ...]]]:
    """Flatten a (name, shape | children) tree the way nn.Module.state_dict() walks registered members."""
    for name, node in children:
        if isinstance(node, tuple):
            yield prefix + name, node
        else:
            yield from _walk(prefix + name + ".", node)


def _shape_linear(out_f: int, in_f: int, bias: bool = True):
    return [("weight", (out_f, in_f))] + ([("bias", (out_f,))] if bias else [])


def _shape_layer_norm(n: int):
    return [("weight", (n,)), ("bias", (n,))]


def _shape_multihead(d_in: int, dk: int, dv: int):
    # modules.py MultiHeadAttention.__init__: three bias-free projections, the norm, then the bias-free output projection
    return [("q_linear", _shape_linear(dk, d_in, False)), ("k_linear", _shape_linear(dk, d_in, False)),
            ("v_linear", _shape_linear(dv, d_in, False)), ("layer_norm", _shape_layer_norm(d_in)),
            ("joint_linear", _shape_linear(d_in, dv, False))]


def _shape_feed_forward(d_in: int, hidden: int):
    # modules.py PositionWiseFeedForward.__init__
    return [("position_wise_1", _shape_linear(hidden, d_in)), ("position_wise_2", _shape_linear(d_in, hidden)),
            ("layer_norm", _shape_layer_norm(d_in))]


def param_shapes(cfg: OracleConfig) -> "Dict[str, Tuple[int, ...]]":
    """state_dict layout (SURVEY.md 8a): the member tree of the reference's Transformer in the order its __init__ methods
    register it (model.py Encoder / Decoder / Transformer, modules.py blocks), flattened like state_dict() does.  Pinned to
    the reference's own key list and shapes by tests/test_oracle.py::test_state_dict_layout."""
    d, dd = cfg.encode_input_size, cfg.decode_input_size
    enc_block = [("multihead_attention", _shape_multihead(d, cfg.encode_q_k_dim, cfg.encode_v_dim)),
                 ("feed_forward", _shape_feed_forward(d, cfg.encode_hidden_size))]
    encoder = []
    if cfg.split_position:
        encoder.append(("object_embedding", _shape_linear(d, cfg.encode_dim_positions - 4, False)))
        encoder.append(("position_embedding", _shape_linear(d, 4, False)))
    else:
        encoder.append(("position_embedding", _shape_linear(d, cfg.encode_dim_positions, False)))
    if cfg.split_image_objects:
        encoder.append(("image_encoder", enc_block))
    encoder += [("feature_embedding", _shape_linear(d, cfg.encode_dim_features, False)), ("norm", _shape_layer_norm(d)),
                ("encoder", [(str(i), enc_block) for i in range(cfg.encode_num_blocks)])]
    dec_block = [("self_attention", _shape_multihead(dd, cfg.decode_q_k_dim, cfg.decode_v_dim)),
                 ("encode_attention", _shape_multihead(dd, cfg.decode_q_k_dim, cfg.decode_v_dim)),
                 ("feed_forward", _shape_feed_forward(dd, cfg.decode_hidden_size))]
    decoder = [("word_embedding", [("weight", (cfg.num_vocab, cfg.dim_word_embedding))]),
               ("word_embedding_linear", _shape_linear(dd, cfg.dim_word_embedding, False)),
               ("position_embedding", [("pos_table", (1, cfg.max_length - 1, dd))]),          # registered buffer
               ("norm", _shape_layer_norm(dd))]
    if cfg.move_first_image_feature:
        decoder += _shape_feed_forward(dd, cfg.decode_hidden_size)      # the decoder's own FFN members, registered inline
    decoder.append(("decoder", [(str(i), dec_block) for i in range(cfg.decode_num_blocks)]))
    tree = [("encoder", encoder), ("decoder", decoder), ("classifer", _shape_linear(cfg.num_vocab, dd))]
    return dict(_walk("", tree))


def init_state_dict(cfg: OracleConfig, seed: int = 0) -> Dict[str, Tensor]:
    """Random init with the reference's DISTRIBUTIONS (SURVEY.md §8a 'Initialisation'); the
    exact random stream of the reference is not reproduced (parity runs share a state_dict)."""
    g = torch.Generator().manual_seed(seed)
    sd: Dict[str, Tensor] = {}
    for name, shape in param_shapes(cfg).items():
        if name.endswith("pos_table"):
            sd[name] = sinusoid_table(shape[1], shape[2])
        elif name.endswith("layer_norm.weight") or name.endswith("norm.weight"):
            sd[name] = torch.ones(shape)
        elif name.endswith("layer_norm.bias") or name.endswith("norm.bias"):
            sd[name] = torch.zeros(shape)
        elif name == "decoder.word_embedding.weight":
            w = torch.randn(shape, generator=g)
            w[cfg.pad_idx] = 0
            sd[name] = w
        elif name.endswith(".bias"):
            fan_in = {"position_wise_1.bias": None}.get(name, None)
            wshape = param_shapes(cfg)[name[:-4] + "weight"]
            bound = 1.0 / math.sqrt(wshape[1])
            sd[name] = (torch.rand(shape, generator=g) * 2 - 1) * bound
        elif any(name.endswith(s) for s in ("q_linear.weight", "k_linear.weight", "v_linear.weight")):
            std = math.sqrt(2.0 / (shape[0] + shape[1]))
            sd[name] = torch.randn(shape, generator=g) * std
        elif any(s in name for s in ("joint_linear", "position_wise", "classifer")):
            std = math.sqrt(2.0 / (shape[0] + shape[1]))  # xavier_normal
            sd[name] = torch.randn(shape, generator=g) * std
        else:  # default nn.Linear init: kaiming_uniform(a=sqrt(5)) == U(-1/sqrt(fan_in), 1/sqrt(fan_in))
            bound = 1.0 / math.sqrt(shape[1])
            sd[name] = (torch.rand(shape, generator=g) * 2 - 1) * bound
    return sd
