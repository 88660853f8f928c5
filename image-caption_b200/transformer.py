"""Drop-in `Transformer` (same constructor / forward / generate_caption_vector / beam_search
signatures and state_dict layout as core/TRANSFORMER/model.py:8-209 of the reference), executing on
libicap.so.  It is an nn.Module so the reference wrapper's `.to(DEVICE)`, `.parameters()`,
`.state_dict()`, `.load_state_dict()`, `.eval()` (core/models.py:63-68,110-113) keep working.

All parameters are views into ONE flat fp32 buffer (registration order == reference order), which
is what the fused Adam / gradient all-reduce operate on.
"""
from __future__ import annotations

import contextlib
import gc
import math
import os
from typing import List, Optional

import numpy as np
import torch
import torch.nn as nn

from .engine import BUFFER_NAMES, CaptionEngine, ModelConfig, RegionBatch, flat_offsets, param_layout
from ._native import IcapError


def _sinusoid_table(num_positions: int, dim: int) -> torch.Tensor:
    """PositionalEncoding._get_sinusoid_encoding_table (model.py:502-514): float64 numpy, then float32."""
    j = np.arange(dim)
    pos = np.arange(num_positions, dtype=np.float64)[:, None]
    table = pos / np.power(10000, 2 * (j // 2) / dim)[None, :]
    table[:, 0::2] = np.sin(table[:, 0::2])
    table[:, 1::2] = np.cos(table[:, 1::2])
    return torch.tensor(table, dtype=torch.float32).unsqueeze(0)


class _Namespace(nn.Module):
    """Empty container used to reproduce the reference's dotted parameter names."""


def _set_nested(root: nn.Module, dotted: str, value, is_buffer: bool) -> None:
    parts = dotted.split(".")
    mod = root
    for p in parts[:-1]:
        if not hasattr(mod, p):
            mod.add_module(p, _Namespace())
        mod = getattr(mod, p)
    if is_buffer:
        mod.register_buffer(parts[-1], value)
    else:
        mod.register_parameter(parts[-1], value)


@contextlib.contextmanager
def _graph_capture(graph: torch.cuda.CUDAGraph):
    """`torch.cuda.graph(graph)` with Python's cycle collector held off.  A model and its captured steps reference each
    other, so a dropped model lives until a collection; if that collection runs inside a capture, it destroys the
    model's CUDA graphs there, and destroying a graph while a stream captures invalidates the capture
    (cudaErrorStreamCaptureInvalidated).  torch does not collect before a capture, so dead models are collected here."""
    enabled = gc.isenabled()
    gc.collect()
    gc.disable()
    try:
        with torch.cuda.graph(graph):
            yield
    finally:
        if enabled:
            gc.enable()


def _check_tape(eng: CaptionEngine, gen: int) -> None:
    """The engine keeps ONE backward tape (the reference's train loop is forward -> backward -> step): a second recorded
    forward, a decode or a no_grad pass between a forward and its backward() replaces / drops it."""
    if eng.tape is None or eng.tape_gen != gen:
        raise IcapError("backward() of a stale forward: another forward / decode ran on this model since (the engine "
                        "keeps one tape -- call backward() right after the forward it belongs to)")


class _LossFn(torch.autograd.Function):
    """Lets `loss.backward()` (core/models.py:125) drive the explicit backward of the engine."""

    @staticmethod
    def forward(ctx, model, record, feats, pos, captions, *params):
        eng = model._engine()
        eng.training = model.training
        eng.shadow_fresh = False                       # an external optimizer may have stepped the weights
        f, p, c = eng.prepare_inputs(feats, pos, captions)
        logits, tgt, count2, dec = eng.forward_logits(f, p, c, record=record)
        out2 = eng.loss_from_logits(logits, tgt, count2, dec, record=record)
        ctx.model, ctx.out2, ctx.recorded, ctx.gen = model, out2, record, eng.tape_gen
        return out2[0].clone()

    @staticmethod
    def backward(ctx, grad_out):
        model, eng = ctx.model, ctx.model._engine()
        if not ctx.recorded:
            raise IcapError("backward() called on a forward that did not record (no_grad / frozen parameters)")
        _check_tape(eng, ctx.gen)
        params = [q for _, q in model.named_parameters()]
        fresh = all(q.grad is None for q in params)
        eng.backward(zero_grads=fresh)                 # existing .grad views => accumulate like autograd does
        from ._native import call
        call("icap_scale", eng.g32.data_ptr(), eng.n_flat, ctx.out2[1:2].data_ptr() if eng.cfg.focal else None,
             1.0, eng._s())
        if not (grad_out.numel() == 1 and float(grad_out) == 1.0):
            eng.g32.mul_(grad_out)
        for name, q in model.named_parameters():
            off = eng.offsets[name]
            q.grad = eng.g32[off:off + q.numel()].view_as(q)
        return (None,) * (5 + len(params))


class _LogitsFn(torch.autograd.Function):
    """Differentiable teacher-forced logits (PolicyNetwork.forward, model_RL.py:75-90): the loss is computed by the
    caller in PyTorch, its gradient w.r.t. the logits re-enters the engine's explicit backward here."""

    @staticmethod
    def forward(ctx, model, record, feats, pos, captions, *params):
        eng = model._engine()
        eng.training = model.training
        eng.shadow_fresh = False
        f, p, c = eng.prepare_inputs(feats, pos, captions)
        logits, tgt, count2, dec = eng.forward_logits(f, p, c, record=record)
        if record:
            eng._append_classifier_bwd(logits, dec)
        ctx.model, ctx.logits, ctx.recorded, ctx.gen = model, logits, record, eng.tape_gen
        B, T = c.shape[0], c.shape[1] - 1
        ctx.shape = (B, T, model.num_vocab)
        # a copy: the engine overwrites its logits buffer with d loss / d logits in the backward
        return logits[:, :model.num_vocab].to(torch.float32, copy=True).reshape(B, T, model.num_vocab)

    @staticmethod
    def backward(ctx, grad_out):
        model, eng = ctx.model, ctx.model._engine()
        if not ctx.recorded:
            raise IcapError("backward() called on a forward that did not record (no_grad / frozen parameters)")
        _check_tape(eng, ctx.gen)
        params = [q for _, q in model.named_parameters()]
        fresh = all(q.grad is None for q in params)
        eng.set_dlogits(ctx.logits, grad_out)
        eng.backward(zero_grads=fresh)
        for name, q in model.named_parameters():
            off = eng.offsets[name]
            q.grad = eng.g32[off:off + q.numel()].view_as(q)
        return (None,) * (5 + len(params))


class _SampleFn(torch.autograd.Function):
    """PolicyNetwork.sample (model_RL.py:93-97): log_softmax over the vocabulary + arg-max, one fused kernel; the
    log-probabilities stay differentiable (the self-critical loss gathers them, loss.py:145-158)."""

    @staticmethod
    def forward(ctx, output):
        from ._native import call
        if not output.is_cuda:
            raise IcapError("PolicyNetwork.sample runs on the GPU only (there is no CPU fallback)")
        x = output.detach().to(torch.float32).contiguous()
        B, T, V = x.shape
        logp = torch.empty_like(x)
        seq = torch.empty(B, T, dtype=torch.int64, device=x.device)
        call("icap_log_softmax_argmax", B * T, V, x.data_ptr(), V, logp.data_ptr(), V, seq.data_ptr(),
             torch.cuda.current_stream(x.device).cuda_stream)
        ctx.save_for_backward(logp)
        ctx.mark_non_differentiable(seq)
        return seq, logp

    @staticmethod
    def backward(ctx, _gseq, glogp):
        from ._native import call
        logp, = ctx.saved_tensors
        B, T, V = logp.shape
        g = glogp.to(torch.float32).contiguous()
        dx = torch.empty_like(logp)
        call("icap_log_softmax_bwd", B * T, V, logp.data_ptr(), V, g.data_ptr(), V, dx.data_ptr(), V,
             torch.cuda.current_stream(logp.device).cuda_stream)
        return dx


class Transformer(nn.Module):
    """Reference signature: model.py:10-36."""

    def __init__(self, num_vocab, max_length,
                 encode_dim_positions,
                 encode_dim_features,
                 device,
                 output_name,
                 encode_mask=False,
                 pad_idx=0,
                 dropout=0.2,

                 encode_input_size=512,
                 encode_q_k_dim=512,
                 encode_v_dim=512,
                 encode_hidden_size=2048,
                 encode_num_blocks=6,
                 encode_num_heads=8,

                 dim_word_embedding=512,
                 decode_input_size=512,
                 decode_q_k_dim=512,
                 decode_v_dim=512,
                 decode_hidden_size=2048,
                 decode_num_blocks=6,
                 decode_num_heads=8,

                 move_first_image_feature=False,
                 split_position=False,
                 split_image_objects=False):
        super().__init__()
        self.max_length = max_length
        self.device = device
        self.num_vocab = num_vocab
        self.pad_idx = pad_idx
        self.cfg = ModelConfig(
            num_vocab=num_vocab, max_length=max_length, encode_dim_positions=encode_dim_positions,
            encode_dim_features=encode_dim_features, output_name=output_name, encode_mask=encode_mask,
            pad_idx=pad_idx, dropout=dropout, encode_input_size=encode_input_size, encode_q_k_dim=encode_q_k_dim,
            encode_v_dim=encode_v_dim, encode_hidden_size=encode_hidden_size, encode_num_blocks=encode_num_blocks,
            encode_num_heads=encode_num_heads, dim_word_embedding=dim_word_embedding,
            decode_input_size=decode_input_size, decode_q_k_dim=decode_q_k_dim, decode_v_dim=decode_v_dim,
            decode_hidden_size=decode_hidden_size, decode_num_blocks=decode_num_blocks,
            decode_num_heads=decode_num_heads, move_first_image_feature=move_first_image_feature,
            split_position=split_position, split_image_objects=split_image_objects)
        # "bf16" (tcgen05 GEMMs) or "fp32" (parity mode); the constructor signature is the reference's,
        # so the switch lives in the environment / an attribute.
        self.precision = os.environ.get("ICAP_PRECISION", "bf16")
        self.log_domain_beam = False          # True = PolicyNetwork scoring (model_RL.py:72)
        self.last_gaps: Optional[torch.Tensor] = None
        self._shapes = param_layout(self.cfg)
        self._offsets, self._n_flat = flat_offsets(self._shapes)
        flat = torch.zeros(self._n_flat, dtype=torch.float32)
        self._flat = flat
        for name, shp in self._shapes.items():
            if name in BUFFER_NAMES:
                _set_nested(self, name, _sinusoid_table(shp[1], shp[2]), is_buffer=True)
            else:
                off = self._offsets[name]
                view = flat[off:off + math.prod(shp)].view(shp)
                _set_nested(self, name, nn.Parameter(view), is_buffer=False)
        self._init_parameters()
        self._eng: Optional[CaptionEngine] = None
        self._decode_graphs: dict = {}
        self._train_graphs: dict = {}

    # ------------------------------------------------------------------ init (SURVEY.md §8a "Initialisation")
    @torch.no_grad()
    def _init_parameters(self) -> None:
        for name, q in self.named_parameters():
            shp = q.shape
            if name.endswith("norm.weight"):
                q.fill_(1.0)
            elif name.endswith("norm.bias"):
                q.zero_()
            elif name == "decoder.word_embedding.weight":           # nn.Embedding: N(0,1), padding row zero
                q.normal_(0.0, 1.0)
                q[self.pad_idx].zero_()
            elif name.endswith(".bias"):                             # nn.Linear default bias
                fan_in = self._shapes[name[:-4] + "weight"][1]
                q.uniform_(-1.0 / math.sqrt(fan_in), 1.0 / math.sqrt(fan_in))
            elif name.endswith(("q_linear.weight", "k_linear.weight", "v_linear.weight")):   # modules.py:45-53
                q.normal_(0.0, math.sqrt(2.0 / (shp[0] + shp[1])))
            elif any(s in name for s in ("joint_linear", "position_wise", "classifer")):     # xavier_normal
                q.normal_(0.0, math.sqrt(2.0 / (shp[0] + shp[1])))
            else:                                                    # nn.Linear default: U(+-1/sqrt(fan_in))
                q.uniform_(-1.0 / math.sqrt(shp[1]), 1.0 / math.sqrt(shp[1]))

    # ------------------------------------------------------------------ flat storage upkeep
    def _apply(self, fn, *args, **kwargs):
        super()._apply(fn, *args, **kwargs)            # moves every parameter separately ...
        first = next(iter(self.parameters()))
        if (first.dtype == torch.float32 and first.device == self._flat.device
                and first.untyped_storage().data_ptr() == self._flat.untyped_storage().data_ptr()):
            return self                                # .to() of the device it already lives on: views, Adam state, graphs stay
        self._reflatten()                              # ... so re-pack them into one buffer
        return self

    @torch.no_grad()
    def _reflatten(self) -> None:
        params = dict(self.named_parameters())
        any_p = next(iter(params.values()))
        flat = torch.zeros(self._n_flat, dtype=torch.float32, device=any_p.device)
        for name, q in params.items():
            off = self._offsets[name]
            flat[off:off + q.numel()].copy_(q.detach().reshape(-1).to(torch.float32))
            q.data = flat[off:off + q.numel()].view(q.shape)
            q.grad = None
        self._flat = flat
        self._eng = None
        self._decode_graphs = {}
        self._train_graphs = {}
        if any_p.is_cuda:
            self.device = any_p.device

    def load_state_dict(self, state_dict, strict=True, **kw):
        out = super().load_state_dict(state_dict, strict=strict, **kw)     # in-place copies: views stay valid
        if self._eng is not None:
            self._eng.shadow_fresh = False
            self._eng.pos_table32.copy_(self.decoder.position_embedding.pos_table.reshape(self._eng.pos_table32.shape))
            self._eng.pos_table_act.copy_(self._eng.pos_table32)
        return out

    def set_precision(self, precision: str) -> "Transformer":
        assert precision in ("bf16", "fp32")
        if precision != self.precision:
            self.precision, self._eng = precision, None
            self._decode_graphs = {}
            self._train_graphs = {}
        return self

    def _engine(self) -> CaptionEngine:
        if not self._flat.is_cuda:
            raise IcapError("image-caption_b200 runs on sm_100a GPUs only: call model.to('cuda') first "
                            "(there is no CPU fallback)")
        if self._eng is None:
            self._eng = CaptionEngine(self.cfg, self._flat, self.decoder.position_embedding.pos_table, self.precision)
        return self._eng

    # ------------------------------------------------------------------ reference API
    def forward(self, object_features, position_features, target_caption):
        """model.py:79-98 -> {'loss': 0-d tensor}."""
        params = [q for _, q in self.named_parameters()]
        record = torch.is_grad_enabled() and any(q.requires_grad for q in params)   # grad mode is off inside apply()
        loss = _LossFn.apply(self, record, object_features, position_features, target_caption, *params)
        return {"loss": loss}

    @torch.no_grad()
    def logits(self, object_features, position_features, target_caption) -> torch.Tensor:
        """Teacher-forced logits [B, T, V] fp32 (== PolicyNetwork.forward, model_RL.py:75-90)."""
        eng = self._engine()
        eng.training = False
        f, p, c = eng.prepare_inputs(object_features, position_features, target_caption)
        lg, _, _, _ = eng.forward_logits(f, p, c, record=False)
        B, T = c.shape[0], c.shape[1] - 1
        return lg[:, :self.num_vocab].float().view(B, T, self.num_vocab)

    def _decode(self, f, p, beam_size: int, log_domain: bool, want_attention: bool, num_samples: int = 0,
                temperature: float = 1.0, seed: Optional[int] = None):
        """KV-cached decode of one batch; the whole fixed-trip-count loop (encoder + max_length-1 steps, ~2000
        launches) is ONE CUDA graph per (batch, regions, beam) shape -- per (batch, regions, samples, temperature) when
        sampling -- unless ICAP_DECODE_GRAPH=0.  seed (sampling): the value of the sampling counter for this call."""
        eng = self._engine()
        eng.shadow_fresh = False                       # an external optimizer may have stepped the fp32 weights
        sample_kw = dict(num_samples=int(num_samples), temperature=float(temperature)) if num_samples else {}
        if os.environ.get("ICAP_DECODE_GRAPH", "1") == "0":
            if seed is not None:
                eng.sample_dev.fill_(seed)
            return eng.decode(f, p, beam_size=beam_size, log_domain=log_domain, want_attention=want_attention,
                              want_gaps=not num_samples, **sample_kw)
        cache = f.cache if isinstance(f, RegionBatch) else None
        key = (f.shape[0], f.shape[1], int(beam_size), bool(log_domain), bool(want_attention), id(eng), id(cache),
               int(num_samples), float(temperature))
        gd = self._decode_graphs.get(key)
        if gd is None:
            if len(self._decode_graphs) >= 4:          # each graph owns its KV-cache pool: keep only a few shapes
                self._decode_graphs.pop(next(iter(self._decode_graphs)))
            gd = GraphedDecode(self, f.shape[0], f.shape[1], beam_size, log_domain=log_domain,
                               want_attention=want_attention, want_gaps=not num_samples, cache=cache, **sample_kw)
            self._decode_graphs[key] = gd
        return gd.run(f.idx, seed=seed) if cache is not None else gd.run(f, p, seed=seed)

    def generate_caption_vector(self, object_features, position_features):
        """model.py:101-132 -> (LongTensor [B, max_length+1], list of max_length-1 float32 arrays [B, R])."""
        with torch.no_grad():
            eng = self._engine()
            f, p, _ = eng.prepare_inputs(object_features, position_features)
            out = self._decode(f, p, 1, False, True)
            B = f.shape[0]
            ids = torch.zeros(B, self.max_length + 1, dtype=torch.long, device=eng.dev)
            ids[:, :self.max_length] = out["ids"].long()
            self.last_gaps = out["gaps"]
            att = out["attention"].cpu().numpy()                      # ONE device->host copy (reference: one per step)
            attention_list: List[np.ndarray] = [att[t] for t in range(att.shape[0])]
        return ids, attention_list

    def beam_search(self, object_features, position_features, beam_size=1):
        """model.py:135-200 -> LongTensor [B, max_length] (beam slot 0)."""
        with torch.no_grad():
            eng = self._engine()
            f, p, _ = eng.prepare_inputs(object_features, position_features)
            out = self._decode(f, p, int(beam_size), self.log_domain_beam, False)
            self.last_gaps = out["gaps"]
            return out["ids"].long().contiguous()

    def sample_captions(self, object_features, position_features, num_samples=1, temperature=1.0, seed=None):
        """num_samples captions per image drawn from the model: every token from softmax(logits / temperature) by the
        KV-cached decoder (icap_sample_tokens).  A caption ends at its first <END> (or <NULL>); the positions after it
        hold <NULL> with log-probability 0.  Inputs are tensors or a RegionBatch (position_features=None), as for
        beam_search.  seed (0 <= seed < 2**31) makes the call reproducible; without it every call advances the model's
        sampling counter and draws new captions.
        -> (ids LongTensor [B, num_samples, max_length] with <START> first,
            logp FloatTensor [B, num_samples, max_length - 1]: log_softmax(logits)[token] at temperature 1, the model's
            log-probability of each token, as a policy gradient needs it)."""
        n = int(num_samples)
        if not 1 <= n <= 16:
            raise ValueError(f"num_samples must be in [1, 16], got {num_samples}")
        temperature = float(temperature)
        if not (math.isfinite(temperature) and temperature > 0 and 1.0 / temperature < 3e38):   # 1 / tau is a float32
            raise ValueError(f"temperature must be finite and > 0, got {temperature}")
        if seed is not None and not 0 <= int(seed) < 2 ** 31:
            raise ValueError(f"seed must be in [0, 2**31), got {seed}")
        with torch.no_grad():
            eng = self._engine()
            f, p, _ = eng.prepare_inputs(object_features, position_features)
            out = self._decode(f, p, 1, False, False, num_samples=n, temperature=temperature,
                               seed=None if seed is None else int(seed))
            return out["ids"].long(), out["logp"].clone()

    def get_attention_key_pad_mask(self, k, q):
        """model.py:202-209 (host-visible helper kept for API parity; kernels build the mask in-register)."""
        assert k.size(0) == q.size(0)
        mask = torch.count_nonzero(k, dim=2).eq(0)
        return mask.unsqueeze(1).expand(k.size(0), q.size(1), k.size(1))

    # ------------------------------------------------------------------ optimizer state (resume; not in the reference)
    def optimizer_state_dict(self) -> dict:
        """Adam state of the fused step (exp_avg / exp_avg_sq over the flat buffer + step count).  The reference saves
        only model.state_dict() and cannot resume (models.py:62-63, SURVEY.md §5); `save()` keeps that format and this
        is stored next to it."""
        eng = self._engine()
        if eng.adam_m is None:
            return {"step": int(eng.step_dev), "exp_avg": None, "exp_avg_sq": None}
        return {"step": int(eng.step_dev), "exp_avg": eng.adam_m.detach().cpu().clone(),
                "exp_avg_sq": eng.adam_v.detach().cpu().clone()}

    def load_optimizer_state_dict(self, state: dict) -> None:
        eng = self._engine()
        eng.step_dev.fill_(int(state["step"]))
        if state.get("exp_avg") is None:
            eng.adam_m = eng.adam_v = None
            self._train_graphs = {}                    # captured steps point at the old moment buffers
            return
        assert state["exp_avg"].numel() == eng.n_flat, "optimizer state belongs to a different model configuration"
        if eng.adam_m is None:
            eng.adam_m = state["exp_avg"].to(eng.dev, torch.float32).clone()
            eng.adam_v = state["exp_avg_sq"].to(eng.dev, torch.float32).clone()
        else:                                          # in place: captured step graphs keep pointing at these buffers
            eng.adam_m.copy_(state["exp_avg"])
            eng.adam_v.copy_(state["exp_avg_sq"])

    # ------------------------------------------------------------------ fused training step
    def train_step_fused(self, object_features, position_features, target_caption, lr: float = 5e-4,
                         train_mode: Optional[bool] = None) -> torch.Tensor:
        """zero_grad + forward + backward + Adam in one stream-ordered launch sequence
        (core/models.py:115-126).  Returns the device loss (0-d view, no host sync)."""
        eng = self._engine()
        f, p, c = eng.prepare_inputs(object_features, position_features, target_caption)
        mode = self.training if train_mode is None else bool(train_mode)
        if os.environ.get("ICAP_TRAIN_GRAPH", "1") == "0":
            return eng.train_step(f, p, c, lr=lr, train_mode=mode)[0]
        # one CUDA graph per (batch, regions, caption length, lr, mode) shape: a replay costs one launch instead of
        # ~330 ctypes calls.  The returned loss is a view of the graph's static output (overwritten by the next step).
        cache = f.cache if isinstance(f, RegionBatch) else None
        key = (f.shape[0], f.shape[1], c.shape[1], float(lr), mode, id(eng), id(cache))
        gs = self._train_graphs.get(key)
        if gs is None:
            if len(self._train_graphs) >= 4:           # every graph owns its activation pool: keep only a few shapes
                self._train_graphs.pop(next(iter(self._train_graphs)))
            gs = GraphedTrainStep(self, f.shape[0], f.shape[1], c.shape[1], lr=lr, cache=cache, train_mode=mode)
            self._train_graphs[key] = gs
        gs.load(f.idx if cache is not None else f, p, c)
        return gs.step()


class PolicyNetwork(Transformer):
    """Drop-in for core/TRANSFORMER/model_RL.py::PolicyNetwork (the repo's shipped default CAPTION_MODEL,
    core/config.py:14): same Encoder / Decoder / classifer parameters, but `forward` returns the teacher-forced
    LOGITS [B, T, V] (differentiable: any PyTorch loss on top back-propagates through the CUDA path), `sample`
    is the argmax "sampler" of model_RL.py:93-97 and beam search scores with LogSoftmax (model_RL.py:72,157,182).
    The reward of SelfCriticNetwork is its injectable reward_fn (image_caption_b200.CaptionReward: CIDEr-D + BLEU-4 on
    the GPU)."""

    def __init__(self, num_vocab, max_length, encode_dim_positions, encode_dim_features, device, pad_idx=0, dropout=0.2,
                 encode_mask=False, encode_input_size=512, encode_q_k_dim=512, encode_v_dim=512, encode_hidden_size=2048,
                 encode_num_blocks=6, encode_num_heads=8, dim_word_embedding=512, decode_input_size=512,
                 decode_q_k_dim=512, decode_v_dim=512, decode_hidden_size=2048, decode_num_blocks=6, decode_num_heads=8,
                 move_first_image_feature=False, split_position=False, split_image_objects=False):
        super().__init__(num_vocab, max_length, encode_dim_positions, encode_dim_features, device, "RL_Transformer",
                         encode_mask=encode_mask, pad_idx=pad_idx, dropout=dropout, encode_input_size=encode_input_size,
                         encode_q_k_dim=encode_q_k_dim, encode_v_dim=encode_v_dim, encode_hidden_size=encode_hidden_size,
                         encode_num_blocks=encode_num_blocks, encode_num_heads=encode_num_heads,
                         dim_word_embedding=dim_word_embedding, decode_input_size=decode_input_size,
                         decode_q_k_dim=decode_q_k_dim, decode_v_dim=decode_v_dim, decode_hidden_size=decode_hidden_size,
                         decode_num_blocks=decode_num_blocks, decode_num_heads=decode_num_heads,
                         move_first_image_feature=move_first_image_feature, split_position=split_position,
                         split_image_objects=split_image_objects)
        self.log_domain_beam = True

    def forward(self, object_features, position_features, target_caption):
        """model_RL.py:75-90 -> logits [B, T, V] (fp32)."""
        params = [q for _, q in self.named_parameters()]
        record = torch.is_grad_enabled() and any(q.requires_grad for q in params)
        return _LogitsFn.apply(self, record, object_features, position_features, target_caption, *params)

    @staticmethod
    def sample(output):
        """model_RL.py:93-97 -> (sequence [B, T] int64, log_probs [B, T, V] fp32, differentiable)."""
        return _SampleFn.apply(output)


class GradBuckets:
    """Bucket schedule over the flat gradient buffer.  Gradients complete from the END of the buffer towards its
    start (reverse registration order); `on_done(lo)` is told, after every backward closure, the lowest offset
    that closure wrote, and answers with the slice [lo, hi) that may be all-reduced now (or None).  Every element
    is handed out exactly once; `flush()` returns the remaining prefix."""

    def __init__(self, total_elems: int, bucket_elems: int, tail_elems: Optional[int] = None,
                 tail_below: Optional[int] = None):
        self.prev_lo = int(total_elems)
        self.bucket_elems = int(bucket_elems)
        # The last slices of a step cannot hide behind anything (the backward is over): below offset `tail_below` the
        # bucket threshold drops to `tail_elems`, so that the final flush is a few MB instead of up to a whole bucket.
        self.tail_elems = int(tail_elems) if tail_elems else self.bucket_elems
        self.tail_below = int(tail_below) if tail_below else 0

    def on_done(self, lo: Optional[int]):
        if lo is None or lo >= self.prev_lo:
            return None
        need = self.tail_elems if lo < self.tail_below else self.bucket_elems
        if self.prev_lo - lo < need:
            return None
        out = (int(lo), self.prev_lo)
        self.prev_lo = int(lo)
        return out

    def flush(self):
        if self.prev_lo <= 0:
            return None
        out = (0, self.prev_lo)
        self.prev_lo = 0
        return out


class PeerReduce:
    """All-reduce of the flat gradient buffer over NVLink peer memory with libicap's own kernels (csrc/p2p.cu) instead of
    NCCL.  The gradient buffer and a few flag words are allocated as torch symmetric memory (CUDA VMM allocations that
    `rendezvous` maps into every rank of the group); the kernels get the peers' device pointers.  They need no shared
    memory, so they run beside the backward's persistent GEMMs."""

    def __init__(self, dist, eng: CaptionEngine):
        import ctypes
        import torch.distributed._symmetric_memory as symm_mem
        self.dist, self.rank, self.world = dist, dist.get_rank(), dist.get_world_size()
        assert self.world <= 8
        dev = eng.dev
        self.g32 = symm_mem.empty(eng.n_flat + 8, dtype=torch.float32, device=dev)
        self.flags = symm_mem.empty(64, dtype=torch.int32, device=dev)
        self._hg = symm_mem.rendezvous(self.g32, dist.group.WORLD)
        self._hf = symm_mem.rendezvous(self.flags, dist.group.WORLD)
        self.g32.zero_()
        self.flags.zero_()
        self.epoch = torch.zeros(1, dtype=torch.int32, device=dev)
        self.err = torch.zeros(1, dtype=torch.int32, device=dev)
        gp, fp = [int(x) for x in self._hg.buffer_ptrs], [int(x) for x in self._hf.buffer_ptrs]
        assert gp[self.rank] == self.g32.data_ptr() and len(gp) == self.world
        arr = ctypes.c_void_p * 8
        self._gp = arr(*(gp + [None] * (8 - self.world)))
        self._fp = arr(*(fp + [None] * (8 - self.world)))
        self.gp = ctypes.cast(self._gp, ctypes.c_void_p)
        self.fp = ctypes.cast(self._fp, ctypes.c_void_p)
        self.ctas = int(os.environ.get("ICAP_DP_PEER_CTAS", "148"))
        # NVSwitch multicast mapping of the gradient buffer (0 when the fabric has none): in-switch reduction
        self.mc = int(getattr(self._hg, "multicast_ptr", 0) or 0)
        self.use_nvls = self.mc != 0 and os.environ.get("ICAP_DP_PEER_NVLS", "1") != "0"
        torch.cuda.synchronize(dev)
        dist.barrier()                                   # every rank's flag words are zero before anyone signals

    def barrier(self, stream: int) -> None:
        from ._native import call
        call("icap_p2p_barrier", self.fp, self.rank, self.world, self.epoch.data_ptr(), self.err.data_ptr(), stream)

    def all_reduce(self, lo: int, hi: int, stream: int) -> None:
        """Reduce [lo, hi) on `stream`; the result may be read after ONE more barrier() (end of the step)."""
        from ._native import call
        self.barrier(stream)
        if self.use_nvls:
            call("icap_p2p_allreduce_nvls", self.mc, self.rank, self.world, lo, hi, self.ctas, stream)
            return
        call("icap_p2p_reduce_scatter", self.gp, self.rank, self.world, lo, hi, self.ctas, stream)
        self.barrier(stream)
        call("icap_p2p_all_gather", self.gp, self.rank, self.world, lo, hi, self.ctas, stream)

    def check(self) -> None:
        e = int(self.err)
        if e:
            raise IcapError(f"peer all-reduce: rank {e - 1} never reached a barrier (rank {self.rank} gave up after 2 s)")


class DataParallel:
    """Data parallelism by image (SURVEY.md §8e): one process per GPU, replicated weights and Adam state.
    Every rank back-propagates the SUM of its token losses (dlogits not divided by the local count); the flat
    gradient buffer carries the local non-pad token count in its tail slot, so the all-reduce(SUM) yields both
    the summed gradients and the global count, and Adam divides by it (gscale).  That reproduces the
    reference's global `mean over non-pad targets` exactly, whatever the per-rank token counts are.

    Overlap: gradients become final from the END of the flat buffer (classifier) towards its start (encoder
    embeddings) as the backward proceeds, so the buffer is reduced in `bucket_mb` slices, each launched on a
    communication stream as soon as its slice is complete (engine.bucket_hook) while the backward continues."""

    def __init__(self, model: "Transformer", dist, bucket_mb: Optional[float] = None, overlap: bool = True):
        self.dist = dist
        self.world = dist.get_world_size()
        if model.cfg.focal:
            # d focal / d ce depends on the GLOBAL mean CE; this protocol all-reduces gradients of the summed token
            # losses and the token count only.  Refuse instead of silently training with plain-CE gradients.
            raise IcapError("DataParallel does not support FocalLoss output names ('FocalLoss' in output_name)")
        eng = model._engine()
        eng.dp_unnormalized = True
        dist.broadcast(eng.p32, src=0)          # identical replicas
        eng.shadow_fresh = False
        self.eng = eng
        self.inv = torch.zeros(1, dtype=torch.float32, device=eng.dev)
        # Exchange back-end.  ICAP_DP_PEER=1: libicap's own NVLink peer-memory kernels (PeerReduce); 0: NCCL; unset: the
        # peer kernels when the fabric offers an NVSwitch multicast mapping of the gradient buffer (in-switch reduction),
        # NCCL otherwise.  Measured on 8 x B200 (profiles/r2_scale8_backends.log, r2_dp_ab_4gpu.log): 4.71 ms/step against NCCL's 5.02 (1 GPU 4.44);
        # on 2 GPUs both take 4.73.
        self.peer: Optional[PeerReduce] = None
        mode = os.environ.get("ICAP_DP_PEER", "auto")
        if mode != "0" and self.world <= 8 and eng.dev.type == "cuda" and dist.get_backend() == "nccl":
            try:
                peer = PeerReduce(dist, eng)
            except Exception as e:                       # no symmetric memory on this fabric / torch build
                if mode == "1":
                    raise
                peer = None
                if dist.get_rank() == 0:
                    print(f"[icap] peer-memory gradient exchange unavailable ({type(e).__name__}: {e}); using NCCL",
                          flush=True)
            # every rank takes the same branch: multicast_ptr is a property of the group's allocation
            if peer is not None and (mode == "1" or peer.use_nvls):
                self.peer = peer
                eng.g32 = peer.g32                       # the engine's gradient buffer IS the exported one
        if bucket_mb is None:
            bucket_mb = float(os.environ.get("ICAP_DP_BUCKET_MB", "16" if self.peer is not None else "48"))
        # SMs left to NCCL while the backward's persistent GEMMs run (0 = none reserved)
        reserve = int(os.environ.get("ICAP_DP_RESERVE_SMS", "0"))
        if reserve > 0:
            sms = torch.cuda.get_device_properties(eng.dev).multi_processor_count
            eng.bwd_gemm_sms = max(16, sms - reserve)
        self.bucket_elems = int(bucket_mb * (1 << 20) / 4)
        self.tail_elems = int(min(bucket_mb, float(os.environ.get("ICAP_DP_TAIL_MB", "8"))) * (1 << 20) / 4)
        self.overlap = overlap and os.environ.get("ICAP_DP_OVERLAP", "1") != "0"
        # Gradient exchange dtype (NCCL back-end only): fp32 (default) or, with ICAP_DP_GRAD_DTYPE=bf16, every bucket
        # rounded to bf16 into a staging buffer, all-reduced there and widened back (half the NVLink bytes; the token
        # count in the tail slot still travels in fp32).  Measured on 2 x B200: 4.736 vs 4.728 ms/step -- the exposed
        # 0.29 ms is not volume (profiles/r2_summary.md), so the exact fp32 exchange stays the default.
        want = "fp32" if self.peer is not None else os.environ.get("ICAP_DP_GRAD_DTYPE", "fp32")
        self.comm_bf16 = want == "bf16"
        self.g16 = torch.empty(eng.n_flat, dtype=torch.bfloat16, device=eng.dev) if self.comm_bf16 else None
        self.comm: Optional[torch.cuda.Stream] = None
        self.plan: Optional[GradBuckets] = None
        self.n_buckets = 0

    @staticmethod
    def allreduce_flat(dist, g32: torch.Tensor, n_flat: int) -> torch.Tensor:
        """In-place SUM all-reduce of [grads | count]; returns the view holding the global token count."""
        dist.all_reduce(g32, op=dist.ReduceOp.SUM)
        return g32[n_flat:n_flat + 1]

    def reduce(self, eng: CaptionEngine) -> None:
        if self.comm_bf16 or self.peer is not None:      # same exchange as the bucketed path, one slice
            if self.comm is None:
                self.comm = torch.cuda.Stream(device=eng.dev)
            self._fire((0, eng.g32.numel()))
            if self.peer is not None:
                with torch.cuda.stream(self.comm):
                    self.peer.barrier(torch.cuda.current_stream(eng.dev).cuda_stream)
            torch.cuda.current_stream(eng.dev).wait_stream(self.comm)
            return
        self.allreduce_flat(self.dist, eng.g32, eng.n_flat)

    # ---- bucketed, overlapped with the backward
    def begin(self, eng: CaptionEngine) -> None:
        """Call before forward_backward: arms the bucket hook."""
        if self.comm is None:
            self.comm = torch.cuda.Stream(device=eng.dev)
        self.plan = GradBuckets(eng.g32.numel(), self.bucket_elems, tail_elems=self.tail_elems,
                                tail_below=2 * self.bucket_elems)       # includes the token-count tail slot
        self.n_buckets = 0
        eng.bucket_hook = self._closure_done

    def _fire(self, sl) -> None:
        if sl is None:
            return
        eng = self.eng
        main = torch.cuda.current_stream(eng.dev)
        self.comm.wait_stream(main)
        if eng._bwd_side is not None:
            self.comm.wait_stream(eng._bwd_side)  # weight gradients are written by the wgrad side stream
        with torch.cuda.stream(self.comm):
            lo, hi = sl
            if self.peer is not None:
                self.peer.all_reduce(lo, hi, torch.cuda.current_stream(eng.dev).cuda_stream)
            elif not self.comm_bf16:
                self.dist.all_reduce(eng.g32[lo:hi], op=self.dist.ReduceOp.SUM)
            else:
                from ._native import call, F32, BF16
                n = eng.n_flat
                hg = min(hi, n)
                if hg > lo:
                    st = torch.cuda.current_stream(eng.dev).cuda_stream
                    call("icap_copy2d", eng.g32.data_ptr() + 4 * lo, F32, hg - lo, self.g16.data_ptr() + 2 * lo, BF16, hg - lo,
                         1, hg - lo, 0, st)
                    self.dist.all_reduce(self.g16[lo:hg], op=self.dist.ReduceOp.SUM)
                    call("icap_copy2d", self.g16.data_ptr() + 2 * lo, BF16, hg - lo, eng.g32.data_ptr() + 4 * lo, F32, hg - lo,
                         1, hg - lo, 0, st)
                if hi > n:
                    self.dist.all_reduce(eng.g32[max(lo, n):hi], op=self.dist.ReduceOp.SUM)
        self.n_buckets += 1

    def _closure_done(self, lo: Optional[int]) -> None:
        self._fire(self.plan.on_done(lo))

    def end(self, eng: CaptionEngine) -> None:
        """Call after forward_backward: reduces what is left and joins the communication stream."""
        eng.bucket_hook = None
        self._fire(self.plan.flush())
        if self.peer is not None:                        # nobody still reads a buffer that the next step zeroes
            with torch.cuda.stream(self.comm):
                self.peer.barrier(torch.cuda.current_stream(eng.dev).cuda_stream)
        torch.cuda.current_stream(eng.dev).wait_stream(self.comm)

    def finish(self, eng: CaptionEngine, lr: float) -> None:
        from ._native import call
        call("icap_reciprocal", eng.g32.data_ptr() + 4 * eng.n_flat, self.inv.data_ptr(), 1.0, eng._s())
        eng.adam_step(lr, gscale_dev=self.inv)

    def step_eager(self, eng: CaptionEngine, feats, pos, cap, lr: float, train_mode: bool = True) -> torch.Tensor:
        """One data-parallel train step without CUDA graphs."""
        if self.overlap:
            self.begin(eng)
            out2 = eng.forward_backward(feats, pos, cap, train_mode)
            self.end(eng)
        else:
            out2 = eng.forward_backward(feats, pos, cap, train_mode)
            self.reduce(eng)
        self.finish(eng, lr)
        return out2


class GraphedDecode:
    """The complete KV-cached greedy / beam / sampled decode of a fixed (batch, regions, beam) shape as ONE CUDA graph:
    encoder, cross-K/V projection, and all max_length-1 steps (the reference's loops have a fixed trip count and
    no EOS exit, model.py:114,169).  Replays cost one launch instead of ~2000 ctypes calls."""

    def __init__(self, model: Transformer, batch: int, regions: int, beam_size: int, log_domain: bool = False,
                 want_attention: bool = False, want_gaps: bool = False, cache=None, num_samples: int = 0,
                 temperature: float = 1.0):
        eng = model._engine()
        cfg = model.cfg
        self.eng = eng
        self.kw = dict(beam_size=int(beam_size), log_domain=log_domain, want_attention=want_attention,
                       want_gaps=want_gaps)
        self.sampling = num_samples > 0                # the graph ticks the sampling counter: replays draw new samples
        if self.sampling:
            self.kw.update(num_samples=int(num_samples), temperature=float(temperature))
        self.cache = cache
        if cache is not None:                          # inputs = image numbers into a device-resident RegionCache
            assert regions == cache.regions
            self.idx = torch.zeros(batch, dtype=torch.int64, device=eng.dev)
            self.feats, self.pos = RegionBatch(cache, self.idx), None
        else:
            self.feats = torch.zeros(batch, regions, cfg.encode_dim_features, device=eng.dev)
            self.pos = torch.zeros(batch, regions, cfg.encode_dim_positions, device=eng.dev)
            self.pos[:, :, 2:4] = 1.0                  # placeholder keeps every region "valid" during warm-up
        self.graph: Optional[torch.cuda.CUDAGraph] = None
        self.out = None
        self._streams: list = []

    def capture(self) -> None:
        eng = self.eng
        with torch.no_grad():
            counter0 = eng.sample_dev.clone() if self.sampling else None
            side = eng.warm_stream()
            side.wait_stream(torch.cuda.current_stream(eng.dev))
            with torch.cuda.stream(side):
                eng.decode(self.feats, self.pos, **self.kw)            # warm-up: function attributes, allocator
            torch.cuda.current_stream(eng.dev).wait_stream(side)
            if counter0 is not None:
                eng.sample_dev.copy_(counter0)                         # the warm-up does not count as a draw
            torch.cuda.synchronize(eng.dev)
            eng.refresh_shadow()
            self.graph = torch.cuda.CUDAGraph()
            # Images are independent (no collective, SURVEY.md 8e): optionally (ICAP_DECODE_STREAMS=n) the batch is cut
            # into n slices decoded on separate streams inside the one graph.  Measured on B200 (batch 512, beam 5):
            # no gain -- the per-step kernels do not overlap usefully -- so the default is one stream.
            B = self.feats.shape[0]
            nsplit = max(1, min(int(os.environ.get("ICAP_DECODE_STREAMS", "1")), B // 64 if B >= 128 else 1))
            if self.sampling:
                nsplit = 1                             # the uniforms are keyed by the row number within the whole batch
            while B % nsplit:
                nsplit -= 1
            with _graph_capture(self.graph):
                if nsplit == 1:
                    self.out = eng.decode(self.feats, self.pos, **self.kw)
                else:
                    main = torch.cuda.current_stream(eng.dev)
                    if len(self._streams) < nsplit:
                        self._streams += [torch.cuda.Stream(device=eng.dev) for _ in range(nsplit - len(self._streams))]
                    bs, outs = B // nsplit, []
                    for i in range(nsplit):
                        st = self._streams[i]
                        st.wait_stream(main)
                        with torch.cuda.stream(st):
                            sl = slice(i * bs, (i + 1) * bs)
                            outs.append(eng.decode(self.feats[sl], None if self.pos is None else self.pos[sl], **self.kw))
                    for i in range(nsplit):
                        main.wait_stream(self._streams[i])
                    self.out = {
                        "ids": torch.cat([o["ids"] for o in outs], dim=0),
                        "attention": torch.cat([o["attention"] for o in outs], dim=1) if outs[0]["attention"] is not None else None,
                        "gaps": torch.cat([o["gaps"] for o in outs], dim=1) if outs[0]["gaps"] is not None else None,
                    }

    def run(self, feats: torch.Tensor, pos: Optional[torch.Tensor] = None, seed: Optional[int] = None):
        """Returns the engine's output dict (static device tensors, overwritten by the next run).  With a region
        cache `feats` is the vector of image numbers.  seed (sampling): set the sampling counter first."""
        if self.graph is None:
            self.capture()
        if self.cache is not None:
            self.idx.copy_(feats, non_blocking=True)
        else:
            self.feats.copy_(feats, non_blocking=True)
            self.pos.copy_(pos, non_blocking=True)
        if seed is not None:
            self.eng.sample_dev.fill_(seed)
        self.eng.refresh_shadow()                      # weights may have been stepped since the capture
        self.graph.replay()
        return self.out


class GraphedTrainStep:
    """One CUDA graph holding H2D-staged inputs -> zero_grad -> forward -> backward -> Adam for a fixed
    batch shape.  Replays cost one launch; dropout masks change per replay because the kernels mix the
    device-side step counter into their seeds."""

    def __init__(self, model: Transformer, batch: int, regions: int, caption_len: int, lr: float = 5e-4,
                 warmup: int = 2, dp: Optional[DataParallel] = None, cache=None, train_mode: bool = True):
        eng = model._engine()
        self.dp = dp
        self.train_mode = bool(train_mode)             # False: dropout off (the reference's eval-mode arithmetic)
        self.graph2: Optional[torch.cuda.CUDAGraph] = None
        cfg = model.cfg
        dev = eng.dev
        self.model, self.eng, self.lr = model, eng, lr
        self.cache = cache
        if cache is not None:                          # inputs = image numbers into a device-resident RegionCache
            assert regions == cache.regions
            self.idx = torch.zeros(batch, dtype=torch.int64, device=dev)
            self.feats, self.pos = RegionBatch(cache, self.idx), None
        else:
            self.feats = torch.zeros(batch, regions, cfg.encode_dim_features, device=dev)
            self.pos = torch.zeros(batch, regions, cfg.encode_dim_positions, device=dev)
            self.pos[:, :, 2:4] = 1.0                  # placeholder keeps every region "valid" during capture
        self.cap = torch.ones(batch, caption_len, dtype=torch.int32, device=dev)
        self.graph: Optional[torch.cuda.CUDAGraph] = None
        self.out2: Optional[torch.Tensor] = None
        self.warmup = warmup
        self.launches_per_step = 0
        self.single_graph_dp = False

    def _one_step(self) -> torch.Tensor:
        return self.eng.train_step(self.feats, self.pos, self.cap, lr=self.lr, train_mode=self.train_mode)

    def load(self, feats: torch.Tensor, pos: Optional[torch.Tensor], cap: torch.Tensor) -> None:
        """Stage one batch (host or device tensors).  With a region cache: load(image_idx, None, captions)."""
        if self.cache is not None:
            assert pos is None
            self.idx.copy_(feats, non_blocking=True)
        else:
            self.feats.copy_(feats, non_blocking=True)
            self.pos.copy_(pos, non_blocking=True)
        self.cap.copy_(cap, non_blocking=True)

    def capture(self) -> None:
        """Capture with whatever is currently staged in the input buffers (call load() first)."""
        from . import _native
        eng = self.eng
        # warm-up on a side stream (allocator + function attributes), then roll the optimizer state back
        p0, step0 = eng.p32.clone(), eng.step_dev.clone()
        m0 = eng.adam_m.clone() if eng.adam_m is not None else None       # a capture in the middle of a training run
        v0 = eng.adam_v.clone() if eng.adam_v is not None else None       # must not disturb the optimizer state
        side = eng.warm_stream()
        side.wait_stream(torch.cuda.current_stream(eng.dev))
        with torch.cuda.stream(side):
            for _ in range(self.warmup):
                if self.dp is None:
                    self._one_step()
                else:
                    self.dp.step_eager(eng, self.feats, self.pos, self.cap, self.lr)
        torch.cuda.current_stream(eng.dev).wait_stream(side)
        eng.p32.copy_(p0)
        eng.step_dev.copy_(step0)
        if m0 is None:
            eng.adam_m.zero_()
            eng.adam_v.zero_()
        else:
            eng.adam_m.copy_(m0)
            eng.adam_v.copy_(v0)
        del p0, m0, v0
        eng.shadow_fresh = False
        eng.refresh_shadow()
        torch.cuda.synchronize(eng.dev)
        self.graph = torch.cuda.CUDAGraph()
        n0 = _native.launch_count
        if self.dp is None:
            with _graph_capture(self.graph):
                self.out2 = self._one_step()
        elif self.dp.overlap:
            # ONE graph: forward, backward with the bucketed NCCL all-reduces on the communication stream, Adam
            try:
                with _graph_capture(self.graph):
                    self.out2 = self.dp.step_eager(eng, self.feats, self.pos, self.cap, self.lr)
                self.single_graph_dp = True
            except Exception as exc:     # NCCL not capturable in this build: fall back to the split graphs below
                import warnings
                warnings.warn(f"capturing NCCL all-reduces failed ({exc!r}); using eager all-reduce between two graphs")
                eng.bucket_hook = None
                self.dp.overlap = False
                torch.cuda.synchronize(eng.dev)
                self.graph = torch.cuda.CUDAGraph()
        if self.dp is not None and not self.dp.overlap:
            # graph 1: zero_grad/forward/backward ; NCCL all-reduce (eager) ; graph 2: 1/count + Adam
            with _graph_capture(self.graph):
                self.out2 = eng.forward_backward(self.feats, self.pos, self.cap)
            self.graph2 = torch.cuda.CUDAGraph()
            with _graph_capture(self.graph2):
                self.dp.finish(eng, self.lr)
        self.launches_per_step = _native.launch_count - n0

    def step(self) -> torch.Tensor:
        if self.graph is None:
            self.capture()
        self.eng.refresh_shadow()                      # fp32 weights changed outside (load_state_dict, another optimizer)
        self.graph.replay()
        if self.graph2 is not None:
            self.dp.reduce(self.eng)
            self.graph2.replay()
        self.eng.shadow_fresh = True                   # the fused Adam wrote the bf16 shadow
        return self.out2[0]
