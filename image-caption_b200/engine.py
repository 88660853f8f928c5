"""Kernel orchestration for the caption Transformer on one B200.

`CaptionEngine` owns the flat parameter / gradient / optimizer buffers and turns one call of the
reference's hot path (core/TRANSFORMER/model.py: Transformer.forward, generate_caption_vector,
beam_search; core/models.py:115-126 train_step) into a sequence of libicap.so launches on the
current CUDA stream.  PyTorch is used only as the device allocator / stream owner; every FLOP and
every byte moved on the device goes through the C ABI (include/icap.h).  There is no CPU path.

Two arithmetic modes:
  * "bf16": activations + weight shadow in bf16, tcgen05 GEMMs, fp32 statistics / softmax / loss /
            master weights / Adam.
  * "fp32": everything fp32 with true-fp32 SIMT GEMMs (parity mode, 1e-4 relative vs the reference).

Backward is explicit (no autograd): each forward block appends a closure to a tape; gradients of
multi-consumer activations are carried as lists and summed inside the fused LayerNorm backward.
"""
from __future__ import annotations

import math
import os
from dataclasses import dataclass
from typing import Callable, Dict, List, Optional, Tuple

import torch

from . import _native as N
from ._native import BF16, F32, call


@dataclass
class ModelConfig:
    """Constructor arguments of the reference Transformer (model.py:10-36)."""
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

    @property
    def focal(self) -> bool:
        return self.output_name.find("FocalLoss") != -1      # model.py:73

    @property
    def T(self) -> int:                                        # decoder positions (model.py:383)
        return self.max_length - 1


ATTN_DROPOUT = 0.1      # ScaledDotProductAttention default, never overridden (modules.py:8,55-56)
LN_EPS = 1e-6
END_IDX = 2             # <END> of the vocabulary (preprocess.py:303); sampled rows stop there


def param_layout(cfg: ModelConfig) -> "Dict[str, Tuple[int, ...]]":
    """Parameter/buffer shapes in the reference's registration order (== state_dict order)."""
    d, F_, E = cfg.encode_input_size, cfg.encode_hidden_size, cfg.dim_word_embedding
    shapes: Dict[str, Tuple[int, ...]] = {}

    def mha(p, d_in, dk, dv):
        shapes[p + ".q_linear.weight"] = (dk, d_in)
        shapes[p + ".k_linear.weight"] = (dk, d_in)
        shapes[p + ".v_linear.weight"] = (dv, d_in)
        shapes[p + ".layer_norm.weight"] = (d_in,)
        shapes[p + ".layer_norm.bias"] = (d_in,)
        shapes[p + ".joint_linear.weight"] = (d_in, dv)

    def ffn(p, d_in, hid):
        shapes[p + ".position_wise_1.weight"] = (hid, d_in)
        shapes[p + ".position_wise_1.bias"] = (hid,)
        shapes[p + ".position_wise_2.weight"] = (d_in, hid)
        shapes[p + ".position_wise_2.bias"] = (d_in,)
        shapes[p + ".layer_norm.weight"] = (d_in,)
        shapes[p + ".layer_norm.bias"] = (d_in,)

    if cfg.split_position:
        shapes["encoder.object_embedding.weight"] = (d, cfg.encode_dim_positions - 4)
        shapes["encoder.position_embedding.weight"] = (d, 4)
    else:
        shapes["encoder.position_embedding.weight"] = (d, cfg.encode_dim_positions)
    if cfg.split_image_objects:
        mha("encoder.image_encoder.multihead_attention", d, cfg.encode_q_k_dim, cfg.encode_v_dim)
        ffn("encoder.image_encoder.feed_forward", d, F_)
    shapes["encoder.feature_embedding.weight"] = (d, cfg.encode_dim_features)
    shapes["encoder.norm.weight"] = (d,)
    shapes["encoder.norm.bias"] = (d,)
    for i in range(cfg.encode_num_blocks):
        mha(f"encoder.encoder.{i}.multihead_attention", d, cfg.encode_q_k_dim, cfg.encode_v_dim)
        ffn(f"encoder.encoder.{i}.feed_forward", d, F_)
    dd, dF = cfg.decode_input_size, cfg.decode_hidden_size
    shapes["decoder.word_embedding.weight"] = (cfg.num_vocab, E)
    shapes["decoder.word_embedding_linear.weight"] = (dd, E)
    shapes["decoder.position_embedding.pos_table"] = (1, cfg.max_length - 1, dd)      # buffer
    shapes["decoder.norm.weight"] = (dd,)
    shapes["decoder.norm.bias"] = (dd,)
    if cfg.move_first_image_feature:
        shapes["decoder.position_wise_1.weight"] = (dF, dd)
        shapes["decoder.position_wise_1.bias"] = (dF,)
        shapes["decoder.position_wise_2.weight"] = (dd, dF)
        shapes["decoder.position_wise_2.bias"] = (dd,)
        shapes["decoder.layer_norm.weight"] = (dd,)
        shapes["decoder.layer_norm.bias"] = (dd,)
    for i in range(cfg.decode_num_blocks):
        mha(f"decoder.decoder.{i}.self_attention", dd, cfg.decode_q_k_dim, cfg.decode_v_dim)
        mha(f"decoder.decoder.{i}.encode_attention", dd, cfg.decode_q_k_dim, cfg.decode_v_dim)
        ffn(f"decoder.decoder.{i}.feed_forward", dd, dF)
    shapes["classifer.weight"] = (cfg.num_vocab, dd)
    shapes["classifer.bias"] = (cfg.num_vocab,)
    return shapes


BUFFER_NAMES = ("decoder.position_embedding.pos_table",)


def flat_offsets(shapes: "Dict[str, Tuple[int, ...]]") -> "Tuple[Dict[str, int], int]":
    """Offsets (in elements) of every PARAMETER in the flat buffers; 8-element aligned so that bf16
    views are 16-byte aligned for TMA and fp32 views for float4."""
    off, offsets = 0, {}
    for name, shp in shapes.items():
        if name in BUFFER_NAMES:
            continue
        offsets[name] = off
        off += (math.prod(shp) + 7) // 8 * 8
    return offsets, off


def _ptr(t: Optional[torch.Tensor]) -> Optional[int]:
    return None if t is None else t.data_ptr()


class RegionBatch:
    """A batch named by image numbers into a device-resident `feed.RegionCache` (SURVEY.md 8f #2).  Accepted wherever
    the engine takes `feats` (with pos=None): the packed encoder input is gathered on the device inside encode()."""

    def __init__(self, cache, idx: torch.Tensor):
        assert idx.dim() == 1 and idx.dtype in (torch.int32, torch.int64)
        self.cache, self.idx = cache, idx

    @property
    def shape(self):
        return (self.idx.shape[0], self.cache.regions, self.cache.dim_features)

    def __getitem__(self, sl):
        return RegionBatch(self.cache, self.idx[sl])


class CaptionEngine:
    def __init__(self, cfg: ModelConfig, flat_params: torch.Tensor, pos_table: torch.Tensor, precision: str = "bf16"):
        assert flat_params.is_cuda and flat_params.dtype == torch.float32
        assert precision in ("bf16", "fp32")
        self.cfg = cfg
        self.dev = flat_params.device
        call("icap_sm_check", self.dev.index if self.dev.index is not None else torch.cuda.current_device())
        self.precision = precision
        self.act = BF16 if precision == "bf16" else F32
        self.tdt = torch.bfloat16 if precision == "bf16" else torch.float32
        self.shapes = param_layout(cfg)
        self.offsets, self.n_flat = flat_offsets(self.shapes)
        assert flat_params.numel() == self.n_flat
        self.p32 = flat_params
        self.g32 = torch.zeros(self.n_flat + 8, dtype=torch.float32, device=self.dev)   # tail slot: DP token count
        self.one = torch.ones(1, dtype=torch.float32, device=self.dev)
        self.dp_unnormalized = False     # data parallel: dlogits are NOT divided by the local token count
        self._prof = None
        self._gemm_log: Optional[List[tuple]] = None     # bench: argument tuples of every GEMM launch of a step
        # backward: weight-gradient GEMMs run on a second stream, concurrently with the dgrad / LayerNorm /
        # attention chain that does not depend on them (joined before the optimizer step)
        self.wgrad_side_stream = os.environ.get("ICAP_WGRAD_STREAM", "1") != "0"
        call("icap_set_pdl", 1 if os.environ.get("ICAP_PDL", "1") == "1" else 0)
        self._side: Optional[torch.cuda.Stream] = None
        self._warm: Optional[torch.cuda.Stream] = None       # warm-up stream of the graph captures (see warm_stream)
        self._bwd_side: Optional[torch.cuda.Stream] = None
        # cross-attention K|V projections of all decoder layers (forward) and their dgrad into the encoder-output
        # gradient (backward) depend only on the encoder output: launched on the side stream
        self.xkv_side = os.environ.get("ICAP_XKV_SIDE", "1") != "0"
        # projection + dropout + residual + LayerNorm as one cluster kernel: 0 never, 1 inference passes, 2 training too
        # (measured on B200: beam-5 decode 17.0 -> 15.8 ms, training step 4.53 -> 4.44 ms)
        self.gemm_ln_mode = int(os.environ.get("ICAP_GEMM_LN", "2"))
        self.p16 = torch.empty(self.n_flat, dtype=torch.bfloat16, device=self.dev) if precision == "bf16" else None
        self.shadow_fresh = False
        self.adam_m: Optional[torch.Tensor] = None
        self.adam_v: Optional[torch.Tensor] = None
        self.step_dev = torch.zeros(1, dtype=torch.int32, device=self.dev)
        # sampled decoding: its own counter (neither the dropout masks nor Adam's step see it) and base seed
        self.sample_dev = torch.zeros(1, dtype=torch.int32, device=self.dev)
        self.sample_seed = 0x243F6A8885A308D3
        self.pos_table32 = pos_table.reshape(-1, pos_table.shape[-1]).contiguous()
        self.pos_table_act = self.pos_table32.to(self.tdt)
        self.base_seed = 0x1234ABCD
        self.tape: Optional[List[Callable[[], None]]] = None
        self.tape_gen = 0                # bumped by every recorded forward: autograd wrappers check they run THEIR tape
        self.gr: Dict[int, List[torch.Tensor]] = {}
        self.keep: List[torch.Tensor] = []
        self.training = False
        self._site = 0
        self._stream = 0
        # data parallel: called after every backward closure with the lowest flat offset it wrote (or None);
        # gradients complete from the END of the flat buffer towards its start (reverse registration order)
        self.bucket_hook: Optional[Callable[[Optional[int]], None]] = None
        # data parallel: persistent-GEMM grid width during the backward (None = all SMs); the SMs left over run the
        # NCCL all-reduce kernels of the gradient buckets (DataParallel sets it)
        self.bwd_gemm_sms: Optional[int] = None
        for k in ("encode_q_k_dim", "encode_v_dim", "decode_q_k_dim", "decode_v_dim"):
            assert getattr(cfg, k) % 8 == 0, f"{k} must be a multiple of 8"
        assert cfg.encode_input_size == cfg.decode_input_size, \
            "cross-attention reads encoder rows with decoder projections: widths must match (as in the reference)"

    def warm_stream(self) -> torch.cuda.Stream:
        """ONE stream for the eager warm-up pass that precedes every graph capture.  The caching allocator keeps freed
        blocks per stream: a fresh stream per capture would strand ~2 GB of cached blocks each time."""
        if self._warm is None:
            self._warm = torch.cuda.Stream(device=self.dev)
        return self._warm

    # ------------------------------------------------------------------ parameter views
    def w(self, name: str, rows: Optional[int] = None, cols: Optional[int] = None):
        """(pointer to the GEMM-dtype copy of a weight, numel offset) for kernels."""
        base = self.p16 if self.precision == "bf16" else self.p32
        return base.data_ptr() + self.offsets[name] * base.element_size()

    def p(self, name: str) -> int:      # fp32 master pointer (LN affine, biases)
        return self.p32.data_ptr() + self.offsets[name] * 4

    def g(self, name: str) -> int:      # fp32 gradient pointer
        return self.g32.data_ptr() + self.offsets[name] * 4

    def refresh_shadow(self) -> None:
        if self.precision == "bf16" and not self.shadow_fresh:
            call("icap_copy2d", self.p32.data_ptr(), F32, self.n_flat, self.p16.data_ptr(), BF16, self.n_flat,
                 1, self.n_flat, 0, self._s())
            self.shadow_fresh = True

    # ------------------------------------------------------------------ small helpers
    def _s(self) -> int:
        return torch.cuda.current_stream(self.dev).cuda_stream

    def new(self, *shape, dtype=None, zero=False) -> torch.Tensor:
        dt = self.tdt if dtype is None else dtype
        t = (torch.zeros if zero else torch.empty)(*shape, dtype=dt, device=self.dev)
        if self.tape is not None:
            self.keep.append(t)
        return t

    def _seed(self) -> int:
        self._site += 1
        return (self.base_seed + 0x9E3779B1 * self._site) & 0xFFFFFFFFFFFFFFFF

    def add_grad(self, x: torch.Tensor, g: torch.Tensor) -> None:
        self.gr.setdefault(id(x), []).append(g)

    def pop_grads(self, x: torch.Tensor) -> List[torch.Tensor]:
        gs = self.gr.pop(id(x), [])
        if len(gs) > 2:      # fold extras so the fused LN backward sees at most two
            acc = gs[1]
            for extra in gs[2:]:
                call("icap_copy2d", extra.data_ptr(), self.act, extra.shape[-1], acc.data_ptr(), self.act,
                     acc.shape[-1], extra.shape[0], extra.shape[-1], 1, self._s())
            gs = gs[:2]
        return gs

    # ------------------------------------------------------------------ primitive launches
    def gemm(self, a: torch.Tensor, a_kmajor: bool, b_ptr: int, ldb: int, b_kmajor: bool, M: int, Nn: int, K: int,
             out: torch.Tensor, ldc: Optional[int] = None, bias: Optional[int] = None, epi: int = 0,
             aux: Optional[torch.Tensor] = None, accumulate: bool = False, split_k: int = 1,
             lda: Optional[int] = None, a_ptr: Optional[int] = None, c_ptr: Optional[int] = None,
             c_dtype: Optional[int] = None, side: bool = False, b_static: bool = False) -> None:
        """b_static: B (and bias) are model weights that the kernel launched just before does not write -- the
        small-footprint kernel may then fetch them before its grid dependency resolves (ICAP_EPI_B_STATIC)."""
        ab = BF16 if self.precision == "bf16" else F32
        if b_static:
            epi |= N.EPI_B_STATIC
        if c_dtype is None:
            c_dtype = F32 if out.dtype == torch.float32 else BF16
        args = (ab, int(a_kmajor), int(b_kmajor), M, Nn, K,
                a.data_ptr() if a_ptr is None else a_ptr, a.shape[-1] if lda is None else lda, b_ptr, ldb,
                out.data_ptr() if c_ptr is None else c_ptr, (out.shape[-1] if ldc is None else ldc), c_dtype,
                bias, epi, _ptr(aux), (aux.shape[-1] if aux is not None else 0), int(accumulate), split_k)
        if self._gemm_log is not None:
            self._gemm_log.append(args)
        if side and self._bwd_side is not None:
            self.side_call("icap_gemm", *args)       # off the critical path: backward side stream
            return
        ev = self._prof_begin()
        call("icap_gemm", *args, self._s())
        self._prof_end(ev, 2.0 * M * Nn * K)

    def wgrad(self, dy: torch.Tensor, x: torch.Tensor, g_ptr: int, Nout: int, Kin: int, rows: int,
              ld_dy: Optional[int] = None, dy_ptr: Optional[int] = None, ldg: Optional[int] = None,
              x_ptr: Optional[int] = None, ldx: Optional[int] = None, side_ok: bool = True) -> None:
        """dW[Nout,Kin] += dy[rows,Nout]^T x[rows,Kin]  (fp32, split-K over rows so the grid fills the GPU)."""
        ab = BF16 if self.precision == "bf16" else F32
        if ab == BF16:
            split = 0           # automatic: the persistent tcgen05 kernel picks tile width + split to fill the SMs
        else:
            tiles = ((Nout + 127) // 128) * ((Kin + 127) // 128)
            split = max(1, min(32, (148 * 2) // max(1, tiles), (rows + 511) // 512))
        args = (ab, 0, 0, Nout, Kin, rows, dy.data_ptr() if dy_ptr is None else dy_ptr,
                dy.shape[-1] if ld_dy is None else ld_dy, x.data_ptr() if x_ptr is None else x_ptr,
                x.shape[-1] if ldx is None else ldx, g_ptr, Kin if ldg is None else ldg,
                F32, None, 0, None, 0, 1, split)
        if self._gemm_log is not None:
            self._gemm_log.append(args)
        if self._bwd_side is not None and side_ok:
            # dy and x stay allocated until the end of backward (self.keep), so the side stream may read them late
            self.side_call("icap_gemm", *args)
            return
        ev = self._prof_begin()
        call("icap_gemm", *args, self._s())
        self._prof_end(ev, 2.0 * Nout * Kin * rows)

    def _prof_begin(self):
        if self._prof is None:
            return None
        e = torch.cuda.Event(enable_timing=True)
        e.record()
        return e

    def _prof_end(self, e0, flops: float) -> None:
        if e0 is None:
            return
        e1 = torch.cuda.Event(enable_timing=True)
        e1.record()
        self._prof.append((e0, e1, flops))

    def profile_gemms(self, fn) -> "List[Tuple[float, float]]":
        """Run fn() eagerly with a CUDA-event pair around every GEMM launch; returns [(ms, flops)]."""
        self._prof = []
        try:
            fn()
            torch.cuda.synchronize(self.dev)
            return [(a.elapsed_time(b), fl) for a, b, fl in self._prof]
        finally:
            self._prof = None

    def record_gemms(self, fn) -> "List[tuple]":
        """Run fn() and return the icap_gemm argument tuple of every GEMM it launched (bench: the GEMM-only graph)."""
        self._gemm_log = []
        try:
            fn()
            return self._gemm_log
        finally:
            self._gemm_log = None

    def replay_gemms(self, log: "List[tuple]") -> float:
        """Re-launch recorded GEMMs on the current stream (timing only: outputs land in recycled activation
        memory); returns their total FLOPs."""
        for args in log:
            call("icap_gemm", *args, self._s())
        return sum(2.0 * a[3] * a[4] * a[5] for a in log)

    def add_ln(self, a: torch.Tensor, res: Optional[torch.Tensor], res_rows: int, norm: str,
               rowscale: Optional[torch.Tensor], p_drop: float):
        M, d = a.shape
        y = self.new(M, d)
        rec = self.tape is not None
        mean = self.new(M, dtype=torch.float32) if rec else None
        rstd = self.new(M, dtype=torch.float32) if rec else None
        seed = self._seed()
        p = p_drop if self.training else 0.0
        call("icap_add_ln_fwd", F32 if a.dtype == torch.float32 else BF16, self.act, M, d, a.data_ptr(), _ptr(res),
             res_rows, self.p(norm + ".weight"), self.p(norm + ".bias"), _ptr(rowscale), y.data_ptr(), _ptr(mean),
             _ptr(rstd), int(rec), p, seed, self.step_dev.data_ptr(), LN_EPS, self._s())
        return y, mean, rstd, seed, p

    def proj_add_ln(self, a: torch.Tensor, w_name: str, K: int, bias: Optional[int], res: torch.Tensor, norm: str,
                    rowscale: Optional[torch.Tensor], p_drop: float):
        """LayerNorm(dropout(a . W^T + bias) + res) [* rowscale]  (modules.py:86-90,117-120).  Returns
        (y, s, mean, rstd, seed, p) with `s` the pre-norm sum the backward reads.  bf16 mode and d in
        {128,256,512,1024}: ONE cluster kernel (icap_gemm_ln, statistics exchanged through DSMEM) when enabled
        (ICAP_GEMM_LN: 0 = never, 1 = inference passes, 2 = training too); otherwise icap_gemm + icap_add_ln_fwd."""
        M, d = a.shape[0], res.shape[1]
        rec = self.tape is not None
        fused = (self.precision == "bf16" and d in (128, 256, 512, 1024) and K % 8 == 0 and self._prof is None
                 and (self.gemm_ln_mode == 2 or (self.gemm_ln_mode == 1 and not rec)))
        if not fused:
            o = self.new(M, d)
            self.gemm(a, True, self.w(w_name), K, True, M, d, K, o, bias=bias)
            y, mean, rstd, seed, p = self.add_ln(o, res, M, norm, rowscale, p_drop)
            return y, o, mean, rstd, seed, p
        y = self.new(M, d)
        ssum = self.new(M, d) if rec else None
        mean = self.new(M, dtype=torch.float32) if rec else None
        rstd = self.new(M, dtype=torch.float32) if rec else None
        seed = self._seed()
        p = p_drop if self.training else 0.0
        call("icap_gemm_ln", M, d, K, a.data_ptr(), a.shape[1], self.w(w_name), K, bias, res.data_ptr(), d,
             self.p(norm + ".weight"), self.p(norm + ".bias"), _ptr(rowscale), y.data_ptr(), d, _ptr(ssum), d,
             _ptr(mean), _ptr(rstd), LN_EPS, p, seed, self.step_dev.data_ptr(), self._s())
        return y, ssum, mean, rstd, seed, p

    def ln_bwd(self, y: torch.Tensor, s: torch.Tensor, mean, rstd, norm: str, rowscale, p: float, seed: int,
               dbias2: Optional[int] = None):
        """Returns (ds, da): gradient for the residual input and for the GEMM-branch input."""
        gs = self.pop_grads(y)
        assert gs, "activation without gradient"
        M, d = s.shape
        ds = self.new(M, d)
        da = self.new(M, d) if p > 0 else None
        dy2 = _ptr(gs[1]) if len(gs) > 1 else None
        if self._bwd_side is None:
            call("icap_add_ln_bwd", self.act, M, d, gs[0].data_ptr(), dy2, s.data_ptr(), mean.data_ptr(), rstd.data_ptr(),
                 self.p(norm + ".weight"), _ptr(rowscale), ds.data_ptr(), _ptr(da), self.g(norm + ".weight"),
                 self.g(norm + ".bias"), dbias2, p, seed, self.step_dev.data_ptr(), self._s())
        else:
            # ds / da on the main stream (the dgrad chain waits for them); the parameter-gradient column sums
            # (dgamma, dbeta, bias of the producing GEMM) only feed the optimizer: side stream
            call("icap_add_ln_bwd_rows", self.act, M, d, gs[0].data_ptr(), dy2, s.data_ptr(), mean.data_ptr(),
                 rstd.data_ptr(), self.p(norm + ".weight"), _ptr(rowscale), ds.data_ptr(), _ptr(da), p, seed,
                 self.step_dev.data_ptr(), self._s())
            self.side_call("icap_add_ln_bwd_params", self.act, M, d, gs[0].data_ptr(), dy2, s.data_ptr(), mean.data_ptr(),
                           rstd.data_ptr(), _ptr(rowscale), ds.data_ptr(), _ptr(da), self.g(norm + ".weight"),
                           self.g(norm + ".bias"), dbias2)
        return ds, (da if da is not None else ds)

    def side_call(self, name: str, *args) -> None:
        """Launch a kernel whose results only feed the optimizer on the backward side stream (after everything
        enqueued on the main stream so far); same stream when the side stream is off.  The stream is appended."""
        if self._bwd_side is None:
            call(name, *args, self._s())
            return
        main = torch.cuda.current_stream(self.dev)
        ev = torch.cuda.Event()
        ev.record(main)
        self._bwd_side.wait_event(ev)
        with torch.cuda.stream(self._bwd_side):
            call(name, *args, self._s())

    # ------------------------------------------------------------------ blocks
    def mha_block(self, prefix: str, xq: torch.Tensor, xkv: torch.Tensor, B: int, Lq: int, Lk: int, H: int,
                  dk_tot: int, dv_tot: int, kvalid: Optional[torch.Tensor], causal: bool,
                  attn_mean: Optional[torch.Tensor] = None, kv_pre=None, report_lo: bool = True) -> torch.Tensor:
        """MultiHeadAttention.forward (modules.py:67-92) with q = xq, k = v = xkv.
        kv_pre = (tensor, event): the packed K|V projection of xkv was already launched on another stream."""
        cfg = self.cfg
        d = xq.shape[1]
        Mq, Mk = B * Lq, B * Lk
        dk, dv = dk_tot // H, dv_tot // H
        self_attn = xkv is xq
        wq = prefix + ".q_linear.weight"
        wk = prefix + ".k_linear.weight"
        if self_attn:
            nqkv = 2 * dk_tot + dv_tot
            qkv = self.new(Mq, nqkv)
            self.gemm(xq, True, self.w(wq), d, True, Mq, nqkv, d, qkv, b_static=True)      # packed [Wq;Wk;Wv]
            q_ptr, k_ptr, v_ptr = qkv.data_ptr(), qkv.data_ptr() + dk_tot * qkv.element_size(), \
                qkv.data_ptr() + 2 * dk_tot * qkv.element_size()
            ldq = ldk = ldv = nqkv
            kvb = None
        else:
            qkv = self.new(Mq, dk_tot)
            self.gemm(xq, True, self.w(wq), d, True, Mq, dk_tot, d, qkv, b_static=True)
            if kv_pre is not None:
                kvb = kv_pre[0]
                torch.cuda.current_stream(self.dev).wait_event(kv_pre[1])
            else:
                kvb = self.new(Mk, dk_tot + dv_tot)
                self.gemm(xkv, True, self.w(wk), d, True, Mk, dk_tot + dv_tot, d, kvb, b_static=True)   # packed [Wk;Wv]
            q_ptr, k_ptr, v_ptr = qkv.data_ptr(), kvb.data_ptr(), kvb.data_ptr() + dk_tot * kvb.element_size()
            ldq, ldk, ldv = dk_tot, dk_tot + dv_tot, dk_tot + dv_tot
        att = self.new(Mq, dv_tot)
        seed_a = self._seed()
        p_att = ATTN_DROPOUT if self.training else 0.0
        call("icap_mha_fwd", self.act, B, H, Lq, Lk, dk, dv, q_ptr, ldq, k_ptr, ldk, v_ptr, ldv, att.data_ptr(), dv_tot,
             _ptr(kvalid), int(causal), p_att, seed_a, self.step_dev.data_ptr(), _ptr(attn_mean), self._s())
        y, o, mean, rstd, seed_l, p_l = self.proj_add_ln(att, prefix + ".joint_linear.weight", dv_tot, None, xq,
                                                         prefix + ".layer_norm", None, cfg.dropout)

        if self.tape is not None:
            def bwd():
                ds, da = self.ln_bwd(y, o, mean, rstd, prefix + ".layer_norm", None, p_l, seed_l)
                self.add_grad(xq, ds)
                self.wgrad(da, att, self.g(prefix + ".joint_linear.weight"), d, dv_tot, Mq)
                datt = self.new(Mq, dv_tot)
                self.gemm(da, True, self.w(prefix + ".joint_linear.weight"), dv_tot, False, Mq, dv_tot, d, datt,
                          b_static=True)
                esz = qkv.element_size()
                if self_attn:
                    dqkv = self.new(Mq, nqkv)
                    call("icap_mha_bwd", self.act, B, H, Lq, Lk, dk, dv, q_ptr, ldq, k_ptr, ldk, v_ptr, ldv,
                         datt.data_ptr(), dv_tot, dqkv.data_ptr(), nqkv, dqkv.data_ptr() + dk_tot * esz, nqkv,
                         dqkv.data_ptr() + 2 * dk_tot * esz, nqkv, _ptr(kvalid), int(causal), p_att, seed_a,
                         self.step_dev.data_ptr(), self._s())
                    self.wgrad(dqkv, xq, self.g(wq), nqkv, d, Mq)
                    dx = self.new(Mq, d)
                    self.gemm(dqkv, True, self.w(wq), d, False, Mq, d, nqkv, dx, b_static=True)
                    self.add_grad(xq, dx)
                else:
                    dq = self.new(Mq, dk_tot)
                    dkv = self.new(Mk, dk_tot + dv_tot)
                    call("icap_mha_bwd", self.act, B, H, Lq, Lk, dk, dv, q_ptr, ldq, k_ptr, ldk, v_ptr, ldv,
                         datt.data_ptr(), dv_tot, dq.data_ptr(), dk_tot, dkv.data_ptr(), dk_tot + dv_tot,
                         dkv.data_ptr() + dk_tot * esz, dk_tot + dv_tot, _ptr(kvalid), int(causal), p_att, seed_a,
                         self.step_dev.data_ptr(), self._s())
                    self.wgrad(dq, xq, self.g(wq), dk_tot, d, Mq)
                    dx = self.new(Mq, d)
                    self.gemm(dq, True, self.w(wq), d, False, Mq, d, dk_tot, dx, b_static=True)
                    self.add_grad(xq, dx)
                    self.wgrad(dkv, xkv, self.g(wk), dk_tot + dv_tot, d, Mk)
                    # all decoder layers accumulate into ONE gradient buffer of the encoder output
                    # (side stream when enabled: only the encoder backward needs it -- encode() appends the join)
                    gl = self.gr.setdefault(id(xkv), [])
                    on_side = self.xkv_side and not cfg.move_first_image_feature
                    if gl:
                        self.gemm(dkv, True, self.w(wk), d, False, Mk, d, dk_tot + dv_tot, gl[0], accumulate=True,
                                  side=on_side)
                    else:
                        dxkv = self.new(Mk, d)
                        self.gemm(dkv, True, self.w(wk), d, False, Mk, d, dk_tot + dv_tot, dxkv, side=on_side)
                        gl.append(dxkv)
            # lowest flat offset this closure writes gradients to (DP buckets: everything from there to the end of the
            # flat buffer must be FINAL when it returns -- callers whose parameters are registered before tensors that
            # complete later pass report_lo=False)
            bwd.lo = self.offsets[wq] if report_lo else None
            self.tape.append(bwd)
        return y

    def ffn_block(self, prefix: str, x: torch.Tensor, hidden: int, rowscale: Optional[torch.Tensor],
                  norm: Optional[str] = None, x_in: Optional[torch.Tensor] = None, report_lo: bool = True) -> torch.Tensor:
        """FeedForward.forward (modules.py:110-122) [+ `*= non_pad_mask`, modules.py:154-155,203-204].
        x_in (move_first_image_feature tail, model.py:451-457): GEMM input differs from the residual."""
        cfg = self.cfg
        M, d = x.shape
        norm = norm or (prefix + ".layer_norm")
        w1, b1 = prefix + ".position_wise_1.weight", prefix + ".position_wise_1.bias"
        w2, b2 = prefix + ".position_wise_2.weight", prefix + ".position_wise_2.bias"
        gin = x if x_in is None else x_in
        h = self.new(M, hidden)
        self.gemm(gin, True, self.w(w1), d, True, M, hidden, d, h, bias=self.p(b1), epi=N.EPI_RELU, b_static=True)
        y, f, mean, rstd, seed_l, p_l = self.proj_add_ln(h, w2, hidden, self.p(b2), x, norm, rowscale, cfg.dropout)

        if self.tape is not None:
            def bwd():
                ds, da = self.ln_bwd(y, f, mean, rstd, norm, rowscale, p_l, seed_l, dbias2=self.g(b2))
                self.add_grad(x, ds)
                self.wgrad(da, h, self.g(w2), d, hidden, M)
                dh = self.new(M, hidden)
                self.gemm(da, True, self.w(w2), hidden, False, M, hidden, d, dh, epi=N.EPI_RELU_MASK, aux=h, b_static=True)
                self.side_call("icap_colsum", self.act, M, hidden, dh.data_ptr(), hidden, self.g(b1))
                self.wgrad(dh, gin, self.g(w1), hidden, d, M)
                dx = self.new(M, d)
                self.gemm(dh, True, self.w(w1), d, False, M, d, hidden, dx, b_static=True)
                self.add_grad(gin, dx)
            # the move_first tail completes out of order; image_encoder.* is registered BEFORE encoder.feature_embedding /
            # encoder.norm, whose gradients are only final at the very end of the backward (report_lo=False)
            bwd.lo = self.offsets[w1] if (prefix != "decoder" and report_lo) else None
            self.tape.append(bwd)
        return y

    # ------------------------------------------------------------------ encoder
    def _cat_width(self) -> int:
        # width of the packed [features | positions | 0] operand: a multiple of 64 elements, so that its row pitch is a
        # multiple of 128 B (a ragged pitch makes every TMA box row straddle two L2 lines: 26.6 vs 18 us for the GEMM)
        cfg = self.cfg
        return (cfg.encode_dim_features + cfg.encode_dim_positions + 63) // 64 * 64

    def _pack_embed_weights(self) -> torch.Tensor:
        """[Wf | Wp (| Wobj) | 0] as one [d, Kc] matrix: feature_embedding + position_embedding
        (+ object_embedding) become ONE GEMM over the concatenated input (model.py:294-307)."""
        cfg = self.cfg
        d, Df, Dp, Kc = cfg.encode_input_size, cfg.encode_dim_features, cfg.encode_dim_positions, self._cat_width()
        wcat = self.new(d, Kc, zero=True)
        src_dt = F32
        call("icap_copy2d", self.p("encoder.feature_embedding.weight"), src_dt, Df, wcat.data_ptr(), self.act, Kc,
             d, Df, 0, self._s())
        esz = wcat.element_size()
        if cfg.split_position:
            call("icap_copy2d", self.p("encoder.position_embedding.weight"), src_dt, 4, wcat.data_ptr() + Df * esz,
                 self.act, Kc, d, 4, 0, self._s())
            call("icap_copy2d", self.p("encoder.object_embedding.weight"), src_dt, Dp - 4,
                 wcat.data_ptr() + (Df + 4) * esz, self.act, Kc, d, Dp - 4, 0, self._s())
        else:
            call("icap_copy2d", self.p("encoder.position_embedding.weight"), src_dt, Dp, wcat.data_ptr() + Df * esz,
                 self.act, Kc, d, Dp, 0, self._s())
        return wcat

    def _unpack_embed_grads(self, dwcat: torch.Tensor) -> None:
        cfg = self.cfg
        d, Df, Dp, Kc = cfg.encode_input_size, cfg.encode_dim_features, cfg.encode_dim_positions, self._cat_width()
        acc = 1
        call("icap_copy2d", dwcat.data_ptr(), F32, Kc, self.g("encoder.feature_embedding.weight"), F32, Df, d, Df, acc,
             self._s())
        if cfg.split_position:
            call("icap_copy2d", dwcat.data_ptr() + Df * 4, F32, Kc, self.g("encoder.position_embedding.weight"), F32, 4,
                 d, 4, acc, self._s())
            call("icap_copy2d", dwcat.data_ptr() + (Df + 4) * 4, F32, Kc, self.g("encoder.object_embedding.weight"), F32,
                 Dp - 4, d, Dp - 4, acc, self._s())
        else:
            call("icap_copy2d", dwcat.data_ptr() + Df * 4, F32, Kc, self.g("encoder.position_embedding.weight"), F32, Dp,
                 d, Dp, acc, self._s())

    def encode(self, feats: torch.Tensor, pos: torch.Tensor):
        """Encoder.forward (model.py:257-332).  feats [B,R,Df] fp32, pos [B,R,Dp] fp32 (device)."""
        cfg = self.cfg
        B, R, Df = feats.shape
        M, d, Kc = B * R, cfg.encode_input_size, self._cat_width()
        H = cfg.encode_num_heads
        kvalid = self.new(M, dtype=torch.uint8)
        rowscale = self.new(M, dtype=torch.float32)
        if isinstance(feats, RegionBatch):      # rows come packed from the device-resident cache: no fp32 staging
            c = feats.cache
            assert c.engine_key == (Kc, self.act, Df, cfg.encode_dim_positions) and c.xcat.device == self.dev, \
                "region cache was built for a different model configuration / precision / device"
            xcat = self.new(M, Kc)
            call("icap_gather_regions", self.act, c.xcat.data_ptr(), c.valid.data_ptr(), c.num_images,
                 feats.idx.data_ptr(), int(feats.idx.dtype == torch.int64), B, R, Kc, xcat.data_ptr(),
                 kvalid.data_ptr(), rowscale.data_ptr(), c.err.data_ptr(), self._s())
        else:
            Dp = pos.shape[2]
            assert Df == cfg.encode_dim_features and Dp == cfg.encode_dim_positions
            call("icap_region_valid", pos.data_ptr(), M, Dp, kvalid.data_ptr(), rowscale.data_ptr(), self._s())
            xcat = self.new(M, Kc, zero=(Kc != Df + Dp))
            call("icap_copy2d", feats.data_ptr(), F32, Df, xcat.data_ptr(), self.act, Kc, M, Df, 0, self._s())
            call("icap_copy2d", pos.data_ptr(), F32, Dp, xcat.data_ptr() + Df * xcat.element_size(), self.act, Kc, M,
                 Dp, 0, self._s())
        wcat = self._pack_embed_weights()
        rec = self.tape is not None
        dwcat = self.new(d, Kc, dtype=torch.float32, zero=True) if rec else None
        if rec:     # runs LAST in the backward: every embedding wgrad has been accumulated into dwcat by then
            self.tape.append(lambda: self._unpack_embed_grads(dwcat))
        if cfg.split_image_objects:
            x = self._encode_split_objects(xcat, wcat, dwcat, kvalid, B, R)
        else:
            e = self.new(M, d)
            self.gemm(xcat, True, wcat.data_ptr(), Kc, True, M, d, Kc, e)
            x0, mean, rstd, _, _ = self.add_ln(e, None, 1, "encoder.norm", None, 0.0)
            x = x0
            if rec:
                def bwd():      # NB: closes over x0 (x is re-bound by the block loop below)
                    ds, _ = self.ln_bwd(x0, e, mean, rstd, "encoder.norm", None, 0.0, 0)
                    self.wgrad(ds, xcat, dwcat.data_ptr(), d, Kc, M, side_ok=False)
                self.tape.append(bwd)
        for i in range(cfg.encode_num_blocks):
            pre = f"encoder.encoder.{i}"
            if cfg.encode_mask:   # key-pad OR causal over region order, rows zeroed after the FFN (model.py:311-326)
                x = self.mha_block(pre + ".multihead_attention", x, x, B, R, R, H, cfg.encode_q_k_dim, cfg.encode_v_dim,
                                   kvalid, True)
                x = self.ffn_block(pre + ".feed_forward", x, cfg.encode_hidden_size, rowscale)
            else:                 # no mask at all (model.py:327-328)
                x = self.mha_block(pre + ".multihead_attention", x, x, B, R, R, H, cfg.encode_q_k_dim, cfg.encode_v_dim,
                                   None, False)
                x = self.ffn_block(pre + ".feed_forward", x, cfg.encode_hidden_size, None)
        if rec:
            def join_side():        # the cross-attention dgrads into d(encoder output) ran on the side stream
                if self._bwd_side is not None:
                    torch.cuda.current_stream(self.dev).wait_stream(self._bwd_side)
            self.tape.append(join_side)
        return x, kvalid

    def _encode_split_objects(self, xcat, wcat, dwcat, kvalid, B, R):
        """split_image_objects branch (model.py:258-292): every region i becomes the 2-token sequence
        [whole image (region 0), region i]; embed + LN, one extra `image_encoder` block with causal + key-pad
        mask, keep token 1, re-add the position embedding, LN again."""
        cfg = self.cfg
        assert not cfg.split_position, "split_position + split_image_objects is a shape error in the reference too"
        M, d, Kc, Df = B * R, cfg.encode_input_size, self._cat_width(), cfg.encode_dim_features
        H = cfg.encode_num_heads
        esz = xcat.element_size()
        rec = self.tape is not None
        # token 0 of pair (b, i) = region 0 of image b ; token 1 = region i
        x2 = self.new(2 * M, Kc)
        call("icap_rows_gather_add", self.act, xcat.data_ptr(), Kc, None, 0, x2.data_ptr(), 2 * Kc, M, Kc, R, R, 0, self._s())
        call("icap_copy2d", xcat.data_ptr(), self.act, Kc, x2.data_ptr() + Kc * esz, self.act, 2 * Kc, M, Kc, 0, self._s())
        kvalid2 = self.new(2 * M, dtype=torch.uint8)
        rowscale2 = self.new(2 * M, dtype=torch.float32)
        # validity of the pair tokens from the packed position columns (same rule: all-zero position row = padding)
        pos2 = self.new(2 * M, Kc - Df, dtype=torch.float32)
        call("icap_copy2d", x2.data_ptr() + Df * esz, self.act, Kc, pos2.data_ptr(), F32, Kc - Df, 2 * M, Kc - Df, 0, self._s())
        call("icap_region_valid", pos2.data_ptr(), 2 * M, Kc - Df, kvalid2.data_ptr(), rowscale2.data_ptr(), self._s())
        e2 = self.new(2 * M, d)
        self.gemm(x2, True, wcat.data_ptr(), Kc, True, 2 * M, d, Kc, e2)
        y2, mean2, rstd2, _, _ = self.add_ln(e2, None, 1, "encoder.norm", None, 0.0)
        if rec:
            def bwd_embed2():
                ds, _ = self.ln_bwd(y2, e2, mean2, rstd2, "encoder.norm", None, 0.0, 0)
                self.wgrad(ds, x2, dwcat.data_ptr(), d, Kc, 2 * M, side_ok=False)
            self.tape.append(bwd_embed2)
        pre = "encoder.image_encoder"
        z = self.mha_block(pre + ".multihead_attention", y2, y2, M, 2, 2, H, cfg.encode_q_k_dim, cfg.encode_v_dim,
                           kvalid2, True, report_lo=False)
        z = self.ffn_block(pre + ".feed_forward", z, cfg.encode_hidden_size, rowscale2, report_lo=False)
        # embedded_feature = output[:, 1]; embedded_position = position_embedding(position)[:, 1]  (model.py:290-292)
        tok1 = self.new(M, d)
        call("icap_copy2d", z.data_ptr() + d * esz, self.act, 2 * d, tok1.data_ptr(), self.act, d, M, d, 0, self._s())
        emb_p = self.new(M, d)
        self.gemm(xcat, True, wcat.data_ptr() + Df * esz, Kc, True, M, d, Kc - Df, emb_p,
                  a_ptr=xcat.data_ptr() + Df * esz, lda=Kc)
        x, mean, rstd, _, _ = self.add_ln(tok1, emb_p, M, "encoder.norm", None, 0.0)
        if rec:
            def bwd_tail():
                ds, _ = self.ln_bwd(x, tok1, mean, rstd, "encoder.norm", None, 0.0, 0)
                # d position-embedding weights (tail columns of the packed matrix)
                self.wgrad(ds, xcat, dwcat.data_ptr() + Df * 4, d, Kc - Df, M, x_ptr=xcat.data_ptr() + Df * esz, ldx=Kc,
                           ldg=Kc, side_ok=False)
                dz = self.new(2 * M, d, zero=True)
                call("icap_copy2d", ds.data_ptr(), self.act, d, dz.data_ptr() + d * esz, self.act, 2 * d, M, d, 0, self._s())
                self.add_grad(z, dz)
            self.tape.append(bwd_tail)
        return x

    # ------------------------------------------------------------------ decoder (teacher forced)
    def decode_train(self, inp: torch.Tensor, tok_valid: torch.Tensor, rowscale: torch.Tensor, enc: torch.Tensor,
                     kvalid_enc: torch.Tensor, B: int, T: int, R: int, ctx_mean: Optional[torch.Tensor] = None):
        """Decoder.forward (model.py:419-459) on the full teacher-forced sequence."""
        cfg = self.cfg
        M, d, E, H = B * T, cfg.decode_input_size, cfg.dim_word_embedding, cfg.decode_num_heads
        emb = self.new(M, E)
        call("icap_embed_fwd", self.act, self.act, inp.data_ptr(), 1, M, E, self.w("decoder.word_embedding.weight"),
             emb.data_ptr(), None, cfg.pad_idx, self._s())
        we = self.new(M, d)
        self.gemm(emb, True, self.w("decoder.word_embedding_linear.weight"), E, True, M, d, E, we)
        x0, mean, rstd, _, _ = self.add_ln(we, self.pos_table_act, T, "decoder.norm", None, 0.0)
        x = x0
        if self.tape is not None:
            def bwd():          # NB: closes over x0 (x is re-bound by the block loop below)
                ds, _ = self.ln_bwd(x0, we, mean, rstd, "decoder.norm", None, 0.0, 0)
                self.wgrad(ds, emb, self.g("decoder.word_embedding_linear.weight"), d, E, M)
                demb = self.new(M, E)
                self.gemm(ds, True, self.w("decoder.word_embedding_linear.weight"), E, False, M, E, d, demb)
                call("icap_embed_bwd", self.act, inp.data_ptr(), M, E, cfg.pad_idx, demb.data_ptr(),
                     self.g("decoder.word_embedding.weight"), self._s())
            bwd.lo = self.offsets["decoder.word_embedding.weight"]
            self.tape.append(bwd)
        kv_pre = [None] * cfg.decode_num_blocks
        if (self.xkv_side and self.tape is not None and self.wgrad_side_stream and self.precision == "bf16"
                and self._prof is None and self._gemm_log is None):
            # K|V projections of the encoder output for every decoder layer, on the side stream while the decoder's
            # self-attention blocks run (the buffers live until the end of the step: self.keep)
            main = torch.cuda.current_stream(self.dev)
            if self._side is None:
                self._side = torch.cuda.Stream(device=self.dev)
            self._side.wait_stream(main)
            nkv = cfg.decode_q_k_dim + cfg.decode_v_dim
            with torch.cuda.stream(self._side):
                for i in range(cfg.decode_num_blocks):
                    kvb = self.new(B * R, nkv)
                    self.gemm(enc, True, self.w(f"decoder.decoder.{i}.encode_attention.k_linear.weight"), d, True, B * R,
                              nkv, d, kvb)
                    ev = torch.cuda.Event()
                    ev.record(self._side)
                    kv_pre[i] = (kvb, ev)
        for i in range(cfg.decode_num_blocks):
            pre = f"decoder.decoder.{i}"
            last = i == cfg.decode_num_blocks - 1
            x = self.mha_block(pre + ".self_attention", x, x, B, T, T, H, cfg.decode_q_k_dim, cfg.decode_v_dim,
                               tok_valid, True)
            x = self.mha_block(pre + ".encode_attention", x, enc, B, T, R, H, cfg.decode_q_k_dim, cfg.decode_v_dim,
                               kvalid_enc, False, attn_mean=ctx_mean if last else None, kv_pre=kv_pre[i])
            x = self.ffn_block(pre + ".feed_forward", x, cfg.decode_hidden_size, rowscale)
        if cfg.move_first_image_feature:
            x = self._move_first_tail(x, enc, B, T, R)
        return x

    def _move_first_tail(self, x, enc, B, T, R, rows_per_image: int = 1):
        """move_first_image_feature tail (model.py:451-457):
        LN(Dropout(W2 relu(W1 (x + enc[:, 0]) + b1) + b2) + x) with the decoder-level position_wise / layer_norm."""
        cfg = self.cfg
        M, d = x.shape
        gin = self.new(M, d)
        # row r belongs to image r // (T * rows_per_image); its first region is row image * R of enc
        call("icap_rows_gather_add", self.act, enc.data_ptr(), d, x.data_ptr(), d, gin.data_ptr(), d, M, d,
             T * rows_per_image, R, 0, self._s())
        y = self.ffn_block("decoder", x, cfg.decode_hidden_size, None, norm="decoder.layer_norm", x_in=gin)
        if self.tape is not None:
            def bwd():          # executed right after ffn_block's backward: gin's gradient flows to x and to enc[:, 0]
                gs = self.gr.pop(id(gin), [])
                assert len(gs) == 1
                self.add_grad(x, gs[0])
                gl = self.gr.setdefault(id(enc), [])
                if not gl:
                    gl.append(self.new(enc.shape[0], d, zero=True))
                call("icap_rows_segsum_add", self.act, gs[0].data_ptr(), d, gl[0].data_ptr(), d, B, T * rows_per_image, d,
                     R, 0, self._s())
            # tape runs in reverse: this closure must run AFTER ffn_block's, so insert it BEFORE that one
            self.tape.insert(len(self.tape) - 1, bwd)
        return y

    # ------------------------------------------------------------------ full passes
    def prepare_inputs(self, feats, pos, captions=None):
        if isinstance(feats, RegionBatch):
            assert pos is None, "a RegionBatch carries its positions"
            if feats.idx.device != self.dev:
                feats = RegionBatch(feats.cache, feats.idx.to(self.dev, non_blocking=True))
        else:
            feats = feats.to(self.dev, torch.float32, non_blocking=True).contiguous()
            pos = pos.to(self.dev, torch.float32, non_blocking=True).contiguous()
        if captions is not None:
            assert captions.dtype in (torch.int32, torch.int64)
            if not captions.is_cuda and captions.numel():
                # the kernels index the embedding table / logits with these ids unchecked (the reference would raise a
                # device assert): validate host batches here, where it costs nothing
                lo, hi = int(captions.min()), int(captions.max())
                if lo < 0 or hi >= self.cfg.num_vocab:
                    raise N.IcapError(f"caption token ids must lie in [0, {self.cfg.num_vocab}): got [{lo}, {hi}] "
                                      "(vocabulary / checkpoint mismatch?)")
            captions = captions.to(self.dev, non_blocking=True).contiguous()
        return feats, pos, captions

    def forward_logits(self, feats, pos, captions, record: bool):
        """Teacher-forced pass up to the classifier (Transformer.forward, model.py:79-93).
        Returns (logits [B*T, ldl] in act dtype, tgt, count2, dec_out)."""
        cfg = self.cfg
        self.refresh_shadow()
        self._site = 0
        self.tape = [] if record else None
        if record:
            self.tape_gen += 1
        self.gr, self.keep = {}, []
        B, R, _ = feats.shape
        L = captions.shape[1]
        T = L - 1
        assert T <= cfg.T, f"caption length {L} exceeds max_length {cfg.max_length}"
        M = B * T
        inp = self.new(M, dtype=torch.int32)
        tgt = self.new(M, dtype=torch.int32)
        tok_valid = self.new(M, dtype=torch.uint8)
        rowscale = self.new(M, dtype=torch.float32)
        count_i = self.new(1, dtype=torch.int32)
        count2 = self.new(2, dtype=torch.float32)
        call("icap_caption_prep", captions.data_ptr(), int(captions.dtype == torch.int64), B, L, cfg.pad_idx,
             inp.data_ptr(), tgt.data_ptr(), tok_valid.data_ptr(), rowscale.data_ptr(), count_i.data_ptr(),
             count2.data_ptr(), self._s())
        enc, kvalid = self.encode(feats, pos)
        dec = self.decode_train(inp, tok_valid, rowscale, enc, kvalid, B, T, R)
        V, d = cfg.num_vocab, cfg.decode_input_size
        ldl = (V + 7) // 8 * 8
        logits = self.new(M, ldl)
        self.gemm(dec, True, self.w("classifer.weight"), d, True, M, V, d, logits, ldc=ldl, bias=self.p("classifer.bias"),
                  b_static=True)
        return logits, tgt, count2, dec

    def loss_from_logits(self, logits, tgt, count2, dec, record: bool) -> torch.Tensor:
        """CrossEntropyLoss(ignore_index, 'mean') / FocalLoss (model.py:73-76,95-96); returns out2 =
        [loss, dloss/dce] on the device.  With record=True the logits buffer becomes dlogits."""
        cfg = self.cfg
        M, ldl = logits.shape
        V, d = cfg.num_vocab, cfg.decode_input_size
        row_loss = self.new(M, dtype=torch.float32)
        out2 = self.new(2, dtype=torch.float32)
        inv_count = count2[1:2]
        grad_scale = self.one if self.dp_unnormalized else inv_count     # DP: divide by the GLOBAL count in Adam
        call("icap_xent", self.act, M, V, logits.data_ptr(), ldl, tgt.data_ptr(), cfg.pad_idx, grad_scale.data_ptr(),
             row_loss.data_ptr(), int(record), self._s())
        if self.dp_unnormalized and record:
            call("icap_copy2d", count2.data_ptr(), F32, 1, self.g32.data_ptr() + 4 * self.n_flat, F32, 1, 1, 1, 1, self._s())
        call("icap_xent_finalize", M, row_loss.data_ptr(), inv_count.data_ptr(), int(cfg.focal), out2.data_ptr(),
             self._s())
        if record:
            self._append_classifier_bwd(logits, dec)
        return out2

    def _append_classifier_bwd(self, logits: torch.Tensor, dec: torch.Tensor) -> None:
        """Backward of `classifer` (model.py:68,93): by the time it runs, `logits` holds d loss / d logits."""
        cfg = self.cfg
        M, ldl = logits.shape
        V, d = cfg.num_vocab, cfg.decode_input_size

        def bwd():
            self.wgrad(logits, dec, self.g("classifer.weight"), V, d, M, ld_dy=ldl)
            self.side_call("icap_colsum", self.act, M, V, logits.data_ptr(), ldl, self.g("classifer.bias"))
            dx = self.new(M, d)
            self.gemm(logits, True, self.w("classifer.weight"), d, False, M, d, V, dx, lda=ldl, b_static=True)
            self.add_grad(dec, dx)
        bwd.lo = self.offsets["classifer.weight"]
        self.tape.append(bwd)

    def set_dlogits(self, logits: torch.Tensor, grad: torch.Tensor) -> None:
        """Overwrite the recorded logits buffer [M, ldl] with an externally computed d loss / d logits [M, V] (fp32):
        the PolicyNetwork path, where the loss lives in user code (model_RL.py:75-90, loss.py:31-219)."""
        M, ldl = logits.shape
        V = self.cfg.num_vocab
        grad = grad.reshape(M, V).to(torch.float32).contiguous()
        call("icap_copy2d", grad.data_ptr(), F32, V, logits.data_ptr(), self.act, ldl, M, V, 0, self._s())

    def backward(self, zero_grads: bool = True) -> None:
        """Run the tape in reverse: fills g32 with d(mean CE)/d(param); focal scaling is applied by
        the caller (icap_scale / Adam gscale) from out2[1]."""
        assert self.tape is not None, "forward was not recorded"
        if zero_grads:
            self.g32.zero_()
        main = torch.cuda.current_stream(self.dev)
        if self.wgrad_side_stream and self.precision == "bf16" and self._prof is None:
            if self._side is None:
                self._side = torch.cuda.Stream(device=self.dev)
            self._bwd_side = self._side
            self._bwd_side.wait_stream(main)          # g32 has been zeroed / the forward is complete
        limit = self.bwd_gemm_sms if self.bucket_hook is not None else None
        if limit:
            call("icap_set_gemm_sms", int(limit))
        try:
            for fn in reversed(self.tape):
                fn()
                if self.bucket_hook is not None:
                    self.bucket_hook(getattr(fn, "lo", None))
        finally:
            if limit:
                call("icap_set_gemm_sms", 0)
            if self._bwd_side is not None:
                main.wait_stream(self._bwd_side)      # every weight gradient has landed in g32
                self._bwd_side = None
        self.tape = None
        self.gr, self.keep = {}, []

    def adam_step(self, lr: float, betas=(0.9, 0.999), eps: float = 1e-8, gscale_dev: Optional[torch.Tensor] = None,
                  gscale: float = 1.0) -> None:
        """torch.optim.Adam semantics over the flat buffers (core/models.py:111-113,126)."""
        if self.adam_m is None:
            self.adam_m = torch.zeros_like(self.p32)
            self.adam_v = torch.zeros_like(self.p32)
        call("icap_adam_step", self.n_flat, self.p32.data_ptr(), self.g32.data_ptr(), self.adam_m.data_ptr(),
             self.adam_v.data_ptr(), _ptr(self.p16), lr, betas[0], betas[1], eps, self.step_dev.data_ptr(), 1,
             _ptr(gscale_dev), gscale, self._s())
        self.shadow_fresh = True

    def train_step(self, feats, pos, captions, lr: float = 5e-4, train_mode: bool = True,
                   betas=(0.9, 0.999), eps: float = 1e-8) -> torch.Tensor:
        """zero_grad -> forward -> backward -> Adam (core/models.py:115-126), all on the current stream.
        Returns the device tensor [loss, dloss/dce] (no host sync).  train_mode=False keeps dropout off
        (the reference's eval-mode arithmetic, used by the parity tests)."""
        out2 = self.forward_backward(feats, pos, captions, train_mode)
        self.adam_step(lr, betas=betas, eps=eps, gscale_dev=out2[1:2] if self.cfg.focal else None)
        return out2

    def forward_backward(self, feats, pos, captions, train_mode: bool = True) -> torch.Tensor:
        """zero_grad + forward + backward; gradients land in g32 (data parallel: all-reduce them next)."""
        self.training = train_mode
        self.g32.zero_()      # before the forward: in DP mode the forward deposits the token count in the tail slot
        logits, tgt, count2, dec = self.forward_logits(feats, pos, captions, record=True)
        out2 = self.loss_from_logits(logits, tgt, count2, dec, record=True)
        self.backward(zero_grads=False)
        return out2

    def _proj_res_ln(self, att: torch.Tensor, resid: torch.Tensor, prefix: str, rows: int, d: int, dv_tot: int):
        """joint_linear -> (+ residual) -> LayerNorm of an attention block in a decode step (modules.py:86-90, eval)."""
        y, *_ = self.proj_add_ln(att, prefix + ".joint_linear.weight", dv_tot, None, resid, prefix + ".layer_norm", None,
                                 0.0)
        return y

    # ------------------------------------------------------------------ KV-cached decoding
    def decode(self, feats: torch.Tensor, pos: torch.Tensor, beam_size: int = 1, log_domain: bool = False,
               want_attention: bool = False, want_gaps: bool = False, num_samples: int = 0, temperature: float = 1.0,
               sample_counter: Optional[torch.Tensor] = None, stop_at_end: bool = False, length_penalty: float = 0.0,
               n_best: int = 0):
        """Greedy (beam_size=1: Transformer.generate_caption_vector, model.py:101-132) or beam search
        (Transformer.beam_search, model.py:135-200) with a KV cache: the reference re-runs the decoder on
        the whole prefix every step (and once per beam); here every step computes ONE position for all
        B*k rows, self-attention reads cached K/V through a beam slot table, cross-attention K/V of the
        encoder output are projected once per layer.  Semantics kept: probability-domain additive beam
        scores (log-domain for the PolicyNetwork variant), no EOS handling, pad-token (id 0) masking of
        generated tokens, result = beam slot 0.

        num_samples = n > 0: sampled decoding instead (icap_sample_tokens): B*n independent rows, n per image, each
        token drawn from softmax(logits / temperature); a row that has emitted <END> or <NULL> continues with <NULL>
        and log-probability 0.  The uniforms are keyed by the int32 device counter `sample_counter` (the engine's
        sample_dev by default), which the decode advances by one at its end.

        stop_at_end: beam search that stops at <END> instead (also for beam_size = 1; icap_beam_select_eos): log-probability
        scores, a hypothesis whose last token is <END> or <NULL> is finished and continues with <NULL> at an unchanged
        score; after the last step the beams are ranked by score / ((5 + len) / 6)^length_penalty (icap_beam_finalize)
        and the n_best (0: all beam_size) best are kept.

        Returns dict(ids int32 [B, T+1] (col 0 = <START>), attention fp32 [T, B, R] | None,
                     gaps fp32 [T, B] | None, score fp32 [B] (beam slot 0) | None)  -- all device tensors, no host sync.
        Sampling: dict(ids int32 [B, n, T+1], logp fp32 [B, n, T] (log_softmax of the token at temperature 1)).
        stop_at_end: dict(ids int32 [B, n, T+1], score fp32 [B, n] (log-probability), len int32 [B, n], gaps | None),
        best first."""
        cfg = self.cfg
        assert self.tape is None
        self.training = False
        self.refresh_shadow()
        self._site = 0
        sampling = num_samples > 0
        if sampling:
            assert not (want_attention or want_gaps), "sampled decoding returns ids and log-probabilities only"
            assert math.isfinite(temperature) and temperature > 0, "the temperature must be finite and > 0"
            if sample_counter is None:
                sample_counter = self.sample_dev
        k = int(num_samples) if sampling else int(beam_size)        # rows per image
        if stop_at_end:
            assert not (sampling or want_attention), "the <END>-aware beam search returns ids, scores and lengths"
            assert math.isfinite(length_penalty) and length_penalty >= 0, "the length penalty must be finite and >= 0"
            n_best = int(n_best) or k
            assert 1 <= n_best <= k, "n_best must be in [1, beam_size]"
        beam = not sampling and (k > 1 or stop_at_end)
        B, R, _ = feats.shape
        T, d, V, E = cfg.T, cfg.decode_input_size, cfg.num_vocab, cfg.dim_word_embedding
        H, dk_tot, dv_tot, hid = cfg.decode_num_heads, cfg.decode_q_k_dim, cfg.decode_v_dim, cfg.decode_hidden_size
        dk, dv = dk_tot // H, dv_tot // H
        nqkv, nkv = 2 * dk_tot + dv_tot, dk_tot + dv_tot
        rows = B * k
        Tmax = T + 1
        esz = 2 if self.precision == "bf16" else 4
        s = self._s
        enc, kvalid = self.encode(feats, pos)
        # cross-attention K/V of every decoder layer, once (the reference recomputes them per step and beam)
        cross = []
        for i in range(cfg.decode_num_blocks):
            kvb = self.new(B * R, nkv)
            self.gemm(enc, True, self.w(f"decoder.decoder.{i}.encode_attention.k_linear.weight"), d, True, B * R, nkv, d, kvb)
            cross.append(kvb)
        # token embedding folded with word_embedding_linear: table[v] = Emb[v] . Wwe^T  (model.py:432-433)
        table = self.new(V, d)
        emb_w = self.p16 if self.precision == "bf16" else self.p32
        self.gemm(emb_w, True, self.w("decoder.word_embedding_linear.weight"), E, True, V, d, E, table,
                  a_ptr=self.w("decoder.word_embedding.weight"), lda=E)
        tok = [torch.zeros(rows, Tmax, dtype=torch.int32, device=self.dev) for _ in range(2)]
        tok[0][:, 0] = 1                                  # <START> (model.py:111,144)
        slot = None
        if beam:
            slot = [torch.zeros(rows, Tmax, dtype=torch.int32, device=self.dev) for _ in range(2)]
            slot[0][:, 0] = torch.arange(rows, dtype=torch.int32, device=self.dev)
            score = [torch.zeros(B, k, dtype=torch.float32, device=self.dev) for _ in range(2)]
            parent = torch.empty(B, k, dtype=torch.int32, device=self.dev)
            newtok = torch.empty(B, k, dtype=torch.int32, device=self.dev)
        caches = [self.new(rows, T, nkv) for _ in range(cfg.decode_num_blocks)]
        attn = torch.zeros(T, rows, R, dtype=torch.float32, device=self.dev) if want_attention else None
        gaps = torch.zeros(T, B, dtype=torch.float32, device=self.dev) if want_gaps else None
        logp = torch.zeros(rows, T, dtype=torch.float32, device=self.dev) if sampling else None
        ldl = (V + 7) // 8 * 8
        cur = 0
        fused_start = d % 8 == 0 and d <= 1024 and os.environ.get("ICAP_DECODE_FUSED_START", "1") != "0"

        def step_input(t, tk, reorder=None):
            """Decoder input of position t (model.py:432-436): folded embedding row + positional row -> decoder.norm;
            with `reorder` = (parent, token, tok_out, slot_in, slot_out) the beam bookkeeping of step t - 1 runs in
            the same launch (icap_decode_embed_ln)."""
            x = self.new(rows, d)
            rowscale = self.new(rows, dtype=torch.float32)
            pos_row = self.pos_table_act.data_ptr() + t * d * esz
            if fused_start:
                par, tokn, tko, sli, slo = reorder if reorder is not None else (None,) * 5
                call("icap_decode_embed_ln", self.act, rows, d, k, Tmax, t, _ptr(par), _ptr(tokn), tk.data_ptr(), _ptr(tko),
                     _ptr(sli), _ptr(slo), table.data_ptr(), pos_row, self.p("decoder.norm.weight"),
                     self.p("decoder.norm.bias"), x.data_ptr(), rowscale.data_ptr(), cfg.pad_idx, LN_EPS, s())
                return x, rowscale
            if reorder is not None:
                par, tokn, tko, sli, slo = reorder
                call("icap_beam_reorder", B, k, Tmax, t - 1, par.data_ptr(), tokn.data_ptr(), tk.data_ptr(), tko.data_ptr(),
                     _ptr(sli), _ptr(slo), s())
                tk = tko
            x0 = self.new(rows, d)
            call("icap_embed_fwd", self.act, self.act, tk.data_ptr() + 4 * t, Tmax, rows, d, table.data_ptr(),
                 x0.data_ptr(), rowscale.data_ptr(), cfg.pad_idx, s())
            call("icap_add_ln_fwd", self.act, self.act, rows, d, x0.data_ptr(), pos_row, 1, self.p("decoder.norm.weight"),
                 self.p("decoder.norm.bias"), None, x.data_ptr(), None, None, 0, 0.0, 0, None, LN_EPS, s())
            return x, rowscale

        x, rowscale = step_input(0, tok[cur])
        for t in range(T):
            tk = tok[cur]
            for i in range(cfg.decode_num_blocks):
                pre = f"decoder.decoder.{i}"
                last = i == cfg.decode_num_blocks - 1
                # --- masked self-attention over the cache (modules.py:190-194)
                qkv = self.new(rows, nqkv)
                self.gemm(x, True, self.w(pre + ".self_attention.q_linear.weight"), d, True, rows, nqkv, d, qkv,
                          b_static=True)
                cache = caches[i]
                att = self.new(rows, dv_tot)
                # K/V of position t are appended to the cache inside the attention kernel
                # (ICAP_DECODE_FUSED_APPEND=0: separate strided copy + plain decode attention, for A/B timing)
                sl = slot[cur].data_ptr() if slot is not None else None
                if os.environ.get("ICAP_DECODE_FUSED_APPEND", "1") == "0":
                    call("icap_copy2d", qkv.data_ptr() + dk_tot * esz, self.act, nqkv, cache.data_ptr() + t * nkv * esz,
                         self.act, T * nkv, rows, nkv, 0, s())
                    call("icap_mha_decode", self.act, rows, H, t + 1, dk, dv, qkv.data_ptr(), nqkv, cache.data_ptr(), nkv,
                         cache.data_ptr() + dk_tot * esz, nkv, T, att.data_ptr(), dv_tot, sl, Tmax, tk.data_ptr(), Tmax,
                         cfg.pad_idx, None, 1, None, s())
                else:
                    call("icap_mha_decode_self", self.act, rows, H, t, dk, dv, qkv.data_ptr(), nqkv,
                         qkv.data_ptr() + dk_tot * esz, qkv.data_ptr() + 2 * dk_tot * esz, nqkv, cache.data_ptr(), nkv,
                         cache.data_ptr() + dk_tot * esz, nkv, T, att.data_ptr(), dv_tot, sl, Tmax, tk.data_ptr(), Tmax,
                         cfg.pad_idx, k, s())
                x1 = self._proj_res_ln(att, x, pre + ".self_attention", rows, d, dv_tot)
                # --- cross-attention over the image regions (modules.py:196-200)
                q2 = self.new(rows, dk_tot)
                self.gemm(x1, True, self.w(pre + ".encode_attention.q_linear.weight"), d, True, rows, dk_tot, d, q2,
                          b_static=True)
                att2 = self.new(rows, dv_tot)
                call("icap_mha_decode", self.act, rows, H, R, dk, dv, q2.data_ptr(), dk_tot, cross[i].data_ptr(), nkv,
                     cross[i].data_ptr() + dk_tot * esz, nkv, R, att2.data_ptr(), dv_tot, None, 0, None, 0, cfg.pad_idx,
                     kvalid.data_ptr(), k, attn[t].data_ptr() if (attn is not None and last) else None, s())
                x2 = self._proj_res_ln(att2, x1, pre + ".encode_attention", rows, d, dv_tot)
                # --- FFN + non-pad row mask (modules.py:202-204)
                x = self.ffn_block(pre + ".feed_forward", x2, hid, rowscale)
            if cfg.move_first_image_feature:
                x = self._move_first_tail(x, enc, B, 1, R, rows_per_image=k)
            logits = self.new(rows, ldl)
            # beam search in bf16: the classifier's epilogue leaves per-128-column (max, 2nd max, sum exp) statistics,
            # so that beam_select does not make its own statistics pass over the k * V logits of every image
            stats = None
            if beam and self.precision == "bf16":
                stats = self.new(rows, 8 * ((V + 255) // 256), dtype=torch.float32)
            self.gemm(x, True, self.w("classifer.weight"), d, True, rows, V, d, logits, ldc=ldl,
                      bias=self.p("classifer.bias"), b_static=True, epi=N.EPI_ROWSTATS if stats is not None else 0,
                      aux=stats)
            if not beam:
                if sampling:
                    call("icap_sample_tokens", self.act, rows, V, logits.data_ptr(), ldl, 1.0 / temperature,
                         self.sample_seed, sample_counter.data_ptr(), t, Tmax, tk.data_ptr(), logp.data_ptr(), T,
                         END_IDX, cfg.pad_idx, s())
                else:
                    call("icap_argmax", self.act, rows, V, logits.data_ptr(), ldl, tk.data_ptr() + 4 * (t + 1), Tmax,
                         gaps[t].data_ptr() if gaps is not None else None, s())
                if t + 1 < T:
                    x, rowscale = step_input(t + 1, tk)
            else:
                kin = 1 if t == 0 else k       # step 0: all beams hold <START>, only beam 0 competes (model.py:146-166)
                args = (self.act, B, kin, V, logits.data_ptr(), ldl * (k if t == 0 else 1),
                        score[cur].data_ptr() if t > 0 else None, k, score[cur ^ 1].data_ptr(), parent.data_ptr(),
                        newtok.data_ptr(), gaps[t].data_ptr() if gaps is not None else None)
                stats_args = (_ptr(stats), (stats.shape[1] * (k if t == 0 else 1)) if stats is not None else 0)
                if stop_at_end:
                    call("icap_beam_select_eos", *args, 1, *stats_args, tk.data_ptr(), Tmax, t, END_IDX, cfg.pad_idx, s())
                else:
                    call("icap_beam_select", *args, int(log_domain), *stats_args, s())
                if t + 1 < T:       # bookkeeping of this step + input of the next one in one launch
                    x, rowscale = step_input(t + 1, tk, (parent, newtok, tok[cur ^ 1], slot[cur], slot[cur ^ 1]))
                else:
                    call("icap_beam_reorder", B, k, Tmax, t, parent.data_ptr(), newtok.data_ptr(), tk.data_ptr(),
                         tok[cur ^ 1].data_ptr(), slot[cur].data_ptr(), slot[cur ^ 1].data_ptr(), s())
                cur ^= 1
        if sampling:
            call("icap_step_tick", sample_counter.data_ptr(), s())        # the next decode draws fresh uniforms
            return {"ids": tok[cur].view(B, k, Tmax), "logp": logp.view(B, k, T)}
        if stop_at_end:
            out_ids = torch.empty(B, n_best, Tmax, dtype=torch.int32, device=self.dev)
            out_score = torch.empty(B, n_best, dtype=torch.float32, device=self.dev)
            out_len = torch.empty(B, n_best, dtype=torch.int32, device=self.dev)
            call("icap_beam_finalize", B, k, Tmax, tok[cur].data_ptr(), score[cur].data_ptr(), END_IDX, cfg.pad_idx,
                 float(length_penalty), n_best, out_ids.data_ptr(), out_score.data_ptr(), out_len.data_ptr(), s())
            return {"ids": out_ids, "score": out_score, "len": out_len, "gaps": gaps}
        ids = tok[cur].view(B, k, Tmax)[:, 0, :]
        if attn is not None:
            attn = attn.view(T, B, k, R)[:, :, 0, :]
        return {"ids": ids, "attention": attn, "gaps": gaps, "score": score[cur][:, 0] if beam else None}
