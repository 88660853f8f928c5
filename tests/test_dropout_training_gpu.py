"""The dropout-on training kernels against fp64, with the masks restated bit for bit in numpy.

The training step drops 0.1 of the attention probabilities and 0.2 (model A), 0.3 (B) or 0.2 (C) after every
projection.  No mask is stored: every kernel re-evaluates a counter hash of (seed, element index), the backward kernels
too (icap_common.cuh).  `keep_oracle` below restates that hash in numpy uint32 / uint64 arithmetic, and every mask a
kernel applies is recovered from its outputs and compared with the oracle on every unmasked element:

* attention (icap_mha_fwd / icap_mha_bwd): one-hot V probes make the forward output the dropped probabilities, one-hot
  dO probes make dV = Pd^T the backward's dropped probabilities.  Element ((b*H + h)*Lq + i) * attn_drop_ld(Lk) + j.
* add + LayerNorm (icap_add_ln_fwd, write_sum=1) and GEMM + LayerNorm (icap_gemm_ln): a dropped element leaves the
  saved sum equal to the residual bitwise, and the inputs are drawn so that a kept one cannot.  Element row*d + col.

Outputs and gradients are compared with fp64 evaluated through the oracle's mask.  Data has the product's layout
(packed QKV [B*L, 3*H*dk] for self-attention, q and packed K|V for cross-attention, gradients into the same layouts);
K / V rows of masked keys hold +-3e4, outputs start as NaN.  Each case checks which kernel ran through torch.profiler.

Errors: attention O and P per (row, head) against the largest reference value of that (row, head); attention gradients
per (batch, head) block against its largest reference value; LayerNorm y, s, ds, da per row against the row's largest
reference value; mean as |mean - ref| * rstd_ref; rstd relative; dgamma / dbeta / dbias2 against the vector's largest
value.  Bounds (derived from the arithmetic, see TOL_*), observed maxima on one NVIDIA B200 (1000 W power limit):

    quantity                                         bound            observed max
    attention O, P: fp32                             2e-5             1.0e-6
    attention O, P: bf16 SIMT / mma                  4e-3 / 8e-3      3.89e-3 / 6.72e-3
    attention dQ dK dV: fp32                         2e-5             7.5e-7
    attention dQ dK dV: bf16 SIMT / mma              4e-3 / 8e-3      3.86e-3 / 6.68e-3 (mixed paths 3.68e-3 / 5.90e-3)
    add+LN y, s: fp32                                2e-5             2.9e-7
    add+LN y, s: bf16 (s: bf16 a)                    4e-3             3.89e-3
    add+LN ds, da: fp32 / bf16                       2e-5 / 4e-3      2.9e-7 / 3.88e-3
    add+LN dgamma dbeta dbias2: fp32 / bf16          2e-5 / 4e-3      3.3e-7 / 2.50e-3
    GEMM+LN y, s                                     4e-3             3.89e-3
    GEMM+LN -> split backward ds, da                 5e-3             4.16e-3
    GEMM+LN -> split backward dgamma dbeta dbias2    4e-3             1.80e-3
    mean, rstd (every LayerNorm)                     2e-6             2.7e-7

172 cases (64 attention, 12 of them mixed-path; 38 add + LN forward, 60 backward; 10 GEMM + LN chains).  Each
attention case also flips the most influential keep decision of every (b, h) and checks that the fp64 O moves by more
than 3x the bound (smallest margin observed: 64x the bound, bf16 mma; 88x bf16 SIMT; 20000x fp32), and that a
different step gives a different mask while the same step gives bitwise-equal outputs.

The mixed-path cases run the forward on one attention kernel and the backward on the other (SIMT forward because of
attn_mean + mma backward; mma forward + SIMT backward under ICAP_MHA_SIMT).  Before the SIMT kernels took the row
stride attn_drop_ld(Lk), they indexed the mask with (Lk + 3) & ~3: all 12 mixed-path cases failed (gradient errors of
94 % to 330 % of the block's largest value), and so did the 24 single-path SIMT cases whose Lk is not a key bucket.
"""
import math
import re
from types import SimpleNamespace

import numpy as np
import pytest
import torch
from torch.profiler import ProfilerActivity, profile

import icap_loader

pytestmark = pytest.mark.gpu

pkg = icap_loader.load()
N = pkg._native
F32, BF16 = N.F32, N.BF16
TNAME = {F32: "float", BF16: "__nv_bfloat16"}
SWITCHES = ("ICAP_MHA_SIMT", "ICAP_LN_NARROW", "ICAP_LN_RPW", "ICAP_GEMM_LN_BN", "ICAP_GEMM_LN_SMALL")
GOLDEN = 0x9E3779B97F4A7C15
SEEDS = (0x2545F491, 0xDEADBEEF12345678)        # the second has its high 32 bits set
STEP = 7                                         # device step counter (seed_dev) of every call
POISON = 3e4
EPS = 1e-6

# bounds; derivations:
#  fp32: fp32 arithmetic on exact inputs, sums of <= 4096 terms: ~1e-6 observed, 2e-5 leaves room for reordering.
#  bf16 outputs rounded once from fp32: 2^-9 of the element, <= 2^-8 = 3.9e-3 of the largest one: 4e-3.
#  bf16 mma attention: P (forward) and P, dS (backward) are rounded to bf16 before the second product as well: 2x.
#  GEMM + LN -> backward: the saved sum is rounded to bf16 but mean / rstd are those of the unrounded sum; that moves
#  rstd by ~2 * 2^-8 / sqrt(3 N) relative (<= 3e-4 for N >= 256) on top of the output rounding: 5e-3.
#  mean, rstd: fp32 statistics of exact inputs, ~3e-7 observed.
TOL_O = {(F32, "simt"): 2e-5, (BF16, "simt"): 4e-3, (BF16, "mma"): 8e-3}
TOL_G = {(F32, "simt"): 2e-5, (BF16, "simt"): 4e-3, (BF16, "mma"): 8e-3}
TOL_LN = {F32: 2e-5, BF16: 4e-3}
TOL_LN_CHAIN_DS = 5e-3
TOL_STATS = 2e-6


def dev():
    return torch.device("cuda:0")


def S():
    return torch.cuda.current_stream().cuda_stream


def dt(code):
    return torch.float32 if code == F32 else torch.bfloat16


def ptr(t):
    return None if t is None else t.data_ptr()


@pytest.fixture
def switches(monkeypatch):
    """set(NAME=value, ...): exactly these ICAP_* switches present, the others removed; libicap re-reads them."""
    def set_(**env):
        for name in SWITCHES:
            monkeypatch.delenv(name, raising=False)
        for name, value in env.items():
            monkeypatch.setenv(name, value)
        N.call("icap_reload_env")
    set_()
    yield set_
    monkeypatch.undo()
    N.call("icap_reload_env")


def launched_kernels(fn):
    """Demangled names of the CUDA kernels `fn` launches, in order (profiler, CUDA activity only)."""
    torch.cuda.synchronize()
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        fn()
        torch.cuda.synchronize()
    return [e.name for e in prof.events() if e.device_type == torch.autograd.DeviceType.CUDA
            and "memcpy" not in e.name.lower() and "memset" not in e.name.lower()]


def assert_kernels(fn, expected):
    names = launched_kernels(fn)
    ok = len(names) == len(expected) and all(re.search(p, n) for p, n in zip(expected, names))
    assert ok, f"expected kernels {expected}, the profiler saw {names}"


# ------------------------------------------------------------------------------------------ mask oracle
U32 = np.uint32


def hash32(x):
    """lowbias32 of icap_common.cuh on a uint32 array (wrapping arithmetic)."""
    x = np.asarray(x, dtype=np.uint32).copy()
    x ^= x >> U32(16)
    x *= U32(0x7FEB352D)
    x ^= x >> U32(15)
    x *= U32(0x846CA68B)
    x ^= x >> U32(16)
    return x


def seed_fold(seed):
    inner = int(hash32([((seed >> 32) + 0x9E3779B9) & 0xFFFFFFFF])[0])
    return int(hash32([(seed & 0xFFFFFFFF) ^ inner])[0])


def threshold(p):
    """dropout_threshold of the float p the kernels receive."""
    t = float(np.float32(p)) * 4294967296.0
    return int(min(max(t, 0.0), 4294967295.0))


def keep_oracle(seed, step, p, elem):
    """Keep decision of dropout elements `elem` (integer array): effective seed = seed + step * golden (mod 2^64),
    pair index elem / 2 hashed with rand32, the low / high 16 bits by element parity, kept iff >= threshold >> 16."""
    e = np.asarray(elem, dtype=np.uint64)
    sf = U32(seed_fold((seed + step * GOLDEN) % 2 ** 64))
    pair = e >> np.uint64(1)
    lo = (pair & np.uint64(0xFFFFFFFF)).astype(np.uint32)
    hi = (pair >> np.uint64(32)).astype(np.uint32)
    h = hash32(lo * U32(0x9E3779B1) + hi * U32(0x85EBCA77) + sf)
    u16 = np.where((e & np.uint64(1)) == 0, h & U32(0xFFFF), h >> U32(16))
    return u16 >= U32(threshold(p) >> 16)


def attn_drop_ld(Lk):
    for b in (16, 32, 48, 64, 128):
        if Lk <= b:
            return b
    return (Lk + 3) & ~3


def attn_keep(seed, step, p, B, H, Lq, Lk):
    """[B, H, Lq, Lk] bool keep mask of the attention probabilities."""
    bh = np.arange(B * H, dtype=np.uint64)[:, None, None]
    i = np.arange(Lq, dtype=np.uint64)[None, :, None]
    j = np.arange(Lk, dtype=np.uint64)[None, None, :]
    e = (bh * np.uint64(Lq) + i) * np.uint64(attn_drop_ld(Lk)) + j
    return torch.from_numpy(keep_oracle(seed, step, p, e).reshape(B, H, Lq, Lk)).to(dev())


def rows_keep(seed, step, p, M, d):
    """[M, d] bool keep mask of add + LayerNorm / GEMM + LayerNorm: element row*d + col."""
    e = np.arange(M * d, dtype=np.uint64).reshape(M, d)
    return torch.from_numpy(keep_oracle(seed, step, p, e)).to(dev())


# ------------------------------------------------------------------------------------------ error measures
def rowhead_err(out, ref, H):
    """max over (row, head) of max |out - ref| / max |ref| of that (row, head); NaN anywhere -> NaN."""
    rows = ref.shape[0]
    o, r = out.double().reshape(rows, H, -1), ref.double().reshape(rows, H, -1)
    e = (o - r).abs().amax(-1) / r.abs().amax(-1).clamp_min(1e-30)
    return float("nan") if torch.isnan(o).any() else float(e.max())


def block_err(out, ref, B, H):
    """[B*L, H*dk] tensors: max over (b, h) of max |out - ref| / max |ref| over that (b, h) block."""
    o, r = out.double().reshape(B, -1, H, out.shape[1] // H), ref.double().reshape(B, -1, H, ref.shape[1] // H)
    e = (o - r).abs().amax((1, 3)) / r.abs().amax((1, 3)).clamp_min(1e-30)
    return float("nan") if torch.isnan(o).any() else float(e.max())


def row_err(out, ref):
    o, r = out.double(), ref.double()
    e = (o - r).abs().amax(-1) / r.abs().amax(-1).clamp_min(1e-30)
    return float("nan") if torch.isnan(o).any() else float(e.max())


def vec_err(out, ref):
    o, r = out.double(), ref.double()
    return float("nan") if torch.isnan(o).any() else float((o - r).abs().max() / r.abs().max())


# ------------------------------------------------------------------------------------------ attention
def k_fwd(X):
    return rf"mha_fwd_mma_kernel<{attn_drop_ld(X.Lk) // 8}>\(" if X.mma else rf"mha_fwd_kernel<{TNAME[X.act]}>\("


def k_bwd(X):
    return rf"mha_bwd_mma_kernel<{attn_drop_ld(X.Lk) // 8}>\(" if X.mma else rf"mha_bwd_kernel<{TNAME[X.act]}>\("


def key_validity(kind, B, Lk, g):
    """uint8 [B, Lk]: "regions" = random holes and a padded suffix, "pads" = pad tokens at random positions; key 0 is
    always valid (no fully masked query row)."""
    if kind is None:
        return None
    kv = (torch.rand(B, Lk, generator=g) > (0.25 if kind == "regions" else 0.2)).to(torch.uint8)
    if kind == "regions":
        kv[1, Lk // 2:] = 0
        kv[0] = 1
    kv[:, 0] = 1
    return kv


def attn_inputs(act, B, H, dk, Lq, Lk, layout, causal, valid, p, seed):
    g = torch.Generator().manual_seed(1000 * H + 37 * Lq + Lk + 7 * causal + int(p * 10) + (seed & 0xFF))
    d, D = H * dk, dev()
    kvalid = key_validity(valid, B, Lk, g)
    X = SimpleNamespace(act=act, B=B, H=H, dk=dk, d=d, Lq=Lq, Lk=Lk, layout=layout, causal=int(causal), p=p, seed=seed,
                        mma=False)
    if layout == "self":
        assert Lq == Lk
        buf = torch.randn(B * Lq, 3 * d, generator=g)
        if kvalid is not None:
            m = kvalid.view(-1) == 0
            buf[m, d:] = (torch.randint(0, 2, (int(m.sum()), 2 * d), generator=g) * 2 - 1) * POISON
        X.qbuf = X.kvbuf = buf.to(dt(act)).to(D)
        X.ldq = X.ldk = X.ldv = 3 * d
        X.koff, X.voff = d, 2 * d
    else:
        X.qbuf = torch.randn(B * Lq, d, generator=g).to(dt(act)).to(D)
        kv = torch.randn(B * Lk, 2 * d, generator=g)
        if kvalid is not None:
            m = kvalid.view(-1) == 0
            kv[m] = (torch.randint(0, 2, (int(m.sum()), 2 * d), generator=g) * 2 - 1) * POISON
        X.kvbuf = kv.to(dt(act)).to(D)
        X.ldq, X.ldk, X.ldv = d, 2 * d, 2 * d
        X.koff, X.voff = 0, d
    X.kvalid = None if kvalid is None else kvalid.contiguous().to(D)
    X.dout = torch.randn(B * Lq, d, generator=g).to(dt(act)).to(D)
    masked = torch.zeros(B, Lq, Lk, dtype=torch.bool, device=D)
    if X.kvalid is not None:
        masked |= (X.kvalid == 0)[:, None, :]
    if causal:
        masked |= torch.triu(torch.ones(Lq, Lk, dtype=torch.bool, device=D), 1)[None]
    X.masked = masked
    X.step = torch.tensor([STEP], dtype=torch.int32, device=D)
    return X


def q_of(X):
    return X.qbuf[:, :X.d]


def k_of(X):
    return X.kvbuf[:, X.koff:X.koff + X.d]


def v_of(X, kvbuf=None):
    return (X.kvbuf if kvbuf is None else kvbuf)[:, X.voff:X.voff + X.d]


def mha_fwd(X, o, kvbuf=None, step=None, am=None):
    esz = X.kvbuf.element_size()
    kvb = X.kvbuf if kvbuf is None else kvbuf
    N.call("icap_mha_fwd", X.act, X.B, X.H, X.Lq, X.Lk, X.dk, X.dk, X.qbuf.data_ptr(), X.ldq,
           X.kvbuf.data_ptr() + X.koff * esz, X.ldk, kvb.data_ptr() + X.voff * esz, X.ldv, o.data_ptr(), X.d,
           ptr(X.kvalid), X.causal, X.p, X.seed, (X.step if step is None else step).data_ptr(), ptr(am), S())


def grad_buffers(X):
    """NaN-filled gradient buffers in the product's layout -> (buffers, (dq, dk, dv) views)."""
    nan = float("nan")
    if X.layout == "self":
        dqkv = torch.full((X.B * X.Lq, 3 * X.d), nan, device=dev(), dtype=dt(X.act))
        return (dqkv,), (dqkv[:, :X.d], dqkv[:, X.d:2 * X.d], dqkv[:, 2 * X.d:])
    dq = torch.full((X.B * X.Lq, X.d), nan, device=dev(), dtype=dt(X.act))
    dkv = torch.full((X.B * X.Lk, 2 * X.d), nan, device=dev(), dtype=dt(X.act))
    return (dq, dkv), (dq, dkv[:, :X.d], dkv[:, X.d:])


def mha_bwd(X, dout, views):
    esz = X.kvbuf.element_size()
    dq, dk, dv = views
    N.call("icap_mha_bwd", X.act, X.B, X.H, X.Lq, X.Lk, X.dk, X.dk, X.qbuf.data_ptr(), X.ldq,
           X.kvbuf.data_ptr() + X.koff * esz, X.ldk, X.kvbuf.data_ptr() + X.voff * esz, X.ldv, dout.data_ptr(), X.d,
           dq.data_ptr(), dq.stride(0), dk.data_ptr(), dk.stride(0), dv.data_ptr(), dv.stride(0), ptr(X.kvalid),
           X.causal, X.p, X.seed, X.step.data_ptr(), S())


def ref_attention(X, keep, grads=True):
    """fp64 O = (softmax(S) * keep / (1-p)) V over the kernel's buffers, P, and dQ, dK, dV for dO = X.dout."""
    B, H, dk, Lq, Lk = X.B, X.H, X.dk, X.Lq, X.Lk
    q = q_of(X).double().reshape(B, Lq, H, dk).requires_grad_(grads)
    k = k_of(X).double().reshape(B, Lk, H, dk).requires_grad_(grads)
    v = v_of(X).double().reshape(B, Lk, H, dk).requires_grad_(grads)
    s = torch.einsum("bihd,bjhd->bhij", q, k) / math.sqrt(dk)
    P = s.masked_fill(X.masked[:, None], float("-inf")).softmax(-1)
    O = torch.einsum("bhij,bjhd->bihd", P * keep / (1 - X.p), v)
    out = SimpleNamespace(O=O.detach().reshape(B * Lq, H * dk), P=P.detach())
    if grads:
        O.backward(X.dout.double().view(B, Lq, H, dk))
        out.dq, out.dk, out.dv = (t.grad.reshape(t.shape[0] * t.shape[1], H * dk) for t in (q, k, v))
    return out


def probe_forward_mask(X, am=None):
    """Dropped probabilities Pd [B, H, Lq, Lk] of the forward: V = one-hot probes V[j, c] = (j == c + chunk*dk)."""
    B, H, dk, Lq, Lk = X.B, X.H, X.dk, X.Lq, X.Lk
    Pd = torch.zeros(B, H, Lq, Lk, dtype=torch.float64, device=dev())
    o = torch.empty(B * Lq, X.d, device=dev(), dtype=dt(X.act))
    for chunk in range((Lk + dk - 1) // dk):
        kvp = X.kvbuf.clone()
        j = torch.arange(Lk, device=dev())
        onehot = (j[:, None] == torch.arange(dk, device=dev())[None, :] + chunk * dk).to(kvp.dtype)   # [Lk, dk]
        v_of(X, kvp).copy_(onehot.repeat(B, H))
        o.fill_(float("nan"))
        if am is not None:
            am.zero_()
        mha_fwd(X, o, kvbuf=kvp, am=am)
        n = min(dk, Lk - chunk * dk)
        Pd[..., chunk * dk:chunk * dk + n] = o.double().view(B, Lq, H, dk)[..., :n].permute(0, 2, 1, 3)
    return Pd


def probe_backward_mask(X):
    """Dropped probabilities Pd [B, H, Lq, Lk] of the backward: dO = one-hot probes dO[i, c] = (i == c + chunk*dk),
    so dV[j, c] = Pd[c + chunk*dk, j]."""
    B, H, dk, Lq, Lk = X.B, X.H, X.dk, X.Lq, X.Lk
    Pd = torch.zeros(B, H, Lq, Lk, dtype=torch.float64, device=dev())
    for chunk in range((Lq + dk - 1) // dk):
        i = torch.arange(Lq, device=dev())
        onehot = (i[:, None] == torch.arange(dk, device=dev())[None, :] + chunk * dk).to(dt(X.act))
        dout = onehot.repeat(B, H).contiguous()
        _, views = grad_buffers(X)
        mha_bwd(X, dout, views)
        n = min(dk, Lq - chunk * dk)
        Pd[:, :, chunk * dk:chunk * dk + n, :] = views[2].double().reshape(B, Lk, H, dk)[..., :n].permute(0, 2, 3, 1)
    return Pd


def check_mask(label, Pd, keep, X, P, tol):
    """Kept set of the recovered Pd == oracle on every unmasked element, masked elements 0, kept Pd * (1-p) == P."""
    valid = ~X.masked[:, None].expand_as(keep)
    kept = Pd != 0
    bad = int((kept != keep)[valid].sum())
    assert bad == 0, f"{label}: {bad} of {int(valid.sum())} keep decisions differ from the oracle"
    assert not bool(kept[~valid].any()), f"{label}: a masked probability is nonzero"
    err = rowhead_err((Pd * (1 - X.p) * keep).permute(0, 2, 1, 3).reshape(X.B * X.Lq, -1),
                      (P * keep).permute(0, 2, 1, 3).reshape(X.B * X.Lq, -1), X.H)
    assert err <= tol, f"{label}: kept probabilities * (1-p) differ from P by {err:.3e} (bound {tol:.0e})"
    return err


def flip_shift(X, keep, ref):
    """Flip the keep decision of the largest probability of every (b, h); min over (b, h) of the largest per-(row,
    head) relative move of the fp64 O."""
    B, H, Lq, Lk = X.B, X.H, X.Lq, X.Lk
    flat = ref.P.reshape(B * H, Lq * Lk).argmax(-1)
    keep2 = keep.clone().view(B * H, -1)
    keep2[torch.arange(B * H, device=dev()), flat] ^= True
    moved = ref_attention(X, keep2.view_as(keep), grads=False).O
    o, r = moved.view(B, Lq, H, -1), ref.O.view(B, Lq, H, -1)
    rel = (o - r).abs().amax(-1) / r.abs().amax(-1).clamp_min(1e-30)       # [B, Lq, H]
    return float(rel.amax(1).min())


def run_attention(X):
    path = "mma" if X.mma else "simt"
    tol_o, tol_g = TOL_O[(X.act, path)], TOL_G[(X.act, path)]
    label = (f"{TNAME[X.act]} {path} B{X.B} H{X.H} dk{X.dk} {X.Lq}x{X.Lk} {X.layout} causal{X.causal} "
             f"p{X.p} seed{X.seed:#x}")
    keep = attn_keep(X.seed, STEP, X.p, X.B, X.H, X.Lq, X.Lk)
    o = torch.full((X.B * X.Lq, X.d), float("nan"), device=dev(), dtype=dt(X.act))
    assert_kernels(lambda: mha_fwd(X, o), [k_fwd(X)])
    bufs, views = grad_buffers(X)
    assert_kernels(lambda: mha_bwd(X, X.dout, views), [k_bwd(X)])
    ref = ref_attention(X, keep)
    e_o = rowhead_err(o, ref.O, X.H)
    e_g = max(block_err(views[0], ref.dq, X.B, X.H), block_err(views[1], ref.dk, X.B, X.H),
              block_err(views[2], ref.dv, X.B, X.H))
    e_pf = check_mask(label + " forward", probe_forward_mask(X), keep, X, ref.P, tol_o)
    e_pb = check_mask(label + " backward", probe_backward_mask(X), keep, X, ref.P, tol_o)
    shift = flip_shift(X, keep, ref)
    print(f"[dropout-attn] {label}: O {e_o:.3e} (bound {tol_o:.0e}), grads {e_g:.3e} (bound {tol_g:.1e}), "
          f"P fwd {e_pf:.3e} bwd {e_pb:.3e}, one flip moves O {shift:.3e} = {shift / tol_o:.0f}x bound")
    assert e_o <= tol_o, f"{label}: O err {e_o:.3e}"
    assert e_g <= tol_g, f"{label}: gradient err {e_g:.3e}"
    assert shift > 3 * tol_o, f"{label}: the bound cannot see one flipped keep decision ({shift:.3e})"
    # the step counter: another step -> another mask; the same step -> bitwise the same output
    o2, o3 = torch.full_like(o, float("nan")), torch.full_like(o, float("nan"))
    mha_fwd(X, o2, step=X.step + 1)
    mha_fwd(X, o3)
    torch.cuda.synchronize()
    assert not torch.equal(o2, o), f"{label}: step + 1 gave the same output"
    assert torch.equal(o3.view(torch.int16 if X.act == BF16 else torch.int32),
                       o.view(torch.int16 if X.act == BF16 else torch.int32)), f"{label}: not reproducible"


# (act, H, dk, Lq, Lk, layout, causal, key validity, switches)
ATTN_PRODUCT = [
    # model A (bf16, 8 heads x 64): encoder 36x36 over regions, decoder 21x21 causal with pads, cross 21x36
    (BF16, 8, 64, 36, 36, "self", 0, "regions", {}),
    (BF16, 8, 64, 21, 21, "self", 1, "pads", {}),
    (BF16, 8, 64, 21, 36, "cross", 0, "regions", {}),
    # model B (32 heads x 8), fp32 and bf16: 36x36, 50x50 causal, 50x36 cross
    *[(act, 32, 8, Lq, Lk, lay, c, v, {}) for act in (F32, BF16)
      for Lq, Lk, lay, c, v in ((36, 36, "self", 0, "regions"), (50, 50, "self", 1, "pads"), (50, 36, "cross", 0, "regions"))],
    # model C (bf16, 16 heads x 64): 100x100, 21x100 cross
    (BF16, 16, 64, 100, 100, "self", 0, "regions", {}),
    (BF16, 16, 64, 21, 100, "cross", 0, "regions", {}),
    # models A and C on the bf16 SIMT kernels, and in fp32
    (BF16, 8, 64, 36, 36, "self", 0, "regions", {"ICAP_MHA_SIMT": "1"}),
    (BF16, 8, 64, 21, 21, "self", 1, "pads", {"ICAP_MHA_SIMT": "1"}),
    (BF16, 16, 64, 21, 100, "cross", 0, "regions", {"ICAP_MHA_SIMT": "1"}),
    (BF16, 16, 64, 100, 100, "self", 0, "regions", {"ICAP_MHA_SIMT": "1"}),
    (F32, 8, 64, 36, 36, "self", 0, "regions", {}),
    (F32, 8, 64, 21, 36, "cross", 0, "regions", {}),
]
# every key bucket of the mma kernels (16 / 32 / 48 / 64 / 128), Lq up to 128 and not a multiple of 16
ATTN_BUCKETS = [(BF16, 4, 64, Lq, Lk, "self" if Lq == Lk else "cross", c, v, {}) for Lq, Lk, c, v in
                ((16, 16, 0, None), (23, 16, 0, "regions"), (40, 21, 0, "regions"), (64, 64, 1, "pads"),
                 (50, 64, 0, None), (128, 128, 0, "regions"), (97, 100, 0, "regions"), (128, 36, 0, None),
                 (7, 128, 0, "regions"))]
ATTN_CASES = ATTN_PRODUCT + ATTN_BUCKETS


@pytest.mark.parametrize("p", [0.1, 0.5])
@pytest.mark.parametrize("act,H,dk,Lq,Lk,layout,causal,valid,env", ATTN_CASES)
def test_attention_dropout(act, H, dk, Lq, Lk, layout, causal, valid, env, p, switches):
    """icap_mha_fwd + icap_mha_bwd with dropout: both masks == oracle, O and dQ / dK / dV == fp64 through it."""
    switches(**env)
    seed = SEEDS[(ATTN_CASES.index((act, H, dk, Lq, Lk, layout, causal, valid, env)) + int(p == 0.5)) % 2]
    X = attn_inputs(act, 3, H, dk, Lq, Lk, layout, causal, valid, p, seed)
    X.mma = act == BF16 and dk == 64 and not env
    run_attention(X)


# (H, Lq, Lk, layout, causal, key validity): the shapes of models A and C whose Lk is not a key bucket
MIXED = [(8, 21, 21, "self", 1, "pads"), (8, 21, 36, "cross", 0, "regions"), (16, 100, 100, "self", 0, "regions")]


@pytest.mark.parametrize("p", [0.1, 0.5])
@pytest.mark.parametrize("direction", ["simt_fwd_mma_bwd", "mma_fwd_simt_bwd"])
@pytest.mark.parametrize("H,Lq,Lk,layout,causal,valid", MIXED)
def test_attention_dropout_mixed_kernels(H, Lq, Lk, layout, causal, valid, direction, p, switches):
    """Forward and backward on different kernels (forward with attn_mean -> SIMT, backward aligned -> mma; forward mma,
    backward under ICAP_MHA_SIMT): the gradients are the fp64 gradients of the mask the forward applied."""
    seed = SEEDS[int(p == 0.5)]
    X = attn_inputs(BF16, 3, H, 64, Lq, Lk, layout, causal, valid, p, seed)
    label = f"mixed {direction} H{H} {Lq}x{Lk} p{p}"
    am = torch.zeros(X.B, Lq, Lk, device=dev()) if direction == "simt_fwd_mma_bwd" else None
    X.mma = am is None
    o = torch.full((X.B * Lq, X.d), float("nan"), device=dev(), dtype=torch.bfloat16)
    assert_kernels(lambda: mha_fwd(X, o, am=am), [k_fwd(X)])
    fwd_keep = probe_forward_mask(X, am=am) != 0
    if direction == "mma_fwd_simt_bwd":
        switches(ICAP_MHA_SIMT="1")
    X.mma = not X.mma
    _, views = grad_buffers(X)
    assert_kernels(lambda: mha_bwd(X, X.dout, views), [k_bwd(X)])
    ref = ref_attention(X, fwd_keep)
    tol = TOL_G[(BF16, "mma" if X.mma else "simt")]
    errs = [block_err(v, r, X.B, X.H) for v, r in zip(views, (ref.dq, ref.dk, ref.dv))]
    print(f"[dropout-attn] {label}: dQ {errs[0]:.3e} dK {errs[1]:.3e} dV {errs[2]:.3e} (bound {tol:.1e})")
    assert max(errs) <= tol, f"{label}: the backward did not use the forward's mask (errors {errs})"
    oracle = attn_keep(seed, STEP, p, X.B, X.H, Lq, Lk)
    valid_el = ~X.masked[:, None].expand_as(oracle)
    assert torch.equal(fwd_keep[valid_el], oracle[valid_el]), f"{label}: forward mask != oracle"


# ------------------------------------------------------------------------------------------ add + LayerNorm
def ln_kernel_names(d, T, TR=None, TY=None, env=None, fwd=True):
    """(row kernel, column kernel) regexes of icap_add_ln_fwd / icap_add_ln_bwd for width d."""
    rpw = int((env or {}).get("ICAP_LN_RPW", "1"))
    wide = d % 8 == 0 and "ICAP_LN_NARROW" not in (env or {})
    if wide:
        nit = 1 if d <= 256 else 2 if d <= 512 else 4
        if fwd:
            return rf"add_ln_fwd8_kernel<{nit}, {rpw}, {T}, {TR}, {TY}>\(", None
        return rf"add_ln_bwd_rows8_kernel<{nit}, {rpw}, {T}>\(", rf"add_ln_bwd_cols8_kernel<{T}>\("
    nit = 1 if d <= 128 else 2 if d <= 256 else 4 if d <= 512 else 8
    if fwd:
        return rf"add_ln_fwd_kernel<{nit}, {T}, {TR}, {TY}>\(", None
    return rf"add_ln_bwd_rows_kernel<{nit}, {T}>\(", rf"add_ln_bwd_cols_kernel<{T}>\("


def away_from_zero(shape, g, lo=0.5, hi=1.5):
    mag = torch.rand(shape, generator=g) * (hi - lo) + lo
    return torch.where(torch.rand(shape, generator=g) < 0.5, -mag, mag)


def ln_params(d, M, g):
    gamma = (torch.randn(d, generator=g) * 0.5 + 1.0).to(dev())
    beta = (torch.randn(d, generator=g) * 0.1).to(dev())
    rs = (torch.rand(M, generator=g) > 0.2).float()
    rs[0] = 0.0
    return gamma, beta, rs.to(dev())


def ln_ref(s64, gamma, beta, rs):
    mean = s64.mean(-1, keepdim=True)
    rstd = 1.0 / torch.sqrt(((s64 - mean) ** 2).mean(-1, keepdim=True) + EPS)
    y = ((s64 - mean) * rstd * gamma.double() + beta.double()) * rs.double()[:, None]
    return y, mean.squeeze(-1), rstd.squeeze(-1)


def check_saved(label, keep, s, res_rows_full, y, mean, rstd, s_ref, gamma, beta, rs, tol):
    """Mask recovered from the saved sum (dropped <=> s == res bitwise) == oracle; s, y, mean, rstd against fp64."""
    dropped = s.double() == res_rows_full.double()
    bad = int((dropped == keep).sum())
    assert bad == 0, f"{label}: {bad} of {keep.numel()} keep decisions differ from the oracle"
    y_ref, mean_ref, rstd_ref = ln_ref(s_ref, gamma, beta, rs)
    e_s, e_y = row_err(s, s_ref), row_err(y, y_ref)
    e_m = float(((mean.double() - mean_ref).abs() * rstd_ref).max())
    e_r = float((rstd.double() / rstd_ref - 1).abs().max())
    print(f"[dropout-ln] {label}: s {e_s:.3e} y {e_y:.3e} (bound {tol:.0e}), mean {e_m:.3e} rstd {e_r:.3e} "
          f"(bound {TOL_STATS:.0e}), keep rate {float(keep.float().mean()):.4f}")
    assert e_s <= tol and e_y <= tol, label
    assert e_m <= TOL_STATS and e_r <= TOL_STATS, label


LN_M = 777            # not a multiple of 16 (nor of 2: the RPW=2 kernels get a half-filled last warp)
LN_PAIRS = [(F32, F32), (BF16, BF16), (F32, BF16)]
LN_FWD = [(ta, tact, d, rr, {}) for ta, tact in LN_PAIRS for d, rr in ((256, LN_M), (512, 21), (1024, LN_M), (260, 50))] + \
         [(ta, tact, 512, LN_M, {"ICAP_LN_NARROW": "1"}) for ta, tact in LN_PAIRS] + \
         [(ta, tact, d, LN_M, {"ICAP_LN_RPW": "2"}) for ta, tact in ((F32, F32), (BF16, BF16)) for d in (256, 1024)]


@pytest.mark.parametrize("p", [0.2, 0.3])
@pytest.mark.parametrize("a_dt,act,d,res_rows,env", LN_FWD)
def test_add_ln_fwd_dropout(a_dt, act, d, res_rows, env, p, switches):
    """icap_add_ln_fwd(write_sum=1): mask == oracle (dropped elements of the saved sum == res bitwise, |a| >= 0.5 so a
    kept one cannot round back to res); y, sum, mean, rstd == fp64."""
    switches(**env)
    M = LN_M
    seed = SEEDS[(d + int(p * 10)) % 2]
    g = torch.Generator().manual_seed(d * 10 + res_rows + int(p * 10) + a_dt * 3 + act)
    a = away_from_zero((M, d), g).to(dt(a_dt)).to(dev())
    res = torch.randn(res_rows, d, generator=g).to(dt(act)).to(dev())
    gamma, beta, rs = ln_params(d, M, g)
    work = a.clone()
    y = torch.full((M, d), float("nan"), device=dev(), dtype=dt(act))
    mean = torch.full((M,), float("nan"), device=dev())
    rstd = torch.full((M,), float("nan"), device=dev())
    step = torch.tensor([STEP], dtype=torch.int32, device=dev())
    kern, _ = ln_kernel_names(d, TNAME[a_dt], TNAME[act], TNAME[act], env)
    assert_kernels(lambda: N.call("icap_add_ln_fwd", a_dt, act, M, d, work.data_ptr(), res.data_ptr(), res_rows,
                                  gamma.data_ptr(), beta.data_ptr(), rs.data_ptr(), y.data_ptr(), mean.data_ptr(),
                                  rstd.data_ptr(), 1, p, seed, step.data_ptr(), EPS, S()), [kern])
    keep = rows_keep(seed, STEP, p, M, d)
    assert abs(float(keep.float().mean()) - (1 - p)) < 5e-3
    res_full = res[torch.arange(M, device=dev()) % res_rows]
    s_ref = keep * a.double() / (1 - p) + res_full.double()
    tol = TOL_LN[F32 if a_dt == F32 and act == F32 else BF16]
    check_saved(f"add_ln_fwd {TNAME[a_dt]}/{TNAME[act]} d{d} res_rows{res_rows} {env} p{p}", keep, work, res_full, y,
                mean, rstd, s_ref, gamma, beta, rs, tol)
    # the next step (device counter + 1, as a replayed CUDA graph sees it) applies the oracle's next mask
    work2 = a.clone()
    N.call("icap_add_ln_fwd", a_dt, act, M, d, work2.data_ptr(), res.data_ptr(), res_rows, gamma.data_ptr(),
           beta.data_ptr(), rs.data_ptr(), y.data_ptr(), mean.data_ptr(), rstd.data_ptr(), 1, p, seed,
           (step + 1).data_ptr(), EPS, S())
    torch.cuda.synchronize()
    keep2 = rows_keep(seed, STEP + 1, p, M, d)
    assert not torch.equal(keep2, keep)
    assert torch.equal(work2.double() != res_full.double(), keep2), "step + 1 did not apply the oracle's mask"


def check_ln_bwd(label, act, M, d, s, mean, rstd, gamma, rs, dy1, dy2, keep, p, seed, has_da, has_db2, split, env,
                 tol_rows=None):
    """icap_add_ln_bwd, or icap_add_ln_bwd_rows then icap_add_ln_bwd_params on a second stream after an event, against
    fp64 autograd of y = (LN(keep * a / (1-p) + r) * gamma + beta) * rs at the saved sum."""
    D = dev()
    g = torch.Generator().manual_seed(M + d)
    pre = [torch.randn(d, generator=g).to(D) for _ in range(3)]          # accumulated into: start nonzero
    dgam, dbet, db2 = (t.clone() for t in pre)
    ds = torch.full((M, d), float("nan"), device=D, dtype=dt(act))
    da = torch.full((M, d), float("nan"), device=D, dtype=dt(act)) if has_da else None
    db2_p = db2 if has_db2 else None
    step = torch.tensor([STEP], dtype=torch.int32, device=D)
    rows_k, cols_k = ln_kernel_names(d, TNAME[act], env=env, fwd=False)
    if not split:
        assert_kernels(lambda: N.call("icap_add_ln_bwd", act, M, d, dy1.data_ptr(), ptr(dy2), s.data_ptr(),
                                      mean.data_ptr(), rstd.data_ptr(), gamma.data_ptr(), rs.data_ptr(), ds.data_ptr(),
                                      ptr(da), dgam.data_ptr(), dbet.data_ptr(), ptr(db2_p), p, seed, step.data_ptr(),
                                      S()), [rows_k, cols_k])
    else:
        assert_kernels(lambda: N.call("icap_add_ln_bwd_rows", act, M, d, dy1.data_ptr(), ptr(dy2), s.data_ptr(),
                                      mean.data_ptr(), rstd.data_ptr(), gamma.data_ptr(), rs.data_ptr(), ds.data_ptr(),
                                      ptr(da), p, seed, step.data_ptr(), S()), [rows_k])
        side = torch.cuda.Stream()

        def params():
            ev = torch.cuda.Event()
            ev.record(torch.cuda.current_stream())
            side.wait_event(ev)
            with torch.cuda.stream(side):
                N.call("icap_add_ln_bwd_params", act, M, d, dy1.data_ptr(), ptr(dy2), s.data_ptr(), mean.data_ptr(),
                       rstd.data_ptr(), rs.data_ptr(), ds.data_ptr(), ptr(da), dgam.data_ptr(), dbet.data_ptr(),
                       ptr(db2_p), side.cuda_stream)
            torch.cuda.current_stream().wait_stream(side)
        assert_kernels(params, [cols_k])
    a64 = torch.zeros(M, d, dtype=torch.float64, device=D, requires_grad=True)
    r64 = s.double().requires_grad_(True)
    g64, b64 = gamma.double().requires_grad_(True), torch.zeros(d, dtype=torch.float64, device=D, requires_grad=True)
    x = keep * a64 / (1 - p) + r64
    y = torch.nn.functional.layer_norm(x, (d,), g64, b64, EPS) * rs.double()[:, None]
    y.backward(dy1.double() + (dy2.double() if dy2 is not None else 0.0))
    tol = TOL_LN[act]
    tol_rows = tol if tol_rows is None else tol_rows
    errs = {"ds": row_err(ds, r64.grad), "dgamma": vec_err(dgam, pre[0].double() + g64.grad),
            "dbeta": vec_err(dbet, pre[1].double() + b64.grad)}
    if has_da:
        errs["da"] = row_err(da, a64.grad)
        nz = (r64.grad != 0) & (rs[:, None] != 0)
        bad = int(((da != 0) != keep)[nz].sum())
        assert bad == 0, f"{label}: {bad} keep decisions of the backward differ from the oracle"
    if has_db2:
        errs["dbias2"] = vec_err(db2, pre[2].double() + (a64.grad if has_da else r64.grad).sum(0))
    print(f"[dropout-ln-bwd] {label}: " + " ".join(f"{k} {v:.3e}" for k, v in errs.items()) +
          f" (bound ds / da {tol_rows:.0e}, parameters {tol:.0e})")
    assert max(v for k, v in errs.items() if k in ("ds", "da")) <= tol_rows, f"{label}: {errs}"
    assert max(v for k, v in errs.items() if k not in ("ds", "da")) <= tol, f"{label}: {errs}"


# (act, d, switches, dy2, da, dbias2, split)
LN_BWD = [(act, d, {}, True, True, True, split) for act in (F32, BF16) for d in (256, 512, 1024, 260)
          for split in (False, True)] + \
         [(act, 512, {}, dy2, da, db2, True) for act in (F32, BF16)
          for dy2, da, db2 in ((False, True, True), (True, False, True), (True, True, False))] + \
         [(act, 512, {"ICAP_LN_NARROW": "1"}, True, True, True, split) for act in (F32, BF16) for split in (False, True)] + \
         [(act, 1024, {"ICAP_LN_RPW": "2"}, True, True, True, split) for act in (F32, BF16) for split in (False, True)]


@pytest.mark.parametrize("p", [0.2, 0.3])
@pytest.mark.parametrize("act,d,env,has_dy2,has_da,has_db2,split", LN_BWD)
def test_add_ln_bwd_dropout(act, d, env, has_dy2, has_da, has_db2, split, p, switches):
    """icap_add_ln_bwd and icap_add_ln_bwd_rows / _params: ds, da (mask == oracle), dgamma, dbeta, dbias2 == fp64."""
    switches(**env)
    M = LN_M
    seed = SEEDS[(d + int(p * 10) + int(split)) % 2]
    g = torch.Generator().manual_seed(d + int(p * 10) + 100 * act)
    s = (torch.randn(M, d, generator=g) * 1.5 + 0.3).to(dt(act)).to(dev())
    s64 = s.double()
    mean = s64.mean(-1).float()
    rstd = (1.0 / torch.sqrt(s64.var(-1, unbiased=False) + EPS)).float()
    gamma, _, rs = ln_params(d, M, g)
    dy1 = torch.randn(M, d, generator=g).to(dt(act)).to(dev())
    dy2 = torch.randn(M, d, generator=g).to(dt(act)).to(dev()) if has_dy2 else None
    keep = rows_keep(seed, STEP, p, M, d)
    label = f"add_ln_bwd {TNAME[act]} d{d} {env} dy2={has_dy2} da={has_da} dbias2={has_db2} split={split} p{p}"
    check_ln_bwd(label, act, M, d, s, mean, rstd, gamma, rs, dy1, dy2, keep, p, seed, has_da, has_db2, split, env)


# ------------------------------------------------------------------------------------------ GEMM + LayerNorm chain
# (M, N, K): model A (d 512, FFN 2048; decoder and encoder row counts), model B (d 256), model C (d 1024, FFN 4096)
GEMM_LN = [(9216, 512, 512), (5376, 512, 2048), (2600, 256, 256), (2600, 256, 1024), (3000, 1024, 4096)]


@pytest.mark.parametrize("bn", [128, 256])
@pytest.mark.parametrize("M,Nn,K", GEMM_LN)
def test_gemm_ln_dropout_chain(M, Nn, K, bn, switches):
    """Training form of icap_gemm_ln (p = 0.2, sum / mean / rstd saved) on gemm_ln_kernel<N/BN, BN>: mask == oracle,
    y / sum / mean / rstd == fp64 of LN(keep * (A W^T + b) / (1-p) + res); then the saved tensors through
    icap_add_ln_bwd_rows and icap_add_ln_bwd_params (second stream) with the same seed == fp64."""
    switches(ICAP_GEMM_LN_BN=str(bn), ICAP_GEMM_LN_SMALL="0")
    p, D = 0.2, dev()
    seed = SEEDS[(M + bn) % 2]
    g = torch.Generator().manual_seed(M + Nn + K + bn)
    A = torch.randn(M, K, generator=g).bfloat16().to(D)
    W = (torch.randn(Nn, K, generator=g) * (0.25 / math.sqrt(K))).bfloat16().to(D)
    bias = away_from_zero((Nn,), g, 1.5, 2.5).to(D)          # |A W^T + b| >= ~0.5: a kept sum cannot round to res
    res = torch.randn(M, Nn, generator=g).bfloat16().to(D)
    gamma, beta, rs = ln_params(Nn, M, g)
    y = torch.full((M, Nn), float("nan"), device=D, dtype=torch.bfloat16)
    ssum = torch.full((M, Nn), float("nan"), device=D, dtype=torch.bfloat16)
    mean = torch.full((M,), float("nan"), device=D)
    rstd = torch.full((M,), float("nan"), device=D)
    step = torch.tensor([STEP], dtype=torch.int32, device=D)
    assert_kernels(lambda: N.call("icap_gemm_ln", M, Nn, K, A.data_ptr(), K, W.data_ptr(), K, bias.data_ptr(),
                                  res.data_ptr(), Nn, gamma.data_ptr(), beta.data_ptr(), rs.data_ptr(), y.data_ptr(), Nn,
                                  ssum.data_ptr(), Nn, mean.data_ptr(), rstd.data_ptr(), EPS, p, seed, step.data_ptr(),
                                  S()), [rf"gemm_ln_kernel<{Nn // bn}, {bn}>\("])
    keep = rows_keep(seed, STEP, p, M, Nn)
    x64 = A.double() @ W.double().t() + bias.double()
    s_ref = keep * x64 / (1 - p) + res.double()
    label = f"gemm_ln M{M} N{Nn} K{K} BN{bn}"
    check_saved(label, keep, ssum, res, y, mean, rstd, s_ref, gamma, beta, rs, TOL_LN[BF16])
    dy1 = torch.randn(M, Nn, generator=g).bfloat16().to(D)
    dy2 = torch.randn(M, Nn, generator=g).bfloat16().to(D)
    check_ln_bwd(label + " -> bwd_rows / bwd_params", BF16, M, Nn, ssum, mean, rstd, gamma, rs, dy1, dy2, keep, p,
                 seed, True, True, True, {}, tol_rows=TOL_LN_CHAIN_DS)
