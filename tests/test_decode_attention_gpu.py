"""Decode-step attention against an fp64 reference, one case per dispatch path, and a check of which kernel ran.

icap_mha_decode (cross-attention, and self-attention over the KV cache) and icap_mha_decode_self (self-attention with
the append of the new key / value fused in) choose among six kernels from the dtype, head dim, beam width, position,
alignment and the ICAP_DECODE_* switches.  Every case names the kernel the dispatch has to pick for it; one call per
case runs under torch.profiler and the demangled kernel names must match, so a case cannot silently test another path.

Data has the product's layout: q inside the packed [rows, 3d] QKV buffer (self) or [rows, d] (cross), KV cache
[rows, 50, 2d], cross K|V [images * R, 2d].  Token / slot tables come from a simulated beam search with the bookkeeping
of icap_beam_reorder: shared prefixes, pad ids in mid-sequence, slot entries pointing to other rows.  What a kernel must
not read is poisoned.  Self mode: every cache entry that no (row, position) pair references, and every pad-masked one,
holds NaN.  Cross mode: masked regions hold finite +-3e4, because the mma kernel multiplies masked tiles by zero.  After
icap_mha_decode_self the whole cache is compared bitwise with the expected one.

Error of a case = max over (row, head) of max |out - ref| / max |ref| of that (row, head).  Bounds, derived from the
arithmetic: fp32 2e-5; bf16 generic / decode64 / row / image-per-CTA 4e-3 (fp32 math, output rounded to bf16, whose
unit roundoff is 2^-8 = 3.9e-3 of the element); bf16 mma 8e-3 (P is rounded to bf16 as well).  attn_mean (fp32):
2e-5 of the row's largest mean probability.  Each case also checks that masking one more valid key per row moves the
fp64 reference by more than 3x the bound.  Observed on one NVIDIA B200 (1000 W power limit):

    cases                                             bound   observed max   smallest one-key-fewer shift / bound
    fp32, every path                                  2e-5    1.2e-6         17000x
    bf16 cross: image-per-CTA, decode64, generic      4e-3    3.87e-3        79x
    bf16 cross: mma                                   8e-3    7.63e-3        43x
    bf16 self, icap_mha_decode                        4e-3    3.89e-3        130x
    bf16 icap_mha_decode_self (row, decode64, generic) 4e-3   3.86e-3        145x
    attn_mean                                         2e-5    4.1e-7
The bf16 maxima sit at the output rounding (2^-8 of the head's largest element), the mma one at about twice that.
"""
import ctypes
import math
import re

import pytest
import torch
from torch.profiler import ProfilerActivity, profile

import icap_loader

pytestmark = pytest.mark.gpu

pkg = icap_loader.load()
N = pkg._native
F32, BF16 = N.F32, N.BF16
TNAME = {F32: "float", BF16: "__nv_bfloat16"}
T_CACHE = 50                    # cache positions per row (MAX_LENGTH 49)
PAD = 0
TOL = {(F32, "any"): 2e-5, (BF16, "simt"): 4e-3, (BF16, "mma"): 8e-3}
AM_TOL = 2e-5
SWITCHES = ("ICAP_DECODE_IMG_CROSS", "ICAP_DECODE_NO_MMA", "ICAP_DECODE_SLOW", "ICAP_DECODE_NO_ROW", "ICAP_DECODE_UB",
            "ICAP_DECODE_NO_IMG_BLOCKS", "ICAP_MHA_SIMT")


def dev():
    return torch.device("cuda:0")


def S():
    return torch.cuda.current_stream().cuda_stream


def dt(code):
    return torch.float32 if code == F32 else torch.bfloat16


def ptr(t):
    return None if t is None else t.data_ptr()


def ptr_dev(t):
    return None if t is None else t.to(dev())


def tol_of(act, mma=False):
    return TOL[(F32, "any")] if act == F32 else TOL[(BF16, "mma" if mma else "simt")]


@pytest.fixture
def switches(monkeypatch):
    """set(NAME=value, ...): exactly these ICAP_DECODE_* switches present (they act when the variable exists, whatever
    its value), the others removed; libicap re-reads them.  Restored at teardown."""
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


# ------------------------------------------------------------------------------------------ which kernel ran
def k_img(G):
    return rf"mha_cross_img_kernel<{G}>\("


def k_mma(Lk):
    nt = 2 if Lk <= 16 else 4 if Lk <= 32 else 6 if Lk <= 48 else 8 if Lk <= 64 else 16
    return rf"mha_fwd_mma_kernel<{nt}>\("


def k_d64(act, G):
    return rf"mha_decode64_kernel<{TNAME[act]}, {G}>\("


def k_gen(act):
    return rf"mha_decode_kernel<{TNAME[act]}>\("


def k_row(act, ub):
    return rf"mha_decode_row_kernel<{TNAME[act]}, 8, {ub}>\("


def k_copy(act):
    return rf"copy2d_kernel<{TNAME[act]}, {TNAME[act]}>\("


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


# ------------------------------------------------------------------------------------------ fp64 reference
def ref_decode_attention(q, kc, vc, H, Lk, kv_rows_per_seq, slot=None, tokens=None, kvalid=None, rows_per_image=1,
                         extra_mask=None):
    """fp64 decode attention over the buffers the kernel reads.  q [rows, H*dk], kc [n, H*dk] and vc [n, H*dv] with
    row i = physical cache row i (views with the kernel's strides).  Self mode (tokens given): key j of a row lives in
    row slot[row, j] * kv_rows_per_seq + j (own row without slot) and is masked iff tokens[row, j] == PAD.  Cross mode:
    key j of row r lives in row (r // rows_per_image) * kv_rows_per_seq + j, masked iff kvalid[image, j] == 0.
    extra_mask [rows, Lk] masks more keys.  Returns (out [rows, H*dv], head-mean of P [rows, Lk], mask [rows, Lk])."""
    rows = q.shape[0]
    dk, dv = q.shape[1] // H, vc.shape[1] // H
    j = torch.arange(Lk, device=q.device)
    r = torch.arange(rows, device=q.device)
    if tokens is not None:
        base = slot[:, :Lk].long() if slot is not None else r[:, None].expand(rows, Lk)
        masked = tokens[:, :Lk] == PAD
    else:
        img = r // rows_per_image
        base = img[:, None].expand(rows, Lk)
        masked = (kvalid.view(-1, Lk)[img] == 0) if kvalid is not None else torch.zeros(rows, Lk, dtype=torch.bool,
                                                                                          device=q.device)
    if extra_mask is not None:
        masked = masked | extra_mask
    phys = (base * kv_rows_per_seq + j).reshape(-1)
    K = kc[phys].double().view(rows, Lk, H, dk)
    V = vc[phys].double().view(rows, Lk, H, dv).masked_fill(masked[:, :, None, None], 0.0)   # poison: 0 * NaN
    s = torch.einsum("rhd,rjhd->rhj", q.double().view(rows, H, dk) / math.sqrt(dk), K)
    p = s.masked_fill(masked[:, None, :], float("-inf")).softmax(-1)
    out = torch.einsum("rhj,rjhd->rhd", p, V).reshape(rows, H * dv)
    return out, p.mean(1), masked


def head_err(out, ref, H):
    """max over (row, head) of max |out - ref| / max |ref| of that (row, head); NaN anywhere -> NaN."""
    rows = ref.shape[0]
    o, r = out.double().reshape(rows, H, -1), ref.double().reshape(rows, H, -1)
    e = (o - r).abs().amax(-1) / r.abs().amax(-1).clamp_min(1e-30)
    return float(e.max()) if not torch.isnan(o).any() else float("nan")


def drop_last_key(masked):
    """[rows, Lk] mask of the last valid key of every row that has at least two valid keys."""
    valid = ~masked
    Lk = valid.shape[1]
    last = (valid * torch.arange(1, Lk + 1, device=valid.device)).argmax(-1)
    drop = torch.zeros_like(masked)
    keep = valid.sum(-1) >= 2
    drop[keep.nonzero().squeeze(1), last[keep]] = True
    return drop


def verify(label, out, ref_args, H, tol, am=None):
    """out against the fp64 reference; the bound must be able to see one key too few (3x margin)."""
    ref, pmean, masked = ref_decode_attention(*ref_args[0], **ref_args[1])
    err = head_err(out, ref, H)
    drop = drop_last_key(masked)
    shift = None
    if drop.any():
        moved, _, _ = ref_decode_attention(*ref_args[0], **ref_args[1], extra_mask=drop)
        shift = head_err(moved, ref, H)
    msg = f"[decode-attn] {label}: err {err:.3e} (bound {tol:.0e})" + (f", one key fewer {shift:.3e}" if shift is not None else "")
    am_err = None
    if am is not None:
        am_err = float((am.double() - pmean).abs().amax(-1).div(pmean.amax(-1)).max())
        msg += f", attn_mean err {am_err:.3e}"
    print(msg)
    assert err <= tol, msg
    if shift is not None:
        assert shift > 3 * tol, f"{msg}: the bound cannot see a dropped key"
    if am is not None:
        assert am_err <= AM_TOL, msg


# ------------------------------------------------------------------------------------------ inputs
def region_mask(B, R, g):
    """kvalid [B, R]: image 0 all valid, 1 a padded suffix, 2 a hole and a padded suffix, 3 a single valid region
    (region 0 = the whole image), the rest random holes."""
    kv = (torch.rand(B, R, generator=g) > 0.25).to(torch.uint8)
    kv[0] = 1
    kv[1] = 1
    kv[1, R // 2:] = 0
    kv[2] = 1
    if R > 3:
        kv[2, 1] = 0
        kv[2, R - 2:] = 0
    kv[3] = 0
    kv[:, 0] = 1
    return kv


def beam_history(B, k, t, Tmax, g, V=50, pad_frac=0.2):
    """tokens / slot [B*k, Tmax] int32 after t beam steps, with the bookkeeping of icap_beam_reorder: at every step the
    rows copy their parent's prefix, then position s holds the new token (id PAD with probability pad_frac) and
    slot[:, s] = the row itself.  Step 1 expands beam 0 only (all beams start from <START>)."""
    rows = B * k
    tok = torch.zeros(rows, Tmax, dtype=torch.int32)
    slot = torch.zeros(rows, Tmax, dtype=torch.int32)
    tok[:, 0] = 1                                   # <START>
    slot[:, 0] = torch.arange(rows, dtype=torch.int32)
    for s in range(1, t + 1):
        parent = torch.zeros(B, k, dtype=torch.long) if s == 1 else torch.randint(0, k, (B, k), generator=g)
        new = torch.randint(1, V, (B, k), generator=g, dtype=torch.int32)
        new[torch.rand(B, k, generator=g) < pad_frac] = PAD
        src = (torch.arange(B)[:, None] * k + parent).view(-1)
        tok[:, :s] = tok[src, :s]
        slot[:, :s] = slot[src, :s]
        tok[:, s] = new.view(-1)
        slot[:, s] = torch.arange(rows, dtype=torch.int32)
    return tok, slot


def poisoned_cache(rows, d, Lk, tok, slot, act, g, nan_cols=()):
    """KV cache [rows, T_CACHE, 2d]: random where a (row, position < Lk) pair references it through slot / tokens, NaN
    everywhere else; positions in nan_cols are NaN in every row."""
    cache = torch.randn(rows, T_CACHE, 2 * d, generator=g).to(dt(act))
    ref = torch.zeros(rows * T_CACHE, dtype=torch.bool)
    base = slot[:, :Lk].long() if slot is not None else torch.arange(rows)[:, None].expand(rows, Lk)
    phys = base * T_CACHE + torch.arange(Lk)
    ref[phys[tok[:, :Lk] != PAD]] = True
    for c in nan_cols:
        ref.view(rows, T_CACHE)[:, c] = False
    cache.view(rows * T_CACHE, 2 * d)[~ref] = float("nan")
    return cache


def cache_views(cache, d):
    flat = cache.view(-1, 2 * d)
    return flat[:, :d], flat[:, d:]


def bits(t):
    return t.view(torch.int16 if t.dtype == torch.bfloat16 else torch.int32)


# ------------------------------------------------------------------------------------------ cross-attention
def run_cross(act, H, dk, k, R, kernel, attn_mean=False, mma=False, B=7, seed=0):
    g = torch.Generator().manual_seed(seed * 1000 + 97 * k + R + H)
    d, rows, esz = H * dk, B * k, 4 if act == F32 else 2
    q = torch.randn(rows, d, generator=g).to(dt(act)).to(dev())
    kvb = torch.randn(B * R, 2 * d, generator=g).to(dt(act))
    kvalid = region_mask(B, R, g)
    kvb_p = kvb.clone()
    m = kvalid.view(-1) == 0
    kvb_p[m] = (torch.randint(0, 2, (int(m.sum()), 2 * d), generator=g) * 6e4 - 3e4).to(dt(act))   # finite poison
    kvb, kvb_p, kvalid = kvb.to(dev()), kvb_p.to(dev()), kvalid.to(dev())
    o = torch.full((rows, d), float("nan"), device=dev(), dtype=dt(act))
    am = torch.zeros(rows, R, device=dev()) if attn_mean else None

    def call(kv, kval):
        N.call("icap_mha_decode", act, rows, H, R, dk, dk, q.data_ptr(), d, kv.data_ptr(), 2 * d,
               kv.data_ptr() + d * esz, 2 * d, R, o.data_ptr(), d, None, 0, None, 0, PAD, ptr(kval), k, ptr(am), S())

    tol = tol_of(act, mma)
    label = f"cross {TNAME[act]} H{H} dk{dk} k{k} R{R}"
    assert_kernels(lambda: call(kvb_p, kvalid), [kernel])
    kc, vc = kvb_p[:, :d], kvb_p[:, d:]
    verify(label, o, ((q, kc, vc, H, R, R), dict(kvalid=kvalid, rows_per_image=k)), H, tol, am)
    # kvalid = NULL: every region is a key (clean K|V; kvalid does not take part in the dispatch)
    o.fill_(float("nan"))
    if am is not None:
        am.zero_()
    call(kvb, None)
    torch.cuda.synchronize()
    verify(label + " kvalid=NULL", o, ((q, kvb[:, :d], kvb[:, d:], H, R, R), dict(rows_per_image=k)), H, tol, am)


IMG_CASES = [(k, H, R) for k in (1, 2, 3, 4, 5, 8) for H in (8, 16) for R in (5, 36, 100, 128)] + \
            [(3, 8, 37), (8, 4, 5)]


@pytest.mark.parametrize("k,H,R", IMG_CASES)
def test_cross_image_per_cta(k, H, R, switches):
    """Opt-in image-per-CTA kernel (TMA staging of the image's K|V block in chunks, online softmax per key slot)."""
    switches(ICAP_DECODE_IMG_CROSS="1")
    run_cross(BF16, H, 64, k, R, k_img(k if k <= 5 else 8))


MMA_CASES = [(k, 8, R) for k in range(2, 9) for R in (5, 16, 32, 36, 48, 64, 100, 128)] + \
            [(5, 16, 100), (3, 8, 37), (8, 4, 5), (2, 8, 128)]


@pytest.mark.parametrize("k,H,R", MMA_CASES)
def test_cross_mma(k, H, R, switches):
    """Default bf16 beam cross-attention: the beams of an image as a tiny full attention on mma.sync, every Lk bucket."""
    run_cross(BF16, H, 64, k, R, k_mma(R), mma=True)


D64_CROSS = [(F32, k, R, am, {}) for k in (1, 2, 3, 4, 5, 8) for R, am in ((36, True), (128, False))] + \
            [(BF16, k, R, False, {"ICAP_DECODE_NO_MMA": "1"}) for k in (2, 3, 4, 5, 8) for R in (36, 100)] + \
            [(BF16, 1, R, False, {}) for R in (5, 36, 100, 128)] + \
            [(BF16, k, 36, True, {}) for k in (1, 2, 3, 4, 5, 8)] + [(BF16, 5, 100, True, {})]


@pytest.mark.parametrize("act,k,R,am,env", D64_CROSS)
def test_cross_decode64(act, k, R, am, env, switches):
    """Head-dim-64 warp-per-(beam group, head) kernel: fp32, bf16 with ICAP_DECODE_NO_MMA, greedy bf16, attn_mean."""
    switches(**env)
    run_cross(act, 8, 64, k, R, k_d64(act, k), attn_mean=am)


GEN_CROSS = [(act, 32, 8, k, R, am, {}) for act in (F32, BF16) for k in (1, 3, 5) for R, am in ((36, True), (100, False))] + \
            [(BF16, 32, 8, 5, 128, True, {})] + \
            [(F32, 8, 64, k, R, False, {}) for k in (6, 7) for R in (36, 100)] + \
            [(BF16, 8, 64, k, R, True, {}) for k in (6, 7) for R in (36, 128)] + \
            [(F32, 8, 64, 5, 36, True, {"ICAP_DECODE_SLOW": "1"}), (BF16, 8, 64, 1, 36, False, {"ICAP_DECODE_SLOW": "1"})]


@pytest.mark.parametrize("act,H,dk,k,R,am,env", GEN_CROSS)
def test_cross_generic(act, H, dk, k, R, am, env, switches):
    """Generic warp-per-(row, head) kernel: head dim 8 x 32 heads (the default model), beam widths 6 / 7 in fp32 and
    with attn_mean, ICAP_DECODE_SLOW; Lk up to 128 uses every 32-key chunk."""
    switches(**env)
    run_cross(act, H, dk, k, R, k_gen(act), attn_mean=am)


# ------------------------------------------------------------------------------------------ self-attention
def self_inputs(act, B, k, H, dk, t, seed):
    """Beam state after t steps, packed QKV [rows, 3d] of position t, poisoned cache."""
    g = torch.Generator().manual_seed(seed * 1000 + 31 * t + 7 * k + H + dk)
    rows, d = B * k, H * dk
    tok, slot = beam_history(B, k, t, T_CACHE + 1, g)
    qkv = torch.randn(rows, 3 * d, generator=g).to(dt(act))
    return g, rows, d, tok, (slot if k > 1 else None), qkv


SELF_DECODE = [(act, 8, 64, k, t, k_d64(act, 1), {}) for act in (F32, BF16) for k in (1, 5) for t in (5, 31, 49)] + \
              [(act, 32, 8, k, t, k_gen(act), {}) for act in (F32, BF16) for k in (1, 5) for t in (5, 35, 49)] + \
              [(act, 8, 64, 5, t, k_gen(act), {"ICAP_DECODE_SLOW": "1"}) for act in (F32, BF16) for t in (5, 49)]


@pytest.mark.parametrize("act,H,dk,k,t,kernel,env", SELF_DECODE)
def test_self_decode(act, H, dk, k, t, kernel, env, switches):
    """icap_mha_decode in self mode (cache already holds position t): decode64<T, 1> at head dim 64, the generic kernel
    at head dim 8 and with ICAP_DECODE_SLOW; attn_mean checked."""
    switches(**env)
    B = 7
    g, rows, d, tok, slot, qkv = self_inputs(act, B, k, H, dk, t, 1)
    Lk = t + 1
    cache = poisoned_cache(rows, d, Lk, tok, slot, act, g)
    tok_d, slot_d, qkv_d, cache_d = tok.to(dev()), ptr_dev(slot), qkv.to(dev()), cache.to(dev())
    esz = qkv.element_size()
    o = torch.full((rows, d), float("nan"), device=dev(), dtype=dt(act))
    am = torch.zeros(rows, Lk, device=dev())
    assert_kernels(lambda: N.call(
        "icap_mha_decode", act, rows, H, Lk, dk, dk, qkv_d.data_ptr(), 3 * d, cache_d.data_ptr(), 2 * d,
        cache_d.data_ptr() + d * esz, 2 * d, T_CACHE, o.data_ptr(), d, ptr(slot_d), T_CACHE + 1, tok_d.data_ptr(),
        T_CACHE + 1, PAD, None, 1, am.data_ptr(), S()), [kernel])
    kc, vc = cache_views(cache_d, d)
    verify(f"self {TNAME[act]} H{H} dk{dk} k{k} t{t}", o,
           ((qkv_d[:, :d], kc, vc, H, Lk, T_CACHE), dict(slot=slot_d, tokens=tok_d)), H, tol_of(act), am)
    assert torch.equal(bits(cache_d), bits(cache.to(dev())))           # read only


def run_decode_self(act, H, dk, k, pos, kernels, B=9, seed=2):
    g, rows, d, tok, slot, qkv = self_inputs(act, B, k, H, dk, pos, seed)
    cache = poisoned_cache(rows, d, pos, tok, slot, act, g, nan_cols=(pos,))
    expected = cache.clone()
    expected[:, pos] = qkv[:, d:]                                       # exactly position pos of every row: k_new | v_new
    tok_d, slot_d, qkv_d, cache_d = tok.to(dev()), ptr_dev(slot), qkv.to(dev()), cache.to(dev())
    esz = qkv.element_size()
    o = torch.full((rows, d), float("nan"), device=dev(), dtype=dt(act))
    assert_kernels(lambda: N.call(
        "icap_mha_decode_self", act, rows, H, pos, dk, dk, qkv_d.data_ptr(), 3 * d, qkv_d.data_ptr() + d * esz,
        qkv_d.data_ptr() + 2 * d * esz, 3 * d, cache_d.data_ptr(), 2 * d, cache_d.data_ptr() + d * esz, 2 * d, T_CACHE,
        o.data_ptr(), d, ptr(slot_d), T_CACHE + 1, tok_d.data_ptr(), T_CACHE + 1, PAD, k, S()), kernels)
    assert torch.equal(bits(cache_d), bits(expected.to(dev()))), "the cache changed outside position pos"
    kc, vc = cache_views(cache_d, d)
    verify(f"decode_self {TNAME[act]} H{H} dk{dk} k{k} pos{pos}", o,
           ((qkv_d[:, :d], kc, vc, H, pos + 1, T_CACHE), dict(slot=slot_d, tokens=tok_d)), H, tol_of(act))


ROW_CASES = [(act, H, k, pos, {}) for act in (F32, BF16) for H in (4, 8, 16) for k in (1, 2, 5) for pos in (0, 5, 30, 31)] + \
            [(act, H, k, pos, {"ICAP_DECODE_UB": "8"}) for act in (F32, BF16) for H in (4, 8, 16) for k in (1, 5)
             for pos in (5, 31)] + \
            [(BF16, H, k, pos, {"ICAP_DECODE_NO_IMG_BLOCKS": "1"}) for H in (8, 16) for k in (2, 5) for pos in (5, 31)] + \
            [(act, 8, 2, 30, {"ICAP_DECODE_UB": "8", "ICAP_DECODE_NO_IMG_BLOCKS": "1"}) for act in (F32, BF16)]


@pytest.mark.parametrize("act,H,k,pos,env", ROW_CASES)
def test_decode_self_row(act, H, k, pos, env, switches):
    """Row-per-warp kernel with the fused append (pos + 1 <= 32, H * 64 % 256 == 0): 4 / 8 positions per batch,
    image-wide or 8-warp blocks, 1 / 2 / 4 warps per row."""
    switches(**env)
    run_decode_self(act, H, 64, k, pos, [k_row(act, 8 if env.get("ICAP_DECODE_UB") == "8" else 4)])


D64_SELF = [(act, H, k, pos, {}) for act in (F32, BF16) for H in (8, 16) for k in (1, 5) for pos in (32, 33, 49)] + \
           [(act, H, 5, pos, {}) for act in (F32, BF16) for H in (2, 6) for pos in (5, 31)] + \
           [(act, 8, 5, pos, {"ICAP_DECODE_NO_ROW": "1"}) for act in (F32, BF16) for pos in (5, 31)]


@pytest.mark.parametrize("act,H,k,pos,env", D64_SELF)
def test_decode_self_decode64(act, H, k, pos, env, switches):
    """decode64<T, 1> with the fused append: positions past the row kernel's 32 (pos 31 is its last), H * 64 not a
    multiple of 256, ICAP_DECODE_NO_ROW."""
    switches(**env)
    run_decode_self(act, H, 64, k, pos, [k_d64(act, 1)])


GEN_SELF = [(act, 32, 8, k, pos, {}) for act in (F32, BF16) for k in (1, 5) for pos in (5, 31, 32, 49)] + \
           [(act, 8, 64, 5, pos, {"ICAP_DECODE_SLOW": "1"}) for act in (F32, BF16) for pos in (5, 40)]


@pytest.mark.parametrize("act,H,dk,k,pos,env", GEN_SELF)
def test_decode_self_generic(act, H, dk, k, pos, env, switches):
    """Generic path of icap_mha_decode_self: two strided copies into the cache, then the generic kernel (head dim 8 x 32
    heads, the default model; ICAP_DECODE_SLOW)."""
    switches(**env)
    run_decode_self(act, H, dk, k, pos, [k_copy(act), k_copy(act), k_gen(act)])


# ------------------------------------------------------------------------------------------ stream order under PDL
def test_row_kernel_reads_tables_of_its_own_step_under_pdl(switches):
    """The sequence of a beam-search step with programmatic dependent launch on: icap_decode_embed_ln (beam reorder of
    the previous step into fresh token / slot tables) -> bf16 QKV GEMM with ICAP_EPI_B_STATIC (it lets its successor
    start before it waits) -> icap_mha_decode_self on the row-per-warp path, which must use the tables written two
    kernels earlier.  The output tables start out holding another valid beam state, so a stale read selects other,
    poisoned cache rows.  A race cannot be forced: this test guards the stream-ordering contract (the row kernel
    reads tokens / slot again after its grid dependency resolves); it is not a reproducer."""
    B, k, H, dh, t, V = 64, 5, 8, 64, 20, 300
    rows, d, Tmax = B * k, H * dh, T_CACHE + 1
    g = torch.Generator().manual_seed(11)
    tok_in, slot_in = beam_history(B, k, t - 1, Tmax, g)
    parent = torch.randint(0, k, (B, k), generator=g, dtype=torch.int32)
    token = torch.randint(1, V, (B, k), generator=g, dtype=torch.int32)
    token[:, 1] = PAD
    src = (torch.arange(B)[:, None] * k + parent.long()).view(-1)
    tok_exp, slot_exp = tok_in.clone(), slot_in.clone()
    tok_exp[:, :t] = tok_in[src, :t]
    slot_exp[:, :t] = slot_in[src, :t]
    tok_exp[:, t] = token.view(-1)
    slot_exp[:, t] = torch.arange(rows, dtype=torch.int32)
    stale_tok, stale_slot = beam_history(B, k, t, Tmax, g)              # another beam state of the same shape
    cache = poisoned_cache(rows, d, t, tok_exp, slot_exp, BF16, g, nan_cols=(t,))
    table = torch.randn(V, d, generator=g).bfloat16()
    pos_row = torch.randn(d, generator=g).bfloat16()
    gamma, beta = torch.rand(d, generator=g) + 0.5, torch.randn(d, generator=g) * 0.1
    W = (torch.randn(3 * d, d, generator=g) / math.sqrt(d)).bfloat16()
    D = dev()
    tok_in, slot_in, parent, token, table, pos_row, gamma, beta, W = (
        x.to(D) for x in (tok_in, slot_in, parent, token, table, pos_row, gamma, beta, W))
    tok_out, slot_out, cache_d = stale_tok.to(D), stale_slot.to(D), cache.to(D)
    y = torch.empty(rows, d, device=D, dtype=torch.bfloat16)
    rowscale = torch.empty(rows, device=D)
    qkv = torch.empty(rows, 3 * d, device=D, dtype=torch.bfloat16)
    o = torch.full((rows, d), float("nan"), device=D, dtype=torch.bfloat16)

    def attention():
        N.call("icap_mha_decode_self", BF16, rows, H, t, dh, dh, qkv.data_ptr(), 3 * d, qkv.data_ptr() + 2 * d,
               qkv.data_ptr() + 4 * d, 3 * d, cache_d.data_ptr(), 2 * d, cache_d.data_ptr() + 2 * d, 2 * d, T_CACHE,
               o.data_ptr(), d, slot_out.data_ptr(), Tmax, tok_out.data_ptr(), Tmax, PAD, k, S())

    pdl = ctypes.c_int.in_dll(N.lib(), "icap_g_pdl")
    prev = pdl.value
    N.call("icap_set_pdl", 1)
    try:
        torch.cuda.synchronize()
        N.call("icap_decode_embed_ln", BF16, rows, d, k, Tmax, t, parent.data_ptr(), token.data_ptr(), tok_in.data_ptr(),
               tok_out.data_ptr(), slot_in.data_ptr(), slot_out.data_ptr(), table.data_ptr(), pos_row.data_ptr(),
               gamma.data_ptr(), beta.data_ptr(), y.data_ptr(), rowscale.data_ptr(), PAD, 1e-6, S())
        N.call("icap_gemm", BF16, 1, 1, rows, 3 * d, d, y.data_ptr(), d, W.data_ptr(), d, qkv.data_ptr(), 3 * d, BF16,
               None, N.EPI_B_STATIC, None, 0, 0, 1, S())
        attention()
        torch.cuda.synchronize()
    finally:
        N.call("icap_set_pdl", prev)
    assert torch.equal(tok_out[:, :t + 1].cpu(), tok_exp[:, :t + 1])
    assert torch.equal(slot_out[:, :t + 1].cpu(), slot_exp[:, :t + 1])
    expected = cache.clone()
    expected[:, t] = qkv[:, d:].cpu()
    assert torch.equal(bits(cache_d), bits(expected.to(D)))
    kc, vc = cache_views(cache_d, d)
    tok_e, slot_e = tok_exp.to(D), slot_exp.to(D)
    verify("decode step under PDL", o, ((qkv[:, :d], kc, vc, H, t + 1, T_CACHE), dict(slot=slot_e, tokens=tok_e)), H,
           tol_of(BF16))
    assert_kernels(attention, [k_row(BF16, 4)])                         # the path the sequence exercised
