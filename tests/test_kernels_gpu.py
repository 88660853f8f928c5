"""Per-kernel parity tests (run on a B200: `pytest -m gpu`).  Every test calls the C ABI of
libicap.so through ctypes on raw device pointers and compares with the same operator evaluated
by plain PyTorch (fp32, or fp64 where the tolerance is tight) on the same inputs."""
import math

import pytest
import torch

import icap_loader

pytestmark = pytest.mark.gpu

pkg = icap_loader.load()
N = pkg._native
F32, BF16 = N.F32, N.BF16


def dev():
    return torch.device("cuda:0")


@pytest.fixture(autouse=True)
def _fresh_env():
    """libicap caches its ICAP_* switches; tests that monkeypatch the environment re-read them (and again on exit)."""
    yield
    N.call("icap_reload_env")


def setenv(monkeypatch, key, value):
    monkeypatch.setenv(key, value)
    N.call("icap_reload_env")


def S():
    return torch.cuda.current_stream().cuda_stream


def dt(code):
    return torch.float32 if code == F32 else torch.bfloat16


def rel_err(a, b):
    a, b = a.double(), b.double()
    return float((a - b).abs().max() / (b.abs().max() + 1e-30))


# ------------------------------------------------------------------------------------------ GEMM
def _gemm_case(ab, a_k, b_k, M, Nn, K, c_dtype=F32, bias=False, epi=0, accumulate=0, split_k=1, seed=0):
    g = torch.Generator(device="cuda").manual_seed(seed)
    tdt = dt(ab)
    A = torch.randn((M, K) if a_k else (K, M), device=dev(), generator=g).to(tdt)
    Bm = torch.randn((Nn, K) if b_k else (K, Nn), device=dev(), generator=g).to(tdt)
    Af = (A if a_k else A.t()).double()
    Bf = (Bm.t() if b_k else Bm).double()
    ref = Af @ Bf
    bias_t = torch.randn(Nn, device=dev(), generator=g) if bias else None
    if bias:
        ref = ref + bias_t.double()
    aux = None
    if (epi & 15) == 1:
        ref = ref.clamp_min(0)
    if (epi & 15) == 2:
        aux = torch.randn(M, Nn, device=dev(), generator=g).to(dt(c_dtype))
        ref = ref * (aux.double() > 0)
    C = torch.randn(M, Nn, device=dev(), generator=g).to(dt(c_dtype)) if accumulate else \
        torch.full((M, Nn), float("nan"), device=dev(), dtype=dt(c_dtype))
    if accumulate:
        ref = ref + C.double()
    N.call("icap_gemm", ab, int(a_k), int(b_k), M, Nn, K, A.data_ptr(), A.shape[1], Bm.data_ptr(), Bm.shape[1],
           C.data_ptr(), Nn, c_dtype, bias_t.data_ptr() if bias else None, epi, aux.data_ptr() if aux is not None else None,
           Nn, accumulate, split_k, S())
    torch.cuda.synchronize()
    return rel_err(C, ref)


LAYOUTS = [(1, 1), (1, 0), (0, 0)]


@pytest.mark.parametrize("a_k,b_k", LAYOUTS)
@pytest.mark.parametrize("M,Nn,K", [(128, 128, 64), (300, 200, 136), (37, 397, 84), (1024, 512, 2048)])
def test_gemm_fp32_layouts(a_k, b_k, M, Nn, K):
    assert _gemm_case(F32, a_k, b_k, M, Nn, K) < 5e-6


def test_gemm_fp32_epilogues():
    assert _gemm_case(F32, 1, 1, 260, 136, 96, bias=True, epi=1) < 2e-6
    assert _gemm_case(F32, 1, 0, 260, 136, 96, epi=2) < 2e-6
    assert _gemm_case(F32, 1, 1, 260, 136, 96, bias=True, accumulate=1) < 2e-6
    assert _gemm_case(F32, 0, 0, 136, 96, 3000, accumulate=1, split_k=7) < 2e-6


@pytest.mark.parametrize("a_k,b_k", LAYOUTS)
@pytest.mark.parametrize("M,Nn,K", [(128, 128, 64), (256, 256, 512), (304, 200, 136), (1000, 392, 2048)])
def test_gemm_bf16_tcgen05_layouts(a_k, b_k, M, Nn, K):
    # bf16 inputs are exact in the fp64 reference; only fp32 accumulation order differs
    assert _gemm_case(BF16, a_k, b_k, M, Nn, K) < 1e-5


def test_gemm_bf16_tcgen05_epilogues():
    assert _gemm_case(BF16, 1, 1, 260, 136, 96, c_dtype=BF16, bias=True, epi=1) < 6e-3
    assert _gemm_case(BF16, 1, 0, 260, 136, 96, c_dtype=BF16, epi=2) < 6e-3
    assert _gemm_case(BF16, 1, 1, 260, 136, 96, c_dtype=F32, bias=True, accumulate=1) < 1e-5
    assert _gemm_case(BF16, 1, 1, 260, 136, 96, c_dtype=BF16, accumulate=1) < 6e-3
    assert _gemm_case(BF16, 0, 0, 136, 96, 3000, accumulate=1, split_k=7) < 1e-5
    assert _gemm_case(BF16, 0, 0, 512, 512, 9216, accumulate=1, split_k=18) < 1e-5


@pytest.mark.parametrize("bn", ["128", "256", "pair"])
def test_gemm_bf16_persistent_multi_tile(bn, monkeypatch):
    """More tiles than SMs: every CTA loops over several tiles (TMEM accumulator double buffering, smem ring
    phases carried across tiles), all tile configurations (128x128, 128x256, cta_group::2 pair 256x256), every
    epilogue, automatic split-K."""
    setenv(monkeypatch, "ICAP_GEMM_BN", bn)
    setenv(monkeypatch, "ICAP_GEMM_SMALL", "0")
    assert _gemm_case(BF16, 1, 1, 9216, 2048, 512, c_dtype=BF16, bias=True, epi=1) < 6e-3      # FFN1 forward
    assert _gemm_case(BF16, 1, 0, 9216, 2048, 512, c_dtype=BF16, epi=2) < 6e-3                 # FFN2 dgrad + ReLU mask
    assert _gemm_case(BF16, 1, 1, 5376, 10000, 512, c_dtype=BF16, bias=True) < 6e-3            # classifier
    assert _gemm_case(BF16, 1, 0, 5376, 512, 10000, c_dtype=BF16) < 6e-3                       # classifier dgrad
    assert _gemm_case(BF16, 1, 1, 4000, 1000, 200, c_dtype=F32, bias=True) < 1e-5              # ragged everything
    assert _gemm_case(BF16, 1, 0, 4000, 1000, 200, c_dtype=F32, accumulate=1) < 1e-5
    assert _gemm_case(BF16, 0, 0, 2048, 512, 9216, accumulate=1, split_k=0) < 1e-5             # wgrad, auto split
    assert _gemm_case(BF16, 0, 0, 10000, 512, 5376, accumulate=1, split_k=0) < 1e-5            # classifier wgrad
    assert _gemm_case(BF16, 0, 0, 512, 2136, 9216, accumulate=1, split_k=0) < 1e-5             # embedding wgrad
    setenv(monkeypatch, "ICAP_GEMM_DIRECT_EPILOGUE", "1")
    assert _gemm_case(BF16, 1, 1, 3000, 1000, 200, c_dtype=BF16, bias=True, epi=1) < 6e-3
    assert _gemm_case(BF16, 1, 0, 3000, 1000, 200, c_dtype=BF16, epi=2) < 6e-3
    assert _gemm_case(BF16, 0, 0, 520, 392, 5000, accumulate=1, split_k=0) < 1e-5


@pytest.mark.parametrize("mode", ["0", "2"])
def test_gemm_bf16_small_footprint_kernel(mode, monkeypatch):
    """The small-footprint 128x128 one-tile-per-CTA kernel (gemm_small.cu: decode-step shapes, 2 CTAs per SM, weight
    prefetch before the grid dependency) against the persistent kernel on the same shapes: ragged M / N / K, bias,
    ReLU, the B_STATIC flag, K shorter and longer than the 3-stage ring, more CTAs than fit at once (mode 2)."""
    setenv(monkeypatch, "ICAP_GEMM_SMALL", mode)
    for epi in (0, N.EPI_B_STATIC):
        assert _gemm_case(BF16, 1, 1, 2560, 1536, 512, c_dtype=BF16, epi=epi) < 6e-3            # decode QKV
        assert _gemm_case(BF16, 1, 1, 2560, 2048, 512, c_dtype=BF16, bias=True, epi=1 | epi) < 6e-3   # decode FFN1
        assert _gemm_case(BF16, 1, 1, 2560, 512, 2048, c_dtype=BF16, bias=True, epi=epi) < 6e-3
        assert _gemm_case(BF16, 1, 1, 260, 136, 96, c_dtype=BF16, bias=True, epi=1 | epi) < 6e-3
        assert _gemm_case(BF16, 1, 1, 37, 1000, 64, c_dtype=BF16, bias=True, epi=epi) < 6e-3
        assert _gemm_case(BF16, 1, 1, 515, 392, 200, c_dtype=BF16, epi=epi) < 6e-3
    if mode == "2":
        assert _gemm_case(BF16, 1, 1, 5376, 10000, 512, c_dtype=BF16, bias=True, epi=N.EPI_B_STATIC) < 6e-3


def test_gemm_bf16_limited_grid_and_weight_prefetch(monkeypatch):
    """icap_set_gemm_sms (data parallel: the backward's persistent GEMMs leave SMs to NCCL) and the B_STATIC flag on the
    persistent kernel (weight tiles of the first ring round requested before the grid dependency): same results."""
    setenv(monkeypatch, "ICAP_GEMM_SMALL", "0")
    try:
        for sms in (0, 132, 17):
            N.call("icap_set_gemm_sms", sms)
            for epi in (0, N.EPI_B_STATIC):
                assert _gemm_case(BF16, 1, 1, 9216, 2048, 512, c_dtype=BF16, bias=True, epi=1 | epi) < 6e-3
                assert _gemm_case(BF16, 1, 0, 5376, 512, 2048, c_dtype=BF16, epi=epi) < 6e-3
                assert _gemm_case(BF16, 1, 0, 4000, 1000, 200, c_dtype=F32, accumulate=1, epi=epi) < 1e-5
                assert _gemm_case(BF16, 1, 1, 300, 264, 72, c_dtype=BF16, epi=epi) < 6e-3        # K shorter than the ring
            # fewer SMs -> fewer K splits -> longer fp32 accumulation chains: 9216-term dot products round to ~1e-5
            assert _gemm_case(BF16, 0, 0, 2048, 512, 9216, accumulate=1, split_k=0) < 3e-5
    finally:
        N.call("icap_set_gemm_sms", 0)


def test_gemm_bf16_vocab_shapes():
    """classifier-like shapes: N = V not a multiple of the tile, padded leading dimension."""
    M, V, d, ldl = 300, 1000, 512, 1000
    g = torch.Generator(device="cuda").manual_seed(1)
    X = torch.randn(M, d, device=dev(), generator=g).bfloat16()
    W = torch.randn(V, d, device=dev(), generator=g).bfloat16()
    b = torch.randn(V, device=dev(), generator=g)
    C = torch.zeros(M, ldl, device=dev(), dtype=torch.bfloat16)
    N.call("icap_gemm", BF16, 1, 1, M, V, d, X.data_ptr(), d, W.data_ptr(), d, C.data_ptr(), ldl, BF16, b.data_ptr(), 0,
           None, 0, 0, 1, S())
    ref = X.double() @ W.double().t() + b.double()
    assert rel_err(C, ref) < 6e-3
    # dgrad: dX = dY[M,V] . W[V,d]   (K = V: TMA zero-fills the K tail)
    dX = torch.zeros(M, d, device=dev(), dtype=torch.bfloat16)
    N.call("icap_gemm", BF16, 1, 0, M, d, V, C.data_ptr(), ldl, W.data_ptr(), d, dX.data_ptr(), d, BF16, None, 0, None, 0,
           0, 1, S())
    assert rel_err(dX, C.double() @ W.double()) < 6e-3
    # wgrad: dW = dY^T X
    dW = torch.zeros(V, d, device=dev())
    N.call("icap_gemm", BF16, 0, 0, V, d, M, C.data_ptr(), ldl, X.data_ptr(), d, dW.data_ptr(), d, F32, None, 0, None, 0,
           1, 1, S())
    assert rel_err(dW, C.double().t() @ X.double()) < 1e-5


def test_mha_decode_self_fused_append():
    """icap_mha_decode_self (KV-cache append fused into the attention) == explicit append + icap_mha_decode, for the
    head-dim-64 fast path and the generic path, with beam slot indirection and pad-token masking."""
    # beam widths 1, 2 and 5 of the head-dim-64 paths are compared with fp64 in test_decode_attention_gpu.py
    for act, dh, rpi, H in ((BF16, 64, 3, 4), (BF16, 64, 4, 8), (F32, 64, 4, 4), (F32, 16, 1, 4)):
        g = torch.Generator(device="cuda").manual_seed(9 + dh)
        tdt = dt(act)
        rows, T, t = 24, 9, 5
        d = H * dh
        q = torch.randn(rows, 3 * d, device=dev(), generator=g).to(tdt)            # packed [q | k_new | v_new]
        cache = torch.randn(rows, T, 2 * d, device=dev(), generator=g).to(tdt)
        tok = torch.randint(0, 4, (rows, T + 1), device=dev(), generator=g, dtype=torch.int32)   # id 0 = pad
        tok[:, 0] = 1
        slot = torch.randint(0, rows, (rows, T + 1), device=dev(), generator=g, dtype=torch.int32)
        slot[:, t] = torch.arange(rows, dtype=torch.int32, device=dev())          # newest position: own row
        if rpi > 1:     # beams of an image share their oldest positions (one ancestor), as after a few beam steps: the
            #             image-per-block kernel stages such rows once; tokens of a shared position are the ancestor's
            first = (torch.arange(rows, device=dev()) // rpi * rpi).int()
            slot[:, :3] = first[:, None]
            slot[1::rpi, 3] = slot[0::rpi, 3]
            tok[:, :3] = tok[first.long(), :3]
            tok[1::rpi, 3] = tok[0::rpi, 3]
        esz = q.element_size()
        ref_cache = cache.clone()
        ref_cache[:, t, :] = q[:, d:]
        o_ref = torch.empty(rows, d, device=dev(), dtype=tdt)
        N.call("icap_mha_decode", act, rows, H, t + 1, dh, dh, q.data_ptr(), 3 * d, ref_cache.data_ptr(), 2 * d,
               ref_cache.data_ptr() + d * esz, 2 * d, T, o_ref.data_ptr(), d, slot.data_ptr(), T + 1, tok.data_ptr(), T + 1,
               0, None, 1, None, S())
        o = torch.empty(rows, d, device=dev(), dtype=tdt)
        N.call("icap_mha_decode_self", act, rows, H, t, dh, dh, q.data_ptr(), 3 * d, q.data_ptr() + d * esz,
               q.data_ptr() + 2 * d * esz, 3 * d, cache.data_ptr(), 2 * d, cache.data_ptr() + d * esz, 2 * d, T,
               o.data_ptr(), d, slot.data_ptr(), T + 1, tok.data_ptr(), T + 1, 0, rpi, S())
        torch.cuda.synchronize()
        assert torch.equal(cache, ref_cache)
        assert rel_err(o, o_ref) < (1e-5 if act == F32 else 1e-2)


@pytest.mark.parametrize("small", ["0", "2"])
@pytest.mark.parametrize("M,Nn,K", [(2560, 512, 512), (77, 512, 512), (300, 256, 256), (129, 1024, 1024),
                                    (640, 512, 2048), (9216, 512, 512), (50, 128, 72), (130, 512, 64), (200, 256, 128)])
def test_gemm_ln_small_footprint(M, Nn, K, small, monkeypatch):
    """Inference form of icap_gemm_ln (no dropout, nothing saved): the small-footprint two-pass kernel (192 threads,
    3-stage ring, accumulator re-read from TMEM, two CTAs per SM) and the original kernel against fp64; K shorter than
    the ring (the residual boxes then land in never-used ring slots), with and without bias / residual / row scale."""
    setenv(monkeypatch, "ICAP_GEMM_LN_SMALL", small)
    g = torch.Generator(device="cuda").manual_seed(M + K)
    A = torch.randn(M, K, device=dev(), generator=g).bfloat16()
    W = (torch.randn(Nn, K, device=dev(), generator=g) / math.sqrt(K)).bfloat16()
    res = torch.randn(M, Nn, device=dev(), generator=g).bfloat16()
    bias = torch.randn(Nn, device=dev(), generator=g)
    gamma = torch.randn(Nn, device=dev(), generator=g)
    beta = torch.randn(Nn, device=dev(), generator=g)
    rs = (torch.rand(M, device=dev(), generator=g) > 0.2).float()
    for use_bias, use_rs, use_res in ((True, True, True), (False, False, True), (True, False, False)):
        y = torch.full((M, Nn), float("nan"), device=dev(), dtype=torch.bfloat16)
        N.call("icap_gemm_ln", M, Nn, K, A.data_ptr(), K, W.data_ptr(), K, bias.data_ptr() if use_bias else None,
               res.data_ptr() if use_res else None, Nn, gamma.data_ptr(), beta.data_ptr(),
               rs.data_ptr() if use_rs else None, y.data_ptr(), Nn, None, 0, None, None, 1e-6, 0.0, 0, None, S())
        x = A.double() @ W.double().t() + (res.double() if use_res else 0.0) + (bias.double() if use_bias else 0.0)
        ref = torch.nn.functional.layer_norm(x, (Nn,), gamma.double(), beta.double(), 1e-6)
        if use_rs:
            ref = ref * rs.double()[:, None]
        torch.cuda.synchronize()
        assert rel_err(y, ref) < 8e-3


@pytest.mark.parametrize("bn", ["auto", "128", "256"])
@pytest.mark.parametrize("M,Nn,K", [(2560, 512, 512), (77, 512, 512), (300, 256, 256), (129, 1024, 1024),
                                    (640, 512, 2048), (9216, 512, 512), (50, 128, 72)])
def test_gemm_ln_cluster_fused(M, Nn, K, bn, monkeypatch):
    """icap_gemm_ln (cluster of N/128 or N/256 CTAs, statistics exchanged through DSMEM) == fp64 reference, and its
    saved sum / mean / rstd and DROPOUT decisions == icap_gemm + icap_add_ln_fwd (so icap_add_ln_bwd can consume them)."""
    if bn != "auto":
        if Nn % int(bn):
            pytest.skip("width not a multiple of the forced tile")
        setenv(monkeypatch, "ICAP_GEMM_LN_BN", bn)
        setenv(monkeypatch, "ICAP_GEMM_LN_SMALL", "0")
    g = torch.Generator(device="cuda").manual_seed(M + K)
    A = torch.randn(M, K, device=dev(), generator=g).bfloat16()
    W = (torch.randn(Nn, K, device=dev(), generator=g) / math.sqrt(K)).bfloat16()
    res = torch.randn(M, Nn, device=dev(), generator=g).bfloat16()
    bias = torch.randn(Nn, device=dev(), generator=g)
    gamma = torch.randn(Nn, device=dev(), generator=g)
    beta = torch.randn(Nn, device=dev(), generator=g)
    rs = (torch.rand(M, device=dev(), generator=g) > 0.2).float()
    step = torch.tensor([3], dtype=torch.int32, device=dev())
    for use_bias, use_rs in ((True, True), (False, False)):
        y = torch.full((M, Nn), float("nan"), device=dev(), dtype=torch.bfloat16)
        N.call("icap_gemm_ln", M, Nn, K, A.data_ptr(), K, W.data_ptr(), K, bias.data_ptr() if use_bias else None,
               res.data_ptr(), Nn, gamma.data_ptr(), beta.data_ptr(), rs.data_ptr() if use_rs else None, y.data_ptr(), Nn,
               None, 0, None, None, 1e-6, 0.0, 0, None, S())
        x = A.double() @ W.double().t() + res.double() + (bias.double() if use_bias else 0.0)
        ref = torch.nn.functional.layer_norm(x, (Nn,), gamma.double(), beta.double(), 1e-6)
        if use_rs:
            ref = ref * rs.double()[:, None]
        torch.cuda.synchronize()
        assert rel_err(y, ref) < 8e-3
    # training form: dropout 0.3, sum / mean / rstd saved -- against the two-kernel path with the same seed
    seed, p = 12345, 0.3
    y = torch.empty(M, Nn, device=dev(), dtype=torch.bfloat16)
    ssum = torch.empty(M, Nn, device=dev(), dtype=torch.bfloat16)
    mean, rstd = torch.empty(M, device=dev()), torch.empty(M, device=dev())
    N.call("icap_gemm_ln", M, Nn, K, A.data_ptr(), K, W.data_ptr(), K, bias.data_ptr(), res.data_ptr(), Nn,
           gamma.data_ptr(), beta.data_ptr(), rs.data_ptr(), y.data_ptr(), Nn, ssum.data_ptr(), Nn, mean.data_ptr(),
           rstd.data_ptr(), 1e-6, p, seed, step.data_ptr(), S())
    o = torch.empty(M, Nn, device=dev(), dtype=torch.bfloat16)
    N.call("icap_gemm", BF16, 1, 1, M, Nn, K, A.data_ptr(), K, W.data_ptr(), K, o.data_ptr(), Nn, BF16, bias.data_ptr(),
           0, None, 0, 0, 1, S())
    y2 = torch.empty_like(y)
    mean2, rstd2 = torch.empty_like(mean), torch.empty_like(rstd)
    N.call("icap_add_ln_fwd", BF16, BF16, M, Nn, o.data_ptr(), res.data_ptr(), M, gamma.data_ptr(), beta.data_ptr(),
           rs.data_ptr(), y2.data_ptr(), mean2.data_ptr(), rstd2.data_ptr(), 1, p, seed, step.data_ptr(), 1e-6, S())
    torch.cuda.synchronize()
    # identical dropout decisions: a dropped element leaves s == res exactly in both paths
    dropped, dropped2 = ssum == res, o == res          # `o` now holds the two-kernel path's pre-norm sum
    assert float((dropped != dropped2).float().mean()) < 2e-3        # (an element whose GEMM value rounds to 0 may differ)
    assert 0.25 < float(dropped.float().mean()) < 0.35
    assert rel_err(ssum, o.double()) < 8e-3            # the two-kernel path rounds the GEMM output to bf16 first
    assert rel_err(mean, mean2.double()) < 5e-3 and rel_err(rstd, rstd2.double()) < 5e-3
    assert rel_err(y, y2.double()) < 1.5e-2


# ------------------------------------------------------------------------------------------ add + LayerNorm
@pytest.mark.parametrize("act", [F32, BF16])
@pytest.mark.parametrize("M,d", [(77, 32), (500, 512), (64, 1024), (33, 256)])
def test_add_ln_fwd_bwd(act, M, d):
    g = torch.Generator(device="cuda").manual_seed(M + d)
    T = 7
    a = torch.randn(M, d, device=dev(), generator=g).to(dt(act))
    res = torch.randn(T, d, device=dev(), generator=g).to(dt(act))
    gamma = torch.randn(d, device=dev(), generator=g)
    beta = torch.randn(d, device=dev(), generator=g)
    rs = (torch.rand(M, device=dev(), generator=g) > 0.3).float()
    dy1 = torch.randn(M, d, device=dev(), generator=g).to(dt(act))
    dy2 = torch.randn(M, d, device=dev(), generator=g).to(dt(act))

    a64 = a.double().requires_grad_(True)
    g64, b64 = gamma.double().requires_grad_(True), beta.double().requires_grad_(True)
    s64 = a64 + res.double()[torch.arange(M, device=dev()) % T]
    y64 = torch.nn.functional.layer_norm(s64, (d,), g64, b64, 1e-6) * rs.double()[:, None]
    y64.backward(dy1.double() + dy2.double())

    a_work = a.clone()
    y = torch.empty(M, d, device=dev(), dtype=dt(act))
    mean = torch.empty(M, device=dev())
    rstd = torch.empty(M, device=dev())
    N.call("icap_add_ln_fwd", act, act, M, d, a_work.data_ptr(), res.data_ptr(), T, gamma.data_ptr(), beta.data_ptr(),
           rs.data_ptr(), y.data_ptr(), mean.data_ptr(), rstd.data_ptr(), 1, 0.0, 0, None, 1e-6, S())
    tol = 2e-5 if act == F32 else 2e-2
    assert rel_err(y, y64.detach()) < tol
    assert rel_err(a_work, s64.detach()) < (1e-6 if act == F32 else 1e-2)
    ds = torch.empty(M, d, device=dev(), dtype=dt(act))
    dgam = torch.zeros(d, device=dev())
    dbet = torch.zeros(d, device=dev())
    dbias2 = torch.zeros(d, device=dev())
    N.call("icap_add_ln_bwd", act, M, d, dy1.data_ptr(), dy2.data_ptr(), a_work.data_ptr(), mean.data_ptr(),
           rstd.data_ptr(), gamma.data_ptr(), rs.data_ptr(), ds.data_ptr(), None, dgam.data_ptr(), dbet.data_ptr(),
           dbias2.data_ptr(), 0.0, 0, None, S())
    torch.cuda.synchronize()
    assert rel_err(ds, a64.grad) < (5e-5 if act == F32 else 3e-2)
    assert rel_err(dgam, g64.grad) < (5e-5 if act == F32 else 3e-2)
    assert rel_err(dbet, b64.grad) < (5e-5 if act == F32 else 3e-2)
    assert rel_err(dbias2, a64.grad.sum(0)) < (5e-4 if act == F32 else 5e-2)


# ------------------------------------------------------------------------------------------ attention
def _ref_attention(q, k, v, kvalid, causal, H):
    B, Lq, _ = q.shape
    Lk = k.shape[1]
    dk, dv = q.shape[2] // H, v.shape[2] // H
    qh = q.view(B, Lq, H, dk).transpose(1, 2)
    kh = k.view(B, Lk, H, dk).transpose(1, 2)
    vh = v.view(B, Lk, H, dv).transpose(1, 2)
    att = (qh / math.sqrt(dk)) @ kh.transpose(2, 3)
    mask = torch.zeros(B, 1, Lq, Lk, dtype=torch.bool, device=q.device)
    if kvalid is not None:
        mask = mask | (~kvalid.bool()).view(B, 1, 1, Lk)
    if causal:
        mask = mask | torch.triu(torch.ones(Lq, Lk, dtype=torch.bool, device=q.device), 1).view(1, 1, Lq, Lk)
    att = att.masked_fill(mask, float("-inf")).softmax(-1)
    return (att @ vh).transpose(1, 2).reshape(B, Lq, H * dv), att


@pytest.mark.parametrize("act", [F32, BF16])
@pytest.mark.parametrize("B,H,Lq,Lk,dk,dv,causal,usevalid",
                         [(3, 8, 36, 36, 64, 64, False, False), (3, 8, 21, 21, 64, 64, True, True),
                          (2, 8, 21, 36, 64, 64, False, True), (2, 4, 7, 5, 8, 4, False, True),
                          (2, 32, 36, 36, 8, 8, True, True), (1, 2, 100, 100, 64, 64, False, True)])
def test_mha_fwd_bwd(act, B, H, Lq, Lk, dk, dv, causal, usevalid):
    g = torch.Generator(device="cuda").manual_seed(B * 100 + Lq)
    tdt = dt(act)
    # packed projections: q in [B*Lq, H*dk + 16] with a row stride, k|v packed in one buffer
    ldq = H * dk + 16
    ldkv = H * dk + H * dv
    qb = torch.randn(B * Lq, ldq, device=dev(), generator=g).to(tdt)
    kvb = torch.randn(B * Lk, ldkv, device=dev(), generator=g).to(tdt)
    kvalid = None
    if usevalid:
        nv = torch.randint(max(1, Lk // 2), Lk + 1, (B,), device=dev(), generator=g)
        kvalid = (torch.arange(Lk, device=dev())[None, :] < nv[:, None]).to(torch.uint8).contiguous()
    q64 = qb[:, :H * dk].double().view(B, Lq, H * dk).requires_grad_(True)
    k64 = kvb[:, :H * dk].double().view(B, Lk, H * dk).requires_grad_(True)
    v64 = kvb[:, H * dk:].double().view(B, Lk, H * dv).requires_grad_(True)
    ref, att_ref = _ref_attention(q64, k64, v64, kvalid, causal, H)
    dout = torch.randn(B * Lq, H * dv, device=dev(), generator=g).to(tdt)
    ref.backward(dout.double().view(B, Lq, H * dv))

    o = torch.empty(B * Lq, H * dv, device=dev(), dtype=tdt)
    amean = torch.zeros(B, Lq, Lk, device=dev())
    esz = qb.element_size()
    N.call("icap_mha_fwd", act, B, H, Lq, Lk, dk, dv, qb.data_ptr(), ldq, kvb.data_ptr(), ldkv,
           kvb.data_ptr() + H * dk * esz, ldkv, o.data_ptr(), H * dv, kvalid.data_ptr() if usevalid else None,
           int(causal), 0.0, 0, None, amean.data_ptr(), S())
    tol = 1e-5 if act == F32 else 1.5e-2
    assert rel_err(o, ref.detach().view(B * Lq, -1)) < tol
    assert rel_err(amean, att_ref.detach().mean(1)) < tol
    # without the attention-mean output the bf16 / head-dim-64 cases take the mma.sync tensor-core kernel
    o2 = torch.empty_like(o)
    N.call("icap_mha_fwd", act, B, H, Lq, Lk, dk, dv, qb.data_ptr(), ldq, kvb.data_ptr(), ldkv,
           kvb.data_ptr() + H * dk * esz, ldkv, o2.data_ptr(), H * dv, kvalid.data_ptr() if usevalid else None,
           int(causal), 0.0, 0, None, None, S())
    assert rel_err(o2, ref.detach().view(B * Lq, -1)) < tol
    dq = torch.zeros(B * Lq, ldq, device=dev(), dtype=tdt)
    dkv = torch.zeros(B * Lk, ldkv, device=dev(), dtype=tdt)
    N.call("icap_mha_bwd", act, B, H, Lq, Lk, dk, dv, qb.data_ptr(), ldq, kvb.data_ptr(), ldkv,
           kvb.data_ptr() + H * dk * esz, ldkv, dout.data_ptr(), H * dv, dq.data_ptr(), ldq, dkv.data_ptr(), ldkv,
           dkv.data_ptr() + H * dk * esz, ldkv, kvalid.data_ptr() if usevalid else None, int(causal), 0.0, 0, None, S())
    torch.cuda.synchronize()
    tolb = 2e-5 if act == F32 else 2e-2
    assert rel_err(dq[:, :H * dk], q64.grad.view(B * Lq, -1)) < tolb
    assert rel_err(dkv[:, :H * dk], k64.grad.view(B * Lk, -1)) < tolb
    assert rel_err(dkv[:, H * dk:], v64.grad.view(B * Lk, -1)) < tolb


def test_mha_decode_matches_full_attention():
    """KV-cached single-query attention == last row of full causal attention (incl. pad-token keys,
    beam slot indirection) and cross-attention with rows_per_image sharing."""
    B, k, H, T, dk, dv, R = 3, 2, 4, 6, 16, 16, 5
    rows = B * k
    g = torch.Generator(device="cuda").manual_seed(5)
    for act in (F32, BF16):
        tdt = dt(act)
        t = 4
        nkv = H * (dk + dv)
        q = torch.randn(rows, H * dk, device=dev(), generator=g).to(tdt)
        cache = torch.randn(rows, T, nkv, device=dev(), generator=g).to(tdt)
        tokens = torch.randint(0, 4, (rows, T + 1), device=dev(), generator=g, dtype=torch.int32)
        tokens[:, 0] = 1
        slot = torch.randint(0, rows, (rows, T + 1), device=dev(), generator=g, dtype=torch.int32)
        o = torch.empty(rows, H * dv, device=dev(), dtype=tdt)
        esz = q.element_size()
        N.call("icap_mha_decode", act, rows, H, t + 1, dk, dv, q.data_ptr(), H * dk, cache.data_ptr(), nkv,
               cache.data_ptr() + H * dk * esz, nkv, T, o.data_ptr(), H * dv, slot.data_ptr(), T + 1, tokens.data_ptr(),
               T + 1, 0, None, 1, None, S())
        # reference
        idx = slot[:, :t + 1].long()
        gathered = cache[idx, torch.arange(t + 1, device=dev())[None, :]]          # [rows, t+1, nkv]
        kk = gathered[:, :, :H * dk].double().view(rows, t + 1, H, dk).transpose(1, 2)
        vv = gathered[:, :, H * dk:].double().view(rows, t + 1, H, dv).transpose(1, 2)
        qq = q.double().view(rows, 1, H, dk).transpose(1, 2)
        att = (qq / math.sqrt(dk)) @ kk.transpose(2, 3)
        att = att.masked_fill((tokens[:, :t + 1] == 0).view(rows, 1, 1, t + 1), float("-inf")).softmax(-1)
        ref = (att @ vv).transpose(1, 2).reshape(rows, H * dv)
        assert rel_err(o, ref) < (1e-5 if act == F32 else 1.5e-2)
        # cross attention
        kvb = torch.randn(B * R, nkv, device=dev(), generator=g).to(tdt)
        kvalid = torch.ones(B, R, dtype=torch.uint8, device=dev())
        kvalid[:, R - 1] = 0
        am = torch.zeros(rows, R, device=dev())
        N.call("icap_mha_decode", act, rows, H, R, dk, dv, q.data_ptr(), H * dk, kvb.data_ptr(), nkv,
               kvb.data_ptr() + H * dk * esz, nkv, R, o.data_ptr(), H * dv, None, 0, None, 0, 0, kvalid.data_ptr(), k,
               am.data_ptr(), S())
        img = torch.arange(rows, device=dev()) // k
        kk = kvb.view(B, R, nkv)[img][:, :, :H * dk].double().view(rows, R, H, dk).transpose(1, 2)
        vv = kvb.view(B, R, nkv)[img][:, :, H * dk:].double().view(rows, R, H, dv).transpose(1, 2)
        att = ((qq / math.sqrt(dk)) @ kk.transpose(2, 3)).masked_fill(
            (kvalid[img] == 0).view(rows, 1, 1, R), float("-inf")).softmax(-1)
        ref = (att @ vv).transpose(1, 2).reshape(rows, H * dv)
        torch.cuda.synchronize()
        assert rel_err(o, ref) < (1e-5 if act == F32 else 1.5e-2)
        assert rel_err(am, att.mean(1).squeeze(1)) < (1e-5 if act == F32 else 1.5e-2)


# ------------------------------------------------------------------------------------------ loss / selection
@pytest.mark.parametrize("log_domain", [0, 1])
@pytest.mark.parametrize("kin,kout,V", [(1, 3, 397), (3, 3, 10000), (5, 5, 10000), (5, 5, 401)])
def test_beam_select(log_domain, kin, kout, V):
    B = 7
    g = torch.Generator(device="cuda").manual_seed(V + kin)
    logits = torch.randn(B * kin, V, device=dev(), generator=g) * 3
    prev = torch.rand(B, kin, device=dev(), generator=g)
    sm = torch.log_softmax(logits, 1) if log_domain else torch.softmax(logits, 1)
    cand = (sm.view(B, kin, V) + prev[:, :, None]).view(B, kin * V)
    ref_s, ref_i = torch.topk(cand, kout + 1, dim=1)
    os_ = torch.empty(B, kout, device=dev())
    op = torch.empty(B, kout, dtype=torch.int32, device=dev())
    ot = torch.empty(B, kout, dtype=torch.int32, device=dev())
    gap = torch.empty(B, device=dev())
    N.call("icap_beam_select", F32, B, kin, V, logits.data_ptr(), V, prev.data_ptr(), kout, os_.data_ptr(), op.data_ptr(),
           ot.data_ptr(), gap.data_ptr(), log_domain, None, 0, S())
    torch.cuda.synchronize()
    assert torch.equal(op.long() * V + ot.long(), ref_i[:, :kout])
    assert torch.allclose(os_, ref_s[:, :kout], rtol=1e-5, atol=1e-7)
    assert torch.allclose(gap, ref_s[:, kout - 1] - ref_s[:, kout], rtol=1e-3, atol=1e-7)


@pytest.mark.parametrize("log_domain", [0, 1])
@pytest.mark.parametrize("case", ["flat", "one_beam_dominates", "ties", "tiny_vocab", "bf16_flat", "bf16_one_beam_dominates",
                                  "bf16_ties", "bf16_tiny_vocab", "bf16_random"])
def test_beam_select_degenerate_distributions(log_domain, case):
    """The candidate threshold must stay exact when the distribution is nearly uniform, when one beam's previous score
    dwarfs the others (all winners from one row -- the additive probability scores of model.py:176-181 make this the
    common case early in training), with exact ties (more tied candidates than the fast path's list: slow path), and
    when whole warps see no vocabulary entries."""
    B, kin, kout, V = 9, 5, 5, 10000
    g = torch.Generator(device="cuda").manual_seed(11)
    dtype, code = torch.float32, F32
    if case.startswith("bf16_"):            # bf16 logits (the decode path)
        dtype, code = torch.bfloat16, BF16
        case = case[5:]
    if case == "flat":
        logits = torch.randn(B * kin, V, device=dev(), generator=g) * 1e-2
        prev = torch.rand(B, kin, device=dev(), generator=g) * 1e-3
    elif case == "random":
        V = 9999                                                   # not a multiple of 8: partial last chunk
        logits = torch.randn(B * kin, V, device=dev(), generator=g) * 3
        prev = torch.rand(B, kin, device=dev(), generator=g)
    elif case == "one_beam_dominates":
        logits = torch.randn(B * kin, V, device=dev(), generator=g) * 0.3
        prev = torch.rand(B, kin, device=dev(), generator=g) * 1e-4
        prev[:, 2] += 0.5 if not log_domain else 5.0
    elif case == "ties":
        logits = torch.zeros(B * kin, V, device=dev())
        logits[:, 4000:6000] = 1.0                                  # 2000 tied maxima per row
        prev = torch.zeros(B, kin, device=dev())
    else:
        V = 300                                                    # threads 38.. of the block see nothing
        logits = torch.randn(B * kin, V, device=dev(), generator=g)
        prev = torch.rand(B, kin, device=dev(), generator=g) * 0.1
    ldl = (V + 7) // 8 * 8
    store = torch.zeros(B * kin, ldl, device=dev(), dtype=dtype)
    store[:, :V] = logits.to(dtype)
    logits = store[:, :V]
    x = logits.float()
    sm = torch.log_softmax(x, 1) if log_domain else torch.softmax(x, 1)
    cand = (sm.view(B, kin, V) + prev[:, :, None]).view(B, kin * V)
    os_ = torch.empty(B, kout, device=dev())
    op = torch.empty(B, kout, dtype=torch.int32, device=dev())
    ot = torch.empty(B, kout, dtype=torch.int32, device=dev())
    gap = torch.empty(B, device=dev())
    N.call("icap_beam_select", code, B, kin, V, logits.data_ptr(), ldl, prev.data_ptr(), kout, os_.data_ptr(), op.data_ptr(),
           ot.data_ptr(), gap.data_ptr(), log_domain, None, 0, S())
    torch.cuda.synchronize()
    idx = op.long() * V + ot.long()
    ref_s = torch.topk(cand, kout + 1, dim=1).values
    if case == "ties":                                             # lowest flat index wins ties (CPU topk order, SURVEY 8a)
        want = torch.arange(4000, 4000 + kout, device=dev()).expand(B, kout)
        assert torch.equal(idx, want)
        assert float(gap.abs().max()) == 0.0
    else:
        # the selected candidates' scores are the k best, in order (indices may differ only between exactly equal scores)
        got = cand.gather(1, idx)
        assert torch.allclose(got, ref_s[:, :kout], rtol=1e-6, atol=1e-9)
        assert torch.allclose(os_, ref_s[:, :kout], rtol=1e-5, atol=1e-7)
        assert len({tuple(r) for r in idx.tolist()}) >= 1 and all(len(set(r)) == kout for r in idx.tolist())
        # log domain: scores are ~ -ln(V) = -9.2, one fp32 ulp there is 1e-6 -- the gap is a difference of two of them
        assert torch.allclose(gap, ref_s[:, kout - 1] - ref_s[:, kout], rtol=1e-2, atol=5e-6 if log_domain else 1e-7)


@pytest.mark.parametrize("log_domain", [0, 1])
@pytest.mark.parametrize("V,flat", [(10000, False), (9999, False), (300, False), (30000, False), (40000, False), (10000, True)])
def test_classifier_rowstats_feed_beam_select(log_domain, V, flat):
    """ICAP_EPI_ROWSTATS: the classifier GEMM's epilogue leaves (max, 2nd max, sum exp) per row and 128 columns of the
    ROUNDED logits it stores; icap_beam_select with that buffer (no statistics pass of its own) picks exactly what it
    picks without it, and the statistics equal torch's on the stored logits.  flat: all logits equal (zero weights) -- every
    candidate ties with the bound and both kernels take their exact fall-back."""
    B, k, d = 6, 5, 512
    rows, ldl, P = B * k, (V + 7) // 8 * 8, 2 * ((V + 255) // 256)
    g = torch.Generator(device="cuda").manual_seed(V)
    X = torch.randn(rows, d, device=dev(), generator=g).bfloat16()
    W = (torch.randn(V, d, device=dev(), generator=g) * (0.0 if flat else 0.05)).bfloat16()
    bias = torch.randn(V, device=dev(), generator=g) * (0.0 if flat else 0.1)
    logits = torch.zeros(rows, ldl, device=dev(), dtype=torch.bfloat16)
    stats = torch.full((rows, 4 * P), float("nan"), device=dev())
    N.call("icap_gemm", BF16, 1, 1, rows, V, d, X.data_ptr(), d, W.data_ptr(), d, logits.data_ptr(), ldl, BF16, bias.data_ptr(),
           N.EPI_ROWSTATS | N.EPI_B_STATIC, stats.data_ptr(), 4 * P, 0, 1, S())
    ref = X.double() @ W.double().t() + bias.double()
    assert flat or rel_err(logits[:, :V], ref) < 6e-3
    x = logits[:, :V].float()
    st = stats.view(rows, P, 4)
    npart = (V + 127) // 128
    for pi in (0, npart // 2, npart - 1):
        seg = x[:, pi * 128:min(V, (pi + 1) * 128)]
        top = seg.topk(min(2, seg.shape[1]), dim=1).values
        assert torch.equal(st[:, pi, 0], top[:, 0])
        if seg.shape[1] > 1:
            assert torch.equal(st[:, pi, 1], top[:, 1])
        assert torch.allclose(st[:, pi, 2], (seg - top[:, :1]).exp().sum(1), rtol=1e-4)
    prev = torch.rand(B, k, device=dev(), generator=g) * 1e-4
    outs = []
    for use in (False, True):
        os_ = torch.empty(B, k, device=dev())
        op = torch.empty(B, k, dtype=torch.int32, device=dev())
        ot = torch.empty(B, k, dtype=torch.int32, device=dev())
        gap = torch.empty(B, device=dev())
        N.call("icap_beam_select", BF16, B, k, V, logits.data_ptr(), ldl, prev.data_ptr(), k, os_.data_ptr(), op.data_ptr(),
               ot.data_ptr(), gap.data_ptr(), log_domain, stats.data_ptr() if use else None, 4 * P if use else 0, S())
        torch.cuda.synchronize()
        outs.append((os_, op, ot, gap))
    assert torch.equal(outs[0][1], outs[1][1]) and torch.equal(outs[0][2], outs[1][2])
    assert torch.allclose(outs[0][0], outs[1][0], rtol=1e-5, atol=1e-8)
    sm = torch.log_softmax(x, 1) if log_domain else torch.softmax(x, 1)
    cand = (sm.view(B, k, V) + prev[:, :, None]).view(B, k * V)
    ref_s = torch.topk(cand, k, dim=1).values
    assert torch.allclose(outs[1][0], ref_s, rtol=1e-5, atol=1e-7)


@pytest.mark.parametrize("code,d,k", [(BF16, 512, 5), (BF16, 1024, 3), (F32, 256, 1), (BF16, 512, 1)])
def test_decode_embed_ln_equals_reorder_embed_ln(code, d, k):
    """icap_decode_embed_ln == icap_beam_reorder -> icap_embed_fwd -> icap_add_ln_fwd, bit for bit (same arithmetic order),
    with and without the beam bookkeeping."""
    dt = torch.float32 if code == F32 else torch.bfloat16
    B, Tmax, t, V, pad = 7, 22, 6, 300, 0
    rows = B * k
    g = torch.Generator(device="cuda").manual_seed(d + k)
    table = torch.randn(V, d, device=dev(), generator=g).to(dt)
    pos = torch.randn(Tmax, d, device=dev(), generator=g).to(dt)
    gamma = torch.rand(d, device=dev(), generator=g) + 0.5
    beta = torch.randn(d, device=dev(), generator=g) * 0.1
    tok_in = torch.randint(0, V, (rows, Tmax), device=dev(), generator=g, dtype=torch.int32)
    slot_in = torch.randint(0, rows, (rows, Tmax), device=dev(), generator=g, dtype=torch.int32)
    parent = torch.randint(0, k, (B, k), device=dev(), generator=g, dtype=torch.int32)
    token = torch.randint(0, V, (B, k), device=dev(), generator=g, dtype=torch.int32)
    token[0, 0] = pad
    for reorder in ([True, False] if k > 1 else [False]):
        # reference: the three separate launches
        if reorder:
            tok_ref, slot_ref = torch.zeros_like(tok_in), torch.zeros_like(slot_in)
            N.call("icap_beam_reorder", B, k, Tmax, t - 1, parent.data_ptr(), token.data_ptr(), tok_in.data_ptr(),
                   tok_ref.data_ptr(), slot_in.data_ptr(), slot_ref.data_ptr(), S())
        else:
            tok_ref, slot_ref = tok_in, slot_in
        x0 = torch.empty(rows, d, device=dev(), dtype=dt)
        rs_ref = torch.empty(rows, device=dev())
        N.call("icap_embed_fwd", code, code, tok_ref.data_ptr() + 4 * t, Tmax, rows, d, table.data_ptr(), x0.data_ptr(),
               rs_ref.data_ptr(), pad, S())
        y_ref = torch.empty(rows, d, device=dev(), dtype=dt)
        N.call("icap_add_ln_fwd", code, code, rows, d, x0.data_ptr(), pos[t].data_ptr(), 1, gamma.data_ptr(), beta.data_ptr(),
               None, y_ref.data_ptr(), None, None, 0, 0.0, 0, None, 1e-6, S())
        # fused
        tok_out, slot_out = torch.zeros_like(tok_in), torch.zeros_like(slot_in)
        y = torch.empty(rows, d, device=dev(), dtype=dt)
        rs = torch.empty(rows, device=dev())
        N.call("icap_decode_embed_ln", code, rows, d, k, Tmax, t, parent.data_ptr() if reorder else None,
               token.data_ptr() if reorder else None, tok_in.data_ptr(), tok_out.data_ptr() if reorder else None,
               slot_in.data_ptr() if reorder else None, slot_out.data_ptr() if reorder else None, table.data_ptr(),
               pos[t].data_ptr(), gamma.data_ptr(), beta.data_ptr(), y.data_ptr(), rs.data_ptr(), pad, 1e-6, S())
        torch.cuda.synchronize()
        assert torch.equal(y, y_ref) and torch.equal(rs, rs_ref)
        if reorder:
            assert torch.equal(tok_out[:, :t + 1], tok_ref[:, :t + 1]) and torch.equal(slot_out[:, :t + 1], slot_ref[:, :t + 1])
            assert float(rs[0]) == 0.0
    with pytest.raises(N.IcapError):
        N.call("icap_decode_embed_ln", code, rows, 30, k, Tmax, t, None, None, tok_in.data_ptr(), None, None, None,
               table.data_ptr(), pos[t].data_ptr(), gamma.data_ptr(), beta.data_ptr(), y.data_ptr(), None, pad, 1e-6, S())


def test_beam_reorder():
    B, k, Tmax, t = 4, 3, 8, 2
    g = torch.Generator(device="cuda").manual_seed(2)
    tok_in = torch.randint(1, 50, (B * k, Tmax), device=dev(), generator=g, dtype=torch.int32)
    slot_in = torch.randint(0, B * k, (B * k, Tmax), device=dev(), generator=g, dtype=torch.int32)
    parent = torch.randint(0, k, (B, k), device=dev(), generator=g, dtype=torch.int32)
    token = torch.randint(1, 50, (B, k), device=dev(), generator=g, dtype=torch.int32)
    tok_out = torch.zeros_like(tok_in)
    slot_out = torch.zeros_like(slot_in)
    N.call("icap_beam_reorder", B, k, Tmax, t, parent.data_ptr(), token.data_ptr(), tok_in.data_ptr(), tok_out.data_ptr(),
           slot_in.data_ptr(), slot_out.data_ptr(), S())
    torch.cuda.synchronize()
    src = (torch.arange(B, device=dev())[:, None] * k + parent.long()).view(-1)
    assert torch.equal(tok_out[:, :t + 1], tok_in[src, :t + 1])
    assert torch.equal(tok_out[:, t + 1], token.view(-1))
    assert torch.equal(slot_out[:, :t + 1], slot_in[src, :t + 1])
    assert torch.equal(slot_out[:, t + 1].long(), torch.arange(B * k, device=dev()))


# ------------------------------------------------------------------------------------------ misc kernels
def test_copy2d_region_valid_caption_prep():
    g = torch.Generator(device="cuda").manual_seed(4)
    src = torch.randn(37, 84, device=dev(), generator=g)
    dst = torch.zeros(37, 96, device=dev(), dtype=torch.bfloat16)
    N.call("icap_copy2d", src.data_ptr(), F32, 84, dst.data_ptr() + 2 * 8, BF16, 96, 37, 84, 0, S())
    assert torch.equal(dst[:, 8:92], src.bfloat16()) and float(dst[:, :8].abs().sum()) == 0
    acc = torch.ones(37, 84, device=dev())
    N.call("icap_copy2d", src.data_ptr(), F32, 84, acc.data_ptr(), F32, 84, 37, 84, 1, S())
    assert torch.allclose(acc, src + 1)
    pos = torch.randn(20, 84, device=dev(), generator=g)
    pos[[3, 7, 19]] = 0
    kv = torch.empty(20, dtype=torch.uint8, device=dev())
    rs = torch.empty(20, device=dev())
    N.call("icap_region_valid", pos.data_ptr(), 20, 84, kv.data_ptr(), rs.data_ptr(), S())
    ref = (pos != 0).any(1)
    assert torch.equal(kv.bool(), ref) and torch.equal(rs, ref.float())
    for cdt in (torch.int32, torch.int64):
        cap = torch.randint(0, 9, (6, 10), device=dev(), generator=g).to(cdt)
        B, L = cap.shape
        inp = torch.empty(B * (L - 1), dtype=torch.int32, device=dev())
        tgt = torch.empty_like(inp)
        tv = torch.empty(B * (L - 1), dtype=torch.uint8, device=dev())
        rsc = torch.empty(B * (L - 1), device=dev())
        ci = torch.empty(1, dtype=torch.int32, device=dev())
        c2 = torch.empty(2, device=dev())
        N.call("icap_caption_prep", cap.data_ptr(), int(cdt == torch.int64), B, L, 0, inp.data_ptr(), tgt.data_ptr(),
               tv.data_ptr(), rsc.data_ptr(), ci.data_ptr(), c2.data_ptr(), S())
        torch.cuda.synchronize()
        assert torch.equal(inp.view(B, L - 1).long(), cap[:, :-1].long())
        assert torch.equal(tgt.view(B, L - 1).long(), cap[:, 1:].long())
        assert torch.equal(tv.view(B, L - 1).bool(), cap[:, :-1] != 0)
        n = int((cap[:, 1:] != 0).sum())
        assert int(ci) == n and float(c2[0]) == n and abs(float(c2[1]) - 1 / n) < 1e-9


def test_embed_colsum_adam():
    g = torch.Generator(device="cuda").manual_seed(6)
    V, E, M = 50, 24, 40
    table = torch.randn(V, E, device=dev(), generator=g)
    tok = torch.randint(0, V, (M, 3), device=dev(), generator=g, dtype=torch.int32)
    out = torch.empty(M, E, device=dev())
    rs = torch.empty(M, device=dev())
    N.call("icap_embed_fwd", F32, F32, tok.data_ptr() + 4, 3, M, E, table.data_ptr(), out.data_ptr(), rs.data_ptr(), 0, S())
    assert torch.equal(out, table[tok[:, 1].long()]) and torch.equal(rs, (tok[:, 1] != 0).float())
    dout = torch.randn(M, E, device=dev(), generator=g)
    dtab = torch.zeros(V, E, device=dev())
    t1 = tok[:, 1].contiguous()
    N.call("icap_embed_bwd", F32, t1.data_ptr(), M, E, 0, dout.data_ptr(), dtab.data_ptr(), S())
    ref = torch.zeros(V, E, device=dev()).index_add_(0, t1.long(), dout)
    ref[0] = 0
    assert torch.allclose(dtab, ref, atol=1e-5)
    x = torch.randn(1000, 77, device=dev(), generator=g)
    cs = torch.ones(77, device=dev())
    N.call("icap_colsum", F32, 1000, 77, x.data_ptr(), 77, cs.data_ptr(), S())
    assert torch.allclose(cs, x.sum(0) + 1, atol=1e-3)
    # 16-byte path (N % 8 == 0), bf16 and fp32, padded leading dimension
    for tdt, code, tol in ((torch.float32, F32, 1e-3), (torch.bfloat16, BF16, 2e-2)):
        xw = torch.randn(3001, 520, device=dev(), generator=g).to(tdt)
        cw = torch.ones(512, device=dev())
        N.call("icap_colsum", code, 3001, 512, xw.data_ptr(), 520, cw.data_ptr(), S())
        ref_w = xw[:, :512].float().sum(0) + 1
        assert float((cw - ref_w).abs().max()) < tol * float(ref_w.abs().max())
    # Adam vs torch.optim.Adam for 3 steps
    n = 4096
    p = torch.randn(n, device=dev(), generator=g)
    p_ref = torch.nn.Parameter(p.clone())
    opt = torch.optim.Adam([p_ref], lr=5e-4)
    m, v = torch.zeros(n, device=dev()), torch.zeros(n, device=dev())
    sh = torch.empty(n, device=dev(), dtype=torch.bfloat16)
    step = torch.zeros(1, dtype=torch.int32, device=dev())
    for _ in range(3):
        gr = torch.randn(n, device=dev(), generator=g)
        p_ref.grad = gr.clone()
        opt.step()
        N.call("icap_adam_step", n, p.data_ptr(), gr.data_ptr(), m.data_ptr(), v.data_ptr(), sh.data_ptr(), 5e-4, 0.9,
               0.999, 1e-8, step.data_ptr(), 1, None, 1.0, S())
    torch.cuda.synchronize()
    assert int(step) == 3
    assert torch.allclose(p, p_ref.detach(), rtol=1e-5, atol=1e-6)
    assert torch.equal(sh, p.bfloat16())


def test_bad_arguments_return_errors_not_crashes():
    with pytest.raises(N.IcapError):
        N.call("icap_gemm", BF16, 0, 1, 128, 128, 64, 16, 64, 16, 64, 16, 128, F32, None, 0, None, 0, 0, 1, S())
    with pytest.raises(N.IcapError):
        N.call("icap_add_ln_fwd", F32, F32, 4, 30, 16, None, 1, 16, 16, None, 16, None, None, 0, 0.0, 0, None, 1e-6, S())
    assert "multiple of 4" in N.last_error()
