"""The beam search that stops at <END> on the GPU (`pytest -m gpu`): icap_beam_select_eos against an fp64 construction of
its candidate set, icap_beam_finalize against numpy, and Transformer.beam_search_nbest against the CPU restatement
(tests/beam_eos_oracle.py), the PolicyNetwork-mode beam_search it must reproduce when no hypothesis can finish, and
itself (graph replay / eager, tensor / region-cache input, one / two decode streams)."""
import os
import subprocess
import sys

import numpy as np
import pytest
import torch

import icap_loader
from beam_eos_oracle import END, NULL, beam_search_eos, hypothesis_length, teacher_forced_logprob
from oracle import caption_oracle as O

pytestmark = pytest.mark.gpu
pkg = icap_loader.load()
N = pkg._native
F32, BF16 = N.F32, N.BF16
DEV = torch.device("cuda:0")
GOLD = os.path.join(os.path.dirname(__file__), "golden")
CASES = ["tiny_default", "tiny_cfgpy", "tiny_variants"]


def S():
    return torch.cuda.current_stream().cuda_stream


# ------------------------------------------------------------------------------------------ icap_beam_select_eos
def select_inputs(path, B, k, V, g, flat=False):
    """Logits of B * k rows as the decode leaves them (fp32 rows, or bf16 rows with the classifier GEMM's ROWSTATS
    buffer) -> (logits, ldl, stats, stats_ld, x64 [B*k, V] the stored values in fp64)."""
    rows, ldl = B * k, (V + 7) // 8 * 8
    if path == "fp32":
        x = torch.zeros(rows, V) if flat else torch.randn(rows, V, generator=g) * 3
        store = torch.zeros(rows, ldl)
        store[:, :V] = x
        logits = store.to(DEV)
        return logits, ldl, None, 0, logits[:, :V].double().cpu()
    d, P = 256, 2 * ((V + 255) // 256)
    X = torch.randn(rows, d, generator=g).to(DEV).bfloat16()
    W = (torch.randn(V, d, generator=g) * (0.0 if flat else 0.15)).to(DEV).bfloat16()
    bias = (torch.randn(V, generator=g) * (0.0 if flat else 0.5)).to(DEV)
    logits = torch.zeros(rows, ldl, device=DEV, dtype=torch.bfloat16)
    stats = torch.full((rows, 4 * P), float("nan"), device=DEV)
    N.call("icap_gemm", BF16, 1, 1, rows, V, d, X.data_ptr(), d, W.data_ptr(), d, logits.data_ptr(), ldl, BF16,
           bias.data_ptr(), N.EPI_ROWSTATS | N.EPI_B_STATIC, stats.data_ptr(), 4 * P, 0, 1, S())
    return logits, ldl, stats, 4 * P, logits[:, :V].double().cpu()


def select_eos(path, B, kin, kout, V, logits, ldl, stats, sld, prev, tokens, Tmax, t):
    out_s = torch.full((B, kout), float("nan"), device=DEV)
    out_p = torch.full((B, kout), -1, dtype=torch.int32, device=DEV)
    out_t = torch.full((B, kout), -1, dtype=torch.int32, device=DEV)
    gap = torch.full((B,), float("nan"), device=DEV)
    N.call("icap_beam_select_eos", F32 if path == "fp32" else BF16, B, kin, V, logits.data_ptr(), ldl,
           None if prev is None else prev.data_ptr(), kout, out_s.data_ptr(), out_p.data_ptr(), out_t.data_ptr(),
           gap.data_ptr(), 1, None if stats is None else stats.data_ptr(), sld, tokens.data_ptr(), Tmax, t, END, NULL, S())
    torch.cuda.synchronize()
    return out_s.cpu(), out_p.cpu(), out_t.cpu(), gap.cpu()


def reference_select(x64, prev, fin, kin, kout, V):
    """fp64 candidate set of the contract: (scores, flat indices) of the kout + 1 best per image, ties to the lower
    index (+ the count of real candidates)."""
    B = prev.shape[0]
    lp = torch.log_softmax(x64, dim=1).view(B, kin, V) + prev.double()[:, :, None]
    cand = lp.clone()
    for b in range(B):
        for r in range(kin):
            if fin[b, r]:
                cand[b, r] = float("-inf")
                cand[b, r, NULL] = float(prev[b, r])
    s, i = torch.sort(cand.view(B, kin * V), dim=1, descending=True, stable=True)
    return s[:, :kout + 1], i[:, :kout + 1]


def finished_pattern(which, B, k, g):
    if which == "none":
        return torch.zeros(B, k, dtype=torch.bool)
    if which == "all":
        return torch.ones(B, k, dtype=torch.bool)
    fin = torch.rand(B, k, generator=g) < 0.5
    fin[0, 0], fin[1, -1] = True, False
    return fin


def token_rows(fin, V, Tmax, t, g):
    B, k = fin.shape
    tok = torch.randint(3, V, (B * k, Tmax), generator=g, dtype=torch.int32)
    tok[:, 0] = 1
    f = fin.reshape(-1)
    alt = torch.arange(B * k) % 2 == 0
    tok[f & alt, t] = END
    tok[f & ~alt, t] = NULL
    return tok.to(DEV)


@pytest.mark.parametrize("path", ["fp32", "bf16_rowstats"])
@pytest.mark.parametrize("V", [397, 9999, 10000, 40000])
@pytest.mark.parametrize("k", [1, 3, 5, 8])
@pytest.mark.parametrize("finished", ["none", "some", "all"])
def test_select_eos_vs_fp64(path, V, k, finished):
    B, Tmax, t = 6, 7, 3
    g = torch.Generator().manual_seed(V * 31 + k * 7 + len(finished))
    logits, ldl, stats, sld, x64 = select_inputs(path, B, k, V, g)
    prev = -torch.rand(B, k, generator=g) * 6
    fin = finished_pattern(finished, B, k, g)
    tokens = token_rows(fin, V, Tmax, t, g)
    s, p, tk, gap = select_eos(path, B, k, k, V, logits, ldl, stats, sld, prev.to(DEV), tokens, Tmax, t)
    ref_s, ref_i = reference_select(x64, prev, fin, k, k, V)
    assert torch.equal(p.long(), ref_i[:, :k] // V) and torch.equal(tk.long(), ref_i[:, :k] % V)
    np.testing.assert_allclose(s.double().numpy(), ref_s[:, :k].numpy(), rtol=1e-5, atol=1e-6)
    ref_gap = (ref_s[:, k - 1] - ref_s[:, k]).numpy()
    inf = np.isinf(ref_gap)                            # an image whose k rows all finished has only k candidates
    assert inf.all() == (finished == "all") and np.array_equal(np.isinf(gap.numpy()), inf)
    np.testing.assert_allclose(gap.double().numpy()[~inf], ref_gap[~inf], rtol=1e-3, atol=2e-5)


@pytest.mark.parametrize("path", ["fp32", "bf16_rowstats"])
@pytest.mark.parametrize("finished", ["none", "some"])
def test_select_eos_exact_fallback_on_flat_logits(path, finished):
    """Flat logits: every token of an unfinished row ties (V = 10000 > the 1024-entry candidate list), so both kernels
    take their exact fall-back; the finished rows' single candidates must still enter it."""
    B, k, V, Tmax, t = 4, 5, 10000, 6, 2
    g = torch.Generator().manual_seed(5)
    logits, ldl, stats, sld, x64 = select_inputs(path, B, k, V, g, flat=True)
    prev = torch.zeros(B, k)
    prev[:, 1] = -12.0                                 # a finished row 1 loses to every unfinished candidate
    fin = finished_pattern(finished, B, k, g)
    if finished == "some":
        fin[:] = False
        fin[:, 1] = fin[:, 3] = True
    tokens = token_rows(fin, V, Tmax, t, g)
    s, p, tk, gap = select_eos(path, B, k, k, V, logits, ldl, stats, sld, prev.to(DEV), tokens, Tmax, t)
    ref_s, ref_i = reference_select(x64, prev, fin, k, k, V)
    assert torch.equal(p.long() * V + tk.long(), ref_i[:, :k])
    np.testing.assert_allclose(s.double().numpy(), ref_s[:, :k].numpy(), rtol=1e-5, atol=1e-6)
    if finished == "some":                             # row 3 (score 0) first, then row 0's tied tokens 0, 1, ...
        assert torch.equal(p[:, 0], torch.full((B,), 3, dtype=torch.int32)) and int(tk[0, 0]) == NULL


@pytest.mark.parametrize("path", ["fp32", "bf16_rowstats"])
@pytest.mark.parametrize("t", [0, 4])
def test_select_eos_equals_log_domain_select_when_nothing_finished(path, t):
    """The same arithmetic in the same order as icap_beam_select(log_domain = 1): bitwise equal outputs."""
    B, k, V, Tmax = 8, 5, 10000, 9
    g = torch.Generator().manual_seed(77 + t)
    kin = 1 if t == 0 else k
    logits, ldl, stats, sld, _ = select_inputs(path, B, kin, V, g)
    prev = None if t == 0 else (-torch.rand(B, k, generator=g) * 4).to(DEV)
    tokens = token_rows(torch.zeros(B, kin, dtype=torch.bool), V, Tmax, t, g)
    a = select_eos(path, B, kin, k, V, logits, ldl, stats, sld, prev, tokens, Tmax, t)
    out = [torch.full((B, k), float("nan"), device=DEV), torch.zeros(B, k, dtype=torch.int32, device=DEV),
           torch.zeros(B, k, dtype=torch.int32, device=DEV), torch.zeros(B, device=DEV)]
    N.call("icap_beam_select", F32 if path == "fp32" else BF16, B, kin, V, logits.data_ptr(), ldl,
           None if prev is None else prev.data_ptr(), k, *(o.data_ptr() for o in out), 1,
           None if stats is None else stats.data_ptr(), sld, S())
    torch.cuda.synchronize()
    for x, y in zip(a, out):
        assert torch.equal(x.view(torch.int32), y.cpu().view(torch.int32))


def test_select_eos_argument_checks():
    x = torch.zeros(4, 16, device=DEV)
    tok = torch.zeros(4, 5, dtype=torch.int32, device=DEV)
    prev = torch.zeros(4, device=DEV)
    o = torch.zeros(4, 4, device=DEV)
    oi = torch.zeros(4, 4, dtype=torch.int32, device=DEV)
    base = lambda kin, kout, t, log_domain=1: (F32, 1, kin, 16, x.data_ptr(), 16, prev.data_ptr(), kout, o.data_ptr(),
                                               oi.data_ptr(), oi.data_ptr(), None, log_domain, None, 0, tok.data_ptr(),
                                               5, t, END, NULL, S())
    N.call("icap_beam_select_eos", *base(4, 4, 1))                      # t >= 1: kin >= kout suffices
    for args in (base(3, 4, 1), base(4, 4, 1, 0), base(4, 4, 4), base(4, 9, 1)):
        with pytest.raises(N.IcapError):
            N.call("icap_beam_select_eos", *args)
    torch.cuda.synchronize()


# ------------------------------------------------------------------------------------------ icap_beam_finalize
@pytest.mark.parametrize("alpha", [0.0, 0.6, 1.0])
@pytest.mark.parametrize("n", [8, 3])
def test_finalize_vs_numpy(alpha, n):
    B, k, Tmax = 5, 8, 12
    rng = np.random.default_rng(int(alpha * 10) + n)
    tok = rng.integers(3, 400, size=(B * k, Tmax)).astype(np.int32)
    tok[:, 0] = 1
    for row in range(B * k):
        kind = row % 4
        if kind == 0:                                  # <END> at a varying position, <NULL> after it
            e = 1 + row % (Tmax - 1)
            tok[row, e], tok[row, e + 1:] = END, NULL
        elif kind == 2:                                # finished on <NULL>
            e = 1 + (row * 3) % (Tmax - 1)
            tok[row, e:] = NULL
        elif kind == 3 and row % 8 == 3:               # <END> as the last token
            tok[row, -1] = END
    score = (-rng.random((B, k)) * 20).astype(np.float32)
    ids = torch.empty(B, n, Tmax, dtype=torch.int32, device=DEV)
    sc = torch.empty(B, n, device=DEV)
    ln = torch.empty(B, n, dtype=torch.int32, device=DEV)
    td, sd = torch.from_numpy(tok).to(DEV), torch.from_numpy(score).to(DEV)
    N.call("icap_beam_finalize", B, k, Tmax, td.data_ptr(), sd.data_ptr(), END, NULL, alpha, n, ids.data_ptr(),
           sc.data_ptr(), ln.data_ptr(), S())
    torch.cuda.synchronize()
    for b in range(B):
        lens = np.array([hypothesis_length(tok[b * k + s]) for s in range(k)])
        norm = score[b].astype(np.float64) / ((5.0 + lens) / 6.0) ** alpha
        order = sorted(range(k), key=lambda s: (-norm[s], s))[:n]
        assert np.array_equal(ids[b].cpu().numpy(), tok[[b * k + s for s in order]])
        assert np.array_equal(sc[b].cpu().numpy(), score[b, order])
        assert np.array_equal(ln[b].cpu().numpy(), lens[order])
    lens_all = [hypothesis_length(r) for r in tok]
    assert len(set(lens_all)) > 5 and Tmax - 1 in lens_all


# ------------------------------------------------------------------------------------------ model level
def build(ctor, sd, precision):
    m = pkg.Transformer(device=DEV, **ctor)
    m.load_state_dict(sd)
    m = m.to(DEV).eval()
    m.set_precision(precision)
    return m


def gold_case(name, end_bias=0.0):
    g = torch.load(os.path.join(GOLD, name + ".pt"), weights_only=False)
    sd = {k: v.clone() for k, v in g["state_dict"].items()}
    sd["classifer.bias"][END] += end_bias
    return g, sd


@pytest.mark.parametrize("precision", ["fp32", "bf16"])
@pytest.mark.parametrize("k", [2, 3, 5])
def test_nbest_equals_policy_beam_when_no_hypothesis_can_finish(precision, k):
    """<END> and <NULL> biased to -1e4: nothing finishes, and with length_penalty 0 the best hypothesis and its score are
    the PolicyNetwork-mode (log-probability) beam search's, bit for bit."""
    g, sd = gold_case("tiny_default")
    sd["classifer.bias"][END] = -1e4
    sd["classifer.bias"][NULL] = -1e4
    m = build(g["ctor"], sd, precision)
    f, p = g["features"], g["positions"]
    ids, scores, lens = m.beam_search_nbest(f, p, beam_size=k, length_penalty=0.0)
    m.log_domain_beam = True
    ref_ids = m.beam_search(f, p, beam_size=k)
    fa, pa, _ = m._engine().prepare_inputs(f, p)
    ref_score = m._decode(fa, pa, k, True, False)["score"]
    assert torch.equal(ids[:, 0], ref_ids)
    assert torch.equal(scores[:, 0].view(torch.int32), ref_score.view(torch.int32))
    assert bool((lens == m.max_length - 1).all())


def assert_nbest_shape(ids, scores, lens, m, alpha):
    B, n, L = ids.shape
    assert L == m.max_length and bool((ids[:, :, 0] == 1).all())
    ids_c, sc, ln = ids.cpu(), scores.cpu().double(), lens.cpu()
    for b in range(B):
        norm = sc[b] / ((5.0 + ln[b].double()) / 6.0) ** alpha
        assert bool((norm[:-1] >= norm[1:] - 1e-6 * norm.abs().max()).all()), norm
        for i in range(n):
            row = ids_c[b, i]
            assert int(ln[b, i]) == hypothesis_length(row)
            stop = [j for j in range(1, L) if int(row[j]) in (END, NULL)]
            if stop:
                assert bool((row[stop[0] + 1:] == NULL).all()), row


def first_differing_step(a, b):
    """Smallest decision t whose prefixes (positions 0..t+1) differ as sets over the n hypotheses, else None."""
    for pos in range(1, a.shape[1]):
        if {tuple(r[:pos + 1].tolist()) for r in a} != {tuple(r[:pos + 1].tolist()) for r in b}:
            return pos - 1
    return None


@pytest.mark.parametrize("name", CASES)
@pytest.mark.parametrize("k,alpha", [(3, 0.6), (5, 0.0), (4, 1.0)])
def test_nbest_fp32_vs_oracle(name, k, alpha):
    g, sd = gold_case(name, end_bias=4.0)
    m = build(g["ctor"], sd, "fp32")
    f, p = g["features"], g["positions"]
    ids, scores, lens = m.beam_search_nbest(f, p, beam_size=k, length_penalty=alpha)
    assert m.last_gaps.shape == (m.max_length - 1, f.shape[0])
    assert_nbest_shape(ids, scores, lens, m, alpha)
    cfg = O.OracleConfig(**g["ctor"])
    r_ids, r_scores, r_lens, trace = beam_search_eos(sd, cfg, f, p, beam_size=k, length_penalty=alpha, return_trace=True)
    ids, scores = ids.cpu(), scores.cpu()
    assert bool((lens.cpu() < m.max_length - 1).any()), "no hypothesis finished: the case does not test <END>"
    for b in range(f.shape[0]):
        if torch.equal(ids[b], r_ids[b]):
            np.testing.assert_allclose(scores[b].numpy(), r_scores[b].numpy(), rtol=1e-4, atol=1e-5)
            continue
        t = first_differing_step(ids[b], r_ids[b])
        if t is None:                                  # same hypotheses, ranked differently: a normalised-score near-tie
            norm = lambda s, n_: s.double() / ((5.0 + n_.double()) / 6.0) ** alpha
            nr = norm(r_scores[b], r_lens[b])
            assert float((nr[:-1] - nr[1:]).abs().min()) < 1e-4, (b, nr)
            print(f"near-tie: image {b}: normalised scores {nr.tolist()} rank in a different order")
            continue
        gap = float(trace[b, t])
        assert gap < 1e-5, f"image {b}: hypotheses differ from step {t} on, oracle gap {gap:.3e}"
        print(f"near-tie: image {b}, step {t}: oracle gap {gap:.3e} < 1e-5")


@pytest.mark.parametrize("name", CASES)
def test_nbest_bf16_scores_are_the_tokens_log_likelihood(name):
    g, sd = gold_case(name, end_bias=4.0)
    m = build(g["ctor"], sd, "bf16")
    f, p = g["features"], g["positions"]
    alpha = 0.6
    ids, scores, lens = m.beam_search_nbest(f, p, beam_size=4, length_penalty=alpha)
    assert_nbest_shape(ids, scores, lens, m, alpha)
    B, n, L = ids.shape
    rows = ids.reshape(B * n, L)
    logits = m.logits(f.repeat_interleave(n, 0), p.repeat_interleave(n, 0), rows.int().cpu())
    ll = teacher_forced_logprob(logits.cpu(), rows.cpu(), m.pad_idx)
    sc = scores.reshape(-1).double().cpu().numpy()
    assert (np.abs(sc - ll) <= 2e-2 * np.maximum(1.0, np.abs(ll))).all(), np.abs(sc - ll).max()


def test_nbest_consistency_graph_cache_streams(monkeypatch):
    """Graph replay == eager decode; a region cache gives the tensor input's result; two decode streams give one's;
    beam_search is unchanged by a beam_search_nbest call in between."""
    kw = dict(num_vocab=500, max_length=12, encode_dim_positions=84, encode_dim_features=256, output_name="x",
              dropout=0.0, encode_input_size=128, encode_q_k_dim=128, encode_v_dim=128, encode_hidden_size=256,
              encode_num_blocks=2, encode_num_heads=4, dim_word_embedding=128, decode_input_size=128,
              decode_q_k_dim=128, decode_v_dim=128, decode_hidden_size=256, decode_num_blocks=2, decode_num_heads=4)
    cfg = O.OracleConfig(**kw)
    sd = O.init_state_dict(cfg, seed=3)
    sd["classifer.bias"][END] += 4.0
    f, p, _ = O.synthetic_batch(128, 13, 256, 84, 12, 500, seed=9)
    for precision in ("bf16", "fp32"):
        m = build(kw, sd, precision)
        before = m.beam_search(f, p, beam_size=4)
        ref = m.beam_search_nbest(f, p, beam_size=5, n_best=3, length_penalty=0.6)
        gaps = m.last_gaps.clone()
        assert torch.equal(m.beam_search(f, p, beam_size=4), before)
        assert bool((ref[2] < 11).any())
        again = m.beam_search_nbest(f, p, beam_size=5, n_best=3, length_penalty=0.6)
        monkeypatch.setenv("ICAP_DECODE_GRAPH", "0")
        eager = m.beam_search_nbest(f, p, beam_size=5, n_best=3, length_penalty=0.6)
        eager_gaps = m.last_gaps.clone()
        monkeypatch.delenv("ICAP_DECODE_GRAPH")
        cache = pkg.RegionCache(m, f, p)
        cached = m.beam_search_nbest(cache.batch(torch.arange(128)), None, beam_size=5, n_best=3, length_penalty=0.6)
        m._decode_graphs = {}
        monkeypatch.setenv("ICAP_DECODE_STREAMS", "2")
        split = m.beam_search_nbest(f, p, beam_size=5, n_best=3, length_penalty=0.6)
        split_gaps = m.last_gaps.clone()
        monkeypatch.delenv("ICAP_DECODE_STREAMS")
        for other in (again, eager, cached, split):
            assert torch.equal(other[0], ref[0]) and torch.equal(other[2], ref[2])
            assert torch.equal(other[1].view(torch.int32), ref[1].view(torch.int32))
        for og in (eager_gaps, split_gaps):
            assert torch.equal(og.view(torch.int32), gaps.view(torch.int32))


# ------------------------------------------------------------------------------------------ CLI
def _run(args, tmp_path):
    pkgdir = os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "image-caption_b200")
    env = dict(os.environ, ICAP_MAX_LENGTH="10", ICAP_SYNTHETIC_VOCAB="500", ICAP_BATCH_SIZE="8", ICAP_NUM_EPOCH="1")
    return subprocess.run([sys.executable, os.path.join(pkgdir, "main.py"), *args], cwd=tmp_path, env=env,
                          capture_output=True, text=True, timeout=600)


def test_cli_evaluation_length_penalty_and_demo_nbest(tmp_path):
    r = _run(["evaluation", "--split", "test", "--epoch", "1", "--length-penalty", "0.6", "--num-images", "16"], tmp_path)
    assert r.returncode == 0, r.stderr[-2000:]
    assert "16 captions" in r.stdout and "length penalty 0.6" in r.stdout and "CIDEr-D" in r.stdout
    r = _run(["demo", "--epoch", "1", "--n-best", "3"], tmp_path)
    assert r.returncode == 0, r.stderr[-2000:]
    lines = [ln for ln in r.stdout.splitlines() if ln.startswith("Beam Caption:")]
    assert len(lines) == 3 and all("log-probability" in ln for ln in lines)
