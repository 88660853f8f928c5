"""Sampled KV-cached decoding (icap_sample_tokens, Transformer.sample_captions) against an fp64 oracle.

The oracle restates the sampler's contract (include/icap.h) in numpy: the uniform of row r at decision t is
u = ((rand32(seed_fold(seed + c * golden), r * Tmax + t) >> 8) + 0.5) * 2^-24 (the dropout hash of icap_common.cuh,
imported from test_dropout_training_gpu), the token is the smallest j whose fp64 running sum of
w_j = exp((x_j - max x) / tau) exceeds u * sum w, and the log-probability is the fp64 log_softmax(x)[token] at tau = 1.
A decision may differ from the oracle's only when u * sum lies within eps of a CDF boundary; every such exemption is
counted and printed.  eps:
  * kernel cases (the same logits on both sides): the fp32 rounding of the device's running sum, at most
    (columns per thread + 17) * 2^-24 of the sum (sequential chunk sum, block scan, expf within 2 ulp), times 1.25;
  * end to end (device logits vs the CPU oracle's, parity 1e-4 of the row's largest logit = delta): a boundary F moves
    by at most F (1 - F) * 2 delta / tau; eps = 1.1 times that plus the kernel's eps.
Model A's classifier at initialisation spreads its logits by ~0.3 over 10000 words, which puts nearly every decision
within that eps of a boundary (a measured 75 % with the 1e-4 parity): the end-to-end cases scale the classifier by 14
(logits ~N(0, 4^2)) and raise the <END> bias by 10 so that captions end at varied lengths.

Bounds, and observed maxima on one NVIDIA B200 (1000 W power limit):

    quantity                                                bound       observed max
    kernel logp vs fp64 log_softmax (fp32 and bf16 logits)  1e-6        9.9e-7
    end-to-end fp32 logp vs the oracle's log_softmax        1e-4        2.9e-5
    bf16 sampler logp vs PolicyNetwork.forward log_softmax  0.1         7.8e-3 (bf16 logits: 2^-8 of ~2)

Observed on that run: 0 near-tie exemptions in 5088 kernel decisions; 3 in 5808 end-to-end decisions (at most 0.19 % of
a case), where the neighbouring row's uniform changes 75 % of the decisions (at least 62 % of a case); 0 at
tau = 1e-3 against greedy; chi-square p = 0.75 (tau 1) and 0.95 (tau 0.5) over 15 degrees of freedom.

81 cases: 60 kernel grid (fp32 / bf16 x V in {7, 300, 9999, 10000, 30000} x aligned / odd ldl x tau in {0.5, 1, 2}),
2 seed / counter, 2 chi-square, 2 argument checks without a GPU, 12 end to end, 1 low temperature, 1 bf16 model A at
512 images, 1 CLI.
"""
import math
import os

import numpy as np
import pytest
import torch

import icap_loader
from oracle import caption_oracle as O
from test_dropout_training_gpu import GOLDEN, hash32, seed_fold

pkg = icap_loader.load()
N = pkg._native
F32, BF16 = N.F32, N.BF16
END, PAD = 2, 0
U32 = np.uint32
KERNEL_SEED = 0x243F6A8885A308D3          # CaptionEngine.sample_seed
DEV = torch.device("cuda:0")


def S():
    return torch.cuda.current_stream().cuda_stream


def uniforms(seed, counter, rows, t, Tmax):
    """u of rows `rows` (integer array) at decision t."""
    sf = U32(seed_fold((seed + counter * GOLDEN) % 2 ** 64))
    idx = np.asarray(rows, dtype=np.uint64) * np.uint64(Tmax) + np.uint64(t)
    lo = (idx & np.uint64(0xFFFFFFFF)).astype(np.uint32)
    hi = (idx >> np.uint64(32)).astype(np.uint32)
    h = hash32(lo * U32(0x9E3779B1) + hi * U32(0x85EBCA77) + sf)
    return ((h >> U32(8)).astype(np.float64) + 0.5) * 2.0 ** -24


def kernel_eps(V):
    per = ((V + 7) // 8 + 255) // 256 * 8
    return 1.25 * (per + 17) * 2.0 ** -24


def oracle_decision(x, inv_tau, u, eps_fn):
    """x: fp64 logits row.  Returns (token, near) with near = u * sum within eps_fn(F) * sum of a boundary F of the
    chosen token's interval."""
    w = np.exp((x - x.max()) * inv_tau)
    c = np.cumsum(w)
    tot = c[-1]
    target = u * tot
    j = int(np.searchsorted(c, target, side="right"))
    if j >= len(x):
        j = int(np.nonzero(w)[0][-1])
    lo = c[j - 1] if j > 0 else 0.0
    near = any(abs(b - target) <= eps_fn(b / tot) * tot for b in (lo, c[j]) if 0.0 < b < tot)
    return j, near


def log_softmax64(x):
    m = x.max()
    return x - m - math.log(np.exp(x - m).sum())


def sample_call(act, logits, ldl, M, V, tau, counter, t, Tmax, tokens, logp, ldp, seed=KERNEL_SEED):
    cdev = torch.tensor([counter], dtype=torch.int32, device=DEV)
    N.call("icap_sample_tokens", act, M, V, logits.data_ptr(), ldl, 1.0 / tau, seed, cdev.data_ptr(), t, Tmax,
           tokens.data_ptr(), logp.data_ptr(), ldp, END, PAD, S())
    torch.cuda.synchronize()


def kernel_inputs(act, V, ldl, M, t, Tmax, g, sigma=4.0):
    dt = torch.float32 if act == F32 else torch.bfloat16
    x = torch.randn(M, V, generator=g) * sigma
    buf = torch.full((M * ldl + 8,), 100.0)             # padding columns would win every draw if they were read
    off = 0 if ldl % 8 == 0 else 1                      # an unaligned ldl also gets an unaligned base
    rows = buf[off:off + M * ldl].view(M, ldl)
    rows[:, :V] = x
    dev_buf = buf.to(DEV, dt)
    logits = dev_buf[off:off + M * ldl]
    x64 = logits.view(M, ldl)[:, :V].double().cpu().numpy()
    tokens = torch.randint(3, V if V > 3 else 4, (M, Tmax), generator=g, dtype=torch.int32)
    tokens[:, 0] = 1
    fin = torch.zeros(M, dtype=torch.bool)
    if t >= 1:
        fin[::7] = True
        tokens[::7, t] = END
        tokens[7::14, t] = PAD
    return logits, x64, tokens.to(DEV), fin


# ------------------------------------------------------------------------------------------ kernel
@pytest.mark.gpu
@pytest.mark.parametrize("act", [F32, BF16])
@pytest.mark.parametrize("V", [7, 300, 9999, 10000, 30000])
@pytest.mark.parametrize("ld", ["aligned", "odd"])
@pytest.mark.parametrize("tau", [0.5, 1.0, 2.0])
def test_kernel_vs_fp64(act, V, ld, tau):
    g = torch.Generator().manual_seed(V * 7 + int(tau * 4) + act)
    M, Tmax = 96, 6
    t = 0 if V == 7 else 3
    ldl = (V + 7) // 8 * 8 + 8 if ld == "aligned" else V + 3
    logits, x64, tokens, fin = kernel_inputs(act, V, ldl, M, t, Tmax, g)
    logp = torch.full((M, Tmax - 1), float("nan"), device=DEV)
    counter = 11
    sample_call(act, logits, ldl, M, V, tau, counter, t, Tmax, tokens, logp, Tmax - 1)
    tok = tokens.cpu().numpy()
    lp = logp.cpu().numpy()
    u = uniforms(KERNEL_SEED, counter, np.arange(M), t, Tmax)
    inv_tau = float(np.float32(1.0 / tau))
    eps = kernel_eps(V)
    near, worst = 0, 0.0
    for r in range(M):
        if fin[r]:
            assert tok[r, t + 1] == PAD and lp[r, t] == 0.0, r
            continue
        j, nr = oracle_decision(x64[r], inv_tau, u[r], lambda F: eps)
        if tok[r, t + 1] != j:
            assert nr, (r, int(tok[r, t + 1]), j)
            near += 1
            print(f"near-tie: row {r}: token {int(tok[r, t + 1])} (CUDA) vs {j} (oracle)")
        k = int(tok[r, t + 1])
        assert 0 <= k < V
        worst = max(worst, abs(lp[r, t] - log_softmax64(x64[r])[k]))
    print(f"V {V} ld {ld} tau {tau}: {near} near-tie exemptions of {int((~fin).sum())}; logp max err {worst:.2e}")
    assert worst < 1e-6
    # the rest of the token rows and logp are untouched
    assert np.isnan(np.delete(lp, t, axis=1)).all()


@pytest.mark.gpu
@pytest.mark.parametrize("act", [F32, BF16])
def test_kernel_same_seed_bitwise_and_counter_changes_tokens(act):
    g = torch.Generator().manual_seed(5)
    M, V, Tmax, t = 512, 300, 4, 1
    logits, _, tokens, fin = kernel_inputs(act, V, 304, M, t, Tmax, g, sigma=1.0)
    outs = []
    for counter in (3, 3, 4):
        tk = tokens.clone()
        lp = torch.zeros(M, Tmax - 1, device=DEV)
        sample_call(act, logits, 304, M, V, 1.0, counter, t, Tmax, tk, lp, Tmax - 1)
        outs.append((tk, lp))
    assert torch.equal(outs[0][0], outs[1][0]) and torch.equal(outs[0][1].view(torch.int32), outs[1][1].view(torch.int32))
    live = ~fin.to(DEV)
    differ = (outs[0][0][live, t + 1] != outs[2][0][live, t + 1]).float().mean()
    assert float(differ) > 0.9, float(differ)


@pytest.mark.gpu
@pytest.mark.parametrize("tau", [1.0, 0.5])
def test_kernel_distribution_chi_square(tau):
    """2^20 rows of one V = 16 logits row in one call: the token histogram against softmax(x / tau)."""
    from scipy.stats import chisquare
    M, V, Tmax = 1 << 20, 16, 2
    x = torch.tensor([0.3, -1.2, 2.0, 0.0, 1.1, -0.5, 0.7, -2.5, 1.6, 0.2, -0.1, 0.9, -3.0, 1.3, 0.4, -0.8])
    logits = x.to(DEV).repeat(M, 1).contiguous()
    tokens = torch.ones(M, Tmax, dtype=torch.int32, device=DEV)
    logp = torch.zeros(M, 1, device=DEV)
    sample_call(F32, logits, V, M, V, tau, 1234, 0, Tmax, tokens, logp, 1)
    hist = torch.bincount(tokens[:, 1].long(), minlength=V).cpu().numpy()
    p = torch.softmax(x.double() / tau, 0).numpy()
    stat, pval = chisquare(hist, p * M)
    print(f"tau {tau}: chi-square {stat:.2f} over {V - 1} degrees of freedom, p = {pval:.3f}")
    assert hist.sum() == M and pval > 1e-3
    lp_ref = torch.log_softmax(x.double(), 0).numpy()
    assert np.abs(logp[:, 0].cpu().numpy() - lp_ref[tokens[:, 1].cpu().numpy()]).max() < 1e-6


def test_kernel_argument_errors_without_a_gpu():
    """Argument checks run before any launch: a bad temperature, shape or pointer is an error code, not a crash."""
    fake = 0x1000
    bad = [(F32, 4, 10, fake, 16, float("inf"), fake, fake),      # tau = 0
           (F32, 4, 10, fake, 16, float("nan"), fake, fake),
           (F32, 4, 10, fake, 16, -1.0, fake, fake),
           (F32, 0, 10, fake, 16, 1.0, fake, fake),
           (F32, 4, 0, fake, 16, 1.0, fake, fake),
           (F32, 4, 10, None, 16, 1.0, fake, fake),
           (F32, 4, 10, fake, 16, 1.0, None, fake),
           (F32, 4, 10, fake, 16, 1.0, fake, None)]
    lib = N.lib()
    for act, M, V, lg, ldl, inv, tk, lp in bad:
        rc = lib.icap_sample_tokens(act, M, V, lg, ldl, inv, 1, None, 0, 4, tk, lp, 3, END, PAD, None)
        assert rc < 0, (M, V, inv)


def test_sample_captions_argument_errors_without_a_gpu():
    m = pkg.Transformer(num_vocab=50, max_length=6, encode_dim_positions=84, encode_dim_features=32, device="cpu",
                        output_name="x", encode_num_blocks=1, decode_num_blocks=1)
    f, p = torch.zeros(1, 3, 32), torch.zeros(1, 3, 84)
    for kw in (dict(num_samples=0), dict(num_samples=17), dict(temperature=0.0), dict(temperature=float("inf")),
               dict(temperature=-1.0), dict(seed=-1), dict(seed=2 ** 31)):
        with pytest.raises(ValueError):
            m.sample_captions(f, p, **kw)


# ------------------------------------------------------------------------------------------ end to end, fp32
def model_a_cfg(**over):
    kw = dict(num_vocab=10000, max_length=12, encode_dim_positions=84, encode_dim_features=2048, output_name="x",
              dropout=0.0, encode_num_blocks=2, decode_num_blocks=2)
    kw.update(over)
    return kw


def spread_state_dict(cfg, seed):
    sd = O.init_state_dict(cfg, seed=seed)
    sd["classifer.weight"] = sd["classifer.weight"] * 14.0
    sd["classifer.bias"] = sd["classifer.bias"] * 14.0
    sd["classifer.bias"][END] += 10.0
    return sd


def build(kw, sd, precision, cls=None):
    m = (cls or pkg.Transformer)(device=DEV, **kw)
    m.load_state_dict(sd)
    m = m.to(DEV).eval()
    m.set_precision(precision)
    return m


def first_stop(row):
    """Index of the first <END> or <NULL> after <START> (len(row) if none)."""
    hit = np.nonzero((row[1:] == END) | (row[1:] == PAD))[0]
    return int(hit[0]) + 1 if len(hit) else len(row)


@pytest.mark.gpu
@pytest.mark.parametrize("variant", ["default", "split_move_first"])
@pytest.mark.parametrize("n", [1, 5, 16])
@pytest.mark.parametrize("tau", [1.0, 0.7])
def test_sampled_decode_vs_oracle_fp32(variant, n, tau):
    over = dict(split_image_objects=True, move_first_image_feature=True) if variant == "split_move_first" else {}
    kw = model_a_cfg(**over)
    cfg = O.OracleConfig(**kw)
    sd = spread_state_dict(cfg, seed=1)
    B = 6
    f, p, _ = O.synthetic_batch(B, 36, 2048, 84, 12, 10000, seed=5)
    m = build(kw, sd, "fp32")
    seed = 77
    ids, logp = m.sample_captions(f, p, num_samples=n, temperature=tau, seed=seed)
    Tmax, T = kw["max_length"], kw["max_length"] - 1
    assert ids.shape == (B, n, Tmax) and logp.shape == (B, n, T) and ids.dtype == torch.long
    rows = ids.reshape(B * n, Tmax).cpu()
    lp = logp.reshape(B * n, T).cpu().numpy()
    rep = torch.arange(B).repeat_interleave(n)
    ref = O.logits_forward(sd, cfg, f[rep], p[rep], rows).double().numpy()     # teacher forced on the samples
    R = rows.numpy()
    inv_tau = float(np.float32(1.0 / tau))
    eps_k = kernel_eps(10000)
    decisions = near = moved = 0
    worst = 0.0
    for r in range(B * n):
        stop = first_stop(R[r])
        assert (R[r, stop + 1:] == PAD).all() and (lp[r, stop:] == 0).all(), r
        u = uniforms(KERNEL_SEED, seed, [r], np.arange(T), Tmax)
        u_nb = uniforms(KERNEL_SEED, seed, [(r + 1) % (B * n)], np.arange(T), Tmax)
        for t in range(min(stop, T)):
            x = ref[r, t]
            delta = 1e-4 * np.abs(x).max()
            j, nr = oracle_decision(x, inv_tau, u[t], lambda F: 1.1 * F * (1 - F) * 2 * delta / tau + eps_k)
            decisions += 1
            if R[r, t + 1] != j:
                assert nr, (r, t, int(R[r, t + 1]), j)
                near += 1
                print(f"near-tie: row {r} decision {t}: token {int(R[r, t + 1])} (CUDA) vs {j} (oracle)")
            moved += oracle_decision(x, inv_tau, u_nb[t], lambda F: 0.0)[0] != R[r, t + 1]
            worst = max(worst, abs(lp[r, t] - log_softmax64(x)[R[r, t + 1]]))
    print(f"{variant} n {n} tau {tau}: {decisions} decisions, {near} near-tie exemptions, neighbour's uniform "
          f"changes {moved}, logp max err {worst:.2e}")
    assert worst < 1e-4
    assert moved > decisions / 2                        # the check above is not vacuous
    assert near <= decisions // 4


@pytest.mark.gpu
def test_low_temperature_reproduces_greedy():
    kw = model_a_cfg()
    cfg = O.OracleConfig(**kw)
    sd = spread_state_dict(cfg, seed=2)
    f, p, _ = O.synthetic_batch(6, 36, 2048, 84, 12, 10000, seed=9)
    m = build(kw, sd, "fp32")
    greedy, _ = m.generate_caption_vector(f, p)
    gaps = m.last_gaps.t().cpu().numpy()                 # [B, T] top-2 logit gap of every greedy decision
    G = greedy[:, :kw["max_length"]].cpu().numpy()
    ids, _ = m.sample_captions(f, p, num_samples=3, temperature=1e-3, seed=5)
    ids = ids.cpu().numpy()
    for b in range(6):
        stop = first_stop(G[b])
        for s in range(3):
            neq = np.nonzero(ids[b, s, :stop + 1] != G[b, :stop + 1])[0]
            if len(neq):
                t = int(neq[0]) - 1
                # a runner-up within 0.03 of the top logit keeps a weight above exp(-30) at tau = 1e-3
                assert gaps[b, t] < 0.03, (b, s, t, float(gaps[b, t]))
                print(f"near-tie: image {b} sample {s} decision {t}: gap {gaps[b, t]:.2e}")


# ------------------------------------------------------------------------------------------ bf16, model A, 512 images
@pytest.mark.gpu
def test_bf16_model_a_512_images(monkeypatch):
    kw = model_a_cfg(max_length=22, encode_num_blocks=6, decode_num_blocks=6)
    torch.manual_seed(0)
    m = pkg.Transformer(device=DEV, **kw).to(DEV).eval()
    f, p, _ = O.synthetic_batch(512, 36, 2048, 84, 22, 10000, seed=4321)
    f, p = f.to(DEV), p.to(DEV)
    eng = m._engine()
    greedy0 = m.generate_caption_vector(f, p)[0].clone()
    beam0 = m.beam_search(f, p, beam_size=5).clone()
    step0 = eng.step_dev.clone()
    ids, logp = m.sample_captions(f, p, num_samples=5, seed=123)
    assert ids.shape == (512, 5, 22) and logp.shape == (512, 5, 21)
    assert bool((ids[:, :, 0] == 1).all()) and int(ids.min()) >= 0 and int(ids.max()) < 10000
    rows, lp = ids.reshape(-1, 22).cpu().numpy(), logp.reshape(-1, 21).cpu().numpy()
    for r in range(rows.shape[0]):
        stop = first_stop(rows[r])
        assert (rows[r, stop + 1:] == PAD).all() and (lp[r, stop:] == 0).all()
    assert np.isfinite(lp).all() and (lp <= 0).all()
    # graph replay == eager; fused step start == three launches
    monkeypatch.setenv("ICAP_DECODE_GRAPH", "0")
    e_ids, e_lp = m.sample_captions(f, p, num_samples=5, seed=123)
    monkeypatch.setenv("ICAP_DECODE_FUSED_START", "0")
    u_ids, u_lp = m.sample_captions(f, p, num_samples=5, seed=123)
    monkeypatch.delenv("ICAP_DECODE_FUSED_START")
    monkeypatch.delenv("ICAP_DECODE_GRAPH")
    for a, b in ((e_ids, e_lp), (u_ids, u_lp)):
        assert torch.equal(a, ids) and torch.equal(b.view(torch.int32), logp.view(torch.int32))
    # a region cache gives the tensor input's samples
    cache = pkg.RegionCache(m, f.cpu(), p.cpu())
    idx = torch.arange(512)
    c_ids, c_lp = m.sample_captions(cache.batch(idx), None, num_samples=5, seed=123)
    assert torch.equal(c_ids, ids) and torch.equal(c_lp.view(torch.int32), logp.view(torch.int32))
    # unseeded calls advance the counter
    a, _ = m.sample_captions(f, p, num_samples=5)
    b, _ = m.sample_captions(f, p, num_samples=5)
    assert not torch.equal(a, b)
    # sampling touches neither the dropout / Adam step counter nor greedy and beam search
    assert torch.equal(eng.step_dev, step0)
    assert torch.equal(m.generate_caption_vector(f, p)[0], greedy0)
    assert torch.equal(m.beam_search(f, p, beam_size=5), beam0)
    # PolicyNetwork.forward teacher forced on the samples: the same log-probabilities within bf16 rounding
    pk = {k: v for k, v in kw.items() if k != "output_name"}
    pn = pkg.PolicyNetwork(device=DEV, **pk)
    pn.load_state_dict(m.state_dict())
    pn = pn.to(DEV).eval()
    pn.set_precision("bf16")
    sub = 64
    srows = ids[:sub].reshape(sub * 5, 22)
    rep = torch.arange(sub, device=DEV).repeat_interleave(5)
    with torch.no_grad():
        lg = pn(f[rep], p[rep], srows)
        tf = torch.log_softmax(lg.double(), 2).gather(2, srows[:, 1:].unsqueeze(2)).squeeze(2).cpu().numpy()
    sl = logp[:sub].reshape(sub * 5, 21).cpu().numpy()
    sr = srows.cpu().numpy()
    worst = 0.0
    for r in range(sub * 5):
        stop = first_stop(sr[r])
        if stop > 0:
            worst = max(worst, float(np.abs(sl[r, :stop] - tf[r, :stop]).max()))
    print(f"bf16 sampler logp vs PolicyNetwork.forward: max abs difference {worst:.3e}")
    assert worst < 0.1


# ------------------------------------------------------------------------------------------ CLI
@pytest.mark.gpu
def test_cli_demo_prints_sampled_captions(tmp_path):
    from test_cli import _run
    r = _run(["demo", "--num-samples", "3", "--temperature", "0.8", "--seed", "4"], tmp_path)
    assert r.returncode == 0, r.stderr[-2000:]
    assert r.stdout.count("Sampled Caption:") == 3, r.stdout
    r = _run(["demo"], tmp_path)
    assert r.returncode == 0 and "Generated Caption:" in r.stdout and "Sampled Caption:" not in r.stdout
