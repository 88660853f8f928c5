"""The vocabulary-side kernels of csrc/loss.cu against fp64, element by element, on every dispatch path, with a check
of which kernel ran.

Kernels and cases (every case runs its call under torch.profiler and matches the demangled kernel name):

* icap_xent, 76 cases: one per dispatch path x form x write_grad (1 and 0).  Paths: xent_reg_kernel<5> (bf16, 16-byte
  rows, V % 8 == 0, V <= 10240, ICAP_XENT_REG not 0); xent_kernel<T> with the row in shared memory (4V <= 48 KB), the
  same past 48 KB (opt-in, V <= 51200), and with the row re-read from memory (V > 51200).  Forms of xent_kernel: vector
  (16-byte base, ldl * size % 16 == 0; scalar tail V & ~3 .. V - 1) and scalar.  fp32 V in {1, 397, 12288, 12289,
  30000, 51200, 51201}, bf16 V in {8, 397, 10000, 10240, 10248, 12296, 30000, 51200, 51208, 60000}, each with an
  aligned ldl and with an odd ldl on a base that is not 16-byte aligned; ICAP_XENT_REG=0 at bf16 V in {8, 10000,
  10240}; M = 37, and M = 256 * 21 = 5376 (the training step's rows) at bf16 V = 10000 and 30000.  The path of a case
  is also checked from the `shared memory` field of its kernel record in the exported Chrome trace: at least 4V bytes
  on the two row-in-shared-memory paths, under 1 KB on the others.
* the bias gradient, 6 cases: icap_xent(write_grad=1) then icap_colsum over the written rows (stride ldl) at M = 5376,
  fp32 and bf16, V in {9999 (colsum_kernel), 10000, 30000 (colsum8_kernel)}.
* icap_xent_finalize, 24 cases: M in {1, 37, 255, 256, 257, 5376} x focal 0 / 1 x mean loss near 1e-3 / near ln 10^4.
* icap_argmax, 73 cases: fp32 and bf16 x V in {1, 7, 8, 300, 2048, 2049, 9999, 10000, 30000} x 16-byte / odd rows x
  gap on / off, M = 40; bf16 M = 512, V = 10000 (model A's greedy decode).  Into column t + 1 of an int32 [M, Tmax]
  token matrix (out_stride = Tmax).
* icap_log_softmax_argmax + icap_log_softmax_bwd, 10 cases: fp32 V in {1, 7, 1000, 10000, 30000} x idx null / not.

Inputs: rows of randn (sigma 1 and 4; argmax: sigma 2 and randint(-3, 4), where ties are everywhere), a logit 100 above
the rest (nearly every probability underflows), all-equal rows, targets at 0, V - 1, in the scalar tail and at the row's
maximum, every fifth row ignored (ignore_index 0, the pad id; -1 in the V = 1 and one bf16 V = 397 case), inv_count
1 / n (aligned cases) and 1 (odd cases, the data-parallel scaling).  Argmax rows place the maximum twice: inside one
thread's 8-column chunk, 8 columns apart (two threads), 2048 apart (one thread, two passes), at 0 and V - 1.  Padding
columns and a guard row on each side hold +100 (a kernel that read them would change its result) and must be bitwise
unchanged afterwards; so must every output element outside the written block (row_loss, out2, token columns other than
t + 1, gap, idx, logp and dx padding).  With write_grad = 0 the whole logits buffer is bitwise unchanged.

References are fp64 on the GPU from the values exactly as stored.  Arg-max indices (first index of the maximum) and
gaps (float32(top1 - top2), top2 counting duplicates: a tie gives 0) must be bit-exact.  Ignored rows must have loss 0
and, with write_grad = 1, an exactly zero gradient row.  Bounds, with u = 2^-24 and n_t = ceil(V / 256), the terms one
thread adds in order:

* lse (fp32): the block sum of exp(x - max) has (n_t + 13) roundings (13: five shuffle levels, eight warp sums) and
  2 ulp per expf; __expf (bf16 mode) is off by 2 + 1.17 |d| ulp at argument d, which adds 1.2 u times the p-weighted
  mean of |x - max|; logf adds 1 ulp of log(sum), max + log one rounding: err_lse = (n_t + 15 + 1.2 w) u +
  (2 |log sum| + |lse|) u.
* row loss: err_lse + (|x_t| + |loss|) u, absolute.
* gradient element j: (r + 2u + err_lse + (4 + 2.2 |x_j - lse|) u) (|ref_j| + [j = t] p_t s) (1 + 2^-8) + 1.01 * 2^-126
  max(1, s).  r = output rounding: 2^-8 in bf16 (half the spacing of its 8-bit significand), u in fp32; 2u for (p - [j = t]) and its product with s; exp(x_j - lse) inherits err_lse and is off by
  its own (4 + 2.2 |x_j - lse|) u (expf / __expf, rounding of the argument).  The target's error scales with p_t s, not
  with its reference (1 - p_t) s, which underflows when the target logit sits 100 above the rest.  The floor covers
  exponentials, probabilities and products flushed to zero below 2^-126 (__expf flushes), times s.
* bias gradient column c: the sum over rows of the gradient bounds, plus (ceil(rows per split / 8) + 8 + splits) u of
  the column's sum of |ref| for the fp32 sum in no fixed order (split count restated from icap_colsum).
* mean loss: (ceil(M / 256) + 14) u relative.  Focal: om = 1 - expf(-ce) cancels for small ce, relative error
  (2 u pt + pt |d ce|) / om + u; loss 2 d_om + d_ce + 3u, d loss / d ce as the sum of its two terms' bounds.
* logp: u |logp| + err_lse (fp32 expf).  dx from the kernel's own logp: (n_t + 17) u (|g_j| + p_j sum |g|).

Largest error observed on one NVIDIA B200 (1000 W power limit), and the largest ratio of an error to its own bound:

    quantity                                          observed max                      max err / bound
    row loss, fp32 / bf16 (absolute)                  3.4e-6 / 1.4e-6                   0.33 / 0.33
    gradient, bf16 (relative to |ref| + p_t s)        3.89e-3 (M = 5376: 3.89e-3)       0.99
    gradient, fp32                                    3.5e-6                            0.25
    bias gradient, fp32 / bf16 (of column sum |ref|)  2.5e-6 / 3.1e-3                   0.05 / 0.79
    mean loss (relative)                              9.8e-8                            0.11
    focal loss, d loss / d ce; ce ~ 1e-3 / ~ 9        9.0e-5 / 6.7e-8 (relative)        0.37 / 0.24
    logp (absolute)                                   3.3e-6                            0.60
    dx (relative to |g_j| + p_j sum |g|)              8.7e-8                            0.08

The fp32 bias-gradient and dx bounds sit 20x and 12x above what was seen: they are worst-case sums, which assume that
all the roundings of a column sum (of a row sum) go the same way; the errors of random data grow like the square root
of their number.  The bf16 gradient bound is the output rounding itself, reached within 1 %.  The whole file runs in
8 s on that card.

Found by these tests: an fp32 row of V = 12288 (and any V in 12281 .. 12288) failed to launch -- 48 KB of dynamic
shared memory next to xent_kernel's 32 static bytes is over the limit without the opt-in, and ensure_smem opted in only
above 48 KB.  It now starts from the kernel's own limit (cudaFuncGetAttributes).
"""
import json
import math
import os
import re
import subprocess
import sys
import xml.etree.ElementTree as ET
from dataclasses import dataclass

import pytest
import torch
import icap_loader
from test_dropout_training_gpu import assert_kernels
from torch.profiler import ProfilerActivity, profile

pkg = icap_loader.load()
N = pkg._native
F32, BF16 = N.F32, N.BF16
TNAME = {F32: "float", BF16: "__nv_bfloat16"}
gpu = pytest.mark.gpu
DEV = torch.device("cuda:0")

U = 2.0 ** -24                  # fp32 unit roundoff
TINY = 2.0 ** -126              # smallest normal fp32: __expf flushes below it
OUT_ROUND = {F32: 2.0 ** -24, BF16: 2.0 ** -8}      # half the spacing of a 24- / 8-bit significand
SENT = 100.0                    # padding / guard value of every input: a kernel that reads it changes its result
PAD = 0                         # the pad id, CrossEntropyLoss(ignore_index=pad)
NT = 256                        # threads per row of every kernel here

# icap_xent's dispatch (loss.cu), restated
REG_MAX_V = 5 * NT * 8          # xent_reg_kernel<5>: the whole row in registers
SMEM_DEFAULT = 48 * 1024        # dynamic shared memory without the opt-in
SMEM_CACHE_MAX = 200 * 1024     # largest row staged in shared memory


# The GPU tests run in a fresh Python process of their own.  Late in a whole-suite process, after the engine tests,
# torch.profiler recorded each launch but delivered no kernel record at all, every session of a test alike (B200,
# 190 GB of device memory free, with or without CUPTI teardown); in a fresh process every kernel record arrives.  The
# kernel checks depend on those records, so the suite's process runs this file's GPU tests once in a child process and
# each test reports the child's outcome.
IN_CHILD = os.environ.get("ICAP_VOCAB_TESTS_CHILD") == "1"


@pytest.fixture(scope="module")
def child_outcomes(tmp_path_factory):
    """{test name: None (passed) | failure text} of this file's GPU tests, run in a fresh process."""
    xml = tmp_path_factory.mktemp("vocab_child") / "junit.xml"
    r = subprocess.run([sys.executable, "-m", "pytest", __file__, "-q", "-m", "gpu", "-p", "no:cacheprovider",
                        f"--junitxml={xml}"], cwd=os.path.dirname(os.path.dirname(os.path.abspath(__file__))),
                       env=dict(os.environ, ICAP_VOCAB_TESTS_CHILD="1"), capture_output=True, text=True)
    out = {}
    if xml.exists():
        for case in ET.parse(xml).getroot().iter("testcase"):
            bad = [e for e in case if e.tag in ("failure", "error", "skipped")]
            out[case.get("name")] = (bad[0].get("message", "") + "\n" + (bad[0].text or ""))[-4000:] if bad else None
    out[None] = (r.stdout + r.stderr)[-4000:]
    return out


def in_parent(request):
    """True in the suite's process, after asserting that this test passed in the fresh child process."""
    if IN_CHILD:
        return False
    out = request.getfixturevalue("child_outcomes")
    name = request.node.name
    assert name in out, f"{name} did not run in the child process; its output:\n{out[None]}"
    assert out[name] is None, f"{name} failed in the child process:\n{out[name]}"
    return True


def S():
    return torch.cuda.current_stream().cuda_stream


def dt(act):
    return torch.float32 if act == F32 else torch.bfloat16


@pytest.fixture
def xent_reg(monkeypatch):
    """xent_reg(on): ICAP_XENT_REG removed (on) or set to 0 (off); libicap re-reads it, and again at the end."""
    def set_(on):
        if on:
            monkeypatch.delenv("ICAP_XENT_REG", raising=False)
        else:
            monkeypatch.setenv("ICAP_XENT_REG", "0")
        N.call("icap_reload_env")
    set_(True)
    yield set_
    monkeypatch.undo()
    N.call("icap_reload_env")


def traced_kernels(fn, tmp_path):
    """(name, args) of every CUDA kernel `fn` launches, from the Chrome trace torch.profiler exports."""
    torch.cuda.synchronize()
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        fn()
        torch.cuda.synchronize()
    path = os.path.join(str(tmp_path), "trace.json")
    prof.export_chrome_trace(path)
    with open(path) as f:
        events = json.load(f)["traceEvents"]
    return [(e["name"], e.get("args", {})) for e in events if e.get("cat") == "kernel"]


def report(what, err, ratio):
    """Largest error of one quantity in one case and its largest ratio to its bound, printed (pytest -s) as the source
    of the docstring's table."""
    print(f"\nOBS {what}: max err {err:.3e}, max err / bound {ratio:.3f}")


# ------------------------------------------------------------------------------------------ padded rows
def leading_dim(V, ld):
    """aligned: a multiple of 8 (16-byte rows in both dtypes); odd: an odd stride (V + 2 or V + 3)."""
    return (V + 7) // 8 * 8 + 8 if ld == "aligned" else V + (2 if V % 2 else 3)


def padded(act, M, V, ldl, ld, fill):
    """A device buffer [guard row, M rows, guard row] of stride ldl, all SENT, with fill(rows) written into the
    [M, V] block; an odd ldl also puts the first row on an element index = 1 mod 8 (a base that is not 16-byte
    aligned, as the kernels see it).  Returns (buffer, rows view [M, ldl], element offset of row 0)."""
    off = 0 if ld == "aligned" else (1 - ldl) % 8
    buf = torch.full((off + (M + 2) * ldl,), SENT, device=DEV, dtype=dt(act))
    rows = buf[off + ldl:off + (M + 1) * ldl].view(M, ldl)
    rows[:, :V] = fill.to(dt(act))
    return buf, rows, off + ldl


def rows_pointer(buf, first, act):
    return buf.data_ptr() + first * (4 if act == F32 else 2)


# ------------------------------------------------------------------------------------------ icap_xent cases
def xent_path(act, V, ldl, aligned, reg_on=True):
    """(path, form) icap_xent takes: reg | smem (row in shared memory, no opt-in) | smem_optin | mem (row re-read from
    global memory); vec (16-byte loads, scalar tail) | scalar."""
    esz = 4 if act == F32 else 2
    vec = aligned and (ldl * esz) % 16 == 0
    if act == BF16 and vec and V % 8 == 0 and V <= REG_MAX_V and reg_on:
        return "reg", "vec"
    smem = 4 * V
    path = "smem" if smem <= SMEM_DEFAULT else "smem_optin" if smem <= SMEM_CACHE_MAX else "mem"
    return path, "vec" if vec else "scalar"


@dataclass(frozen=True)
class XCase:
    act: int
    V: int
    ld: str             # aligned | odd
    write_grad: int
    M: int = 37
    reg_on: bool = True
    ignore: int = PAD

    @property
    def ldl(self):
        return leading_dim(self.V, self.ld)

    @property
    def path(self):
        return xent_path(self.act, self.V, self.ldl, self.ld == "aligned", self.reg_on)

    @property
    def kernel(self):
        return r"xent_reg_kernel<(\(int\))?5>" if self.path[0] == "reg" else rf"::xent_kernel<{TNAME[self.act]}>"

    @property
    def name(self):
        return (f"{'f32' if self.act == F32 else 'bf16'}-V{self.V}-{self.ld}-M{self.M}-grad{self.write_grad}"
                f"{'' if self.reg_on else '-REG0'}{'' if self.ignore == PAD else f'-ignore{self.ignore}'}"
                f"-{self.path[0]}-{self.path[1]}")


XENT_V = {F32: (1, 397, 12288, 12289, 30000, 51200, 51201),
          BF16: (8, 397, 10000, 10240, 10248, 12296, 30000, 51200, 51208, 60000)}
XCASES = [XCase(act, V, ld, wg, ignore=-1 if V == 1 or (act == BF16 and V == 397 and ld == "odd") else PAD)
          for act in (F32, BF16) for V in XENT_V[act] for ld in ("aligned", "odd") for wg in (1, 0)]
XCASES += [XCase(BF16, V, "aligned", wg, reg_on=False) for V in (8, 10000, 10240) for wg in (1, 0)]
XCASES += [XCase(BF16, V, "aligned", 1, M=256 * 21) for V in (10000, 30000)]     # model A / model C training step


def xent_rows(M, V, ignore, seed):
    """Logits [M, V] (fp32, device) and int32 targets.  Rows: randn with sigma 1 (even) / 4 (odd); per 37 rows one
    logit 100 above the rest (target on it, and elsewhere), an all-equal row, targets at 0, at V - 1, at the first
    column of the scalar tail V & ~3 (V - 1 when V % 4 == 0) and at the row's maximum; every fifth row ignored."""
    g = torch.Generator(device=DEV).manual_seed(seed)
    r = torch.arange(M, device=DEV)
    x = torch.randn(M, V, device=DEV, generator=g) * torch.where(r % 2 == 0, 1.0, 4.0)[:, None]
    tgt = torch.randint(0, V, (M,), device=DEV, generator=g)
    k = r % 37
    spike = (r * 7919) % V
    for kind in (1, 2):
        rows = (k == kind).nonzero().flatten()
        x[rows, spike[rows]] = x[rows].amax(1) + 100.0
    tgt = torch.where(k == 1, spike, tgt)
    tgt = torch.where((k == 2) & (tgt == spike), (spike + 1) % V, tgt)
    x[k == 3] = 0.75
    tgt = torch.where(k == 4, 0, tgt)
    tgt = torch.where(k == 6, V - 1, tgt)
    tgt = torch.where(k == 7, (V & ~3) if V % 4 else V - 1, tgt)
    tgt = torch.where(k == 8, x.argmax(1), tgt)
    tgt = torch.where(r % 5 == 0, ignore, tgt)
    return x, tgt.to(torch.int32)


def lse_error(x64, sum_exp, lse, fast_exp):
    """Bound on |fp32 lse - lse| per row.  Every thread sums ceil(V / 256) terms in order, the block adds its 256 sums
    in 5 shuffle levels and 8 warp sums in order: (ceil(V / 256) + 13) u of the sum, plus 2 u for the exponentials
    (expf: 2 ulp).  __expf (bf16 mode) is off by 2 + 1.17 |d| ulp at argument d, which adds the p-weighted mean of
    1.2 |x - max| u.  logf is within 1 ulp of log(sum), and the sum max + log rounds once more."""
    mx = x64.amax(1, keepdim=True)
    n_t = math.ceil(x64.shape[1] / NT)
    w = ((x64 - mx).exp() * (x64 - mx).abs()).sum(1) / sum_exp if fast_exp else 0.0
    eps_sum = (n_t + 15 + 1.2 * w) * U
    return eps_sum + (2 * sum_exp.log().abs() + lse.abs()) * U


@gpu
@pytest.mark.parametrize("cs", XCASES, ids=[c.name for c in XCASES])
def test_xent_path(cs, xent_reg, tmp_path, request):
    if in_parent(request):
        return
    act, V, M, ldl = cs.act, cs.V, cs.M, cs.ldl
    xent_reg(cs.reg_on)
    x, tgt = xent_rows(M, V, cs.ignore, seed=V * 11 + act + 3 * cs.write_grad + M)
    buf, rows, first = padded(act, M, V, ldl, cs.ld, x)
    before = buf.clone()
    valid = tgt != cs.ignore
    n = int(valid.sum())
    inv = torch.tensor([1.0 / max(n, 1) if cs.ld == "aligned" else 1.0], device=DEV)
    row_loss = torch.full((M + 2,), -7.0, device=DEV)              # one guard element on each side

    def run():
        N.call("icap_xent", act, M, V, rows_pointer(buf, first, act), ldl, tgt.data_ptr(), cs.ignore, inv.data_ptr(),
               row_loss.data_ptr() + 4, cs.write_grad, S())
    recs = traced_kernels(run, tmp_path)
    assert len(recs) == 1 and re.search(cs.kernel, recs[0][0]), f"expected {cs.kernel}, the trace has {recs}"
    args = recs[0][1]
    if "shared memory" not in args:
        pytest.fail(f"the profiler's kernel record carries no 'shared memory' field (fields: {sorted(args)}): the "
                    "shared-memory path of icap_xent cannot be checked with this torch build")
    smem = int(args["shared memory"])
    if cs.path[0] in ("smem", "smem_optin"):
        assert smem >= 4 * V, (cs.path, smem)
    else:
        assert smem < 1024, (cs.path, smem)

    # fp64 reference from the logits as stored
    x64 = before[first:first + M * ldl].view(M, ldl)[:, :V].double()
    mx = x64.amax(1, keepdim=True)
    sum_exp = (x64 - mx).exp().sum(1)
    lse = mx.squeeze(1) + sum_exp.log()
    t = tgt.long().clamp(0, V - 1)
    xt = x64.gather(1, t[:, None]).squeeze(1)
    loss_ref = torch.where(valid, lse - xt, 0.0)
    eps_lse = lse_error(x64, sum_exp, lse, act == BF16)

    loss = row_loss[1:M + 1].double()
    assert float(row_loss[0]) == -7.0 and float(row_loss[M + 1]) == -7.0, "row_loss written outside [0, M)"
    assert torch.equal(loss[~valid], torch.zeros_like(loss[~valid])), "ignored rows must have loss 0"
    err = (loss - loss_ref).abs()
    bound = eps_lse + (xt.abs() + loss_ref.abs()) * U
    report(f"xent row loss {cs.name}", float(err.max()), float((err / bound).max()))
    bad = (err > bound).nonzero().flatten()
    assert len(bad) == 0, f"row loss: rows {bad[:8].tolist()} err {err[bad[:8]].tolist()} bound {bound[bad[:8]].tolist()}"

    after = buf
    outside = torch.ones_like(buf, dtype=torch.bool)
    outside[first:first + M * ldl].view(M, ldl)[:, :V] = False
    assert torch.equal(after[outside].view(torch.int16 if act == BF16 else torch.int32),
                       before[outside].view(torch.int16 if act == BF16 else torch.int32)), \
        "padding columns or guard rows changed"
    grad = after[first:first + M * ldl].view(M, ldl)[:, :V]
    if not cs.write_grad:
        assert torch.equal(after.view(torch.int16 if act == BF16 else torch.int32),
                           before.view(torch.int16 if act == BF16 else torch.int32)), "write_grad=0 wrote the logits"
        return
    assert torch.equal(grad[~valid].double(), torch.zeros_like(grad[~valid], dtype=torch.float64)), \
        "ignored rows must have an exactly zero gradient"
    s = torch.where(valid, float(inv), 0.0).double()
    p = (x64 - lse[:, None]).exp()
    onehot = torch.zeros_like(p).scatter_(1, t[:, None], 1.0)
    ref = (p - onehot) * s[:, None]
    # per element: rounding of (p - [j = t]) * s and of the output; p_j = exp(x_j - lse) is off by the error of lse
    # plus (expf / __expf, argument rounding) (4 + 2.2 |x_j - lse|) u.  The target element's error scales with p_t s,
    # not with its reference |p_t - 1| s (a logit 100 above the rest: p_t - 1 underflows, p_t s does not).  Below
    # TINY * max(1, s) an exponential, a probability or a product may have flushed to 0.
    eps = OUT_ROUND[act] + 2 * U + eps_lse[:, None] + (4 + 2.2 * (x64 - lse[:, None]).abs()) * U
    scale = ref.abs() + onehot * p * s[:, None]
    floor = 1.01 * TINY * max(1.0, float(inv))
    bound = eps * scale * (1 + 2.0 ** -8) + floor
    err = (grad.double() - ref).abs()
    rel = torch.where(scale > floor / OUT_ROUND[act], err / scale.clamp_min(1e-300), 0.0)   # above the flush range
    bad = (err > bound).nonzero()
    report(f"xent gradient / (|ref| + [j=t] p_t s) {cs.name}", float(rel.max()), float((err / bound).max()))
    assert len(bad) == 0, (f"gradient: {len(bad)} elements out of bound, first (row, col) {bad[:6].tolist()}: "
                           f"err {err[tuple(bad[:6].t())].tolist()} bound {bound[tuple(bad[:6].t())].tolist()} "
                           f"ref {ref[tuple(bad[:6].t())].tolist()}")
    if cs.ld == "aligned" and n > 0:
        # the mean loss over the non-ignored rows from these row losses (CrossEntropyLoss(reduction='mean'))
        out2 = torch.empty(2, device=DEV)
        N.call("icap_xent_finalize", M, row_loss.data_ptr() + 4, inv.data_ptr(), 0, out2.data_ptr(), S())
        ce_ref = float(loss_ref.sum()) / n
        bound = float(bound_sum(M) * ce_ref + (eps_lse + (xt.abs() + loss_ref.abs()) * U)[valid].sum() / n) + \
            abs(float(inv) * n - 1) * ce_ref
        assert abs(float(out2[0]) - ce_ref) <= bound, (float(out2[0]), ce_ref, bound)


def bound_sum(M):
    """Relative error of xent_finalize's fp32 sum of M non-negative row losses times inv_count: ceil(M / 256) terms per
    thread, 13 levels of block reduction, one product."""
    return (math.ceil(M / NT) + 14) * U


def test_xent_case_table_reaches_every_path():
    """CPU: the cases reach every row of icap_xent's path table (register, row in shared memory without and with the
    opt-in, row re-read from memory), each xent_kernel path in its vector and its scalar form, for both dtypes, with
    write_grad 1 and 0; the register path also switched off by ICAP_XENT_REG=0."""
    rows = {(c.act, *c.path, c.write_grad) for c in XCASES}
    for act in (F32, BF16):
        for path in ("smem", "smem_optin", "mem"):
            for form in ("vec", "scalar"):
                for wg in (0, 1):
                    assert (act, path, form, wg) in rows, (act, path, form, wg)
    assert (F32, "reg", "vec", 1) not in rows
    assert (BF16, "reg", "vec", 1) in rows and (BF16, "reg", "vec", 0) in rows
    off = [c for c in XCASES if not c.reg_on]
    assert off and all(c.path == ("smem", "vec") and c.V % 8 == 0 and c.V <= REG_MAX_V for c in off)
    # the boundaries of the table sit inside the cases
    assert xent_path(F32, 12288, 12296, True) == ("smem", "vec") and xent_path(F32, 12289, 12304, True)[0] == "smem_optin"
    assert xent_path(F32, 51200, 51208, True)[0] == "smem_optin" and xent_path(F32, 51201, 51216, True)[0] == "mem"
    assert xent_path(BF16, 10240, 10248, True) == ("reg", "vec") and xent_path(BF16, 10248, 10256, True)[0] == "smem"
    for c in XCASES:
        assert bool(re.search(c.kernel, "void (anonymous namespace)::xent_reg_kernel<5>(int, __nv_bfloat16 *, long)")) \
            == (c.path[0] == "reg"), c.name
    assert any(c.ignore == -1 for c in XCASES) and {c.M for c in XCASES} == {37, 5376}


# ------------------------------------------------------------------------------------------ bias gradient chain
@gpu
@pytest.mark.parametrize("act", [F32, BF16])
@pytest.mark.parametrize("V", [9999, 10000, 30000])
def test_xent_then_colsum_bias_gradient(act, V, request):
    if in_parent(request):
        return
    M = 256 * 21
    ldl = leading_dim(V, "aligned")
    x, tgt = xent_rows(M, V, PAD, seed=V + 17 * act)
    buf, rows, first = padded(act, M, V, ldl, "aligned", x)
    x64 = rows[:, :V].double()
    valid = tgt != PAD
    inv = torch.tensor([1.0 / int(valid.sum())], device=DEV)
    out = torch.zeros(V, device=DEV)
    row_loss = torch.empty(M, device=DEV)
    eight = V % 8 == 0
    pat = rf"{'colsum8_kernel' if eight else 'colsum_kernel'}<{TNAME[act]}>"

    def run():
        N.call("icap_xent", act, M, V, rows_pointer(buf, first, act), ldl, tgt.data_ptr(), PAD, inv.data_ptr(),
               row_loss.data_ptr(), 1, S())
        N.call("icap_colsum", act, M, V, rows_pointer(buf, first, act), ldl, out.data_ptr(), S())
    xent_pat = r"xent_reg_kernel" if xent_path(act, V, ldl, True)[0] == "reg" else rf"::xent_kernel<{TNAME[act]}>"
    assert_kernels(run, [xent_pat, pat])

    mx = x64.amax(1, keepdim=True)
    sum_exp = (x64 - mx).exp().sum(1)
    lse = mx.squeeze(1) + sum_exp.log()
    p = (x64 - lse[:, None]).exp()
    t = tgt.long()
    onehot = torch.zeros_like(p).scatter_(1, t[:, None], 1.0)
    s = torch.where(valid, float(inv), 0.0).double()[:, None]
    ref = (p - onehot) * s
    # column c: the sum of the per-element bounds of test_xent_path over the rows, plus the fp32 summation: a thread adds
    # every 8th row of its row split in order, the block its 8 row lanes, and one atomic per split adds the block's sum
    # in no fixed order (the split count restated from icap_colsum)
    if eight:
        splits = max(1, min(math.ceil(148 * 4 / math.ceil(V / 256)), math.ceil(M / 32)))
    else:
        splits = max(1, min(math.ceil(148 * 8 / math.ceil(V / 32)), math.ceil(M / 64)))
    n_round = math.ceil(math.ceil(M / splits) / 8) + 8 + splits
    eps = OUT_ROUND[act] + 2 * U + lse_error(x64, sum_exp, lse, act == BF16)[:, None] + \
        (4 + 2.2 * (x64 - lse[:, None]).abs()) * U
    elem = (eps * (ref.abs() + onehot * p * s) * (1 + 2.0 ** -8) + 1.01 * TINY).sum(0)
    abs_sum = ref.abs().sum(0)
    bound = elem + n_round * U * abs_sum * (1 + OUT_ROUND[act])
    err = (out.double() - ref.sum(0)).abs()
    report(f"colsum of xent gradient / column sum |ref| ({'f32' if act == F32 else 'bf16'} V{V})",
           float((err / abs_sum).max()), float((err / bound).max()))
    bad = (err > bound).nonzero().flatten()
    assert len(bad) == 0, f"columns {bad[:8].tolist()}: err {err[bad[:8]].tolist()} bound {bound[bad[:8]].tolist()}"


# ------------------------------------------------------------------------------------------ icap_xent_finalize
@gpu
@pytest.mark.parametrize("M", [1, 37, 255, 256, 257, 5376])
@pytest.mark.parametrize("focal", [0, 1])
@pytest.mark.parametrize("level", ["near0", "lnV"])
def test_xent_finalize(M, focal, level, request):
    if in_parent(request):
        return
    g = torch.Generator(device=DEV).manual_seed(M * 4 + focal * 2 + (level == "lnV"))
    r = torch.arange(M, device=DEV)
    u = torch.rand(M, device=DEV, generator=g)
    row_loss = (u * 2e-3) if level == "near0" else (math.log(10000) + u - 0.5)
    row_loss = torch.where(r % 5 == 4, 0.0, row_loss)                 # ignored rows carry loss 0
    n = int((r % 5 != 4).sum())
    inv = torch.tensor([1.0 / n], device=DEV)
    out = torch.full((4,), -7.0, device=DEV)
    assert_kernels(lambda: N.call("icap_xent_finalize", M, row_loss.data_ptr(), inv.data_ptr(), focal,
                                  out.data_ptr() + 4, S()), [r"xent_finalize_kernel"])
    assert float(out[0]) == -7.0 and float(out[3]) == -7.0, "written outside out2[0:2]"
    ce_ref = float(row_loss.double().sum()) * float(inv)
    eps_ce = bound_sum(M)                                             # relative error of the fp32 ce
    o0, o1 = float(out[1]), float(out[2])
    if not focal:
        report(f"finalize ce M{M} {level}", abs(o0 - ce_ref) / ce_ref, abs(o0 - ce_ref) / (eps_ce * ce_ref))
        assert abs(o0 - ce_ref) <= eps_ce * ce_ref
        assert o1 == 1.0
        return
    ce = torch.tensor(ce_ref, dtype=torch.float64, requires_grad=True)
    fl = (1 - torch.exp(-ce)) ** 2 * ce
    fl.backward()
    f_ref, d_ref = float(fl.detach()), float(ce.grad)
    # pt = expf(-ce) (2 ulp, plus the ce error), om = 1 - pt: cancellation for small ce makes om's relative error
    # (2 u pt + pt |d ce|) / om + u; the products add a rounding each
    pt = math.exp(-ce_ref)
    om = 1 - pt
    d_om = (2 * U * pt + pt * eps_ce * ce_ref) / om + U
    d_pt = 2 * U + eps_ce * ce_ref
    b0 = (2 * d_om + eps_ce + 3 * U) * abs(f_ref)
    A, B = 2 * om * pt * ce_ref, om * om
    b1 = A * (d_om + d_pt + eps_ce + 3 * U) + B * (2 * d_om + U) + U * (A + B)
    report(f"finalize focal M{M} {level}: loss, d loss / d ce relative",
           max(abs(o0 - f_ref) / abs(f_ref), abs(o1 - d_ref) / abs(d_ref)), max(abs(o0 - f_ref) / b0, abs(o1 - d_ref) / b1))
    assert abs(o0 - f_ref) <= b0, (o0, f_ref, b0)
    assert abs(o1 - d_ref) <= b1, (o1, d_ref, b1)


# ------------------------------------------------------------------------------------------ icap_argmax
def argmax_rows(act, M, V, seed):
    """Even rows randn * 2, odd rows randint(-3, 4) (ties nearly everywhere); row 0 all equal; rows 1-4 hold a maximum
    50 twice: inside one thread's 8-column chunk, 8 columns apart (two threads), 2048 columns apart (one thread, two
    passes), at 0 and V - 1; rows 5 / 6 a single maximum at V - 1 / 0."""
    g = torch.Generator(device=DEV).manual_seed(seed)
    r = torch.arange(M, device=DEV)[:, None]
    x = torch.where(r % 2 == 0, torch.randn(M, V, device=DEV, generator=g) * 2,
                    torch.randint(-3, 4, (M, V), device=DEV, generator=g).float())
    x[0] = 1.5
    q = V // 16 * 8
    for row, cols in ((1, (q + 1, q + 5)), (2, (q, q + 8)), (3, (5, 2053)), (4, (0, V - 1)), (5, (V - 1,)), (6, (0,))):
        if row < M and max(cols) < V:
            x[row, list(cols)] = 50.0
    return x.to(dt(act)).float()


def first_max_and_gap(x):
    mx = x.amax(1)
    V = x.shape[1]
    idx = torch.where(x == mx[:, None], torch.arange(V, device=x.device), V).amin(1)
    top2 = x.topk(2, dim=1).values[:, 1] if V > 1 else torch.full_like(mx, -math.inf)
    return idx, (mx.double() - top2.double()).float()


ARGMAX_CASES = [(act, V, ld, gap, 40) for act in (F32, BF16) for V in (1, 7, 8, 300, 2048, 2049, 9999, 10000, 30000)
                for ld in ("aligned", "odd") for gap in (1, 0)]
ARGMAX_CASES.append((BF16, 10000, "aligned", 1, 512))          # model A's greedy decode: 512 images


@gpu
@pytest.mark.parametrize("act,V,ld,with_gap,M", ARGMAX_CASES,
                         ids=[f"{'f32' if a == F32 else 'bf16'}-V{V}-{ld}-gap{g}-M{M}" for a, V, ld, g, M in ARGMAX_CASES])
def test_argmax(act, V, ld, with_gap, M, request):
    if in_parent(request):
        return
    x = argmax_rows(act, M, V, seed=V * 3 + act)
    ldl = leading_dim(V, ld)
    buf, rows, first = padded(act, M, V, ldl, ld, x)
    before = buf.clone()
    Tmax, t = 6, 2
    tok = torch.full((M, Tmax), -7, dtype=torch.int32, device=DEV)
    gap = torch.full((M + 1,), -5.0, device=DEV)
    assert_kernels(lambda: N.call("icap_argmax", act, M, V, rows_pointer(buf, first, act), ldl,
                                  tok.data_ptr() + 4 * (t + 1), Tmax, gap.data_ptr() if with_gap else None, S()),
                   [rf"argmax_kernel<{TNAME[act]}>"])
    idx, gap_ref = first_max_and_gap(rows[:, :V].float())
    assert torch.equal(tok[:, t + 1].long(), idx), (tok[:, t + 1] != idx).nonzero().flatten()[:8].tolist()
    others = torch.ones(Tmax, dtype=torch.bool)
    others[t + 1] = False
    assert bool((tok[:, others] == -7).all()), "wrote outside column t + 1 of the token matrix"
    if with_gap:
        assert torch.equal(gap[:M].view(torch.int32), gap_ref.view(torch.int32)), \
            (gap[:M] != gap_ref).nonzero().flatten()[:8].tolist()
    assert float(gap[M]) == -5.0 and (with_gap or bool((gap == -5.0).all()))
    assert torch.equal(buf.view(torch.int16 if act == BF16 else torch.int32),
                       before.view(torch.int16 if act == BF16 else torch.int32))
    if V > 1:
        assert int((gap_ref == 0).sum()) >= 2, "the rows hold no ties"


# ------------------------------------------------------------------------------------------ log_softmax + argmax
@gpu
@pytest.mark.parametrize("V", [1, 7, 1000, 10000, 30000])
@pytest.mark.parametrize("with_idx", [1, 0])
def test_log_softmax_argmax_and_bwd(V, with_idx, request):
    if in_parent(request):
        return
    M = 24
    g = torch.Generator(device=DEV).manual_seed(V + with_idx)
    x = torch.randn(M, V, device=DEV, generator=g) * 3
    x[0] = -0.5                                                        # all equal
    for row, cols in ((1, (0, V - 1)), (2, (V // 2, V // 2 + 1)), (3, (3, 3 + NT)), (4, (V - 1,))):
        if max(cols) < V:
            x[row, list(cols)] = 40.0
    ldx, ldo, ldd, ldg = V + 5, V + 3, V + 7, V + 9
    xb, xr, xf = padded(F32, M, V, ldx, "odd", x)
    lb, lr, lf = padded(F32, M, V, ldo, "odd", torch.full((M, V), -3.0, device=DEV))
    lb[:] = -3.0
    dg = torch.randn(M, V, device=DEV, generator=g)
    gb, gr, gf = padded(F32, M, V, ldd, "odd", dg)
    db, dr, df = padded(F32, M, V, ldg, "odd", torch.full((M, V), -3.0, device=DEV))
    db[:] = -3.0
    idx = torch.full((M + 1,), -9, dtype=torch.int64, device=DEV)
    assert_kernels(lambda: N.call("icap_log_softmax_argmax", M, V, rows_pointer(xb, xf, F32), ldx,
                                  rows_pointer(lb, lf, F32), ldo, idx.data_ptr() if with_idx else None, S()),
                   [r"log_softmax_argmax_kernel"])
    assert_kernels(lambda: N.call("icap_log_softmax_bwd", M, V, rows_pointer(lb, lf, F32), ldo,
                                  rows_pointer(gb, gf, F32), ldd, rows_pointer(db, df, F32), ldg, S()),
                   [r"log_softmax_bwd_kernel"])
    x64 = xr[:, :V].double()
    if with_idx:
        ref_idx, _ = first_max_and_gap(xr[:, :V])
        assert torch.equal(idx[:M], ref_idx), (idx[:M] != ref_idx).nonzero().flatten()[:8].tolist()
    assert int(idx[M]) == -9 and (with_idx or bool((idx == -9).all()))
    for b, r, f, ld, what in ((lb, lr, lf, ldo, "logp"), (db, dr, df, ldg, "dx")):
        outside = torch.ones_like(b, dtype=torch.bool)
        outside[f:f + M * ld].view(M, ld)[:, :V] = False
        assert bool((b[outside] == -3.0).all()), f"{what} written outside its [M, V] block"
    mx = x64.amax(1, keepdim=True)
    sum_exp = (x64 - mx).exp().sum(1)
    lse = mx.squeeze(1) + sum_exp.log()
    lp_ref = x64 - lse[:, None]
    lp = lr[:, :V].double()
    # lp_j = fl(x_j - lse32): half an ulp of the result plus the error of lse (lse_error, expf)
    bound = U * lp_ref.abs() + lse_error(x64, sum_exp, lse, False)[:, None]
    err = (lp - lp_ref).abs()
    report(f"log_softmax logp V{V}", float(err.max()), float((err / bound).max()))
    assert bool((err <= bound).all()), f"logp: worst err / bound {float((err / bound).max()):.3g}"
    # dx_j = fl(g_j - expf(lp_j) * fl(sum g)) from the kernel's own logp: the fp32 sum of g in the order of lse_error,
    # expf 2 ulp, product and difference one rounding each
    gg = gr[:, :V].double()
    pk = lp.exp()
    dx_ref = gg - pk * gg.sum(1, keepdim=True)
    scale = gg.abs() + pk * gg.abs().sum(1, keepdim=True)
    bound = (math.ceil(V / NT) + 13 + 4) * U * scale
    err = (dr[:, :V].double() - dx_ref).abs()
    report(f"log_softmax_bwd dx / (|g_j| + p_j sum |g|) V{V}", float((err / scale).max()), float((err / bound).max()))
    assert bool((err <= bound).all()), f"dx: worst err / bound {float((err / bound).max()):.3g}"


# ------------------------------------------------------------------------------------------ argument checks
def test_vocab_kernel_argument_errors_without_a_gpu():
    """Row strides below V, V >= 2^31 and M >= 2^31 are argument errors, returned before any launch (fake pointers)."""
    fake, big = 0x1000, 2 ** 31
    lib = N.lib()
    calls = [
        ("icap_xent", lambda M, V, ld: lib.icap_xent(F32, M, V, fake, ld, fake, 0, fake, fake, 1, None)),
        ("icap_xent", lambda M, V, ld: lib.icap_xent(BF16, M, V, fake, ld, fake, 0, fake, fake, 0, None)),
        ("icap_argmax", lambda M, V, ld: lib.icap_argmax(BF16, M, V, fake, ld, fake, 4, fake, None)),
        ("icap_log_softmax_argmax", lambda M, V, ld: lib.icap_log_softmax_argmax(M, V, fake, ld, fake, V, fake, None)),
        ("icap_log_softmax_argmax", lambda M, V, ld: lib.icap_log_softmax_argmax(M, V, fake, V, fake, ld, None, None)),
        ("icap_log_softmax_bwd", lambda M, V, ld: lib.icap_log_softmax_bwd(M, V, fake, ld, fake, V, fake, V, None)),
        ("icap_log_softmax_bwd", lambda M, V, ld: lib.icap_log_softmax_bwd(M, V, fake, V, fake, ld, fake, V, None)),
        ("icap_log_softmax_bwd", lambda M, V, ld: lib.icap_log_softmax_bwd(M, V, fake, V, fake, V, fake, ld, None)),
    ]
    for name, fn in calls:
        for M, V, ld in ((4, 10, 9), (4, 10, 1), (4, big, big), (big, 10, 10)):
            assert fn(M, V, ld) < 0, (name, M, V, ld)
            assert N.last_error().startswith(name + ": bad logits shape"), (name, N.last_error())
    assert lib.icap_xent_finalize(big, fake, fake, 0, fake, None) < 0
    assert N.last_error() == "icap_xent_finalize: too many rows"
