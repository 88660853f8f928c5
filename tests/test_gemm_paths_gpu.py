"""icap_gemm on integer data, one or more cases per kernel and dispatch path, bit-exact against fp64, and a check of
which kernel ran.

icap_gemm chooses among 25 kernels: gemm_tc_kernel in three tile configurations (128x128, 128x256, the 256x256 CTA
pair) x three operand layouts x two C dtypes, plus its row-statistics build; gemm_small_kernel<2> and <3>; and the fp32
gemm_f32_kernel in four layouts.  Inside those, C leaves through a TMA store, a TMA reduce-add, direct stores or
atomics.  Every case below names the kernel it must run; its one icap_gemm call runs under torch.profiler and the
demangled kernel name must match, so a case cannot silently test another path.

Exact data: A and B hold integers in [-8, 8], bias integers in [-64, 64], the initial C of accumulating cases integers,
the ReLU-mask operand integers including 0 and -0.0.  Every partial sum is then an integer below 2^24, exact in fp32 in
any order and for any split of K, so the fp32 C must equal the fp64 reference exactly and the bf16 C must equal it
rounded to bf16.  Accumulating into bf16 C gives bf16(C + bf16(v)) on every store path (include/icap.h).  The
comparison is by value: it fails on any NaN and on any differing bit except the sign of a zero.

Guard band: C lives inside a larger buffer (ldc > N, rows above and below) filled with a NaN sentinel; afterwards every
element outside the [M, N] block must still hold the sentinel's bits.  The same holds for the row-statistics buffer
beyond the statistics the kernel writes, and the padding of A and B holds NaN, which a read would carry into C.
"""
import re
from dataclasses import dataclass

import pytest
import torch

import icap_loader

pkg = icap_loader.load()
N = pkg._native
F32, BF16 = N.F32, N.BF16
gpu = pytest.mark.gpu

# every ICAP_GEMM_* switch icap_gemm reads; a case sets the ones it names and removes the others
SWITCHES = ("ICAP_GEMM_BN", "ICAP_GEMM_SMALL", "ICAP_GEMM_SMALL_STAGES", "ICAP_GEMM_DIRECT_EPILOGUE",
            "ICAP_GEMM_NO_PAIR", "ICAP_GEMM_NO_B_PREFETCH", "ICAP_GEMM_SMS", "ICAP_GEMM_DEBUG")
TC_CFGS = ("128", "256", "pair")
TC_LAYOUTS = ((1, 1), (1, 0), (0, 0))          # (A K-major, B K-major); (0, 1) has no tcgen05 instantiation
SENTINEL = {F32: 0x7FA1A1A1, BF16: 0x7FA1}      # NaN payloads: bits no kernel writes
BIG_M = 8_391_936                              # stem GEMM of 669 crops (12544 rows each): ceil(M / 128) > 65535


# ------------------------------------------------------------------------------------------ kernels and their names
def tc(cfg, layout, c):
    return ("tc", cfg, layout[0], layout[1], c)


STATS = ("stats",)


def small(stages):
    return ("small", stages)


def f32k(layout):
    return ("f32", layout[0], layout[1])


ALL_KERNELS = ([tc(cfg, lay, c) for cfg in TC_CFGS for lay in TC_LAYOUTS for c in (F32, BF16)] + [STATS]
               + [small(2), small(3)] + [f32k(lay) for lay in ((1, 1), (1, 0), (0, 0), (0, 1))])


def _b(x):
    return r"(?:\(bool\))?" + ("(?:1|true)" if x else "(?:0|false)")


def _i(x):
    return rf"(?:\(int\))?{x}"


def kernel_regex(k):
    """Regex of the demangled name (with or without the demangler's (int) / (bool) casts)."""
    if k[0] in ("tc", "stats"):
        cfg, ak, bk, c, st = ("256", 1, 1, BF16, 1) if k[0] == "stats" else (*k[1:], 0)
        bn, two = (128, 0) if cfg == "128" else (256, int(cfg == "pair"))
        t = "float" if c == F32 else "__nv_bfloat16"
        return rf"gemm_tc_kernel<{_i(bn)}, {_b(two)}, {_b(ak)}, {_b(bk)}, {t}, {_b(st)}>\("
    if k[0] == "small":
        return rf"gemm_small_kernel<{_i(k[1])}>\("
    return rf"gemm_f32_kernel<{_b(k[1])}, {_b(k[2])}>\("


def kernel_of(name):
    """The ALL_KERNELS entry whose regex matches a demangled kernel name (None: not a GEMM kernel of icap_gemm)."""
    hits = [k for k in ALL_KERNELS if re.search(kernel_regex(k), name)]
    return hits[0] if len(hits) == 1 else None


def launched_kernels(fn):
    """Demangled names of the CUDA kernels `fn` launches, in order (profiler, CUDA activity only)."""
    from torch.profiler import ProfilerActivity, profile
    torch.cuda.synchronize()
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        fn()
        torch.cuda.synchronize()
    return [e.name for e in prof.events() if e.device_type == torch.autograd.DeviceType.CUDA
            and "memcpy" not in e.name.lower() and "memset" not in e.name.lower()]


# ------------------------------------------------------------------------------------------ cases
@dataclass(frozen=True)
class Case:
    name: str
    kernel: tuple                # expected kernel (None: record whichever runs)
    M: int
    N: int
    K: int
    ab: int = BF16
    layout: tuple = (1, 1)
    c: int = BF16                # C dtype
    bias: bool = False
    epi: int = 0                 # 0 none, 1 ReLU, 2 ReLU-mask, 3 row statistics
    acc: int = 0
    split_k: int = 1
    b_static: bool = False
    env: tuple = ()              # ((switch, value), ...)
    sms: int = 0                 # icap_set_gemm_sms
    amp: int = 8                 # A, B in [-amp, amp]
    bias_amp: int = 64
    lda: int = 0                 # 0: the operand's width rounded up to 8 (bf16) or itself (fp32), plus ld_pad
    ldb: int = 0
    ld_pad: int = 0
    ldc: int = 0                 # 0: N rounded up to 8, plus 8
    ldaux: int = 0               # 0: ldc
    a_off: int = 0               # pointer offsets in elements from a 256-byte boundary
    b_off: int = 0
    c_off: int = 0
    aux_off: int = 0


def env(**kw):
    return tuple(sorted(kw.items()))


def bn(cfg, **kw):
    return env(ICAP_GEMM_BN=cfg, ICAP_GEMM_SMALL="0", **kw)


def lay_name(lay):
    return {(1, 1): "kk", (1, 0): "km", (0, 0): "mm", (0, 1): "mk"}[lay]


def c_name(c):
    return "f32" if c == F32 else "bf16"


def build_cases():
    cs = []
    # --- all 18 gemm_tc_kernel instantiations, ragged: M % 128 != 0; pair: M % 256 in (0, 128] and in (128, 256);
    # N < 32 and N % 32 != 0; K in {8, 40}, K % 64 in {8, 56}, K longer than the smem ring (384 / 256 / 384) with a tail;
    # more tiles than SMs, so the TMEM accumulator stages and smem ring phases wrap
    shapes = {"128": [(300, 20, 8), (385, 200, 40), (1000, 392, 1032), (9000, 2100, 72), (130, 1000, 568), (700, 33, 136)],
              "256": [(300, 20, 40), (385, 300, 8), (1000, 392, 1032), (9000, 2100, 120), (130, 1000, 568), (700, 257, 136)],
              "pair": [(300, 20, 8), (400, 300, 40), (1000, 392, 1032), (9000, 2100, 72), (556, 1000, 568),
                       (1200, 257, 136)]}
    for cfg in TC_CFGS:
        i = 0
        for lay in TC_LAYOUTS:
            for c in (F32, BF16):
                M, Nn, K = shapes[cfg][i]
                cs.append(Case(f"tc-{cfg}-{lay_name(lay)}-{c_name(c)}-{M}x{Nn}x{K}", tc(cfg, lay, c), M, Nn, K, layout=lay,
                               c=c, bias=i % 2 == 1, env=bn(cfg)))
                i += 1
    # --- epilogues on each configuration and C dtype: TMA store (none / bias / ReLU / ReLU-mask) and reduce-add
    for cfg in TC_CFGS:
        for c in (F32, BF16):
            e = bn(cfg)
            base = dict(M=1000, N=392, K=1032, c=c, env=e)
            p = f"epi-{cfg}-{c_name(c)}"
            cs += [Case(f"{p}-bias", tc(cfg, (1, 1), c), bias=True, **base),
                   Case(f"{p}-bias-relu", tc(cfg, (1, 1), c), bias=True, epi=1, **base),
                   Case(f"{p}-mask", tc(cfg, (1, 0), c), layout=(1, 0), epi=2, **base),
                   Case(f"{p}-mask-aux-off4", tc(cfg, (1, 0), c), layout=(1, 0), epi=2, aux_off=4 // (4 if c == F32 else 2),
                        **base),
                   Case(f"{p}-acc", tc(cfg, (1, 1), c), bias=True, acc=1, **base),
                   Case(f"{p}-acc-mm", tc(cfg, (0, 0), c), layout=(0, 0), acc=1, **base)]
    # --- direct stores: forced, and natural (odd ldc, C not 16-byte aligned); plain and accumulating
    for cfg in TC_CFGS:
        for c in (F32, BF16):
            esz = 4 if c == F32 else 2
            p = f"direct-{cfg}-{c_name(c)}"
            base = dict(M=1000, N=392, K=1032, c=c, bias=True)
            for acc in (0, 1):
                a = "-acc" if acc else ""
                cs += [Case(f"{p}-forced{a}", tc(cfg, (1, 1), c), epi=0 if acc else 1, acc=acc,
                            env=bn(cfg, ICAP_GEMM_DIRECT_EPILOGUE="1"), **base),
                       Case(f"{p}-odd-ldc{a}", tc(cfg, (1, 1), c), acc=acc, ldc=393, env=bn(cfg), **base),
                       Case(f"{p}-c-off{esz}{a}", tc(cfg, (1, 0), c), layout=(1, 0), acc=acc, c_off=1, env=bn(cfg), **base)]
            # rows that end inside a 16-byte chunk: the TMA store would spill past N, so these leave through direct stores
            cs += [Case(f"{p}-ragged-n{a}", tc(cfg, (1, 1), c), 1000, 389, 200, c=c, bias=not acc, acc=acc,
                        env=bn(cfg))
                   for acc, a in ((0, ""), (1, "-acc"))]
            cs.append(Case(f"{p}-forced-mask-aux-off4", tc(cfg, (1, 0), c), layout=(1, 0), epi=2, aux_off=4 // esz,
                           env=bn(cfg, ICAP_GEMM_DIRECT_EPILOGUE="1"), M=1000, N=392, K=1032, c=c))
    # --- split-K (fp32 C): reduce-add on the staged path, atomics on the direct one; 3 splits, more splits than
    # k-blocks (K = 200: 4 k-blocks), automatic
    for cfg in TC_CFGS:
        for lay in ((0, 0), (1, 0)):
            p = f"splitk-{cfg}-{lay_name(lay)}"
            base = dict(c=F32, layout=lay, acc=1)
            cs += [Case(f"{p}-3", tc(cfg, lay, F32), 520, 392, 1032, split_k=3, env=bn(cfg), **base),
                   Case(f"{p}-9-of-4", tc(cfg, lay, F32), 520, 392, 200, split_k=9, env=bn(cfg), **base),
                   Case(f"{p}-auto", tc(cfg, lay, F32), 520, 392, 5000, split_k=0, env=bn(cfg), **base),
                   Case(f"{p}-3-atomics", tc(cfg, lay, F32), 520, 392, 1032, split_k=3, c_off=1, env=bn(cfg), **base),
                   Case(f"{p}-auto-atomics", tc(cfg, lay, F32), 520, 392, 5000, split_k=0,
                        env=bn(cfg, ICAP_GEMM_DIRECT_EPILOGUE="1"), **base)]
    # --- B_STATIC weight prefetch on the single-CTA configurations; with split-K, CTAs whose first tile is a split > 0
    for cfg in ("128", "256"):
        for lay in ((1, 1), (1, 0)):
            cs += [Case(f"bstatic-{cfg}-{lay_name(lay)}", tc(cfg, lay, BF16), 1000, 392, 1032, layout=lay, bias=True,
                        b_static=True, env=bn(cfg)),
                   Case(f"bstatic-{cfg}-{lay_name(lay)}-short-k", tc(cfg, lay, BF16), 300, 200, 40, layout=lay,
                        b_static=True, env=bn(cfg)),
                   Case(f"bstatic-{cfg}-{lay_name(lay)}-split-first", tc(cfg, lay, F32), 300, 200, 1032, layout=lay,
                        c=F32, acc=1, split_k=3, b_static=True, env=bn(cfg))]
    # --- row statistics (the one 128x256 build, chosen for any N): small operands so the exp-sums see many terms
    for Nn in (1, 127, 128, 129, 255, 257, 10000):
        cs.append(Case(f"rowstats-n{Nn}", STATS, 300, Nn, 40, bias=True, epi=3, amp=1, bias_amp=2, b_static=Nn == 10000))
    # --- the small-footprint kernel, forced (ICAP_GEMM_SMALL=2), each stage count
    for st in (2, 3):
        e = env(ICAP_GEMM_SMALL="2", ICAP_GEMM_SMALL_STAGES=str(st))
        cs += [Case(f"small{st}-bias-relu", small(st), 300, 200, 40, bias=True, epi=1, env=e),
               Case(f"small{st}-bias-long-k", small(st), 37, 1000, 1032, bias=True, env=e),
               Case(f"small{st}-n24-k8", small(st), 130, 24, 8, env=e),
               Case(f"small{st}-bstatic", small(st), 2560, 1536, 512, bias=True, epi=1, b_static=True, env=e),
               Case(f"small{st}-ragged", small(st), 515, 392, 200, env=e)]
    # ... and every reason it declines a GEMM: the persistent kernel runs it instead (N <= 128: 128x128 tiles)
    e = env(ICAP_GEMM_SMALL="2")
    cs += [Case("small-declines-acc", tc("128", (1, 1), BF16), 300, 100, 200, acc=1, env=e),
           Case("small-declines-f32-c", tc("128", (1, 1), F32), 300, 100, 200, c=F32, bias=True, env=e),
           Case("small-declines-ldc", tc("128", (1, 1), BF16), 300, 100, 200, bias=True, ldc=102, env=e),
           Case("small-declines-c-off", tc("128", (1, 1), BF16), 300, 100, 200, bias=True, c_off=1, env=e),
           Case("small-declines-mask", tc("128", (1, 1), BF16), 300, 100, 200, epi=2, env=e),
           Case("small-declines-ragged-n", tc("128", (1, 1), BF16), 300, 20, 200, bias=True, env=e),
           Case("small-declines-big-m", tc("128", (1, 1), BF16), BIG_M, 64, 64, env=e)]
    # --- the fp32 SIMT kernel: 4 layouts; vector and scalar loads (lda % 4 != 0, A not 16-byte aligned); epilogues;
    # split-K (atomics)
    for lay in ((1, 1), (1, 0), (0, 0), (0, 1)):
        p = f"f32-{lay_name(lay)}"
        base = dict(ab=F32, c=F32, layout=lay)
        k = f32k(lay)
        cs += [Case(f"{p}-vec", k, 300, 200, 136, **base),
               Case(f"{p}-scalar", k, 300, 200, 136, ld_pad=1, a_off=1, b_off=3, **base),
               Case(f"{p}-bias-relu", k, 259, 131, 1032, bias=True, epi=1, **base),
               Case(f"{p}-mask", k, 259, 131, 72, epi=2, aux_off=1, **base),
               Case(f"{p}-acc-bias", k, 259, 131, 72, bias=True, acc=1, ldc=133, **base),
               Case(f"{p}-splitk3", k, 259, 131, 1032, acc=1, split_k=3, **base)]
    cs.append(Case("f32-big-m", f32k((1, 1)), BIG_M, 64, 152, ab=F32, c=F32))
    # --- icap_set_gemm_sms: a pair needs two SMs, so one SM runs the forced pair on 128x128 tiles
    for cfg in TC_CFGS:
        for n in (1, 2, 3, 17, 0):
            want = "128" if (cfg == "pair" and n == 1) else cfg
            cs.append(Case(f"sms{n}-{cfg}", tc(want, (1, 1), BF16), 1000, 392, 1032, bias=True, epi=1, sms=n, env=bn(cfg)))
        cs.append(Case(f"sms{1}-{cfg}-splitk", tc("128" if cfg == "pair" else cfg, (0, 0), F32), 520, 392, 1032,
                       layout=(0, 0), c=F32, acc=1, split_k=3, sms=1, env=bn(cfg)))
    cs.append(Case("env-sms1-pair", tc("128", (1, 1), BF16), 1000, 392, 1032, bias=True, env=bn("pair", ICAP_GEMM_SMS="1")))
    cs.append(Case("env-sms1-auto", tc("256", (1, 1), F32), 1000, 392, 5184, c=F32, env=env(ICAP_GEMM_SMS="1")))
    # --- automatic dispatch: never the pair for M <= 128, even with a k loop long enough (81 k-blocks) to take it
    cs.append(Case("auto-m100-no-pair", tc("128", (1, 1), F32), 100, 300, 5184, c=F32))
    cs.append(Case("auto-m300-pair", tc("pair", (1, 1), F32), 300, 300, 5184, c=F32))
    return cs


CASES = build_cases()
assert len({c.name for c in CASES}) == len(CASES)


# ------------------------------------------------------------------------------------------ fixtures
@pytest.fixture
def switches(monkeypatch):
    """set(NAME=value, ...): exactly these ICAP_GEMM_* switches present, the others removed; libicap re-reads them.
    The grid limit of icap_set_gemm_sms is reset at teardown."""
    def set_(pairs=()):
        for name in SWITCHES:
            monkeypatch.delenv(name, raising=False)
        for name, value in pairs:
            monkeypatch.setenv(name, value)
        N.call("icap_reload_env")
    set_()
    yield set_
    monkeypatch.undo()
    N.call("icap_reload_env")
    N.call("icap_set_gemm_sms", 0)


# ------------------------------------------------------------------------------------------ data and reference
def dev():
    return torch.device("cuda:0")


def tdt(code):
    return torch.float32 if code == F32 else torch.bfloat16


def itype(code):
    return torch.int32 if code == F32 else torch.int16


def ints(shape, lo, hi, g):
    return torch.randint(lo, hi + 1, shape, device=dev(), generator=g, dtype=torch.int32).float()


def placed(rows, cols, ld, off, dtype, fill):
    """[rows, cols] view with row stride ld inside a fresh buffer, `off` elements past a 256-byte boundary; the rest
    of the buffer keeps `fill` (a tensor: the view's values, or NaN padding)."""
    buf = torch.full((off + rows * ld + 64,), float("nan"), device=dev(), dtype=dtype)
    v = buf[off:off + rows * ld].view(rows, ld)[:, :cols]
    v.copy_(fill)
    return buf, v


def operand(rows, cols, ld, off, code, amp, g):
    vals = ints((rows, cols), -amp, amp, g)
    return placed(rows, cols, ld, off, tdt(code), vals)[1]


def matmul64(A, B, a_k, b_k, rows=1 << 20):
    """fp64 op(A) @ op(B), in row chunks (exact for the integer data: every partial sum is below 2^53)."""
    Bd = (B.t() if b_k else B).double()
    M = A.shape[0] if a_k else A.shape[1]
    out = torch.empty(M, Bd.shape[1], dtype=torch.float64, device=dev())
    for r in range(0, M, rows):
        Ar = A[r:r + rows] if a_k else A[:, r:r + rows].t()
        out[r:r + rows] = Ar.double() @ Bd
    return out


def stats_expected(x, Nn):
    """(largest, second largest, sum exp(x - largest), 0) per row and 128 columns of the stored logits x [M, N]; an
    empty column half reads (-inf, -inf, 0, 0)."""
    M, P = x.shape[0], 2 * ((Nn + 255) // 256)
    out = torch.empty(M, P, 4, dtype=torch.float64, device=dev())
    for s in range(P):
        seg = x[:, s * 128:min(Nn, (s + 1) * 128)].double()
        if seg.shape[1] == 0:
            out[:, s] = torch.tensor([float("-inf"), float("-inf"), 0.0, 0.0], dtype=torch.float64, device=dev())
            continue
        top = seg.topk(min(2, seg.shape[1]), dim=1).values
        out[:, s, 0] = top[:, 0]
        out[:, s, 1] = top[:, 1] if seg.shape[1] > 1 else float("-inf")
        out[:, s, 2] = (seg - top[:, :1]).exp().sum(1)
        out[:, s, 3] = 0.0
    return out


def mismatch(got, exp):
    bad = got.double() != exp.double()
    if not bool(bad.any()):
        return None
    idx = bad.nonzero()[0].tolist()
    return f"{int(bad.sum())} elements differ, first at {idx}: got {got[tuple(idx)].item()}, want {exp[tuple(idx)].item()}"


def run_case(cs, switches, check_kernel=True):
    """Run one case; assert its results (and its kernel, if named).  Returns (demangled GEMM kernel names, C)."""
    switches(cs.env)
    N.call("icap_set_gemm_sms", cs.sms)
    g = torch.Generator(device="cuda").manual_seed(hash((cs.M, cs.N, cs.K, cs.layout, cs.ab)) & 0xFFFFFFFF)
    M, Nn, K = cs.M, cs.N, cs.K
    a_k, b_k = cs.layout
    r8 = (lambda x: (x + 7) // 8 * 8) if cs.ab == BF16 else (lambda x: x)
    a_rows, a_cols = (M, K) if a_k else (K, M)
    b_rows, b_cols = (Nn, K) if b_k else (K, Nn)
    lda = cs.lda or r8(a_cols) + cs.ld_pad
    ldb = cs.ldb or r8(b_cols) + cs.ld_pad
    A = operand(a_rows, a_cols, lda, cs.a_off, cs.ab, cs.amp, g)
    B = operand(b_rows, b_cols, ldb, cs.b_off, cs.ab, cs.amp, g)
    bias = ints((Nn,), -cs.bias_amp, cs.bias_amp, g) if cs.bias else None
    ldc = cs.ldc or (Nn + 7) // 8 * 8 + 8
    esz = 4 if cs.c == F32 else 2
    ref = matmul64(A, B, a_k, b_k)
    if bias is not None:
        ref += bias.double()
    aux = stats = None
    if cs.epi == 1:
        ref.clamp_min_(0)
    elif cs.epi == 2:
        av = ints((M, Nn), -2, 2, g)
        av[(av == 0) & (torch.rand(M, Nn, device=dev(), generator=g) < 0.5)] = -0.0
        ldaux = cs.ldaux or ldc
        aux_buf, aux = placed(M, Nn, ldaux, cs.aux_off, tdt(cs.c), av)
        ref = torch.where(aux.double() > 0, ref, torch.zeros_like(ref))
    # C: the [M, N] block at row stride ldc inside a sentinel-filled buffer with guard rows above and below
    lead = 256 // esz + cs.c_off
    cbuf = torch.empty(lead + (M + 2) * ldc + 64, device=dev(), dtype=tdt(cs.c))
    cbuf.view(itype(cs.c)).fill_(SENTINEL[cs.c])
    C = cbuf[lead:lead + M * ldc].view(M, ldc)[:, :Nn]
    if cs.acc:
        c0 = ints((M, Nn), -1000, 1000, g).to(tdt(cs.c))
        C.copy_(c0)
        v = ref if cs.c == F32 else ref.to(torch.bfloat16).double()
        ref = c0.double() + v
    assert float(ref.abs().max()) < 2 ** 24, "the case leaves the exact fp32 range"
    expected = ref.to(tdt(cs.c))
    epi = cs.epi | (N.EPI_B_STATIC if cs.b_static else 0)
    if cs.epi == 3:
        P = 2 * ((Nn + 255) // 256)
        ldaux = 4 * P + 4
        stats = torch.full((M + 2, ldaux), float("nan"), device=dev())
        stats.view(torch.int32).fill_(SENTINEL[F32])
        aux_ptr = stats.data_ptr()
    else:
        ldaux = aux.stride(0) if aux is not None else 0
        aux_ptr = aux.data_ptr() if aux is not None else None

    def call():
        N.call("icap_gemm", cs.ab, a_k, b_k, M, Nn, K, A.data_ptr(), lda, B.data_ptr(), ldb, C.data_ptr(), ldc, cs.c,
               bias.data_ptr() if bias is not None else None, epi, aux_ptr, ldaux, cs.acc, cs.split_k,
               torch.cuda.current_stream().cuda_stream)
    names = launched_kernels(call)
    gemm_names = [n for n in names if "gemm_" in n]
    assert len(gemm_names) == 1, f"{cs.name}: expected one GEMM kernel, the profiler saw {names}"
    if check_kernel and cs.kernel is not None:
        assert re.search(kernel_regex(cs.kernel), gemm_names[0]), \
            f"{cs.name}: expected {kernel_regex(cs.kernel)}, the profiler saw {gemm_names[0]}"
    err = mismatch(C, expected)
    assert err is None, f"{cs.name} ({gemm_names[0]}): {err}"
    # guard band: every element outside the block keeps its sentinel bits
    bits = cbuf.view(itype(cs.c)).clone()
    bits[lead:lead + M * ldc].view(M, ldc)[:, :Nn] = SENTINEL[cs.c]
    nbad = int((bits != SENTINEL[cs.c]).sum())
    assert nbad == 0, f"{cs.name}: {nbad} elements outside the [M, N] block of C were written"
    if stats is not None:
        st = stats[:M, :4 * P].view(M, P, 4)
        es = stats_expected(C, Nn)
        for j, what in ((0, "largest"), (1, "second largest"), (3, "pad")):
            e = mismatch(st[:, :, j], es[:, :, j])
            assert e is None, f"{cs.name}: row statistics, {what}: {e}"
        assert torch.allclose(st[:, :, 2].double(), es[:, :, 2], rtol=1e-4, atol=0), f"{cs.name}: row statistics, exp-sum"
        sbits = stats.view(torch.int32).clone()
        sbits[:M, :4 * P] = SENTINEL[F32]
        assert bool((sbits == SENTINEL[F32]).all()), f"{cs.name}: statistics written outside [M, 8 ceil(N / 256)]"
    return gemm_names, C.clone()


# ------------------------------------------------------------------------------------------ tests
def test_case_table_names_every_kernel():
    """CPU: the cases name all 25 kernels icap_gemm can launch, and each name pattern picks exactly one of them."""
    named = {c.kernel for c in CASES}
    assert len(ALL_KERNELS) == 25 and len(set(ALL_KERNELS)) == 25
    missing = [k for k in ALL_KERNELS if k not in named]
    assert not missing, f"no case runs {missing}"
    b = {0: "(bool)0", 1: "(bool)1"}
    names = []
    for k in ALL_KERNELS:       # demangled as cu++filt prints the library's symbols
        if k[0] == "small":
            names.append(f"void <unnamed>::gemm_small_kernel<(int){k[1]}>(CUtensorMap_st, CUtensorMap_st, CUtensorMap_st, "
                         "<unnamed>::SmallArgs)")
        elif k[0] == "f32":
            names.append(f"void <unnamed>::gemm_f32_kernel<{b[k[1]]}, {b[k[2]]}>(int, int, int, const float *, long)")
        else:
            cfg, ak, bk, c, st = ("256", 1, 1, BF16, 1) if k == STATS else (*k[1:], 0)
            bnv, two = (128, 0) if cfg == "128" else (256, int(cfg == "pair"))
            t = "float" if c == F32 else "__nv_bfloat16"
            names.append(f"void <unnamed>::gemm_tc_kernel<(int){bnv}, {b[two]}, {b[ak]}, {b[bk]}, {t}, {b[st]}>"
                         "(CUtensorMap_st, CUtensorMap_st, CUtensorMap_st, <unnamed>::GemmArgs)")
    for k, name in zip(ALL_KERNELS, names):
        assert kernel_of(name) == k, (k, name)
        plain = name.replace("(int)", "").replace("(bool)0", "false").replace("(bool)1", "true")
        assert kernel_of(plain) == k, (k, plain)


@gpu
@pytest.mark.parametrize("cs", CASES, ids=[c.name for c in CASES])
def test_gemm_path(cs, switches):
    run_case(cs, switches)


@gpu
@pytest.mark.parametrize("cfg", TC_CFGS)
def test_bf16_accumulate_same_bits_at_any_alignment(cfg, switches):
    """C += into bf16: the TMA reduce-add (aligned C), the vector direct stores and the scalar direct stores (C 2 bytes
    off) leave identical bits."""
    outs = []
    for c_off, ldc, extra in ((0, 400, {}), (0, 400, {"ICAP_GEMM_DIRECT_EPILOGUE": "1"}), (1, 400, {}), (0, 393, {})):
        cs = Case(f"acc-align-{cfg}", tc(cfg, (1, 1), BF16), 1000, 392, 1032, bias=True, acc=1, c_off=c_off, ldc=ldc,
                  env=bn(cfg, **extra))
        outs.append(run_case(cs, switches)[1].view(torch.int16))
    for o in outs[1:]:
        assert torch.equal(o, outs[0])


# ---------------------------------------------------------------------- GEMMs of the product's steps, replayed
def _signature(args):
    (ab, a_k, b_k, M, Nn, K, A, lda, B, ldb, C, ldc, c, bias, epi, aux, ldaux, acc, split_k) = args
    esz_ab = 4 if ab == F32 else 2
    esz_c = 4 if c == F32 else 2
    return (ab, a_k, b_k, M, Nn, K, lda, ldb, ldc, c, bias is not None, epi, ldaux if aux else 0, acc, split_k,
            (A % 256) // esz_ab, (B % 256) // esz_ab, (C % 256) // esz_c, ((aux or 0) % 256) // esz_c)


def _case_of(sig, i):
    (ab, a_k, b_k, M, Nn, K, lda, ldb, ldc, c, has_bias, epi, ldaux, acc, split_k, ao, bo, co, xo) = sig
    e = epi & 15
    return Case(f"step-{i}", None, M, Nn, K, ab=ab, layout=(a_k, b_k), c=c, bias=has_bias, epi=e, acc=acc,
                split_k=split_k, b_static=bool(epi & 16), lda=lda, ldb=ldb, ldc=ldc, ldaux=ldaux if e == 2 else 0,
                a_off=ao, b_off=bo, c_off=co, aux_off=xo, amp=1 if e == 3 else 8, bias_amp=2 if e == 3 else 64)


def _record(kind):
    from oracle import caption_oracle as O
    kw = dict(num_vocab=10000, max_length=22, encode_dim_positions=84, encode_dim_features=2048, output_name="x",
              dropout=0.2)                                   # model A
    torch.manual_seed(0)
    m = pkg.Transformer(device=dev(), **kw).to(dev())
    m.set_precision("fp32" if kind == "train_fp32" else "bf16")
    eng = m._engine()
    batch = {"train_bf16": 256, "train_fp32": 8, "decode_beam5": 512}[kind]
    f, p, c = O.synthetic_batch(batch, 36, 2048, 84, 22, 10000, seed=5)
    f, p, c = f.to(dev()), p.to(dev()), c.to(dev())
    if kind == "decode_beam5":
        m.eval()
        log = eng.record_gemms(lambda: eng.decode(f, p, beam_size=5))
    else:
        m.train()
        log = eng.record_gemms(lambda: eng.train_step(f, p, c, lr=5e-4))
    torch.cuda.synchronize()
    del m, eng
    return log


@gpu
@pytest.mark.parametrize("kind", ["train_bf16", "train_fp32", "decode_beam5"])
def test_product_step_gemms(kind, switches):
    """Every distinct GEMM of a model-A step (argument signature: shapes, leading dimensions, epilogue, pointer
    alignment mod 256 bytes), replayed on integer data and compared exactly.  The kernel each one runs is printed;
    asserted are only the documented rules: row statistics run on the 128x256 build, the pair is never chosen for
    M <= 128, and the M = 2560 projections of the beam-5 decode (512 images) run the small-footprint kernel."""
    sigs = list(dict.fromkeys(_signature(a) for a in _record(kind)))
    torch.cuda.empty_cache()
    rows = []
    for i, sig in enumerate(sigs):
        cs = _case_of(sig, i)
        name = run_case(cs, switches)[0][0]
        k = kernel_of(name)
        rows.append((cs, k))
        if cs.epi == 3:
            assert k == STATS, (cs, name)
        if cs.M <= 128:
            assert k is not None and k[1] != "pair", (cs, name)
        eligible = (cs.layout == (1, 1) and cs.c == BF16 and cs.epi in (0, 1) and not cs.acc and cs.c_off % 8 == 0
                    and cs.ldc % 8 == 0)
        if kind == "decode_beam5" and cs.M == 2560 and eligible:
            assert k is not None and k[0] == "small", (cs, name)
    print(f"\n{kind}: {len(sigs)} distinct GEMMs")
    print("   M      N      K  layout  C     epi  acc  split  kernel")
    for cs, k in rows:
        print(f"{cs.M:6d} {cs.N:6d} {cs.K:6d}  {lay_name(cs.layout):6s}  {c_name(cs.c):4s}  {cs.epi:3d}  {cs.acc:3d}  "
              f"{cs.split_k:5d}  {k}")
    if kind == "decode_beam5":
        assert any(cs.M == 2560 for cs, _ in rows)
