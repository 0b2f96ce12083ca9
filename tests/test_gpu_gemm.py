"""The tcgen05 3xTF32 GEMM (csrc/gemm_tc.cu), every dispatch path of re2e_gemm_tf32x3, against fp64.

Each case is pinned to one kernel.  ``plan`` restates the host dispatch of re2e_gemm_tf32x3 (tile width BN, the split-K
slice search, per-tile or persistent kernel, epilogue); a case states the path it was built for, the test asserts that
``plan`` agrees, and that torch.profiler saw exactly that kernel with those template arguments -- and the zero-fill of C
when the case splits K without accumulating.  A change in the dispatch therefore breaks a test instead of quietly moving
a case onto another path.

Three checks per case:
  (a) exact: A, B, bias (and C for ``accumulate``) are integers in [-4, 4].  TF32 holds them exactly (lo = 0) and every
      partial sum is an integer below 2^24 (K <= 6400), so C must equal the fp64 product bit for bit.
  (b) exact split terms (K <= 960): operands sign(i) (|i| + t 2^-12), i in {+-1, +-2}, t in {0, 1}.  Truncated or rounded
      to TF32 such a value gives hi = i and lo = +-t 2^-12 exactly (an offset towards zero would not: 1 - 2^-12
      truncates to 1 - 2^-11).  Every partial sum of hi.hi + lo.hi + hi.lo then lies on the 2^-12 grid below 2^12, which
      fp32 holds, so C must equal the fp64 sum of those three terms (no lo.lo) bit for bit.  This is the only check that
      sees the lo copies the converter warps write.
  (c) accuracy on random data: max-norm error < 1e-5 (2e-5 with ``accumulate``) and, element by element,
      |C - ref| <= TAU (|A||B|^T + |bias| + |C0|).  Non-split paths must also be bit-identical over two calls.
Every call has NaN in the operands' padding (pitch columns and two rows past the matrix) and NaN guards around C (pitch
columns, rows before and after); no NaN may reach C and every guard must stay NaN.
"""
import collections

import pytest
import torch
import torch.nn.functional as F

from helpers import rel_err
from robust_e2e_gan_b200 import _lib
from robust_e2e_gan_b200.linear import linear
from test_gpu_frontend_paths import _template_args

gpu = pytest.mark.gpu
DEV = "cuda:0"
E_ARG, E_UNSUPPORTED = -1, -2
B200_SMS = 148
TILE, PERSIST = "gemm_tf32x3_kernel", "gemm_tf32x3_persist_kernel"
TAU = 1e-5
LAYOUTS = ((0, 0), (0, 1), (1, 0), (1, 1))


def _cdiv(a, b):
    return -(-a // b)


def _pad4(n):
    return _cdiv(n, 4) * 4


# ---- the host dispatch of re2e_gemm_tf32x3, restated ----------------------------------------------------------------
Plan = collections.namedtuple("Plan", "kernel targs splits epilogue")


def plan(M, N, K, a_mn, b_mn, ldc, c_off, sms):
    """Kernel, template arguments <A_MN, B_MN, BN, STAGES>, number of k slices and epilogue that re2e_gemm_tf32x3 picks
    (C at ``c_off`` floats past a 16 B boundary).  Epilogues: per-tile 'tma' (TMA store, or TMA reduce-add when split or
    accumulating) / 'scalar'; persistent 'vec' (16 B stores / red.global.add.v4) / 'scalar'."""
    BN = 256 if (N % 256 == 0 or N > 1024) else 160
    nkb = _cdiv(K, 32)
    kb_per = nkb
    if nkb > 24:
        tiles = _cdiv(M, 128) * _cdiv(N, BN)
        best = None
        for kp in range(12, 21):
            cost = _cdiv(tiles * _cdiv(nkb, kp), sms) * (kp + 4)
            if best is None or cost < best:
                best, kb_per = cost, kp
    splits = _cdiv(nkb, kb_per)
    items = _cdiv(M, 128) * _cdiv(N, BN) * splits
    c16 = ldc % 4 == 0 and c_off == 0
    targs = ("true" if a_mn else "false", "true" if b_mn else "false", str(BN), "2" if BN == 256 else "3")
    if items > sms:
        return Plan(PERSIST, targs, splits, "vec" if c16 else "scalar")
    return Plan(TILE, targs, splits, "tma" if (c16 and N >= 4) else "scalar")


def describe(p):
    """'tile 160 whole tma', 'persist 256 split vec', ..."""
    return "%s %s %s %s" % ("persist" if p.kernel == PERSIST else "tile", p.targs[2], "split" if p.splits > 1 else "whole",
                            p.epilogue)


class Case(object):
    """One call: C[M,N] (+)= Aop Bop^T (+ bias).  lda / ldb default to the padded pitch + 4 (so that every operand has
    NaN pitch columns); ldc defaults to the padded pitch; C sits ``c_off`` floats past a 16 B boundary."""

    def __init__(self, M, N, K, a_mn=0, b_mn=0, path=None, ldc=None, lda=None, ldb=None, c_off=0, bias=True,
                 accumulate=False):
        self.M, self.N, self.K, self.a_mn, self.b_mn, self.path = M, N, K, a_mn, b_mn, path
        self.ldc = _pad4(N) if ldc is None else ldc
        self.lda = _pad4(M if a_mn else K) + 4 if lda is None else lda
        self.ldb = _pad4(N if b_mn else K) + 4 if ldb is None else ldb
        self.c_off, self.bias, self.accumulate = c_off, bias, accumulate

    def plan(self, sms):
        return plan(self.M, self.N, self.K, self.a_mn, self.b_mn, self.ldc, self.c_off, sms)

    def __repr__(self):
        return "%dx%dx%d a%d b%d ldc%d off%d%s%s" % (self.M, self.N, self.K, self.a_mn, self.b_mn, self.ldc, self.c_off,
                                                 "" if self.bias else " nobias", " acc" if self.accumulate else "")


def P(name, M, N, K, ab, path, **kw):
    return pytest.param(Case(M, N, K, ab[0], ab[1], path, **kw), id=name)


# The shapes of this file's first test, with the unaligned pitch ldc = N + 3 (4236 for N = 4233 is TMA-addressable).
FIRST_SHAPES = [(128, 160, 32), (300, 200, 96), (6400, 320, 320), (777, 4233, 320), (1000, 320, 4236)]


def first_cases(M, N, K, a_mn, b_mn):
    """The first test's two calls: with bias, then accumulating without."""
    return [Case(M, N, K, a_mn, b_mn, ldc=N + 3), Case(M, N, K, a_mn, b_mn, ldc=N + 3, bias=False, accumulate=True)]

CASES = [
    # ---- per-tile kernel
    *[P("tile-tma-store-%d%d" % ab, 6400, 320, 320, ab, "tile 160 whole tma") for ab in LAYOUTS],
    P("tile-bn256-n512", 300, 512, 96, (0, 0), "tile 256 whole tma"),
    P("tile-bn256-n512-mn", 300, 512, 96, (1, 1), "tile 256 whole tma"),
    P("tile-split-tma-reduce", 320, 320, 6400, (1, 1), "tile 160 split tma"),
    P("tile-split-tma-reduce-k4236", 1000, 320, 4236, (0, 0), "tile 160 split tma"),
    P("tile-k768-whole", 256, 160, 768, (0, 0), "tile 160 whole tma"),
    P("tile-k769-split", 256, 160, 769, (0, 1), "tile 160 split tma"),
    P("tile-k4233-split", 256, 160, 4233, (1, 0), "tile 160 split tma"),
    P("tile-unaligned-c", 640, 320, 320, (0, 0), "tile 160 whole scalar", c_off=1),
    P("tile-split-unaligned-c", 320, 320, 6400, (0, 0), "tile 160 split scalar", c_off=1),
    # ---- persistent kernel
    P("persist-149-items", 19072, 160, 64, (0, 0), "persist 160 whole vec"),
    P("persist-150-items", 19073, 160, 64, (1, 0), "persist 160 whole vec"),
    *[P("persist-bn256-vec-%d%d" % ab, 6400, 4233, 320, ab, "persist 256 whole vec") for ab in LAYOUTS],
    *[P("persist-bn160-vec-%d%d" % ab, 6400, 480, 320, ab, "persist 160 whole vec") for ab in LAYOUTS],
    P("persist-scalar-ldc4237", 6400, 4233, 320, (0, 0), "persist 256 whole scalar", ldc=4237),
    P("persist-scalar-unaligned-c", 6400, 4233, 320, (0, 1), "persist 256 whole scalar", c_off=1),
    P("persist-split-bn256-00", 6400, 512, 1024, (0, 0), "persist 256 split vec"),
    P("persist-split-bn256-10", 6400, 512, 1024, (1, 0), "persist 256 split vec"),
    P("persist-split-bn160-ctc-dx", 6400, 320, 4233, (0, 1), "persist 160 split vec"),
    P("persist-split-bn160-ctc-dw", 4233, 320, 6400, (1, 1), "persist 160 split vec"),
    P("persist-split-scalar", 6400, 320, 4233, (0, 0), "persist 160 split scalar", ldc=323),
    # ---- edges
    P("m1", 1, 4233, 320, (0, 0), "tile 256 whole tma"),
    P("m127", 127, 320, 320, (1, 0), "tile 160 whole tma"),
    P("m129", 129, 320, 320, (0, 1), "tile 160 whole tma"),
    P("m4233", 4233, 160, 320, (1, 1), "tile 160 whole tma"),
    P("n1", 129, 1, 40, (0, 0), "tile 160 whole scalar", ldc=4),
    P("n2", 129, 2, 40, (1, 1), "tile 160 whole scalar", ldc=4),
    P("n3", 129, 3, 40, (0, 1), "tile 160 whole scalar", ldc=4),
    P("n163-tail-only-block", 640, 163, 320, (0, 0), "tile 160 whole tma", ldc=164),
    P("n163-tail-split", 640, 163, 1024, (1, 0), "tile 160 split tma", ldc=164),
    P("k300", 640, 320, 300, (0, 0), "tile 160 whole tma"),
    P("acc-bias-tile", 6400, 320, 320, (0, 1), "tile 160 whole tma", accumulate=True),
    P("acc-bias-tile-scalar", 640, 163, 320, (1, 0), "tile 160 whole scalar", ldc=167, accumulate=True),
    P("acc-bias-persist", 6400, 4233, 320, (0, 0), "persist 256 whole vec", accumulate=True),
    P("acc-bias-persist-scalar", 6400, 4233, 320, (1, 1), "persist 256 whole scalar", ldc=4237, accumulate=True),
    P("acc-split-tile", 320, 320, 6400, (1, 1), "tile 160 split tma", accumulate=True),
    P("acc-split-persist", 6400, 320, 4233, (0, 1), "persist 160 split vec", accumulate=True, bias=False),
    P("no-bias-tile", 640, 163, 320, (0, 0), "tile 160 whole tma", ldc=164, bias=False),
    P("no-bias-persist", 6400, 480, 320, (1, 1), "persist 160 whole vec", bias=False),
]


# ---- operands, C with guards, the call ------------------------------------------------------------------------------
def _store(X, mn, ld):
    """X (rows, K) in the kernel's layout, [rows][ld] (K-major) or [K][ld] (MN-major), on the GPU.  Every element
    outside the matrix -- the pitch columns and two rows past it -- is NaN."""
    src = X.t() if mn else X
    S = torch.full((src.shape[0] + 2, ld), float("nan"), device=DEV)
    S[:src.shape[0], :src.shape[1]] = src.to(DEV)
    return S


class CBuf(object):
    """C (M, N) with pitch ldc inside a NaN-filled buffer: four pitch rows before it, two after, the pitch columns."""

    def __init__(self, case, C0=None):
        self.case = case
        self.start = 4 * case.ldc + case.c_off
        self.buf = torch.full((self.start + (case.M + 2) * case.ldc,), float("nan"), device=DEV)
        self.C = self.buf[self.start:self.start + case.M * case.ldc].view(case.M, case.ldc)[:, :case.N]
        if C0 is not None:
            self.C.copy_(C0)
        self.ptr = self.C.data_ptr()

    def guards_intact(self):
        g = self.buf.clone()
        g[self.start:self.start + self.case.M * self.case.ldc].view(self.case.M, self.case.ldc)[:, :self.case.N] = \
            float("nan")
        return bool(torch.isnan(g).all())


def _gemm(case, As, Bs, cptr, bias):
    return _lib.lib().re2e_gemm_tf32x3(As.data_ptr(), case.lda, case.a_mn, Bs.data_ptr(), case.ldb, case.b_mn, cptr,
                                       case.ldc, _lib.ptr(bias), case.M, case.N, case.K, int(case.accumulate),
                                       _lib.stream_ptr())


def _profiled(fn):
    """fn() under torch.profiler: (its result, {(kernel, template args)} of the GEMM kernels that ran, whether a memset
    ran -- the runtime call or its device activity)."""
    torch.cuda.synchronize()
    with torch.profiler.profile(activities=[torch.profiler.ProfilerActivity.CUDA]) as prof:
        rc = fn()
        torch.cuda.synchronize()
    names = []
    for e in prof.events():
        names.append(e.name)
        names.extend(k.name for k in getattr(e, "kernels", []))
    ran = {(f, tuple(_template_args(n, f))) for n in names for f in (TILE, PERSIST) if f in n}
    return rc, ran, any("emset" in n for n in names)


def _run(case, A, B, bias, C0, profile=False):
    """One call on fresh guarded buffers; returns C (and, when profiled, what ran)."""
    As, Bs = _store(A, case.a_mn, case.lda), _store(B, case.b_mn, case.ldb)
    bias_d = bias.to(DEV) if bias is not None else None
    cb = CBuf(case, C0.to(DEV) if C0 is not None else None)
    n0 = _lib.launch_count()
    if profile:
        rc, ran, memset = _profiled(lambda: _gemm(case, As, Bs, cb.ptr, bias_d))
    else:
        rc, ran, memset = _gemm(case, As, Bs, cb.ptr, bias_d), None, None
        torch.cuda.synchronize()
    assert rc == 0, (case, rc)
    assert _lib.launch_count() == n0 + 1, case
    assert cb.guards_intact(), "%s: a write outside C" % case
    assert not torch.isnan(cb.C).any(), "%s: NaN in C (a read outside an operand)" % case
    return cb.C, ran, memset


# ---- data ---------------------------------------------------------------------------------------------------------------
def _seed(case, kind):
    return (case.M * 1000003 + case.N * 10007 + case.K * 101 + 2 * case.bias + case.accumulate) * 4 + "abc".index(kind)


def integer_data(case):
    """(a): integers in [-4, 4]."""
    g = torch.Generator().manual_seed(_seed(case, "a"))
    r = lambda *s: torch.randint(-4, 5, s, generator=g).float()
    return (r(case.M, case.K), r(case.N, case.K), r(case.N) if case.bias else None,
            r(case.M, case.N) if case.accumulate else None)


def split_term_values(shape, g):
    """(b): (x, hi, lo) with x = sign(i) (|i| + t 2^-12), i in {-2, -1, 1, 2}, t in {0, 1}: hi = i, lo = x - i."""
    i = torch.tensor([-2.0, -1.0, 1.0, 2.0])[torch.randint(0, 4, shape, generator=g)]
    lo = torch.sign(i) * torch.randint(0, 2, shape, generator=g).float() * 2.0 ** -12
    return i + lo, i, lo


def split_term_data(case):
    g = torch.Generator().manual_seed(_seed(case, "b"))
    A = split_term_values((case.M, case.K), g)
    B = split_term_values((case.N, case.K), g)
    bias = split_term_values((case.N,), g)[0] if case.bias else None
    C0 = torch.randint(-4, 5, (case.M, case.N), generator=g).float() if case.accumulate else None
    return A, B, bias, C0


def random_data(case):
    """(c): standard normal A, B, bias and C0; the same for every layout of a shape."""
    g = torch.Generator().manual_seed(_seed(case, "c"))
    return (torch.randn(case.M, case.K, generator=g), torch.randn(case.N, case.K, generator=g),
            torch.randn(case.N, generator=g) if case.bias else None,
            torch.randn(case.M, case.N, generator=g) if case.accumulate else None)


def _d(x):
    return None if x is None else x.to(DEV, torch.float64)


def _affine(A, B, bias, C0):
    """A B^T + bias + C0 in fp64 on the GPU (None terms left out)."""
    out = _d(A) @ _d(B).t()
    if bias is not None:
        out += _d(bias)
    if C0 is not None:
        out += _d(C0)
    return out


def _assert_exact(case, got, ref, what):
    diff = got.double() != ref
    if diff.any():
        idx = diff.nonzero()[0].tolist()
        raise AssertionError("%s: %s: %d of %d elements differ, first at %s: %r != %r" % (
            case, what, int(diff.sum()), diff.numel(), idx, float(got[tuple(idx)]), float(ref[tuple(idx)])))


def check_case(case, checks="abc"):
    sms = torch.cuda.get_device_properties(0).multi_processor_count
    p = case.plan(sms)
    if case.path is not None:
        assert describe(p) == case.path, "%s: dispatch restated as '%s', case built for '%s'" % (case, describe(p),
                                                                                                 case.path)
    # (a) exact integers, run under the profiler: the kernel the plan names, and the zero-fill exactly when it is needed
    A, B, bias, C0 = integer_data(case)
    C, ran, memset = _run(case, A, B, bias, C0, profile=True)
    assert ran == {(p.kernel, p.targs)}, "%s: expected %s<%s>, ran %s" % (case, p.kernel, ", ".join(p.targs), ran)
    assert memset == (p.splits > 1 and not case.accumulate), "%s: split-K zero-fill %s" % (case, memset)
    _assert_exact(case, C, _affine(A, B, bias, C0), "(a) integers")
    # (b) exact hi.hi + lo.hi + hi.lo
    if "b" in checks and case.K <= 960:
        (A, Ahi, Alo), (B, Bhi, Blo), bias, C0 = split_term_data(case)
        C, _, _ = _run(case, A, B, bias, C0)
        ref = _affine(Ahi, Bhi, bias, C0) + _d(Ahi) @ _d(Blo).t() + _d(Alo) @ _d(Bhi).t()
        _assert_exact(case, C, ref, "(b) split terms")
    # (c) accuracy on random data; determinism of the non-split paths
    if "c" in checks:
        A, B, bias, C0 = random_data(case)
        C, _, _ = _run(case, A, B, bias, C0)
        ref = _affine(A, B, bias, C0)
        scale = _affine(A.abs(), B.abs(), None if bias is None else bias.abs(), None if C0 is None else C0.abs())
        err = (C.double() - ref).abs()
        rel = float(err.max() / ref.abs().max())
        ratio = float((err / scale).max())
        print("gemm accuracy %-40s rel_err %.2e  element ratio %.2e" % (case, rel, ratio))
        assert rel < (2e-5 if case.accumulate else 1e-5), (case, rel)
        assert ratio < TAU, (case, ratio)
        if p.splits == 1:
            assert torch.equal(_run(case, A, B, bias, C0)[0], C), "%s: not deterministic" % case


# ---- the cases ------------------------------------------------------------------------------------------------------------
@gpu
@pytest.mark.parametrize("M,N,K", FIRST_SHAPES)
@pytest.mark.parametrize("a_mn,b_mn", LAYOUTS)
def test_gemm_matches_fp64(M, N, K, a_mn, b_mn):
    for case in first_cases(M, N, K, a_mn, b_mn):
        check_case(case)


@gpu
@pytest.mark.parametrize("case", CASES)
def test_gemm_path_matches_fp64(case):
    check_case(case)


def _table_cases():
    return [prm.values[0] for prm in CASES] + [c for M, N, K in FIRST_SHAPES for a_mn, b_mn in LAYOUTS
                                               for c in first_cases(M, N, K, a_mn, b_mn)]


def test_case_table_covers_every_gemm_path():
    """At the B200's 148 SMs the cases reach all 16 instantiations (two kernels x four majors x two BN), split and
    whole K on both kernels, and every epilogue; each case's stated path is the restated dispatch's."""
    plans = []
    for case in _table_cases():
        p = case.plan(B200_SMS)
        assert case.path is None or describe(p) == case.path, (case, describe(p))
        plans.append((p, case.accumulate))
    insts = {(p.kernel,) + p.targs for p, _ in plans}
    assert insts == {(k, a, b, bn, st) for k in (TILE, PERSIST) for a in ("false", "true") for b in ("false", "true")
                     for bn, st in (("160", "3"), ("256", "2"))}
    kinds = {(p.kernel, p.splits > 1, p.epilogue, acc) for p, acc in plans}
    for k, epis in ((TILE, ("tma", "scalar")), (PERSIST, ("vec", "scalar"))):
        for split in (False, True):
            for e in epis:
                assert (k, split, e, False) in kinds, (k, split, e)
            assert (k, split, epis[0], True) in kinds, (k, split, "accumulate")


def test_split_term_values_are_what_the_kernel_splits():
    """The operands of check (b) split, as the kernel splits them (tcgen05 reads the truncated TF32, the converters
    write lo = cvt.rna.tf32(x - hi)), into exactly hi = i and lo = x - i."""
    x, i, lo = split_term_values((4096,), torch.Generator().manual_seed(0))
    hi_k, lo_k = tf32_split(x)
    assert torch.equal(hi_k, i) and torch.equal(lo_k, lo)
    assert set(lo.unique().tolist()) == {-2.0 ** -12, 0.0, 2.0 ** -12}


# ---- the bounds of check (c) reject weaker GEMMs -----------------------------------------------------------------------
def tf32_split(x):
    """(hi, lo) of fp32 x as the kernel splits it: hi = x truncated to TF32 (what the tensor core reads of an fp32
    operand), lo = x - hi rounded to TF32, nearest with ties away from zero."""
    x = x.float().contiguous()
    hi = (x.view(torch.int32) & -8192).view(torch.float32)
    lo = (((x - hi).view(torch.int32) + 4096) & -8192).view(torch.float32)
    return hi, lo


def test_accuracy_bounds_reject_weaker_gemms():
    """On the data of every accuracy case, two weaker products emulated in fp64 break both bounds of check (c): the
    3xTF32 product without its hi.lo term, and a single TF32 pass.  (The emulation leaves out the truncating TMEM
    accumulator; the kernel's own error against the bounds is printed by the GPU cases.)"""
    seen = set()
    for case in _table_cases():
        key = (case.M, case.N, case.K, case.bias, case.accumulate)
        if key in seen:
            continue
        seen.add(key)
        A, B, bias, C0 = random_data(case)
        (Ah, Al), (Bh, Bl) = tf32_split(A), tf32_split(B)
        extra = (0.0 if bias is None else bias.double()) + (0.0 if C0 is None else C0.double())
        ref = A.double() @ B.double().t() + extra
        scale = A.double().abs() @ B.double().abs().t() + (0.0 if bias is None else bias.double().abs()) + \
            (0.0 if C0 is None else C0.double().abs())
        hh = Ah.double() @ Bh.double().t() + extra
        for name, emu in (("no hi.lo", hh + Al.double() @ Bh.double().t()), ("1xTF32", hh)):
            err = (emu - ref).abs()
            rel = float(err.max() / ref.abs().max())
            ratio = float((err / scale).max())
            assert rel > (2e-5 if case.accumulate else 1e-5), (case, name, rel)
            assert ratio > TAU, (case, name, ratio)


# ---- the products of the benchmarked step, replayed ---------------------------------------------------------------------
@pytest.fixture(scope="module")
def bench_products():
    """Every distinct re2e_gemm_tf32x3 call of one eager HotPath.step at DEFAULT_CFG and one Decoder.forward + backward
    on the decoder_forward_bench workload, as Cases with the recorded pitches and C alignment."""
    from robust_e2e_gan_b200.hotpath import DEFAULT_CFG, HotPath, make_batch
    from test_gpu_decoder import training_case
    L = _lib.lib()
    real = L.re2e_gemm_tf32x3
    calls = []

    def record(A, lda, a_mn, B, ldb, b_mn, C, ldc, bias, M, N, K, acc, stream):
        calls.append((M, N, K, a_mn, b_mn, lda, ldb, ldc, (C % 16) // 4, bias is not None, bool(acc)))
        return real(A, lda, a_mn, B, ldb, b_mn, C, ldc, bias, M, N, K, acc, stream)

    with pytest.MonkeyPatch.context() as mp:
        mp.setattr(L, "re2e_gemm_tf32x3", record)
        cfg = dict(DEFAULT_CFG)
        HotPath(cfg, seed=4000).to(DEV).step(make_batch(cfg, seed=4001).to(DEV))
        dec, _, hpad, hlen, ys, _, _ = training_case("bench")
        loss, _ = dec(hpad.to(DEV).requires_grad_(True), hlen, [y.to(DEV) for y in ys], 0.0)
        loss.backward()
        torch.cuda.synchronize()
    return [Case(M, N, K, a, b, ldc=ldc, lda=lda, ldb=ldb, c_off=off, bias=bias, accumulate=acc)
            for M, N, K, a, b, lda, ldb, ldc, off, bias, acc in sorted(set(calls))]


@gpu
def test_bench_products_match_fp64(bench_products):
    """Checks (a) and (c) on every product of the benchmarked step, at its recorded shape, pitches and flags."""
    ctc_lo = {(6400, 4233, 320, 0, 0), (6400, 320, 4233, 0, 1), (4233, 320, 6400, 1, 1)}   # fwd, dX, dW
    sms = torch.cuda.get_device_properties(0).multi_processor_count
    got = {(c.M, c.N, c.K, c.a_mn, c.b_mn) for c in bench_products if c.plan(sms).kernel == PERSIST}
    assert ctc_lo <= got, sorted(got)
    for case in bench_products:
        check_case(case, checks="ac")


# ---- argument errors --------------------------------------------------------------------------------------------------------
@gpu
def test_gemm_rejects_bad_arguments_without_launching():
    M, N, K = 200, 160, 64
    A = torch.randn(M + 8, K + 8, device=DEV)       # room for every pitch / major below
    B = torch.randn(N + 8, K + 8, device=DEV)
    Cb = torch.full((M, N + 4), 7.0, device=DEV)
    L = _lib.lib()
    good = dict(A=A.data_ptr(), lda=K + 8, a_mn=0, B=B.data_ptr(), ldb=K + 8, b_mn=0, C=Cb.data_ptr(), ldc=N + 4,
                bias=None, M=M, N=N, K=K, acc=0)

    def call(**kw):
        a = dict(good, **kw)
        return L.re2e_gemm_tf32x3(a["A"], a["lda"], a["a_mn"], a["B"], a["ldb"], a["b_mn"], a["C"], a["ldc"], a["bias"],
                                  a["M"], a["N"], a["K"], a["acc"], _lib.stream_ptr())

    bad = [dict(lda=K + 2), dict(ldb=K + 6), dict(A=A.data_ptr() + 4), dict(B=B.data_ptr() + 8),
           dict(lda=K - 4), dict(ldb=K - 4), dict(a_mn=1, lda=M - 4), dict(b_mn=1, ldb=N - 4), dict(ldc=N - 1),
           dict(M=0), dict(N=0), dict(K=0), dict(M=-1), dict(N=-128), dict(K=-32), dict(A=None), dict(C=None)]
    for kw in bad:
        n0 = _lib.launch_count()
        assert call(**kw) == E_ARG, kw
        torch.cuda.synchronize()
        assert _lib.launch_count() == n0, kw
        assert bool((Cb == 7.0).all()), kw
    n0 = _lib.launch_count()
    assert call() == 0
    torch.cuda.synchronize()
    assert _lib.launch_count() == n0 + 1
    assert not bool((Cb[:, :N] == 7.0).any()) and bool((Cb[:, N:] == 7.0).all())


# ---- the autograd wrapper linear.linear ------------------------------------------------------------------------------------
@gpu
@pytest.mark.parametrize("lead,K,N,has_bias,grad", [
    pytest.param((300,), 320, 320, True, "rows", id="2d"),
    pytest.param((4, 75), 320, 200, False, "rows", id="3d-no-bias"),
    pytest.param((2, 333), 320, 4233, True, "rows", id="3d-n4233"),
    pytest.param((300,), 320, 4233, True, "transposed", id="2d-n4233-transposed-grad"),
    pytest.param((4, 75), 320, 320, True, "transposed", id="3d-transposed-grad"),
])
def test_linear_matches_fp64(lead, K, N, has_bias, grad):
    g = torch.Generator().manual_seed(N + K + len(lead))
    x = torch.randn(*lead, K, generator=g).to(DEV).requires_grad_(True)
    w = torch.randn(N, K, generator=g).to(DEV).requires_grad_(True)
    b = torch.randn(N, generator=g).to(DEV).requires_grad_(True) if has_bias else None
    if grad == "rows":
        gy = torch.randn(*lead, N, generator=g).to(DEV)
    else:   # a gradient whose last dimension is not the contiguous one: the wrapper copies it into rows
        gy = torch.randn(N, *lead, generator=g).to(DEV).permute(*range(1, len(lead) + 1), 0)
    y = linear(x, w, b)
    assert y.shape == (*lead, N)
    if N % 4:      # the output is the row-padded view of a (M, pad4(N)) buffer
        ld, strides = _pad4(N), []
        for n in reversed(lead):
            strides.insert(0, ld)
            ld *= n
        assert y.stride() == (*strides, 1)
    y.backward(gy)
    x64 = x.detach().double().requires_grad_(True)
    w64 = w.detach().double().requires_grad_(True)
    b64 = b.detach().double().requires_grad_(True) if has_bias else None
    y64 = F.linear(x64, w64, b64)
    y64.backward(gy.double())
    assert rel_err(y, y64) < 1e-5
    assert rel_err(x.grad, x64.grad) < 1e-5
    assert rel_err(w.grad, w64.grad) < 1e-5
    if has_bias:
        assert rel_err(b.grad, b64.grad) < 1e-5


@gpu
@pytest.mark.parametrize("needs", ["x", "weight"])
def test_linear_skips_the_unneeded_gradient_product(needs):
    g = torch.Generator().manual_seed(5)
    x = torch.randn(300, 320, generator=g).to(DEV).requires_grad_(needs == "x")
    w = torch.randn(200, 320, generator=g).to(DEV).requires_grad_(needs == "weight")
    gy = torch.randn(300, 200, generator=g).to(DEV)
    n0 = _lib.launch_count()
    y = linear(x, w)
    torch.cuda.synchronize()
    assert _lib.launch_count() == n0 + 1
    y.backward(gy)
    torch.cuda.synchronize()
    assert _lib.launch_count() == n0 + 2        # one product: dX or dW, not both
    if needs == "x":
        assert w.grad is None and rel_err(x.grad, gy.double() @ w.detach().double()) < 1e-5
    else:
        assert x.grad is None and rel_err(w.grad, gy.double().t() @ x.detach().double()) < 1e-5


# ---- re2e_skinny_nt / re2e_skinny_nn --------------------------------------------------------------------------------------
@gpu
@pytest.mark.parametrize("nn", [0, 1], ids=["nt", "nn"])
@pytest.mark.parametrize("M,N,K,x_off,acc", [
    (1, 37, 45, 0, 0),        # odd K: scalar staging
    (31, 37, 64, 1, 0),       # K % 4 == 0 but X one float past 16 B: scalar staging
    (32, 1200, 300, 0, 0),    # vector staging
    (33, 50, 45, 0, 1),
    (70, 33, 320, 1, 1),      # three rows per lane
    (70, 1200, 300, 0, 1),
])
def test_skinny_matches_fp64(nn, M, N, K, x_off, acc):
    g = torch.Generator().manual_seed(M * N + K + nn)
    X = torch.randn(M, K, generator=g)
    W = torch.randn(K, N, generator=g) if nn else torch.randn(N, K, generator=g)
    out0 = torch.randn(M, N, generator=g) if acc else None
    xb = torch.full((M * K + 8,), float("nan"), device=DEV)
    xb[x_off:x_off + M * K] = X.flatten().to(DEV)
    ob = torch.full((M * N + 64,), float("nan"), device=DEV)
    out = ob[32:32 + M * N].view(M, N)
    if acc:
        out.copy_(out0)
    Wd = W.to(DEV)
    fn = _lib.lib().re2e_skinny_nn if nn else _lib.lib().re2e_skinny_nt
    n0 = _lib.launch_count()
    assert fn(xb.data_ptr() + 4 * x_off, Wd.data_ptr(), out.data_ptr(), M, N, K, acc, _lib.stream_ptr()) == 0
    torch.cuda.synchronize()
    assert _lib.launch_count() == n0 + 1
    assert torch.isnan(ob[:32]).all() and torch.isnan(ob[32 + M * N:]).all()
    Wt = W.double() if nn else W.double().t()
    ref = X.double() @ Wt + (out0.double() if acc else 0.0)
    scale = X.double().abs() @ Wt.abs() + (out0.double().abs() if acc else 0.0)
    # fp32 FMA chains of <= K terms plus the accumulate add: |error| <= (K + 2) u (sum |x||w| + |out0|), u = 2^-24
    ratio = float(((out.cpu().double() - ref).abs() / scale).max())
    assert ratio <= (K + 2) * 2.0 ** -24, ratio
    assert rel_err(out, ref) < 1e-5


@gpu
@pytest.mark.parametrize("nn", [0, 1], ids=["nt", "nn"])
def test_skinny_rejects_shapes_over_its_shared_memory(nn):
    M, N, K = 64, 32, 800      # 4 (64 * 801 + 16 * 800) B = 256 KB > 200 KB
    X = torch.randn(M, K, device=DEV)
    W = torch.randn(N, K, device=DEV)
    out = torch.full((M, N), 7.0, device=DEV)
    fn = _lib.lib().re2e_skinny_nn if nn else _lib.lib().re2e_skinny_nt
    n0 = _lib.launch_count()
    assert fn(X.data_ptr(), W.data_ptr(), out.data_ptr(), M, N, K, 0, _lib.stream_ptr()) == E_UNSUPPORTED
    torch.cuda.synchronize()
    assert _lib.launch_count() == n0 and bool((out == 7.0).all())


# ---- column sums --------------------------------------------------------------------------------------------------------------
@gpu
@pytest.mark.parametrize("rows,cols,pad", [(6400, 4233, 3), (1, 5, 0), (257, 320, 0), (130, 129, 7)])
def test_colsum_matches_fp64_and_is_deterministic(rows, cols, pad):
    from robust_e2e_gan_b200.linear import colsum
    g = torch.Generator().manual_seed(rows + cols)
    X = torch.randn(rows, cols + pad, generator=g).to(DEV)
    out = colsum(X[:, :cols])
    assert rel_err(out, X[:, :cols].double().sum(0)) < 1e-5
    assert torch.equal(out, colsum(X[:, :cols]))
