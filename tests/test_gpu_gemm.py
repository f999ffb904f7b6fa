"""GPU: the GEMM engines every layer runs on -- the tcgen05 kernels (one tile per CTA with split-K clusters, and the
persistent variant), the CUDA-core kernels, the K-group split of deep and skinny GEMMs and the GEMM chain's store phase --
against float64, variant by variant and epilogue by epilogue.

Two operand regimes:
  * exact: every operand is k / 8 with integer k in [-8, 8].  Such values have 4 significant bits, so TMA's TF32
    conversion keeps them, every product is a multiple of 2^-6 and every partial sum is one of magnitude <= K < 2^18:
    the fp32 accumulator is exact whatever the summation order, split, K group or tile walk.  The pre-activation then
    equals the float64 reference bit for bit, and so does every epilogue step that is one rounded fp32 operation of exact
    values.  ELU, tanh, sin and cos are held to the CUDA Programming Guide's ulp bounds.
  * Gaussian: He-scaled randn operands against float64, measured per slice (worst 128 x bn tile, last row and column
    tile, worst row and column), so that a kernel that quietly dropped to a coarser format still fails.

Outputs, pre-activations and derivative operands live inside guard buffers filled with a NaN bit pattern; the margins
must come back bit-identical.  Operand padding between the logical K (or M / N) and the pitch is NaN too.
"""
import math
import re

import pytest
import torch

gpu = pytest.mark.gpu

DEV = "cuda"
NAN_BITS = 0x7FC0DEAD          # a quiet NaN whose payload no kernel produces
ROW_MARGIN, COL_MARGIN = 128, 256
SMS = 148                      # the persistent kernel needs >= 4 tiles per SM
ULP_BOUND = {"elu": 1, "tanh": 2, "sin": 2, "cos_pre": 2}  # CUDA Programming Guide: expm1f, tanhf, sinf, cosf

# Gaussian-regime bars (rel-L2 of the error over the slice), about 3x the worst measured over every case of this file on
# an NVIDIA B200 at a 1000 W power limit (stated beside each; the module prints them again when run with -s).
TF32_BARS = {"tile": 1e-3,        # measured 3.3e-4
             "row_tile": 1e-3,    # 3.1e-4
             "col_tile": 1e-3,    # 3.1e-4
             "row": 1.5e-3,       # 5.1e-4
             "col": 1.3e-3}       # 4.3e-4
FP32_BARS = {"tile": 5e-7,        # 1.6e-7
             "row_tile": 5e-7,    # 1.6e-7
             "col_tile": 5e-7,    # 1.6e-7
             "row": 1e-6,         # 3.4e-7
             "col": 1.1e-6}       # 3.6e-7

_WORST = {}                    # bar name -> worst Gaussian error seen, printed at the end of the module
_ULPS = {}                     # transcendental -> worst ulp seen


def _lib():
    from rlrep_b200 import _lib as L
    return L


# ------------------------------------------------------------------------------------------------ buffers
def _nan_fill(rows, cols):
    return torch.full((rows, cols), NAN_BITS, dtype=torch.int32, device=DEV).view(torch.float32)


class Guarded:
    """A [rows, cols] view into a NaN-filled buffer with ROW_MARGIN rows and COL_MARGIN columns on every side; `off`
    shifts the view right by that many floats (an unaligned C / aux / pre_out)."""

    def __init__(self, rows, cols, off=0, init=None):
        self.buf = _nan_fill(rows + 2 * ROW_MARGIN, cols + 2 * COL_MARGIN + 4)
        self.view = self.buf[ROW_MARGIN:ROW_MARGIN + rows, COL_MARGIN + off:COL_MARGIN + off + cols]
        if init is not None:
            self.view.copy_(init)
        self.mask = torch.ones_like(self.buf, dtype=torch.bool)
        self.mask[ROW_MARGIN:ROW_MARGIN + rows, COL_MARGIN + off:COL_MARGIN + off + cols] = False

    def margins_intact(self):
        bits = self.buf.view(torch.int32)[self.mask]
        return bool((bits == NAN_BITS).all())


def _operand(rows, cols, draw, pad=0):
    """[rows, cols] operand in a buffer pitch cols + pad (pitch a multiple of 4 floats); the padding is NaN."""
    pitch = (cols + pad + 3) // 4 * 4
    buf = _nan_fill(rows, pitch)
    buf[:, :cols] = draw((rows, cols))
    return buf[:, :cols]


def _exact(shape, gen, lo=-8, hi=8):
    return torch.randint(lo, hi + 1, shape, generator=gen, device=DEV).float() / 8


def _gauss(shape, gen, K):
    return torch.randn(shape, generator=gen, device=DEV) * math.sqrt(2.0 / K)


def _gen(seed):
    g = torch.Generator(device=DEV)
    g.manual_seed(seed)
    return g


# ------------------------------------------------------------------------------------------------ reference
def _f32(x):
    return x.float().double()


def _ulp(x):
    a = x.abs().float()
    return (torch.nextafter(a, torch.full_like(a, math.inf)) - a).double()


def _act64(v, act):
    if act == "elu":
        return torch.where(v > 0, v, torch.expm1(v))
    if act == "relu":
        return torch.clamp(v, min=0)
    if act == "tanh":
        return torch.tanh(v)
    if act == "sin":
        return torch.sin(v)
    return v


def _dact64(h, dact):
    if dact == "elu_out":
        return torch.where(h > 0, torch.ones_like(h), h + 1)
    if dact == "relu_out":
        return (h > 0).double()
    if dact == "tanh_out":
        return 1 - h * h
    if dact == "cos_pre":
        return torch.cos(h)
    return torch.ones_like(h)


class Epi:
    """One epilogue configuration with its operands (exact grid values), the library struct and the float64 model."""

    def __init__(self, M, N, gen, act="none", dact="none", bias=False, scale=1.0, r1=False, pre_out=False,
                 accumulate=False, off=0):
        self.act, self.dact, self.scale, self.accumulate = act, dact, scale, accumulate
        # a bias offset by one float when the store under test is the unaligned one
        self.bias = None
        if bias:
            b = _nan_fill(1, N + 8)[0]
            b[off:off + N] = _exact((N,), gen)
            self.bias = b[off:off + N]
        self.r1 = None
        if r1:  # inside longer buffers: a store past the last row / column reads NaN, not past the allocation
            u, w = _nan_fill(1, M + 8)[0], _nan_fill(1, N + 8)[0]
            u[:M], w[:N] = _exact((M,), gen), _exact((N,), gen)
            self.r1 = (u[:M], w[:N])
        self.aux = None
        if dact != "none":
            lo = -16 if dact == "cos_pre" else -8
            self.aux = Guarded(M, N, off, _exact((M, N), gen, lo=lo))
        self.pre = Guarded(M, N, off) if pre_out else None
        self.c0 = _exact((M, N), gen) if accumulate else None

    def struct(self):
        L = _lib()
        return L.make_epilogue(bias=self.bias, r1=self.r1, aux=self.aux.view if self.aux else None,
                               pre_out=self.pre.view if self.pre else None, act=self.act, dact=self.dact,
                               accumulate=self.accumulate, scale=self.scale)

    def output(self, M, N, off=0):
        return Guarded(M, N, off, self.c0 if self.accumulate else None)

    def pre64(self, acc):
        v = acc * self.scale
        if self.r1 is not None:
            v = v + self.r1[0].double()[:, None] * self.r1[1].double()[None, :]
        if self.bias is not None:
            v = v + self.bias.double()[None, :]
        return v

    def check(self, acc, C, what):
        """Compares the library's C (and pre_out) with the float64 model of the epilogue applied to the exact
        accumulator `acc`.  Bit for bit where every step is one rounded fp32 operation of exact values; within the
        transcendental's ulp bound otherwise."""
        v = self.pre64(acc)
        assert torch.equal(_f32(v), v), f"{what}: operands are not exact in fp32 (test premise)"
        if self.pre is not None:
            assert torch.equal(self.pre.view.double(), v), f"{what}: pre_out differs"
            assert self.pre.margins_intact(), f"{what}: pre_out written outside [M, N]"
        a = _act64(v, self.act)
        d = _dact64(self.aux.view.double(), self.dact) if self.aux is not None else None
        bound = ULP_BOUND.get(self.act, 0) + ULP_BOUND.get(self.dact, 0)
        a32 = _f32(a)
        out = a32 if d is None else _f32(a32 * _f32(d))
        if self.accumulate:
            out = _f32(out + self.c0.double())
        got = C.view.double()
        assert C.margins_intact(), f"{what}: C written outside [M, N]"
        if self.aux is not None:
            assert self.aux.margins_intact(), f"{what}: aux buffer modified"
        if bound == 0:
            bad = (got != out) & ~(torch.isnan(got) & torch.isnan(out))
            assert not bad.any(), f"{what}: {int(bad.sum())} elements differ, first at {bad.nonzero()[0].tolist()}"
            return
        assert not torch.isnan(got).any(), f"{what}: NaN in C"
        # kernel act within B ulp of the exact value, the model's within 0.5: then one rounding per later fp32 step
        dd = torch.ones_like(a) if d is None else d.abs()
        tol = (ULP_BOUND.get(self.act, 0) + 0.5) * _ulp(a) * dd + 2 * _ulp(out) + 1e-37
        if self.dact == "cos_pre":
            tol = tol + (ULP_BOUND["cos_pre"] + 0.5) * _ulp(d) * a.abs()
        if self.accumulate or d is not None:
            tol = tol + _ulp(a32 * (1 if d is None else _f32(d)))
        err = (got - out).abs()
        assert (err <= tol).all(), f"{what}: worst excess {(err - tol).max().item():.3e}"
        if d is None and not self.accumulate:  # the activation alone: its ulp error against float64
            ulps = ((got - a).abs() / _ulp(a)).max().item()
            _ULPS[self.act] = max(_ULPS.get(self.act, 0.0), ulps)
        elif self.dact == "cos_pre" and self.act == "none" and not self.accumulate:
            ref = a * d
            ulps = ((got - ref).abs() / torch.maximum(_ulp(ref), _ulp(a) * 1e-30)).max().item()
            _ULPS["cos_pre"] = max(_ULPS.get("cos_pre", 0.0), ulps)


def _acc64(A, B, a_mn, b_mn):
    a = A.double() if a_mn else A.double().t()          # [K, M]
    b = B.double() if b_mn else B.double().t()          # [K, N]
    return a.t() @ b


def _slices(err, ref, bn, what, bars, label):
    """Per-slice rel-L2 of err against ref: worst 128 x bn tile, last row / column tile, worst row and column."""
    M, N = ref.shape
    e2, r2 = err.square(), ref.square()
    tm, tn = (M + 127) // 128, (N + bn - 1) // bn
    pe = torch.zeros(tm * 128, tn * bn, dtype=torch.float64, device=DEV)
    pr = torch.zeros_like(pe)
    pe[:M, :N], pr[:M, :N] = e2, r2
    te = pe.view(tm, 128, tn, bn).sum((1, 3))
    tr = pr.view(tm, 128, tn, bn).sum((1, 3))
    rel = lambda e, r: (e / r.clamp_min(1e-300)).sqrt()
    got = {"tile": rel(te, tr).max().item(), "row_tile": rel(te[-1].sum(), tr[-1].sum()).item(),
           "col_tile": rel(te[:, -1].sum(), tr[:, -1].sum()).item(), "row": rel(e2.sum(1), r2.sum(1)).max().item(),
           "col": rel(e2.sum(0), r2.sum(0)).max().item()}
    for k, v in got.items():
        key = f"{label}:{k}"
        _WORST[key] = max(_WORST.get(key, 0.0), v)
        assert v < bars[k], f"{what}: {k} rel-L2 {v:.3e} >= {bars[k]:.1e}"


# ------------------------------------------------------------------------------------------------ premise
def test_exact_operands_make_fp32_sums_order_independent():
    """CPU: for k / 8 operands an fp32 matmul equals the float64 one bit for bit in any summation order -- a random
    permutation of K, and K cut into chunks summed separately -- up to K = 39,200."""
    g = torch.Generator().manual_seed(0)
    for M, N, K in ((16, 8, 39200), (64, 48, 507), (3, 5, 17)):
        A = torch.randint(-8, 9, (M, K), generator=g).float() / 8
        B = torch.randint(-8, 9, (N, K), generator=g).float() / 8
        ref = A.double() @ B.double().t()
        assert ref.abs().max().item() < 2 ** 18
        assert torch.equal((A @ B.t()).double(), ref)
        perm = torch.randperm(K, generator=g)
        assert torch.equal((A[:, perm] @ B[:, perm].t()).double(), ref)
        chunks = [A[:, i:i + 97] @ B[:, i:i + 97].t() for i in range(0, K, 97)]
        total = torch.zeros(M, N)
        for c in reversed(chunks):
            total = total + c
        assert torch.equal(total.double(), ref)
        # and the epilogue's pre-activation (scale by a power of two, rank-1 term, bias) stays on the grid
        u, w, b = (torch.randint(-8, 9, (n,), generator=g).float() / 8 for n in (M, N, N))
        v32 = torch.addcmul(total * 0.5, u[:, None], w[None, :]) + b
        assert torch.equal(v32.double(), ref * 0.5 + u.double()[:, None] * w.double()[None, :] + b.double())


# ------------------------------------------------------------------------------------------------ tensor cores
def _tc_plan_ok(K, split):
    nkb = (K + 31) // 32
    return split == 1 or (split - 1) * ((nkb + split - 1) // split) < nkb   # make_tc_plan's non-empty-split rule


def _tc_shape(bn, a_mn, b_mn, split, ragged):
    if not ragged:
        return 256, 2 * bn, 768                                                   # 24 k-blocks
    M = 224 if a_mn else 300
    N = bn + 32 if b_mn else bn + 13                                              # N % 4 != 0 where B allows it
    K = 507 if split > 1 else {32: 8, 64: 17, 128: 23, 256: 203}[bn]              # K % 32 != 0
    return M, N, K


def _majors():
    return [(0, 0), (0, 1), (1, 0), (1, 1)]


TC_CASES = [(bn, a_mn, b_mn, split, ragged) for bn in (32, 64, 128, 256) for a_mn, b_mn in _majors()
            for split in (1, 2, 4, 8) for ragged in (False, True)]


def _operands(M, N, K, a_mn, b_mn, draw):
    A = _operand(K, M, draw, pad=8) if a_mn else _operand(M, K, draw, pad=5)
    B = _operand(K, N, draw, pad=8) if b_mn else _operand(N, K, draw, pad=5)
    return A, B


def _run_tc(A, B, a_mn, b_mn, epi, C, bn, split, path="tc"):
    L = _lib()
    if path == "tc":
        L.gemm(A, B, C, a_mn=bool(a_mn), b_mn=bool(b_mn), path="tc", epi=epi, bn=bn, split_k=split)
    else:
        L.gemm(A, B, C, a_mn=bool(a_mn), b_mn=bool(b_mn), path=path, epi=epi)


@gpu
@pytest.mark.parametrize("bn,a_mn,b_mn,split,ragged", TC_CASES)
def test_tc_variant(lib, bn, a_mn, b_mn, split, ragged):
    """Every (bn, majors, split-K) variant of the one-tile-per-CTA kernel, on an interior shape (fast store) and a
    ragged one (M % 128, N % bn, N % 4, K % 32 != 0): exact operands with bias + ReLU bit for bit, Gaussian per slice."""
    M, N, K = _tc_shape(bn, a_mn, b_mn, split, ragged)
    assert _tc_plan_ok(K, split), (M, N, K, split)
    what = f"tc bn={bn} a_mn={a_mn} b_mn={b_mn} split={split} {M}x{N}x{K}"
    g = _gen(hash((bn, a_mn, b_mn, split, ragged)) & 0xFFFF)
    A, B = _operands(M, N, K, a_mn, b_mn, lambda s: _exact(s, g))
    e = Epi(M, N, g, act="relu", bias=True)
    C = e.output(M, N)
    _run_tc(A, B, a_mn, b_mn, e.struct(), C.view, bn, split)
    e.check(_acc64(A, B, a_mn, b_mn), C, what)
    A, B = _operands(M, N, K, a_mn, b_mn, lambda s: _gauss(s, g, K))
    C = Guarded(M, N)
    _run_tc(A, B, a_mn, b_mn, None, C.view, bn, split)
    ref = _acc64(A, B, a_mn, b_mn)
    assert C.margins_intact(), what
    _slices(C.view.double() - ref, ref, bn, what, TF32_BARS, "tf32")


@gpu
@pytest.mark.parametrize("a_mn,b_mn", _majors())
@pytest.mark.parametrize("shape", [(256, 2048, 1024), (256, 256, 2048), (2048, 1024, 256), (200, 136, 100),
                                   (128, 128, 32), (64, 32, 64)])
def test_tc_planner_choice(lib, a_mn, b_mn, shape):
    """The planner's own (bn, split) over the shapes the agents use, Gaussian operands with bias + ELU."""
    M, N, K = shape
    M = (M + 31) // 32 * 32 if a_mn else M
    N = (N + 31) // 32 * 32 if b_mn else N
    g = _gen(7)
    A, B = _operands(M, N, K, a_mn, b_mn, lambda s: _gauss(s, g, K))
    bias = torch.randn(N, generator=g, device=DEV)
    C = Guarded(M, N)
    _run_tc(A, B, a_mn, b_mn, _lib().make_epilogue(bias=bias, act="elu"), C.view, 0, 0)
    ref = _act64(_acc64(A, B, a_mn, b_mn) + bias.double(), "elu")
    assert C.margins_intact()
    _slices(C.view.double() - ref, ref, 32, f"tc auto {shape} {a_mn}{b_mn}", TF32_BARS, "tf32")


@gpu
def test_tc_refuses_unfetchable_operands(lib):
    """MN-major operands with mn % 32 != 0, and bases that are not 16-byte aligned, are refused loudly on the tensor
    cores (the CUDA-core path takes them)."""
    L = _lib()
    g = _gen(3)
    A, B, C = _exact((64, 100), g), _exact((64, 72), g), torch.empty(100, 72, device=DEV)
    with pytest.raises(L.RlrepError):
        L.gemm(A, B, C, a_mn=True, b_mn=True, path="tc")
    with pytest.raises(L.RlrepError):
        L.gemm(A[:, :96], B, C[:96], a_mn=True, b_mn=True, path="tc")   # N = 72
    Ab = torch.zeros(64, 68, device=DEV)
    with pytest.raises(L.RlrepError):
        L.gemm(Ab[:, 1:65], B[:, :64], C[:64, :64], path="tc")          # A base 4 bytes past a 16-byte boundary
    L.gemm(A, B, C, a_mn=True, b_mn=True, path="simt")
    assert torch.equal(C.double(), A.double().t() @ B.double())


# ------------------------------------------------------------------------------------------------ epilogue matrix
PAIRS = [("none", "none"), ("elu", "none"), ("relu", "none"), ("tanh", "none"), ("sin", "none"),
         ("none", "elu_out"), ("none", "relu_out"), ("none", "tanh_out"), ("none", "cos_pre"),
         ("relu", "elu_out")]          # the last is outside RLREP_EPILOGUE_SWITCH: the run-time (-1, -1) epilogue
EXTRAS = [{}, {"scale": 0.5}, {"r1": True}, {"pre_out": True}, {"accumulate": True},
          {"scale": 2.0, "r1": True, "pre_out": True, "accumulate": True}]

# store path -> (M, N, K, bn, split, offset of C / bias / aux / pre_out in floats)
TC_STORES = {
    "fast": (256, 128, 96, 64, 1, 0),         # store_tile_fast, specialised without extras, run-time with them
    "push": (256, 128, 256, 64, 4, 0),        # split-K pushed into the owner's shared memory, local reduction
    "slice": (256, 512, 256, 256, 2, 0),      # bn = 256: pull over DSMEM into registers, then the stores
    "slice8": (128, 256, 512, 256, 8, 0),
    "edge": (300, 77, 75, 32, 1, 0),          # store_tile_general: ragged M and N, N % 4 != 0
    "edge_split": (300, 141, 507, 128, 4, 0),
    "offset": (256, 128, 96, 64, 1, 1),       # store_tile_general: C, bias, aux, pre_out one float off alignment
}


def _epilogue_matrix(run, M, N, K, off, a_mn, b_mn, seed, what):
    g = _gen(seed)
    A, B = _operands(M, N, K, a_mn, b_mn, lambda s: _exact(s, g))
    acc = _acc64(A, B, a_mn, b_mn)
    for act, dact in PAIRS:
        for bias in (False, True):
            for ex in EXTRAS:
                e = Epi(M, N, g, act=act, dact=dact, bias=bias, off=off, **ex)
                C = e.output(M, N, off)
                run(A, B, e.struct(), C.view)
                e.check(acc, C, f"{what} act={act} dact={dact} bias={bias} {ex}")


@gpu
@pytest.mark.parametrize("store", list(TC_STORES))
def test_tc_epilogue_matrix(lib, store):
    """Every (act, dact) case of the epilogue switch and one outside it, with and without bias, with scale, rank-1
    term, pre-activation copy and accumulate alone and combined, through each store path of the tcgen05 kernel."""
    M, N, K, bn, split, off = TC_STORES[store]
    assert _tc_plan_ok(K, split)
    _epilogue_matrix(lambda A, B, e, C: _run_tc(A, B, 0, 0, e, C, bn, split), M, N, K, off, 0, 0, 11,
                     f"tc {store}")


@gpu
@pytest.mark.parametrize("a_mn,b_mn", _majors())
def test_tc_epilogue_mn_major(lib, a_mn, b_mn):
    """The derivative and extras epilogue on the wgrad / dgrad operand layouts (split-K push, ragged M)."""
    M, N, K = 224, 96, 256
    _epilogue_matrix(lambda A, B, e, C: _run_tc(A, B, a_mn, b_mn, e, C, 32, 2), M, N, K, 0, a_mn, b_mn, 12,
                     f"tc mn {a_mn}{b_mn}")


# ------------------------------------------------------------------------------------------------ persistent kernel
def _persist_shape(bn, ragged):
    M = 4096 + 96                                       # 33 row tiles; MN-major A needs M % 32 == 0
    N = {32: 640, 64: 1280, 128: 2304, 256: 4608}[bn]
    K = {32: 512, 64: 480, 128: 64, 256: 47}[bn]        # nkb <= 16 (bn 32 / 64), <= 2 (bn 128 / 256)
    if ragged:
        N -= 3
    return M, N, K


PERSIST_CASES = [(bn, a_mn, b_mn, store) for bn in (32, 64, 128, 256) for a_mn, b_mn in _majors()
                 for store in ("vector", "scalar")]


def _kernel_names(fn):
    """Names of the CUDA kernels `fn` launches.  `fn` must be idempotent: a profiler session that recorded no device
    activity at all (seen now and then when several sessions run in one process) is repeated."""
    from torch.profiler import ProfilerActivity, profile
    for _ in range(3):
        with profile(activities=[ProfilerActivity.CUDA]) as prof:
            fn()
            torch.cuda.synchronize()
        names = {e.name for e in prof.events() if e.device_type == torch.autograd.DeviceType.CUDA}
        if names:
            break
    return names


@gpu
@pytest.mark.parametrize("bn,a_mn,b_mn,store", PERSIST_CASES)
def test_tc_persistent(lib, bn, a_mn, b_mn, store):
    """>= 592 tiles without split: one CTA per SM walks the tiles.  Its transposed vector store, and the scalar store
    for ragged N (K-major B) or an unaligned C (MN-major B, whose N stays a multiple of 32)."""
    ragged = store == "scalar" and not b_mn
    off = 1 if store == "scalar" and b_mn else 0
    M, N, K = _persist_shape(bn, ragged)
    tiles = ((M + 127) // 128) * ((N + bn - 1) // bn)
    assert tiles >= 4 * SMS
    what = f"persistent bn={bn} a_mn={a_mn} b_mn={b_mn} {store} {M}x{N}x{K}"
    g = _gen(bn + 2 * a_mn + b_mn)
    A, B = _operands(M, N, K, a_mn, b_mn, lambda s: _exact(s, g))
    acc = _acc64(A, B, a_mn, b_mn)
    # the plan does not depend on the epilogue: one plain launch shows which kernel runs
    names = _kernel_names(lambda: _run_tc(A, B, a_mn, b_mn, None, torch.empty(M, N, device=DEV), bn, 1))
    assert any("gemm_tf32_persistent" in n for n in names), (what, names)
    assert not any("gemm_tf32_kernel" in n for n in names), (what, names)
    for kw in (dict(act="relu", bias=True), dict(dact="elu_out", scale=0.5, r1=True, accumulate=True)):
        e = Epi(M, N, g, off=off, **kw)
        C = e.output(M, N, off)
        _run_tc(A, B, a_mn, b_mn, e.struct(), C.view, bn, 1)
        e.check(acc, C, f"{what} {kw}")
    A, B = _operands(M, N, K, a_mn, b_mn, lambda s: _gauss(s, g, K))
    C = Guarded(M, N, off)
    _run_tc(A, B, a_mn, b_mn, None, C.view, bn, 1)
    ref = _acc64(A, B, a_mn, b_mn)
    assert C.margins_intact(), what
    _slices(C.view.double() - ref, ref, bn, what, TF32_BARS, "tf32")


# ------------------------------------------------------------------------------------------------ CUDA cores
# kernel -> (M, N, K, a_mn, b_mn); launch_simt picks the kernel from the shape
SIMT_SHAPES = {
    "tiled": (200, 100, 77, 0, 0),
    "tiled_mn": (200, 100, 77, 1, 1),
    "tiled_amn": (130, 70, 45, 1, 0),
    "tiled_bmn": (70, 130, 45, 0, 1),
    "rowwarp": (100, 23, 300, 0, 0),
    "rowwarp_bmn": (100, 32, 64, 0, 1),
    "rowthread8": (100, 6, 300, 1, 1),
    "rowthread16": (100, 12, 300, 1, 1),
    "rowthread32": (100, 23, 300, 1, 1),
    "rowthread_t8": (6, 100, 300, 1, 1),       # M <= 32: the transposed problem
    "rowthread_t16": (12, 100, 300, 1, 1),
    "rowthread_t32": (23, 100, 300, 1, 1),
}


def _run_simt(A, B, a_mn, b_mn, epi, C, A2=None):
    _lib().gemm(A, B, C, a_mn=bool(a_mn), b_mn=bool(b_mn), path="simt", epi=epi, A2=A2)


@gpu
@pytest.mark.parametrize("kernel", list(SIMT_SHAPES))
def test_simt_kernel(lib, kernel):
    """Each CUDA-core kernel on its shape: the epilogue matrix on exact operands bit for bit, Gaussian near 1e-6."""
    M, N, K, a_mn, b_mn = SIMT_SHAPES[kernel]
    _epilogue_matrix(lambda A, B, e, C: _run_simt(A, B, a_mn, b_mn, e, C), M, N, K, 0, a_mn, b_mn, 21,
                     f"simt {kernel}")
    g = _gen(22)
    A, B = _operands(M, N, K, a_mn, b_mn, lambda s: _gauss(s, g, K))
    C = Guarded(M, N, 1)
    _run_simt(A, B, a_mn, b_mn, None, C.view)
    ref = _acc64(A, B, a_mn, b_mn)
    assert C.margins_intact()
    _slices(C.view.double() - ref, ref, 64, f"simt {kernel}", FP32_BARS, "fp32")


@gpu
def test_simt_two_segment_input(lib):
    """cat(s, a) read from two buffers (first layers), K1 not a multiple of 4 or of 16, with a tanh epilogue, a
    derivative epilogue with rank-1 term and accumulate, and a pre-activation copy."""
    L = _lib()
    M, N = 64, 40
    for K1, K2 in ((17, 6), (18, 5), (20, 9), (40, 23)):
        g = _gen(K1)
        X1, X2 = _operand(M, K1, lambda s: _exact(s, g), 3), _operand(M, K2, lambda s: _exact(s, g), 1)
        W = _operand(N, K1 + K2, lambda s: _exact(s, g), 2)
        acc = torch.cat([X1, X2], 1).double() @ W.double().t()
        for kw in (dict(act="tanh", bias=True), dict(dact="elu_out", r1=True, accumulate=True), dict(pre_out=True)):
            e = Epi(M, N, g, **kw)
            C = e.output(M, N)
            L.gemm(X1, W, C.view, path="simt", A2=X2, epi=e.struct())
            e.check(acc, C, f"two-segment K1={K1} K2={K2} {kw}")


# ------------------------------------------------------------------------------------------------ K groups
KGROUP_CASES = [(M, N, K) for M in (256, 100) for N in (50, 64, 200) for K in (39200, 32768 + 17)]


@gpu
@pytest.mark.parametrize("M,N,K", KGROUP_CASES)
def test_runner_k_groups(lib, M, N, K):
    """Deep and skinny GEMMs through the agents' runner: K cut into groups, each reduced by its own split-K cluster,
    then kgroup_finish sums the groups and applies the epilogue (accumulate included)."""
    g = _gen(M + N)
    A, B = _operands(M, N, K, 0, 0, lambda s: _exact(s, g))
    acc = _acc64(A, B, 0, 0)
    names = _kernel_names(lambda: _run_tc(A, B, 0, 0, None, torch.empty(M, N, device=DEV), 0, 0, path="runner"))
    assert any("kgroup_finish" in n for n in names), names
    for kw in (dict(act="relu", bias=True), dict(act="tanh", bias=True), dict(accumulate=True, scale=0.5)):
        e = Epi(M, N, g, **kw)
        C = e.output(M, N)
        _run_tc(A, B, 0, 0, e.struct(), C.view, 0, 0, path="runner")
        e.check(acc, C, f"k groups {M}x{N}x{K} {kw}")
    A, B = _operands(M, N, K, 0, 0, lambda s: _gauss(s, g, K))
    C = Guarded(M, N)
    _run_tc(A, B, 0, 0, None, C.view, 0, 0, path="runner")
    ref = _acc64(A, B, 0, 0)
    assert C.margins_intact()
    _slices(C.view.double() - ref, ref, 128, f"k groups {M}x{N}x{K}", TF32_BARS, "tf32")


# ------------------------------------------------------------------------------------------------ chain
CHAIN_EXTRAS = {"scale": dict(scale=0.5, bias=True, act="relu"),
                "r1_derivative": dict(r1=True, dact="tanh_out"),
                "pre_out": dict(pre_out=True, bias=True, act="relu"),
                "accumulate": dict(accumulate=True, dact="relu_out")}


@gpu
@pytest.mark.parametrize("bn,split_k", [(0, 0), (64, 2)])
@pytest.mark.parametrize("extra", list(CHAIN_EXTRAS))
def test_chain_epilogue_extras(lib, extra, bn, split_k):
    """The GEMM chain's own store code for scale, rank-1 term + derivative, pre_out and accumulate, bit for bit."""
    L = _lib()
    g = _gen(31)
    M, N, K = 256, 160, 256
    A, B = _operands(M, N, K, 0, 0, lambda s: _exact(s, g))
    e = Epi(M, N, g, **CHAIN_EXTRAS[extra])
    C = e.output(M, N)
    L.gemm_chain([(A, B, C.view, dict(epi=e.struct()))], bn=bn, split_k=split_k, iters=1)
    torch.cuda.synchronize()
    e.check(_acc64(A, B, 0, 0), C, f"chain {extra} bn={bn} split={split_k}")


# ------------------------------------------------------------------------------------------------ determinism
DETERMINISM_CASES = {
    "push": (256, 256, 2048, 64, 4, "tc"),
    "pull": (256, 512, 2048, 256, 8, "tc"),
    "persistent": (4192, 640, 512, 32, 1, "tc"),
    "k_groups": (256, 200, 39200, 0, 0, "runner"),
}


@gpu
@pytest.mark.parametrize("case", list(DETERMINISM_CASES))
def test_repeated_launches_are_bit_identical(lib, case):
    M, N, K, bn, split, path = DETERMINISM_CASES[case]
    g = _gen(41)
    A, B = _operands(M, N, K, 0, 0, lambda s: _gauss(s, g, K))
    outs = []
    for _ in range(3):
        C = torch.empty(M, N, device=DEV)
        _run_tc(A, B, 0, 0, None, C, bn, split, path=path)
        outs.append(C)
    torch.cuda.synchronize()
    assert all(torch.equal(o.view(torch.int32), outs[0].view(torch.int32)) for o in outs[1:]), case


# ------------------------------------------------------------------------------------------------ coverage
@gpu
def test_gemm_paths_are_reached(lib):
    """The shapes of this file launch all 16 one-tile and all 16 persistent tcgen05 instantiations, every CUDA-core
    kernel and width, the K-group finish and the chain kernel.  If the planner or the dispatch stops reaching one of
    them at these sizes, this test says so."""
    L = _lib()
    g = _gen(51)
    draw = lambda s: _exact(s, g)

    def launch_all():
        for bn, a_mn, b_mn, split, ragged in TC_CASES:
            M, N, K = _tc_shape(bn, a_mn, b_mn, split, ragged)
            A, B = _operands(M, N, K, a_mn, b_mn, draw)
            _run_tc(A, B, a_mn, b_mn, None, torch.empty(M, N, device=DEV), bn, split)
        for bn, a_mn, b_mn, store in PERSIST_CASES:
            M, N, K = _persist_shape(bn, store == "scalar" and not b_mn)
            A, B = _operands(M, N, K, a_mn, b_mn, draw)
            _run_tc(A, B, a_mn, b_mn, None, torch.empty(M, N, device=DEV), bn, 1)
        for M, N, K, a_mn, b_mn in SIMT_SHAPES.values():
            A, B = _operands(M, N, K, a_mn, b_mn, draw)
            _run_simt(A, B, a_mn, b_mn, None, torch.empty(M, N, device=DEV))
        M, N, K = KGROUP_CASES[0]
        A, B = _operands(M, N, K, 0, 0, draw)
        _run_tc(A, B, 0, 0, None, torch.empty(M, N, device=DEV), 0, 0, path="runner")
        A, B = _operands(256, 160, 256, 0, 0, draw)
        L.gemm_chain([(A, B, torch.empty(256, 160, device=DEV), {})], iters=1)

    names = _kernel_names(launch_all)
    found = set()
    for n in names:
        m = re.search(r"(gemm_tf32_kernel|gemm_tf32_persistent_kernel)<(\d+), (true|false), (true|false)>", n)
        if m:
            found.add((m.group(1), int(m.group(2)), m.group(3) == "true", m.group(4) == "true"))
    missing = [(k, bn, a, b) for k in ("gemm_tf32_kernel", "gemm_tf32_persistent_kernel") for bn in (32, 64, 128, 256)
               for a in (False, True) for b in (False, True) if (k, bn, a, b) not in found]
    assert not missing, (missing, sorted(names))
    rowthread = {int(m.group(1)) for n in names for m in [re.search(r"skinny_rowthread_kernel<(\d+)>", n)] if m}
    assert rowthread == {8, 16, 32}, sorted(names)
    for want in ("gemm_tiled_kernel", "skinny_rowwarp_kernel", "kgroup_finish_kernel", "gemm_chain_kernel"):
        assert any(want in n for n in names), (want, sorted(names))


@gpu
def test_report_measured_worst():
    """Prints the worst Gaussian-regime error per bar and the worst ulp per transcendental seen by this module (run
    with -s); the bars beside TF32_BARS / FP32_BARS are about 3x these on a B200."""
    for k in sorted(_WORST):
        print(f"gemm worst {k}: {_WORST[k]:.3e}")
    for k in sorted(_ULPS):
        print(f"gemm worst ulp {k}: {_ULPS[k]:.2f} (bound {ULP_BOUND[k]})")
