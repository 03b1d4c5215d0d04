"""Every per-sweep contraction kernel (csrc/contract.cu, csrc/mttkrp_tc.cu, csrc/tc_gemm.cu) against float64.

`admmq_mttkrp_kernel` names the kernel, tile width, grid and split count an MTTKRP call runs with (include/admmq.h,
ADMMQ_MTTKRP_*).  The case list holds every mode of the ResNet-18 headline layers and the two matrix workloads at
both precisions, plus the edges of every path: fold groups that do not fill a 128-row tile, long-fold tiles that
straddle two output rows, every tile width the query can return at 148 SMs, K tails against the stage depths of the
tile product, ranks of 1 .. 1141 and the split counts of the float64 sum.

CPU: the case list reaches every kernel and width, the headline maps to HEADLINE_KERNELS, the query's edges.
GPU, per MTTKRP case (and admmq_gemm_nt's own operand path):
  - precision 1: |F - F64| <= (nx + 48) u mag + ulp(F) / 2 elementwise (see `tc_bound`);
  - precision 0: on inputs whose contraction float64 holds exactly (see `exact_inputs`), F is the correctly rounded
    float32 of the exact result on every element, with and without the split of the sum over p;
  - the fold gives the same bits at every forced tile width;
  - hygiene: the output starts as NaN inside NaN guard words, the workspace as 0xFF bytes; afterwards the guards
    and the inputs are unchanged, no NaN is left, and a second call and a call with a zeroed workspace give the
    same bits.
Also on the GPU: the float32 Gram-Hadamard product, unfold3, permute_myx, the reconstruction error and the float64
pieces of the ALS / EPC initialisation.
"""
import ctypes
import os
import re
from collections import namedtuple
from types import SimpleNamespace

import numpy as np
import pytest
import torch

REPO = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
U32 = 2.0 ** -24                 # unit roundoff of float32
U64 = 2.0 ** -53                 # ... of float64
GUARD = 64                       # guard words on each side of an output
SENTINEL = 0x7FA5A5A5            # a NaN: what an output and its guards hold before the call

# op: "mttkrp" (admmq_mttkrp at precision 0, admmq_permute_myx + admmq_mttkrp_tc at precision 1) or "gemm_nt"
# (admmq_gemm_nt, B split on the fly); ny = 1 for a matrix
Case = namedtuple("Case", "op M nx ny R precision")


def _kernel_ids():
    text = open(os.path.join(REPO, "include", "admmq.h")).read()
    return {k: int(v) for k, v in re.findall(r"#define ADMMQ_MTTKRP_(\w+) (\d+)", text)}


IDS = _kernel_ids()
BASES = {"GEMM": (16, 32, 64, 128), "FOLD": tuple(range(16, 129, 16)), "FOLDLONG": (80, 96, 112, 128)}
ALL_KERNELS = {IDS["F64_16"], IDS["F64_64"]} | {IDS[b] + w for b, ws in BASES.items() for w in ws}


def kernel_name(kid):
    for b in ("FOLDLONG", "FOLD", "GEMM"):
        if kid > IDS[b]:
            return f"{b}{kid - IDS[b]}"
    return next(k for k, v in IDS.items() if v == kid)


def _nat():
    from source import _native
    return _native


def _sm_count():
    return torch.cuda.get_device_properties(0).multi_processor_count if torch.cuda.is_available() else 148


def query(case, sms):
    """(id, grid, splits) of the case; admmq_gemm_nt has the matrix path's cost model without the 128 width."""
    return _nat().mttkrp_kernel(case.M, case.nx, case.ny, case.R, case.precision, sms)


def headline_layers():
    import bench
    units, _ = bench.workload_units(SimpleNamespace(workload="resnet18", reduction_rate=2.0, bits=4))
    return list(dict.fromkeys((bench.unit_shape(u), bench.unit_rank(u)) for u in units))


def headline_matrices():
    """resnet50-l4 conv3 and llama7b q_proj: (M, nx, R) of both orientations."""
    import bench
    out = []
    for wl, shape in (("resnet50-l4", (2048, 512)), ("llama7b", (4096, 4096))):
        units, _ = bench.workload_units(SimpleNamespace(workload=wl, reduction_rate=2.0, bits=4))
        R = next(bench.unit_rank(u) for u in units if bench.unit_shape(u) == shape)
        out += list(dict.fromkeys([(shape[0], shape[1], R), (shape[1], shape[0], R)]))
    return out


def modes(shape):
    """(M, nx, ny) of the three MTTKRPs of a 3-way tensor, as the solver calls them (nx, ny in mode order)."""
    I, J, K = shape
    return [(I, J, K), (J, I, K), (K, I, J)]


# what the headline runs on at 148 SMs (precision 1: tensor-core MTTKRP; bench.py's default)
HEADLINE_KERNELS = {
    ((64, 64, 9), 134): ("FOLD16", "FOLD16", "FOLD16"),
    ((128, 64, 9), 183): ("FOLD16", "FOLD16", "FOLD16"),
    ((128, 128, 9), 278): ("FOLD32", "FOLD32", "FOLD32"),
    ((256, 128, 9), 375): ("FOLD64", "FOLD32", "FOLD32"),
    ((256, 256, 9), 566): ("FOLD96", "FOLD96", "FOLDLONG80"),
    ((512, 256, 9), 759): ("FOLD96", "FOLD112", "FOLDLONG96"),
    ((512, 512, 9), 1141): ("FOLD96", "FOLD96", "FOLDLONG96"),
    ((2048, 512), 204): ("GEMM32", "GEMM16"),
    ((4096, 4096), 1024): ("GEMM128", "GEMM128"),
}


def build_cases(sms):
    cases = []

    def add(M, nx, ny, R, precisions=(1,), op="mttkrp"):
        for p in precisions:
            c = Case(op, M, nx, ny, R, p)
            if c not in cases:
                cases.append(c)

    # headline: every mode of every ResNet-18 layer and both matrix workloads, at both precisions
    for shape, R in headline_layers():
        for M, nx, ny in modes(shape):
            add(M, nx, ny, R, (1, 0))
    for M, nx, R in headline_matrices():
        add(M, nx, 1, R, (1, 0))
    # fold: two m per row of 64, a last tile with fewer than mg m (37 = 2 x 14 + 9) and Mout * ny = 333 not a multiple
    # of 128, one m per tile (ny = 127 leaves a row of the box unused, ny = 128 fills it), more tiles than CTAs
    add(5, 64, 2, 17)
    add(37, 65, 9, 134)
    add(3, 31, 127, 15)
    add(2, 130, 128, 1141)
    add(300, 129, 9, 1141)
    # long fold: Mout = 1 (a second tile with one row), tiles that straddle two m (ny = 129, 200, 255, 257), tiles
    # inside one m (256, 640), more tiles than CTAs
    add(1, 64, 129, 17)
    add(3, 64, 129, 1141)
    add(5, 31, 200, 15)
    add(4, 65, 255, 1)
    add(2, 130, 256, 134)
    add(3, 3, 257, 1141)
    add(2, 129, 640, 17)
    add(17, 130, 200, 1141)
    # K tails: nx = 1 .. 130 covers ldv padding, a partial swizzle atom and 1 .. 3 K-blocks, on every path
    for nx in (1, 3, 31, 64, 65, 129, 130):
        add(40, nx, 9, 33)
        add(200, nx, 1, 17)
        add(2, nx, 200, 134)
        add(130, nx, 1, 1141)
    # ranks
    for R in (1, 15, 17, 1141):
        add(64, 64, 9, R)
        add(17, 3, 200, R)
    # every tensor-core width the query can return: the smallest shape that selects it
    want = {IDS["GEMM"] + w for w in BASES["GEMM"]} | {IDS["FOLD"] + w for w in BASES["FOLD"]} | \
        {IDS["FOLDLONG"] + w for w in BASES["FOLDLONG"]}
    cands = sorted(((M, 64, ny, R) for ny in (1, 9, 129) for M in (1, 9, 17, 64, 128, 200, 256, 512, 1000)
                    for R in (1, 17, 134, 300, 700, 1000, 1141, 1500)), key=lambda s: s[0] * s[2] * s[3])
    for w in sorted(want):
        if any(query(c, sms)[0] == w for c in cases if c.precision == 1):
            continue
        found = next((s for s in cands if _nat().mttkrp_kernel(*s, 1, sms)[0] == w), None)
        assert found is not None, f"no shape selects {kernel_name(w)}"
        add(*found)
    # admmq_gemm_nt's own operand path at the widths it has (16, 32, 64)
    for w in (16, 32, 64):
        s = next(c for c in cases if c.precision == 1 and query(c, sms)[0] == IDS["GEMM"] + w)
        add(s.M, s.nx, 1, s.R, op="gemm_nt")
    add(130, 65, 1, 17, op="gemm_nt")
    # precision 0: 16- and 64-row tiles, one slice (P < 512), P not a multiple of 16, the cap of 64 slices
    add(16, 31, 9, 15, (0,))
    add(17, 31, 9, 15, (0,))
    add(16, 128, 128, 64, (0,))
    add(9, 1, 3, 1, (0,))
    add(17, 129, 130, 1141, (0,))
    return cases


CASES = build_cases(_sm_count())


def case_id(c):
    return f"{c.op}-{c.M}x{c.nx}x{c.ny}-R{c.R}-p{c.precision}"


# ------------------------------------------------------------------------------------------------ CPU
def test_case_list_reaches_every_kernel_and_width():
    sms = 148
    cases = build_cases(sms)
    reached = {query(c, sms)[0] for c in cases if c.op == "mttkrp"}
    assert reached == ALL_KERNELS, sorted(kernel_name(k) for k in ALL_KERNELS ^ reached)
    gemm_nt = {query(c, sms)[0] - IDS["GEMM"] for c in cases if c.op == "gemm_nt"}
    assert gemm_nt == {16, 32, 64}, gemm_nt
    splits = {query(c, sms)[2] for c in cases if c.precision == 0}
    assert 1 in splits and 64 in splits and max(splits) == 64, sorted(splits)
    # at least one long-fold case with a 128-row tile that holds rows of two m
    assert any(c.ny > 128 and any((t * 128) // c.ny != min(t * 128 + 127, c.M * c.ny - 1) // c.ny
                                  for t in range((c.M * c.ny + 127) // 128)) for c in cases)


def test_headline_runs_on_the_published_kernels():
    nat = _nat()
    layers = dict(headline_layers())
    mats = headline_matrices()
    assert set(HEADLINE_KERNELS) == {(s, r) for s, r in layers.items()} | {((M, nx), R) for M, nx, R in mats[::2]}
    for (shape, R), names in HEADLINE_KERNELS.items():
        ms = modes(shape) if len(shape) == 3 else [(shape[0], shape[1], 1), (shape[1], shape[0], 1)]
        got = tuple(kernel_name(nat.mttkrp_kernel(M, nx, ny, R, 1, 148)[0]) for M, nx, ny in ms)
        assert got == names, (shape, R, got)
        par = {kernel_name(nat.mttkrp_kernel(M, nx, ny, R, 0, 148)[0]) for M, nx, ny in ms}
        assert par <= {"F64_16", "F64_64"}, (shape, R, par)


def test_kernel_query_edges(monkeypatch):
    nat = _nat()
    k = lambda M, nx, ny, R, p=1, s=148: kernel_name(nat.mttkrp_kernel(M, nx, ny, R, p, s)[0])   # noqa: E731
    assert k(9, 512, 128, 1141).startswith("FOLD") and not k(9, 512, 128, 1141).startswith("FOLDLONG")
    assert k(9, 512, 129, 1141).startswith("FOLDLONG")
    assert k(9, 512, 1, 1141).startswith("GEMM") and k(9, 512, 2, 1141).startswith("FOLD")
    assert k(16, 64, 9, 64, 0) == "F64_16" and k(17, 64, 9, 64, 0) == "F64_64"
    assert nat.mttkrp_kernel(16, 31, 9, 15, 0, 148)[2] == 1                  # P < 512: one slice
    assert nat.mttkrp_kernel(16, 128, 128, 64, 0, 148)[2] == 64              # the cap
    assert nat.mttkrp_kernel(4096, 4096, 1, 1024, 1, 148)[1:] == (148, 1)    # 256 tiles on 148 CTAs
    monkeypatch.setenv("ADMMQ_FOLD_BN", "48")
    assert k(512, 512, 9, 1141) == "FOLD48" and k(9, 512, 129, 1141) == "FOLDLONG96"
    monkeypatch.setenv("ADMMQ_FOLD_BN", "50")                                # not a multiple of 16: ignored
    assert k(512, 512, 9, 1141) == "FOLD96"
    for bad in ((0, 5, 9, 5, 1, 148), (5, 0, 9, 5, 1, 148), (5, 5, 0, 5, 1, 148), (5, 5, 9, 0, 1, 148),
                (5, 5, 9, 5, 2, 148), (5, 5, 9, 5, -1, 148), (5, 5, 9, 5, 1, 0)):
        with pytest.raises(ValueError):
            nat.mttkrp_kernel(*bad)


# ------------------------------------------------------------------------------------------------ reference pieces
def exact_inputs(g, M, nx, ny, R):
    """Wn, X, Y whose MTTKRP float64 computes exactly, in any order: W holds 11-bit integers times 2^-14, X and Y
    13-bit integers times 2^-12.  Every product X Y is exact in float64 (26 bits), every term W X Y a multiple of
    2^-38 below 2^-4, and every partial sum of at most 2^18 terms below 2^14, i.e. at most 2^52 units of 2^-38.  So the
    float64 reference is the exact contraction, the kernel's float64 accumulation is exact too, and its float32 result
    must be the correctly rounded value - no band of ambiguous elements.  (With Gaussian inputs the worst-case
    float64 error 2 P 2^-53 sum|terms| reaches about a quarter of a float32 ulp at the headline depth P = 2^18, and
    about half the elements would fall inside it.)"""
    assert nx * ny <= 2 ** 18
    ri = lambda shape, b, e: (torch.randint(-2 ** b, 2 ** b + 1, shape, generator=g) * 2.0 ** e).float()   # noqa: E731
    Y = ri((ny, R), 12, -12) if ny > 1 else None
    return ri((M, nx * ny), 10, -14), ri((nx, R), 12, -12), Y


def gauss_inputs(g, M, nx, ny, R):
    Y = torch.randn(ny, R, generator=g) if ny > 1 else None
    return torch.randn(M, nx * ny, generator=g) * 0.05, torch.randn(nx, R, generator=g), Y


def mttkrp64(Wn, X, Y):
    """F64 = Wn . KhatriRao(X, Y) in float64 on the device (T = W x X per y, then the weighted sum over y)."""
    Wn, X = Wn.double(), X.double()
    if Y is None:
        return Wn @ X
    M, nx, ny = Wn.shape[0], X.shape[0], Y.shape[0]
    T = torch.einsum("mxy,xr->myr", Wn.view(M, nx, ny), X)
    return (T * Y.double()[None]).sum(1)


def tc_bound(F, mag, nx):
    """3xTF32 bound: the split of both operands into tf32 hi + lo drops lo.lo and rounds the lo parts (3 * 2^-22 =
    12 u per product); an accumulator update of the MMA may truncate (1 ulp = 2 u), and a product passes at most
    3 * ceil(nx / 8) of them plus the sums inside an MMA and the sum of the two accumulators: (nx + 48) u times
    sum |W X| for an element of T.  The fold over y (float64, the products Y T exact) carries this into
    (nx + 48) u sum |Wn KR| = (nx + 48) u mag, and the result is rounded to float32 once: + ulp(F) / 2."""
    a = F.abs()
    half_ulp = (torch.nextafter(a, torch.full_like(a, float("inf"))) - a).double() / 2
    return (nx + 48) * U32 * mag + half_ulp


def guarded(n, dtype=torch.float32):
    """(buffer, view): n elements of NaN between GUARD NaN words on each side."""
    buf = torch.full((n + 2 * GUARD,), SENTINEL, dtype=torch.int32, device="cuda").view(dtype) if dtype == torch.float32 \
        else torch.full((n + 2 * GUARD,), float("nan"), dtype=dtype, device="cuda")
    return buf, buf[GUARD:GUARD + n]


def bits(t):
    return t.contiguous().view(torch.int32 if t.element_size() == 4 else torch.int64)


def same(a, b):
    return torch.equal(bits(a), bits(b))


def guards_intact(buf):
    ref = guarded(0, buf.dtype)[0][:GUARD]
    return same(buf[:GUARD], ref) and same(buf[-GUARD:], ref)


def ptr(t):
    return ctypes.c_void_p(t.data_ptr())


def stream():
    return ctypes.c_void_p(torch.cuda.current_stream().cuda_stream)


class Runner:
    """One contraction call on fixed inputs, output in a guarded NaN buffer, workspace of 0xFF bytes."""

    def __init__(self, case, Wn, X, Y):
        nat = self.nat = _nat()
        self.case, self.Wn, self.X, self.Y = case, Wn, X, Y
        M, nx, ny, R = case.M, case.nx, case.ny, case.R
        self.ldv = (nx + 3) // 4 * 4
        if case.op == "gemm_nt":
            self.A = torch.zeros(M, self.ldv, device="cuda")
            self.A[:, :nx] = Wn
            self.B = torch.zeros(R, self.ldv, device="cuda")
            self.B[:, :nx] = X.t()
            self.inputs = (self.A, self.B)
            need = 0
        elif case.precision == 1:
            self.V = nat.permute_myx(Wn, nx, ny)
            self.inputs = (self.V, X) + ((Y,) if Y is not None else ())
            need = nat.mttkrp_tc_workspace_bytes(M, nx, ny, R)
        else:
            self.inputs = (Wn, X) + ((Y,) if Y is not None else ())
            need = nat.mttkrp_workspace_bytes(M, nx, ny, R, 0)
        self.need = max(need, 256)
        self.before = [t.clone() for t in self.inputs]

    def __call__(self, ws_fill=0xFF, ws_bytes=None):
        c, nat = self.case, self.nat
        buf, F = guarded(c.M * c.R)
        ws = torch.full((self.need,), ws_fill, dtype=torch.uint8, device="cuda")
        nb = self.need if ws_bytes is None else ws_bytes
        Yp = None if self.Y is None else ptr(self.Y)
        if c.op == "gemm_nt":
            rc = nat.lib.admmq_gemm_nt(ptr(self.A), self.ldv, c.M, ptr(self.B), self.ldv, c.R, c.nx, ptr(F), c.R, stream())
        elif c.precision == 1:
            rc = nat.lib.admmq_mttkrp_tc(ptr(self.V), c.M, ptr(self.X), c.nx, Yp, c.ny, c.R, ptr(F), ptr(ws), nb, stream())
        else:
            rc = nat.lib.admmq_mttkrp(ptr(self.Wn), c.M, ptr(self.X), c.nx, Yp, c.ny, c.R, ptr(F), 0, ptr(ws), nb,
                                      stream())
        nat.check(rc)
        assert guards_intact(buf), "a guard word was overwritten"
        assert not bool(torch.isnan(F).any()), "an output element was never written"
        assert all(same(a, b) for a, b in zip(self.inputs, self.before)), "an input changed"
        return F.view(c.M, c.R)


# ------------------------------------------------------------------------------------------------ GPU: MTTKRP
@pytest.mark.gpu
@pytest.mark.parametrize("case", CASES, ids=[case_id(c) for c in CASES])
def test_mttkrp_kernel(case, capsys, monkeypatch):
    monkeypatch.delenv("ADMMQ_FOLD_BN", raising=False)
    sms = _sm_count()
    kid, grid, splits = query(case, sms)
    g = torch.Generator().manual_seed(7000 + CASES.index(case))
    M, nx, ny, R = case.M, case.nx, case.ny, case.R
    Wn, X, Y = ((exact_inputs if case.precision == 0 else gauss_inputs)(g, M, nx, ny, R))
    Wn, X = Wn.cuda(), X.cuda()
    Y = None if Y is None else Y.cuda()
    run = Runner(case, Wn, X, Y)
    F = run()
    F64 = mttkrp64(Wn, X, Y)
    if case.precision == 1:
        mag = mttkrp64(Wn.abs(), X.abs(), None if Y is None else Y.abs())
        ratio = float(((F.double() - F64).abs() / tc_bound(F, mag, nx)).max())
        assert ratio <= 1.0, f"off by {ratio:.3g} x the 3xTF32 bound"
        detail = f"error {ratio:.3f} of bound"
    else:
        exact32 = F64.float()
        wrong = int((bits(F) != bits(exact32)).sum())
        assert wrong == 0, f"{wrong} elements are not the correctly rounded float32 of the exact contraction"
        # the same sum in one slice: a workspace too small for the partials
        if splits > 1:
            assert same(run(ws_bytes=splits * M * R * 8 - 8), F), "the one-slice fallback differs"
        detail = f"{splits} slices, exact"
    # the same bits again, and with a zeroed workspace
    assert same(run(), F), "a second call differs"
    assert same(run(ws_fill=0), F), "the result depends on the workspace's previous contents"
    # the fold sums over k in the same order at every tile width
    if case.op == "mttkrp" and case.precision == 1 and 1 < ny <= 128:
        for w in BASES["FOLD"]:
            monkeypatch.setenv("ADMMQ_FOLD_BN", str(w))
            assert query(case, sms)[0] == IDS["FOLD"] + w
            assert same(run(), F), f"tile width {w} gives other bits than {kernel_name(kid)}"
        monkeypatch.delenv("ADMMQ_FOLD_BN")
    with capsys.disabled():
        print(f"\n[mttkrp] {case_id(case)} {kernel_name(kid)} grid {grid}: {detail}", end="")


# ------------------------------------------------------------------------------------------------ GPU: the others
def gram_pairs():
    """(n1, n2, R) of the Gram-Hadamard products: the headline operand pairs (n2 = 0: U2 = NULL, the matrix case),
    R of 1 and around a 32-wide tile edge, and a one-row U1."""
    pairs = []
    for shape, R in headline_layers():
        for _, nx, ny in modes(shape):
            pairs.append((nx, ny, R))
    for M, nx, R in headline_matrices():
        pairs.append((nx, 0, R))
    for R in (1, 31, 32, 33):
        pairs += [(64, 9, R), (64, 0, R)]
    pairs += [(1, 9, 33), (1, 0, 134)]
    return list(dict.fromkeys(pairs))


def _rounding_candidates(x64, band):
    """The float32 values the correctly rounded result can take when x64 is within `band` of the exact value."""
    return (x64 - band).float(), (x64 + band).float()


@pytest.mark.gpu
def test_gram_hadamard(capsys):
    """G = fl32(fl32(G1) * fl32(G2)), each Gram the float64 sum of the exact float32 products, rounded once.  The
    kernel's and the reference's float64 Grams each lie within n u64 sum|products| of the exact one; where twice that
    band contains no float32 rounding boundary, G must be bit for bit the float32 product of the rounded Grams;
    elsewhere it must lie between the products of the candidate roundings.  G must be bitwise symmetric."""
    nat = _nat()
    g = torch.Generator().manual_seed(31)
    worst_amb = 0.0
    for n1, n2, R in gram_pairs():
        U1 = torch.randn(n1, R, generator=g).cuda()
        U2 = torch.randn(n2, R, generator=g).cuda() if n2 else None
        buf, G = guarded(R * R)
        before = [t.clone() for t in (U1, U2) if t is not None]
        nat.check(nat.lib.admmq_gram_hadamard(ptr(U1), n1, None if U2 is None else ptr(U2), n2, R, ptr(G), stream()))
        G = G.view(R, R)
        assert guards_intact(buf) and not bool(torch.isnan(G).any()), (n1, n2, R)
        assert all(same(a, b) for a, b in zip(before, [t for t in (U1, U2) if t is not None]))
        lo, hi, amb = None, None, torch.zeros(R, R, dtype=torch.bool, device="cuda")
        for U, n in ((U1, n1), (U2, n2)):
            if U is None:
                continue
            Ud = U.double()
            band = 2 * n * U64 * (Ud.abs().T @ Ud.abs()) * (1 + 1e-9)
            a, b = _rounding_candidates(Ud.T @ Ud, band)
            amb |= a != b
            if lo is None:
                lo, hi = a, b
            else:
                prods = torch.stack([lo * a, lo * b, hi * a, hi * b])
                lo, hi = prods.min(0).values, prods.max(0).values
        exact = ~amb
        assert same(G[exact], lo[exact]), f"{int((bits(G[exact]) != bits(lo[exact])).sum())} products differ ({n1}, {n2}, {R})"
        assert bool(((G >= lo) & (G <= hi)).all()), (n1, n2, R)
        assert same(G, G.T.contiguous()), f"G is not symmetric ({n1}, {n2}, {R})"
        worst_amb = max(worst_amb, float(amb.double().mean()))
    with capsys.disabled():
        print(f"\n[gram] {len(gram_pairs())} products, ambiguous share at most {worst_amb:.2e}", end="")



def unfold_shapes():
    return [s for s, _ in headline_layers()] + [(5, 7, 3), (13, 31, 9), (3, 129, 2)]


@pytest.mark.gpu
def test_unfold3_and_permute_myx():
    """Both are copies: bitwise equal to numpy.  permute_myx zeroes the pad columns [nx, ldv) of V."""
    nat = _nat()
    g = torch.Generator().manual_seed(5)
    for I, J, K in unfold_shapes():
        W = torch.randn(I, J, K, generator=g)
        Wd = W.cuda()
        Wn = W.numpy()
        for mode, (M, nx, ny) in enumerate(modes((I, J, K))):
            ref = np.ascontiguousarray(np.moveaxis(Wn, mode, 0)).reshape(M, nx * ny)
            buf, out = guarded(M * nx * ny)
            nat.check(nat.lib.admmq_unfold3(ptr(Wd), I, J, K, mode, ptr(out), stream()))
            assert guards_intact(buf)
            assert np.array_equal(out.view(M, nx * ny).cpu().numpy().view(np.int32), ref.view(np.int32)), ((I, J, K), mode)
            # V[(m, y), x] = Wn[m, x * ny + y], ld = nx rounded up to 4, written into a V full of NaN
            unf = torch.from_numpy(ref).cuda()
            ldv = (nx + 3) // 4 * 4
            vbuf, V = guarded(M * ny * ldv)
            nat.check(nat.lib.admmq_permute_myx(ptr(unf), M, nx, ny, ptr(V), stream()))
            assert guards_intact(vbuf)
            V = V.view(M * ny, ldv).cpu().numpy()
            vref = ref.reshape(M, nx, ny).transpose(0, 2, 1).reshape(M * ny, nx)
            assert np.array_equal(V[:, :nx].view(np.int32), vref.view(np.int32)), ((I, J, K), mode)
            assert np.array_equal(V[:, nx:].view(np.int32), np.zeros((M * ny, ldv - nx), np.int32)), ((I, J, K), mode)
            assert same(Wd, W.cuda())


def recon_problems():
    """(M, nx, ny, R) of the mode-0 reconstruction errors: every headline layer and the llama matrix."""
    out = [(s[0], s[1], s[2], R) for s, R in headline_layers()]
    M, nx, R = next(m for m in headline_matrices() if m[0] == 4096)
    return out + [(M, nx, 1, R), (65, 31, 3, 17)]


@pytest.mark.gpu
def test_recon_error(capsys):
    """out2 = {sum (W - rec)^2, sum W^2} with rec the float32 rounding of the float64 inner product over r, the difference
    and its square float32, the two sums float64 (csrc/contract.cu).  The kernel's and the reference's rec64 each lie
    within R u64 sum|terms| (+ one rounding) of the exact one; an element whose band holds a float32 rounding boundary
    may contribute either candidate's square.  The den sum must agree to 1e-13, the num sum to the ambiguous elements'
    spread plus 1e-13 (positive terms: both fixed-order float64 sums are within ~40 u64 of exact)."""
    nat = _nat()
    g = torch.Generator().manual_seed(41)
    worst = 0.0
    for M, nx, ny, R in recon_problems():
        A = (torch.randn(M, R, generator=g) / R ** 0.5).cuda()
        X = torch.randn(nx, R, generator=g).cuda()
        Y = torch.randn(ny, R, generator=g).cuda() if ny > 1 else None
        KR = X.double() if Y is None else (X.double()[:, None, :] * Y.double()[None, :, :]).reshape(nx * ny, R)
        rec64 = A.double() @ KR.T
        W0 = (rec64.float() + 0.1 * torch.randn(M, nx * ny, generator=g).cuda()).contiguous()
        band = (2 * R + 2) * U64 * (A.double().abs() @ KR.abs().T) * (1 + 1e-9)
        lo, hi = _rounding_candidates(rec64, band)
        sq = lambda rec: ((W0 - rec) * (W0 - rec)).double()   # noqa: E731  (float32 difference and square)
        num_ref = float(sq(rec64.float()).sum())
        den_ref = float((W0 * W0).double().sum())
        spread = float((sq(lo) - sq(hi)).abs().sum())
        need = nat.recon_error_workspace_bytes(M, nx, ny)
        out = torch.full((2,), float("nan"), dtype=torch.float64, device="cuda")
        sums = []
        for fill in (0xFF, 0):
            ws = torch.full((need,), fill, dtype=torch.uint8, device="cuda")
            nat.check(nat.lib.admmq_recon_error(ptr(W0), M, ptr(A), ptr(X), nx, None if Y is None else ptr(Y), ny, R,
                                                ptr(out), ptr(ws), need, stream()))
            sums.append(out.clone())
        assert same(sums[0], sums[1]), "the result depends on the workspace's previous contents"
        num, den = (float(v) for v in sums[0].cpu())
        assert abs(den - den_ref) <= 1e-13 * den_ref, (M, nx, ny, R, den, den_ref)
        assert abs(num - num_ref) <= spread + 1e-13 * num_ref, (M, nx, ny, R, num, num_ref, spread)
        worst = max(worst, abs(num - num_ref) / num_ref)
    with capsys.disabled():
        print(f"\n[recon] {len(recon_problems())} problems, worst relative num difference {worst:.2e}", end="")


@pytest.mark.gpu
def test_float64_initialisation_pieces():
    """mttkrp_f64 and gram_hadamard_f64 on every mode of one headline layer, against float64 torch on the device:
    the kernel's fixed-order sum of P terms (one rounding for the product X Y, P - 1 for the sums, one per slice) and
    the reference's (nx + ny + 3 roundings) stay within (P + nx + ny + splits + 4) u64 mag, which is below
    2 P u64 mag here.  normalize_columns_f64: norms within (n + 4) u64, zero columns untouched with norm 1, U divided
    and carry multiplied by exactly those norms."""
    nat = _nat()
    g = torch.Generator().manual_seed(51)
    shape, R = next((s, r) for s, r in headline_layers() if s == (256, 128, 9))
    facs = [torch.randn(d, R, generator=g, dtype=torch.float64).cuda() for d in shape]
    W = torch.randn(*shape, generator=g, dtype=torch.float64).cuda()
    for mode, (M, nx, ny) in enumerate(modes(shape)):
        others = [k for k in range(3) if k != mode]
        X, Y = facs[others[0]], facs[others[1]]
        Wn = W.movedim(mode, 0).reshape(M, nx * ny).contiguous()
        splits = nat.mttkrp_kernel(M, nx, ny, R, 0, _sm_count())[2]
        F = nat.mttkrp_f64(Wn, X, Y)
        mag = mttkrp64(Wn.abs(), X.abs(), Y.abs())
        bound = (nx * ny + nx + ny + splits + 4) * U64 * mag * (1 + 1e-9)
        assert bool(((F - mttkrp64(Wn, X, Y)).abs() <= bound).all()), mode
        assert nx * ny + nx + ny + splits + 4 <= 2 * nx * ny
        G = nat.gram_hadamard_f64(X, Y)
        gm = (X.abs().T @ X.abs()) * (Y.abs().T @ Y.abs())
        assert bool(((G - (X.T @ X) * (Y.T @ Y)).abs() <= (2 * (nx + ny) + 4) * U64 * gm * (1 + 1e-9)).all()), mode
    U = torch.randn(300, 37, generator=g, dtype=torch.float64).cuda()
    U[:, [0, 5, 36]] = 0.0
    U0 = U.clone()
    carry = torch.randn(37, generator=g, dtype=torch.float64).cuda()
    c0 = carry.clone()
    norms = nat.normalize_columns_f64(U, carry)
    ref = torch.linalg.vector_norm(U0, dim=0)
    zero = ref == 0
    assert bool((norms[zero] == 1).all()) and same(U[:, zero], U0[:, zero])
    assert bool(((norms[~zero] - ref[~zero]).abs() <= (300 + 4) * U64 * ref[~zero]).all())
    assert same(U, U0 / norms) and same(carry, c0 * norms)
