"""Every kernel of the ADMM inner loop (csrc/admm_loop*.cu*) against one float64 definition of an iteration.

`admmq_admm_loop_kernel` names the kernel a call runs (include/admmq.h, ADMMQ_LOOP_*).  The case list holds the factors
of the ResNet-18 headline at the SM budgets bench.py gives them, plus the edges of every kernel (empty CTAs of the
clusters, strip widths of the tap kernel, the shared-memory limits that switch kernels, every tensor-core tile width)
and every kernel with every scheme and bit width.

CPU: the case list reaches every kernel the query can return, and the headline factors map to the kernels listed in
HEADLINE_KERNELS.  GPU, per case:
  - one iteration against float64: the ridge product H_ls (recovered from the outputs as H' - (U' - U)) within a
    rounding-error bound of RHS . (G + rho I)^-1, the projection of V = H_ls - U (scale, clip candidate, codes) and
    the consistency of codes, H', U' and the reported residuals;
  - 30 calls of one iteration equal one call of 30 iterations bit for bit, the exit test stops at exactly the
    iteration it must, and admmq_admm_loop equals admmq_admm_iteration;
  - the kernel writes nothing outside H, U and codes, and a workspace full of 0xFF bytes gives the same bits as a
    zeroed one.
"""
import os
import re
from collections import namedtuple
from types import SimpleNamespace

import numpy as np
import pytest
import torch

REPO = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
MSE, MINMAX, SYM, AFFINE = "tensor_mseminmax_symmetric", "tensor_minmax", "tensor_symmetric", "tensor_affine"
U32 = 2.0 ** -24                 # unit roundoff of float32
STEPS = 30                       # iterations of the composition test

Case = namedtuple("Case", "I R precision budget scheme bits attempts")


def _kernel_ids():
    text = open(os.path.join(REPO, "include", "admmq.h")).read()
    return {k: int(v) for k, v in re.findall(r"#define ADMMQ_LOOP_(\w+) (\d+)", text)}


IDS = _kernel_ids()
TC = IDS["TC"]
TC_WIDTHS = range(16, 161, 16)
ALL_KERNELS = {v for k, v in IDS.items() if k != "TC"} | {TC + w for w in TC_WIDTHS}


def kernel_name(kid):
    if kid > TC:
        return f"TC{kid - TC}"
    return next(k for k, v in IDS.items() if v == kid)


def _nat():
    from source import _native
    return _native


def _sm_count():
    return torch.cuda.get_device_properties(0).multi_processor_count if torch.cuda.is_available() else 148


def _grid(budget, sms):
    return budget if 0 < budget < sms else sms


def kernel_of(case, sms):
    return _nat().loop_kernel(case.I, case.R, case.attempts, case.precision, _grid(case.budget, sms))


def headline_units(sms):
    """Distinct (shape, R, budget) of the ResNet-18 headline, budgets as bench.py gives them (cost-proportional, at
    least one SM each)."""
    import bench
    from source import workloads as wl
    units, _ = bench.workload_units(SimpleNamespace(workload="resnet18", reduction_rate=2.0, bits=4))
    shapes = [bench.unit_shape(u) for u in units]
    ranks = [bench.unit_rank(u) for u in units]
    budgets = bench.allocate_ctas([wl.solve_cost(s, r) for s, r in zip(shapes, ranks)], sms, 1)
    out = []
    for s, r, b in zip(shapes, ranks, budgets):
        if (s, r, b) not in out:
            out.append((s, r, b))
    return out


# what the headline factors run on at the budgets of a 148-SM B200 (precision 1; precision 0 takes the parity tiles)
HEADLINE_KERNELS = {
    ((64, 64, 9), 134, 1): ("RESIDENT", "RESIDENT", "RESIDENT"),
    ((128, 64, 9), 183, 1): ("TC96", "TC96", "SKINNY9"),
    ((128, 128, 9), 278, 2): ("TC144", "TC144", "SKINNY9"),
    ((256, 128, 9), 375, 3): ("TC128", "TC128", "SKINNY9"),
    ((256, 256, 9), 566, 7): ("TC96", "TC96", "SKINNY9"),
    ((512, 256, 9), 759, 14): ("TC112", "TC112", "SKINNY9"),
    ((512, 512, 9), 1141, 33): ("TC144", "TC144", "SKINNY9"),
}


def build_cases(sms):
    cases = []

    def add(I, R, precisions, budgets, scheme=MSE, bits=4, attempts=200):
        for p in precisions:
            for b in budgets:
                c = Case(I, R, p, b, scheme, bits, attempts)
                if c not in cases:
                    cases.append(c)

    for shape, R, b in headline_units(sms):
        for I in dict.fromkeys(shape):
            add(I, R, (1, 0), (b,))
    P12 = (1, 2)
    # shared-memory-resident kernel (budget 1)
    for I, R in ((1, 1), (3, 5), (64, 136), (17, 135)):
        add(I, R, P12, (1,))
    # clusters of 4 and 8: CTAs without rows, candidate counts
    add(1, 7, P12, (8,))
    add(3, 20, P12, (8,))
    for att in (1, 7, 1024):
        add(33, 77, P12, (4, 8), attempts=att)
    # tap cluster: last CTA without columns at R = 137 / 161, one row, the widest rank; 9 x 641 falls to the strips
    for I, R in ((9, 137), (9, 161), (1, 200), (9, 640), (9, 641)):
        add(I, R, P12, (8,))
    # column strips
    for I in (9, 10, 16):
        for R in (1, 3, 77, 1141):
            add(I, R, P12, (3,))
    add(9, 1141, P12, (2, 14, 148))
    add(16, 1024, P12, (3,))      # I * Rp == kRhsFloats: still the strips
    add(16, 1025, P12, (3,))      # one float4 more: FFMA tiles
    # float32 FFMA tiles
    add(200, 300, (2,), (2, 37, 148))
    add(63, 300, (1,), (37,))
    add(300, 31, (1,), (37,))
    # tensor cores: both thresholds, odd shapes, then one budget for every tile width
    add(64, 32, (1,), (2, 3))
    add(65, 33, (1,), (2,))
    add(129, 1141, (1,), (33, 148))
    nat = _nat()
    for w in TC_WIDTHS:
        if any(kernel_of(c, sms) == TC + w for c in cases):
            continue
        found = next(((I, R, b) for I, R in ((128, 183), (256, 375), (512, 759), (512, 1141), (129, 1141))
                      for b in range(1, sms + 1) if nat.loop_kernel(I, R, 200, 1, _grid(b, sms)) == TC + w), None)
        assert found is not None, f"no budget selects tile width {w}"
        add(found[0], found[1], (1,), (found[2],))
    # parity tiles of 64 and 32
    for I, R in ((65, 33), (200, 301)):
        for b in (1, 2, 148):
            add(I, R, (0,), (b,))
    # every kernel with every scheme and with 1, 2, 4 and 8 bits, on its smallest case of at least 64 elements (a
    # factor of one element has min == max: the minmax and affine grids degenerate)
    by_kernel = {}
    size = lambda c: (c.I * c.R < 64, c.I * c.R)   # noqa: E731
    for c in cases:
        k = kernel_of(c, sms)
        if k not in by_kernel or size(c) < size(by_kernel[k]):
            by_kernel[k] = c
    for k, c in sorted(by_kernel.items()):
        for scheme in (MINMAX, SYM, AFFINE):
            add(c.I, c.R, (c.precision,), (c.budget,), scheme=scheme, attempts=c.attempts)
        for bits in (1, 2, 8):
            add(c.I, c.R, (c.precision,), (c.budget,), bits=bits, attempts=c.attempts)
    return cases


CASES = build_cases(_sm_count())


def case_id(c):
    return f"{c.I}x{c.R}-p{c.precision}-b{c.budget}-{c.scheme.split('_')[1]}{c.bits}-n{c.attempts}"


# ------------------------------------------------------------------------------------------------ CPU
def test_case_list_reaches_every_kernel():
    sms = 148
    reached = {kernel_of(c, sms) for c in build_cases(sms)}
    assert reached == ALL_KERNELS, sorted(kernel_name(k) for k in ALL_KERNELS ^ reached)
    # and every kernel with every scheme and bit width
    combos = {(kernel_of(c, sms), c.scheme, c.bits) for c in build_cases(sms)}
    for k in ALL_KERNELS:
        for s in (MSE, MINMAX, SYM, AFFINE):
            assert (k, s, 4) in combos, (kernel_name(k), s)
        for bits in (1, 2, 4, 8):
            assert (k, MSE, bits) in combos, (kernel_name(k), bits)


def test_headline_factors_run_on_the_published_kernels():
    units = headline_units(148)
    assert {(s, r, b) for s, r, b in units} == set(HEADLINE_KERNELS)
    nat = _nat()
    for (shape, R, b), names in HEADLINE_KERNELS.items():
        got = tuple(kernel_name(nat.loop_kernel(I, R, 200, 1, b)) for I in shape)
        assert got == names, (shape, R, b, got)
        par = {kernel_name(nat.loop_kernel(I, R, 200, 0, b)) for I in shape}
        assert par <= {"F64_64", "F64_32"}, (shape, R, b, par)


def test_kernel_query_edges():
    nat = _nat()
    k = lambda I, R, p, g, n=200: kernel_name(nat.loop_kernel(I, R, n, p, g))   # noqa: E731
    assert k(64, 136, 1, 1) == "RESIDENT" and k(64, 137, 1, 1) != "RESIDENT"
    assert k(33, 77, 1, 4) == "CLUSTER4" and k(33, 77, 1, 8) == "CLUSTER8" and k(33, 77, 1, 148) == "CLUSTER8"
    assert k(33, 77, 1, 2).startswith("FFMA")
    assert k(9, 640, 1, 8) == "TAP" and k(9, 641, 1, 8) == "SKINNY9" and k(9, 640, 1, 7) == "SKINNY9"
    assert k(16, 1024, 1, 3) == "SKINNY16" and k(16, 1025, 1, 3).startswith("FFMA")
    assert k(64, 32, 1, 2) == "TC16" and k(63, 32, 1, 2).startswith("FFMA") and k(64, 31, 1, 2).startswith("FFMA")
    assert k(64, 32, 2, 2).startswith("FFMA") and k(9, 134, 0, 1) in ("F64_64", "F64_32")
    assert k(33, 77, 1, 8, 1025) != "CLUSTER8"
    with pytest.raises(ValueError):
        nat.loop_kernel(0, 5, 200, 1, 1)
    with pytest.raises(ValueError):
        nat.loop_kernel(5, 5, 200, 3, 1)


# ------------------------------------------------------------------------------------------------ reference pieces
def _f32(x):
    return np.asarray(x, dtype=np.float32)


def _levels(bits):
    q = 2 ** (bits - 1)
    return q, 2 * q - 1


def _codes(x, scheme, bits, scale, aux):
    """Integer codes of the kernels' projection (include/admmq.h) of float32 x for a given scale and aux (minmax: the
    minimum; affine: the zero point).  Every one is monotone in x."""
    q, denom = _levels(bits)
    x = _f32(x)
    s = np.float32(scale)
    if scheme in (MSE, SYM):
        return np.clip(np.rint(x / s), -q, q - 1)
    if scheme == AFFINE:
        return np.clip(np.rint(x / s) + np.float32(aux), -q, q - 1)
    if bits == 1:
        return np.sign(x)
    n = np.float32(2 ** bits - 1)
    unit = (x - np.float32(aux)) / s
    return np.floor(unit * n + np.float32(0.5)) - q


def _values(codes, scheme, bits, scale, aux):
    """H of the codes under the scheme's code convention."""
    c = _f32(codes)
    s = np.float32(scale)
    if scheme in (MSE, SYM):
        return c * s
    if scheme == AFFINE:
        return (c - np.float32(aux)) * s
    if bits == 1:
        return c - np.float32(1.0)
    q = np.float32(2 ** (bits - 1))
    n = np.float32(2 ** bits - 1)
    return (c + q) * s / n + np.float32(aux)


def _problem(case, seed):
    """Seeded H, U, F and a Gram-Hadamard G (float32, CPU) with H_ls of order one."""
    g = torch.Generator().manual_seed(seed)
    I, R = case.I, case.R
    B, C = torch.randn(96, R, generator=g), torch.randn(9, R, generator=g) / 3
    G = (B.T @ B) * (C.T @ C)
    F = (torch.randn(I, R, generator=g) @ G).contiguous()
    H = torch.randn(I, R, generator=g)
    U = torch.randn(I, R, generator=g) * 0.1
    return H, U, F, G


def _bound_factor(kid, R):
    """|H_ls(kernel) - H_ls(float64)| <= factor * (|RHS| . |Minv|), elementwise (u = 2^-24):
      parity tiles: float64 products and sums against the float64 inverse, one rounding to float32: 4 u;
      cluster: float64 products and sums against the float32 inverse (u per element) plus the output rounding: 4 u;
      float32 FFMA (resident, tap, strips, tiles): at most R + 16 roundings on the path of any product (an FMA chain
        over k plus the fixed-order sums of the partial results), plus the float32 inverse: (R + 20) u;
      3xTF32 on tcgen05: the split of both operands into tf32 hi + lo drops lo.lo and rounds the lo parts (3 * 2^-22 =
        12 u per product); an accumulator update of the MMA may truncate (1 ulp = 2 u), and a product passes at most
        3 * ceil(R / 8) of them plus the sums inside an MMA: (R + 48) u."""
    if kid in (IDS["F64_64"], IDS["F64_32"], IDS["CLUSTER4"], IDS["CLUSTER8"]):
        return 4 * U32
    if kid > TC:
        return (R + 48) * U32
    return (R + 20) * U32


def _spacing(x):
    return np.spacing(np.abs(_f32(x))).astype(np.float64)


def check_one_step(case, kid, H0, U0, F, G, H1, U1, codes, rep):
    """The float64 reference of one iteration; returns (worst ratio to the ridge bound, ambiguous share, mismatches)."""
    I, R, bits, scheme = case.I, case.R, case.bits, case.scheme
    q, denom = _levels(bits)
    H0, U0, F, G = (t.numpy() for t in (H0, U0, F, G))
    H1, U1, codes = H1.cpu().numpy(), U1.cpu().numpy(), codes.cpu().numpy().astype(np.float32)
    tr = np.float32(np.trace(G.astype(np.float64)))
    rho = np.float32(rep.rho)                               # trace(G) / R as the kernel summed it
    assert abs(rho - np.float32(tr / np.float32(R))) <= np.spacing(rho), (rep.rho, tr / R)
    rhs = F + rho * (H0 + U0)                                                  # float32, the kernels' own formula
    A = G.astype(np.float64)
    A[np.diag_indices(R)] = (np.diag(G) + rho).astype(np.float64)            # G + rho I as float32, then widened
    Minv = np.linalg.inv(A)
    hls64 = rhs.astype(np.float64) @ Minv
    mag = np.abs(rhs.astype(np.float64)) @ np.abs(Minv)
    # the kernel's H_ls from its outputs: U' = fl(U + fl(H' - H_ls)) -> H_ls = H' - (U' - U) up to two half-ulps
    du = U1.astype(np.float64) - U0.astype(np.float64)
    hls_k = H1.astype(np.float64) - du
    delta = _spacing(U1) + _spacing(du)
    # 1. ridge product
    bound = _bound_factor(kid, R) * mag + delta
    ratio = float(np.max(np.abs(hls_k - hls64) / bound))
    assert ratio <= 1.0, f"ridge product off by {ratio:.3g} x its bound"
    # 2. projection of V = fl(H_ls - U) (kernel's V within band of v64)
    v64 = hls_k - U0.astype(np.float64)
    band = delta + _spacing(v64)
    absmax = np.float32(rep.absmax)
    # where V is the reported extreme it is known exactly (tensor_symmetric puts it on a rounding boundary: a tie)
    ext = np.abs(_f32(v64)) == absmax
    v64, band = np.where(ext, np.sign(v64) * float(absmax), v64), np.where(ext, 0.0, band)
    v32 = _f32(v64)
    assert abs(float(absmax) - float(np.max(np.abs(v64)))) <= float(np.max(band)), (rep.absmax, np.max(np.abs(v64)))
    vmin, vmax = np.float32(v32.min()), np.float32(v32.max())
    if -vmin == absmax:
        tmin, tmax = -absmax, vmax
    elif vmax == absmax:
        tmin, tmax = vmin, absmax
    else:                                                   # extreme not recovered exactly: take the nearer one
        tmin, tmax = (-absmax, vmax) if abs(-vmin - absmax) < abs(vmax - absmax) else (vmin, absmax)
    scale = np.float32(rep.scale)
    aux = np.float32(0.0)
    ext_tol = 2 * float(np.max(band))
    if scheme == MSE:
        from oracle import admm_oracle as orc
        clip = orc.candidate_grid(float(absmax), case.attempts)
        assert 0 <= rep.best_index < case.attempts
        assert scale == np.float32(np.float32(2 * clip[rep.best_index]) / np.float32(denom)), (scale, rep.best_index)
        _, _, _, ref_best, mses = orc.project_mse(torch.from_numpy(v32.copy()), bits, case.attempts, "exact")
        if rep.best_index != ref_best:
            gap = abs(float(mses[rep.best_index]) - float(mses[ref_best])) / float(mses[ref_best])
            assert gap < 3e-7, (rep.best_index, ref_best, gap)
    elif scheme == SYM:
        assert rep.best_index == -1
        assert scale == np.float32(np.float32(2 * absmax) / np.float32(denom)), (scale, absmax)
    elif scheme == MINMAX:
        assert abs(float(scale) - float(np.float32(tmax - tmin))) <= ext_tol + float(_spacing(scale)), (scale, tmin, tmax)
        if bits > 1:   # the minimum itself has level 0, whose value is the minimum: aux exactly
            lows = H1[codes == -q]
            assert lows.size > 0 and np.all(lows == lows[0])
            aux = np.float32(lows[0])
            assert abs(float(aux) - float(tmin)) <= ext_tol
    else:
        assert abs(float(scale) - float(np.float32((tmax - tmin) / np.float32(denom)))) <= ext_tol + float(_spacing(scale))
        aux = np.float32(np.clip(np.trunc(np.float32(-q) - np.trunc(np.float32(tmin) / scale)), -q, q - 1))
    outward = lambda x, to: np.where(band > 0, np.nextafter(_f32(x), np.float32(to)), v32)   # noqa: E731
    lo = _codes(outward(v64 - band, -np.inf), scheme, bits, scale, aux)
    hi = _codes(outward(v64 + band, np.inf), scheme, bits, scale, aux)
    ambiguous = lo != hi
    amb_share = float(ambiguous.mean())
    mismatches = int(np.count_nonzero((codes != lo) & ~ambiguous))
    assert mismatches == 0, f"{mismatches} codes differ from the exact projection of V"
    assert amb_share <= 1e-3, amb_share
    # 3. consistency: codes and H, the dual update, the residuals
    assert np.array_equal(_values(codes, scheme, bits, scale, aux), H1), "codes and H disagree"
    # U' = fl(U + fl(H' - h)) for a float32 h within two ulps of the recovered H_ls, on every element
    h = _f32(hls_k)
    for _ in range(2):
        h = np.nextafter(h, np.float32(-np.inf))
    dual_ok = np.zeros(h.shape, dtype=bool)
    for _ in range(5):
        dual_ok |= (U0 + (H1 - h)) == U1
        h = np.nextafter(h, np.float32(np.inf))
    assert dual_ok.all(), f"{int((~dual_ok).sum())} elements of U' are not U + (H' - H_ls)"
    h64, h0 = H1.astype(np.float64), H0.astype(np.float64)
    r64 = float(np.sum((h64 - hls_k) ** 2) / np.sum(h64 ** 2))
    s64 = float(np.sum((h64 - h0) ** 2) / np.sum(U1.astype(np.float64) ** 2))
    assert abs(rep.r - r64) <= 1e-3 * r64 and abs(rep.s - s64) <= 1e-3 * s64, (rep.r, r64, rep.s, s64)
    return ratio, amb_share, mismatches


def _state(H, U, codes):
    return H.clone(), U.clone(), codes.clone()


def _equal(a, b):
    return all(torch.equal(x.view(torch.uint8) if x.dtype != torch.int8 else x,
                           y.view(torch.uint8) if y.dtype != torch.int8 else y) for x, y in zip(a, b))


# ------------------------------------------------------------------------------------------------ GPU
@pytest.mark.gpu
@pytest.mark.parametrize("case", CASES, ids=[case_id(c) for c in CASES])
def test_loop_kernel(case, capsys):
    nat = _nat()
    sms = _sm_count()
    kid = kernel_of(case, sms)
    seed = 1000 + CASES.index(case)
    H0, U0, F, G = _problem(case, seed)
    I, R, p, b, scheme, bits, na = case.I, case.R, case.precision, case.budget, case.scheme, case.bits, case.attempts
    d = lambda t: t.cuda().contiguous()   # noqa: E731
    Fd, Gd = d(F), d(G)
    # ---- b. one iteration against float64
    H, U = d(H0), d(U0)
    codes = torch.empty(I, R, dtype=torch.int8, device="cuda")
    rep = nat.read_report(nat.admm_iteration_inplace(H, U, Fd, Gd, 2, 0.0, bits, scheme, na, codes=codes, precision=p,
                                                     max_ctas=b))
    assert rep.iterations == 1 and rep.status == 0, (rep.iterations, rep.status)
    ratio, amb, mism = check_one_step(case, kid, H0, U0, F, G, H, U, codes, rep)
    # ---- c. composition: STEPS calls of one iteration == one call of STEPS iterations, bit for bit
    inv = nat.spd_inverse(Gd, minv64=True, max_ctas=b)
    Minv, rho, st, m64 = inv
    m64 = m64 if p == 0 else None
    ws = torch.empty(nat.admm_loop_workspace_bytes(I, R, na), dtype=torch.uint8, device="cuda")

    def loop(Hx, Ux, cx, iters, eps, workspace=ws):
        r = nat.admm_loop_inplace(Hx, Ux, Fd, Minv, rho, st, iters + 1, eps, bits, scheme, na, codes=cx, ws=workspace,
                                  precision=p, max_ctas=b, minv64=m64)
        return nat.read_report(r)

    H, U = d(H0), d(U0)
    codes = torch.empty(I, R, dtype=torch.int8, device="cuda")
    snaps, reps = [], []
    for _ in range(STEPS):
        reps.append(loop(H, U, codes, 1, 0.0))
        snaps.append(_state(H, U, codes))
    Hk, Uk = d(H0), d(U0)
    ck = torch.empty(I, R, dtype=torch.int8, device="cuda")
    rk = loop(Hk, Uk, ck, STEPS, 0.0)
    last = reps[-1]
    assert rk.iterations == STEPS
    assert _equal((Hk, Uk, ck), snaps[-1]), f"{STEPS} iterations in one call differ from {STEPS} single calls"
    assert (rk.r, rk.s, rk.scale, rk.best_index) == (last.r, last.s, last.scale, last.best_index)
    # exit at exactly iteration j: the last strict record low of max(r, s) before the last iteration (the cluster and
    # tap kernels test iteration j after the first barrier of iteration j + 1)
    m = [max(x.r, x.s) for x in reps]
    j = max(i for i in range(STEPS - 1) if all(m[i] < m[k] for k in range(i)))
    eps = float(np.nextafter(np.float32(m[j]), np.float32(np.inf)))
    He, Ue = d(H0), d(U0)
    ce = torch.empty(I, R, dtype=torch.int8, device="cuda")
    re_ = loop(He, Ue, ce, STEPS, eps)
    assert re_.iterations == j + 1 and re_.status & nat.ST_CONVERGED, (re_.iterations, j + 1, re_.status)
    assert _equal((He, Ue, ce), snaps[j]), "the exit left another state than the single steps"
    # admmq_admm_loop == admmq_admm_iteration
    Hi, Ui = d(H0), d(U0)
    ci = torch.empty(I, R, dtype=torch.int8, device="cuda")
    ri = nat.read_report(nat.admm_iteration_inplace(Hi, Ui, Fd, Gd, STEPS + 1, 0.0, bits, scheme, na, codes=ci,
                                                    precision=p, max_ctas=b))
    assert _equal((Hi, Ui, ci), (Hk, Uk, ck)) and ri.iterations == STEPS
    # ---- d. memory hygiene: guards around H, U, codes; F, G untouched; a 0xFF workspace gives the same bits
    gd = 64
    sentinel = torch.tensor([0x7FA5A5A5], dtype=torch.int32).view(torch.float32).item()
    Hb = torch.full((I * R + 2 * gd,), sentinel, device="cuda")
    Ub = Hb.clone()
    cb = torch.full((I * R + 2 * gd * 4,), 0x5A, dtype=torch.int8, device="cuda")
    Hg, Ug = Hb[gd:gd + I * R].view(I, R), Ub[gd:gd + I * R].view(I, R)
    cg = cb[gd * 4:gd * 4 + I * R].view(I, R)
    Hg.copy_(d(H0))
    Ug.copy_(d(U0))
    F_before, G_before = Fd.clone(), Gd.clone()
    ws.fill_(0xFF)
    loop(Hg, Ug, cg, 3, 0.0)
    for buf in (Hb, Ub):
        assert _equal((buf[:gd], buf[-gd:]), (torch.full((gd,), sentinel, device="cuda"),) * 2), "guard overwritten"
    assert bool((cb[:gd * 4] == 0x5A).all()) and bool((cb[-gd * 4:] == 0x5A).all()), "codes guard overwritten"
    assert _equal((Fd, Gd), (F_before, G_before)), "F or G changed"
    ws.zero_()
    Hz, Uz = d(H0), d(U0)
    cz = torch.empty(I, R, dtype=torch.int8, device="cuda")
    loop(Hz, Uz, cz, 3, 0.0)
    assert _equal((Hg, Ug, cg), (Hz, Uz, cz)), "the result depends on the workspace's previous contents"
    with capsys.disabled():
        print(f"\n[loop] {case_id(case)} {kernel_name(kid)}: ridge error {ratio:.3f} of bound, ambiguous "
              f"{amb:.2e}, code mismatches {mism}, exit at {j + 1}", end="")
