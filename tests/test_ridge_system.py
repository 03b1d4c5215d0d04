"""The ridge-system inverse `k_spd_inverse` (csrc/spd_inverse.cuh) against float64, and its failure path through every
caller.

`admmq_spd_inverse` forms rho = trace(G) / R and A = fl32(G + rho I), factors A by a blocked float64 Cholesky on a
cooperative grid and writes Minv (float32) and Minv64 (float64).  The case list holds every (R, budget) pair bench.py
gives the inverse on a 148-SM B200, the ranks where the 32-wide tiles and the padded leading dimension have their
edges, the grids around the panel count, and six kinds of G from well to badly conditioned.

CPU: the case list holds every benchmark pair and every edge; the kinds of G span the conditioning they claim; the
reference tells a float64-formed diagonal apart from the right one; every failing system fails torch.linalg.cholesky.
GPU, per case: Minv64 within tau = 4 R kappa 2^-53 |X|max of X = cho_solve(A); Minv == fl32(Minv64); both bitwise
symmetric with +0.0 pad columns; rho == torch.trace(G) / R bitwise; the same bits at every grid, after a scaling of G
by 4^+-20 (scaled back) and with NaN above the diagonal of G; nothing written outside the outputs and no dependence on
the previous contents of the outputs, the status word or the workspace.
Failure path: G = 0, a NaN below the diagonal at every panel, +Inf on the diagonal and a negative last pivot set the
status at every grid and leave rho written; a good call afterwards resets the status; every loop kernel leaves H, U and
codes untouched when the status is set; LayerSolver, admm_iteration, factorize and factorize_batch raise LinAlgError.
"""
import ctypes
import sys
from collections import namedtuple
from types import SimpleNamespace

import numpy as np
import pytest
import scipy.linalg
import torch

import test_loop_kernels as tlk

MSE = "tensor_mseminmax_symmetric"
U64 = 2.0 ** -53                 # unit roundoff of float64
EDGE_RANKS = (1, 2, 3, 4, 5, 31, 32, 33, 63, 64, 65, 96, 97, 160)
ABOVE = 4096                     # a max_ctas no device can hold co-resident: the call only launches if it clamps
KINDS = ("gram", "solver", "mean", "rank1", "dead", "diag")
KIND_RANKS = (2, 33, 97, 134, 1141, 1522)        # ranks of the kinds other than "gram" and "solver"
SOLVER_LAYERS = ("layer1.0.conv1", "layer4.1.conv2")   # headline layers whose G snapshots are taken
NB = 32                          # tile edge of the blocked factorization (csrc/spd_inverse.cuh kNB)

Case = namedtuple("Case", "R kind grids src")


def _nat():
    from source import _native
    return _native


def _bench_args(workload):
    """bench.py's defaults for `workload` (reduction rate, bits, round size)."""
    import bench
    argv = sys.argv
    sys.argv = ["bench.py"]
    try:
        args = bench.parse_args()
    finally:
        sys.argv = argv
    args.workload = workload
    return args


def bench_pairs(sms):
    """{(R, budget): shape} for every distinct pair bench.py gives the inverse on `sms` SMs: the concurrent workloads
    with budgets proportional to solve_cost (run_native), and sweep256 in rounds of --round-size units in LPT order by
    unit_cost (run_sweep256).  The shape is the first layer of that rank (the kind "gram" takes its initial factors)."""
    import bench
    from source import workloads as wl
    out = {}
    for name in ("resnet18", "resnet50-l4", "llama7b"):
        units, _ = bench.workload_units(_bench_args(name))
        shapes = [bench.unit_shape(u) for u in units]
        ranks = [bench.unit_rank(u) for u in units]
        budgets = bench.allocate_ctas([wl.solve_cost(s, r) for s, r in zip(shapes, ranks)], sms, 1)
        for s, r, b in zip(shapes, ranks, budgets):
            out.setdefault((r, b), s)
    args = _bench_args("sweep256")
    units, _ = bench.workload_units(args)
    jobs = [(bench.unit_shape(u), bench.unit_rank(u), u[7]) for u in units]
    jobs = sorted(jobs, key=lambda j: -wl.unit_cost(j[0], j[1], j[2]))
    for i in range(0, len(jobs), args.round_size):
        rd = jobs[i:i + args.round_size]
        for (s, r, _), b in zip(rd, bench.allocate_ctas([wl.unit_cost(s, r, bits) for s, r, bits in rd], sms, 1)):
            out.setdefault((r, b), s)
    return out


def standard_grids(R, sms):
    nb = -(-R // NB)
    return {g for g in (1, 2, nb - 1, nb, nb + 1, sms, ABOVE) if g >= 1}


def build_cases(sms):
    pairs = bench_pairs(sms)
    shape_of, budgets = {}, {}
    for (r, b), s in pairs.items():
        shape_of.setdefault(r, s)
        budgets.setdefault(r, set()).add(b)
    cases = []
    for R in sorted(set(shape_of) | set(EDGE_RANKS)):
        grids = sorted(standard_grids(R, sms) | budgets.get(R, set()))
        cases.append(Case(R, "gram", tuple(grids), shape_of.get(R, (64, 512, 9))))
    import bench
    units, _ = bench.workload_units(_bench_args("resnet18"))
    headline = {(s, r): b for s, r, b in tlk.headline_units(sms)}
    for name in SOLVER_LAYERS:
        u = next(u for u in units if u[1] == name)
        R = bench.unit_rank(u)
        cases.append(Case(R, "solver", (headline[bench.unit_shape(u), R], sms), name))
    for kind in ("mean", "rank1", "dead", "diag"):
        for R in KIND_RANKS:
            nb = -(-R // NB)
            cases.append(Case(R, kind, tuple(sorted({1, 2, nb, sms})), (64, 512, 9)))
    return cases


CASES = build_cases(tlk._sm_count())


def case_id(c):
    return f"R{c.R}-{c.kind}" + (f"-{c.src}" if c.kind == "solver" else "")


# ------------------------------------------------------------------------------------------------ G of every kind
def _gram(U1, U2=None):
    """(U1^T U1) * (U2^T U2): the native kernel on CUDA tensors, float64 rounded to float32 on the CPU."""
    if U1.is_cuda:
        return _nat().gram_hadamard(U1, U2)
    g = U1.double().T @ U1.double()
    if U2 is not None:
        g = g * (U2.double().T @ U2.double())
    return g.float()


def make_g(kind, shape, R, seed, device="cpu"):
    """G (float32, on `device`) of one kind; mode 0 of a layer of `shape`:
      gram  - the benchmark's random initial factors (bench.py: random_init with seed 42), kappa 3 .. 5 at its ranks;
      mean  - factors 1 + 0.3 randn: a common mean, kappa in the hundreds;
      rank1 - every column one vector plus 1e-3 noise: kappa close to R + 1;
      dead  - the gram factors with one zero column: a zero row and column of G;
      diag  - diag(2^24, 1, ..., 1), whose float32 running trace (2^24) differs from the float64 one."""
    from source import workloads as wl
    if kind == "diag":
        G = torch.eye(R)
        G[0, 0] = 2.0 ** 24
        return G.to(device)
    g = torch.Generator().manual_seed(seed)
    if kind == "gram":
        fac = wl.random_init(shape, R, 42)[1:]
    elif kind == "mean":
        fac = [1.0 + 0.3 * torch.randn(d, R, generator=g) for d in shape[1:]]
    elif kind == "rank1":
        fac = [torch.randn(d, 1, generator=g) + 1e-3 * torch.randn(d, R, generator=g) for d in shape[1:]]
    elif kind == "dead":
        fac = wl.random_init(shape, R, 42)[1:]
        fac[0][:, R // 2] = 0.0
    else:
        raise ValueError(kind)
    fac = [f.to(device) for f in fac]
    return _gram(fac[0], fac[1] if len(fac) > 1 else None)


# ------------------------------------------------------------------------------------------------ reference
def rho_of(G):
    """rho as the reference forms it (source/admm.py:53): ATen's CPU trace (accumulated in double), over R, in float32."""
    Gt = torch.as_tensor(G).cpu()
    return np.float32((torch.trace(Gt) / Gt.shape[0]).item())


def ridge_matrix(G, rho, f64_diagonal=False):
    """A64 = float64(fl32(G + rho I)): off-diagonal G_ij, diagonal fl32(G_ii + rho).  f64_diagonal forms the diagonal
    as G_ii + rho in float64 instead (the error the reference must catch)."""
    G = np.asarray(G, dtype=np.float32)
    A = G.astype(np.float64)
    d = np.diag(G).astype(np.float64) + float(rho) if f64_diagonal else (np.diag(G) + np.float32(rho)).astype(np.float64)
    A[np.diag_indices(G.shape[0])] = d
    return A


def reference(A):
    """(X, kappa, tau): X = A^-1 by LAPACK's Cholesky, kappa from the eigenvalues and tau = 4 R kappa 2^-53 |X|max, the
    Cholesky-inverse bound that covers both the kernel's error and LAPACK's."""
    R = A.shape[0]
    X = scipy.linalg.cho_solve(scipy.linalg.cho_factor(A, lower=True), np.eye(R))
    ev = scipy.linalg.eigvalsh(A)
    kappa = float(ev[-1] / ev[0])
    return X, kappa, 4.0 * R * kappa * U64 * float(np.abs(X).max())


# ------------------------------------------------------------------------------------------------ failing systems
FAIL_RANKS = (134, 1141)


def failing_systems(R):
    """[(name, panel where the factorization must fail)]: G = 0 (rho = 0), a NaN at G[r, 0] and G[0, r] (a NaN in a
    factor would poison the diagonal and rho: only an off-diagonal NaN reaches a later panel), +Inf on the diagonal,
    and a last pivot made negative by scaling the coupling of the last row and column."""
    out = [("zero", 0), ("inf", 0), ("negative-last-pivot", (R - 1) // NB)]
    out += [(f"nan-{r}", r // NB) for r in (1, 31, 32, 33, R - 1)]
    return out


def failing_g(name, R):
    G = make_g("gram", (64, 512, 9), R, 0).numpy().copy()
    if name == "zero":
        G[:] = 0.0
    elif name == "inf":
        G[R // 3, R // 3] = np.inf
    elif name.startswith("nan-"):
        r = int(name[4:])
        G[r, 0] = G[0, r] = np.nan
    else:   # scale the last coupling so that the Schur complement of the last pivot is about -A_nn
        A = ridge_matrix(G, rho_of(G))
        a = A[:-1, -1]
        q = float(a @ np.linalg.solve(A[:-1, :-1], a))
        c = np.float32(np.sqrt(2.0 * A[-1, -1] / q))
        G[:-1, -1] *= c
        G[-1, :-1] *= c
    return torch.from_numpy(G)


def last_pivot(A):
    n = A.shape[0] - 1
    return A[n, n] - A[:n, n] @ np.linalg.solve(A[:n, :n], A[:n, n])


# ------------------------------------------------------------------------------------------------ CPU
def test_case_list_holds_every_benchmark_pair_and_edge():
    sms = 148
    cases = build_cases(sms)
    gram = {c.R: c for c in cases if c.kind == "gram"}
    pairs = bench_pairs(sms)
    for (R, b) in pairs:
        assert R in gram and b in gram[R].grids, (R, b)
    # the ranks the benchmark runs, as the documents state them
    ranks = {R for R, _ in pairs}
    assert min(ranks) == 67 and max(ranks) == 1522, sorted(ranks)
    assert {134, 183, 278, 375, 566, 759, 1141, 204, 1024, 1492} <= ranks
    # the headline's budgets of the largest and the smallest factor
    assert (1141, 33) in pairs and (134, 1) in pairs
    nat = _nat()
    assert set(EDGE_RANKS) <= set(gram)
    assert {R % NB for R in gram} >= {0, 1, NB - 1}
    assert {nat.lib.admmq_padded_ld(R) - R for R in EDGE_RANKS} == {0, 1, 2, 3}
    for R, c in gram.items():
        assert standard_grids(R, sms) <= set(c.grids) and ABOVE in c.grids, (R, c.grids)
    for R in (1, 33, 1141):
        assert {1, 2, sms, ABOVE} <= set(gram[R].grids)
    # every kind, and the kinds besides gram at one rank of every tile-fill edge and at the benchmark's extremes
    assert {c.kind for c in cases} == set(KINDS)
    for kind in ("mean", "rank1", "dead", "diag"):
        assert {c.R for c in cases if c.kind == kind} == set(KIND_RANKS)
    assert {c.src for c in cases if c.kind == "solver"} == set(SOLVER_LAYERS)


@pytest.mark.parametrize("R", (134, 1141))
def test_kinds_span_the_conditioning(R):
    kappa = {}
    for kind in ("gram", "mean", "rank1", "dead", "diag"):
        G = make_g(kind, (64, 512, 9), R, 7).numpy()
        assert np.array_equal(G, G.T), kind
        kappa[kind] = reference(ridge_matrix(G, rho_of(G)))[1]
        if kind == "dead":
            assert not G[R // 2].any() and not G[:, R // 2].any()
    assert 2.0 < kappa["gram"] < 10.0 and 2.0 < kappa["dead"] < 10.0, kappa
    assert 100.0 < kappa["mean"] < 2000.0, kappa
    assert 0.9 * (R + 1) < kappa["rank1"] <= (R + 1) * (1 + 1e-6), kappa
    assert 0.9 * (R + 1) < kappa["diag"] <= (R + 1) * (1 + 1e-6), kappa


def test_diag_kind_pins_the_double_accumulated_trace():
    G = make_g("diag", None, 134, 0)
    run32 = np.float32(0.0)
    for v in np.diag(G.numpy()):
        run32 = np.float32(run32 + v)
    exact = np.float32(np.trace(G.numpy().astype(np.float64)))
    assert run32 != exact
    assert np.float32(torch.trace(G).item()) == exact
    assert rho_of(G) == np.float32(exact / np.float32(134))


@pytest.mark.parametrize("R,kind", [(134, "gram"), (1141, "gram"), (1522, "gram"), (1141, "mean"), (1522, "rank1")])
def test_reference_catches_a_float64_diagonal(R, kind):
    """fl32(G_ii + rho) against G_ii + rho in float64: the inverses differ by far more than tau, so the check sees a
    kernel that forms the diagonal in float64."""
    G = make_g(kind, (64, 512, 9), R, 3).numpy()
    rho = rho_of(G)
    X, _, tau = reference(ridge_matrix(G, rho))
    Xw = reference(ridge_matrix(G, rho, f64_diagonal=True))[0]
    assert np.abs(Xw - X).max() > 10.0 * tau, (np.abs(Xw - X).max(), tau)


@pytest.mark.parametrize("R", FAIL_RANKS)
def test_failing_systems_fail_on_the_cpu(R):
    for name, panel in failing_systems(R):
        G = failing_g(name, R)
        rho = torch.trace(G) / R
        A = G + rho * torch.eye(R)
        with pytest.raises(torch.linalg.LinAlgError):
            torch.linalg.cholesky(A)
        assert 0 <= panel < -(-R // NB)
        if name == "negative-last-pivot":
            assert torch.equal(torch.diagonal(G), torch.diagonal(make_g("gram", (64, 512, 9), R, 0)))
            A64 = ridge_matrix(G.numpy(), rho_of(G))
            torch.linalg.cholesky(torch.from_numpy(A64[:-1, :-1]))   # the leading minor is positive definite
            assert last_pivot(A64) < -0.5 * A64[-1, -1]


def test_nan_above_the_diagonal_is_not_read_by_the_reference():
    G = make_g("gram", (64, 512, 9), 40, 0)
    A = G + (torch.trace(G) / 40) * torch.eye(40)
    up = A.clone()
    up[torch.triu(torch.ones(40, 40, dtype=torch.bool), 1)] = float("nan")
    assert torch.equal(torch.linalg.cholesky(up), torch.linalg.cholesky(A))
    lo = A.clone()
    lo[39, 0] = float("nan")
    with pytest.raises(torch.linalg.LinAlgError):
        torch.linalg.cholesky(lo)


# ------------------------------------------------------------------------------------------------ GPU helpers
GUARD = 64
F32_GUARD = 0x7FA5A5A5                 # a NaN payload the kernel never writes
F64_GUARD = 0x7FF5A5A5A5A5A5A5
STATUS_GARBAGE = 0x5EADBEEF


class Guarded:
    """A tensor of `n` elements between GUARD guard words, prefilled with a fill pattern."""

    def __init__(self, n, dtype, guard, fill):
        ity = {torch.float32: torch.int32, torch.float64: torch.int64, torch.int32: torch.int32}[dtype]
        self.raw = torch.full((n + 2 * GUARD,), guard, dtype=ity, device="cuda")
        self.raw[GUARD:GUARD + n] = fill
        self.guard, self.n, self.dtype = guard, n, dtype
        self.t = self.raw.view(dtype)[GUARD:GUARD + n]

    def guards_intact(self):
        return bool((self.raw[:GUARD] == self.guard).all()) and bool((self.raw[-GUARD:] == self.guard).all())


def run_inverse(G, grid, ws_fill=0x00, ws=None, status=None, minv64=True):
    """One admmq_spd_inverse into NaN-filled, guarded outputs and a status word prefilled with garbage.  Returns
    (Minv, Minv64 or None, rho, status, the guarded buffers)."""
    nat = _nat()
    R = G.shape[0]
    ld = nat.lib.admmq_padded_ld(R)
    nan32 = 0x7FC00000
    nan64 = 0x7FF8000000000000
    M = Guarded(R * ld, torch.float32, F32_GUARD, nan32)
    M64 = Guarded(R * ld, torch.float64, F64_GUARD, nan64) if minv64 else None
    rho = Guarded(1, torch.float32, F32_GUARD, nan32)
    st = Guarded(1, torch.int32, F32_GUARD, STATUS_GARBAGE) if status is None else status
    if ws is None:
        ws = torch.full((nat.spd_inverse_workspace_bytes(R),), ws_fill, dtype=torch.uint8, device="cuda")
    nat.spd_inverse(G, out=(M.t.view(R, ld), rho.t, st.t), ws=ws, max_ctas=grid,
                    minv64=None if M64 is None else M64.t.view(R, ld))
    torch.cuda.synchronize()
    return M.t.view(R, ld), None if M64 is None else M64.t.view(R, ld), rho.t, st.t, (M, M64, rho, st)


def bits(t):
    t = t.detach().cpu().contiguous()
    return t.view({torch.float32: torch.int32, torch.float64: torch.int64, torch.int32: torch.int32}[t.dtype])


def same_bits(a, b):
    return torch.equal(bits(a), bits(b))


_SNAPSHOTS = {}


def solver_snapshots(name, budget):
    """G entering every loop call of the first two sweeps of a headline layer, as bench.py runs it (initial factors with
    seed 42, its SM budget, the tensor-core MTTKRP and ridge product), with 200 inner iterations per call."""
    key = (name, budget)
    if key not in _SNAPSHOTS:
        import bench
        from source import workloads as wl
        from source.solver import LayerSolver
        u = next(u for u in bench.workload_units(_bench_args("resnet18"))[0] if u[1] == name)
        W = wl.layer_weight_as_tensor(wl.synthetic_weight(*u[2:6], 42, name)).contiguous()
        R = bench.unit_rank(u)
        s = LayerSolver(W.cuda(), [f.cuda() for f in wl.random_init(W.shape, R, 42)], 4, MSE, max_iter_admm=200,
                        mttkrp_precision=1, solve_precision=1, max_ctas=budget)
        s.snapshot_inputs = True
        gs = []
        for _ in range(2):
            s.sweep()
            gs += [s.snapshots[m][3].clone() for m in range(s.N)]
        _SNAPSHOTS[key] = gs
    return _SNAPSHOTS[key]


def gs_of(case):
    if case.kind == "solver":
        return solver_snapshots(case.src, case.grids[0])
    return [make_g(case.kind, case.src, case.R, 100 + case.R, device="cuda")]


WORST = {}


# ------------------------------------------------------------------------------------------------ GPU
@pytest.mark.gpu
@pytest.mark.parametrize("case", CASES, ids=[case_id(c) for c in CASES])
def test_inverse(case, capsys):
    nat = _nat()
    R = case.R
    ld = nat.lib.admmq_padded_ld(R)
    worst = 0.0
    for G in gs_of(case):
        G = G.contiguous()
        Gh = G.cpu()
        G_before = G.clone()
        rho_ref = rho_of(Gh)
        X, kappa, tau = reference(ridge_matrix(Gh.numpy(), rho_ref))
        g0 = case.grids[0]
        M, M64, rho, st, bufs = run_inverse(G, g0, ws_fill=0xFF)
        # ---- status, rho, the guards, G, no NaN left
        assert int(st.item()) == 0, int(st.item())
        assert same_bits(rho, torch.tensor([rho_ref], dtype=torch.float32)), (rho.item(), rho_ref)
        assert all(b.guards_intact() for b in bufs), "a guard word was overwritten"
        assert same_bits(G, G_before), "G changed"
        assert not bool(torch.isnan(M).any()) and not bool(torch.isnan(M64).any()), "an output element was not written"
        # ---- against float64
        Mh, M64h = M.cpu(), M64.cpu()
        err = float(np.abs(M64h[:, :R].numpy() - X).max())
        worst = max(worst, err / tau)
        assert err <= tau, f"|Minv64 - X| = {err:.3g} is {err / tau:.3g} x tau (kappa {kappa:.3g})"
        assert same_bits(Mh, M64h.float()), "Minv is not Minv64 rounded to float32"
        assert same_bits(Mh[:, :R], Mh[:, :R].T) and same_bits(M64h[:, :R], M64h[:, :R].T), "not bitwise symmetric"
        if ld > R:
            assert same_bits(Mh[:, R:], torch.zeros(R, ld - R)), "pad columns of Minv are not +0.0"
            assert same_bits(M64h[:, R:], torch.zeros(R, ld - R, dtype=torch.float64)), "pad columns of Minv64"
        # ---- the same bits at every grid, from a zeroed workspace, and a second call
        for g in case.grids:
            Mg, M64g, rg, sg, bg = run_inverse(G, g, ws_fill=0x00 if g != g0 else 0xFF)
            assert int(sg.item()) == 0 and all(b.guards_intact() for b in bg), g
            assert same_bits(Mg, Mh) and same_bits(M64g, M64h) and same_bits(rg, rho), f"grid {g} differs from grid {g0}"
        Mz = run_inverse(G, g0, ws_fill=0x00)[0]
        assert same_bits(Mz, Mh), "the result depends on the workspace's previous contents"
        # ---- without Minv64 the same Minv
        Mn, none, rn, sn, _ = run_inverse(G, case.grids[-1], minv64=False)
        assert none is None and int(sn.item()) == 0 and same_bits(Mn, Mh) and same_bits(rn, rho)
        # ---- scaling by 4^k is exact through sqrt, division and fma: Minv(4^k G) == 4^-k Minv(G)
        for k in (20, -20):
            s = 4.0 ** k
            Gs = G * s
            assert torch.equal(Gs / s, G) and not bool(((Gs != 0) & (Gs.abs() < 2.0 ** -126)).any())
            Ms, M64s, rs, ss, _ = run_inverse(Gs, case.grids[-1])
            assert int(ss.item()) == 0, k
            assert same_bits(rs, rho * s), (k, rs.item(), rho.item())
            assert same_bits(Ms, Mh.cuda() / s) and same_bits(M64s, M64h.cuda() / s), f"Minv(4^{k} G) != 4^{-k} Minv(G)"
        # ---- only the lower triangle of G is read
        Gu = G.clone()
        Gu[torch.triu(torch.ones(R, R, dtype=torch.bool, device="cuda"), 1)] = float("nan")
        Mu, M64u, ru, su, _ = run_inverse(Gu, case.grids[-1])
        assert int(su.item()) == 0 and same_bits(Mu, Mh) and same_bits(M64u, M64h) and same_bits(ru, rho), \
            "NaN above the diagonal of G changed the result"
    WORST[case.kind] = max(WORST.get(case.kind, 0.0), worst)
    with capsys.disabled():
        print(f"\n[ridge] {case_id(case)} grids {case.grids}: |Minv64 - X| / tau {worst:.3g} (kappa {kappa:.3g}); "
              f"worst of kind {case.kind} so far {WORST[case.kind]:.3g}", end="")


FAIL_CASES = [(R, name) for R in FAIL_RANKS for name, _ in failing_systems(R)]


@pytest.mark.gpu
@pytest.mark.parametrize("R,name", FAIL_CASES, ids=[f"R{R}-{n}" for R, n in FAIL_CASES])
def test_failing_system_sets_the_status(R, name):
    """At every grid: the call returns ADMMQ_OK (spd_inverse raises on any other code), the status reads ADMMQ_E_NOT_PD
    and rho is written.  A good call on the same status word and workspace afterwards writes status 0 and the bits of a
    fresh call."""
    nat = _nat()
    sms = tlk._sm_count()
    G = failing_g(name, R).cuda()
    rho_ref = rho_of(G)
    good = make_g("gram", (64, 512, 9), R, 1, device="cuda")
    nb = -(-R // NB)
    for grid in sorted({1, 2, 3, nb, sms}):
        ws = torch.full((nat.spd_inverse_workspace_bytes(R),), 0xFF, dtype=torch.uint8, device="cuda")
        _, _, rho, st, bufs = run_inverse(G, grid, ws=ws)
        assert int(st.item()) == nat.E_NOT_PD, (grid, int(st.item()))
        assert same_bits(rho, torch.tensor([rho_ref], dtype=torch.float32)), (grid, rho.item(), rho_ref)
        assert all(b.guards_intact() for b in bufs), grid
        M, M64, rho2, st2, _ = run_inverse(good, grid, ws=ws, status=bufs[3])
        assert int(st2.item()) == 0, (grid, int(st2.item()))
        Mf, M64f, rhof, _, _ = run_inverse(good, grid)
        assert same_bits(M, Mf) and same_bits(M64, M64f) and same_bits(rho2, rhof), grid


def _loop_cases(sms):
    """One case per loop kernel id of test_loop_kernels.build_cases (its smallest of at least 64 elements)."""
    by_kernel = {}
    size = lambda c: (c.I * c.R < 64, c.I * c.R)   # noqa: E731
    for c in tlk.build_cases(sms):
        k = tlk.kernel_of(c, sms)
        if k not in by_kernel or size(c) < size(by_kernel[k]):
            by_kernel[k] = c
    return [c for _, c in sorted(by_kernel.items())]


LOOP_CASES = _loop_cases(tlk._sm_count())


def test_loop_cases_reach_every_kernel():
    assert {tlk.kernel_of(c, 148) for c in _loop_cases(148)} == tlk.ALL_KERNELS
    # the two kernels of test_layer_solver_raises
    nat = _nat()
    for precision, budget, name in ((0, 3, "F64_32"), (1, 1, "RESIDENT")):
        assert {tlk.kernel_name(nat.loop_kernel(I, 40, 200, precision, budget)) for I in (32, 24, 9)} == {name}


@pytest.mark.gpu
@pytest.mark.parametrize("case", LOOP_CASES, ids=[tlk.case_id(c) for c in LOOP_CASES])
def test_loop_kernel_leaves_everything_after_a_failed_inverse(case):
    """inv_status = ADMMQ_E_NOT_PD and a NaN inverse: the kernel touches neither H, U nor codes and reports iterations 0,
    the status, rho as given and zeros elsewhere; read_report raises LinAlgError."""
    nat = _nat()
    I, R, p = case.I, case.R, case.precision
    ld = nat.lib.admmq_padded_ld(R)
    H0, U0, F, _ = tlk._problem(case, 7000 + LOOP_CASES.index(case))
    H, U, Fd = H0.cuda(), U0.cuda(), F.cuda()
    codes = (torch.arange(I * R, dtype=torch.int32) % 251 - 125).to(torch.int8).view(I, R).cuda()
    codes0 = codes.clone()
    Minv = torch.full((R, ld), float("nan"), device="cuda")
    M64 = torch.full((R, ld), float("nan"), dtype=torch.float64, device="cuda") if p == 0 else None
    rho = torch.tensor([0.375], device="cuda")
    st = torch.tensor([nat.E_NOT_PD], dtype=torch.int32, device="cuda")
    report = torch.full((ctypes.sizeof(nat.LoopReport),), 0x5A, dtype=torch.uint8, device="cuda")
    nat.admm_loop_inplace(H, U, Fd, Minv, rho, st, 50, 0.0, case.bits, case.scheme, case.attempts, codes=codes,
                          report=report, precision=p, max_ctas=case.budget, minv64=M64)
    torch.cuda.synchronize()
    assert same_bits(H, H0) and same_bits(U, U0) and torch.equal(codes, codes0), "the loop touched its state"
    rep = nat.LoopReport.from_buffer_copy(bytes(report.cpu().numpy().tobytes()))
    got = (rep.iterations, rep.status, rep.rho, rep.scale, rep.r, rep.s, rep.best_index, rep.absmax, list(rep.phase_ns))
    assert got == (0, nat.E_NOT_PD, 0.375, 0.0, 0.0, 0.0, -1, 0.0, [0, 0, 0, 0]), got
    with pytest.raises(torch.linalg.LinAlgError):
        nat.read_report(report)


@pytest.mark.gpu
def test_admm_iteration_raises_at_a_late_panel():
    from source.admm import admm_iteration
    R = 134
    G = failing_g(f"nan-{R - 1}", R).cuda()
    g = torch.Generator().manual_seed(3)
    H, F = torch.randn(64, R, generator=g).cuda(), torch.randn(64, R, generator=g).cuda()
    for precision in (0, 1):
        with pytest.raises(torch.linalg.LinAlgError):
            admm_iteration(H, torch.zeros_like(H), F, G, 5, 1e-8, 4, MSE, precision=precision)


def _bad_factors(shape, R, how, seed=5):
    g = torch.Generator().manual_seed(seed)
    fac = [torch.randn(d, R, generator=g) for d in shape]
    if how == "zero":
        fac[1].zero_()
    else:
        fac[1][len(fac[1]) // 2, R // 3] = float("nan")
    return fac


@pytest.mark.gpu
@pytest.mark.parametrize("how", ("nan", "zero"))
@pytest.mark.parametrize("path", ("collect", "host"))
@pytest.mark.parametrize("precision,budget", ((0, 3), (1, 1)), ids=("F64_32-b3", "RESIDENT-b1"))
def test_layer_solver_raises(how, path, precision, budget):
    """A factor with a NaN or all zero makes the next mode's ridge system fail: the loop leaves that mode's factor as it
    was, and both ways of reading a sweep's reports raise.  The factors run on a cooperative kernel (parity tiles) and
    on the shared-memory kernel, whose early exits are separate code."""
    from source.solver import LayerSolver
    g = torch.Generator().manual_seed(9)
    W = (torch.randn(32, 24, 9, generator=g) * 0.05).cuda()
    R = 40
    fac = _bad_factors(W.shape, R, how)
    s = LayerSolver(W, [f.cuda() for f in fac], 4, MSE, max_iter_admm=20, solve_precision=precision,
                    mttkrp_precision=precision, max_ctas=budget)
    if path == "collect":
        with pytest.raises(torch.linalg.LinAlgError):
            s.sweep()
    else:
        s.enqueue_sweep()
        host = lambda ts: [torch.empty(t.shape, dtype=t.dtype).pin_memory() for t in ts]   # noqa: E731
        reports = torch.empty(s.N * s.reports_dev[0].numel(), dtype=torch.uint8).pin_memory()
        err = torch.empty(2, 2, dtype=torch.float64).pin_memory()
        s.store_to_host(host(s.factors), host(s.duals), host(s.factors_q), err, reports)
        torch.cuda.synchronize()
        with pytest.raises(torch.linalg.LinAlgError):
            s.check_host_reports(reports)
    torch.cuda.synchronize()
    assert same_bits(s.factors[0], fac[0]) and not bool(s.duals[0].any()), "the failed mode's loop ran"


@pytest.mark.gpu
@pytest.mark.parametrize("ndim", (3, 2))
def test_factorize_raises(ndim):
    nat = _nat()
    g = torch.Generator().manual_seed(11)
    shape = (32, 24, 9) if ndim == 3 else (48, 40)
    R = 20
    W = (torch.randn(*shape, generator=g) * 0.05).cuda()
    fac = [f.cuda() for f in _bad_factors(shape, R, "zero")]
    du = [torch.zeros_like(f) for f in fac]
    with pytest.raises(torch.linalg.LinAlgError):
        nat.factorize(W, fac, du, 4, MSE, 3, 20, solve_precision=1, mttkrp_precision=1)
    torch.cuda.synchronize()


@pytest.mark.gpu
def test_factorize_batch_raises_for_one_bad_problem():
    nat = _nat()
    g = torch.Generator().manual_seed(12)
    jobs = []
    for k in range(3):
        W = (torch.randn(32, 24, 9, generator=g) * 0.05).cuda()
        fac = _bad_factors(W.shape, 40, "nan", seed=20 + k)
        if k != 1:
            fac[1] = torch.randn(24, 40, generator=g)
        fac = [f.cuda() for f in fac]
        jobs.append({"W": W, "factors": fac, "duals": [torch.zeros_like(f) for f in fac], "bits": 4, "qscheme": MSE,
                     "max_iter_als": 2, "max_iter_admm": 20, "max_ctas": 4})
    with pytest.raises(torch.linalg.LinAlgError):
        nat.factorize_batch(jobs)
    torch.cuda.synchronize()
