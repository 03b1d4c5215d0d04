"""The FP4 E2M1 grid `tensor_mseminmax_e2m1` (include/admmq.h, csrc/numerics.cuh, DESIGN.md 2b).

CPU: the host rounding onto E2M1 against a table (every boundary, every tie, +-0, saturation), the closed-form
thresholds against a neighbour-float search with the exact division, host threshold-form sums against host direct sums
and float64, the argument checks (bits != 4 is a ValueError), and the channel_* names still raising.
GPU: the projection against a numpy restatement of the definition; the device codes against the hardware conversion;
threshold-form against direct sums; every loop kernel id of test_loop_kernels.build_cases with E2M1 codes (one step
against float64, 30 single steps against one call, the exit test, a NaN input as on the integer grid, an all-zero V);
the two-block splitting;
LayerSolver against admmq_factorize_cp3 on layer1.0.conv1; scripts/factorize.py.
"""
import ctypes
import os
import subprocess
import sys

import numpy as np
import pytest
import torch

import test_loop_kernels as tlk

REPO = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
PKG = os.path.join(REPO, "admm-quantization_b200")
E2M1 = "tensor_mseminmax_e2m1"
MAG = np.array([0.0, 0.5, 1.0, 1.5, 2.0, 3.0, 4.0, 6.0])
BOUNDS = np.array([0.25, 0.75, 1.25, 1.75, 2.5, 3.5, 5.0])   # boundary k separates magnitudes k and k + 1


def e2m1_round(t):
    """Codes of float32 t: nearest of +-MAG, ties to the even mantissa (even index), saturating at +-6."""
    t = np.asarray(t, dtype=np.float32)
    a = np.abs(t.astype(np.float64))
    idx = np.zeros(a.shape, dtype=np.int64)
    for k, b in enumerate(BOUNDS):
        idx += (a > b) if k % 2 == 0 else (a >= b)   # a tie at an even boundary stays below, at an odd one goes up
    return (idx | np.where(np.signbit(t), 8, 0)).astype(np.int8)


def e2m1_values(codes):
    c = np.asarray(codes).astype(np.int64)
    v = MAG[c & 7].astype(np.float32)
    return np.where(c & 8, -v, v).astype(np.float32)


def quantize(x, scale):
    """(codes, values) of float32 x on the grid of float32 scale, as the definition states them."""
    x = np.asarray(x, dtype=np.float32)
    s = np.float32(scale)
    codes = e2m1_round(x / s)
    return codes, (e2m1_values(codes) * s).astype(np.float32)


def candidate_scales(absmax, nc):
    from oracle import admm_oracle as orc
    return (orc.candidate_grid(float(absmax), nc) / np.float32(6.0)).astype(np.float32)


def candidate_sums(x, absmax, nc):
    """float64 sum((x - Q_c(x))**2) for every candidate c."""
    x = np.asarray(x, dtype=np.float32).reshape(-1)
    x64 = x.astype(np.float64)
    out = np.empty(nc)
    for c, s in enumerate(candidate_scales(absmax, nc)):
        out[c] = float(((x64 - quantize(x, s)[1].astype(np.float64)) ** 2).sum())
    return out


def fp(a):
    return a.ctypes.data_as(ctypes.c_void_p)


@pytest.fixture(scope="session")
def hc(tmp_path_factory):
    so = str(tmp_path_factory.mktemp("e2m1") / "libe2m1check.so")
    subprocess.check_call(["g++", "-O2", "-ffp-contract=off", "-std=c++17", "-shared", "-fPIC",
                           os.path.join(REPO, "tests", "hostcheck", "e2m1check.cpp"), "-o", so])
    return ctypes.CDLL(so)


def _nat():
    from source import _native
    return _native


# ------------------------------------------------------------------------------------------------ CPU
def _rounding_table():
    """(t, code) on every boundary, every tie, their neighbours, +-0 and saturation."""
    f = np.float32
    rows = [(0.0, 0), (-0.0, 8), (0.1, 0), (-0.1, 8), (6.0, 7), (-6.0, 15), (7.0, 7), (1e30, 7), (-1e30, 15),
            (np.inf, 7), (-np.inf, 15)]
    for i, m in enumerate(MAG):
        rows += [(m, i), (-m, 8 | i)]
    for k, b in enumerate(BOUNDS):
        tie = k if k % 2 == 0 else k + 1
        up, down = np.nextafter(f(b), f(np.inf)), np.nextafter(f(b), f(0))
        for sgn, sb in ((1.0, 0), (-1.0, 8)):
            rows += [(sgn * b, sb | tie), (sgn * float(up), sb | (k + 1)), (sgn * float(down), sb | k)]
    t = np.array([r[0] for r in rows], dtype=np.float32)
    return t, np.array([r[1] for r in rows], dtype=np.int8)


def test_host_rounding_matches_the_table(hc):
    t, want = _rounding_table()
    got = np.empty(t.size, np.int8)
    hc.hc_e2m1_round(fp(t), ctypes.c_longlong(t.size), fp(got))
    assert np.array_equal(got, want), [(float(a), int(b), int(c)) for a, b, c in zip(t, got, want) if b != c]
    assert np.array_equal(e2m1_round(t), want)
    # the numpy restatement and the host rounding on random quotients of every magnitude
    g = np.random.default_rng(3)
    t = np.concatenate([g.standard_normal(20000) * 3, g.uniform(-7, 7, 20000)]).astype(np.float32)
    got = np.empty(t.size, np.int8)
    hc.hc_e2m1_round(fp(t), ctypes.c_longlong(t.size), fp(got))
    assert np.array_equal(got, e2m1_round(t))
    values = np.empty(16, np.float32)
    assert hc.hc_e2m1_value_mismatches(fp(values)) == 0
    assert np.array_equal(values.view(np.uint32), e2m1_values(np.arange(16)).view(np.uint32))


def test_closed_form_thresholds_equal_the_search(hc):
    theta = np.empty(14, np.float32)
    g = torch.Generator().manual_seed(11)
    scales = [np.float32(float(torch.rand(1, generator=g) + 0.01) * 10 ** float(torch.randint(-9, 9, (1,), generator=g)))
              for _ in range(500)]
    for e in (-46, -40, -23, -1, 0, 1, 7, 24, 37):
        for mant in (1.0, 1.5, 1.0 + 2.0 ** -23, 2.0 - 2.0 ** -23, 1.25, 1.0 + 2.0 ** -12, 4.0 / 3.0):
            scales.append(np.float32(mant * 2.0 ** e))
    for s in scales:
        assert hc.hc_e2m1_thresholds(ctypes.c_float(s), fp(theta)) == 0, s
        assert np.all(np.diff(theta) > 0), s
        # theta is the first float32 whose code reaches the next value (the numpy restatement agrees)
        below = np.nextafter(theta, np.float32(-np.inf))
        lv = np.sort(np.unique(e2m1_values(np.arange(16))))
        assert np.all(e2m1_values(quantize(theta, s)[0]) >= lv[1:]) and np.all(e2m1_values(quantize(below, s)[0]) < lv[1:])


def test_host_threshold_sums_match_direct_sums(hc):
    g = torch.Generator().manual_seed(77)
    for shape, nc in [((64, 134), 200), ((9, 134), 200), ((33, 57), 7), ((1, 1), 200), ((40, 40), 1000), ((7, 5), 1)]:
        for trial in range(2):
            xt = torch.randn(*shape, generator=g) * float(10 ** torch.randint(-3, 3, (1,), generator=g).item())
            x = np.ascontiguousarray(xt.numpy()).reshape(-1)
            mx = np.float32(np.abs(x).max())
            direct, thr, best = np.empty(nc), np.empty(nc), ctypes.c_int()
            hc.hc_e2m1_sums(fp(x), ctypes.c_longlong(x.size), ctypes.c_float(mx), nc, fp(direct), fp(thr), ctypes.byref(best))
            floor = 1e-13 * float((x.astype(np.float64) ** 2).sum()) + 1e-300
            assert np.all(np.abs(thr - direct) <= 3e-6 * np.abs(direct) + floor), (shape, nc)
            exact = candidate_sums(x, mx, nc)
            assert np.all(np.abs(thr - exact) <= 1e-9 * exact + floor), (shape, nc)
            ref = int(np.argmin(exact))
            if best.value != ref:
                assert abs(exact[best.value] - exact[ref]) <= 3e-7 * exact[ref], (shape, best.value, ref)


def test_bits_other_than_4_raise_value_error():
    nat = _nat()
    buf = (ctypes.c_float * 64)()
    p = ctypes.cast(buf, ctypes.c_void_p)
    for bits in (1, 3, 5, 8):
        with pytest.raises(ValueError, match="bits = 4"):
            nat.check(nat.lib.admmq_project(p, 4, bits, 4, 200, None, None, p, None, None, p, 1 << 20, None))
        with pytest.raises(ValueError, match="bits = 4"):
            nat.check(nat.lib.admmq_clip_search_sums_scheme(p, 4, bits, 4, 200, 1, 0, p, p, 1 << 20, None))
        with pytest.raises(ValueError, match="bits = 4"):
            nat.check(nat.lib.admmq_admm_loop(p, p, p, p, None, p, None, 2, 2, 3, 0.0, bits, 4, 200, 1, 0, None, p, p,
                                              1 << 20, None))
        with pytest.raises(ValueError, match="bits = 4"):
            nat.check(nat.lib.admmq_split_loop(p, p, p, p, 4, 1.0, 3, 0.0, bits, 4, 200, 0, None, p, p, 1 << 20, None))
    with pytest.raises(ValueError, match="no clip search"):
        nat.check(nat.lib.admmq_clip_search_sums_scheme(p, 4, 4, 2, 200, 1, 0, p, p, 1 << 20, None))
    with pytest.raises(ValueError, match="unknown qscheme"):
        nat.check(nat.lib.admmq_project(p, 4, 4, 5, 200, None, None, p, None, None, p, 1 << 20, None))
    assert nat.QSCHEME_IDS[E2M1] == 4


def test_channel_schemes_still_raise_not_implemented():
    from source.quantization import quantize_tensor
    for name in ("channel_symmetric", "channel_affine"):
        with pytest.raises(NotImplementedError):
            quantize_tensor(torch.randn(4, 4), 4, name)
    with pytest.raises(NotImplementedError):
        _nat().qscheme_id("channel_mseminmax_e2m1")


# ------------------------------------------------------------------------------------------------ GPU
def _tensors():
    g = torch.Generator().manual_seed(21)
    out = [("normal_64x134", torch.randn(64, 134, generator=g), 200),
           ("normal_512x1141", torch.randn(512, 1141, generator=g) * 0.03, 200),
           ("laplace_9x566", torch.distributions.Laplace(0.0, 1.0).sample((9, 566)), 200),
           ("tiny_neg", -torch.rand(40, 40, generator=g) * 1e-3, 200),
           ("attempts_1", torch.randn(33, 57, generator=g), 1),
           ("attempts_7", torch.randn(33, 57, generator=g), 7),
           ("attempts_1000", torch.randn(50, 50, generator=g), 1000),
           ("single", torch.tensor([[-0.37]]), 200),
           ("huge_direct", torch.randn(20, 30, generator=g) * 1e13, 200),
           ("small_direct", torch.randn(20, 30, generator=g) * 1e-13, 200)]
    x = torch.randn(64, 64, generator=g)
    x[0, :8] = torch.tensor([0.0, -0.0, 1e-30, -1e-30, 5.0, -5.0, 2.5, -2.5])
    out.append(("edges", x, 200))
    return out


@pytest.mark.gpu
@pytest.mark.parametrize("name,x,nc", _tensors(), ids=[t[0] for t in _tensors()])
def test_project_matches_the_definition(name, x, nc):
    nat = _nat()
    xq, codes, info = nat.project(x.cuda(), 4, E2M1, num_attempts=nc, want_codes=True, want_info=True)
    xv = np.ascontiguousarray(x.numpy()).reshape(-1)
    absmax = np.float32(np.abs(xv).max())
    scale, aux, best, mx = info.cpu().numpy()
    assert mx == absmax and aux == 0.0
    best = int(best)
    sums = candidate_sums(xv, absmax, nc)
    ref = int(np.argmin(sums))
    if best != ref:   # ambiguous within the resolution of the kernels' sums: the two MSEs must agree
        assert abs(sums[best] - sums[ref]) <= 3e-7 * sums[ref], (name, best, ref)
    assert scale == candidate_scales(absmax, nc)[best]
    want_codes, want_values = quantize(xv, scale)
    assert np.array_equal(codes.cpu().numpy().reshape(-1), want_codes), name
    assert np.array_equal(xq.cpu().numpy().reshape(-1).view(np.uint32), want_values.view(np.uint32)), name
    # the device codes are the hardware conversion of fl(x / s)
    t = torch.from_numpy((xv / np.float32(scale)).astype(np.float32)).cuda()
    assert torch.equal(nat.e2m1_encode(t).reshape(-1), codes.reshape(-1)), name
    # quantize_tensor passes num_attempts through
    from source.quantization import quantize_tensor
    assert torch.equal(quantize_tensor(x.cuda(), 4, E2M1, num_attempts=nc), xq.reshape(x.shape))


@pytest.mark.gpu
def test_hardware_conversion_equals_the_host_rounding():
    t, want = _rounding_table()
    g = np.random.default_rng(5)
    rnd = np.concatenate([g.standard_normal(100000) * 3, g.uniform(-8, 8, 100000)]).astype(np.float32)
    every = np.concatenate([t, rnd, np.nextafter(np.float32(BOUNDS), np.float32(np.inf)) * -1])
    codes = _nat().e2m1_encode(torch.from_numpy(every).cuda()).cpu().numpy()
    assert np.array_equal(codes[:t.size], want)
    assert np.array_equal(codes, e2m1_round(every))


@pytest.mark.gpu
def test_threshold_and_direct_sums_agree():
    nat = _nat()
    g = torch.Generator().manual_seed(8)
    for tag, x, nc in [("64x134", torch.randn(64, 134, generator=g), 200),
                       ("512x1141", torch.randn(512, 1141, generator=g) * 0.02, 200),
                       ("9x278", torch.randn(9, 278, generator=g) * 5, 1000),
                       ("3x7", torch.randn(3, 7, generator=g), 33)]:
        xd = x.cuda()
        n = x.numel()
        direct = nat.clip_search_sums(xd, 4, nc, method=0, qscheme=E2M1).cpu().numpy()
        thr = nat.clip_search_sums(xd, 4, nc, method=1, qscheme=E2M1).cpu().numpy()
        floor = 1e-13 * float((x.double() ** 2).sum()) + 1e-300
        assert np.all(np.abs(thr - direct) <= 3e-6 * np.abs(direct) + floor), tag
        exact = candidate_sums(x.numpy(), np.float32(x.abs().max()), nc)
        assert np.all(np.abs(thr - exact) <= 1e-9 * exact + floor), tag
        mse_d, mse_t = (direct / n).astype(np.float32), (thr / n).astype(np.float32)
        bd, bt = int(np.argmin(mse_d)), int(np.argmin(mse_t))
        if bd != bt:
            assert abs(float(mse_d[bd]) - float(mse_d[bt])) <= 3e-7 * float(mse_d[bd]), (tag, bd, bt)
        assert np.array_equal(thr, nat.clip_search_sums(xd, 4, nc, method=1, qscheme=E2M1).cpu().numpy()), tag
        for ctas in (1, 3, 7):
            few = nat.clip_search_sums(xd, 4, nc, method=1, max_ctas=ctas, qscheme=E2M1).cpu().numpy()
            assert np.all(np.abs(few - thr) <= 1e-11 * np.abs(thr) + floor), (tag, ctas)
            fewd = nat.clip_search_sums(xd, 4, nc, method=0, max_ctas=ctas, qscheme=E2M1).cpu().numpy()
            assert np.all(np.abs(fewd - direct) <= 1e-11 * np.abs(direct) + floor), (tag, ctas)
        # the uniform scheme through the new entry point is the old one
        old = torch.empty(nc, dtype=torch.float64, device="cuda")
        ws = torch.empty(nat.project_workspace_bytes(n, nc), dtype=torch.uint8, device="cuda")
        nat.call(xd.device, nat.lib.admmq_clip_search_sums, nat.ptr(xd), n, 4, nc, 1, 0, nat.ptr(old), nat.ptr(ws),
                 ws.numel(), nat.stream_ptr(xd.device))
        assert torch.equal(old, nat.clip_search_sums(xd, 4, nc, method=1)), tag


def _loop_cases(sms):
    """One case per loop kernel id of test_loop_kernels.build_cases (its smallest of at least 64 elements), on E2M1."""
    by_kernel = {}
    size = lambda c: (c.I * c.R < 64, c.I * c.R)   # noqa: E731
    for c in tlk.build_cases(sms):
        k = tlk.kernel_of(c, sms)
        if k not in by_kernel or size(c) < size(by_kernel[k]):
            by_kernel[k] = c
    return [c._replace(scheme=E2M1, bits=4) for _, c in sorted(by_kernel.items())]


LOOP_CASES = _loop_cases(tlk._sm_count())


def test_loop_cases_reach_every_kernel():
    assert {tlk.kernel_of(c, 148) for c in _loop_cases(148)} == tlk.ALL_KERNELS


def check_one_step(case, kid, H0, U0, F, G, H1, U1, codes, rep):
    """One iteration on the E2M1 grid against float64: ridge product within the kernel's bound, candidate and codes of
    V = H_ls - U, H = codes * scale, the dual update and the residuals.  Returns the ambiguous share."""
    I, R = case.I, case.R
    H0, U0, F, G = (t.numpy() for t in (H0, U0, F, G))
    H1, U1, codes = H1.cpu().numpy(), U1.cpu().numpy(), codes.cpu().numpy()
    rho = np.float32(rep.rho)
    rhs = F + rho * (H0 + U0)
    A = G.astype(np.float64)
    A[np.diag_indices(R)] = (np.diag(G) + rho).astype(np.float64)
    Minv = np.linalg.inv(A)
    hls64 = rhs.astype(np.float64) @ Minv
    mag = np.abs(rhs.astype(np.float64)) @ np.abs(Minv)
    du = U1.astype(np.float64) - U0.astype(np.float64)
    hls_k = H1.astype(np.float64) - du
    delta = tlk._spacing(U1) + tlk._spacing(du)
    ratio = float(np.max(np.abs(hls_k - hls64) / (tlk._bound_factor(kid, R) * mag + delta)))
    assert ratio <= 1.0, f"ridge product off by {ratio:.3g} x its bound"
    v64 = hls_k - U0.astype(np.float64)
    band = delta + tlk._spacing(v64)
    absmax = np.float32(rep.absmax)
    ext = np.abs(tlk._f32(v64)) == absmax
    v64, band = np.where(ext, np.sign(v64) * float(absmax), v64), np.where(ext, 0.0, band)
    v32 = tlk._f32(v64)
    scale = np.float32(rep.scale)
    assert 0 <= rep.best_index < case.attempts
    assert scale == candidate_scales(absmax, case.attempts)[rep.best_index]
    sums = candidate_sums(v32, absmax, case.attempts)
    ref = int(np.argmin(sums))
    if rep.best_index != ref:
        assert abs(sums[rep.best_index] - sums[ref]) <= 3e-7 * sums[ref], (rep.best_index, ref)
    outward = lambda x, to: np.where(band > 0, np.nextafter(tlk._f32(x), np.float32(to)), v32)   # noqa: E731
    lo = quantize(outward(v64 - band, -np.inf), scale)[0]
    hi = quantize(outward(v64 + band, np.inf), scale)[0]
    ambiguous = lo != hi
    assert int(np.count_nonzero((codes != lo) & ~ambiguous)) == 0, "codes differ from the exact projection of V"
    assert float(ambiguous.mean()) <= 1e-3
    assert np.array_equal((e2m1_values(codes) * scale).astype(np.float32).view(np.uint32), H1.view(np.uint32))
    h = tlk._f32(hls_k)
    for _ in range(2):
        h = np.nextafter(h, np.float32(-np.inf))
    dual_ok = np.zeros(h.shape, dtype=bool)
    for _ in range(5):
        dual_ok |= (U0 + (H1 - h)) == U1
        h = np.nextafter(h, np.float32(np.inf))
    assert dual_ok.all()
    h64, h0 = H1.astype(np.float64), H0.astype(np.float64)
    r64 = float(np.sum((h64 - hls_k) ** 2) / np.sum(h64 ** 2))
    s64 = float(np.sum((h64 - h0) ** 2) / np.sum(U1.astype(np.float64) ** 2))
    assert abs(rep.r - r64) <= 1e-3 * r64 and abs(rep.s - s64) <= 1e-3 * s64, (rep.r, r64, rep.s, s64)
    return float(ambiguous.mean())


@pytest.mark.gpu
@pytest.mark.parametrize("case", LOOP_CASES, ids=[tlk.case_id(c) for c in LOOP_CASES])
def test_loop_kernel_e2m1(case, capsys):
    nat = _nat()
    sms = tlk._sm_count()
    kid = tlk.kernel_of(case, sms)
    H0, U0, F, G = tlk._problem(case, 5000 + LOOP_CASES.index(case))
    I, R, p, b, na = case.I, case.R, case.precision, case.budget, case.attempts
    d = lambda t: t.cuda().contiguous()   # noqa: E731
    Fd, Gd = d(F), d(G)
    H, U = d(H0), d(U0)
    codes = torch.empty(I, R, dtype=torch.int8, device="cuda")
    rep = nat.read_report(nat.admm_iteration_inplace(H, U, Fd, Gd, 2, 0.0, 4, E2M1, na, codes=codes, precision=p, max_ctas=b))
    assert rep.iterations == 1 and rep.status == 0, (rep.iterations, rep.status)
    amb = check_one_step(case, kid, H0, U0, F, G, H, U, codes, rep)
    Minv, rho, st, m64 = nat.spd_inverse(Gd, minv64=True, max_ctas=b)
    m64 = m64 if p == 0 else None
    ws = torch.empty(nat.admm_loop_workspace_bytes(I, R, na), dtype=torch.uint8, device="cuda")

    def loop(Hx, Ux, cx, iters, eps, Fx=Fd):
        return nat.read_report(nat.admm_loop_inplace(Hx, Ux, Fx, Minv, rho, st, iters + 1, eps, 4, E2M1, na, codes=cx,
                                                     ws=ws, precision=p, max_ctas=b, minv64=m64))

    H, U = d(H0), d(U0)
    codes = torch.empty(I, R, dtype=torch.int8, device="cuda")
    snaps, reps = [], []
    for _ in range(tlk.STEPS):
        reps.append(loop(H, U, codes, 1, 0.0))
        snaps.append(tlk._state(H, U, codes))
    Hk, Uk = d(H0), d(U0)
    ck = torch.empty(I, R, dtype=torch.int8, device="cuda")
    rk = loop(Hk, Uk, ck, tlk.STEPS, 0.0)
    assert rk.iterations == tlk.STEPS
    assert tlk._equal((Hk, Uk, ck), snaps[-1]), "30 iterations in one call differ from 30 single calls"
    last = reps[-1]
    assert (rk.r, rk.s, rk.scale, rk.best_index) == (last.r, last.s, last.scale, last.best_index)
    assert int(ck.min()) >= 0 and int(ck.max()) <= 15
    m = [max(x.r, x.s) for x in reps]
    j = max(i for i in range(tlk.STEPS - 1) if all(m[i] < m[k] for k in range(i)))
    eps = float(np.nextafter(np.float32(m[j]), np.float32(np.inf)))
    He, Ue = d(H0), d(U0)
    ce = torch.empty(I, R, dtype=torch.int8, device="cuda")
    re_ = loop(He, Ue, ce, tlk.STEPS, eps)
    assert re_.iterations == j + 1 and re_.status & nat.ST_CONVERGED, (re_.iterations, j + 1, re_.status)
    assert tlk._equal((He, Ue, ce), snaps[j]), "the exit left another state than the single steps"
    # a NaN in the input: the status, the iteration count and where NaN ends up as with the integer grid
    nan_runs = []
    for scheme in (E2M1, tlk.MSE):
        Hn, Un = d(H0), d(U0)
        Hn.view(-1)[I * R // 2] = float("nan")
        r = nat.read_report(nat.admm_loop_inplace(Hn, Un, Fd, Minv, rho, st, 4, 0.0, 4, scheme, na, ws=ws, precision=p,
                                                  max_ctas=b, minv64=m64))
        nan_runs.append((r.status, r.iterations, torch.isnan(Hn).cpu(), torch.isnan(Un).cpu()))
    (s0, i0, h0, u0), (s1, i1, h1, u1) = nan_runs
    assert (s0, i0) == (s1, i1) and torch.equal(h0, h1) and torch.equal(u0, u1), (s0, i0, s1, i1)
    # an all-zero V: the degenerate range of the clip search
    Hz, Uz = d(torch.zeros(I, R)), d(torch.zeros(I, R))
    rz = loop(Hz, Uz, torch.empty(I, R, dtype=torch.int8, device="cuda"), 3, 0.0, Fx=torch.zeros_like(Fd))
    assert rz.status & nat.ST_NONFINITE and rz.iterations == 1 and bool(torch.isnan(Hz).all()), (rz.status, rz.iterations)
    with capsys.disabled():
        print(f"\n[e2m1 loop] {tlk.case_id(case)} {tlk.kernel_name(kid)}: ambiguous {amb:.2e}, exit at {j + 1}", end="")


@pytest.mark.gpu
def test_split_loop_runs_e2m1():
    """One step of the two-block splitting (scripts/factorize_lowrank.py:85-88) on E2M1, then a longer run."""
    nat = _nat()
    g = torch.Generator().manual_seed(13)
    n = 40000
    W, H2, H, U = (torch.randn(n, generator=g) for _ in range(4))
    rho = 0.7
    Hd, Ud = H.cuda(), (U * 0.1).cuda()
    U0 = Ud.cpu().numpy()
    codes = torch.empty(n, dtype=torch.int8, device="cuda")
    rep = nat.read_report(nat.split_loop_inplace(Hd, Ud, W.cuda(), H2.cuda(), rho, 2, 0.0, 4, E2M1, codes=codes))
    assert rep.iterations == 1 and rep.status == 0
    r = np.float32(rho)
    hls = ((r * (H.numpy() + U0) + W.numpy() - H2.numpy()) / (np.float32(1.0) + r)).astype(np.float32)
    v = (hls - U0).astype(np.float32)
    absmax = np.float32(np.abs(v).max())
    assert rep.absmax == absmax
    sums = candidate_sums(v, absmax, 200)
    ref = int(np.argmin(sums))
    if rep.best_index != ref:
        assert abs(sums[rep.best_index] - sums[ref]) <= 3e-7 * sums[ref]
    scale = np.float32(rep.scale)
    assert scale == candidate_scales(absmax, 200)[rep.best_index]
    want_codes, want_values = quantize(v, scale)
    assert np.array_equal(codes.cpu().numpy(), want_codes)
    assert np.array_equal(Hd.cpu().numpy().view(np.uint32), want_values.view(np.uint32))
    assert np.array_equal(Ud.cpu().numpy(), (U0 + (want_values - hls)).astype(np.float32))
    rep = nat.read_report(nat.split_loop_inplace(Hd, Ud, W.cuda(), H2.cuda(), rho, 50, 0.0, 4, E2M1, codes=codes))
    assert rep.iterations == 49 and rep.status == 0
    assert np.array_equal(e2m1_values(codes.cpu().numpy()) * np.float32(rep.scale), Hd.cpu().numpy())


@pytest.mark.gpu
def test_layer_solver_equals_factorize_cp3_on_layer1_conv1():
    """A few sweeps of layer1.0.conv1 (64 x 64 x 9, rank 134) in both solver paths; every quantized factor on s x E2M1."""
    from source import workloads as wl
    from source.solver import LayerSolver
    nat = _nat()
    g = torch.Generator().manual_seed(17)
    W = (torch.randn(64, 64, 9, generator=g) * 0.05).cuda()
    R = 134
    init = wl.random_init((64, 64, 9), R, 3)
    for prec in (0, 1):
        s = LayerSolver(W, [f.cuda() for f in init], 4, E2M1, max_iter_admm=30, solve_precision=prec, mttkrp_precision=prec)
        n_py = s.run(3)
        fac = [f.clone().cuda() for f in init]
        du = [torch.zeros_like(f) for f in fac]
        hist, histq, n_c, fq = nat.factorize(W, fac, du, 4, E2M1, 3, 30, solve_precision=prec, mttkrp_precision=prec)
        assert n_c == n_py and hist == s.loss_hist and histq == s.loss_quant_hist, (prec, hist, s.loss_hist)
        for a, b in zip(fac + du + fq, s.factors + s.duals + s.factors_q):
            assert torch.equal(a, b)
        for f, q in zip(fac, fq):
            xq, codes, info = nat.project(f, 4, E2M1, want_codes=True, want_info=True)
            assert torch.equal(xq, q)
            scale = np.float32(info[0].item())
            assert np.array_equal(e2m1_values(codes.cpu().numpy()) * scale, q.cpu().numpy())
        assert all(np.isfinite(hist)) and histq[-1] < histq[0] * 1.5


@pytest.mark.gpu
def test_factorize_script_runs_e2m1(tmp_path):
    w = torch.randn(64, 64, 3, 3, generator=torch.Generator().manual_seed(1)) * 0.05
    wf = tmp_path / "w.pt"
    torch.save(w, wf)
    out = tmp_path / "out"
    r = subprocess.run([sys.executable, os.path.join(PKG, "scripts", "factorize.py"), "--model-name", "resnet18",
                        "--method", "admm", "--layer", "layer1.0.conv1", "--reduction-rate", "2", "--bits", "4",
                        "--qscheme", E2M1, "--seed", "0", "--max_iter_als", "2", "--max_iter_admm", "20",
                        "--weight-file", str(wf), "--outdir", str(out)], capture_output=True, text=True, cwd=str(tmp_path))
    assert r.returncode == 0, r.stdout[-2000:] + r.stderr[-2000:]
    files = sorted(os.listdir(out))
    assert any(f.endswith("_losshist.pt") for f in files), files
    assert sum(f.endswith(tuple(f"_mode_{m}.pt" for m in range(3))) for f in files) == 3, files
