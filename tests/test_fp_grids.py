"""The FP8 (E4M3, E5M2) and FP6 (E3M2, E2M3) grids `tensor_mseminmax_e4m3 / _e5m2 / _e3m2 / _e2m3` (include/admmq.h,
csrc/numerics.cuh, DESIGN.md 2c), each test over the four formats.

CPU: the host rounding against an enumerated table (every value, every boundary and its two neighbours, +-0, subnormals,
saturation, +-inf) and, for FP8, against torch's float8 dtypes; the closed-form thresholds against a neighbour-float
search with the exact division; host threshold-form sums against host direct sums and float64; the argument checks.
GPU: the projection against a numpy restatement of the definition; the hardware conversion against the host rounding;
threshold-form against direct sums; every loop kernel id of test_loop_kernels.build_cases (one step against float64,
30 single steps against one call, the exit test, a NaN input as on the integer grid, an all-zero V); the two-block
splitting; LayerSolver against admmq_factorize_cp3 on layer1.0.conv1; scripts/factorize.py.
"""
import ctypes
import os
import subprocess
import sys
from collections import namedtuple

import numpy as np
import pytest
import torch

import test_loop_kernels as tlk

REPO = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
PKG = os.path.join(REPO, "admm-quantization_b200")

Fmt = namedtuple("Fmt", "name id bits ebits mbits bias top max dtype")
FORMATS = [
    Fmt("tensor_mseminmax_e4m3", 6, 8, 4, 3, 7, 126, 448.0, torch.float8_e4m3fn),
    Fmt("tensor_mseminmax_e5m2", 7, 8, 5, 2, 15, 123, 57344.0, torch.float8_e5m2),
    Fmt("tensor_mseminmax_e3m2", 8, 6, 3, 2, 3, 31, 28.0, None),
    Fmt("tensor_mseminmax_e2m3", 9, 6, 2, 3, 1, 31, 7.5, None),
]
FMT_IDS = [f.name.split("_")[-1] for f in FORMATS]
by_fmt = pytest.mark.parametrize("f", FORMATS, ids=FMT_IDS)


def magnitudes(f):
    """float64 value of the magnitude codes 0 .. top, from the encoding."""
    k = np.arange(f.top + 1)
    e, m = k >> f.mbits, k & ((1 << f.mbits) - 1)
    return np.where(e == 0, m * 2.0 ** (1 - f.bias - f.mbits), (2 ** f.mbits + m) * 2.0 ** (e - f.bias - f.mbits))


def values(f, codes):
    """float32 value of codes (int8 storage of the byte, or 0 .. 63)."""
    c = np.asarray(codes).astype(np.int64) & 0xff
    sign = 1 << (f.bits - 1)
    v = magnitudes(f)[c & (sign - 1)].astype(np.float32)
    return np.where(c & sign, -v, v).astype(np.float32)


def fp_round(f, t):
    """Codes (int8) of float32 t: nearest value of the format, ties to the even mantissa, saturating at +-max."""
    t = np.asarray(t, dtype=np.float32)
    a = np.abs(t.astype(np.float64))
    mags = magnitudes(f)
    lo = np.clip(np.searchsorted(mags, a, side="right") - 1, 0, f.top)
    hi = np.minimum(lo + 1, f.top)
    mid = (mags[lo] + mags[hi]) / 2
    up = (a > mid) | ((a == mid) & (hi % 2 == 0))
    k = np.where(a >= f.max, f.top, np.where(up & (lo < f.top), hi, lo))
    code = k | np.where(np.signbit(t), 1 << (f.bits - 1), 0)
    return code.astype(np.uint8).view(np.int8)


def quantize(f, x, scale):
    """(codes, values) of float32 x on the grid of float32 scale, as the definition states them."""
    x = np.asarray(x, dtype=np.float32)
    codes = fp_round(f, x / np.float32(scale))
    return codes, (values(f, codes) * np.float32(scale)).astype(np.float32)


def candidate_scales(f, absmax, nc):
    from oracle import admm_oracle as orc
    return (orc.candidate_grid(float(absmax), nc) / np.float32(f.max)).astype(np.float32)


def candidate_sums(f, x, absmax, nc):
    """float64 sum((x - Q_c(x))**2) for every candidate c."""
    x = np.asarray(x, dtype=np.float32).reshape(-1)
    x64 = x.astype(np.float64)
    out = np.empty(nc)
    for c, s in enumerate(candidate_scales(f, absmax, nc)):
        out[c] = float(((x64 - quantize(f, x, s)[1].astype(np.float64)) ** 2).sum())
    return out


def fp(a):
    return a.ctypes.data_as(ctypes.c_void_p)


@pytest.fixture(scope="session")
def hc(tmp_path_factory):
    so = str(tmp_path_factory.mktemp("fp") / "libfpcheck.so")
    subprocess.check_call(["g++", "-O2", "-ffp-contract=off", "-std=c++17", "-shared", "-fPIC",
                           os.path.join(REPO, "tests", "hostcheck", "fpcheck.cpp"), "-o", so])
    return ctypes.CDLL(so)


def _nat():
    from source import _native
    return _native


def host_round(hc, f, t):
    t = np.ascontiguousarray(t, dtype=np.float32)
    out = np.empty(t.size, np.int8)
    hc.hc_fp_round(f.id, fp(t), ctypes.c_longlong(t.size), fp(out))
    return out


# ------------------------------------------------------------------------------------------------ CPU
def rounding_table(f):
    """(t, code) on every value, every boundary and its two neighbours, +-0, saturation and +-inf, built from the
    encoding alone."""
    f32 = np.float32
    sign = 1 << (f.bits - 1)
    mags = magnitudes(f)
    rows = [(0.0, 0), (-0.0, sign), (f.max * 1.25, f.top), (-f.max * 1.25, sign | f.top), (1e30, f.top),
            (-1e30, sign | f.top), (np.inf, f.top), (-np.inf, sign | f.top)]
    for k, m in enumerate(mags):
        rows += [(m, k), (-m, sign | k)]
    for k in range(f.top):
        b = f32((mags[k] + mags[k + 1]) / 2)
        assert float(b) == (mags[k] + mags[k + 1]) / 2   # the boundary is exact in float32
        tie = k if k % 2 == 0 else k + 1
        up, down = np.nextafter(b, f32(np.inf)), np.nextafter(b, f32(0))
        for sgn, sb in ((1.0, 0), (-1.0, sign)):
            rows += [(sgn * float(b), sb | tie), (sgn * float(up), sb | (k + 1)), (sgn * float(down), sb | k)]
    t = np.array([r[0] for r in rows], dtype=np.float32)
    return t, np.array([r[1] for r in rows], dtype=np.int64).astype(np.uint8).view(np.int8)


def random_quotients(f, n, seed):
    """float32 quotients over the whole range of a format: log-uniform from below the smallest subnormal to above max,
    random signs, plus uniform values inside [-max, max]."""
    g = np.random.default_rng(seed)
    lo = np.log2(magnitudes(f)[1]) - 2
    a = 2.0 ** g.uniform(lo, np.log2(f.max) + 1, n) * g.choice([-1.0, 1.0], n)
    return np.concatenate([a, g.uniform(-f.max, f.max, n)]).astype(np.float32)


@by_fmt
def test_format_descriptor(hc, f):
    ints, mx = (ctypes.c_int * 6)(), ctypes.c_float()
    hc.hc_fp_format(f.id, ints, ctypes.byref(mx))
    assert list(ints)[:5] == [f.bits, f.ebits, f.mbits, f.bias, f.top] and mx.value == f.max
    assert ints[5] == (1 if f.name.endswith("e4m3") else 0)
    assert magnitudes(f)[-1] == f.max
    if f.dtype is not None:   # max and the codes below it are torch's float8 values
        byte = torch.arange(f.top + 1, dtype=torch.uint8).view(torch.int8).view(f.dtype).float().numpy()
        assert np.array_equal(byte, magnitudes(f).astype(np.float32))
        assert f.max == float(torch.finfo(f.dtype).max)
    # values from the bits: every code of the grid, sign and -0 included
    codes = np.arange(1 << f.bits, dtype=np.int32)
    codes = codes[(codes & ((1 << (f.bits - 1)) - 1)) <= f.top]
    out = np.empty(codes.size, np.float32)
    hc.hc_fp_value(f.id, fp(codes), codes.size, fp(out))
    assert np.array_equal(out.view(np.uint32), values(f, codes).view(np.uint32))
    # the ascending grid of 2 top + 1 values, +-0 merged
    levels, gcodes = np.empty(2 * f.top + 1, np.float32), np.empty(2 * f.top + 1, np.int32)
    assert hc.hc_fp_grid(f.id, fp(levels), fp(gcodes)) == 2 * f.top + 1
    assert np.all(np.diff(levels) > 0) and levels[f.top] == 0 and not np.signbit(levels[f.top])
    assert np.array_equal(levels, values(f, gcodes)) and levels[-1] == f.max and levels[0] == -f.max


@by_fmt
def test_host_rounding_matches_the_table(hc, f):
    t, want = rounding_table(f)
    got = host_round(hc, f, t)
    assert np.array_equal(got, want), [(float(a), int(b), int(c)) for a, b, c in zip(t, got, want) if b != c][:10]
    assert np.array_equal(fp_round(f, t), want)
    t = random_quotients(f, 20000, 3 + f.id)
    assert np.array_equal(host_round(hc, f, t), fp_round(f, t))


@pytest.mark.parametrize("f", FORMATS[:2], ids=FMT_IDS[:2])
def test_host_rounding_matches_torch_float8(hc, f):
    """torch's CPU conversion rounds to nearest even but does not saturate: clamp to +-max first."""
    t = np.concatenate([random_quotients(f, 50000, 31 + f.id), rounding_table(f)[0]])
    t = t[np.isfinite(t)]
    ref = torch.from_numpy(t).clamp(-f.max, f.max).to(f.dtype).view(torch.int8).numpy()
    assert np.array_equal(host_round(hc, f, t), ref)


@by_fmt
def test_closed_form_thresholds_equal_the_search(hc, f):
    theta = np.empty(2 * f.top, np.float32)
    g = torch.Generator().manual_seed(11 + f.id)
    scales = [np.float32(float(torch.rand(1, generator=g) + 0.01) * 10 ** float(torch.randint(-9, 9, (1,), generator=g)))
              for _ in range(500)]
    # scale = clip / max with clip in 0.2 .. 1.2 x abs-max, abs-max in [2^-40, 2^40] (the binned range)
    for e in (-58, -46, -40, -23, -1, 0, 1, 7, 24, 37):
        for mant in (1.0, 1.5, 1.0 + 2.0 ** -23, 2.0 - 2.0 ** -23, 1.25, 1.0 + 2.0 ** -12, 4.0 / 3.0):
            scales.append(np.float32(mant * 2.0 ** e))
    lv = np.sort(np.unique(values(f, np.arange(1 << f.bits)[(np.arange(1 << f.bits) & ((1 << (f.bits - 1)) - 1)) <= f.top])))
    for s in scales:
        assert hc.hc_fp_thresholds(f.id, ctypes.c_float(s), fp(theta)) == 0, s
        assert np.all(np.diff(theta) > 0), s
        # theta is the first float32 whose code reaches the next value (the numpy restatement agrees)
        below = np.nextafter(theta, np.float32(-np.inf))
        assert np.all(values(f, quantize(f, theta, s)[0]) >= lv[1:]) and np.all(values(f, quantize(f, below, s)[0]) < lv[1:])


@by_fmt
def test_host_threshold_sums_match_direct_sums(hc, f):
    g = torch.Generator().manual_seed(77)
    for shape, nc in [((64, 134), 200), ((9, 134), 200), ((33, 57), 7), ((1, 1), 200), ((40, 40), 1000), ((7, 5), 1)]:
        for trial in range(2):
            xt = torch.randn(*shape, generator=g) * float(10 ** torch.randint(-3, 3, (1,), generator=g).item())
            x = np.ascontiguousarray(xt.numpy()).reshape(-1)
            mx = np.float32(np.abs(x).max())
            direct, thr, best = np.empty(nc), np.empty(nc), ctypes.c_int()
            hc.hc_fp_sums(f.id, fp(x), ctypes.c_longlong(x.size), ctypes.c_float(mx), nc, fp(direct), fp(thr),
                          ctypes.byref(best))
            floor = 1e-13 * float((x.astype(np.float64) ** 2).sum()) + 1e-300
            assert np.all(np.abs(thr - direct) <= 3e-6 * np.abs(direct) + floor), (shape, nc)
            exact = candidate_sums(f, x, mx, nc)
            assert np.all(np.abs(thr - exact) <= 1e-9 * exact + floor), (shape, nc)
            ref = int(np.argmin(exact))
            if best.value != ref:
                assert abs(exact[best.value] - exact[ref]) <= 3e-7 * exact[ref], (shape, best.value, ref)
            scales = np.empty(nc, np.float32)
            hc.hc_fp_scales(f.id, ctypes.c_float(mx), nc, fp(scales))
            assert np.array_equal(scales, candidate_scales(f, mx, nc))


def test_argument_checks():
    nat = _nat()
    buf = (ctypes.c_float * 64)()
    p = ctypes.cast(buf, ctypes.c_void_p)
    for f in FORMATS:
        assert nat.QSCHEME_IDS[f.name] == f.id and f.name in nat.CLIP_SEARCH_SCHEMES
        for bits in (1, 4, 5, 6, 7, 8):
            if bits == f.bits:
                continue
            msg = f"{f.name} needs bits = {f.bits}"
            with pytest.raises(ValueError, match=msg):
                nat.check(nat.lib.admmq_project(p, 4, bits, f.id, 200, None, None, p, None, None, p, 1 << 20, None))
            with pytest.raises(ValueError, match=msg):
                nat.check(nat.lib.admmq_clip_search_sums_scheme(p, 4, bits, f.id, 200, 1, 0, p, p, 1 << 20, None))
            with pytest.raises(ValueError, match=msg):
                nat.check(nat.lib.admmq_admm_loop(p, p, p, p, None, p, None, 2, 2, 3, 0.0, bits, f.id, 200, 1, 0, None,
                                                  p, p, 1 << 20, None))
            with pytest.raises(ValueError, match=msg):
                nat.check(nat.lib.admmq_split_loop(p, p, p, p, 4, 1.0, 3, 0.0, bits, f.id, 200, 0, None, p, p, 1 << 20,
                                                   None))
        with pytest.raises(ValueError, match="num_attempts"):
            nat.check(nat.lib.admmq_project(p, 4, f.bits, f.id, 0, None, None, p, None, None, p, 1 << 20, None))
    for bad in (5, 10, -1):
        with pytest.raises(ValueError, match="unknown qscheme"):
            nat.check(nat.lib.admmq_project(p, 4, 8, bad, 200, None, None, p, None, None, p, 1 << 20, None))
        with pytest.raises(ValueError, match="unknown qscheme"):
            nat.check(nat.lib.admmq_split_loop(p, p, p, p, 4, 1.0, 3, 0.0, 8, bad, 200, 0, None, p, p, 1 << 20, None))
    assert 5 not in nat.QSCHEME_IDS.values()
    for bad in (0, 4, 5, 10):
        with pytest.raises(ValueError, match="no FP8 / FP6 grid"):
            nat.check(nat.lib.admmq_fp_encode(p, 4, bad, p, None))
    with pytest.raises(NotImplementedError):
        nat.qscheme_id("channel_mseminmax_e4m3")


# ------------------------------------------------------------------------------------------------ GPU
def _tensors():
    g = torch.Generator().manual_seed(21)
    out = [("normal_64x134", torch.randn(64, 134, generator=g), 200),
           ("normal_128x1141", torch.randn(128, 1141, generator=g) * 0.03, 200),
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
    x[1, :4] = torch.tensor([1e-7, -1e-7, 3e-6, -3e-6])   # subnormal quotients on the finer grids
    out.append(("edges", x, 200))
    return out


TENSORS = _tensors()


@pytest.mark.gpu
@by_fmt
@pytest.mark.parametrize("name,x,nc", TENSORS, ids=[t[0] for t in TENSORS])
def test_project_matches_the_definition(f, name, x, nc):
    nat = _nat()
    xq, codes, info = nat.project(x.cuda(), f.bits, f.name, num_attempts=nc, want_codes=True, want_info=True)
    xv = np.ascontiguousarray(x.numpy()).reshape(-1)
    absmax = np.float32(np.abs(xv).max())
    scale, aux, best, mx = info.cpu().numpy()
    assert mx == absmax and aux == 0.0
    best = int(best)
    sums = candidate_sums(f, xv, absmax, nc)
    ref = int(np.argmin(sums))
    if best != ref:   # ambiguous within the resolution of the kernels' sums: the two MSEs must agree
        assert abs(sums[best] - sums[ref]) <= 3e-7 * sums[ref], (name, best, ref)
    assert scale == candidate_scales(f, absmax, nc)[best]
    want_codes, want_values = quantize(f, xv, scale)
    got = codes.cpu().numpy().reshape(-1)
    assert np.array_equal(got, want_codes), name
    assert np.array_equal(xq.cpu().numpy().reshape(-1).view(np.uint32), want_values.view(np.uint32)), name
    if f.dtype is not None:   # the codes are the FP8 tensor
        fq = (codes.view(f.dtype).float() * float(scale)).cpu().numpy().reshape(-1)
        assert np.array_equal(fq.view(np.uint32), xq.cpu().numpy().reshape(-1).view(np.uint32)), name
    # the device codes are the hardware conversion of fl(x / s)
    t = torch.from_numpy((xv / np.float32(scale)).astype(np.float32)).cuda()
    assert torch.equal(nat.fp_encode(t, f.name).reshape(-1), codes.reshape(-1)), name
    # quantize_tensor passes num_attempts through, quantize_tensor_codes returns the same codes
    from source.quantization import quantize_tensor, quantize_tensor_codes
    assert torch.equal(quantize_tensor(x.cuda(), f.bits, f.name, num_attempts=nc), xq.reshape(x.shape))
    out, c2, _ = quantize_tensor_codes(x.cuda(), f.bits, f.name, num_attempts=nc)
    assert torch.equal(c2.reshape(-1), codes.reshape(-1)) and torch.equal(out, xq.reshape(x.shape))


@pytest.mark.gpu
@by_fmt
def test_hardware_conversion_equals_the_host_rounding(hc, f):
    t, want = rounding_table(f)
    rnd = random_quotients(f, 50000, 5 + f.id)
    every = np.concatenate([t, rnd])
    codes = _nat().fp_encode(torch.from_numpy(every).cuda(), f.name).cpu().numpy()
    assert np.array_equal(codes[:t.size], want)
    assert np.array_equal(codes, host_round(hc, f, every))
    assert np.array_equal(codes, fp_round(f, every))


@pytest.mark.gpu
@by_fmt
def test_threshold_and_direct_sums_agree(f):
    nat = _nat()
    g = torch.Generator().manual_seed(8)
    for tag, x, nc in [("64x134", torch.randn(64, 134, generator=g), 200),
                       ("256x1141", torch.randn(256, 1141, generator=g) * 0.02, 200),
                       ("9x278", torch.randn(9, 278, generator=g) * 5, 1000),
                       ("3x7", torch.randn(3, 7, generator=g), 33)]:
        xd = x.cuda()
        n = x.numel()
        direct = nat.clip_search_sums(xd, f.bits, nc, method=0, qscheme=f.name).cpu().numpy()
        thr = nat.clip_search_sums(xd, f.bits, nc, method=1, qscheme=f.name).cpu().numpy()
        floor = 1e-13 * float((x.double() ** 2).sum()) + 1e-300
        assert np.all(np.abs(thr - direct) <= 3e-6 * np.abs(direct) + floor), tag
        exact = candidate_sums(f, x.numpy(), np.float32(x.abs().max()), nc)
        assert np.all(np.abs(thr - exact) <= 1e-9 * exact + floor), tag
        mse_d, mse_t = (direct / n).astype(np.float32), (thr / n).astype(np.float32)
        bd, bt = int(np.argmin(mse_d)), int(np.argmin(mse_t))
        if bd != bt:
            assert abs(float(mse_d[bd]) - float(mse_d[bt])) <= 3e-7 * float(mse_d[bd]), (tag, bd, bt)
        assert np.array_equal(thr, nat.clip_search_sums(xd, f.bits, nc, method=1, qscheme=f.name).cpu().numpy()), tag
        for ctas in (1, 3, 7):
            few = nat.clip_search_sums(xd, f.bits, nc, method=1, max_ctas=ctas, qscheme=f.name).cpu().numpy()
            assert np.all(np.abs(few - thr) <= 1e-11 * np.abs(thr) + floor), (tag, ctas)
            fewd = nat.clip_search_sums(xd, f.bits, nc, method=0, max_ctas=ctas, qscheme=f.name).cpu().numpy()
            assert np.all(np.abs(fewd - direct) <= 1e-11 * np.abs(direct) + floor), (tag, ctas)


def _loop_cases(sms):
    """One case per loop kernel id of test_loop_kernels.build_cases (its smallest of at least 64 elements), on each
    format."""
    by_kernel = {}
    size = lambda c: (c.I * c.R < 64, c.I * c.R)   # noqa: E731
    for c in tlk.build_cases(sms):
        k = tlk.kernel_of(c, sms)
        if k not in by_kernel or size(c) < size(by_kernel[k]):
            by_kernel[k] = c
    return [(f, c._replace(scheme=f.name, bits=f.bits)) for f in FORMATS for _, c in sorted(by_kernel.items())]


LOOP_CASES = _loop_cases(tlk._sm_count())


def test_loop_cases_reach_every_kernel_on_every_format():
    cases = _loop_cases(148)
    for f in FORMATS:
        assert {tlk.kernel_of(c, 148) for g, c in cases if g is f} == tlk.ALL_KERNELS


def check_one_step(f, case, kid, H0, U0, F, G, H1, U1, codes, rep):
    """One iteration on an FP grid against float64: ridge product within the kernel's bound, candidate and codes of
    V = H_ls - U, H = value(codes) * scale, the dual update and the residuals.  Returns the ambiguous share."""
    R = case.R
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
    assert scale == candidate_scales(f, absmax, case.attempts)[rep.best_index]
    sums = candidate_sums(f, v32, absmax, case.attempts)
    ref = int(np.argmin(sums))
    if rep.best_index != ref:
        assert abs(sums[rep.best_index] - sums[ref]) <= 3e-7 * sums[ref], (rep.best_index, ref)
    outward = lambda x, to: np.where(band > 0, np.nextafter(tlk._f32(x), np.float32(to)), v32)   # noqa: E731
    lo = quantize(f, outward(v64 - band, -np.inf), scale)[0]
    hi = quantize(f, outward(v64 + band, np.inf), scale)[0]
    ambiguous = lo != hi
    assert int(np.count_nonzero((codes != lo) & ~ambiguous)) == 0, "codes differ from the exact projection of V"
    assert float(ambiguous.mean()) <= 1e-3
    assert np.array_equal((values(f, codes) * scale).astype(np.float32).view(np.uint32), H1.view(np.uint32))
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
@pytest.mark.parametrize("f,case", LOOP_CASES, ids=[f"{f.name.split('_')[-1]}-{tlk.case_id(c)}" for f, c in LOOP_CASES])
def test_loop_kernel_fp(f, case, capsys):
    nat = _nat()
    sms = tlk._sm_count()
    kid = tlk.kernel_of(case, sms)
    H0, U0, F, G = tlk._problem(case, 6000 + LOOP_CASES.index((f, case)))
    I, R, p, b, na, bits = case.I, case.R, case.precision, case.budget, case.attempts, f.bits
    d = lambda t: t.cuda().contiguous()   # noqa: E731
    Fd, Gd = d(F), d(G)
    H, U = d(H0), d(U0)
    codes = torch.empty(I, R, dtype=torch.int8, device="cuda")
    rep = nat.read_report(nat.admm_iteration_inplace(H, U, Fd, Gd, 2, 0.0, bits, f.name, na, codes=codes, precision=p,
                                                     max_ctas=b))
    assert rep.iterations == 1 and rep.status == 0, (rep.iterations, rep.status)
    amb = check_one_step(f, case, kid, H0, U0, F, G, H, U, codes, rep)
    Minv, rho, st, m64 = nat.spd_inverse(Gd, minv64=True, max_ctas=b)
    m64 = m64 if p == 0 else None
    ws = torch.empty(nat.admm_loop_workspace_bytes(I, R, na), dtype=torch.uint8, device="cuda")

    def loop(Hx, Ux, cx, iters, eps, Fx=Fd):
        return nat.read_report(nat.admm_loop_inplace(Hx, Ux, Fx, Minv, rho, st, iters + 1, eps, bits, f.name, na, codes=cx,
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
    assert np.array_equal((values(f, ck.cpu().numpy()) * np.float32(rk.scale)).view(np.uint32),
                          Hk.cpu().numpy().view(np.uint32))
    if f.bits == 6:
        assert int(ck.min()) >= 0 and int(ck.max()) <= 63
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
    for scheme in (f.name, tlk.MSE):
        Hn, Un = d(H0), d(U0)
        Hn.view(-1)[I * R // 2] = float("nan")
        r = nat.read_report(nat.admm_loop_inplace(Hn, Un, Fd, Minv, rho, st, 4, 0.0, bits, scheme, na, ws=ws, precision=p,
                                                  max_ctas=b, minv64=m64))
        nan_runs.append((r.status, r.iterations, torch.isnan(Hn).cpu(), torch.isnan(Un).cpu()))
    (s0, i0, h0, u0), (s1, i1, h1, u1) = nan_runs
    assert (s0, i0) == (s1, i1) and torch.equal(h0, h1) and torch.equal(u0, u1), (s0, i0, s1, i1)
    # an all-zero V: the degenerate range of the clip search
    Hz, Uz = d(torch.zeros(I, R)), d(torch.zeros(I, R))
    rz = loop(Hz, Uz, torch.empty(I, R, dtype=torch.int8, device="cuda"), 3, 0.0, Fx=torch.zeros_like(Fd))
    assert rz.status & nat.ST_NONFINITE and rz.iterations == 1 and bool(torch.isnan(Hz).all()), (rz.status, rz.iterations)
    with capsys.disabled():
        print(f"\n[fp loop] {f.name} {tlk.case_id(case)} {tlk.kernel_name(kid)}: ambiguous {amb:.2e}, exit at {j + 1}",
              end="")


@pytest.mark.gpu
@by_fmt
def test_split_loop_runs_fp(f):
    """One step of the two-block splitting (scripts/factorize_lowrank.py:85-88) on each format, then a longer run."""
    nat = _nat()
    g = torch.Generator().manual_seed(13)
    n = 40000
    W, H2, H, U = (torch.randn(n, generator=g) for _ in range(4))
    rho = 0.7
    Hd, Ud = H.cuda(), (U * 0.1).cuda()
    U0 = Ud.cpu().numpy()
    codes = torch.empty(n, dtype=torch.int8, device="cuda")
    rep = nat.read_report(nat.split_loop_inplace(Hd, Ud, W.cuda(), H2.cuda(), rho, 2, 0.0, f.bits, f.name, codes=codes))
    assert rep.iterations == 1 and rep.status == 0
    r = np.float32(rho)
    hls = ((r * (H.numpy() + U0) + W.numpy() - H2.numpy()) / (np.float32(1.0) + r)).astype(np.float32)
    v = (hls - U0).astype(np.float32)
    absmax = np.float32(np.abs(v).max())
    assert rep.absmax == absmax
    sums = candidate_sums(f, v, absmax, 200)
    ref = int(np.argmin(sums))
    if rep.best_index != ref:
        assert abs(sums[rep.best_index] - sums[ref]) <= 3e-7 * sums[ref]
    scale = np.float32(rep.scale)
    assert scale == candidate_scales(f, absmax, 200)[rep.best_index]
    want_codes, want_values = quantize(f, v, scale)
    assert np.array_equal(codes.cpu().numpy(), want_codes)
    assert np.array_equal(Hd.cpu().numpy().view(np.uint32), want_values.view(np.uint32))
    assert np.array_equal(Ud.cpu().numpy(), (U0 + (want_values - hls)).astype(np.float32))
    rep = nat.read_report(nat.split_loop_inplace(Hd, Ud, W.cuda(), H2.cuda(), rho, 50, 0.0, f.bits, f.name, codes=codes))
    assert rep.iterations == 49 and rep.status == 0
    assert np.array_equal(values(f, codes.cpu().numpy()) * np.float32(rep.scale), Hd.cpu().numpy())


@pytest.mark.gpu
@by_fmt
def test_layer_solver_equals_factorize_cp3_on_layer1_conv1(f):
    """A few sweeps of layer1.0.conv1 (64 x 64 x 9, rank 134) in both solver paths; every quantized factor on the grid."""
    from source import workloads as wl
    from source.solver import LayerSolver
    nat = _nat()
    g = torch.Generator().manual_seed(17)
    W = (torch.randn(64, 64, 9, generator=g) * 0.05).cuda()
    R = 134
    init = wl.random_init((64, 64, 9), R, 3)
    for prec in (0, 1):
        s = LayerSolver(W, [t.cuda() for t in init], f.bits, f.name, max_iter_admm=30, solve_precision=prec,
                        mttkrp_precision=prec)
        n_py = s.run(3)
        fac = [t.clone().cuda() for t in init]
        du = [torch.zeros_like(t) for t in fac]
        hist, histq, n_c, fq = nat.factorize(W, fac, du, f.bits, f.name, 3, 30, solve_precision=prec,
                                             mttkrp_precision=prec)
        assert n_c == n_py and hist == s.loss_hist and histq == s.loss_quant_hist, (prec, hist, s.loss_hist)
        for a, b in zip(fac + du + fq, s.factors + s.duals + s.factors_q):
            assert torch.equal(a, b)
        for t, q in zip(fac, fq):
            xq, codes, info = nat.project(t, f.bits, f.name, want_codes=True, want_info=True)
            assert torch.equal(xq, q)
            scale = np.float32(info[0].item())
            assert np.array_equal(values(f, codes.cpu().numpy()) * scale, q.cpu().numpy())
        assert all(np.isfinite(hist)) and histq[-1] < histq[0] * 1.5


@pytest.mark.gpu
def test_factorize_script_runs_e4m3(tmp_path):
    w = torch.randn(64, 64, 3, 3, generator=torch.Generator().manual_seed(1)) * 0.05
    wf = tmp_path / "w.pt"
    torch.save(w, wf)
    out = tmp_path / "out"
    r = subprocess.run([sys.executable, os.path.join(PKG, "scripts", "factorize.py"), "--model-name", "resnet18",
                        "--method", "admm", "--layer", "layer1.0.conv1", "--reduction-rate", "2", "--bits", "8",
                        "--qscheme", "tensor_mseminmax_e4m3", "--seed", "0", "--max_iter_als", "2", "--max_iter_admm",
                        "20", "--weight-file", str(wf), "--outdir", str(out)], capture_output=True, text=True,
                       cwd=str(tmp_path))
    assert r.returncode == 0, r.stdout[-2000:] + r.stderr[-2000:]
    files = sorted(os.listdir(out))
    assert any(f.endswith("_losshist.pt") for f in files), files
    assert sum(f.endswith(tuple(f"_mode_{m}.pt" for m in range(3))) for f in files) == 3, files
