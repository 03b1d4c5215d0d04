"""CP layers on the FP8 tensor cores from their factor codes (csrc/code_gemm.cu, DESIGN.md 2d): the code -> FP8 operand
mapping, per-row E4M3 activations, the tcgen05 kind::f8f6f4 code GEMM against float64, the CPLayerFP8 modules against a
float64 restatement and against the float32 CP layer, a trained model's top-1, and calibrate.py --execute fp8."""
import ctypes
import math
import os
import subprocess
import sys

import numpy as np
import pytest
import torch

REPO = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
PKG = os.path.join(REPO, "admm-quantization_b200")

E4M3, E5M2 = "tensor_mseminmax_e4m3", "tensor_mseminmax_e5m2"
SYM, MSE = "tensor_symmetric", "tensor_mseminmax_symmetric"
IDS = {MSE: 0, "tensor_minmax": 1, SYM: 2, "tensor_affine": 3, "tensor_mseminmax_e2m1": 4, E4M3: 6, E5M2: 7,
       "tensor_mseminmax_e3m2": 8, "tensor_mseminmax_e2m3": 9}
# (qscheme, bits) of every grid with an exact FP8 operand, and the operand format
GRIDS = [(MSE, b) for b in range(1, 6)] + [(SYM, b) for b in range(2, 6)] + [
    ("tensor_mseminmax_e2m1", 4), (E4M3, 8), (E5M2, 8), ("tensor_mseminmax_e3m2", 6), ("tensor_mseminmax_e2m3", 6)]


def _nat():
    from source import _native
    return _native


# ---------------------------------------------------------------------------------------------------- the definition
def levels(qscheme, bits):
    """{code: grid level} of every code of the grid, computed from the format's definition (not from the library)."""
    if qscheme in (MSE, SYM):
        q = 2 ** (bits - 1)
        return {c: float(c) for c in range(-q, q)}
    if qscheme == "tensor_mseminmax_e2m1":
        mag = [0.0, 0.5, 1.0, 1.5, 2.0, 3.0, 4.0, 6.0]
        return {c: math.copysign(mag[c & 7], -1.0 if c & 8 else 1.0) for c in range(16)}
    if qscheme in ("tensor_mseminmax_e3m2", "tensor_mseminmax_e2m3"):
        eb, mb, bias = (3, 2, 3) if qscheme.endswith("e3m2") else (2, 3, 1)
        out = {}
        for c in range(64):
            e, m = (c >> mb) & ((1 << eb) - 1), c & ((1 << mb) - 1)
            mag = m * 2.0 ** (1 - bias - mb) if e == 0 else (1 + m / 2 ** mb) * 2.0 ** (e - bias)
            out[c] = math.copysign(mag, -1.0 if c & 32 else 1.0)
        return out
    dt = torch.float8_e4m3fn if qscheme == E4M3 else torch.float8_e5m2
    vals = torch.arange(256, dtype=torch.int32).to(torch.uint8).view(dt).float().tolist()
    return {(c - 256 if c > 127 else c): v for c, v in enumerate(vals) if math.isfinite(v)}


def fp8_lut(qscheme, bits):
    """256-entry uint8 table, indexed by the code's byte: the operand byte of the definition (torch's own E4M3 cast of
    the level; the FP8 grids pass through)."""
    lut = np.zeros(256, np.uint8)
    for c, v in levels(qscheme, bits).items():
        if qscheme in (E4M3, E5M2):
            lut[c & 0xFF] = c & 0xFF
        else:
            lut[c & 0xFF] = torch.tensor([v]).to(torch.float8_e4m3fn).view(torch.uint8).item()
    return lut


def fp8_values(b, fmt):
    """float64 values of uint8 FP8 bytes."""
    dt = torch.float8_e5m2 if fmt == E5M2 else torch.float8_e4m3fn
    return torch.as_tensor(b).cpu().contiguous().view(dt).to(torch.float64)


def ref_quantize_rows(x):
    """Host restatement of the activation rule: float32 division, clamp to +-448, torch's float8_e4m3fn cast."""
    x = x.detach().cpu().to(torch.float32)
    amax = x.abs().amax(dim=1)
    s = amax / torch.tensor(448.0)
    s = torch.where(torch.isfinite(amax), s, torch.full_like(s, float("nan")))
    t = (x / s[:, None]).clamp(-448.0, 448.0)
    q = t.to(torch.float8_e4m3fn).view(torch.uint8)
    q = torch.where((s == 0)[:, None], torch.zeros_like(q), q)
    return q, s


@pytest.fixture(scope="module")
def hc(tmp_path_factory):
    so = str(tmp_path_factory.mktemp("code8") / "libcode8check.so")
    subprocess.check_call(["g++", "-O2", "-ffp-contract=off", "-std=c++17", "-shared", "-fPIC",
                           os.path.join(REPO, "tests", "hostcheck", "code8check.cpp"), "-o", so])
    return ctypes.CDLL(so)


# ---------------------------------------------------------------------------------------------------- CPU
@pytest.mark.parametrize("qscheme,bits", GRIDS)
def test_every_code_maps_to_its_level(hc, qscheme, bits):
    """Every code's operand byte, read as float8_e4m3fn (E5M2 for that grid), is the grid level exactly, +-0 included;
    the FP8 grids pass through unchanged."""
    fmt = E5M2 if qscheme == E5M2 else E4M3
    assert hc.hc_fp8_operand_format(IDS[qscheme], bits) == IDS[fmt]
    for c, level in levels(qscheme, bits).items():
        b = hc.hc_code_to_fp8(IDS[qscheme], c)
        v = fp8_values(torch.tensor([b], dtype=torch.uint8), fmt).item()
        assert v == level and math.copysign(1.0, v) == math.copysign(1.0, level), (qscheme, bits, c, b, v, level)
        if qscheme in (E4M3, E5M2):
            assert b == c & 0xFF
    assert np.array_equal(fp8_lut(qscheme, bits), np.array([hc.hc_code_to_fp8(IDS[qscheme], c - 256 if c > 127 else c)
                                                            if (c - 256 if c > 127 else c) in levels(qscheme, bits) else 0
                                                            for c in range(256)], np.uint8))


def test_operand_format_and_its_refusals():
    nat = _nat()
    for qs, bits in GRIDS:
        assert nat.fp8_operand_format(bits, qs) == (E5M2 if qs == E5M2 else E4M3)
    bad = [(MSE, 6, "bits 1 .. 5"), (MSE, 8, "17 is not"), (SYM, 6, "17 is not"), ("tensor_affine", 4, "zero point"),
           ("tensor_minmax", 4, "minimum"), (E4M3, 4, "bits = 8"), ("tensor_mseminmax_e2m1", 8, "bits = 4"),
           ("tensor_mseminmax_e3m2", 8, "bits = 6")]
    for qs, bits, why in bad:
        with pytest.raises(ValueError, match=why):
            nat.fp8_operand_format(bits, qs)
        with pytest.raises(ValueError):   # refused before anything touches a device
            nat.codes_to_fp8(torch.zeros(4, 4, dtype=torch.int8), bits, qs)
    with pytest.raises(NotImplementedError):
        nat.fp8_operand_format(4, "channel_symmetric")


def test_entry_points_check_their_arguments():
    """Argument checks run before any device work: they hold on a machine without a GPU."""
    nat = _nat()
    lib, p = nat.lib, ctypes.c_void_p(256)
    gemm = lambda lda, ldb, M, N, K, fmt=6, ldd=None: int(lib.admmq_code_gemm(
        p, lda, p, M, p, ldb, p, fmt, N, K, None, p, N if ldd is None else ldd, None))
    assert gemm(64, 64, 8, 8, 0) == nat.E_BADARG                  # K <= 0
    assert gemm(40, 64, 8, 8, 33) == nat.E_BADARG                 # lda not a multiple of 16
    assert gemm(48, 32, 8, 8, 33) == nat.E_BADARG                 # ldb < K
    assert gemm(64, 64, 8, 8, 33, fmt=4) == nat.E_BADARG          # B format neither E4M3 nor E5M2
    assert gemm(64, 64, 8, 8, 33, ldd=7) == nat.E_BADARG          # ldd < N
    assert gemm(1 << 16, 64, 1 << 15, 8, 33) == nat.E_UNSUPPORTED   # M * lda = 2^31
    q = lambda ldx, M, K, ldq: int(lib.admmq_fp8_quantize_rows(p, ldx, M, K, p, ldq, p, None))
    assert q(8, 4, 0, 16) == nat.E_BADARG
    assert q(8, 4, 9, 16) == nat.E_BADARG                         # ldx < K
    assert q(32, 4, 20, 24) == nat.E_BADARG                       # ldq not a multiple of 16
    assert q(1 << 16, 1 << 15, 20, 32) == nat.E_UNSUPPORTED
    c = lambda rows, cols, bits, qs, tr, ldo: int(lib.admmq_codes_to_fp8(p, rows, cols, bits, qs, tr, p, ldo, None))
    assert c(4, 20, 4, 0, 0, 16) == nat.E_BADARG                  # ldo < cols
    assert c(20, 4, 4, 0, 1, 16) == nat.E_BADARG                  # transposed: ldo < rows
    assert c(4, 20, 4, 3, 0, 32) == nat.E_BADARG                  # tensor_affine
    assert c(1 << 27, 16, 4, 0, 1, 1 << 27) == nat.E_UNSUPPORTED   # 16 x 2^27 output bytes


def test_tile_width_rule_reaches_every_width():
    """admmq_code_gemm_kernel: whole waves of 128 x bn tiles; every width 16 .. 256 is the choice for some shape."""
    nat = _nat()
    seen = {}
    for N in range(1, 1200):
        for M in (128, 128 * 148, 128 * 148 * 4 + 1):
            bn, grid = nat.code_gemm_kernel(M, N, 64, 148)
            assert bn % 16 == 0 and 16 <= bn <= 256 and 1 <= grid <= 148
            seen.setdefault(bn, (M, N))
    assert sorted(seen) == list(range(16, 257, 16)), sorted(seen)
    assert nat.code_gemm_kernel(8192, 8192, 8192, 148)[0] == 256


# ---------------------------------------------------------------------------------------------------- GPU: operands
def _factor_shapes():
    from source import workloads as wl
    from source.shapes import rank_from_reduction_rate
    shapes = set()
    for name, cout, cin, kh, kw in wl.resnet18_conv_layers() + wl.llama7b_linear_layers():
        W = torch.empty(cout, cin, kh * kw) if kh * kw > 1 else torch.empty(cout, cin)
        R = rank_from_reduction_rate(W, 2.0)
        shapes |= {(cout, R), (cin, R)} | ({(kh * kw, R)} if kh * kw > 1 else set())
    return sorted(shapes) + [(1, 1), (3, 17), (17, 3), (33, 129), (130, 15)]


def _random_codes(qscheme, bits, shape, seed):
    g = torch.Generator().manual_seed(seed)
    valid = torch.tensor(sorted(levels(qscheme, bits)), dtype=torch.int64)
    return valid[torch.randint(0, len(valid), shape, generator=g)].to(torch.int8)


@pytest.mark.gpu
def test_codes_to_fp8_bit_exact_at_every_factor_shape():
    nat = _nat()
    for i, (rows, cols) in enumerate(_factor_shapes()):
        qs, bits = GRIDS[i % len(GRIDS)]
        codes = _random_codes(qs, bits, (rows, cols), i)
        lut = torch.from_numpy(fp8_lut(qs, bits))
        want = lut[codes.to(torch.int64) & 0xFF]
        for tr in (False, True):
            got = nat.codes_to_fp8(codes.cuda(), bits, qs, transpose=tr).cpu()
            w = want.t() if tr else want
            assert got.shape == (w.shape[0], nat.ld16(w.shape[1]))
            assert torch.equal(got[:, :w.shape[1]], w), (rows, cols, qs, tr)
            assert not got[:, w.shape[1]:].any(), "pad columns must be zero"


def _activation_cases():
    g = torch.Generator().manual_seed(7)
    cases = []
    for K in (1, 15, 16, 17, 64, 130, 1141):
        x = torch.randn(37, K, generator=g) * torch.logspace(-3, 3, 37)[:, None]
        x[3] = 0.0                                                           # zero row
        x[5] = torch.randn(K, generator=g) * 1e-3
        x[5, K // 2] = 1e4                                                   # one outlier: the rest goes subnormal / zero
        x[7] = torch.randn(K, generator=g) * 1e-44                           # abs-max whose scale underflows to 0
        x[9] = torch.randn(K, generator=g) * 3e-36                           # tiny but representable scale
        cases.append((f"K{K}", x))
    x = torch.randn(12, 100, generator=g)
    x[2, 17] = float("nan")
    x[6, 3] = float("inf")
    x[8, 50] = -float("inf")
    cases.append(("nonfinite", x))
    return cases


@pytest.mark.gpu
@pytest.mark.parametrize("name,x", _activation_cases(), ids=[c[0] for c in _activation_cases()])
def test_fp8_quantize_rows_bit_exact(name, x):
    nat = _nat()
    q, s = nat.fp8_quantize_rows(x.cuda())
    q, s = q.cpu(), s.cpu()
    qr, sr = ref_quantize_rows(x)
    K = x.shape[1]
    assert q.shape == (x.shape[0], nat.ld16(K)) and not q[:, K:].any()
    bad = ~torch.isfinite(x).all(dim=1)                     # NaN or infinite abs-max: s = NaN, every code NaN
    assert torch.isnan(s[bad]).all() and ((q[bad, :K] & 0x7F) == 0x7F).all()
    ok = ~bad
    assert torch.equal(s[ok].view(torch.int32), sr[ok].view(torch.int32)), name
    assert torch.equal(q[ok, :K], qr[ok]), name
    if name == "K64":
        assert s[3] == 0 and not q[3].any() and s[7] == 0 and not q[7].any()   # zero row, underflowing scale
        assert ((q[5, :K] & 0x7F) < 8).sum() > K // 2                              # the outlier row: subnormal codes


# ---------------------------------------------------------------------------------------------------- GPU: code GEMM
def _fp8_operand(shape, fmt, g, spread=2.0):
    """Random finite FP8 bytes of `fmt`: float values of several magnitudes cast to the format."""
    v = torch.randn(shape, generator=g) * torch.exp(torch.randn(shape, generator=g) * spread)
    dt = torch.float8_e5m2 if fmt == E5M2 else torch.float8_e4m3fn
    top = 57344.0 if fmt == E5M2 else 448.0
    return v.clamp(-top, top).to(dt).view(torch.uint8)


def _padded(b, ld):
    out = torch.zeros(b.shape[0], ld, dtype=torch.uint8)
    out[:, :b.shape[1]] = b
    return out


def gemm_check(M, N, K, fmt, with_bias, seed, worst):
    """code_gemm against float64 of the decoded operands.  Bound (DESIGN.md 2d):
    |D - D64| <= (K/32) 2^-22 |s_a s_w| sum_k |a_k b_k| + 2^-23 |P64| (+ 2^-23 |D64| with a bias), P64 = s_a s_w sum a b."""
    nat = _nat()
    g = torch.Generator().manual_seed(seed)
    a = _fp8_operand((M, K), E4M3, g)
    b = _fp8_operand((N, K), fmt, g)
    sa = torch.rand(M, generator=g) * 1e-2 + 1e-4
    sw = torch.rand(1, generator=g) * 1e-2 + 1e-4
    bias = torch.randn(N, generator=g) if with_bias else None
    ld = nat.ld16(K)
    D = nat.code_gemm(_padded(a, ld).cuda(), sa.cuda(), _padded(b, ld).cuda(), sw.cuda(), K, fmt,
                      None if bias is None else bias.cuda()).double()
    D = D.cuda()   # the float64 reference runs on the device too (FP64 pipe): the Llama shapes are 10^11 operations
    A64, B64 = fp8_values(a, E4M3).cuda(), fp8_values(b, fmt).cuda()
    s64 = sa.double().cuda()[:, None] * sw.double().cuda()
    P64 = (A64 @ B64.t()) * s64
    absum = (A64.abs() @ B64.abs().t()) * s64
    D64 = P64 + (bias.double().cuda()[None, :] if with_bias else 0.0)
    bound = (K / 32) * 2.0 ** -22 * absum + 2.0 ** -23 * P64.abs() + (2.0 ** -23 * D64.abs() if with_bias else 0.0)
    err = (D - D64).abs()
    assert torch.isfinite(D).all()
    zero = bound == 0
    assert torch.equal(err[zero], torch.zeros_like(err[zero])), (M, N, K)
    ratio = (err[~zero] / bound[~zero]).max().item() if (~zero).any() else 0.0
    worst[0] = max(worst[0], ratio)
    assert ratio <= 1.0, (M, N, K, fmt, with_bias, ratio)


_MS, _NS, _KS = (1, 2, 127, 128, 129, 4096), (1, 15, 16, 17, 255, 256, 257, 1141), (1, 31, 32, 33, 127, 128, 129, 4096)


def _gemm_shapes():
    shapes = {(129, n, k) for n in _NS for k in _KS}
    shapes |= {(m, n, 129) for m in _MS for n in _NS}
    shapes |= {(m, 257, k) for m in _MS for k in _KS}
    from source import workloads as wl
    from source.shapes import rank_from_reduction_rate
    for name, cout, cin, kh, kw in wl.resnet18_conv_layers():
        R = rank_from_reduction_rate(torch.empty(cout, cin, kh * kw), 2.0)
        hw = {64: 56, 128: 28, 256: 14, 512: 7}[cout]
        stride = 2 if (cin != cout and name.endswith("conv1")) else 1
        hin = hw * stride
        shapes |= {(64 * hin * hin, R, cin), (64 * hw * hw, cout, R)}
    for name, cout, cin, _, _ in wl.llama7b_linear_layers():
        R = rank_from_reduction_rate(torch.empty(cout, cin), 2.0)
        shapes |= {(m, R, cin) for m in (1, 128, 4096)} | {(m, cout, R) for m in (1, 128, 4096)}
    return sorted(shapes)


@pytest.mark.gpu
def test_code_gemm_against_float64(capsys):
    """Every shape of the grid M x N x K of DESIGN.md 2d, the ResNet-18 CP conv GEMMs and the Llama-7B ones; E4M3 / E5M2
    weights and bias alternate.  Measured worst ratio on a B200: 0.876 (no split of K over accumulators is needed)."""
    worst = [0.0]
    for i, (M, N, K) in enumerate(_gemm_shapes()):
        fmt = E5M2 if i % 2 else E4M3
        gemm_check(M, N, K, fmt, with_bias=(i // 2) % 2 == 1, seed=i, worst=worst)
    with capsys.disabled():
        print(f"\n[code_gemm] {len(_gemm_shapes())} shapes, worst |D - D64| / bound = {worst[0]:.4f}")


@pytest.mark.gpu
@pytest.mark.parametrize("fmt", [E4M3, E5M2])
@pytest.mark.parametrize("with_bias", [False, True])
def test_code_gemm_variants(fmt, with_bias):
    worst = [0.0]
    for M, N, K in ((300, 257, 1000), (4096, 1141, 512), (1, 16, 4096)):
        gemm_check(M, N, K, fmt, with_bias, seed=M + N + K, worst=worst)


@pytest.mark.gpu
def test_code_gemm_same_bits_every_width_and_call_no_stray_writes(monkeypatch):
    nat = _nat()
    g = torch.Generator().manual_seed(3)
    M, N, K, ldd = 300, 257, 700, 270
    a = _padded(_fp8_operand((M, K), E4M3, g), nat.ld16(K)).cuda()
    b = _padded(_fp8_operand((N, K), E4M3, g), nat.ld16(K)).cuda()
    sa, sw, bias = torch.rand(M).cuda() + 0.5, torch.rand(1).cuda() + 0.5, torch.randn(N).cuda()
    ref = nat.code_gemm(a, sa, b, sw, K, E4M3, bias)
    assert torch.equal(ref, nat.code_gemm(a, sa, b, sw, K, E4M3, bias))
    for w in range(16, 257, 16):
        monkeypatch.setenv("ADMMQ_CODE_GEMM_BN", str(w))
        assert nat.code_gemm_kernel(M, N, K, 148)[0] == w
        big = torch.full((M + 3, ldd), -7.25, device="cuda")
        out = big[:M, :N]
        nat.code_gemm(a, sa, b, sw, K, E4M3, bias, out=out)
        assert torch.equal(out.view(torch.int32), ref.view(torch.int32)), w
        assert (big[:M, N:] == -7.25).all() and (big[M:] == -7.25).all(), w


# ---------------------------------------------------------------------------------------------------- GPU: layers
def _record(monkeypatch):
    """Wrap the two native steps of CPLayerFP8 so that the test sees every intermediate the module produced."""
    nat = _nat()
    log = []
    fq, fg = nat.fp8_quantize_rows, nat.code_gemm

    def quantize(x, *a, **k):
        q, s = fq(x, *a, **k)
        log.append(("q", x.clone(), q, s))
        return q, s

    def gemm(q, s, w8, sw, K, fmt, bias=None, *a, **k):
        D = fg(q, s, w8, sw, K, fmt, bias, *a, **k)
        log.append(("g", q, s, w8, sw, K, fmt, bias, D.clone()))
        return D

    monkeypatch.setattr(nat, "fp8_quantize_rows", quantize)
    monkeypatch.setattr(nat, "code_gemm", gemm)
    return log


def _check_stage(qrec, grec):
    """One pointwise stage: the activation codes equal the host restatement bit for bit, the GEMM is within its bound."""
    _, x, q, s = qrec
    qr, sr = ref_quantize_rows(x)
    K = x.shape[1]
    assert torch.equal(q.cpu()[:, :K], qr) and torch.equal(s.cpu(), sr)
    _, q2, s2, w8, sw, K2, fmt, bias, D = grec
    assert q2.data_ptr() == q.data_ptr() and K2 == K
    A64 = fp8_values(q.cpu()[:, :K], E4M3)
    B64 = fp8_values(w8.cpu()[:, :K], fmt)
    s64 = s.cpu().double()[:, None] * sw.cpu().double()
    P64 = (A64 @ B64.t()) * s64
    D64 = P64 + (0.0 if bias is None else bias.cpu().double()[None, :])
    bound = (K / 32) * 2.0 ** -22 * ((A64.abs() @ B64.abs().t()) * s64) + 2.0 ** -23 * P64.abs() + \
        (0.0 if bias is None else 2.0 ** -23 * D64.abs())
    assert ((D.cpu().double() - D64).abs() <= bound).all()
    return D


def _layer_cases():
    return [("conv3x3_s1", dict(kind="conv", cin=64, cout=64, k=3, stride=1, hw=14)),
            ("conv3x3_s2", dict(kind="conv", cin=64, cout=128, k=3, stride=2, hw=14)),
            ("conv1x1_s2", dict(kind="conv1x1", cin=64, cout=128, k=1, stride=2, hw=14)),
            ("linear", dict(kind="linear", cin=512, cout=300, k=1, stride=1, hw=0))]


# Relative Frobenius error of the FP8-executed layer against the float32 CP layer on the same decoded factors: measured
# 3.48e-2 .. 3.67e-2 over these cases on a B200 (the two E4M3 activation roundings, <= 2^-4 each); asserted at twice that.
_FP32_GAP_BOUND = 7.4e-2


@pytest.mark.gpu
@pytest.mark.parametrize("qscheme,bits", [(MSE, 4), (E4M3, 8)])
@pytest.mark.parametrize("name,c", _layer_cases(), ids=[n for n, _ in _layer_cases()])
def test_layer_matches_float64_restatement(monkeypatch, capsys, name, c, qscheme, bits):
    from torch import nn
    from source.models import build_cpfc_layer, replace_with_cp, replace_with_cp_fp8
    from source.quantization import quantize_tensor_codes
    from source.shapes import layer_weight_as_tensor, rank_from_reduction_rate
    g = torch.Generator().manual_seed(11)
    if c["kind"] == "linear":
        layer = nn.Linear(c["cin"], c["cout"], bias=True)
        x = torch.randn(4, 25, c["cin"], generator=g)
    else:
        k = c["k"]
        layer = nn.Conv2d(c["cin"], c["cout"], k, stride=c["stride"], padding=k // 2, bias=True)
        x = torch.randn(2, c["cin"], c["hw"], c["hw"], generator=g)
    layer = layer.cuda()
    W = layer_weight_as_tensor(layer.weight.detach())
    R = rank_from_reduction_rate(W, 2.0)
    factors = [torch.randn(d, R, generator=g).cuda() * 0.3 for d in W.shape]
    fp8_model = nn.Sequential(layer)
    decoded = [quantize_tensor_codes(f, bits, qscheme)[0] for f in factors]
    log = _record(monkeypatch)
    new = replace_with_cp_fp8(fp8_model, "0", factors, bits, qscheme)
    x = x.cuda()
    y = new(x)
    assert [e[0] for e in log] == ["q", "g", "q", "g"]
    D1 = _check_stage(log[0], log[1])
    D2 = _check_stage(log[2], log[3])
    # the layout steps around the GEMMs, restated
    if c["kind"] == "linear":
        assert torch.equal(log[0][1], x.reshape(-1, c["cin"]))
        assert torch.equal(y, D2.reshape(4, 25, c["cout"]))
        assert torch.equal(log[2][1], D1)
    else:
        xs = x if c["kind"] == "conv" else x[:, :, ::c["stride"], ::c["stride"]]
        assert torch.equal(log[0][1], xs.permute(0, 2, 3, 1).reshape(-1, c["cin"]))
        n, _, h, w = xs.shape
        if c["kind"] == "conv":
            y1 = D1.double().reshape(n, h, w, R).permute(0, 3, 1, 2)
            y2 = torch.nn.functional.conv2d(y1, new.dw.double(), stride=c["stride"], padding=c["k"] // 2, groups=R)
            rows2 = y2.permute(0, 2, 3, 1).reshape(-1, R)
            tol = 1e-6 * torch.nn.functional.conv2d(y1.abs(), new.dw.double().abs(), stride=c["stride"],
                                                    padding=c["k"] // 2, groups=R).permute(0, 2, 3, 1).reshape(-1, R)
            assert ((log[2][1].double() - rows2).abs() <= tol).all()
            h, w = y2.shape[2:]
        else:
            assert torch.equal(log[2][1], D1)
        assert torch.equal(y, D2.reshape(n, h, w, c["cout"]).permute(0, 3, 1, 2))
    # against today's float32 CP layer on the same decoded factors
    if c["kind"] == "linear":
        ref_layer = build_cpfc_layer(R, decoded, layer.bias.detach(), c["cin"], c["cout"]).cuda()
    else:
        ref_layer = replace_with_cp(nn.Sequential(layer), "0", decoded, R)
    with torch.no_grad():
        y32 = ref_layer(x)
    rel = ((y.double() - y32.double()).norm() / y32.double().norm()).item()
    with capsys.disabled():
        print(f"\n[cp fp8 layer] {name} {qscheme}: relative Frobenius error against the float32 CP layer {rel:.3e}")
    assert rel <= _FP32_GAP_BOUND


# ---------------------------------------------------------------------------------------------------- GPU: model
@pytest.mark.gpu
@pytest.mark.parametrize("qscheme,bits", [(MSE, 4), (E4M3, 8)])
def test_model_top1_fp8_execution_vs_float32_cp(capsys, qscheme, bits):
    """The prototype-task ResNet-18 of test_gpu_parity.py, its four layer1 convolutions factorized by LayerSolver (rr = 2,
    2 sweeps x 30 inner iterations); the float32 CP model on the re-projected (decoded) factors and the model executed on
    the FP8 tensor cores from the same codes, both BN-calibrated the same way, scored on 16384 held-out images."""
    import copy
    import torchvision
    from test_gpu_parity import _PrototypeTask
    from source import workloads as wl
    from source.models import get_submodule, replace_with_cp, replace_with_cp_fp8
    from source.quantization import quantize_tensor_codes
    from source.solver import LayerSolver, layer_weight_as_tensor, rank_from_reduction_rate
    from source.utils import bncalibrate_model, top1_accuracy
    torch.set_num_threads(4)
    torch.manual_seed(42)
    torch.backends.cudnn.deterministic, torch.backends.cudnn.benchmark = True, False
    base = torchvision.models.resnet18(weights=None, num_classes=10).cuda()
    opt = torch.optim.SGD(base.parameters(), lr=0.05, momentum=0.9)
    base.train()
    for x, y in _PrototypeTask(120, 128, seed=5):
        opt.zero_grad()
        torch.nn.functional.cross_entropy(base(x), y).backward()
        opt.step()
    base.eval()
    fp32, fp8 = copy.deepcopy(base), copy.deepcopy(base)
    for path in ("layer1.0.conv1", "layer1.0.conv2", "layer1.1.conv1", "layer1.1.conv2"):
        W = layer_weight_as_tensor(get_submodule(base, path).weight.detach()).contiguous()
        R = rank_from_reduction_rate(W, 2.0)
        s = LayerSolver(W, [f.cuda() for f in wl.random_init(W.shape, R, 42)], bits, qscheme, max_iter_admm=30,
                        solve_precision=1, mttkrp_precision=1)
        for _ in range(2):
            s.sweep()
        replace_with_cp(fp32, path, [quantize_tensor_codes(f, bits, qscheme)[0] for f in s.factors], R)
        replace_with_cp_fp8(fp8, path, [f.clone() for f in s.factors], bits, qscheme)
    accs = []
    for m in (fp32, fp8):
        bncalibrate_model(m, _PrototypeTask(18, 64, seed=1), num_samples=1000, device="cuda")
        accs.append(top1_accuracy(m, _PrototypeTask(128, 128, seed=2), "cuda"))
    torch.set_num_threads(1)
    with capsys.disabled():
        print(f"\n[top-1 fp8] {qscheme} {bits}-bit: float32 CP model {accs[0]:.2f} %, FP8-executed {accs[1]:.2f} % "
              f"(gap {accs[1] - accs[0]:+.2f} pp)")
    assert abs(accs[1] - accs[0]) <= 0.5


@pytest.mark.gpu
def test_calibrate_execute_fp8_runs_on_factorize_output(tmp_path):
    w = torch.randn(64, 64, 3, 3, generator=torch.Generator().manual_seed(1)) * 0.05
    wf = tmp_path / "w.pt"
    torch.save(w, wf)
    out = tmp_path / "factors"
    r = subprocess.run([sys.executable, os.path.join(PKG, "scripts", "factorize.py"), "--model-name", "resnet18",
                        "--method", "admm", "--layer", "layer1.0.conv1", "--reduction-rate", "2", "--bits", "4",
                        "--qscheme", MSE, "--seed", "0", "--max_iter_als", "2", "--max_iter_admm", "20",
                        "--weight-file", str(wf), "--outdir", str(out)], capture_output=True, text=True, cwd=str(tmp_path))
    assert r.returncode == 0, r.stdout[-2000:] + r.stderr[-2000:]
    r = subprocess.run([sys.executable, os.path.join(PKG, "scripts", "calibrate.py"), "--bits", "4", "--qscheme", MSE,
                        "--seed", "0", "--layers", "layer1.0.conv1", "--factor-dir", str(out), "--execute", "fp8",
                        "--calibration-samples", "128", "--eval-batches", "2", "--batch-size", "32", "--image-size", "32"],
                       capture_output=True, text=True, cwd=str(tmp_path))
    assert r.returncode == 0, r.stdout[-2000:] + r.stderr[-2000:]
    assert "top-1 agreement" in r.stdout
