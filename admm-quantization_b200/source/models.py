"""CP-format layers built from factor matrices - the consumer side of the factor files the solver writes
(reference source/models.py:24-74, used by scripts/calibrate.py:151-189).

A rank-R CP factorization W[o, i, k] = sum_r A[o, r] B[i, r] C[k, r] of a (Cout, Cin, kh*kw) convolution weight is
the composition of three convolutions: a 1x1 Cin -> R with weight B^T, a depthwise kh x kw on the R channels with
the r-th filter C[:, r] (which carries the padding and stride of the original layer), and a 1x1 R -> Cout with
weight A (which carries the bias).  A 1x1 convolution (2-D factorization W = A B^T) needs only the two pointwise
layers.  Module and parameter names (conv1 / conv2 / conv3, fc1 / fc2) follow the reference so that state dicts are
interchangeable.
"""
from collections import OrderedDict

import torch
from torch import nn


def _set(conv, weight, bias=None):
    assert tuple(conv.weight.shape) == tuple(weight.shape), \
        f"Expected shape: {tuple(conv.weight.shape)}, but got {tuple(weight.shape)}"
    with torch.no_grad():
        conv.weight = nn.Parameter(weight.detach().clone().contiguous(), requires_grad=True)
        if bias is not None:
            assert tuple(conv.bias.shape) == tuple(bias.shape), \
                f"Expected shape: {tuple(conv.bias.shape)}, but got {tuple(bias.shape)}"
            conv.bias = nn.Parameter(bias.detach().clone(), requires_grad=True)


def build_cp_layer(rank, factors, bias, cin, cout, kernel_size, padding, stride, groups):
    """reference source/models.py:24-50.  factors = [A (cout, R), B (cin, R), C (kh*kw, R)] or None/[] for an
    uninitialised skeleton."""
    has_bias = bias is not None
    seq = nn.Sequential(OrderedDict([
        ("conv1", nn.Conv2d(cin, rank, kernel_size=(1, 1), groups=groups, bias=False)),
        ("conv2", nn.Conv2d(rank, rank, kernel_size=kernel_size, groups=rank, padding=padding, stride=stride, bias=False)),
        ("conv3", nn.Conv2d(rank, cout, kernel_size=(1, 1), bias=has_bias)),
    ]))
    if factors:
        A, B, C = factors
        kh, kw = kernel_size
        _set(seq.conv1, B.t()[:, :, None, None])                                   # (R, cin, 1, 1)
        _set(seq.conv2, C.reshape(kh, kw, rank).permute(2, 0, 1)[:, None, :, :])   # (R, 1, kh, kw)
        _set(seq.conv3, A[:, :, None, None], bias if has_bias else None)          # (cout, R, 1, 1)
    return seq


def build_cp2conv_layer(rank, factors, bias, cin, cout, padding, stride):
    """reference source/models.py:53-74: a factorized 1x1 convolution, factors = [A (cout, R), B (cin, R)]."""
    has_bias = bias is not None
    seq = nn.Sequential(OrderedDict([
        ("conv1", nn.Conv2d(cin, rank, kernel_size=(1, 1), padding=padding, stride=stride, bias=False)),
        ("conv2", nn.Conv2d(rank, cout, kernel_size=(1, 1), bias=has_bias)),
    ]))
    if factors:
        A, B = factors
        _set(seq.conv1, B.t()[:, :, None, None])
        _set(seq.conv2, A[:, :, None, None], bias if has_bias else None)
    return seq


def build_cpfc_layer(rank, factors, bias, fin, fout):
    """reference source/models.py:77-95: a factorized linear layer, factors = [A (fout, R), B (fin, R)]."""
    has_bias = bias is not None
    seq = nn.Sequential(OrderedDict([
        ("fc1", nn.Linear(fin, rank, bias=False)),
        ("fc2", nn.Linear(rank, fout, bias=has_bias)),
    ]))
    if factors:
        A, B = factors
        _set(seq.fc1, B.t())
        _set(seq.fc2, A, bias if has_bias else None)
    return seq


def get_submodule(model, path):
    mod = model
    for attr in path.split("."):
        mod = getattr(mod, attr)
    return mod


def replace_with_cp(model, layer_path, factors, rank=None):
    """Swap the convolution at `layer_path` for its CP form built from `factors` (the loop body of
    reference scripts/calibrate.py:161-189).  Returns the new module."""
    layer = get_submodule(model, layer_path)
    rank = factors[0].shape[1] if rank is None else rank
    bias = layer.bias.detach() if layer.bias is not None else None
    dev = layer.weight.device
    factors = [f.to(device=dev, dtype=torch.float32) for f in factors]
    if tuple(layer.kernel_size) != (1, 1):
        new = build_cp_layer(rank, factors, bias, layer.in_channels, layer.out_channels, tuple(layer.kernel_size),
                             layer.padding, layer.stride, layer.groups)
    else:
        new = build_cp2conv_layer(rank, factors, bias, layer.in_channels, layer.out_channels, layer.padding, layer.stride)
    new = new.to(dev)
    parent_path, _, leaf = layer_path.rpartition(".")
    setattr(get_submodule(model, parent_path) if parent_path else model, leaf, new)
    return new


# ---------------------------------------------------------------------------------------------------------------------
# The same three CP shapes executed on the FP8 tensor cores from the factor codes (DESIGN.md 2d).  Each pointwise layer
# (conv1 / conv3, conv1 / conv2, fc1 / fc2) is a code GEMM: the input rows are quantized to per-row E4M3, the factor's
# codes are the FP8 operand as they are (E4M3 / E5M2) or widened exactly into E4M3, and the two scales s_a[m] s_w are
# applied to the float32 accumulator.  The depthwise kh x kw layer stays a float32 torch convolution with the decoded
# factor (level x s_w); it is not where the time goes.
class CPLayerFP8(nn.Module):
    """Inference-only CP layer on the FP8 tensor cores.  `factors` = [(codes, info)] of A (out, R), B (in, R) and, for a
    kh x kw convolution, C (kh*kw, R), each from quantize_tensor_codes(f, bits, qscheme).  kind: "conv" (build_cp_layer),
    "conv1x1" (build_cp2conv_layer) or "linear" (build_cpfc_layer)."""

    def __init__(self, kind, rank, factors, bias, bits, qscheme, cin, cout, kernel_size=(1, 1), padding=(0, 0),
                 stride=(1, 1)):
        super().__init__()
        from . import _native
        assert kind in ("conv", "conv1x1", "linear"), kind
        self.kind, self.rank, self.cin, self.cout = kind, int(rank), int(cin), int(cout)
        self.kernel_size, self.padding, self.stride = tuple(kernel_size), tuple(padding), tuple(stride)
        self.fmt = _native.fp8_operand_format(bits, qscheme)
        (a_codes, a_info), (b_codes, b_info) = factors[0], factors[1]
        assert tuple(a_codes.shape) == (cout, rank) and tuple(b_codes.shape) == (cin, rank), (a_codes.shape, b_codes.shape)
        self.register_buffer("w1", _native.codes_to_fp8(b_codes, bits, qscheme, transpose=True))   # (R, ld16(cin))
        self.register_buffer("s1", b_info[:1].to(torch.float32).clone())
        self.register_buffer("w2", _native.codes_to_fp8(a_codes, bits, qscheme))                   # (cout, ld16(R))
        self.register_buffer("s2", a_info[:1].to(torch.float32).clone())
        self.register_buffer("bias", None if bias is None else bias.detach().to(torch.float32).contiguous().clone())
        if kind == "conv":
            c_codes, c_info = factors[2]
            kh, kw = self.kernel_size
            assert tuple(c_codes.shape) == (kh * kw, rank), c_codes.shape
            c = _native.codes_to_fp8(c_codes, bits, qscheme)[:, :rank].view(_native.FP8_DTYPES[self.fmt]).float()
            c = c * c_info[:1].to(torch.float32)
            self.register_buffer("dw", c.reshape(kh, kw, rank).permute(2, 0, 1)[:, None, :, :].contiguous())

    def _pointwise(self, rows, w8, sw, K, bias=None):
        from . import _native
        q, s = _native.fp8_quantize_rows(rows)
        return _native.code_gemm(q, s, w8, sw, K, self.fmt, bias)

    @torch.no_grad()
    def forward(self, x):
        x = x.to(torch.float32)
        if self.kind == "linear":
            lead = x.shape[:-1]
            y = self._pointwise(x.reshape(-1, self.cin).contiguous(), self.w1, self.s1, self.cin)
            y = self._pointwise(y, self.w2, self.s2, self.rank, self.bias)
            return y.reshape(*lead, self.cout)
        if self.kind == "conv1x1":   # conv1 carries the padding and stride of the original layer
            ph, pw = self.padding
            if ph or pw:
                x = torch.nn.functional.pad(x, (pw, pw, ph, ph))
            x = x[:, :, ::self.stride[0], ::self.stride[1]]
        n, _, h, w = x.shape
        y = self._pointwise(x.permute(0, 2, 3, 1).reshape(-1, self.cin).contiguous(), self.w1, self.s1, self.cin)
        if self.kind == "conv":
            y = y.reshape(n, h, w, self.rank).permute(0, 3, 1, 2)
            y = torch.nn.functional.conv2d(y, self.dw, stride=self.stride, padding=self.padding, groups=self.rank)
            n, _, h, w = y.shape
            y = y.permute(0, 2, 3, 1).reshape(-1, self.rank).contiguous()
        y = self._pointwise(y, self.w2, self.s2, self.rank, self.bias)
        return y.reshape(n, h, w, self.cout).permute(0, 3, 1, 2).contiguous()


def build_cp_layer_fp8(rank, factors, bias, cin, cout, kernel_size, padding, stride, groups, bits, qscheme):
    """build_cp_layer on the FP8 tensor cores; factors = [(codes, info)] of A, B, C."""
    if groups != 1:
        raise NotImplementedError("CPLayerFP8: grouped convolutions (groups != 1) are not supported")
    return CPLayerFP8("conv", rank, factors, bias, bits, qscheme, cin, cout, kernel_size, _pair(padding), _pair(stride))


def build_cp2conv_layer_fp8(rank, factors, bias, cin, cout, padding, stride, bits, qscheme):
    """build_cp2conv_layer on the FP8 tensor cores; factors = [(codes, info)] of A, B."""
    return CPLayerFP8("conv1x1", rank, factors, bias, bits, qscheme, cin, cout, (1, 1), _pair(padding), _pair(stride))


def build_cpfc_layer_fp8(rank, factors, bias, fin, fout, bits, qscheme):
    """build_cpfc_layer on the FP8 tensor cores; factors = [(codes, info)] of A, B."""
    return CPLayerFP8("linear", rank, factors, bias, bits, qscheme, fin, fout)


def _pair(v):
    return tuple(v) if isinstance(v, (tuple, list)) else (int(v), int(v))


def replace_with_cp_fp8(model, layer_path, factors, bits, qscheme, num_attempts=200):
    """replace_with_cp for execution on the FP8 tensor cores: each float factor is re-projected with
    quantize_tensor_codes (the re-projection behind the solver's quant_rec_error), and the convolution or linear layer at
    `layer_path` is swapped for a CPLayerFP8 built from the codes.  Returns the new module."""
    from .quantization import quantize_tensor_codes
    layer = get_submodule(model, layer_path)
    dev = layer.weight.device
    coded = []
    for f in factors:
        _, codes, info = quantize_tensor_codes(f.to(device=dev, dtype=torch.float32).contiguous(), bits, qscheme,
                                               num_attempts=num_attempts)
        coded.append((codes, info))
    rank = factors[0].shape[1]
    bias = layer.bias.detach() if layer.bias is not None else None
    if isinstance(layer, nn.Linear):
        new = build_cpfc_layer_fp8(rank, coded, bias, layer.in_features, layer.out_features, bits, qscheme)
    elif tuple(layer.kernel_size) != (1, 1):
        new = build_cp_layer_fp8(rank, coded, bias, layer.in_channels, layer.out_channels, tuple(layer.kernel_size),
                                 layer.padding, layer.stride, layer.groups, bits, qscheme)
    else:
        if layer.groups != 1:
            raise NotImplementedError("CPLayerFP8: grouped convolutions (groups != 1) are not supported")
        new = build_cp2conv_layer_fp8(rank, coded, bias, layer.in_channels, layer.out_channels, layer.padding, layer.stride,
                                      bits, qscheme)
    parent_path, _, leaf = layer_path.rpartition(".")
    setattr(get_submodule(model, parent_path) if parent_path else model, leaf, new)
    return new
