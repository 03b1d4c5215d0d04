"""Grid projection, drop-in for the reference's source/quantization.py:12-144 (tensor_* schemes).

Everything runs in libadmmq.so (csrc/project.cu); CUDA tensors only, no CPU path."""
import torch

from . import _native

_TENSOR_SCHEMES = tuple(_native.QSCHEME_IDS)
_CHANNEL_SCHEMES = ("channel_symmetric", "channel_affine")


def get_tensor_stats(tensor, qscheme, mode=0):
    """(max, min) over the whole tensor (reference source/quantization.py:12-45, tensor schemes)."""
    if qscheme in ("tensor_affine", "tensor_symmetric", "tensor_log"):
        return tensor.max(), tensor.min()
    if qscheme in _CHANNEL_SCHEMES:
        raise NotImplementedError(
            f"{qscheme}: the per-channel schemes are unreachable from the solver (dim=None) and raise in the "
            "reference as well (SURVEY App. A.2)")
    raise TypeError("Can't collect statistics. Unknown quantization scheme: {}".format(qscheme))


def min_max_quantize(input, bits, min_val=None, max_val=None):
    """reference source/quantization.py:48-66."""
    assert bits >= 1, bits
    if min_val is not None and max_val is not None:
        raise NotImplementedError("explicit min_val/max_val are not used on the solver path")
    return _native.project(input, bits, "tensor_minmax")[0].reshape(input.shape)


def quantize_tensor(tensor, bits, qscheme, dim=None, **kwargs):
    """reference source/quantization.py:69-115: project `tensor` onto the `bits`-bit grid of `qscheme`.
    kwargs: num_attempts (every clip search), tmin/tmax (affine).  tensor_mseminmax_e2m1 (bits 4), _e4m3 / _e5m2
    (bits 8) and _e3m2 / _e2m3 (bits 6) are this project's own schemes (no reference counterpart): the clip search onto
    the FP4, FP8 and FP6 grids of the B200's tensor cores."""
    if qscheme in _CHANNEL_SCHEMES:
        get_tensor_stats(tensor, qscheme, mode=dim)
    if qscheme not in _TENSOR_SCHEMES:
        raise NotImplementedError(qscheme)
    if qscheme == "tensor_mseminmax_symmetric":
        return quantize_tensor_mse(tensor, bits, **kwargs)
    if qscheme in _native.CLIP_SEARCH_SCHEMES:   # the clip search on a grid other than the uniform one
        out, _, _ = _native.project(tensor, bits, qscheme, num_attempts=kwargs.get("num_attempts", 200))
        return out.reshape(tensor.shape)
    out, _, _ = _native.project(tensor, bits, qscheme, tmin=kwargs.get("tmin"), tmax=kwargs.get("tmax"))
    return out.reshape(tensor.shape)


def quantize_tensor_mse(x, bits, num_attempts=200):
    """reference source/quantization.py:118-144: 200-candidate clip search by MSE."""
    out, _, _ = _native.project(x, bits, "tensor_mseminmax_symmetric", num_attempts=num_attempts)
    return out.reshape(x.shape)


def quantize_tensor_codes(tensor, bits, qscheme, **kwargs):
    """Extension (the reference never stores codes): (dequantized, int8 codes, info[scale, zp|min, index, absmax]).
    On the FP8 grids a code is the byte of the FP8 value (codes.view(torch.float8_e4m3fn) for tensor_mseminmax_e4m3,
    torch.float8_e5m2 for _e5m2), on the FP6 grids the encoding 0 .. 63, on E2M1 the encoding 0 .. 15."""
    out, codes, info = _native.project(tensor, bits, qscheme, num_attempts=kwargs.get("num_attempts", 200),
                                       tmin=kwargs.get("tmin"), tmax=kwargs.get("tmax"), want_codes=True,
                                       want_info=True)
    return out.reshape(tensor.shape), codes.reshape(tensor.shape), info
