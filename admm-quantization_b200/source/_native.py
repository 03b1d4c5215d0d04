"""ctypes binding of libadmmq.so (include/admmq.h).  There is no CPU fallback: importing this
module without the built library, or calling it with non-CUDA tensors, raises."""
import ctypes
import os
import threading

import torch

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.environ.get("ADMMQ_LIB") or os.path.join(os.path.dirname(_HERE), "lib", "libadmmq.so")

QSCHEME_IDS = {
    "tensor_mseminmax_symmetric": 0,
    "tensor_minmax": 1,
    "tensor_symmetric": 2,
    "tensor_affine": 3,
    "tensor_mseminmax_e2m1": 4,   # FP4 E2M1 grid, bits = 4 (include/admmq.h)
    "tensor_mseminmax_e4m3": 6,   # FP8 E4M3 grid, bits = 8 (id 5 is unassigned)
    "tensor_mseminmax_e5m2": 7,   # FP8 E5M2 grid, bits = 8
    "tensor_mseminmax_e3m2": 8,   # FP6 E3M2 grid, bits = 6
    "tensor_mseminmax_e2m3": 9,   # FP6 E2M3 grid, bits = 6
}
CLIP_SEARCH_SCHEMES = ("tensor_mseminmax_symmetric", "tensor_mseminmax_e2m1", "tensor_mseminmax_e4m3",
                       "tensor_mseminmax_e5m2", "tensor_mseminmax_e3m2", "tensor_mseminmax_e2m3")   # scale from the clip search

E_BADARG, E_WORKSPACE, E_CUDA, E_NOT_PD, E_UNSUPPORTED = -1, -2, -3, -4, -5
ST_CONVERGED, ST_NONFINITE = 1, 2


class LoopReport(ctypes.Structure):
    _fields_ = [("iterations", ctypes.c_int32), ("status", ctypes.c_int32), ("rho", ctypes.c_float),
                ("scale", ctypes.c_float), ("r", ctypes.c_float), ("s", ctypes.c_float),
                ("best_index", ctypes.c_int32), ("absmax", ctypes.c_float), ("phase_ns", ctypes.c_uint64 * 4)]


class FactorizeParams(ctypes.Structure):
    _fields_ = [("max_iter_als", ctypes.c_int32), ("max_iter_admm", ctypes.c_int32), ("eps", ctypes.c_float),
                ("tol", ctypes.c_double), ("bits", ctypes.c_int32), ("qscheme", ctypes.c_int32),
                ("num_attempts", ctypes.c_int32), ("solve_precision", ctypes.c_int32),
                ("mttkrp_precision", ctypes.c_int32), ("max_ctas", ctypes.c_int32), ("init_is_random", ctypes.c_int32)]


class Problem(ctypes.Structure):
    _fields_ = [("W", ctypes.c_void_p), ("ndim", ctypes.c_int32), ("shape", ctypes.c_int32 * 3), ("rank", ctypes.c_int32),
                ("factors", ctypes.c_void_p * 3), ("duals", ctypes.c_void_p * 3), ("factors_q", ctypes.c_void_p * 3),
                ("params", FactorizeParams), ("loss_hist", ctypes.c_void_p), ("loss_quant_hist", ctypes.c_void_p),
                ("sweeps_done", ctypes.POINTER(ctypes.c_int32)), ("workspace", ctypes.c_void_p),
                ("workspace_bytes", ctypes.c_size_t), ("stream", ctypes.c_void_p)]


def _load():
    if not os.path.exists(LIB_PATH):
        raise ImportError(
            f"{LIB_PATH} is missing: build it with `python admm-quantization_b200/csrc/build.py` "
            "(the solver has no CPU or PyTorch fallback)")
    lib = ctypes.CDLL(LIB_PATH)
    c_int, c_i64, c_sz, c_f, vp = ctypes.c_int, ctypes.c_int64, ctypes.c_size_t, ctypes.c_float, ctypes.c_void_p
    sig = {
        "admmq_version": (c_int, []),
        "admmq_last_error": (ctypes.c_char_p, []),
        "admmq_device_info": (c_int, [ctypes.POINTER(c_int)] * 3),
        "admmq_launch_count": (ctypes.c_uint64, []),
        "admmq_project_workspace_bytes": (c_sz, [c_i64, c_int]),
        "admmq_project": (c_int, [vp, c_i64, c_int, c_int, c_int, vp, vp, vp, vp, vp, vp, c_sz, vp]),
        "admmq_clip_search_sums": (c_int, [vp, c_i64, c_int, c_int, c_int, c_int, vp, vp, c_sz, vp]),
        "admmq_clip_search_sums_scheme": (c_int, [vp, c_i64, c_int, c_int, c_int, c_int, c_int, vp, vp, c_sz, vp]),
        "admmq_e2m1_encode": (c_int, [vp, c_i64, vp, vp]),
        "admmq_fp_encode": (c_int, [vp, c_i64, c_int, vp, vp]),
        "admmq_gram_hadamard": (c_int, [vp, c_int, vp, c_int, c_int, vp, vp]),
        "admmq_unfold3": (c_int, [vp, c_int, c_int, c_int, c_int, vp, vp]),
        "admmq_mttkrp_workspace_bytes": (c_sz, [c_int, c_int, c_int, c_int, c_int]),
        "admmq_mttkrp": (c_int, [vp, c_int, vp, c_int, vp, c_int, c_int, vp, c_int, vp, c_sz, vp]),
        "admmq_permute_myx": (c_int, [vp, c_int, c_int, c_int, vp, vp]),
        "admmq_mttkrp_tc_workspace_bytes": (c_sz, [c_int, c_int, c_int, c_int]),
        "admmq_mttkrp_tc": (c_int, [vp, c_int, vp, c_int, vp, c_int, c_int, vp, vp, c_sz, vp]),
        "admmq_mttkrp_kernel": (c_int, [c_int, c_int, c_int, c_int, c_int, c_int, ctypes.POINTER(c_int),
                                        ctypes.POINTER(c_int)]),
        "admmq_mttkrp_f64_workspace_bytes": (c_sz, [c_int, c_int, c_int, c_int]),
        "admmq_mttkrp_f64": (c_int, [vp, c_int, vp, c_int, vp, c_int, c_int, vp, vp, c_sz, vp]),
        "admmq_gram_hadamard_f64": (c_int, [vp, c_int, vp, c_int, c_int, vp, vp]),
        "admmq_normalize_columns_f64": (c_int, [vp, c_int, c_int, vp, vp, vp]),
        "admmq_recon_error_workspace_bytes": (c_sz, [c_int, c_int, c_int]),
        "admmq_recon_error": (c_int, [vp, c_int, vp, vp, c_int, vp, c_int, c_int, vp, vp, c_sz, vp]),
        "admmq_gemm_nt": (c_int, [vp, c_int, c_int, vp, c_int, c_int, c_int, vp, c_int, vp]),
        "admmq_fp8_operand_format": (c_int, [c_int, c_int]),
        "admmq_codes_to_fp8": (c_int, [vp, c_int, c_int, c_int, c_int, c_int, vp, c_int, vp]),
        "admmq_fp8_quantize_rows": (c_int, [vp, c_int, c_int, c_int, vp, c_int, vp, vp]),
        "admmq_code_gemm_kernel": (c_int, [c_int, c_int, c_int, c_int, ctypes.POINTER(c_int)]),
        "admmq_code_gemm": (c_int, [vp, c_int, vp, c_int, vp, c_int, vp, c_int, c_int, c_int, vp, vp, c_int, vp]),
        "admmq_padded_ld": (c_int, [c_int]),
        "admmq_spd_inverse_workspace_bytes": (c_sz, [c_int]),
        "admmq_spd_inverse": (c_int, [vp, c_int, vp, vp, vp, vp, c_int, vp, c_sz, vp]),
        "admmq_admm_loop_kernel": (c_int, [c_int, c_int, c_int, c_int, c_int]),
        "admmq_admm_loop_workspace_bytes": (c_sz, [c_int, c_int, c_int]),
        "admmq_admm_loop": (c_int, [vp, vp, vp, vp, vp, vp, vp, c_int, c_int, c_int, c_f, c_int, c_int, c_int, c_int, c_int,
                                    vp, vp, vp, c_sz, vp]),
        "admmq_split_loop_workspace_bytes": (c_sz, [c_i64, c_int]),
        "admmq_split_loop": (c_int, [vp, vp, vp, vp, c_i64, c_f, c_int, c_f, c_int, c_int, c_int, c_int, vp, vp, vp, c_sz, vp]),
        "admmq_factorize_workspace_bytes": (c_sz, [c_int, ctypes.POINTER(c_int), c_int, ctypes.POINTER(FactorizeParams)]),
        "admmq_factorize_cp3": (c_int, [vp, c_int, c_int, c_int, c_int] + [vp] * 9 +
                                [ctypes.POINTER(FactorizeParams), vp, vp, ctypes.POINTER(c_int), vp, c_sz, vp]),
        "admmq_factorize_mat": (c_int, [vp, c_int, c_int, c_int] + [vp] * 6 +
                                [ctypes.POINTER(FactorizeParams), vp, vp, ctypes.POINTER(c_int), vp, c_sz, vp]),
        "admmq_factorize_batch": (c_int, [c_int, ctypes.POINTER(Problem)]),
        "admmq_admm_iteration_workspace_bytes": (c_sz, [c_int, c_int, c_int]),
        "admmq_admm_iteration": (c_int, [vp, vp, vp, vp, c_int, c_int, c_int, c_f, c_int, c_int, c_int, c_int, c_int,
                                         vp, vp, vp, c_sz, vp]),
    }
    for name, (res, args) in sig.items():
        fn = getattr(lib, name)
        fn.restype = res
        fn.argtypes = args
    return lib


lib = _load()
EXPORTS = ("admmq_version admmq_last_error admmq_device_info admmq_launch_count admmq_project_workspace_bytes "
           "admmq_project admmq_clip_search_sums admmq_clip_search_sums_scheme admmq_e2m1_encode admmq_fp_encode admmq_admm_loop_kernel admmq_admm_loop_workspace_bytes admmq_admm_loop admmq_gemm_nt "
           "admmq_gram_hadamard admmq_unfold3 admmq_mttkrp_workspace_bytes admmq_mttkrp admmq_permute_myx "
           "admmq_mttkrp_tc_workspace_bytes admmq_mttkrp_tc admmq_mttkrp_kernel admmq_mttkrp_f64_workspace_bytes "
           "admmq_mttkrp_f64 "
           "admmq_gram_hadamard_f64 admmq_normalize_columns_f64 "
           "admmq_recon_error_workspace_bytes admmq_recon_error admmq_padded_ld admmq_spd_inverse_workspace_bytes "
           "admmq_spd_inverse admmq_admm_iteration_workspace_bytes admmq_admm_iteration "
           "admmq_factorize_workspace_bytes admmq_factorize_cp3 admmq_factorize_mat admmq_factorize_batch "
           "admmq_split_loop_workspace_bytes admmq_split_loop "
           "admmq_fp8_operand_format admmq_codes_to_fp8 admmq_fp8_quantize_rows admmq_code_gemm_kernel admmq_code_gemm").split()


def last_error() -> str:
    return lib.admmq_last_error().decode()


def check(rc: int):
    """Translate an ADMMQ_E_* code into the exception type the reference raises (SURVEY 8(b))."""
    if rc == 0:
        return
    msg = last_error()
    if rc == E_BADARG:
        raise ValueError(msg)
    if rc == E_NOT_PD:
        raise torch.linalg.LinAlgError(msg)
    if rc == E_UNSUPPORTED:
        raise NotImplementedError(msg)
    raise RuntimeError(f"libadmmq error {rc}: {msg}")


def qscheme_id(qscheme: str) -> int:
    if qscheme not in QSCHEME_IDS:
        raise NotImplementedError(qscheme)  # source/quantization.py:115
    return QSCHEME_IDS[qscheme]


def require_cuda(*tensors):
    """Every tensor of a call must live on ONE CUDA device (the library launches on a single device and stream)."""
    dev = None
    for t in tensors:
        if t is None:
            continue
        if not t.is_cuda:
            raise RuntimeError("libadmmq kernels need CUDA tensors (there is no CPU fallback); got device "
                               f"{t.device}")
        if dev is None:
            dev = t.device
        elif t.device != dev:
            raise RuntimeError(f"libadmmq: all tensors of a call must share one device, got {dev} and {t.device}")


def call(device, fn, *args):
    """Run a library entry point with `device` made current: the C side resolves the device (SM count, cooperative
    launch, kernel launches, memsets) with cudaGetDevice(), and the stream passed in belongs to `device`."""
    device = torch.device(device)
    if torch.cuda.current_device() == device.index:
        return check(fn(*args))
    with torch.cuda.device(device):
        return check(fn(*args))


def ptr(t):
    return None if t is None else ctypes.c_void_p(t.data_ptr())


def stream_ptr(device):
    return ctypes.c_void_p(torch.cuda.current_stream(device).cuda_stream)


_tls = threading.local()


def workspace(nbytes: int, device, tag: str = "main") -> torch.Tensor:
    """Caller-owned scratch (the library never allocates).  One growing buffer per (thread, device, STREAM, tag): the
    scratch holds barrier counters and accumulators of persistent kernels, so two calls that may run concurrently
    (different streams) must never share it.  A buffer that has to grow is replaced; the old one is handed back to
    the caching allocator with `record_stream`, so kernels still using it on that stream finish first."""
    cache = getattr(_tls, "ws", None)
    if cache is None:
        cache = _tls.ws = {}
    device = torch.device(device)
    stream = torch.cuda.current_stream(device)
    key = (device.index, stream.cuda_stream, tag)
    buf = cache.get(key)
    if buf is None or buf.numel() < nbytes:
        if buf is not None:
            buf.record_stream(stream)
        with torch.cuda.device(device):
            buf = torch.empty(max(int(nbytes), 256), dtype=torch.uint8, device=device)
        cache[key] = buf
    return buf


def f32c(t: torch.Tensor) -> torch.Tensor:
    return t.detach().to(torch.float32).contiguous()


# ------------------------------------------------------------------------------- thin wrappers
# Every wrapper takes optional `out=` / `ws=` tensors so that a solver can preallocate once and enqueue
# sweeps without touching the allocator; without them a result tensor / the thread-local scratch is used.
def _ws(nbytes, device, ws):
    if ws is None:
        return workspace(nbytes, device)
    assert ws.is_cuda and ws.numel() * ws.element_size() >= nbytes, "workspace too small"
    return ws


def project_workspace_bytes(n, num_attempts=200):
    return int(lib.admmq_project_workspace_bytes(int(n), int(num_attempts)))


def project(x, bits, qscheme, num_attempts=200, tmin=None, tmax=None, want_codes=False, want_info=False,
            out=None, codes=None, info=None, ws=None):
    require_cuda(x)
    xc = f32c(x)
    n = xc.numel()
    out = torch.empty_like(xc) if out is None else out
    if want_codes and codes is None:
        codes = torch.empty(xc.shape, dtype=torch.int8, device=xc.device)
    if want_info and info is None:
        info = torch.empty(4, dtype=torch.float32, device=xc.device)
    ws = _ws(project_workspace_bytes(n, num_attempts), xc.device, ws)
    tmin_t = None if tmin is None else torch.as_tensor(tmin, dtype=torch.float32, device=xc.device).reshape(1)
    tmax_t = None if tmax is None else torch.as_tensor(tmax, dtype=torch.float32, device=xc.device).reshape(1)
    call(xc.device, lib.admmq_project, ptr(xc), n, int(bits), qscheme_id(qscheme), int(num_attempts), ptr(tmin_t), ptr(tmax_t),
                            ptr(out), ptr(codes), ptr(info), ptr(ws), ws.numel(), stream_ptr(xc.device))
    return out, codes, info


def clip_search_sums(x, bits, num_attempts=200, method=1, max_ctas=0, qscheme="tensor_mseminmax_symmetric"):
    """Per-candidate sum((x - Q_c(x))**2) as float64: method 0 = direct evaluation, 1 = threshold form (parity tests),
    for any clip-search scheme."""
    require_cuda(x)
    xc = f32c(x)
    n = xc.numel()
    sums = torch.empty(int(num_attempts), dtype=torch.float64, device=xc.device)
    ws = _ws(project_workspace_bytes(n, num_attempts), xc.device, None)
    call(xc.device, lib.admmq_clip_search_sums_scheme, ptr(xc), n, int(bits), qscheme_id(qscheme), int(num_attempts),
         int(method), int(max_ctas), ptr(sums), ptr(ws), ws.numel(), stream_ptr(xc.device))
    return sums


def e2m1_encode(t):
    """E2M1 codes (int8, 0 .. 15) of float32 t by the hardware conversion cvt.rn.satfinite.e2m1x2.f32."""
    require_cuda(t)
    tc = f32c(t)
    codes = torch.empty(tc.shape, dtype=torch.int8, device=tc.device)
    call(tc.device, lib.admmq_e2m1_encode, ptr(tc), tc.numel(), ptr(codes), stream_ptr(tc.device))
    return codes


def fp_encode(t, qscheme):
    """FP8 / FP6 codes (int8) of float32 t by the hardware conversion cvt.rn.satfinite.<fmt>x2.f32 for one of the
    schemes tensor_mseminmax_e4m3 / _e5m2 / _e3m2 / _e2m3: the FP8 byte, or the FP6 encoding 0 .. 63."""
    require_cuda(t)
    tc = f32c(t)
    codes = torch.empty(tc.shape, dtype=torch.int8, device=tc.device)
    call(tc.device, lib.admmq_fp_encode, ptr(tc), tc.numel(), qscheme_id(qscheme), ptr(codes), stream_ptr(tc.device))
    return codes


def gram_hadamard(U1, U2=None, out=None):
    require_cuda(U1, U2)
    U1 = f32c(U1)
    U2 = None if U2 is None else f32c(U2)
    R = U1.shape[1]
    G = torch.empty(R, R, dtype=torch.float32, device=U1.device) if out is None else out
    call(U1.device, lib.admmq_gram_hadamard, ptr(U1), U1.shape[0], ptr(U2), 0 if U2 is None else U2.shape[0], R, ptr(G),
                                  stream_ptr(U1.device))
    return G


def unfold3(W, mode, out=None):
    require_cuda(W)
    W = f32c(W)
    I, J, K = W.shape
    shape = [(I, J * K), (J, I * K), (K, I * J)][mode]
    out = torch.empty(shape, dtype=torch.float32, device=W.device) if out is None else out
    call(W.device, lib.admmq_unfold3, ptr(W), I, J, K, int(mode), ptr(out), stream_ptr(W.device))
    return out


def mttkrp_workspace_bytes(M, nx, ny, R, precision=0):
    return int(lib.admmq_mttkrp_workspace_bytes(int(M), int(nx), int(ny), int(R), int(precision)))


def mttkrp(Wn, X, Y=None, precision=0, out=None, ws=None):
    """F = Wn @ khatri_rao(X, Y); Wn is the (M, nx*ny) unfolding."""
    require_cuda(Wn, X, Y)
    Wn, X = f32c(Wn), f32c(X)
    Y = None if Y is None else f32c(Y)
    M, R = Wn.shape[0], X.shape[1]
    nx, ny = X.shape[0], (1 if Y is None else Y.shape[0])
    assert Wn.shape[1] == nx * ny, (Wn.shape, nx, ny)
    F = torch.empty(M, R, dtype=torch.float32, device=Wn.device) if out is None else out
    ws = _ws(mttkrp_workspace_bytes(M, nx, ny, R, precision), Wn.device, ws)
    call(Wn.device, lib.admmq_mttkrp, ptr(Wn), M, ptr(X), nx, ptr(Y), ny, R, ptr(F), int(precision), ptr(ws), ws.numel(),
                           stream_ptr(Wn.device))
    return F


def permute_myx(Wn, nx, ny):
    """V[(m, y), x] = Wn[m, x*ny + y] as an (M*ny, ldv) tensor, ldv = nx rounded up to 4 (operand of mttkrp_tc)."""
    require_cuda(Wn)
    Wn = f32c(Wn)
    M = Wn.shape[0]
    assert Wn.shape[1] == nx * ny
    ldv = (nx + 3) // 4 * 4
    V = torch.empty(M * ny, ldv, dtype=torch.float32, device=Wn.device)
    call(Wn.device, lib.admmq_permute_myx, ptr(Wn), M, int(nx), int(ny), ptr(V), stream_ptr(Wn.device))
    return V


def mttkrp_tc_workspace_bytes(M, nx, ny, R):
    return int(lib.admmq_mttkrp_tc_workspace_bytes(int(M), int(nx), int(ny), int(R)))


def mttkrp_tc(V, M, X, Y=None, out=None, ws=None):
    """F = MTTKRP in 3xTF32 on the tensor cores; V from `permute_myx` (or the (M, nx) matrix itself when Y is None)."""
    require_cuda(V, X, Y)
    X = f32c(X)
    Y = None if Y is None else f32c(Y)
    nx, R = X.shape
    ny = 1 if Y is None else Y.shape[0]
    assert V.dtype == torch.float32 and V.is_contiguous() and V.shape == (M * ny, (nx + 3) // 4 * 4)
    F = torch.empty(M, R, dtype=torch.float32, device=V.device) if out is None else out
    ws = _ws(mttkrp_tc_workspace_bytes(M, nx, ny, R), V.device, ws)
    call(V.device, lib.admmq_mttkrp_tc, ptr(V), int(M), ptr(X), nx, ptr(Y), ny, R, ptr(F), ptr(ws), ws.numel(), stream_ptr(V.device))
    return F


def mttkrp_kernel(M, nx, ny, R, precision, sm_count):
    """(id, grid, splits) of the MTTKRP kernel (include/admmq.h ADMMQ_MTTKRP_*) a call runs on `sm_count` SMs;
    precision 1 = mttkrp_tc, ny = 1 for a matrix."""
    grid, splits = ctypes.c_int(0), ctypes.c_int(0)
    rc = int(lib.admmq_mttkrp_kernel(int(M), int(nx), int(ny), int(R), int(precision), int(sm_count),
                                     ctypes.byref(grid), ctypes.byref(splits)))
    check(min(rc, 0))
    return rc, grid.value, splits.value


# ---- float64 pieces of the ALS + EPC initialisation (source/parafac_epc.py)
def _f64c(t):
    assert t.dtype == torch.float64 and t.is_contiguous(), "float64 contiguous tensor expected"
    return t


def mttkrp_f64(Wn, X, Y=None, out=None, ws=None):
    """F = Wn @ khatri_rao(X, Y) in float64 without materialising the Khatri-Rao operand; Wn is the (M, nx*ny) unfolding."""
    require_cuda(Wn, X, Y, out, ws)
    Wn, X = _f64c(Wn), _f64c(X)
    Y = None if Y is None else _f64c(Y)
    M, R = Wn.shape[0], X.shape[1]
    nx, ny = X.shape[0], (1 if Y is None else Y.shape[0])
    assert Wn.shape[1] == nx * ny, (Wn.shape, nx, ny)
    F = torch.empty(M, R, dtype=torch.float64, device=Wn.device) if out is None else _f64c(out)
    ws = _ws(int(lib.admmq_mttkrp_f64_workspace_bytes(M, nx, ny, R)), Wn.device, ws)
    call(Wn.device, lib.admmq_mttkrp_f64, ptr(Wn), M, ptr(X), nx, ptr(Y), ny, R, ptr(F), ptr(ws), ws.numel(),
         stream_ptr(Wn.device))
    return F


def gram_hadamard_f64(U1, U2=None, out=None):
    """G = (U1^T U1) * (U2^T U2) in float64."""
    require_cuda(U1, U2, out)
    U1 = _f64c(U1)
    U2 = None if U2 is None else _f64c(U2)
    R = U1.shape[1]
    G = torch.empty(R, R, dtype=torch.float64, device=U1.device) if out is None else _f64c(out)
    call(U1.device, lib.admmq_gram_hadamard_f64, ptr(U1), U1.shape[0], ptr(U2), 0 if U2 is None else U2.shape[0], R, ptr(G),
         stream_ptr(U1.device))
    return G


def normalize_columns_f64(U, carry=None, norms=None):
    """In place: U[:, c] /= ||U[:, c]|| (zero columns untouched), carry[c] *= ||U[:, c]||.  Returns the norms."""
    require_cuda(U, carry, norms)
    U = _f64c(U)
    n, R = U.shape
    norms = torch.empty(R, dtype=torch.float64, device=U.device) if norms is None else _f64c(norms)
    if carry is not None:
        _f64c(carry)
    call(U.device, lib.admmq_normalize_columns_f64, ptr(U), n, R, ptr(norms), ptr(carry), stream_ptr(U.device))
    return norms


def recon_error_workspace_bytes(M, nx, ny):
    return int(lib.admmq_recon_error_workspace_bytes(int(M), int(nx), int(ny)))


def recon_error_sums(W0, A, X, Y=None, out=None, ws=None):
    """Device double[2] = {sum (W - [[A, X, Y]])^2, sum W^2}; W0 is the (M, nx*ny) mode-0 unfolding."""
    require_cuda(W0, A, X, Y)
    W0, A, X = f32c(W0), f32c(A), f32c(X)
    Y = None if Y is None else f32c(Y)
    M, R = A.shape
    nx, ny = X.shape[0], (1 if Y is None else Y.shape[0])
    assert W0.shape == (M, nx * ny)
    out = torch.empty(2, dtype=torch.float64, device=W0.device) if out is None else out
    ws = _ws(recon_error_workspace_bytes(M, nx, ny), W0.device, ws)
    call(W0.device, lib.admmq_recon_error, ptr(W0), M, ptr(A), ptr(X), nx, ptr(Y), ny, R, ptr(out), ptr(ws), ws.numel(),
                                stream_ptr(W0.device))
    return out


def gemm_nt(A, B, out=None):
    """C = A @ B.T in 3xTF32 on the tensor cores; A (M, K), B (N, K) float32 with K % 4 == 0 (or zero padded)."""
    require_cuda(A, B)
    assert A.dtype == torch.float32 and B.dtype == torch.float32 and A.stride(1) == 1 and B.stride(1) == 1
    M, K = A.shape
    N = B.shape[0]
    assert B.shape[1] == K
    C = torch.empty(M, N, dtype=torch.float32, device=A.device) if out is None else out
    call(A.device, lib.admmq_gemm_nt, ptr(A), A.stride(0), M, ptr(B), B.stride(0), N, K, ptr(C), C.stride(0), stream_ptr(A.device))
    return C


# ---- CP layers on the FP8 tensor cores (include/admmq.h, DESIGN.md 2d)
FP8_DTYPES = {"tensor_mseminmax_e4m3": torch.float8_e4m3fn, "tensor_mseminmax_e5m2": torch.float8_e5m2}


def ld16(n):
    """Row stride (elements) of an FP8 operand with n columns: n rounded up to 16 bytes."""
    return (int(n) + 15) // 16 * 16


def fp8_operand_format(bits, qscheme):
    """The FP8 format the codes of (bits, qscheme) run as: "tensor_mseminmax_e4m3" or "tensor_mseminmax_e5m2" (the scheme
    whose torch dtype FP8_DTYPES gives).  ValueError, with the reason, for a grid without an exact FP8 form."""
    rc = int(lib.admmq_fp8_operand_format(int(bits), qscheme_id(qscheme)))
    check(min(rc, 0))
    return "tensor_mseminmax_e5m2" if rc == QSCHEME_IDS["tensor_mseminmax_e5m2"] else "tensor_mseminmax_e4m3"


def codes_to_fp8(codes, bits, qscheme, transpose=False):
    """FP8 operand bytes (uint8) of a 2-D int8 code tensor: (rows, ld16(cols)), or with transpose=True
    (cols, ld16(rows)) holding codes.T; pad columns zero.  View the result as FP8_DTYPES[fp8_operand_format(...)]."""
    fp8_operand_format(bits, qscheme)
    require_cuda(codes)
    assert codes.dtype == torch.int8 and codes.dim() == 2
    c = codes.contiguous()
    rows, cols = c.shape
    out_rows, out_cols = (cols, rows) if transpose else (rows, cols)
    out = torch.empty(out_rows, ld16(out_cols), dtype=torch.uint8, device=c.device)
    call(c.device, lib.admmq_codes_to_fp8, ptr(c), rows, cols, int(bits), qscheme_id(qscheme), 1 if transpose else 0,
         ptr(out), out.shape[1], stream_ptr(c.device))
    return out


def fp8_quantize_rows(x, out=None, scale=None):
    """Per-row dynamic E4M3 codes of a 2-D float32 tensor x (M, K) with unit column stride: (q uint8 (M, ld16(K)) with
    zero pad columns, s float32 (M,)), s_m = fl(amax_m / 448), q = E4M3(fl(x / s_m))."""
    require_cuda(x, out, scale)
    assert x.dtype == torch.float32 and x.dim() == 2 and x.stride(1) == 1
    M, K = x.shape
    q = torch.empty(M, ld16(K), dtype=torch.uint8, device=x.device) if out is None else out
    s = torch.empty(M, dtype=torch.float32, device=x.device) if scale is None else scale
    call(x.device, lib.admmq_fp8_quantize_rows, ptr(x), x.stride(0), M, K, ptr(q), q.stride(0), ptr(s), stream_ptr(x.device))
    return q, s


def code_gemm(a8, a_scale, b8, b_scale, K, b_format="tensor_mseminmax_e4m3", bias=None, out=None):
    """D (M, N) float32 = fl(acc * fl(a_scale[m] * b_scale[0])) (+ bias[n]) with acc = a8[:, :K] . b8[:, :K]^T summed on
    the FP8 tensor cores: a8 (M, lda) E4M3 bytes, b8 (N, ldb) bytes of b_format, both uint8 with unit column stride;
    a_scale (M,), b_scale (>= 1,) and bias (N,) float32 on the device."""
    require_cuda(a8, a_scale, b8, b_scale, bias, out)
    assert a8.dtype == torch.uint8 and b8.dtype == torch.uint8 and a8.stride(1) == 1 and b8.stride(1) == 1
    for t in (a_scale, b_scale, bias):
        assert t is None or (t.dtype == torch.float32 and t.is_contiguous())
    M, N = a8.shape[0], b8.shape[0]
    assert a_scale.numel() >= M and (bias is None or bias.numel() >= N)
    D = torch.empty(M, N, dtype=torch.float32, device=a8.device) if out is None else out
    assert D.dtype == torch.float32 and D.stride(1) == 1 and D.shape[0] >= M and D.shape[1] >= N
    call(a8.device, lib.admmq_code_gemm, ptr(a8), a8.stride(0), ptr(a_scale), M, ptr(b8), b8.stride(0), ptr(b_scale),
         qscheme_id(b_format), N, int(K), ptr(bias), ptr(D), D.stride(0), stream_ptr(a8.device))
    return D


def code_gemm_kernel(M, N, K, sm_count):
    """(tile width, grid) a code_gemm of this shape runs on `sm_count` SMs."""
    grid = ctypes.c_int(0)
    rc = int(lib.admmq_code_gemm_kernel(int(M), int(N), int(K), int(sm_count), ctypes.byref(grid)))
    check(min(rc, 0))
    return rc, grid.value


def spd_inverse_workspace_bytes(R):
    return int(lib.admmq_spd_inverse_workspace_bytes(int(R)))


def spd_inverse(G, out=None, ws=None, max_ctas=0, minv64=None):
    """(Minv [R, ld], rho [1], status [1]) of G + trace(G)/R * I.  `out` = preallocated (Minv, rho, status);
    `minv64` = preallocated float64 [R, ld] that also receives the inverse before its rounding to float32 (the
    operand of the loop's parity mode), or True to allocate it (it is then returned as a fourth element)."""
    require_cuda(G)
    G = f32c(G)
    R = G.shape[0]
    ld = lib.admmq_padded_ld(R)
    if out is None:
        Minv = torch.empty(R, ld, dtype=torch.float32, device=G.device)
        rho = torch.empty(1, dtype=torch.float32, device=G.device)
        status = torch.empty(1, dtype=torch.int32, device=G.device)
    else:
        Minv, rho, status = out
    made = minv64 is True
    if made:
        minv64 = torch.empty(R, ld, dtype=torch.float64, device=G.device)
    if minv64 is not None:
        assert minv64.dtype == torch.float64 and minv64.is_contiguous() and minv64.shape == (R, ld)
    require_cuda(G, Minv, rho, status, minv64)
    ws = _ws(spd_inverse_workspace_bytes(R), G.device, ws)
    call(G.device, lib.admmq_spd_inverse, ptr(G), R, ptr(Minv), ptr(minv64), ptr(rho), ptr(status), int(max_ctas), ptr(ws),
         ws.numel(), stream_ptr(G.device))
    return (Minv, rho, status, minv64) if made else (Minv, rho, status)


def admm_iteration_inplace(H, U, F, G, max_iter, eps, bits, qscheme, num_attempts=200, codes=None, precision=0,
                           max_ctas=0):
    """Runs the persistent loop on contiguous float32 CUDA tensors, updating H and U in place.
    Returns the device report (uint8[32]); decode with `read_report` (synchronises)."""
    require_cuda(H, U, F, G)
    for t in (H, U, F, G):
        assert t.dtype == torch.float32 and t.is_contiguous()
    I, R = H.shape
    assert U.shape == H.shape and F.shape == H.shape and G.shape == (R, R)
    report = torch.empty(ctypes.sizeof(LoopReport), dtype=torch.uint8, device=H.device)
    nbytes = lib.admmq_admm_iteration_workspace_bytes(I, R, int(num_attempts))
    ws = workspace(nbytes, H.device)
    call(H.device, lib.admmq_admm_iteration, ptr(H), ptr(U), ptr(F), ptr(G), I, R, int(max_iter), float(eps), int(bits),
                                   qscheme_id(qscheme), int(num_attempts), int(precision), int(max_ctas), ptr(codes),
                                   ptr(report), ptr(ws), ws.numel(), stream_ptr(H.device))
    return report


def loop_kernel(I, R, num_attempts, precision, grid):
    """Id of the loop kernel (include/admmq.h ADMMQ_LOOP_*) a call on a cooperative grid of `grid` CTAs runs."""
    rc = int(lib.admmq_admm_loop_kernel(int(I), int(R), int(num_attempts), int(precision), int(grid)))
    check(min(rc, 0))
    return rc


def admm_loop_workspace_bytes(I, R, num_attempts=200):
    return int(lib.admmq_admm_loop_workspace_bytes(int(I), int(R), int(num_attempts)))


def new_report(device):
    return torch.empty(ctypes.sizeof(LoopReport), dtype=torch.uint8, device=device)


def admm_loop_inplace(H, U, F, Minv, rho, inv_status, max_iter, eps, bits, qscheme, num_attempts=200, codes=None,
                      report=None, ws=None, precision=0, max_ctas=0, minv64=None):
    """The persistent loop alone, given (Minv, rho, status[, Minv64]) from `spd_inverse`; H and U are updated in place.
    precision 0 (parity mode) needs `minv64`."""
    require_cuda(H, U, F, Minv, rho, inv_status, minv64, codes, report, ws)
    for t in (H, U, F, Minv):
        assert t.dtype == torch.float32 and t.is_contiguous()
    I, R = H.shape
    assert U.shape == H.shape and F.shape == H.shape and Minv.shape == (R, lib.admmq_padded_ld(R))
    if int(precision) == 0 and minv64 is None:
        raise ValueError("admm_loop_inplace: precision 0 (parity mode) needs minv64 from spd_inverse(..., minv64=...)")
    if minv64 is not None:
        assert minv64.dtype == torch.float64 and minv64.is_contiguous() and minv64.shape == Minv.shape
    report = new_report(H.device) if report is None else report
    ws = _ws(admm_loop_workspace_bytes(I, R, num_attempts), H.device, ws)
    call(H.device, lib.admmq_admm_loop, ptr(H), ptr(U), ptr(F), ptr(Minv), ptr(minv64), ptr(rho), ptr(inv_status), I, R,
         int(max_iter), float(eps), int(bits), qscheme_id(qscheme), int(num_attempts), int(precision), int(max_ctas),
         ptr(codes), ptr(report), ptr(ws), ws.numel(), stream_ptr(H.device))
    return report


def split_loop_inplace(H, U, W, H2, rho, max_iter, eps, bits, qscheme, num_attempts=200, max_ctas=0, codes=None,
                       report=None, ws=None):
    """Quantized block of the two-block splitting W ~ W_q + W_r (scripts/factorize_lowrank.py:84-99); H and U
    (contiguous float32 CUDA tensors) are updated in place."""
    require_cuda(H, U, W, H2)
    for t in (H, U, W, H2):
        assert t.dtype == torch.float32 and t.is_contiguous() and t.numel() == H.numel()
    n = H.numel()
    report = new_report(H.device) if report is None else report
    ws = _ws(int(lib.admmq_split_loop_workspace_bytes(n, int(num_attempts))), H.device, ws)
    call(H.device, lib.admmq_split_loop, ptr(H), ptr(U), ptr(W), ptr(H2), n, float(rho), int(max_iter), float(eps), int(bits),
                               qscheme_id(qscheme), int(num_attempts), int(max_ctas), ptr(codes), ptr(report), ptr(ws),
                               ws.numel(), stream_ptr(H.device))
    return report


def factorize(W, factors, duals, bits, qscheme, max_iter_als, max_iter_admm=1000, eps=1e-8, tol=1e-5, num_attempts=200,
              solve_precision=0, mttkrp_precision=0, max_ctas=0, init_is_random=True, ws=None):
    """The whole outer loop in one C call (admmq_factorize_cp3 / admmq_factorize_mat; scripts/factorize.py:207-310).
    `factors` and `duals` (lists of contiguous float32 CUDA tensors) are updated in place.  Returns
    (loss_hist, loss_quant_hist, sweeps_done, factors_q)."""
    import numpy as np
    require_cuda(W, *factors, *duals)
    Wc = f32c(W)
    N = Wc.ndim
    assert N in (2, 3), "Incorrect number of dimentions in weight tensor"
    for t in list(factors) + list(duals):
        assert t.dtype == torch.float32 and t.is_contiguous()
    R = factors[0].shape[1]
    prm = FactorizeParams(int(max_iter_als), int(max_iter_admm), float(eps), float(tol), int(bits), qscheme_id(qscheme),
                          int(num_attempts), int(solve_precision), int(mttkrp_precision), int(max_ctas),
                          1 if init_is_random else 0)
    shape = (ctypes.c_int * N)(*[int(d) for d in Wc.shape])
    need = int(lib.admmq_factorize_workspace_bytes(N, shape, R, ctypes.byref(prm)))
    ws = _ws(need, Wc.device, ws)
    fq = [torch.empty_like(f) for f in factors]
    hist = np.zeros(int(max_iter_als) + 1, np.float32)
    histq = np.zeros(int(max_iter_als) + 1, np.float32)
    done = ctypes.c_int(0)
    hp, hqp = hist.ctypes.data_as(ctypes.c_void_p), histq.ctypes.data_as(ctypes.c_void_p)
    if N == 3:
        call(Wc.device, lib.admmq_factorize_cp3, ptr(Wc), *[int(d) for d in Wc.shape], R, *[ptr(t) for t in factors],
             *[ptr(t) for t in duals], *[ptr(t) for t in fq], ctypes.byref(prm), hp, hqp,
             ctypes.byref(done), ptr(ws), ws.numel(), stream_ptr(Wc.device))
    else:
        call(Wc.device, lib.admmq_factorize_mat, ptr(Wc), *[int(d) for d in Wc.shape], R, *[ptr(t) for t in factors],
             *[ptr(t) for t in duals], *[ptr(t) for t in fq], ctypes.byref(prm), hp, hqp,
             ctypes.byref(done), ptr(ws), ws.numel(), stream_ptr(Wc.device))
    n = done.value + (0 if init_is_random else 1)
    return [float(v) for v in hist[:n]], [float(v) for v in histq[:n]], done.value, fq


def factorize_batch(jobs):
    """Several independent solves side by side (admmq_factorize_batch).  jobs: list of dicts with W, factors, duals
    (updated in place), bits, qscheme, max_iter_als and optionally max_iter_admm, eps, tol, num_attempts,
    solve_precision, mttkrp_precision, max_ctas, init_is_random, stream (torch.cuda.Stream).  Returns one
    (loss_hist, loss_quant_hist, sweeps_done, factors_q) per job."""
    import numpy as np
    n = len(jobs)
    arr = (Problem * n)()
    keep = []
    for k, j in enumerate(jobs):
        Wc = f32c(j["W"])
        require_cuda(Wc, *j["factors"], *j["duals"])
        if keep and keep[0][0].device != Wc.device:
            raise RuntimeError("factorize_batch: all problems of one batch must live on one device")
        N = Wc.ndim
        R = j["factors"][0].shape[1]
        prm = FactorizeParams(int(j["max_iter_als"]), int(j.get("max_iter_admm", 1000)), float(j.get("eps", 1e-8)),
                              float(j.get("tol", 1e-5)), int(j["bits"]), qscheme_id(j["qscheme"]),
                              int(j.get("num_attempts", 200)), int(j.get("solve_precision", 0)),
                              int(j.get("mttkrp_precision", 0)), int(j.get("max_ctas", 0)),
                              1 if j.get("init_is_random", True) else 0)
        shape = (ctypes.c_int * N)(*[int(d) for d in Wc.shape])
        need = int(lib.admmq_factorize_workspace_bytes(N, shape, R, ctypes.byref(prm)))
        ws = j.get("ws")
        if ws is None:
            ws = torch.empty(need, dtype=torch.uint8, device=Wc.device)
        assert ws.numel() >= need
        fq = [torch.empty_like(f) for f in j["factors"]]
        hist = np.zeros(prm.max_iter_als + 1, np.float32)
        histq = np.zeros(prm.max_iter_als + 1, np.float32)
        done = ctypes.c_int32(0)
        stream = j.get("stream") or torch.cuda.Stream(device=Wc.device)
        stream.wait_stream(torch.cuda.current_stream(Wc.device))
        q = arr[k]
        q.W, q.ndim, q.rank = Wc.data_ptr(), N, R
        for m in range(N):
            q.shape[m] = int(Wc.shape[m])
            q.factors[m], q.duals[m], q.factors_q[m] = j["factors"][m].data_ptr(), j["duals"][m].data_ptr(), fq[m].data_ptr()
        q.params = prm
        q.loss_hist, q.loss_quant_hist = hist.ctypes.data, histq.ctypes.data
        q.sweeps_done = ctypes.pointer(done)
        q.workspace, q.workspace_bytes, q.stream = ws.data_ptr(), ws.numel(), stream.cuda_stream
        keep.append((Wc, ws, fq, hist, histq, done, stream, prm))
    call(keep[0][0].device, lib.admmq_factorize_batch, n, arr)   # all problems of a batch live on one device
    out = []
    for Wc, ws, fq, hist, histq, done, stream, prm in keep:
        torch.cuda.current_stream(Wc.device).wait_stream(stream)
        cnt = done.value + (0 if prm.init_is_random else 1)
        out.append(([float(v) for v in hist[:cnt]], [float(v) for v in histq[:cnt]], done.value, fq))
    return out


def launch_count() -> int:
    return int(lib.admmq_launch_count())


def decode_report(raw: bytes) -> LoopReport:
    rep = LoopReport.from_buffer_copy(raw)
    if rep.status == E_NOT_PD:
        raise torch.linalg.LinAlgError("admm_iteration: G + rho*I is not positive-definite (Cholesky failed)")
    return rep


def read_report(report: torch.Tensor) -> LoopReport:
    return decode_report(bytes(report.cpu().numpy().tobytes()))
