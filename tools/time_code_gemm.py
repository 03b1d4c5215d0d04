"""Time the FP8 code GEMM (admmq_code_gemm, tcgen05 kind::f8f6f4) at the shapes the CP layers run, against the 3xTF32
admmq_gemm_nt on the decoded values and torch._scaled_mm, and the FP8-executed CP conv layer against the float32 CP layer.

    python tools/time_code_gemm.py [--out results/code_gemm.json]

Shapes: the two GEMMs of every ResNet-18 CP conv at ImageNet activations (batch 64, layer1 at 56 x 56 ...), both Llama-7B
matrices of the llama7b workload at M = 4096 tokens, and M = N = K = 8192.  Each timing is CUDA events around many calls
after warm-up, with the same operands every call: a shape whose operands and output fit in the 126 MB L2 runs from L2
after the first call ("l2_resident" in the output).  The card's name, power limit and maximum SM clock are read in the
same run.  TFLOP/s are 2 M N K / time against the 4,500 TFLOP/s data-sheet dense FP8 rate (1,125 TF32).
"""
import argparse
import json
import os
import subprocess
import sys

import torch

REPO = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, os.path.join(REPO, "admm-quantization_b200"))

from source import _native as nat  # noqa: E402
from source import workloads as wl  # noqa: E402
from source.models import build_cp_layer, build_cp_layer_fp8  # noqa: E402
from source.quantization import quantize_tensor_codes  # noqa: E402
from source.shapes import rank_from_reduction_rate  # noqa: E402

FP8_PEAK, TF32_PEAK, L2_BYTES = 4500.0, 1125.0, 126e6


def card():
    try:
        return subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                              capture_output=True, text=True, timeout=30).stdout.strip().splitlines()[0]
    except (OSError, IndexError, subprocess.SubprocessError) as e:
        return f"unknown ({e})"


def timed(fn, budget_s=0.5):
    """Mean time per call in ms: 3 warm-up calls, then enough calls for about budget_s, between two CUDA events."""
    for _ in range(3):
        fn()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    fn()
    e1.record()
    e1.synchronize()
    n = int(min(500, max(10, budget_s * 1e3 / max(e0.elapsed_time(e1), 1e-3))))
    e0.record()
    for _ in range(n):
        fn()
    e1.record()
    e1.synchronize()
    return e0.elapsed_time(e1) / n


def gemm_shapes():
    out, seen = [], set()
    for name, cout, cin, kh, kw in wl.resnet18_conv_layers():
        R = rank_from_reduction_rate(torch.empty(cout, cin, kh * kw), 2.0)
        hw = {64: 56, 128: 28, 256: 14, 512: 7}[cout]
        hin = hw * (2 if cin != cout else 1)    # the first conv of stages 2-4 has stride 2
        for label, shape in ((f"{name} gemm1", (64 * hin * hin, R, cin)), (f"{name} gemm2", (64 * hw * hw, cout, R))):
            if shape not in seen:
                seen.add(shape)
                out.append((label,) + shape)
    for name, cout, cin, _, _ in wl.llama7b_linear_layers():
        R = rank_from_reduction_rate(torch.empty(cout, cin), 2.0)
        out += [(f"llama7b {name} fc1", 4096, R, cin), (f"llama7b {name} fc2", 4096, cout, R)]
    out.append(("square 8192", 8192, 8192, 8192))
    return out


def fp8_bytes(shape, g):
    v = torch.randn(shape, generator=g, device="cuda")
    return v.to(torch.float8_e4m3fn).view(torch.uint8)


def time_gemm(label, M, N, K, g):
    ld = nat.ld16(K)
    a = torch.zeros(M, ld, dtype=torch.uint8, device="cuda")
    b = torch.zeros(N, ld, dtype=torch.uint8, device="cuda")
    a[:, :K] = fp8_bytes((M, K), g)
    b[:, :K] = fp8_bytes((N, K), g)
    sa = torch.rand(M, generator=g, device="cuda") + 0.5
    sw = torch.rand(1, generator=g, device="cuda") + 0.5
    D = torch.empty(M, N, device="cuda")
    flop = 2.0 * M * N * K
    t8 = timed(lambda: nat.code_gemm(a, sa, b, sw, K, out=D))
    bn, grid = nat.code_gemm_kernel(M, N, K, torch.cuda.get_device_properties(0).multi_processor_count)
    row = {"shape": label, "M": M, "N": N, "K": K, "tile_width": bn, "grid": grid, "code_gemm_ms": t8,
           "code_gemm_tflops": flop / t8 / 1e9, "l2_resident": (M * ld + N * ld + 4 * M * N) < L2_BYTES}
    row["code_gemm_share_of_fp8_peak"] = row["code_gemm_tflops"] / FP8_PEAK
    # 3xTF32 on the decoded values (float32 operands, K padded to 4)
    ld4 = (K + 3) // 4 * 4
    af = torch.zeros(M, ld4, device="cuda")
    bf = torch.zeros(N, ld4, device="cuda")
    af[:, :K] = a[:, :K].view(torch.float8_e4m3fn).float() * sa[:, None]
    bf[:, :K] = b[:, :K].view(torch.float8_e4m3fn).float() * sw
    C = torch.empty(M, N, device="cuda")
    t32 = timed(lambda: nat.gemm_nt(af, bf, out=C))
    row["gemm_nt_3xtf32_ms"], row["gemm_nt_3xtf32_tflops"] = t32, flop / t32 / 1e9
    row["rel_diff_vs_3xtf32"] = ((D - C).norm() / C.norm()).item()
    del af, bf, C
    # torch._scaled_mm with row-wise scales, where it runs (K and N multiples of 16)
    try:
        a8 = a[:, :K].contiguous().view(torch.float8_e4m3fn)
        b8 = b[:, :K].contiguous().view(torch.float8_e4m3fn)
        sb = sw.expand(N).reshape(1, N).contiguous()
        out = torch._scaled_mm(a8, b8.t(), scale_a=sa.reshape(M, 1), scale_b=sb, out_dtype=torch.bfloat16)
        ts = timed(lambda: torch._scaled_mm(a8, b8.t(), scale_a=sa.reshape(M, 1), scale_b=sb, out_dtype=torch.bfloat16))
        row["scaled_mm_ms"], row["scaled_mm_tflops"] = ts, flop / ts / 1e9
        row["scaled_mm_rel_diff"] = ((D - out.float()).norm() / D.norm()).item()
    except Exception as e:  # noqa: BLE001 - reported, not fatal: the yardstick does not run at every shape
        row["scaled_mm"] = f"did not run: {type(e).__name__}: {str(e).splitlines()[0][:120]}"
    return row


def time_layer(name, cout, cin, g):
    R = rank_from_reduction_rate(torch.empty(cout, cin, 9), 2.0)
    hw = {64: 56, 128: 28, 256: 14, 512: 7}[cout]
    stride = 2 if cin != cout else 1
    x = torch.randn(64, cin, hw * stride, hw * stride, generator=g, device="cuda")
    facs = [torch.randn(d, R, generator=g, device="cuda") * 0.3 for d in (cout, cin, 9)]
    coded = [quantize_tensor_codes(f, 4, "tensor_mseminmax_symmetric") for f in facs]
    bias = torch.randn(cout, generator=g, device="cuda")
    f8 = build_cp_layer_fp8(R, [(c, i) for _, c, i in coded], bias, cin, cout, (3, 3), (1, 1), (stride, stride), 1, 4,
                            "tensor_mseminmax_symmetric")
    f32 = build_cp_layer(R, [d for d, _, _ in coded], bias, cin, cout, (3, 3), (1, 1), (stride, stride), 1).cuda()
    with torch.no_grad():
        t8 = timed(lambda: f8(x))
        t32 = timed(lambda: f32(x))
        y8, y32 = f8(x), f32(x)
    return {"layer": name, "rank": R, "input": list(x.shape), "fp8_forward_ms": t8, "fp32_forward_ms": t32,
            "rel_frobenius_vs_fp32": ((y8 - y32).norm() / y32.norm()).item()}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    assert torch.cuda.is_available(), "time_code_gemm.py measures on the GPU; there is no CPU path"
    g = torch.Generator(device="cuda").manual_seed(0)
    res = {"card": card(), "gemms": [], "layers": []}
    print(f"card (name, power limit, max SM clock): {res['card']}")
    for label, M, N, K in gemm_shapes():
        row = time_gemm(label, M, N, K, g)
        res["gemms"].append(row)
        print(json.dumps(row))
    torch.backends.cudnn.benchmark = True
    for name, cout, cin, _, _ in wl.resnet18_conv_layers():
        if name.endswith("conv1") and name.split(".")[1] == "0":
            row = time_layer(name, cout, cin, g)
            res["layers"].append(row)
            print(json.dumps(row))
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            json.dump(res, f, indent=1)


if __name__ == "__main__":
    main()
