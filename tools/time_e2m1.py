"""E2M1 (`tensor_mseminmax_e2m1`) against the 4-bit uniform clip search (`tensor_mseminmax_symmetric`), or with
`--scheme` / `--bits` any other clip-search grids against the uniform grid of the same width (FP8: `--bits 8 --scheme
tensor_mseminmax_e4m3 tensor_mseminmax_e5m2`, FP6: `--bits 6 --scheme tensor_mseminmax_e3m2 tensor_mseminmax_e2m3`):

  1. per-iteration time of the ADMM inner loop (admmq_admm_loop, precision 1) for the factors of the ResNet-18 headline
     at the CTA budgets bench.py gives them; CUDA events around `--iters` iterations, the two schemes alternated
     `--reps` times, median reported;
  2. the quantized reconstruction error of the 16 ResNet-18 3x3 conv layers (bench.py's synthetic Kaiming-normal
     weights, rank from reduction rate 2, random init) after `--sweeps` outer sweeps of LayerSolver.

    python tools/time_e2m1.py [--scheme S ...] [--bits B] [--iters 200] [--reps 3] [--sweeps 10] [--inner 300]
                              [--out result.json]
Needs a CUDA device.  Prints two tables and one JSON line (written to --out as well)."""
import argparse
import json
import os
import sys
from types import SimpleNamespace

REPO = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
for p in (REPO, os.path.join(REPO, "admm-quantization_b200")):
    if p not in sys.path:
        sys.path.insert(0, p)

import numpy as np  # noqa: E402
import torch  # noqa: E402

UNIFORM, E2M1 = "tensor_mseminmax_symmetric", "tensor_mseminmax_e2m1"


def tag(scheme):
    """Key and column name of a scheme: "uniform", or the format ("e2m1", "e4m3", ...)."""
    return "uniform" if scheme == UNIFORM else scheme.rsplit("_", 1)[-1]


def loop_times(iters, reps, schemes=(E2M1,), bits=4):
    import bench
    from source import _native as nat, workloads as wl
    sms = torch.cuda.get_device_properties(0).multi_processor_count
    units, _ = bench.workload_units(SimpleNamespace(workload="resnet18", reduction_rate=2.0, bits=4))
    shapes = [bench.unit_shape(u) for u in units]
    ranks = [bench.unit_rank(u) for u in units]
    budgets = bench.allocate_ctas([wl.solve_cost(s, r) for s, r in zip(shapes, ranks)], sms, 1)
    seen, rows = set(), []
    g = torch.Generator().manual_seed(0)
    for shape, R, b in zip(shapes, ranks, budgets):
        for I in shape:
            if (I, R, b) in seen:
                continue
            seen.add((I, R, b))
            B, C = torch.randn(96, R, generator=g), torch.randn(9, R, generator=g) / 3
            G = ((B.T @ B) * (C.T @ C)).cuda()
            F = (torch.randn(I, R, generator=g).cuda() @ G).contiguous()
            H0, U0 = torch.randn(I, R, generator=g).cuda(), (torch.randn(I, R, generator=g) * 0.1).cuda()
            Minv, rho, st = nat.spd_inverse(G, max_ctas=b)[:3]
            ws = torch.empty(nat.admm_loop_workspace_bytes(I, R, 200), dtype=torch.uint8, device="cuda")
            codes = torch.empty(I, R, dtype=torch.int8, device="cuda")
            order = (UNIFORM,) + tuple(schemes)
            us = {s: [] for s in order}

            def run(scheme):
                H, U = H0.clone(), U0.clone()
                e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                e0.record()
                nat.admm_loop_inplace(H, U, F, Minv, rho, st, iters + 1, 0.0, bits, scheme, 200, codes=codes, ws=ws,
                                      precision=1, max_ctas=b)
                e1.record()
                torch.cuda.synchronize()
                return e0.elapsed_time(e1) * 1e3 / iters

            for scheme in order:   # warm-up: module load, shared-memory attributes
                run(scheme)
            for _ in range(reps):
                for scheme in order:
                    us[scheme].append(run(scheme))
            kid = nat.loop_kernel(I, R, 200, 1, b if 0 < b < sms else sms)
            row = {"I": I, "R": R, "budget": b, "kernel": kid}
            row.update({tag(s) + "_us": float(np.median(us[s])) for s in order})
            row.update({tag(s) + "_runs": us[s] for s in order})
            rows.append(row)
    return rows


def quantized_errors(sweeps, inner, schemes=(E2M1,), bits=4):
    from source import workloads as wl
    from source.solver import LayerSolver
    rows = []
    for name, cout, cin, kh, kw in wl.resnet18_conv_layers():
        W = wl.layer_weight_as_tensor(wl.synthetic_weight(cout, cin, kh, kw, 42, name)).contiguous()
        R = wl.rank_from_reduction_rate(W, 2.0)
        init = wl.random_init(W.shape, R, 42)
        row = {"layer": name, "rank": R}
        for scheme in (UNIFORM,) + tuple(schemes):
            s = LayerSolver(W.cuda(), [f.cuda() for f in init], bits, scheme, max_iter_admm=inner, solve_precision=1,
                            mttkrp_precision=1)
            s.run(sweeps)
            row[tag(scheme)] = float(s.loss_quant_hist[-1])
            row[tag(scheme) + "_unquantized"] = float(s.loss_hist[-1])
        rows.append(row)
    return rows


def main():
    ap = argparse.ArgumentParser(description=__doc__, formatter_class=argparse.RawDescriptionHelpFormatter)
    ap.add_argument("--scheme", nargs="+", default=[E2M1], help="clip-search grids to set against the uniform one")
    ap.add_argument("--bits", type=int, default=4, help="the width of every scheme (E2M1 4, FP8 8, FP6 6)")
    ap.add_argument("--iters", type=int, default=200)
    ap.add_argument("--reps", type=int, default=3)
    ap.add_argument("--sweeps", type=int, default=10)
    ap.add_argument("--inner", type=int, default=300)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("time_e2m1.py needs a CUDA device")
    from source import _native as nat
    dev = torch.cuda.get_device_properties(0)
    tags = [tag(s) for s in args.scheme]
    head = "".join(f" {t.upper()} |" for t in tags) + "".join(f" {t.upper()} / uniform |" for t in tags)
    rule = "---|" * (2 * len(tags))
    loops = loop_times(args.iters, args.reps, args.scheme, args.bits)
    print(f"per-iteration loop time, us ({dev.name}, precision 1, median of {args.reps} alternated runs of {args.iters})")
    print(f"| factor | budget | kernel | uniform {args.bits}-bit |{head}")
    print(f"|---|---|---|---|{rule}")
    for r in loops:
        k = r["kernel"]
        kname = f"TC{k - 1000}" if k > 1000 else {v: n for n, v in _kernel_ids().items()}.get(k, str(k))
        cols = "".join(f" {r[t + '_us']:.2f} |" for t in tags) + "".join(f" {r[t + '_us'] / r['uniform_us']:.3f} |"
                                                                          for t in tags)
        print(f"| {r['I']} x {r['R']} | {r['budget']} | {kname} | {r['uniform_us']:.2f} |{cols}")
    errs = quantized_errors(args.sweeps, args.inner, args.scheme, args.bits)
    print(f"\nquantized reconstruction error after {args.sweeps} sweeps (max_iter_admm {args.inner}, {args.bits} bits)")
    print(f"| layer | rank | uniform {args.bits}-bit |{head}")
    print(f"|---|---|---|{rule}")
    for r in errs:
        cols = "".join(f" {r[t]:.5f} |" for t in tags) + "".join(f" {r[t] / r['uniform']:.3f} |" for t in tags)
        print(f"| {r['layer']} | {r['rank']} | {r['uniform']:.5f} |{cols}")
    res = {"device": dev.name, "loops": loops, "errors": errs, "sweeps": args.sweeps, "inner": args.inner,
           "iters": args.iters, "reps": args.reps, "launches": int(nat.launch_count())}
    line = json.dumps(res)
    print(line)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            f.write(line + "\n")


def _kernel_ids():
    import re
    text = open(os.path.join(REPO, "include", "admmq.h")).read()
    return {k: int(v) for k, v in re.findall(r"#define ADMMQ_LOOP_(\w+) (\d+)", text)}


if __name__ == "__main__":
    main()
