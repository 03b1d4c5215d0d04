#!/usr/bin/env python
"""Whole-model / sweep driver (new: the reference has only the per-layer CLI and external shell loops).

    torchrun --nproc-per-node 8 scripts/factorize_model.py --model-name resnet18 --bits 3 4 6 8 \
        --reduction-rate 1.5 2 3 4 --qscheme tensor_mseminmax_symmetric --seed 42 --max_iter_als 1000

Enumerates layers x reduction rates x bit-widths (BASELINE configs 2, 3 and 5; layer lists of
source/layer_map.py:10-31), shards the independent solves over the ranks (LPT on the cost model), runs every rank's
units in rounds of `--round-size` concurrent solves through `admmq_factorize_batch` (each solve on its own stream with
an SM budget proportional to its cost, the whole outer loop incl. the reference's stop rules inside the C call),
gathers the factors once (NCCL), and writes the reference's file layout
(`{bits}bit_{qscheme}/factors_admm_seed{seed}/{layer}_admm_{init}_rank_{rank}_mode_{m}.pt`) on rank 0.
No arithmetic crosses a shard boundary: N-GPU results are bitwise identical to 1-GPU results.
"""
import os
import sys
import time
from argparse import ArgumentParser

import numpy as np
import torch
import torch.distributed as dist

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from source import _native, workloads as wl  # noqa: E402
from source.admm import init_factors  # noqa: E402
from source.distributed import gather_results, shard_units  # noqa: E402
from source.solver import layer_weight_as_tensor, rank_from_reduction_rate  # noqa: E402


def parse_args(argv=None):
    ap = ArgumentParser()
    ap.add_argument("--model-name", default="resnet18", choices=["resnet18", "resnet50", "llama7b"])
    ap.add_argument("--bits", type=int, nargs="+", default=[4])
    ap.add_argument("--reduction-rate", type=float, nargs="+", default=[2.0])
    ap.add_argument("--qscheme", default="tensor_mseminmax_symmetric",
                    help="a tensor_* scheme; the clip search also onto FP4 (tensor_mseminmax_e2m1, bits 4), FP8 "
                         "(tensor_mseminmax_e4m3 / _e5m2, bits 8) or FP6 (tensor_mseminmax_e3m2 / _e2m3, bits 6)")
    ap.add_argument("--init", default="random")
    ap.add_argument("--seed", type=int, default=42)
    ap.add_argument("--max_iter_als", type=int, default=5000)
    ap.add_argument("--max_iter_admm", type=int, default=1000)
    ap.add_argument("--solve-precision", type=int, default=1)
    ap.add_argument("--mttkrp-precision", type=int, default=1)
    ap.add_argument("--round-size", type=int, default=16, help="solves that run concurrently on one GPU")
    ap.add_argument("--outroot", default=".")
    ap.add_argument("--layers", nargs="*", default=None, help="subset of layer names")
    ap.add_argument("--backend", default="nccl")
    return ap.parse_args(argv)


def allocate(costs, sm_count):
    """SM budgets proportional to cost, at least one CTA each (0 = every SM for a lone solve)."""
    n = len(costs)
    if n == 1:
        return [0]
    if n >= sm_count:
        return [1] * n
    total = float(sum(costs))
    raw = [max(1.0, c / total * sm_count) for c in costs]
    out = [max(1, int(r)) for r in raw]
    while sum(out) > sm_count:
        out[out.index(max(out))] -= 1
    return out


def main(argv=None):
    args = parse_args(argv)
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise SystemExit("factorize_model.py needs CUDA devices: the solver has no CPU path")
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1:
        dist.init_process_group(args.backend, device_id=dev if args.backend == "nccl" else None)
    layers = wl.model_layers(args.model_name)
    if args.layers:
        layers = [l for l in layers if l[0] in args.layers]
    units = []
    for name, cout, cin, kh, kw in layers:
        W = layer_weight_as_tensor(wl.synthetic_weight(cout, cin, kh, kw, args.seed, name)).contiguous()
        for rr in args.reduction_rate:
            r = rank_from_reduction_rate(W, rr)
            for bits in args.bits:
                units.append({"key": (name, rr, bits), "W": W, "shape": tuple(W.shape), "rank": r, "bits": bits})
    owner = shard_units(units, world)
    sm_count = torch.cuda.get_device_properties(dev).multi_processor_count
    t0 = time.time()
    mine = [u for u, o in zip(units, owner) if o == rank]
    for u in mine:
        u["cost"] = wl.unit_cost(u["shape"], u["rank"], u["bits"])
    mine.sort(key=lambda u: -u["cost"])
    results = {}
    wdev = {}
    for r0 in range(0, len(mine), args.round_size):
        rd = mine[r0:r0 + args.round_size]
        jobs = []
        for u, g in zip(rd, allocate([u["cost"] for u in rd], sm_count)):
            name = u["key"][0]
            if name not in wdev:
                wdev[name] = u["W"].to(dev)
            np.random.seed(args.seed)   # scripts/factorize.py:21-24: the ALS initialisation draws from numpy's global stream
            factors = init_factors(wdev[name], rank=u["rank"], init=args.init, device=dev, seed=args.seed)
            factors = [f.to(dev).contiguous() for f in factors]
            jobs.append(dict(W=wdev[name], factors=factors, duals=[torch.zeros_like(f) for f in factors], bits=u["bits"],
                             qscheme=args.qscheme, max_iter_als=args.max_iter_als, max_iter_admm=args.max_iter_admm,
                             solve_precision=args.solve_precision, mttkrp_precision=args.mttkrp_precision, max_ctas=g,
                             init_is_random=(args.init == "random")))
        out = _native.factorize_batch(jobs)
        torch.cuda.synchronize()
        for u, j, (hist, histq, sweeps, fq) in zip(rd, jobs, out):
            results[u["key"]] = {"factors": [f.detach().cpu() for f in j["factors"]], "loss": hist, "loss_quant": histq}
            print(f"[rank {rank}] {u['key']} rank {u['rank']} on {j['max_ctas'] or sm_count} SMs: {sweeps} sweeps, "
                  f"rec_error {hist[-1]:.6f}, quant {histq[-1]:.6f}", flush=True)
    merged = gather_results(results, device=dev if args.backend == "nccl" else torch.device("cpu"))
    if rank == 0:
        for (name, rr, bits), res in merged.items():
            r = res["factors"][0].shape[1]
            outdir = os.path.join(args.outroot, f"{bits}bit_{args.qscheme}", f"factors_admm_seed{args.seed}")
            os.makedirs(outdir, exist_ok=True)
            prefix = f"{name}_admm_{args.init}_rank_{r}"
            for m, f in enumerate(res["factors"]):
                torch.save(f.clone(), os.path.join(outdir, prefix + f"_mode_{m}.pt"))
            torch.save(res["loss"], os.path.join(outdir, prefix + "_losshist.pt"))
            torch.save(res["loss_quant"], os.path.join(outdir, prefix + "_lossquanthist.pt"))
        print(f"{len(merged)} solves on {world} GPU(s) in {time.time() - t0:.1f} s")
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
