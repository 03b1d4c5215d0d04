#!/usr/bin/env python
"""`scripts/factorize.py` of the reference (:38-357) on the B200 kernels: same flags, same output files.

    python scripts/factorize.py --model-name resnet18 --method admm --init random --layer layer1.0.conv1 \
        --reduction-rate 2 --bits 4 --qscheme tensor_mseminmax_symmetric --seed 42

Differences that are deliberate:
  * the layer lookup + reshape the reference left commented out (:130-147) is implemented (the committed script only
    works for `deit`): walk `model.<layer path>`, conv (Cout,Cin,kh,kw) -> (Cout,Cin,kh*kw), 1x1 -> (Cout,Cin);
  * `--weights {pretrained,random}` (default random: there is no network for checkpoints) and
    `--weight-file` (a .pt tensor or state_dict) as additional optional flags;
  * `--eps`, `--tol`, `--num-attempts`, `--solve-precision`, `--outdir` expose the reference's hard-coded constants with
    identical defaults (:179-180, source/quantization.py:118).
"""
import os
import random
import sys
import time
from argparse import ArgumentParser

import numpy as np
import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from source.admm import init_factors, squared_relative_diff  # noqa: E402
from source.parafac_epc import parafac_als, parafac_epc  # noqa: E402
from source.quantization import quantize_tensor  # noqa: E402
from source.solver import LayerSolver, layer_weight_as_tensor  # noqa: E402


def set_seed(seed):
    torch.manual_seed(seed)
    np.random.seed(seed)
    random.seed(seed)


def run_name(args):
    return "_".join([args.method, f"l={args.layer}", f"r={args.rank}", f"b={args.bits}", f"s={args.seed}",
                     f"i={args.init}", f"{args.qscheme}"])


def parse_args(argv=None):
    parser = ArgumentParser()
    parser.add_argument("--model-name", type=str, required=True, help="[resnet18, resnet50]")
    parser.add_argument("--with-wandb", action="store_true", help="Whether to enable experiment logging to wandb.")
    parser.add_argument("--method", type=str, required=True, help="[admm, parafac, parafac-epc]")
    parser.add_argument("--init", type=str, required=False, default="random", help="[random, parafac-epc]")
    parser.add_argument("--layer", type=str, required=True,
                        help="Name of a layer to decompose(for example, layer2.1.conv1 means model.layer2[1].conv1)")
    parser.add_argument("--rank", type=int, required=False, help="Rank for decomposition.")
    parser.add_argument("--reduction-rate", type=float, required=False,
                        help="Rank is computed such that number of parameters reduce <reduction_rate> times.")
    parser.add_argument("--bits", required=True, type=int, help="Number of quantization bits.")
    parser.add_argument("--max_iter_als", required=False, default=5000, type=int)
    parser.add_argument("--max_iter_admm", required=False, default=1000, type=int)
    parser.add_argument("--max_iter_epc", required=False, default=5000, type=int)
    parser.add_argument("--seed", required=True, type=int, help="Random seed.")
    parser.add_argument("--qscheme", required=True, type=str, help="[tensor_mseminmax_symmetric, tensor_minmax, tensor_mseminmax_e2m1 (bits 4), "
                        "tensor_mseminmax_e4m3 / tensor_mseminmax_e5m2 (bits 8), tensor_mseminmax_e3m2 / tensor_mseminmax_e2m3 (bits 6)]")
    # additions (defaults reproduce the reference's hard-coded values)
    parser.add_argument("--weights", default="pretrained", choices=["pretrained", "random"],
                        help="pretrained (default, what the reference loads: `resnet18(pretrained=True)`): fails loudly when the "
                             "checkpoint is neither cached nor downloadable; random: the architecture's own initialisation "
                             "(must be asked for explicitly - the output directory is then tagged `_randomweights`)")
    parser.add_argument("--weight-file", default=None, help=".pt file holding the layer's weight tensor or a state_dict")
    parser.add_argument("--eps", type=float, default=1e-8)
    parser.add_argument("--tol", type=float, default=1e-5)
    parser.add_argument("--num-attempts", type=int, default=200)
    parser.add_argument("--solve-precision", type=int, default=0,
                        help="0 parity mode (float64 product with the float64 inverse), 1 3xTF32 tcgen05, 2 float32 FFMA")
    parser.add_argument("--outdir", default=None)
    args = parser.parse_args(argv)
    if args.rank is None and args.reduction_rate is None:
        raise ValueError("One of [--rank, --reduction-rate] arguments must be specified.")
    if args.method not in ["admm", "parafac", "parafac-epc"]:
        raise ValueError("Method must be on of [admm, parafac, parafac-epc].")
    return args


def load_weight(args):
    if args.weight_file is not None:
        obj = torch.load(args.weight_file, map_location="cpu")
        if isinstance(obj, dict):
            obj = obj[args.layer + ".weight"]
        return obj.detach().float()
    if args.model_name not in ("resnet18", "resnet50"):
        raise ValueError(f"unrecognized model name: {args.model_name}")
    import torchvision
    ctor = getattr(torchvision.models, args.model_name)
    if args.weights == "pretrained":
        try:
            model = ctor(weights="DEFAULT")
        except Exception as e:  # noqa: BLE001 - no network / no cached checkpoint: never fall back to random weights silently
            raise RuntimeError(f"could not load the pretrained {args.model_name} checkpoint ({type(e).__name__}: {e}); pass "
                               "--weight-file with a local checkpoint, or --weights random to factorize the architecture's "
                               "random initialisation on purpose") from e
    else:
        print("WARNING: --weights random: factorizing RANDOMLY INITIALISED weights (not the reference's pretrained model)")
        model = ctor(weights=None)
    layer = model
    for attr in args.layer.split("."):
        layer = layer[int(attr)] if attr.isdigit() else getattr(layer, attr)
    return layer.weight.detach().float()


def main(argv=None):
    if not torch.cuda.is_available():
        raise SystemExit("factorize.py needs a CUDA device: the B200 solver has no CPU path")
    device = torch.device("cuda:0")
    print("Running on:", device)
    args = parse_args(argv)
    print("Args:", args)
    set_seed(args.seed)
    weight = layer_weight_as_tensor(load_weight(args)).contiguous().to(device)
    if weight.ndim == 3:
        ein_op = "ir,jr,kr->ijk"
    elif weight.ndim == 2:
        ein_op = "ir,jr->ij"
    else:
        raise ValueError("Incorrect number of dimentions in weight tensor")
    if args.rank is None:
        args.rank = int(weight.numel() / sum(list(weight.shape)) / args.reduction_rate)
    outdir = args.outdir or f"{args.bits}bit_{args.qscheme}/factors_{args.method}_seed{args.seed}"
    if args.outdir is None and args.weights == "random" and args.weight_file is None:
        outdir += "_randomweights"   # never under the reference's name: calibrate.py would score meaningless factors
    os.makedirs(outdir, exist_ok=True)
    fileprefix = f"{args.layer}_{args.method}_{args.init}_rank_{args.rank}"
    run = None
    if args.with_wandb:
        import wandb
        run = wandb.init(config=args, name=run_name(args))

    start = time.time()
    if args.method == "admm":
        if run:
            run.config.update({"tol": args.tol, "eps": args.eps})
        factors = init_factors(weight, rank=args.rank, init=args.init, device=device, seed=args.seed)
        solver = LayerSolver(weight, factors, args.bits, args.qscheme, max_iter_admm=args.max_iter_admm, eps=args.eps,
                             tol=args.tol, num_attempts=args.num_attempts, init_is_random=(args.init == "random"),
                             solve_precision=args.solve_precision)
        if run and solver.loss_hist:
            run.log({"rec_error": solver.loss_hist[0], "quant_rec_error": solver.loss_quant_hist[0]})
        try:
            from tqdm import tqdm
            iterator = tqdm(range(args.max_iter_als))
        except ImportError:
            iterator = range(args.max_iter_als)
        for _ in iterator:
            err, errq = solver.sweep()
            if run:
                run.log({"rec_error": err, "quant_rec_error": errq})
            if solver.should_stop():
                break
        factors, factors_quantized = solver.factors, solver.factors_q
        torch.save(solver.loss_hist, os.path.join(outdir, fileprefix + "_losshist.pt"))
        torch.save(solver.loss_quant_hist, os.path.join(outdir, fileprefix + "_lossquanthist.pt"))
    elif args.method == "parafac":
        _, factors = parafac_als(weight, args.rank, n_iter_max=args.max_iter_als, tol=1e-8, random_state=args.seed)
        factors_quantized = [quantize_tensor(f, qscheme=args.qscheme, bits=args.bits) for f in factors]
    else:  # parafac-epc
        _, factors = parafac_epc(weight, rank=args.rank, init=args.init, als_maxiter=args.max_iter_als,
                                 epc_maxiter=args.max_iter_epc)
        factors = [f.to(torch.float) for f in factors]
        factors_quantized = [quantize_tensor(f, qscheme=args.qscheme, bits=args.bits) for f in factors]
    torch.cuda.synchronize()
    end = time.time()
    print("Factorization took {} minutes".format((end - start) / 60))

    for mode, factor in enumerate(factors):
        torch.save(factor.detach().cpu(), os.path.join(outdir, fileprefix + f"_mode_{mode}.pt"))
    error = squared_relative_diff(weight, torch.einsum(ein_op, *factors))
    quantized_error = squared_relative_diff(weight, torch.einsum(ein_op, *factors_quantized))
    print("Factorization error is {} for usual and {} for quantized".format(error, quantized_error))
    if run:
        run.log({"rec_error": error, "quant_rec_error": quantized_error})
        run.finish()
    return error, quantized_error


if __name__ == "__main__":
    main()
