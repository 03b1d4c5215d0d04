"""Factor files -> CP model -> BN calibration -> top-1: the consumer side of scripts/factorize.py
(reference scripts/calibrate.py:151-189 + source/utils.py:134-155), on SYNTHETIC images because neither ImageNet nor
pretrained checkpoints exist offline: the model is torchvision's architecture with seeded random weights
(the weights scripts/factorize.py factorizes with `--weights random`), images are standard normal, labels are the original model's
own predictions.

    python admm-quantization_b200/scripts/calibrate.py --model-name resnet18 --method admm --init random \
        --reduction-rate 2 --bits 4 --qscheme tensor_mseminmax_symmetric --seed 42 [--layers layer1.0.conv1 ...] \
        [--execute fp8]

`--execute fp32` (default) builds float32 CP layers from the factor values; `--execute fp8` re-projects every factor
onto the `--bits/--qscheme` grid and runs the CP layers on the FP8 tensor cores from the codes (replace_with_cp_fp8).

Factor files are read from `{bits}bit_{qscheme}/factors_{method}_seed{seed}/{layer}_{method}_{init}_rank_{rank}_mode_{m}.pt`
(the naming of scripts/factorize.py:164-166, 345-347).
"""
import argparse
import copy
import os
import sys

import torch

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, os.path.dirname(HERE))

from source.models import get_submodule, replace_with_cp, replace_with_cp_fp8  # noqa: E402
from source.solver import layer_weight_as_tensor, rank_from_reduction_rate  # noqa: E402
from source.utils import SyntheticImages, bncalibrate_model, top1_accuracy  # noqa: E402
from source.workloads import resnet18_conv_layers  # noqa: E402


def parse_args(argv=None):
    ap = argparse.ArgumentParser()
    ap.add_argument("--model-name", default="resnet18")
    ap.add_argument("--method", default="admm")
    ap.add_argument("--init", default="random")
    ap.add_argument("--reduction-rate", type=float, default=2.0)
    ap.add_argument("--bits", type=int, required=True)
    ap.add_argument("--qscheme", required=True)
    ap.add_argument("--seed", type=int, required=True)
    ap.add_argument("--layers", nargs="*", default=None, help="default: every factorized 3x3 conv of the model")
    ap.add_argument("--factor-dir", default=None)
    ap.add_argument("--calibration-samples", type=int, default=1000)
    ap.add_argument("--eval-batches", type=int, default=16)
    ap.add_argument("--batch-size", type=int, default=64)
    ap.add_argument("--image-size", type=int, default=64)
    ap.add_argument("--execute", choices=("fp32", "fp8"), default="fp32",
                    help="fp8: run the CP layers on the FP8 tensor cores from the factor codes")
    return ap.parse_args(argv)


def build_model(name, seed):
    import torchvision
    if name != "resnet18":
        raise ValueError(f"unsupported model {name}")
    torch.manual_seed(seed)
    return torchvision.models.resnet18(weights=None)


def main(argv=None):
    args = parse_args(argv)
    device = "cuda" if torch.cuda.is_available() else "cpu"
    model = build_model(args.model_name, args.seed).to(device).eval()
    teacher = copy.deepcopy(model)
    layers = args.layers or [l[0] for l in resnet18_conv_layers()]
    fdir = args.factor_dir or os.path.join(f"{args.bits}bit_{args.qscheme}", f"factors_{args.method}_seed{args.seed}")
    for path in layers:
        w = layer_weight_as_tensor(get_submodule(model, path).weight.detach())
        rank = rank_from_reduction_rate(w, args.reduction_rate)
        prefix = os.path.join(fdir, f"{path}_{args.method}_{args.init}_rank_{rank}_")
        factors = [torch.load(prefix + f"mode_{m}.pt") for m in range(w.ndim)]
        assert all(f.dtype == torch.float32 for f in factors)
        if args.execute == "fp8":
            replace_with_cp_fp8(model, path, factors, args.bits, args.qscheme)
        else:
            replace_with_cp(model, path, factors, rank)
    calib = SyntheticImages(args.calibration_samples // args.batch_size + 2, args.batch_size, args.image_size, seed=1, device=device)
    bncalibrate_model(model, calib, num_samples=args.calibration_samples, device=device)
    evalset = SyntheticImages(args.eval_batches, args.batch_size, args.image_size, seed=2, device=device, labels_from=teacher)
    acc = top1_accuracy(model, evalset, device)
    print(f"top-1 agreement with the uncompressed model on synthetic images: {acc:.2f} % "
          f"({args.eval_batches * args.batch_size} images, {len(layers)} factorized layers)")
    return acc


if __name__ == "__main__":
    main()
