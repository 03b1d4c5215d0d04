import os, sys
REPO = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path[:0] = [REPO, os.path.join(REPO, "admm-quantization_b200")]
import torch
from oracle import admm_oracle as orc
from source import _native as nat
MSE="tensor_mseminmax_symmetric"
torch.set_num_threads(1)
g = torch.Generator().manual_seed(33)
for (I, R, bits, qs) in [(64, 134, 4, MSE), (9, 134, 4, MSE), (64, 134, 3, MSE), (48, 100, 8, "tensor_minmax"), (64, 134, 4, "tensor_affine")]:
    Bf, Cf = torch.randn(64, R, generator=g), torch.randn(9, R, generator=g)
    G = (Bf.T @ Bf) * (Cf.T @ Cf)
    F = torch.randn(I, R, generator=g) * 24
    H0 = torch.randn(I, R, generator=g)
    U0 = torch.randn(I, R, generator=g) * 0.1
    for iters in (2, 4):
        Uo = U0.clone()
        Ho, Uo, _ = orc.admm_iteration(H0.clone(), Uo, F, G, iters, 1e-8, bits, qs)
        outs = []
        for ctas in (1, 0):
            H, U = H0.clone().cuda(), U0.clone().cuda()
            rep = nat.read_report(nat.admm_iteration_inplace(H, U, F.cuda(), G.cuda(), iters, 1e-8, bits, qs, precision=0, max_ctas=ctas))
            outs.append((H.cpu(), U.cpu(), rep))
        def cf(a, b):
            tol = 1e-4 * float(b.abs().max()); return float(((a - b).abs() <= tol).float().mean())
        print(I, R, bits, qs, iters, "H res-vs-oracle", cf(outs[0][0], Ho), "gen-vs-oracle", cf(outs[1][0], Ho), "res-vs-gen", cf(outs[0][0], outs[1][0]),
              "U res-vs-oracle", cf(outs[0][1], Uo), "gen-vs-oracle", cf(outs[1][1], Uo), "scale", outs[0][2].scale, outs[1][2].scale, "best", outs[0][2].best_index, outs[1][2].best_index)
