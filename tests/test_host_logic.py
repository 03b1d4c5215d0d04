"""CPU-only tests of the host-side logic: rank / reshape rules against the reference's tables, the LPT sharding,
the ALS + EPC initialisation (property tests - parity unpinned, see DESIGN.md), the CLI argument contract, and the
N > 1 gather path on the gloo backend with two processes."""
import json
import os
import sys

import numpy as np
import pytest
import torch
import torch.distributed as dist
import torch.multiprocessing as mp

REPO = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
PKG = os.path.join(REPO, "admm-quantization_b200")
torch.set_num_threads(1)


def test_rank_rule_reproduces_the_reference_rank_tables():
    from source import workloads as wl
    from source.solver import layer_weight_as_tensor, rank_from_reduction_rate
    table = json.load(open(os.path.join(REPO, "tests", "golden", "rank_table.json")))["table"]
    layers = {n: (co, ci, kh, kw) for n, co, ci, kh, kw in wl.resnet18_conv_layers()}
    assert len(layers) == 16
    checked = 0
    for rate, ranks in table.items():
        for name, ref_rank in ranks.items():
            if name not in layers:
                continue
            co, ci, kh, kw = layers[name]
            W = layer_weight_as_tensor(torch.empty(co, ci, kh, kw))
            assert W.shape == (co, ci, kh * kw)
            assert rank_from_reduction_rate(W, float(rate)) == ref_rank, (rate, name)
            checked += 1
    assert checked >= 60
    assert layer_weight_as_tensor(torch.empty(8, 4, 1, 1)).shape == (8, 4)


def test_lpt_sharding_is_balanced_and_complete():
    from source import workloads as wl
    from source.distributed import shard_units
    units = [{"shape": (co, ci, kh * kw), "rank": int(co * ci * kh * kw / (co + ci + kh * kw) / 2)}
             for _, co, ci, kh, kw in wl.resnet18_conv_layers()]
    costs = [wl.solve_cost(u["shape"], u["rank"]) for u in units]
    for ws in (1, 2, 4, 8):
        owner = shard_units(units, ws)
        assert sorted(set(owner)) == list(range(ws))
        load = [sum(c for c, o in zip(costs, owner) if o == r) for r in range(ws)]
        # the largest unit bounds what any schedule can do (SURVEY 8(e): ~4.2x on 8 GPUs for one ResNet-18)
        assert max(load) <= max(sum(costs) / ws, max(costs)) * 1.34
    assert sum(costs) / max(costs) == pytest.approx(4.2, abs=0.4)


def test_parafac_epc_oracle_properties_and_no_cpu_path():
    """ALS + EPC (parity unpinned: tensorly / musco are absent): the CPU restatement of the published algorithms
    (oracle.admm_oracle.als_fp64 / epc_sweep_fp64 / parafac_epc_fp64, the checker of the GPU test) has the properties
    the method is defined by; the product (source/parafac_epc.py) has no CPU path."""
    from oracle import admm_oracle as orc
    g = torch.Generator().manual_seed(3)
    W = torch.randn(14, 10, 6, generator=g)
    Y = W.double()
    w, fac, errs = orc.als_fp64(Y, 12, 40, 1e-7, np.random.RandomState(5), normalize=True)
    rec = torch.einsum("r,ir,jr,kr->ijk", w, *fac)
    delta = float(torch.linalg.norm(Y - rec))
    assert delta / float(torch.linalg.norm(Y)) < 0.75          # ALS does reduce the error
    assert all(b <= a + 1e-12 for a, b in zip(errs, errs[1:]))  # monotonically
    fac[-1] = fac[-1] * w

    def intensity2(fs):
        lam = torch.ones(12, dtype=torch.float64)
        for f in fs:
            lam = lam * torch.linalg.norm(f, dim=0)
        return float((lam ** 2).sum())

    prev = intensity2(fac)
    for _ in range(8):
        fac = orc.epc_sweep_fp64(Y, fac, delta)
        err = float(torch.linalg.norm(Y - torch.einsum("ir,jr,kr->ijk", *fac)))
        cur = intensity2(fac)
        assert err <= delta * (1 + 1e-6)                       # the error bound is preserved
        assert cur <= prev * (1 + 1e-9)                        # the intensity never grows
        prev = cur
    lam, Us = orc.parafac_epc_fp64(W, 12, als_maxiter=15, epc_maxiter=4, epc_rounds=2, rng=np.random.RandomState(3))
    assert [tuple(u.shape) for u in Us] == [(14, 12), (10, 12), (6, 12)] and Us[0].dtype == torch.float64   # original mode order
    rel = float(torch.linalg.norm(Y - torch.einsum("ir,jr,kr->ijk", *Us)) / torch.linalg.norm(Y))
    assert rel < 0.8 and lam.shape == (12,)
    from source.parafac_epc import parafac_epc
    with pytest.raises(NotImplementedError):
        parafac_epc(W, 4, init="svd")
    if not torch.cuda.is_available():
        with pytest.raises(RuntimeError, match="no CPU fallback"):
            parafac_epc(W, 4)


def test_init_factors_random_matches_reference_generator_semantics():
    from source.admm import init_factors
    W = torch.zeros(5, 4, 3)
    a = init_factors(W, 7, init="random", device=None, seed=42)
    gen = torch.Generator().manual_seed(42)
    ref = [torch.randn(d, 7, generator=gen) for d in W.shape]   # source/admm.py:22-28: one generator, modes in order
    assert all(torch.equal(x, y) for x, y in zip(a, ref))
    with pytest.raises(NotImplementedError):
        init_factors(W, 7, init="bogus", seed=1)


def test_cli_argument_contract():
    sys.path.insert(0, os.path.join(PKG, "scripts"))
    import importlib
    fz = importlib.import_module("factorize")
    base = ["--model-name", "resnet18", "--method", "admm", "--layer", "layer1.0.conv1", "--bits", "4", "--seed", "42",
            "--qscheme", "tensor_mseminmax_symmetric"]
    with pytest.raises(ValueError):
        fz.parse_args(base)                                     # neither --rank nor --reduction-rate (:98-99)
    with pytest.raises(ValueError):
        fz.parse_args([a if a != "admm" else "bogus" for a in base] + ["--rank", "3"])   # (:100-101)
    a = fz.parse_args(base + ["--reduction-rate", "2"])
    assert (a.max_iter_als, a.max_iter_admm, a.max_iter_epc, a.init) == (5000, 1000, 5000, "random")
    assert fz.run_name(fz.parse_args(base + ["--rank", "134"])) == "admm_l=layer1.0.conv1_r=134_b=4_s=42_i=random_tensor_mseminmax_symmetric"


def test_bench_output_dump_whole_under_the_limit_and_a_fixed_sample_above(tmp_path, monkeypatch):
    """bench.py --dump-outputs: every array of every unit is written whole while they fit the size limit; above it each
    large array is replaced by a sample at the same seeded positions in every run, and the files stay within the limit."""
    import importlib.util
    # bench.py sets this at import for the processes it runs; keep it out of the test process
    monkeypatch.setenv("CUDA_DEVICE_MAX_CONNECTIONS", os.environ.get("CUDA_DEVICE_MAX_CONNECTIONS", "32"))
    spec = importlib.util.spec_from_file_location("bench", os.path.join(REPO, "bench.py"))
    bench = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(bench)
    g = torch.Generator().manual_seed(0)
    fac = [torch.randn(d, 40, generator=g) for d in (300, 200, 9)]
    units = [("layer1.0.conv1/rr2.0/b4", fac, [f.round() for f in fac], 0.5, 0.25)]
    name = "layer1.0.conv1_rr2.0_b4"
    bench.dump_outputs(str(tmp_path / "whole"), units, 1)
    whole = {p.name: np.load(p) for p in (tmp_path / "whole").iterdir()}
    assert sorted(whole) == sorted([f"{name}.rec_error.npy"] + [f"{name}.factor{m}{q}.npy" for m in range(3)
                                                                for q in ("", "_quantized")])
    assert whole[f"{name}.rec_error.npy"].dtype == np.float64 and whole[f"{name}.rec_error.npy"].tolist() == [0.5, 0.25]
    for m in range(3):
        assert whole[f"{name}.factor{m}.npy"].dtype == np.float32
        assert np.array_equal(whole[f"{name}.factor{m}.npy"], fac[m].numpy())
        assert np.array_equal(whole[f"{name}.factor{m}_quantized.npy"], fac[m].round().numpy())
    monkeypatch.setattr(bench, "DUMP_LIMIT_BYTES", 100_000)
    runs = []
    for k in range(2):
        d = tmp_path / f"sampled{k}"
        bench.dump_outputs(str(d), units, 1)
        assert sum(p.stat().st_size for p in d.iterdir()) <= 100_000
        runs.append({p.name: np.load(p) for p in d.iterdir()})
    assert sorted(runs[0]) == sorted(whole) and sorted(runs[1]) == sorted(whole)
    sample = runs[0][f"{name}.factor0.npy"]
    assert 0 < sample.size < fac[0].numel() and np.isin(sample, fac[0].numpy()).all()
    assert np.array_equal(runs[0][f"{name}.factor2.npy"], fac[2].numpy())     # small arrays stay whole
    assert all(np.array_equal(runs[0][n], runs[1][n]) for n in runs[0])


def _gather_worker(rank, world, port, out):
    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port), RANK=str(rank), WORLD_SIZE=str(world))
    sys.path[:0] = [REPO, PKG]
    from source.distributed import gather_results, shard_units
    dist.init_process_group("gloo", rank=rank, world_size=world)
    units = [{"key": f"u{i}", "seed": 100 + i, "shape": (8 + i, 6, 3), "rank": 5 + i} for i in range(5)]
    owner = shard_units(units, world)
    local = {}
    for u, o in zip(units, owner):
        if o == rank:
            g = torch.Generator().manual_seed(u["seed"])
            local[u["key"]] = {"factors": [torch.randn(d, u["rank"], generator=g) for d in u["shape"]],
                               "loss": [0.5, 0.4], "loss_quant": [0.6]}
    merged = gather_results(local)
    if rank == 0:
        ok = sorted(merged) == [u["key"] for u in units]
        for u in units:
            g = torch.Generator().manual_seed(u["seed"])
            ref = [torch.randn(d, u["rank"], generator=g) for d in u["shape"]]
            ok = ok and all(torch.equal(a, b) for a, b in zip(merged[u["key"]]["factors"], ref))
            ok = ok and merged[u["key"]]["loss"] == [0.5, 0.4]
        out.put(ok)
    else:
        assert merged is None
    dist.destroy_process_group()


def test_two_rank_gather_on_gloo_is_bitwise_identical():
    """world_size 2 on CPU: units sharded by LPT, results gathered once; the merged factors equal what a single
    process computes (no arithmetic crosses a shard boundary)."""
    ctx = mp.get_context("spawn")
    out = ctx.SimpleQueue()
    port = 29500 + (os.getpid() % 2000)
    procs = [ctx.Process(target=_gather_worker, args=(r, 2, port, out)) for r in range(2)]
    for p in procs:
        p.start()
    for p in procs:
        p.join(120)
        assert p.exitcode == 0
    assert out.get() is True


# ------------------------------------------------------------------ factor files -> CP model (SURVEY 8(f-1))
def test_cp_layers_reproduce_the_convolution_they_factorize():
    """reference source/models.py:24-74: conv1 (B^T) -> depthwise conv2 (C) -> conv3 (A, bias) equals the dense
    convolution with W[o,i,k] = sum_r A[o,r] B[i,r] C[k,r]; same for the two-layer form of a 1x1 convolution."""
    import torch
    from source.models import build_cp_layer, build_cp2conv_layer, build_cpfc_layer
    g = torch.Generator().manual_seed(0)
    R = 5
    A, B, C = (torch.randn(n, R, generator=g) for n in (8, 6, 9))
    conv = torch.nn.Conv2d(6, 8, 3, padding=1, stride=2, bias=True)
    with torch.no_grad():
        conv.weight.copy_(torch.einsum("or,ir,kr->oik", A, B, C).reshape(8, 6, 3, 3))
    cp = build_cp_layer(R, [A, B, C], conv.bias.detach(), 6, 8, (3, 3), (1, 1), (2, 2), 1)
    assert [n for n, _ in cp.named_children()] == ["conv1", "conv2", "conv3"]
    x = torch.randn(2, 6, 10, 10, generator=g)
    assert torch.allclose(conv(x), cp(x), atol=1e-4)
    pw = torch.nn.Conv2d(6, 8, 1, stride=2, bias=False)
    with torch.no_grad():
        pw.weight.copy_((A @ B.t())[:, :, None, None])
    cp2 = build_cp2conv_layer(R, [A, B], None, 6, 8, (0, 0), (2, 2))
    assert torch.allclose(pw(x), cp2(x), atol=1e-4)
    fc = build_cpfc_layer(R, [A, B], torch.zeros(8), 6, 8)
    v = torch.randn(3, 6, generator=g)
    assert torch.allclose(fc(v), v @ (A @ B.t()).t(), atol=1e-4)
    with pytest.raises(AssertionError):   # wrong factor shape (reference: the shape asserts of source/models.py:39-41)
        build_cp_layer(R, [A[:7], B, C], None, 6, 8, (3, 3), (1, 1), (1, 1), 1)


def test_replace_calibrate_and_score_on_synthetic_images():
    """replace_with_cp + bncalibrate_model + top1_accuracy (reference scripts/calibrate.py:161-189,
    source/utils.py:134-155) on a seeded ResNet-18: exact rank-full factors keep every prediction."""
    import copy
    import torch
    import torchvision
    from source.models import get_submodule, replace_with_cp
    from source.utils import SyntheticImages, bncalibrate_model, top1_accuracy
    torch.manual_seed(3)
    model = torchvision.models.resnet18(weights=None).eval()
    teacher = copy.deepcopy(model)
    w = get_submodule(model, "layer1.0.conv1").weight.detach()          # (64, 64, 3, 3)
    # an exact CP representation: one component per (input channel, tap) pair
    cin, taps = 64, 9
    A = w.reshape(64, cin * taps).clone()
    B = torch.eye(cin).repeat_interleave(taps, dim=1)
    C = torch.eye(taps).repeat(1, cin)
    replace_with_cp(model, "layer1.0.conv1", [A, B, C])
    ev = SyntheticImages(2, 8, image_size=32, seed=2, labels_from=teacher)
    assert top1_accuracy(model, ev, "cpu") == 100.0
    bn_before = model.bn1.running_mean.clone()
    bncalibrate_model(model, SyntheticImages(3, 8, image_size=32, seed=1), num_samples=16, device="cpu")
    assert not torch.equal(bn_before, model.bn1.running_mean)            # statistics were re-estimated
    assert not model.training and all(not p.requires_grad for p in model.parameters())


def test_modelled_sm_budgets_follow_the_wave_structure():
    """source/workloads.py: the tensor-core ridge product takes whole waves of tiles, so budgets are moved from wave
    boundary to wave boundary; the budgets never exceed the SM count and the slowest predicted layer is not starved."""
    from source import workloads as wl
    costs = [wl.product_cost(512, 1141, g) for g in range(1, 149)]
    assert all(a >= b for a, b in zip(costs, costs[1:]))                         # more CTAs never hurt ...
    assert len(set(costs)) < 40                                                  # ... but only at wave boundaries
    assert wl.product_cost(512, 1141, 36) == 144.0 < wl.product_cost(512, 1141, 35)   # 36 tiles of 128: one wave
    assert wl.product_cost(9, 1141, 8) == pytest.approx(2 * wl.product_cost(9, 1141, 16))                      # skinny: 1 / g
    big = (297.0, 31, [(512, 1141, 61.0, 40.8, 999), (512, 1141, 61.0, 40.8, 999), (9, 1141, 17.0, 20.0, 999)])
    mid = (270.0, 7, [(256, 566, 40.0, 51.0, 999), (256, 566, 40.0, 51.0, 999), (9, 566, 18.0, 19.0, 999)])
    small = (112.0, 2, [(64, 134, 17.0, 28.0, 999), (64, 134, 17.0, 28.0, 999), (9, 134, 10.0, 19.0, 999)])
    assert wl.predict_sweep_ms(*big[:2], 31, big[2]) == pytest.approx(297.0)
    assert wl.predict_sweep_ms(*big[:2], 36, big[2]) < wl.predict_sweep_ms(*big[:2], 32, big[2]) < 297.0
    layers = [small] * 4 + [mid] * 4 + [big] * 3
    g = wl.allocate_ctas_modelled(layers, 148)
    assert sum(g) <= 148 and min(g) >= 1 and g[-1] > g[4] > g[0]
    t = [wl.predict_sweep_ms(m, g0, gi, mo) for (m, g0, mo), gi in zip(layers, g)]
    assert max(t) < 297.0                                   # better than the measured starting point
    assert wl.allocate_ctas_modelled(layers, 8) == [1] * 11  # more solves than SMs: one CTA each
