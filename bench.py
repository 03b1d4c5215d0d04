#!/usr/bin/env python
"""Benchmark of the quantization-aware CP factorization hot path (BASELINE.json metric).

  python bench.py --gpus N --steps K --warmup W            # this repo's CUDA path (one process per GPU)
  python bench.py --impl reference --gpus N --steps K ...  # the reference's own functions on the host CPU
  python bench.py --full [--init parafac-epc]              # the metric's second half: factorize time to the stop rule

Default workload (BASELINE.json configs[1]): every 3x3 conv layer of ResNet-18 (16 layers, synthetic
Kaiming-normal weights, rank from reduction-rate 2.0), ADMM with 4-bit tensor_mseminmax_symmetric
projection, max_iter_admm = 1000.  One STEP = one outer sweep over all 16 layers = 16 x 3 factor updates
x 999 inner ADMM iterations (+ Gram, MTTKRP, ridge inverse, re-projection, two reconstruction errors).
Metric: inner ADMM iterations per second (SURVEY 8(d): the unit of work is one inner iteration of one
factor), counted from the kernels' device reports (the inner loop may leave early exactly where the reference's
does, tests/golden/early_exit.npz).

With N GPUs ONE job is sharded: the independent units (layers; with --workload sweep256 the 256 units
layer x reduction-rate {1.5, 2, 3, 4} x bits {3, 4, 6, 8} of configs[2]) are assigned to the ranks by
longest-processing-time-first (source/distributed.py), every rank runs its units concurrently on its own SM budgets,
there is no data-path collective, and the packed factors are gathered once with one NCCL all_gather after the timed
region -> "scaling": "strong".  `--seed-replicas` keeps round 1's weak-scaling mode (every rank the whole layer set for
its own seed) as a labelled extra.

Prints ONE JSON line on rank 0.
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

# One hardware work queue per layer stream: with the default of 8 connections, streams that share a queue falsely
# serialise behind each other's long-running persistent kernels (measured: the last-launched layers started 0.4 s late).
os.environ.setdefault("CUDA_DEVICE_MAX_CONNECTIONS", "32")

REPO = os.path.dirname(os.path.abspath(__file__))
PKG = os.path.join(REPO, "admm-quantization_b200")
for p in (REPO, PKG):
    if p not in sys.path:
        sys.path.insert(0, p)

QSCHEME = "tensor_mseminmax_symmetric"
METRIC = "admm_inner_iter_per_s"
UNIT = "inner ADMM iterations/s"
SWEEP_RATES = (1.5, 2.0, 3.0, 4.0)
SWEEP_BITS = (3, 4, 6, 8)
DUMP_LIMIT_BYTES = 64 * 10**6     # --dump-outputs: all files of one run together
DUMP_WHOLE_ELEMENTS = 4096        # arrays up to this size are never sampled


def parse_args():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=3)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="native", choices=["native", "reference"])
    ap.add_argument("--workload", default="resnet18", choices=["resnet18", "layer1", "resnet50-l4", "llama7b", "sweep256"])
    ap.add_argument("--bits", type=int, default=4)
    ap.add_argument("--reduction-rate", type=float, default=2.0)
    ap.add_argument("--max-iter-admm", type=int, default=1000)
    ap.add_argument("--cpu-budget-s", type=float, default=15.0, help="CPU seconds for the cpu_baseline sample")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--no-parity-leg", action="store_true",
                    help="skip the one-step measurement of the same workload in the parity mode (precision 0: FP64 pipe, ~10x slower)")
    ap.add_argument("--no-eager-reference", action="store_true",
                    help="skip the informative second bar: the reference's own Python run eagerly on this GPU")
    ap.add_argument("--mttkrp-precision", type=int, default=1,
                    help="0 = float64-accumulating CUDA-core MTTKRP, 1 = 3xTF32 tcgen05 MTTKRP (default)")
    ap.add_argument("--concurrency", default="prop", choices=["off", "prop"],
                    help="off: layers run one after the other on every SM; prop: every layer gets a share of the SMs "
                         "proportional to its cost and all layers run concurrently on their own streams")
    ap.add_argument("--min-ctas", type=int, default=2,
                    help="--full, and the first warm-up step of --balance model / prop: SMs at least per unit")
    ap.add_argument("--balance", default="cost", choices=["cost", "model", "prop"],
                    help="SM budgets of the concurrent units: 'cost' (default) = proportional to the cost model and fixed, "
                         "so that runs with the same arguments compute the same numbers; re-balanced during warm-up from "
                         "measured times: 'model' = wave model of the tensor-core product fitted to the reported phase "
                         "times (source/workloads.py), 'prop' = proportional to time x CTAs.  The loop kernel a factor runs "
                         "on depends on its budget, so with measured budgets the results differ from run to run in the "
                         "last bits, which the solver amplifies")
    ap.add_argument("--budgets", default=None,
                    help="experiment knob: comma-separated SM budgets, one per layer in workload order; fixes the budgets "
                         "(no re-balancing during warm-up; single GPU)")
    ap.add_argument("--trace-layer", default=None, help="print the per-kernel-group times of this layer's last sweep")
    ap.add_argument("--placement", action="store_true",
                    help="report the SMs (%%smid) the last loop launch of every unit ran on (diagnostics of die / GPC locality)")
    ap.add_argument("--reserve-sms", type=int, default=0,
                    help="SMs kept out of the cooperative-grid budgets so that the ordinary kernels between the loops "
                         "(Gram, MTTKRP, projection, errors) never wait for a persistent kernel to finish")
    ap.add_argument("--solve-precision", type=int, default=1,
                    help="ridge product inside the ADMM loop: 0 = parity mode (float64 product with the float64 inverse), "
                         "1 = 3xTF32 on tcgen05 (default), 2 = float32 FFMA")
    ap.add_argument("--seed-replicas", action="store_true",
                    help="round 1's weak-scaling mode: every rank factorizes the whole unit set for its own seed")
    ap.add_argument("--round-size", type=int, default=32, help="sweep256: units that run concurrently on one GPU (measured on one B200: 8 -> 6.27 s, 16 -> 4.92 s, 32 -> 4.50 s per sweep of all 256 units)")
    ap.add_argument("--full", action="store_true",
                    help="run every unit to the reference's stop rule (scripts/factorize.py:259-263) and report the "
                         "factorize time (init + ADMM) instead of the per-sweep throughput")
    ap.add_argument("--init", default="random", choices=["random", "parafac-epc"], help="--full: factor initialisation")
    ap.add_argument("--max-iter-als", type=int, default=1000, help="--full: sweep budget per unit")
    ap.add_argument("--dump-outputs", default=None, metavar="DIR",
                    help="after the timed steps, write what the last step computed for every unit (factors, quantized "
                         "factors, the two reconstruction errors) as DIR/<unit>.<array>.npy, so that two builds can be "
                         f"compared output for output; above {DUMP_LIMIT_BYTES // 10**6} MB in all, every large array is "
                         "replaced by the same seeded sample of its elements")
    return ap.parse_args()


# ------------------------------------------------------------------------------------------ workloads
def workload_units(args):
    """[(key, name, cout, cin, kh, kw, reduction_rate, bits)] and a description.  Pure Python (no native library)."""
    from source import workloads as wl
    name = args.workload
    if name == "sweep256":
        units = [(f"{l[0]}/rr{rr}/b{b}", *l, rr, b) for rr in SWEEP_RATES for b in SWEEP_BITS for l in wl.resnet18_conv_layers()]
        return units, ("ResNet-18 sweep: 16 3x3 conv layers x reduction-rate {1.5,2,3,4} x bits {3,4,6,8} = 256 independent "
                       "solves (admmq_factorize_batch)")
    if name == "resnet18":
        layers, desc = wl.resnet18_conv_layers(), "ResNet-18 all 16 3x3 conv layers"
    elif name == "layer1":
        layers, desc = wl.resnet18_conv_layers()[:1], "ResNet-18 layer1.0.conv1 (64x64x3x3)"
    elif name == "resnet50-l4":
        layers, desc = wl.resnet50_layer4_layers(), "ResNet-50-shaped layer4 (512x512x3x3, 2048x512 1x1)"
    else:
        layers, desc = wl.llama7b_linear_layers(), "Llama-7B-shaped linear (4096x4096, 11008x4096)"
    return [(l[0], *l, args.reduction_rate, args.bits) for l in layers], desc


def unit_shape(u):
    _, _, cout, cin, kh, kw, _, _ = u
    return (cout, cin, kh * kw) if kh * kw > 1 else (cout, cin)


def unit_rank(u):
    from source.shapes import rank_for_shape
    return rank_for_shape(unit_shape(u), u[6])


def config_dict(args, desc, extra=None):
    if args.workload == "sweep256":
        what = f"{desc}, {QSCHEME}"
    else:
        what = f"{desc}, ADMM {args.bits}-bit {QSCHEME}, reduction-rate {args.reduction_rate}"
    cfg = {"workload": f"{what}, init=random, max_iter_admm={args.max_iter_admm}; one step = one outer sweep over every unit",
           "bits": args.bits, "qscheme": QSCHEME, "reduction_rate": args.reduction_rate,
           "max_iter_admm": args.max_iter_admm, "num_attempts": 200,
           "solve_precision": args.solve_precision, "mttkrp_precision": args.mttkrp_precision,
           "ridge_product": {0: "float64 product with the float64 inverse (parity mode)", 1: "3xTF32 tcgen05",
                             2: "float32 FFMA"}[args.solve_precision]}
    if extra:
        cfg.update(extra)
    return cfg


# ------------------------------------------------------------------------------------------ clocks
class ClockSampler:
    """nvidia-smi sampled every 200 ms during the timed region (B200_PROFILING.md clocks line)."""
    FIELDS = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,"
              "clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
              "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index):
        self.rows, self.proc, self.gpu = [], None, gpu_index

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.gpu), f"--query-gpu={self.FIELDS}",
                                          "--format=csv,noheader,nounits", "-lms", "200"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            threading.Thread(target=self._read, daemon=True).start()
        except OSError:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append([c.strip() for c in line.split(",")])

    def stop(self):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        try:
            self.proc.wait(timeout=5)
        except subprocess.TimeoutExpired:
            self.proc.kill()
        sm = sorted(float(r[1]) for r in self.rows if len(r) >= 9 and r[1].replace(".", "").isdigit())
        mx = [float(r[2]) for r in self.rows if len(r) >= 9 and r[2].replace(".", "").isdigit()]
        pw = [float(r[3]) for r in self.rows if len(r) >= 9 and r[3].replace(".", "").isdigit()]
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        reasons = [n for k, n in enumerate(names) if any(len(r) >= 9 and r[5 + k].lower() == "active" for r in self.rows)]
        return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "power_w_max": max(pw) if pw else None, "samples": len(sm), "reasons": reasons}


# ------------------------------------------------------------------------------------------ reference arm
def load_reference():
    """(admm_iteration callable with the reference's signature, kind).  kind "reference": the UNMODIFIED reference
    functions (from /root/reference in the dev container, else the byte-compiled build product oracle/_ref made by
    oracle/build_ref.py); kind "port": the oracle's restatement when neither exists."""
    try:
        from oracle.ref_import import import_reference, reference_available
        if reference_available():
            ref = import_reference()
            return ref.admm_iteration, "reference"
    except Exception as e:  # noqa: BLE001 - fall back to the pinned restatement, and say so in `kind`
        sys.stderr.write(f"[bench] reference import failed ({e}); timing the oracle port instead\n")
    from oracle import admm_oracle as orc

    def port(H, U, F, G, max_iter, eps, bits, qscheme):
        h, u, _ = orc.admm_iteration(H, U, F, G, max_iter, eps, bits, qscheme)
        return h, u
    return port, "port"


def reference_sample(args, units, budget_s, device="cpu", thread_cache=None):
    """Times the reference's `admm_iteration` (source/admm.py:51-67 incl. the Cholesky set-up and the 200-candidate
    projection of source/quantization.py:118-144) on every distinct factor shape of the workload for a few inner
    iterations and converts to the workload's inner-iterations/s.  On the CPU the thread count is chosen PER SHAPE
    (best of {1, 4, nproc/2, nproc}: small shapes get slower with threads).  Returns a dict."""
    import torch
    admm_iteration, kind = load_reference()
    if device != "cpu" and kind != "reference":
        raise RuntimeError("the eager-on-GPU bar needs the reference's own functions (oracle/_ref is missing)")
    nproc = os.cpu_count() or 1
    shapes = {}
    for u in units:
        dims, rank, bits = unit_shape(u), unit_rank(u), u[7]
        for m, d in enumerate(dims):
            others = [x for k, x in enumerate(dims) if k != m]
            shapes.setdefault((d, rank, bits), [0, others])[0] += 1
    g = torch.Generator().manual_seed(7)

    def one(I, R, bits, others, iters):
        mats = [torch.randn(o, R, generator=g).to(device) for o in others]
        G = mats[0].T @ mats[0]
        for M in mats[1:]:
            G = G * (M.T @ M)
        scale = 1.0
        for o in others:
            scale *= o
        F = (torch.randn(I, R, generator=g) * scale ** 0.5).to(device)
        H = torch.randn(I, R, generator=g).to(device)
        U = torch.zeros(I, R, device=device)
        if device != "cpu":
            torch.cuda.synchronize()
        t0 = time.perf_counter()
        admm_iteration(H, U, F, G, iters + 1, 1e-8, bits, QSCHEME)
        if device != "cpu":
            torch.cuda.synchronize()
        return (time.perf_counter() - t0) / iters

    thread_cache = {} if thread_cache is None else thread_cache
    t_start = time.perf_counter()
    total_s_per_sweep, sampled = 0.0, 0
    share = budget_s / len(shapes)          # equal time per distinct shape
    used_threads = set()
    for (I, R, bits), (count, others) in sorted(shapes.items()):
        if device == "cpu":
            if (I, R, bits) not in thread_cache:
                best = None
                for t in sorted({1, min(4, nproc), max(1, nproc // 2), nproc}):
                    torch.set_num_threads(t)
                    dt = min(one(I, R, bits, others, 1), one(I, R, bits, others, 1)) if I * R < 200000 else one(I, R, bits, others, 1)
                    if best is None or dt < best[1]:
                        best = (t, dt)
                thread_cache[(I, R, bits)] = best
            threads, probe = thread_cache[(I, R, bits)]
            torch.set_num_threads(threads)
            used_threads.add(threads)
        else:
            probe = one(I, R, bits, others, 1)
            probe = one(I, R, bits, others, 2)
        iters = int(min(60, max(2, round((share - 2 * probe) / probe))))
        per_iter = one(I, R, bits, others, iters)
        sampled += iters
        total_s_per_sweep += count * (args.max_iter_admm - 1) * per_iter
    if device == "cpu":
        torch.set_num_threads(1)
    inner_per_sweep = sum(c for c, _ in shapes.values()) * (args.max_iter_admm - 1)
    where = (f"torch-CPU float32, threads chosen per shape from {{1, 4, {max(1, nproc // 2)}, {nproc}}}, used {sorted(used_threads)}"
             if device == "cpu" else "eager PyTorch on the B200 (stock ATen / cuBLAS / cuSOLVER kernels, ~2000 launches and 3 host "
                                     "syncs per inner iteration)")
    what = "the reference's own source/admm.py::admm_iteration" if kind == "reference" else "oracle admm_iteration (port)"
    return {"value": inner_per_sweep / total_s_per_sweep, "kind": kind, "cores": max(used_threads) if used_threads else 0,
            "sample": (f"{what} ({where}): {sampled} timed inner iterations spread over the {len(shapes)} distinct factor "
                       f"shapes of the workload (Cholesky set-up included), extrapolated to one sweep = {inner_per_sweep} "
                       f"inner iterations; Gram/MTTKRP/error terms (<1 % of the time) not included"),
            "seconds": round(time.perf_counter() - t_start, 1), "threads_per_shape": {f"{k[0]}x{k[1]}@{k[2]}b": v[0] for k, v in thread_cache.items()}}


def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return 0
    units, desc = workload_units(args)
    vals, cache, res = [], {}, None
    t0 = time.perf_counter()
    per_step = 4.0 if args.workload != "sweep256" else 12.0
    for i in range(args.warmup + args.steps):
        res = reference_sample(args, units, per_step, "cpu", cache)
        if i >= args.warmup:
            vals.append(res["value"])
    value = len(vals) / sum(1.0 / v for v in vals)
    inner = sum(len(unit_shape(u)) for u in units) * (args.max_iter_admm - 1)
    line = {"impl": "reference", "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": args.gpus, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": inner / value * 1e3, "higher_is_better": True, "scaling": "strong",
            "vs_baseline": None, "dtype": "f32", "data": "synthetic", "config": config_dict(args, desc),
            "cpu_baseline": {"value": value, "unit": UNIT, "cores": res["cores"], "kind": res["kind"], "sample": res["sample"],
                             "host_cores": os.cpu_count(), "threads_per_shape": res["threads_per_shape"]},
            "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
            "gpu_launches": 0, "wall_s": time.perf_counter() - t0,
            "note": "ms_per_step is the extrapolated CPU time of one full sweep; each timed step ran a bounded sample"}
    print(json.dumps(line), flush=True)
    return 0


def mttkrp_roofline(problems, dev, peaks):
    """GPU time of the tensor-core MTTKRP (scripts/factorize.py:217,227,237) on the workload's largest 3-D unit, per mode:
    20 calls captured into one CUDA graph (no host launch gaps, transpose / split kernel included), replayed three times
    and timed with CUDA events on the capturing stream; against the 3xTF32 roof from MEASURED_PEAKS.json."""
    import torch
    from source import _native as nat
    cands = [p for p in problems if p[1].ndim == 3]
    if not cands:
        return None
    name, W, rank, init = max(cands, key=lambda p: p[1].numel())[:4]
    W = W.to(dev)
    I, J, K = W.shape
    fac = [f.to(dev) for f in init]
    unf = [W.reshape(I, J * K), nat.unfold3(W, 1), nat.unfold3(W, 2)]
    dims = [I, J, K]
    flop = 2.0 * I * J * K * rank
    us = []
    for mode in range(3):
        o = [k for k in range(3) if k != mode]
        X, Y = fac[o[0]], fac[o[1]]
        V = nat.permute_myx(unf[mode], X.shape[0], Y.shape[0])
        ws = torch.empty(nat.mttkrp_tc_workspace_bytes(dims[mode], X.shape[0], Y.shape[0], rank), dtype=torch.uint8, device=dev)
        F = torch.empty(dims[mode], rank, device=dev)
        fn = lambda: nat.mttkrp_tc(V, dims[mode], X, Y, out=F, ws=ws)
        fn()
        torch.cuda.synchronize()
        st = torch.cuda.Stream(device=dev)
        with torch.cuda.stream(st):
            fn()
            graph = torch.cuda.CUDAGraph()
            with torch.cuda.graph(graph, stream=st):
                for _ in range(20):
                    fn()
            graph.replay()
            st.synchronize()
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record(st)
            for _ in range(3):
                graph.replay()
            e1.record(st)
            st.synchronize()
        us.append(e0.elapsed_time(e1) / 60.0 * 1e3)
    sustained = float(peaks.get("bf16_tflops_sustained", 2250.0 * 0.62)) / 6.0
    burst = float(peaks.get("bf16_tflops", 2250.0 * 0.74)) / 6.0
    tf = [flop / (u * 1e-6) / 1e12 for u in us]
    return {"kernel": "k_mttkrp_fold_tc / k_mttkrp_foldlong_tc (+ transpose / split)", "unit_name": name, "shape": [I, J, K], "rank": rank,
            "bound": "tensor", "us_per_mode": [round(u, 2) for u in us], "achieved": [round(t, 1) for t in tf], "unit": "TFLOP/s",
            "peak": sustained, "frac": [round(t / sustained, 3) for t in tf], "peak_burst": burst,
            "frac_of_burst": [round(t / burst, 3) for t in tf],
            "how": "fp32-equivalent flop 2 I J K R per mode (the hardware executes 3x that in TF32) / GPU time per call in a CUDA "
                   "graph of 20 calls (timed alone, after the sweeps); peak = MEASURED_PEAKS.json bf16 / 2 / 3"}


def allocate_ctas(costs, sm_count, min_ctas):
    """Share of the SMs for every independent solve, proportional to its estimated cost (largest-remainder rounding,
    at least `min_ctas` each, sum == sm_count when there are enough SMs)."""
    n = len(costs)
    total = float(sum(costs))
    if n * min_ctas >= sm_count:
        return [max(1, sm_count // n)] * n
    spare = sm_count - n * min_ctas
    raw = [c / total * spare for c in costs]
    out = [min_ctas + int(r) for r in raw]
    rest = sm_count - sum(out)
    for i in sorted(range(n), key=lambda k: raw[k] - int(raw[k]), reverse=True)[:rest]:
        out[i] += 1
    return out


def dump_outputs(out_dir, units, world):
    """Write what the last timed step computed for every unit of this rank - factors, quantized factors and the two
    reconstruction errors - as out_dir/<unit>.<array>.npy (float32; the errors float64).  The ranks of a job share
    DUMP_LIMIT_BYTES.  When a rank's arrays need more, every array of more than DUMP_WHOLE_ELEMENTS elements is replaced
    by the same fraction of its elements, at positions drawn with a fixed seed, so that runs with the same arguments
    sample the same positions.  units: [(key, factors, factors_q, rec_error, quant_rec_error)]."""
    import numpy as np
    arrays = {}
    for key, factors, factors_q, err, errq in units:
        name = key.replace("/", "_")
        arrays[f"{name}.rec_error"] = np.array([err, errq], dtype=np.float64)
        for m, (f, q) in enumerate(zip(factors, factors_q)):
            arrays[f"{name}.factor{m}"] = f.float().cpu().numpy()
            arrays[f"{name}.factor{m}_quantized"] = q.float().cpu().numpy()
    room = DUMP_LIMIT_BYTES // world - 256 * len(arrays)     # 256 B per file covers the .npy header
    whole = sum(a.nbytes for a in arrays.values() if a.size <= DUMP_WHOLE_ELEMENTS)
    big = sum(a.nbytes for a in arrays.values()) - whole
    keep = min(1.0, max(room - whole, 0) / big) if big else 1.0
    os.makedirs(out_dir, exist_ok=True)
    for name, a in arrays.items():
        if keep < 1.0 and a.size > DUMP_WHOLE_ELEMENTS:
            pos = np.random.default_rng(0).choice(a.size, int(a.size * keep), replace=False)
            a = a.reshape(-1)[np.sort(pos)]
        np.save(os.path.join(out_dir, name + ".npy"), a)


# ------------------------------------------------------------------------------------------ native arm
class Rank:
    """Process-group plumbing of one rank."""

    def __init__(self):
        import torch
        import torch.distributed as dist
        self.torch, self.dist = torch, dist
        self.rank = int(os.environ.get("RANK", "0"))
        self.world = int(os.environ.get("WORLD_SIZE", "1"))
        self.local = int(os.environ.get("LOCAL_RANK", "0"))
        torch.cuda.set_device(self.local)
        self.dev = torch.device("cuda", self.local)
        if self.world > 1:
            dist.init_process_group("nccl", device_id=self.dev)
            # bring the communicator up before anything is timed (lazy connection set-up cost 0.2 - 1.3 s in round 1)
            warm = torch.zeros(8, device=self.dev)
            dist.all_reduce(warm)
            out = torch.empty(8 * self.world, device=self.dev)
            dist.all_gather_into_tensor(out, warm)
            torch.cuda.synchronize()

    def barrier(self):
        if self.world > 1:
            self.dist.barrier()
        self.torch.cuda.synchronize()

    def reduce(self, value, op):
        t = self.torch.tensor([float(value)], dtype=self.torch.float64, device=self.dev)
        if self.world > 1:
            self.dist.all_reduce(t, op=getattr(self.dist.ReduceOp, op))
        return float(t.item())

    def gather_objects(self, obj):
        if self.world == 1:
            return [obj]
        out = [None] * self.world
        self.dist.all_gather_object(out, obj)
        return out

    def gather_factors(self, tensors):
        """The job's only collective: ONE all_gather of the packed factors (padded to the largest rank's payload),
        timed on the device.  Returns (ms, bytes of this rank's payload)."""
        torch, dist = self.torch, self.dist
        if self.world == 1:
            return None, 0
        flat = torch.cat([t.reshape(-1) for t in tensors]) if tensors else torch.zeros(1, device=self.dev)
        width = int(self.reduce(flat.numel(), "MAX"))
        padded = torch.zeros(width, dtype=torch.float32, device=self.dev)
        padded[:flat.numel()] = flat
        out = torch.empty(width * self.world, dtype=torch.float32, device=self.dev)
        torch.cuda.synchronize()
        dist.barrier()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        dist.all_gather_into_tensor(out, padded)
        e1.record()
        torch.cuda.synchronize()
        return self.reduce(e0.elapsed_time(e1), "MAX"), flat.numel() * 4


def shard(args, units, rk):
    """Owner rank of every unit: LPT over the cost model (source/distributed.py); seed replicas: everything everywhere."""
    if args.seed_replicas or rk.world == 1:
        return [rk.rank] * len(units)
    from source.distributed import shard_units
    return shard_units([{"shape": unit_shape(u), "rank": unit_rank(u), "bits": u[7]} for u in units], rk.world)


def run_native(args):
    import torch
    from source import _native, workloads as wl
    from source.solver import LayerSolver
    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device - the solver has no CPU path (use --impl reference for the CPU arm)")
    rk = Rank()
    rank, world, dev = rk.rank, rk.world, rk.dev
    units, desc = workload_units(args)
    owner = shard(args, units, rk)
    mine = [u for u, o in zip(units, owner) if o == rank]
    init_seed = 42 + (rank if args.seed_replicas else 0)
    sm_count = torch.cuda.get_device_properties(dev).multi_processor_count
    if args.workload == "sweep256":
        return run_sweep256(args, rk, units, owner, mine, desc, sm_count)
    if args.full:
        return run_full(args, rk, units, owner, mine, desc, sm_count)

    problems = []
    for key, name, cout, cin, kh, kw, rr, bits in mine:
        W = wl.layer_weight_as_tensor(wl.synthetic_weight(cout, cin, kh, kw, 42, name)).contiguous()
        rnk = wl.rank_from_reduction_rate(W, rr)
        problems.append((key, W, rnk, wl.random_init(W.shape, rnk, init_seed), bits))
    host, solvers = [], []   # pinned host state for the end-to-end leg
    concurrent = args.concurrency == "prop" and len(problems) > 0
    # fixed budgets give the small units one SM each, where the re-balancing from measured times always ends
    budgets = allocate_ctas([wl.solve_cost(W.shape, rnk) for _, W, rnk, _, _ in problems], sm_count - args.reserve_sms,
                            1 if args.balance == "cost" else args.min_ctas) if concurrent else [0] * len(problems)
    if args.budgets and concurrent and world == 1:
        budgets = [int(x) for x in args.budgets.split(",")]
        assert len(budgets) == len(problems) and sum(budgets) <= sm_count, (len(problems), sum(budgets), sm_count)
    streams = [torch.cuda.Stream(device=dev) for _ in problems] if concurrent else None
    rep_bytes = _native.new_report(dev).numel()
    for (key, W, rnk, init, bits), g in zip(problems, budgets):
        solvers.append(LayerSolver(W.to(dev), [f.to(dev) for f in init], bits, QSCHEME,
                                   max_iter_admm=args.max_iter_admm, mttkrp_precision=args.mttkrp_precision,
                                   solve_precision=args.solve_precision, time_loops=True, max_ctas=g))
        host.append({"W": W.pin_memory(), "factors": [f.clone().pin_memory() for f in init],
                     "duals": [torch.zeros_like(f).pin_memory() for f in init],
                     "factors_q": [torch.zeros_like(f).pin_memory() for f in init],
                     "err": torch.zeros(2, 2, dtype=torch.float64).pin_memory(),
                     "reports": torch.zeros(W.ndim * rep_bytes, dtype=torch.uint8).pin_memory()})
    for (key, _, _, _, _), s in zip(problems, solvers):
        if args.trace_layer and key == args.trace_layer:
            s.part_events = []
    inner_per_step = sum(s.inner_iterations_per_sweep() for s in solvers)
    flush = torch.empty(256 << 20, dtype=torch.uint8, device=dev)   # > 126 MB L2
    sweep_events = []

    def enqueue_all(prepare=None):
        """One sweep of every local unit.  Concurrent mode: every unit on its own stream (fork from / join into the
        current stream with events, so CUDA events recorded on the current stream bracket all of the work)."""
        if streams is None:
            for k, s in enumerate(solvers):
                if prepare is not None:
                    prepare(k)
                s.enqueue_sweep()
            return
        main = torch.cuda.current_stream()
        fork = torch.cuda.Event(enable_timing=True)
        fork.record(main)
        sweep_events.clear()
        for k, (s, st) in enumerate(zip(solvers, streams)):
            st.wait_event(fork)
            with torch.cuda.stream(st):
                if prepare is not None:
                    prepare(k)
                s.enqueue_sweep()
                join = torch.cuda.Event(enable_timing=True)
                join.record(st)
            main.wait_event(join)
            sweep_events.append((fork, join))

    def step():
        enqueue_all()
        return [s.collect() for s in solvers]

    def step_e2e():
        """The same sweep through the public solver API starting from HOST buffers: weights, factors and duals go
        host->device (pinned), results (factors, duals, re-projected factors, error sums, loop reports) come back."""
        moved = [0, 0]

        def h2d_copy(k):
            moved[0] += solvers[k].load_from_host(host[k]["W"], host[k]["factors"], host[k]["duals"])

        enqueue_all(prepare=h2d_copy)
        for s, h in zip(solvers, host):   # results come back on the (joined) current stream
            moved[1] += s.store_to_host(h["factors"], h["duals"], h["factors_q"], h["err"], h["reports"])
        torch.cuda.synchronize()
        for s, h in zip(solvers, host):   # a non-PD ridge system raises here like the reference's cholesky
            s.check_host_reports(h["reports"])
        return moved[0], moved[1]

    tried = []   # (step ms, budgets) of every warm-up step: the timed steps run with the best MEASURED budgets
    if streams is not None:
        step()   # one-time costs (module load, kernel attributes, allocator) stay out of the comparison below
    for w in range(args.warmup):
        flush.fill_(1)
        w0, w1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        w0.record()
        step()
        w1.record()
        torch.cuda.synchronize()
        tried.append((w0.elapsed_time(w1), [s.max_ctas for s in solvers]))
        if streams is not None and w < args.warmup - 1 and args.balance != "cost" and not args.budgets and len(solvers) > 1:
            # re-balance the SM budgets from what was just measured: per unit the sweep time and, per factor, the
            # phase times its persistent kernel reported, through the wave model of source/workloads.py
            fitted = []
            for (a, b), s in zip(sweep_events, solvers):
                modes = []
                for f, r in zip(s.factors, s.last_reports):
                    it = max(r.iterations, 1)
                    modes.append((f.shape[0], s.R, r.phase_ns[0] / 1e3 / it, (r.phase_ns[1] + r.phase_ns[2]) / 1e3 / it, it))
                fitted.append((a.elapsed_time(b), max(s.max_ctas, 1), modes))
            new = wl.allocate_ctas_modelled(fitted, sm_count - args.reserve_sms, args.solve_precision) \
                if args.balance == "model" else \
                allocate_ctas([m * g0 for m, g0, _ in fitted], sm_count - args.reserve_sms, 1)
            for s, g in zip(solvers, new):
                s.max_ctas = g
    if streams is not None and len(tried) > 1:
        best_ms, best = min((ms, b) for ms, b in tried)
        for s, g in zip(solvers, best):
            s.max_ctas = g
    budgets[:] = [s.max_ctas for s in solvers]
    for s in solvers:
        s.loop_events.clear()
    sampler = ClockSampler(rk.local)
    if rank == 0:
        sampler.start()
    launches0 = _native.launch_count()
    step_ms = []
    # inner iterations actually executed in the timed steps, per unit and factor, from the kernels' device reports (the
    # loop leaves early where the reference's own exit test fires, source/admm.py:64-65) - the metric counts these
    done = [[0] * s.N for s in solvers]
    early, nonfinite = [], 0
    errs = []
    rk.barrier()
    for stp in range(args.steps):
        flush.fill_(1)                      # L2 flush between timed steps (outside the event pair)
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        errs = step()
        e1.record()
        torch.cuda.synchronize()
        step_ms.append(e0.elapsed_time(e1))
        for k, sv in enumerate(solvers):
            for m, r in enumerate(sv.last_reports):
                done[k][m] += int(r.iterations)
                if int(r.iterations) < sv.max_iter_admm - 1:
                    early.append({"unit": problems[k][0], "mode": m, "step": stp, "sweep": len(sv.loss_hist) - 1,
                                  "iterations": int(r.iterations), "r": float(r.r), "s": float(r.s), "rows": sv.factors[m].shape[0]})
                nonfinite += bool(int(r.status) & _native.ST_NONFINITE)
    rk.barrier()
    done_total = sum(sum(d) for d in done)
    launches = _native.launch_count() - launches0
    clocks = sampler.stop() if rank == 0 else None
    total_ms = rk.reduce(sum(step_ms), "MAX")
    done_all = rk.reduce(done_total, "SUM")
    value = done_all / (total_ms / 1e3)
    if args.dump_outputs and (rank == 0 or not args.seed_replicas):   # seed replicas: every rank has the same units
        dump_outputs(args.dump_outputs, [(p[0], s.factors, s.factors_q, *e) for p, s, e in zip(problems, solvers, errs)],
                     1 if args.seed_replicas else world)

    # ---- the dominant kernel (persistent ADMM loop), timed with CUDA events on its own stream.  In concurrent mode a
    # launch holds only its share g of the SMs, so its duration is weighted by g / SMs: the sum is the time the whole
    # GPU would have been busy with these launches (equals the plain sum when every launch uses every SM).
    loop_ms, loop_gpu_ms, per_layer, sweep_ms = 0.0, 0.0, {}, {}
    for k, ((key, _, _, _, _), s) in enumerate(zip(problems, solvers)):
        ms = sum(a.elapsed_time(b) for _, a, b in s.loop_events)
        loop_ms += ms
        loop_gpu_ms += ms * ((s.max_ctas or sm_count) / sm_count)
        per_layer[key] = round(sum(done[k]) / (ms / 1e3), 1) if ms > 0 else None
    for (key, _, _, _, _), ev in zip(problems, sweep_events):
        sweep_ms[key] = round(ev[0].elapsed_time(ev[1]), 1)
    n_loop = sum(len(s.loop_events) for s in solvers)
    # algorithmic work of the iterations that ran (DESIGN.md section 5)
    alg_bytes = sum(it * (16 * f.shape[0] * s.R + 4 * s.R * s.R) for s, d in zip(solvers, done) for f, it in zip(s.factors, d))
    evals = sum(it * (s.num_attempts if s.qscheme == QSCHEME else 0) * f.shape[0] * s.R
                for s, d in zip(solvers, done) for f, it in zip(s.factors, d))
    flops = sum(it * 2 * f.shape[0] * s.R * s.R for s, d in zip(solvers, done) for f, it in zip(s.factors, d))
    peaks = {}
    try:
        peaks = json.load(open(os.path.join(REPO, "MEASURED_PEAKS.json")))
    except OSError:
        pass
    traffic = None
    try:
        traffic = json.load(open(os.path.join(REPO, "profiles", "roofline_traffic.json")))
    except OSError:
        pass
    hbm_peak = float(peaks.get("hbm_gbs", 6650.0))
    # The kernel's dominant phase is the ridge product H_ls = RHS . Minv (2 I R^2 flop per inner iteration, float32
    # accuracy through three TF32 tensor-core products per term), so it is reported against the tensor roofline:
    # dense TF32 = bf16 / 2, 3xTF32 = TF32 / 3, from the MEASURED sustained bf16 rate (the kernel runs inside a long step).
    bf16 = float(peaks.get("bf16_tflops_sustained", peaks.get("bf16_tflops", 2250.0 * 0.62)))
    tensor_peak = bf16 / 2.0 / 3.0
    roofline = None
    if loop_gpu_ms > 0:
        achieved = flops / (loop_gpu_ms / 1e3) / 1e12
        hbm_achieved = alg_bytes / (loop_gpu_ms / 1e3) / 1e9
        roofline = {"kernel": "k_admm_loop (persistent ADMM inner loop: ridge product on tcgen05 + clip search + dual update)",
                    "bound": "tensor", "achieved": achieved, "peak": tensor_peak, "unit": "TFLOP/s", "frac": achieved / tensor_peak,
                    "peak_source": ("MEASURED_PEAKS.json bf16_tflops_sustained / 2 (tf32) / 3 (3xTF32 split), fp32-equivalent" if peaks
                                    else "fallback: 0.62 x 2250 bf16 TFLOP/s / 6"),
                    "traffic": (traffic or {}).get("bytes") if isinstance(traffic, dict) else traffic,
                    "traffic_note": (traffic or {}).get("note") if isinstance(traffic, dict) else None,
                    "launches": n_loop, "avg_launch_ms": loop_ms / max(n_loop, 1),
                    "gpu_share_weighted_ms": loop_gpu_ms, "share_of_step": loop_gpu_ms / sum(step_ms),
                    "algorithmic_flops_per_launch": flops / max(n_loop, 1),
                    "algorithmic_bytes_per_launch": alg_bytes / max(n_loop, 1),
                    "rank": 0,
                    "note": "rank 0's launches; achieved = 2 I R^2 flop per inner iteration (fp32-equivalent; the hardware "
                            "executes 3x that in TF32) / (launch duration x the launch's share of the SMs); the launch also "
                            "contains the clip search, the dual update and three device-wide barriers per iteration, so frac "
                            "is a lower bound for the product itself (tools/microbench/tcprof.cu times the product alone)",
                    "hbm": {"achieved_gbs": hbm_achieved, "peak_gbs": hbm_peak, "frac": hbm_achieved / hbm_peak,
                            "note": "state is L2-resident by design (ncu: see traffic), HBM is not the binding resource"},
                    "clip_search": {"candidates_x_elements_per_s": evals / (loop_gpu_ms / 1e3),
                                    "note": "threshold form: O(1) work per element + (2^bits - 1) x candidates thresholds per CTA"}}

    if roofline is not None and world == 1 and args.mttkrp_precision == 1:
        try:
            roofline["mttkrp"] = mttkrp_roofline(problems, dev, peaks)
        except Exception as e:  # noqa: BLE001 - a side measurement must not take the bench line down
            roofline["mttkrp"] = {"error": str(e)[:200]}

    # ---- end to end through the public API with host buffers
    e2e = None
    if not args.no_e2e:
        step_e2e()
        rk.barrier()
        t_e2e = []
        h2d = d2h = 0
        done_e2e = 0
        for _ in range(args.steps):
            flush.fill_(1)
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            h2d, d2h = step_e2e()
            e1.record()
            torch.cuda.synchronize()
            t_e2e.append(e0.elapsed_time(e1))
            done_e2e += sum(int(r.iterations) for sv in solvers for r in sv.last_reports)
        rk.barrier()
        tot = rk.reduce(sum(t_e2e), "MAX")
        cnt = rk.reduce(done_e2e, "SUM")
        e2e = {"value": cnt / (tot / 1e3), "unit": UNIT, "h2d_bytes_per_step": int(rk.reduce(h2d, "SUM")),
               "d2h_bytes_per_step": int(rk.reduce(d2h, "SUM")), "ms_per_step": tot / args.steps}

    if args.placement:
        torch.cuda.synchronize()
        import numpy as np
        for (key, *_), sv in zip(problems, solvers):
            ms = sweep_ms.get(key, float("nan"))
            words = sv.ws_loop[64:96].cpu().numpy().view(np.uint32)
            smids = [32 * w + b for w in range(8) for b in range(32) if (int(words[w]) >> b) & 1]
            print(f"[placement] {key:16s} {ms:7.1f} ms  {len(smids):3d} SMs: {smids}", file=sys.stderr, flush=True)

    # ---- the job's only collective: final factor gather over NCCL (once per job, outside the timed region)
    gather_ms, gather_bytes = rk.gather_factors([f for s in solvers for f in s.factors])
    per_rank = rk.gather_objects({"rank": rank, "units": [p[0] for p in problems], "ctas": dict(zip([p[0] for p in problems], budgets)),
                                  "ms_per_step": sum(step_ms) / args.steps, "inner_iterations": done_total / args.steps,
                                  "sweep_ms": sweep_ms, "per_unit_inner_iter_per_s": per_layer, "early": early,
                                  "nonfinite": nonfinite, "launches": launches, "gather_bytes": gather_bytes,
                                  "rec_error": {p[0]: round(e[0], 6) for p, e in zip(problems, errs)}})
    # ---- the same sweep in the PARITY mode (precision 0: float64 ridge product against the float64 inverse, float64-
    # accumulating MTTKRP) - the mode the bit-level claims are made in; one warm-up + one timed step, same SM budgets
    parity = None
    if world == 1 and args.solve_precision != 0 and not args.no_parity_leg and streams is not None:
        psolvers = [LayerSolver(W.to(dev), [f.to(dev) for f in init], bits, QSCHEME, max_iter_admm=args.max_iter_admm,
                                mttkrp_precision=0, solve_precision=0, max_ctas=g)
                    for (key, W, rnk, init, bits), g in zip(problems, budgets)]
        times = []
        for _ in range(2):
            flush.fill_(1)
            main = torch.cuda.current_stream()
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record(main)
            joins = []
            for s, st in zip(psolvers, streams):   # fork every stream from e0, join them all afterwards
                st.wait_event(e0)
                with torch.cuda.stream(st):
                    s.enqueue_sweep()
                    j = torch.cuda.Event()
                    j.record(st)
                joins.append(j)
            for j in joins:
                main.wait_event(j)
            e1.record(main)
            for s in psolvers:
                s.collect()
            torch.cuda.synchronize()
            times.append(e0.elapsed_time(e1))
        pdone = sum(int(r.iterations) for s in psolvers for r in s.last_reports)
        parity = {"solve_precision": 0, "mttkrp_precision": 0, "ms_per_step": times[-1], "value": pdone / (times[-1] / 1e3),
                  "unit": UNIT, "steps": 1, "warmup": 1,
                  "note": "same workload and SM budgets in the parity mode (second sweep of a fresh run)"}
        del psolvers
    cpu = eager = None
    if rank == 0 and world == 1 and not args.no_cpu_baseline:
        r = reference_sample(args, units, args.cpu_budget_s, "cpu")
        cpu = {"value": r["value"], "unit": UNIT, "cores": r["cores"], "kind": r["kind"], "sample": r["sample"],
               "host_cores": os.cpu_count(), "seconds": r["seconds"], "threads_per_shape": r["threads_per_shape"]}
    if rank == 0 and world == 1 and not args.no_eager_reference:
        try:
            r = reference_sample(args, units, 6.0, "cuda")
            eager = {"value": r["value"], "unit": UNIT, "kind": r["kind"], "sample": r["sample"], "seconds": r["seconds"]}
        except Exception as e:  # noqa: BLE001 - informative bar only
            eager = {"unavailable": str(e)[:200]}
    if rank == 0 and args.trace_layer:
        for (key, _, _, _, _), s in zip(problems, solvers):
            if s.part_events:
                sys.stderr.write(f"[trace {key}] " + ", ".join(f"{k} {v:.1f}" for k, v in s.part_times_ms()) + "\n")
    if rank == 0:
        all_early = [e for pr in per_rank for e in pr["early"]]
        n_loops = args.steps * sum(len(unit_shape(u)) for u in units) * (world if args.seed_replicas else 1)
        par = (f"{world} independent seeds, one per GPU" if args.seed_replicas else
               f"one job, {len(units)} units sharded over {world} GPU(s) by LPT on the cost model") + "; no data-path collective"
        line = {"metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps,
                "warmup": args.warmup, "ms_per_step": total_ms / args.steps, "higher_is_better": True,
                "scaling": "weak" if args.seed_replicas else "strong", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
                "config": config_dict(args, desc, {"l2": "flushed between timed steps (256 MiB write)",
                                                   "concurrency": args.concurrency, "balance": args.balance,
                                                   "units_per_rank": [len(pr["units"]) for pr in per_rank],
                                                   "ctas_per_unit": {k: v for pr in per_rank for k, v in pr["ctas"].items()},
                                                   "parallelism": par,
                                                   "inner_iterations_per_step": done_all / args.steps,
                                                   "inner_iterations_nominal_per_step": inner_per_step if world == 1 else
                                                   sum(len(unit_shape(u)) for u in units) * (args.max_iter_admm - 1) * (world if args.seed_replicas else 1),
                                                   "loops_left_early": f"{len(all_early)} of {n_loops} (exit test r < eps and s < eps, "
                                                                       "eps = 1e-8: source/admm.py:62-65; the unmodified reference "
                                                                       "leaves at the same iteration from the same state, "
                                                                       "tests/golden/early_exit.npz)",
                                                   "loops_nonfinite": sum(pr["nonfinite"] for pr in per_rank)}),
                "clocks": clocks, "e2e": e2e, "gpu_launches": sum(pr["launches"] for pr in per_rank), "roofline": roofline,
                "cpu_baseline": cpu, "reference_eager_b200": eager, "parity_mode": parity,
                "per_unit_inner_iter_per_s": {k: v for pr in per_rank for k, v in pr["per_unit_inner_iter_per_s"].items()},
                "per_unit_sweep_ms_last_step": {k: v for pr in per_rank for k, v in pr["sweep_ms"].items()},
                "per_rank_ms_per_step": [round(pr["ms_per_step"], 2) for pr in per_rank],
                "rec_error_last_step": {k: v for pr in per_rank for k, v in pr["rec_error"].items()},
                "early_exits": all_early[:64],
                "factor_gather_ms": gather_ms, "factor_gather_bytes_per_rank": [pr["gather_bytes"] for pr in per_rank]}
        print(json.dumps(line), flush=True)
    if world > 1:
        rk.dist.destroy_process_group()
    return 0


# ------------------------------------------------------------------------------------------ config 3: 256 units
def run_sweep256(args, rk, units, owner, mine, desc, sm_count):
    """BASELINE configs[2]: layer x reduction-rate x bits as independent solves through admmq_factorize_batch.  A rank's
    units run in ROUNDS of --round-size units of similar cost (LPT order), every unit of a round on its own stream with
    an SM budget proportional to its cost; one step = one outer sweep of every unit (one batch call per round with
    max_iter_als = 1: set-up of the unfoldings included, factors and duals carried from step to step)."""
    import torch
    from source import _native, workloads as wl
    rank, world, dev = rk.rank, rk.world, rk.dev
    jobs = []
    weights = {}
    for key, name, cout, cin, kh, kw, rr, bits in mine:
        if name not in weights:
            weights[name] = wl.layer_weight_as_tensor(wl.synthetic_weight(cout, cin, kh, kw, 42, name)).contiguous()
        W = weights[name]
        rnk = wl.rank_from_reduction_rate(W, rr)
        init = wl.random_init(W.shape, rnk, 42)
        jobs.append({"key": key, "Wh": W, "rank": rnk, "bits": bits, "init": init,
                     "cost": wl.unit_cost(W.shape, rnk, bits)})
    jobs.sort(key=lambda j: -j["cost"])
    rounds = [jobs[i:i + args.round_size] for i in range(0, len(jobs), args.round_size)]
    wdev = {n: w.to(dev) for n, w in weights.items()}
    for rd in rounds:
        ctas = allocate_ctas([j["cost"] for j in rd], sm_count, 1)
        for j, g in zip(rd, ctas):
            name = j["key"].split("/")[0]
            j.update(W=wdev[name], factors=[f.to(dev) for f in j["init"]], qscheme=QSCHEME, max_iter_als=1,
                     max_iter_admm=args.max_iter_admm, solve_precision=args.solve_precision,
                     mttkrp_precision=args.mttkrp_precision, max_ctas=g, stream=torch.cuda.Stream(device=dev))
            j["duals"] = [torch.zeros_like(f) for f in j["factors"]]
            need = int(_native.lib.admmq_factorize_workspace_bytes(
                j["W"].ndim, (_native.ctypes.c_int * j["W"].ndim)(*j["W"].shape), j["rank"],
                _native.ctypes.byref(_native.FactorizeParams(1, args.max_iter_admm, 1e-8, 1e-5, j["bits"], 0, 200,
                                                             args.solve_precision, args.mttkrp_precision, g, 1))))
            j["ws"] = torch.empty(need, dtype=torch.uint8, device=dev)
            j["host"] = {"factors": [f.clone().pin_memory() for f in j["init"]],
                         "duals": [torch.zeros_like(f).pin_memory() for f in j["init"]],
                         "factors_q": [torch.zeros_like(f).pin_memory() for f in j["init"]]}
    n_modes = sum(j["W"].ndim for j in jobs)
    inner_nominal = n_modes * (args.max_iter_admm - 1)

    def step(e2e=False):
        moved = [0, 0]
        errs = {}
        for rd in rounds:
            if e2e:
                for j in rd:
                    with torch.cuda.stream(j["stream"]):
                        for dst, src in zip(j["factors"] + j["duals"], j["host"]["factors"] + j["host"]["duals"]):
                            dst.copy_(src, non_blocking=True)
                            moved[0] += dst.numel() * 4
            out = _native.factorize_batch(rd)
            for j, (hist, histq, n, fq) in zip(rd, out):
                errs[j["key"]] = hist[-1]
                j["last"] = (fq, hist[-1], histq[-1])
                if e2e:
                    for dst, src in zip(j["host"]["factors"] + j["host"]["duals"] + j["host"]["factors_q"],
                                        j["factors"] + j["duals"] + fq):
                        dst.copy_(src, non_blocking=True)
                        moved[1] += src.numel() * 4
        torch.cuda.synchronize()
        return errs, moved

    flush = torch.empty(256 << 20, dtype=torch.uint8, device=dev)
    for _ in range(max(args.warmup, 1)):
        step()
    sampler = ClockSampler(rk.local)
    if rank == 0:
        sampler.start()
    launches0 = _native.launch_count()
    step_ms, errs = [], {}
    rk.barrier()
    for _ in range(args.steps):
        flush.fill_(1)
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        errs, _ = step()
        e1.record()
        torch.cuda.synchronize()
        step_ms.append(e0.elapsed_time(e1))
    rk.barrier()
    launches = _native.launch_count() - launches0
    clocks = sampler.stop() if rank == 0 else None
    total_ms = rk.reduce(sum(step_ms), "MAX")
    # the batch entry point keeps the loop reports on the device; the nominal budget is counted (tap factors of wide
    # layers leave early in later sweeps, so this is an upper bound of the executed iterations by a few per cent)
    inner_all = rk.reduce(inner_nominal * args.steps, "SUM")
    value = inner_all / (total_ms / 1e3)
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, [(j["key"], j["factors"], *j["last"]) for j in jobs], world)
    e2e = None
    if not args.no_e2e:
        step(e2e=True)
        rk.barrier()
        t, moved = [], [0, 0]
        for _ in range(args.steps):
            flush.fill_(1)
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            _, moved = step(e2e=True)
            e1.record()
            torch.cuda.synchronize()
            t.append(e0.elapsed_time(e1))
        rk.barrier()
        tot = rk.reduce(sum(t), "MAX")
        e2e = {"value": inner_all / (tot / 1e3), "unit": UNIT, "h2d_bytes_per_step": int(rk.reduce(moved[0], "SUM")),
               "d2h_bytes_per_step": int(rk.reduce(moved[1], "SUM")), "ms_per_step": tot / args.steps}
    gather_ms, gather_bytes = rk.gather_factors([f for j in jobs for f in j["factors"]])
    per_rank = rk.gather_objects({"rank": rank, "units": len(jobs), "rounds": len(rounds), "ms_per_step": sum(step_ms) / args.steps,
                                  "launches": launches, "gather_bytes": gather_bytes,
                                  "cost": sum(j["cost"] for j in jobs)})
    if rank == 0:
        line = {"metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
                "ms_per_step": total_ms / args.steps, "higher_is_better": True, "scaling": "strong", "vs_baseline": None,
                "dtype": "f32", "data": "synthetic",
                "config": config_dict(args, desc, {"l2": "flushed between timed steps (256 MiB write)",
                                                   "parallelism": f"one job, {len(units)} units sharded over {world} GPU(s) by LPT; "
                                                                  f"rounds of {args.round_size} concurrent units per GPU; no data-path collective",
                                                   "units_per_rank": [pr["units"] for pr in per_rank],
                                                   "rounds_per_rank": [pr["rounds"] for pr in per_rank],
                                                   "inner_iterations_per_step": inner_all / args.steps,
                                                   "inner_iterations_counted": "nominal budget (max_iter_admm - 1 per factor update)"}),
                "clocks": clocks, "e2e": e2e, "gpu_launches": sum(pr["launches"] for pr in per_rank), "roofline": None,
                "cpu_baseline": None, "per_rank_ms_per_step": [round(pr["ms_per_step"], 2) for pr in per_rank],
                "per_rank_cost_share": [round(pr["cost"] / sum(p["cost"] for p in per_rank), 4) for pr in per_rank],
                "rec_error_sample": dict(list(errs.items())[:8]),
                "factor_gather_ms": gather_ms, "factor_gather_bytes_per_rank": [pr["gather_bytes"] for pr in per_rank]}
        print(json.dumps(line), flush=True)
    if world > 1:
        rk.dist.destroy_process_group()
    return 0


# ------------------------------------------------------------------------------------------ the metric's second half
def run_full(args, rk, units, owner, mine, desc, sm_count):
    """"Full factorize time" (reference: the printed "took N minutes", scripts/factorize.py:177, 342-343): every unit
    from its initialisation (`--init random | parafac-epc`, source/admm.py:21-48) to the reference's stop rule
    (:259-263), all local units concurrently on their SM budgets.  Reports init seconds, ADMM seconds and sweeps per
    unit and the job's wall time = max over ranks."""
    import torch
    from source import _native, workloads as wl
    from source.admm import init_factors
    from source.solver import LayerSolver
    rank, world, dev = rk.rank, rk.world, rk.dev
    import numpy as np
    problems = []
    for key, name, cout, cin, kh, kw, rr, bits in mine:
        W = wl.layer_weight_as_tensor(wl.synthetic_weight(cout, cin, kh, kw, 42, name)).contiguous()
        problems.append((key, W, wl.rank_from_reduction_rate(W, rr), bits))
    rk.barrier()
    t_job = time.perf_counter()
    init_s, solvers = {}, []
    budgets = allocate_ctas([wl.solve_cost(W.shape, r) for _, W, r, _ in problems], sm_count, args.min_ctas) \
        if len(problems) > 1 else [0] * len(problems)
    # Initialisation of every local unit, concurrently: one host thread and one CUDA stream per unit.  An EPC pass is
    # bound by the latency of the R x R symmetric eigen-decomposition (cuSOLVER, a small part of the GPU), so independent
    # units overlap almost perfectly.  Every unit draws its ALS start from RandomState(42) - the stream a fresh process
    # of the reference gets from np.random.seed(42) (scripts/factorize.py:21-24).
    from concurrent.futures import ThreadPoolExecutor
    init_info = {}

    def init_unit(k):
        key, W, rnk, bits = problems[k]
        torch.cuda.set_device(dev)
        st = torch.cuda.Stream(device=dev)
        t0 = time.perf_counter()
        with torch.cuda.stream(st):
            Wd = W.to(dev)
            fac = init_factors(Wd, rank=rnk, init=args.init, device=dev if args.init != "random" else None, seed=42,
                               rng=np.random.RandomState(42))
            fac = [f.to(dev).contiguous() for f in fac]
        st.synchronize()
        init_s[key] = time.perf_counter() - t0
        return Wd, fac

    if args.init != "random":   # torch loads its CUDA linear-algebra library lazily and not thread-safely: do it here
        eye = torch.eye(4, dtype=torch.float64, device=dev)
        torch.linalg.solve(eye, eye)
        torch.linalg.eigh(eye)
        torch.cuda.synchronize()
    t_init = time.perf_counter()
    with ThreadPoolExecutor(max_workers=max(1, min(len(problems), 16))) as pool:
        inits = list(pool.map(init_unit, range(len(problems))))
    torch.cuda.synchronize()
    init_wall = time.perf_counter() - t_init
    for (key, W, rnk, bits), g, (Wd, fac) in zip(problems, budgets, inits):
        solvers.append(LayerSolver(Wd, fac, bits, QSCHEME, max_iter_admm=args.max_iter_admm, init_is_random=(args.init == "random"),
                                   mttkrp_precision=args.mttkrp_precision, solve_precision=args.solve_precision, max_ctas=g))
    streams = [torch.cuda.Stream(device=dev) for _ in solvers]
    torch.cuda.synchronize()
    t_admm = time.perf_counter()
    active = list(range(len(solvers)))
    sweeps = {p[0]: 0 for p in problems}
    admm_s = {}
    inner = 0
    while active:
        for k in active:
            streams[k].wait_stream(torch.cuda.current_stream())
            with torch.cuda.stream(streams[k]):
                solvers[k].enqueue_sweep()
        nxt = []
        for k in active:
            streams[k].synchronize()
            solvers[k].collect()
            inner += sum(int(r.iterations) for r in solvers[k].last_reports)
            sweeps[problems[k][0]] += 1
            if solvers[k].should_stop() or sweeps[problems[k][0]] >= args.max_iter_als:
                admm_s[problems[k][0]] = time.perf_counter() - t_admm
            else:
                nxt.append(k)
        if len(nxt) < len(active) and len(nxt) > 0:   # units that finished hand their SMs to the others
            for k, g in zip(nxt, allocate_ctas([wl.solve_cost(problems[k][1].shape, problems[k][2]) for k in nxt], sm_count,
                                               args.min_ctas if len(nxt) > 1 else sm_count)):
                solvers[k].max_ctas = g if len(nxt) > 1 else 0
        active = nxt
    torch.cuda.synchronize()
    wall = time.perf_counter() - t_job
    job_s = rk.reduce(wall, "MAX")
    inner_all = rk.reduce(inner, "SUM")
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, [(p[0], s.factors, s.factors_q, s.loss_hist[-1], s.loss_quant_hist[-1])
                                         for p, s in zip(problems, solvers)], world)
    gather_ms, _ = rk.gather_factors([f for s in solvers for f in s.factors])
    per_rank = rk.gather_objects({"init_s": {k: round(v, 3) for k, v in init_s.items()},
                                  "admm_s": {k: round(v, 3) for k, v in admm_s.items()}, "sweeps": sweeps,
                                  "rec_error": {p[0]: round(s.loss_hist[-1], 6) for p, s in zip(problems, solvers)},
                                  "quant_rec_error": {p[0]: round(s.loss_quant_hist[-1], 6) for p, s in zip(problems, solvers)},
                                  "wall_s": wall, "init_wall_s": init_wall})
    if rank == 0:
        merged = {f: {k: v for pr in per_rank for k, v in pr[f].items()} for f in ("init_s", "admm_s", "sweeps", "rec_error", "quant_rec_error")}
        line = {"metric": "full_factorize_time_s", "value": job_s, "unit": "s", "n_gpus": world, "steps": 1, "warmup": 0,
                "higher_is_better": False, "scaling": "strong", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
                "config": config_dict(args, desc, {"init": args.init, "max_iter_als": args.max_iter_als,
                                                   "stop_rule": "scripts/factorize.py:259-263 (|d rec_error| < 1e-5 or divergence guard)",
                                                   "parallelism": f"{len(units)} units sharded over {world} GPU(s) by LPT; no data-path collective"}),
                "inner_iterations": inner_all, "inner_iter_per_s_incl_init": inner_all / job_s,
                "per_rank_wall_s": [round(pr["wall_s"], 2) for pr in per_rank],
                "per_rank_init_wall_s": [round(pr["init_wall_s"], 2) for pr in per_rank],
                "note": "init_s / admm_s are per unit (units of a rank run concurrently: init on one host thread + stream each, "
                        "ADMM on SM budgets); value = the job's wall time = max over ranks of (init + ADMM to the stop rule)",
                "factor_gather_ms": gather_ms, **merged}
        print(json.dumps(line), flush=True)
    if world > 1:
        rk.dist.destroy_process_group()
    return 0


def main():
    args = parse_args()
    if args.steps < 1 or args.warmup < 0:
        raise SystemExit("--steps >= 1 and --warmup >= 0")
    if args.dump_outputs and args.impl == "reference":
        raise SystemExit("--dump-outputs: the reference arm times samples, not the workload's outputs")
    sys.exit(run_reference(args) if args.impl == "reference" else run_native(args))


if __name__ == "__main__":
    main()
