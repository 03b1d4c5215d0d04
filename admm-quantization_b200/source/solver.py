"""Outer AO-ADMM loop of the reference CLI (scripts/factorize.py:176-318) as a reusable object.

One `LayerSolver` owns one layer's problem on one GPU: the unfoldings of W (made once), the
factors, the scaled duals, every scratch buffer and the loss histories.  `enqueue_sweep()` puts one
outer iteration on the current CUDA stream without allocating or synchronising - per mode the
Gram-Hadamard, the MTTKRP, the ridge-system inverse, the persistent ADMM kernel and the
re-projection, then the two reconstruction-error reductions - and `collect()` reads the two error
sums and the loop reports back (one host sync per sweep) to apply the reference's stop rules
(:259-263 / :303-307).  Several solvers can be enqueued back to back before the first `collect()`.
"""
import numpy as np
import torch

from . import _native
from .shapes import layer_weight_as_tensor, rank_from_reduction_rate  # noqa: F401  (re-exported)


def _bytes(n, device):
    return torch.empty(max(int(n), 256), dtype=torch.uint8, device=device)


class LayerSolver:
    def __init__(self, weight, factors, bits, qscheme, max_iter_admm=1000, eps=1e-8, tol=1e-5,
                 num_attempts=200, mttkrp_precision=0, init_is_random=True, time_loops=False, solve_precision=0,
                 max_ctas=0):
        _native.require_cuda(weight)
        assert weight.ndim in (2, 3), "Incorrect number of dimentions in weight tensor"
        self.W = _native.f32c(weight)
        self.N = self.W.ndim
        self.bits, self.qscheme = int(bits), qscheme
        _native.qscheme_id(qscheme)
        self.max_iter_admm, self.eps, self.tol = int(max_iter_admm), float(eps), float(tol)
        self.num_attempts, self.mttkrp_precision = int(num_attempts), int(mttkrp_precision)
        self.solve_precision = int(solve_precision)
        self.max_ctas = int(max_ctas)   # cooperative-grid budget of this solver (0 = every SM), see include/admmq.h
        dev = self.W.device
        self.factors = [_native.f32c(f).to(dev).clone() for f in factors]
        self.duals = [torch.zeros_like(f) for f in self.factors]       # :209-212 / :272-273
        self.factors_q = [torch.empty_like(f) for f in self.factors]
        self.loss_hist, self.loss_quant_hist = [], []
        self.R = R = self.factors[0].shape[1]
        if self.N == 3:
            I, J, K = self.W.shape
            self.unfoldings = [self.W.reshape(I, J * K), _native.unfold3(self.W, 1), _native.unfold3(self.W, 2)]
        else:
            self.unfoldings = [self.W, self.W.t().contiguous()]
        # ---- preallocated scratch (the C ABI never allocates; neither does a sweep)
        dims = [f.shape[0] for f in self.factors]
        ld = _native.lib.admmq_padded_ld(R)
        self.G = torch.empty(R, R, dtype=torch.float32, device=dev)
        self.F = [torch.empty(d, R, dtype=torch.float32, device=dev) for d in dims]
        self.Minv = torch.empty(R, ld, dtype=torch.float32, device=dev)
        # parity mode (solve_precision 0): the loop multiplies by the float64 inverse and accumulates in float64
        self.Minv64 = torch.empty(R, ld, dtype=torch.float64, device=dev) if self.solve_precision == 0 else None
        self.rho = torch.empty(1, dtype=torch.float32, device=dev)
        self.inv_status = torch.zeros(1, dtype=torch.int32, device=dev)
        self.reports_dev = [_native.new_report(dev) for _ in range(self.N)]
        self.err_sums = torch.zeros(2, 2, dtype=torch.float64, device=dev)
        others = [[k for k in range(self.N) if k != m] for m in range(self.N)]
        self._others = others
        nxny = [(dims[o[0]], dims[o[1]] if self.N == 3 else 1) for o in others]
        self.ws_inv = _bytes(_native.spd_inverse_workspace_bytes(R), dev)
        self.ws_loop = _bytes(max(_native.admm_loop_workspace_bytes(d, R, self.num_attempts) for d in dims), dev)
        self.ws_proj = _bytes(_native.project_workspace_bytes(max(dims) * R, self.num_attempts), dev)
        if self.mttkrp_precision == 1:
            # tensor-core MTTKRP: the (m, y, x) permutations of W are constant, make them once (include/admmq.h)
            self.permuted = [_native.permute_myx(self.unfoldings[m], nxny[m][0], nxny[m][1]) for m in range(self.N)]
            self.ws_mttkrp = _bytes(max(_native.mttkrp_tc_workspace_bytes(dims[m], nxny[m][0], nxny[m][1], R)
                                        for m in range(self.N)), dev)
        else:
            self.permuted = None
            self.ws_mttkrp = _bytes(max(_native.mttkrp_workspace_bytes(dims[m], nxny[m][0], nxny[m][1], R, 0)
                                        for m in range(self.N)), dev)
        self.ws_err = _bytes(_native.recon_error_workspace_bytes(dims[0], nxny[0][0], nxny[0][1]), dev)
        self.time_loops = bool(time_loops)
        self.loop_events = []      # (mode, start, stop) CUDA events around the persistent kernel
        self.part_events = None    # set to [] to record an event after every kernel group of a sweep (diagnostics)
        self.last_reports = []
        self._pending = False
        self.snapshot_inputs = False   # diagnostics: keep clones of (H, U, F, G) entering every loop call of a sweep
        self.snapshots = {}
        if not init_is_random:                                          # :192-201
            fq = [_native.project(f, self.bits, qscheme, self.num_attempts)[0] for f in self.factors]
            self.loss_hist.append(self._error(self.factors))
            self.loss_quant_hist.append(self._error(fq))

    # ---- pieces
    def _error_sums(self, fac, out=None):
        y = fac[2] if self.N == 3 else None
        return _native.recon_error_sums(self.unfoldings[0], fac[0], fac[1], y, out=out, ws=self.ws_err)

    @staticmethod
    def _finish_error(sums):
        num, den = (np.float32(v) for v in sums)
        return float(np.sqrt(np.float32(num / den)))                    # source/admm.py:15 in float32

    def _error(self, fac):
        return self._finish_error(self._error_sums(fac).cpu().numpy())

    def update_mode(self, mode, codes=None):
        """One ALS step for `mode`: scripts/factorize.py:215-224 (and the two analogous blocks)."""
        o = self._others[mode]
        X = self.factors[o[0]]
        Y = self.factors[o[1]] if self.N == 3 else None
        self._mark(f"m{mode}:start")
        _native.gram_hadamard(X, Y, out=self.G)                                          # :215
        self._mark(f"m{mode}:gram")
        if self.permuted is not None:
            _native.mttkrp_tc(self.permuted[mode], self.F[mode].shape[0], X, Y, out=self.F[mode], ws=self.ws_mttkrp)
        else:
            _native.mttkrp(self.unfoldings[mode], X, Y, 0, out=self.F[mode], ws=self.ws_mttkrp)  # :217
        self._mark(f"m{mode}:mttkrp")
        _native.spd_inverse(self.G, out=(self.Minv, self.rho, self.inv_status), ws=self.ws_inv,
                            max_ctas=self.max_ctas, minv64=self.Minv64)  # source/admm.py:52-54
        self._mark(f"m{mode}:inverse")
        if self.snapshot_inputs:
            self.snapshots[mode] = (self.factors[mode].clone(), self.duals[mode].clone(), self.F[mode].clone(), self.G.clone())
        if self.time_loops:
            ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            ev0.record()
        _native.admm_loop_inplace(self.factors[mode], self.duals[mode], self.F[mode], self.Minv, self.rho,
                                  self.inv_status, self.max_iter_admm, self.eps, self.bits, self.qscheme,
                                  self.num_attempts, codes, report=self.reports_dev[mode], ws=self.ws_loop,
                                  precision=self.solve_precision, max_ctas=self.max_ctas, minv64=self.Minv64)  # :218
        if self.time_loops:
            ev1.record()
            self.loop_events.append((mode, ev0, ev1))
        self._mark(f"m{mode}:loop")
        _native.project(self.factors[mode], self.bits, self.qscheme, self.num_attempts,
                        out=self.factors_q[mode], ws=self.ws_proj)                       # :222
        self._mark(f"m{mode}:project")

    def _mark(self, label):
        if self.part_events is not None:
            ev = torch.cuda.Event(enable_timing=True)
            ev.record()
            self.part_events.append((label, ev))

    def part_times_ms(self):
        """[(label, ms since the previous mark)] of the last recorded sweep (after a synchronise)."""
        ev = self.part_events or []
        return [(ev[i][0], ev[i - 1][1].elapsed_time(ev[i][1])) for i in range(1, len(ev))]

    def enqueue_sweep(self):
        """One outer iteration (:214-255) on the current stream; no allocation, no host sync."""
        if self.part_events is not None:
            self.part_events.clear()
        for mode in range(self.N):
            self.update_mode(mode)
        self._error_sums(self.factors, out=self.err_sums[0])           # :246-248
        self._error_sums(self.factors_q, out=self.err_sums[1])         # :249-253
        self._mark("errors")
        self._pending = True

    def collect(self):
        """Host side of the sweep: read errors + reports (synchronises), append to the histories."""
        assert self._pending, "collect() without enqueue_sweep()"
        sums = self.err_sums.cpu().numpy()
        self.last_reports = [_native.read_report(r) for r in self.reports_dev]  # LinAlgError on a non-PD system
        err, errq = self._finish_error(sums[0]), self._finish_error(sums[1])
        self.loss_hist.append(err)
        self.loss_quant_hist.append(errq)
        self._pending = False
        return err, errq

    def sweep(self):
        self.enqueue_sweep()
        return self.collect()

    # ---- host-buffer interface (the call a user with CPU tensors makes; bench.py's end-to-end leg)
    def load_from_host(self, weight, factors, duals):
        """Host -> device copy of the layer state (pinned tensors copy asynchronously on the current stream)
        and re-derivation of the unfoldings.  Returns the number of bytes copied."""
        n = 0
        self.W.copy_(weight.reshape(self.W.shape), non_blocking=True)
        n += self.W.numel() * 4
        if self.N == 3:
            _native.unfold3(self.W, 1, out=self.unfoldings[1])
            _native.unfold3(self.W, 2, out=self.unfoldings[2])
        else:
            self.unfoldings[1].copy_(self.W.t())
        if self.permuted is not None:
            dims = [f.shape[0] for f in self.factors]
            for m in range(self.N):
                o = self._others[m]
                _native.call(self.W.device, _native.lib.admmq_permute_myx, _native.ptr(self.unfoldings[m]), dims[m],
                             dims[o[0]], dims[o[1]] if self.N == 3 else 1, _native.ptr(self.permuted[m]),
                             _native.stream_ptr(self.W.device))
        for dst, src in zip(self.factors + self.duals, list(factors) + list(duals)):
            dst.copy_(src, non_blocking=True)
            n += dst.numel() * 4
        return n

    def store_to_host(self, factors, duals, factors_q, err_sums, reports=None):
        """Device -> host copy of the sweep's results into (pinned) host tensors; asynchronous - synchronise
        the stream, then call `check_host_reports(reports)`, before reading them.  `reports` is a pinned uint8 tensor
        of N * sizeof(LoopReport) bytes that receives the loop reports: a ridge system that was not positive definite
        (loop skipped, factors untouched) or a non-finite loop must not go unnoticed on this path either.  Without
        `reports` the sweep stays pending and `collect()` must still be called.  Returns the number of bytes copied."""
        n = 0
        for dst, src in zip(list(factors) + list(duals) + list(factors_q), self.factors + self.duals + self.factors_q):
            dst.copy_(src, non_blocking=True)
            n += src.numel() * 4
        err_sums.copy_(self.err_sums, non_blocking=True)
        n += self.err_sums.numel() * 8
        if reports is not None:
            size = self.reports_dev[0].numel()
            for m, r in enumerate(self.reports_dev):
                reports[m * size:(m + 1) * size].copy_(r, non_blocking=True)
            n += self.N * size
            self._pending = False
        return n

    def check_host_reports(self, reports):
        """Decode the loop reports `store_to_host` copied (after the stream was synchronised): raises
        torch.linalg.LinAlgError for a non-positive-definite ridge system like `collect()` and the reference's
        torch.linalg.cholesky; returns the reports."""
        size = self.reports_dev[0].numel()
        self.last_reports = [_native.decode_report(bytes(reports[m * size:(m + 1) * size].numpy().tobytes()))
                             for m in range(self.N)]
        return self.last_reports

    def should_stop(self):
        """Stop rules of scripts/factorize.py:259-263 (3-D) and :303-307 (2-D)."""
        h = self.loss_hist
        if len(h) > 1 and abs(h[-2] - h[-1]) < self.tol:
            return True
        back = 5 if self.N == 3 else 10
        if len(h) > 10 and h[-1] - h[-back] > 1e-3:
            return True
        return False

    def run(self, max_iter_als, progress=None):
        sweeps = 0
        it = range(max_iter_als) if progress is None else progress(range(max_iter_als))
        for _ in it:
            self.sweep()
            sweeps += 1
            if self.should_stop():
                break
        return sweeps

    # ---- accounting used by bench.py (SURVEY 8(d): the unit of work is one inner iteration of one factor)
    def inner_iterations_per_sweep(self):
        return self.N * max(self.max_iter_admm - 1, 0)

    def loop_algorithmic_bytes_per_sweep(self):
        """16 B per element of H (read H, U, F; write H, U - counted once) + one pass over Minv, per inner
        iteration, summed over the modes of one sweep (DESIGN.md 'roofline')."""
        it = max(self.max_iter_admm - 1, 0)
        return sum(it * (16 * f.shape[0] * self.R + 4 * self.R * self.R) for f in self.factors)

    def candidate_evaluations_per_sweep(self):
        it = max(self.max_iter_admm - 1, 0)
        nc = self.num_attempts if self.qscheme in _native.CLIP_SEARCH_SCHEMES else 0
        return sum(it * nc * f.shape[0] * self.R for f in self.factors)

    def solve_flops_per_sweep(self):
        it = max(self.max_iter_admm - 1, 0)
        return sum(it * 2 * f.shape[0] * self.R * self.R for f in self.factors)
