"""GPU parity tests: the CUDA path (through the C ABI, via source._native) against the golden
vectors produced by the unmodified reference and against the CPU oracle on seeded inputs.

Tolerances (north_star): integer codes / grid values of the projection bit-exact given identical
input; one ADMM step from identical state >= 99.9 % identical codes (the ridge solve is a float32
product with a float64-computed inverse instead of LAPACK potrs, so H_ls differs in the last
bits); reconstruction errors within 1e-3 relative."""
import os

import numpy as np
import pytest
import torch

pytestmark = pytest.mark.gpu
MSE = "tensor_mseminmax_symmetric"


@pytest.fixture(scope="module")
def nat():
    from source import _native
    return _native


def dev(a):
    return torch.from_numpy(np.ascontiguousarray(a)).cuda()


def bits_equal(a, b):
    return np.array_equal(np.asarray(a, dtype=np.float32).view(np.uint32), np.asarray(b, dtype=np.float32).view(np.uint32))


# ------------------------------------------------------------------ projection
def test_projection_bit_exact_on_reference_vectors(nat, golden_projection):
    gp = golden_projection
    for m in gp.meta:
        if "scheme" in m:
            continue
        n = m["name"]
        x = dev(gp[n + "/x"])
        out, codes, info = nat.project(x, m["bits"], MSE, m["num_attempts"], want_codes=True, want_info=True)
        out, codes, info = out.cpu().numpy(), codes.cpu().numpy(), info.cpu().numpy()
        if n == "all_zero_b4":
            assert np.isnan(out).all()  # reference: scale 0 -> NaN everywhere
            continue
        idx, scale = gp[n + "/idx_scale"]
        assert int(info[2]) == int(idx), (n, info, idx)
        assert np.float32(info[0]) == np.float32(scale), n
        assert np.array_equal(codes, gp[n + "/codes"]), n
        assert bits_equal(out, gp[n + "/xq"]), n


def test_other_schemes_bit_exact(nat, golden_projection):
    gp = golden_projection
    for m in gp.meta:
        if "scheme" not in m:
            continue
        n = m["name"]
        out, _, _ = nat.project(dev(gp[n + "/x"]), m["bits"], m["scheme"])
        assert bits_equal(out.cpu().numpy(), gp[n + "/xq"]), n


def test_projection_matches_oracle_on_random_tensors(nat):
    """Seeded sweep over shapes / bit-widths / candidate counts incl. ragged and tiny inputs."""
    from oracle import admm_oracle as orc
    torch.set_num_threads(1)
    g = torch.Generator().manual_seed(2024)
    shapes = [(1, 1), (1, 7), (3, 5), (9, 134), (64, 67), (17, 333), (128, 183), (2, 4097)]
    checked = 0
    for shape in shapes:
        for bits in (2, 3, 4, 6, 8):
            for nc in (200, 33):
                x = torch.randn(*shape, generator=g) * float(10 ** torch.randint(-3, 3, (1,), generator=g).item())
                xq, codes, scale, best, mses = orc.project_mse(x, bits, nc, "aten")
                out, c, info = nat.project(x.cuda(), bits, MSE, nc, want_codes=True, want_info=True)
                info = info.cpu().numpy()
                if int(info[2]) != best:
                    # tolerated only when the two candidates are tied to within float32 summation noise
                    gap = abs(float(mses[int(info[2])]) - float(mses[best])) / float(mses[best])
                    assert gap < 3e-7, (shape, bits, nc, best, info, gap)
                    continue
                assert np.array_equal(c.cpu().numpy(), codes.numpy()), (shape, bits, nc)
                assert bits_equal(out.cpu().numpy(), xq.numpy()), (shape, bits, nc)
                checked += 1
    assert checked >= 70


def test_projection_full_size_layer4(nat):
    """BASELINE config-2 size (512 x 1141) and the slow-path: oracle still finishes in seconds."""
    from oracle import admm_oracle as orc
    torch.set_num_threads(4)
    g = torch.Generator().manual_seed(7)
    x = torch.randn(512, 1141, generator=g) * 0.05
    xq, codes, scale, best, _ = orc.project_mse(x, 4, 200, "aten")
    out, c, info = nat.project(x.cuda(), 4, MSE, 200, want_codes=True, want_info=True)
    assert int(info[2].item()) == best
    assert np.array_equal(c.cpu().numpy(), codes.numpy())
    assert bits_equal(out.cpu().numpy(), xq.numpy())
    # size-independent properties
    vals = torch.unique(out)
    assert vals.numel() <= 16
    again, _, _ = nat.project(out, 4, MSE, 200)
    assert torch.unique(again).numel() <= 16
    torch.set_num_threads(1)


def test_threshold_search_against_direct_evaluation(nat):
    """The product's threshold form of the clip search (csrc/numerics.cuh) against the direct evaluation of every
    (element, candidate) pair with the reference's float32 operations, incl. BASELINE full sizes, skewed / grid-valued
    / outlier inputs and every bit-width: sums agree to float32 summation noise, the argmin is the same (or a near
    tie), the result does not depend on the grid beyond fixed-point rounding and is bit-reproducible run to run."""
    g = torch.Generator().manual_seed(99)
    cases = []
    for shape, bits, nc in [((512, 1141), 4, 200), ((4096, 1024), 4, 200), ((64, 134), 4, 200), ((9, 1141), 4, 200),
                            ((256, 566), 3, 200), ((128, 278), 8, 200), ((64, 134), 8, 1000), ((300, 77), 2, 200),
                            ((37, 41), 1, 200), ((1, 5), 4, 200), ((2048, 204), 6, 200), ((1, 1), 4, 7)]:
        cases.append((torch.randn(*shape, generator=g) * 0.07, bits, nc, "randn"))
    x = torch.randn(256, 566, generator=g)
    x[17, 3] = 250.0
    cases.append((x, 4, 200, "outlier"))
    cases.append((torch.randn(200, 300, generator=g).abs() + 5.0, 4, 200, "offset"))
    cases.append((torch.randint(-8, 8, (128, 278), generator=g).float() * 0.013, 4, 200, "grid-valued"))
    cases.append((torch.full((64, 64), 0.37), 4, 200, "constant"))
    cases.append((torch.randn(128, 128, generator=g) * 1e-9, 4, 200, "small"))
    cases.append((torch.randn(128, 128, generator=g) * 1e9, 4, 200, "large"))
    for x, bits, nc, tag in cases:
        xd = x.cuda()
        direct = nat.clip_search_sums(xd, bits, nc, method=0).cpu().numpy()
        thr = nat.clip_search_sums(xd, bits, nc, method=1).cpu().numpy()
        n = x.numel()
        floor = 1e-13 * float((x.double() ** 2).sum()) + 1e-300
        assert np.all(np.abs(thr - direct) <= 3e-6 * np.abs(direct) + floor), (tag, tuple(x.shape), bits, nc)
        mse_d, mse_t = (direct / n).astype(np.float32), (thr / n).astype(np.float32)
        bd, bt = int(np.argmin(mse_d)), int(np.argmin(mse_t))
        if bd != bt:
            assert abs(float(mse_d[bd]) - float(mse_d[bt])) <= 3e-7 * float(mse_d[bd]), (tag, bd, bt)
        again = nat.clip_search_sums(xd, bits, nc, method=1).cpu().numpy()
        assert np.array_equal(thr, again), tag
        few = nat.clip_search_sums(xd, bits, nc, method=1, max_ctas=3).cpu().numpy()
        assert np.all(np.abs(few - thr) <= 1e-11 * np.abs(thr) + floor), tag


def test_projection_in_place_and_repeatable(nat):
    g = torch.Generator().manual_seed(3)
    x = torch.randn(300, 77, generator=g).cuda()
    a, ca, _ = nat.project(x, 4, MSE, want_codes=True)
    b, cb, _ = nat.project(x, 4, MSE, want_codes=True)
    assert torch.equal(a, b) and torch.equal(ca, cb)


def test_bad_arguments_raise(nat):
    x = torch.randn(4, 4).cuda()
    with pytest.raises(NotImplementedError):
        nat.project(x, 4, "channel_affine")
    with pytest.raises(ValueError):
        nat.project(x, 0, MSE)
    with pytest.raises(ValueError):
        nat.project(x, 4, MSE, num_attempts=5000)
    with pytest.raises(RuntimeError):
        nat.project(torch.randn(4, 4), 4, MSE)


# ------------------------------------------------------------------ contractions
def test_contractions_against_reference_and_float64(nat, golden_contractions):
    gc = golden_contractions
    for m in gc.meta:
        n = m["name"]
        W = gc[n + "/W"]
        fac = [gc[n + "/" + k] for k in "ABC"[: m["ndim"]]]
        fd = [dev(f) for f in fac]
        f64 = [f.astype(np.float64) for f in fac]
        if m["ndim"] == 3:
            I, J, K = m["dims"]
            unf = [dev(W.reshape(I, J * K)), nat.unfold3(dev(W), 1), nat.unfold3(dev(W), 2)]
            assert np.array_equal(unf[1].cpu().numpy(), np.moveaxis(W, 1, 0).reshape(J, -1))
            assert np.array_equal(unf[2].cpu().numpy(), np.moveaxis(W, 2, 0).reshape(K, -1))
            subs = ["abc,br,cr->ar", "abc,ar,cr->br", "abc,ar,br->cr"]
        else:
            unf = [dev(W), dev(W.T.copy())]
        for mode in range(m["ndim"]):
            others = [k for k in range(m["ndim"]) if k != mode]
            G = nat.gram_hadamard(fd[others[0]], fd[others[1]] if m["ndim"] == 3 else None).cpu().numpy()
            Gref = gc[f"{n}/G{mode}"]
            G64 = np.ones((m["rank"],) * 2)
            for k in others:
                G64 = G64 * (f64[k].T @ f64[k]).astype(np.float32).astype(np.float64)
            assert np.abs(G - G64).max() <= 2e-7 * np.abs(G64).max()
            assert np.abs(G - Gref).max() <= 2e-5 * np.abs(Gref).max()
            F = nat.mttkrp(unf[mode], fd[others[0]], fd[others[1]] if m["ndim"] == 3 else None).cpu().numpy()
            if m["ndim"] == 3:
                F64 = np.einsum(subs[mode], W.astype(np.float64), f64[others[0]], f64[others[1]])
            else:
                F64 = W.astype(np.float64) @ f64[1] if mode == 0 else W.astype(np.float64).T @ f64[0]
            assert np.array_equal(F, F64.astype(np.float32)) or np.abs(F - F64).max() <= 1.2e-7 * np.abs(F64).max()
            assert np.abs(F - gc[f"{n}/F{mode}"]).max() <= 2e-5 * np.abs(F64).max()
        sums = nat.recon_error_sums(unf[0], fd[0], fd[1], fd[2] if m["ndim"] == 3 else None).cpu().numpy()
        err = float(np.sqrt(np.float32(np.float32(sums[0]) / np.float32(sums[1]))))
        assert abs(err - float(gc[n + "/err"][0])) <= 1e-5 * err


def test_tensor_core_mttkrp_and_gemm(nat, golden_contractions):
    """3xTF32 tcgen05 paths against float64: admmq_gemm_nt and the permuted-operand MTTKRP, incl. ragged shapes.
    Tolerance 4e-6 of the largest output (measured 3e-6 at K = 1141; cuBLAS float32 gives 1.5e-6)."""
    g = torch.Generator().manual_seed(77)
    for (M, N, K) in [(128, 32, 64), (100, 50, 72), (512, 300, 1144), (9, 1141, 512), (64, 134, 136)]:
        A, B = torch.randn(M, K, generator=g), torch.randn(N, K, generator=g)
        C = nat.gemm_nt(A.cuda(), B.cuda()).cpu().double()
        ref = A.double() @ B.double().T
        assert (C - ref).abs().max() <= 4e-6 * ref.abs().max(), (M, N, K)
    gc = golden_contractions
    for m in gc.meta:
        n = m["name"]
        W = gc[n + "/W"]
        fac = [gc[n + "/" + k] for k in "ABC"[: m["ndim"]]]
        fd = [dev(f) for f in fac]
        f64 = [f.astype(np.float64) for f in fac]
        if m["ndim"] == 3:
            I, J, K = m["dims"]
            unf = [dev(W.reshape(I, J * K)), nat.unfold3(dev(W), 1), nat.unfold3(dev(W), 2)]
            subs = ["abc,br,cr->ar", "abc,ar,cr->br", "abc,ar,br->cr"]
        else:
            unf = [dev(W), dev(W.T.copy())]
        for mode in range(m["ndim"]):
            others = [k for k in range(m["ndim"]) if k != mode]
            X = fd[others[0]]
            Y = fd[others[1]] if m["ndim"] == 3 else None
            V = nat.permute_myx(unf[mode], X.shape[0], 1 if Y is None else Y.shape[0])
            F = nat.mttkrp_tc(V, unf[mode].shape[0], X, Y).cpu().numpy()
            if m["ndim"] == 3:
                F64 = np.einsum(subs[mode], W.astype(np.float64), f64[others[0]], f64[others[1]])
            else:
                F64 = W.astype(np.float64) @ f64[1] if mode == 0 else W.astype(np.float64).T @ f64[0]
            assert np.abs(F - F64).max() <= 4e-6 * np.abs(F64).max(), (n, mode)


def test_spd_inverse(nat):
    g = torch.Generator().manual_seed(11)
    for R, n in ((5, 9), (32, 40), (33, 64), (134, 64), (300, 128)):
        B = torch.randn(n, R, generator=g)
        C = torch.randn(9, R, generator=g)
        G = (B.T @ B) * (C.T @ C)
        Minv, rho, status = nat.spd_inverse(G.cuda())
        assert int(status.item()) == 0
        rho_ref = torch.trace(G) / R
        assert float(rho.item()) == float(rho_ref)
        A = (G + rho_ref * torch.eye(R)).double()
        M = Minv[:, :R].cpu().double()
        assert torch.allclose(M, M.T, atol=0, rtol=0)
        resid = (A @ M - torch.eye(R, dtype=torch.float64)).abs().max().item()
        assert resid < 5e-6, (R, resid)
        if Minv.shape[1] > R:
            assert float(Minv[:, R:].abs().max()) == 0.0
        # the float64 inverse of the parity mode: same matrix before its rounding to float32, residual at float64 level
        Minv2, _, _, M64 = nat.spd_inverse(G.cuda(), minv64=True)
        assert torch.equal(Minv2, Minv) and torch.equal(M64.float(), Minv)
        resid64 = (A @ M64[:, :R].cpu() - torch.eye(R, dtype=torch.float64)).abs().max().item()
        assert resid64 < 1e-12 * R, (R, resid64)


def test_not_positive_definite_raises(nat):
    from source.admm import admm_iteration
    R = 40
    G = -torch.eye(R).cuda()
    H = torch.randn(8, R).cuda()
    with pytest.raises(torch.linalg.LinAlgError):
        admm_iteration(H, torch.zeros_like(H), torch.randn(8, R).cuda(), G, 5, 1e-8, 4, MSE)


# ------------------------------------------------------------------ ADMM inner loop
def _grid_codes(h):
    """Integer codes of a grid-valued tensor, recovered from the values alone: level index counted
    from the smallest value, with the level spacing taken as the smallest gap between distinct
    values.  The reference never stores codes; the last bits of its *scale* depend on the last bits
    of the ridge solve (LAPACK potrs there, a float32 product with the float64-computed inverse
    here), so parity is defined on the integer codes (north_star) plus a tolerance on the scale."""
    h = np.asarray(h, dtype=np.float64)
    u = np.unique(h)
    if u.size < 2:
        return np.zeros(h.shape, np.int64), 0.0
    step = np.diff(u).min()
    step = (u[-1] - u[0]) / np.rint((u[-1] - u[0]) / step)  # average spacing: no float32 granularity noise
    return np.rint((h - u[0]) / step).astype(np.int64), float(step)


def _agreement(a, b):
    """Fraction of identical integer codes + relative difference of the grid spacing."""
    ca, sa = _grid_codes(a)
    cb, sb = _grid_codes(b)
    return float(np.mean(ca == cb)), abs(sa - sb) / max(abs(sb), 1e-300)


@pytest.mark.parametrize("precision", [0, 1])
def test_admm_teacher_forced_steps(golden_admm, precision):
    """From the reference's own state at inner iteration k, one step must land on the reference's
    state at k+1: same clip candidate, >= 99.9 % identical grid values.  Checked for both forms of the
    ridge product: float32 FFMA (precision 0) and 3xTF32 on the tensor cores (precision 1)."""
    from source.admm import admm_iteration
    ga = golden_admm
    worst = 1.0
    for m in ga.meta:
        n = m["name"]
        keep = list(ga[n + "/keep"])
        F, G = dev(ga[n + "/F"]), dev(ga[n + "/G"])
        for pos in range(len(keep) - 1):
            if keep[pos + 1] != keep[pos] + 1:
                continue
            H = dev(ga[n + "/H"][pos])
            U = dev(ga[n + "/U"][pos])
            Hn, Un = admm_iteration(H, U, F, G, 2, 1e-8, m["bits"], m["qscheme"], precision=precision)
            assert Un is U
            agree, dscale = _agreement(Hn.cpu().numpy(), ga[n + "/H"][pos + 1])
            worst = min(worst, agree)
            assert agree >= 0.999 and dscale <= 5e-6, (n, keep[pos], agree, dscale)
            du = np.abs(Un.cpu().numpy() - ga[n + "/U"][pos + 1])
            assert np.quantile(du, 0.999) <= 1e-4 * np.abs(ga[n + "/U"][pos + 1]).max() + 1e-6
    print(f"worst teacher-forced agreement (precision {precision})", worst)


@pytest.mark.parametrize("precision", [0, 1])
def test_admm_free_running_first_iterations(golden_admm, capsys, precision):
    """Same start as the reference, one call: report N = the first inner iteration with any differing
    code (north_star: "bit-exact for the first N iterations"), require N > 3 and >= 99 % identical
    codes over the first 12 iterations.  (Measured on B200: 4-bit cases show no mismatch in 60
    iterations; the 3-bit case flips its first element at iteration ~10 - one boundary flip is enough
    for the chaotic trajectory to separate, SURVEY App. E.)"""
    from source.admm import admm_iteration
    ga = golden_admm
    for m in ga.meta:
        n = m["name"]
        keep = list(ga[n + "/keep"])
        F, G = dev(ga[n + "/F"]), dev(ga[n + "/G"])
        first_mismatch = None
        for pos, k in enumerate(keep):
            H = dev(ga[n + "/H0"])
            U = torch.zeros_like(H)
            Hn, _ = admm_iteration(H, U, F, G, k + 2, 1e-8, m["bits"], m["qscheme"], precision=precision)
            agree, dscale = _agreement(Hn.cpu().numpy(), ga[n + "/H"][pos])
            if agree < 1.0 and first_mismatch is None:
                first_mismatch = (k + 1, agree)
            if k < 12:
                assert agree >= 0.99 and dscale <= 1e-5, (n, k, agree, dscale)
        # float32 ridge product: no case flips before iteration 5; 3xTF32 (about twice the rounding noise) may flip
        # an element of the 255-level grid one or two iterations earlier
        assert first_mismatch is None or first_mismatch[0] > (3 if precision == 0 else 1), (n, first_mismatch)
        with capsys.disabled():
            print(f"\n[first-N] precision {precision} {n}: first inner iteration with any differing code: {first_mismatch}")


def test_admm_iteration_semantics(nat):
    """max_iter-1 iterations, U updated in place, fresh H, report fields, codes consistent."""
    from source import admm as A
    g = torch.Generator().manual_seed(5)
    I, R = 24, 40
    H0 = torch.randn(I, R, generator=g).cuda()
    U = torch.zeros(I, R).cuda()
    Bf = torch.randn(30, R, generator=g).cuda()
    G = nat.gram_hadamard(Bf)
    F = torch.randn(I, R, generator=g).cuda()
    keepH = H0.clone()
    H, U2, codes = A.admm_iteration(H0, U, F, G, 7, 1e-8, 4, MSE, return_codes=True)
    assert U2 is U and torch.equal(H0, keepH) and H.data_ptr() != H0.data_ptr()
    rep = A.last_report
    assert rep.iterations == 6 and rep.status == 0 and rep.best_index >= 0
    assert torch.equal(codes.float() * rep.scale, H)
    assert torch.unique(H).numel() <= 16
    # max_iter = 1 -> no iteration (range(1, 1) is empty): H is returned unchanged
    H1, _ = A.admm_iteration(H0, torch.zeros_like(H0), F, G, 1, 1e-8, 4, MSE)
    assert torch.equal(H1, H0) and A.last_report.iterations == 0
    # deterministic
    Ua, Ub = torch.zeros_like(H0), torch.zeros_like(H0)
    Ha, _ = A.admm_iteration(H0, Ua, F, G, 30, 1e-8, 4, MSE)
    Hb, _ = A.admm_iteration(H0, Ub, F, G, 30, 1e-8, 4, MSE)
    assert torch.equal(Ha, Hb) and torch.equal(Ua, Ub)
    # exit test fires with a huge eps (source/admm.py:64-65)
    Hc, _ = A.admm_iteration(H0, torch.zeros_like(H0), F, G, 50, 1e30, 4, MSE)
    assert A.last_report.iterations == 1 and A.last_report.status & 1


@pytest.mark.parametrize("precision", [0, 1])
def test_admm_full_size_step_against_oracle(precision):
    """Two inner iterations at the layer4 size (512 x 1141) against the CPU oracle."""
    from oracle import admm_oracle as orc
    from source.admm import admm_iteration
    torch.set_num_threads(4)
    g = torch.Generator().manual_seed(21)
    I, R = 512, 1141
    Bf, Cf = torch.randn(512, R, generator=g), torch.randn(9, R, generator=g)
    G = (Bf.T @ Bf) * (Cf.T @ Cf)
    F = torch.randn(I, R, generator=g) * 30
    H0 = torch.randn(I, R, generator=g)
    U0 = torch.randn(I, R, generator=g) * 0.1
    Uo = U0.clone()
    Ho, Uo, _ = orc.admm_iteration(H0.clone(), Uo, F, G, 3, 1e-8, 4, MSE)
    Ud = U0.clone().cuda()
    Hd, _ = admm_iteration(H0.cuda(), Ud, F.cuda(), G.cuda(), 3, 1e-8, 4, MSE, precision=precision)
    agree, dscale = _agreement(Hd.cpu().numpy(), Ho.numpy())
    assert agree >= 0.999 and dscale <= 5e-6, (agree, dscale)
    torch.set_num_threads(1)


def test_shared_memory_resident_loop_for_small_factors(nat):
    """A factor that fits in shared memory (64 x 134, 9 x 134) on a budget of one CTA runs the resident kernel (float32
    FFMA arithmetic: precision 1 or 2; the parity mode, precision 0, always takes the general kernel)
    (csrc/admm_loop_resident.cuh): same float32 recipe as the general kernel up to the summation order of the ridge
    product, so codes agree with the CPU oracle and with the general kernel; U is updated in place, the exit test and
    the NaN semantics of a degenerate projection are those of the general kernel."""
    from oracle import admm_oracle as orc
    torch.set_num_threads(1)
    g = torch.Generator().manual_seed(33)
    for (I, R, bits, qs) in [(64, 134, 4, MSE), (9, 134, 4, MSE), (64, 134, 3, MSE), (48, 100, 8, "tensor_minmax"), (64, 134, 4, "tensor_affine")]:
        Bf, Cf = torch.randn(64, R, generator=g), torch.randn(9, R, generator=g)
        G = (Bf.T @ Bf) * (Cf.T @ Cf)
        F = torch.randn(I, R, generator=g) * 24
        H0 = torch.randn(I, R, generator=g)
        U0 = torch.randn(I, R, generator=g) * 0.1
        def close_frac(a, b, ref):   # share of elements that agree to 1e-4 of the scale of ref
            return float(((a - b).abs() <= 1e-4 * float(ref.abs().max())).float().mean())
        for max_iter, need in ((2, 0.9999), (4, 0.999)):
            Uo = U0.clone()
            Ho, Uo, _ = orc.admm_iteration(H0.clone(), Uo, F, G, max_iter, 1e-8, bits, qs)
            outs = []
            for ctas in (1, 0):
                H, U = H0.clone().cuda(), U0.clone().cuda()
                rep = nat.read_report(nat.admm_iteration_inplace(H, U, F.cuda(), G.cuda(), max_iter, 1e-8, bits, qs, precision=2, max_ctas=ctas))
                assert rep.iterations == max_iter - 1
                outs.append((H.cpu(), U.cpu()))
            assert close_frac(outs[0][0], Ho, Ho) >= need, (I, R, bits, qs, max_iter)
            assert close_frac(outs[0][0], outs[1][0], Ho) >= need, (I, R, bits, qs, max_iter)
            if max_iter == 2:
                # one step from identical state: the dual agrees too (later a single flipped code moves a whole row of
                # the next H_ls, SURVEY App. E; U = u + (H - H_ls) is compared on the scale of H)
                assert close_frac(outs[0][1], Uo, Ho) >= need and close_frac(outs[0][1], outs[1][1], Ho) >= need, (I, R, bits, qs)
    # long run: stays on the general kernel's trajectory for dozens of iterations
    Bf, Cf = torch.randn(64, 134, generator=g), torch.randn(9, 134, generator=g)
    G = ((Bf.T @ Bf) * (Cf.T @ Cf)).cuda()
    F = (torch.randn(64, 134, generator=g) * 24).cuda()
    H0 = torch.randn(64, 134, generator=g).cuda()
    res = []
    for ctas in (1, 0):
        H, U = H0.clone(), torch.zeros_like(H0)
        nat.admm_iteration_inplace(H, U, F, G, 41, 1e-8, 4, MSE, precision=2, max_ctas=ctas)
        res.append(H.cpu().numpy())
    agree, _ = _agreement(res[0], res[1])
    assert agree >= 0.99, agree
    # degenerate projection: all-zero state -> NaN everywhere, status NONFINITE (reference: scale 0)
    Z = torch.zeros(64, 134).cuda()
    H, U = Z.clone(), Z.clone()
    rep = nat.read_report(nat.admm_iteration_inplace(H, U, Z.clone(), G, 5, 1e-8, 4, MSE, precision=2, max_ctas=1))
    assert rep.status & nat.ST_NONFINITE and torch.isnan(H).all()


def test_tensor_core_tile_product_random_shapes(nat):
    """Ragged shapes through both operand paths of the 3xTF32 tile product (pre-split B via mttkrp_tc incl. 128-wide
    tiles, on-the-fly split via gemm_nt): one- and two-K-block products, many tiles per CTA, single rows; against
    float64.  (tools/stress_tc.py runs the long version.)"""
    g = torch.Generator().manual_seed(4)
    ri = lambda lo, hi: int(torch.randint(lo, hi + 1, (1,), generator=g))
    shapes = [(1, 1, 1), (5, 3, 2), (129, 17, 64), (130, 129, 65), (700, 1141, 130), (4608, 300, 512)]
    shapes += [(ri(1, 900), ri(1, 1500), ri(1, 1300)) for _ in range(10)]
    for M, R, nx in shapes:
        W = torch.randn(M, nx, generator=g).cuda()
        X = torch.randn(nx, R, generator=g).cuda()
        ldv = (nx + 3) // 4 * 4
        V = torch.zeros(M, ldv, device="cuda")
        V[:, :nx] = W
        ref = W.double() @ X.double()
        scale = float(ref.abs().max().clamp_min(1e-30))
        F = nat.mttkrp_tc(V, M, X, None)
        assert float((F.double() - ref).abs().max()) <= 2e-5 * scale, (M, R, nx)
        Xt = torch.zeros(R, ldv, device="cuda")
        Xt[:, :nx] = X.t()
        C = nat.gemm_nt(V, Xt)
        assert float((C.double() - ref).abs().max()) <= 2e-5 * scale, (M, R, nx)


def test_tensor_core_product_is_independent_of_the_sm_budget(nat):
    """The 3xTF32 ridge product picks its tile width from the CTA budget (16 .. 128 columns with two accumulators, 1 .. 3
    operand stages); every such width accumulates over k in the same order, so ten inner iterations at the layer4 size
    give BIT-IDENTICAL H and U on 148 CTAs (32-wide tiles), 36 (128-wide, one wave), 24 (96-wide) and 7 CTAs - and they
    agree with the CPU oracle like the full-grid run does.  On 32 .. 35 CTAs the product takes 144-wide tiles with a
    single accumulator (one wave instead of two; round-toward-zero accumulation of 3x as many MMAs: ~3x the rounding
    error of the narrower tiles), whose H agrees to rounding."""
    from oracle import admm_oracle as orc
    torch.set_num_threads(4)
    g = torch.Generator().manual_seed(22)
    I, R = 512, 1141
    Bf, Cf = torch.randn(512, R, generator=g), torch.randn(9, R, generator=g)
    G = ((Bf.T @ Bf) * (Cf.T @ Cf)).cuda()
    F = (torch.randn(I, R, generator=g) * 30).cuda()
    H0 = torch.randn(I, R, generator=g)
    U0 = torch.randn(I, R, generator=g) * 0.1
    outs = []
    for ctas in (0, 36, 24, 7, 33):
        H, U = H0.clone().cuda(), U0.clone().cuda()
        rep = nat.admm_iteration_inplace(H, U, F, G, 11 if ctas != 33 else 2, 1e-8, 4, MSE, precision=1, max_ctas=ctas)
        assert nat.read_report(rep).iterations == (10 if ctas != 33 else 1)
        outs.append((H.cpu(), U.cpu()))
    for H, U in outs[1:4]:
        assert torch.equal(H, outs[0][0]) and torch.equal(U, outs[0][1])
    H1, U1 = H0.clone().cuda(), U0.clone().cuda()
    nat.admm_iteration_inplace(H1, U1, F, G, 2, 1e-8, 4, MSE, precision=1, max_ctas=36)
    wide, _ = _agreement(outs[4][0].numpy(), H1.cpu().numpy())
    assert wide >= 0.9995, wide
    Uo = U0.clone()
    Ho, Uo, _ = orc.admm_iteration(H0.clone(), Uo, F.cpu(), G.cpu(), 3, 1e-8, 4, MSE)
    H, U = H0.clone().cuda(), U0.clone().cuda()
    nat.admm_iteration_inplace(H, U, F, G, 3, 1e-8, 4, MSE, precision=1, max_ctas=36)
    agree, dscale = _agreement(H.cpu().numpy(), Ho.numpy())
    assert agree >= 0.999 and dscale <= 5e-6, (agree, dscale)
    torch.set_num_threads(1)


# ------------------------------------------------------------------ outer loop
@pytest.mark.parametrize("precision", [0, 1])
def test_outer_loop_against_reference_history(golden_outer, capsys, precision):
    from source.solver import LayerSolver
    go = golden_outer
    m = go.case("config1_short")
    W = dev(go["config1/W"])
    init = [dev(go[f"config1_short/init{k}"]) for k in range(3)]
    s = LayerSolver(W, init, m["bits"], m["qscheme"], max_iter_admm=m["max_iter_admm"], solve_precision=precision)
    for _ in range(m["sweeps"]):
        s.sweep()
    ref, refq = go["config1_short/loss"], go["config1_short/lossq"]
    rel = np.abs(np.array(s.loss_hist) - ref) / ref
    relq = np.abs(np.array(s.loss_quant_hist) - refq) / refq
    with capsys.disabled():
        print(f"\n[outer] precision {precision} rel. diff of rec_error per sweep:", np.array2string(rel, precision=2),
              "quant:", np.array2string(relq, precision=2))
    assert rel[0] <= 1e-3 and relq[0] <= 1e-3 and rel[1] <= 1e-3
    # From sweep 2 on the yardstick is the UNMODIFIED reference against itself on this very configuration when the output
    # of its own ridge solve is jittered by +-3e-7 / +-6e-8 per inner iteration (tests/golden/short_divergence.npz, made by
    # oracle/make_golden.py --only short_divergence: spread 2.9e-4, 7.9e-4, 3.6e-3, 3.1e-3 in sweeps 2 .. 5): every sweep
    # within north_star's 1e-3 or twice that spread, whichever is larger - no blanket bound.
    sd = np.load(os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "short_divergence.npz"))
    trials = [k for k in sd.files if k.startswith("trial") and k.endswith("/loss")]
    spread = np.max([np.abs(sd[k] - ref) / ref for k in trials], axis=0)
    spreadq = np.max([np.abs(sd[k + "q"] - refq) / refq for k in trials], axis=0)
    assert len(trials) == 8 and np.all(rel <= np.maximum(1e-3, 2 * spread)), (rel, spread)
    assert np.all(relq <= np.maximum(1e-3, 2 * spreadq)), (relq, spreadq)
    # 2-D branch
    mm = go.case("mat")
    s2 = LayerSolver(dev(go["mat/W"]), [dev(go["mat/init0"]), dev(go["mat/init1"])], mm["bits"], mm["qscheme"],
                     max_iter_admm=mm["max_iter_admm"], solve_precision=precision)
    for _ in range(mm["sweeps"]):
        s2.sweep()
    rel2 = np.abs(np.array(s2.loss_hist) - go["mat/loss"]) / go["mat/loss"]
    with capsys.disabled():
        print(f"[outer] precision {precision} 2-D case, rel. diff of rec_error per sweep:", np.array2string(rel2, precision=2))
    # the reference does not move on this case under the same jitter (mat_trial* of short_divergence.npz: <= 9e-8 in all
    # five sweeps), so every sweep is held to north_star's 1e-3
    spread2 = np.max([np.abs(sd[k] - go["mat/loss"]) / go["mat/loss"] for k in sd.files if k.startswith("mat_trial")], axis=0)
    assert spread2.max() <= 1e-6 and rel2.max() <= 1e-3, (rel2, spread2)


def test_outer_loop_with_tensor_core_mttkrp(golden_outer, capsys):
    """Throughput configuration (3xTF32 MTTKRP + 3xTF32 ridge product): the first three sweeps track the reference
    history within north_star's 1e-3 (the reference's own spread there is <= 2.9e-4, short_divergence.npz)."""
    from source.solver import LayerSolver
    go = golden_outer
    m = go.case("config1_short")
    W = dev(go["config1/W"])
    init = [dev(go[f"config1_short/init{k}"]) for k in range(3)]
    s = LayerSolver(W, init, m["bits"], m["qscheme"], max_iter_admm=m["max_iter_admm"], solve_precision=1, mttkrp_precision=1)
    for _ in range(3):
        s.sweep()
    rel = np.abs(np.array(s.loss_hist) - go["config1_short/loss"][:3]) / go["config1_short/loss"][:3]
    with capsys.disabled():
        print("\n[outer] throughput mode (tensor-core MTTKRP + ridge product), rel. diff of rec_error per sweep:", np.array2string(rel, precision=2))
    assert rel.max() <= 1e-3, rel


@pytest.mark.parametrize("precision", [0, 1])
def test_outer_loop_full_inner_budget_first_sweep(golden_outer, capsys, precision):
    """BASELINE config 1 with max_iter_admm = 1000, free-running first sweep (2997 inner iterations): rec_error within
    north_star's 1e-3 relative of the reference.  Yardsticks made from the UNMODIFIED reference: against itself with
    every MTTKRP output jittered by +-6e-8 it moves 1.3e-4 .. 1.6e-4 in sweep 0 (self_divergence.npz); with the OUTPUT
    OF ITS RIDGE SOLVE jittered by +-3e-7 per inner iteration (LAPACK potrs' own distance from the exact solution) it
    moves 3e-4 .. 6e-4 (solve_divergence.npz).  Precision 0 forms the correctly rounded solve (float64 product with
    the float64 inverse); round 1's float32 product (5.9e-7 from exact) was at 1.35e-3."""
    from source.solver import LayerSolver
    go = golden_outer
    W = dev(go["config1/W"])
    init = [dev(go[f"config1_full/init{k}"]) for k in range(3)]
    s = LayerSolver(W, init, 4, MSE, max_iter_admm=1000, solve_precision=precision)
    err, errq = s.sweep()
    ref, refq = float(go["config1_full/loss"][0]), float(go["config1_full/lossq"][0])
    sd = np.load(os.path.join(os.path.dirname(__file__), "golden", "self_divergence.npz"))
    self_div = max(abs(float(sd[f"trial{t}/loss"][0]) - ref) / ref for t in range(2))
    sv = np.load(os.path.join(os.path.dirname(__file__), "golden", "solve_divergence.npz"))
    solve_div = [abs(float(sv[f"trial{t}/loss"][0]) - ref) / ref for t in range(5)]
    with capsys.disabled():
        print(f"\n[outer-full] precision {precision} sweep 0: rec_error {err:.6f} vs reference {ref:.6f} (rel {abs(err - ref) / ref:.2e}); "
              f"quant {errq:.6f} vs {refq:.6f}; reference self-divergence: {self_div:.2e} under +-6e-8 jitter of F, "
              f"{min(solve_div):.1e}..{max(solve_div):.1e} under +-3e-7 jitter of the solve")
    assert abs(err - ref) <= 1e-3 * ref
    assert abs(errq - refq) <= 1e-3 * refq
    assert all(r.iterations == 999 for r in s.last_reports)  # the exit test never fires (SURVEY 0.2)


def test_c_level_outer_loop_equals_python_orchestration(nat, golden_outer):
    """admmq_factorize_cp3 / admmq_factorize_mat (the whole loop of scripts/factorize.py:207-310 in one C call) run
    the same kernels in the same order as source/solver.py::LayerSolver: identical histories and factors, stop rules
    included; and the first sweep matches the reference's recorded history."""
    from source import workloads as wl
    from source.solver import LayerSolver
    g = torch.Generator().manual_seed(5)
    for shape, R, sweeps, inner in [((24, 20, 9), 30, 4, 25), ((40, 28), 12, 12, 15)]:
        W = (torch.randn(*shape, generator=g) * 0.05).cuda()
        init = wl.random_init(shape, R, 7)
        for prec in (0, 1):
            s = LayerSolver(W, [f.cuda() for f in init], 4, MSE, max_iter_admm=inner, solve_precision=prec, mttkrp_precision=prec)
            n_py = s.run(sweeps)
            fac = [f.clone().cuda() for f in init]
            du = [torch.zeros_like(f) for f in fac]
            hist, histq, n_c, fq = nat.factorize(W, fac, du, 4, MSE, sweeps, inner, solve_precision=prec, mttkrp_precision=prec)
            assert n_c == n_py and hist == s.loss_hist and histq == s.loss_quant_hist, (shape, prec, hist, s.loss_hist)
            for a, b in zip(fac + du + fq, s.factors + s.duals + s.factors_q):
                assert torch.equal(a, b)
    # non-random init: one leading history entry (scripts/factorize.py:192-201)
    W = (torch.randn(16, 12, 9, generator=g) * 0.05).cuda()
    fac = [f.cuda() for f in wl.random_init((16, 12, 9), 10, 3)]
    hist, histq, n, _ = nat.factorize(W, fac, [torch.zeros_like(f) for f in fac], 4, MSE, 2, 10, init_is_random=False)
    assert n == 2 and len(hist) == 3 and len(histq) == 3
    with pytest.raises(ValueError):
        nat.factorize(W, fac, [torch.zeros_like(f) for f in fac], 9, MSE, 2, 10)
    # the reference's recorded history (config 1, short budget) through the C entry point
    go = golden_outer
    m = go.case("config1_short")
    fac = [dev(go[f"config1_short/init{k}"]) for k in range(3)]
    hist, _, n, _ = nat.factorize(dev(go["config1/W"]), fac, [torch.zeros_like(f) for f in fac], m["bits"], m["qscheme"],
                                  m["sweeps"], m["max_iter_admm"], tol=0.0)
    ref = go["config1_short/loss"]
    assert n == m["sweeps"] and abs(hist[0] - ref[0]) <= 1e-3 * ref[0] and abs(hist[1] - ref[1]) <= 1e-3 * ref[1]


def test_batched_solves_equal_individual_calls(nat):
    """admmq_factorize_batch: independent problems (two tensors, one matrix; different ranks, bit-widths, budgets and
    stop points) interleaved sweep by sweep on their own streams give exactly what one call per problem gives."""
    from source import workloads as wl
    g = torch.Generator().manual_seed(8)
    specs = [((24, 20, 9), 30, 4, 5, 20, 3), ((32, 16, 9), 17, 3, 3, 15, 2), ((40, 28), 12, 8, 12, 12, 0)]
    jobs, ref = [], []
    for shape, R, bits, sweeps, inner, ctas in specs:
        W = (torch.randn(*shape, generator=g) * 0.05).cuda()
        init = wl.random_init(shape, R, 11)
        fa = [f.clone().cuda() for f in init]
        da = [torch.zeros_like(f) for f in fa]
        ref.append((nat.factorize(W, fa, da, bits, MSE, sweeps, inner, solve_precision=1, mttkrp_precision=1, max_ctas=ctas), fa, da))
        fb = [f.clone().cuda() for f in init]
        jobs.append(dict(W=W, factors=fb, duals=[torch.zeros_like(f) for f in fb], bits=bits, qscheme=MSE, max_iter_als=sweeps,
                         max_iter_admm=inner, solve_precision=1, mttkrp_precision=1, max_ctas=ctas))
    out = nat.factorize_batch(jobs)
    torch.cuda.synchronize()
    for (hist, histq, n, fq), ((rh, rhq, rn, rfq), fa, da), job in zip(out, ref, jobs):
        assert n == rn and hist == rh and histq == rhq
        for a, b in zip(job["factors"] + job["duals"] + fq, fa + da + rfq):
            assert torch.equal(a, b)


def test_two_block_splitting_quantized_block_bit_exact(nat):
    """admmq_split_loop (quantized block of scripts/factorize_lowrank.py:84-101) against the CPU restatement: the
    least-squares step is elementwise in the reference's operation order and the projection is bit-exact, so H and U
    agree BIT FOR BIT up to the common exit iteration for the grid-from-min/max schemes, and codes agree for the clip search."""
    from oracle import lowrank_oracle as lo
    from source.lowrank import admm_iteration_quantized, factorize_lowrank, project_rank
    torch.set_num_threads(1)
    g = torch.Generator().manual_seed(21)
    for shape, bits, qs in [((96, 80), 4, "tensor_minmax"), ((64, 48), 3, "tensor_symmetric"), ((50, 70), 8, "tensor_affine"),
                            ((120, 64), 4, MSE)]:
        W = torch.randn(*shape, generator=g) * 0.02
        H = torch.randn(*shape, generator=g)
        H2 = lo.project_rank(torch.randn(*shape, generator=g), 4) * 0.01
        U = torch.zeros(*shape)
        trace = []
        Hr, Ur = lo.admm_iteration(H.clone(), U.clone(), W, H2, lo.quantize_func(bits, qs), rho=1.0, max_iter=50, trace=trace)
        Ud = U.clone().cuda()
        Hd, Ud2, rep = admm_iteration_quantized(H.cuda(), Ud, W.cuda(), H2.cuda(), bits, qs, rho=1.0, max_iter=50)
        assert Ud2 is Ud                                            # U updated in place, like the reference
        r = nat.read_report(rep)
        assert r.iterations == len(trace), (shape, qs, r.iterations, len(trace))   # same exit iteration (:97)
        if qs == MSE:
            same = (Hd.cpu() == Hr).float().mean().item()
            assert same >= 0.999, (shape, same)
        else:
            assert bits_equal(Hd.cpu().numpy(), Hr.numpy()), (shape, qs)
            assert bits_equal(Ud.cpu().numpy(), Ur.numpy()), (shape, qs)
    # outer loop (scripts/factorize_lowrank.py:130-170) against the same loop on the CPU restatement, from the same start
    Wb = torch.randn(64, 48, generator=g) * 0.02
    torch.manual_seed(1)
    Wq0, Wr0 = torch.randn(64, 48), lo.project_rank(torch.randn(64, 48), 6)
    Wq, Uq, Wr, Ur = Wq0.clone(), torch.zeros(64, 48), Wr0.clone(), torch.zeros(64, 48)
    ref_hist = []
    for _ in range(3):
        Wq, Uq = lo.admm_iteration(Wq, Uq, Wb, Wr, lo.quantize_func(4, "tensor_minmax"), max_iter=20)
        Wr, Ur = lo.admm_iteration(Wr, Ur, Wb, Wq, lambda X: lo.project_rank(X, 6), max_iter=20)
        ref_hist.append(float(torch.linalg.norm(Wb - Wr - Wq) / torch.linalg.norm(Wb)))
    from source.lowrank import admm_iteration_projected
    Wd = Wb.cuda()
    Wq, Uq, Wr, Ur = Wq0.cuda(), torch.zeros(64, 48).cuda(), Wr0.cuda(), torch.zeros(64, 48).cuda()
    hist = []
    for _ in range(3):
        Wq, Uq, _ = admm_iteration_quantized(Wq, Uq, Wd, Wr, 4, "tensor_minmax", max_iter=20)
        Wr, Ur = admm_iteration_projected(Wr, Ur, Wd, Wq, lambda X: project_rank(X, 6), max_iter=20)
        hist.append(float(torch.linalg.norm(Wd - Wr - Wq) / torch.linalg.norm(Wd)))
    assert np.allclose(hist, ref_hist, rtol=2e-3), (hist, ref_hist)
    sv = torch.linalg.svdvals(Wr.double())
    assert hist[-1] < hist[0] and float(sv[6]) <= 1e-5 * float(sv[0])   # W_r keeps rank 6 (to float32 rounding)
    W_q, W_r, h2 = factorize_lowrank(Wd, 4, 6, "tensor_minmax", max_iter=2, seed=1, inner_max_iter=10)
    assert len(h2) == 2 and W_q.shape == Wd.shape and W_r.shape == Wd.shape
    assert torch.unique(W_q).numel() <= 16
    torch.set_num_threads(1)


# ------------------------------------------------------------------ model level (north_star: top-1 on synthetic-calibrated weights)
class _PrototypeTask:
    """10-class synthetic image task with a real decision margin: class prototype + unit Gaussian noise."""

    def __init__(self, n_batches, batch_size, seed, device="cuda"):
        self.n_batches, self.batch_size, self.seed, self.device = n_batches, batch_size, seed, device
        self.protos = torch.randn(10, 3, 32, 32, generator=torch.Generator().manual_seed(1234))

    def __iter__(self):
        g = torch.Generator().manual_seed(self.seed)
        for _ in range(self.n_batches):
            y = torch.randint(0, 10, (self.batch_size,), generator=g)
            x = 1.0 * self.protos[y] + torch.randn(self.batch_size, 3, 32, 32, generator=g)
            yield x.to(self.device), y.to(self.device)


@pytest.mark.parametrize("precision", [0, 1])
def test_model_top1_with_our_factors_vs_reference_factors(capsys, precision):
    """north_star: "ResNet-18 top-1 must stay within 0.1 pp on synthetic-calibrated weights".  A ResNet-18 is trained
    for a few steps on a synthetic 10-class task (no dataset or checkpoint exists offline), its four layer1
    convolutions are factorized with the CPU oracle (2 sweeps x 30 inner iterations, random init) and with the CUDA
    solver; every factor set goes through source/models.py into a CP model, is BN-calibrated on the same synthetic images
    (source/utils.py) and scored on 16384 held-out images.

    The solver is chaotic at the 1-ulp level from the second sweep on (SURVEY 0.6: one flipped code never heals), so two
    runs that are not bit-identical - including the reference against itself from an init perturbed by half a float32
    ulp - end in different, equally good factor sets whose models differ by +-0.2 pp.  The 0.1 pp requirement is therefore
    asserted the way code parity is (SURVEY 8(c)): TEACHER-FORCED AT THE SWEEP BOUNDARY - the CUDA solver runs the last
    sweep from the reference's own state (factors and duals after sweep 1).  The free-running CUDA result is reported
    next to the band the reference spans against itself, with a loose bound."""
    import copy
    import torchvision
    from oracle import admm_oracle as orc
    from source import workloads as wl
    from source.models import get_submodule, replace_with_cp
    from source.solver import LayerSolver, layer_weight_as_tensor, rank_from_reduction_rate
    from source.utils import bncalibrate_model, top1_accuracy
    torch.set_num_threads(4)   # (8 threads crawled on a contended GPU box: OpenMP oversubscription)
    torch.manual_seed(42)
    torch.backends.cudnn.deterministic, torch.backends.cudnn.benchmark = True, False   # reproducible training run
    base = torchvision.models.resnet18(weights=None, num_classes=10).cuda()
    opt = torch.optim.SGD(base.parameters(), lr=0.05, momentum=0.9)
    base.train()
    for x, y in _PrototypeTask(120, 128, seed=5):
        opt.zero_grad()
        torch.nn.functional.cross_entropy(base(x), y).backward()
        opt.step()
    base.eval()
    acc_base = top1_accuracy(base, _PrototypeTask(32, 64, seed=2), "cuda")
    forced, free, ref = copy.deepcopy(base), copy.deepcopy(base), copy.deepcopy(base)
    variants = [copy.deepcopy(base) for _ in range(3)]   # the reference against itself: init * (1 +- 6e-8)
    errs, agree = [], []
    for path in ("layer1.0.conv1", "layer1.0.conv2", "layer1.1.conv1", "layer1.1.conv2"):
        W = layer_weight_as_tensor(get_submodule(base, path).weight.detach()).contiguous()
        R = rank_from_reduction_rate(W, 2.0)
        init = wl.random_init(W.shape, R, 42)
        fac1, _, _, _, duals1 = orc.factorize(W.cpu(), init, 4, MSE, 1, 30, stop_rules=False)     # reference state after sweep 1
        fac, _, loss, _, _ = orc.factorize(W.cpu(), init, 4, MSE, 2, 30, stop_rules=False)        # ... and after sweep 2
        replace_with_cp(ref, path, fac, R)
        # free-running CUDA solver
        s = LayerSolver(W, [f.cuda() for f in init], 4, MSE, max_iter_admm=30, solve_precision=precision,
                        mttkrp_precision=precision)
        for _ in range(2):
            s.sweep()
        replace_with_cp(free, path, [f.clone() for f in s.factors], R)
        # last sweep from the reference's state
        t = LayerSolver(W, [f.cuda() for f in fac1], 4, MSE, max_iter_admm=30, solve_precision=precision,
                        mttkrp_precision=precision)
        for d, src in zip(t.duals, duals1):
            d.copy_(src)
        t.sweep()
        replace_with_cp(forced, path, [f.clone() for f in t.factors], R)
        errs.append((round(t.loss_hist[-1], 5), round(s.loss_hist[-1], 5), round(loss[-1], 5)))
        agree.append(min(_agreement(a.cpu().numpy(), b.numpy())[0] for a, b in zip(t.factors, fac)))
        for v, model in enumerate(variants):
            gj = torch.Generator().manual_seed(1000 + v)
            jit = [f * (1 + 6e-8 * (torch.randint(0, 2, f.shape, generator=gj).float() * 2 - 1)) for f in init]
            fv, _, _, _, _ = orc.factorize(W.cpu(), jit, 4, MSE, 2, 30, stop_rules=False)
            replace_with_cp(model, path, fv, R)
    accs = []
    for m in [forced, free, ref] + variants:
        bncalibrate_model(m, _PrototypeTask(18, 64, seed=1), num_samples=1000, device="cuda")
        accs.append(top1_accuracy(m, _PrototypeTask(128, 128, seed=2), "cuda"))
    a_forced, a_free, a_ref = accs[:3]
    with capsys.disabled():
        print(f"\n[top-1] precision {precision}: uncompressed {acc_base:.2f} %; CP model from the reference's factors {a_ref:.2f} %; "
              f"from our factors, last sweep from the reference's state {a_forced:.2f} % (code agreement per layer "
              f"{[round(a, 5) for a in agree]}); free-running {a_free:.2f} %; reference re-run from half-ulp-jittered inits "
              f"{', '.join(f'{a:.2f}' for a in accs[3:])} % (16384 held-out synthetic images, 4-bit, rr = 2, BN-calibrated); "
              f"rec_error forced / free / reference per layer {errs}")
    assert acc_base >= 95.0                      # the synthetic task was learnt: the labels carry a margin
    lo, hi = min(accs[2:]), max(accs[2:])        # the reference against itself (unperturbed + half-ulp-jittered inits)
    if precision == 0:
        # parity mode: north_star's code and top-1 criteria, teacher-forced at the sweep boundary
        for ef, es, l in errs:
            assert abs(ef - l) <= 1e-3 * l and abs(es - l) <= 5e-3 * l
        assert min(agree) >= 0.999               # final code agreement >= 99.9 %
        assert abs(a_forced - a_ref) <= 0.1      # top-1 within 0.1 pp
    else:
        # throughput mode: a single flipped code early in the sweep can separate one layer's trajectory within the sweep
        # (measured: 3 of 4 layers bit-identical, one at 81 %); the models stay inside the band the reference spans
        # against itself
        for ef, es, l in errs:
            assert abs(ef - l) <= 5e-3 * l and abs(es - l) <= 5e-3 * l
        assert sorted(agree)[len(agree) // 2] >= 0.999
        assert lo - 0.1 <= a_forced <= hi + 0.1
    assert lo - 0.5 <= a_free <= hi + 0.5        # free-running: different, equally good local solutions
    torch.set_num_threads(1)


# ------------------------------------------------------------------ CLI and file contract (SURVEY 8(a) a15, 8(b))
def test_factorize_cli_writes_the_reference_file_set(tmp_path, monkeypatch):
    """scripts/factorize.py: flags, output directory and file names of the reference (:164-166, 315-318, 345-347) and
    the consumer side (scripts/calibrate.py) reading exactly those files."""
    import importlib.util
    monkeypatch.chdir(tmp_path)
    def load(name):
        spec = importlib.util.spec_from_file_location(name, os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))),
                                                                         "admm-quantization_b200", "scripts", name + ".py"))
        mod = importlib.util.module_from_spec(spec)
        spec.loader.exec_module(mod)
        return mod
    fz = load("factorize")
    err, errq = fz.main(["--model-name", "resnet18", "--method", "admm", "--init", "random", "--layer", "layer1.0.conv1",
                         "--reduction-rate", "2", "--bits", "4", "--qscheme", MSE, "--seed", "42",
                         "--max_iter_als", "2", "--max_iter_admm", "20", "--weights", "random",
                         "--outdir", f"4bit_{MSE}/factors_admm_seed42"])
    d = tmp_path / f"4bit_{MSE}" / "factors_admm_seed42"
    names = sorted(p.name for p in d.iterdir())
    prefix = "layer1.0.conv1_admm_random_rank_134_"
    assert names == sorted(prefix + s for s in ("losshist.pt", "lossquanthist.pt", "mode_0.pt", "mode_1.pt", "mode_2.pt"))
    shapes = [tuple(torch.load(d / (prefix + f"mode_{m}.pt")).shape) for m in range(3)]
    assert shapes == [(64, 134), (64, 134), (9, 134)]
    assert torch.load(d / (prefix + "mode_0.pt")).dtype == torch.float32
    hist = torch.load(d / (prefix + "losshist.pt"))
    assert len(hist) == 2 and 0.5 < hist[-1] < 1.0 and abs(err - hist[-1]) < 1e-3 and abs(errq - err) < 1e-2
    with pytest.raises(SystemExit):
        fz.parse_args(["--model-name", "resnet18"])                       # required flags (:38-102)
    # the reference loads the PRETRAINED model: that is the default, and without network / cache it fails loudly instead
    # of factorizing random weights under the reference's file names.  The checkpoint fetch is replaced by one that
    # fails the way it does offline, so the test neither reads the user's download cache nor reaches the network.
    base = ["--model-name", "resnet18", "--method", "admm", "--layer", "layer1.0.conv1", "--reduction-rate", "2", "--bits", "4",
            "--qscheme", MSE, "--seed", "42"]
    assert fz.parse_args(base).weights == "pretrained"
    import torchvision.models._api

    def offline(url, *_a, **_k):
        raise OSError(f"no network and no cached checkpoint for {url}")
    monkeypatch.setattr(torchvision.models._api, "load_state_dict_from_url", offline)
    with pytest.raises(RuntimeError, match="pretrained"):
        fz.main(base + ["--max_iter_als", "1", "--max_iter_admm", "5"])
    acc = load("calibrate").main(["--bits", "4", "--qscheme", MSE, "--seed", "42", "--layers", "layer1.0.conv1",
                                  "--eval-batches", "2", "--batch-size", "16", "--calibration-samples", "32"])
    assert 0.0 <= acc <= 100.0
