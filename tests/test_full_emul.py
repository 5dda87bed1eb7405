"""The whole C ABI on the CPU under the SIMT emulator (tests/emul_lib.py, tests/host_emul): csrc/vggp.cu with its 45
kernel launches rewritten, every kernel of csrc/*.cuh compiled unchanged by g++.  The same oracle parity checks the GPU
suite makes (tests/test_gpu_elbo.py) are made here at small sizes.  Two purposes:
  * the emulator is validated on the paths that passed on B200 (raw / packed layouts, the fused B1 grid side and the
    dense grid side of the B0 / SVGP / VFF families, DMMA and SIMT GEMMs);
  * the paths that have NOT run on a GPU yet -- the binned layout end to end through vggp_obs_bin_prepare / _pack /
    vggp_obs_fwd_bwd_binned, both streaming variants -- get the same parity check before their first GPU run.
Test infrastructure only; the product library has no CPU path."""
import numpy as np
import pytest
import torch

import emul_lib
from oracle import vggp_oracle as O
from test_gpu_elbo import make_problem, oracle_value_and_grads


@pytest.fixture(scope="module")
def emu():
    got = emul_lib.load()
    if got is None:
        pytest.skip("g++ not available")
    return got


def relerr(a, b):
    a = np.asarray(a, dtype=np.float64).reshape(-1)
    b = b.detach().cpu().to(torch.float64).reshape(-1).numpy()
    return float(np.linalg.norm(a - b) / max(np.linalg.norm(b), 1e-300))


def check_against_oracle(plan, out, dtheta, dm, dL, elbo_ref, g_ref, N, tol):
    D = plan.D
    assert plan.read_info() == 0
    assert out[3] == N
    assert abs(out[0] - elbo_ref.item()) <= tol * abs(elbo_ref.item()), (out, elbo_ref)
    assert relerr(dtheta[:D], g_ref[0]) < tol * 10
    assert relerr(dtheta[D:2 * D], g_ref[1]) < tol * 10
    assert relerr(dtheta[2 * D], g_ref[2]) < tol * 10
    assert relerr(dm, g_ref[3]) < tol * 10
    off = 0
    for d, n in enumerate(plan.m_per_dim):
        dLd = dL[off:off + n * n].reshape(n, n)
        off += n * n
        assert np.count_nonzero(np.triu(dLd, 1)) == 0
        assert relerr(np.tril(dLd), torch.tril(g_ref[4 + d])) < tol * 10, ("dL", d)


B1_CASES = [((12,), 500), ((9, 7), 700), ((6, 14, 5), 900)]
LAYOUTS = ["raw", "packed_sorted", "packed_unsorted", "binned_ldg", "binned_tma"]


@pytest.mark.parametrize("layout", LAYOUTS)
@pytest.mark.parametrize("knots,N", B1_CASES)
@pytest.mark.parametrize("dtype,tol", [(np.float64, 1e-9), (np.float32, 1e-3)])
def test_b1_step_matches_oracle_under_emulation(emu, knots, N, dtype, tol, layout):
    lib, L = emu
    D = len(knots)
    meshes, X, y, l, s2, noise, m, Ls = make_problem(knots, N, seed=42 + D)
    tdt = torch.float64 if dtype == np.float64 else torch.float32
    Xq, yq = X.to(tdt), y.to(tdt)
    scale = 1.7
    elbo_ref, g_ref = oracle_value_and_grads(O.B1_ASVGP, meshes, Xq.to(torch.float64), yq.to(torch.float64),
                                             l, s2, noise, m, Ls, scale=scale)
    plan = emul_lib.EmuPlan(lib, L, L.B1_ASVGP, [t.numpy() for t in meshes], dtype)
    theta = torch.cat([l, s2, noise.reshape(1)]).numpy().copy()
    mm = m.numpy().copy()
    Lcat = torch.cat([Lx.reshape(-1) for Lx in Ls]).numpy().copy()
    xs = [np.ascontiguousarray(Xq[:, d].numpy()) for d in range(D)]
    yy = np.ascontiguousarray(yq.numpy())
    lib.vggp_set_binned_stream(1 if layout == "binned_tma" else 0)
    try:
        if layout == "raw":
            out, dtheta, dm, dL = plan.step(theta, mm, Lcat, xs, yy, ell_scale=scale)
        elif layout.startswith("packed"):
            out, dtheta, dm, dL = plan.step(theta, mm, Lcat, plan.pack(xs, yy, layout == "packed_sorted"), None, scale)
        else:
            binned = plan.bin(xs, yy, run_cap=16)
            assert binned[2].n == N and binned[2].n_tasks == (binned[2].n_runs + 31) // 32
            out, dtheta, dm, dL = plan.step(theta, mm, Lcat, binned, None, scale)
        check_against_oracle(plan, out, dtheta, dm, dL, elbo_ref, g_ref, N, tol)
    finally:
        lib.vggp_set_binned_stream(0)
        plan.close()


@pytest.mark.parametrize("knots,N", [((600,), 900), ((70, 45), 1500), ((40, 33, 35), 1200)])
def test_fused_grid_side_larger_meshes_under_emulation(emu, knots, N):
    """csrc/grid_b1.cuh beyond the small meshes above: several chunks in the generator scan (k_b1_gens), lanes owning more
    than 16 elements of a fibre (600 knots: the shared-memory sweep of fp_fibre), tiles that straddle fibres of different
    outer index (3-D middle mode), partial tiles."""
    lib, L = emu
    D = len(knots)
    meshes, X, y, l, s2, noise, m, Ls = make_problem(knots, N, seed=77 + D)
    elbo_ref, g_ref = oracle_value_and_grads(O.B1_ASVGP, meshes, X, y, l, s2, noise, m, Ls, scale=1.3)
    plan = emul_lib.EmuPlan(lib, L, L.B1_ASVGP, [t.numpy() for t in meshes], np.float64)
    theta = torch.cat([l, s2, noise.reshape(1)]).numpy().copy()
    xs = [np.ascontiguousarray(X[:, d].numpy()) for d in range(D)]
    out, dtheta, dm, dL = plan.step(theta, m.numpy().copy(), torch.cat([Lx.reshape(-1) for Lx in Ls]).numpy().copy(),
                                    plan.bin(xs, y.numpy().copy(), run_cap=64), None, 1.3)
    check_against_oracle(plan, out, dtheta, dm, dL, elbo_ref, g_ref, N, 1e-9)
    plan.close()


def test_fast_and_generic_fibre_kernels_agree_under_emulation(emu):
    """k_fibre_pass_fast (M_d <= 512, the default) against the generic k_fibre_pass on the same step (2-D and 3-D, sizes that
    leave partial tiles, partial lanes and absent fibres)."""
    lib, L = emu
    # the power-of-two meshes fill their window of the 512-slot row exactly: full tiles take the SIMPLE specialisation of
    # ff_pass_body (validity = slot < 512, addresses in arithmetic progression), partial ones the general form
    for knots, N in (((37, 50), 1200), ((21, 13, 18), 900), ((300,), 700), ((70, 130), 1500), ((9, 200, 33), 1500),
                     ((64, 128), 1500), ((16, 64, 8), 900), ((512,), 700), ((64, 9), 700)):
        D = len(knots)
        meshes, X, y, l, s2, noise, m, Ls = make_problem(knots, N, seed=5 + D)
        theta = torch.cat([l, s2, noise.reshape(1)]).numpy().copy()
        xs = [np.ascontiguousarray(X[:, d].numpy()) for d in range(D)]
        res = []
        # 5 = fast kernel with fibre packing forced (2, 4 or 8 fibres per 512-slot row: contiguous and strided modes, windows
        # wider than n, partial rows and tiles), 3 = fast kernel without packing, 0 = generic kernel
        for fast in (5, 3, 0):
            lib.vggp_debug_fp_fast(fast)
            try:
                plan = emul_lib.EmuPlan(lib, L, L.B1_ASVGP, [t.numpy() for t in meshes], np.float64)
                res.append(plan.step(theta, m.numpy().copy(), torch.cat([Lx.reshape(-1) for Lx in Ls]).numpy().copy(),
                                     plan.bin(xs, y.numpy().copy(), run_cap=64), None, 1.1))
                plan.close()
            finally:
                lib.vggp_debug_fp_fast(1)
        for other in res[:2]:
            for a, b in zip(other, res[2]):
                assert relerr(a, torch.from_numpy(np.asarray(b, dtype=np.float64))) < 1e-11


@pytest.mark.parametrize("layout", ["packed_sorted", "binned_ldg"])
def test_two_wave_run_length_under_emulation(emu, layout):
    """Enough observations that the packed layout needs two waves of chunks per resident warp (the emulated device
    has 24 resident warps): run length and chunk count come out balanced, and the step still matches the oracle."""
    import ctypes as C
    lib, L = emu
    knots, N = (33,), 420000
    meshes, X, y, l, s2, noise, m, Ls = make_problem(knots, N, seed=17)
    Xq, yq = X.to(torch.float32), y.to(torch.float32)
    elbo_ref, g_ref = oracle_value_and_grads(O.B1_ASVGP, meshes, Xq.to(torch.float64), yq.to(torch.float64),
                                             l, s2, noise, m, Ls, scale=1.0)
    plan = emul_lib.EmuPlan(lib, L, L.B1_ASVGP, [t.numpy() for t in meshes], np.float32)
    npk, run = C.c_int64(), C.c_int()
    plan.check(lib.vggp_obs_pack_geometry(plan.h, N, C.byref(npk), C.byref(run)))
    chunks = npk.value // (32 * run.value)
    assert run.value % 4 == 0 and run.value < 512 and 44 <= chunks <= 48          # just below 2 x 24 warps
    theta = torch.cat([l, s2, noise.reshape(1)]).numpy().copy()
    xs = [np.ascontiguousarray(Xq[:, 0].numpy())]
    yy = np.ascontiguousarray(yq.numpy())
    obs = plan.pack(xs, yy, True) if layout == "packed_sorted" else plan.bin(xs, yy, run_cap=256)
    out, dtheta, dm, dL = plan.step(theta, m.numpy().copy(), Ls[0].reshape(-1).numpy().copy(), obs, None, 1.0)
    check_against_oracle(plan, out, dtheta, dm, dL, elbo_ref, g_ref, N, 1e-3)
    plan.close()


@pytest.mark.parametrize("knots,N", [((11,), 300), ((8, 7), 300)])
def test_b0_family_under_emulation(emu, knots, N):
    lib, L = emu
    D = len(knots)
    meshes, X, y, l, s2, noise, m, Ls = make_problem(knots, N, seed=3, family=O.B0_GRIDDED)
    elbo_ref, g_ref = oracle_value_and_grads(O.B0_GRIDDED, meshes, X, y, l, s2, noise, m, Ls, scale=1.0)
    plan = emul_lib.EmuPlan(lib, L, L.B0_GRIDDED, [t.numpy() for t in meshes], np.float64)
    theta = torch.cat([l, s2, noise.reshape(1)]).numpy().copy()
    xs = [np.ascontiguousarray(X[:, d].numpy()) for d in range(D)]
    out, dtheta, dm, dL = plan.step(theta, m.numpy().copy(), torch.cat([Lx.reshape(-1) for Lx in Ls]).numpy().copy(),
                                    xs, y.numpy().copy(), 1.0)
    check_against_oracle(plan, out, dtheta, dm, dL, elbo_ref, g_ref, N, 1e-8)
    plan.close()


@pytest.mark.parametrize("knots,N", [((11,), 300), ((8, 7), 300), ((70, 6), 250)])
@pytest.mark.parametrize("dtype,tol", [(np.float64, 1e-8), (np.float32, 1e-3)])
def test_svgp_product_grid_family_under_emulation(emu, knots, N, dtype, tol):
    """Product-grid SVGP (kronecker_structure.py:287-338, Matern12SVGP): inducing points on non-uniform per-dimension grids,
    features s2 exp(-|x - z_i| / l), Kuu_d the kernel matrix of the points; the whole step (dense Cholesky path, dense-feature
    per-observation kernel with the feature-path hyper-parameter gradients) against the oracle, observations outside the hull
    of the inducing points included."""
    lib, L = emu
    D = len(knots)
    meshes, X, y, l, s2, noise, m, Ls = make_problem(knots, N, seed=13 + D, family=O.SVGP_GRID, x_lo=-0.2, x_hi=1.2)
    meshes = [(t ** (1.0 + 0.3 * d)).to(torch.float32) for d, t in enumerate(meshes)]          # strictly increasing, non-uniform
    tdt = torch.float64 if dtype == np.float64 else torch.float32
    Xq, yq = X.to(tdt), y.to(tdt)
    elbo_ref, g_ref = oracle_value_and_grads(O.SVGP_GRID, meshes, Xq.to(torch.float64), yq.to(torch.float64), l, s2, noise, m, Ls, scale=1.1)
    plan = emul_lib.EmuPlan(lib, L, L.SVGP_GRID, [t.numpy() for t in meshes], dtype)
    assert plan.m_per_dim == list(knots)
    theta = torch.cat([l, s2, noise.reshape(1)]).numpy().copy()
    xs = [np.ascontiguousarray(Xq[:, d].numpy()) for d in range(D)]
    out, dtheta, dm, dL = plan.step(theta, m.numpy().copy(), torch.cat([Lx.reshape(-1) for Lx in Ls]).numpy().copy(),
                                    xs, np.ascontiguousarray(yq.numpy()), 1.1)
    check_against_oracle(plan, out, dtheta, dm, dL, elbo_ref, g_ref, N, tol)
    # the exported dense features are the oracle's
    phi = plan.features_dense(0, xs[0], theta)
    ref = O.svgp_features_dense(meshes[0], Xq[:, 0], l[0], s2[0]).numpy()
    assert np.max(np.abs(phi - ref)) <= (1e-13 if dtype == np.float64 else 1e-6) * np.max(np.abs(ref))
    plan.close()


@pytest.mark.parametrize("knots,N", [((9,), 300), ((7, 11), 300), ((71, 5), 250)])
@pytest.mark.parametrize("dtype,tol", [(np.float64, 1e-8), (np.float32, 1e-3)])
def test_vff_family_under_emulation(emu, knots, N, dtype, tol):
    """Variational Fourier features (kronecker_structure.py:347-514 Matern12VFFGP, fourier.py:58-88): cosines / sines on a domain
    smaller than the data (so the exp(-r / l) branch outside [a, b) and its lengthscale gradient are exercised), Kuu_d =
    diag(alpha) + beta beta^T through the dense Cholesky path; the whole step against the oracle (float64 semantics)."""
    lib, L = emu
    D = len(knots)
    meshes, X, y, l, s2, noise, m, Ls = make_problem(knots, N, seed=17 + D, family=O.VFF_GRID, x_lo=-0.2, x_hi=1.2)
    tdt = torch.float64 if dtype == np.float64 else torch.float32
    Xq, yq = X.to(tdt), y.to(tdt)
    Xq[::7, 0] = 0.0                                   # on the lower end of the domain (inside), and on the upper end (outside)
    Xq[3::11, D - 1] = 1.0
    elbo_ref, g_ref = oracle_value_and_grads(O.VFF_GRID, meshes, Xq.to(torch.float64), yq.to(torch.float64), l, s2, noise, m, Ls, scale=1.2)
    plan = emul_lib.EmuPlan(lib, L, L.VFF_GRID, [t.numpy() for t in meshes], dtype)
    assert plan.m_per_dim == list(knots)
    theta = torch.cat([l, s2, noise.reshape(1)]).numpy().copy()
    xs = [np.ascontiguousarray(Xq[:, d].numpy()) for d in range(D)]
    out, dtheta, dm, dL = plan.step(theta, m.numpy().copy(), torch.cat([Lx.reshape(-1) for Lx in Ls]).numpy().copy(),
                                    xs, np.ascontiguousarray(yq.numpy()), 1.2)
    check_against_oracle(plan, out, dtheta, dm, dL, elbo_ref, g_ref, N, tol)
    phi = plan.features_dense(0, xs[0], theta)
    ref = O.vff_features_dense(meshes[0], Xq[:, 0], l[0], s2[0], ref_quirks=False).numpy()
    assert np.max(np.abs(phi - ref)) <= (1e-12 if dtype == np.float64 else 2e-5)
    plan.close()


@pytest.mark.parametrize("name", ["lin11_01", "lin129_01", "lin16_02", "lin21_m3_7", "padded21_pad2"])
@pytest.mark.parametrize("tag,dtype", [("f64", np.float64), ("f32", np.float32)])
def test_b1_stencil_kernel_bit_exact_vs_reference_golden(emu, golden_dir, name, tag, dtype):
    """k_b1_stencil / k_b1_dense (emulated with -ffp-contract=off, IEEE float arithmetic) against the fixtures produced by
    the reference's own bspline.py: identical cell index and identical weight bits."""
    import os
    lib, L = emu
    sten = np.load(os.path.join(golden_dir, "b1_stencil.npz"))
    mesh, x, phi_ref = sten[f"{name}.{tag}.mesh"], sten[f"{name}.{tag}.x"], sten[f"{name}.{tag}.phi"]
    plan = emul_lib.EmuPlan(lib, L, L.B1_ASVGP, [mesh], dtype)
    phi = plan.features_dense(0, x)
    assert phi.dtype == phi_ref.dtype and np.array_equal(phi, phi_ref)
    c, wl, wh = plan.b1_stencil(0, x)
    co, wlo, who = O.b1_stencil(torch.from_numpy(mesh), torch.from_numpy(x))
    assert np.array_equal(c.astype(np.int64), co.numpy())
    assert np.array_equal(wl, wlo.numpy()) and np.array_equal(wh, who.numpy())
    plan.close()


def test_point_prediction_under_emulation(emu):
    """k_predict_b1 against the dense formulas mean = phi^T alpha, var = kff - phi^T P phi + phi^T Q phi built from the
    workspace-independent oracle pieces."""
    lib, L = emu
    knots, N = (9, 7), 400
    meshes, X, y, l, s2, noise, m, Ls = make_problem(knots, N, seed=8)
    plan = emul_lib.EmuPlan(lib, L, L.B1_ASVGP, [t.numpy() for t in meshes], np.float64)
    theta = torch.cat([l, s2, noise.reshape(1)]).numpy().copy()
    plan.grid_forward(theta, m.numpy().copy(), torch.cat([Lx.reshape(-1) for Lx in Ls]).numpy().copy())
    xs = [np.ascontiguousarray(X[:, d].numpy()) for d in range(2)]
    mean, var = plan.predict(xs)
    Ks = [O.kuu_factor(O.B1_ASVGP, meshes[d], l[d], s2[d], ref_quirks=False) for d in range(2)]
    Ps = [torch.linalg.inv(K) for K in Ks]
    Ss = [torch.tril(Lx) @ torch.tril(Lx).T for Lx in Ls]
    Qs = [P @ S @ P for P, S in zip(Ps, Ss)]
    alpha = (Ps[0] @ m.reshape(9, 7) @ Ps[1].T)
    phis = [O.b1_features_dense(meshes[d], X[:, d]) for d in range(2)]          # (M_d, N)
    mu_ref = torch.einsum("in,ij,jn->n", phis[0], alpha, phis[1])
    p = [torch.einsum("in,ij,jn->n", phis[d], Ps[d], phis[d]) for d in range(2)]
    q = [torch.einsum("in,ij,jn->n", phis[d], Qs[d], phis[d]) for d in range(2)]
    inside = (phis[0].sum(0) > 0) & (phis[1].sum(0) > 0)
    var_ref = torch.where(inside, s2[0] * s2[1] - p[0] * p[1] + q[0] * q[1], s2[0] * s2[1])
    mu_ref = torch.where(inside, mu_ref, torch.zeros_like(mu_ref))
    assert np.allclose(mean, mu_ref.numpy(), rtol=1e-9, atol=1e-11)
    assert np.allclose(var, var_ref.numpy(), rtol=1e-9, atol=1e-11)
    plan.close()


@pytest.mark.parametrize("knots,N", [((11,), 400), ((8, 7), 500), ((5, 12), 300)])
@pytest.mark.parametrize("dtype,tol", [(np.float64, 1e-8), (np.float32, 1e-3)])
def test_b0_step_scan_form_matches_oracle_under_emulation(emu, knots, N, dtype, tol):
    """The B0 family through the binned layout = scan form (k_obs_b0s + table construction + adjoint stage, b0scan.cuh):
    ELBO and every gradient against the oracle's dense-feature evaluation, observations outside the mesh included."""
    lib, L = emu
    D = len(knots)
    meshes, X, y, l, s2, noise, m, Ls = make_problem(knots, N, seed=21 + D, family=O.B0_GRIDDED, x_lo=-0.2, x_hi=1.2)
    tdt = torch.float64 if dtype == np.float64 else torch.float32
    Xq, yq = X.to(tdt), y.to(tdt)
    scale = 1.3
    elbo_ref, g_ref = oracle_value_and_grads(O.B0_GRIDDED, meshes, Xq.to(torch.float64), yq.to(torch.float64),
                                             l, s2, noise, m, Ls, scale=scale)
    plan = emul_lib.EmuPlan(lib, L, L.B0_GRIDDED, [t.numpy() for t in meshes], dtype)
    theta = torch.cat([l, s2, noise.reshape(1)]).numpy().copy()
    xs = [np.ascontiguousarray(Xq[:, d].numpy()) for d in range(D)]
    yy = np.ascontiguousarray(yq.numpy())
    binned = plan.bin(xs, yy, run_cap=16)
    assert binned[2].n_inside == N                      # every observation has an extended cell
    out, dtheta, dm, dL = plan.step(theta, m.numpy().copy(), torch.cat([Lx.reshape(-1) for Lx in Ls]).numpy().copy(),
                                    binned, None, scale)
    check_against_oracle(plan, out, dtheta, dm, dL, elbo_ref, g_ref, N, tol)
    plan.close()


@pytest.mark.parametrize("knots,N", [((71,), 300), ((41, 76), 350), ((100, 34), 350)])
def test_b0_segmented_sweeps_under_emulation(emu, knots, N):
    """The segmented sweeps of the scan form (k_b0s_scan_seg / k_b0s_scan_adj_seg: a fibre cut into ceil(M / 16) segments with
    carries folded through shared memory; here 3 - 7 segments with a partial last one, row and column fibres, the tangent
    variant included) against the one-thread-per-fibre kernels on the same step, and against the oracle."""
    lib, L = emu
    D = len(knots)
    meshes, X, y, l, s2, noise, m, Ls = make_problem(knots, N, seed=31 + D, family=O.B0_GRIDDED, x_lo=-0.1, x_hi=1.1)
    l = l * 0.04                                         # l ~ delta: the float32-rounded Toeplitz row of the reference stays positive definite
    elbo_ref, g_ref = oracle_value_and_grads(O.B0_GRIDDED, meshes, X, y, l, s2, noise, m, Ls, scale=1.2)
    theta = torch.cat([l, s2, noise.reshape(1)]).numpy().copy()
    xs = [np.ascontiguousarray(X[:, d].numpy()) for d in range(D)]
    res = []
    for seg in (1, 0):
        lib.vggp_debug_b0s_seg(seg)
        try:
            plan = emul_lib.EmuPlan(lib, L, L.B0_GRIDDED, [t.numpy() for t in meshes], np.float64)
            out = plan.step(theta, m.numpy().copy(), torch.cat([Lx.reshape(-1) for Lx in Ls]).numpy().copy(),
                            plan.bin(xs, np.ascontiguousarray(y.numpy()), run_cap=16), None, 1.2)
            if seg:
                check_against_oracle(plan, *out, elbo_ref, g_ref, N, 1e-7)
            res.append(out)
            plan.close()
        finally:
            lib.vggp_debug_b0s_seg(1)
    for a, b in zip(res[0], res[1]):
        assert relerr(torch.from_numpy(np.asarray(a, dtype=np.float64)), torch.from_numpy(np.asarray(b, dtype=np.float64))) < 1e-10


@pytest.mark.parametrize("knots", [(11,), (8, 7)])
@pytest.mark.parametrize("dtype,tol", [(np.float64, 1e-9), (np.float32, 2e-4)])
def test_b0_point_prediction_scan_form_under_emulation(emu, knots, dtype, tol):
    """vggp_predict for the B0 family = the scan form of csrc/b0scan.cuh (per-cell tables from dense products, O(1) work
    per point) against the dense formulas with the reference's dense features; points outside the mesh and on knots
    included."""
    lib, L = emu
    D = len(knots)
    meshes, X, y, l, s2, noise, m, Ls = make_problem(knots, 300, seed=12, family=O.B0_GRIDDED, x_lo=-0.3, x_hi=1.3)
    plan = emul_lib.EmuPlan(lib, L, L.B0_GRIDDED, [t.numpy() for t in meshes], dtype)
    theta = torch.cat([l, s2, noise.reshape(1)]).numpy().copy()
    plan.grid_forward(theta, m.numpy().copy(), torch.cat([Lx.reshape(-1) for Lx in Ls]).numpy().copy())
    tdt = torch.float64 if dtype == np.float64 else torch.float32
    Xq = X.to(tdt)
    xs = [np.ascontiguousarray(Xq[:, d].numpy()) for d in range(D)]
    mean, var = plan.predict(xs)
    Ms = [k - 1 for k in knots]
    Ks = [O.kuu_factor(O.B0_GRIDDED, meshes[d], l[d], s2[d], ref_quirks=False).to(torch.float64) for d in range(D)]
    Ps = [torch.linalg.inv(K) for K in Ks]
    Qs = [P @ torch.tril(Lx) @ torch.tril(Lx).T @ P for P, Lx in zip(Ps, Ls)]
    phis = [O.b0_features_dense(meshes[d], Xq[:, d].to(torch.float64), l[d], s2[d]) for d in range(D)]
    A = m.reshape(Ms)
    for d in range(D):
        A = O.mode_product(A, Ps[d], d)
    mu_ref = phis[0].T @ A if D == 1 else torch.einsum("in,ij,jn->n", phis[0], A, phis[1])
    pp = torch.ones_like(mu_ref)
    qq = torch.ones_like(mu_ref)
    for d in range(D):
        pp = pp * (phis[d] * (Ps[d] @ phis[d])).sum(0)
        qq = qq * (phis[d] * (Qs[d] @ phis[d])).sum(0)
    var_ref = torch.prod(s2) - pp + qq
    scale_mu = float(mu_ref.abs().max())
    assert np.max(np.abs(mean - mu_ref.numpy())) <= tol * scale_mu
    assert np.max(np.abs(var - var_ref.numpy())) <= tol * float(var_ref.abs().max())
    plan.close()


@pytest.mark.parametrize("dtype,tol", [(np.float64, 1e-12), (np.float32, 1e-5)])
def test_metrics_kernels_under_emulation(emu, dtype, tol):
    """vggp_metrics / vggp_predict_metrics against the reference's formulas (src/utils/evaluationmetrics.py:6-54)."""
    lib, L = emu
    rng = np.random.default_rng(1)
    n = 7001
    t = (50.0 + rng.standard_normal(n)).astype(dtype)             # large mean: the pivoted one-pass TSS must not cancel
    p = (t + 0.3 * rng.standard_normal(n)).astype(dtype)
    out = np.full(4, np.nan)
    assert lib.vggp_metrics(L.F32 if dtype == np.float32 else L.F64, emul_lib.ptr(t), emul_lib.ptr(p), n, emul_lib.ptr(out), None) == 0
    t64, p64 = t.astype(np.float64), p.astype(np.float64)
    mse = np.mean((t64 - p64) ** 2)
    mae = np.mean(np.abs(t64 - p64))
    r2 = 1 - np.sum((t64 - p64) ** 2) / np.sum((t64 - t64.mean()) ** 2)
    assert abs(out[0] / n - mse) <= tol * mse and abs(out[1] / n - mae) <= tol * mae
    assert abs((1 - out[0] / (out[3] - out[2] ** 2 / n)) - r2) <= 10 * tol
    assert lib.vggp_metrics(L.F64, None, None, 0, emul_lib.ptr(out), None) == 0 and not out.any()
    # fused with the prediction
    knots, N = (9, 7), 500
    meshes, X, y, l, s2, noise, m, Ls = make_problem(knots, N, seed=8)
    plan = emul_lib.EmuPlan(lib, L, L.B1_ASVGP, [tt.numpy() for tt in meshes], dtype)
    theta = torch.cat([l, s2, noise.reshape(1)]).numpy().copy()
    plan.grid_forward(theta, m.numpy().copy(), torch.cat([Lx.reshape(-1) for Lx in Ls]).numpy().copy())
    xs = [np.ascontiguousarray(X[:, d].numpy().astype(dtype)) for d in range(2)]
    yy = y.numpy().astype(dtype)
    mean, _ = plan.predict(xs)
    sums = plan.predict_metrics(xs, yy)
    e = yy.astype(np.float64) - mean.astype(np.float64)
    assert abs(sums[0] - np.sum(e ** 2)) <= 1e-12 * np.sum(e ** 2) and abs(sums[1] - np.sum(np.abs(e))) <= 1e-12 * np.sum(np.abs(e))
    c = yy.astype(np.float64) - float(yy[0])
    assert abs(sums[2] - c.sum()) <= 1e-9 * max(1.0, abs(c.sum())) and abs(sums[3] - np.sum(c ** 2)) <= 1e-12 * np.sum(c ** 2)
    plan.close()


@pytest.mark.parametrize("dtype", [np.float64, np.float32])
def test_minmax_scaling_bit_exact_under_emulation(emu, dtype):
    """vggp_minmax / vggp_minmax_scale against the reference's torch expressions (src/utils/dataprocessors.py:3-44)."""
    lib, L = emu
    code = L.F32 if dtype == np.float32 else L.F64
    rng = np.random.default_rng(4)
    for n in (1, 255, 70001):
        x = (rng.standard_normal(n) * 37.0 + 11.0).astype(dtype)
        mm = np.zeros(2, dtype=dtype)
        assert lib.vggp_minmax(code, emul_lib.ptr(x), n, emul_lib.ptr(mm), None) == 0
        assert mm[0] == x.min() and mm[1] == x.max()
        if n == 1:
            continue
        y = np.zeros_like(x)
        assert lib.vggp_minmax_scale(code, emul_lib.ptr(x), n, emul_lib.ptr(mm), 0, emul_lib.ptr(y), None) == 0
        t = torch.from_numpy(x)
        ref = (t - torch.min(t)) / (torch.max(t) - torch.min(t))
        assert np.array_equal(y, ref.numpy())
        back = np.zeros_like(x)
        assert lib.vggp_minmax_scale(code, emul_lib.ptr(y), n, emul_lib.ptr(mm), 1, emul_lib.ptr(back), None) == 0
        ref_back = ref * (torch.max(t) - torch.min(t)) + torch.min(t)
        assert np.array_equal(back, ref_back.numpy())
    assert lib.vggp_minmax(code, None, 0, emul_lib.ptr(mm), None) == -1


@pytest.mark.parametrize("family", ["B1", "B0"])
def test_binned_shards_sum_to_the_full_batch_under_emulation(emu, family):
    """Sharding contract of SURVEY.md section 8e for the binned layouts: two ranks run the per-observation stage on their
    halves, the gradient buffers are summed (what the all-reduce does), and the grid backward on the sum reproduces the
    single-rank step.  For the B0 scan form this also checks that the adjoint stage is linear in the raw sums."""
    lib, L = emu
    fam = L.B1_ASVGP if family == "B1" else L.B0_GRIDDED
    ofam = O.B1_ASVGP if family == "B1" else O.B0_GRIDDED
    knots, N = (9, 7), 800
    meshes, X, y, l, s2, noise, m, Ls = make_problem(knots, N, seed=31, family=ofam, x_lo=-0.1, x_hi=1.1)
    theta = torch.cat([l, s2, noise.reshape(1)]).numpy().copy()
    mm = m.numpy().copy()
    Lcat = torch.cat([Lx.reshape(-1) for Lx in Ls]).numpy().copy()
    xs = [np.ascontiguousarray(X[:, d].numpy()) for d in range(2)]
    yy = y.numpy().copy()
    full = emul_lib.EmuPlan(lib, L, fam, [t.numpy() for t in meshes], np.float64)
    ref = full.step(theta, mm, Lcat, full.bin(xs, yy, run_cap=16), None, 1.0)
    ranks = [emul_lib.EmuPlan(lib, L, fam, [t.numpy() for t in meshes], np.float64) for _ in range(2)]
    cut = 317
    total = np.zeros(ranks[0].gbuf_bytes, dtype=np.uint8)
    acc_obs = np.zeros(ranks[0].gbuf_obs_elems)
    acc_scal = np.zeros(8)
    for r, (lo, hi) in zip(ranks, ((0, cut), (cut, N))):
        r.grid_forward(theta, mm, Lcat)
        r.obs_fwd_bwd(r.bin([x[lo:hi].copy() for x in xs], yy[lo:hi].copy(), run_cap=16))
        acc_obs += r.gbuf[: r.gbuf_obs_elems * 8].view(np.float64)
        acc_scal += r.gbuf[r.gbuf_scalar_offset: r.gbuf_scalar_offset + 64].view(np.float64)
    r0 = ranks[0]
    r0.gbuf[: r0.gbuf_obs_elems * 8].view(np.float64)[:] = acc_obs
    r0.gbuf[r0.gbuf_scalar_offset: r0.gbuf_scalar_offset + 64].view(np.float64)[:] = acc_scal
    got = r0.grid_backward(theta, mm, Lcat, 1.0)
    for a, b in zip(got, ref):
        assert np.allclose(a, b, rtol=1e-10, atol=1e-12)
    for pl in [full] + ranks:
        pl.close()


def test_binned_abi_edge_cases_under_emulation(emu):
    lib, L = emu
    meshes = [np.linspace(0, 1, 9, dtype=np.float32), np.linspace(0, 1, 7, dtype=np.float32)]
    plan = emul_lib.EmuPlan(lib, L, L.B1_ASVGP, meshes, np.float64)
    rng = np.random.default_rng(0)
    theta = np.array([0.3, 0.4, 1.0, 0.9, 0.05])
    m = 0.1 * rng.standard_normal(63)
    Lcat = np.concatenate([np.eye(n).reshape(-1) for n in (9, 7)])
    empty = [np.zeros(0), np.zeros(0)]
    out_b, *_ = plan.step(theta, m, Lcat, plan.bin(empty, np.zeros(0)), None, 1.0)
    out_r, *_ = plan.step(theta, m, Lcat, empty, np.zeros(0), 1.0)
    assert out_b[3] == 0 and np.allclose(out_b, out_r, rtol=1e-12, atol=0)
    xo = [np.full(50, 3.0), rng.random(50)]
    yo = rng.standard_normal(50)
    b1 = plan.bin(xo, yo)
    assert b1[2].n_tasks == 0 and b1[2].n_inside == 0
    out_b, dth_b, dm_b, _ = plan.step(theta, m, Lcat, b1, None, 1.0)
    out_r, dth_r, dm_r, _ = plan.step(theta, m, Lcat, xo, yo, 1.0)
    assert np.allclose(out_b, out_r, rtol=1e-12) and np.allclose(dth_b, dth_r, rtol=1e-10) and np.allclose(dm_b, dm_r)
    # a descriptor from another prepare is refused
    d1 = plan.bin([rng.random(40), rng.random(40)], rng.standard_normal(40))[2]
    desc = L.BinnedDesc()
    import ctypes as C
    xs = [rng.random(30), rng.random(30)]
    plan.check(lib.vggp_obs_bin_prepare(plan.h, plan._xptrs(xs), 30, 16, C.byref(desc), None))
    buf = np.zeros(int(d1.bytes) + 512, dtype=np.uint8)
    assert lib.vggp_obs_bin_pack(plan.h, C.byref(d1), plan._xptrs(xs), emul_lib.ptr(rng.standard_normal(30)), emul_lib.ptr(buf), None) == -1      # VGGP_E_ARG
    plan.close()


@pytest.mark.parametrize("knots,N,chunk", [((17, 12), 1500, 200), ((9, 7, 5), 900, 128), ((40,), 700, 64)])
def test_host_entry_point_chunked_transfer_under_emulation(emu, knots, N, chunk):
    """vggp_elbo_host (the whole step from host buffers): with the observations crossing in chunks -- copy stream, one
    event per chunk, the per-observation kernel accumulating chunk by chunk into one gradient buffer -- the results equal
    those of the one-shot step, and the count the kernel reports is the shard's, not a chunk's."""
    import ctypes as C
    lib, L = emu
    D = len(knots)
    meshes, X, y, l, s2, noise, m, Ls = make_problem(knots, N, seed=9 + D)
    theta = torch.cat([l, s2, noise.reshape(1)]).numpy().copy()
    mm = m.numpy().copy()
    Lcat = torch.cat([Lx.reshape(-1) for Lx in Ls]).numpy().copy()
    xs = [np.ascontiguousarray(X[:, d].numpy()) for d in range(D)]
    yy = np.ascontiguousarray(y.numpy())
    plan = emul_lib.EmuPlan(lib, L, L.B1_ASVGP, [t.numpy() for t in meshes], np.float64)
    ref = plan.step(theta, mm, Lcat, xs, yy, 1.4)
    res = []
    for target in (chunk, 1 << 23):
        lib.vggp_debug_host_chunk(target)
        try:
            out, dth = np.zeros(4), np.zeros(2 * D + 1)
            dm, dL = np.zeros(plan.M), np.zeros(plan.L_total)
            ptrs = (C.c_void_p * D)(*[x.ctypes.data for x in xs])
            rc = lib.vggp_elbo_host(plan.h, ptrs, yy.ctypes.data, N, theta.ctypes.data, mm.ctypes.data, Lcat.ctypes.data,
                                    C.c_double(1.4), out.ctypes.data, dth.ctypes.data, dm.ctypes.data, dL.ctypes.data, None)
            assert rc == 0, lib.vggp_last_error()
            res.append((out, dth, dm, dL))
        finally:
            lib.vggp_debug_host_chunk(1 << 23)
    assert res[0][0][3] == N and res[1][0][3] == N
    for got in res:
        for a, b in zip(got, ref):
            assert relerr(torch.from_numpy(a), torch.from_numpy(np.asarray(b, dtype=np.float64))) < 1e-11
    plan.close()


@pytest.mark.parametrize("D", [2, 3])
@pytest.mark.parametrize("dtype", [np.float32, np.float64])
def test_track_generator_under_emulation(emu, D, dtype):
    """vggp_generate_tracks (the synthetic along-track data set of the bench, generated by the library) against the torch
    restatement in bench.py: identical coordinates (integer hash + separately rounded float64 operations), targets equal up to
    the last bits of sin / cos; a shard [lo, hi) is the corresponding slice of the whole data set."""
    import ctypes as C
    import bench
    lib, L = emu
    n_total, seed = 6000, 3
    tdt = torch.float32 if dtype == np.float32 else torch.float64
    xs_ref, y_ref = bench.make_tracks_torch(0, n_total, n_total, torch.device("cpu"), tdt, seed=seed, D=D)

    def gen(lo, hi):
        xs = [np.zeros(hi - lo, dtype=dtype) for _ in range(D)]
        y = np.zeros(hi - lo, dtype=dtype)
        ptrs = (C.c_void_p * D)(*[x.ctypes.data for x in xs])
        rc = lib.vggp_generate_tracks(L.F32 if dtype == np.float32 else L.F64, D, n_total, lo, hi, seed, bench.PASSES,
                                      C.c_double(bench.TRACK_GRADIENT), ptrs, y.ctypes.data, None)
        assert rc == 0, lib.vggp_last_error()
        return xs, y

    xs, y = gen(0, n_total)
    for d in range(D):
        assert np.array_equal(xs[d], xs_ref[d].numpy()), d
    tol = 2e-7 if dtype == np.float32 else 1e-14
    assert np.max(np.abs(y - y_ref.numpy())) <= tol * max(1.0, float(y_ref.abs().max()))
    assert 0.0 <= min(x.min() for x in xs) and max(x.max() for x in xs) <= 1.0
    xs_s, y_s = gen(1234, 4321)
    for d in range(D):
        assert np.array_equal(xs_s[d], xs[d][1234:4321])
    assert np.array_equal(y_s, y[1234:4321])


def test_automatic_run_cap_under_emulation(emu):
    """vggp_obs_bin_prepare with run_cap = 0 picks the cap from the shard size (never below 32, 256 for large shards); the
    step over that layout equals the step over an explicit cap."""
    lib, L = emu
    knots, N = (9, 7), 4000
    meshes, X, y, l, s2, noise, m, Ls = make_problem(knots, N, seed=2)
    theta = torch.cat([l, s2, noise.reshape(1)]).numpy().copy()
    mm, Lcat = m.numpy().copy(), torch.cat([Lx.reshape(-1) for Lx in Ls]).numpy().copy()
    xs = [np.ascontiguousarray(X[:, d].numpy()) for d in range(2)]
    yy = np.ascontiguousarray(y.numpy())
    plan = emul_lib.EmuPlan(lib, L, L.B1_ASVGP, [t.numpy() for t in meshes], np.float64)
    auto = plan.bin(xs, yy, run_cap=0)
    assert auto[2].run_cap == 32
    ref = plan.step(theta, mm, Lcat, plan.bin(xs, yy, run_cap=32), None, 1.0)
    got = plan.step(theta, mm, Lcat, auto, None, 1.0)
    for a, b in zip(got, ref):
        assert relerr(torch.from_numpy(np.asarray(a, dtype=np.float64)), torch.from_numpy(np.asarray(b, dtype=np.float64))) < 1e-12
    plan.close()


@pytest.mark.parametrize("knots,N", B1_CASES)
@pytest.mark.parametrize("dtype,tol", [(np.float64, 1e-9), (np.float32, 1e-3)])
def test_deterministic_mode_matches_oracle_under_emulation(emu, knots, N, dtype, tol):
    """vggp_set_deterministic (include/vggp.h): run records + ordered reductions instead of the atomics of the per-observation
    kernel, per-CTA partials instead of the atomics of the fibre passes -- same ELBO and gradients as the oracle, identical
    bits from two runs, and the plain-array entry point refuses while the mode is on."""
    lib, L = emu
    D = len(knots)
    meshes, X, y, l, s2, noise, m, Ls = make_problem(knots, N, seed=7 + D)
    tdt = torch.float64 if dtype == np.float64 else torch.float32
    Xq, yq = X.to(tdt), y.to(tdt)
    scale = 1.3
    elbo_ref, g_ref = oracle_value_and_grads(O.B1_ASVGP, meshes, Xq.to(torch.float64), yq.to(torch.float64),
                                             l, s2, noise, m, Ls, scale=scale)
    plan = emul_lib.EmuPlan(lib, L, L.B1_ASVGP, [t.numpy() for t in meshes], dtype)
    theta = torch.cat([l, s2, noise.reshape(1)]).numpy().copy()
    mm = m.numpy().copy()
    Lcat = torch.cat([Lx.reshape(-1) for Lx in Ls]).numpy().copy()
    xs = [np.ascontiguousarray(Xq[:, d].numpy()) for d in range(D)]
    yy = np.ascontiguousarray(yq.numpy())
    try:
        binned = plan.bin(xs, yy, run_cap=8)          # cells split into several runs: the ordered sum has something to order
        plain = plan.step(theta, mm, Lcat, binned, None, scale)
        plan.check(lib.vggp_set_deterministic(plan.h, 1))
        a = plan.step(theta, mm, Lcat, binned, None, scale)
        b = plan.step(theta, mm, Lcat, binned, None, scale)
        check_against_oracle(plan, *a, elbo_ref, g_ref, N, tol)
        for u, v in zip(a, b):
            assert np.array_equal(np.asarray(u), np.asarray(v))
        for u, v in zip(a, plain):
            assert relerr(u, torch.from_numpy(np.asarray(v, dtype=np.float64))) < tol * 10
        rc = lib.vggp_obs_fwd_bwd(plan.h, plan._xptrs(xs), emul_lib.ptr(yy), N, emul_lib.ptr(plan.gbuf), None)
        assert rc == -6
        plan.check(lib.vggp_set_deterministic(plan.h, 0))
        c = plan.step(theta, mm, Lcat, binned, None, scale)
        for u, v in zip(c, plain):
            assert relerr(u, torch.from_numpy(np.asarray(v, dtype=np.float64))) < tol * 10
    finally:
        plan.close()


def test_workspace_bytes_under_emulation(emu):
    """vggp_workspace_bytes (include/vggp.h, SURVEY.md section 8b): the plan-owned memory is fixed at creation, the gradient
    buffer size equals vggp_gbuf_layout's, and the scratch figure grows when an opt-in path (here the plain-array entry point)
    stages observations."""
    lib, L = emu
    meshes, X, y, l, s2, noise, m, Ls = make_problem((9, 7), 300, seed=3)
    plan = emul_lib.EmuPlan(lib, L, L.B1_ASVGP, [t.numpy() for t in meshes], np.float32)
    try:
        a, b, c = emul_lib.C.c_int64(), emul_lib.C.c_int64(), emul_lib.C.c_int64()
        plan.check(lib.vggp_workspace_bytes(plan.h, emul_lib.C.byref(a), emul_lib.C.byref(b), emul_lib.C.byref(c)))
        assert a.value > 8 * plan.M and b.value == plan.gbuf_bytes and c.value == 0
        theta = torch.cat([l, s2, noise.reshape(1)]).numpy().copy()
        xs = [np.ascontiguousarray(X[:, d].numpy().astype(np.float32)) for d in range(2)]
        plan.step(theta, m.numpy().copy(), torch.cat([Lx.reshape(-1) for Lx in Ls]).numpy().copy(), xs, y.numpy().astype(np.float32))
        a2, c2 = emul_lib.C.c_int64(), emul_lib.C.c_int64()
        plan.check(lib.vggp_workspace_bytes(plan.h, emul_lib.C.byref(a2), None, emul_lib.C.byref(c2)))
        assert a2.value == a.value and c2.value >= 300 * 4 * 3
        assert lib.vggp_workspace_bytes(None, None, None, None) == -1
    finally:
        plan.close()


def test_b1_plan_holds_only_the_fused_grid_side_under_emulation(emu):
    """A B1 plan has no dense factor path: VGGP_WS_K and VGGP_WS_Q are refused (the step never forms the Cholesky factor or
    the full Q_d), the views the fused grid side does provide stay available, and the plan-owned memory is what the fused
    grid side, the per-observation kernel and those views use, plus a few scalars."""
    import ctypes as C
    lib, L = emu
    knots = (40, 33)
    meshes = [np.linspace(0, 1, k, dtype=np.float32) for k in knots]
    plan = emul_lib.EmuPlan(lib, L, L.B1_ASVGP, meshes, np.float32)
    try:
        ptr, n = C.c_void_p(), C.c_int64()
        for which in (L.WS_K, L.WS_Q):
            assert lib.vggp_workspace_ptr(plan.h, which, 0, C.byref(ptr), C.byref(n)) == -6      # VGGP_E_UNSUPPORTED
            assert b"VGGP_WS_QBAND" in lib.vggp_last_error()
        for which in (L.WS_P, L.WS_R, L.WS_QBAND, L.WS_KRAW):
            assert lib.vggp_workspace_ptr(plan.h, which, 1, C.byref(ptr), C.byref(n)) == 0
        a = C.c_int64()
        plan.check(lib.vggp_workspace_bytes(plan.h, C.byref(a), None, None))
        M, sn, tsz = int(np.prod(knots)), sum(knots), 4
        kept = (8 * sum(3 * k * k for k in knots)         # K_d and P_d (filled on demand), R_d
                + 8 * (2 + 3 + 3) * sn                    # band of Q_d, generators [pd | ru | rl], band accumulators of dK_d
                + 8 * 3 * M                               # alpha, the two mode-product tensors
                + tsz * (M + 8 * sn + 128 * 4 * sn)       # alpha in the observation dtype, per-cell tables, band replicas
                + 2 * 4 * sn)                             # the knots, twice
        assert kept <= a.value <= kept + 256, (a.value, kept)
    finally:
        plan.close()


def test_splitk_fixup_mode_product_under_emulation(emu):
    """A group with fewer tiles than SMs is cut along k; the partial tiles meet in a workspace and the last CTA of a tile adds
    them in split order (gemm.cuh gemm_fixup) -- no destination clear, no float64 atomics.  vggp_mode_product on a 140-knot
    dimension (3 x 3 tiles, k = 139 -> two splits) against numpy, twice (the tile counters return to zero), into a destination
    full of NaNs (nothing may be accumulated into it), and the dense-path step with both forms of the split."""
    lib, L = emu
    meshes = [np.linspace(0, 1, 140, dtype=np.float32), np.linspace(0, 1, 9, dtype=np.float32)]
    plan = emul_lib.EmuPlan(lib, L, L.B0_GRIDDED, meshes, np.float64)
    try:
        n0, n1 = plan.m_per_dim
        rng = np.random.default_rng(0)
        A = rng.standard_normal((n0, n0))
        src = rng.standard_normal((n0, n1))
        for _ in range(2):
            dst = np.full((n0, n1), np.nan)
            plan.check(lib.vggp_mode_product(plan.h, 0, emul_lib.ptr(A), emul_lib.ptr(src), emul_lib.ptr(dst), None))
            ref = A @ src if np.allclose(dst, A @ src, rtol=1e-12, atol=1e-12) else A.T @ src
            assert np.allclose(dst, ref, rtol=1e-12, atol=1e-12)
    finally:
        plan.close()
    knots, N = (140, 7), 600
    meshes_t, X, y, l, s2, noise, m, Ls = make_problem(knots, N, seed=21, family=O.B0_GRIDDED)
    l = torch.tensor([0.03, 0.3], dtype=torch.float64)      # l / delta small enough for the float32-rounded Toeplitz row to stay PD
    elbo_ref, g_ref = oracle_value_and_grads(O.B0_GRIDDED, meshes_t, X, y, l, s2, noise, m, Ls, scale=1.2)
    res = []
    for fix in (1, 0):
        lib.vggp_debug_splitk_fixup(fix)
        try:
            plan = emul_lib.EmuPlan(lib, L, L.B0_GRIDDED, [t.numpy() for t in meshes_t], np.float64)
            theta = torch.cat([l, s2, noise.reshape(1)]).numpy().copy()
            xs = [np.ascontiguousarray(X[:, d].numpy()) for d in range(2)]
            res.append(plan.step(theta, m.numpy().copy(), torch.cat([Lx.reshape(-1) for Lx in Ls]).numpy().copy(),
                                 xs, y.numpy().copy(), 1.2))
            if fix:
                check_against_oracle(plan, *res[-1], elbo_ref, g_ref, N, 1e-7)
            plan.close()
        finally:
            lib.vggp_debug_splitk_fixup(1)
    for a, b in zip(res[0], res[1]):
        assert relerr(a, torch.from_numpy(np.asarray(b, dtype=np.float64))) < 1e-9


def test_deterministic_mode_edge_cases_under_emulation(emu):
    """Deterministic mode on an empty shard and on a shard with every observation outside the mesh (no run at all): same
    results as the plain-array path."""
    lib, L = emu
    meshes = [np.linspace(0, 1, 9, dtype=np.float32), np.linspace(0, 1, 7, dtype=np.float32)]
    plan = emul_lib.EmuPlan(lib, L, L.B1_ASVGP, meshes, np.float64)
    try:
        rng = np.random.default_rng(0)
        theta = np.array([0.3, 0.4, 1.0, 0.9, 0.05])
        m = 0.1 * rng.standard_normal(63)
        Lcat = np.concatenate([np.eye(n).reshape(-1) for n in (9, 7)])
        empty = [np.zeros(0), np.zeros(0)]
        xo = [np.full(50, 3.0), rng.random(50)]
        yo = rng.standard_normal(50)
        ref_e = plan.step(theta, m, Lcat, empty, np.zeros(0), 1.0)
        ref_o = plan.step(theta, m, Lcat, xo, yo, 1.0)
        b_e, b_o = plan.bin(empty, np.zeros(0)), plan.bin(xo, yo)
        assert b_o[2].n_tasks == 0
        plan.check(lib.vggp_set_deterministic(plan.h, 1))
        for obs, ref in ((b_e, ref_e), (b_o, ref_o)):
            got = plan.step(theta, m, Lcat, obs, None, 1.0)
            for u, v in zip(got, ref):
                assert np.allclose(u, v, rtol=1e-10, atol=1e-12)
    finally:
        plan.close()
