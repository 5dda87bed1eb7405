"""GPU parity of the libvggp building blocks against the CPU oracle / torch float64 (run with -m gpu on a B200).
Everything goes through the C ABI (ctypes)."""
import os

import numpy as np
import pytest
import torch

from oracle import vggp_oracle as O

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def vg():
    import vggp_b200
    vggp_b200._lib.load()
    return vggp_b200


@pytest.fixture(scope="module")
def dev():
    assert torch.cuda.is_available(), "these tests need a CUDA device"
    return torch.device("cuda", 0)


# ---------------------------------------------------------------------------------------------------------
# GEMM (DMMA tensor-core loop and its SIMT cross-check)
# ---------------------------------------------------------------------------------------------------------
GEMM_SHAPES = [(64, 64, 64), (100, 37, 53), (513, 130, 257), (1, 7, 300), (200, 1, 5), (128, 128, 1)]


@pytest.mark.parametrize("use_mma", [True, False])
@pytest.mark.parametrize("shape", GEMM_SHAPES)
def test_gemm_plain(vg, dev, use_mma, shape):
    m, n, k = shape
    g = torch.Generator(device="cpu").manual_seed(m * 1000 + n * 10 + k)
    A = torch.randn(m, k, generator=g, dtype=torch.float64).to(dev)
    B = torch.randn(k, n, generator=g, dtype=torch.float64).to(dev)
    C = vg.gemm_f64(A, B, use_mma=use_mma)
    ref = A @ B
    assert torch.allclose(C, ref, rtol=1e-12, atol=1e-11), (C - ref).abs().max().item()


@pytest.mark.parametrize("use_mma", [True, False])
def test_gemm_strided_transposed_batched_splitk(vg, dev, use_mma):
    g = torch.Generator(device="cpu").manual_seed(7)
    A = torch.randn(3, 90, 140, generator=g, dtype=torch.float64).to(dev)      # use A^T: (3, 140, 90)
    B = torch.randn(3, 70, 90, generator=g, dtype=torch.float64).to(dev)       # use B^T: (3, 90, 70)
    At, Bt = A.transpose(1, 2), B.transpose(1, 2)
    C = vg.gemm_f64(At, Bt, use_mma=use_mma)
    assert torch.allclose(C, At @ Bt, rtol=1e-12, atol=1e-11)
    # split-K accumulates atomically into a pre-filled C (beta*C must already be there)
    C0 = torch.randn(140, 70, generator=g, dtype=torch.float64).to(dev)
    C1 = vg.gemm_f64(At[0], Bt[0], use_mma=use_mma, splitk=4, alpha=-0.5, C_in=C0.clone())
    assert torch.allclose(C1, C0 - 0.5 * (At[0] @ Bt[0]), rtol=1e-12, atol=1e-11)
    # beta path
    C2 = vg.gemm_f64(At[1], Bt[1], use_mma=use_mma, alpha=2.0, beta=3.0, C_in=C0.clone())
    assert torch.allclose(C2, 3.0 * C0 + 2.0 * (At[1] @ Bt[1]), rtol=1e-12, atol=1e-11)


@pytest.mark.parametrize("dims", [(7,), (9, 70), (5, 66, 3), (130, 4, 65)])
def test_mode_product(vg, dev, dims):
    meshes = [torch.linspace(0, 1, n) for n in dims]
    plan = vg.GridPlan(vg.B1_ASVGP, meshes, torch.float64, dev)
    g = torch.Generator(device="cpu").manual_seed(11)
    T = torch.randn(*dims, generator=g, dtype=torch.float64)
    for d, n in enumerate(dims):
        A = torch.randn(n, n, generator=g, dtype=torch.float64)
        ref = O.mode_product(T, A, d)
        out = plan.mode_product(d, A.to(dev).contiguous(), T.reshape(-1).to(dev).contiguous()).reshape(*dims)
        assert torch.allclose(out.cpu(), ref, rtol=1e-12, atol=1e-11), (d, (out.cpu() - ref).abs().max().item())


# ---------------------------------------------------------------------------------------------------------
# B1 stencil: bit-exact against the fixtures produced by the reference's own bspline.py
# ---------------------------------------------------------------------------------------------------------
MESHES = ["lin11_01", "lin129_01", "lin16_02", "lin21_m3_7", "padded21_pad2"]


@pytest.mark.parametrize("name", MESHES)
@pytest.mark.parametrize("tag", ["f64", "f32"])
def test_b1_features_bit_exact_vs_reference_fixture(vg, dev, golden_dir, name, tag):
    sten = np.load(os.path.join(golden_dir, "b1_stencil.npz"))
    mesh = torch.from_numpy(sten[f"{name}.{tag}.mesh"])
    x = torch.from_numpy(sten[f"{name}.{tag}.x"])
    phi_ref = sten[f"{name}.{tag}.phi"]
    plan = vg.GridPlan(vg.B1_ASVGP, [mesh], x.dtype, dev)
    phi = plan.features_dense(0, x.to(dev)).cpu().numpy()
    assert phi.dtype == phi_ref.dtype
    assert np.array_equal(phi, phi_ref)          # numerical equality: -0.0 == 0.0
    c, wl, wh = plan.b1_stencil(0, x.to(dev))
    co, wlo, who = O.b1_stencil(mesh, x)
    assert np.array_equal(c.cpu().numpy().astype(np.int64), co.numpy())
    assert np.array_equal(wl.cpu().numpy(), wlo.numpy())
    assert np.array_equal(wh.cpu().numpy(), who.numpy())


@pytest.mark.parametrize("dtype", [torch.float32, torch.float64])
@pytest.mark.parametrize("K", [3, 12, 129, 512, 515])
def test_b1_stencil_bit_exact_random(vg, dev, dtype, K):
    mesh = torch.linspace(-0.3, 1.7, K)
    g = torch.Generator().manual_seed(K)
    x = (torch.rand(200_000, generator=g, dtype=torch.float64) * 2.2 - 0.4).to(dtype)
    x = torch.cat([x, mesh.to(dtype), torch.tensor([float("nan"), float("inf"), -float("inf")], dtype=dtype)])
    plan = vg.GridPlan(vg.B1_ASVGP, [mesh], dtype, dev)
    c, wl, wh = plan.b1_stencil(0, x.to(dev))
    co, wlo, who = O.b1_stencil(mesh, x)
    assert np.array_equal(c.cpu().numpy().astype(np.int64), co.numpy())
    assert np.array_equal(wl.cpu().numpy(), wlo.numpy())
    assert np.array_equal(wh.cpu().numpy(), who.numpy())


def test_b1_stencil_nonuniform_mesh_uses_search(vg, dev):
    # a mesh far from uniform: the arithmetic guess is disabled at plan creation and a binary search is used
    mesh = torch.tensor([0.0, 0.01, 0.02, 0.5, 0.51, 0.9, 2.0, 2.5, 2.50001, 3.0])
    g = torch.Generator().manual_seed(3)
    x = torch.rand(50_000, generator=g, dtype=torch.float64) * 3.4 - 0.2
    x = torch.cat([x, mesh.to(torch.float64)])
    plan = vg.GridPlan(vg.B1_ASVGP, [mesh], torch.float64, dev)
    c, wl, wh = plan.b1_stencil(0, x.to(dev))
    co, wlo, who = O.b1_stencil(mesh, x)
    assert np.array_equal(c.cpu().numpy().astype(np.int64), co.numpy())
    assert np.array_equal(wl.cpu().numpy(), wlo.numpy())
    assert np.array_equal(wh.cpu().numpy(), who.numpy())


def test_empty_inputs(vg, dev):
    mesh = torch.linspace(0, 1, 9)
    plan = vg.GridPlan(vg.B1_ASVGP, [mesh], torch.float64, dev)
    c, wl, wh = plan.b1_stencil(0, torch.empty(0, dtype=torch.float64, device=dev))
    assert c.numel() == 0 and wl.numel() == 0 and wh.numel() == 0


@pytest.mark.parametrize("dtype,tol", [(torch.float64, 1e-13), (torch.float32, 2e-6)])
def test_b0_features_dense(vg, dev, dtype, tol):
    mesh = torch.linspace(0, 1, 14)
    g = torch.Generator().manual_seed(5)
    x = (torch.rand(3000, generator=g, dtype=torch.float64) * 1.4 - 0.2).to(dtype)
    x = torch.cat([x, mesh.to(dtype)])
    l, s2 = torch.tensor(0.37, dtype=torch.float64), torch.tensor(1.3, dtype=torch.float64)
    theta = torch.tensor([0.37, 1.3, 0.1], dtype=torch.float64, device=dev)
    plan = vg.GridPlan(vg.B0_GRIDDED, [mesh], dtype, dev)
    phi = plan.features_dense(0, x.to(dev), theta).cpu()
    ref = O.b0_features_dense(mesh, x.to(torch.float64), l, s2)
    assert torch.allclose(phi.to(torch.float64), ref, rtol=tol, atol=tol), (phi.to(torch.float64) - ref).abs().max().item()


# ---------------------------------------------------------------------------------------------------------
# grid-side forward pieces against float64 torch
# ---------------------------------------------------------------------------------------------------------
_GF_KNOTS = [(9,), (70, 12), (131, 5, 66), (300, 7), (700,)]
_GF_PATHS = [(0, "b1_fused"), (1, "b0_dense")]


# B0 family at (700,): the reference's float32 Toeplitz row is indefinite at this l / delta (the test below covers that
# case), so the combination is not generated
@pytest.mark.parametrize("family,knots",
                         [pytest.param(f, k, id=f"{name}-{'x'.join(map(str, k))}")
                          for (f, name) in _GF_PATHS for k in _GF_KNOTS if not (f == 1 and max(k) > 400)])
def test_grid_forward_pieces(vg, dev, family, knots):
    """family 0 (B1): the fused fibre passes over the twisted factorisation; family 1 (B0): the dense blocked Cholesky +
    triangular inverse, whose Cholesky factor and full Q_d are checked too."""
    D = len(knots)
    dense = family != 0
    meshes = [torch.linspace(0, 1 + 0.5 * d, k) for d, k in enumerate(knots)]
    plan = vg.GridPlan(family, meshes, torch.float64, dev)
    g = torch.Generator().manual_seed(100 + D)
    # B0 family: the reference's float32 rounding of (k +- 1) * delta (gridded_kronecker_structure.py:1312-1316)
    # makes the Toeplitz factor numerically indefinite once l / delta is large (min eigenvalue -8e-7 at 130 cells,
    # l = 0.68); keep the lengthscales where the reference's own factor is positive definite
    l = torch.rand(D, generator=g, dtype=torch.float64) * (0.5 if family == 0 else 0.1) + (0.2 if family == 0 else 0.05)
    s2 = torch.rand(D, generator=g, dtype=torch.float64) + 0.5
    noise = torch.tensor([0.05], dtype=torch.float64)
    theta = torch.cat([l, s2, noise])
    Ms = plan.m_per_dim
    m = torch.randn(plan.M, generator=g, dtype=torch.float64) * 0.3
    Ls = [torch.eye(n, dtype=torch.float64) * 0.7 + 0.1 * torch.randn(n, n, generator=g, dtype=torch.float64) for n in Ms]
    Lcat = torch.cat([L.reshape(-1) for L in Ls])
    plan.grid_forward(theta.to(dev), m.to(dev), Lcat.to(dev))
    assert plan.read_info() == 0
    alpha_ref = m.reshape(Ms)
    logdetK, logdetS, trs = [], [], []
    for d in range(D):
        K_ref = O.kuu_factor(family, meshes[d], l[d], s2[d], ref_quirks=False).to(torch.float64)
        K = plan.workspace(vg._lib.WS_KRAW, d).cpu()
        assert torch.allclose(K, K_ref, rtol=1e-12, atol=1e-14), (d, (K - K_ref).abs().max().item())
        C_ref = torch.linalg.cholesky(K_ref)
        if dense:
            C = torch.tril(plan.workspace(vg._lib.WS_K, d).cpu())
            assert torch.allclose(C, C_ref, rtol=1e-9, atol=1e-10), (d, (C - C_ref).abs().max().item())
        P = plan.workspace(vg._lib.WS_P, d).cpu()
        P_ref = torch.cholesky_inverse(C_ref)
        scale = P_ref.abs().max().item()
        assert (P - P_ref).abs().max().item() < 1e-9 * scale, (d, (P - P_ref).abs().max().item(), scale)
        Lt = torch.tril(Ls[d])
        R_ref = P_ref @ Lt
        R = plan.workspace(vg._lib.WS_R, d).cpu()
        assert (R - R_ref).abs().max().item() < 1e-9 * R_ref.abs().max().item()
        if dense:
            Q = plan.workspace(vg._lib.WS_Q, d).cpu()
            Q_ref = R_ref @ R_ref.T
            assert (Q - Q_ref).abs().max().item() < 1e-9 * Q_ref.abs().max().item()
        alpha_ref = O.mode_product(alpha_ref, P_ref, d)
        logdetK.append(2 * torch.log(torch.diagonal(C_ref)).sum())
        logdetS.append(2 * torch.log(torch.diagonal(Lt).abs()).sum())
        trs.append((R_ref * Lt).sum())
    alpha = plan.workspace(vg._lib.WS_ALPHA).cpu().reshape(Ms)
    assert (alpha - alpha_ref).abs().max().item() < 1e-8 * alpha_ref.abs().max().item()
    sc = plan.workspace(vg._lib.WS_SCAL).cpu()
    for d in range(D):
        assert abs(sc[0 + d] - logdetK[d]) < 1e-8 * max(1.0, abs(logdetK[d]))
        assert abs(sc[3 + d] - logdetS[d]) < 1e-10 * max(1.0, abs(logdetS[d]))
        assert abs(sc[6 + d] - trs[d]) < 1e-8 * abs(trs[d])
    ma = (m * alpha_ref.reshape(-1)).sum()
    assert abs(sc[9] - ma) < 1e-8 * max(1.0, abs(ma))


def test_reference_b0_factor_indefinite_is_reported(vg, dev):
    """The reference's own B0 Toeplitz factor is indefinite here (float32-rounded exponents); the reference would
    raise LinAlgError / add jitter (6_gulf_stream_experiement.ipynb cell 13 warning).  The library must flag it."""
    mesh = torch.linspace(0, 1, 131)
    K = O.kuu_b0(mesh, torch.tensor(0.6819, dtype=torch.float64), torch.tensor(1.4908, dtype=torch.float64))
    assert torch.linalg.eigvalsh(K).min() < 0
    plan = vg.GridPlan(vg.B0_GRIDDED, [mesh], torch.float64, dev)
    theta = torch.tensor([0.6819, 1.4908, 0.1], dtype=torch.float64, device=dev)
    m = torch.zeros(130, dtype=torch.float64, device=dev)
    L = torch.eye(130, dtype=torch.float64, device=dev).reshape(-1).contiguous()
    plan.grid_forward(theta, m, L)
    assert plan.read_info() == 1


def test_not_positive_definite_is_reported(vg, dev):
    # a negative outputscale makes K_d negative definite: the factorisation must flag dimension 1
    mesh = torch.linspace(0, 1, 20)
    plan = vg.GridPlan(vg.B1_ASVGP, [mesh], torch.float64, dev)
    theta = torch.tensor([0.3, -1.0, 0.1], dtype=torch.float64, device=dev)
    m = torch.zeros(20, dtype=torch.float64, device=dev)
    L = torch.eye(20, dtype=torch.float64, device=dev).reshape(-1).contiguous()
    plan.grid_forward(theta, m, L)
    assert plan.read_info() == 1
