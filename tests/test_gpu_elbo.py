"""GPU parity of the fused ELBO forward/backward against the structured CPU oracle (oracle/vggp_oracle.py,
itself pinned to the reference by tests/test_oracle_golden.py and tests/test_oracle_identities.py).

Tolerances (BASELINE.json north_star): float64 observations 1e-5 relative (we assert much tighter), float32
observations 1e-3 relative; gradients are compared in the norm of each parameter block."""
import importlib
import math

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
    assert torch.cuda.is_available()
    return torch.device("cuda", 0)


def make_problem(knots, N, seed, family=O.B1_ASVGP, x_lo=-0.05, x_hi=1.05):
    D = len(knots)
    g = torch.Generator().manual_seed(seed)
    meshes = [torch.linspace(0, 1, k) for k in knots]
    X = torch.rand(N, D, generator=g, dtype=torch.float64) * (x_hi - x_lo) + x_lo
    # a few observations exactly on knots / boundaries
    for d in range(D):
        X[d::97, d] = meshes[d][(torch.arange(len(X[d::97, d])) * 3) % knots[d]].to(torch.float64)
    y = torch.sin(3 * X[:, 0]) + (torch.cos(5 * X[:, -1]) if D > 1 else 0) + 0.1 * torch.randn(N, generator=g, dtype=torch.float64)
    l = torch.rand(D, generator=g, dtype=torch.float64) * 0.4 + 0.2
    s2 = torch.rand(D, generator=g, dtype=torch.float64) * 0.8 + 0.6
    noise = torch.tensor(0.07, dtype=torch.float64)
    Ms = [O.n_inducing(family, m) for m in meshes]
    M = int(np.prod(Ms))
    m = torch.randn(M, generator=g, dtype=torch.float64) * 0.2
    Ls = [torch.eye(n, dtype=torch.float64) * 0.6 + 0.05 * torch.randn(n, n, generator=g, dtype=torch.float64) for n in Ms]
    return meshes, X, y, l, s2, noise, m, Ls


def oracle_value_and_grads(family, meshes, X, y, l, s2, noise, m, Ls, scale=1.0):
    l = l.clone().requires_grad_(True)
    s2 = s2.clone().requires_grad_(True)
    noise = noise.clone().requires_grad_(True)
    m = m.clone().requires_grad_(True)
    Ls = [L.clone().requires_grad_(True) for L in Ls]
    elbo = O.elbo_structured(family, meshes, X, y, l, s2, noise, m, Ls, ref_quirks=False, scale=scale)
    grads = torch.autograd.grad(elbo, [l, s2, noise, m] + Ls)
    return elbo.detach(), grads


def relerr(a, b):
    a = a.detach().cpu().to(torch.float64).reshape(-1)
    b = b.detach().cpu().to(torch.float64).reshape(-1)
    return ((a - b).norm() / b.norm().clamp_min(1e-300)).item()


CASES = [
    # knots, N
    ((12,), 700),
    ((9, 7), 900),
    ((70, 13), 5000),
    ((6, 66, 5), 4000),
    ((130, 9), 3000),
    ((150, 70), 3000),
    ((37, 70, 9), 2500),
]


@pytest.mark.parametrize("layout", ["raw", "packed_sorted", "packed_unsorted"])
@pytest.mark.parametrize("knots,N", CASES)
@pytest.mark.parametrize("dtype,tol", [(torch.float64, 1e-9), (torch.float32, 1e-3)])
def test_elbo_and_grads_match_oracle_b1(vg, dev, knots, N, dtype, tol, layout):
    D = len(knots)
    meshes, X, y, l, s2, noise, m, Ls = make_problem(knots, N, seed=42 + D)
    Xq = X.to(dtype)          # quantise the observations once so oracle and kernel see identical inputs
    yq = y.to(dtype)
    scale = 1.7
    elbo_ref, g_ref = oracle_value_and_grads(O.B1_ASVGP, meshes, Xq.to(torch.float64), yq.to(torch.float64),
                                             l, s2, noise, m, Ls, scale=scale)
    plan = vg.GridPlan(vg.B1_ASVGP, meshes, dtype, dev)
    theta = torch.cat([l, s2, noise.reshape(1)]).to(dev)
    Lcat = torch.cat([L.reshape(-1) for L in Ls]).to(dev)
    xs = [Xq[:, d].contiguous().to(dev) for d in range(D)]
    if layout == "raw":
        out, dtheta, dm, dL = plan.step(theta, m.to(dev), Lcat, xs, yq.to(dev), ell_scale=scale)
    else:
        packed = plan.pack(xs, yq.to(dev), sort_by_cell=(layout == "packed_sorted"))
        assert packed.n == N and packed.run_len % 4 == 0
        out, dtheta, dm, dL = plan.step(theta, m.to(dev), Lcat, packed, None, ell_scale=scale)
    assert plan.read_info() == 0
    assert out[3].item() == N
    assert abs(out[0].item() - elbo_ref.item()) <= tol * abs(elbo_ref.item()), (out.cpu(), elbo_ref)
    assert relerr(dtheta[:D], g_ref[0]) < tol * 10, ("dl", dtheta[:D].cpu(), g_ref[0])
    assert relerr(dtheta[D:2 * D], g_ref[1]) < tol * 10, ("ds2", dtheta[D:2 * D].cpu(), g_ref[1])
    assert relerr(dtheta[2 * D], g_ref[2]) < tol * 10, ("dnoise", dtheta[2 * D].cpu(), g_ref[2])
    assert relerr(dm, g_ref[3]) < tol * 10, "dm"
    off = 0
    for d, n in enumerate(plan.m_per_dim):
        dLd = dL[off:off + n * n].reshape(n, n).cpu()
        off += n * n
        assert torch.count_nonzero(torch.triu(dLd, 1)) == 0
        assert relerr(torch.tril(dLd), torch.tril(g_ref[4 + d])) < tol * 10, ("dL", d)


B0_CASES = [((14,), 600), ((10, 8), 700), ((71, 14), 1500)]


@pytest.mark.parametrize("knots,N", B0_CASES)
@pytest.mark.parametrize("dtype,tol", [(torch.float64, 1e-8), (torch.float32, 1e-3)])
def test_elbo_and_grads_match_oracle_b0(vg, dev, knots, N, dtype, tol):
    """B0 (cell-integrated Matern-1/2) family: dense, hyper-parameter dependent features; observations partly outside
    the mesh (the features are non-zero there)."""
    D = len(knots)
    meshes, X, y, l, s2, noise, m, Ls = make_problem(knots, N, seed=77 + D, family=O.B0_GRIDDED)
    l = l * 0.3 + 0.03            # keep l / delta where the reference's float32-rounded Toeplitz factor is PD
    Xq, yq = X.to(dtype), y.to(dtype)
    scale = 1.3
    elbo_ref, g_ref = oracle_value_and_grads(O.B0_GRIDDED, meshes, Xq.to(torch.float64), yq.to(torch.float64),
                                             l, s2, noise, m, Ls, scale=scale)
    plan = vg.GridPlan(vg.B0_GRIDDED, meshes, dtype, dev)
    theta = torch.cat([l, s2, noise.reshape(1)]).to(dev)
    Lcat = torch.cat([L.reshape(-1) for L in Ls]).to(dev)
    xs = [Xq[:, d].contiguous().to(dev) for d in range(D)]
    out, dtheta, dm, dL = plan.step(theta, m.to(dev), Lcat, xs, yq.to(dev), ell_scale=scale)
    assert plan.read_info() == 0
    assert out[3].item() == N
    assert abs(out[0].item() - elbo_ref.item()) <= tol * abs(elbo_ref.item()), (out.cpu(), elbo_ref)
    assert relerr(dtheta[:D], g_ref[0]) < tol * 10, ("dl", dtheta[:D].cpu(), g_ref[0])
    assert relerr(dtheta[D:2 * D], g_ref[1]) < tol * 10, ("ds2", dtheta[D:2 * D].cpu(), g_ref[1])
    assert relerr(dtheta[2 * D], g_ref[2]) < tol * 10, ("dnoise", dtheta[2 * D].cpu(), g_ref[2])
    assert relerr(dm, g_ref[3]) < tol * 10, "dm"
    off = 0
    for d, n in enumerate(plan.m_per_dim):
        dLd = dL[off:off + n * n].reshape(n, n).cpu()
        off += n * n
        assert relerr(torch.tril(dLd), torch.tril(g_ref[4 + d])) < tol * 10, ("dL", d)


@pytest.mark.parametrize("pset", ["raw0", "raw1"])
def test_b0_1d_matches_reference_collapsed_bound_at_optimal_q(vg, dev, golden_dir, pset):
    """Direct pin to numbers produced by the reference's own code (oracle/make_golden.py, case G3:
    gridded_univariate_structure.Matern12GriddedGP): in 1-D every covariance is a 'Kronecker product of one factor', so
    the CUDA uncollapsed bound evaluated at the reference's optimal q(v) = N(m*, S*) must equal the reference's
    collapsed `_elbo()`."""
    import os
    ref = np.load(os.path.join(golden_dir, "reference_models.npz"))
    key = f"G3_griddedgp1d.{pset}"
    x = torch.from_numpy(ref["g3.x"])
    y = torch.from_numpy(ref["g3.y"])
    m_star = torch.from_numpy(ref[key + ".q_mean"])
    S_star = torch.from_numpy(ref[key + ".q_cov"])
    elbo_ref = float(ref[key + ".elbo"])
    raw = {"raw0": (0.0, 0.0, 0.0), "raw1": (-0.3, 0.5, -3.0)}[pset]       # (raw_l, raw_s, raw_noise), make_golden.py
    l, s2, noise = O.constrain(torch.tensor([raw[0]], dtype=torch.float64), torch.tensor([raw[1]], dtype=torch.float64),
                               torch.tensor(raw[2], dtype=torch.float64))
    mesh = torch.linspace(0.0, 2.0, 33)
    S_sym = 0.5 * (S_star + S_star.T)
    Lc = torch.linalg.cholesky(S_sym)
    plan = vg.GridPlan(vg.B0_GRIDDED, [mesh], torch.float64, dev)
    theta = torch.cat([l, s2, noise.reshape(1)]).to(dev)
    out, dtheta, dm, dL = plan.step(theta, m_star.to(dev).contiguous(), Lc.reshape(-1).to(dev).contiguous(),
                                    [x.to(dev).contiguous()], y.to(dev).contiguous())
    assert plan.read_info() == 0
    assert abs(out[0].item() - elbo_ref) < 1e-6 * abs(elbo_ref), (out[0].item(), elbo_ref)
    # (m*, S*) is the maximiser of the uncollapsed bound: its gradient w.r.t. m vanishes there
    alpha = plan.workspace(vg._lib.WS_ALPHA)
    assert dm.abs().max().item() < 1e-6 * alpha.abs().max().item()


def test_simt_and_dmma_paths_agree(vg, dev):
    """The dense grid side (B0 family) with the DMMA and the SIMT inner loop of its GEMMs, whole step."""
    knots, N = B0_CASES[2]
    meshes, X, y, l, s2, noise, m, Ls = make_problem(knots, N, seed=5, family=O.B0_GRIDDED)
    l = l * 0.3 + 0.03            # as in the B0 parity test: the reference's float32-rounded Toeplitz factor stays PD
    plan = vg.GridPlan(vg.B0_GRIDDED, meshes, torch.float64, dev)
    theta = torch.cat([l, s2, noise.reshape(1)]).to(dev)
    Lcat = torch.cat([L.reshape(-1) for L in Ls]).to(dev)
    xs = [X[:, d].contiguous().to(dev) for d in range(2)]
    res = []
    try:
        for mode in (1, 0):
            vg._lib.load().vggp_set_gemm_mode(mode)
            out, dtheta, dm, dL = plan.step(theta, m.to(dev), Lcat, xs, y.to(dev))
            res.append((out.clone(), dtheta.clone(), dm.clone(), dL.clone()))
    finally:
        vg._lib.load().vggp_set_gemm_mode(1)
    for a, b in zip(res[0], res[1]):
        assert relerr(a, b) < 1e-10


def test_all_observations_outside_the_mesh(vg, dev):
    meshes = [torch.linspace(0, 1, 8), torch.linspace(0, 1, 6)]
    N = 300
    X = torch.rand(N, 2, dtype=torch.float64) + 2.0
    y = torch.randn(N, dtype=torch.float64)
    _, _, _, l, s2, noise, m, Ls = make_problem((8, 6), 10, seed=1)
    elbo_ref, g_ref = oracle_value_and_grads(O.B1_ASVGP, meshes, X, y, l, s2, noise, m, Ls)
    plan = vg.GridPlan(vg.B1_ASVGP, meshes, torch.float64, dev)
    theta = torch.cat([l, s2, noise.reshape(1)]).to(dev)
    Lcat = torch.cat([L.reshape(-1) for L in Ls]).to(dev)
    out, dtheta, dm, dL = plan.step(theta, m.to(dev), Lcat, [X[:, 0].contiguous().to(dev), X[:, 1].contiguous().to(dev)], y.to(dev))
    assert abs(out[0].item() - elbo_ref.item()) < 1e-9 * abs(elbo_ref.item())
    assert relerr(dm, g_ref[3]) < 1e-8


def test_empty_shard(vg, dev):
    # n = 0 observations: ELBO = -KL, gradients finite
    meshes, X, y, l, s2, noise, m, Ls = make_problem((9, 7), 10, seed=2)
    elbo_ref, g_ref = oracle_value_and_grads(O.B1_ASVGP, meshes, X[:0], y[:0], l, s2, noise, m, Ls)
    plan = vg.GridPlan(vg.B1_ASVGP, meshes, torch.float64, dev)
    theta = torch.cat([l, s2, noise.reshape(1)]).to(dev)
    Lcat = torch.cat([L.reshape(-1) for L in Ls]).to(dev)
    e = torch.empty(0, dtype=torch.float64, device=dev)
    out, dtheta, dm, dL = plan.step(theta, m.to(dev), Lcat, [e, e], e)
    assert abs(out[0].item() - elbo_ref.item()) < 1e-9 * abs(elbo_ref.item())
    assert abs(out[0].item() + out[2].item()) < 1e-9 * abs(out[2].item())
    assert relerr(dm, g_ref[3]) < 1e-8


def test_linearity_in_shards(vg, dev):
    """Size-independent property: the gradient buffer of a data set is the sum of the buffers of its shards
    (this is what the all-reduce relies on)."""
    meshes, X, y, l, s2, noise, m, Ls = make_problem((33, 21), 20000, seed=9)
    plan = vg.GridPlan(vg.B1_ASVGP, meshes, torch.float64, dev)
    theta = torch.cat([l, s2, noise.reshape(1)]).to(dev)
    Lcat = torch.cat([L.reshape(-1) for L in Ls]).to(dev)
    plan.grid_forward(theta, m.to(dev), Lcat)
    xs = [X[:, d].contiguous().to(dev) for d in range(2)]
    yd = y.to(dev)
    plan.obs_fwd_bwd(xs, yd)
    full = plan.gbuf.clone().view(torch.float64)
    acc = torch.zeros_like(full)
    for lo, hi in ((0, 7000), (7000, 7001), (7001, 20000)):
        plan.obs_fwd_bwd([x[lo:hi].contiguous() for x in xs], yd[lo:hi].contiguous())
        acc += plan.gbuf.view(torch.float64)
    assert relerr(acc, full) < 1e-12


def _model_module(name):
    return importlib.import_module(f"variational-gridded-gaussian-processes_b200.models.sparse.{name}")


def test_model_class_training_loop_api(vg, dev):
    """Drop-in API: constructor signature, .to(float64), parameters(), -_elbo().backward(), Adam step; ELBO and raw
    parameter gradients against the oracle with the same softplus parameterisation."""
    gks = _model_module("gridded_kronecker_structure")
    g = torch.Generator().manual_seed(0)
    N = 625
    X = torch.rand(N, 2, generator=g, dtype=torch.float64)
    y = torch.sin(5 * X[:, 0]) + torch.cos(7 * X[:, 1]) + 0.05 * torch.randn(N, generator=g, dtype=torch.float64)
    model = gks.GriddedMatern12ASVGP(X, y, 10, 1, (0, 1), (0, 1)).to(torch.float64).to(dev)
    names = [n for n, _ in model.named_parameters()]
    for want in ("likelihood.noise_covar.raw_noise", "kernel_1.raw_outputscale", "kernel_1.base_kernel.raw_lengthscale",
                 "kernel_2.raw_outputscale", "kernel_2.base_kernel.raw_lengthscale", "variational_mean",
                 "variational_chol_1", "variational_chol_2"):
        assert want in names
    with torch.no_grad():
        model.variational_mean.normal_(0, 0.1, generator=None)
        model.kernel_1.base_kernel.lengthscale = 0.4
        model.likelihood.noise = 0.05
    assert abs(model.kernel_1.base_kernel.lengthscale.item() - 0.4) < 1e-12
    elbo = model._elbo()
    assert elbo.dim() == 0 and elbo.requires_grad
    (-elbo).backward()
    # oracle with raw parameters
    raw_l = torch.stack([model.kernel_1.base_kernel.raw_lengthscale.detach().cpu().reshape(()),
                         model.kernel_2.base_kernel.raw_lengthscale.detach().cpu().reshape(())]).requires_grad_(True)
    raw_s = torch.stack([model.kernel_1.raw_outputscale.detach().cpu(), model.kernel_2.raw_outputscale.detach().cpu()]).requires_grad_(True)
    raw_n = model.likelihood.noise_covar.raw_noise.detach().cpu().reshape(()).requires_grad_(True)
    l, s2, noise = O.constrain(raw_l, raw_s, raw_n)
    meshes = [O.make_padded_mesh(0, 1, 10, 1)] * 2
    m = model.variational_mean.detach().cpu()
    Ls = [model.variational_chol_1.detach().cpu(), model.variational_chol_2.detach().cpu()]
    ref = O.elbo_structured(O.B1_ASVGP, meshes, X, y, l, s2, noise, m, Ls, ref_quirks=False)
    gl, gs, gn = torch.autograd.grad(-ref, [raw_l, raw_s, raw_n])
    assert abs(elbo.item() - ref.item()) < 1e-9 * abs(ref.item())
    assert abs(model.kernel_1.base_kernel.raw_lengthscale.grad.item() - gl[0].item()) < 1e-7 * abs(gl[0].item())
    assert abs(model.kernel_2.raw_outputscale.grad.item() - gs[1].item()) < 1e-7 * abs(gs[1].item())
    assert abs(model.likelihood.noise_covar.raw_noise.grad.item() - gn.item()) < 1e-7 * abs(gn.item())
    # a few Adam steps must increase the bound
    opt = torch.optim.Adam(model.parameters(), lr=0.05)
    first = None
    for it in range(15):
        opt.zero_grad()
        loss = -model._elbo()
        loss.backward()
        opt.step()
        first = loss.item() if first is None else first
    assert (-model._elbo()).item() < first


def test_packing_is_a_permutation(vg, dev):
    """vggp_obs_pack keeps every observation exactly once (multiset equality), pads with NaN / 0, and with
    sort_by_cell orders each lane's run by flat cell id."""
    meshes = [torch.linspace(0, 1, 40), torch.linspace(0, 1, 23)]
    g = torch.Generator().manual_seed(3)
    N = 10007
    X = (torch.rand(N, 2, generator=g, dtype=torch.float64) * 1.2 - 0.1).to(torch.float32)
    y = torch.randn(N, generator=g, dtype=torch.float64).to(torch.float32)
    plan = vg.GridPlan(vg.B1_ASVGP, meshes, torch.float32, dev)
    xs = [X[:, d].contiguous().to(dev) for d in range(2)]
    for sort in (False, True):
        pk = plan.pack(xs, y.to(dev), sort_by_cell=sort)
        R = pk.run_len
        yp = pk.yp.cpu()
        x1p, x2p = pk.xp[0].cpu(), pk.xp[1].cpu()
        real = ~torch.isnan(x1p)
        assert int(real.sum()) == N
        assert torch.all(yp[~real] == 0) and torch.all(torch.isnan(x2p[~real]))
        key_in = torch.sort(X[:, 0].to(torch.float64) * 7.0 + X[:, 1].to(torch.float64) * 13.0 + y.to(torch.float64))[0]
        key_pk = torch.sort(x1p[real].to(torch.float64) * 7.0 + x2p[real].to(torch.float64) * 13.0 + yp[real].to(torch.float64))[0]
        assert torch.equal(key_in, key_pk)
        # un-transpose: stream position s = (32 w + l) R + j  lives at  w*32R + (j//4)*128 + l*4 + j%4
        nw = x1p.numel() // (32 * R)
        st = x1p.reshape(nw, R // 4, 32, 4).permute(0, 2, 1, 3).reshape(-1)[:N]
        st2 = x2p.reshape(nw, R // 4, 32, 4).permute(0, 2, 1, 3).reshape(-1)[:N]
        if not sort:
            assert torch.equal(st, X[:, 0]) and torch.equal(st2, X[:, 1])
        else:
            c1, _, _ = O.b1_stencil(meshes[0], st.to(torch.float32))
            c2, _, _ = O.b1_stencil(meshes[1], st2.to(torch.float32))
            ncell = 39 * 22
            key = torch.where((c1 >= 0) & (c2 >= 0), c1 * 22 + c2, torch.full_like(c1, ncell))
            assert torch.all(key[1:] >= key[:-1])


@pytest.mark.parametrize("dtype,tol", [(torch.float64, 1e-9), (torch.float32, 2e-4)])
def test_point_prediction_matches_dense_formulas(vg, dev, dtype, tol):
    """posterior(x*) marginals against the dense formulas of kronecker_structure.py:199-230 written with (m, S):
    mean = Kuf*^T Kuu^-1 m,  var = k** - diag(Kuf*^T Kuu^-1 Kuf*) + diag(Kuf*^T Kuu^-1 S Kuu^-1 Kuf*)."""
    knots = (11, 8)
    meshes, X, y, l, s2, noise, m, Ls = make_problem(knots, 50, seed=21)
    g = torch.Generator().manual_seed(4)
    Xs = (torch.rand(400, 2, generator=g, dtype=torch.float64) * 1.2 - 0.1).to(dtype)
    Kuu, Kuf, _, _ = O.dense_Kuu_Kuf(O.B1_ASVGP, meshes, Xs.to(torch.float64), l, s2, ref_quirks=False)
    S = O.kron_cov_from_factors(Ls)
    A = torch.linalg.solve(Kuu, Kuf)
    mean_ref = A.T @ m
    var_ref = torch.prod(s2) - (Kuf * A).sum(0) + (A * (S @ A)).sum(0)
    plan = vg.GridPlan(vg.B1_ASVGP, meshes, dtype, dev)
    theta = torch.cat([l, s2, noise.reshape(1)]).to(dev)
    Lcat = torch.cat([L.reshape(-1) for L in Ls]).to(dev)
    plan.grid_forward(theta, m.to(dev), Lcat)
    mean, var = plan.predict([Xs[:, 0].contiguous().to(dev), Xs[:, 1].contiguous().to(dev)])
    scale = max(1.0, mean_ref.abs().max().item())
    assert (mean.cpu().to(torch.float64) - mean_ref).abs().max().item() < tol * scale
    assert (var.cpu().to(torch.float64) - var_ref).abs().max().item() < tol * max(1.0, var_ref.abs().max().item())
    # model-level API
    gks = _model_module("kronecker_structure")
    model = gks.Matern12B1SplineASVGP(X, y, 9, (0, 1), (0, 1)).to(dtype).to(dev)
    post = model.posterior(Xs.to(dev))
    pred = model.posterior_predictive(Xs.to(dev))
    assert post.mean.shape == (400,) and torch.all(pred.variance > post.variance)
    lo, hi = post.confidence_region()
    assert torch.all(hi >= lo)


def test_q_v_cell_integrals_match_dense_formulas(vg, dev):
    """GriddedMatern12ASVGP.q_v() marginals against the dense matrices the reference builds (_Kvu :831-845,
    _Kvv :847-901) with the intended covariance  Kvv - Kvu Kuu^-1 Kuv + Kvu Kuu^-1 S Kuu^-1 Kuv."""
    gks = _model_module("gridded_kronecker_structure")
    g = torch.Generator().manual_seed(12)
    nb, pad = 6, 1
    X = torch.rand(200, 2, generator=g, dtype=torch.float64)
    y = torch.sin(4 * X[:, 0]) + 0.1 * torch.randn(200, generator=g, dtype=torch.float64)
    model = gks.GriddedMatern12ASVGP(X, y, nb, pad, (0, 1), (0, 1)).to(torch.float64).to(dev)
    with torch.no_grad():
        model.variational_mean.copy_(torch.randn(model.M, generator=g, dtype=torch.float64).to(dev))
        for c in model._chols():
            c.add_(0.1 * torch.randn(c.shape, generator=g, dtype=torch.float64).to(dev))
        model.kernel_1.base_kernel.lengthscale = 0.3
        model.kernel_2.outputscale = 1.4
    qv = model.q_v()
    # dense reference construction on the CPU
    meshes = [O.make_padded_mesh(0, 1, nb, pad)] * 2
    l = torch.stack([model.kernel_1.base_kernel.lengthscale.detach().cpu().reshape(()),
                     model.kernel_2.base_kernel.lengthscale.detach().cpu().reshape(())])
    s2 = torch.stack([model.kernel_1.outputscale.detach().cpu(), model.kernel_2.outputscale.detach().cpu()])
    Ks = [O.kuu_b1(meshes[d], l[d], s2[d], ref_quirks=False) for d in range(2)]
    Kuu = torch.kron(Ks[0], Ks[1])
    Kd = meshes[0].numel()
    delta = (meshes[0][1] - meshes[0][0]).to(torch.float64)
    first_row = torch.nn.functional.pad(torch.stack([delta, delta]), (pad, Kd - (pad + 2)))
    Kvu_d = torch.vstack([torch.roll(first_row, i) for i in range(nb)])
    Kvu = torch.kron(Kvu_d, Kvu_d)
    b0mesh = torch.linspace(0, 1, nb + 1)
    Kvv = torch.kron(O.kuu_b0(b0mesh, l[0], s2[0]), O.kuu_b0(b0mesh, l[1], s2[1]))
    m = model.variational_mean.detach().cpu()
    S = O.kron_cov_from_factors([c.detach().cpu() for c in model._chols()])
    A = torch.linalg.solve(Kuu, Kvu.T)
    mean_ref = A.T @ m
    cov_ref = Kvv - Kvu @ A + A.T @ S @ A
    assert relerr(qv.mean, mean_ref) < 1e-9
    assert relerr(qv.variance, torch.diagonal(cov_ref)) < 1e-9


def test_full_size_properties_bench_config(vg, dev):
    """BASELINE.json configs[2] / [4] shape (2-D along-track observations, 512 x 512 grid, float32), N = 2^24, where
    the oracle cannot run: size-independent properties instead.
      (1) the cell-sorted packed layout, the acquisition-order packed layout and the plain-array entry point give the
          same ELBO and gradients (different summation orders only);
      (2) linearity: the gradient buffer of the data set equals the sum of the buffers of two shards;
      (3) every observation is counted once (out[3] == N) and the ELBO is finite and negative."""
    import bench
    N = 1 << 24
    meshes = [torch.linspace(0, 1, k) for k in bench.KNOTS]
    xs, y = bench.make_tracks(0, N, N, dev, torch.float32)
    theta, m, Ls = bench.make_params(meshes, dev)
    theta, m = theta.to(dev), m.to(dev)
    Lcat = torch.cat([L.reshape(-1) for L in Ls]).to(dev).contiguous()
    plan = vg.GridPlan(vg.B1_ASVGP, meshes, torch.float32, dev)
    pk_sorted = plan.pack(xs, y, sort_by_cell=True)
    pk_acq = plan.pack(xs, y, sort_by_cell=False)
    res = []
    for obs, yy in ((pk_sorted, None), (pk_acq, None), (xs, y)):
        out, dtheta, dm, dL = plan.step(theta, m, Lcat, obs, yy)
        res.append((out.clone(), dtheta.clone(), dm.clone(), dL.clone()))
    assert plan.read_info() == 0
    assert res[0][0][3].item() == N and torch.isfinite(res[0][0]).all() and res[0][0][0].item() < 0
    for k in (1, 2):
        assert abs(res[k][0][0].item() - res[0][0][0].item()) < 1e-5 * abs(res[0][0][0].item())
        for a, b in zip(res[k][1:], res[0][1:]):
            assert relerr(a, b) < 1e-3
    # linearity in shards on the sorted layout
    plan.grid_forward(theta, m, Lcat)
    plan.obs_fwd_bwd(pk_sorted)
    obs_full, scal_full = [t.clone() for t in plan.gbuf_views()]
    half = N // 2 + 12345
    acc_obs = torch.zeros_like(obs_full, dtype=torch.float64)
    acc_scal = torch.zeros_like(scal_full)
    for lo, hi in ((0, half), (half, N)):
        pk = plan.pack([x[lo:hi].contiguous() for x in xs], y[lo:hi].contiguous(), sort_by_cell=True)
        plan.obs_fwd_bwd(pk)
        o, sc = plan.gbuf_views()
        acc_obs += o.to(torch.float64)
        acc_scal += sc
    assert relerr(acc_obs, obs_full) < 1e-4
    assert abs(acc_scal[1].item() - N) == 0 and abs(acc_scal[0].item() - scal_full[0].item()) < 1e-5 * abs(scal_full[0].item())


def test_bench_configuration_two_wave_run_length(vg, dev):
    """The bench configuration itself (N = 2^26, 512 x 512, float32): above 48.5 M observations per GPU the packed layout
    balances the run length to two waves of chunks per resident warp (pack_geometry).  The ELBO must be the one every
    round-1 run of this data set and these parameters produced (-177008473.3, layouts agreeing to 1e-9), and every
    observation must be counted once."""
    import bench
    N = bench.N_TOTAL
    meshes = [torch.linspace(0, 1, k) for k in bench.KNOTS]
    xs, y = bench.make_tracks(0, N, N, dev, torch.float32)
    theta, m, Ls = bench.make_params(meshes, dev)
    plan = vg.GridPlan(vg.B1_ASVGP, meshes, torch.float32, dev)
    pk = plan.pack(xs, y, sort_by_cell=True)
    assert pk.run_len % 4 == 0 and 16 <= pk.run_len <= 512
    out, dtheta, dm, dL = plan.step(theta.to(dev), m.to(dev), torch.cat([L.reshape(-1) for L in Ls]).to(dev).contiguous(), pk, None)
    assert plan.read_info() == 0 and out[3].item() == N
    assert abs(out[0].item() - (-177008473.3)) < 1e-6 * 177008473.3
    assert torch.isfinite(dtheta).all() and torch.isfinite(dm).all() and torch.isfinite(dL).all()


@pytest.mark.parametrize("dtype,tol", [(torch.float64, 1e-9), (torch.float32, 1e-3)])
def test_first_knot_hit_followed_by_points_left_of_the_mesh(vg, dev, dtype, tol):
    """Regression: an observation exactly on the first knot followed, in the same lane run of an UNSORTED stream, by
    observations left of the mesh (they must contribute y^2 only).  Found under the SIMT emulator
    (tests/test_device_emul.py); the plain-array entry point keeps the input order."""
    meshes = [torch.linspace(0, 1, 5)]
    g = torch.Generator().manual_seed(5)
    N = 64
    x = 0.025 + 0.2 * torch.rand(N, generator=g, dtype=torch.float64)          # everything in cell 0 ...
    x[10] = 0.0                                                                # ... one exact first-knot hit ...
    x[11:20] = -0.05 * torch.arange(1, 10, dtype=torch.float64)                # ... then points left of the mesh
    y = torch.sin(3 * x) + 0.1 * torch.randn(N, generator=g, dtype=torch.float64)
    l, s2, noise = torch.tensor([0.3], dtype=torch.float64), torch.tensor([0.9], dtype=torch.float64), torch.tensor(0.07, dtype=torch.float64)
    m = 0.2 * torch.randn(5, generator=g, dtype=torch.float64)
    Ls = [torch.eye(5, dtype=torch.float64) * 0.6 + 0.05 * torch.randn(5, 5, generator=g, dtype=torch.float64)]
    xq, yq = x.to(dtype), y.to(dtype)
    elbo_ref, g_ref = oracle_value_and_grads(O.B1_ASVGP, meshes, xq.to(torch.float64).reshape(-1, 1), yq.to(torch.float64),
                                             l, s2, noise, m, Ls)
    plan = vg.GridPlan(vg.B1_ASVGP, meshes, dtype, dev)
    theta = torch.cat([l, s2, noise.reshape(1)]).to(dev)
    for layout in ("raw", "packed_unsorted"):
        obs = [xq.to(dev)] if layout == "raw" else plan.pack([xq.to(dev)], yq.to(dev), sort_by_cell=False)
        out, dtheta, dm, dL = plan.step(theta, m.to(dev), Ls[0].reshape(-1).to(dev), obs, yq.to(dev) if layout == "raw" else None)
        assert abs(out[0].item() - elbo_ref.item()) <= tol * abs(elbo_ref.item()), layout
        assert relerr(dm, g_ref[3]) < tol * 10, layout


def test_model_refuses_cpu(vg):
    ks = _model_module("kronecker_structure")
    X = torch.rand(10, 2, dtype=torch.float64)
    y = torch.rand(10, dtype=torch.float64)
    model = ks.Matern12B1SplineASVGP(X, y, 5, (0, 1), (0, 1))
    with pytest.raises(RuntimeError):
        model._elbo()


def test_two_live_plans_of_different_sizes(vg, dev):
    """The dynamic-shared-memory opt-in of a kernel is a per-function, process-wide attribute: creating (and using) a
    second, smaller plan must not lower what an earlier, larger plan needs (1-D, 1100 knots, float64: the band tables of
    the per-observation kernel and the staging of the theta kernel are both above the 48 KB default)."""
    def run(plan, prob, packed):
        meshes, X, y, l, s2, noise, m, Ls = prob
        theta = torch.cat([l, s2, noise.reshape(1)]).to(dev)
        Lcat = torch.cat([L.reshape(-1) for L in Ls]).to(dev)
        xs = [X[:, d].contiguous().to(dev) for d in range(X.shape[1])]
        if packed:
            out = plan.step(theta, m.to(dev), Lcat, plan.pack(xs, y.to(dev), sort_by_cell=True), None)
        else:
            out = plan.step(theta, m.to(dev), Lcat, xs, y.to(dev))
        torch.cuda.synchronize()
        assert plan.read_info() == 0
        return [t.clone() for t in out]

    big = make_problem((1100,), 6000, seed=5)
    small = make_problem((9, 7), 500, seed=6)
    plan_big = vg.GridPlan(vg.B1_ASVGP, big[0], torch.float64, dev)
    first = [run(plan_big, big, packed) for packed in (False, True)]
    plan_small = vg.GridPlan(vg.B1_ASVGP, small[0], torch.float64, dev)
    for packed in (False, True):
        run(plan_small, small, packed)
    plan_1d = vg.GridPlan(vg.B1_ASVGP, [torch.linspace(0, 1, 12)], torch.float32, dev)      # what B1SplineBasis._plan makes
    assert plan_1d.M == 12
    again = [run(plan_big, big, packed) for packed in (False, True)]
    for which, (a, b) in enumerate(zip(first, again)):
        for k, (ta, tb) in enumerate(zip(a, b)):
            assert relerr(ta, tb) < 1e-9, ("the large plan changed its results after smaller plans were used", which, k)
    # and it is the right answer (1100 knots: the factor's condition number limits the agreement, not the kernels)
    elbo_ref, g_ref = oracle_value_and_grads(O.B1_ASVGP, *big)
    for which in range(2):
        assert abs(again[which][0][0].item() - elbo_ref.item()) <= 1e-6 * abs(elbo_ref.item()), (which, again[which][0][0].item(), elbo_ref.item())


@pytest.mark.parametrize("dtype,tol", [(torch.float64, 1e-10), (torch.float32, 2e-5)])
def test_host_entry_point_matches_device_step(vg, dev, dtype, tol):
    """vggp_elbo_host (pinned host buffers in, host results out; the call bench.py's e2e leg times): single-shot for a small
    shard, and with the observations crossing PCIe in chunks on a second stream while the per-observation kernel of the
    previous chunk runs (chunk size lowered through the debug hook so that 300 000 observations make 5 chunks)."""
    import ctypes as C
    knots, N = (70, 33), 300_000
    D = len(knots)
    meshes, X, y, l, s2, noise, m, Ls = make_problem(knots, N, seed=8)
    Xq, yq = X.to(dtype), y.to(dtype)
    plan = vg.GridPlan(vg.B1_ASVGP, meshes, dtype, dev)
    theta = torch.cat([l, s2, noise.reshape(1)])
    Lcat = torch.cat([L.reshape(-1) for L in Ls]).contiguous()
    xs = [Xq[:, d].contiguous() for d in range(D)]
    ref = plan.step(theta.to(dev), m.to(dev), Lcat.to(dev), [x.to(dev) for x in xs], yq.to(dev), ell_scale=1.3)
    ref = [t.cpu().clone() for t in ref]
    lib = vg._lib.load()
    xs_h = [x.pin_memory() for x in xs]
    y_h, th_h, m_h, L_h = yq.pin_memory(), theta.pin_memory(), m.pin_memory(), Lcat.pin_memory()
    stream = torch.cuda.current_stream(dev).cuda_stream
    for chunk in (1 << 23, 65536):
        lib.vggp_debug_host_chunk(chunk)
        try:
            out_h = torch.empty(4, dtype=torch.float64).pin_memory()
            dth_h = torch.empty(2 * D + 1, dtype=torch.float64).pin_memory()
            dm_h = torch.empty(plan.M, dtype=torch.float64).pin_memory()
            dL_h = torch.empty(plan.L_total, dtype=torch.float64).pin_memory()
            ptrs = (C.c_void_p * D)(*[t.data_ptr() for t in xs_h])
            for _ in range(2):          # the second call reuses the staging buffers, the copy stream and the events
                vg._lib.check(lib.vggp_elbo_host(plan.handle, ptrs, y_h.data_ptr(), N, th_h.data_ptr(), m_h.data_ptr(),
                                                 L_h.data_ptr(), 1.3, out_h.data_ptr(), dth_h.data_ptr(), dm_h.data_ptr(),
                                                 dL_h.data_ptr(), stream))
            assert out_h[3].item() == N
            for got, want in zip((out_h, dth_h, dm_h, dL_h), ref):
                assert relerr(got, want) < tol, chunk
        finally:
            lib.vggp_debug_host_chunk(1 << 23)


@pytest.mark.parametrize("knots,N", [((14,), 600), ((10, 8), 700), ((70, 14), 1500)])
@pytest.mark.parametrize("dtype,tol", [(torch.float64, 1e-8), (torch.float32, 1e-3)])
def test_elbo_and_grads_match_oracle_svgp(vg, dev, knots, N, dtype, tol):
    """Product-grid SVGP family (kronecker_structure.py:287-338 Matern12SVGP): kernel features s2 exp(-|x - z_i| / l) at
    non-uniformly spaced inducing points, Kuu_d = k_d(Z, Z); dense-feature kernel + dense factor path, every gradient block."""
    D = len(knots)
    meshes, X, y, l, s2, noise, m, Ls = make_problem(knots, N, seed=55 + D, family=O.SVGP_GRID, x_lo=-0.2, x_hi=1.2)
    meshes = [(t ** (1.0 + 0.3 * d)).to(torch.float32) for d, t in enumerate(meshes)]
    Xq, yq = X.to(dtype), y.to(dtype)
    scale = 1.3
    elbo_ref, g_ref = oracle_value_and_grads(O.SVGP_GRID, meshes, Xq.to(torch.float64), yq.to(torch.float64),
                                             l, s2, noise, m, Ls, scale=scale)
    plan = vg.GridPlan(vg.SVGP_GRID, meshes, dtype, dev)
    assert plan.m_per_dim == list(knots)
    theta = torch.cat([l, s2, noise.reshape(1)]).to(dev)
    Lcat = torch.cat([L.reshape(-1) for L in Ls]).to(dev)
    xs = [Xq[:, d].contiguous().to(dev) for d in range(D)]
    out, dtheta, dm, dL = plan.step(theta, m.to(dev), Lcat, xs, yq.to(dev), ell_scale=scale)
    assert plan.read_info() == 0
    assert out[3].item() == N
    assert abs(out[0].item() - elbo_ref.item()) <= tol * abs(elbo_ref.item())
    assert relerr(dtheta[:D], g_ref[0]) < tol * 10
    assert relerr(dtheta[D:2 * D], g_ref[1]) < tol * 10
    assert relerr(dtheta[2 * D], g_ref[2]) < tol * 10
    assert relerr(dm, g_ref[3]) < tol * 10
    off = 0
    for d, n in enumerate(plan.m_per_dim):
        dLd = dL[off:off + n * n].reshape(n, n).cpu()
        off += n * n
        assert relerr(torch.tril(dLd), torch.tril(g_ref[4 + d])) < tol * 10, ("dL", d)
    phi = plan.features_dense(0, xs[0], theta)
    ref = O.svgp_features_dense(meshes[0], Xq[:, 0], l[0], s2[0])
    assert relerr(phi, ref) < (1e-13 if dtype == torch.float64 else 1e-6)
    with pytest.raises(RuntimeError):
        plan.bin(xs, yq.to(dev))                     # this family takes plain observation arrays


def test_svgp_model_class_on_the_gpu(vg, dev):
    """kronecker_structure.Matern12SVGP as a drop-in class on the device: ELBO against the oracle, Adam improves the bound,
    posterior() finite."""
    ks = importlib.import_module("variational-gridded-gaussian-processes_b200.models.sparse.kronecker_structure")
    g = torch.Generator().manual_seed(3)
    N = 2000
    X = torch.rand(N, 2, generator=g, dtype=torch.float64)
    y = torch.sin(5 * X[:, 0]) + torch.cos(7 * X[:, 1]) + 0.05 * torch.randn(N, generator=g, dtype=torch.float64)
    Z = torch.stack([torch.linspace(0, 1, 12), torch.linspace(0, 1, 12) ** 1.2], dim=1)
    model = ks.Matern12SVGP(X, y, Z).to(torch.float64).to(dev)
    with torch.no_grad():
        model.variational_mean.normal_(0, 0.1, generator=None)
        model.kernel_1.base_kernel.lengthscale = 0.3
        model.likelihood.noise = 0.05
    elbo = model._elbo()
    l = torch.stack([model.kernel_1.base_kernel.lengthscale.detach().reshape(()), model.kernel_2.base_kernel.lengthscale.detach().reshape(())]).cpu()
    s2 = torch.stack([model.kernel_1.outputscale.detach().reshape(()), model.kernel_2.outputscale.detach().reshape(())]).cpu()
    ref = O.elbo_structured(O.SVGP_GRID, [model.Z[:, 0].cpu(), model.Z[:, 1].cpu()], X, y, l.to(torch.float64), s2.to(torch.float64),
                            model.likelihood.noise.detach().reshape(()).cpu().to(torch.float64), model.variational_mean.detach().cpu(),
                            [model.variational_chol_1.detach().cpu(), model.variational_chol_2.detach().cpu()], ref_quirks=False)
    assert abs(elbo.item() - ref.item()) < 1e-8 * abs(ref.item())
    opt = torch.optim.Adam(model.parameters(), lr=0.02)
    losses = []
    for _ in range(5):
        opt.zero_grad()
        loss = -model._elbo()
        loss.backward()
        opt.step()
        losses.append(loss.item())
    assert losses[-1] < losses[0]
    post = model.posterior(X[:64].to(dev))
    assert torch.isfinite(post.mean).all() and (post.variance > 0).all()


@pytest.mark.parametrize("knots,N", [((9,), 600), ((7, 11), 700), ((71, 13), 1500)])
@pytest.mark.parametrize("dtype,tol", [(torch.float64, 1e-8), (torch.float32, 1e-3)])
def test_elbo_and_grads_match_oracle_vff(vg, dev, knots, N, dtype, tol):
    """Variational Fourier features (kronecker_structure.py:347-514 Matern12VFFGP, fourier.py:58-88) on domains smaller than
    the data: cosine / sine features inside, exp(-r / l) outside, Kuu_d = diag(alpha) + beta beta^T; every gradient block."""
    D = len(knots)
    meshes, X, y, l, s2, noise, m, Ls = make_problem(knots, N, seed=66 + D, family=O.VFF_GRID, x_lo=-0.2, x_hi=1.2)
    Xq, yq = X.to(dtype), y.to(dtype)
    scale = 1.3
    elbo_ref, g_ref = oracle_value_and_grads(O.VFF_GRID, meshes, Xq.to(torch.float64), yq.to(torch.float64),
                                             l, s2, noise, m, Ls, scale=scale)
    plan = vg.GridPlan(vg.VFF_GRID, meshes, dtype, dev)
    assert plan.m_per_dim == list(knots)
    theta = torch.cat([l, s2, noise.reshape(1)]).to(dev)
    Lcat = torch.cat([L.reshape(-1) for L in Ls]).to(dev)
    xs = [Xq[:, d].contiguous().to(dev) for d in range(D)]
    out, dtheta, dm, dL = plan.step(theta, m.to(dev), Lcat, xs, yq.to(dev), ell_scale=scale)
    assert plan.read_info() == 0
    assert out[3].item() == N
    assert abs(out[0].item() - elbo_ref.item()) <= tol * abs(elbo_ref.item())
    assert relerr(dtheta[:D], g_ref[0]) < tol * 10
    assert relerr(dtheta[D:2 * D], g_ref[1]) < tol * 10
    assert relerr(dtheta[2 * D], g_ref[2]) < tol * 10
    assert relerr(dm, g_ref[3]) < tol * 10
    off = 0
    for d, n in enumerate(plan.m_per_dim):
        dLd = dL[off:off + n * n].reshape(n, n).cpu()
        off += n * n
        assert relerr(torch.tril(dLd), torch.tril(g_ref[4 + d])) < tol * 10, ("dL", d)
    with pytest.raises(RuntimeError):
        vg.GridPlan(vg.VFF_GRID, [torch.linspace(0, 1, 8)], dtype, dev)          # 2 M + 1 knots


def test_vff_model_class_on_the_gpu(vg, dev):
    """kronecker_structure.Matern12VFFGP on the device: ELBO against the oracle, Adam improves the bound, posterior() finite."""
    ks = importlib.import_module("variational-gridded-gaussian-processes_b200.models.sparse.kronecker_structure")
    g = torch.Generator().manual_seed(4)
    N = 2000
    X = torch.rand(N, 2, generator=g, dtype=torch.float64)
    y = torch.sin(5 * X[:, 0]) + torch.cos(7 * X[:, 1]) + 0.05 * torch.randn(N, generator=g, dtype=torch.float64)
    model = ks.Matern12VFFGP(X, y, 6, (-0.125, 1.125), (0.125, 0.875)).to(torch.float64).to(dev)
    with torch.no_grad():
        model.variational_mean.normal_(0, 0.1)
        model.kernel_1.base_kernel.lengthscale = 0.3
        model.likelihood.noise = 0.05
    elbo = model._elbo()
    l = torch.stack([model.kernel_1.base_kernel.lengthscale.detach().reshape(()), model.kernel_2.base_kernel.lengthscale.detach().reshape(())]).cpu()
    s2 = torch.stack([model.kernel_1.outputscale.detach().reshape(()), model.kernel_2.outputscale.detach().reshape(())]).cpu()
    meshes = [torch.linspace(-0.125, 1.125, 13), torch.linspace(0.125, 0.875, 13)]
    ref = O.elbo_structured(O.VFF_GRID, meshes, X, y, l.to(torch.float64), s2.to(torch.float64),
                            model.likelihood.noise.detach().reshape(()).cpu().to(torch.float64), model.variational_mean.detach().cpu(),
                            [model.variational_chol_1.detach().cpu(), model.variational_chol_2.detach().cpu()], ref_quirks=False)
    assert abs(elbo.item() - ref.item()) < 1e-8 * abs(ref.item())
    opt = torch.optim.Adam(model.parameters(), lr=0.02)
    losses = []
    for _ in range(5):
        opt.zero_grad()
        loss = -model._elbo()
        loss.backward()
        opt.step()
        losses.append(loss.item())
    assert losses[-1] < losses[0]
    post = model.posterior(X[:64].to(dev))
    assert torch.isfinite(post.mean).all() and (post.variance > 0).all()
