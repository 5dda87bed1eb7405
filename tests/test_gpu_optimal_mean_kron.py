"""GPU tests of the Kronecker-preconditioned optimal-mean solve (vggp_meanopt_solve_pc with VGGP_MEANOPT_KRONECKER,
csrc/meanopt.cuh): parity with the mean of the reference's q_u(), stationarity of the existing step at full size on the
track data and theta of tools/mg_oracle_iterations.py (so that the counts compare with the CPU oracle's), 3-D B1 included,
and GriddedVariationalGP.set_optimal_mean(preconditioner="kronecker") on the model classes."""
import importlib

import pytest
import torch

import bench
from oracle import vggp_oracle as O
from test_gpu_optimal_mean import _b1_model, _problem, _relerr, _setup

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def vg():
    if not torch.cuda.is_available():
        pytest.skip("no CUDA device")
    return importlib.import_module("variational-gridded-gaussian-processes_b200")


@pytest.fixture(scope="module")
def dev(vg):
    return torch.device("cuda", 0)


@pytest.mark.parametrize("markov", [False, True])
@pytest.mark.parametrize("knots,N", [((11,), 5000), ((33, 29), 5000), ((12, 10, 8), 5000)])
@pytest.mark.parametrize("dtype,tol", [(torch.float64, 1e-8), (torch.float32, 1e-4)])
def test_kronecker_optimal_mean_matches_reference_q_u(vg, dev, markov, knots, N, dtype, tol):
    meshes, X, y, l, s2, noise, Ls = _problem(markov, knots, N, seed=7 + len(knots))
    Xq, yq = X.to(dtype).to(torch.float64), y.to(dtype).to(torch.float64)
    ref = O.optimal_q(O.SVGP_GRID if markov else O.B1_ASVGP, meshes, Xq, yq, l, s2, noise, ref_quirks=False)[0]
    plan, theta, Lcat, obs = _setup(vg, dev, markov, meshes, Xq, yq, l, s2, noise, Ls, dtype)
    plan.grid_forward(theta, torch.zeros(plan.M, dtype=torch.float64, device=dev), Lcat)
    plan.meanopt_assemble(obs)
    m, iters, relres = plan.meanopt_solve(1e-12, 20000, "kronecker")
    assert iters > 0 and relres <= 1e-12
    assert _relerr(m, ref) <= tol
    # the Jacobi solve of the same system agrees
    plan.grid_forward(theta, torch.zeros(plan.M, dtype=torch.float64, device=dev), Lcat)
    mj, _, _ = plan.meanopt_solve(1e-12, 20000, "jacobi")
    assert _relerr(m, mj) <= 1e-9


# data and theta of tools/mg_oracle_iterations.py; oracle Kronecker-PCG counts to rtol 1e-8 from m = 0 in DESIGN.md
@pytest.mark.parametrize("markov,knots,N,max_iter,oracle_iters", [
    (False, (512, 512), 1 << 22, 20000, 196), (True, (512, 512), 1 << 22, 20000, None),
    (False, (64, 64, 16), 1 << 20, 20000, None), (True, (64, 64, 16), 1 << 20, 20000, None)])
def test_full_size_kronecker_solve_is_stationary_for_the_step(vg, dev, markov, knots, N, max_iter, oracle_iters):
    D = len(knots)
    meshes = [torch.linspace(0, 1, k) for k in knots]
    xs, y = bench.make_tracks_torch(0, N, N, torch.device("cpu"), torch.float32, 0, D=D)
    xs, y = [x.to(dev) for x in xs], y.to(dev)
    plan = vg.GridPlan(vg.SVGP_MARKOV if markov else vg.B1_ASVGP, meshes, torch.float32, dev)
    obs = plan.bin(xs, y)
    theta = torch.tensor([0.3] * D + [0.8] * D + [0.05], dtype=torch.float64, device=dev)
    Lcat = torch.cat([(0.5 * torch.eye(k, dtype=torch.float64)).reshape(-1) for k in knots]).to(dev)
    zero = torch.zeros(plan.M, dtype=torch.float64, device=dev)
    plan.grid_forward(theta, zero, Lcat)
    plan.meanopt_assemble(obs)
    jac_scratch = plan.workspace_bytes()["scratch"]
    m, iters, relres = plan.meanopt_solve(1e-8, max_iter, "kronecker")
    assert relres <= 1e-8, (iters, relres)
    if oracle_iters is not None:
        assert abs(iters - oracle_iters) <= 0.1 * oracle_iters, (iters, oracle_iters)
    dm0 = plan.step(theta, zero, Lcat, obs, None)[2].norm().item()
    dms = plan.step(theta, m, Lcat, obs, None)[2].norm().item()
    assert dms <= 1e-3 * dm0, (dms, dm0)
    assert plan.workspace_bytes()["scratch"] == jac_scratch + 8 * (plan.M + 3 * sum(knots) + 1)


def test_b1_model_set_optimal_mean_kronecker(vg, dev):
    mdl = _b1_model(dev)
    with torch.no_grad():
        mdl.variational_mean.normal_(0.0, 0.1)
    mdl.zero_grad()
    mdl._elbo().backward()
    g0 = mdl.variational_mean.grad.norm().item()
    res = mdl.set_optimal_mean(preconditioner="kronecker")
    assert res["relres"] <= 1e-10 and res["iterations"] > 0
    xt = torch.rand(2000, 2, dtype=torch.float64).to(dev)
    assert _relerr(mdl.posterior(xt).mean, mdl.posterior_dense(xt, optimal=True).mean) <= 1e-8
    mdl.zero_grad()
    mdl._elbo().backward()
    assert mdl.variational_mean.grad.norm().item() <= 1e-6 * g0
    before = mdl.variational_mean.detach().clone()
    with pytest.raises(ValueError, match="preconditioner"):
        mdl.set_optimal_mean(preconditioner="multigrid")
    assert torch.equal(mdl.variational_mean.detach(), before)


def test_markov_model_set_optimal_mean_kronecker(vg, dev):
    ks = importlib.import_module("variational-gridded-gaussian-processes_b200.models.sparse.kronecker_structure")
    g = torch.Generator().manual_seed(71)
    N = 20000
    X = torch.rand(N, 2, generator=g, dtype=torch.float64) * 1.2 - 0.1
    y = torch.sin(4 * X[:, 0]) * torch.cos(3 * X[:, 1]) + 0.05 * torch.randn(N, generator=g, dtype=torch.float64)
    Z = torch.stack([torch.linspace(0, 1, 30), torch.linspace(0, 1, 30) ** 1.2], dim=1)
    torch.manual_seed(0)
    dense = ks.Matern12SVGP(X, y, Z, markov=False).to(torch.float64).to(dev)
    markov = ks.Matern12SVGP(X, y, Z, markov=True).to(torch.float64).to(dev)
    res = markov.set_optimal_mean(preconditioner="kronecker")
    assert res["relres"] <= 1e-10
    dense.load_state_dict(markov.state_dict())
    xt = torch.rand(2000, 2, dtype=torch.float64).to(dev) * 1.4 - 0.2
    assert _relerr(markov.posterior(xt).mean, dense.posterior_dense(xt, optimal=True).mean) <= 1e-8
    with pytest.raises(ValueError, match="preconditioner"):
        markov.set_optimal_mean(preconditioner="Kronecker")
