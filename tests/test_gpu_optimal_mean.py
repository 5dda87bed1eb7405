"""GPU tests of the optimal variational mean (vggp_meanopt_assemble / vggp_meanopt_solve, csrc/meanopt.cuh): parity with the
mean of the reference's q_u() (vggp_oracle.optimal_q) for the B1 family and the Markov SVGP form, stationarity of the existing
step at full size, and GriddedVariationalGP.set_optimal_mean() on the model classes."""
import importlib

import pytest
import torch

from oracle import vggp_oracle as O

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def vg():
    if not torch.cuda.is_available():
        pytest.skip("no CUDA device")
    return importlib.import_module("variational-gridded-gaussian-processes_b200")


@pytest.fixture(scope="module")
def dev(vg):
    return torch.device("cuda", 0)


def _problem(markov, knots, N, seed, x_lo=-0.2, x_hi=1.2, uniform=False):
    D = len(knots)
    g = torch.Generator().manual_seed(seed)
    meshes = [torch.linspace(0, 1, k) for k in knots]
    if markov and not uniform:
        meshes = [(t ** (1.0 + 0.3 * d)).to(torch.float32) for d, t in enumerate(meshes)]
    X = torch.rand(N, D, generator=g, dtype=torch.float64) * (x_hi - x_lo) + x_lo
    y = torch.sin(3 * X[:, 0]) + (torch.cos(5 * X[:, -1]) if D > 1 else 0) + 0.1 * torch.randn(N, generator=g, dtype=torch.float64)
    l = torch.rand(D, generator=g, dtype=torch.float64) * 0.4 + 0.2
    s2 = torch.rand(D, generator=g, dtype=torch.float64) * 0.8 + 0.6
    noise = torch.tensor(0.07, dtype=torch.float64)
    Ls = [torch.eye(n, dtype=torch.float64) * 0.6 for n in knots]
    return meshes, X, y, l, s2, noise, Ls


def _relerr(a, b):
    a = a.detach().cpu().to(torch.float64).reshape(-1)
    b = b.detach().cpu().to(torch.float64).reshape(-1)
    return ((a - b).norm() / b.norm().clamp_min(1e-300)).item()


def _setup(vg, dev, markov, meshes, X, y, l, s2, noise, Ls, dtype):
    plan = vg.GridPlan(vg.SVGP_MARKOV if markov else vg.B1_ASVGP, meshes, dtype, dev)
    theta = torch.cat([l, s2, noise.reshape(1)]).to(dev)
    Lcat = torch.cat([L.reshape(-1) for L in Ls]).to(dev)
    xs = [X[:, d].to(dev, dtype).contiguous() for d in range(len(meshes))]
    obs = plan.bin(xs, y.to(dev, dtype).contiguous())
    return plan, theta, Lcat, obs


def _optimal(plan, theta, m, Lcat, obs, rtol=1e-12, max_iter=20000):
    plan.grid_forward(theta, m, Lcat)
    plan.meanopt_assemble(obs)
    return plan.meanopt_solve(rtol, max_iter)


@pytest.mark.parametrize("markov", [False, True])
@pytest.mark.parametrize("knots,N", [((11,), 5000), ((33, 29), 5000), ((12, 10, 8), 5000)])
@pytest.mark.parametrize("dtype,tol", [(torch.float64, 1e-8), (torch.float32, 1e-4)])
def test_optimal_mean_matches_reference_q_u(vg, dev, markov, knots, N, dtype, tol):
    meshes, X, y, l, s2, noise, Ls = _problem(markov, knots, N, seed=7 + len(knots))
    Xq, yq = X.to(dtype).to(torch.float64), y.to(dtype).to(torch.float64)
    ref = O.optimal_q(O.SVGP_GRID if markov else O.B1_ASVGP, meshes, Xq, yq, l, s2, noise, ref_quirks=False)[0]
    plan, theta, Lcat, obs = _setup(vg, dev, markov, meshes, Xq, yq, l, s2, noise, Ls, dtype)
    m, iters, relres = _optimal(plan, theta, torch.zeros(plan.M, dtype=torch.float64, device=dev), Lcat, obs)
    assert iters > 0 and relres <= 1e-12
    assert _relerr(m, ref) <= tol


# 3-D B1: Jacobi-preconditioned CG does not reach rtol 1e-8 within the default iteration limit (60000 iterations leave
# relres 2.3e-4 on one B200); a stronger preconditioner is the documented next step (DESIGN.md section 7)
@pytest.mark.parametrize("markov,knots,N", [
    (False, (512, 512), 1 << 22), (True, (512, 512), 1 << 22), (True, (64, 64, 16), 1 << 20),
    pytest.param(False, (64, 64, 16), 1 << 20, marks=pytest.mark.xfail(strict=True, reason="Jacobi-CG too slow for the 3-D B1 prior"))])
def test_full_size_solve_is_stationary_for_the_step(vg, dev, markov, knots, N):
    gen = importlib.import_module("variational-gridded-gaussian-processes_b200.utils.dataloaders")
    models = importlib.import_module("variational-gridded-gaussian-processes_b200.models._gridded")
    D = len(knots)
    meshes = [torch.linspace(0, 1, k) for k in knots]
    xs, y = gen.generate_tracks(0, N, N, dev, torch.float32, seed=3, D=D)
    plan = vg.GridPlan(vg.SVGP_MARKOV if markov else vg.B1_ASVGP, meshes, torch.float32, dev)
    obs = plan.bin(xs, y)
    theta = torch.tensor([0.3] * D + [0.8] * D + [0.05], dtype=torch.float64, device=dev)
    Lcat = torch.cat([(0.5 * torch.eye(k, dtype=torch.float64)).reshape(-1) for k in knots]).to(dev)
    zero = torch.zeros(plan.M, dtype=torch.float64, device=dev)
    m, iters, relres = _optimal(plan, theta, zero, Lcat, obs, rtol=1e-8,
                                max_iter=models.GriddedVariationalGP.MEANOPT_MAX_ITER)
    assert relres <= 1e-8, (iters, relres)
    dm0 = plan.step(theta, zero, Lcat, obs, None)[2].norm().item()
    dms = plan.step(theta, m, Lcat, obs, None)[2].norm().item()
    assert dms <= 1e-3 * dm0, (dms, dm0)
    assert plan.workspace_bytes()["scratch"] > 0


def _b1_model(dev):
    ks = importlib.import_module("variational-gridded-gaussian-processes_b200.models.sparse.kronecker_structure")
    g = torch.Generator().manual_seed(3)
    N = 6000
    X = torch.rand(N, 2, generator=g, dtype=torch.float64) * 1.2 - 0.1
    y = torch.sin(4 * X[:, 0]) * torch.cos(3 * X[:, 1]) + 0.05 * torch.randn(N, generator=g, dtype=torch.float64)
    return ks.Matern12B1SplineASVGP(X, y, 40, (0, 1), (0, 1)).to(torch.float64).to(dev)


def test_b1_model_set_optimal_mean(vg, dev):
    mdl = _b1_model(dev)
    assert mdl.M <= 4096
    with torch.no_grad():
        mdl.variational_mean.normal_(0.0, 0.1)
    mdl.zero_grad()
    mdl._elbo().backward()
    g0 = mdl.variational_mean.grad.norm().item()
    e0 = mdl._elbo().item()
    res = mdl.set_optimal_mean()
    assert res["relres"] <= 1e-10 and res["iterations"] > 0
    xt = torch.rand(2000, 2, dtype=torch.float64).to(dev)
    assert _relerr(mdl.posterior(xt).mean, mdl.posterior_dense(xt, optimal=True).mean) <= 1e-8
    mdl.zero_grad()
    e1 = mdl._elbo()
    assert e1.item() >= e0
    e1.backward()
    assert mdl.variational_mean.grad.norm().item() <= 1e-6 * g0
    # a forced non-convergence raises and leaves the mean as it was
    with torch.no_grad():
        mdl.variational_mean.zero_()
    with pytest.raises(RuntimeError, match="unchanged"):
        mdl.set_optimal_mean(max_iter=1)
    assert not bool(mdl.variational_mean.any())
    # the dense-feature families point at the dense closed form
    ks = importlib.import_module("variational-gridded-gaussian-processes_b200.models.sparse.kronecker_structure")
    b0 = ks.Matern12B0SplineGriddedGP(mdl.train_inputs[0].cpu(), mdl.train_targets.cpu(), 10, (0, 1), (0, 1))
    with pytest.raises(NotImplementedError, match="set_optimal_q"):
        b0.to(torch.float64).to(dev).set_optimal_mean()


def test_markov_model_set_optimal_mean(vg, dev):
    ks = importlib.import_module("variational-gridded-gaussian-processes_b200.models.sparse.kronecker_structure")
    g = torch.Generator().manual_seed(71)
    N = 20000
    X = torch.rand(N, 2, generator=g, dtype=torch.float64) * 1.2 - 0.1
    y = torch.sin(4 * X[:, 0]) * torch.cos(3 * X[:, 1]) + 0.05 * torch.randn(N, generator=g, dtype=torch.float64)
    Z = torch.stack([torch.linspace(0, 1, 30), torch.linspace(0, 1, 30) ** 1.2], dim=1)
    torch.manual_seed(0)
    dense = ks.Matern12SVGP(X, y, Z, markov=False).to(torch.float64).to(dev)
    markov = ks.Matern12SVGP(X, y, Z, markov=True).to(torch.float64).to(dev)
    with torch.no_grad():
        markov.variational_mean.normal_(0.0, 0.1)
    markov.zero_grad()
    markov._elbo().backward()
    g0 = markov.variational_mean.grad.norm().item()
    e0 = markov._elbo().item()
    res = markov.set_optimal_mean()
    assert res["relres"] <= 1e-10
    dense.load_state_dict(markov.state_dict())
    xt = torch.rand(2000, 2, dtype=torch.float64).to(dev) * 1.4 - 0.2
    assert _relerr(markov.posterior(xt).mean, dense.posterior_dense(xt, optimal=True).mean) <= 1e-8
    markov.zero_grad()
    e1 = markov._elbo()
    assert e1.item() >= e0
    e1.backward()
    assert markov.variational_mean.grad.norm().item() <= 1e-6 * g0
    with torch.no_grad():
        markov.variational_mean.normal_(0.0, 0.1)
    before = markov.variational_mean.detach().clone()
    with pytest.raises(RuntimeError, match="unchanged"):
        markov.set_optimal_mean(max_iter=1)
    assert torch.equal(markov.variational_mean.detach(), before)
    with pytest.raises(NotImplementedError, match="set_optimal_q"):
        dense.set_optimal_mean()
