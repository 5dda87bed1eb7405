"""GPU tests of the collapsed ELBO (vggp_logdet_system / vggp_collapsed_terms, csrc/collapsed.cuh): unit-probe parity with the
reference's collapsed bound at D = 1..3, bitwise reproducibility, the D = 1 identity with the Kronecker-optimal uncollapsed
bound, the Rademacher estimate against the exact value at 64 x 64, full-size runs and the model method."""
import importlib
import math

import pytest
import torch

from oracle import collapsed as CO
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


def _problem(markov, knots, N, seed, x_lo=-0.2, x_hi=1.2):
    D = len(knots)
    g = torch.Generator().manual_seed(seed)
    meshes = [torch.linspace(0, 1, k) for k in knots]
    if markov:
        meshes = [(t ** (1.0 + 0.3 * d)).to(torch.float32) for d, t in enumerate(meshes)]
    X = torch.rand(N, D, generator=g, dtype=torch.float64) * (x_hi - x_lo) + x_lo
    y = torch.sin(3 * X[:, 0]) + (torch.cos(5 * X[:, -1]) if D > 1 else 0) + 0.1 * torch.randn(N, generator=g, dtype=torch.float64)
    l = torch.rand(D, generator=g, dtype=torch.float64) * 0.4 + 0.2
    s2 = torch.rand(D, generator=g, dtype=torch.float64) * 0.8 + 0.6
    return meshes, X, y, l, s2, torch.tensor(0.07, dtype=torch.float64)


def _solved_plan(vg, dev, markov, meshes, xs, y, theta, cg_rtol=1e-12, pc="kronecker"):
    plan = vg.GridPlan(vg.SVGP_MARKOV if markov else vg.B1_ASVGP, meshes, y.dtype, dev)
    obs = plan.bin(xs, y)
    Lcat = torch.cat([torch.eye(t.numel(), dtype=torch.float64).reshape(-1) for t in meshes]).to(dev)
    plan.grid_forward(theta, torch.zeros(plan.M, dtype=torch.float64, device=dev), Lcat)
    plan.meanopt_assemble(obs)
    _, it, rr = plan.meanopt_solve(cg_rtol, 20000, pc)
    assert rr <= cg_rtol, (it, rr)
    return plan, obs


@pytest.mark.parametrize("markov", [False, True])
@pytest.mark.parametrize("knots,N", [((37,), 4000), ((13, 11), 6000), ((7, 6, 5), 8000)])
@pytest.mark.parametrize("dtype,tol", [(torch.float64, 1e-9), (torch.float32, 1e-5)])
def test_unit_probes_give_the_collapsed_bound(vg, dev, markov, knots, N, dtype, tol):
    meshes, X, y, l, s2, noise = _problem(markov, knots, N, seed=len(knots) + 10 * markov)
    X, y = X.to(dtype).to(torch.float64), y.to(dtype).to(torch.float64)
    theta = torch.cat([l, s2, noise.reshape(1)]).to(dev)
    xs = [X[:, d].to(dev, dtype).contiguous() for d in range(len(knots))]
    plan, obs = _solved_plan(vg, dev, markov, meshes, xs, y.to(dev, dtype), theta)
    terms = [float(v) for v in plan.collapsed_terms(obs).cpu()]
    want = float(O.elbo_collapsed_woodbury(O.SVGP_GRID if markov else O.B1_ASVGP, meshes, X, y, l, s2, noise,
                                           ref_quirks=False))
    for pc in ("kronecker", "jacobi"):
        ld = plan.logdet_system(plan.M, 0, pc, "unit", plan.M + 8, 1e-14)
        assert ld["converged"] == plan.M
        got = CO.collapsed_elbo(*terms, ld["logdet"], float(noise), s2.numpy(), markov)
        assert abs(got - want) <= tol * abs(want), (pc, got, want)


@pytest.mark.parametrize("markov", [False, True])
def test_same_seed_same_bits(vg, dev, markov):
    meshes, X, y, l, s2, noise = _problem(markov, (40, 30), 50000, seed=3)
    theta = torch.cat([l, s2, noise.reshape(1)]).to(dev)
    xs = [X[:, d].to(dev, torch.float32).contiguous() for d in range(2)]
    plan, obs = _solved_plan(vg, dev, markov, meshes, xs, y.to(dev, torch.float32), theta)
    for pc in ("kronecker", "jacobi"):
        a = plan.logdet_system(16, 7, pc, "rademacher", 200, 1e-8, per_probe=True)
        b = plan.logdet_system(16, 7, pc, "rademacher", 200, 1e-8, per_probe=True)
        assert a["logdet"] == b["logdet"] and a["stderr"] == b["stderr"] and torch.equal(a["per_probe"], b["per_probe"])
    t1, t2 = plan.collapsed_terms(obs), plan.collapsed_terms(obs)
    assert torch.equal(t1, t2)


def _model(vg, markov, X, y, meshes, l, s2, noise, dev, dtype=torch.float64):
    gm = importlib.import_module("variational-gridded-gaussian-processes_b200.models._gridded")

    class Model(gm.GriddedVariationalGP):
        pass

    Model.family = vg.SVGP_MARKOV if markov else vg.B1_ASVGP
    mdl = Model(X, y, meshes).to(dtype).to(dev)
    for d, k in enumerate(mdl._kernels):
        k.base_kernel.lengthscale = l[d].reshape(1, 1).to(dev)
        k.outputscale = s2[d].to(dev)
    mdl.likelihood.noise = noise.to(dev)
    return mdl


@pytest.mark.parametrize("markov", [False, True])
def test_1d_collapsed_equals_the_kronecker_optimal_uncollapsed_bound(vg, dev, markov):
    meshes, X, y, l, s2, noise = _problem(markov, (512,), 1 << 20, seed=21)
    mdl = _model(vg, markov, X, y, meshes, l, s2, noise, dev)
    res = mdl.collapsed_elbo(n_probes=512, probes="unit", rtol=1e-13, max_steps=520, cg_rtol=1e-13)
    assert res["converged"] and res["stderr"] == 0.0
    mdl.set_optimal_mean(rtol=1e-13, preconditioner="kronecker")
    mdl.set_optimal_covariance()
    unc = mdl._elbo().item()
    assert abs(res["elbo"] - unc) <= 1e-8 * abs(unc), (res, unc)


@pytest.mark.parametrize("markov", [False, True])
def test_64x64_tracks_rademacher_against_exact(vg, dev, markov):
    gen = importlib.import_module("variational-gridded-gaussian-processes_b200.utils.dataloaders")
    N = 1 << 20
    xs, y = gen.generate_tracks(0, N, N, dev, torch.float32, seed=5, D=2)
    meshes = [torch.linspace(0, 1, 64)] * 2
    theta = torch.tensor([0.3, 0.3, 0.8, 0.8, 0.05], dtype=torch.float64, device=dev)
    plan, obs = _solved_plan(vg, dev, markov, meshes, xs, y, theta)
    exact = plan.logdet_system(plan.M, 0, "kronecker", "unit", 1000, 1e-13)
    assert exact["converged"] == plan.M
    for pc in ("kronecker", "jacobi"):
        est = plan.logdet_system(32, 0, pc, "rademacher", 200, 1e-6)
        assert est["converged"] == 32 and est["stderr"] > 0.0
        assert abs(est["logdet"] - exact["logdet"]) <= 4.0 * est["stderr"], (pc, est, exact["logdet"])
    # the Kronecker-optimal uncollapsed bound lies below the collapsed one
    X = torch.stack([x.double().cpu() for x in xs], 1)
    l, s2, noise = torch.tensor([0.3, 0.3]), torch.tensor([0.8, 0.8]), torch.tensor(0.05)
    mdl = _model(vg, markov, X, y.double().cpu(), meshes, l.double(), s2.double(), noise.double(), dev, torch.float32)
    col = mdl.collapsed_elbo(n_probes=plan.M, probes="unit", rtol=1e-13, max_steps=1000)
    mdl.set_optimal_mean(rtol=1e-10, preconditioner="kronecker")
    mdl.set_optimal_covariance(rtol=1e-7)
    unc = mdl._elbo().item()
    assert unc < col["elbo"], (unc, col)
    print(f"64 x 64 markov={markov}: collapsed {col['elbo']:.6e}, Kronecker-optimal uncollapsed {unc:.6e}")


@pytest.mark.parametrize("markov,knots", [(False, (512, 512)), (True, (512, 512)), (False, (256, 256, 64))])
def test_full_size_two_seeds_agree(vg, dev, markov, knots):
    gen = importlib.import_module("variational-gridded-gaussian-processes_b200.utils.dataloaders")
    N, D = 1 << 26, len(knots)
    xs, y = gen.generate_tracks(0, N, N, dev, torch.float32, seed=0, D=D)
    theta = torch.tensor([0.3] * D + [0.8] * D + [0.05], dtype=torch.float64, device=dev)
    plan, obs = _solved_plan(vg, dev, markov, [torch.linspace(0, 1, k) for k in knots], xs, y, theta,
                             cg_rtol=1e-8 if D == 3 else 1e-10)
    del xs, y
    a = plan.logdet_system(16, 0, "kronecker", "rademacher", 1000, 1e-6)
    b = plan.logdet_system(16, 1, "kronecker", "rademacher", 1000, 1e-6)
    for r in (a, b):
        assert r["converged"] == 16 and math.isfinite(r["logdet"]) and r["stderr"] > 0.0, r
    assert abs(a["logdet"] - b["logdet"]) <= 5.0 * math.hypot(a["stderr"], b["stderr"]), (a, b)
    terms = plan.collapsed_terms(obs).cpu()
    assert torch.isfinite(terms).all() and terms[0].item() == N


def test_model_method_and_refusals(vg, dev):
    meshes, X, y, l, s2, noise = _problem(False, (20, 18), 20000, seed=8)
    mdl = _model(vg, False, X, y, meshes, l, s2, noise, dev)
    m0 = mdl.variational_mean.detach().clone()
    res = mdl.collapsed_elbo(n_probes=16, seed=3)
    assert set(res) == {"elbo", "stderr", "logdet_sigma", "quad", "trace_term", "cg_iterations", "lanczos_steps", "converged"}
    assert torch.equal(mdl.variational_mean.detach(), m0)
    exact = mdl.collapsed_elbo(n_probes=mdl.M, probes="unit", rtol=1e-13, max_steps=mdl.M + 8)
    want = float(O.elbo_collapsed_woodbury(O.B1_ASVGP, meshes, X, y, l, s2, noise, ref_quirks=False))
    assert abs(exact["elbo"] - want) <= 1e-9 * abs(want)
    assert abs(res["elbo"] - want) <= 5.0 * res["stderr"] + 1e-9 * abs(want)
    with pytest.raises(RuntimeError, match="Lanczos"):
        mdl.collapsed_elbo(n_probes=4, max_steps=2, rtol=1e-14)
    mdl.shard_observations(0, 2, group=None)
    with pytest.raises(NotImplementedError, match="sharded"):
        mdl.collapsed_elbo()
    ks = importlib.import_module("variational-gridded-gaussian-processes_b200.models.sparse.kronecker_structure")
    dense = ks.Matern12SVGP(X[:2000, :2], y[:2000], torch.stack([torch.linspace(0, 1, 10)] * 2, 1),
                            markov=False).to(torch.float64).to(dev)
    with pytest.raises(NotImplementedError):
        dense.collapsed_elbo()
