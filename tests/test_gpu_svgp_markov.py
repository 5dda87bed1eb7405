"""GPU tests of the product-grid SVGP family in its O(1)-per-observation Markov form (SVGP_MARKOV, csrc/svgpm.cuh): parity
with the dense SVGP oracle, agreement with the dense-feature SVGP_GRID plan on the same inputs, full-size runs against
oracle/svgp_markov.py, CUDA-graph replay, and the Matern12SVGP(markov=True) model."""
import importlib

import numpy as np
import pytest
import torch

from oracle import svgp_markov as SM
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


def _problem(knots, N, seed, x_lo=-0.2, x_hi=1.2, uniform=False):
    D = len(knots)
    g = torch.Generator().manual_seed(seed)
    meshes = [torch.linspace(0, 1, k) for k in knots]
    if not uniform:
        meshes = [(t ** (1.0 + 0.3 * d)).to(torch.float32) for d, t in enumerate(meshes)]
    X = torch.rand(N, D, generator=g, dtype=torch.float64) * (x_hi - x_lo) + x_lo
    y = torch.sin(3 * X[:, 0]) + (torch.cos(5 * X[:, -1]) if D > 1 else 0) + 0.1 * torch.randn(N, generator=g, dtype=torch.float64)
    l = torch.rand(D, generator=g, dtype=torch.float64) * 0.4 + 0.2
    s2 = torch.rand(D, generator=g, dtype=torch.float64) * 0.8 + 0.6
    noise = torch.tensor(0.07, dtype=torch.float64)
    Ms = list(knots)
    m = torch.randn(int(np.prod(Ms)), generator=g, dtype=torch.float64) * 0.2
    Ls = [torch.eye(n, dtype=torch.float64) * 0.6 + 0.05 * torch.randn(n, n, generator=g, dtype=torch.float64) / n ** 0.5
          for n in Ms]
    return meshes, X, y, l, s2, noise, m, Ls


def _relerr(a, b):
    a = a.detach().cpu().to(torch.float64).reshape(-1)
    b = b.detach().cpu().to(torch.float64).reshape(-1)
    return ((a - b).norm() / b.norm().clamp_min(1e-300)).item()


def _step(vg, dev, family, meshes, X, y, l, s2, noise, m, Ls, dtype, scale=1.0):
    plan = vg.GridPlan(family, meshes, dtype, dev)
    theta = torch.cat([l, s2, noise.reshape(1)]).to(dev)
    Lcat = torch.cat([L.reshape(-1) for L in Ls]).to(dev)
    xs = [X[:, d].to(dev, dtype).contiguous() for d in range(len(meshes))]
    yy = y.to(dev, dtype).contiguous()
    obs, yarg = (plan.bin(xs, yy), None) if family == vg.SVGP_MARKOV else (xs, yy)
    res = plan.step(theta, m.to(dev), Lcat, obs, yarg, ell_scale=scale)
    return plan, res, (theta, Lcat, xs, yy, obs)


def _check(plan, res, ref, gref, N, tol):
    out, dtheta, dm, dL = res
    D = plan.D
    assert plan.read_info() == 0
    assert out[3].item() == N
    assert abs(out[0].item() - ref.item()) <= tol * abs(ref.item()), (out.cpu(), ref)
    assert _relerr(dtheta[:D], gref[0]) < tol * 10, ("dl", dtheta[:D].cpu(), gref[0])
    assert _relerr(dtheta[D:2 * D], gref[1]) < tol * 10, ("ds2", dtheta[D:2 * D].cpu(), gref[1])
    assert _relerr(dtheta[2 * D], gref[2]) < tol * 10, "dnoise"
    assert _relerr(dm, gref[3]) < tol * 10, "dm"
    off = 0
    for d, n in enumerate(plan.m_per_dim):
        dLd = dL[off:off + n * n].reshape(n, n).cpu()
        off += n * n
        assert torch.count_nonzero(torch.triu(dLd, 1)) == 0
        assert _relerr(torch.tril(dLd), torch.tril(gref[4 + d])) < tol * 10, ("dL", d)


CASES = [((11,), 700), ((9, 7), 900), ((70, 13), 5000), ((6, 9, 5), 3000)]


@pytest.mark.parametrize("knots,N", CASES)
@pytest.mark.parametrize("dtype,tol", [(torch.float64, 1e-8), (torch.float32, 1e-3)])
def test_markov_matches_dense_svgp_oracle(vg, dev, knots, N, dtype, tol):
    meshes, X, y, l, s2, noise, m, Ls = _problem(knots, N, seed=31 + len(knots))
    Xq, yq = X.to(dtype).to(torch.float64), y.to(dtype).to(torch.float64)
    ls = [L.clone().requires_grad_(True) for L in Ls]
    args = [t.clone().requires_grad_(True) for t in (l, s2, noise, m)]
    ref = O.elbo_structured(O.SVGP_GRID, meshes, Xq, yq, *args, ls, ref_quirks=False, scale=1.4)
    gref = torch.autograd.grad(ref, args + ls)
    plan, res, _ = _step(vg, dev, vg.SVGP_MARKOV, meshes, Xq, yq, l, s2, noise, m, Ls, dtype, scale=1.4)
    _check(plan, res, ref.detach(), gref, N, tol)


@pytest.mark.parametrize("dtype,tol", [(torch.float64, 1e-9), (torch.float32, 1e-3)])
def test_markov_plan_agrees_with_dense_svgp_plan(vg, dev, dtype, tol):
    knots, N = (24, 19), 20000
    meshes, X, y, l, s2, noise, m, Ls = _problem(knots, N, seed=41)
    Xq, yq = X.to(dtype).to(torch.float64), y.to(dtype).to(torch.float64)
    pm, rm, (theta, Lcat, xs, _, _) = _step(vg, dev, vg.SVGP_MARKOV, meshes, Xq, yq, l, s2, noise, m, Ls, dtype, scale=1.1)
    pg, rg, _ = _step(vg, dev, vg.SVGP_GRID, meshes, Xq, yq, l, s2, noise, m, Ls, dtype, scale=1.1)
    assert pm.read_info() == 0 and pg.read_info() == 0
    for a, b, name in zip(rm, rg, ("out", "dtheta", "dm", "dL")):
        assert _relerr(a, b) < tol * 10, name
    # predictions: the Markov plan's vggp_predict against the dense features and workspace of the SVGP_GRID plan
    xt = [torch.linspace(-0.3, 1.3, 4001, dtype=torch.float64).to(dev, dtype), torch.rand(4001, dtype=torch.float64).to(dev, dtype)]
    mean, var = pm.predict(xt)
    phis = [pg.features_dense(d, xt[d], theta).to(torch.float64) for d in range(2)]
    A = pg.workspace(vg._lib.WS_ALPHA).reshape(knots)
    mref = torch.einsum("in,ij,jn->n", phis[0], A, phis[1])
    p = torch.ones_like(mref)
    q = torch.ones_like(mref)
    for d in range(2):
        p = p * (phis[d] * (pg.workspace(vg._lib.WS_P, d) @ phis[d])).sum(0)
        q = q * (phis[d] * (pg.workspace(vg._lib.WS_Q, d) @ phis[d])).sum(0)
    vref = torch.prod(theta[2:4]) - p + q
    ptol = 1e-9 if dtype == torch.float64 else 1e-4
    assert (mean.to(torch.float64) - mref).abs().max().item() <= ptol * 10
    assert (var.to(torch.float64) - vref).abs().max().item() <= ptol * 10


@pytest.mark.parametrize("knots,N", [((512, 512), 1 << 22), ((64, 64, 16), 1 << 20)])
def test_markov_full_size_matches_markov_oracle(vg, dev, knots, N):
    meshes, X, y, l, s2, noise, m, Ls = _problem(knots, N, seed=51, x_lo=-0.05, x_hi=1.05, uniform=True)
    Xq, yq = X.to(torch.float32).to(torch.float64), y.to(torch.float32).to(torch.float64)
    ref, gref = SM.value_and_grads(meshes, Xq, yq, l, s2, noise, m, Ls)
    plan, res, _ = _step(vg, dev, vg.SVGP_MARKOV, meshes, Xq, yq, l, s2, noise, m, Ls, torch.float32)
    _check(plan, res, ref, gref, N, 1e-3)


def test_markov_graphed_step_equals_eager(vg, dev):
    knots, N = (96, 80), 1 << 18
    meshes, X, y, l, s2, noise, m, Ls = _problem(knots, N, seed=61)
    plan, eager, (theta, Lcat, xs, yy, obs) = _step(vg, dev, vg.SVGP_MARKOV, meshes, X, y, l, s2, noise, m, Ls, torch.float64)
    eager = [t.clone() for t in eager]
    mm = m.to(dev)
    gs = plan.graphed_step(theta, mm, Lcat, obs)
    for _ in range(2):
        got = gs.replay()
    torch.cuda.synchronize()
    for a, b in zip(got, eager):
        assert _relerr(a, b) < 1e-12
    # new parameter values written into the static buffers are picked up by the replay
    theta.copy_(theta * 1.05)
    got = [t.clone() for t in gs.replay()]
    again = plan.step(theta, mm, Lcat, obs, None)
    for a, b in zip(got, again):
        assert _relerr(a, b) < 1e-12


def test_matern12svgp_markov_model(vg, dev):
    ks = importlib.import_module("variational-gridded-gaussian-processes_b200.models.sparse.kronecker_structure")
    g = torch.Generator().manual_seed(71)
    N = 20000
    X = torch.rand(N, 2, generator=g, dtype=torch.float64) * 1.2 - 0.1
    y = torch.sin(4 * X[:, 0]) * torch.cos(3 * X[:, 1]) + 0.05 * torch.randn(N, generator=g, dtype=torch.float64)
    Z = torch.stack([torch.linspace(0, 1, 30), torch.linspace(0, 1, 30) ** 1.2], dim=1)
    models = []
    for markov in (False, True):
        torch.manual_seed(0)
        mdl = ks.Matern12SVGP(X, y, Z, markov=markov).to(torch.float64).to(dev)
        with torch.no_grad():
            mdl.variational_mean.copy_(0.1 * torch.randn(mdl.M, generator=g, dtype=torch.float64).to(dev))
        models.append(mdl)
    dense, markov = models
    markov.load_state_dict(dense.state_dict())
    xt = torch.rand(3000, 2, dtype=torch.float64).to(dev) * 1.4 - 0.2
    pd_, pm_ = dense.posterior(xt), markov.posterior(xt)
    assert (pd_.mean - pm_.mean).abs().max().item() < 1e-9
    assert (pd_.variance - pm_.variance).abs().max().item() < 1e-9
    e_dense, e_markov = dense._elbo(), markov._elbo()
    assert abs(e_dense.item() - e_markov.item()) <= 1e-9 * abs(e_dense.item())
    opt = torch.optim.Adam(markov.parameters(), lr=0.02)
    losses = []
    for _ in range(5):
        opt.zero_grad()
        loss = -markov._elbo()
        loss.backward()
        opt.step()
        losses.append(loss.item())
    assert losses[-1] < losses[0]
    with pytest.raises(NotImplementedError):
        markov._elbo(batch=torch.arange(100, device=dev))
