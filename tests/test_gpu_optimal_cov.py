"""GPU tests of the optimal Kronecker-factored covariance (vggp_covopt_update, csrc/covopt.cuh): parity with the float64
oracle (oracle/optimal_cov.py), the uncollapsed == collapsed identity for D = 1 after set_optimal_mean() and
set_optimal_covariance(), full-size convergence, the model method and a two-process sharded run."""
import importlib
import os
import socket

import pytest
import torch

from oracle import optimal_cov as OC
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
    noise = torch.tensor(0.07, dtype=torch.float64)
    m = 0.2 * torch.randn(int(torch.tensor(knots).prod()), generator=g, dtype=torch.float64)
    Ls = [torch.eye(n, dtype=torch.float64) * 0.6 + 0.02 * torch.randn(n, n, generator=g, dtype=torch.float64) for n in knots]
    return meshes, X, y, l, s2, noise, m, Ls


def _relerr(a, b):
    a = a.detach().cpu().to(torch.float64).reshape(-1)
    b = b.detach().cpu().to(torch.float64).reshape(-1)
    return ((a - b).norm() / b.norm().clamp_min(1e-300)).item()


def _blocks(plan, Lcat):
    out, off = [], 0
    for n in plan.m_per_dim:
        out.append(Lcat[off:off + n * n].reshape(n, n))
        off += n * n
    return out


def _update(plan, d, theta, m, Lcat, obs, change):
    plan.grid_forward(theta, m, Lcat)
    plan.obs_fwd_bwd(obs)
    plan.covopt_update(d, plan.gbuf, 1.0, Lcat, change)


@pytest.mark.parametrize("markov", [False, True])
@pytest.mark.parametrize("knots,N", [((40,), 5000), ((33, 29), 5000), ((12, 10, 8), 5000)])
@pytest.mark.parametrize("dtype,tol", [(torch.float64, 1e-10), (torch.float32, 1e-5)])
def test_update_matches_oracle(vg, dev, markov, knots, N, dtype, tol):
    family = O.SVGP_GRID if markov else O.B1_ASVGP
    meshes, X, y, l, s2, noise, m, Ls = _problem(markov, knots, N, seed=7 + len(knots))
    Xq = X.to(dtype).to(torch.float64)
    plan = vg.GridPlan(vg.SVGP_MARKOV if markov else vg.B1_ASVGP, meshes, dtype, dev)
    theta = torch.cat([l, s2, noise.reshape(1)]).to(dev)
    Lcat = torch.cat([L.reshape(-1) for L in Ls]).to(dev)
    obs = plan.bin([Xq[:, d].to(dev, dtype).contiguous() for d in range(len(knots))], y.to(dev, dtype).contiguous())
    change = torch.zeros(1, dtype=torch.float64, device=dev)
    for d in range(len(knots)):
        prev = [b.cpu().clone() for b in _blocks(plan, Lcat)]
        ref = OC.update(family, meshes, Xq, l, s2, noise, prev, d)
        _update(plan, d, theta, m.to(dev), Lcat, obs, change)
        got = _blocks(plan, Lcat)[d]
        assert _relerr(got, ref) <= tol, (d, _relerr(got, ref))
    assert plan.read_info() == 0


@pytest.mark.parametrize("markov", [False, True])
def test_uncollapsed_bound_reaches_the_collapsed_bound_in_1d(vg, dev, markov):
    family = O.SVGP_GRID if markov else O.B1_ASVGP
    meshes, X, y, l, s2, noise, m, Ls = _problem(markov, (60,), 3000, seed=5)
    model = importlib.import_module("variational-gridded-gaussian-processes_b200.models._gridded")

    class Model(model.GriddedVariationalGP):
        pass

    Model.family = vg.SVGP_MARKOV if markov else vg.B1_ASVGP
    mdl = Model(X, y, meshes).to(torch.float64).to(dev)
    mdl.kernel.base_kernel.lengthscale = l.to(dev)
    mdl.kernel.outputscale = s2.to(dev)
    mdl.likelihood.noise = noise.to(dev)
    ls, os_, nz = [t.detach().cpu().reshape(-1) for t in mdl._hyper()]
    mdl.set_optimal_mean(rtol=1e-13)
    res = mdl.set_optimal_covariance()
    assert res["sweeps"] == 2                      # one update gives the optimum; the second sweep confirms it
    ref = O.elbo_collapsed_literal(family, meshes, X, y, ls, os_, nz.reshape(()), ref_quirks=False)
    got = mdl._elbo().item()
    assert abs(got - ref.item()) <= 1e-8 * abs(ref.item()), (got, ref.item())
    assert abs(res["elbo"] - got) <= 1e-10 * abs(got)


@pytest.mark.parametrize("markov,knots,N", [(False, (512, 512), 1 << 22), (True, (512, 512), 1 << 22),
                                            (False, (64, 64, 16), 1 << 20), (True, (64, 64, 16), 1 << 20)])
def test_full_size_sweeps_converge_and_ascend(vg, dev, markov, knots, N):
    gen = importlib.import_module("variational-gridded-gaussian-processes_b200.utils.dataloaders")
    D = len(knots)
    meshes = [torch.linspace(0, 1, k) for k in knots]
    xs, y = gen.generate_tracks(0, N, N, dev, torch.float32, seed=3, D=D)
    plan = vg.GridPlan(vg.SVGP_MARKOV if markov else vg.B1_ASVGP, meshes, torch.float32, dev)
    obs = plan.bin(xs, y)
    theta = torch.tensor([0.3] * D + [0.8] * D + [0.05], dtype=torch.float64, device=dev)
    Lcat = torch.cat([torch.eye(k, dtype=torch.float64).reshape(-1) for k in knots]).to(dev)
    m = torch.zeros(plan.M, dtype=torch.float64, device=dev)
    change = torch.zeros(1, dtype=torch.float64, device=dev)
    # float32 observations: the float32 band sums of the gradient buffer change in their last bits from one data pass to the
    # next (atomics), which leaves the change of a sweep at a floor near 3e-8 (512 x 512 Markov, one B200); rtol 1e-7 here
    rtol = 1e-7
    elbos = [plan.step(theta, m, Lcat, obs, None)[0][0].item()]
    for sweep in range(100):
        change.zero_()
        for d in range(D):
            _update(plan, d, theta, m, Lcat, obs, change)
            elbos.append(plan.step(theta, m, Lcat, obs, None)[0][0].item())
        if change.item() <= rtol:
            break
    assert change.item() <= rtol, (sweep, change.item())
    # float32 observations: the gradient buffer carries ~1e-7 relative noise, so ascent holds up to that
    assert all(b >= a - 1e-6 * abs(a) for a, b in zip(elbos, elbos[1:])), elbos
    print(f"{knots} markov={markov}: {sweep + 1} sweeps, ELBO {elbos[0]:.6e} -> {elbos[-1]:.6e}")


def test_markov_model_set_optimal_covariance(vg, dev):
    ks = importlib.import_module("variational-gridded-gaussian-processes_b200.models.sparse.kronecker_structure")
    g = torch.Generator().manual_seed(71)
    N = 20000
    X = torch.rand(N, 2, generator=g, dtype=torch.float64) * 1.2 - 0.1
    y = torch.sin(4 * X[:, 0]) * torch.cos(3 * X[:, 1]) + 0.05 * torch.randn(N, generator=g, dtype=torch.float64)
    Z = torch.stack([torch.linspace(0, 1, 30), torch.linspace(0, 1, 30) ** 1.2], dim=1)
    mdl = ks.Matern12SVGP(X, y, Z, markov=True).to(torch.float64).to(dev)
    mdl.set_optimal_mean()
    e0 = mdl._elbo().item()
    start = [c.detach().clone() for c in mdl._chols()]
    with pytest.raises(RuntimeError, match="unchanged"):
        mdl.set_optimal_covariance(max_sweeps=1)
    assert all(torch.equal(a, b.detach()) for a, b in zip(start, mdl._chols()))
    res = mdl.set_optimal_covariance()
    assert 1 < res["sweeps"] <= 100 and res["change"] <= 1e-8
    mdl.zero_grad()
    e1 = mdl._elbo()
    assert e1.item() > e0 and abs(res["elbo"] - e1.item()) <= 1e-10 * abs(e1.item())
    e1.backward()
    for c in mdl._chols():                     # stationary in every factor
        assert torch.tril(c.grad).norm().item() <= 1e-5 * abs(e1.item())
    dense = ks.Matern12SVGP(X, y, Z, markov=False).to(torch.float64).to(dev)
    with pytest.raises(NotImplementedError, match="set_optimal_q"):
        dense.set_optimal_covariance()


def _free_port():
    s = socket.socket()
    s.bind(("127.0.0.1", 0))
    p = s.getsockname()[1]
    s.close()
    return p


def _sharded_factors(rank, world, port, out_dir):
    import torch.distributed as dist
    import vggp_b200 as vg
    os.environ["MASTER_ADDR"] = "127.0.0.1"
    os.environ["MASTER_PORT"] = str(port)
    torch.cuda.set_device(rank)
    dev = torch.device("cuda", rank)
    dist.init_process_group("nccl", rank=rank, world_size=world, device_id=dev)
    mdl = _sharded_model(vg, dev, rank, world)
    res = mdl.set_optimal_covariance()
    if rank == 0:
        torch.save({"res": res, "L": [c.detach().cpu() for c in mdl._chols()]}, os.path.join(out_dir, "covopt.pt"))
    dist.barrier()
    dist.destroy_process_group()


def _sharded_model(vg, dev, rank, world):
    model = importlib.import_module("variational-gridded-gaussian-processes_b200.models._gridded")
    meshes, X, y, l, s2, noise, m, Ls = _problem(False, (40, 30), 20000, seed=13)
    mdl = model.GriddedVariationalGP(X, y, meshes).to(torch.float64).to(dev)
    if world > 1:
        mdl.shard_observations(rank, world)
    return mdl


def test_sharded_model_matches_one_process(vg, tmp_path):
    if torch.cuda.device_count() < 2:
        pytest.skip("needs 2 GPUs")
    import torch.multiprocessing as mp
    mp.spawn(_sharded_factors, args=(2, _free_port(), str(tmp_path)), nprocs=2, join=True)
    got = torch.load(os.path.join(str(tmp_path), "covopt.pt"))
    mdl = _sharded_model(vg, torch.device("cuda", 0), 0, 1)
    res = mdl.set_optimal_covariance()
    assert res["sweeps"] == got["res"]["sweeps"]
    for a, b in zip(got["L"], mdl._chols()):
        assert _relerr(a, b) <= 1e-10
