"""GPU tests of the epoch-shuffled minibatches in the binned layout (GridPlan.bin_epoch, csrc/minibatch.cuh): every batch view
is byte-identical to GridPlan.bin of its observations, the index sets follow the numpy restatement of the sampling law,
the batches of an epoch add up to the full data pass, a batch step matches the oracle on its subset, and the model API
(minibatches() + _elbo(batch=...)) trains, replays in a graph and refuses what it cannot do."""
import importlib
import os
import socket

import numpy as np
import pytest
import torch

from chunked_oracle import elbo_and_grads_chunked
from oracle import svgp_markov as SM
from oracle import vggp_oracle as O
from test_minibatch import epoch_batches

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def vg():
    if not torch.cuda.is_available():
        pytest.skip("no CUDA device")
    return importlib.import_module("variational-gridded-gaussian-processes_b200")


@pytest.fixture(scope="module")
def dev(vg):
    return torch.device("cuda", 0)


FAMILIES = [("b1", 1), ("b1", 2), ("b1", 3), ("markov", 1), ("markov", 2), ("markov", 3), ("b0", 1), ("b0", 2)]
KNOTS = {1: (37,), 2: (21, 17), 3: (9, 8, 7)}


def _family(vg, name):
    return {"b1": vg.B1_ASVGP, "markov": vg.SVGP_MARKOV, "b0": vg.B0_GRIDDED}[name]


def _problem(knots, N, seed, lo=-0.15, hi=1.15):
    D = len(knots)
    g = torch.Generator().manual_seed(seed)
    meshes = [torch.linspace(0, 1, k) for k in knots]
    X = torch.rand(N, D, generator=g, dtype=torch.float64) * (hi - lo) + lo
    y = torch.sin(3 * X[:, 0]) + (torch.cos(5 * X[:, -1]) if D > 1 else 0) + 0.1 * torch.randn(N, generator=g, dtype=torch.float64)
    return meshes, X, y


def _params(plan, seed):
    g = torch.Generator().manual_seed(seed)
    D = plan.D
    l = torch.rand(D, generator=g, dtype=torch.float64) * 0.3 + 0.2
    s2 = torch.rand(D, generator=g, dtype=torch.float64) * 0.8 + 0.6
    noise = torch.tensor(0.07, dtype=torch.float64)
    m = torch.randn(plan.M, generator=g, dtype=torch.float64) * 0.2
    Ls = [torch.eye(n, dtype=torch.float64) * 0.6 + 0.05 * torch.randn(n, n, generator=g, dtype=torch.float64) / n ** 0.5
          for n in plan.m_per_dim]
    return l, s2, noise, m, Ls


def _dev_inputs(plan, dev, l, s2, noise, m, Ls):
    theta = torch.cat([l, s2, noise.reshape(1)]).to(dev)
    return theta, m.to(dev), torch.cat([L.reshape(-1) for L in Ls]).to(dev)


def _sections(bo):
    d, T = bo.desc, int(bo.desc.n_tasks)
    buf = bo.buf

    def sec(off, nbytes):
        return buf[int(off):int(off) + nbytes].cpu()
    return {"header": sec(0, 256), "task_off": sec(d.off_task_off, 8 * T), "task_R": sec(d.off_task_R, 4 * T),
            "run_cell": sec(d.off_run_cell, 128 * T), "run_n": sec(d.off_run_n, 128 * T),
            "run_start": sec(d.off_run_start, 128 * T), "data": sec(d.off_data, int(d.data_elems) * bo.elem_size)}


def _assert_same_layout(got, want):
    for f in ("n", "n_inside", "n_tasks", "n_runs", "data_elems", "run_cap", "D"):
        assert getattr(got.desc, f) == getattr(want.desc, f), f
    a, b = _sections(got), _sections(want)
    # header[0] is the float64 sum of y^2 outside the mesh: k_bin_sum_y2 adds one partial per CTA atomically, so with more than
    # 256 such observations its last bit depends on the order the CTAs finish in, in GridPlan.bin as well
    ha, hb = a.pop("header"), b.pop("header")
    assert torch.equal(ha[8:], hb[8:])
    sa, sb = ha[:8].view(torch.float64).item(), hb[:8].view(torch.float64).item()
    assert abs(sa - sb) <= 1e-14 * abs(sb)
    for k in b:      # bitwise; NaN padding compares equal as bytes
        assert torch.equal(a[k], b[k]), k


@pytest.mark.parametrize("dtype", [torch.float32, torch.float64])
@pytest.mark.parametrize("name,D", FAMILIES)
def test_batches_are_the_binned_subsets(vg, dev, name, D, dtype):
    meshes, X, y = _problem(KNOTS[D], 3000, seed=D)
    plan = vg.GridPlan(_family(vg, name), meshes, dtype, dev)
    xs = [X[:, d].to(dev, dtype).contiguous() for d in range(D)]
    yy = y.to(dev, dtype).contiguous()
    # n % B != 0, one cell over run_cap, B = n, B = 1
    for B, cap, seed, epoch in ((700, 16, 1, 0), (1024, 256, 2, 5), (3000, 64, 3, 1), (1, 4, 4, 2)):
        if B == 1:
            xs1, yy1 = [x[:40].contiguous() for x in xs], yy[:40].contiguous()
        else:
            xs1, yy1 = xs, yy
        n = yy1.numel()
        ep = plan.bin_epoch(xs1, yy1, B, seed, epoch, run_cap=cap)
        sets = epoch_batches(n, B, seed, epoch)
        assert len(ep) == len(sets) == n // B
        for bo, idx in zip(ep, sets):
            assert bo.n == B and bo.scale == n / B
            it = torch.as_tensor(idx, device=dev)
            ref = plan.bin([x[it].contiguous() for x in xs1], yy1[it].contiguous(), cap)
            _assert_same_layout(bo, ref)


@pytest.mark.parametrize("name", ["b1", "markov", "b0"])
def test_dense_cell_and_sparse_cells(vg, dev, name):
    """One cell far above run_cap, and a fine mesh with one observation per cell (every run padded from 1 to 4)."""
    fam = _family(vg, name)
    plan = vg.GridPlan(fam, [torch.linspace(0, 1, 2001)], torch.float64, dev)
    x = ((torch.arange(1500, dtype=torch.float64) + 0.5) / 2000)[torch.randperm(1500, generator=torch.Generator().manual_seed(0))]
    x[:400] = 0.1234
    y = torch.randn(1500, dtype=torch.float64, generator=torch.Generator().manual_seed(1))
    xs, yy = [x.to(dev)], y.to(dev)
    ep = plan.bin_epoch(xs, yy, 500, 7, 3, run_cap=32)
    for bo, idx in zip(ep, epoch_batches(1500, 500, 7, 3)):
        it = torch.as_tensor(idx, device=dev)
        _assert_same_layout(bo, plan.bin([xs[0][it].contiguous()], yy[it].contiguous(), 32))


def test_draws_are_disjoint_and_fresh_per_epoch_and_seed():
    n, B = 10007, 1000
    sets = epoch_batches(n, B, 5, 0)
    allidx = np.concatenate(sets)
    assert all(s.size == B for s in sets) and len(sets) == n // B
    assert np.unique(allidx).size == allidx.size == (n // B) * B
    for other in (epoch_batches(n, B, 5, 1), epoch_batches(n, B, 6, 0)):
        assert not np.array_equal(other[0], sets[0])


def test_deterministic_step_on_a_batch_is_bitwise_the_subset_step(vg, dev):
    meshes, X, y = _problem((33, 29), 20000, seed=11)
    plan = vg.GridPlan(vg.B1_ASVGP, meshes, torch.float64, dev)
    plan.set_deterministic(True)
    theta, m, L = _dev_inputs(plan, dev, *_params(plan, 3))
    xs = [X[:, d].to(dev).contiguous() for d in range(2)]
    yy = y.to(dev)
    ep = plan.bin_epoch(xs, yy, 6000, 9, 0, run_cap=64)
    for bo, idx in zip(ep, epoch_batches(20000, 6000, 9, 0)):
        it = torch.as_tensor(idx, device=dev)
        ref = plan.bin([x[it].contiguous() for x in xs], yy[it].contiguous(), 64)
        a = [t.clone() for t in plan.step(theta, m, L, bo, None, ell_scale=bo.scale)]
        b = [t.clone() for t in plan.step(theta, m, L, ref, None, ell_scale=bo.scale)]
        for u, v in zip(a, b):
            assert torch.equal(u, v)


@pytest.mark.parametrize("name,D", FAMILIES)
def test_batches_of_an_epoch_sum_to_the_full_pass(vg, dev, name, D):
    meshes, X, y = _problem(KNOTS[D], 4000, seed=20 + D)
    plan = vg.GridPlan(_family(vg, name), meshes, torch.float64, dev)
    theta, m, L = _dev_inputs(plan, dev, *_params(plan, 4))
    xs = [X[:, d].to(dev).contiguous() for d in range(D)]
    yy = y.to(dev)
    plan.grid_forward(theta, m, L)
    full = torch.empty_like(plan.gbuf)
    plan.obs_fwd_bwd(plan.bin(xs, yy), gbuf=full)
    acc_o, acc_s = None, None
    g = torch.empty_like(plan.gbuf)
    for bo in plan.bin_epoch(xs, yy, 500, 1, 0):
        plan.obs_fwd_bwd(bo, gbuf=g)
        o, s = plan.gbuf_views(g)
        acc_o = o.clone() if acc_o is None else acc_o + o
        acc_s = s.clone() if acc_s is None else acc_s + s
    fo, fs = plan.gbuf_views(full)
    assert (acc_o - fo).abs().max().item() <= 1e-12 * max(1.0, fo.abs().max().item())
    assert (acc_s - fs).abs().max().item() <= 1e-12 * max(1.0, fs.abs().max().item())


ORACLE_CASES = [("b1", (14, 11)), ("b0", (10, 8)), ("markov", (12, 9))]


@pytest.mark.parametrize("dtype,tol", [(torch.float64, 1e-8), (torch.float32, 1e-3)])
@pytest.mark.parametrize("name,knots", ORACLE_CASES)
def test_batch_step_matches_oracle_on_its_subset(vg, dev, name, knots, dtype, tol):
    N, B = 2400, 700
    meshes, X, y = _problem(knots, N, seed=31)
    fam = _family(vg, name)
    plan = vg.GridPlan(fam, meshes, dtype, dev)
    l, s2, noise, m, Ls = _params(plan, 5)
    theta, md, L = _dev_inputs(plan, dev, l, s2, noise, m, Ls)
    Xq, yq = X.to(dtype).to(torch.float64), y.to(dtype).to(torch.float64)
    xs = [Xq[:, d].to(dev, dtype).contiguous() for d in range(2)]
    ep = plan.bin_epoch(xs, yq.to(dev, dtype).contiguous(), B, 2, 1)
    idx = torch.as_tensor(epoch_batches(N, B, 2, 1)[1])
    bo = ep[1]
    out, dtheta, dm, dL = plan.step(theta, md, L, bo, None, ell_scale=bo.scale)
    if fam == vg.SVGP_MARKOV:
        ref, gref = SM.value_and_grads(meshes, Xq[idx], yq[idx], l, s2, noise, m, Ls, scale=N / B)
    else:
        ref, gref = elbo_and_grads_chunked(O.B1_ASVGP if fam == vg.B1_ASVGP else O.B0_GRIDDED, meshes, Xq[idx], yq[idx], l, s2,
                                           noise, m, Ls, scale=N / B)

    def rel(a, b):
        a, b = a.detach().cpu().to(torch.float64).reshape(-1), b.detach().cpu().to(torch.float64).reshape(-1)
        return ((a - b).norm() / b.norm().clamp_min(1e-300)).item()
    assert abs(out[0].item() - ref.item()) <= tol * abs(ref.item())
    assert rel(dtheta[:2], gref[0]) < 10 * tol and rel(dtheta[2:4], gref[1]) < 10 * tol and rel(dtheta[4], gref[2]) < 10 * tol
    assert rel(dm, gref[3]) < 10 * tol
    off = 0
    for d, n in enumerate(plan.m_per_dim):
        assert rel(torch.tril(dL[off:off + n * n].reshape(n, n)), torch.tril(gref[4 + d])) < 10 * tol
        off += n * n


def _model(name, X, y):
    ks = importlib.import_module("variational-gridded-gaussian-processes_b200.models.sparse.kronecker_structure")
    gk = importlib.import_module("variational-gridded-gaussian-processes_b200.models.sparse.gridded_kronecker_structure")
    if name == "b1":
        return gk.GriddedMatern12ASVGP(X, y, 20, 2, (0, 1), (0, 1))
    if name == "b0":
        return gk.Matern12GriddedGP(X, y, 20, (0, 1), (0, 1))
    return ks.Matern12SVGP(X, y, torch.stack([torch.linspace(0, 1, 20), torch.linspace(0, 1, 20)], 1), markov=True)


@pytest.mark.parametrize("name", ["b1", "b0", "markov"])
def test_model_minibatch_training_and_graph_replay(vg, dev, name):
    meshes, X, y = _problem((2, 2), 6000, seed=41, lo=0.0, hi=1.0)
    mdl = _model(name, X.to(torch.float32), y.to(torch.float32)).to(dev)
    opt = torch.optim.Adam(mdl.parameters(), lr=0.01)
    mb = mdl.minibatches(2000, seed=3)
    losses = []
    for e in range(2):
        batches = list(mb.epoch(e))
        assert len(batches) == 3
        for bo in batches:
            opt.zero_grad()
            loss = -mdl._elbo(batch=bo)
            loss.backward()
            opt.step()
            losses.append(loss.item())
            assert all(torch.isfinite(p.grad).all() for p in mdl.parameters() if p.grad is not None)
    assert all(np.isfinite(losses))
    mdl.check_factorisation()
    # a graph captured on one batch replays that batch's step
    plan = mdl._ensure_plan()
    bo = batches[0]
    theta = mdl._theta()
    m = mdl.variational_mean.detach().to(torch.float64).contiguous()
    L = torch.cat([c.detach().to(torch.float64).reshape(-1) for c in mdl._chols()]).contiguous()
    eager = [t.clone() for t in plan.step(theta, m, L, bo, None, ell_scale=bo.scale)]
    gs = plan.graphed_step(theta, m, L, bo, None, ell_scale=bo.scale)
    replay = gs.replay()
    torch.cuda.synchronize()
    for a, b in zip(replay, eager):      # float32 observations: the gradient sums are atomic, their order varies per run
        assert ((a - b).norm() / b.norm().clamp_min(1e-300)).item() < 1e-3
    if name == "markov":
        with pytest.raises(NotImplementedError, match="minibatches"):
            mdl._elbo(batch=torch.arange(10, device=dev))


def test_refusals(vg, dev):
    ks = importlib.import_module("variational-gridded-gaussian-processes_b200.models.sparse.kronecker_structure")
    meshes, X, y = _problem((8, 8), 200, seed=2, lo=0.0, hi=1.0)
    Z = torch.stack([torch.linspace(0, 1, 8)] * 2, 1)
    dense = ks.Matern12SVGP(X, y, Z, markov=False).to(torch.float64).to(dev)
    with pytest.raises(NotImplementedError):
        dense.minibatches(50)
    for fam, knots in ((vg.SVGP_GRID, (8, 8)), (vg.VFF_GRID, (9, 9)), (vg.B0_GRIDDED, (6, 5, 4))):
        plan = vg.GridPlan(fam, [torch.linspace(0, 1, k) for k in knots], torch.float64, dev)
        xs = [torch.rand(100, dtype=torch.float64, device=dev) for _ in knots]
        with pytest.raises(RuntimeError, match="status -6"):
            plan.bin_epoch(xs, torch.rand(100, dtype=torch.float64, device=dev), 10, 0, 0)
    plan = vg.GridPlan(vg.B1_ASVGP, meshes, torch.float64, dev)
    xs = [X[:, d].to(dev).contiguous() for d in range(2)]
    for B in (0, 201):
        with pytest.raises(RuntimeError, match="status -1"):
            plan.bin_epoch(xs, y.to(dev), B, 0, 0)


def _free_port():
    s = socket.socket()
    s.bind(("127.0.0.1", 0))
    p = s.getsockname()[1]
    s.close()
    return p


def _sharded_model(dev, rank, world):
    gk = importlib.import_module("variational-gridded-gaussian-processes_b200.models.sparse.gridded_kronecker_structure")
    _, X, y = _problem((2, 2), 9000, seed=51, lo=0.0, hi=1.0)
    mdl = gk.GriddedMatern12ASVGP(X, y, 20, 2, (0, 1), (0, 1)).to(torch.float64).to(dev)
    if world > 1:
        mdl.shard_observations(rank, world)
    return mdl, X, y


def _sharded_run(rank, world, port, out_dir):
    import torch.distributed as dist
    os.environ["MASTER_ADDR"] = "127.0.0.1"
    os.environ["MASTER_PORT"] = str(port)
    torch.cuda.set_device(rank)
    dev = torch.device("cuda", rank)
    dist.init_process_group("nccl", rank=rank, world_size=world, device_id=dev)
    mdl, _, _ = _sharded_model(dev, rank, world)
    bo = next(iter(mdl.minibatches(1000, seed=4).epoch(2)))
    e = mdl._elbo(batch=bo)
    e.backward()
    if rank == 0:
        torch.save({"elbo": e.item(), "gm": mdl.variational_mean.grad.cpu()}, os.path.join(out_dir, "mb.pt"))
    dist.barrier()
    dist.destroy_process_group()


def test_sharded_batches_match_one_process_on_the_union(vg, tmp_path):
    if torch.cuda.device_count() < 2:
        pytest.skip("needs 2 GPUs")
    import torch.multiprocessing as mp
    mp.spawn(_sharded_run, args=(2, _free_port(), str(tmp_path)), nprocs=2, join=True)
    got = torch.load(os.path.join(str(tmp_path), "mb.pt"))
    dev = torch.device("cuda", 0)
    mdl, X, y = _sharded_model(dev, 0, 1)
    dist_mod = importlib.import_module("variational-gridded-gaussian-processes_b200.dist")
    idx = []
    for r in range(2):
        lo, hi = dist_mod.shard_bounds(9000, r, 2)
        idx.append(lo + epoch_batches(hi - lo, 1000, 4, 2, rank=r)[0])
    union = torch.as_tensor(np.concatenate(idx))
    plan = mdl._ensure_plan()
    obs = plan.bin([X[union, d].to(dev).contiguous() for d in range(2)], y[union].to(dev).contiguous())
    m = mdl.variational_mean.detach().to(torch.float64).contiguous()
    L = torch.cat([c.detach().to(torch.float64).reshape(-1) for c in mdl._chols()]).contiguous()
    out, _, dm, _ = plan.step(mdl._theta(), m, L, obs, None, ell_scale=4500 / 1000)
    assert abs(out[0].item() - got["elbo"]) <= 1e-10 * abs(got["elbo"])
    assert ((dm.cpu() - got["gm"]).norm() / got["gm"].norm()).item() <= 1e-10
