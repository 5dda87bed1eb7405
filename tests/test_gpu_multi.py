"""Two-rank GPU tests (skipped with fewer than two GPUs; `python -m pytest tests/test_gpu_multi.py -m gpu` on a machine with two):
the library's peer-memory all-reduce kernel (vggp_allreduce_gbuf) against NCCL on the same buffers, and a sharded step
through it against the single-process step on the whole data set."""
import os
import socket

import pytest
import torch

pytestmark = pytest.mark.gpu


def _free_port():
    s = socket.socket()
    s.bind(("127.0.0.1", 0))
    p = s.getsockname()[1]
    s.close()
    return p


def _worker(rank, world, port, dtype_name, out_dir):
    import torch.distributed as dist
    import vggp_b200 as vg
    from test_gpu_elbo import make_problem
    os.environ["MASTER_ADDR"] = "127.0.0.1"
    os.environ["MASTER_PORT"] = str(port)
    torch.cuda.set_device(rank)
    dev = torch.device("cuda", rank)
    dist.init_process_group("nccl", rank=rank, world_size=world, device_id=dev)
    dtype = getattr(torch, dtype_name)
    knots, N = (70, 45), 20000
    meshes, X, y, l, s2, noise, m, Ls = make_problem(knots, N, seed=31)
    theta = torch.cat([l, s2, noise.reshape(1)]).to(dev)
    Lcat = torch.cat([L.reshape(-1) for L in Ls]).to(dev)
    lo, hi = vg.shard_bounds(N, rank, world)
    xs = [X[lo:hi, d].to(dtype).contiguous().to(dev) for d in range(2)]
    ys = y[lo:hi].to(dtype).to(dev)
    res = {}
    for mode in ("nccl", "peer"):
        plan = vg.GridPlan(vg.B1_ASVGP, meshes, dtype, dev)
        if mode == "peer":
            res["multicast"] = plan.enable_peer_allreduce()
        obs = plan.bin(xs, ys, run_cap=64)
        for rep in range(3):                      # several calls: the barrier sequence numbers advance
            out, dtheta, dm, dL = plan.step(theta, m.to(dev), Lcat, obs, None, 1.0, group="world")
        torch.cuda.synchronize()
        if mode == "peer":
            assert not plan.peer_allreduce_failed()
        gobs, gscal = plan.gbuf_views()
        res[mode] = [t.detach().cpu().double() for t in (out, dtheta, dm, dL, gobs, gscal)]
    if rank == 0:
        torch.save(res, os.path.join(out_dir, f"res_{dtype_name}.pt"))
    dist.barrier()
    dist.destroy_process_group()


@pytest.mark.parametrize("dtype_name", ["float32", "float64"])
def test_peer_allreduce_matches_nccl_and_single_process(tmp_path, dtype_name):
    if torch.cuda.device_count() < 2:
        pytest.skip("needs 2 GPUs")
    import torch.multiprocessing as mp
    import vggp_b200 as vg
    from test_gpu_elbo import make_problem, relerr
    mp.spawn(_worker, args=(2, _free_port(), dtype_name, str(tmp_path)), nprocs=2, join=True)
    res = torch.load(os.path.join(str(tmp_path), f"res_{dtype_name}.pt"))
    tol = 1e-10 if dtype_name == "float64" else 1e-5       # the two collectives sum in different orders
    for a, b in zip(res["peer"], res["nccl"]):
        assert relerr(a, b) < tol
    # against the single-process step on the whole data set
    dev = torch.device("cuda", 0)
    dtype = getattr(torch, dtype_name)
    knots, N = (70, 45), 20000
    meshes, X, y, l, s2, noise, m, Ls = make_problem(knots, N, seed=31)
    plan = vg.GridPlan(vg.B1_ASVGP, meshes, dtype, dev)
    xs = [X[:, d].to(dtype).contiguous().to(dev) for d in range(2)]
    out, dtheta, dm, dL = plan.step(torch.cat([l, s2, noise.reshape(1)]).to(dev), m.to(dev),
                                    torch.cat([L.reshape(-1) for L in Ls]).to(dev), plan.bin(xs, y.to(dtype).to(dev), run_cap=64), None)
    for a, b in zip(res["peer"][:4], (out, dtheta, dm, dL)):
        assert relerr(a, b) < (1e-10 if dtype_name == "float64" else 1e-4)
    print("multicast path:", res["multicast"])
