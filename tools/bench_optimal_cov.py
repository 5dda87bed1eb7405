"""Benchmark of the optimal Kronecker-factored covariance (vggp_covopt_update, csrc/covopt.cuh).  Prints one JSON line per
workload; also appends them to --out if given.

Workloads: N = 2^26 float32 track observations (vggp_generate_tracks) on 512 x 512 points (tracks512) and on 256 x 256 x 64
points (3d), each for the B1 family and the Markov SVGP family, theta of tools/bench_svgp_markov.py.  Per workload:
  mean       m* first (Kronecker-preconditioned CG to rtol --mean-rtol, at most --mean-max-iter iterations); every number below
             is at m = m*
  sweeps     coordinate sweeps from L_d = I until the summed factor change of a sweep is <= --rtol: sweep count, the change of
             every sweep, wall time (host clock around the synchronising read of the change that ends every sweep)
  update     one update (grid forward + the family's per-observation kernel + vggp_covopt_update) and one sweep, host clock
             around a synchronising call, median of --reps
  kernels    device time of the update kernels (k_co_*) and of the per-observation kernel of the same updates, torch.profiler
             over one sweep in a run of its own
  elbo       at (m*, I), after the sweeps, and after Adam (lr --lr) on the L_d alone, eager steps, for the wall time the sweeps took
The card's name and power limit are read in the same run."""
import argparse
import importlib
import json
import os
import sys
import time

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tools"))
import bench_svgp_markov as BS        # noqa: E402  (gpu_info, params)
import bench_optimal_mean as BM       # noqa: E402  (kernel_totals)


def eye_factors(knots, dev):
    return torch.cat([torch.eye(k, dtype=torch.float64).reshape(-1) for k in knots]).to(dev)


def workload(vg, gen, name, family, knots, n, dev, args):
    D = len(knots)
    meshes = [torch.linspace(0, 1, k) for k in knots]
    xs, y = gen.generate_tracks(0, n, n, dev, torch.float32, seed=0, D=D)
    plan = vg.GridPlan(family, meshes, torch.float32, dev)
    obs = plan.bin(xs, y)
    del xs, y
    theta, _, _ = BS.params(knots, dev)
    L0 = eye_factors(knots, dev)
    zero = torch.zeros(plan.M, dtype=torch.float64, device=dev)
    plan.grid_forward(theta, zero, L0)
    plan.meanopt_assemble(obs)
    m, mit, mrr = plan.meanopt_solve(args.mean_rtol, args.mean_max_iter, "kronecker")
    rec = {"bench": "optimal_cov", "workload": name, "family": "B1" if family == vg.B1_ASVGP else "SVGP_MARKOV",
           "knots": list(knots), "n": n, "obs_dtype": "float32", **BS.gpu_info(), "mean_iters": mit, "mean_relres": mrr}
    change = torch.zeros(1, dtype=torch.float64, device=dev)
    kname = "k_obs_b1_binned" if family == vg.B1_ASVGP else "k_obs_svgpm_binned"

    def update(d, L):
        plan.grid_forward(theta, m, L)
        plan.obs_fwd_bwd(obs)
        plan.covopt_update(d, plan.gbuf, 1.0, L, change)

    def sweep(L):
        change.zero_()
        for d in range(D):
            update(d, L)
        return change.item()

    sweep(L0.clone())                                   # first call: allocation, module load
    elbo = lambda L: plan.step(theta, m, L, obs, None)[0][0].item()       # noqa: E731
    rec["elbo_identity"] = elbo(L0)
    # sweeps from L_d = I
    L = L0.clone()
    changes = []
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    while len(changes) < args.max_sweeps:
        changes.append(sweep(L))
        if changes[-1] <= args.rtol:
            break
    wall = time.perf_counter() - t0
    rec.update({"rtol": args.rtol, "sweeps": len(changes), "converged": changes[-1] <= args.rtol, "changes": changes,
                "sweeps_wall_ms": wall * 1e3, "elbo_after": elbo(L), "scratch_bytes": plan.workspace_bytes()["scratch"]})
    # one update and one sweep, host clock around a synchronising call
    Lw = L.clone()
    up, sw = [], []
    for _ in range(args.reps):
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        update(D - 1, Lw)
        torch.cuda.synchronize()
        up.append((time.perf_counter() - t0) * 1e3)
        t0 = time.perf_counter()
        sweep(Lw)
        sw.append((time.perf_counter() - t0) * 1e3)
    up.sort()
    sw.sort()
    rec.update({"update_ms_median": up[len(up) // 2], "sweep_ms_median": sw[len(sw) // 2]})
    # device times over one sweep, in a run of its own
    names = ["k_co_factor", "k_co_b1_x", "k_co_b1_rq", "k_co_markov", "k_co_change", kname]
    kt = BM.kernel_totals(lambda: sweep(Lw), names)
    co_ms = sum(kt[k][0] for k in names[:-1])
    rec["kernels_one_sweep"] = {k: {"ms": v[0], "launches": v[1]} for k, v in kt.items()}
    rec["covopt_kernels_ms_per_update"] = co_ms / D
    rec["data_pass_kernel_ms_per_update"] = kt[kname][0] / max(kt[kname][1], 1)
    rec["covopt_over_data_pass"] = rec["covopt_kernels_ms_per_update"] / rec["data_pass_kernel_ms_per_update"]
    # Adam on the L_d alone for the wall time of the sweeps
    P = L0.clone().requires_grad_(True)
    opt = torch.optim.Adam([P], lr=args.lr)
    steps = 0
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    while time.perf_counter() - t0 < wall:
        _, _, _, dL = plan.step(theta, m, P.detach(), obs, None)
        P.grad = -dL
        opt.step()
        steps += 1
        torch.cuda.synchronize()
    rec.update({"adam_lr": args.lr, "adam_steps": steps, "elbo_adam_same_wall": elbo(P.detach())})
    del plan, obs
    torch.cuda.empty_cache()
    return rec


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--n", type=int, default=1 << 26)
    ap.add_argument("--reps", type=int, default=10)
    ap.add_argument("--rtol", type=float, default=1e-8)
    ap.add_argument("--max-sweeps", type=int, default=100)
    ap.add_argument("--mean-rtol", type=float, default=1e-8)
    ap.add_argument("--mean-max-iter", type=int, default=20000)
    ap.add_argument("--lr", type=float, default=0.01)
    ap.add_argument("--only", default=None, help="comma-separated workload names")
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("bench_optimal_cov needs a CUDA device")
    vg = importlib.import_module("variational-gridded-gaussian-processes_b200")
    gen = importlib.import_module("variational-gridded-gaussian-processes_b200.utils.dataloaders")
    dev = torch.device("cuda", 0)
    wls = [("tracks512_b1", vg.B1_ASVGP, (512, 512)), ("tracks512_markov", vg.SVGP_MARKOV, (512, 512)),
           ("3d_b1", vg.B1_ASVGP, (256, 256, 64)), ("3d_markov", vg.SVGP_MARKOV, (256, 256, 64))]
    for name, fam, knots in wls:
        if args.only and name not in args.only.split(","):
            continue
        line = json.dumps(workload(vg, gen, name, fam, knots, args.n, dev, args))
        print(line, flush=True)
        if args.out:
            with open(args.out, "a") as f:
                f.write(line + "\n")


if __name__ == "__main__":
    main()
