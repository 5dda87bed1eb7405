"""Benchmark of the optimal variational mean (vggp_meanopt_assemble / vggp_meanopt_solve, csrc/meanopt.cuh).  Prints one JSON
line per workload; also appends them to --out if given.

Workloads: N = 2^26 float32 track observations (vggp_generate_tracks) on 512 x 512 points (tracks512) and on 256 x 256 x 64
points (3d), each for the B1 family and the Markov SVGP family, theta of tools/bench_svgp_markov.py.  Per workload:
  assemble   the whole call (zeroing of G and b + the per-observation kernel) by CUDA events over --reps launches, and the
             kernel alone (torch.profiler); its algorithmic bytes (D + 1) sizeof(T) N and their share of the HBM copy rate
             measured in the same run (device-to-device copy of 2 GiB)
  k1         the per-observation ELBO kernel of the family (k_obs_b1_binned / k_obs_svgpm_binned) on the same binned buffer:
             the whole call by events and the kernel alone, in launches alternated with the assemble launches
  solve      cold start (m = 0) to rtol --rtol: iterations, total ms, ms per iteration, relative residual
  elbo       at m = 0, at m*, and after Adam (lr --lr) on m alone, eager steps, for the wall time of assemble + solve
With --preconditioner jacobi,kronecker it measures the solves instead, one record per workload: every listed preconditioner
on the same assembled system, cold start (m = 0) to rtol --rtol: iterations, relative residual, solve time (host clock
around the synchronising call, after one untimed solve), time per iteration, the step's ||dm|| at m* over ||dm|| at 0, and
from torch.profiler (CUPTI activity records of a solve of its own with rtol = 0, so that all --profile-iters iterations
do work and no launch returns early on a converged status) the device time of one stencil product (k_mo_matvec) and of one
preconditioner application (the D k_mo_kron_sweep launches of one iteration).
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
import bench_svgp_markov as BS        # noqa: E402  (gpu_info, params, timed)


def copy_rate_gbs(dev, nbytes=1 << 31, reps=10):
    src = torch.empty(nbytes // 4, dtype=torch.float32, device=dev)
    dst = torch.empty_like(src)
    dst.copy_(src)
    ms = BS.timed(lambda: dst.copy_(src), reps)
    del src, dst
    return 2 * nbytes / (ms * 1e-3) / 1e9


def kernel_ms(fn, name, reps):
    """Mean device time of the kernels whose name contains `name` over `reps` calls of fn (torch.profiler)."""
    from torch.profiler import ProfilerActivity, profile
    torch.cuda.synchronize()
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        for _ in range(reps):
            fn()
        torch.cuda.synchronize()
    tot, cnt = 0.0, 0
    for e in prof.events():
        if name in e.name and e.device_type == torch.autograd.DeviceType.CUDA:
            tot += e.device_time_total if hasattr(e, "device_time_total") else e.cuda_time_total
            cnt += 1
    return tot / max(cnt, 1) / 1e3, cnt


def kernel_totals(fn, names):
    """{name: (total device ms, launches)} of the kernels whose name contains each of `names` in one call of fn"""
    from torch.profiler import ProfilerActivity, profile
    torch.cuda.synchronize()
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        fn()
        torch.cuda.synchronize()
    out = {k: [0.0, 0] for k in names}
    for e in prof.events():
        if e.device_type != torch.autograd.DeviceType.CUDA:
            continue
        for k in names:
            if k in e.name:
                out[k][0] += (e.device_time_total if hasattr(e, "device_time_total") else e.cuda_time_total) / 1e3
                out[k][1] += 1
    return {k: tuple(v) for k, v in out.items()}


def solve_workload(vg, gen, name, family, knots, n, dev, args):
    D = len(knots)
    meshes = [torch.linspace(0, 1, k) for k in knots]
    xs, y = gen.generate_tracks(0, n, n, dev, torch.float32, seed=0, D=D)
    plan = vg.GridPlan(family, meshes, torch.float32, dev)
    obs = plan.bin(xs, y)
    del xs, y
    theta, _, L = BS.params(knots, dev)
    zero = torch.zeros(plan.M, dtype=torch.float64, device=dev)
    plan.grid_forward(theta, zero, L)
    plan.meanopt_assemble(obs)                        # one assembled system for every solve below
    dm0 = plan.step(theta, zero, L, obs, None)[2].norm().item()
    rec = {"bench": "optimal_mean_kron", "workload": name, "family": "B1" if family == vg.B1_ASVGP else "SVGP_MARKOV",
           "knots": list(knots), "n": n, "obs_dtype": "float32", **BS.gpu_info(), "solve_rtol": args.rtol,
           "max_iter": args.max_iter, "dm_norm_m0": dm0}
    for pc in args.preconditioner.split(","):
        def solve(max_iter=args.max_iter, rtol=args.rtol):
            plan.grid_forward(theta, zero, L)         # cold start; the B1 system does not depend on theta, Markov's is
            return plan.meanopt_solve(rtol, max_iter, pc)          # at the same theta
        solve(min(args.max_iter, 64))                 # first call: allocation, module load
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        mstar, iters, relres = solve()
        ms = (time.perf_counter() - t0) * 1e3
        dms = plan.step(theta, mstar, L, obs, None)[2].norm().item()
        # rtol = 0: every profiled iteration runs (a converged solve would leave the rest of its batch as empty launches)
        n_prof = min(args.profile_iters, args.max_iter)
        kt = kernel_totals(lambda: solve(n_prof, 0.0), ["k_mo_matvec", "k_mo_kron_sweep"])
        mv_ms, mv_n = kt["k_mo_matvec"]
        sw_ms, sw_n = kt["k_mo_kron_sweep"]
        rec[pc] = {"iters": iters, "relres": relres, "converged": relres <= args.rtol, "solve_ms": ms,
                   "ms_per_iter": ms / max(iters, 1), "dm_norm_mstar_over_m0": dms / dm0,
                   "profiled_iters": n_prof, "matvec_kernel_ms": mv_ms / max(mv_n, 1), "matvec_launches": mv_n,
                   "precond_apply_kernel_ms": sw_ms / max(sw_n // D, 1) if sw_n else None, "sweep_launches": sw_n,
                   "scratch_bytes": plan.workspace_bytes()["scratch"]}
    del plan, obs
    torch.cuda.empty_cache()
    return rec


def workload(vg, gen, name, family, knots, n, dev, args, hbm_gbs):
    D = len(knots)
    meshes = [torch.linspace(0, 1, k) for k in knots]
    xs, y = gen.generate_tracks(0, n, n, dev, torch.float32, seed=0, D=D)
    plan = vg.GridPlan(family, meshes, torch.float32, dev)
    obs = plan.bin(xs, y)
    del xs, y
    theta, m_rand, L = BS.params(knots, dev)
    zero = torch.zeros(plan.M, dtype=torch.float64, device=dev)
    plan.grid_forward(theta, zero, L)
    assemble = lambda: plan.meanopt_assemble(obs)        # noqa: E731
    k1 = lambda: plan.obs_fwd_bwd(obs)                   # noqa: E731
    for _ in range(3):
        assemble()
        k1()
    a_ms, k_ms = [], []
    for _ in range(args.reps):                           # alternated
        a_ms.append(BS.timed(assemble, 1))
        k_ms.append(BS.timed(k1, 1))
    a_ms.sort()
    k_ms.sort()
    kname = "k_obs_b1_binned" if family == vg.B1_ASVGP else "k_obs_svgpm_binned"
    akern, na = kernel_ms(assemble, "assemble", args.reps)
    kkern, nk = kernel_ms(k1, kname, args.reps)
    abytes = (D + 1) * 4 * n
    rec = {"bench": "optimal_mean", "workload": name, "family": "B1" if family == vg.B1_ASVGP else "SVGP_MARKOV",
           "knots": list(knots), "n": n, "obs_dtype": "float32", **BS.gpu_info(), "hbm_copy_gbs": hbm_gbs,
           "assemble_call_ms_median": a_ms[len(a_ms) // 2], "assemble_kernel_ms": akern, "assemble_kernel_launches": na,
           "assemble_bytes": abytes, "assemble_kernel_gbs": abytes / (akern * 1e-3) / 1e9,
           "assemble_kernel_copy_fraction": abytes / (akern * 1e-3) / 1e9 / hbm_gbs,
           "k1_kernel": kname, "k1_call_ms_median": k_ms[len(k_ms) // 2], "k1_kernel_ms": kkern, "k1_kernel_launches": nk,
           "assemble_over_k1_kernel": akern / kkern, "streamed_bytes": obs.streamed_bytes}
    # cold solve from m = 0
    plan.grid_forward(theta, zero, L)
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    assemble()
    mstar, iters, relres = plan.meanopt_solve(args.rtol, args.max_iter)
    torch.cuda.synchronize()
    wall = time.perf_counter() - t0
    t1 = time.perf_counter()
    plan.grid_forward(theta, zero, L)
    plan.meanopt_solve(args.rtol, args.max_iter)
    solve_ms = (time.perf_counter() - t1) * 1e3
    rec.update({"solve_rtol": args.rtol, "solve_iters": iters, "solve_relres": relres, "solve_ms": solve_ms,
                "solve_ms_per_iter": solve_ms / max(iters, 1), "assemble_plus_solve_wall_ms": wall * 1e3,
                "scratch_bytes": plan.workspace_bytes()["scratch"]})
    elbo = lambda m: plan.step(theta, m, L, obs, None)[0][0].item()     # noqa: E731
    rec["elbo_m0"] = elbo(zero)
    rec["elbo_mstar"] = elbo(mstar)
    rec["dm_norm_m0"] = plan.step(theta, zero, L, obs, None)[2].norm().item()
    rec["dm_norm_mstar"] = plan.step(theta, mstar, L, obs, None)[2].norm().item()
    # Adam on m alone for the same wall time
    m = zero.clone().requires_grad_(True)
    opt = torch.optim.Adam([m], lr=args.lr)
    steps = 0
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    while time.perf_counter() - t0 < wall:
        _, _, dm, _ = plan.step(theta, m.detach(), L, obs, None)
        m.grad = -dm
        opt.step()
        steps += 1
        torch.cuda.synchronize()
    rec.update({"adam_lr": args.lr, "adam_steps": steps, "elbo_adam_same_wall": elbo(m.detach())})
    del plan, obs
    torch.cuda.empty_cache()
    return rec


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--n", type=int, default=1 << 26)
    ap.add_argument("--reps", type=int, default=20)
    ap.add_argument("--rtol", type=float, default=1e-8)
    ap.add_argument("--max-iter", type=int, default=100000)
    ap.add_argument("--lr", type=float, default=0.01)
    ap.add_argument("--only", default=None, help="comma-separated workload names")
    ap.add_argument("--out", default=None)
    ap.add_argument("--preconditioner", default=None,
                    help="comma-separated jacobi,kronecker: compare the solves on the same assembled system")
    ap.add_argument("--profile-iters", type=int, default=64, help="iterations of the profiled solve (--preconditioner)")
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("bench_optimal_mean needs a CUDA device")
    vg = importlib.import_module("variational-gridded-gaussian-processes_b200")
    gen = importlib.import_module("variational-gridded-gaussian-processes_b200.utils.dataloaders")
    dev = torch.device("cuda", 0)
    hbm = None if args.preconditioner else copy_rate_gbs(dev)
    wls = [("tracks512_b1", vg.B1_ASVGP, (512, 512)), ("tracks512_markov", vg.SVGP_MARKOV, (512, 512)),
           ("3d_b1", vg.B1_ASVGP, (256, 256, 64)), ("3d_markov", vg.SVGP_MARKOV, (256, 256, 64))]
    for name, fam, knots in wls:
        if args.only and name not in args.only.split(","):
            continue
        if args.preconditioner:
            line = json.dumps(solve_workload(vg, gen, name, fam, knots, args.n, dev, args))
        else:
            line = json.dumps(workload(vg, gen, name, fam, knots, args.n, dev, args, hbm))
        print(line, flush=True)
        if args.out:
            with open(args.out, "a") as f:
                f.write(line + "\n")


if __name__ == "__main__":
    main()
