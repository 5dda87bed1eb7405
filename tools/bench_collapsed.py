"""Benchmark of the collapsed ELBO (vggp_collapsed_terms, vggp_logdet_system; csrc/collapsed.cuh).  Prints one JSON line per
(workload, preconditioner, probe count); also appends them to --out if given.

Workloads: float32 track observations (vggp_generate_tracks), theta of tools/bench_svgp_markov.py: 64 x 64 points with 2^20
observations (where the dense float64 slogdet of A, M = 4096, is the reference) and, with --n (default 2^26), 512 x 512 points
and 256 x 256 x 64 points, each for the B1 family and the Markov SVGP family.  Per workload: the optimal-mean system is
assembled once and solved by Kronecker-preconditioned CG to --cg-rtol (time, iterations, final residual; 3-D Markov is
reported whether it converges or not); the exact terms (time); then for k = 16 / 32 / 64 Rademacher probes and both
preconditioners the SLQ estimate of log det A (time, Lanczos steps, probes converged, standard error of the ELBO relative to
|ELBO|).  --steps-study S1,S2,..: instead, for the 3-D workloads, 16 probes with rtol = 0 (no early stop) and max_steps = S1,
S2, .. for both preconditioners, to see how the estimate moves with the number of Lanczos steps.  Times are host clocks around calls that end in a device synchronisation, median of --reps.  The card's name and
power limit are read in the same run."""
import argparse
import importlib
import json
import math
import os
import sys
import time

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tools"))
import bench_svgp_markov as BS        # noqa: E402  (gpu_info, params)


def elbo_from(terms, logdet_a, theta, D, markov):
    N, yy, bx, tr, ldk = terms
    noise = float(theta[2 * D])
    s2 = float(torch.prod(theta[D:2 * D]))
    ldf = -ldk if markov else ldk
    return (-0.5 * (N * math.log(2 * math.pi) + N * math.log(noise) + logdet_a - ldf + (yy - bx) / noise)
            - (N * s2 - tr) / (2 * noise))


def timed(fn, reps):
    ts, out = [], None
    for _ in range(reps):
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        out = fn()
        torch.cuda.synchronize()
        ts.append((time.perf_counter() - t0) * 1e3)
    ts.sort()
    return out, ts[len(ts) // 2]


def dense_logdet(plan, vg, family, knots, theta, xs, y):
    """float64 slogdet of A formed densely from the features (M <= 4096)"""
    import numpy as np
    sys.path.insert(0, ROOT)
    from oracle import optimal_mean as OM
    from oracle import vggp_oracle as O
    meshes = [torch.linspace(0, 1, k) for k in knots]
    D = len(knots)
    X = torch.stack([x.double().cpu() for x in xs], 1)
    th = theta.cpu()
    fam = O.B1_ASVGP if family == vg.B1_ASVGP else O.SVGP_GRID
    A, _, _ = OM.system(fam, meshes, X, y.double().cpu(), th[:D], th[D:2 * D], th[2 * D])
    return float(np.linalg.slogdet(A.numpy())[1])


def workload(vg, gen, name, family, knots, n, dev, args):
    D = len(knots)
    meshes = [torch.linspace(0, 1, k) for k in knots]
    xs, y = gen.generate_tracks(0, n, n, dev, torch.float32, seed=0, D=D)
    plan = vg.GridPlan(family, meshes, torch.float32, dev)
    obs = plan.bin(xs, y)
    theta, _, L = BS.params(knots, dev)
    markov = family == vg.SVGP_MARKOV
    base = {"bench": "collapsed", "workload": name, "family": "SVGP_MARKOV" if markov else "B1", "knots": list(knots), "n": n,
            "obs_dtype": "float32", **BS.gpu_info()}
    ref = dense_logdet(plan, vg, family, knots, theta, xs, y) if plan.M <= 4096 else None
    del xs, y
    plan.grid_forward(theta, torch.zeros(plan.M, dtype=torch.float64, device=dev), L)
    plan.meanopt_assemble(obs)
    (_, it, rr), cg_ms = timed(lambda: plan.meanopt_solve(args.cg_rtol, args.cg_max_iter, "kronecker"), 1)
    terms, terms_ms = timed(lambda: plan.collapsed_terms(obs).cpu(), args.reps)
    terms = [float(v) for v in terms]
    base.update({"cg_iterations": it, "cg_relres": rr, "cg_ms": cg_ms, "terms_ms": terms_ms, "terms": terms,
                 "dense_logdet_a": ref})
    recs = []
    if args.steps_study:
        for pc in ("kronecker", "jacobi"):
            for ms in (int(v) for v in args.steps_study.split(",")):
                rec = dict(base, preconditioner=pc, n_probes=16, rtol=0.0, max_steps=ms, study="steps")
                plan.logdet_system(16, 0, pc, "rademacher", 8, 0.0)
                ld, t = timed(lambda: plan.logdet_system(16, 0, pc, "rademacher", ms, 0.0), 1)
                rec.update({"slq_ms": t, "ms_per_step": t / ld["steps"], "lanczos_steps": ld["steps"],
                            "logdet_a": ld["logdet"], "logdet_a_stderr": ld["stderr"],
                            "elbo": elbo_from(terms, ld["logdet"], theta.cpu(), D, markov)})
                recs.append(rec)
                print(json.dumps(rec), flush=True)
        del plan, obs
        torch.cuda.empty_cache()
        return recs
    for pc in ("kronecker", "jacobi"):
        for k in (int(v) for v in args.probes.split(",")):
            rec = dict(base, preconditioner=pc, n_probes=k, rtol=args.rtol, max_steps=args.max_steps)
            try:
                plan.logdet_system(k, 0, pc, "rademacher", args.max_steps, args.rtol)      # allocation, module load
                ld, ms = timed(lambda: plan.logdet_system(k, 0, pc, "rademacher", args.max_steps, args.rtol), args.reps)
                ld1 = plan.logdet_system(k, 1, pc, "rademacher", args.max_steps, args.rtol)
            except RuntimeError as e:
                rec["error"] = str(e)
                recs.append(rec)
                continue
            elbo = elbo_from(terms, ld["logdet"], theta.cpu(), D, markov)
            rec.update({"slq_ms": ms, "lanczos_steps": ld["steps"], "probes_converged": ld["converged"],
                        "logdet_a": ld["logdet"], "logdet_a_stderr": ld["stderr"], "logdet_p": ld["logdet_p"],
                        "elbo": elbo, "elbo_stderr_rel": 0.5 * ld["stderr"] / abs(elbo),
                        "seed1_logdet_a": ld1["logdet"], "seed1_stderr": ld1["stderr"],
                        "scratch_bytes": plan.workspace_bytes()["scratch"]})
            if ref is not None:
                rec["dense_err_in_stderr"] = (ld["logdet"] - ref) / ld["stderr"]
            recs.append(rec)
            print(json.dumps(rec), flush=True)
    del plan, obs
    torch.cuda.empty_cache()
    return recs


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--n", type=int, default=1 << 26)
    ap.add_argument("--reps", type=int, default=3)
    ap.add_argument("--rtol", type=float, default=1e-6)
    ap.add_argument("--max-steps", type=int, default=1000)
    ap.add_argument("--probes", default="16,32,64", help="comma-separated probe counts")
    ap.add_argument("--cg-rtol", type=float, default=1e-10)
    ap.add_argument("--cg-max-iter", type=int, default=20000)
    ap.add_argument("--steps-study", default=None, help="comma-separated max_steps values (3-D workloads)")
    ap.add_argument("--only", default=None, help="comma-separated workload names")
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("bench_collapsed needs a CUDA device")
    vg = importlib.import_module("variational-gridded-gaussian-processes_b200")
    gen = importlib.import_module("variational-gridded-gaussian-processes_b200.utils.dataloaders")
    dev = torch.device("cuda", 0)
    wls = [("tracks64_b1", vg.B1_ASVGP, (64, 64), 1 << 20), ("tracks64_markov", vg.SVGP_MARKOV, (64, 64), 1 << 20),
           ("tracks512_b1", vg.B1_ASVGP, (512, 512), args.n), ("tracks512_markov", vg.SVGP_MARKOV, (512, 512), args.n),
           ("3d_b1", vg.B1_ASVGP, (256, 256, 64), args.n), ("3d_markov", vg.SVGP_MARKOV, (256, 256, 64), args.n)]
    for name, fam, knots, n in wls:
        if args.only and name not in args.only.split(","):
            continue
        for rec in workload(vg, gen, name, fam, knots, n, dev, args):
            if args.out:
                with open(args.out, "a") as f:
                    f.write(json.dumps(rec) + "\n")


if __name__ == "__main__":
    main()
