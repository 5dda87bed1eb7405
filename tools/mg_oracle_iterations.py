"""Iteration counts of the optimal-mean solve on the CPU, from the float64 oracles, to rtol --rtol from m = 0:
  mg       multigrid-preconditioned CG (oracle/optimal_mean_mg.py, Galerkin hierarchy), one count per smoother of --smoothers:
           chebyshev (degree 2, the design's point smoother, lambda_max from 10 power iterations), chebyshev50 (the same
           with 50 power iterations), l1 (two l1-Jacobi sweeps), line (two l1 line-block Jacobi sweeps
           along the finest dimension, the one with the most nodes, full coarsening), line_semi (the same smoother with
           semi-coarsening: the line dimension is not coarsened)
  jacobi   Jacobi-preconditioned CG, the library's solver (scipy's CG with the same stopping rule), with --jacobi-max
  kron     CG preconditioned by the Kronecker product kron_d (F_d + g I) of the per-dimension prior factors F_d (B1: K_d,
           Markov: K_d^-1), g = mean(diag(G) / noise)^(1 / D), applied exactly by dense per-dimension inverses
Data: the track data set of bench.py (torch restatement), theta of tools/bench_svgp_markov.py.  One line per grid and family."""
import argparse
import os
import sys
import time

import numpy as np
import scipy.sparse.linalg as spla
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import bench                                   # noqa: E402
from oracle import optimal_mean_mg as MG       # noqa: E402
from oracle import svgp_markov as SM           # noqa: E402
from oracle import vggp_oracle as O            # noqa: E402


def jacobi_iters(A, rhs, rtol, max_iter):
    n = [0]
    dinv = 1.0 / A.diagonal()
    Mop = spla.LinearOperator(A.shape, matvec=lambda v: dinv * v)
    spla.cg(A, rhs, rtol=rtol, atol=0.0, maxiter=max_iter, M=Mop, callback=lambda _: n.__setitem__(0, n[0] + 1))
    return n[0]


def kron_preconditioner(family, meshes, l, s2, A, prior):
    D = len(meshes)
    knots = [int(t.numel()) for t in meshes]
    if family == O.B1_ASVGP:
        F = [O.kuu_b1(meshes[d], l[d], s2[d], ref_quirks=False).numpy() for d in range(D)]
    else:
        F = [SM.tridiag(*SM.precision_band(meshes[d], l[d], s2[d])[:2]).numpy() for d in range(D)]
    g = float(np.mean((A - prior).diagonal())) ** (1.0 / D)
    inv = [np.linalg.inv(f + g * np.eye(f.shape[0])) for f in F]

    def apply(r):
        t = r.reshape(knots)
        for d in range(D):
            t = np.moveaxis(np.tensordot(inv[d], np.moveaxis(t, d, 0), 1), 0, d)
        return t.reshape(-1)
    return apply


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--grids", default="64x64x16:20,128x128:20", help="comma-separated KNOTSxKNOTS[xKNOTS]:LOG2_N")
    ap.add_argument("--rtol", type=float, default=1e-8)
    ap.add_argument("--max-iter", type=int, default=2000)
    ap.add_argument("--jacobi-max", type=int, default=0, help="also count Jacobi-CG up to this many iterations")
    ap.add_argument("--kron", action="store_true", help="also count CG with the Kronecker preconditioner")
    ap.add_argument("--smoothers", default="chebyshev,chebyshev50,l1,line,line_semi")
    args = ap.parse_args()
    for spec in args.grids.split(","):
        g, logn = spec.split(":")
        knots = tuple(int(k) for k in g.split("x"))
        D, n = len(knots), 1 << int(logn)
        xs, y = bench.make_tracks_torch(0, n, n, torch.device("cpu"), torch.float32, 0, D=D)
        X = torch.stack(xs, 1)
        meshes = [torch.linspace(0, 1, k) for k in knots]
        l = torch.full((D,), 0.3, dtype=torch.float64)
        s2 = torch.full((D,), 0.8, dtype=torch.float64)
        noise = torch.tensor(0.05, dtype=torch.float64)
        for fam, name in ((O.B1_ASVGP, "B1"), (O.SVGP_GRID, "MARKOV")):
            A, rhs, prior = MG.system(fam, meshes, X, y, l, s2, noise)
            line = f"{g} N=2^{logn} {name} rtol={args.rtol:g}"
            line_dim = int(np.argmax(knots))
            for sm in args.smoothers.split(","):
                if sm.startswith("line"):
                    kw = {"kind": "line", "line_dim": line_dim, "semi": sm == "line_semi"}
                elif sm == "chebyshev50":
                    kw = {"kind": "chebyshev", "power_iters": 50}
                else:
                    kw = {"kind": sm}
                t0 = time.perf_counter()
                H = MG.hierarchy(A, knots, **kw)
                _, it, rel = MG.pcg(A, rhs, H, rtol=args.rtol, max_iter=args.max_iter)
                line += (f" | {sm}: levels={len(H)} coarsest={H[-1]['dims']} iters={it} relres={rel:.2e}"
                         f" cpu_s={time.perf_counter() - t0:.1f}")
            if args.jacobi_max:
                line += f" | jacobi_iters={jacobi_iters(A, rhs, args.rtol, args.jacobi_max)}"
            if args.kron:
                apply = kron_preconditioner(fam, meshes, l, s2, A, prior)
                _, itk, relk = MG.pcg(A, rhs, None, rtol=args.rtol, max_iter=args.max_iter,
                                      precondition=apply)
                line += f" | kron_iters={itk} kron_relres={relk:.2e}"
            print(line, flush=True)


if __name__ == "__main__":
    main()
