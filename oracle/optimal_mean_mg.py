"""TEST INFRASTRUCTURE / DESIGN VALIDATION -- a geometric multigrid preconditioner for the optimal-mean solve
(csrc/meanopt.cuh), stated in float64 numpy / scipy on the sparse form of the stencil system of oracle.optimal_mean
(A = prior + W W^T / noise, a 3^D-point stencil on the node grid), with the preconditioned CG of the library's solve.
It measures the design before any device code exists: DESIGN.md section 4 (K1m, multigrid) records its iteration counts.

Hierarchy: level 0 is the node grid.  A dimension with n > 3 nodes keeps its even indices and its last index (n // 2 + 1
nodes), one with n <= 3 is not coarsened, and neither is the dimension `keep` (semi-coarsening, for line smoothing);
coarsening stops at <= `coarsest` nodes or when no dimension can be coarsened.  P = kron_d P_d with P_d the index-space
linear interpolation (1/2, 1, 1/2) between kept nodes (identity for a dimension that is not coarsened), R = P^T,
A_{l+1} = P^T A_l P.  The same smoother runs before and after the coarse correction (the pre-smoothing starts from zero), so
the V-cycle is a symmetric positive definite operator:
  chebyshev  Chebyshev polynomial of degree 2 in D^-1 A over [lambda_max / 30, 1.1 lambda_max], lambda_max of D^-1 A from
             10 power iterations from a fixed start vector (the smoother the design specifies)
  l1         two sweeps of l1-Jacobi, x += (r - A x) / sum_j |a_ij|
  line       two sweeps of l1 line-block Jacobi along dimension `line_dim`: the couplings within a line of that dimension are
             solved exactly, the absolute couplings to other lines are added to the diagonal
Coarsest level: exact dense solve."""
import math
from typing import Sequence

import numpy as np
import scipy.sparse as sp
import scipy.sparse.linalg as spla
import torch

from . import svgp_markov as SM
from . import vggp_oracle as O

COARSEST = 512


def _weights(family, meshes, X, l):
    """per dimension (first node, w_lo, w_hi) of every observation: weights of nodes c and c + 1 (B1 outside the mesh:
    c = -1 and both weights 0; Markov: c = -1 or c = M - 1 in the virtual cells, where the missing node is dropped)"""
    out = []
    for d, mesh in enumerate(meshes):
        if family == O.B1_ASVGP:
            c, wlo, whi = O.b1_stencil(mesh, X[:, d])
            out.append((c, wlo.to(torch.float64), whi.to(torch.float64)))
        else:
            e, wlo, whi = SM.cell_weights(mesh, X[:, d], l[d])
            out.append((e - 1, wlo, whi))
    return out


def system(family: int, meshes: Sequence[torch.Tensor], X: torch.Tensor, y: torch.Tensor, l, s2, noise):
    """(A, rhs, prior) of oracle.optimal_mean.system as scipy CSR matrices and a numpy vector (any grid size)."""
    D = len(meshes)
    N = y.numel()
    Ms = [int(t.numel()) for t in meshes]
    strides = [math.prod(Ms[d + 1:]) for d in range(D)]
    M = math.prod(Ms)
    X = X.reshape(N, D).to(torch.float64)
    if family == O.B1_ASVGP:
        bands = [O.kuu_b1(meshes[d], l[d], s2[d], ref_quirks=False).to(torch.float64).numpy() for d in range(D)]
        facs = [sp.csr_matrix(b) for b in bands]
    elif family == O.SVGP_GRID:
        facs = []
        for d in range(D):
            dg, of, _ = SM.precision_band(meshes[d], l[d], s2[d])
            facs.append(sp.diags([of.numpy(), dg.numpy(), of.numpy()], [-1, 0, 1], format="csr"))
    else:
        raise ValueError("the stencil system exists for the B1 family and the Markov form of SVGP_GRID")
    cells = _weights(family, meshes, X, l)
    rows, cols, vals = [], [], []
    ar = np.arange(N)
    for corner in range(2 ** D):
        w = torch.ones(N, dtype=torch.float64)
        idx = torch.zeros(N, dtype=torch.long)
        ok = torch.ones(N, dtype=torch.bool)
        for d in range(D):
            c, wlo, whi = cells[d]
            bit = (corner >> (D - 1 - d)) & 1
            node = c + bit
            ok = ok & (node >= 0) & (node < Ms[d])
            w = w * (whi if bit else wlo)
            idx = idx + node.clamp(0, Ms[d] - 1) * strides[d]
        okn = ok.numpy()
        rows.append(idx.numpy()[okn])
        cols.append(ar[okn])
        vals.append(w.numpy()[okn])
    W = sp.csr_matrix((np.concatenate(vals), (np.concatenate(rows), np.concatenate(cols))), shape=(M, N))
    prior = facs[0]
    for f in facs[1:]:
        prior = sp.kron(prior, f, format="csr")
    nz = float(noise)
    A = (prior + (W @ W.T) / nz).tocsr()
    rhs = W @ y.reshape(-1).to(torch.float64).numpy() / nz
    return A, rhs, prior


def coarse_n(n: int) -> int:
    return n // 2 + 1 if n > 3 else n


def level_dims(dims: Sequence[int], coarsest: int = COARSEST, keep=None):
    """dimensions of every level; dimension `keep` (if given) is never coarsened"""
    def nxt(t):
        return tuple(n if d == keep else coarse_n(n) for d, n in enumerate(t))
    out = [tuple(int(n) for n in dims)]
    while math.prod(out[-1]) > coarsest and nxt(out[-1]) != out[-1]:
        out.append(nxt(out[-1]))
    return out


def interp(n: int, nc=None):
    """P_d (n x coarse_n(n)): kept fine node f = min(2 c, n - 1) takes coarse c; a dropped (odd) node averages its neighbours.
    The identity when the dimension is not coarsened (nc == n)."""
    nc = coarse_n(n) if nc is None else nc
    if nc == n:
        return sp.identity(n, format="csr")
    r, c, v = [], [], []
    for i in range(n):
        if i % 2 == 0 or i == n - 1:
            r.append(i); c.append(min(i // 2, nc - 1) if i != n - 1 else nc - 1); v.append(1.0)
        else:
            r += [i, i]; c += [(i - 1) // 2, (i + 1) // 2]; v += [0.5, 0.5]
    return sp.csr_matrix((v, (r, c)), shape=(n, nc))


def prolongation(dims, coarse_dims):
    P = interp(dims[0], coarse_dims[0])
    for n, nc in zip(dims[1:], coarse_dims[1:]):
        P = sp.kron(P, interp(n, nc), format="csr")
    return P


def lambda_max(A, dinv, iters=10):
    """power-iteration estimate of the largest eigenvalue of D^-1 A from the fixed start vector 1 + sin(i)"""
    v = 1.0 + np.sin(np.arange(A.shape[0], dtype=np.float64))
    lam = 0.0
    for _ in range(iters):
        v = v / np.linalg.norm(v)
        w = dinv * (A @ v)
        lam = float(np.linalg.norm(w))
        v = w
    return lam


def smoother(A, dims, kind="chebyshev", line_dim=None, power_iters=10):
    """s(r, x): the smoothing step of one level for A x = r, started from x"""
    if kind == "l1":
        dl1 = 1.0 / np.asarray(abs(A).sum(axis=1)).ravel()

        def s(r, x):
            for _ in range(2):
                x = x + dl1 * (r - A @ x)
            return x
        return s
    if kind == "chebyshev":
        dinv = 1.0 / A.diagonal()
        lmax = 1.1 * lambda_max(A, dinv, power_iters)
        lmin = lmax / (1.1 * 30.0)
        theta, delta = 0.5 * (lmax + lmin), 0.5 * (lmax - lmin)
        sigma = theta / delta
        rho1 = 1.0 / (2.0 * sigma - 1.0 / sigma)

        def s(r, x):
            d = dinv * (r - A @ x) / theta
            x = x + d
            d = rho1 / sigma * d + 2.0 * rho1 / delta * dinv * (r - A @ x)
            return x + d
        return s
    if kind == "line":
        A = A.tocoo()
        ci = np.unravel_index(A.row, dims)
        cj = np.unravel_index(A.col, dims)
        same = np.ones(A.nnz, dtype=bool)
        for d in range(len(dims)):
            if d != line_dim:
                same &= ci[d] == cj[d]
        off = np.bincount(A.row[~same], weights=np.abs(A.data[~same]), minlength=A.shape[0]).astype(np.float64)
        B = sp.csc_matrix((A.data[same], (A.row[same], A.col[same])), shape=A.shape) + sp.diags(off)
        lu = spla.splu(B.tocsc())
        A = A.tocsr()

        def s(r, x):
            for _ in range(2):
                x = x + lu.solve(r - A @ x)
            return x
        return s
    raise ValueError(f"unknown smoother {kind!r}")


def hierarchy(A, dims, coarsest: int = COARSEST, kind: str = "chebyshev", line_dim=None, semi: bool = False,
              power_iters: int = 10):
    """levels [{A, dims, smooth, P (to the next level)}], the last one with the dense inverse `inv`.  `semi`: do not coarsen
    `line_dim` (semi-coarsening across the lines of the line smoother).  `power_iters`: of the Chebyshev lambda_max estimate;
    when it falls short of lambda_max / 1.1 the smoother amplifies the top of the spectrum and PCG slows down."""
    H = []
    lv = level_dims(dims, coarsest, keep=line_dim if semi else None)
    for k, dd in enumerate(lv):
        A = A.tocsr()
        ent = {"A": A, "dims": dd}
        if k + 1 < len(lv):
            ent["smooth"] = smoother(A, dd, kind, line_dim, power_iters)
            ent["P"] = prolongation(dd, lv[k + 1])
            H.append(ent)
            A = ent["P"].T @ A @ ent["P"]
        else:
            ent["inv"] = np.linalg.inv(A.toarray())
            H.append(ent)
    return H


def vcycle(H, r, k=0):
    lev = H[k]
    if "inv" in lev:
        return lev["inv"] @ r
    A, s, P = lev["A"], lev["smooth"], lev["P"]
    x = s(r, np.zeros_like(r))
    x = x + P @ vcycle(H, P.T @ (r - A @ x), k + 1)
    return s(r, x)


def pcg(A, rhs, H, x0=None, rtol=1e-8, max_iter=1000, precondition=None):
    """(x, iterations, ||r|| / ||rhs||) of CG preconditioned by the V-cycle of H (or by `precondition`, z = precondition(r));
    the stopping rule of the library's solve, ||r|| <= rtol ||rhs||"""
    if precondition is None:
        precondition = lambda v: vcycle(H, v)       # noqa: E731
    x = np.zeros_like(rhs) if x0 is None else np.array(x0, dtype=np.float64)
    bn = np.linalg.norm(rhs)
    if bn == 0.0:
        return np.zeros_like(rhs), 0, 0.0
    r = rhs - A @ x
    rel = np.linalg.norm(r) / bn
    it = 0
    if rel <= rtol:
        return x, 0, rel
    z = precondition(r)
    p = z.copy()
    rz = r @ z
    while it < max_iter:
        q = A @ p
        a = rz / (p @ q)
        x += a * p
        r -= a * q
        it += 1
        rel = np.linalg.norm(r) / bn
        if rel <= rtol:
            break
        z = precondition(r)
        rz, rz_old = r @ z, rz
        p = z + (rz / rz_old) * p
    return x, it, rel


def optimal_mean(family, meshes, X, y, l, s2, noise, rtol=1e-12, max_iter=1000, coarsest: int = COARSEST, **kw):
    """(m*, iterations) by multigrid-preconditioned CG from m = 0 (`kw`: smoother options of hierarchy())"""
    A, rhs, prior = system(family, meshes, X, y, l, s2, noise)
    H = hierarchy(A, [int(t.numel()) for t in meshes], coarsest, **kw)
    x, it, _ = pcg(A, rhs, H, rtol=rtol, max_iter=max_iter)
    return (prior @ x if family == O.B1_ASVGP else x), it
