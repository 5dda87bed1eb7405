"""TEST INFRASTRUCTURE / DESIGN VALIDATION -- the optimal variational mean of the B1 and VGGP_SVGP_MARKOV families as the dense
linear systems the library solves (csrc/meanopt.cuh), in float64 torch.  The m-dependent part of the ELBO,
-(1 / 2 noise) ||y - mu(m)||^2 - (1 / 2) m^T Kuu^-1 m, does not depend on S, so its maximiser m* solves
    B1:      (Kuu + Phi Phi^T / noise) alpha = Phi y / noise,   m* = Kuu alpha*      (mu = Phi^T alpha, alpha = Kuu^-1 m)
    Markov:  (Kuu^-1 + Psi Psi^T / noise) m = Psi y / noise                          (mu = Psi^T m, Psi = Kuu^-1 Kuf)
which is the mean of the reference's q_u(), m* = Kuu Sigma^-1 Kuf y / noise (vggp_oracle.optimal_q)."""
import math
from typing import Sequence

import torch

from . import svgp_markov as SM
from . import vggp_oracle as O


def system(family: int, meshes: Sequence[torch.Tensor], X: torch.Tensor, y: torch.Tensor, l, s2, noise):
    """(A, rhs, prior) of the stencil system: A = prior + W W^T / noise, rhs = W y / noise, with W = Phi and prior = Kuu for B1,
    W = Psi and prior = Kuu^-1 for the Markov form (family SVGP_GRID of the oracle: the same model)."""
    D = len(meshes)
    N = y.numel()
    Xc = X.reshape(N, D).to(torch.float64)
    yy = y.reshape(-1).to(torch.float64)
    if family == O.B1_ASVGP:
        Kuu, Phi, _, _ = O.dense_Kuu_Kuf(O.B1_ASVGP, meshes, Xc, l, s2, ref_quirks=False)
        prior, W = Kuu, Phi
    elif family == O.SVGP_GRID:
        Ms = [int(t.numel()) for t in meshes]
        strides = [math.prod(Ms[d + 1:]) for d in range(D)]
        W = torch.zeros(math.prod(Ms), N, dtype=torch.float64)
        cells = [SM.cell_weights(meshes[d], Xc[:, d], l[d]) for d in range(D)]
        cols = torch.arange(N)
        for corner in range(2 ** D):
            w = torch.ones(N, dtype=torch.float64)
            idx = torch.zeros(N, dtype=torch.long)
            ok = torch.ones(N, dtype=torch.bool)
            for d in range(D):
                e, wlo, whi = cells[d]
                bit = (corner >> (D - 1 - d)) & 1
                node = e - 1 + bit
                ok = ok & (node >= 0) & (node < Ms[d])
                w = w * (whi if bit else wlo)
                idx = idx + node.clamp(0, Ms[d] - 1) * strides[d]
            W.index_put_((idx[ok], cols[ok]), w[ok], accumulate=True)
        P = torch.ones(1, 1, dtype=torch.float64)
        for d in range(D):
            dg, of, _ = SM.precision_band(meshes[d], l[d], s2[d])
            P = torch.kron(P, SM.tridiag(dg, of))
        prior = P
    else:
        raise ValueError("the stencil system exists for the B1 family and the Markov form of SVGP_GRID")
    A = prior + (W @ W.T) / noise
    rhs = (W @ yy) / noise
    return A, rhs, prior


def optimal_mean(family: int, meshes, X, y, l, s2, noise) -> torch.Tensor:
    """m* of the stencil system (dense Cholesky solve)."""
    A, rhs, prior = system(family, meshes, X, y, l, s2, noise)
    sol = torch.cholesky_solve(rhs.unsqueeze(-1), torch.linalg.cholesky(A)).squeeze(-1)
    return prior @ sol if family == O.B1_ASVGP else sol
