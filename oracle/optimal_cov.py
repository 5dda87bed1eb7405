"""TEST INFRASTRUCTURE / DESIGN VALIDATION -- the optimal Kronecker-factored variational covariance of the B1 and
VGGP_SVGP_MARKOV families (csrc/covopt.cuh) as a float64 torch statement built from dense features.

With theta, m and every S_e, e != d, fixed, the S_d-dependent part of the ELBO (ell_scale s) is
    -(1/2) tr(S_d A_d) + (M / (2 M_d)) log det S_d,   maximised by S_d = (M / M_d) A_d^-1,
    T_d = (s / noise) H_d + c_d F_d,   H_d = W_d diag(prod_{e != d} q_e) W_d^T,   c_d = prod_{e != d} tr(Kuu_e^-1 S_e)
    Markov:  W_d = Psi_d = K_d^-1 k_d(Z, x),  F_d = K_d^-1,  q_e = w_e^T S_e w_e,          A_d = T_d
    B1:      W_d = Phi_d (hat features),      F_d = K_d,     q_e = w_e^T P_e S_e P_e w_e,  A_d = P_d T_d P_d   (P = K^-1)
For D = 1 one update is the reference's S* = Kuu Sigma^-1 Kuu (vggp_oracle.optimal_q).  The second half states the device
construction of the Cholesky factor in numpy: the UL factorisation of T_d, the column recurrences of U^-T and the RQ sweep."""
import math
from typing import Sequence

import numpy as np
import torch

from . import svgp_markov as SM
from . import vggp_oracle as O


def features(family: int, mesh: torch.Tensor, x: torch.Tensor, l) -> torch.Tensor:
    """(M_d, N) float64 weights of one dimension: B1 hat features, or the two Markov weights of the extended cell."""
    xx = x.to(torch.float64)
    if family == O.B1_ASVGP:
        return O.b1_features_dense(mesh, xx)
    M, N = mesh.numel(), xx.numel()
    e, wlo, whi = SM.cell_weights(mesh, xx, l)
    W = torch.zeros(M, N, dtype=torch.float64)
    cols = torch.arange(N)
    for node, w in ((e - 1, wlo), (e, whi)):
        ok = (node >= 0) & (node < M)
        W.index_put_((node[ok], cols[ok]), w[ok], accumulate=True)
    return W


def prior(family: int, mesh, l, s2):
    """(K_d, F_d): the per-dimension prior covariance factor and the tridiagonal factor of T_d."""
    if family == O.B1_ASVGP:
        K = O.kuu_b1(mesh, l, s2, ref_quirks=False).to(torch.float64)
        return K, K
    dg, of, _ = SM.precision_band(mesh, l, s2)
    F = SM.tridiag(dg, of)
    return torch.linalg.inv(F), F


def system(family: int, meshes: Sequence[torch.Tensor], X, l, s2, noise, Ls, d: int, scale: float = 1.0):
    """T_d, K_d and the constant M / M_d of the update of dimension d."""
    D = len(meshes)
    N = X.shape[0]
    Xc = X.reshape(N, D)
    Ms = [int(t.numel()) for t in meshes]
    Ws = [features(family, meshes[e], Xc[:, e], l[e]) for e in range(D)]
    pri = [prior(family, meshes[e], l[e], s2[e]) for e in range(D)]
    prod_q = torch.ones(N, dtype=torch.float64)
    c = torch.ones((), dtype=torch.float64)
    for e in range(D):
        if e == d:
            continue
        Lt = torch.tril(Ls[e].to(torch.float64))
        S = Lt @ Lt.T
        Ke = pri[e][0]
        Pe = torch.linalg.inv(Ke)
        Q = Pe @ S @ Pe if family == O.B1_ASVGP else S
        prod_q = prod_q * (Ws[e] * (Q @ Ws[e])).sum(0)
        c = c * torch.trace(Pe @ S)
    H = (Ws[d] * prod_q) @ Ws[d].T
    Kd, Fd = pri[d]
    T = (scale / noise) * H + c * Fd
    return T, Kd, math.prod(Ms) / Ms[d]


def update(family: int, meshes, X, l, s2, noise, Ls, d: int, scale: float = 1.0) -> torch.Tensor:
    """Cholesky factor of the optimal S_d given the other factors."""
    T, Kd, r = system(family, meshes, X, l, s2, noise, Ls, d, scale)
    Tinv = torch.linalg.inv(T)
    S = r * (Kd @ Tinv @ Kd if family == O.B1_ASVGP else Tinv)
    return torch.linalg.cholesky(0.5 * (S + S.T))


def elbo(family: int, meshes, X, y, l, s2, noise, m, Ls, scale: float = 1.0) -> torch.Tensor:
    """The library's uncollapsed bound of the family (float64)."""
    if family == O.B1_ASVGP:
        return O.elbo_structured(O.B1_ASVGP, meshes, X, y, l, s2, noise, m, Ls, ref_quirks=False, scale=scale)
    return SM.elbo(meshes, X, y, l, s2, noise, m, Ls, scale)


def grad_L(family: int, meshes, X, y, l, s2, noise, m, Ls, d: int, scale: float = 1.0) -> torch.Tensor:
    """d ELBO / d tril(L_d) by autograd."""
    Ls = [L.detach().clone().requires_grad_(e == d) for e, L in enumerate(Ls)]
    val = elbo(family, meshes, X, y, l, s2, noise, m, Ls, scale)
    return torch.tril(torch.autograd.grad(val, Ls[d])[0])


def change(L_new, L_old) -> float:
    """||L_new / ||L_new|| - L_old / ||L_old|| ||_F of the lower triangles."""
    a, b = torch.tril(L_new), torch.tril(L_old)
    return float((a / a.norm() - b / b.norm()).norm())


# ---- the device construction, in numpy ------------------------------------------------------------------------
def ul_factor(td: np.ndarray, to: np.ndarray):
    """T = U U^T for a tridiagonal T (diag td, super-diagonal to): U upper bidiagonal with diagonal b and U[k-1][k] = e[k]
    (e[0] = 0), by the backward recurrence b_k^2 = T[k][k] - e_{k+1}^2, e_k = T[k-1][k] / b_k.  None if a pivot fails."""
    n = td.size
    b, e = np.zeros(n), np.zeros(n)
    ek = 0.0
    for k in range(n - 1, -1, -1):
        piv = td[k] - ek * ek
        if not (piv > 0.0 and np.isfinite(piv)):
            return None
        b[k] = math.sqrt(piv)
        ek = to[k - 1] / b[k] if k > 0 else 0.0
        e[k] = ek
    return b, e


def uinv_t(b: np.ndarray, e: np.ndarray) -> np.ndarray:
    """U^-T column by column: y_j = 1 / b_j, y_k = -(e_k / b_k) y_{k-1}."""
    n = b.size
    Y = np.zeros((n, n))
    for j in range(n):
        y = 1.0 / b[j]
        Y[j, j] = y
        for k in range(j + 1, n):
            y *= -e[k] / b[k]
            Y[k, j] = y
    return Y


def rq_lower(X: np.ndarray) -> np.ndarray:
    """Lower-triangular L with L L^T = X X^T for a lower Hessenberg X: Givens rotation k mixes columns k and k + 1 and
    zeroes X[k][k+1], k = 0..n-2; the last column's sign is made positive."""
    A = X.copy()
    n = A.shape[0]
    for k in range(n - 1):
        a, bb = A[k, k], A[k, k + 1]
        rho = math.hypot(a, bb)
        c, s = (a / rho, bb / rho) if rho > 0 else (1.0, 0.0)
        ck, ck1 = A[:, k].copy(), A[:, k + 1].copy()
        A[:, k] = c * ck + s * ck1
        A[:, k + 1] = c * ck1 - s * ck
    A[:, n - 1] *= np.sign(A[n - 1, n - 1]) or 1.0
    return np.tril(A)


def device_factor(family: int, T: np.ndarray, K: np.ndarray, r: float) -> np.ndarray:
    """The Cholesky factor of S_d the way csrc/covopt.cuh builds it from T_d (tridiagonal), K_d and r = M / M_d."""
    b, e = ul_factor(np.diag(T).copy(), np.append(np.diag(T, 1), 0.0))
    Y = math.sqrt(r) * uinv_t(b, e)
    if family != O.B1_ASVGP:
        return Y
    return rq_lower(K @ Y)
