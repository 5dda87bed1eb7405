"""TEST INFRASTRUCTURE / DESIGN VALIDATION -- the O(1)-per-observation ("Markov") form of the product-grid SVGP family
(kronecker_structure.py:287-338, Matern12SVGP), stated in float64 torch with gradients by autograd.  It is the reference of
the VGGP_SVGP_MARKOV kernels (csrc/svgpm.cuh) and is itself checked against the dense SVGP statement of vggp_oracle
(elbo_structured with family SVGP_GRID), which is pinned to the reference's own class through tests/golden.

With a Matern-1/2 kernel, K_d = s2_d exp(-|z_i - z_j| / l_d) on sorted points z is the covariance of an Ornstein-Uhlenbeck
process, so, with rho_i = exp(-h_i / l), h_i = z_{i+1} - z_i, u_i = 1 / (1 - rho_i^2):
    K_d^-1 = tridiag / s2:  diag u_0, u_{i-1} + u_i - 1, u_{M-2};  off -rho_i u_i
    log det K_d = M_d log s2_d - sum_i log u_i
    psi_d(x) = K_d^-1 k_d(Z, x) has two non-zeros: for x in [z_c, z_{c+1}], a = (z_{c+1} - x) / l, b = (x - z_c) / l,
        wlo = sinh(a) / sinh(h_c / l) at c,   whi = sinh(b) / sinh(h_c / l) at c + 1;
    left of z_0 only exp(-(z_0 - x) / l) at 0, right of z_{M-1} only exp(-(x - z_{M-1}) / l) at M - 1.
The extended cell of x is e = #{knots < x} in 0..M_d (e = 0 and e = M_d are the virtual cells outside the points); its two
slots are the nodes e - 1 and e.  Per observation
    mu = sum_corners prod_d w_d m[corner],   var = prod s2_d - prod_d w_d^T K_d[e] w_d + prod_d w_d^T S_d[e] w_d
with K_d[e], S_d[e] the 2 x 2 diagonal blocks of K_d and S_d = tril(L_d) tril(L_d)^T.  O(N 2^D) per step."""
import math
from typing import Sequence

import torch


def cell_weights(z: torch.Tensor, x: torch.Tensor, l: torch.Tensor):
    """Extended cell e (0..M) of every x and the weights (wlo at node e - 1, whi at node e); the weight of a node that does
    not exist is zero.  Stable for any h / l: sinh ratios written with expm1."""
    zz = z.to(torch.float64)
    M = zz.numel()
    xx = x.to(torch.float64).contiguous()
    e = torch.searchsorted(zz, xx, right=False)                      # number of knots < x
    left, right = e == 0, e == M
    t0 = zz[(e - 1).clamp(0, M - 1)]
    t1 = zz[e.clamp(0, M - 1)]
    a = ((t1 - xx) / l).clamp(min=0)
    b = ((xx - t0) / l).clamp(min=0)
    eta = torch.where(left | right, torch.ones((), dtype=torch.float64), (t1 - t0) / l)
    den = -torch.expm1(-2 * eta)
    wlo = torch.exp(-b) * (-torch.expm1(-2 * a)) / den
    whi = torch.exp(-a) * (-torch.expm1(-2 * b)) / den
    zero = torch.zeros((), dtype=torch.float64)
    wlo = torch.where(left, zero, torch.where(right, torch.exp(-b), wlo))
    whi = torch.where(right, zero, torch.where(left, torch.exp(-a), whi))
    return e, wlo, whi


def precision_band(z: torch.Tensor, l: torch.Tensor, s2: torch.Tensor):
    """(diag, off) of K_d^-1 (M and M - 1 values) and log det K_d, closed form."""
    zz = z.to(torch.float64)
    h = zz[1:] - zz[:-1]
    rho = torch.exp(-h / l)
    u = -1.0 / torch.expm1(-2 * h / l)                                 # 1 / (1 - rho^2)
    diag = torch.cat([u[:1], u[:-1] + u[1:] - 1, u[-1:]]) / s2
    off = -rho * u / s2
    logdet = zz.numel() * torch.log(s2) - torch.log(u).sum()
    return diag, off, logdet


def tridiag(diag: torch.Tensor, off: torch.Tensor) -> torch.Tensor:
    return torch.diag(diag) + torch.diag(off, 1) + torch.diag(off, -1)


def mode_product(T: torch.Tensor, A: torch.Tensor, d: int) -> torch.Tensor:
    return torch.movedim(torch.tensordot(A, T, dims=([1], [d])), 0, d)


def elbo(meshes: Sequence[torch.Tensor], X, y, l, s2, noise, m, Ls: Sequence[torch.Tensor], scale: float = 1.0):
    """ELBO of the uncollapsed bound, q(u) = N(m, kron_d L_d L_d^T), in the Markov form.  Same arguments and value as
    vggp_oracle.elbo_structured(SVGP_GRID, ...)."""
    D = len(meshes)
    N = y.numel()
    Xc = X.reshape(N, D).to(torch.float64)
    Ms = [int(t.numel()) for t in meshes]
    M = math.prod(Ms)
    strides = [math.prod(Ms[d + 1:]) for d in range(D)]
    Lt = [torch.tril(L) for L in Ls]
    Ss = [L @ L.T for L in Lt]
    mu = torch.zeros(N, dtype=torch.float64)
    p = torch.ones(N, dtype=torch.float64)
    q = torch.ones(N, dtype=torch.float64)
    cells = []
    for d in range(D):
        e, wlo, whi = cell_weights(meshes[d], Xc[:, d], l[d])
        cells.append((e, wlo, whi))
        zz = meshes[d].to(torch.float64)
        lo, hi = (e - 1).clamp(0, Ms[d] - 1), e.clamp(0, Ms[d] - 1)
        kx = s2[d] * torch.exp(-(zz[hi] - zz[lo]) / l[d])
        p = p * (s2[d] * (wlo * wlo + whi * whi) + 2 * kx * wlo * whi)
        S = Ss[d]
        q = q * (S[lo, lo] * wlo * wlo + 2 * S[lo, hi] * wlo * whi + S[hi, hi] * whi * whi)
    mf = m.reshape(-1)
    for corner in range(2 ** D):
        w = torch.ones(N, dtype=torch.float64)
        idx = torch.zeros(N, dtype=torch.long)
        for d in range(D):
            e, wlo, whi = cells[d]
            bit = (corner >> (D - 1 - d)) & 1
            w = w * (whi if bit else wlo)
            idx = idx + (e - 1 + bit).clamp(0, Ms[d] - 1) * strides[d]
        mu = mu + w * mf[idx]
    var = torch.prod(s2) - p + q
    ell = (-0.5 * torch.log(2 * math.pi * noise) - ((y.to(torch.float64) - mu) ** 2 + var) / (2 * noise)).sum()
    tr = torch.ones((), dtype=torch.float64)
    lds = torch.zeros((), dtype=torch.float64)
    Km = m.reshape(Ms)
    for d in range(D):
        dg, of, ldk = precision_band(meshes[d], l[d], s2[d])
        tr = tr * ((dg * torch.diagonal(Ss[d])).sum() + 2 * (of * torch.diagonal(Ss[d], 1)).sum())
        lds = lds + (M / Ms[d]) * (ldk - 2 * torch.log(torch.diagonal(Lt[d]).abs()).sum())
        Km = mode_product(Km, tridiag(dg, of), d)
    kl = 0.5 * (tr + (m.reshape(-1) * Km.reshape(-1)).sum() - M + lds)
    return scale * ell - kl


def value_and_grads(meshes, X, y, l, s2, noise, m, Ls, scale: float = 1.0):
    """ELBO and its gradients (l, s2, noise, m, L_1..L_D) by autograd."""
    l = l.detach().clone().requires_grad_(True)
    s2 = s2.detach().clone().requires_grad_(True)
    noise = noise.detach().clone().requires_grad_(True)
    m = m.detach().clone().requires_grad_(True)
    Ls = [L.detach().clone().requires_grad_(True) for L in Ls]
    val = elbo(meshes, X, y, l, s2, noise, m, Ls, scale)
    grads = torch.autograd.grad(val, [l, s2, noise, m] + Ls)
    return val.detach(), grads


def predict(meshes, x, l, s2, m, Ls):
    """Marginal mean and variance of q(f(x*)) in the Markov form."""
    D = len(meshes)
    xx = x.reshape(x.shape[0], D).to(torch.float64)
    Ms = [int(t.numel()) for t in meshes]
    strides = [math.prod(Ms[d + 1:]) for d in range(D)]
    n = xx.shape[0]
    mu = torch.zeros(n, dtype=torch.float64)
    p = torch.ones(n, dtype=torch.float64)
    q = torch.ones(n, dtype=torch.float64)
    cells = []
    for d in range(D):
        e, wlo, whi = cell_weights(meshes[d], xx[:, d], l[d])
        cells.append((e, wlo, whi))
        zz = meshes[d].to(torch.float64)
        lo, hi = (e - 1).clamp(0, Ms[d] - 1), e.clamp(0, Ms[d] - 1)
        kx = s2[d] * torch.exp(-(zz[hi] - zz[lo]) / l[d])
        p = p * (s2[d] * (wlo * wlo + whi * whi) + 2 * kx * wlo * whi)
        Lt = torch.tril(Ls[d])
        S = Lt @ Lt.T
        q = q * (S[lo, lo] * wlo * wlo + 2 * S[lo, hi] * wlo * whi + S[hi, hi] * whi * whi)
    for corner in range(2 ** D):
        w = torch.ones(n, dtype=torch.float64)
        idx = torch.zeros(n, dtype=torch.long)
        for d in range(D):
            e, wlo, whi = cells[d]
            bit = (corner >> (D - 1 - d)) & 1
            w = w * (whi if bit else wlo)
            idx = idx + (e - 1 + bit).clamp(0, Ms[d] - 1) * strides[d]
        mu = mu + w * m.reshape(-1)[idx]
    return mu, torch.prod(s2) - p + q
