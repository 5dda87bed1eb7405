"""TEST INFRASTRUCTURE / DESIGN VALIDATION -- the Kronecker preconditioner of the optimal-mean solve (vggp_meanopt_solve_pc
with VGGP_MEANOPT_KRONECKER, csrc/meanopt.cuh) in the form the device computes it, float64 numpy:

    z = kron_d (F_d + g I)^-1 r,    g = (trace(G) / (noise M))^(1 / D) = mean(diag(A - prior))^(1 / D)

with F_d the tridiagonal prior factor of dimension d (B1: K_d; Markov: K_d^-1).  Per dimension the Thomas factors
[l | 1 / d' | off] of F_d + g I, then one forward and one backward recurrence along every fibre of each mode of the
row-major (M_1, ..., M_D) tensor:
    forward   y_i = x_i - l_i y_{i-1}                (l_0 = 0)
    backward  z_i = (y_i - off_i z_{i+1}) / d'_i     (off_{n-1} = 0)
The dense version (explicit inverses, tools/mg_oracle_iterations.py) is its cross-check in tests/test_optimal_mean_kron.py."""
import math

import numpy as np
import torch

from oracle import svgp_markov as SM
from oracle import vggp_oracle as O


def prior_bands(family, meshes, l, s2):
    """(diag, off) of F_d per dimension, float64 numpy (off has n - 1 values)"""
    out = []
    for d, mesh in enumerate(meshes):
        if family == O.B1_ASVGP:
            K = O.kuu_b1(mesh, l[d], s2[d], ref_quirks=False).to(torch.float64).numpy()
            out.append((np.diag(K).copy(), np.diag(K, 1).copy()))
        else:
            dg, of, _ = SM.precision_band(mesh, l[d], s2[d])
            out.append((dg.numpy().copy(), of.numpy().copy()))
    return out


def shift(A, prior, D):
    """g = mean(diag(G) / noise)^(1 / D) from the system matrix and its prior part (dense or scipy sparse)"""
    dg = np.asarray(A.diagonal()) - np.asarray(prior.diagonal())
    return float(np.mean(dg)) ** (1.0 / D)


def thomas(bd, bo, g):
    """[l, 1 / d', off] (n each) of the LU factorisation of tridiag(bo, bd + g, bo), as k_mo_kron_factors"""
    n = bd.size
    l, invd, off = np.zeros(n), np.zeros(n), np.zeros(n)
    off[:n - 1] = bo[:n - 1]
    invd[0] = 1.0 / (bd[0] + g)
    for i in range(1, n):
        l[i] = bo[i - 1] * invd[i - 1]
        invd[i] = 1.0 / (bd[i] + g - l[i] * bo[i - 1])
    return l, invd, off


def factors(family, meshes, l, s2, g):
    return [thomas(bd, bo, g) for bd, bo in prior_bands(family, meshes, l, s2)]


def sweep(t, fac, d):
    """tridiagonal solve along mode d of the tensor t (all fibres at once)"""
    l, invd, off = fac
    x = np.moveaxis(t, d, -1).copy()
    n = x.shape[-1]
    for i in range(1, n):
        x[..., i] -= l[i] * x[..., i - 1]
    x[..., n - 1] *= invd[n - 1]
    for i in range(n - 2, -1, -1):
        x[..., i] = (x[..., i] - off[i] * x[..., i + 1]) * invd[i]
    return np.moveaxis(x, -1, d)


def apply(facs, knots, r):
    """z = kron_d (F_d + g I)^-1 r, one sweep per mode in the order of the device (0, ..., D - 1)"""
    t = np.asarray(r, dtype=np.float64).reshape(knots)
    for d in range(len(knots)):
        t = sweep(t, facs[d], d)
    return t.reshape(-1)


def dense(family, meshes, l, s2, g):
    """kron_d (F_d + g I)^-1 formed densely (small grids only)"""
    out = np.ones((1, 1))
    for bd, bo in prior_bands(family, meshes, l, s2):
        F = np.diag(bd + g) + np.diag(bo[:bd.size - 1], 1) + np.diag(bo[:bd.size - 1], -1)
        out = np.kron(out, np.linalg.inv(F))
    return out


def preconditioner(family, meshes, l, s2, A, prior):
    """the apply function of the Kronecker preconditioner for the system (A, prior) of oracle.optimal_mean(_mg).system"""
    knots = [int(t.numel()) for t in meshes]
    facs = factors(family, meshes, l, s2, shift(A, prior, len(knots)))
    assert math.prod(knots) == A.shape[0]
    return lambda r: apply(facs, knots, r)
