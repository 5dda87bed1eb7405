"""TEST INFRASTRUCTURE / DESIGN VALIDATION -- the collapsed bound of the B1 and VGGP_SVGP_MARKOV families as the library
computes it (csrc/collapsed.cuh, vggp_logdet_system / vggp_collapsed_terms), float64 numpy, dense matrices (small M only).

With A = F + G / noise the optimal-mean system (oracle.optimal_mean.system: F = Kuu for B1, Kuu^-1 for Markov), x* its
solution and b its right-hand side times noise,
    ELBO = -1/2 [N log 2 pi + N log noise + log det A - log det F + (y^T y - b^T x*) / noise] - (N prod s2 - tr(F^-1 G)) / (2 noise)
log det A by preconditioned stochastic Lanczos quadrature: P = C C^T, log det A = log det P + tr log(C^-1 A C^-T), the trace
estimated from probes eps_j by Gauss quadrature on the Lanczos tridiagonal of each probe.  The Rademacher probes use the
counter hash of the device (mb_mix32 of csrc/minibatch.cuh keyed by seed and probe), so the same seed gives the same signs;
the convergence rule is the device's (quadrature checked every CHECK steps up to 16 CHECK, then every
steps / 8 rounded down to a multiple of CHECK; stop at a relative change <= rtol between checks)."""
import math

import numpy as np
import scipy.linalg as sla

CHECK = 8
_M32 = 0xFFFFFFFF


def mix32(x):
    """mb_mix32 of csrc/minibatch.cuh on uint64 arrays holding 32-bit values"""
    x = np.asarray(x, dtype=np.uint64) & _M32
    x ^= x >> np.uint64(16)
    x = (x * np.uint64(0x7FEB352D)) & _M32
    x ^= x >> np.uint64(15)
    x = (x * np.uint64(0x846CA68B)) & _M32
    x ^= x >> np.uint64(16)
    return x


def probe_key(seed: int, probe: int) -> int:
    h = int(mix32(seed & _M32))
    h = int(mix32(h ^ ((seed >> 32) & _M32)))
    return int(mix32(h ^ (((probe + 1) * 0x9E3779B9) & _M32)))


def rademacher(seed: int, probe: int, M: int) -> np.ndarray:
    """the probe eps_j of vggp_logdet_system: +1 / -1 from the top bit of mix32(key ^ node)"""
    h = mix32(np.uint64(probe_key(seed, probe)) ^ np.arange(M, dtype=np.uint64))
    return np.where((h >> np.uint64(31)) & np.uint64(1), -1.0, 1.0)


def kronecker_factor(thomas):
    """dense C = kron_d L_d D_d^(1/2) from the Thomas factors (l, 1 / d', off) of F_d + g I (tests/kron_oracle.thomas)"""
    C = np.ones((1, 1))
    for l, invd, _ in thomas:
        n = l.size
        Ld = np.eye(n) + np.diag(l[1:], -1)
        C = np.kron(C, Ld * np.sqrt(1.0 / invd)[None, :])
    return C


def jacobi_factor(A):
    return np.diag(np.sqrt(np.diag(A)))


def gauss_log(alpha, beta):
    """sum_i tau_i^2 log theta_i of the Lanczos tridiagonal (alpha, beta[:-1])"""
    theta, vec = sla.eigh_tridiagonal(np.asarray(alpha), np.asarray(beta[:len(alpha) - 1]))
    return float(np.sum(vec[0] ** 2 * np.log(theta)))


def lanczos_quadrature(B, v, max_steps, rtol):
    """eps^T log(B) eps / ||eps||^2 for v = eps / ||eps||, with the device's stopping rule; returns (value, steps, converged)"""
    M = B.shape[0]
    v0, v1 = np.zeros(M), v.copy()
    alpha, beta = [], []
    q, conv = math.nan, False
    check = CHECK
    for step in range(max_steps):
        y = B @ v1
        a = float(y @ v1)
        y = y - a * v1 - (beta[-1] if beta else 0.0) * v0
        bb = float(np.sqrt(y @ y))
        alpha.append(a)
        beta.append(bb)
        exhausted = not bb > 1e-13 * abs(a) or step + 1 >= M
        last = exhausted or step + 1 >= max_steps
        if step + 1 == check or last:
            check = step + 1 + CHECK * max(1, (step + 1) // (8 * CHECK))
            qprev, q = q, gauss_log(alpha, beta)
            if exhausted or abs(q - qprev) <= rtol * abs(q):
                return q, step + 1, True
        if last:
            break
        v0, v1 = v1, y / bb
    return q, len(alpha), conv


def logdet_slq(A, C, kind="rademacher", n_probes=32, seed=0, first=0, max_steps=200, rtol=1e-8):
    """(estimate, standard error, log det P, per-probe values, steps) of log det A with the preconditioner P = C C^T
    (C lower triangular).  kind "unit": probes e_first .. e_{first + n_probes - 1}, estimate = log det P + their sum."""
    M = A.shape[0]
    Ci = sla.solve_triangular(C, np.eye(M), lower=True)
    B = Ci @ A @ Ci.T
    B = 0.5 * (B + B.T)
    logdet_p = 2.0 * float(np.sum(np.log(np.diag(C))))
    vals, steps = [], []
    for j in range(n_probes):
        if kind == "unit":
            v, norm2 = np.eye(M)[first + j], 1.0
        else:
            v, norm2 = rademacher(seed, j, M) / math.sqrt(M), float(M)
        q, s, _ = lanczos_quadrature(B, v, max_steps, rtol)
        vals.append(norm2 * q)
        steps.append(s)
    vals = np.array(vals)
    if kind == "unit":
        return logdet_p + vals.sum(), 0.0, logdet_p, vals, steps
    se = float(vals.std(ddof=1) / math.sqrt(n_probes)) if n_probes > 1 else 0.0
    return logdet_p + vals.mean(), se, logdet_p, vals, steps


def collapsed_elbo(N, yy, bx, trace, logdet_kuu, logdet_a, noise, s2, markov):
    """the bound from its terms (the composition of GriddedVariationalGP.collapsed_elbo)"""
    logdet_f = -logdet_kuu if markov else logdet_kuu
    quad = (yy - bx) / noise
    return (-0.5 * (N * math.log(2 * math.pi) + N * math.log(noise) + logdet_a - logdet_f + quad)
            - (N * float(np.prod(s2)) - trace) / (2 * noise))
