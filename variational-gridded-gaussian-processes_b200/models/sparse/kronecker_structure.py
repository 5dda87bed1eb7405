"""2-D Kronecker-structured sparse models: drop-in names of src/models/sparse/kronecker_structure.py."""
from typing import Tuple

import torch

from ... import _lib
from ...basis import B0SplineBasis, B1SplineBasis
from .._gridded import GriddedMarginals, GriddedVariationalGP, linspace_mesh


class KroneckerStructure(GriddedVariationalGP):
    """kronecker_structure.py:15-278 (base class name kept)."""


class _TwoDimMesh(KroneckerStructure):
    def __init__(self, X, y, nknots: int, dim1lims: Tuple[float, float], dim2lims: Tuple[float, float]):
        self.nknots = nknots
        self.dim1lims = dim1lims
        self.dim2lims = dim2lims
        mesh_1 = linspace_mesh(dim1lims, nknots)
        mesh_2 = linspace_mesh(dim2lims, nknots)
        super().__init__(X, y, [mesh_1, mesh_2])
        self.mesh_1, self.mesh_2 = mesh_1, mesh_2
        self.delta_1 = mesh_1[1] - mesh_1[0]
        self.delta_2 = mesh_2[1] - mesh_2[0]


class Matern12B1SplineASVGP(_TwoDimMesh):
    """kronecker_structure.py:524-662."""
    family = _lib.B1_ASVGP

    def __init__(self, X, y, nknots, dim1lims, dim2lims):
        super().__init__(X, y, nknots, dim1lims, dim2lims)
        self.delta = self.delta_1
        self.basis_1 = B1SplineBasis(self.mesh_1)
        self.basis_2 = B1SplineBasis(self.mesh_2)


class Matern12B0SplineGriddedGP(_TwoDimMesh):
    """kronecker_structure.py:671-849."""
    family = _lib.B0_GRIDDED

    def __init__(self, X, y, nknots, dim1lims, dim2lims):
        super().__init__(X, y, nknots, dim1lims, dim2lims)
        self.basis_1 = B0SplineBasis(self.mesh_1)
        self.basis_2 = B0SplineBasis(self.mesh_2)

    def q_v(self, optimal: bool = False):
        """q(v) = q(u): the inducing variables are the cell integrals (kronecker_structure.py:825-849 returns the
        closed-form optimum: `optimal=True`; default: the learned q(u))."""
        return self.q_u(optimal)


class _DenseFeatureModel(KroneckerStructure):
    """Families whose per-observation work goes through the dense-feature kernel (SVGP points, Fourier features): plain
    observation arrays, and point predictions assembled from the exported dense features."""

    def posterior(self, x: torch.Tensor) -> GriddedMarginals:
        """Marginals of q(f(x*)) (kronecker_structure.py:199-230 restricted to its diagonal) from the dense per-dimension
        features and the workspace of the last forward: mean = phi_1^T A phi_2, var = kff - prod_d phi_d^T P_d phi_d +
        prod_d phi_d^T Q_d phi_d (device torch ops; small grids)."""
        plan = self._ensure_plan()
        theta = self._theta()
        m = self.variational_mean.detach().to(torch.float64).contiguous()
        L = torch.cat([c.detach().to(torch.float64).reshape(-1) for c in self._chols()]).contiguous()
        plan.grid_forward(theta, m, L)
        x = x.reshape(x.shape[0], -1).to(device=plan.device, dtype=plan.obs_dtype)
        phis = [plan.features_dense(d, x[:, d].contiguous(), theta).to(torch.float64) for d in range(self.D)]
        A = plan.workspace(_lib.WS_ALPHA).reshape(self.m_per_dim)
        mean = torch.einsum("in,ij,jn->n", phis[0], A, phis[1])
        p = torch.ones_like(mean)
        q = torch.ones_like(mean)
        for d in range(self.D):
            p = p * (phis[d] * (plan.workspace(_lib.WS_P, d) @ phis[d])).sum(0)
            q = q * (phis[d] * (plan.workspace(_lib.WS_Q, d) @ phis[d])).sum(0)
        kff = torch.prod(theta[self.D:2 * self.D])
        return GriddedMarginals(mean.to(plan.obs_dtype), (kff - p + q).to(plan.obs_dtype))


class Matern12SVGP(_DenseFeatureModel):
    """kronecker_structure.py:287-338: SVGP with inducing POINTS on a product grid, Z (m x 2) holding the per-dimension
    locations in its columns (`Kuu = kron(k_1(Z), k_2(Z))`, `Kuf = k(cartesian_prod(Z[:, 0], Z[:, 1]), x)`).

    Same constructor as the reference.  Differences: the step is the uncollapsed bound (explicit q(u), like every class
    here); the columns of Z are sorted (the library wants increasing knots; the product grid is the same set); and Z is a
    fixed buffer -- the reference registers it as a parameter, d ELBO / d Z is not computed here.  Per-observation work
    goes through the dense-feature kernel (k_obs_b0 with s2 exp(-|x - z| / l) features): O(M + sum M_d^2) per observation,
    the reference's own dense algorithm, meant for the grid sizes the reference uses (tens of points per dimension).

    `markov=True` evaluates the same model (same ELBO, gradients and predictions) in its O(1)-per-observation Markov form
    (family SVGP_MARKOV, csrc/svgpm.cuh): K_d^-1 is tridiagonal for a Matern-1/2 kernel on sorted points, so every
    observation touches two inducing points per dimension, the grid side is O(M + sum M_d^2), and 512 x 512 grids with
    2^26 observations are in reach.  Full-batch `_elbo()` only (a minibatch raises NotImplementedError).  The default stays
    the dense path for now; the intended follow-up makes `markov=True` the default and keeps SVGP_GRID as the test
    reference."""
    family = _lib.SVGP_GRID

    def __init__(self, X, y, Z: torch.Tensor, markov: bool = False):
        self.markov = bool(markov)
        if self.markov:
            self.family = _lib.SVGP_MARKOV
        Z = torch.as_tensor(Z).detach()
        if Z.dim() != 2 or Z.shape[1] != 2:
            raise ValueError("Z must be (m, 2): one column of inducing locations per dimension")
        cols = [torch.sort(Z[:, d].to(torch.float32)).values for d in range(2)]
        for c in cols:
            if not bool((c[1:] > c[:-1]).all()):
                raise ValueError("the inducing locations of a dimension must be distinct")
        super().__init__(X, y, cols)
        self.register_buffer("Z", torch.stack(cols, dim=1))

    def posterior(self, x: torch.Tensor) -> GriddedMarginals:
        """Marginals of q(f(x*)): the dense-feature assembly, or with `markov=True` the library's O(1)-per-point prediction
        (vggp_predict)."""
        if self.markov:
            return GriddedVariationalGP.posterior(self, x)
        return super().posterior(x)


class Matern12VFFGP(_DenseFeatureModel):
    """kronecker_structure.py:347-514: variational Fourier features for a Matern-1/2 kernel, `nfrequencies` frequencies per
    dimension on the domains `dim1lims`, `dim2lims` (2 nfrequencies + 1 inducing features per dimension: cosines, then sines;
    `Kuu_d = diag(alpha) + beta beta^T`, `Kuf_d = FourierBasisMatern12(x)`, src/basis/fourier.py:58-88).  Same constructor as
    the reference.  Differences: the uncollapsed bound with explicit q(u); float64 throughout (the reference's float32
    frequency tensor makes its Kuu and Kuf float32 before the final cast -- `ref_quirks` in the oracle reproduces that and is
    pinned to the reference's own output); the limits are stored as float32 knots."""
    family = _lib.VFF_GRID

    def __init__(self, X, y, nfrequencies: int, dim1lims: Tuple[float, float], dim2lims: Tuple[float, float]):
        self.nfrequencies = int(nfrequencies)
        self.dim1lims, self.dim2lims = dim1lims, dim2lims
        n = 2 * self.nfrequencies + 1
        super().__init__(X, y, [linspace_mesh(dim1lims, n), linspace_mesh(dim2lims, n)])
        import math
        self.omegas_1 = 2 * math.pi * torch.arange(self.nfrequencies + 1) / (dim1lims[1] - dim1lims[0])
        self.omegas_2 = 2 * math.pi * torch.arange(self.nfrequencies + 1) / (dim2lims[1] - dim2lims[0])
