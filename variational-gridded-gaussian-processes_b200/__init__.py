"""B200-native (sm_100a) ELBO forward/backward for variational GPs with gridded, Kronecker-structured inducing
variables.  Host side = PyTorch plumbing over the C ABI of libvggp.so (include/vggp.h); there is no CPU path.

Module layout mirrors the reference's `src/` for the classes on the hot path:
    <pkg>.basis.bspline                                  B0SplineBasis, B1SplineBasis
    <pkg>.models.sparse.univariate_structure             Matern12B1SplineASVGP, Matern12B0SplineGriddedGP (1-D)
    <pkg>.models.sparse.kronecker_structure              Matern12B1SplineASVGP, Matern12B0SplineGriddedGP (2-D)
    <pkg>.models.sparse.gridded_univariate_structure     GriddedMatern12ASVGP, Matern12GriddedGP (1-D)
    <pkg>.models.sparse.gridded_kronecker_structure      GriddedMatern12ASVGP, Matern12GriddedGP (2-D)
"""
from . import _lib  # noqa: F401
from .plan import GridPlan, gridded_elbo, gemm_f64  # noqa: F401
from .dist import shard_bounds, init_from_env, spatial_reshard  # noqa: F401
from .models._gridded import GriddedVariationalGP  # noqa: F401

B1_ASVGP = _lib.B1_ASVGP
B0_GRIDDED = _lib.B0_GRIDDED
SVGP_GRID = _lib.SVGP_GRID
VFF_GRID = _lib.VFF_GRID
SVGP_MARKOV = _lib.SVGP_MARKOV
