"""The multigrid statement of the optimal-mean solve (oracle/optimal_mean_mg.py), without a GPU:
  * its sparse stencil system is the dense one of oracle/optimal_mean.py (any grid size, both families, D = 1, 2, 3);
  * the hierarchy follows its rules: even indices and the last index kept, dimensions of <= 3 nodes not coarsened,
    interpolation exact on constants, coarse operators P^T A P;
  * the V-cycle is a symmetric positive definite operator, and multigrid-preconditioned CG reaches the dense Cholesky m*
    (non-uniform Markov points, observations outside the points, hierarchies of 2 and 3 levels), for each smoother of the
    statement: Chebyshev, l1-Jacobi, and l1 line-block Jacobi with full coarsening or with semi-coarsening across the lines."""
import numpy as np
import pytest
import torch

pytest.importorskip("scipy")

from oracle import optimal_mean as OM  # noqa: E402
from oracle import optimal_mean_mg as MG  # noqa: E402
from oracle import vggp_oracle as O  # noqa: E402
from test_optimal_mean import _problem, _relerr  # noqa: E402

FAMILIES = [O.B1_ASVGP, O.SVGP_GRID]
SMOOTHERS = {"chebyshev": {}, "l1": {"kind": "l1"}, "line": {"kind": "line", "line_dim": 0},
             "line_semi": {"kind": "line", "line_dim": 0, "semi": True}}


@pytest.mark.parametrize("family", FAMILIES)
@pytest.mark.parametrize("knots", [(11,), (9, 6), (7, 5, 4)])
def test_sparse_system_is_the_dense_system(family, knots):
    meshes, X, y, l, s2, noise, m, Ls = _problem(family, knots, 400, seed=5 + len(knots))
    A, rhs, prior = MG.system(family, meshes, X, y, l, s2, noise)
    Ad, rd, pd = OM.system(family, meshes, X, y, l, s2, noise)
    assert np.abs(A.toarray() - Ad.numpy()).max() <= 1e-13 * np.abs(Ad.numpy()).max()
    assert np.abs(prior.toarray() - pd.numpy()).max() <= 1e-13 * np.abs(pd.numpy()).max()
    assert _relerr(rhs, rd) <= 1e-13


def test_level_dims_and_interpolation():
    assert MG.level_dims((64, 64, 16)) == [(64, 64, 16), (33, 33, 9), (17, 17, 5), (9, 9, 3)]
    assert MG.level_dims((512, 512)) == [(512, 512), (257, 257), (129, 129), (65, 65), (33, 33), (17, 17)]
    assert MG.level_dims((9, 6), coarsest=8) == [(9, 6), (5, 4), (3, 3)]
    assert MG.level_dims((7, 5, 3), coarsest=1) == [(7, 5, 3), (4, 3, 3), (3, 3, 3)]
    assert MG.level_dims((100,)) == [(100,)]
    assert MG.level_dims((9, 6, 5), coarsest=1, keep=0) == [(9, 6, 5), (9, 4, 3), (9, 3, 3)]
    assert MG.prolongation((9, 6), (9, 4)).toarray().tolist() == np.kron(np.eye(9), MG.interp(6).toarray()).tolist()
    for n in range(2, 12):
        P = MG.interp(n).toarray()
        assert np.allclose(P.sum(axis=1), 1.0)                       # exact on constants
        if n <= 3:
            assert np.array_equal(P, np.eye(n))
            continue
        assert P.shape == (n, n // 2 + 1)
        kept = [i for i in range(n) if i % 2 == 0 or i == n - 1]
        assert np.array_equal(P[kept], np.eye(len(kept)))            # end nodes and even nodes are coarse nodes
        for i in set(range(n)) - set(kept):
            assert sorted(P[i][P[i] != 0]) == [0.5, 0.5]


@pytest.mark.parametrize("family", FAMILIES)
def test_coarse_operators_are_galerkin(family):
    meshes, X, y, l, s2, noise, m, Ls = _problem(family, (9, 6), 300, seed=3)
    A, _, _ = MG.system(family, meshes, X, y, l, s2, noise)
    H = MG.hierarchy(A, (9, 6), coarsest=8)
    assert [h["dims"] for h in H] == [(9, 6), (5, 4), (3, 3)]
    Ad = A.toarray()
    for k in range(len(H) - 1):
        P = np.kron(MG.interp(H[k]["dims"][0]).toarray(), MG.interp(H[k]["dims"][1]).toarray())
        Ad = P.T @ Ad @ P
        got = H[k + 1]["A"].toarray()
        assert np.abs(got - Ad).max() <= 1e-12 * np.abs(Ad).max()
        assert got.shape == (np.prod(H[k + 1]["dims"]),) * 2


@pytest.mark.parametrize("smoother", list(SMOOTHERS))
@pytest.mark.parametrize("family", FAMILIES)
@pytest.mark.parametrize("knots", [(9, 6), (5, 4, 3)])
def test_vcycle_is_symmetric_positive_definite(family, knots, smoother):
    meshes, X, y, l, s2, noise, m, Ls = _problem(family, knots, 300, seed=7)
    A, _, _ = MG.system(family, meshes, X, y, l, s2, noise)
    H = MG.hierarchy(A, knots, coarsest=6, **SMOOTHERS[smoother])
    assert len(H) >= 2
    M = A.shape[0]
    Z = np.stack([MG.vcycle(H, e) for e in np.eye(M)], 1)
    assert np.linalg.norm(Z - Z.T) <= 1e-12 * np.linalg.norm(Z)
    assert np.linalg.eigvalsh(0.5 * (Z + Z.T)).min() > 0
    # a convergent smoother and an exact coarsest solve make the V-cycle a contraction in the A norm: eig(Z A) in (0, 1]
    ev = np.linalg.eigvals(Z @ A.toarray()).real
    assert ev.min() > 0 and ev.max() <= 1 + 1e-10


@pytest.mark.parametrize("smoother", list(SMOOTHERS))
@pytest.mark.parametrize("family", FAMILIES)
@pytest.mark.parametrize("knots,N", [((11,), 400), ((9, 6), 600), ((7, 5, 4), 700)])
def test_multigrid_pcg_reaches_the_dense_optimal_mean(family, knots, N, smoother):
    meshes, X, y, l, s2, noise, m, Ls = _problem(family, knots, N, seed=23 + len(knots))
    assert bool((X < 0).any()) and bool((X > 1).any())
    ref = OM.optimal_mean(family, meshes, X, y, l, s2, noise)
    got, it = MG.optimal_mean(family, meshes, X, y, l, s2, noise, rtol=1e-13, coarsest=8, **SMOOTHERS[smoother])
    assert 0 < it < 1000
    assert _relerr(got, ref) <= 1e-10, (it, _relerr(got, ref))


@pytest.mark.parametrize("family", FAMILIES)
def test_pcg_edge_cases(family):
    knots = (9, 6)
    meshes, X, y, l, s2, noise, m, Ls = _problem(family, knots, 300, seed=41)
    A, rhs, _ = MG.system(family, meshes, X, y, l, s2, noise)
    H = MG.hierarchy(A, knots, coarsest=8)
    x, it, rel = MG.pcg(A, rhs, H, rtol=1e-12)
    assert rel <= 1e-12
    _, it2, rel2 = MG.pcg(A, rhs, H, x0=x, rtol=1e-10)               # a start at the solution
    assert it2 <= 1 and rel2 <= 1e-10
    _, it1, rel1 = MG.pcg(A, rhs, H, rtol=1e-10, max_iter=1)          # the iteration limit
    assert it1 == 1 and rel1 > 1e-10
    x0, it0, rel0 = MG.pcg(A, np.zeros_like(rhs), H, x0=np.ones_like(rhs))   # b = 0: m* = 0
    assert it0 == 0 and rel0 == 0.0 and not np.any(x0)
