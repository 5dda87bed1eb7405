"""Kronecker-preconditioned CG for the optimal variational mean (vggp_meanopt_solve_pc with VGGP_MEANOPT_KRONECKER,
csrc/meanopt.cuh) without a GPU:
  * the Thomas form of the preconditioner (tests/kron_oracle.py) equals kron_d (F_d + g I)^-1 formed densely, and the
    dense-inverse version of tools/mg_oracle_iterations.py;
  * under the SIMT emulator: the device application (through the first CG iterate), the solve against the dense Cholesky
    m* of oracle/optimal_mean.py, its iteration count against the oracle's PCG, the warm start, the edge cases, the
    refusals, and the Jacobi choice of the new entry point against vggp_meanopt_solve bit for bit."""
import ctypes as C
import os
import sys

import numpy as np
import pytest
import torch

import emul_lib
import kron_oracle as KO
from oracle import optimal_mean as OM
from oracle import optimal_mean_mg as MG
from oracle import vggp_oracle as O
from test_optimal_mean import _arrays, _assemble, _plan, _problem, _relerr

E_ARG, E_UNSUPPORTED = -1, -6
SHAPES = [(7,), (5, 37), (37, 5), (3, 4, 29)]


def _meshes(family, knots):
    meshes = [torch.linspace(0, 1, k, dtype=torch.float32) for k in knots]
    if family != O.B1_ASVGP:            # the Markov form takes any sorted points
        meshes = [(t ** (1.0 + 0.3 * d)).to(torch.float32) for d, t in enumerate(meshes)]
    return meshes


@pytest.mark.parametrize("family", [O.B1_ASVGP, O.SVGP_GRID])
@pytest.mark.parametrize("knots", SHAPES + [(2560,)])
def test_thomas_apply_equals_dense_inverse(family, knots):
    D = len(knots)
    meshes = _meshes(family, knots)
    l = torch.linspace(0.2, 0.4, D, dtype=torch.float64)
    s2 = torch.linspace(0.7, 1.1, D, dtype=torch.float64)
    g = 0.37
    facs = KO.factors(family, meshes, l, s2, g)
    r = np.random.default_rng(len(knots)).standard_normal(int(np.prod(knots)))
    got = KO.apply(facs, list(knots), r)
    if int(np.prod(knots)) <= 1024:
        want = KO.dense(family, meshes, l, s2, g) @ r
    else:                               # 1-D only: one dense solve
        bd, bo = KO.prior_bands(family, meshes, l, s2)[0]
        want = np.linalg.solve(np.diag(bd + g) + np.diag(bo, 1) + np.diag(bo, -1), r)
    assert _relerr(got, want) <= 1e-12


@pytest.mark.parametrize("family", [O.B1_ASVGP, O.SVGP_GRID])
def test_thomas_apply_matches_the_dense_tool_version(family):
    sys.path.insert(0, os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "tools"))
    from mg_oracle_iterations import kron_preconditioner
    meshes, X, y, l, s2, noise, m, Ls = _problem(family, (6, 5, 4), 700, seed=3)
    A, rhs, prior = MG.system(family, meshes, X, y, l, s2, noise)
    r = np.random.default_rng(2).standard_normal(A.shape[0])
    want = kron_preconditioner(family, meshes, l, s2, A, prior)(r)
    got = KO.preconditioner(family, meshes, l, s2, A, prior)(r)
    assert _relerr(got, want) <= 1e-12


# ---- the C ABI under the SIMT emulator ------------------------------------------------------------------------
@pytest.fixture(scope="module")
def emu():
    got = emul_lib.load()
    if got is None:
        pytest.skip("g++ not available")
    return got


def _solve_pc(plan, precond, rtol=1e-12, max_iter=10000):
    out = np.full(plan.M, np.nan)
    it, rr = C.c_int(-1), C.c_double(-1.0)
    plan.check(plan.lib.vggp_meanopt_solve_pc(plan.h, precond, rtol, max_iter, emul_lib.ptr(out), C.byref(it),
                                              C.byref(rr), None))
    return out, it.value, rr.value


def _setup(emu, family, knots, N, seed, dtype=np.float64, m0=None):
    meshes, X, y, l, s2, noise, m, Ls = _problem(family, knots, N, seed=seed)
    tq = torch.float32 if dtype == np.float32 else torch.float64
    Xq, yq = X.to(tq).to(torch.float64), y.to(tq).to(torch.float64)
    plan = _plan(emu, family, meshes, dtype)
    theta, mm, Lcat, xs, yy = _arrays(plan, Xq, yq, l, s2, noise, m, Ls, dtype)
    obs = plan.bin(xs, yy, run_cap=16)
    plan.grid_forward(theta, np.zeros(plan.M) if m0 is None else m0, Lcat)
    _assemble(plan, obs)
    return plan, (meshes, Xq, yq, l, s2, noise), (theta, Lcat, obs)


@pytest.mark.parametrize("family", [O.B1_ASVGP, O.SVGP_GRID])
@pytest.mark.parametrize("knots", SHAPES + [(2560,), (1536, 256)])
def test_emulated_application_matches_oracle_through_the_first_iterate(emu, family, knots):
    """From x0 = 0 the first iterate is x1 = (r0.z0 / z0.A z0) z0 with z0 = P b: it carries the device's P to 1e-12.
    (2560,): the longest mesh of a plan, one row per block in shared memory.  (1536, 256): with the emulator's 3 SMs the
    contiguous mode gets 2 segments per row, whose 32-row tile exceeds the shared-memory budget, so the segment count
    doubles until the tile fits."""
    N = min(20000, 60 * int(np.prod(knots)) // len(knots))
    plan, (meshes, X, y, l, s2, noise), _ = _setup(emu, family, knots, N, seed=5)
    got, it, rr = _solve_pc(plan, emu[1].MEANOPT_KRONECKER, rtol=0.0, max_iter=1)
    assert it == 1 and rr > 0.0
    A, rhs, prior = MG.system(family, meshes, X, y, l, s2, noise)
    z0 = KO.preconditioner(family, meshes, l, s2, A, prior)(rhs)
    x1 = (rhs @ z0) / (z0 @ A @ z0) * z0
    want = prior @ x1 if family == O.B1_ASVGP else x1
    tol = 1e-12
    if family == O.B1_ASVGP:            # the epilogue m = Kuu x cancels: its rounding grows with || |Kuu| |x| || / ||Kuu x||
        tol = max(tol, 2e-16 * np.linalg.norm(abs(prior) @ abs(x1)) / np.linalg.norm(want))
    assert _relerr(got, want) <= tol, (_relerr(got, want), tol)
    plan.close()


@pytest.mark.parametrize("family", [O.B1_ASVGP, O.SVGP_GRID])
@pytest.mark.parametrize("knots,N", [((11,), 400), ((8, 7), 600), ((6, 5, 4), 700)])
@pytest.mark.parametrize("dtype,tol", [(np.float64, 1e-8), (np.float32, 1e-4)])
def test_emulated_kronecker_solve_matches_oracle(emu, family, knots, N, dtype, tol):
    plan, (meshes, X, y, l, s2, noise), _ = _setup(emu, family, knots, N, seed=23 + len(knots), dtype=dtype)
    ref = OM.optimal_mean(family, meshes, X, y, l, s2, noise)
    got, it, rr = _solve_pc(plan, emu[1].MEANOPT_KRONECKER)
    assert 0 < it <= 10000 and rr <= 1e-12
    assert _relerr(got, ref) <= tol, (it, rr, _relerr(got, ref))
    if dtype == np.float64:             # the oracle's PCG on the same system takes the same number of iterations
        A, rhs, prior = (t.numpy() for t in OM.system(family, meshes, X, y, l, s2, noise))
        _, it_ref, _ = MG.pcg(A, rhs, None, rtol=1e-12, max_iter=10000,
                              precondition=KO.preconditioner(family, meshes, l, s2, A, prior))
        assert abs(it - it_ref) <= 2, (it, it_ref)
    plan.close()


@pytest.mark.parametrize("family", [O.B1_ASVGP, O.SVGP_GRID])
def test_kronecker_warm_start_edge_cases_and_scratch(emu, family):
    lib, L = emu
    plan, _, (theta, Lcat, obs) = _setup(emu, family, (8, 7), 300, seed=41)
    sc = C.c_int64()
    plan.check(lib.vggp_workspace_bytes(plan.h, None, None, C.byref(sc)))
    before = sc.value
    mstar, it, rr = _solve_pc(plan, L.MEANOPT_KRONECKER, rtol=1e-10)
    assert it > 0 and rr <= 1e-10
    plan.check(lib.vggp_workspace_bytes(plan.h, None, None, C.byref(sc)))
    assert sc.value - before == 8 * (plan.M + 3 * (8 + 7) + 1)
    # warm start: a forward at m* makes the next solve start at its own result
    plan.grid_forward(theta, mstar, Lcat)
    _assemble(plan, obs)
    _, it2, rr2 = _solve_pc(plan, L.MEANOPT_KRONECKER, rtol=1e-10)
    assert it2 <= 1 and rr2 <= 1e-10
    # one iteration on a non-trivial problem: status 0, relres above rtol
    plan.grid_forward(theta, np.zeros(plan.M), Lcat)
    _, it, rr = _solve_pc(plan, L.MEANOPT_KRONECKER, rtol=1e-10, max_iter=1)
    assert it == 1 and rr > 1e-10
    # no data: m* = 0, 0 iterations, relres 0
    _assemble(plan, plan.bin([np.zeros(0)] * 2, np.zeros(0)))
    got, it, rr = _solve_pc(plan, L.MEANOPT_KRONECKER)
    assert it == 0 and rr == 0.0 and not np.any(got)
    # an unknown preconditioner
    out = np.zeros(plan.M)
    i, r = C.c_int(), C.c_double()
    for bad in (-1, 2):
        assert lib.vggp_meanopt_solve_pc(plan.h, bad, 1e-10, 10, emul_lib.ptr(out), C.byref(i), C.byref(r), None) == E_ARG
        assert b"precond" in lib.vggp_last_error()
    plan.close()


@pytest.mark.parametrize("family", [O.B1_ASVGP, O.SVGP_GRID])
@pytest.mark.parametrize("knots", [(11,), (8, 7), (6, 5, 4)])
def test_jacobi_through_the_new_entry_point_is_bitwise_the_old_solve(emu, family, knots):
    lib, L = emu
    plan, _, _ = _setup(emu, family, knots, 500, seed=7)
    a, ita, rra = _solve_pc(plan, L.MEANOPT_JACOBI, rtol=1e-10)
    b = np.full(plan.M, np.nan)
    itb, rrb = C.c_int(-1), C.c_double(-1.0)
    plan.check(lib.vggp_meanopt_solve(plan.h, 1e-10, 10000, emul_lib.ptr(b), C.byref(itb), C.byref(rrb), None))
    assert ita == itb.value and rra == rrb.value and np.array_equal(a, b)
    # a Kronecker solve in between leaves the Jacobi solve unchanged
    _solve_pc(plan, L.MEANOPT_KRONECKER, rtol=1e-10)
    c, itc, rrc = _solve_pc(plan, L.MEANOPT_JACOBI, rtol=1e-10)
    assert itc == ita and rrc == rra and np.array_equal(a, c)
    plan.close()


def test_kronecker_refusals(emu):
    lib, L = emu
    out = np.zeros(64)
    it, rr = C.c_int(), C.c_double()
    for family, knots in ((L.B0_GRIDDED, (5, 6)), (L.SVGP_GRID, (5, 6)), (L.VFF_GRID, (5, 7))):
        meshes = [np.linspace(0, 1, k, dtype=np.float32) for k in knots]
        plan = emul_lib.EmuPlan(lib, L, family, meshes, np.float64)
        for pc in (L.MEANOPT_JACOBI, L.MEANOPT_KRONECKER):
            rc = lib.vggp_meanopt_solve_pc(plan.h, pc, 1e-10, 10, emul_lib.ptr(out), C.byref(it), C.byref(rr), None)
            assert rc == E_UNSUPPORTED
        plan.close()
    for family in (L.B1_ASVGP, L.SVGP_MARKOV):
        plan = emul_lib.EmuPlan(lib, L, family, [np.linspace(0, 1, 8, dtype=np.float32)] * 2, np.float64)
        rc = lib.vggp_meanopt_solve_pc(plan.h, L.MEANOPT_KRONECKER, 1e-10, 10, emul_lib.ptr(out), C.byref(it),
                                       C.byref(rr), None)
        assert rc == E_ARG and b"assemble" in lib.vggp_last_error()
        plan.close()
