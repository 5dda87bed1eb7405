"""Optimal variational mean (vggp_meanopt_assemble / vggp_meanopt_solve, csrc/meanopt.cuh) without a GPU:
  * the dense statement of the stencil systems (oracle/optimal_mean.py) gives the mean of the reference's q_u() (vggp_oracle,
    pinned to reference-run goldens) for the B1 family and the Markov form of SVGP_GRID, D = 1, 2, 3;
  * assembly + conjugate gradients under the SIMT emulator (tests/host_emul) against that oracle, the existing step's d m at
    the result (zero at the optimum), the warm start, the edge cases and the refusals."""
import ctypes as C

import numpy as np
import pytest
import torch

import emul_lib
from oracle import optimal_mean as OM
from oracle import vggp_oracle as O
from test_gpu_elbo import make_problem


def _problem(family, knots, N, seed, x_lo=-0.3, x_hi=1.3):
    meshes, X, y, l, s2, noise, m, Ls = make_problem(knots, N, seed=seed, family=O.B1_ASVGP if family == O.B1_ASVGP else O.SVGP_GRID,
                                                     x_lo=x_lo, x_hi=x_hi)
    if family != O.B1_ASVGP:       # the Markov form takes any sorted points (B1 meshes are uniform)
        meshes = [(t ** (1.0 + 0.3 * d)).to(torch.float32) for d, t in enumerate(meshes)]
    return meshes, X.contiguous(), y, l, s2, noise, m, Ls


def _relerr(a, b):
    a = torch.as_tensor(np.asarray(a), dtype=torch.float64).reshape(-1)
    b = torch.as_tensor(np.asarray(b), dtype=torch.float64).reshape(-1)
    return float((a - b).norm() / b.norm().clamp_min(1e-300))


@pytest.mark.parametrize("family", [O.B1_ASVGP, O.SVGP_GRID])
@pytest.mark.parametrize("knots", [(11,), (8, 7), (6, 5, 4)])
def test_stencil_system_gives_the_reference_optimal_mean(family, knots):
    meshes, X, y, l, s2, noise, m, Ls = _problem(family, knots, 500, seed=11 + len(knots))
    assert bool((X < 0).any()) and bool((X > 1).any())
    ref = O.optimal_q(family, meshes, X, y, l, s2, noise, ref_quirks=False)[0]
    got = OM.optimal_mean(family, meshes, X, y, l, s2, noise)
    assert _relerr(got, ref) <= 1e-10


# ---- the C ABI under the SIMT emulator ------------------------------------------------------------------------
@pytest.fixture(scope="module")
def emu():
    got = emul_lib.load()
    if got is None:
        pytest.skip("g++ not available")
    return got


FAMILIES = {O.B1_ASVGP: "B1_ASVGP", O.SVGP_GRID: "SVGP_MARKOV"}


def _plan(emu, family, meshes, dtype):
    lib, L = emu
    return emul_lib.EmuPlan(lib, L, getattr(L, FAMILIES[family]), [t.numpy() for t in meshes], dtype)


def _arrays(plan, X, y, l, s2, noise, m, Ls, dtype):
    theta = torch.cat([l, s2, noise.reshape(1)]).numpy().copy()
    Lcat = torch.cat([L.reshape(-1) for L in Ls]).numpy().copy()
    xs = [np.ascontiguousarray(X[:, d].numpy().astype(dtype)) for d in range(plan.D)]
    return theta, m.numpy().copy(), Lcat, xs, np.ascontiguousarray(y.numpy().astype(dtype))


def _assemble(plan, obs):
    plan.check(plan.lib.vggp_meanopt_assemble(plan.h, C.byref(obs[2]), emul_lib.ptr(obs[1]), None))


def _solve(plan, rtol=1e-12, max_iter=10000):
    out = np.full(plan.M, np.nan)
    it, rr = C.c_int(-1), C.c_double(-1.0)
    plan.check(plan.lib.vggp_meanopt_solve(plan.h, rtol, max_iter, emul_lib.ptr(out), C.byref(it), C.byref(rr), None))
    return out, it.value, rr.value


def _optimal(plan, theta, m, Lcat, obs, **kw):
    """forward at (theta, m), assemble, solve"""
    plan.grid_forward(theta, m, Lcat)
    _assemble(plan, obs)
    return _solve(plan, **kw)


@pytest.mark.parametrize("family", [O.B1_ASVGP, O.SVGP_GRID])
@pytest.mark.parametrize("knots,N", [((11,), 400), ((8, 7), 600), ((6, 5, 4), 700)])
@pytest.mark.parametrize("dtype,tol", [(np.float64, 1e-8), (np.float32, 1e-4)])
def test_emulated_optimal_mean_matches_oracle(emu, family, knots, N, dtype, tol):
    meshes, X, y, l, s2, noise, m, Ls = _problem(family, knots, N, seed=23 + len(knots))
    tq = torch.float32 if dtype == np.float32 else torch.float64
    Xq, yq = X.to(tq).to(torch.float64), y.to(tq).to(torch.float64)
    ref = OM.optimal_mean(family, meshes, Xq, yq, l, s2, noise)
    plan = _plan(emu, family, meshes, dtype)
    theta, mm, Lcat, xs, yy = _arrays(plan, Xq, yq, l, s2, noise, m, Ls, dtype)
    obs = plan.bin(xs, yy, run_cap=16)
    got, it, rr = _optimal(plan, theta, np.zeros(plan.M), Lcat, obs)
    assert 0 < it <= 10000 and rr <= 1e-12
    assert _relerr(got, ref) <= tol, (it, rr, _relerr(got, ref))
    plan.close()


@pytest.mark.parametrize("family", [O.B1_ASVGP, O.SVGP_GRID])
@pytest.mark.parametrize("knots", [(9, 8), (6, 5, 4)])
def test_existing_step_is_stationary_at_the_optimal_mean(emu, family, knots):
    meshes, X, y, l, s2, noise, m, Ls = _problem(family, knots, 800, seed=31 + len(knots))
    plan = _plan(emu, family, meshes, np.float64)
    theta, mm, Lcat, xs, yy = _arrays(plan, X, y, l, s2, noise, m, Ls, np.float64)
    obs = plan.bin(xs, yy, run_cap=16)
    mstar, it, rr = _optimal(plan, theta, np.zeros(plan.M), Lcat, obs)
    out0, _, dm0, _ = plan.step(theta, mm, Lcat, obs)
    e0, dm0 = out0[0], dm0.copy()
    outs, _, dms, _ = plan.step(theta, mstar, Lcat, obs)
    estar = outs[0]
    assert np.linalg.norm(dms) <= 1e-7 * np.linalg.norm(dm0), (np.linalg.norm(dms), np.linalg.norm(dm0))
    assert estar >= e0
    v = np.random.default_rng(5).standard_normal(plan.M)
    for sgn in (1.0, -1.0):
        assert estar >= plan.step(theta, mstar + sgn * 1e-3 * v, Lcat, obs)[0][0]
    # warm start: a forward at m* makes the next solve start at its own result
    _, it2, rr2 = _optimal(plan, theta, mstar, Lcat, obs, rtol=1e-10)
    assert it2 <= 1 and rr2 <= 1e-10
    plan.close()


@pytest.mark.parametrize("family", [O.B1_ASVGP, O.SVGP_GRID])
def test_empty_and_outside_and_iteration_limit(emu, family):
    knots, N = (8, 7), 300
    meshes, X, y, l, s2, noise, m, Ls = _problem(family, knots, N, seed=41)
    plan = _plan(emu, family, meshes, np.float64)
    theta, mm, Lcat, xs, yy = _arrays(plan, X, y, l, s2, noise, m, Ls, np.float64)
    # empty binned set
    got, it, rr = _optimal(plan, theta, mm, Lcat, plan.bin([np.zeros(0) for _ in range(2)], np.zeros(0)))
    assert it == 0 and rr == 0.0 and not np.any(got)
    # every observation outside the mesh in dimension 0, on both sides
    Xo = X.clone()
    Xo[:, 0] = torch.where(torch.arange(N) % 2 == 0, -0.5 - X[:, 0].abs(), 1.5 + X[:, 0].abs())
    _, _, _, xo, _ = _arrays(plan, Xo, y, l, s2, noise, m, Ls, np.float64)
    got, it, rr = _optimal(plan, theta, np.zeros(plan.M), Lcat, plan.bin(xo, yy, run_cap=16))
    if family == O.B1_ASVGP:            # zero features: m* = 0
        assert it == 0 and not np.any(got)
    else:                               # the Markov weights reach outside the points
        assert rr <= 1e-12 and _relerr(got, OM.optimal_mean(family, meshes, Xo, y, l, s2, noise)) <= 1e-8
    # one iteration on a non-trivial problem: status 0, relres above rtol
    got, it, rr = _optimal(plan, theta, np.zeros(plan.M), Lcat, plan.bin(xs, yy), rtol=1e-10, max_iter=1)
    assert it == 1 and rr > 1e-10
    plan.close()


def test_refusals(emu):
    lib, L = emu
    E_ARG, E_UNSUPPORTED = -1, -6
    out = np.zeros(64)
    it, rr = C.c_int(), C.c_double()
    for family, knots in ((L.B0_GRIDDED, (5, 6)), (L.SVGP_GRID, (5, 6)), (L.VFF_GRID, (5, 7))):
        meshes = [np.linspace(0, 1, k, dtype=np.float32) for k in knots]
        plan = emul_lib.EmuPlan(lib, L, family, meshes, np.float64)
        desc = L.BinnedDesc()
        desc.D = 2
        assert lib.vggp_meanopt_assemble(plan.h, C.byref(desc), None, None) == E_UNSUPPORTED
        assert lib.vggp_meanopt_solve(plan.h, 1e-10, 10, emul_lib.ptr(out), C.byref(it), C.byref(rr), None) == E_UNSUPPORTED
        plan.close()
    for family in (L.B1_ASVGP, L.SVGP_MARKOV):
        plan = emul_lib.EmuPlan(lib, L, family, [np.linspace(0, 1, 8, dtype=np.float32)] * 2, np.float64)
        assert lib.vggp_meanopt_solve(plan.h, 1e-10, 10, emul_lib.ptr(out), C.byref(it), C.byref(rr), None) == E_ARG
        assert b"assemble" in lib.vggp_last_error()
        plan.close()
