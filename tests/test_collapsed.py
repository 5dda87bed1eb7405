"""Collapsed ELBO (vggp_logdet_system / vggp_collapsed_terms, csrc/collapsed.cuh) without a GPU:
  * the oracle restatement of the estimator (oracle/collapsed.py): unit probes give torch.linalg.slogdet, Rademacher probes are
    unbiased over seeds;
  * under the SIMT emulator (tests/host_emul), B1 and Markov, D = 1..3, both observation dtypes, observations outside the mesh:
    unit-probe log det A and the exact terms give the reference's collapsed bound (elbo_collapsed_woodbury), the Rademacher
    estimate equals the oracle's for the same seed, the output is bitwise reproducible, and the refusals."""
import ctypes as C
import math

import numpy as np
import pytest
import torch

import emul_lib
import kron_oracle as KO
from oracle import collapsed as CO
from oracle import optimal_mean as OM
from oracle import vggp_oracle as O
from test_optimal_mean import _arrays, _plan, _problem

E_ARG, E_UNSUPPORTED = -1, -6


def _dense_system(family, knots, N, seed, dtype=np.float64):
    meshes, X, y, l, s2, noise, m, Ls = _problem(family, knots, N, seed=seed)
    tq = torch.float32 if dtype == np.float32 else torch.float64
    X, y = X.to(tq).to(torch.float64), y.to(tq).to(torch.float64)
    A, rhs, prior = (t.numpy() for t in OM.system(family, meshes, X, y, l, s2, noise))
    return (meshes, X, y, l, s2, noise, m, Ls), A, prior


def _factor(kind, family, meshes, l, s2, A, prior):
    if kind == "jacobi":
        return CO.jacobi_factor(A)
    return CO.kronecker_factor(KO.factors(family, meshes, l, s2, KO.shift(A, prior, len(meshes))))


@pytest.mark.parametrize("family", [O.B1_ASVGP, O.SVGP_GRID])
@pytest.mark.parametrize("knots", [(7,), (6, 5), (4, 5, 3)])
@pytest.mark.parametrize("pc", ["jacobi", "kronecker"])
def test_oracle_unit_probes_give_slogdet(family, knots, pc):
    (meshes, X, y, l, s2, noise, m, Ls), A, prior = _dense_system(family, knots, 300, seed=3)
    M = A.shape[0]
    est, se, ldp, vals, steps = CO.logdet_slq(A, _factor(pc, family, meshes, l, s2, A, prior), kind="unit", n_probes=M,
                                              max_steps=M, rtol=1e-14)
    want = float(torch.linalg.slogdet(torch.from_numpy(A))[1])
    assert se == 0.0 and abs(est - want) <= 1e-10 * abs(want), (est, want)


@pytest.mark.parametrize("pc", ["jacobi", "kronecker"])
def test_oracle_rademacher_is_unbiased(pc):
    family = O.B1_ASVGP
    (meshes, X, y, l, s2, noise, m, Ls), A, prior = _dense_system(family, (6, 5), 300, seed=4)
    Cf = _factor(pc, family, meshes, l, s2, A, prior)
    want = float(torch.linalg.slogdet(torch.from_numpy(A))[1])
    vals = np.concatenate([CO.logdet_slq(A, Cf, n_probes=8, seed=s, max_steps=30, rtol=1e-12)[3] for s in range(60)])
    ldp = 2.0 * np.log(np.diag(Cf)).sum()
    err = ldp + vals.mean() - want
    assert abs(err) <= 4.0 * vals.std(ddof=1) / math.sqrt(vals.size), (err, vals.std())


# ---- the C ABI under the SIMT emulator ------------------------------------------------------------------------
@pytest.fixture(scope="module")
def emu():
    got = emul_lib.load()
    if got is None:
        pytest.skip("g++ not available")
    return got


def _logdet(plan, pc, kind, k, seed, max_steps, rtol, per_probe=False):
    out = np.full(plan.L.LOGDET_FIELDS, np.nan)
    pp = np.full(k, np.nan) if per_probe else None
    plan.check(plan.lib.vggp_logdet_system(plan.h, pc, kind, k, seed, max_steps, rtol, emul_lib.ptr(out), emul_lib.ptr(pp),
                                           None))
    return out, pp


def _terms(plan, obs):
    out = np.full(plan.L.CT_FIELDS, np.nan)
    plan.check(plan.lib.vggp_collapsed_terms(plan.h, C.byref(obs[2]), emul_lib.ptr(obs[1]), emul_lib.ptr(out), None))
    return out


def _setup(emu, family, knots, N, seed, dtype, pc):
    lib, L = emu
    meshes, X, y, l, s2, noise, m, Ls = _problem(family, knots, N, seed=seed)
    tq = torch.float32 if dtype == np.float32 else torch.float64
    Xq, yq = X.to(tq).to(torch.float64), y.to(tq).to(torch.float64)
    plan = _plan(emu, family, meshes, dtype)
    theta, mm, Lcat, xs, yy = _arrays(plan, Xq, yq, l, s2, noise, m, Ls, dtype)
    obs = plan.bin(xs, yy, run_cap=16)
    plan.grid_forward(theta, np.zeros(plan.M), Lcat)
    plan.check(lib.vggp_meanopt_assemble(plan.h, C.byref(obs[2]), emul_lib.ptr(obs[1]), None))
    mstar = np.zeros(plan.M)
    it, rr = C.c_int(), C.c_double()
    plan.check(lib.vggp_meanopt_solve_pc(plan.h, pc, 1e-13, 20000, emul_lib.ptr(mstar), C.byref(it), C.byref(rr), None))
    assert rr.value <= 1e-13
    return plan, obs, (meshes, Xq, yq, l, s2, noise)


@pytest.mark.parametrize("family", [O.B1_ASVGP, O.SVGP_GRID])
@pytest.mark.parametrize("knots,N", [((7,), 300), ((6, 5), 500), ((4, 5, 3), 600)])
@pytest.mark.parametrize("dtype,tol", [(np.float64, 1e-9), (np.float32, 1e-5)])
def test_emulated_unit_probes_give_the_collapsed_bound(emu, family, knots, N, dtype, tol):
    lib, L = emu
    pcs = [L.MEANOPT_KRONECKER, L.MEANOPT_JACOBI]
    plan, obs, (meshes, X, y, l, s2, noise) = _setup(emu, family, knots, N, 50 + len(knots), dtype, pcs[0])
    assert bool((X < 0).any()) and bool((X > 1).any())
    if family == O.B1_ASVGP:
        assert obs[2].n_inside < obs[2].n
    terms = _terms(plan, obs)
    assert terms[0] == N
    np.testing.assert_allclose(terms[1], float(y @ y), rtol=1e-12)
    want = float(O.elbo_collapsed_woodbury(family, meshes, X, y, l, s2, noise, ref_quirks=False))
    M = plan.M
    for pc in pcs:
        out, pp = _logdet(plan, pc, L.PROBE_UNIT, M, 0, M + 8, 1e-14, per_probe=True)
        assert out[1] == 0.0 and out[4] == M and out[5] == M and out[3] <= M
        np.testing.assert_allclose(out[0], out[2] + pp.sum(), rtol=1e-13)
        got = CO.collapsed_elbo(*terms, out[0], float(noise), s2.numpy(), family != O.B1_ASVGP)
        assert abs(got - want) <= tol * abs(want), (pc, got, want)
    plan.close()


@pytest.mark.parametrize("family", [O.B1_ASVGP, O.SVGP_GRID])
@pytest.mark.parametrize("knots,pc", [((7,), "jacobi"), ((6, 5), "jacobi"), ((4, 5, 3), "jacobi"), ((7,), "kronecker"),
                                      ((6, 5), "kronecker"), ((4, 5, 3), "kronecker"), ((40,), "kronecker"),
                                      ((12, 20), "kronecker")])
def test_emulated_rademacher_estimate_equals_the_oracle(emu, family, knots, pc):
    """(40,) and (12, 20): the half-sweeps cut the 40- and 20-node fibres into 8 and 4 segments (the emulator has 3 SMs), so
    the carries between segments are exercised; the short fibres of the other shapes run as one segment."""
    lib, L = emu
    code = L.MEANOPT_JACOBI if pc == "jacobi" else L.MEANOPT_KRONECKER
    plan, obs, (meshes, X, y, l, s2, noise) = _setup(emu, family, knots, 400, 70 + len(knots), np.float64, code)
    A, rhs, prior = (t.numpy() for t in OM.system(family, meshes, X, y, l, s2, noise))
    k, seed = 6, 12345678901
    out, pp = _logdet(plan, code, L.PROBE_RADEMACHER, k, seed, 60, 1e-12, per_probe=True)
    est, se, ldp, vals, steps = CO.logdet_slq(A, _factor(pc, family, meshes, l, s2, A, prior), n_probes=k, seed=seed,
                                              max_steps=60, rtol=1e-12)
    assert out[4] == k and out[5] == k
    np.testing.assert_allclose(out[2], ldp, rtol=1e-12)
    np.testing.assert_allclose(pp, vals, rtol=1e-10, atol=1e-10 * abs(ldp))
    np.testing.assert_allclose(out[0], est, rtol=1e-10)
    np.testing.assert_allclose(out[1], se, rtol=1e-8)
    # the same seed again: the same bits
    again, pp2 = _logdet(plan, code, L.PROBE_RADEMACHER, k, seed, 60, 1e-12, per_probe=True)
    assert np.array_equal(out, again) and np.array_equal(pp, pp2)
    plan.close()


def test_emulated_step_limit_and_scratch(emu):
    lib, L = emu
    plan, obs, _ = _setup(emu, O.SVGP_GRID, (6, 5), 400, 9, np.float64, L.MEANOPT_JACOBI)
    sc = C.c_int64()
    plan.check(lib.vggp_workspace_bytes(plan.h, None, None, C.byref(sc)))
    before = sc.value
    out, _ = _logdet(plan, L.MEANOPT_JACOBI, L.PROBE_RADEMACHER, 4, 1, 3, 1e-14)
    assert out[3] == 3 and out[4] == 0 and out[5] == 4 and np.isfinite(out[0])
    plan.check(lib.vggp_workspace_bytes(plan.h, None, None, C.byref(sc)))
    assert sc.value - before >= 8 * (4 * 4 + 1) * plan.M
    plan.close()


def test_refusals(emu):
    lib, L = emu
    out = np.zeros(8)
    for family, knots in ((L.B0_GRIDDED, (5, 6)), (L.SVGP_GRID, (5, 6)), (L.VFF_GRID, (5, 7))):
        plan = emul_lib.EmuPlan(lib, L, family, [np.linspace(0, 1, k, dtype=np.float32) for k in knots], np.float64)
        assert lib.vggp_logdet_system(plan.h, 0, 0, 4, 0, 10, 1e-6, emul_lib.ptr(out), None, None) == E_UNSUPPORTED
        desc = L.BinnedDesc()
        desc.D = 2
        assert lib.vggp_collapsed_terms(plan.h, C.byref(desc), None, emul_lib.ptr(out), None) == E_UNSUPPORTED
        plan.close()
    for family in (O.B1_ASVGP, O.SVGP_GRID):
        code = L.B1_ASVGP if family == O.B1_ASVGP else L.SVGP_MARKOV
        plan = emul_lib.EmuPlan(lib, L, code, [np.linspace(0, 1, 6, dtype=np.float32)] * 2, np.float64)
        assert lib.vggp_logdet_system(plan.h, 0, 0, 4, 0, 10, 1e-6, emul_lib.ptr(out), None, None) == E_ARG
        assert b"assemble" in lib.vggp_last_error()
        plan.close()
        # assembled but not solved: the terms refuse, the log-determinant runs
        plan, obs, _ = _setup(emu, family, (6, 5), 200, 5, np.float64, L.MEANOPT_JACOBI)
        plan.check(lib.vggp_meanopt_assemble(plan.h, C.byref(obs[2]), emul_lib.ptr(obs[1]), None))
        assert lib.vggp_collapsed_terms(plan.h, C.byref(obs[2]), emul_lib.ptr(obs[1]), emul_lib.ptr(out), None) == E_ARG
        assert b"solve" in lib.vggp_last_error()
        M = plan.M
        for pc, kind, k, first in ((2, 0, 4, 0), (-1, 0, 4, 0), (0, 0, 0, 0), (0, 2, 4, 0), (0, 1, 4, M - 3), (0, 1, 1, M)):
            assert lib.vggp_logdet_system(plan.h, pc, kind, k, first, 10, 1e-6, emul_lib.ptr(out), None, None) == E_ARG
        assert lib.vggp_logdet_system(plan.h, 0, 0, 65536, 0, 10, 1e-6, emul_lib.ptr(out), None, None) == E_ARG
        _logdet(plan, L.MEANOPT_KRONECKER, L.PROBE_UNIT, 3, M - 3, 10, 1e-6)
        plan.close()
        # solved, then: another binned set, and a grid forward after the solve
        plan, obs, (meshes, X, y, l, s2, noise) = _setup(emu, family, (6, 5), 200, 5, np.float64, L.MEANOPT_JACOBI)
        _terms(plan, obs)
        xs = [np.ascontiguousarray(X[:150, d].numpy()) for d in range(2)]
        other = plan.bin(xs, np.ascontiguousarray(y[:150].numpy()), run_cap=16)
        assert lib.vggp_collapsed_terms(plan.h, C.byref(other[2]), emul_lib.ptr(other[1]), emul_lib.ptr(out), None) == E_ARG
        assert b"binned set" in lib.vggp_last_error()
        theta, Lcat = plan._keep[0], plan._keep[2]
        plan.grid_forward(theta, np.zeros(plan.M), Lcat)
        assert lib.vggp_collapsed_terms(plan.h, C.byref(obs[2]), emul_lib.ptr(obs[1]), emul_lib.ptr(out), None) == E_ARG
        assert b"grid_forward" in lib.vggp_last_error()
        plan.close()
