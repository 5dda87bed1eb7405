"""Optimal Kronecker-factored variational covariance (vggp_covopt_update, csrc/covopt.cuh) without a GPU:
  * the dense statement (oracle/optimal_cov.py) gives the reference's S* = Kuu Sigma^-1 Kuu for D = 1, zeroes the ELBO's
    gradient in L_d after updating d, and its sweeps raise the ELBO monotonically and converge, D = 2, 3;
  * the device construction (UL factorisation, U^-T columns, RQ sweep) in numpy equals numpy's Cholesky factor of S_d;
  * the C ABI under the SIMT emulator (tests/host_emul) against the oracle, the step's dL_d after the update, sharded
    gradient buffers, the failed pivot, aliasing and the refusals."""
import ctypes as C

import numpy as np
import pytest
import torch

import emul_lib
from oracle import optimal_cov as OC
from oracle import vggp_oracle as O
from test_gpu_elbo import make_problem

FAMILIES = [O.B1_ASVGP, O.SVGP_GRID]          # SVGP_GRID of the oracle is the model of the library's SVGP_MARKOV


def _problem(family, knots, N, seed, x_lo=-0.3, x_hi=1.3):
    meshes, X, y, l, s2, noise, m, Ls = make_problem(knots, N, seed=seed, family=family, x_lo=x_lo, x_hi=x_hi)
    if family != O.B1_ASVGP:       # the Markov form takes any sorted points (B1 meshes are uniform)
        meshes = [(t ** (1.0 + 0.3 * d)).to(torch.float32) for d, t in enumerate(meshes)]
    return meshes, X.contiguous(), y, l, s2, noise, m, Ls


def _relerr(a, b):
    a = torch.as_tensor(np.asarray(a), dtype=torch.float64).reshape(-1)
    b = torch.as_tensor(np.asarray(b), dtype=torch.float64).reshape(-1)
    return float((a - b).norm() / b.norm().clamp_min(1e-300))


def _sweeps(family, meshes, X, y, l, s2, noise, m, Ls, rtol=1e-8, max_sweeps=200):
    Ls = [L.clone() for L in Ls]
    elbos = [float(OC.elbo(family, meshes, X, y, l, s2, noise, m, Ls))]
    for sweep in range(1, max_sweeps + 1):
        ch = 0.0
        for d in range(len(meshes)):
            new = OC.update(family, meshes, X, l, s2, noise, Ls, d)
            ch += OC.change(new, Ls[d])
            Ls[d] = new
            elbos.append(float(OC.elbo(family, meshes, X, y, l, s2, noise, m, Ls)))
        if ch <= rtol:
            return Ls, elbos, sweep
    raise AssertionError(f"no convergence after {max_sweeps} sweeps (change {ch:.2e})")


@pytest.mark.parametrize("family", FAMILIES)
def test_one_update_is_the_reference_optimal_covariance_in_1d(family):
    meshes, X, y, l, s2, noise, m, Ls = _problem(family, (13,), 400, seed=3)
    ref = O.optimal_q(family, meshes, X, y, l, s2, noise, ref_quirks=False)[1]
    Ln = OC.update(family, meshes, X, l, s2, noise, Ls, 0)
    assert _relerr(Ln @ Ln.T, ref) <= 1e-10


@pytest.mark.parametrize("family", FAMILIES)
@pytest.mark.parametrize("knots,N", [((8, 7), 600), ((6, 5, 4), 700)])
def test_update_zeroes_the_gradient_and_sweeps_ascend(family, knots, N):
    meshes, X, y, l, s2, noise, m, Ls = _problem(family, knots, N, seed=5 + len(knots))
    for d in range(len(knots)):
        g0 = OC.grad_L(family, meshes, X, y, l, s2, noise, m, Ls, d)
        Lu = list(Ls)
        Lu[d] = OC.update(family, meshes, X, l, s2, noise, Ls, d)
        g1 = OC.grad_L(family, meshes, X, y, l, s2, noise, m, Lu, d)
        assert float(g1.norm()) <= 1e-9 * float(g0.norm()), (d, float(g1.norm()), float(g0.norm()))
    _, elbos, sweeps = _sweeps(family, meshes, X, y, l, s2, noise, m, [torch.eye(k, dtype=torch.float64) for k in knots])
    assert all(b >= a - 1e-9 * abs(a) for a, b in zip(elbos, elbos[1:])), elbos
    assert 1 < sweeps <= 60


@pytest.mark.parametrize("family", FAMILIES)
def test_device_construction_is_the_cholesky_factor(family):
    meshes, X, y, l, s2, noise, m, Ls = _problem(family, (9, 40), 900, seed=17)
    T, K, r = OC.system(family, meshes, X, l, s2, noise, Ls, 1)
    Tn, Kn = T.numpy(), K.numpy()
    S = r * (Kn @ np.linalg.inv(Tn) @ Kn if family == O.B1_ASVGP else np.linalg.inv(Tn))
    ref = np.linalg.cholesky(0.5 * (S + S.T))
    got = OC.device_factor(family, Tn, Kn, r)
    assert np.allclose(np.triu(got, 1), 0.0)
    assert np.all(np.diag(got) > 0)
    assert _relerr(got, ref) <= 1e-12
    # a non-positive pivot is reported, not factored
    assert OC.ul_factor(np.zeros(4), np.zeros(4)) is None


# ---- the C ABI under the SIMT emulator ------------------------------------------------------------------------
@pytest.fixture(scope="module")
def emu():
    got = emul_lib.load()
    if got is None:
        pytest.skip("g++ not available")
    return got


LIBFAM = {O.B1_ASVGP: "B1_ASVGP", O.SVGP_GRID: "SVGP_MARKOV"}


def _plan(emu, family, meshes, dtype):
    lib, L = emu
    return emul_lib.EmuPlan(lib, L, getattr(L, LIBFAM[family]), [t.numpy() for t in meshes], dtype)


def _arrays(plan, X, y, l, s2, noise, m, Ls, dtype):
    theta = torch.cat([l, s2, noise.reshape(1)]).numpy().copy()
    Lcat = torch.cat([L.reshape(-1) for L in Ls]).numpy().copy()
    xs = [np.ascontiguousarray(X[:, d].numpy().astype(dtype)) for d in range(plan.D)]
    return theta, m.numpy().copy(), Lcat, xs, np.ascontiguousarray(y.numpy().astype(dtype))


def _update(plan, d, theta, m, Lcat, obs, L_out=None, gbuf=None):
    """forward at (theta, m, Lcat), data pass (unless a gbuf is given), covopt_update of dimension d"""
    plan.grid_forward(theta, m, Lcat)
    if gbuf is None:
        plan.obs_fwd_bwd(obs)
        gbuf = plan.gbuf
    out = Lcat if L_out is None else L_out
    change = np.zeros(1)
    plan.check(plan.lib.vggp_covopt_update(plan.h, d, emul_lib.ptr(gbuf), 1.0, emul_lib.ptr(Lcat), emul_lib.ptr(out),
                                           emul_lib.ptr(change), None))
    return change[0]


def _block(plan, Lcat, d):
    off = sum(n * n for n in plan.m_per_dim[:d])
    n = plan.m_per_dim[d]
    return Lcat[off:off + n * n].reshape(n, n)


@pytest.mark.parametrize("family", FAMILIES)
@pytest.mark.parametrize("knots,N,dtype,tol", [
    (knots, N, dtype, tol) for knots, N in [((11,), 400), ((8, 7), 600), ((6, 5, 4), 700)]
    for dtype, tol in [(np.float64, 1e-10), (np.float32, 1e-5)]] + [((300,), 2000, np.float64, 1e-10)])   # 300 > CO_THREADS rows
def test_emulated_update_matches_oracle(emu, family, knots, N, dtype, tol):
    meshes, X, y, l, s2, noise, m, Ls = _problem(family, knots, N, seed=23 + len(knots))
    assert bool((X < 0).any()) and bool((X > 1).any())            # observations outside the points on both sides
    tq = torch.float32 if dtype == np.float32 else torch.float64
    Xq, yq = X.to(tq).to(torch.float64), y.to(tq).to(torch.float64)
    plan = _plan(emu, family, meshes, dtype)
    theta, mm, Lcat, xs, yy = _arrays(plan, Xq, yq, l, s2, noise, m, Ls, dtype)
    obs = plan.bin(xs, yy, run_cap=16)
    for d in range(len(knots)):
        Lprev = [torch.from_numpy(_block(plan, Lcat, e).copy()) for e in range(len(knots))]
        ref = OC.update(family, meshes, Xq, l, s2, noise, Lprev, d)
        ch = _update(plan, d, theta, mm, Lcat, obs)
        got = _block(plan, Lcat, d)
        assert np.all(np.triu(got, 1) == 0.0)
        assert _relerr(got, ref) <= tol, (d, _relerr(got, ref))
        assert abs(ch - OC.change(ref, Lprev[d])) <= 1e-6 * max(ch, 1e-3)
    plan.close()


@pytest.mark.parametrize("family", FAMILIES)
@pytest.mark.parametrize("knots", [(9, 8), (6, 5, 4)])
def test_step_gradient_vanishes_after_update_and_shards_add_up(emu, family, knots):
    N = 800
    meshes, X, y, l, s2, noise, m, Ls = _problem(family, knots, N, seed=31 + len(knots))
    plan = _plan(emu, family, meshes, np.float64)
    theta, mm, Lcat, xs, yy = _arrays(plan, X, y, l, s2, noise, m, Ls, np.float64)
    obs = plan.bin(xs, yy, run_cap=16)
    # the update from the sum of two shards' gradient buffers equals the update from the full buffer
    half = N // 3
    shards = [plan.bin([x[:half] for x in xs], yy[:half], run_cap=16), plan.bin([x[half:] for x in xs], yy[half:], run_cap=16)]
    d = len(knots) - 1
    for e in range(d):
        _update(plan, e, theta, mm, Lcat, obs)
    dL0 = _block(plan, plan.step(theta, mm, Lcat, obs)[3], d).copy()
    L_full = Lcat.copy()
    _update(plan, d, theta, mm, L_full, obs)
    L_sh2 = Lcat.copy()
    _update(plan, d, theta, mm, L_sh2, None, gbuf=_sharded_gbuf(plan, theta, mm, Lcat, shards))
    assert _relerr(_block(plan, L_sh2, d), _block(plan, L_full, d)) <= 1e-12
    dL1 = _block(plan, plan.step(theta, mm, L_full, obs)[3], d)
    assert np.linalg.norm(np.tril(dL1)) <= 1e-9 * np.linalg.norm(np.tril(dL0)), (np.linalg.norm(dL1), np.linalg.norm(dL0))
    plan.close()


def _sharded_gbuf(plan, theta, m, Lcat, shards):
    plan.grid_forward(theta, m, Lcat)
    obs_bytes = plan.gbuf_obs_elems * plan.dtype.itemsize
    so = plan.gbuf_scalar_offset
    total = np.zeros_like(plan.gbuf)
    for sh in shards:
        plan.obs_fwd_bwd(sh)
        total[:obs_bytes].view(np.float64)[:] += plan.gbuf[:obs_bytes].view(np.float64)
        total[so:].view(np.float64)[:] += plan.gbuf[so:].view(np.float64)
    return total


@pytest.mark.parametrize("family", FAMILIES)
def test_aliasing_failed_pivot_and_refusals(emu, family):
    lib, Lmod = emu
    E_ARG, E_UNSUPPORTED = -1, -6
    knots = (8, 7)
    meshes, X, y, l, s2, noise, m, Ls = _problem(family, knots, 300, seed=41)
    plan = _plan(emu, family, meshes, np.float64)
    theta, mm, Lcat, xs, yy = _arrays(plan, X, y, l, s2, noise, m, Ls, np.float64)
    obs = plan.bin(xs, yy, run_cap=16)
    change = np.zeros(1)
    # no forward yet
    assert lib.vggp_covopt_update(plan.h, 0, emul_lib.ptr(plan.gbuf), 1.0, emul_lib.ptr(Lcat), emul_lib.ptr(Lcat),
                                  emul_lib.ptr(change), None) == E_ARG
    assert b"grid_forward" in lib.vggp_last_error()
    # separate output == in place; the other blocks of the output are untouched
    out = np.full_like(Lcat, 7.0)
    _update(plan, 1, theta, mm, Lcat, obs, L_out=out)
    inplace = Lcat.copy()
    plan.check(lib.vggp_covopt_update(plan.h, 1, emul_lib.ptr(plan.gbuf), 1.0, emul_lib.ptr(inplace), emul_lib.ptr(inplace),
                                      emul_lib.ptr(change), None))                   # same forward, same gradient buffer
    assert np.array_equal(_block(plan, out, 1), _block(plan, inplace, 1))
    assert np.all(_block(plan, out, 0) == 7.0)
    for bad in (-1, 2):
        assert lib.vggp_covopt_update(plan.h, bad, emul_lib.ptr(plan.gbuf), 1.0, emul_lib.ptr(Lcat), emul_lib.ptr(Lcat),
                                      emul_lib.ptr(change), None) == E_ARG
    assert lib.vggp_covopt_update(plan.h, 0, emul_lib.ptr(plan.gbuf), 1.0, None, emul_lib.ptr(Lcat),
                                  emul_lib.ptr(change), None) == E_ARG
    # L_0 = 0 and no data: T_1 = 0, the pivot fails, the flag is set and the output is left alone
    Lz = Lcat.copy()
    _block(plan, Lz, 0)[:] = 0.0
    empty = plan.bin([np.zeros(0) for _ in knots], np.zeros(0))
    before = Lz.copy()
    ch = _update(plan, 1, theta, mm, Lz, empty)
    assert plan.read_info() == 2 and ch == np.inf
    assert np.array_equal(Lz, before)
    plan.close()
    for fam, kn in ((Lmod.B0_GRIDDED, (5, 6)), (Lmod.SVGP_GRID, (5, 6)), (Lmod.VFF_GRID, (5, 7))):
        p = emul_lib.EmuPlan(lib, Lmod, fam, [np.linspace(0, 1, k, dtype=np.float32) for k in kn], np.float64)
        Lp = np.zeros(p.L_total)
        assert lib.vggp_covopt_update(p.h, 0, emul_lib.ptr(p.gbuf), 1.0, emul_lib.ptr(Lp), emul_lib.ptr(Lp),
                                      emul_lib.ptr(change), None) == E_UNSUPPORTED
        p.close()
