"""Product-grid SVGP in its O(1)-per-observation Markov form (family SVGP_MARKOV, csrc/svgpm.cuh), without a GPU:
  * the Markov oracle (oracle/svgp_markov.py) equals the dense SVGP statement of the same model (vggp_oracle, pinned to the
    reference's class through tests/golden) in float64, over non-uniform points, observations on both sides outside them,
    h / l from 1e-3 to 30 and D = 1, 2, 3;
  * the whole C ABI of the family under the SIMT emulator (tests/host_emul): ELBO, d theta, d m, d L and predictions
    against the Markov oracle, shard sums, an empty shard, observations all outside the points, and the refusals."""
import ctypes as C

import numpy as np
import pytest
import torch

import emul_lib
from oracle import svgp_markov as SM
from oracle import vggp_oracle as O
from test_gpu_elbo import make_problem, oracle_value_and_grads


def _problem(knots, N, seed, lscale=1.0):
    meshes, X, y, l, s2, noise, m, Ls = make_problem(knots, N, seed=seed, family=O.SVGP_GRID, x_lo=-0.3, x_hi=1.3)
    meshes = [(t ** (1.0 + 0.3 * d)).to(torch.float32) for d, t in enumerate(meshes)]    # strictly increasing, non-uniform
    return meshes, X.contiguous(), y, l * lscale, s2, noise, m, Ls


def _relerr(a, b):
    a = torch.as_tensor(np.asarray(a), dtype=torch.float64).reshape(-1)
    b = b.detach().to(torch.float64).reshape(-1)
    return float((a - b).norm() / b.norm().clamp_min(1e-300))


# (knots, N, lengthscale factor, tolerance): l in [0.2, 0.6] times the factor against point spacings of ~0.01 .. 0.2 spans
# h / l from ~1e-3 (l >> h, the normal regime) to ~30.  At h / l ~ 1e-3 the dense reference itself loses digits: its Cholesky
# of K_d (condition ~ M_d l / h) and the cancellation in s2 - k^T K^-1 k leave ~1e-9 of relative error in the ELBO.
ORACLE_CASES = [((11,), 400, 1.0, 1e-10), ((11,), 400, 300.0, 1e-8), ((11,), 400, 30.0, 1e-8), ((11,), 400, 0.02, 1e-10),
                ((8, 7), 400, 1.0, 1e-10), ((8, 7), 400, 60.0, 1e-8), ((8, 7), 400, 0.015, 1e-10),
                ((6, 5, 4), 400, 1.0, 1e-10), ((6, 5, 4), 400, 40.0, 1e-8), ((6, 5, 4), 400, 0.02, 1e-10)]


@pytest.mark.parametrize("knots,N,lscale,tol", ORACLE_CASES)
def test_markov_oracle_equals_dense_svgp_oracle(knots, N, lscale, tol):
    meshes, X, y, l, s2, noise, m, Ls = _problem(knots, N, seed=3 + len(knots), lscale=lscale)
    assert bool((X < 0).any()) and bool((X > 1).any())
    ref, gref = oracle_value_and_grads(O.SVGP_GRID, meshes, X, y, l, s2, noise, m, Ls, scale=1.3)
    val, g = SM.value_and_grads(meshes, X, y, l, s2, noise, m, Ls, scale=1.3)
    assert abs(float(val - ref)) <= tol * abs(float(ref))
    for a, b in zip(g, gref):
        assert float((a - b).norm()) <= tol * max(float(b.norm()), 1e-300)


def test_markov_oracle_predictions_equal_dense():
    meshes, X, y, l, s2, noise, m, Ls = _problem((8, 7), 300, seed=9)
    mu, var = SM.predict(meshes, X, l, s2, m, Ls)
    Kuu, Kuf, _, _ = O.dense_Kuu_Kuf(O.SVGP_GRID, meshes, X, l, s2, False)
    B = torch.linalg.solve(Kuu, Kuf)
    S = O.kron_cov_from_factors(Ls)
    mu_ref = B.T @ m
    var_ref = torch.prod(s2) - (Kuf * B).sum(0) + (B * (S @ B)).sum(0)
    assert float((mu - mu_ref).abs().max()) < 1e-10
    assert float((var - var_ref).abs().max()) < 1e-10


# ---- the C ABI under the SIMT emulator ------------------------------------------------------------------------
@pytest.fixture(scope="module")
def emu():
    got = emul_lib.load()
    if got is None:
        pytest.skip("g++ not available")
    return got


def _inputs(plan, X, y, l, s2, noise, m, Ls, dtype):
    theta = torch.cat([l, s2, noise.reshape(1)]).numpy().copy()
    Lcat = torch.cat([L.reshape(-1) for L in Ls]).numpy().copy()
    xs = [np.ascontiguousarray(X[:, d].numpy().astype(dtype)) for d in range(plan.D)]
    return theta, m.numpy().copy(), Lcat, xs, np.ascontiguousarray(y.numpy().astype(dtype))


def _check(plan, res, ref, gref, N, tol):
    out, dtheta, dm, dL = res
    D = plan.D
    assert plan.read_info() == 0
    assert out[3] == N
    assert abs(out[0] - float(ref)) <= tol * abs(float(ref)), (out, ref)
    assert _relerr(dtheta[:D], gref[0]) < tol * 10, ("dl", dtheta[:D], gref[0])
    assert _relerr(dtheta[D:2 * D], gref[1]) < tol * 10, ("ds2", dtheta[D:2 * D], gref[1])
    assert _relerr(dtheta[2 * D:], gref[2]) < tol * 10, "dnoise"
    assert _relerr(dm, gref[3]) < tol * 10, "dm"
    off = 0
    for d, n in enumerate(plan.m_per_dim):
        dLd = dL[off:off + n * n].reshape(n, n)
        off += n * n
        assert np.count_nonzero(np.triu(dLd, 1)) == 0
        assert _relerr(np.tril(dLd), torch.tril(gref[4 + d])) < tol * 10, ("dL", d)


EMU_CASES = [((11,), 500), ((8, 7), 600), ((6, 5, 4), 700)]


@pytest.mark.parametrize("knots,N", EMU_CASES)
@pytest.mark.parametrize("dtype,tol", [(np.float64, 1e-8), (np.float32, 1e-3)])
def test_markov_step_matches_oracle_under_emulation(emu, knots, N, dtype, tol):
    lib, L = emu
    meshes, X, y, l, s2, noise, m, Ls = _problem(knots, N, seed=21 + len(knots))
    Xq = X.to(torch.float32 if dtype == np.float32 else torch.float64).to(torch.float64)
    yq = y.to(torch.float32 if dtype == np.float32 else torch.float64).to(torch.float64)
    ref, gref = SM.value_and_grads(meshes, Xq, yq, l, s2, noise, m, Ls, scale=1.2)
    plan = emul_lib.EmuPlan(lib, L, L.SVGP_MARKOV, [t.numpy() for t in meshes], dtype)
    assert plan.m_per_dim == list(knots)
    theta, mm, Lcat, xs, yy = _inputs(plan, Xq, yq, l, s2, noise, m, Ls, dtype)
    obs = plan.bin(xs, yy, run_cap=16)
    assert obs[2].n_inside == N                 # extended cells: every observation is streamed
    _check(plan, plan.step(theta, mm, Lcat, obs, None, 1.2), ref, gref, N, tol)
    # predictions (vggp_predict) and the fused metrics (vggp_predict_metrics) from the same forward
    mean, var = plan.predict(xs)
    mu_ref, var_ref = SM.predict(meshes, Xq, l, s2, m, Ls)
    ptol = 1e-10 if dtype == np.float64 else 2e-5
    assert np.max(np.abs(mean - mu_ref.numpy())) <= ptol * 10
    assert np.max(np.abs(var - var_ref.numpy())) <= ptol * 10
    met = plan.predict_metrics(xs, yy)
    assert abs(met[0] - float(((yq - mu_ref) ** 2).sum())) <= 1e-3 * float(((yq - mu_ref) ** 2).sum())
    # the dense features are the SVGP family's k_d(Z, x)
    phi = plan.features_dense(0, xs[0], theta)
    fref = O.svgp_features_dense(meshes[0], Xq[:, 0], l[0], s2[0]).numpy()
    assert np.max(np.abs(phi - fref)) <= (1e-13 if dtype == np.float64 else 1e-6) * np.max(np.abs(fref))
    plan.close()


@pytest.mark.parametrize("knots", [(8, 7), (6, 5, 4)])
def test_markov_shard_gbufs_sum_to_full_batch(emu, knots):
    lib, L = emu
    N = 600
    meshes, X, y, l, s2, noise, m, Ls = _problem(knots, N, seed=5)
    plan = emul_lib.EmuPlan(lib, L, L.SVGP_MARKOV, [t.numpy() for t in meshes], np.float64)
    theta, mm, Lcat, xs, yy = _inputs(plan, X, y, l, s2, noise, m, Ls, np.float64)
    plan.grid_forward(theta, mm, Lcat)
    plan.obs_fwd_bwd(plan.bin(xs, yy))
    full = plan.gbuf.copy()
    obs_f, sc_f = full[:plan.gbuf_scalar_offset].view(np.float64), full[plan.gbuf_scalar_offset:].view(np.float64)
    acc_o, acc_s = np.zeros_like(obs_f), np.zeros_like(sc_f)
    for lo, hi in ((0, 250), (250, 251), (251, 251), (251, N)):
        plan.obs_fwd_bwd(plan.bin([x[lo:hi].copy() for x in xs], yy[lo:hi].copy()))
        acc_o += plan.gbuf[:plan.gbuf_scalar_offset].view(np.float64)
        acc_s += plan.gbuf[plan.gbuf_scalar_offset:].view(np.float64)
    assert np.allclose(acc_o, obs_f, rtol=1e-12, atol=1e-12)
    assert np.allclose(acc_s, sc_f, rtol=1e-12, atol=1e-12)
    plan.close()


def test_markov_empty_shard_and_all_outside(emu):
    lib, L = emu
    knots, N = (8, 7), 300
    meshes, X, y, l, s2, noise, m, Ls = _problem(knots, N, seed=6)
    # every observation outside the points in at least one dimension, on both sides
    X[:, 0] = torch.where(torch.arange(N) % 2 == 0, -0.5 - X[:, 0].abs(), 1.5 + X[:, 0].abs())
    plan = emul_lib.EmuPlan(lib, L, L.SVGP_MARKOV, [t.numpy() for t in meshes], np.float64)
    theta, mm, Lcat, xs, yy = _inputs(plan, X, y, l, s2, noise, m, Ls, np.float64)
    ref, gref = SM.value_and_grads(meshes, X, y, l, s2, noise, m, Ls)
    _check(plan, plan.step(theta, mm, Lcat, plan.bin(xs, yy), None, 1.0), ref, gref, N, 1e-8)
    # empty shard: ELL is zero, the ELBO is -KL
    empty = [np.zeros(0) for _ in range(2)]
    out, dtheta, dm, dL = plan.step(theta, mm, Lcat, plan.bin(empty, np.zeros(0)), None, 1.0)
    ref0, gref0 = SM.value_and_grads(meshes, X[:0], y[:0], l, s2, noise, m, Ls)
    assert out[3] == 0 and abs(out[0] - float(ref0)) <= 1e-9 * abs(float(ref0))
    assert _relerr(dm, gref0[3]) < 1e-8
    plan.close()


def test_markov_refusals(emu):
    lib, L = emu
    meshes, X, y, l, s2, noise, m, Ls = _problem((8, 7), 50, seed=7)
    plan = emul_lib.EmuPlan(lib, L, L.SVGP_MARKOV, [t.numpy() for t in meshes], np.float64)
    theta, mm, Lcat, xs, yy = _inputs(plan, X, y, l, s2, noise, m, Ls, np.float64)
    plan.grid_forward(theta, mm, Lcat)
    E = -6                                                   # VGGP_E_UNSUPPORTED
    xp = (C.c_void_p * 2)(*[x.ctypes.data for x in xs])
    assert lib.vggp_obs_fwd_bwd(plan.h, xp, yy.ctypes.data, yy.size, plan.gbuf.ctypes.data, None) == E
    assert lib.vggp_obs_fwd_bwd_packed(plan.h, xp, yy.ctypes.data, yy.size, plan.gbuf.ctypes.data, None) == E
    outs = [np.zeros(k) for k in (4, 5, plan.M, plan.L_total)]
    assert lib.vggp_elbo_host(plan.h, xp, yy.ctypes.data, yy.size, theta.ctypes.data, mm.ctypes.data, Lcat.ctypes.data, 1.0,
                              *[o.ctypes.data for o in outs], None) == E
    assert b"binned layout" in lib.vggp_last_error()
    assert lib.vggp_set_deterministic(plan.h, 1) == E
    ptr, n = C.c_void_p(), C.c_int64()
    assert lib.vggp_workspace_ptr(plan.h, L.WS_P, 0, C.byref(ptr), C.byref(n)) == E
    assert lib.vggp_set_deterministic(plan.h, 0) == 0
    plan.close()
