"""No GPU needed: the sampling law of the epoch-shuffled minibatches (csrc/minibatch.cuh) restated in numpy, and the whole
epoch binning (vggp_epoch_bin_prepare / _pack / vggp_epoch_batch: key kernel, radix sorts, device run planner, table and
gather kernels) under the SIMT emulator, batch by batch against vggp_obs_bin_pack of the same observations."""
import ctypes as C

import numpy as np
import pytest

import emul_lib

M32 = 0xFFFFFFFF
ROUNDS = 4


def _mix32(x):
    x = np.asarray(x, dtype=np.uint64) & M32
    x ^= x >> np.uint64(16)
    x = (x * np.uint64(0x7FEB352D)) & np.uint64(M32)
    x ^= x >> np.uint64(15)
    x = (x * np.uint64(0x846CA68B)) & np.uint64(M32)
    x ^= x >> np.uint64(16)
    return x


def permutation(n, seed, epoch, rank):
    """pi(i) for i = 0..n-1: balanced Feistel network on the smallest even k >= 2 with 2^k >= n, 4 rounds of a 32-bit mixing
    hash of (seed, epoch, rank, round, half), cycle-walking below n."""
    k = 2
    while (1 << k) < n:
        k += 2
    half = np.uint64(k // 2)
    mask = np.uint64((1 << (k // 2)) - 1)
    h = _mix32(seed & M32)
    h = _mix32(h ^ np.uint64(seed >> 32))
    h = _mix32(h ^ np.uint64(epoch & M32))
    h = _mix32(h ^ np.uint64(epoch >> 32))
    h = _mix32(h ^ np.uint64(rank))
    keys = [_mix32(h ^ np.uint64(((r + 1) * 0x9E3779B9) & M32)) for r in range(ROUNDS)]
    v = np.arange(n, dtype=np.uint64)
    todo = np.ones(n, dtype=bool)
    while todo.any():
        w = v[todo]
        L, R = w >> half, w & mask
        for kr in keys:
            L, R = R, L ^ (_mix32(kr ^ R) & mask)
        v[todo] = (L << half) | R
        todo = v >= n
    return v.astype(np.int64)


def epoch_batches(n, B, seed, epoch, rank=0, n_batches=0):
    """The index sets of the P batches of one epoch, each in ascending order."""
    P = n_batches or n // B
    b = permutation(n, seed, epoch, rank) // B
    order = np.argsort(b, kind="stable")
    return [order[i * B:(i + 1) * B] for i in range(P)] if P else []


@pytest.mark.parametrize("n", [1, 2, 3, 4, 5, 15, 16, 17, 63, 64, 65, 1000, 4097, 65537, 1 << 18])
def test_permutation_is_a_bijection(n):
    for seed, epoch, rank in ((0, 0, 0), (7, 3, 1), (2 ** 40 + 5, 2 ** 33 + 1, 5)):
        q = permutation(n, seed, epoch, rank)
        assert q.min() >= 0 and q.max() < n
        assert np.array_equal(np.sort(q), np.arange(n))


def test_permutation_depends_on_every_key():
    n = 5000
    base = permutation(n, 1, 2, 0)
    for other in (permutation(n, 2, 2, 0), permutation(n, 1, 3, 0), permutation(n, 1, 2, 1), permutation(n, 1 + 2 ** 32, 2, 0)):
        assert (other != base).mean() > 0.9
    # a batch is a fair sample: its mean index is near n / 2
    for bset in epoch_batches(n, 1000, 11, 0):
        assert abs(bset.mean() - n / 2) < 0.1 * n


@pytest.fixture(scope="module")
def emu():
    got = emul_lib.load()
    if got is None:
        pytest.skip("g++ not available")
    return got


def _epoch(plan, xs, y, B, seed, epoch, run_cap, rank=0, n_batches=0):
    lib, L = plan.lib, plan.L
    n = y.size
    P = n_batches or n // B
    desc = L.EpochDesc()
    tot = np.zeros(max(1, L.EPOCH_TOTALS * P), dtype=np.int64)
    tptr = tot.ctypes.data_as(C.POINTER(C.c_int64))
    plan.check(lib.vggp_epoch_bin_prepare(plan.h, plan._xptrs(xs), n, B, n_batches, run_cap, seed, epoch, rank, C.byref(desc),
                                          tptr, None))
    raw = np.full(int(desc.bytes) + 256, 0xAB, dtype=np.uint8)
    off = (-raw.ctypes.data) % 256
    buf = raw[off:off + int(desc.bytes)]
    plan.check(lib.vggp_epoch_bin_pack(plan.h, C.byref(desc), tptr, plan._xptrs(xs), emul_lib.ptr(y), emul_lib.ptr(buf), None))
    views = []
    for b in range(P):
        bd, vo = L.BinnedDesc(), C.c_int64()
        plan.check(lib.vggp_epoch_batch(C.byref(desc), tptr, b, C.byref(bd), C.byref(vo)))
        views.append((bd, buf[int(vo.value):]))
    return desc, views, raw


def _sections(bd, buf, dtype):
    T = int(bd.n_tasks)

    def sec(off, n, dt):
        return buf[int(off):int(off) + n * np.dtype(dt).itemsize].view(dt)
    return {"header": buf[:256].copy(), "task_off": sec(bd.off_task_off, T, np.int64), "task_R": sec(bd.off_task_R, T, np.int32),
            "run_cell": sec(bd.off_run_cell, 32 * T, np.uint32), "run_n": sec(bd.off_run_n, 32 * T, np.int32),
            "run_start": sec(bd.off_run_start, 32 * T, np.uint32), "data": sec(bd.off_data, int(bd.data_elems), dtype)}


def assert_batch_equals_bin(plan, bd, vbuf, xs, y, idx, run_cap, dtype):
    """Batch view == vggp_obs_bin_pack of x[idx], y[idx], section by section, bitwise (data NaN-aware)."""
    sub = [np.ascontiguousarray(x[idx]) for x in xs]
    ref = plan.bin(sub, np.ascontiguousarray(y[idx]), run_cap)
    rd, rbuf = ref[2], ref[1]
    for f in ("n", "n_inside", "n_tasks", "n_runs", "data_elems", "run_cap", "D"):
        assert getattr(bd, f) == getattr(rd, f), f
    got, want = _sections(bd, vbuf, dtype), _sections(rd, rbuf, dtype)
    for k in want:
        a, b = got[k], want[k]
        if k == "data":
            a, b = a.view(np.uint32 if dtype == np.float32 else np.uint64), b.view(np.uint32 if dtype == np.float32 else np.uint64)
        assert np.array_equal(a, b), k


FAMILIES = [("b1", 0, 1), ("b1", 0, 2), ("b1", 0, 3), ("markov", 4, 1), ("markov", 4, 2), ("markov", 4, 3), ("b0", 1, 1),
            ("b0", 1, 2)]
KNOTS = {1: (9,), 2: (6, 5), 3: (4, 5, 3)}


def _data(D, n, rng, dtype, case):
    X = rng.uniform(-0.15, 1.15, size=(n, D))                    # some observations outside the mesh
    if case == "overflow":
        X[: n // 2] = 0.31                                        # one cell holds half the data: several runs of it
    elif case == "sparse":
        X = rng.uniform(0.0, 1.0, size=(n, D))
    return [np.ascontiguousarray(X[:, d], dtype=dtype) for d in range(D)], rng.standard_normal(n).astype(dtype)


@pytest.mark.parametrize("dtype", [np.float32, np.float64])
@pytest.mark.parametrize("name,family,D", FAMILIES)
def test_epoch_layout_identity(emu, name, family, D, dtype):
    lib, L = emu
    rng = np.random.default_rng(100 * family + D)
    meshes = [np.linspace(0, 1, k, dtype=np.float32) for k in KNOTS[D]]
    plan = emul_lib.EmuPlan(lib, L, family, meshes, dtype)
    try:
        # (n, B, run_cap, case): remainder dropped, a cell overflowing run_cap, B = n, B = 1, a fine mesh with one
        # observation per cell (every run padded from 1 to 4)
        cases = [(203, 40, 8, "mixed"), (160, 80, 4, "overflow"), (37, 37, 16, "mixed"), (9, 1, 4, "mixed")]
        for n, B, cap, case in cases:
            xs, y = _data(D, n, rng, dtype, case)
            for seed, epoch in ((3, 0), (3, 1)):
                desc, views, _ = _epoch(plan, xs, y, B, seed, epoch, cap)
                sets = epoch_batches(n, B, seed, epoch)
                assert desc.n_batches == len(sets) == n // B
                for (bd, vbuf), idx in zip(views, sets):
                    assert_batch_equals_bin(plan, bd, vbuf, xs, y, idx, cap, dtype)
    finally:
        plan.close()
    if D == 1:
        fine = emul_lib.EmuPlan(lib, L, family, [np.linspace(0, 1, 401, dtype=np.float32)], dtype)
        try:
            x = np.ascontiguousarray((np.arange(300) + 0.5) / 400.0, dtype=dtype)[rng.permutation(300)]
            y = rng.standard_normal(300).astype(dtype)
            _, views, _ = _epoch(fine, [x], y, 100, 9, 4, 32)
            for (bd, vbuf), idx in zip(views, epoch_batches(300, 100, 9, 4)):
                assert bd.n_runs == 100
                assert_batch_equals_bin(fine, bd, vbuf, [x], y, idx, 32, dtype)
        finally:
            fine.close()


def test_epoch_planner_random_cell_counts(emu):
    """Random per-cell counts (many cells empty, a few far above run_cap) in every batch: the device planner against plan_bins."""
    lib, L = emu
    rng = np.random.default_rng(5)
    meshes = [np.linspace(0, 1, 13, dtype=np.float32), np.linspace(0, 1, 7, dtype=np.float32)]
    plan = emul_lib.EmuPlan(lib, L, 0, meshes, np.float64)
    try:
        centres = np.array([(a + 0.5) / 12 for a in range(12)])
        for trial in range(3):
            w = rng.pareto(1.0, size=12 * 6) * (rng.random(12 * 6) < 0.5)
            w = w / w.sum()
            n = 1500
            cell = rng.choice(12 * 6, size=n, p=w)
            x0 = centres[cell // 6] + rng.uniform(-0.03, 0.03, n)
            x1 = (cell % 6 + 0.5) / 6 + rng.uniform(-0.05, 0.05, n)
            xs = [np.ascontiguousarray(x0), np.ascontiguousarray(x1)]
            y = rng.standard_normal(n)
            B, cap = [(500, 12), (300, 20), (1500, 8)][trial]
            _, views, _ = _epoch(plan, xs, y, B, 17, trial, cap)
            for (bd, vbuf), idx in zip(views, epoch_batches(n, B, 17, trial)):
                assert_batch_equals_bin(plan, bd, vbuf, xs, y, idx, cap, np.float64)
    finally:
        plan.close()


def test_epoch_rank_and_batch_count(emu):
    """A rank key gives its own permutation; n_batches below n / B draws that many batches of the same law."""
    lib, L = emu
    rng = np.random.default_rng(8)
    plan = emul_lib.EmuPlan(lib, L, 4, [np.linspace(0, 1, 6, dtype=np.float32)] * 2, np.float64)
    try:
        xs, y = _data(2, 150, rng, np.float64, "mixed")
        desc, views, _ = _epoch(plan, xs, y, 30, 5, 2, 8, rank=3, n_batches=2)
        sets = epoch_batches(150, 30, 5, 2, rank=3, n_batches=2)
        assert desc.n_batches == 2 and len(views) == 2
        for (bd, vbuf), idx in zip(views, sets):
            assert_batch_equals_bin(plan, bd, vbuf, xs, y, idx, 8, np.float64)
    finally:
        plan.close()


def test_epoch_refusals(emu):
    lib, L = emu
    rng = np.random.default_rng(1)
    desc = L.EpochDesc()
    tot = np.zeros(64, dtype=np.int64)
    tptr = tot.ctypes.data_as(C.POINTER(C.c_int64))
    for family, knots in ((L.SVGP_GRID, (5, 6)), (L.VFF_GRID, (5, 7)), (L.B0_GRIDDED, (5, 6, 4))):
        meshes = [np.linspace(0, 1, k, dtype=np.float32) for k in knots]
        plan = emul_lib.EmuPlan(lib, L, family, meshes, np.float64)
        xs, y = _data(len(knots), 20, rng, np.float64, "mixed")
        assert lib.vggp_epoch_bin_prepare(plan.h, plan._xptrs(xs), 20, 5, 0, 8, 0, 0, 0, C.byref(desc), tptr, None) == -6
        plan.close()
    plan = emul_lib.EmuPlan(lib, L, L.B1_ASVGP, [np.linspace(0, 1, 5, dtype=np.float32)], np.float64)
    xs, y = _data(1, 20, rng, np.float64, "mixed")
    for n, B, P in ((20, 0, 0), (20, 21, 0), (1 << 31, 5, 0), (20, 5, 5), (0, 1, 0)):
        assert lib.vggp_epoch_bin_prepare(plan.h, plan._xptrs(xs), n, B, P, 8, 0, 0, 0, C.byref(desc), tptr, None) == -1
    # a pack needs its own prepare, with the descriptor it returned
    buf = np.zeros(1 << 16, dtype=np.uint8)
    assert lib.vggp_epoch_bin_pack(plan.h, C.byref(desc), tptr, plan._xptrs(xs), emul_lib.ptr(y), emul_lib.ptr(buf), None) == -1
    assert lib.vggp_epoch_bin_prepare(plan.h, plan._xptrs(xs), 20, 5, 0, 8, 0, 0, 0, C.byref(desc), tptr, None) == 0
    bad = L.EpochDesc.from_buffer_copy(desc)
    bad.epoch = 1
    assert lib.vggp_epoch_bin_pack(plan.h, C.byref(bad), tptr, plan._xptrs(xs), emul_lib.ptr(y), emul_lib.ptr(buf), None) == -1
    bd, vo = L.BinnedDesc(), C.c_int64()
    assert lib.vggp_epoch_batch(C.byref(desc), tptr, 4, C.byref(bd), C.byref(vo)) == -1
    assert lib.vggp_epoch_batch(C.byref(desc), tptr, 3, C.byref(bd), C.byref(vo)) == 0 and vo.value == 3 * 256
    plan.close()
