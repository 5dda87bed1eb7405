#!/usr/bin/env python
"""bench.py -- ELBO forward+backward throughput of the gridded variational GP hot path on B200.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl reference] [--dump-outputs DIR]
    python -m torch.distributed.run --nnodes=1 --nproc-per-node N ... bench.py --gpus N --steps K --warmup W

Workload (BASELINE.json configs[4], the configuration the metric is quoted on; it fits one GPU): 2-D
B1-spline ASVGP (GriddedMatern12ASVGP / Matern12B1SplineASVGP feature family), 512 x 512 grid of inducing
variables, N = 2^26 synthetic along-track observations in acquisition order, float32 observations, float64
grid side, full batch.  The observation axis is sharded over the ranks (total N fixed -> "strong" scaling); one
step = grid forward + fused per-observation forward/backward + one all-reduce + grid backward, i.e. the ELBO and
every gradient.  One JSON line is printed by rank 0.

`--impl reference` times the reference's CPU algorithm (the structured torch restatement in oracle/, the only
form of the reference's maths that can run at this size: SURVEY.md section 0 fact 5) on the host cores, on a
bounded sample of the same workload.
"""
import argparse
import json
import math
import os
import subprocess
import sys
import tempfile
import threading
import time

import numpy as np
import torch

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

METRIC = "elbo_fwd_bwd_observations_per_sec"
UNIT = "obs/s"
N_TOTAL = 1 << 26
KNOTS = (512, 512)
PASSES = 1024          # ascending passes; as many descending ones (SURVEY.md section 8d, config 3 geometry)
TRACK_GRADIENT = 2.0

# The headline line is `tracks512` (BASELINE.json configs[4], the configuration the metric is quoted on).  The other
# workloads are the remaining GPU configurations of BASELINE.json, run with --workload for the profiles / DESIGN.md tables.
WORKLOADS = {
    "tracks512": {"family": "B1_ASVGP", "knots": (512, 512), "n_total": 1 << 26,
                  "desc": "configs[4]: 2-D B1-spline ASVGP, 512x512 inducing grid, N=2^26 synthetic along-track "
                          "observations (acquisition order), fp32 observations / fp64 grid side, full batch"},
    "b1_cfg3": {"family": "B1_ASVGP", "knots": (512, 512), "n_total": 1 << 24,
                "desc": "configs[2]: 2-D B1-spline ASVGP (GriddedMatern12ASVGP), 512x512 grid, N=2^24 along-track observations, fp32"},
    "b0_cfg3": {"family": "B0_GRIDDED", "knots": (512, 512), "n_total": 1 << 24,
                "desc": "configs[2]: 2-D cell-integrated Matern-1/2 features (Matern12GriddedGP), 511x511 cells, N=2^24 "
                        "along-track observations, fp32 observations / fp64 grid side, scan form of the features"},
    "3d": {"family": "B1_ASVGP", "knots": (256, 256, 64), "n_total": 1 << 26,
           "desc": "configs[3]: 3-D (lon, lat, time) B1-spline ASVGP, 256x256x64 inducing grid, N=2^26 along-track observations "
                   "with time increasing along the acquisition order, fp32 observations / fp64 grid side"},
}


def workload_config(n_total, world, extra=None, workload="tracks512"):
    w = WORKLOADS[workload]
    D = len(w["knots"])
    cfg = {
        "workload": w["desc"], "workload_key": workload,
        "n_obs_total": n_total, "grid": list(w["knots"]), "family": w["family"], "obs_dtype": "float32",
        "sharding": f"observation axis, {world} contiguous shard(s), one all-reduce(sum) of the gradient buffer",
        "l2_policy": f"inputs larger than L2 ({n_total * (D + 1) * 4 / 1e6:.0f} MB of observations per step vs 126 MB L2); no explicit flush",
    }
    if extra:
        cfg.update(extra)
    return cfg


# ---------------------------------------------------------------------------------------------------------
# synthetic satellite-track-shaped data (geometry of src/utils/dataloaders.py:290-377 generate_track)
# ---------------------------------------------------------------------------------------------------------
def field(x1, x2):
    return (torch.sin(5 * x1) + torch.cos(7 * x2) + 0.5 * torch.sin(15 * x1) + 0.5 * torch.cos(12 * x2))


def _hash_uniform(idx, salt):
    """Counter-based uniform(0,1) from the global observation index (int64 LCG + xorshift mix, wrap-around
    arithmetic): the data set does not depend on how it is sharded over ranks."""
    def wrap(v):                              # Python int -> two's-complement int64
        v &= (1 << 64) - 1
        return v - (1 << 64) if v >= (1 << 63) else v
    h = idx * wrap(6364136223846793005) + wrap(1442695040888963407 + salt * 7046029254386353131)
    h = h ^ ((h >> 29) & ((1 << 35) - 1))     # logical shift
    h = h * wrap(0xBF58476D1CE4E5B9)
    h = h ^ ((h >> 32) & ((1 << 32) - 1))
    return ((h >> 11) & ((1 << 40) - 1)).to(torch.float64) / float(1 << 40)


def make_tracks(lo, hi, n_total, device, dtype, seed=0, D=2):
    """Observations lo..hi-1 (global acquisition order) of the synthetic track data set: generated by the library on the device
    (vggp_generate_tracks); the torch restatement below serves the CPU arm and the tests (bit-identical arithmetic)."""
    if torch.device(device).type == "cuda":
        import importlib
        import vggp_b200 as vg
        gen = importlib.import_module(vg.__name__ + ".utils.dataloaders")
        return gen.generate_tracks(lo, hi, n_total, device, dtype, seed=seed, D=D, passes=PASSES, trajectory_gradient=TRACK_GRADIENT)
    return make_tracks_torch(lo, hi, n_total, device, dtype, seed, D)


def make_tracks_torch(lo, hi, n_total, device, dtype, seed=0, D=2):
    """Observations lo..hi-1 (global acquisition order) of the synthetic track data set.  D = 3 adds the acquisition time
    as third coordinate (monotone along the concatenated passes, SURVEY.md section 8d config 4) and a slow drift of the
    field in time."""
    idx = torch.arange(lo, hi, device=device, dtype=torch.int64)
    per_pass = max(1, n_total // (2 * PASSES))
    j = torch.clamp(idx // per_pass, max=2 * PASSES - 1)
    k = idx - j * per_pass
    jitter = _hash_uniform(idx, 2 * seed + 1)
    t = ((k.to(torch.float64) + jitter) / float(per_pass)).clamp_(0.0, 1.0)       # monotone along a pass
    asc = j < PASSES
    off = (j % PASSES).to(torch.float64) / PASSES
    x1 = off + t / TRACK_GRADIENT
    x1 = x1 - torch.floor(x1)
    x2 = torch.where(asc, t, 1.0 - t)
    # noise: sum of 4 uniforms (Irwin-Hall), variance 4/12 -> scaled to sigma = 0.05
    u = sum(_hash_uniform(idx, 2 * seed + 10 + q) for q in range(4)) - 2.0
    y = field(x1, x2) + 0.05 * math.sqrt(3.0) * u
    if D == 3:
        x3 = ((idx.to(torch.float64) + _hash_uniform(idx, 2 * seed + 31)) / float(n_total)).clamp_(0.0, 1.0)
        y = y + 0.3 * torch.sin(4.0 * x3) * torch.cos(3.0 * x1)
        return [x1.to(dtype).contiguous(), x2.to(dtype).contiguous(), x3.to(dtype).contiguous()], y.to(dtype).contiguous()
    return [x1.to(dtype).contiguous(), x2.to(dtype).contiguous()], y.to(dtype).contiguous()


def b1_factor(mesh, l, s2):
    """Per-dimension RKHS Gram factor of the B1/ASVGP family, (l A + B / l + BC) / (2 s2)
    (gridded_kronecker_structure.py:731-780), float64, from the float32 knot spacing."""
    n = mesh.numel()
    d = (mesh[1] - mesh[0]).to(torch.float64)
    A = torch.zeros(n, n, dtype=torch.float64)
    B = torch.zeros(n, n, dtype=torch.float64)
    i = torch.arange(n)
    A[i, i] = 2.0 / 3.0 * d
    B[i, i] = 2.0 / d
    A[i[:-1], i[:-1] + 1] = A[i[:-1] + 1, i[:-1]] = d / 6.0
    B[i[:-1], i[:-1] + 1] = B[i[:-1] + 1, i[:-1]] = -1.0 / d
    for e in (0, n - 1):
        A[e, e] -= d / 3.0
        B[e, e] -= 1.0 / d
    BC = torch.zeros(n, n, dtype=torch.float64)
    BC[0, 0] = BC[n - 1, n - 1] = 1.0
    return (A * l + B / l + BC) / (2.0 * s2)


def b0_factor(mesh, l, s2):
    """Cov of the B0 cell integrals of a Matern-1/2 process along one dimension (gridded_kronecker_structure.py:1286-1323),
    float64 throughout (only used to place the variational parameters of the bench)."""
    m = mesh.numel() - 1
    d = (mesh[1] - mesh[0]).to(torch.float64)
    k = torch.arange(m, dtype=torch.float64)
    row = torch.exp(-(k - 1) * d / l) + torch.exp(-(k + 1) * d / l) - 2 * torch.exp(-k * d / l)
    row[0] = 2 * (torch.exp(-d / l) + d / l - 1)
    i = torch.arange(m)
    return row[(i[:, None] - i[None, :]).abs()] * (l * l * s2)


def make_params(meshes, device, seed=1, family="B1_ASVGP"):
    """A sensible point of the optimisation: theta as non_informative_initialise(lmbda=5, kappa=10) would set it,
    m = Kuu f0 (so that the predictive mean interpolates the field f0 at the knots / cell centres) plus noise, and
    L_d = chol(K_d) (I/2 + small random lower-triangular matrix) (q(u) between prior and posterior)."""
    g = torch.Generator().manual_seed(seed)
    D = len(meshes)
    l = torch.full((D,), 0.2887 / 5.0, dtype=torch.float64)
    s2 = torch.full((D,), 1.2, dtype=torch.float64)
    noise = torch.tensor([1.2 / 100.0], dtype=torch.float64)
    theta = torch.cat([l, s2, noise])
    if family == "B1_ASVGP":
        Ks = [b1_factor(meshes[d], l[d], s2[d]) for d in range(D)]
        pts = [m.to(torch.float64) for m in meshes]
    else:
        Ks = [b0_factor(meshes[d], l[d], s2[d]) for d in range(D)]
        pts = [0.5 * (m[1:] + m[:-1]).to(torch.float64) for m in meshes]
    grids = torch.meshgrid(*pts, indexing="ij")
    f0 = field(grids[0], grids[1] if D > 1 else grids[0])     # smooth: its RKHS norm (the <m, alpha> term of the KL) stays moderate
    mt = f0
    for d in range(D):
        mt = torch.movedim(torch.tensordot(Ks[d], mt, dims=([1], [d])), 0, d)
    m = mt.reshape(-1).contiguous()
    Ls = []
    for K in Ks:
        C = torch.linalg.cholesky(K)
        n = K.shape[0]
        G = 0.5 * torch.eye(n, dtype=torch.float64) + 0.05 * torch.tril(torch.randn(n, n, generator=g, dtype=torch.float64)) / math.sqrt(n)
        Ls.append(C @ G)          # S_d = C G G^T C^T: a whitened perturbation of K_d / 4
    return theta, m, Ls


# ---------------------------------------------------------------------------------------------------------
class ClockSampler:
    """nvidia-smi clocks / throttle reasons sampled while the timed region runs."""
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap,utilization.gpu")

    def __init__(self, gpu_index):
        self.gpu = gpu_index
        self.proc = None
        self.path = None

    def start(self):
        try:
            fd, self.path = tempfile.mkstemp(suffix=".csv")
            os.close(fd)
            self.f = open(self.path, "w")
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.gpu), f"--query-gpu={self.Q}",
                                          "--format=csv,noheader,nounits", "-lms", "20"],
                                         stdout=self.f, stderr=subprocess.DEVNULL)
        except Exception:
            self.proc = None

    def n_samples(self):
        try:
            self.f.flush()
            return sum(1 for _ in open(self.path))
        except Exception:
            return 0

    def stop(self):
        out = {"sm_mhz": None, "sm_max_mhz": None, "reasons": [], "samples": 0}
        if self.proc is None:
            return out
        try:
            self.proc.terminate()
            self.proc.wait(timeout=5)
            self.f.close()
            rows = [r.strip().split(",") for r in open(self.path) if r.strip()]
            sm, mx = [], []
            reasons = set()
            names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
            loaded = []
            for r in rows:
                r = [c.strip() for c in r]
                try:
                    if len(r) > 9 and float(r[9]) >= 50.0:
                        loaded.append(r)
                except Exception:
                    pass
            use = loaded if loaded else [[c.strip() for c in r] for r in rows]
            for r in use:
                try:
                    sm.append(float(r[1]))
                    mx.append(float(r[2]))
                except Exception:
                    continue
                for name, val in zip(names, r[5:9]):
                    if val.lower().startswith("active"):
                        reasons.add(name)
            if sm:
                sm.sort()
                out = {"sm_mhz": sm[len(sm) // 2], "sm_max_mhz": max(mx), "reasons": sorted(reasons), "samples": len(sm)}
        except Exception:
            pass
        finally:
            try:
                os.unlink(self.path)
            except Exception:
                pass
        return out


def k1_traffic(layout, run_cap):
    """DRAM bytes per launch of the per-observation kernel from the committed ncu --set full capture of the SAME kernel
    and configuration (profiles/r2_k1_traffic.json lists layout, run_cap and n_obs it was taken on); None otherwise."""
    try:
        with open(os.path.join(ROOT, "profiles", "r2_k1_traffic.json")) as f:
            rec = json.load(f)
        if rec.get("layout") == layout and int(rec.get("run_cap", -1)) == int(run_cap) and int(rec.get("n_obs", -1)) == N_TOTAL:
            return float(rec["traffic"])
    except Exception:
        pass
    return None


def dmma_peak():
    """FP64 tensor-pipe peak measured on a B200 of this pool by tools/microbench/dmma_peak.cu (pure mma.sync.m8n8k4.f64 on
    register operands); MEASURED_PEAKS.json has no FP64 entry and the profiling recipe states no fallback for it."""
    try:
        with open(os.path.join(ROOT, "profiles", "r2_dmma_peak.json")) as f:
            return float(json.load(f)["dmma_f64_tflops"]), "measured (profiles/r2_dmma_peak.json, tools/microbench/dmma_peak.cu)"
    except Exception:
        return None, "unmeasured"


def tensor_roofline(vg, plan, device, reps=20):
    """The Kronecker mode-n products of the dense grid side (B0 family: alpha = (P_1 x P_2) m and its reverse), timed alone
    through vggp_mode_product = k_gemm_group (4-stage cp.async pipeline, mma.sync.m8n8k4.f64): FLOPs = 2 M M_d per product."""
    M = plan.M
    src = torch.randn(M, dtype=torch.float64, device=device)
    per_dim, flops, ms_tot = [], 0.0, 0.0
    for d, n in enumerate(plan.m_per_dim):
        A = plan.workspace(vg._lib.WS_P, d).clone()
        for _ in range(3):
            plan.mode_product(d, A, src)
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        torch.cuda.synchronize()
        a.record()
        for _ in range(reps):
            plan.mode_product(d, A, src)
        b.record()
        torch.cuda.synchronize()
        ms = a.elapsed_time(b) / reps
        f = 2.0 * M * n
        per_dim.append({"mode": d, "m_d": n, "ms": ms, "tflops": f / (ms * 1e-3) / 1e12})
        flops += f
        ms_tot += ms
    peak, src_txt = dmma_peak()
    achieved = flops / (ms_tot * 1e-3) / 1e12
    # The same kernel on a batch of 64 independent products of the same size in ONE launch: a 511^3 product alone is 7 us of
    # DMMA work behind ~ 15 us of launch, destination clear (k-split), pipeline fill and drain, so it measures latency; the
    # batch measures the kernel's rate (ncu: profiles/r2_ncu_summary_gemm_steady.txt, DMMA pipe 85 % active at 4096 x 4096 x 1024).
    nb, n0 = 64, plan.m_per_dim[0]
    Ab = torch.randn(nb, n0, n0, dtype=torch.float64, device=device)
    Bb = torch.randn(nb, n0, n0, dtype=torch.float64, device=device)
    Cb = torch.zeros(nb, n0, n0, dtype=torch.float64, device=device)
    for _ in range(3):
        vg.gemm_f64(Ab, Bb, C_in=Cb)
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    torch.cuda.synchronize()
    a.record()
    for _ in range(reps):
        vg.gemm_f64(Ab, Bb, C_in=Cb)
    b.record()
    torch.cuda.synchronize()
    ms_b = a.elapsed_time(b) / reps
    tf_b = 2.0 * nb * n0 ** 3 / (ms_b * 1e-3) / 1e12
    steady = {"batch": nb, "m_d": n0, "ms": ms_b, "tflops": tf_b, "frac": (tf_b / peak) if peak else None,
              "what": "one launch of k_gemm_one over a batch of %d independent %d^3 products" % (nb, n0)}
    return {"bound": "tensor", "kernel": "k_gemm_group (Kronecker mode-n products T x_d P_d, mma.sync.m8n8k4.f64 = DMMA)",
            "achieved": achieved, "peak": peak, "unit": "TFLOP/s", "frac": (achieved / peak) if peak else None,
            "steady_state": steady,
            "peak_source": src_txt, "flops": flops, "per_mode": per_dim,
            "timing": "CUDA events around %d back-to-back launches per mode on the current stream, after 3 warm-up launches" % reps,
            "note": "FP64 only: the grid side needs float64 (cond(K_d) ~ 1e7) and tcgen05 has no f64 kind, so the tensor "
                    "instruction is the warp-level DMMA"}


DUMP_NAMES = ("out", "dtheta", "dm", "dL")       # what plan.step returns; out = [ELBO, scaled log-likelihood, KL, n]
DUMP_LIMIT = 64 << 20


def dump_outputs(path, tensors):
    """Write the arrays of one step as <path>/<name>.npy (float64), so that two builds can be compared output for output:
    the data and the parameters are functions of the arguments alone (make_tracks, make_params)."""
    arrays = {name: t.numpy() for name, t in zip(DUMP_NAMES, tensors)}
    total = sum(a.nbytes for a in arrays.values())
    if total > DUMP_LIMIT:
        raise SystemExit(f"--dump-outputs: {total} bytes of outputs exceed the {DUMP_LIMIT}-byte limit")
    os.makedirs(path, exist_ok=True)
    for name, a in arrays.items():
        np.save(os.path.join(path, name + ".npy"), a)


def measured_peaks():
    path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    try:
        with open(path) as f:
            p = json.load(f)
        return float(p["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
    except Exception:
        return 6650.0, "fallback (B200_PROFILING.md 6.65 TB/s)"


# ---------------------------------------------------------------------------------------------------------
# CPU baseline: the oracle's structured ELBO (float32 per-observation arithmetic) + autograd on the host cores
# ---------------------------------------------------------------------------------------------------------
def cpu_oracle_step_fn(n_sample, seed=0, workload="tracks512"):
    from oracle import vggp_oracle as O
    w = WORKLOADS[workload]
    meshes = [torch.linspace(0, 1, k) for k in w["knots"]]
    D = len(meshes)
    xs, y = make_tracks(0, n_sample, n_sample, torch.device("cpu"), torch.float32, seed, D=D)
    X = torch.stack(xs, dim=1).to(torch.float64)
    y = y.to(torch.float64)
    theta, m, Ls = make_params(meshes, "cpu", family=w["family"])
    ofam = O.B1_ASVGP if w["family"] == "B1_ASVGP" else O.B0_GRIDDED

    def step():
        l = theta[:D].clone().requires_grad_(True)
        s2 = theta[D:2 * D].clone().requires_grad_(True)
        nz = theta[2 * D].clone().requires_grad_(True)
        mm = m.clone().requires_grad_(True)
        LL = [L.clone().requires_grad_(True) for L in Ls]
        elbo = O.elbo_structured(ofam, meshes, X, y, l, s2, nz, mm, LL, ref_quirks=False,
                                 work_dtype=torch.float32)
        torch.autograd.grad(elbo, [l, s2, nz, mm] + LL)
        return float(elbo.detach())

    return step


def _calib_n(workload):
    """First sample size of the CPU legs: the dense-feature (B0) oracle costs O(N M_d^2), the stencil one O(N)."""
    return 1 << (12 if WORKLOADS[workload]["family"] != "B1_ASVGP" else 17)


def time_cpu_baseline(budget_s=20.0, steps=3, warmup=1, n_cap=1 << 22, workload="tracks512"):
    cores = os.cpu_count() or 1
    torch.set_num_threads(cores)
    n = _calib_n(workload)
    step = cpu_oracle_step_fn(n, workload=workload)
    step()
    t0 = time.perf_counter()
    step()
    dt = time.perf_counter() - t0
    # grid-side cost is constant; scale the sample so that (steps + warmup) runs fit the budget
    scale = max(1.0, budget_s / max(dt * (steps + warmup), 1e-3))
    n_sample = int(min(n_cap, max(n, (1 << int(math.log2(n * scale))))))
    if n_sample != n:
        step = cpu_oracle_step_fn(n_sample, workload=workload)
    for _ in range(warmup):
        step()
    t0 = time.perf_counter()
    for _ in range(steps):
        step()
    dt = (time.perf_counter() - t0) / steps
    grid = "x".join(str(k) for k in WORKLOADS[workload]["knots"])
    return {"value": n_sample / dt, "unit": UNIT, "cores": int(torch.get_num_threads()), "kind": "port",
            "sample": f"{n_sample} observations of the same track workload on the full {grid} grid, fp32 "
                      f"per-observation arithmetic, {steps} timed fwd+bwd steps after {warmup} warm-up "
                      f"({dt * 1e3:.1f} ms/step), torch CPU + autograd",
            "ms_per_step": dt * 1e3, "n_sample": n_sample}


def run_reference_arm(args, rank, world):
    if rank != 0:
        return
    cores = os.cpu_count() or 1
    torch.set_num_threads(cores)
    # bounded sample: calibrate on a small sample, then size the sample so the whole run ends in ~2 minutes
    workload = args.workload
    n = _calib_n(workload)
    step = cpu_oracle_step_fn(n, workload=workload)
    step()
    t0 = time.perf_counter()
    step()
    dt = time.perf_counter() - t0
    total = args.steps + args.warmup
    scale = max(1.0, 120.0 / max(dt * total, 1e-3))
    n_sample = int(min(1 << 22, max(n, 1 << int(math.log2(n * scale)))))
    if n_sample != n:
        step = cpu_oracle_step_fn(n_sample, workload=workload)
    for _ in range(args.warmup):
        step()
    t0 = time.perf_counter()
    for _ in range(args.steps):
        step()
    dt = (time.perf_counter() - t0) / max(1, args.steps)
    value = n_sample / dt
    line = {
        "impl": "reference", "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": args.gpus, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": dt * 1e3, "higher_is_better": True, "scaling": "strong",
        "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": workload_config(WORKLOADS[workload]["n_total"], world, {"cpu_sample_obs": n_sample}, workload),
        "cpu_baseline": {"value": value, "unit": UNIT, "cores": int(torch.get_num_threads()), "kind": "port",
                         "sample": f"{n_sample} observations per step (bounded sample of the workload), full "
                                   f"grid, structured torch-CPU restatement of the reference maths + autograd"},
        "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line), flush=True)


# ---------------------------------------------------------------------------------------------------------
def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--workload", default="tracks512", choices=sorted(WORKLOADS),
                    help="tracks512 = BASELINE.json configs[4] (the headline); b1_cfg3 / b0_cfg3 = configs[2]; 3d = configs[3]")
    ap.add_argument("--n-obs", type=int, default=None, help="total observations over all ranks (default: the workload's)")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--deterministic", action="store_true",
                    help="vggp_set_deterministic: bitwise reproducible steps (B1 family, binned layout); reports its cost")
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--obs-layout", default="binned", choices=["packed", "binned"],
                    help="layout the fused per-observation kernel streams: 'binned' = k_obs_b1_binned (per-cell runs in "
                         "warp tasks, default since round 2); 'packed' = k_obs_b1 (round-1 kernel, cross-check)")
    ap.add_argument("--run-cap", type=int, default=256,
                    help="binned layout: longest run of one cell (0 = automatic, smaller caps for thin shards: measured equal to "
                         "256 at 2 x B200, profiles/r2_s3/multi2/run_cap.txt)")
    ap.add_argument("--binned-stream", default="ldg", choices=["ldg", "tma"],
                    help="binned layout: 16-byte global loads into registers, or a per-warp shared-memory ring "
                         "filled by TMA bulk copies (vggp_set_binned_stream)")
    ap.add_argument("--cuda-graph", dest="cuda_graph", action="store_true", default=True,
                    help="replay the step from CUDA graphs (default; an NCCL all-reduce stays outside the graphs, the "
                         "library's own collective is captured with the rest)")
    ap.add_argument("--no-cuda-graph", dest="cuda_graph", action="store_false",
                    help="launch the ~8 kernels of a step eagerly (three C calls per step)")
    ap.add_argument("--allreduce", default="auto", choices=["auto", "nccl", "peer"],
                    help="the one collective of a sharded step: NCCL, or the library's own one-kernel all-reduce over NVLink "
                         "peer memory (vggp_allreduce_gbuf: in-switch multimem reduction; captured into the step's CUDA graph). "
                         "auto = peer from 4 ranks up (measured on 8 x B200: 0.118 vs 0.149 ms per step), NCCL for 2 ranks "
                         "(0.173 vs 0.186 ms) and whenever peer memory cannot be set up")
    ap.add_argument("--reshard-balance", default="count", choices=["count", "cells"],
                    help="--spatial-reshard: cut the cell ranges at observation-count quantiles (default) or evenly")
    ap.add_argument("--spatial-reshard", action="store_true",
                    help="multi-GPU: exchange the acquisition-order shards by grid-cell range at setup "
                         "(dist.spatial_reshard; measured slower at 8 x B200 in round 1, off by default)")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="after the timed steps, write what the last timed step returned (ELBO terms, dtheta, dm, dL) "
                         "as DIR/<name>.npy in float64")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "b200":
        ap.error("--dump-outputs writes the outputs of the CUDA path (--impl b200)")
    args.warmup = max(args.warmup, 3) if args.impl == "b200" else args.warmup

    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))

    if args.impl == "reference":
        run_reference_arm(args, rank, world)
        return

    import vggp_b200 as vg
    import torch.distributed as dist
    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device (there is no CPU path); use --impl reference for the CPU arm")
    torch.cuda.set_device(local_rank)
    device = torch.device("cuda", local_rank)
    if world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        dist.init_process_group("nccl", rank=rank, world_size=world, device_id=device)
    lib = vg._lib.load()

    wl = WORKLOADS[args.workload]
    knots, fam_name = wl["knots"], wl["family"]
    n_total = int(args.n_obs) if args.n_obs else wl["n_total"]
    lo, hi = vg.shard_bounds(n_total, rank, world)
    n_local = hi - lo
    dtype = torch.float32
    meshes = [torch.linspace(0, 1, k) for k in knots]
    is_b1 = fam_name == "B1_ASVGP"
    if not is_b1:
        args.obs_layout = "binned"          # the B0 family streams per-cell runs too (scan form); there is no packed layout for it
    plan = vg.GridPlan(vg.B1_ASVGP if is_b1 else vg.B0_GRIDDED, meshes, dtype, device)
    multicast = None
    if args.allreduce == "auto":
        args.allreduce = "peer" if world >= 4 else "nccl"
        if world >= 4:
            try:
                multicast = plan.enable_peer_allreduce()
            except Exception as exc:          # no peer access / symmetric memory: every rank fails alike
                if rank == 0:
                    print(f"peer-memory all-reduce unavailable ({exc}); using NCCL", file=sys.stderr)
                args.allreduce = "nccl"
    elif world > 1 and args.allreduce == "peer":
        multicast = plan.enable_peer_allreduce()
    xs, y = make_tracks(lo, hi, n_total, device, dtype, D=len(knots))
    sharding = "contiguous in acquisition order"
    if world > 1 and args.spatial_reshard:
        # one-time setup exchange: every rank ends up owning a contiguous range of grid cells (dist.spatial_reshard)
        keys = plan.cell_keys(xs)
        xs, y = vg.spatial_reshard(xs, y, keys, plan.n_cells, balance=args.reshard_balance)
        n_local = int(y.numel())
        sharding = "by grid-cell range (one-time all-to-all of the acquisition-order shards at setup)"
        del keys
    # one-time setup (X is constant over optimisation steps): bin the observations by grid cell and store them
    # in the packed layout the fused kernel streams; the acquisition-order packing is timed as a second leg
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    if args.obs_layout == "binned":
        lib.vggp_set_binned_stream(1 if args.binned_stream == "tma" else 0)
        packed = plan.bin(xs, y, run_cap=args.run_cap)
    else:
        packed = plan.pack(xs, y, sort_by_cell=True)
    if args.deterministic:
        plan.set_deterministic(True)
    torch.cuda.synchronize()
    setup_ms = (time.perf_counter() - t0) * 1e3
    theta, m, Ls = make_params(meshes, device, family=fam_name)
    theta_d = theta.to(device)
    m_d = m.to(device)
    L_d = torch.cat([L.reshape(-1) for L in Ls]).to(device).contiguous()
    group = "world" if world > 1 else None
    ev_a = [torch.cuda.Event(enable_timing=True) for _ in range(args.steps)]
    ev_b = [torch.cuda.Event(enable_timing=True) for _ in range(args.steps)]

    def step(i=None, obs=None):
        plan.grid_forward(theta_d, m_d, L_d)
        if i is not None:
            ev_a[i].record()
        if isinstance(obs, tuple):
            plan.obs_fwd_bwd(obs[0], obs[1])          # plain arrays in the order given (the e2e leg: what was just copied in)
        else:
            plan.obs_fwd_bwd(packed if obs is None else obs)
        if i is not None:
            ev_b[i].record()
        if group is not None:
            plan.allreduce_gbuf(None)
        return plan.grid_backward(theta_d, m_d, L_d, 1.0)

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    graphed = None
    launches_per_step = None
    plain_step = step
    if args.cuda_graph:
        c0 = lib.vggp_launch_count()
        step()
        launches_per_step = lib.vggp_launch_count() - c0      # kernels of this library in one step (replayed by the graphs)
        graphed = plan.graphed_step(theta_d, m_d, L_d, packed, None, 1.0, group)
        # an instrumented twin of the same step for the roofline: captured with the library's timing on, it holds two event-record
        # nodes around the per-observation kernel (they cost ~10 us per replay, so the timed region replays the clean graph)
        plan.k1_timing(True)
        graphed_timed = plan.graphed_step(theta_d, m_d, L_d, packed, None, 1.0, group, warmup=1)
        plan.k1_timing(False)

        def step(i=None, obs=None):          # noqa: F811  (the graphs hold the cell-sorted observations)
            if obs is not None:
                return plain_step(i, obs)
            return graphed.replay()

    sampler = ClockSampler(local_rank)
    if rank == 0:
        sampler.start()
    for _ in range(args.warmup):
        out = step()
    barrier()
    if plan.read_info() != 0:
        raise SystemExit("factorisation failed in the bench configuration")
    # the timed region can be shorter than one nvidia-smi sampling period: keep the identical step loop running
    # (untimed) until the sampler has produced a few samples under load, then go straight into the timed steps
    extra_warm = 0
    t_w = time.perf_counter()
    flag = torch.zeros(1, dtype=torch.int32, device=device)
    while True:
        if rank == 0:
            flag.fill_(1 if (sampler.n_samples() >= 6 or time.perf_counter() - t_w > 3.0) else 0)
        if world > 1:
            dist.broadcast(flag, 0)
        if int(flag.item()) == 1:
            break
        for _ in range(20):
            out = step()
        extra_warm += 20
        torch.cuda.synchronize()
    launches0 = lib.vggp_launch_count()
    barrier()
    if graphed is None:
        plan.k1_timing(True)          # the library brackets the per-observation kernel itself with CUDA events
    t_start = torch.cuda.Event(enable_timing=True)
    t_end = torch.cuda.Event(enable_timing=True)
    t_start.record()
    for i in range(args.steps):
        out = step(i)
    t_end.record()
    barrier()
    dumped = [t.cpu() for t in out] if (args.dump_outputs and rank == 0) else None
    launches = lib.vggp_launch_count() - launches0
    if plan.peer_allreduce_failed():
        raise SystemExit("a barrier of the peer-memory all-reduce timed out (a rank went missing)")
    if graphed is not None:
        launches = launches_per_step * args.steps
    clocks = sampler.stop() if rank == 0 else None
    ms_total = t_start.elapsed_time(t_end)
    if graphed is not None:
        # The instrumented twin graph holds two external event-record nodes around the per-observation kernel; every replay
        # re-records the same pair, so each sample is one replay of the whole step followed by the read (a synchronisation).
        samples = []
        for _ in range(args.steps):
            graphed_timed.replay()
            samples.append(plan.k1_graph_time_read())
        k1_kernel_ms, k1_launches = sum(samples) / len(samples), len(samples)
        # the whole C call (memset + kernel + band-replica reduction) cannot be bracketed inside the graph: eager loop
        torch.cuda.synchronize()
        for i in range(args.steps):
            ev_a[i].record()
            plan.obs_fwd_bwd(packed)
            ev_b[i].record()
        torch.cuda.synchronize()
    else:
        k1_kernel_ms, k1_launches = plan.k1_time_read()       # the kernel alone (events inside the C call, same stream)
        plan.k1_timing(False)
    k1_call_ms = sum(a.elapsed_time(b) for a, b in zip(ev_a, ev_b)) / args.steps   # whole vggp_obs_fwd_bwd* call
    tt = torch.tensor([ms_total, k1_kernel_ms, k1_call_ms, float(n_local)], dtype=torch.float64, device=device)
    if world > 1:
        dist.all_reduce(tt, op=dist.ReduceOp.MAX)
    ms_step = tt[0].item() / args.steps
    k1_ms = tt[1].item()
    k1_call_ms = tt[2].item()
    n_local_max = int(tt[3].item())        # the roofline pairs the slowest rank's kernel time with the largest shard
    value = n_total / (ms_step * 1e-3)

    # ---- secondary leg: same step on observations left in acquisition (along-track) order (B1 family: the packed kernel
    # takes any order; the B0 scan form needs per-cell runs)
    acq_ms = None
    if is_b1 and not args.deterministic:       # deterministic mode takes the binned layout only
        packed_acq = plan.pack(xs, y, sort_by_cell=False)
        for _ in range(2):
            step(None, packed_acq)
        barrier()
        a0, a1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        acq_steps = max(3, min(args.steps, 10))
        a0.record()
        for _ in range(acq_steps):
            step(None, packed_acq)
        a1.record()
        barrier()
        ta = torch.tensor([a0.elapsed_time(a1) / acq_steps], dtype=torch.float64, device=device)
        if world > 1:
            dist.all_reduce(ta, op=dist.ReduceOp.MAX)
        acq_ms = ta.item()
        del packed_acq

    # ---- end-to-end leg: host buffers, H2D of the step's inputs and D2H of its results inside the timed region
    e2e = None
    if not args.no_e2e and not args.deterministic:      # vggp_elbo_host streams plain arrays: not a deterministic-mode path
        xs_h = [x.cpu().pin_memory() for x in xs]
        y_h = y.cpu().pin_memory()
        th_h, m_h, L_h = theta.pin_memory(), m.pin_memory(), torch.cat([L.reshape(-1) for L in Ls]).pin_memory()
        D = len(meshes)
        out_h = torch.empty(4, dtype=torch.float64).pin_memory()
        dth_h = torch.empty(2 * D + 1, dtype=torch.float64).pin_memory()
        dm_h = torch.empty(plan.M, dtype=torch.float64).pin_memory()
        dL_h = torch.empty(plan.L_total, dtype=torch.float64).pin_memory()
        h2d = sum(t.numel() * t.element_size() for t in xs_h + [y_h, th_h, m_h, L_h])
        d2h = sum(t.numel() * t.element_size() for t in (out_h, dth_h, dm_h, dL_h))
        import ctypes as C
        stream = torch.cuda.current_stream(device).cuda_stream

        def e2e_step():
            if not is_b1:
                # B0 family: host observations -> device, per-cell runs (sort + gather: the scan form needs them), step
                for dst, src in zip(xs + [y], xs_h + [y_h]):
                    dst.copy_(src, non_blocking=True)
                theta_d.copy_(th_h, non_blocking=True)
                m_d.copy_(m_h, non_blocking=True)
                L_d.copy_(L_h, non_blocking=True)
                o, dth, dm, dL = step(None, plan.bin(xs, y, run_cap=args.run_cap))
                out_h.copy_(o, non_blocking=True)
                dth_h.copy_(dth, non_blocking=True)
                dm_h.copy_(dm, non_blocking=True)
                dL_h.copy_(dL, non_blocking=True)
                torch.cuda.synchronize()
            elif world == 1:
                ptrs = (C.c_void_p * D)(*[t.data_ptr() for t in xs_h])
                vg._lib.check(lib.vggp_elbo_host(plan.handle, ptrs, y_h.data_ptr(), n_local, th_h.data_ptr(),
                                                 m_h.data_ptr(), L_h.data_ptr(), 1.0, out_h.data_ptr(),
                                                 dth_h.data_ptr(), dm_h.data_ptr(), dL_h.data_ptr(), stream))
            else:
                for dst, src in zip(xs + [y], xs_h + [y_h]):
                    dst.copy_(src, non_blocking=True)
                theta_d.copy_(th_h, non_blocking=True)
                m_d.copy_(m_h, non_blocking=True)
                L_d.copy_(L_h, non_blocking=True)
                o, dth, dm, dL = plain_step(None, (xs, y))          # the step consumes the arrays that were just copied in
                out_h.copy_(o, non_blocking=True)
                dth_h.copy_(dth, non_blocking=True)
                dm_h.copy_(dm, non_blocking=True)
                dL_h.copy_(dL, non_blocking=True)
                torch.cuda.synchronize()

        e2e_steps = max(3, min(args.steps, 10))
        for _ in range(2):
            e2e_step()
        barrier()
        t0 = time.perf_counter()
        for _ in range(e2e_steps):
            e2e_step()
        barrier()
        dt = (time.perf_counter() - t0) / e2e_steps
        te = torch.tensor([dt], dtype=torch.float64, device=device)
        if world > 1:
            dist.all_reduce(te, op=dist.ReduceOp.MAX)
        e2e = {"value": n_total / te.item(), "unit": UNIT, "h2d_bytes_per_step": int(h2d), "d2h_bytes_per_step": int(d2h),
               "ms_per_step": te.item() * 1e3, "steps": e2e_steps,
               "path": "vggp_elbo_host (C ABI, pinned host buffers)" if (world == 1 and is_b1) else
                       "pinned host -> device copies" + ("" if is_b1 else " + vggp_obs_bin_* (per-cell runs)")
                       + " + plan.step + device -> host of ELBO and gradients"}

    if rank == 0:
        peak, peak_src = measured_peaks()
        alg_bytes = n_local_max * (len(knots) + 1) * 4 + 2 * plan.M * 4
        achieved = alg_bytes / (k1_ms * 1e-3) / 1e9
        line = {
            "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
            "ms_per_step": ms_step, "higher_is_better": True, "scaling": "strong", "vs_baseline": None,
            "dtype": "f32", "data": "synthetic",
            "config": workload_config(n_total, world, {
                "n_obs_per_gpu": n_local_max, "observation_sharding": sharding,
                **({"run_len": packed.run_len,
                    "layout": "observations binned by grid cell + warp-transposed packing, done once at setup "
                              "(X is constant over optimisation steps); setup is outside the timed region"}
                   if args.obs_layout == "packed" else
                   {"deterministic": bool(args.deterministic), "binned_stream": args.binned_stream, "run_cap": packed.run_cap, "n_runs": packed.n_runs,
                    "n_tasks": packed.n_tasks,
                    "streamed_bytes": packed.streamed_bytes,
                    "layout": "per-cell runs, 32 equally long runs per warp task (vggp_obs_bin_pack), done once at "
                              "setup; setup is outside the timed region"}),
                "setup_ms": setup_ms, "cuda_graph": bool(args.cuda_graph),
                "allreduce": (None if world == 1 else
                              ("NCCL" if args.allreduce == "nccl" else
                               "vggp_allreduce_gbuf (one kernel over NVLink peer memory, %s)"
                               % ("multimem in-switch reduction" if multicast else "two-shot P2P loads/stores"))),
                "acquisition_order": ({"ms_per_step": acq_ms, "value": n_total / (acq_ms * 1e-3),
                                       "note": "same step without the cell binning (along-track order kept)"}
                                      if acq_ms is not None else None)}, args.workload),
            "elbo": out[0][0].item(),
            "roofline": {"bound": "hbm", "kernel": (("k_obs_b1" if args.obs_layout == "packed" else "k_obs_b1_binned") if is_b1
                                                    else "k_obs_b0s") + " (fused per-observation ELBO forward+backward)",
                         "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak,
                         "traffic": (k1_traffic(args.obs_layout, packed.run_cap if args.obs_layout == "binned" else args.run_cap)
                                     if (world == 1 and args.workload == "tracks512" and n_total == N_TOTAL) else None),
                         "peak_source": peak_src, "kernel_ms": k1_ms, "kernel_launches_timed": k1_launches,
                         "timing": ("CUDA events recorded by the library immediately around the kernel launch, on the "
                                    "launching stream, inside the timed region (vggp_k1_timing)" if graphed is None else
                                    "CUDA events recorded by event-record nodes immediately around the kernel inside a replayed "
                                    "graph of the whole step (vggp_k1_graph_time_read): %d replays, right after the timed region, "
                                    "of a twin of the timed graph that differs only by the two event nodes (they cost ~10 us "
                                    "per replay, hence the twin)" % k1_launches),
                         "call_ms": k1_call_ms,
                         "call_note": "whole vggp_obs_fwd_bwd* call: gradient-buffer memset + kernel + band-replica reduction",
                         "algorithmic_bytes": alg_bytes,
                         "share_of_step": k1_ms / ms_step},
            "gpu_launches": int(launches),
            "clocks": dict(clocks, window="sampled every 20 ms over the last warm-up steps and the timed region "
                                          "(identical step loop; %d extra untimed steps)" % extra_warm),
        }
        if not is_b1:
            line["tensor_roofline"] = tensor_roofline(vg, plan, device)
        if e2e is not None:
            line["e2e"] = e2e
        if not args.no_cpu_baseline and world == 1:
            line["cpu_baseline"] = time_cpu_baseline(workload=args.workload)
        if dumped is not None:
            dump_outputs(args.dump_outputs, dumped)
        print(json.dumps(line), flush=True)
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
