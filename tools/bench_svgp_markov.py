"""Benchmark of the product-grid SVGP family in its O(1)-per-observation Markov form (SVGP_MARKOV, csrc/svgpm.cuh).  Prints
one JSON line; also writes it to --out if given.

  headline  N = 2^26 track observations (vggp_generate_tracks), float32, Z = 512 x 512 linspace(0, 1) points, CUDA-graph replay:
            step ms and obs/s, the per-observation kernel (vggp_k1_graph_time_read) and its share of the project's measured HBM
            peak (6552.6 GB/s, VERDICT.md row "K1 roofline"; bytes = the binned stream the kernel reads), grid forward + backward ms
  dense     the dense-feature SVGP_GRID step against the Markov step on the same inputs (32 x 32 Z, N = 2^20, eager steps)
  3d        Z = 256 x 256 x 64, N = 2^26 track observations (D = 3), CUDA-graph replay
The card's name and power limit are read in the same run (nvidia-smi query)."""
import argparse
import importlib
import json
import os
import subprocess
import sys

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
HBM_PEAK_GBS = 6552.6


def gpu_info():
    try:
        q = subprocess.run(["nvidia-smi", "-i", "0", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                           capture_output=True, text=True, timeout=30).stdout.strip()
    except Exception as e:          # the name from torch is still recorded
        q = f"nvidia-smi unavailable: {e}"
    return {"gpu": torch.cuda.get_device_name(0), "nvidia_smi": q}


def params(knots, dev, seed=0):
    g = torch.Generator().manual_seed(seed)
    D = len(knots)
    M = 1
    for k in knots:
        M *= k
    theta = torch.cat([torch.full((D,), 0.3, dtype=torch.float64), torch.full((D,), 0.8, dtype=torch.float64),
                       torch.tensor([0.05], dtype=torch.float64)]).to(dev)
    m = (0.1 * torch.randn(M, generator=g, dtype=torch.float64)).to(dev)
    L = torch.cat([(0.5 * torch.eye(k, dtype=torch.float64)).reshape(-1) for k in knots]).to(dev)
    return theta, m, L


def timed(fn, iters):
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record()
    for _ in range(iters):
        fn()
    b.record()
    b.synchronize()
    return a.elapsed_time(b) / iters


def graph_run(vg, gen, knots, n, dev, steps, warmup):
    D = len(knots)
    meshes = [torch.linspace(0, 1, k) for k in knots]
    xs, y = gen.generate_tracks(0, n, n, dev, torch.float32, seed=0, D=D)
    plan = vg.GridPlan(vg.SVGP_MARKOV, meshes, torch.float32, dev)
    obs = plan.bin(xs, y)
    del xs, y
    theta, m, L = params(knots, dev)
    plan.k1_timing(True)
    gs = plan.graphed_step(theta, m, L, obs, warmup=warmup)
    for _ in range(warmup):
        gs.replay()
    step_ms = timed(gs.replay, steps)
    k1 = []
    for _ in range(min(steps, 20)):
        gs.replay()
        k1.append(plan.k1_graph_time_read())
    k1.sort()
    k1_ms = k1[len(k1) // 2]
    # grid side alone: forward + backward on the gbuf of the last step
    def grid():
        plan.grid_forward(theta, m, L)
        plan.grid_backward(theta, m, L, 1.0)
    for _ in range(warmup):
        grid()
    grid_ms = timed(grid, steps)
    out = gs.replay()[0].cpu().tolist()
    bytes_k1 = obs.streamed_bytes
    return {"knots": list(knots), "n": n, "step_ms": step_ms, "obs_per_s": n / (step_ms * 1e-3), "k1_ms": k1_ms,
            "k1_bytes": bytes_k1, "k1_gbs": bytes_k1 / (k1_ms * 1e-3) / 1e9,
            "k1_hbm_fraction": bytes_k1 / (k1_ms * 1e-3) / 1e9 / HBM_PEAK_GBS, "grid_fwd_bwd_ms": grid_ms,
            "elbo": out[0], "plan_bytes": plan.workspace_bytes()}


def dense_vs_markov(vg, gen, dev, steps, warmup, knots=(32, 32), n=1 << 20):
    meshes = [torch.linspace(0, 1, k) for k in knots]
    xs, y = gen.generate_tracks(0, n, n, dev, torch.float32, seed=0, D=2)
    theta, m, L = params(knots, dev)
    res = {"knots": list(knots), "n": n}
    for name, fam in (("dense", vg.SVGP_GRID), ("markov", vg.SVGP_MARKOV)):
        plan = vg.GridPlan(fam, meshes, torch.float32, dev)
        obs, yy = (plan.bin(xs, y), None) if fam == vg.SVGP_MARKOV else (xs, y)
        step = lambda: plan.step(theta, m, L, obs, yy)        # noqa: E731
        for _ in range(warmup):
            step()
        res[name + "_step_ms"] = timed(step, steps)
        res[name + "_elbo"] = plan.step(theta, m, L, obs, yy)[0][0].item()
    res["speedup"] = res["dense_step_ms"] / res["markov_step_ms"]
    return res


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--steps", type=int, default=50)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--n", type=int, default=1 << 26)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("bench_svgp_markov needs a CUDA device")
    vg = importlib.import_module("variational-gridded-gaussian-processes_b200")
    gen = importlib.import_module("variational-gridded-gaussian-processes_b200.utils.dataloaders")
    dev = torch.device("cuda", 0)
    rec = {"bench": "svgp_markov", **gpu_info()}
    rec["headline"] = graph_run(vg, gen, (512, 512), args.n, dev, args.steps, args.warmup)
    torch.cuda.empty_cache()
    rec["dense_vs_markov"] = dense_vs_markov(vg, gen, dev, max(5, args.steps // 5), 2)
    torch.cuda.empty_cache()
    rec["3d"] = graph_run(vg, gen, (256, 256, 64), args.n, dev, args.steps, args.warmup)
    line = json.dumps(rec)
    print(line)
    if args.out:
        with open(args.out, "w") as f:
            f.write(line + "\n")


if __name__ == "__main__":
    main()
