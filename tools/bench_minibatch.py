"""Benchmark of the epoch-shuffled binned minibatches (GridPlan.bin_epoch, csrc/minibatch.cuh).  Prints one JSON line per
(workload, batch size); also appends them to --out if given.

Workloads: float32 track observations (vggp_generate_tracks): N = 2^26 on 512 x 512 points for B1 and Markov SVGP, N = 2^26 on
256 x 256 x 64 points for B1 and Markov SVGP, N = 2^24 on 511 x 511 cells for B0 (BASELINE.json configs[2]); theta of
tools/bench_svgp_markov.py.  Batch sizes B = 2^18, 2^20, 2^22, 2^24.  Per line, device events after warm-up, the paths
alternated within every repetition:
  bin_full_ms       GridPlan.bin of all N observations (prepare + pack, both synchronise)
  bin_epoch_ms      GridPlan.bin_epoch: all P = N / B batches of one epoch
  step_ms           one eager step (grid forward, per-observation kernel, grid backward) on a batch, mean over the epoch
  graph_step_ms     replay of a graph captured on one batch
  index_step_ms     B1 and B0: _elbo(batch=idx)'s path at the same B, i.e. the torch gather x[idx], y[idx] plus the plain-array
                    step (B1: raw per-observation kernel, B0: dense-feature kernel); idx drawn before the timed window
  k1_batch_ms       the per-observation kernel on one batch (the library's own events, vggp_k1_timing), against
  k1_full_scaled_ms B / N times its time on the full data
The card's name and power limit are read in the same run."""
import argparse
import importlib
import json
import os
import sys

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tools"))
import bench_svgp_markov as BS        # noqa: E402  (gpu_info, params)


def ev_ms(fn):
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record()
    fn()
    b.record()
    b.synchronize()
    return a.elapsed_time(b)


def median(v):
    v = sorted(v)
    return v[len(v) // 2]


def workload(vg, gen, name, family, knots, n, batch_sizes, dev, args):
    D = len(knots)
    meshes = [torch.linspace(0, 1, k) for k in knots]
    xs, y = gen.generate_tracks(0, n, n, dev, torch.float32, seed=0, D=D)
    plan = vg.GridPlan(family, meshes, torch.float32, dev)
    mk = list(plan.m_per_dim)
    theta, m, L = BS.params(mk, dev)
    fam = {vg.B1_ASVGP: "B1", vg.B0_GRIDDED: "B0", vg.SVGP_MARKOV: "SVGP_MARKOV"}[family]
    full = plan.bin(xs, y)                                    # warm-up of the full-data binning and of the step
    plan.step(theta, m, L, full, None)
    plan.k1_timing(True)
    for _ in range(args.reps):
        plan.step(theta, m, L, full, None)
    k1_full, _ = plan.k1_time_read()
    plan.k1_timing(False)
    del full
    out = []
    for B in batch_sizes:
        rec = {"bench": "minibatch", "workload": name, "family": fam, "knots": list(knots), "n": n, "batch_size": B,
               "n_batches": n // B, "obs_dtype": "float32", "run_cap": 256, **BS.gpu_info()}
        ep = plan.bin_epoch(xs, y, B, 0, 0)                   # warm-up
        del ep
        tf, te, ts, ti = [], [], [], []
        for r in range(args.reps):
            tf.append(ev_ms(lambda: plan.bin(xs, y)))
            holder = {}
            te.append(ev_ms(lambda: holder.setdefault("ep", plan.bin_epoch(xs, y, B, 0, r + 1))))
            ep = holder.pop("ep")
            plan.step(theta, m, L, ep[0], None, ep[0].scale)
            ts.append(ev_ms(lambda: [plan.step(theta, m, L, bo, None, bo.scale) for bo in ep]) / len(ep))
            if family != vg.SVGP_MARKOV:
                idx = torch.randint(0, n, (B,), device=dev)
                plan.step(theta, m, L, [x[idx].contiguous() for x in xs], y[idx].contiguous(), n / B)
                ib = torch.randperm(n, device=dev)[:B]
                ti.append(ev_ms(lambda: plan.step(theta, m, L, [x[ib].contiguous() for x in xs], y[ib].contiguous(), n / B)))
        rec.update({"bin_full_ms": median(tf), "bin_epoch_ms": median(te), "step_ms": median(ts),
                    "bin_full_ms_all": tf, "bin_epoch_ms_all": te})
        if ti:
            rec["index_step_ms"] = median(ti)
        bo = ep[0]
        gs = plan.graphed_step(theta, m, L, bo, None, bo.scale)
        gs.replay()
        rec["graph_step_ms"] = ev_ms(lambda: [gs.replay() for _ in range(args.graph_iters)]) / args.graph_iters
        plan.k1_timing(True)
        for bo in ep:
            plan.step(theta, m, L, bo, None, bo.scale)
        k1_b, nb = plan.k1_time_read()
        plan.k1_timing(False)
        rec.update({"k1_batch_ms": k1_b, "k1_full_ms": k1_full, "k1_full_scaled_ms": k1_full * B / n,
                    "epoch_bytes": int(ep.buf.numel())})
        del ep, gs, bo
        torch.cuda.empty_cache()
        out.append(rec)
    del plan, xs, y
    torch.cuda.empty_cache()
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--graph-iters", type=int, default=50)
    ap.add_argument("--scale", type=int, default=0, help="shift N and every B right by this many bits (rehearsals)")
    ap.add_argument("--only", default=None, help="comma-separated workload names")
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("bench_minibatch needs a CUDA device")
    vg = importlib.import_module("variational-gridded-gaussian-processes_b200")
    gen = importlib.import_module("variational-gridded-gaussian-processes_b200.utils.dataloaders")
    dev = torch.device("cuda", 0)
    s = args.scale
    bs = [1 << (k - s) for k in (18, 20, 22, 24)]
    wls = [("tracks512_b1", vg.B1_ASVGP, (512, 512), 1 << (26 - s)), ("tracks512_markov", vg.SVGP_MARKOV, (512, 512), 1 << (26 - s)),
           ("3d_b1", vg.B1_ASVGP, (256, 256, 64), 1 << (26 - s)), ("3d_markov", vg.SVGP_MARKOV, (256, 256, 64), 1 << (26 - s)),
           ("b0_cfg2", vg.B0_GRIDDED, (512, 512), 1 << (24 - s))]
    for name, fam, knots, n in wls:
        if args.only and name not in args.only.split(","):
            continue
        for rec in workload(vg, gen, name, fam, knots, n, [b for b in bs if b <= n], dev, args):
            line = json.dumps(rec)
            print(line, flush=True)
            if args.out:
                with open(args.out, "a") as f:
                    f.write(line + "\n")


if __name__ == "__main__":
    main()
