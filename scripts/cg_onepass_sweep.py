"""Plain CG, one pass per iteration (KL_OPT_CG_ONEPASS = 1, 48n B) against the two-kernel path (0, 64n B) over the
grid size, to place the auto threshold.  Manufactured problem b = A 1, tol 0, default options (host poll every 32
iterations, batches replayed as CUDA graphs).  The two settings alternate, REPS runs each; time = the solve's CUDA-event
window (kl_stats solve_ms).
Usage: python scripts/cg_onepass_sweep.py [--out FILE] [ns ...]   (default 1024 2048 4096 8192 16384); writes the
table as JSON to FILE (default: cg_onepass_sweep.json in the current directory)"""
import argparse, json, os, statistics, subprocess, sys
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import torch
import gmres_b200 as kl

KL_OPT_CG_ONEPASS = 22
ap = argparse.ArgumentParser()
ap.add_argument("--out", default="cg_onepass_sweep.json")
ap.add_argument("sizes", nargs="*", type=int)
args = ap.parse_args()
REPS = 5
ITS = {1024: 3200, 2048: 1600, 4096: 448, 8192: 128, 16384: 64}    # ~0.1-0.2 s per solve

gpu = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                     capture_output=True, text=True).stdout.strip()
h = kl.Handle(0)
out = dict(gpu=gpu, reps=REPS, note="ms per iteration, CUDA events around the iteration loop; median (min..max) of REPS "
           "alternating runs", sizes={})
for ns in args.sizes or sorted(ITS):
    its = ITS.get(ns, 128)
    b = h.apply(kl.stvec, torch.ones(ns * ns, dtype=torch.float64, device="cuda"), ns, ns)
    ms = {0: [], 1: []}
    hist = {}
    for rep in range(REPS + 1):                 # rep 0 warms up both settings (module load, graph capture)
        for v in (0, 1):
            h.set_option(KL_OPT_CG_ONEPASS, v)
            r = h.cg_omp(kl.stvec, b, 0.0, its, nx=ns, ny=ns)
            assert r.stats["algorithmic_bytes"] / its / (ns * ns) == (48.0 if v else 64.0)
            hist[v] = r.history
            if rep:
                ms[v].append(r.stats["solve_ms"] / its)
    # first 50 iterations: tol = 0 runs the small grids far past convergence, where the point-wise ratio of two
    # correct residual histories is noise (tests/parity.py)
    rel = float((torch.as_tensor(hist[1][:50]) / torch.as_tensor(hist[0][:50]) - 1).abs().max())
    row = {}
    for v, label in ((0, "two_kernel_64n"), (1, "onepass_48n")):
        med = statistics.median(ms[v])
        row[label] = dict(ms_per_it=round(med, 5), min=round(min(ms[v]), 5), max=round(max(ms[v]), 5),
                          gbs=round((48.0 if v else 64.0) * ns * ns / (med * 1e-3) / 1e9, 1))
    row["speedup"] = round(row["two_kernel_64n"]["ms_per_it"] / row["onepass_48n"]["ms_per_it"], 3)
    row["history_rel_diff_first50"] = rel
    row["iterations"] = its
    out["sizes"][str(ns)] = row
    print(ns, row, flush=True)
    del b
    torch.cuda.empty_cache()
h.set_option(KL_OPT_CG_ONEPASS, -1)
if os.path.dirname(args.out):
    os.makedirs(os.path.dirname(args.out), exist_ok=True)
with open(args.out, "w") as f:
    json.dump(out, f, indent=1)
