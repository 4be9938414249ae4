"""Plain CG in pairs of passes (KL_OPT_CG_ONEPASS = 2, 36n B per iteration) against one pass per iteration (1, 48n B)
over the grid size, to place the auto threshold of pair mode.  Manufactured problem b = A 1, tol 0, default options
(host poll every 32 iterations, batches replayed as CUDA graphs).  The two settings alternate, REPS runs each; time =
the solve's CUDA-event window (kl_stats solve_ms).  The two settings must agree bit for bit (history and x).
Usage: python scripts/cg_pair_sweep.py [--out FILE] [ns ...]   (default 2048 4096 8192 16384); writes the table as
JSON to FILE (default: cg_pair_sweep.json in the current directory)"""
import argparse, json, os, statistics, subprocess, sys
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import torch
import gmres_b200 as kl

KL_OPT_CG_ONEPASS = 22
ap = argparse.ArgumentParser()
ap.add_argument("--out", default="cg_pair_sweep.json")
ap.add_argument("sizes", nargs="*", type=int)
args = ap.parse_args()
REPS = 5
ITS = {2048: 1600, 4096: 448, 8192: 128, 16384: 64}    # even (no flush of x), ~0.1-0.2 s per solve
BYTES = {1: 48.0, 2: 36.0}
LABEL = {1: "onepass_48n", 2: "pair_36n"}

gpu = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                     capture_output=True, text=True).stdout.strip()
h = kl.Handle(0)
out = dict(gpu=gpu, reps=REPS, note="ms per iteration, CUDA events around the iteration loop; median (min..max) of REPS "
           "alternating runs", sizes={})
for ns in args.sizes or sorted(ITS):
    its = ITS.get(ns, 128)
    b = h.apply(kl.stvec, torch.ones(ns * ns, dtype=torch.float64, device="cuda"), ns, ns)
    ms = {1: [], 2: []}
    res = {}
    for rep in range(REPS + 1):                 # rep 0 warms up both settings (module load, graph capture)
        for v in (1, 2):
            h.set_option(KL_OPT_CG_ONEPASS, v)
            r = h.cg_omp(kl.stvec, b, 0.0, its, nx=ns, ny=ns)
            assert r.stats["algorithmic_bytes"] / its / (ns * ns) == BYTES[v]
            res[v] = (r.history, r.x)
            if rep:
                ms[v].append(r.stats["solve_ms"] / its)
    same = bool(torch.equal(torch.as_tensor(res[1][0]), torch.as_tensor(res[2][0])) and torch.equal(res[1][1], res[2][1]))
    row = {}
    for v in (1, 2):
        med = statistics.median(ms[v])
        row[LABEL[v]] = dict(ms_per_it=round(med, 5), min=round(min(ms[v]), 5), max=round(max(ms[v]), 5),
                             gbs=round(BYTES[v] * ns * ns / (med * 1e-3) / 1e9, 1))
    row["speedup"] = round(row[LABEL[1]]["ms_per_it"] / row[LABEL[2]]["ms_per_it"], 3)
    row["bit_identical"] = same
    row["iterations"] = its
    out["sizes"][str(ns)] = row
    print(ns, row, flush=True)
    del b, res, r
    torch.cuda.empty_cache()
h.set_option(KL_OPT_CG_ONEPASS, -1)
if os.path.dirname(args.out):
    os.makedirs(os.path.dirname(args.out), exist_ok=True)
with open(args.out, "w") as f:
    json.dump(out, f, indent=1)
