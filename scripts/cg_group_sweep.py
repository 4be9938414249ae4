"""Plain CG in groups of G passes (KL_OPT_CG_ONEPASS = 3: G - 1 passes that store nothing, one that stores r, p and x;
(16 (G - 1) + 48) / G n B per iteration) against pairs of passes (2, 36n B) over the grid size, to place the auto
threshold of group mode.  Manufactured problem b = A 1, tol 0, default options (host poll every 32 iterations, batches
replayed as CUDA graphs).  The settings alternate, REPS runs each; time = the solve's CUDA-event window (kl_stats
solve_ms).  Groups and pairs agree within rounding (the reduction order of alpha and beta differs); the largest
relative difference of the residual histories and of x is reported.
--passes: also time every pass of a group of each size G at the largest grid with KL_OPT_PROFILE (a run of its own)
and project ms per iteration = (sum of the group's pass times) / G.
Usage: python scripts/cg_group_sweep.py [--out FILE] [--groups G ...] [--passes] [NXxNY | N ...]
(default sizes 8192 8192x16384 16384, default group size 4); writes JSON to FILE (default cg_group_sweep.json)"""
import argparse, json, os, statistics, subprocess, sys
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import torch
import gmres_b200 as kl

KL_OPT_PROFILE = 8
KL_OPT_CG_ONEPASS = 22
ap = argparse.ArgumentParser()
ap.add_argument("--out", default="cg_group_sweep.json")
ap.add_argument("--groups", nargs="*", type=int, default=[4])
ap.add_argument("--passes", action="store_true")
ap.add_argument("sizes", nargs="*")
args = ap.parse_args()
REPS = 5
ITS = 96     # a multiple of 2, 3 and 4: whole pairs and groups, ~0.1-0.2 s per solve at these sizes


def parse(s):
    a, _, b = s.partition("x")
    return int(a), int(b or a)


def handle(g):
    """Handles read the group size from the environment when they are created."""
    if g:
        os.environ["KL_CG_GROUP"] = str(g)
    hd = kl.Handle(0)
    os.environ.pop("KL_CG_GROUP", None)
    return hd


def group_bytes(g):
    return (16.0 * (g - 1) + 48.0) / g


gpu = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                     capture_output=True, text=True).stdout.strip()
arms = [("pair_36n", 2, None)] + [(f"group{g}_{group_bytes(g):.1f}n", 3, g) for g in args.groups]
hs = {label: handle(g) for label, _, g in arms}
for label, mode, _ in arms:
    hs[label].set_option(KL_OPT_CG_ONEPASS, mode)
out = dict(gpu=gpu, reps=REPS, iterations=ITS, note="ms per iteration, CUDA events around the iteration loop; median "
           "(min..max) of REPS alternating runs; rel_hist / rel_x: largest relative difference from pairs", sizes={})
sizes = [parse(s) for s in args.sizes] or [(8192, 8192), (8192, 16384), (16384, 16384)]
for nx, ny in sizes:
    n = nx * ny
    h0 = hs["pair_36n"]
    b = h0.apply(kl.stvec, torch.ones(n, dtype=torch.float64, device="cuda"), nx, ny)
    ms = {label: [] for label, _, _ in arms}
    res = {}
    for rep in range(REPS + 1):                 # rep 0 warms up every setting (module load, graph capture)
        for label, mode, g in arms:
            r = hs[label].cg_omp(kl.stvec, b, 0.0, ITS, nx=nx, ny=ny)
            want = 36.0 if mode == 2 else group_bytes(g)
            assert abs(r.stats["algorithmic_bytes"] / ITS / n - want) < 1e-9, (label, r.stats["algorithmic_bytes"])
            res[label] = (torch.as_tensor(r.history), r.x)
            if rep:
                ms[label].append(r.stats["solve_ms"] / ITS)
    row = {}
    ref_h, ref_x = res["pair_36n"]
    for label, mode, g in arms:
        med = statistics.median(ms[label])
        byt = 36.0 if mode == 2 else group_bytes(g)
        row[label] = dict(ms_per_it=round(med, 5), min=round(min(ms[label]), 5), max=round(max(ms[label]), 5),
                          gbs=round(byt * n / (med * 1e-3) / 1e9, 1))
        if mode == 3:
            hh, xx = res[label]
            row[label]["speedup"] = round(row["pair_36n"]["ms_per_it"] / med, 3)
            row[label]["rel_hist"] = float(((hh - ref_h).abs() / ref_h.abs()).max())
            row[label]["rel_x"] = float(((xx - ref_x).abs().max() / ref_x.abs().max()).item())
    out["sizes"][f"{nx}x{ny}"] = row
    print(nx, ny, row, flush=True)
    del b, res, r
    torch.cuda.empty_cache()

if args.passes:
    nx, ny = sizes[-1]
    n = nx * ny
    passes = {}
    for label, mode, g in arms:
        h = hs[label]
        b = h.apply(kl.stvec, torch.ones(n, dtype=torch.float64, device="cuda"), nx, ny)
        h.set_option(KL_OPT_PROFILE, 1)
        h.cg_omp(kl.stvec, b, 0.0, ITS, nx=nx, ny=ny)           # warm-up
        r = h.cg_omp(kl.stvec, b, 0.0, ITS, nx=nx, ny=ny)
        prof = h.profile()
        h.set_option(KL_OPT_PROFILE, 0)
        rows = [dict(name=p["name"], us=round(1e3 * p["ms"] / p["launches"], 1), launches=p["launches"],
                     gbs=round(p["algorithmic_bytes"] / p["launches"] / (p["ms"] / p["launches"] * 1e-3) / 1e9, 1))
                for p in prof]
        passes[label] = dict(passes=rows, projected_ms_per_it=round(sum(p["ms"] for p in prof) / ITS, 4),
                             solve_ms_per_it=round(r.stats["solve_ms"] / ITS, 4))
        print(label, passes[label], flush=True)
        del b
        torch.cuda.empty_cache()
    out["passes"] = {"grid": f"{nx}x{ny}", **passes}

for hd in hs.values():
    hd.close()
if os.path.dirname(args.out):
    os.makedirs(os.path.dirname(args.out), exist_ok=True)
with open(args.out, "w") as f:
    json.dump(out, f, indent=1)
