"""Warm starts (KL_OPT_X0) on a sequence of related systems A x_k = b_k, b_k = A u_k, where u_k is a Gaussian bump
(width 0.1 of the unit square) whose centre moves by 0.002 per system: the situation of a time stepper or a parameter
sweep.  Each system is solved cold (x0 = 0) and warm (x0 = the previous system's warm solution; the first system is
solved cold in both columns) with
  - CG at 8192^2, tol 1e-9 absolute (tests/test_cg.f90:20), default options;
  - GMRES(95) + cheb(6) at 2048^2, tol 1e-8 relative to ||b||, interval from 30 Lanczos steps (scripts/cheb_sweep.py).
Reports iterations and the call time (kl_stats total_ms: CUDA events around the whole call, the residual prologue of a
warm start included) per system, and max |x - u_k| of both solves.  Vectors stay on the device.
Usage: python scripts/warm_start.py [--out FILE] [--systems K]   (JSON to FILE, default warm_start.json)"""
import argparse, json, os, subprocess, sys
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import torch
import gmres_b200 as kl

ap = argparse.ArgumentParser()
ap.add_argument("--out", default="warm_start.json")
ap.add_argument("--systems", type=int, default=10)
args = ap.parse_args()

gpu = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                     capture_output=True, text=True).stdout.strip()
h = kl.Handle(0)
h.set_option(3, 0)      # KL_OPT_VERR: no v_err epilogue


def bump(ns, k):
    t = (torch.arange(ns, dtype=torch.float64, device="cuda") + 1) / (ns + 1)
    cx, cy, s = 0.4 + 0.002 * k, 0.5, 0.1
    gx, gy = torch.exp(-(t - cx) ** 2 / (2 * s * s)), torch.exp(-(t - cy) ** 2 / (2 * s * s))
    return (gy[:, None] * gx[None, :]).reshape(-1)      # idx = i + j*nx


def sequence(name, ns, run, count):
    rows, prev = [], None
    run(h.apply(kl.stvec, bump(ns, 0), ns, ns), None)        # warm-up: modules, CUDA graphs
    for k in range(args.systems):
        u = bump(ns, k)
        b = h.apply(kl.stvec, u, ns, ns)
        cold = run(b, None)
        warm = cold if prev is None else run(b, prev)
        prev = warm.x
        row = dict(k=k, cold_its=count(cold), warm_its=count(warm), cold_ms=round(cold.stats["total_ms"], 2),
                   warm_ms=round(warm.stats["total_ms"], 2), cold_ok=cold.status == 0, warm_ok=warm.status == 0,
                   cold_err=float((cold.x - u).abs().max()), warm_err=float((warm.x - u).abs().max()))
        rows.append(row)
        print(name, row, flush=True)
    tail = rows[1:]
    its = (sum(r["cold_its"] for r in tail), sum(r["warm_its"] for r in tail))
    ms = (sum(r["cold_ms"] for r in tail), sum(r["warm_ms"] for r in tail))
    summary = dict(systems_after_first=len(tail), cold_its=its[0], warm_its=its[1], cold_ms=round(ms[0], 1),
                   warm_ms=round(ms[1], 1), iteration_ratio=round(its[1] / its[0], 3), time_ratio=round(ms[1] / ms[0], 3))
    print(name, summary, flush=True)
    return dict(rows=rows, summary=summary)


out = dict(gpu=gpu, note="per system: iterations and kl_stats total_ms of a cold (x0 = 0) and a warm (x0 = previous warm "
           "solution) solve; summary over the systems after the first", systems=args.systems)

ns = 8192
out["cg8192"] = sequence("cg8192", ns, lambda b, x0: h.cg_omp(kl.stvec, b, 1e-9, 200000, nx=ns, ny=ns, x0=x0),
                         lambda r: r.iter)
out["cg8192"].update(tol=1e-9, mode="default options (pairs of passes at 2^26 unknowns)")
torch.cuda.empty_cache()

ns, m = 2048, 95
lo, hi = h.lanczos(kl.stvec, ns, ns, 30)
prm = h.cheb_interval_from_ritz(hi, 6)
out["gmres2048_cheb6"] = sequence(
    "gmres2048_cheb6", ns,
    lambda b, x0: h.gmres_mgsr_omp(kl.stvec, b, m, 1e-8, kl.cheb(6), prm, nx=ns, ny=ns, x0=x0),
    lambda r: (r.restart_out - 1) * m + r.n_out)
out["gmres2048_cheb6"].update(tol=1e-8, m=m, cheb_interval=prm, ritz=(lo, hi))
h.close()
if os.path.dirname(args.out):
    os.makedirs(os.path.dirname(args.out), exist_ok=True)
with open(args.out, "w") as f:
    json.dump(out, f, indent=1)
