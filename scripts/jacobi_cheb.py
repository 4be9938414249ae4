"""Measurements of the Jacobi-scaled Chebyshev preconditioner (KL_PC_JACOBI_CHEB) on the variable-coefficient operator.

1. Time of one application z = M^-1 r at ns^2 (default 8192^2), degrees 0..8, the temporally blocked pass (ChJacCheb)
   against one pass per step (KL_OPT_CHAIN = 0): device-resident vectors, CUDA events on the handle's stream, the two
   paths alternated over several rounds (median, min, max of the per-round means).  Bytes are the algorithmic traffic of
   each path (chain: r, kx, ky in, z out = 32n; steps: start 40n, each step 56n), the share is of the measured HBM
   rate 6547 GB/s.
2. Time to tolerance at ss^2 (default 4096^2) on a contrast-1e4, anisotropy-100 field: CG, PCG + cbpr2 with the
   drivers' Lanczos policy, PCG + jacobi_cheb(k) for k in {0, 2, 4, 6}, GMRES(95) without and with jacobi_cheb(4).

Usage: python scripts/jacobi_cheb.py --out results.json [--ns 8192] [--ss 4096]
"""
import argparse
import json
import os
import subprocess
import sys
import time

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import numpy as np
import torch

import gmres_b200 as kl

PEAK_GBS = 6547.0
KL_OPT_MAX_RESTARTS = 2


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm,clocks.sm", "--format=csv,noheader"],
                       capture_output=True, text=True).stdout.strip().splitlines()
    return q[0] if q else "unknown"


def fields(n, seed, contrast=1e4, aniso=100.0):
    g = torch.Generator(device="cuda").manual_seed(seed)
    lc = float(np.log(contrast) / 2)
    kx = torch.exp((torch.rand(n, dtype=torch.float64, device="cuda", generator=g) * 2 - 1) * lc)
    ky = torch.exp((torch.rand(n, dtype=torch.float64, device="cuda", generator=g) * 2 - 1) * lc) / aniso
    return kx, ky


def bytes_per_app(k, chain, n):
    if k == 0:
        return 32 * n
    if chain:
        return 32 * n if k <= 6 else 40 * n + 56 * n * (k - 6)
    return 40 * n + 56 * n * k


def apply_times(h, st, ns, rounds, reps):
    n = ns * ns
    A = kl.aniso_var(*fields(n, 1))
    r = torch.randn(n, dtype=torch.float64, device="cuda", generator=torch.Generator(device="cuda").manual_seed(2))
    z = torch.empty_like(r)
    prm = h.cheb_interval_from_ritz(2.0 / 1.025, 4)
    out = {}
    with torch.cuda.stream(st):
        for k in range(9):
            per = {1: [], 0: []}
            for _ in range(rounds):
                for chain in (1, 0):
                    h.set_option(kl.KL_OPT_CHAIN, chain)
                    for _ in range(2):
                        h.set_output_buffer(z)
                        h.apply_precond(kl.jacobi_cheb(k), A, r, prm, ns, ns)
                    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                    e0.record(st)
                    for _ in range(reps):
                        h.set_output_buffer(z)
                        h.apply_precond(kl.jacobi_cheb(k), A, r, prm, ns, ns)
                    e1.record(st)
                    st.synchronize()
                    per[chain].append(e0.elapsed_time(e1) * 1e3 / reps)
            h.set_option(kl.KL_OPT_CHAIN, 1)
            row = {}
            for chain, name in ((1, "chain"), (0, "stepwise")):
                us = np.array(per[chain])
                med = float(np.median(us))
                b = bytes_per_app(k, chain, n)
                row[name] = dict(us_median=round(med, 1), us_min=round(float(us.min()), 1), us_max=round(float(us.max()), 1),
                                 bytes=b, gbs=round(b / med / 1e3, 1), share=round(b / med / 1e3 / PEAK_GBS, 3))
            row["speedup"] = round(row["stepwise"]["us_median"] / row["chain"]["us_median"], 2)
            out[f"degree{k}"] = row
            print(f"jacobi_cheb({k}) {ns}^2: chain {row['chain']['us_median']:8.1f} us "
                  f"[{row['chain']['us_min']:.1f}, {row['chain']['us_max']:.1f}] {row['chain']['share'] * 100:5.1f}%   "
                  f"stepwise {row['stepwise']['us_median']:8.1f} us [{row['stepwise']['us_min']:.1f}, "
                  f"{row['stepwise']['us_max']:.1f}] {row['stepwise']['share'] * 100:5.1f}%   x{row['speedup']}", flush=True)
    return out


def solves(h, ss, cg_cap, gmres_cycles):
    n = ss * ss
    A = kl.aniso_var(*fields(n, 3))
    b = h.apply(A, torch.ones(n, dtype=torch.float64, device="cuda"), ss, ss)
    torch.cuda.synchronize()
    out = {}

    def run(name, fn, m=None):
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        g = fn()
        torch.cuda.synchronize()
        sec = time.perf_counter() - t0
        its = g.iter if m is None else (g.restart_out - 1) * m + g.n_out
        err = float((g.x - 1).abs().max())
        out[name] = dict(iterations=int(its), seconds=round(sec, 3), status=int(g.status), max_err=err)
        print(f"{ss}^2 {name:24s} {its:8d} its {sec:9.3f} s status {g.status} max|x-1| {err:.2e}", flush=True)

    lo, hi = h.lanczos(A, ss, ss, 30)
    cb = h.cheb_params_from_ritz(lo, hi)
    out["lanczos"] = dict(theta_min=lo, theta_max=hi, cbpr2_params=cb)
    run("cg", lambda: h.cg_omp(A, b, 1e-9, cg_cap))
    run("pcg_cbpr2_lanczos", lambda: h.pcg_omp(A, b, 1e-9, cg_cap, kl.cbpr2, cb))
    for k in (0, 2, 4, 6):
        prm = (0.0, 0.0) if k == 0 else h.cheb_interval_from_ritz(2.0 / 1.025, k)
        run(f"pcg_jacobi_cheb{k}", lambda: h.pcg_omp(A, b, 1e-9, cg_cap, kl.jacobi_cheb(k), prm))
    h.set_option(KL_OPT_MAX_RESTARTS, gmres_cycles)
    run("gmres95", lambda: h.gmres_mgsr_omp(A, b, 95, 1e-8, None, None), m=95)
    prm = h.cheb_interval_from_ritz(2.0 / 1.025, 4)
    run("gmres95_jacobi_cheb4", lambda: h.gmres_mgsr_omp(A, b, 95, 1e-8, kl.jacobi_cheb(4), prm), m=95)
    h.set_option(KL_OPT_MAX_RESTARTS, 1000)
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--ns", type=int, default=8192)
    ap.add_argument("--ss", type=int, default=4096)
    ap.add_argument("--rounds", type=int, default=5)
    ap.add_argument("--reps", type=int, default=10)
    ap.add_argument("--cg-cap", type=int, default=60000)
    ap.add_argument("--gmres-cycles", type=int, default=100)
    ap.add_argument("--out", required=True, help="JSON file the results are written to")
    a = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("no CUDA device: these are GPU measurements")
    st = torch.cuda.Stream()
    h = kl.Handle(0, stream=st.cuda_stream)
    res = dict(card=card(), ns=a.ns, rounds=a.rounds, reps=a.reps, peak_gbs=PEAK_GBS)
    print(res["card"], flush=True)
    res["apply"] = apply_times(h, st, a.ns, a.rounds, a.reps)
    res["solves"] = dict(ss=a.ss, cg_cap=a.cg_cap, gmres_cycles=a.gmres_cycles, results=solves(h, a.ss, a.cg_cap,
                                                                                                a.gmres_cycles))
    res["card_after"] = card()
    h.close()
    os.makedirs(os.path.dirname(a.out) or ".", exist_ok=True)
    json.dump(res, open(a.out, "w"), indent=1)


if __name__ == "__main__":
    main()
