"""Convection-diffusion (KL_OP_STENCIL5) on one GPU: the fused paths against aniso(1, 0.01) and against the generic
path, and time to tolerance of GMRES(95) with the Chebyshev preconditioners on the exact spectrum interval.

1. Rate: BiCGSTAB + cbpr2 at 8192^2 and GMRES-MGSR(95) + cbpr2 at 4096^2, a fixed number of iterations, on
   convdiff(0.5, 0.25) and aniso(1, 0.01), fused (default options) and with KL_OPT_FUSE = 0 (one kernel per reference
   loop: the path a KL_OP_USER callback gets).  it/s from the library's CUDA-event solve time; GB/s = the executed
   kernels' algorithmic bytes over that time (kl_stats_t).
2. Time to rtol 1e-8 of GMRES(95) at 2048^2 (at most 100 cycles) with no preconditioner, cbpr2, cheb(4) and cheb(6), on the exact interval
   [lam_min, lam_max] of kl_stencil5_spectrum and on the cut interval [lam_max/ratio(k), lam_max] of the library's
   ratio table (kl_cheb_interval_from_ritz), for central px = 0.5, central px = 0.9 and upwind px = 2.

    python scripts/convdiff.py --out results.json [--n-tol 2048]
"""
import argparse
import json
import os
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

import torch  # noqa: E402

import gmres_b200 as kl  # noqa: E402

FUSE, MAX_RESTARTS = 7, 2


def gpu_info():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm,clocks.sm", "--format=csv,noheader"],
                       capture_output=True, text=True).stdout.strip().split("\n")[0]
    name, pl, smmax, sm = [s.strip() for s in q.split(",")]
    return dict(gpu=name, power_limit=pl, sm_clock_max=smmax, sm_clock_at_start=sm)


def ones(n):
    return torch.ones(n, dtype=torch.float64, device="cuda")


def rate(h, kind, A, n, its, fuse):
    b = h.apply(A, ones(n * n), n, n)
    # cbpr2 on the exact interval (aniso(ex, ey) is stencil5(2(ex + ey), ex, ex, ey, ey))
    S = A if A.kind == kl.api.KL_OP_STENCIL5 else kl.stencil5(2.0 * (A.eps_x + A.eps_y), A.eps_x, A.eps_x, A.eps_y, A.eps_y)
    lo, hi = kl.stencil5_spectrum(S, n, n)
    prm = (hi, lo)
    h.set_option(FUSE, fuse)
    try:
        def run():
            if kind == "bicgstab":
                return h.pbicgstab_omp(A, b, 1e-300, its, kl.cbpr2, prm)
            h.set_option(MAX_RESTARTS, its // 95)
            return h.gmres_mgsr_omp(A, b, 95, 1e-300, kl.cbpr2, prm)
        run()
        best = None
        for _ in range(3):
            r = run()
            st = r.stats
            it = st["iterations"]
            v = dict(iterations=it, solve_ms=st["solve_ms"], it_per_s=it / (st["solve_ms"] / 1e3),
                     gb_per_s=st["algorithmic_bytes"] / (st["solve_ms"] / 1e3) / 1e9,
                     bytes_per_it=st["algorithmic_bytes"] / it, launches=st["kernel_launches"])
            if best is None or v["solve_ms"] < best["solve_ms"]:
                best = v
        return best
    finally:
        h.set_option(FUSE, 1)
        h.set_option(MAX_RESTARTS, 1000)


def to_tol(h, A, n, pc, k, interval):
    b = h.apply(A, ones(n * n), n, n)
    lo, hi = kl.stencil5_spectrum(A, n, n)
    if pc is None:
        M, prm = None, None
    else:
        M = kl.cbpr2 if pc == "cbpr2" else kl.cheb(k)
        prm = (hi, lo) if interval == "exact" else h.cheb_interval_from_ritz(hi / 1.025, 1 if pc == "cbpr2" else k)
    h.set_option(MAX_RESTARTS, 100)
    try:
        t0 = time.perf_counter()
        r = h.gmres_mgsr_omp(A, b, 95, 1e-8, M, prm)
        wall = time.perf_counter() - t0
    finally:
        h.set_option(MAX_RESTARTS, 1000)
    its = (r.restart_out - 1) * 95 + r.n_out
    err = float((r.x - 1).abs().max())
    return dict(precond=pc if pc != "cheb" else f"cheb({k})", interval=interval if pc else None,
                params=list(prm) if prm else None, status=r.status, iterations=its, solve_ms=r.stats["solve_ms"],
                wall_s=wall, err_inf=err)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", required=True, help="JSON file the results are written to")
    ap.add_argument("--n-tol", type=int, default=2048)
    args = ap.parse_args()
    h = kl.Handle(0)
    out = dict(info=gpu_info(), rate=[], to_tol=[])
    for kind, n, its in (("bicgstab", 8192, 200), ("gmres95", 4096, 190)):
        for name, A in (("convdiff(0.5, 0.25)", kl.convdiff(0.5, 0.25)), ("aniso(1, 0.01)", kl.aniso(1.0, 0.01))):
            for fuse in (1, 0):
                v = rate(h, kind, A, n, its, fuse)
                v.update(solver=f"{kind}+cbpr2", n=n, operator=name, fuse=fuse)
                print(json.dumps(v), flush=True)
                out["rate"].append(v)
    n = args.n_tol
    for name, A in (("central px=0.5", kl.convdiff(0.5, 0.0)), ("central px=0.9", kl.convdiff(0.9, 0.0)),
                    ("upwind px=2", kl.convdiff(2.0, 0.0, upwind=True))):
        lo, hi = kl.stencil5_spectrum(A, n, n)
        for pc, k, interval in ((None, 0, None), ("cbpr2", 0, "exact"), ("cbpr2", 0, "cut"), ("cheb", 4, "exact"),
                                ("cheb", 4, "cut"), ("cheb", 6, "exact"), ("cheb", 6, "cut")):
            v = to_tol(h, A, n, pc, k, interval)
            v.update(operator=name, n=n, lam_min=lo, lam_max=hi)
            print(json.dumps(v), flush=True)
            out["to_tol"].append(v)
    out["info"]["sm_clock_at_end"] = gpu_info()["sm_clock_at_start"]
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as f:
        json.dump(out, f, indent=1)
    h.close()


if __name__ == "__main__":
    main()
