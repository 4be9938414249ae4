"""Measurements of the sparse-matrix operator KL_OP_CSR (kl_csr.cu k_csr_spmv).

(a) y = A x for the CSR assembly of the 5-point Poisson matrix at 2048^2 (x, 34 MB, fits in the 126 MB L2) and 4096^2
    (x, 134 MB, does not), beside the built-in stencil KL_OP_POISSON5 on the same grid.
(b) y = A x for an irregular matrix: 2^22 rows of 1..64 random off-diagonal entries plus the diagonal, and four rows
    of 10^4 entries (tests/csr_twin.py irregular()).
(c) CG iterations per second on CSR Poisson 4096^2 beside KL_OP_POISSON5 (fixed iteration count, tolerance 0).

Every operator time is the mean over --reps device-mode applications (default 200) after warm-up, taken with CUDA
events around the whole batch, in --rounds rounds (median, min, max reported).  Bytes are algorithmic: CSR reads val
and col_ind (12 nnz), row_ptr (8(n+1)) and x once (8n) and writes y (8n); the stencil 16n.  Rates are bytes over time,
shares are of the HBM rate measured in the same run by a device-to-device copy of 2 GB (read + write) and of the
6547 GB/s measured earlier on this project's B200.  The card name and power limit are read in the same run.

Usage: python scripts/csr_bench.py --out profiles/r09_csr.json [--reps 200] [--rounds 5] [--label hints]
       [--compare-lib PATH --compare-label LABEL]   (repeats (a) and (b) with another build of the library)
"""
import argparse
import json
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))
import numpy as np
import torch

PEAK_GBS = 6547.0


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True).stdout.strip().splitlines()
    return q[0] if q else "unknown"


def copy_gbs(st):
    a = torch.empty(1 << 28, dtype=torch.float64, device="cuda")
    b = torch.empty_like(a)
    with torch.cuda.stream(st):
        for _ in range(3):
            b.copy_(a)
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record(st)
        for _ in range(20):
            b.copy_(a)
        e1.record(st)
    st.synchronize()
    ms = e0.elapsed_time(e1) / 20
    return 2 * a.numel() * 8 / ms / 1e6


def time_apply(h, st, A, x, nx, ny, reps, rounds):
    y = torch.empty_like(x)
    us = []
    with torch.cuda.stream(st):
        for _ in range(3):
            h.set_output_buffer(y)
            h.apply(A, x, nx, ny)
        for _ in range(rounds):
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record(st)
            for _ in range(reps):
                h.set_output_buffer(y)
                h.apply(A, x, nx, ny)
            e1.record(st)
            st.synchronize()
            us.append(e0.elapsed_time(e1) * 1e3 / reps)
    return np.array(us)


def row(us, nbytes, hbm):
    med = float(np.median(us))
    return dict(us_median=round(med, 2), us_min=round(float(us.min()), 2), us_max=round(float(us.max()), 2),
                bytes=int(nbytes), gbs=round(nbytes / med / 1e3, 1), share_measured_copy=round(nbytes / med / 1e3 / hbm, 3),
                share_6547=round(nbytes / med / 1e3 / PEAK_GBS, 3))


def csr_bytes(n, nnz):
    return 12 * nnz + 8 * (n + 1) + 8 * n + 8 * n


def operator_rates(kl, h, st, reps, rounds, hbm):
    import csr_twin as twin
    out = {}
    g = torch.Generator(device="cuda").manual_seed(1)
    for ns in (2048, 4096):
        n = ns * ns
        P = twin.poisson5(ns)
        A = kl.csr(P)
        x = torch.randn(n, dtype=torch.float64, device="cuda", generator=g)
        r = row(time_apply(h, st, A, x, n, 1, reps, rounds), csr_bytes(n, P.nnz), hbm)
        s = row(time_apply(h, st, kl.stvec, x, ns, ns, reps, rounds), 16 * n, hbm)
        out[f"poisson{ns}"] = dict(n=n, nnz=int(P.nnz), width=twin.width(n, P.nnz), csr=r, stencil=s,
                                   csr_over_stencil_time=round(r["us_median"] / s["us_median"], 2))
        print(f"CSR Poisson {ns}^2: {r['us_median']:8.1f} us  {r['gbs']:7.1f} GB/s  {r['share_measured_copy'] * 100:5.1f}% "
              f"of copy  {r['share_6547'] * 100:5.1f}% of 6547   | stencil {s['us_median']:6.1f} us", flush=True)
        del A, P
    n = 1 << 22
    ip, ix, dv = twin.irregular(n, 22)
    A = kl.csr((ip, ix, dv), n)
    x = torch.randn(n, dtype=torch.float64, device="cuda", generator=g)
    r = row(time_apply(h, st, A, x, n, 1, reps, rounds), csr_bytes(n, dv.size), hbm)
    out["irregular_2_22"] = dict(n=n, nnz=int(dv.size), width=twin.width(n, dv.size),
                                 longest_row=int(np.diff(ip).max()), csr=r)
    print(f"irregular 2^22 (nnz {dv.size}): {r['us_median']:8.1f} us  {r['gbs']:7.1f} GB/s  "
          f"{r['share_measured_copy'] * 100:5.1f}% of copy", flush=True)
    return out


def cg_rates(kl, h, st, its):
    import csr_twin as twin
    ns = 4096
    n = ns * ns
    A = kl.csr(twin.poisson5(ns))
    b = torch.randn(n, dtype=torch.float64, device="cuda", generator=torch.Generator(device="cuda").manual_seed(3))
    out = {}
    with torch.cuda.stream(st):
        for name, op in (("csr", A), ("poisson5", kl.stvec)):
            h.cg_omp(op, b, 0.0, 20)
            r = h.cg_omp(op, b, 0.0, its)
            ms = r.stats["solve_ms"]
            out[name] = dict(iterations=its, solve_ms=round(ms, 2), its_per_s=round(its / ms * 1e3, 1))
            print(f"CG 4096^2 {name}: {its / ms * 1e3:8.1f} it/s ({ms:.1f} ms for {its})", flush=True)
    out["csr_over_poisson5_time"] = round(out["csr"]["solve_ms"] / out["poisson5"]["solve_ms"], 2)
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", required=True)
    ap.add_argument("--reps", type=int, default=200)
    ap.add_argument("--rounds", type=int, default=5)
    ap.add_argument("--cg-its", type=int, default=300)
    ap.add_argument("--label", default="shipped")
    ap.add_argument("--operator-only", action="store_true")
    ap.add_argument("--compare-lib")
    ap.add_argument("--compare-label", default="compare")
    a = ap.parse_args()
    import gmres_b200 as kl
    h = kl.Handle(0)
    st = torch.cuda.Stream()
    hbm = copy_gbs(st)
    res = dict(card=card(), hbm_copy_gbs=round(hbm, 1), reps=a.reps, rounds=a.rounds)
    print(res["card"], f"copy {hbm:.1f} GB/s", flush=True)
    res[a.label] = operator_rates(kl, h, st, a.reps, a.rounds, hbm)
    if not a.operator_only:
        res["cg_4096"] = cg_rates(kl, h, st, a.cg_its)
    h.close()
    if a.compare_lib:
        tmp = a.out + ".compare.json"
        env = dict(os.environ, KRYLOV_B200_LIB=os.path.abspath(a.compare_lib))
        subprocess.check_call([sys.executable, os.path.abspath(__file__), "--out", tmp, "--reps", str(a.reps),
                               "--rounds", str(a.rounds), "--label", a.compare_label, "--operator-only"], env=env)
        with open(tmp) as f:
            other = json.load(f)
        os.remove(tmp)
        res[a.compare_label] = other[a.compare_label]
        res[a.compare_label + "_card"] = other["card"]
    with open(a.out, "w") as f:
        json.dump(res, f, indent=1)


if __name__ == "__main__":
    main()
