#!/usr/bin/env python
"""bench.py -- Krylov iterations/s on synthetic Poisson grids, B200 vs the CPU path.

    python bench.py --gpus N --steps K --warmup W [--workload cg16384|gmres4096|...]
    python bench.py --impl reference --gpus N --steps K --warmup W
    python bench.py --gpus 1 --steps K --warmup W --dump-outputs DIR

A "step" is ONE Krylov iteration.  The primary workload is BASELINE.json configs[3]:
CG on the 16384 x 16384 Poisson grid (268 M unknowns), strong-scaled over N GPUs by
row slabs (halo send/recv + scalar all-reduces).  At N=1 the JSON line also carries
`extra` results for configs[2] (Chebyshev-preconditioned GMRES-MGSR(95), 4096^2),
configs[1] (Householder GMRES(95), 1024^2) and configs[4] (BiCGSTAB, 8192^2/GPU).

Bytes: `roofline` and `roofline_iter` use the bytes the kernels actually have to move (kl_get_stats /
kl_get_profile, listed per kernel in DESIGN.md section 3): plain CG executes 64n B per iteration (the operator
is applied twice instead of storing A p; SURVEY.md section 8d assumed 80n), PCG + cbpr2 80n, BiCGSTAB + cbpr2
160n.  `roofline.traffic` is the DRAM traffic ncu measured for the dominant kernel (profiles/r02_traffic.json).

Inputs are synthetic and deterministic (x_true = 1, b = A*1; no RNG), resident in HBM
before the timed region; vectors (2.1 GB each) are far larger than the 126 MB L2, so no
L2 flush is needed between iterations.  Timing: CUDA events on the launching stream
around exactly K iterations (tol = 0 so nothing converges early), barrier + device sync
on both sides, MAX over ranks.

`--dump-outputs DIR`: after the timed call, what it returned is written as DIR/<name>.npy (float64): the solution
x (for more than 2^21 unknowns, its entries at up to 2^21 seeded random positions, which x_index lists), the iteration
count, the final residual, the status and the residual history (GMRES: final_err, v_err, n_out, restart_out as
well).  The inputs carry no randomness, so two builds run with the same arguments can be compared file by file.
With several ranks, each writes its own slab's files with a _rank<r> suffix.

`--impl reference`: the reference is Fortran and no Fortran compiler exists on the
build or GPU box, so this arm times the C/OpenMP restatement of the reference's
`cg_omp` (oracle/, same loop/barrier structure) on all host cores, on a bounded
number of iterations of the same workload.
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

P_REF = (8.2, 0.2)  # tests/test_poisson_mf.f90:38

WORKLOADS = {
    # name: (solver, nx, ny_per_gpu_or_global, scaling, precond, m, bytes_per_iter_per_unknown)
    "cg16384": dict(solver="cg_omp", nx=16384, ny=16384, scaling="strong", pc=None, m=0),
    "pcg16384": dict(solver="pcg_omp", nx=16384, ny=16384, scaling="strong", pc="cbpr2", m=0),
    "gmres4096": dict(solver="gmres_mgsr_omp", nx=4096, ny=4096, scaling="strong", pc="cbpr2", m=95),
    "gmres4096sel": dict(solver="gmres_mgsr_omp", nx=4096, ny=4096, scaling="strong", pc="cbpr2", m=95, ortho=2, eta=300),
    "hh1024": dict(solver="gmres_hh_omp", nx=1024, ny=1024, scaling="strong", pc=None, m=95),
    "bicgstab8192": dict(solver="pbicgstab_omp", nx=8192, ny=8192, scaling="weak", pc="cbpr2", m=0,
                         aniso=(1.0, 0.01)),
    "gmres300": dict(solver="gmres_mgsr_omp", nx=300, ny=300, scaling="strong", pc="cbpr2", m=95),
    "cg4096": dict(solver="cg_omp", nx=4096, ny=4096, scaling="strong", pc=None, m=0),
    # degree-4 Chebyshev (4 operator applications per preconditioner call, one HBM pass: kl_chain_tma.cuh)
    "pcg8192cheb4": dict(solver="pcg_omp", nx=8192, ny=8192, scaling="strong", pc="cheb4", m=0),
    "gmres4096cheb4": dict(solver="gmres_mgsr_omp", nx=4096, ny=4096, scaling="strong", pc="cheb4", m=95),
}


def load_peaks():
    try:
        with open(os.path.join(ROOT, "MEASURED_PEAKS.json")) as f:
            return float(json.load(f)["hbm_gbs"]), "measured"
    except Exception:
        return 6650.0, "fallback"   # B200_PROFILING.md fallback


class ClockSampler:
    """nvidia-smi clocks / throttle reasons sampled DURING the timed region."""

    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,"
         "clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index=0):
        self.gpu = gpu_index
        self.proc = None
        self.lines = []

    def start(self):
        try:
            self.proc = subprocess.Popen(
                ["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits", "-lms", "20",
                 "-i", str(self.gpu)], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.t = threading.Thread(target=self._read, daemon=True)
            self.t.start()
        except Exception:
            self.proc = None

    def _read(self):
        for ln in self.proc.stdout:
            self.lines.append(ln.strip())

    def stop(self):
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.15)
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except Exception:
            self.proc.kill()
        sm, mx, reasons, pw = [], [], set(), []
        for ln in self.lines:
            f = [s.strip() for s in ln.split(",")]
            if len(f) < 9:
                continue
            try:
                sm.append(float(f[1])); mx.append(float(f[2])); pw.append(float(f[3]))
            except ValueError:
                continue
            for name, val in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"),
                                 f[5:9]):
                if val.lower().startswith("active"):
                    reasons.add(name)
        if not sm:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["no samples"]}
        # "under load": the samples taken while the GPU drew more than half of the highest power seen
        load = sorted(c for c, p in zip(sm, pw) if p >= 0.5 * max(pw)) or sorted(sm)
        return {"sm_mhz": load[len(load) // 2], "sm_max_mhz": max(mx), "reasons": sorted(reasons),
                "samples": len(sm), "samples_under_load": len(load), "power_w_max": max(pw)}


def workload_string(name, world):
    """the same string in both arms (the driver compares config.workload of the b200 and the reference line)"""
    w = WORKLOADS[name]
    nx, ny = w["nx"], w["ny"] * (world if w["scaling"] == "weak" else 1)
    pc = f" + {w['pc']}" if w["pc"] else ""
    m = f"({w['m']})" if w["m"] else ""
    op = f"anisotropic diffusion (eps {w['aniso'][0]:g}, {w['aniso'][1]:g})" if w.get("aniso") else "Poisson"
    return (f"{w['solver']}{m}{pc}, {op} 2D 5-point matrix-free {nx}x{ny} ({nx * ny} unknowns), FP64, x_true=1, "
            f"fixed K iterations (tol=0)")


def history_parity(name, hist, r0):
    """Residuals of the timed run against the committed history of the same workload (tests/golden/bench_history.json:
    the CPU oracle's and the single-GPU run's first iterations) -- carries correctness into every bench line,
    multi-GPU ones included.  max_rel = max |h_k/h'_k - 1|, max_norm = max |h_k - h'_k| / ||r_0||."""
    try:
        with open(os.path.join(ROOT, "tests", "golden", "bench_history.json")) as f:
            ref = json.load(f)[name]
    except Exception:
        return None
    out = {}
    for src in ("oracle", "gpu_n1"):
        hr = ref.get(src)
        if not hr:
            continue
        k = min(len(hr), len(hist))
        if k == 0:
            continue
        rel = max(abs(hist[i] / hr[i] - 1.0) for i in range(k))
        nrm = max(abs(hist[i] - hr[i]) for i in range(k)) / r0
        out[src] = {"max_rel": rel, "max_norm": nrm, "iterations_compared": k}
    if not out:
        return None
    best = out.get("oracle") or out.get("gpu_n1")
    return {"max_rel": best["max_rel"], "max_norm": best["max_norm"], "iterations_compared": best["iterations_compared"],
            "against": ref.get("source", ""), "detail": out}


DUMP_SAMPLE = 1 << 21   # solution entries kept by --dump-outputs when x is longer (16 MB of float64)


def solver_outputs(r):
    """What a caller of the timed solver call receives (x and the result fields beside it) as float64 host arrays.
    An x longer than DUMP_SAMPLE is reduced to the entries at a fixed, seeded set of positions, stored as x_index."""
    import dataclasses
    import numpy as np
    import torch

    out = {}
    for f in dataclasses.fields(r):
        v = getattr(r, f.name)
        if f.name == "stats":
            continue
        if f.name == "x":
            if v.numel() > DUMP_SAMPLE:
                idx = np.unique(np.random.default_rng(0).integers(0, v.numel(), DUMP_SAMPLE))
                out["x_index"] = idx.astype(np.float64)
                v = v[torch.from_numpy(idx).to(v.device)]
            out["x"] = v.cpu().numpy().astype(np.float64)
        else:
            out[f.name] = np.asarray(v, dtype=np.float64)
    return out


def make_ops(kl, w):
    A = kl.aniso(*w["aniso"]) if w.get("aniso") else kl.stvec
    M = kl.cbpr2 if w["pc"] == "cbpr2" else (kl.cheb(int(w["pc"][4:])) if (w["pc"] or "").startswith("cheb") else None)
    return A, M


def run_gpu_solver(kl, h, w, b, nx, ny, iters, profile=False):
    """Run exactly `iters` iterations (tol = 0 => never converges).  Returns result."""
    A, M = make_ops(kl, w)
    h.set_option(3, 0)        # KL_OPT_VERR off: the epilogue is not part of an iteration
    h.set_option(8, 1 if profile else 0)
    s = w["solver"]
    if s in ("cg_omp", "pcg_omp", "pbicgstab_omp"):
        h.set_option(4, max(iters, 1))   # one host poll at the end
        if s == "cg_omp":
            return h.cg_omp(A, b, 0.0, iters, nx=nx, ny=ny)
        if s == "pcg_omp":
            return h.pcg_omp(A, b, 0.0, iters, M, P_REF, nx=nx, ny=ny)
        return h.pbicgstab_omp(A, b, 0.0, iters, M, P_REF, nx=nx, ny=ny)
    m = w["m"]
    cycles = max(1, iters // m)
    h.set_option(2, cycles)   # KL_OPT_MAX_RESTARTS
    if s == "gmres_mgsr_omp":
        h.set_ortho(w.get("ortho", 1))
        h.set_option(11, w.get("eta", 300))   # KL_OPT_REORTH_ETA (selective mode only)
        try:
            return h.gmres_mgsr_omp(A, b, m, 0.0, M, P_REF, nx=nx, ny=ny)
        finally:
            h.set_ortho(1)
            h.set_option(11, 300)
    if s == "gmres_hh_omp":
        return h.gmres_hh_omp(A, b, m, 0.0, nx=nx, ny=ny)
    raise ValueError(s)


def gpu_arm(args):
    import numpy as np
    import torch
    import gmres_b200 as kl

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device (no CPU fallback in the product path)")
    torch.cuda.set_device(local)
    dist = None
    if world > 1:
        import torch.distributed as dist
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    h = kl.Handle(local)
    if world > 1:
        ids = [h.unique_id() if rank == 0 else None]
        dist.broadcast_object_list(ids, src=0)
        h.comm_init(rank, world, ids[0])

    def barrier():
        torch.cuda.synchronize()
        if dist:
            dist.barrier()
        torch.cuda.synchronize()

    def max_over_ranks(v):
        if not dist:
            return v
        t = torch.tensor([v], dtype=torch.float64, device="cuda")
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item())

    def measure(name, steps, warmup, with_e2e, with_profile, keep_outputs=False):
        w = WORKLOADS[name]
        nx = w["nx"]
        ny = w["ny"] * (world if w["scaling"] == "weak" else 1)   # global lines
        j0, nyl = h.partition(ny)
        n_loc = nx * nyl
        A, M = make_ops(kl, w)
        # b = A*1 built by the operator itself on this rank's slab (+ global boundary rows)
        ones = torch.ones(n_loc, dtype=torch.float64, device="cuda")
        b = h.apply(A, ones, nx, ny)
        del ones
        m = w["m"] or 1
        steps_eff = max(m, (steps // m) * m) if w["m"] else steps
        warm_eff = max(m, (warmup // m) * m) if w["m"] else max(warmup, 3)
        smp = ClockSampler(local)
        if rank == 0:
            smp.start()          # 20 ms period, started before the warm-up so that the short timed region is covered
        run_gpu_solver(kl, h, w, b, nx, ny, warm_eff)                    # warm-up (untimed)
        barrier()
        r = run_gpu_solver(kl, h, w, b, nx, ny, steps_eff)               # timed: events inside the library
        barrier()
        clocks = smp.stop() if rank == 0 else None
        outputs = solver_outputs(r) if keep_outputs else None
        ms = max_over_ranks(r.stats["solve_ms"])
        its = r.stats["iterations"]
        launches = r.stats["kernel_launches"]
        r0 = 1.0 if w["m"] else float(np.sqrt(4.0 * nx + 8.0)) if (nx == ny and not w.get("aniso")) else None
        parity = history_parity(name, [float(v) for v in r.history], r0) if r0 else None
        out = dict(workload=name, iterations=its, ms=ms, ms_per_step=ms / max(its, 1), parity=parity,
                   its_per_s=its / (ms * 1e-3), launches=int(launches), clocks=clocks,
                   bytes_per_iter=r.stats["algorithmic_bytes"] / max(its, 1) * world,
                   n_unknowns=nx * ny, nx=nx, ny=ny, outputs=outputs)
        peak, which = load_peaks()
        out["roofline_iter"] = dict(
            bound="hbm", achieved=r.stats["algorithmic_bytes"] / (ms * 1e-3) / 1e9, peak=peak, unit="GB/s",
            frac=r.stats["algorithmic_bytes"] / (ms * 1e-3) / 1e9 / peak, peak_source=which,
            note="per-GPU algorithmic bytes of all executed kernels / CUDA-event time of the iteration loop")
        if with_profile:
            rp = run_gpu_solver(kl, h, w, b, nx, ny, steps_eff, profile=True)
            barrier()
            prof = h.profile()
            tot = sum(p["ms"] for p in prof) or 1.0
            for p in prof:
                p["avg_us"] = 1e3 * p["ms"] / p["launches"]
                p["gbs"] = p["algorithmic_bytes"] / (p["ms"] * 1e-3) / 1e9 if p["ms"] > 0 else 0.0
                p["frac_of_peak"] = p["gbs"] / peak
                p["share"] = p["ms"] / tot
            out["kernels"] = prof
            dom = max(prof, key=lambda p: p["ms"]) if prof else None
            if dom:
                traffic, tsrc = None, None
                try:
                    tpath = os.path.join(ROOT, "profiles", "r02_traffic.json")
                    if not os.path.exists(tpath):
                        tpath = os.path.join(ROOT, "profiles", "r01_traffic.json")
                    with open(tpath) as tf:
                        tj = json.load(tf)
                    key = dom["name"].split(" ")[0]
                    ent = tj["bytes_per_unknown"].get(key)
                    if ent and "measured" in ent:
                        traffic = ent["measured"] * n_loc      # bytes per launch on this rank
                        tsrc = tj["source"]
                except Exception:
                    pass
                out["roofline"] = dict(bound="hbm", achieved=dom["gbs"], peak=peak, unit="GB/s",
                                       frac=dom["gbs"] / peak, traffic=traffic, kernel=dom["name"],
                                       algorithmic_bytes_per_launch=dom["algorithmic_bytes"] / dom["launches"],
                                       avg_launch_us=dom["avg_us"], peak_source=which, traffic_source=tsrc)
            h.set_option(8, 0)
        if with_e2e:
            # the reference-facing call with HOST buffers: H2D of b and D2H of x inside the timed region
            bh = torch.empty(n_loc, dtype=torch.float64).pin_memory()
            bh.copy_(b)
            del b
            torch.cuda.empty_cache()
            bn = bh.numpy()
            xh = torch.empty(n_loc, dtype=torch.float64).pin_memory()
            run_gpu_solver(kl, h, w, bn, nx, ny, min(steps_eff, max(m, 3)))   # warm the host-buffer path
            barrier()
            h.set_output_buffer(xh.numpy())
            t0 = time.perf_counter()
            r2 = run_gpu_solver(kl, h, w, bn, nx, ny, steps_eff)
            barrier()
            wall = max_over_ranks(time.perf_counter() - t0)
            tot_ms = max_over_ranks(r2.stats["total_ms"])
            # the same call with PAGEABLE host arrays (what a Fortran `allocate` gives the drivers)
            pageable = None
            try:
                bp = np.array(bn, copy=True)
                h.set_output_buffer(np.empty_like(bp))
                barrier()
                r3 = run_gpu_solver(kl, h, w, bp, nx, ny, steps_eff)
                barrier()
                pageable = r3.stats["iterations"] / (max_over_ranks(r3.stats["total_ms"]) * 1e-3)
                del bp
            except Exception as ex:  # pragma: no cover
                pageable = str(ex)[:100]
            out["e2e"] = dict(value=r2.stats["iterations"] / (tot_ms * 1e-3), unit="iterations/s",
                              value_pageable_host=pageable,
                              h2d_bytes_per_step=r2.stats["h2d_bytes"] * world / max(r2.stats["iterations"], 1),
                              d2h_bytes_per_step=r2.stats["d2h_bytes"] * world / max(r2.stats["iterations"], 1),
                              total_ms=tot_ms, wall_ms=wall * 1e3,
                              note="one solver call of K iterations through the C ABI with pinned host buffers "
                                   "(b uploaded, x downloaded once per call; device event time incl. copies); "
                                   "value_pageable_host = the same with ordinary (pageable) host arrays")
        return out

    primary = measure(args.workload, args.steps, args.warmup, True, True, keep_outputs=bool(args.dump_outputs))
    if args.dump_outputs:
        os.makedirs(args.dump_outputs, exist_ok=True)
        suffix = f"_rank{rank}" if world > 1 else ""
        for k, v in primary["outputs"].items():
            np.save(os.path.join(args.dump_outputs, f"{k}{suffix}.npy"), v)
    extras = {}
    if world == 1 and args.extras:
        for name, st in (("gmres4096", 95), ("gmres4096sel", 95), ("pcg16384", args.steps), ("bicgstab8192", args.steps),
                         ("hh1024", 95), ("gmres300", 475)):
            if name == args.workload or (args.only_extras and name not in args.only_extras.split(",")):
                continue
            try:
                e = measure(name, st, st if WORKLOADS[name]["m"] else 3, False, True)
                extras[name] = {k: e[k] for k in ("iterations", "ms_per_step", "its_per_s", "launches",
                                                    "roofline_iter", "kernels", "parity") if k in e}
            except Exception as ex:  # pragma: no cover
                extras[name] = {"error": str(ex)[:200]}

    cpu = None
    if rank == 0 and world == 1 and args.cpu_baseline:
        cpu = cpu_baseline(args.workload, budget_s=args.cpu_budget)

    if rank == 0:
        w = WORKLOADS[args.workload]
        line = {
            "metric": "krylov_iterations_per_s", "value": primary["its_per_s"], "unit": "iterations/s",
            "n_gpus": world, "steps": primary["iterations"], "warmup": args.warmup,
            "ms_per_step": primary["ms_per_step"], "higher_is_better": True, "scaling": w["scaling"],
            "vs_baseline": None, "dtype": "f64", "data": "synthetic (x_true=1, b=A*1, no RNG)",
            "config": {"workload": workload_string(args.workload, world),
                       "name": args.workload, "partition": f"row-slab x{world}",
                       "comm": ("none" if world == 1 else ("nvlink-peer-memory (IPC) all-reduce + halo push"
                                                            if h.get_option(10) else "nccl send/recv + allreduce")),
                       "l2": "inputs larger than L2 (no flush needed)", "bytes_per_iteration": primary["bytes_per_iter"],
                       "roofline_iter_frac": primary["roofline_iter"]["frac"],
                       "parity": primary.get("parity"),
                       "extras": {k: {"its_per_s": round(v["its_per_s"], 2), "ms_per_step": round(v["ms_per_step"], 5),
                                      "roofline_iter_frac": round(v["roofline_iter"]["frac"], 4),
                                      "parity_max_rel": (v.get("parity") or {}).get("max_rel")}
                                  for k, v in extras.items() if "its_per_s" in v}},
            "clocks": primary["clocks"], "gpu_launches": primary["launches"],
            "roofline": primary.get("roofline"), "roofline_iter": primary["roofline_iter"],
            "kernels": primary.get("kernels"), "e2e": primary.get("e2e"),
            "cpu_baseline": cpu, "extra": extras,
        }
        print(json.dumps(line))
    if dist:
        dist.barrier()
        dist.destroy_process_group()


def cpu_baseline(workload, budget_s=20.0, threads=None, with_six=True):
    """Time the oracle (C/OpenMP restatement of the reference's *_omp routine) on the host cores of this box.
    Built here with the reference's own flags (-O3 -fopenmp -march=native -funroll-loops, CMakeLists.txt:5).
    `value` = all host cores; `value_6_threads` = the reference drivers' own setting (tests/test_cg.f90:25)."""
    import numpy as np
    from oracle import oracle as ko

    so = ko.build_native()
    w = WORKLOADS[workload]
    cores = threads or os.cpu_count()
    ns = w["nx"]
    n = ns * ns
    A = ko.stvec_fn()
    M = ko.cbpr2_fn() if w["pc"] else None
    b = np.zeros(n)
    b.reshape(ns, ns)[0, :] += 1; b.reshape(ns, ns)[-1, :] += 1
    b.reshape(ns, ns)[:, 0] += 1; b.reshape(ns, ns)[:, -1] += 1       # b = A*1 (values 0/1/2)

    def run(iters):
        t0 = time.perf_counter()
        if w["solver"] == "cg_omp":
            ko.cg_omp(A, b, 0.0, iters, history_cap=1)
        elif w["solver"] == "pcg_omp":
            ko.pcg_omp(A, b, 0.0, iters, M, P_REF, history_cap=1)
        elif w["solver"] == "pbicgstab_omp":
            ko.pbicgstab_omp(A, b, 0.0, iters, M, P_REF, history_cap=1)
        elif w["solver"] == "gmres_mgsr_omp":
            ko.gmres_mgsr_omp(A, b, iters, 0.0, M, P_REF, max_restarts=1, skip_verr=True, history_cap=1)
        else:
            ko.gmres_hh(A, b, iters, 0.0, None, max_stages=1, skip_verr=True, history_cap=1)
        return time.perf_counter() - t0

    def rate(nthreads, budget):
        # a short run (setup + i0 iterations), then a longer one; rate from the difference
        ko.set_threads(nthreads)
        i0 = 2
        t_short = run(i0)
        per_it = max(t_short / (i0 + 2), 1e-4)
        i1 = int(min(max((budget * 0.6) / per_it, i0 + 3), 400))
        if w["m"]:
            i1 = min(i1, w["m"])
        t_long = run(i1)
        return (i1 - i0) / max(t_long - t_short, 1e-9), i0, i1, t_short, t_long

    r_all, i0, i1, t_short, t_long = rate(cores, budget_s * (0.6 if with_six else 1.0))
    out = {"value": r_all, "unit": "iterations/s", "cores": cores, "kind": "port",
           "sample": f"{w['solver']} on {ns}x{ns}: ({i1}-{i0}) iterations, time difference of two runs "
                     f"({t_long:.2f}s - {t_short:.2f}s) so that allocation/first-touch cancels; "
                     f"oracle/krylov_oracle.c, gcc -O3 -fopenmp -march=native -funroll-loops built on this box "
                     f"({os.path.basename(so)}), OMP threads = {cores}"}
    if with_six and cores > 6:
        r6, j0, j1, _, _ = rate(6, budget_s * 0.4)
        out["value_6_threads"] = r6
        out["sample"] += f"; value_6_threads: the reference drivers' own 6 threads (tests/test_cg.f90:25), ({j1}-{j0}) iterations"
    ko.set_threads(1)
    return out


def reference_arm(args):
    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    w = WORKLOADS[args.workload]
    cb = cpu_baseline(args.workload, budget_s=max(10.0, min(120.0, 2.0 * (args.steps + args.warmup))))
    line = {
        "impl": "reference", "metric": "krylov_iterations_per_s", "value": cb["value"], "unit": "iterations/s",
        "n_gpus": world, "steps": args.steps, "warmup": args.warmup, "ms_per_step": 1e3 / cb["value"],
        "higher_is_better": True, "scaling": w["scaling"], "vs_baseline": None, "dtype": "f64",
        "data": "synthetic (x_true=1, b=A*1, no RNG)",
        "config": {"workload": workload_string(args.workload, world), "name": args.workload,
                   "note": "reference is Fortran; no Fortran compiler on this box: C/OpenMP restatement "
                           "(oracle/) of the same routine on all host cores"},
        "cpu_baseline": cb,
        "e2e": {"value": cb["value"], "unit": "iterations/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=50)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--workload", default="cg16384", choices=sorted(WORKLOADS))
    ap.add_argument("--no-extras", dest="extras", action="store_false")
    ap.add_argument("--only-extras", default="", help="comma-separated subset of the extra workloads")
    ap.add_argument("--no-cpu-baseline", dest="cpu_baseline", action="store_false")
    ap.add_argument("--cpu-budget", type=float, default=20.0)
    ap.add_argument("--dump-outputs", metavar="DIR", default="",
                    help="write what the timed solver call returned (x, iteration counts, residual history) "
                         "as DIR/<name>.npy")
    args = ap.parse_args()
    if args.dump_outputs and args.impl == "reference":
        ap.error("--dump-outputs applies to the GPU implementation")
    if args.impl == "reference":
        reference_arm(args)
    else:
        gpu_arm(args)


if __name__ == "__main__":
    main()
