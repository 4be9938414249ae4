"""The C++ twins of the reference's driver programs (drivers/*.cpp = tests/*.f90 of the reference), run as
executables against libkrylov_b200.so: the iteration counts they PRINT must be the oracle's (and, where a golden
exists, the reference's own: tests/golden/reference_f90.json).  Plus: the ISO_C_BINDING shim and the reference's
Fortran drivers are compiled and run when a Fortran compiler exists (skipped otherwise -- none in this image)."""
import os
import re
import shutil
import subprocess

import numpy as np
import pytest

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
DRV = os.path.join(ROOT, "drivers")
P = (8.2, 0.2)


def run(*argv, timeout=600):
    exe = os.path.join(DRV, argv[0])
    if not os.path.exists(exe):
        subprocess.check_call(["make", "-C", DRV], stdout=subprocess.DEVNULL)
    out = subprocess.run([exe, *map(str, argv[1:])], capture_output=True, text=True, timeout=timeout, check=True).stdout
    return out


def test_test_poisson_mf_prints_the_oracle_counts(ko):
    """tests/test_poisson_mf.f90:27-85 at BASELINE config 1 (300^2, m = 95, rtol 1e-8): HH+cbpr2 then MGSR+cbpr2."""
    out = run("test_poisson_mf", 300, 95, "1e-8")
    its = [(int(a), int(b)) for a, b in re.findall(r"Iterations until convergence:\s+(\d+)\s+Stages=\s*(\d+)", out)]
    b = ko.manufactured_rhs(ko.stvec_fn(), 300)
    hh = ko.gmres_hh(ko.stvec_fn(), b, 95, 1e-8, ko.cbpr2_fn(), P, skip_verr=True)
    mg = ko.gmres_mgsr_omp(ko.stvec_fn(), b, 95, 1e-8, ko.cbpr2_fn(), P, skip_verr=True)
    assert its == [(hh.iterations, hh.restart_out), (mg.iterations, mg.restart_out)] == [(439, 5), (439, 5)], out
    lmax = [float(v) for v in re.findall(r"Max error L_max:\s+(\S+)", out)]
    assert len(lmax) == 2 and max(lmax) < 1e-4
    # and at the reference driver's own tolerance on a small grid, against the reference's OWN printed numbers
    import json
    with open(os.path.join(ROOT, "tests", "golden", "reference_f90.json")) as f:
        ref = json.load(f)["cases"]["program_test_poisson_mf_24_20"]
    want = [r[1] for r in ref["records"] if r and r[0] == "Iterations until convergence:"]
    out = run("test_poisson_mf", 24, 20)
    got = [int(a) for a in re.findall(r"Iterations until convergence:\s+(\d+)", out)]
    assert len(got) == 2 and all(abs(g - w) <= 1 for g, w in zip(got, want)), (got, want)


def test_test_cg_and_test_bicgstab_tables(ko):
    """tests/test_cg.f90:37-52 / tests/test_bicgstab.f90:37-53: grids 300, 350, 400 (first three of the 15)."""
    out = run("test_cg", "cg", 3)
    rows = [ln.split() for ln in out.splitlines() if re.match(r"^\s+\d+\s+\d+\s+\d+\s", ln)]
    assert [int(r[1]) for r in rows] == [300 * 300, 350 * 350, 400 * 400]
    for r in rows:
        ns = int(round(np.sqrt(int(r[1]))))
        o = ko.pcg_omp(ko.stvec_fn(), ko.manufactured_rhs(ko.stvec_fn(), ns), 1e-9, 10000, ko.cbpr2_fn(), P)
        assert abs(int(r[2]) - o.iter) <= 1, (ns, r[2], o.iter)
        assert float(r[4]) < 1e-9 and float(r[6]) < 1e-8
    out = run("test_cg", "bicgstab", 2)
    rows = [ln.split() for ln in out.splitlines() if re.match(r"^\s+\d+\s+\d+\s+\d+\s", ln)]
    for r in rows:
        ns = int(round(np.sqrt(int(r[1]))))
        o = ko.pbicgstab_omp(ko.stvec_fn(), ko.manufactured_rhs(ko.stvec_fn(), ns), 1e-9, 10000, ko.cbpr2_fn(), P)
        assert abs(int(r[2]) - o.iter) <= max(3, o.iter // 10) and float(r[6]) < 1e-6


def _table(out):
    return [ln.split() for ln in out.splitlines() if re.match(r"^\s*\d+\s+\d+\s+\d+\s+\d+\s+\d+\s", ln)]


def test_restart_sweep_and_grid_sweep_and_strong_scaling(ko):
    """tests/weak_scaling.f90:47-62 (restart-size sweep), tests/test1.f90:34-45 (grid sweep, m = 90) and
    tests/strong_scaling.f90:44-55 (six solves, m = 50): the printed counts equal the oracle's."""
    rows = _table(run("restart_sweep", 100, 3, "mgsr"))
    b = ko.manufactured_rhs(ko.stvec_fn(), 100)
    for r, m in zip(rows, (20, 25, 30)):
        o = ko.gmres_mgsr_omp(ko.stvec_fn(), b, m, 1e-8, ko.cbpr2_fn(), P, skip_verr=True)
        assert int(r[4]) == m and int(r[2]) == o.iterations and int(r[3]) == o.restart_out, (r, o.iterations)
    rows = _table(run("restart_sweep", 100, 2, "hh"))
    for r, m in zip(rows, (20, 25)):
        o = ko.gmres_hh(ko.stvec_fn(), b, m, 1e-8, ko.cbpr2_fn(), P, skip_verr=True)
        assert int(r[2]) == o.iterations, (r, o.iterations)
    rows = _table(run("test1", 2, 100, 30, "1e-10"))          # grids 100, 130 at m = 90
    assert [int(r[1]) for r in rows] == [100 * 100, 130 * 130]
    for r in rows:
        ns = int(round(np.sqrt(int(r[1]))))
        o = ko.gmres_mgsr_omp(ko.stvec_fn(), ko.manufactured_rhs(ko.stvec_fn(), ns), 90, 1e-10, ko.cbpr2_fn(), P, skip_verr=True)
        assert int(r[4]) == 90 and abs(int(r[2]) - o.iterations) <= 1 and float(r[7]) < 1e-6
    rows = _table(run("strong_scaling", 128, 6, "1e-10"))
    o = ko.gmres_mgsr_omp(ko.stvec_fn(), ko.manufactured_rhs(ko.stvec_fn(), 128), 50, 1e-10, ko.cbpr2_fn(), P, skip_verr=True)
    assert len(rows) == 6 and all(int(r[2]) == int(rows[0][2]) for r in rows)      # six identical solves
    assert abs(int(rows[0][2]) - o.iterations) <= 1


def test_fortran_shim_compiles_and_reference_driver_runs():
    """fortran/krylov_b200.f90 (ISO_C_BINDING shim with the reference's module names) + the reference's own
    tests/test_poisson_mf.f90, when a Fortran compiler exists and KRYLOV_REFERENCE names the reference's source tree
    (it is not part of this repository)."""
    fc = shutil.which("gfortran") or shutil.which("flang") or shutil.which("nvfortran")
    ref = os.environ.get("KRYLOV_REFERENCE", "")
    if not fc:
        pytest.skip("no Fortran compiler in this image (gfortran / flang / nvfortran all absent)")
    if not ref or not os.path.exists(os.path.join(ref, "tests", "test_poisson_mf.f90")):
        pytest.skip("set KRYLOV_REFERENCE to the reference's source tree (AlexanderGSC/gmres) to run its driver")
    import tempfile
    with tempfile.TemporaryDirectory() as td:
        exe = os.path.join(td, "test_poisson_mf")
        subprocess.check_call([fc, "-O2", "-J", td, "-o", exe, os.path.join(ROOT, "fortran", "krylov_b200.f90"),
                               os.path.join(ref, "tests", "test_poisson_mf.f90"), "-L" + os.path.join(ROOT, "gmres_b200"),
                               "-lkrylov_b200", "-Wl,-rpath," + os.path.join(ROOT, "gmres_b200")])
        out = subprocess.run([exe, "100", "95"], capture_output=True, text=True, timeout=600, check=True).stdout
        its = [int(a) for a in re.findall(r"Iterations until convergence:\s+(\d+)", out)]
        assert len(its) == 2 and all(abs(i - 152) <= 2 for i in its), out
