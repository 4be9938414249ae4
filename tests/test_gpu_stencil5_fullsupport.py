"""KL_OP_STENCIL5 (convection-diffusion, kl.stencil5 / kl.convdiff) on right-hand sides with support on the whole grid,
at the benchmark's grid sizes: what test_gpu_fullsupport.py does for the Poisson and anisotropic operators, for the
general 5-point operator.  Its fused, TMA and temporally blocked kernels (cbpr2, ChCheb / ChChebCont, ChGmresStep,
ChBiDir / ChBiS, ChCgPass, the generic S5<F> kernels) are separate instantiations that compile unlike their
KL_OP_ANISO5 twins (DESIGN.md section 3.2), and for every convection-diffusion weight set A*1 is zero away from the
boundary, so the b = A*1 tests of test_gpu_stencil5.py leave the interior CTAs multiplying zeros.  Here every input is
a seeded standard normal vector generated on the device, and

  A. point-wise kernels (operator, cbpr2, cheb(k)) are compared BIT FOR BIT with the CPU twin (tests/stencil5_twin.c)
     or the oracle's preconditioners run on it, at the bench sizes, over the geometry options and the edge shapes;
  B. solver paths the code promises to be bit-identical are compared bit for bit: GMRES with the one-pass step
     (ChGmresStep) against the two kernels, pair CG against one-pass CG, eager launches against graph replay;
  C. CG's fused reductions are compared with np.longdouble sums;
  D. the solvers are compared with restatements of the reference recurrences in FP64 torch (bench sizes), which are
     calibrated against np.longdouble in the same run.

Every bar of C and D (below) is >= 10x the largest deviation observed on a B200 (1000 W power limit), >= 10x the FP64
reference's own deviation from np.longdouble at the calibration size, and <= 1/100 of what a one-CTA defect in the
reference operator (wu * x_up dropped on one interior 240-column patch) moves.  Each test prints what it observes
(pytest -s).
"""
import contextlib

import numpy as np
import pytest

import stencil5_twin as tw
from parity import hist_rel
from test_gpu_fullsupport import (EDGE_NX, EDGE_NY, VERR, NpOps, TorchOps, _defect, _free, _ld_first_residual,
                                  cbpr2_ref, cheb_ref, hrel, ld, ld_ok, needs_ld, oracle_threads, randn, ref_bicgstab,
                                  ref_cg, ref_gmres_cycle, xrel)
from test_gpu_fullsupport import opts as _fs_opts

gpu = pytest.mark.gpu

# include/krylov_b200.h (the options test_gpu_fullsupport.py does not name)
ORTHO, USE_GRAPH, FUSE = 1, 5, 7

W = (4.1, 1.37, 0.61, 0.83, 1.29)           # nonsymmetric, real spectrum (test_gpu_stencil5.py)
CENTRAL = (4.0, 1.5, 0.5, 0.75, 1.25)       # kl.convdiff(0.5, 0.25): central differences
UPWIND = (8.0, 5.0, 1.0, 1.0, 1.0)          # kl.convdiff(2, 0, upwind=True)
SHIFTED = (4.1, 1.0, 1.0, 1.0, 1.0)         # symmetric: the shifted Laplacian
ANISO_SYM = (2.07, 1.0, 1.0, 0.01, 0.01)    # symmetric: (2(a + b) + sigma, a, a, b, b), a = 1, b = 0.01, sigma = 0.05
NONSYM = (W, CENTRAL, UPWIND)
DEGREES = (1, 2, 3, 4, 5, 6, 8, 12)         # one chain, the continuation chunks, the LEAN interior march

# bars (see the module docstring; the calibrations are test_cg_reductions_vs_longdouble, test_solvers_1024_vs_longdouble
# and test_gmres_vs_longdouble; the defects test_cg_16384_all_modes, test_bicgstab_8192_three_paths and
# test_gmres_4096_one_cycle)
BAR_RED1 = 1e-14        # CG history[0] against a longdouble sum: observed <= 2.2e-16
BAR_RED2 = 1e-14        # CG history[1] against the FP64 reference: observed <= 3.3e-16
BAR_CG = 1e-13          # CG on the shifted Laplacian, 24 / 25 iterations: observed <= 1.3e-15; reference 6.7e-16
BAR_PCG = 1e-13         # PCG (cbpr2 20 iterations, cheb(4) 12): observed <= 3.3e-15; reference 9.0e-16
# PBiCGSTAB on convdiff(0.5, 0.25), both preconditioners on the exact interval.  The FP64 recurrence leaves longdouble's
# in jumps that depend on b (numpy float64 against np.longdouble at 1024^2, four seeds): with cbpr2 by 10-100x per
# iteration from the sixth on (3.4e-13 after 6, 5.7e-12 after 7, 0.28 after 12), with cheb(4) up to 2.1e-13 after
# 6 iterations and 4.4e-12 after 7 (1.7e-11 after 12 in the FP64 torch reference on the B200).  Hence 5 and 6.
ITS_BICG = {"cbpr2": 5, "cheb4": 6}
BAR_BICG = {"cbpr2": 1e-12,         # observed <= 1.2e-14; reference 2.7e-15
            "cheb4": 1e-11}         # observed <= 1.5e-13 (1024^2), 1.9e-14 (8192^2); reference 2.1e-14
BAR_GMRES = 1e-11       # one GMRES(95) cycle (CGS2, MGS2, selective): observed <= 8.2e-14; the FP64 reference's own
                        # deviation from longdouble reaches 2.2e-13 (cheb(4), 256^2)
BAR_HH = 1e-9           # Householder GMRES(95) against the multi-threaded oracle: observed <= 1.0e-11 (x); the
                        # oracle's own deviation from longdouble is 5.6e-13 at 256^2, the kernels' 1.2e-14


@contextlib.contextmanager
def opts(h, **kv):
    """test_gpu_fullsupport.opts, plus ORTHO, USE_GRAPH and FUSE"""
    more = {globals()[k]: kv.pop(k) for k in ("ORTHO", "USE_GRAPH", "FUSE") if k in kv}
    with _fs_opts(h, **kv):
        old = {k: h.get_option(k) for k in more}
        try:
            for k, v in more.items():
                h.set_option(k, v)
            yield
        finally:
            for k, v in old.items():
                h.set_option(k, v)


# ---------------------------------------------------------------------------------------------------------------
# references
# ---------------------------------------------------------------------------------------------------------------
def np_s5(w, nx, ny, defect=None):
    """numpy restatement of KL_OP_STENCIL5, y = c x - ((wl x_l + wr x_r) + (wd x_d + wu x_u)) with zero Dirichlet
    boundary (idx = i + j*nx, "d" = j+1, "u" = j-1), in any float dtype.  `defect` (test_gpu_fullsupport._defect)
    adds wu * x_u back on one patch, i.e. drops that CTA's upper halo line."""
    c, wl, wr, wd, wu = w

    def A(x):
        X = x.reshape(ny, nx)
        Pd = np.pad(X, 1)
        y = c * X - ((wl * Pd[1:-1, :-2] + wr * Pd[1:-1, 2:]) + (wd * Pd[2:, 1:-1] + wu * Pd[:-2, 1:-1]))
        if defect:
            j, c0, c1 = defect
            y[j, c0:c1] += wu * X[j - 1, c0:c1]
        return y.reshape(-1)
    return A


def t_s5(torch, w, nx, ny, defect=None):
    """the same on torch tensors"""
    c, wl, wr, wd, wu = w

    def A(x):
        X = x.view(ny, nx)
        Pd = torch.nn.functional.pad(X, (1, 1, 1, 1))
        y = c * X - ((wl * Pd[1:-1, :-2] + wr * Pd[1:-1, 2:]) + (wd * Pd[2:, 1:-1] + wu * Pd[:-2, 1:-1]))
        del Pd
        if defect:
            j, c0, c1 = defect
            y[j, c0:c1] += wu * X[j - 1, c0:c1]
        return y.reshape(-1)
    return A


def interval(kl, w, nx, ny):
    """the exact spectrum of the operator on the grid, as the (hi, lo) params of cbpr2 and cheb(k)"""
    lo, hi = kl.stencil5_spectrum(kl.stencil5(*w), nx, ny)
    return hi, lo


def _identity(r):
    return r


# ---------------------------------------------------------------------------------------------------------------
# CPU: both references against the oracle run on the twin (64^2, random b)
# ---------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("kind", ["torch", "longdouble"])
def test_references_match_oracle_on_twin(ko, kind):
    import gmres_b200 as kl
    if kind == "longdouble" and not ld_ok():
        pytest.skip("np.longdouble is no wider than float64 on this platform")
    assert kl.convdiff(0.5, 0.25).w5 == CENTRAL and kl.convdiff(2, 0, upwind=True).w5 == UPWIND
    ns, n = 64, 64 * 64
    b = np.random.default_rng(6464).standard_normal(n)
    if kind == "torch":
        import torch
        ops, bv, op = TorchOps, torch.from_numpy(b.copy()), lambda w, **kw: t_s5(torch, w, ns, ns, **kw)
    else:
        ops, bv, op = NpOps, b.astype(np.longdouble), lambda w, **kw: np_s5(w, ns, ns, **kw)
    S, C, Wo = op(SHIFTED), op(CENTRAL), op(W)
    ps, pc, pw = interval(kl, SHIFTED, ns, ns), interval(kl, CENTRAL, ns, ns), interval(kl, W, ns, ns)
    out = {}
    o = ko.cg_omp(tw.stencil_fn(ko, SHIFTED), b, 0.0, 60)
    out["cg shifted"] = (ref_cg(ops, S, bv, 60), o)
    o = ko.pcg_omp(tw.stencil_fn(ko, SHIFTED), b, 0.0, 20, ko.cheb_fn(4), ps)
    out["pcg cheb4 shifted"] = (ref_cg(ops, S, bv, 20, cheb_ref(S, 4, ps)), o)
    o = ko.pbicgstab_omp(tw.stencil_fn(ko, CENTRAL), b, 0.0, ITS_BICG["cbpr2"], ko.cbpr2_fn(), pc)
    out["bicgstab cbpr2 central"] = (ref_bicgstab(ops, C, bv, ITS_BICG["cbpr2"], cbpr2_ref(C, pc)), o)
    o = ko.gmres_mgsr_omp(tw.stencil_fn(ko, W), b, 40, 0.0, ko.cbpr2_fn(), pw, max_restarts=1, skip_verr=True)
    out["gmres40 cbpr2 W"] = (ref_gmres_cycle(ops, Wo, bv, 40, cbpr2_ref(Wo, pw)), o)
    for name, ((hist, x), o) in out.items():
        d, dx = hrel(hist, o.history), xrel(x, o.x)
        print(f"{kind} reference vs oracle on the twin, {name} at 64^2: history {d:.2e}, x {dx:.2e}")
        assert d < 1e-12 and dx < 1e-12, name
    # the defect is visible at this size too
    hist, _ = ref_cg(ops, op(SHIFTED, defect=_defect(ns, ns)), bv, 60)
    assert hrel(hist, out["cg shifted"][1].history) > 1e-6
    fe, _ = ref_gmres_cycle(ops, op(W, defect=_defect(ns, ns)), bv, 40, cbpr2_ref(op(W, defect=_defect(ns, ns)), pw))
    assert hrel(fe, out["gmres40 cbpr2 W"][1].history) > 1e-6


# ---------------------------------------------------------------------------------------------------------------
# GPU fixtures
# ---------------------------------------------------------------------------------------------------------------
@pytest.fixture(scope="module")
def env():
    import torch
    import gmres_b200 as kl
    h = kl.Handle(0)
    h.set_option(VERR, 0)
    yield kl, h, torch
    h.close()
    torch.cuda.empty_cache()


# ---------------------------------------------------------------------------------------------------------------
# A. point-wise kernels, bit for bit
# ---------------------------------------------------------------------------------------------------------------
@gpu
@pytest.mark.parametrize("n", [16384, 8192])
def test_pointwise_bench_size_vs_twin(env, ko, n):
    """The operator for the three nonsymmetric weight sets against the twin; cbpr2 (16384^2) and cheb(k) (8192^2) on W
    against the oracle's cbpr2 / ko_cheb run on the twin."""
    kl, h, torch = env
    x = randn(torch, n * n, n + 55)
    xh = x.cpu().numpy()
    with oracle_threads(ko):
        for w in NONSYM:
            y = h.apply(kl.stencil5(*w), x, n, n).cpu().numpy()
            yo = ko.apply(tw.stencil_fn(ko, w), xh, n, parallel=True)
            assert np.array_equal(y, yo), (n, w, np.abs(y - yo).max())
            del y, yo
        A, prm = kl.stencil5(*W), interval(kl, W, n, n)
        pcs = [(kl.cbpr2, ko.cbpr2_fn)] if n == 16384 else [(kl.cheb(k), lambda k=k: ko.cheb_fn(k)) for k in DEGREES]
        for M, Mo in pcs:
            z = h.apply_precond(M, A, x, prm, n, n).cpu().numpy()
            zo = ko.apply_precond(Mo(), tw.stencil_fn(ko, W), xh, prm, n, parallel=True)
            assert np.array_equal(z, zo), (n, M, np.abs(z - zo).max())
            del z, zo
    del x, xh
    _free(torch)


@gpu
@pytest.mark.parametrize("what", ["apply", "cbpr2", "cheb4"])
def test_geometry_option_sweep_8192(env, ko, what):
    """All 160 combinations of the stencil kernels' geometry options give the twin's (or the oracle-on-twin's) bits.
    Rows = 8 makes more tiles than the reduction buffer's 16384 slots: stencil_geometry's fallback."""
    kl, h, torch = env
    n = 8192
    x = randn(torch, n * n, 58)
    xh = x.cpu().numpy()
    A, prm = kl.stencil5(*W), interval(kl, W, n, n)
    with oracle_threads(ko):
        if what == "apply":
            ref = ko.apply(tw.stencil_fn(ko, W), xh, n, parallel=True)
            run = lambda: h.apply(A, x, n, n)
        else:
            M, Mo = (kl.cbpr2, ko.cbpr2_fn()) if what == "cbpr2" else (kl.cheb(4), ko.cheb_fn(4))
            ref = ko.apply_precond(Mo, tw.stencil_fn(ko, W), xh, prm, n, parallel=True)
            run = lambda: h.apply_precond(M, A, x, prm, n, n)
    ref = torch.from_numpy(ref).cuda()
    bad = []
    for tma in (1, 0):
        for pers in (0, 1):
            for stag in (0, 1):
                for tail in (-1, 0, 3, 7):
                    for rows in (0, 8, 13, 61, 128):
                        with opts(h, TMA=tma, PERSISTENT=pers, STAGGER=stag, TAIL=tail, ROWS=rows):
                            y = run()
                        if not torch.equal(y, ref):
                            bad.append((tma, pers, stag, tail, rows, float((y - ref).abs().max())))
    assert not bad, bad
    del x, xh, ref
    _free(torch)


@gpu
@pytest.mark.parametrize("nx", EDGE_NX)
def test_edge_shapes_pointwise(env, nx):
    """The edge shapes of test_gpu_fullsupport.py (strip widths, odd nx, short grids): the operator against the twin
    (rectangular grids), cbpr2 and cheb(k) on the chained / TMA path against one kernel per application on the
    generic S5<F> path (CHAIN = 0, TMA = 0).  A shape the library rejects must raise."""
    kl, h, torch = env
    rejected = []
    for ny in EDGE_NY:
        x = randn(torch, nx * ny, nx * 1000 + ny + 5)
        xh = x.cpu().numpy()
        try:
            y = h.apply(kl.stencil5(*W), x, nx, ny)
        except kl.KrylovError as e:
            rejected.append((ny, str(e)))
            continue
        assert np.array_equal(y.cpu().numpy(), tw.apply_xy(W, xh, nx, ny)), (nx, ny, W)
        for w in (CENTRAL, UPWIND):
            assert np.array_equal(h.apply(kl.stencil5(*w), x, nx, ny).cpu().numpy(), tw.apply_xy(w, xh, nx, ny)), \
                (nx, ny, w)
        for w in (W, CENTRAL):
            A, prm = kl.stencil5(*w), interval(kl, w, nx, ny)
            for M in [kl.cbpr2] + [kl.cheb(k) for k in DEGREES]:
                z = h.apply_precond(M, A, x, prm, nx, ny)
                with opts(h, CHAIN=0, TMA=0):
                    zs = h.apply_precond(M, A, x, prm, nx, ny)
                assert torch.equal(z, zs), (nx, ny, w, M, float((z - zs).abs().max()))
    print(f"nx {nx}: rejected {rejected}")
    assert all(ny < 25 for ny, _ in rejected), rejected


@gpu
@pytest.mark.parametrize("ns", [63, 64, 65, 66, 226, 240, 242, 254, 256, 257, 542])
def test_edge_shapes_square_vs_oracle(env, ko, ns):
    kl, h, torch = env
    x = randn(torch, ns * ns, ns + 5)
    xh = x.cpu().numpy()
    for w in NONSYM:
        y = h.apply(kl.stencil5(*w), x, ns, ns).cpu().numpy()
        assert np.array_equal(y, ko.apply(tw.stencil_fn(ko, w), xh, ns)), (ns, w)
    A, prm = kl.stencil5(*W), interval(kl, W, ns, ns)
    for M, Mo in [(kl.cbpr2, ko.cbpr2_fn)] + [(kl.cheb(k), lambda k=k: ko.cheb_fn(k)) for k in DEGREES]:
        z = h.apply_precond(M, A, x, prm, ns, ns).cpu().numpy()
        assert np.array_equal(z, ko.apply_precond(Mo(), tw.stencil_fn(ko, W), xh, prm, ns)), (ns, M)


# ---------------------------------------------------------------------------------------------------------------
# B. solver paths that are bit-identical by construction
# ---------------------------------------------------------------------------------------------------------------
@gpu
@pytest.mark.parametrize("nx,ny,m", [(1024, 1024, 30), (2048, 640, 20), (130, 76, 12)])
def test_gmres_one_pass_step_equals_two_kernels(env, nx, ny, m):
    """GMRES-MGSR + cbpr2, three restart cycles: V_j = w/h, z = A V_j and w = cbpr2(z) as one temporally blocked pass
    (ChGmresStep) against the two kernels (CHAIN = 0), and eager launches (USE_GRAPH = 0) against the replayed
    restart-cycle graph: history, final_err and x bit for bit."""
    kl, h, torch = env
    for w in (W, CENTRAL):
        A, prm = kl.stencil5(*w), interval(kl, w, nx, ny)
        b = randn(torch, nx * ny, nx + ny + m)
        runs = {}
        for name, kv in (("chained", {}), ("two kernels", dict(CHAIN=0)), ("eager", dict(USE_GRAPH=0)),
                         ("two kernels eager", dict(CHAIN=0, USE_GRAPH=0))):
            with opts(h, MAX_RESTARTS=3, **kv):
                runs[name] = h.gmres_mgsr_omp(A, b, m, 0.0, kl.cbpr2, prm, nx=nx, ny=ny)
        g = runs["chained"]
        assert (g.n_out, g.restart_out) == (m, 3) and g.history.size == 3 * m
        for name, u in runs.items():
            assert (u.n_out, u.restart_out) == (g.n_out, g.restart_out), (w, name)
            assert np.array_equal(u.history, g.history), (w, name, hist_rel(u.history, g.history))
            assert np.array_equal(u.final_err, g.final_err) and torch.equal(u.x, g.x), (w, name)
    _free(torch)


@gpu
@pytest.mark.parametrize("n", [4096, 8192])
def test_cg_pair_equals_one_pass(env, n):
    """Pairs of passes (CG_ONEPASS = 2) against one pass per iteration (1) on both symmetric weight sets, bit for bit:
    24 iterations polled every 8 (graph-replayed batches) and 25 polled every 5 (batches that start on a pass B, a run
    that ends with the x flush), each with and without CUDA-graph replay."""
    kl, h, torch = env
    for w in (SHIFTED, ANISO_SYM):
        A = kl.stencil5(*w)
        b = randn(torch, n * n, n + int(100 * w[0]))
        for its, ce in ((24, 8), (25, 5)):
            runs = {}
            for mode in (1, 2):
                for graph in (1, 0):
                    with opts(h, CG_ONEPASS=mode, CHECK_EVERY=ce, USE_GRAPH=graph):
                        runs[mode, graph] = h.cg_omp(A, b, 0.0, its, nx=n, ny=n)
            g = runs[1, 1]
            for key, u in runs.items():
                assert u.iter == its and u.history.size == its, (w, its, key)
                assert np.array_equal(u.history, g.history), (w, its, key, hist_rel(u.history, g.history))
                assert torch.equal(u.x, g.x), (w, its, key)
            del runs, g
        del b
    _free(torch)


# ---------------------------------------------------------------------------------------------------------------
# C. CG's fused reductions against np.longdouble
# ---------------------------------------------------------------------------------------------------------------
@gpu
@needs_ld
@pytest.mark.parametrize("nx,ny", [(16384, 16384), (8192, 8192), (4112, 301), (542, 49), (256, 25), (66, 5),
                                   (240, 1000), (257, 49), (4096, 4096)])
def test_cg_reductions_vs_longdouble(env, nx, ny):
    """history[0] = ||b - alpha0 A b|| through one reduction of each CG mode against longdouble sums; history[1]
    (predicted beta, the pass's four fused sums) against the FP64 reference of two iterations.  Shifted Laplacian."""
    kl, h, torch = env
    A, At = kl.stencil5(*SHIFTED), t_s5(torch, SHIFTED, nx, ny)
    b = randn(torch, nx * ny, 13 * nx + ny)
    want0 = _ld_first_residual(b, At(b))
    want = ref_cg(TorchOps, At, b, 2)[0]
    for mode in (0, 1, 2):
        with opts(h, CG_ONEPASS=mode):
            g1 = h.cg_omp(A, b, 0.0, 1, nx=nx, ny=ny)
            g2 = h.cg_omp(A, b, 0.0, 2, nx=nx, ny=ny)
        d0, d1 = abs(g1.history[0] / want0 - 1), abs(g2.history[1] / want[1] - 1)
        print(f"cg reductions {nx}x{ny} mode {mode}: history[0] {d0:.2e} (bar {BAR_RED1:.0e}), "
              f"history[1] {d1:.2e} (bar {BAR_RED2:.0e})")
        assert g1.history.size == 1 and g2.history.size == 2 and g2.history[0] == g1.history[0]
        assert d0 < BAR_RED1 and d1 < BAR_RED2, (mode, d0, d1)
    del b
    _free(torch)


# ---------------------------------------------------------------------------------------------------------------
# D. calibration: the kernels and the FP64 torch reference against np.longdouble
# ---------------------------------------------------------------------------------------------------------------
@gpu
@needs_ld
def test_solvers_1024_vs_longdouble(env):
    """CG (all three modes), PCG and PBiCGSTAB at 1024^2 against np.longdouble, and the FP64 torch reference's own
    deviation from it, which bounds the bars of the bench-size tests."""
    kl, h, torch = env
    n = 1024
    b = randn(torch, n * n, 1029)
    ps, pc = interval(kl, SHIFTED, n, n), interval(kl, CENTRAL, n, n)
    S, C = kl.stencil5(*SHIFTED), kl.stencil5(*CENTRAL)
    cg_runs = {f"mode {m} check_every {c}": (lambda m=m, c=c: _cg_run(h, S, b, n, m, 25, c))
               for m in (0, 1, 2) for c in (8, 5)}
    cases = [
        ("cg shifted", BAR_CG, cg_runs, lambda o, A_, b_: ref_cg(o, A_, b_, 25), SHIFTED),
        ("pcg cbpr2 shifted", BAR_PCG, {"": lambda: h.pcg_omp(S, b, 0.0, 20, kl.cbpr2, ps, nx=n, ny=n)},
         lambda o, A_, b_: ref_cg(o, A_, b_, 20, cbpr2_ref(A_, ps)), SHIFTED),
        ("pcg cheb4 shifted", BAR_PCG, {"": lambda: h.pcg_omp(S, b, 0.0, 12, kl.cheb(4), ps, nx=n, ny=n)},
         lambda o, A_, b_: ref_cg(o, A_, b_, 12, cheb_ref(A_, 4, ps)), SHIFTED),
    ]
    for pcn, M, Mr in (("cbpr2", kl.cbpr2, cbpr2_ref), ("cheb4", kl.cheb(4), lambda A_, p: cheb_ref(A_, 4, p))):
        runs = {name: (lambda kv=kv, M=M, its=ITS_BICG[pcn]: _bicg_run(h, C, b, n, M, pc, its, kv))
                for name, kv in (("default", {}), ("chain 0", dict(CHAIN=0)), ("fuse 0", dict(FUSE=0)))}
        cases.append((f"bicgstab {pcn} central", BAR_BICG[pcn], runs,
                      lambda o, A_, b_, Mr=Mr, its=ITS_BICG[pcn]: ref_bicgstab(o, A_, b_, its, Mr(A_, pc)), CENTRAL))
    for name, bar, runs, ref, w in cases:
        hl, xl = ref(NpOps, np_s5(w, n, n), ld(b))
        ht, xt = ref(TorchOps, t_s5(torch, w, n, n), b)
        dt, dxt = hrel(ht, hl), xrel(xt.cpu().numpy(), xl)
        print(f"{name} 1024^2: FP64 torch reference vs longdouble: history {dt:.2e}, x {dxt:.2e} (bar {bar:.0e})")
        assert dt < bar / 10 and dxt < bar / 10, name
        for rn, run in runs.items():
            g = run()
            d, dx = hrel(g.history, hl), xrel(g.x.cpu().numpy(), xl)
            print(f"{name} {rn} 1024^2: kernels vs longdouble: history {d:.2e}, x {dx:.2e} (bar {bar:.0e})")
            assert d < bar and dx < bar, (name, rn, d, dx)
    _free(torch)


def _cg_run(h, A, b, n, mode, its, ce):
    with opts(h, CG_ONEPASS=mode, CHECK_EVERY=ce):
        return h.cg_omp(A, b, 0.0, its, nx=n, ny=n)


def _bicg_run(h, A, b, n, M, prm, its, kv):
    with opts(h, CHECK_EVERY=8, **kv):
        return h.pbicgstab_omp(A, b, 0.0, its, M, prm, nx=n, ny=n)


@gpu
@needs_ld
@pytest.mark.parametrize("n", [256, 512])
def test_gmres_vs_longdouble(env, ko, n):
    """One GMRES(95) cycle on convdiff(0.5, 0.25) (cbpr2; at 256^2 also cheb(4) and none, and Householder GMRES on W
    with the oracle) against np.longdouble: the kernels and the FP64 references.  Two sizes show whether the
    reference's own deviation grows with n."""
    kl, h, torch = env
    m = 95
    b = randn(torch, n * n, n + 95)
    pc = interval(kl, CENTRAL, n, n)
    An, At = np_s5(CENTRAL, n, n), t_s5(torch, CENTRAL, n, n)
    pcs = [("cbpr2", kl.cbpr2, lambda A_: cbpr2_ref(A_, pc))]
    if n == 256:
        pcs += [("cheb4", kl.cheb(4), lambda A_: cheb_ref(A_, 4, pc)), ("none", None, lambda A_: _identity)]
    for name, M, Mr in pcs:
        fl, xl = ref_gmres_cycle(NpOps, An, ld(b), m, Mr(An))
        ft, xt = ref_gmres_cycle(TorchOps, At, b, m, Mr(At))
        with opts(h, MAX_RESTARTS=1):
            g = h.gmres_mgsr_omp(kl.stencil5(*CENTRAL), b, m, 0.0, M, pc, nx=n, ny=n)
        d, dx, dt, dxt = hrel(g.history, fl), xrel(g.x.cpu().numpy(), xl), hrel(ft, fl), xrel(xt.cpu().numpy(), xl)
        print(f"gmres {name} {n}^2 m {m} vs longdouble: kernels history {d:.2e} x {dx:.2e}; "
              f"FP64 torch reference {dt:.2e} {dxt:.2e} (bar {BAR_GMRES:.0e})")
        assert g.n_out == m and dt < BAR_GMRES / 10 and dxt < BAR_GMRES / 10
        assert d < BAR_GMRES and dx < BAR_GMRES
    if n == 256:
        # Householder GMRES is held to the oracle (FP64) at 1024^2: the oracle's own deviation from longdouble here
        fl, xl = ref_gmres_cycle(NpOps, np_s5(W, n, n), ld(b), m, _identity)
        bh = b.cpu().numpy()
        o = ko.gmres_hh(tw.stencil_fn(ko, W), bh, m, 0.0, None, max_stages=1, skip_verr=True)
        do, dxo = hrel(o.history, fl), xrel(o.x, xl)
        print(f"hh oracle on the twin {n}^2 m {m} vs longdouble: history {do:.2e}, x {dxo:.2e} (bar {BAR_HH:.0e})")
        assert do < BAR_HH / 10 and dxo < BAR_HH / 10
        with opts(h, MAX_RESTARTS=1):
            for mode in (1, 0):
                with opts(h, HH_MODE=mode):
                    g = h.gmres_hh_omp(kl.stencil5(*W), bh, m, 0.0)
                d, dx = hrel(g.history, fl), xrel(g.x, xl)
                print(f"hh mode {mode} {n}^2 vs longdouble: history {d:.2e}, x {dx:.2e} (bar {BAR_HH:.0e})")
                assert d < BAR_HH and dx < BAR_HH
    _free(torch)


# ---------------------------------------------------------------------------------------------------------------
# D. the bench sizes against the FP64 torch reference
# ---------------------------------------------------------------------------------------------------------------
@gpu
def test_cg_16384_all_modes(env):
    """Shifted Laplacian at 16384^2: pairs (auto), one pass and two kernels, 24 iterations polled every 8 and 25 polled
    every 5; and the one-CTA defect against the bar."""
    kl, h, torch = env
    n = 16384
    A = kl.stencil5(*SHIFTED)
    b = randn(torch, n * n, 16384 + 41)
    At = t_s5(torch, SHIFTED, n, n)
    refs = {its: ref_cg(TorchOps, At, b, its) for its in (24, 25)}
    for mode in (-1, 1, 0):
        for its, ce in ((24, 8), (25, 5)):
            g = _cg_run(h, A, b, n, mode, its, ce)
            hr, xr = refs[its]
            d, dx = hrel(g.history, hr), xrel(g.x, xr)
            print(f"cg shifted {n}^2 mode {mode} its {its} check_every {ce}: history {d:.2e}, x {dx:.2e} "
                  f"(bar {BAR_CG:.0e})")
            assert g.iter == its and d < BAR_CG and dx < BAR_CG, (mode, its, d, dx)
            del g
    hd, xd = ref_cg(TorchOps, t_s5(torch, SHIFTED, n, n, defect=_defect(n, n)), b, 24)
    sh, sx = hrel(hd, refs[24][0]), xrel(xd, refs[24][1])
    print(f"cg shifted {n}^2 one-CTA defect: history {sh:.2e}, x {sx:.2e}: {min(sh, sx) / BAR_CG:.1e} x the bar")
    assert min(sh, sx) > 100 * BAR_CG
    del b, refs, hd, xd
    _free(torch)


@gpu
@pytest.mark.parametrize("case", ["pcg16384cbpr2", "pcg8192cheb4"])
def test_pcg_bench_size(env, case):
    kl, h, torch = env
    n = 16384 if case == "pcg16384cbpr2" else 8192
    b = randn(torch, n * n, n + 43)
    At, prm = t_s5(torch, SHIFTED, n, n), interval(kl, SHIFTED, n, n)
    M, Mr, its = (kl.cbpr2, cbpr2_ref(At, prm), 20) if n == 16384 else (kl.cheb(4), cheb_ref(At, 4, prm), 12)
    hr, xr = ref_cg(TorchOps, At, b, its, Mr)
    with opts(h, CHECK_EVERY=8):
        g = h.pcg_omp(kl.stencil5(*SHIFTED), b, 0.0, its, M, prm, nx=n, ny=n)
    d, dx = hrel(g.history, hr), xrel(g.x, xr)
    print(f"{case} shifted: history {d:.2e}, x {dx:.2e} (bar {BAR_PCG:.0e})")
    assert g.iter == its and d < BAR_PCG and dx < BAR_PCG
    del b, g, xr
    _free(torch)


@gpu
@pytest.mark.parametrize("pc", ["cbpr2", "cheb4"])
def test_bicgstab_8192_three_paths(env, pc):
    """PBiCGSTAB on convdiff(0.5, 0.25) at 8192^2: the default (ChBiDir / ChBiS), CHAIN = 0 and FUSE = 0; and the
    one-CTA defect against the bar."""
    kl, h, torch = env
    n = 8192
    b = randn(torch, n * n, 8192 + len(pc))
    At, prm = t_s5(torch, CENTRAL, n, n), interval(kl, CENTRAL, n, n)
    M, Mr = (kl.cbpr2, cbpr2_ref(At, prm)) if pc == "cbpr2" else (kl.cheb(4), cheb_ref(At, 4, prm))
    its, bar = ITS_BICG[pc], BAR_BICG[pc]
    hr, xr = ref_bicgstab(TorchOps, At, b, its, Mr)
    for name, kv in (("default", {}), ("chain 0", dict(CHAIN=0)), ("fuse 0", dict(FUSE=0))):
        g = _bicg_run(h, kl.stencil5(*CENTRAL), b, n, M, prm, its, kv)
        d, dx = hrel(g.history, hr), xrel(g.x, xr)
        print(f"bicgstab {pc} central 8192^2 {name} {its} its: history {d:.2e}, x {dx:.2e} (bar {bar:.0e})")
        assert g.iter == its and d < bar and dx < bar, (name, d, dx)
        del g
    Ad = t_s5(torch, CENTRAL, n, n, defect=_defect(n, n))
    hd, xd = ref_bicgstab(TorchOps, Ad, b, its, cbpr2_ref(Ad, prm) if pc == "cbpr2" else cheb_ref(Ad, 4, prm))
    sh, sx = hrel(hd, hr), xrel(xd, xr)
    print(f"bicgstab {pc} central 8192^2 one-CTA defect: history {sh:.2e}, x {sx:.2e}: {min(sh, sx) / bar:.1e} x the bar")
    assert min(sh, sx) > 100 * bar
    del b, xr, xd
    _free(torch)


@gpu
def test_gmres_4096_one_cycle(env):
    """One GMRES(95) cycle on convdiff(0.5, 0.25) at 4096^2: cbpr2 (ChGmresStep), cheb(4) and no preconditioner;
    CGS2, MGS2 and selective reorthogonalisation; gmres_mgsr_mf; and the one-CTA defect against the bar."""
    kl, h, torch = env
    n, m = 4096, 95
    b = randn(torch, n * n, 4096 + 95)
    A, At, prm = kl.stencil5(*CENTRAL), t_s5(torch, CENTRAL, n, n), interval(kl, CENTRAL, n, n)
    pcs = {"cbpr2": (kl.cbpr2, cbpr2_ref(At, prm)), "cheb4": (kl.cheb(4), cheb_ref(At, 4, prm)),
           "none": (None, _identity)}
    cases = [("cbpr2", 1, False), ("cheb4", 1, False), ("none", 1, False), ("cbpr2", 0, False), ("cbpr2", 2, False),
             ("cbpr2", 1, True)]
    refs, bad = {}, []
    for pcn, ortho, mf in cases:
        if pcn not in refs:
            refs[pcn] = ref_gmres_cycle(TorchOps, At, b, m, pcs[pcn][1])
        fr, xr = refs[pcn]
        with opts(h, MAX_RESTARTS=1, REORTH_ETA=300, ORTHO=ortho):
            g = (h.gmres_mgsr_mf if mf else h.gmres_mgsr_omp)(A, b, m, 0.0, pcs[pcn][0], prm, nx=n, ny=n)
        d, dx = hrel(g.history, fr), xrel(g.x, xr)
        print(f"gmres {pcn} ortho {ortho}{' mf' if mf else ''} central 4096^2: history {d:.2e}, x {dx:.2e} "
              f"(bar {BAR_GMRES:.0e})")
        if not (g.n_out == m and d < BAR_GMRES and dx < BAR_GMRES):
            bad.append((pcn, ortho, mf, g.n_out, d, dx))
        del g
    Ad = t_s5(torch, CENTRAL, n, n, defect=_defect(n, n))
    fd, xd = ref_gmres_cycle(TorchOps, Ad, b, m, cbpr2_ref(Ad, prm))
    sh, sx = hrel(fd, refs["cbpr2"][0]), xrel(xd, refs["cbpr2"][1])
    print(f"gmres cbpr2 central 4096^2 one-CTA defect: history {sh:.2e}, x {sx:.2e}: "
          f"{min(sh, sx) / BAR_GMRES:.1e} x the bar")
    assert not bad, bad
    assert min(sh, sx) > 100 * BAR_GMRES
    del b, refs, fd, xd
    _free(torch)


@gpu
def test_hh1024_vs_oracle(env, ko):
    """Householder GMRES(95), one cycle at 1024^2 on W, both HH_MODEs, against the oracle's gmres_hh run
    multi-threaded on the twin."""
    kl, h, torch = env
    ns, m = 1024, 95
    b = np.random.default_rng(1024 + 5).standard_normal(ns * ns)
    with oracle_threads(ko):
        o = ko.gmres_hh(tw.stencil_fn(ko, W), b, m, 0.0, None, max_stages=1, skip_verr=True)
    with opts(h, MAX_RESTARTS=1):
        for mode in (1, 0):
            with opts(h, HH_MODE=mode):
                g = h.gmres_hh_omp(kl.stencil5(*W), b, m, 0.0)
            d, dx = hist_rel(g.history, o.history), xrel(g.x, o.x)
            print(f"hh1024 W mode {mode}: history {d:.2e}, x {dx:.2e} (bar {BAR_HH:.0e})")
            assert (g.n_out, g.restart_out) == (m, 1) and d < BAR_HH and dx < BAR_HH
