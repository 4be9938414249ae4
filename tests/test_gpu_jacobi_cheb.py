"""GPU tests of the Jacobi-scaled Chebyshev preconditioner on the variable-coefficient operator (KL_PC_JACOBI_CHEB:
ChJacCheb in kl_chain_tma.cuh, k_jacobi_cheb_step in kl_ops.cu).

Bar: every application is BIT-IDENTICAL to the CPU twin (tests/jacobi_cheb_twin.c), on the chained
path and on the one-pass-per-step path alike; the solvers agree with the oracle solvers run with the twin.  Inputs
are full-support random vectors and log-uniform coefficient fields (contrast up to 1e4, anisotropy up to 100).
"""
import ctypes as C

import numpy as np
import pytest

import jacobi_cheb_twin as twin
from parity import hist_rel

pytestmark = pytest.mark.gpu

PRM = (0.01, 2.0)                       # an interval inside (0, 2]
SHAPES = [(64, 64), (300, 300), (130, 77), (1000, 70), (66, 1000), (240, 24), (482, 150),   # the chain tests' shapes
          (301, 97), (129, 64), (40, 33), (62, 200)]                                         # odd nx, nx < 64
DEGREES = (0, 1, 2, 3, 4, 5, 6, 7, 8, 9, 13)


@pytest.fixture(scope="module")
def kl():
    import gmres_b200 as m
    return m


@pytest.fixture(scope="module")
def h(kl):
    hd = kl.Handle(0)
    yield hd
    hd.close()


def fields(nx, ny, seed, contrast=1e4, aniso=100.0):
    rng = np.random.default_rng(seed)
    lc = np.log(contrast) / 2
    kx = np.exp(rng.uniform(-lc, lc, nx * ny))
    ky = np.exp(rng.uniform(-lc, lc, nx * ny)) / aniso
    return kx, ky


def _with(h, opts, fn):
    old = {k: h.get_option(k) for k in opts}
    for k, v in opts.items():
        h.set_option(k, v)
    try:
        return fn()
    finally:
        for k, v in old.items():
            h.set_option(k, v)


@pytest.mark.parametrize("nx,ny", SHAPES)
def test_bit_identical_to_oracle_twin_chained_and_stepwise(kl, h, ko, nx, ny):
    kx, ky = fields(nx, ny, nx * 3 + ny)
    A = kl.aniso_var(kx, ky)
    r = np.random.default_rng(nx + 7 * ny).standard_normal(nx * ny)
    for k in DEGREES:
        prm = () if k == 0 else PRM
        ref = twin.jacobi_cheb(kx, ky, r, k, prm, nx, ny)
        z = h.apply_precond(kl.jacobi_cheb(k), A, r, prm, nx, ny)
        assert np.array_equal(z, ref), (nx, ny, k, np.abs(z - ref).max())
        zs = _with(h, {kl.KL_OPT_CHAIN: 0}, lambda: h.apply_precond(kl.jacobi_cheb(k), A, r, prm, nx, ny))
        assert np.array_equal(zs, ref), (nx, ny, k, "stepwise")
    # the other switches that turn the chain off, and the reversed interval
    for opt in (kl.KL_OPT_TMA, kl.KL_OPT_FUSE):
        z = _with(h, {opt: 0}, lambda: h.apply_precond(kl.jacobi_cheb(4), A, r, PRM, nx, ny))
        assert np.array_equal(z, twin.jacobi_cheb(kx, ky, r, 4, PRM, nx, ny)), opt
    z = h.apply_precond(kl.jacobi_cheb(5), A, r, PRM[::-1], nx, ny)
    assert np.array_equal(z, twin.jacobi_cheb(kx, ky, r, 5, PRM[::-1], nx, ny))


def test_bit_identical_to_oracle_twin_8192(kl, h, ko):
    n = 8192
    kx, ky = fields(n, n, 81)
    A = kl.aniso_var(kx, ky)
    r = np.random.default_rng(82).standard_normal(n * n)
    Ao = ko.aniso_var_fn(kx, ky)
    ko.set_threads(ko.max_threads())      # the twin is point-wise: the thread count does not change its bits
    try:
        for k in (0, 4, 6, 9):
            prm = (0.0, 0.0) if k == 0 else PRM
            ref = ko.apply_precond(twin.precond_fn(ko, kx, ky, k), Ao, r, prm, n, parallel=True)
            z = h.apply_precond(kl.jacobi_cheb(k), A, r, prm, n, n)
            assert np.array_equal(z, ref), (k, np.abs(z - ref).max())
    finally:
        ko.set_threads(1)


def test_rows_option_and_pointer_modes(kl, h):
    import torch
    nx, ny = 1024, 1030
    kx, ky = fields(nx, ny, 5)
    A = kl.aniso_var(kx, ky)
    r = np.random.default_rng(6).standard_normal(nx * ny)
    for k in (3, 6, 8):
        ref = h.apply_precond(kl.jacobi_cheb(k), A, r, PRM, nx, ny)
        for rows in (7, 16, 33, 200):
            z = _with(h, {kl.KL_OPT_STENCIL_ROWS: rows}, lambda: h.apply_precond(kl.jacobi_cheb(k), A, r, PRM, nx, ny))
            assert np.array_equal(z, ref), (k, rows)
        zd = h.apply_precond(kl.jacobi_cheb(k), A, torch.from_numpy(r).cuda(), PRM, nx, ny)
        torch.cuda.synchronize()
        assert np.array_equal(zd.cpu().numpy(), ref), k
    zd = h.apply_precond(kl.jacobi_cheb(0), A, torch.from_numpy(r).cuda(), (), nx, ny)
    torch.cuda.synchronize()
    assert np.array_equal(zd.cpu().numpy(), h.apply_precond(kl.jacobi_cheb(0), A, r, (), nx, ny))


@pytest.mark.parametrize("c", [1.0, 0.37])
def test_constant_fields_are_scaled_cheb(kl, h, c):
    """kx = ky = c: D = 4c, so the polynomial on D^-1 A over (a, b) is 1/c times KL_PC_CHEB on stvec over (4a, 4b)"""
    nx, ny = 200, 130
    A = kl.aniso_var(np.full(nx * ny, c), np.full(nx * ny, c))
    r = np.random.default_rng(3).standard_normal(nx * ny)
    a, b = 0.05, 1.9
    for k in (1, 2, 4, 6, 9):
        z = h.apply_precond(kl.jacobi_cheb(k), A, r, (a, b), nx, ny)
        ref = h.apply_precond(kl.cheb(k), kl.stvec, r, (4 * a, 4 * b), nx, ny) / c
        assert np.linalg.norm(z - ref) / np.linalg.norm(ref) < 1e-13, k


def test_one_launch_per_application(kl, h):
    nx, ny = 256, 256
    A = kl.aniso_var(*fields(nx, ny, 9))
    r = np.random.default_rng(10).standard_normal(nx * ny)
    for k in range(0, 7):
        before = h.stats()["kernel_launches"]
        h.apply_precond(kl.jacobi_cheb(k), A, r, PRM, nx, ny)
        assert h.stats()["kernel_launches"] - before == 1, k


def _solver_case(kl, ko, ns, seed, contrast):
    kx, ky = fields(ns, ns, seed, contrast)
    A, Ao = kl.aniso_var(kx, ky), ko.aniso_var_fn(kx, ky)
    b = ko.manufactured_rhs(Ao, ns)
    return A, Ao, b, (kx, ky)


def _its(g, m):
    return (g.restart_out - 1) * m + g.n_out


@pytest.mark.parametrize("ns,k", [(96, 4), (127, 3), (128, 8)])
def test_solvers_against_oracle_with_twin(kl, h, ko, ns, k):
    A, Ao, b, (kx, ky) = _solver_case(kl, ko, ns, ns + k, 1e2)
    M, prm = kl.jacobi_cheb(k), PRM

    def Mo():
        return twin.precond_fn(ko, kx, ky, k)

    for run, orun in ((lambda: h.pcg_omp(A, b, 1e-9, 20000, M, prm), lambda: ko.pcg_omp(Ao, b, 1e-9, 20000, Mo(), prm)),
                      (lambda: h.pcg(A, b, 1e-9, 20000, M, prm), lambda: ko.pcg(Ao, b, 1e-9, 20000, Mo(), prm))):
        g, o = run(), orun()
        assert g.status == 0 and abs(g.iter - o.iter) <= max(1, o.iter // 100), (g.iter, o.iter)
        assert hist_rel(g.history[:50], o.history[:50]) < 1e-10
        assert np.linalg.norm(b - h.apply(A, g.x, ns, ns)) < 1e-8
    m = 40
    for gfn, ofn in ((h.gmres_mgsr_omp, ko.gmres_mgsr_omp), (h.gmres_mgsr_mf, ko.gmres_mgsr_mf)):
        g = gfn(A, b, m, 1e-8, M, prm)
        o = ofn(Ao, b, m, 1e-8, Mo(), prm, max_restarts=1000)
        assert g.status == 0 and abs(_its(g, m) - o.iterations) <= max(1, o.iterations // 100), (_its(g, m), o.iterations)
        assert hist_rel(g.history[:m], o.history[:m]) < 1e-10
    g = h.gmres_hh_prec_omp(A, b, m, 1e-8, M, prm)
    o = ko.gmres_hh(Ao, b, m, 1e-8, Mo(), prm)
    assert g.status == 0 and abs(_its(g, m) - o.iterations) <= max(1, o.iterations // 100), (_its(g, m), o.iterations)
    assert hist_rel(g.history[:m], o.history[:m]) < 1e-10
    for run, orun in ((lambda: h.pbicgstab(A, b, 1e-9, 20000, M, prm), lambda: ko.pbicgstab(Ao, b, 1e-9, 20000, Mo(), prm)),
                      (lambda: h.pbicgstab_omp(A, b, 1e-9, 20000, M, prm),
                       lambda: ko.pbicgstab_omp(Ao, b, 1e-9, 20000, Mo(), prm))):
        g, o = run(), orun()
        assert g.status == 0 and abs(g.iter - o.iter) <= max(2, o.iter * 5 // 100), (g.iter, o.iter)
        assert np.abs(g.x - o.x).max() < 1e-6


def test_pcg_jacobi_cheb_halves_cg_iterations(kl, h, ko):
    ns = 512
    A, Ao, b, _ = _solver_case(kl, ko, ns, 512, 1e4)
    prm = h.cheb_interval_from_ritz(2.0 / 1.025, 4)
    plain = h.cg_omp(A, b, 1e-9, 400000)
    pre = h.pcg_omp(A, b, 1e-9, 400000, kl.jacobi_cheb(4), prm)
    jac = h.pcg_omp(A, b, 1e-9, 400000, kl.jacobi_cheb(0), ())
    print(f"512^2 contrast 1e4: cg {plain.iter}, pcg+jacobi {jac.iter}, pcg+jacobi_cheb(4) {pre.iter}")
    assert plain.status == 0 and pre.status == 0 and jac.status == 0
    assert 2 * pre.iter < plain.iter


def _status(kl, h, M, op, params, nx=64, ny=64):
    L = kl.load_library()
    r = np.ones(nx * ny)
    z = np.zeros(nx * ny)
    L.kl_set_pointer_mode(h._h, kl.api.KL_POINTER_HOST)
    o, keep = op._c()
    p, keep_p = M._c()
    pr = np.ascontiguousarray(params if len(params) else (0.0,), dtype=np.float64)
    return L.kl_apply_precond(h._h, C.byref(p), C.byref(o), C.c_void_p(r.ctypes.data), C.c_void_p(z.ctypes.data),
                              pr.ctypes.data_as(C.POINTER(C.c_double)), len(params), nx, ny)


def test_error_paths(kl, h, ko):
    A = kl.aniso_var(*fields(64, 64, 1))
    assert _status(kl, h, kl.jacobi_cheb(0), A, ()) == 0
    assert _status(kl, h, kl.jacobi_cheb(3), A, PRM) == 0
    for op in (kl.stvec, kl.aniso(1.0, 0.01), kl.stv_poisson):
        assert _status(kl, h, kl.jacobi_cheb(3), op, PRM) == -5          # KL_ERR_UNSUPPORTED
        assert _status(kl, h, kl.jacobi_cheb(0), op, ()) == -5
    assert "KL_PC_CHEB" in kl.load_library().kl_last_error(h._h).decode()
    assert _status(kl, h, kl.jacobi_cheb(-1), A, PRM) == -1                 # KL_ERR_INVALID
    assert _status(kl, h, kl.jacobi_cheb(2), A, (2.0,)) == -1
    assert _status(kl, h, kl.jacobi_cheb(2), A, ()) == -1
    for bad in ((0.0, 2.0), (-0.1, 2.0), (1.0, 1.0), (np.inf, 2.0), (0.1, np.nan), (0.1, -2.0)):
        assert _status(kl, h, kl.jacobi_cheb(2), A, bad) == -1, bad
    # the solvers return the same statuses
    b = np.ones(64 * 64)
    with pytest.raises(kl.KrylovError, match="error -5"):
        h.pcg_omp(kl.stvec, b, 1e-9, 100, kl.jacobi_cheb(2), PRM)
    with pytest.raises(kl.KrylovError, match="error -1"):
        h.gmres_mgsr_omp(A, b, 10, 1e-8, kl.jacobi_cheb(2), (1.0, 1.0))
