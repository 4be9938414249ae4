"""GPU tests of the temporally blocked ("chained") stencil kernels (kl_chain_tma.cuh):
several dependent operator applications in one pass over HBM.

Bar: every point-wise result is BIT-IDENTICAL to the one-pass-per-application kernels
(KL_OPT_CHAIN = 0) and to the CPU oracle (oracle/krylov_extras.c ko_cheb); solver-level
differences come only from the summation order of the fused dot products.
"""
import numpy as np
import pytest

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def kl():
    import gmres_b200 as m
    return m


@pytest.fixture(scope="module")
def h(kl):
    hd = kl.Handle(0)
    yield hd
    hd.close()


def _no_chain(kl, h, fn):
    h.set_option(kl.KL_OPT_CHAIN, 0)
    try:
        return fn()
    finally:
        h.set_option(kl.KL_OPT_CHAIN, 1)


@pytest.mark.parametrize("nx,ny", [(64, 64), (300, 300), (130, 77), (1000, 70), (66, 1000), (240, 24), (482, 150)])
def test_cheb_chain_bit_identical_to_stepwise(kl, h, nx, ny):
    rng = np.random.default_rng(nx * 7 + ny)
    r = rng.standard_normal(nx * ny)
    for op in (kl.stvec, kl.stv_poisson, kl.aniso(1.0, 0.01)):
        for k in (1, 2, 3, 4, 5, 6, 7, 8, 9, 12, 13):   # <= 6 one chain, 7..12 two chains, 13 = chain of 6 + 7 passes
            zc = h.apply_precond(kl.cheb(k), op, r, (0.2, 8.2), nx, ny)
            zs = _no_chain(kl, h, lambda: h.apply_precond(kl.cheb(k), op, r, (0.2, 8.2), nx, ny))
            assert np.array_equal(zc, zs), (nx, ny, k, op.kind, np.abs(zc - zs).max())


@pytest.mark.parametrize("ns", [64, 300, 512])
def test_cheb_chain_bit_identical_to_oracle(kl, h, ko, ns):
    rng = np.random.default_rng(ns + 5)
    r = rng.standard_normal(ns * ns)
    for k in (2, 4, 6, 8):
        zc = h.apply_precond(kl.cheb(k), kl.stvec, r, (0.2, 8.2), ns, ns)
        assert np.array_equal(zc, ko.apply_precond(ko.cheb_fn(k), ko.stvec_fn(), r, (0.2, 8.2), ns))


def test_cheb_chain_rows_option_and_large_grid(kl, h):
    # CTA height must not change the bits; 4096 x 1030 exercises many CTAs in both directions
    nx, ny = 4096, 1030
    rng = np.random.default_rng(11)
    r = rng.standard_normal(nx * ny)
    ref = _no_chain(kl, h, lambda: h.apply_precond(kl.cheb(4), kl.stvec, r, (0.2, 8.2), nx, ny))
    for rows in (0, 7, 16, 33, 200):
        h.set_option(kl.KL_OPT_STENCIL_ROWS, rows)
        try:
            z = h.apply_precond(kl.cheb(4), kl.stvec, r, (0.2, 8.2), nx, ny)
        finally:
            h.set_option(kl.KL_OPT_STENCIL_ROWS, 0)
        assert np.array_equal(z, ref), rows


def test_pcg_with_chained_chebyshev(kl, h, ko):
    ns = 300
    b = ko.manufactured_rhs(ko.stvec_fn(), ns)
    lo, hi = h.lanczos(kl.stvec, ns, ns, 30)
    prm = h.cheb_params_from_ritz(lo, hi)
    g = h.pcg_omp(kl.stvec, b, 1e-9, 10000, kl.cheb(4), (prm[1], prm[0]))
    s = _no_chain(kl, h, lambda: h.pcg_omp(kl.stvec, b, 1e-9, 10000, kl.cheb(4), (prm[1], prm[0])))
    o = ko.pcg_omp(ko.stvec_fn(), b, 1e-9, 10000, ko.cheb_fn(4), (prm[1], prm[0]))
    print(f"pcg+cheb(4) {ns}: chain {g.iter} stepwise {s.iter} oracle {o.iter}")
    assert g.status == 0 and abs(g.iter - o.iter) <= 1 and abs(g.iter - s.iter) <= 1
    k = min(g.history.size, s.history.size, 40)
    assert np.allclose(g.history[:k], s.history[:k], rtol=1e-10)
    assert np.abs(g.x - 1).max() < 1e-7


@pytest.mark.parametrize("ns", [100, 300, 1024])
def test_pbicgstab_chain_matches_two_pass(kl, h, ko, ns):
    b = h.apply(kl.stvec, np.ones(ns * ns), ns, ns)
    P = (8.2, 0.2)
    # a few iterations: x agrees to rounding (alpha, omega come from differently ordered sums)
    for its in (1, 2, 5):
        g = h.pbicgstab_omp(kl.stvec, b, 0.0, its, kl.cbpr2, P)
        s = _no_chain(kl, h, lambda: h.pbicgstab_omp(kl.stvec, b, 0.0, its, kl.cbpr2, P))
        assert np.allclose(g.x, s.x, rtol=1e-11, atol=1e-13), (its, np.abs(g.x - s.x).max())
        assert np.allclose(g.history, s.history, rtol=1e-11)
    g = h.pbicgstab_omp(kl.stvec, b, 1e-9, 10000, kl.cbpr2, P)
    s = _no_chain(kl, h, lambda: h.pbicgstab_omp(kl.stvec, b, 1e-9, 10000, kl.cbpr2, P))
    print(f"pbicgstab {ns}: chain {g.iter} two-pass {s.iter}; bytes/it {g.stats['algorithmic_bytes'] / max(g.iter, 1) / (ns * ns):.0f}n")
    # BiCGSTAB amplifies rounding differences ~x2.5 per iteration (DESIGN.md "Parity"): the two variants
    # differ only in the summation order of the dot products, yet their counts drift apart on larger
    # grids (795 vs 914 at 1024^2) exactly as two CPU restatements do; both reach the tolerance.
    assert g.status == 0 and s.status == 0 and abs(g.iter - s.iter) <= max(3, 0.2 * s.iter)
    assert g.res < 1e-9 and np.abs(g.x - 1).max() < 1e-6
    assert np.allclose(g.history[:10], s.history[:10], rtol=1e-9)


def test_pbicgstab_chain_anisotropic_rectangular(kl, h):
    nx, ny = 512, 200
    A = kl.aniso(1.0, 0.01)
    b = h.apply(A, np.ones(nx * ny), nx, ny)
    prm = (2.0 * (1.0 + 0.01) * 2.0, 0.05)
    g = h.pbicgstab_omp(A, b, 0.0, 4, kl.cbpr2, prm, nx, ny)
    s = _no_chain(kl, h, lambda: h.pbicgstab_omp(A, b, 0.0, 4, kl.cbpr2, prm, nx, ny))
    assert np.allclose(g.history[:4], s.history[:4], rtol=1e-9)
    assert np.allclose(g.x, s.x, rtol=1e-8, atol=1e-10)


@pytest.mark.parametrize("nx,ny", [(300, 300), (1000, 64), (128, 515)])
def test_cg_operator_twice_matches_stored_ap(kl, h, nx, ny):
    # default plain CG never stores A p (64n B/iteration: K2 recomputes p = r + beta*p_old and A p);
    # KL_OPT_CHAIN = 0 keeps the variant that stores it (72n B).  Same arithmetic per point.
    b = h.apply(kl.stvec, np.ones(nx * ny), nx, ny)
    for its in (1, 2, 7):
        g = h.cg_omp(kl.stvec, b, 0.0, its, nx=nx, ny=ny)
        s = _no_chain(kl, h, lambda: h.cg_omp(kl.stvec, b, 0.0, its, nx=nx, ny=ny))
        assert np.allclose(g.x, s.x, rtol=1e-12, atol=1e-14), (its, np.abs(g.x - s.x).max())
        assert np.allclose(g.history, s.history, rtol=1e-12)
    g = h.cg_omp(kl.stvec, b, 1e-9, 20000, nx=nx, ny=ny)
    s = _no_chain(kl, h, lambda: h.cg_omp(kl.stvec, b, 1e-9, 20000, nx=nx, ny=ny))
    assert g.status == 0 and abs(g.iter - s.iter) <= 1
    assert g.stats["algorithmic_bytes"] / g.iter / (nx * ny) == pytest.approx(64.0)
    assert np.abs(g.x - 1).max() < 1e-7 and np.abs(g.x - s.x).max() < 1e-9


@pytest.mark.parametrize("nx,ny,m", [(1024, 1024, 30), (2048, 640, 20), (1200, 1000, 24), (300, 300, 50), (130, 76, 12), (512, 500, 24)])
def test_gmres_one_pass_step_bit_identical_to_two_kernels(kl, h, nx, ny, m):
    """GMRES-MGSR + cbpr2: V_j = w/h, z = A V_j and w = cbpr2(z) as ONE temporally blocked pass (ChGmresStep,
    kl_gmres.cu) against the two separate kernels (KL_OPT_CHAIN = 0).  Every point sees the same divisions and the
    same fma, the orthogonalisation kernels are the same ones: the residual history, H and x are bit-identical.
    Both with and without CUDA-graph replay of the restart cycle."""
    P = (8.2, 0.2)
    h.set_option(2, 6)              # six restart cycles are enough to compare (the thin grids need hundreds to converge)
    try:
        for op in (kl.stvec, kl.aniso(1.0, 0.05)):
            b = h.apply(op, np.ones(nx * ny), nx, ny)
            run = lambda: h.gmres_mgsr_omp(op, b, m, 1e-9, kl.cbpr2, P, nx=nx, ny=ny)
            g = run()
            u = _no_chain(kl, h, run)
            assert g.status in (0, 1) and (g.status, g.n_out, g.restart_out) == (u.status, u.n_out, u.restart_out)
            assert g.history.size >= min(m, 20) and np.array_equal(g.history, u.history) and np.array_equal(g.x, u.x)
            assert np.array_equal(g.final_err, u.final_err)
            h.set_option(5, 0)          # KL_OPT_USE_GRAPH off: eager launches
            try:
                e = run()
            finally:
                h.set_option(5, 1)
            assert np.array_equal(e.history, g.history) and np.array_equal(e.x, g.x)
    finally:
        h.set_option(2, 1000)


@pytest.mark.parametrize("ns,m", [(100, 95), (300, 50), (512, 30)])
def test_cooperative_cgs2_step_bit_identical_to_three_kernels(kl, h, ns, m):
    """KL_OPT_COOP: the three tall-skinny passes of a CGS2 step as ONE cooperative kernel with two grid barriers
    (k_cgs2_coop) against three separate launches.  Same device code; the grids differ (the cooperative kernel is
    limited to co-resident CTAs), hence the partition of the partial sums: agreement to rounding, same counts."""
    P = (8.2, 0.2)
    b = h.apply(kl.stvec, np.ones(ns * ns), ns, ns)
    h.set_option(2, 8)           # eight restart cycles
    try:
        u = h.gmres_mgsr_omp(kl.stvec, b, m, 1e-9, kl.cbpr2, P)
        h.set_option(20, 1)          # KL_OPT_COOP on (off by default: measured slower than graph-replayed launches)
        try:
            g = h.gmres_mgsr_omp(kl.stvec, b, m, 1e-9, kl.cbpr2, P)
        finally:
            h.set_option(20, 0)
    finally:
        h.set_option(2, 1000)
    assert g.status in (0, 1) and (g.status, g.n_out, g.restart_out) == (u.status, u.n_out, u.restart_out)
    assert np.abs(g.history / u.history - 1).max() < 1e-11 and np.abs(g.x - u.x).max() < 1e-12
    assert g.stats["kernel_launches"] < u.stats["kernel_launches"]


@pytest.mark.parametrize("nx,ny", [(1024, 1024), (1000, 64), (128, 515)])
def test_cg_operator_twice_matches_stored_ap_random_rhs(kl, h, nx, ny):
    """As test_cg_operator_twice_matches_stored_ap with a random b (support on the whole grid)."""
    b = np.random.default_rng(nx + 2 * ny).standard_normal(nx * ny)
    h.set_option(22, 0)          # KL_OPT_CG_ONEPASS off: the two-kernel iteration at every size
    try:
        for its in (1, 2, 7, 40):
            g = h.cg_omp(kl.stvec, b, 0.0, its, nx=nx, ny=ny)
            s = _no_chain(kl, h, lambda: h.cg_omp(kl.stvec, b, 0.0, its, nx=nx, ny=ny))
            assert np.abs(g.x - s.x).max() < 1e-12 * np.abs(s.x).max(), (its, np.abs(g.x - s.x).max())
            assert np.allclose(g.history, s.history, rtol=1e-12, atol=0)
    finally:
        h.set_option(22, -1)


@pytest.mark.parametrize("nx,ny,m", [(1024, 1024, 30), (2048, 640, 20), (130, 76, 12)])
def test_gmres_one_pass_step_bit_identical_to_two_kernels_random_rhs(kl, h, nx, ny, m):
    """As test_gmres_one_pass_step_bit_identical_to_two_kernels with a random b (support on the whole grid)."""
    P = (8.2, 0.2)
    b = np.random.default_rng(nx + ny + m).standard_normal(nx * ny)
    h.set_option(2, 3)
    try:
        for op in (kl.stvec, kl.aniso(1.0, 0.05)):
            run = lambda: h.gmres_mgsr_omp(op, b, m, 0.0, kl.cbpr2, P, nx=nx, ny=ny)
            g = run()
            u = _no_chain(kl, h, run)
            assert (g.n_out, g.restart_out) == (u.n_out, u.restart_out) and g.history.size == 3 * m
            assert np.array_equal(g.history, u.history) and np.array_equal(g.x, u.x)
    finally:
        h.set_option(2, 1000)
