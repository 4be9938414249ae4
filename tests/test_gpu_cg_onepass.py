"""GPU tests of plain CG in one temporally blocked pass per iteration (ChCg, kl_cg.cu; KL_OPT_CG_ONEPASS).

The pass does the two-kernel path's point-wise fmas on the same operands; only beta is formed differently (predicted
from three dot products of the same pass, tests/test_cg_onepass_numerics.py).  Bars: against the oracle the ones
test_cg_parity uses; against the two-kernel path (option 0) 1e-12 over a few iterations.
"""
import numpy as np
import pytest

from parity import hist_bar, hist_norm

pytestmark = pytest.mark.gpu

KL_OPT_CG_ONEPASS = 22      # include/krylov_b200.h


@pytest.fixture(scope="module")
def kl():
    import gmres_b200 as m
    return m


@pytest.fixture(scope="module")
def h(kl):
    hd = kl.Handle(0)
    yield hd
    hd.close()


def _with(h, value, fn):
    h.set_option(KL_OPT_CG_ONEPASS, value)
    try:
        return fn()
    finally:
        h.set_option(KL_OPT_CG_ONEPASS, -1)


def _bytes_per_point(r, nx, ny):
    return r.stats["algorithmic_bytes"] / r.stats["iterations"] / (nx * ny)


@pytest.mark.parametrize("ns", [100, 300])
def test_onepass_parity_with_oracle(kl, h, ko, ns):
    b = ko.manufactured_rhs(ko.stvec_fn(), ns)
    o = ko.cg_omp(ko.stvec_fn(), b, 1e-9, 10000)
    g = _with(h, 1, lambda: h.cg_omp(kl.stvec, b, 1e-9, 10000))
    assert _bytes_per_point(g, ns, ns) == pytest.approx(48.0)
    assert g.status == 0 and abs(g.iter - o.iter) <= 1
    k = min(g.history.size, o.history.size)
    rel = np.abs(g.history[:k] / o.history[:k] - 1)
    print(f"cg one-pass {ns}: iters gpu {g.iter} oracle {o.iter}; history rel diff head {rel[:50].max():.2e} all {rel.max():.2e}")
    assert rel[:50].max() < 1e-10
    assert rel.max() < hist_bar(f"cg_omp_{ns}"), (rel.max(), hist_bar(f"cg_omp_{ns}"))
    assert hist_norm(g.history, o.history, float(np.linalg.norm(b))) < 1e-10
    assert np.abs(g.x - o.x).max() / np.abs(o.x).max() < 1e-9
    assert np.abs(g.x - 1).max() < 1e-9


@pytest.mark.parametrize("nx,ny", [(300, 300), (1000, 64), (128, 515), (301, 200)])
@pytest.mark.parametrize("aniso", [False, True])
def test_onepass_matches_two_kernel_path(kl, h, nx, ny, aniso):
    op = kl.aniso(1.0, 0.01) if aniso else kl.stvec
    b = h.apply(op, np.ones(nx * ny), nx, ny)
    for its in (1, 2, 7):
        g = _with(h, 1, lambda: h.cg_omp(op, b, 0.0, its, nx=nx, ny=ny))
        s = _with(h, 0, lambda: h.cg_omp(op, b, 0.0, its, nx=nx, ny=ny))
        # odd nx: the chain kernel needs column pairs, the two-kernel path runs
        assert _bytes_per_point(g, nx, ny) == pytest.approx(64.0 if nx % 2 else 48.0)
        assert _bytes_per_point(s, nx, ny) == pytest.approx(64.0)
        assert g.history.size == s.history.size == its
        assert np.allclose(g.history, s.history, rtol=1e-12, atol=0), (its, np.abs(g.history / s.history - 1).max())
        assert np.allclose(g.x, s.x, rtol=1e-12, atol=1e-14), (its, np.abs(g.x - s.x).max())


def test_onepass_not_converged_leaves_iter(kl, h):
    ns = 300
    b = h.apply(kl.stvec, np.ones(ns * ns), ns, ns)
    g = _with(h, 1, lambda: h.cg_omp(kl.stvec, b, 1e-9, 25))
    assert g.status == kl.api.KL_NOT_CONVERGED and g.iter == 25 and g.history.size == 25
    assert g.stats["iterations"] == 25


@pytest.mark.parametrize("device", [False, True])
def test_onepass_early_convergence_both_parities(kl, h, device):
    """Convergence after an odd and after an even number of iterations, with odd and even maxit: x is ping-ponged
    from the first iteration on, and the result must come back in the caller's buffer either way."""
    ns = 300
    b = h.apply(kl.stvec, np.ones(ns * ns), ns, ns)
    if device:
        import torch
        b = torch.from_numpy(b).cuda()
    run = lambda tol, its: _with(h, 1, lambda: h.cg_omp(kl.stvec, b, tol, its, nx=ns, ny=ns))
    hist = run(0.0, 40).history
    hist = hist.cpu().numpy() if hasattr(hist, "cpu") else np.asarray(hist)
    seen = set()
    for k in range(2, 40):
        if k % 2 in seen or not hist[k - 1] < hist[: k - 1].min():
            continue
        seen.add(k % 2)
        tol = 0.5 * (hist[k - 1] + hist[: k - 1].min())        # first met at iteration k
        ref = run(0.0, k)
        for maxit in (k + 6, k + 7):
            g = run(tol, maxit)
            assert g.status == 0 and g.iter == k and g.history.size == k
            gx, rx = (g.x.cpu().numpy(), ref.x.cpu().numpy()) if device else (g.x, ref.x)
            assert np.array_equal(gx, rx), (k, maxit)
    assert seen == {0, 1}


def test_onepass_bit_identical_reruns(kl, h):
    ns = 1000
    b = h.apply(kl.stvec, np.ones(ns * ns), ns, ns)
    run = lambda: _with(h, 1, lambda: h.cg_omp(kl.stvec, b, 1e-9, 200))
    g1, g2 = run(), run()       # batches after the first are captured and replayed as CUDA graphs
    assert g1.iter == g2.iter == 200
    assert np.array_equal(g1.history, g2.history) and np.array_equal(g1.x, g2.x)


def test_onepass_auto_threshold(kl, h):
    import torch
    for ns, want in ((300, 64.0), (1000, 64.0), (1024, 48.0), (2048, 48.0)):   # from 2^20 unknowns on
        b = h.apply(kl.stvec, torch.ones(ns * ns, dtype=torch.float64, device="cuda"), ns, ns)
        g = h.cg_omp(kl.stvec, b, 0.0, 4, nx=ns, ny=ns)
        assert _bytes_per_point(g, ns, ns) == pytest.approx(want), ns


@pytest.mark.parametrize("nx,ny", [(1024, 1024), (1000, 64), (128, 515)])
@pytest.mark.parametrize("aniso", [False, True])
def test_onepass_matches_two_kernel_path_random_rhs(kl, h, nx, ny, aniso):
    """As above with a random b, which has support on the whole grid from the first iteration on."""
    op = kl.aniso(1.0, 0.01) if aniso else kl.stvec
    b = np.random.default_rng(nx * 3 + ny).standard_normal(nx * ny)
    for its in (1, 2, 7, 40):
        g = _with(h, 1, lambda: h.cg_omp(op, b, 0.0, its, nx=nx, ny=ny))
        s = _with(h, 0, lambda: h.cg_omp(op, b, 0.0, its, nx=nx, ny=ny))
        assert g.history.size == s.history.size == its
        assert np.allclose(g.history, s.history, rtol=1e-12, atol=0), (its, np.abs(g.history / s.history - 1).max())
        assert np.abs(g.x - s.x).max() < 1e-12 * np.abs(s.x).max(), (its, np.abs(g.x - s.x).max())
