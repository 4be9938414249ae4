"""GPU tests of plain CG in pairs of temporally blocked passes (ChCgPass<kCgPairA / kCgPairB>, kl_cg.cu;
KL_OPT_CG_ONEPASS = 2).

A pair stores p and x only in its second pass, which rebuilds p_{k+1} = r_{k+1} + beta_k p_k and forms x_{k+2} with
the same fmas the one-pass path (option 1) executes, on the same operands and in the same reduction order.  So every
result is compared with option 1 bit for bit, not within a tolerance.
"""
import numpy as np
import pytest

from parity import hist_bar, hist_norm

pytestmark = pytest.mark.gpu

KL_OPT_CHECK_EVERY = 4      # include/krylov_b200.h
KL_OPT_CG_ONEPASS = 22
PAIR_MIN = 1 << 24          # kCgPairMin (kl_cg.cu): auto picks pairs from this many unknowns on


@pytest.fixture(scope="module")
def kl():
    import gmres_b200 as m
    return m


@pytest.fixture(scope="module")
def h(kl):
    hd = kl.Handle(0)
    yield hd
    hd.close()


def _with(h, value, fn, check_every=None):
    h.set_option(KL_OPT_CG_ONEPASS, value)
    old = h.get_option(KL_OPT_CHECK_EVERY)
    if check_every is not None:
        h.set_option(KL_OPT_CHECK_EVERY, check_every)
    try:
        return fn()
    finally:
        h.set_option(KL_OPT_CG_ONEPASS, -1)
        h.set_option(KL_OPT_CHECK_EVERY, old)


def _bytes_per_point(r, nx, ny):
    return r.stats["algorithmic_bytes"] / r.stats["iterations"] / (nx * ny)


def _pair_bytes(its):
    """Bytes per point and iteration of `its` iterations in pairs: 24 per pass A, 48 per pass B, 24 for the flush
    of x after a final pass A."""
    return (24.0 * ((its + 1) // 2) + 48.0 * (its // 2) + 24.0 * (its % 2)) / its


def _np(v):
    return v.cpu().numpy() if hasattr(v, "cpu") else np.asarray(v)


def _same(a, b):
    return np.array_equal(_np(a.history), _np(b.history)) and np.array_equal(_np(a.x), _np(b.x))


@pytest.mark.parametrize("nx,ny", [(300, 300), (1000, 64), (128, 515), (1024, 1024), (301, 200)])
@pytest.mark.parametrize("aniso", [False, True])
def test_pair_bit_identical_to_onepass(kl, h, nx, ny, aniso):
    op = kl.aniso(1.0, 0.01) if aniso else kl.stvec
    b = h.apply(op, np.ones(nx * ny), nx, ny)
    for its in (1, 2, 3, 7, 8, 64):
        g = _with(h, 2, lambda: h.cg_omp(op, b, 0.0, its, nx=nx, ny=ny))
        s = _with(h, 1, lambda: h.cg_omp(op, b, 0.0, its, nx=nx, ny=ny))
        # odd nx: the chain kernels need column pairs, the two-kernel path runs in both settings
        assert _bytes_per_point(g, nx, ny) == pytest.approx(64.0 if nx % 2 else _pair_bytes(its)), its
        if its % 2 == 0 and nx % 2 == 0:
            assert _bytes_per_point(g, nx, ny) == pytest.approx(36.0)
        assert g.iter == s.iter == its and g.history.size == s.history.size == its
        assert _same(g, s), (its, np.abs(g.history / s.history - 1).max(), np.abs(g.x - s.x).max())


@pytest.mark.parametrize("check_every", [5, 3])
def test_pair_batches_starting_on_second_pass(kl, h, check_every):
    """An odd poll interval makes every second batch start on the second pass of a pair (run eagerly)."""
    ns = 300
    b = h.apply(kl.stvec, np.ones(ns * ns), ns, ns)
    for its in (16, 17):
        g = _with(h, 2, lambda: h.cg_omp(kl.stvec, b, 0.0, its), check_every)
        s = _with(h, 1, lambda: h.cg_omp(kl.stvec, b, 0.0, its), check_every)
        assert g.iter == its
        assert _same(g, s), its


def test_pair_graph_replay_bit_identical(kl, h):
    ns = 1000
    b = h.apply(kl.stvec, np.ones(ns * ns), ns, ns)
    run = lambda v: _with(h, v, lambda: h.cg_omp(kl.stvec, b, 1e-9, 200))
    g1, g2 = run(2), run(2)     # batches after the first are captured and replayed as CUDA graphs
    assert g1.iter == g2.iter == 200
    assert _same(g1, g2)
    assert _same(g1, run(1))


@pytest.mark.parametrize("device", [False, True])
def test_pair_early_convergence_both_parities(kl, h, device):
    """Convergence after an odd iteration (ends on a first pass: x is flushed) and after an even one, each with an
    odd and an even maxit: the passes after convergence are gated off and x must come back in the caller's buffer."""
    ns = 300
    b = h.apply(kl.stvec, np.ones(ns * ns), ns, ns)
    if device:
        import torch
        b = torch.from_numpy(b).cuda()
    run = lambda tol, its: _with(h, 2, lambda: h.cg_omp(kl.stvec, b, tol, its, nx=ns, ny=ns))
    hist = _np(run(0.0, 40).history)
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
            assert np.array_equal(_np(g.x), _np(ref.x)), (k, maxit)
    assert seen == {0, 1}


@pytest.mark.parametrize("maxit", [25, 26])
def test_pair_not_converged_leaves_iter(kl, h, maxit):
    ns = 300
    b = h.apply(kl.stvec, np.ones(ns * ns), ns, ns)
    g = _with(h, 2, lambda: h.cg_omp(kl.stvec, b, 1e-9, maxit))
    assert g.status == kl.api.KL_NOT_CONVERGED and g.iter == maxit and g.history.size == maxit
    assert g.stats["iterations"] == maxit
    assert _bytes_per_point(g, ns, ns) == pytest.approx(_pair_bytes(maxit))


@pytest.mark.parametrize("ns", [100, 300])
def test_pair_parity_with_oracle(kl, h, ko, ns):
    b = ko.manufactured_rhs(ko.stvec_fn(), ns)
    o = ko.cg_omp(ko.stvec_fn(), b, 1e-9, 10000)
    g = _with(h, 2, lambda: h.cg_omp(kl.stvec, b, 1e-9, 10000))
    assert _bytes_per_point(g, ns, ns) == pytest.approx(_pair_bytes(g.iter))
    assert g.status == 0 and abs(g.iter - o.iter) <= 1
    k = min(g.history.size, o.history.size)
    rel = np.abs(g.history[:k] / o.history[:k] - 1)
    assert rel[:50].max() < 1e-10
    assert rel.max() < hist_bar(f"cg_omp_{ns}"), (rel.max(), hist_bar(f"cg_omp_{ns}"))
    assert hist_norm(g.history, o.history, float(np.linalg.norm(b))) < 1e-10
    assert np.abs(g.x - o.x).max() / np.abs(o.x).max() < 1e-9
    assert np.abs(g.x - 1).max() < 1e-9


def test_pair_auto_threshold(kl, h):
    import torch
    # two kernels below 2^20 unknowns, one pass per iteration from 2^20, pairs from PAIR_MIN on
    for ns in (1000, 1024, 2048, 4096, 8192):
        want = 64.0 if ns * ns < (1 << 20) else (36.0 if ns * ns >= PAIR_MIN else 48.0)
        b = h.apply(kl.stvec, torch.ones(ns * ns, dtype=torch.float64, device="cuda"), ns, ns)
        g = h.cg_omp(kl.stvec, b, 0.0, 4, nx=ns, ny=ns)
        assert _bytes_per_point(g, ns, ns) == pytest.approx(want), ns
        del b, g
        torch.cuda.empty_cache()


@pytest.mark.parametrize("nx,ny", [(1024, 1024), (1000, 64), (128, 515), (300, 300)])
@pytest.mark.parametrize("aniso", [False, True])
def test_pair_bit_identical_to_onepass_random_rhs(kl, h, nx, ny, aniso):
    """As above with a random b: b = A*1 leaves the grid's interior zero for many iterations, so there agreement
    says nothing about the CTAs away from the boundary."""
    op = kl.aniso(1.0, 0.01) if aniso else kl.stvec
    b = np.random.default_rng(nx + ny).standard_normal(nx * ny)
    for its in (1, 2, 7, 8, 64):
        g = _with(h, 2, lambda: h.cg_omp(op, b, 0.0, its, nx=nx, ny=ny))
        s = _with(h, 1, lambda: h.cg_omp(op, b, 0.0, its, nx=nx, ny=ny))
        assert g.iter == s.iter == its
        assert _same(g, s), (its, np.abs(g.history / s.history - 1).max(), np.abs(g.x - s.x).max())
