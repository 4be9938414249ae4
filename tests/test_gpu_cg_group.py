"""GPU tests of plain CG in groups of passes (ChCgLook<J, STORE>, kl_cg.cu; KL_OPT_CG_ONEPASS = 3).

A group starts from the stored r_k, p_k, x_k; its pass j replays j iterations from them and only its last pass stores
r, p and x.  Every point-wise value is the one-pass path's fma on the same operands, but a pass of J + 1 levels has a
CTA grid of its own, so its block-partial sums (alpha, beta) differ from the one-pass path's at rounding level.  So
against option 1 the results agree within a tolerance; within option 3 (graph replay against eager batches, early
convergence against tol = 0 runs, repeats) they agree bit for bit.
"""
import numpy as np
import pytest

from parity import hist_bar, hist_norm

pytestmark = pytest.mark.gpu

KL_OPT_CHECK_EVERY = 4      # include/krylov_b200.h
KL_OPT_CG_ONEPASS = 22
GROUP_MIN = 1 << 27         # kCgGroupMin (kl_cg.cu): auto picks groups from this many unknowns on
G = 4                       # passes per group (the handle's default)
# mode 3 against mode 1 over the first 8 iterations: the bar the one-pass path met against the two-kernel path
BAR_SHORT = 1e-12
_worst = {}


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


def _np(v):
    return v.cpu().numpy() if hasattr(v, "cpu") else np.asarray(v)


def _same(a, b):
    return np.array_equal(_np(a.history), _np(b.history)) and np.array_equal(_np(a.x), _np(b.x))


def _group_bytes(its, maxit):
    """Bytes per point and iteration: 16 per pass that stores nothing, 48 per store pass.  A group cut short by maxit
    ends on a store pass; one cut short by convergence ends on a pass that stores nothing plus the finishing pass."""
    full, t = divmod(its, G)
    tail = 0.0 if t == 0 else 16.0 * (t - 1 if its == maxit else t) + 48.0
    return (full * (16.0 * (G - 1) + 48.0) + tail) / its


def _ops(kl):
    return {"stvec": kl.stvec, "aniso": kl.aniso(1.0, 0.01),
            "stencil5": kl.stencil5(4.5, 1.0, 1.0, 1.25, 1.25)}     # symmetric, shifted


def _rel(a, b):
    a, b = _np(a), _np(b)
    return float(np.max(np.abs(a - b)) / np.max(np.abs(b))) if np.max(np.abs(b)) > 0 else float(np.max(np.abs(a)))


@pytest.mark.parametrize("nx,ny", [(300, 300), (1000, 64), (128, 515), (1024, 1024)])
@pytest.mark.parametrize("opname", ["stvec", "aniso", "stencil5"])
@pytest.mark.parametrize("rhs", ["ones", "random"])
def test_group_matches_onepass(kl, h, nx, ny, opname, rhs):
    op = _ops(kl)[opname]
    b = (h.apply(op, np.ones(nx * ny), nx, ny) if rhs == "ones"
         else np.random.default_rng(nx + 7 * ny).standard_normal(nx * ny))
    for its in (1, 2, 3, 4, 5, 7, 8, 64):
        g = _with(h, 3, lambda: h.cg_omp(op, b, 0.0, its, nx=nx, ny=ny))
        s = _with(h, 1, lambda: h.cg_omp(op, b, 0.0, its, nx=nx, ny=ny))
        assert g.iter == s.iter == its and g.history.size == s.history.size == its
        assert g.stats["algorithmic_bytes"] / its / (nx * ny) == pytest.approx(_group_bytes(its, its)), its
        rh = np.abs(_np(g.history) / _np(s.history) - 1)
        rx = _rel(g.x, s.x)
        key = "first8" if its <= 8 else "its64"
        _worst[key] = max(_worst.get(key, (0, 0)), (float(rh.max()), rx))
        if its <= 8:
            assert rh.max() < BAR_SHORT and rx < BAR_SHORT, (its, rh.max(), rx)
        else:
            assert rh.max() < hist_bar("cg_omp_300"), (its, rh.max())
            assert hist_norm(g.history, s.history, float(np.linalg.norm(b))) < 1e-10
            assert rx < 1e-10, (its, rx)
    print(f"group vs one-pass, worst so far (history rel, x rel): {_worst}")


@pytest.mark.parametrize("check_every", [3, 4, 5, 6, 7])
def test_group_batches_starting_at_every_phase(kl, h, check_every):
    """Poll intervals that are not multiples of G start batches at every phase of a group (run eagerly); the
    results equal a run polled every two groups (batches replayed as CUDA graphs) and a run polled never, bit for
    bit."""
    ns = 300
    b = h.apply(kl.stvec, np.ones(ns * ns), ns, ns)
    for its in (24, 25, 26, 27, 40):
        g = _with(h, 3, lambda: h.cg_omp(kl.stvec, b, 0.0, its), check_every)
        s = _with(h, 3, lambda: h.cg_omp(kl.stvec, b, 0.0, its), 2 * G)
        t = _with(h, 3, lambda: h.cg_omp(kl.stvec, b, 0.0, its), 1000)
        assert g.iter == its
        assert _same(g, s) and _same(g, t), its


def test_group_graph_replay_bit_identical(kl, h):
    ns = 1000
    b = h.apply(kl.stvec, np.ones(ns * ns), ns, ns)
    run = lambda ce: _with(h, 3, lambda: h.cg_omp(kl.stvec, b, 1e-9, 200), ce)
    g1, g2 = run(24), run(24)     # batches of an even number of groups after the first are replayed as CUDA graphs
    e = run(25)                   # batches that start mid-group run eagerly
    assert g1.iter == g2.iter == e.iter == 200
    assert _same(g1, g2) and _same(g1, e)


@pytest.mark.parametrize("device", [False, True])
def test_group_early_convergence_every_phase(kl, h, device):
    """Convergence at every pass j = 1..G of a group: the later passes are gated off, a pass j < G is followed by one
    store pass that forms x; x equals the tol = 0 run of that many iterations bit for bit."""
    ns = 300
    b = h.apply(kl.stvec, np.ones(ns * ns), ns, ns)
    if device:
        import torch
        b = torch.from_numpy(b).cuda()
    run = lambda tol, its: _with(h, 3, lambda: h.cg_omp(kl.stvec, b, tol, its, nx=ns, ny=ns))
    hist = _np(run(0.0, 120).history)
    seen = set()
    for k in range(2, 120):
        if k % G in seen or not hist[k - 1] < hist[: k - 1].min():
            continue
        seen.add(k % G)
        tol = 0.5 * (hist[k - 1] + hist[: k - 1].min())        # first met at iteration k
        ref = run(0.0, k)
        for maxit in (k + 5, k + 6, k + 7):
            g = run(tol, maxit)
            assert g.status == 0 and g.iter == k and g.history.size == k
            assert np.array_equal(_np(g.history), _np(ref.history))
            assert np.array_equal(_np(g.x), _np(ref.x)), (k, maxit)
            assert g.stats["algorithmic_bytes"] / k / (ns * ns) == pytest.approx(_group_bytes(k, maxit))
    assert seen == set(range(G))


@pytest.mark.parametrize("maxit", [25, 26, 27])
def test_group_not_converged_leaves_iter(kl, h, maxit):
    ns = 300
    b = h.apply(kl.stvec, np.ones(ns * ns), ns, ns)
    g = _with(h, 3, lambda: h.cg_omp(kl.stvec, b, 1e-9, maxit))
    assert g.status == kl.api.KL_NOT_CONVERGED and g.iter == maxit and g.history.size == maxit
    assert g.stats["iterations"] == maxit
    assert g.stats["algorithmic_bytes"] / maxit / (ns * ns) == pytest.approx(_group_bytes(maxit, maxit))


@pytest.mark.parametrize("ns", [100, 300])
def test_group_parity_with_oracle(kl, h, ko, ns):
    b = ko.manufactured_rhs(ko.stvec_fn(), ns)
    o = ko.cg_omp(ko.stvec_fn(), b, 1e-9, 10000)
    g = _with(h, 3, lambda: h.cg_omp(kl.stvec, b, 1e-9, 10000))
    assert g.status == 0 and abs(g.iter - o.iter) <= 1
    k = min(g.history.size, o.history.size)
    rel = np.abs(g.history[:k] / o.history[:k] - 1)
    assert rel[:50].max() < 1e-10
    assert rel.max() < hist_bar(f"cg_omp_{ns}"), (rel.max(), hist_bar(f"cg_omp_{ns}"))
    assert hist_norm(g.history, o.history, float(np.linalg.norm(b))) < 1e-10
    assert np.abs(g.x - o.x).max() / np.abs(o.x).max() < 1e-9
    assert np.abs(g.x - 1).max() < 1e-9


@pytest.mark.parametrize("its", [24, 25])
def test_group_warm_start(kl, h, its):
    """KL_OPT_X0: the recurrence never reads x, so a warm start is the cold solve of b - A x0, plus x0."""
    ns = 300
    rng = np.random.default_rng(its)
    b = rng.standard_normal(ns * ns)
    x0 = rng.standard_normal(ns * ns)
    shifted = b - h.apply(kl.stvec, x0, ns, ns)
    w = _with(h, 3, lambda: h.cg_omp(kl.stvec, b, 0.0, its, x0=x0))              # (x0= sets KL_OPT_X0)
    z = _with(h, 3, lambda: h.cg_omp(kl.stvec, b, 0.0, its, x0=np.zeros(ns * ns)))
    cold = _with(h, 3, lambda: h.cg_omp(kl.stvec, shifted, 0.0, its))
    cold_b = _with(h, 3, lambda: h.cg_omp(kl.stvec, b, 0.0, its))
    assert np.abs(_np(w.history) / _np(cold.history) - 1).max() < 1e-12
    assert np.abs(_np(w.x) - (x0 + _np(cold.x))).max() / np.abs(_np(w.x)).max() < 1e-14
    assert _same(z, cold_b)


def test_group_auto_threshold(kl, h):
    """The default picks groups from GROUP_MIN unknowns on: 8192 x 16384 (2^27) runs groups, 8192^2 pairs."""
    import torch
    for nx, ny in ((8192, 8192), (8192, 16384)):
        n = nx * ny
        want = _group_bytes(G, G) if n >= GROUP_MIN else 36.0
        b = h.apply(kl.stvec, torch.ones(n, dtype=torch.float64, device="cuda"), nx, ny)
        g = h.cg_omp(kl.stvec, b, 0.0, 2 * G, nx=nx, ny=ny)
        assert g.stats["algorithmic_bytes"] / (2 * G) / n == pytest.approx(want), (nx, ny)
        del b, g
        torch.cuda.empty_cache()
