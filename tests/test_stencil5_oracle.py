"""CPU: KL_OP_STENCIL5's definition and its host-side pieces (no GPU needed).

- the CPU twin (tests/stencil5_twin.c) equals a dense matrix built from the weights, on rectangular grids;
- kl_stencil5_spectrum equals the extreme eigenvalues of that matrix (numpy.linalg.eigvals) on grids up to 12 x 12, and
  refuses a complex spectrum;
- kl.convdiff builds the documented weights;
- the Python mirror rejects malformed weights before any call into the library.
"""
import ctypes as C
import math

import numpy as np
import pytest

import stencil5_twin as tw

# nonsymmetric, real spectrum: central px = 0.5, py = 0.25 ; upwind ; negative weights on both sides ; reaction-diffusion
W_REAL = [
    (4.0, 1.5, 0.5, 0.75, 1.25),
    (7.0, 3.0, 1.0, 1.0, 2.0),
    (1.5, -0.5, -2.0, -0.25, -1.0),
    (4.3, 1.0, 1.0, 1.0, 1.0),
    (3.0, 0.9, 0.1, 1.7, 0.3),
]
W_COMPLEX = [
    (4.0, 2.5, -0.5, 1.0, 1.0),     # central px = 1.5
    (4.0, 1.0, 1.0, 0.5, -1.0),
    (4.0, -1.0, 1.0, -1.0, 1.0),
]


@pytest.mark.parametrize("nx,ny", [(1, 1), (2, 3), (5, 4), (7, 9), (12, 5), (3, 12)])
@pytest.mark.parametrize("w", W_REAL + W_COMPLEX)
def test_twin_is_the_dense_matrix(w, nx, ny):
    rng = np.random.default_rng(nx * 100 + ny)
    A = tw.dense(w, nx, ny)
    # small integers: every product and sum is exact, so the twin's rounding order cannot show
    xi = rng.integers(-8, 9, nx * ny).astype(np.float64)
    wi = (8.0, 3.0, -2.0, 1.0, 5.0)
    assert np.array_equal(tw.apply_xy(wi, xi, nx, ny), tw.dense(wi, nx, ny) @ xi)
    x = rng.standard_normal(nx * ny)
    y = tw.apply_xy(w, x, nx, ny)
    assert np.allclose(y, A @ x, rtol=0, atol=1e-13 * (np.abs(A).sum(axis=1).max() * np.abs(x).max()))


def test_twin_evaluation_order_is_aniso_var_on_constant_fields(ko):
    """c = ((a+a)+b)+b, wl = wr = a, wd = wu = b reproduces the oracle's ko_aniso_var on kx = a, ky = b bit for bit."""
    n = 23
    rng = np.random.default_rng(5)
    for a, b in ((1.0, 0.01), (0.37, 2.9), (1.3e-3, 7.1)):
        x = rng.standard_normal(n * n)
        kx, ky = np.full(n * n, a), np.full(n * n, b)
        ref = ko.apply(ko.aniso_var_fn(kx, ky), x, n)
        assert np.array_equal(tw.apply_xy((((a + a) + b) + b, a, a, b, b), x, n, n), ref)


def _lib():
    from gmres_b200.api import load_library
    return load_library()


def _spectrum(w, nx, ny):
    from gmres_b200.api import kl_stencil5_t
    lo, hi = C.c_double(), C.c_double()
    rc = _lib().kl_stencil5_spectrum(C.byref(kl_stencil5_t(*w)), nx, ny, C.byref(lo), C.byref(hi))
    return rc, lo.value, hi.value


@pytest.mark.parametrize("nx,ny", [(1, 1), (2, 2), (3, 7), (6, 6), (9, 4), (12, 12), (12, 1)])
@pytest.mark.parametrize("w", W_REAL)
def test_spectrum_is_exact(w, nx, ny):
    rc, lo, hi = _spectrum(w, nx, ny)
    assert rc == 0
    ev = np.linalg.eigvals(tw.dense(w, nx, ny))
    assert np.abs(ev.imag).max() < 1e-6            # real up to the eigenvalues' conditioning
    scale = max(abs(lo), abs(hi))
    assert abs(lo - ev.real.min()) <= 1e-10 * scale and abs(hi - ev.real.max()) <= 1e-10 * scale


# (central |p| -> 1 is left out: the eigenvalues numpy computes are then ill-conditioned far beyond 1e-10 -- the diagonal
# similarity that makes the spectrum real scales by ((1+p)/(1-p))^(n/2) -- and |p| = 1 is a defective matrix)
@pytest.mark.parametrize("px,py,upwind", [(0.5, 0.5, False), (0.5, 0.25, False), (-0.4, 0.3, False), (0.0, 0.5, False),
                                          (2.0, 0.0, True), (-3.0, 0.5, True), (0.5, 0.25, True)])
def test_spectrum_of_convdiff(px, py, upwind):
    import gmres_b200 as kl
    op = kl.convdiff(px, py, upwind)
    for nx, ny in ((8, 8), (12, 10)):
        lo, hi = kl.stencil5_spectrum(op, nx, ny)
        ev = np.linalg.eigvals(tw.dense(op.w5, nx, ny)).real
        assert abs(lo - ev.min()) <= 1e-10 * hi and abs(hi - ev.max()) <= 1e-10 * hi


@pytest.mark.parametrize("w", W_COMPLEX)
def test_spectrum_refuses_a_complex_spectrum(w):
    rc, lo, hi = _spectrum(w, 8, 8)
    assert rc == -5 and math.isnan(lo) and math.isnan(hi)       # KL_ERR_UNSUPPORTED
    assert np.abs(np.linalg.eigvals(tw.dense(w, 8, 8)).imag).max() > 1e-3
    import gmres_b200 as kl
    with pytest.raises(kl.KrylovError, match="complex"):
        kl.stencil5_spectrum(kl.stencil5(*w), 8, 8)
    with pytest.raises(kl.KrylovError, match="complex"):
        kl.stencil5_spectrum(kl.convdiff(1.5, 0.0), 8, 8)


def test_spectrum_argument_checks():
    from gmres_b200.api import kl_stencil5_t
    lo, hi = C.c_double(), C.c_double()
    L = _lib()
    w = kl_stencil5_t(4.0, 1.0, 1.0, 1.0, 1.0)
    assert L.kl_stencil5_spectrum(None, 4, 4, C.byref(lo), C.byref(hi)) == -1
    assert L.kl_stencil5_spectrum(C.byref(w), 0, 4, C.byref(lo), C.byref(hi)) == -1
    assert L.kl_stencil5_spectrum(C.byref(kl_stencil5_t(4.0, float("nan"), 1.0, 1.0, 1.0)), 4, 4,
                                  C.byref(lo), C.byref(hi)) == -1
    # Poisson: 4 -+ 4 cos(pi/(n+1))
    assert L.kl_stencil5_spectrum(C.byref(w), 7, 7, C.byref(lo), C.byref(hi)) == 0
    assert lo.value == pytest.approx(4 - 4 * math.cos(math.pi / 8), rel=1e-15)
    assert hi.value == pytest.approx(4 + 4 * math.cos(math.pi / 8), rel=1e-15)


@pytest.mark.parametrize("px,py", [(0.5, 0.5), (0.5, 0.25), (-0.9, 0.3), (2.0, -1.5), (0.0, 0.0)])
def test_convdiff_weights(px, py):
    import gmres_b200 as kl
    assert kl.convdiff(px, py).w5 == (4.0, 1 + px, 1 - px, 1 - py, 1 + py)
    c, wl, wr, wd, wu = kl.convdiff(px, py, upwind=True).w5
    assert c == (4.0 + 2 * abs(px)) + 2 * abs(py)
    assert (wl, wr) == ((1 + 2 * abs(px), 1.0) if px >= 0 else (1.0, 1 + 2 * abs(px)))
    assert (wu, wd) == ((1 + 2 * abs(py), 1.0) if py >= 0 else (1.0, 1 + 2 * abs(py)))
    # upwinding is central differencing with the artificial diffusion |p| added on each axis
    cc, cl, cr, cd, cu = kl.convdiff(px, py).w5
    assert np.allclose((c, wl, wr, wd, wu), (cc + 2 * abs(px) + 2 * abs(py), cl + abs(px), cr + abs(px),
                                              cd + abs(py), cu + abs(py)), rtol=0, atol=1e-15)


def test_stencil5_descriptor():
    import gmres_b200 as kl
    from gmres_b200.api import KL_OP_STENCIL5, kl_stencil5_t
    op = kl.stencil5(4, 1.5, 0.5, np.float64(0.75), np.int64(1))
    assert op.kind == KL_OP_STENCIL5 == 5 and op.w5 == (4.0, 1.5, 0.5, 0.75, 1.0)
    o, keep = op._c()
    w = C.cast(o.user, C.POINTER(kl_stencil5_t)).contents
    assert (w.c, w.wl, w.wr, w.wd, w.wu) == op.w5 and isinstance(keep, kl_stencil5_t)


@pytest.mark.parametrize("bad", [float("nan"), float("inf"), -float("inf"), "1.0", None, True, 1 + 2j, [1.0]])
@pytest.mark.parametrize("pos", range(5))
def test_malformed_weights_raise_before_the_library(monkeypatch, bad, pos):
    import gmres_b200 as kl
    from gmres_b200 import api

    def no_library():
        raise AssertionError("the library was called")

    monkeypatch.setattr(api, "load_library", no_library)
    w = [4.0, 1.0, 1.0, 1.0, 1.0]
    w[pos] = bad
    with pytest.raises(kl.KrylovError):
        kl.stencil5(*w)
    if pos < 2:
        with pytest.raises(kl.KrylovError):
            kl.convdiff(*([0.5, bad] if pos else [bad, 0.5]))


def test_spectrum_rejects_other_operators_before_the_library(monkeypatch):
    import gmres_b200 as kl
    from gmres_b200 import api

    def no_library():
        raise AssertionError("the library was called")

    monkeypatch.setattr(api, "load_library", no_library)
    for op in (kl.stvec, kl.aniso(1.0, 0.01), None):
        with pytest.raises(kl.KrylovError):
            kl.stencil5_spectrum(op, 8, 8)
    with pytest.raises(kl.KrylovError):
        kl.stencil5_spectrum(kl.convdiff(0.5, 0.5), 0, 8)
