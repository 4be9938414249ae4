"""CPU check of the one-reduction CG recurrence that the one-pass GPU path runs (ChCg / PostCgOnePass, kl_cg.cu).

One pass per iteration produces r' = r - alpha A p, p' = r' + beta p, x' = x + alpha p and the sums rho = r'.r',
gamma = p'.Ap', sigma = r'.Ap', delta = Ap'.Ap'.  alpha' = rho / gamma is the textbook formula on true dot products;
beta' = rho_hat / rho with rho_hat = rho - 2 alpha' sigma + alpha'^2 delta = ||r' - alpha' Ap'||^2 expanded, i.e. the
next iteration's r.r predicted from this one's sums.  The residual history and the stopping test use the true rho.

Restated here in numpy (matrix-free 5-point operator, b = A 1, sequential sums) against textbook Hestenes-Stiefel CG:
the same iteration count, the history within the bars the GPU parity tests use against the reference
(tests/parity.py), and the same solution.
"""
import numpy as np
import pytest

from parity import hist_bar, hist_rel


def _apply(v, n):
    X = v.reshape(n, n)
    P = np.zeros((n + 2, n + 2))
    P[1:-1, 1:-1] = X
    return (4 * X - (((P[1:-1, :-2] + P[1:-1, 2:]) + P[2:, 1:-1]) + P[:-2, 1:-1])).reshape(-1)


def _cg_hs(b, n, tol, maxit):
    x = np.zeros_like(b); r = b.copy(); p = np.zeros_like(b); beta = 0.0; rr = r @ r; hist = []
    for k in range(maxit):
        p = r + beta * p
        ap = _apply(p, n)
        alpha = rr / (ap @ p)
        x += alpha * p
        r -= alpha * ap
        rn = r @ r
        hist.append(np.sqrt(rn))
        beta = rn / rr
        rr = rn
        if hist[-1] < tol:
            return x, np.array(hist), k + 1
    return x, np.array(hist), maxit


def _cg_onepass(b, n, tol, maxit):
    def scalars(rho, gam, sig, dl):           # PostCgOnePass / cg_onepass_scalars (kl_posts.cuh)
        alpha = rho / gam
        return alpha, (rho - 2.0 * alpha * sig + alpha * alpha * dl) / rho

    x = np.zeros_like(b); r = b.copy(); p = r.copy(); ap = _apply(p, n); hist = []
    alpha, beta = scalars(r @ r, p @ ap, r @ ap, ap @ ap)     # prologue: p_0 = r_0
    for k in range(maxit):
        x = x + alpha * p
        r = r - alpha * ap
        p = r + beta * p
        ap = _apply(p, n)
        rho = r @ r
        hist.append(np.sqrt(rho))
        if hist[-1] < tol:
            return x, np.array(hist), k + 1
        alpha, beta = scalars(rho, p @ ap, r @ ap, ap @ ap)
    return x, np.array(hist), maxit


@pytest.mark.parametrize("ns", [100, 300])
def test_onepass_recurrence_matches_hestenes_stiefel(ns):
    b = _apply(np.ones(ns * ns), ns)
    x0, h0, k0 = _cg_hs(b, ns, 1e-9, 10000)
    x1, h1, k1 = _cg_onepass(b, ns, 1e-9, 10000)
    assert k1 == k0
    rel = np.abs(h1 / h0 - 1)
    assert rel[:50].max() < 1e-10
    assert hist_rel(h1, h0) < hist_bar(f"cg_omp_{ns}")
    assert np.abs(x1 - x0).max() < 1e-12 and np.abs(x1 - 1).max() < 1e-9
