"""CPU check of the recomputation behind CG in groups of passes (ChCgLook, kl_cg.cu; KL_OPT_CG_ONEPASS = 3).

A group stores r_k, p_k, x_k once; its pass j replays the iterations k .. k+j-1 from them with the alphas and betas
the earlier passes of the group found, and then forms the sums of iteration k+j.  Restated here in numpy (matrix-free
5-point operator, sequential sums): the replayed r, p, x and sums are the one-pass sequence's bit for bit, because
every vector operation is the same operation on the same operands.  Only the order of the block-partial sums differs
on the GPU, which this restatement does not model.
"""
import numpy as np
import pytest


def _apply(v, n):
    X = v.reshape(n, n)
    P = np.zeros((n + 2, n + 2))
    P[1:-1, 1:-1] = X
    return (4 * X - (((P[1:-1, :-2] + P[1:-1, 2:]) + P[2:, 1:-1]) + P[:-2, 1:-1])).reshape(-1)


def _scalars(r, p, ap):                  # PostCgOnePass / cg_onepass_scalars (kl_posts.cuh)
    rho, gam, sig, dl = r @ r, p @ ap, r @ ap, ap @ ap
    alpha = rho / gam
    return rho, alpha, (rho - 2.0 * alpha * sig + alpha * alpha * dl) / rho


def _onepass(b, n, maxit):
    """One pass per iteration: every r, p, x stored; history and the final x."""
    r = b.copy(); p = r.copy(); x = np.zeros_like(b)
    _, alpha, beta = _scalars(r, p, _apply(p, n))
    hist = []
    for _ in range(maxit):
        ap = _apply(p, n)
        x = x + alpha * p
        r = r - alpha * ap
        p = r + beta * p
        rho, alpha, beta = _scalars(r, p, _apply(p, n))
        hist.append(np.sqrt(rho))
    return np.array(hist), x


def _groups(b, n, maxit, G):
    """Groups of G passes: pass j replays j iterations from the group's stored r_k, p_k, x_k; only the last pass of a
    group (or of a group cut short by maxit) stores r, p, x."""
    r = b.copy(); p = r.copy(); x = np.zeros_like(b)
    _, alpha, beta = _scalars(r, p, _apply(p, n))
    al, be, hist = [alpha], [beta], []          # alpha_{k+l}, beta_{k+l} of the current group
    it = 0
    while it < maxit:
        J = min(G, maxit - it)
        for j in range(1, J + 1):
            rr, pp, xx = r, p, x
            for lv in range(j):                 # levels 1..j
                ap = _apply(pp, n)
                xx = xx + al[lv] * pp
                rr = rr - al[lv] * ap
                pp = rr + be[lv] * pp
            rho, alpha, beta = _scalars(rr, pp, _apply(pp, n))      # level j + 1
            hist.append(np.sqrt(rho))
            al.append(alpha); be.append(beta)
        r, p, x = rr, pp, xx                    # the store pass
        al, be = al[J:], be[J:]
        it += J
    return np.array(hist), x


@pytest.mark.parametrize("G", [2, 3, 4])
@pytest.mark.parametrize("maxit", [1, 2, 3, 4, 5, 7, 8, 25])
def test_group_replay_is_onepass_exactly(G, maxit):
    n = 24
    rng = np.random.default_rng(maxit)
    for b in (_apply(np.ones(n * n), n), rng.standard_normal(n * n)):
        h1, x1 = _onepass(b, n, maxit)
        hg, xg = _groups(b, n, maxit, G)
        assert np.array_equal(h1, hg) and np.array_equal(x1, xg), (G, maxit)
