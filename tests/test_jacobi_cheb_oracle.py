"""CPU twin of the Jacobi-scaled Chebyshev preconditioner (KL_PC_JACOBI_CHEB, tests/jacobi_cheb_twin.c): the spectral
bound its interval rests on, the recurrence against a dense numpy evaluation, and its operator against the oracle's."""
import numpy as np
import pytest

import jacobi_cheb_twin as twin


def _fields(nx, ny, seed, contrast=1e4, aniso=100.0):
    rng = np.random.default_rng(seed)
    lc = np.log(contrast) / 2
    kx = np.exp(rng.uniform(-lc, lc, nx * ny))
    ky = np.exp(rng.uniform(-lc, lc, nx * ny)) / aniso
    return kx, ky


def _dense_op(kx, ky, nx, ny):
    n = nx * ny
    A = np.zeros((n, n))
    e = np.zeros(n)
    for k in range(n):
        e[k] = 1.0
        A[:, k] = twin.aniso_var_xy(kx, ky, e, nx, ny)
        e[k] = 0.0
    return A


def _recurrence(A, dinv, r, k, a, b):
    """Saad Alg. 12.1 on D^-1 A, written out with numpy (no fma: agreement to rounding, not bits)"""
    s = r * dinv
    if k == 0:
        return s
    theta, delta = (b + a) / 2.0, abs(b - a) / 2.0
    sigma = theta / delta
    rho_prev = 1.0 / sigma
    d = s / theta
    z = d.copy()
    for _ in range(k):
        rho = 1.0 / (2.0 * sigma - rho_prev)
        d = rho * rho_prev * d + (2.0 * rho / delta) * ((r - A @ z) * dinv)
        z = z + d
        rho_prev = rho
    return z


@pytest.mark.parametrize("nx,ny", [(24, 17), (31, 31)])
def test_jacobi_scaled_spectrum_in_0_2(ko, nx, ny):
    kx, ky = _fields(nx, ny, nx * ny)
    A = _dense_op(kx, ky, nx, ny)
    assert np.array_equal(A, A.T)
    dinv = twin.dinv(kx, ky, nx, ny)
    assert np.array_equal(dinv, 1.0 / np.diag(A))
    # D^-1 A is similar to the symmetric D^-1/2 A D^-1/2
    ds = np.sqrt(dinv)
    ev = np.linalg.eigvalsh(ds[:, None] * A * ds[None, :])
    assert ev.min() > 0.0 and ev.max() <= 2.0, (ev.min(), ev.max())


@pytest.mark.parametrize("nx,ny", [(24, 17), (31, 31)])
def test_twin_matches_dense_recurrence(ko, nx, ny):
    kx, ky = _fields(nx, ny, 7 + nx)
    A = _dense_op(kx, ky, nx, ny)
    dinv = 1.0 / np.diag(A)
    r = np.random.default_rng(3).standard_normal(nx * ny)
    for a, b in ((0.02, 2.0), (2.0, 0.1)):
        for k in range(9):
            z = twin.jacobi_cheb(kx, ky, r, k, (a, b), nx, ny)
            ref = _recurrence(A, dinv, r, k, a, b)
            rel = np.linalg.norm(z - ref) / np.linalg.norm(ref)
            assert rel < 1e-13, (k, a, b, rel)


def test_degree_zero_is_point_jacobi(ko):
    nx, ny = 37, 23
    kx, ky = _fields(nx, ny, 5)
    r = np.random.default_rng(9).standard_normal(nx * ny)
    A = _dense_op(kx, ky, nx, ny)
    z = twin.jacobi_cheb(kx, ky, r, 0, (), nx, ny)
    assert np.array_equal(z, r * (1.0 / np.diag(A)))


@pytest.mark.parametrize("n", [5, 32, 47])
def test_twin_operator_is_ko_aniso_var_on_square_grids(ko, n):
    kx, ky = _fields(n, n, n)
    x = np.random.default_rng(n).standard_normal(n * n)
    y = twin.aniso_var_xy(kx, ky, x, n, n)
    assert np.array_equal(y, ko.apply(ko.aniso_var_fn(kx, ky), x, n))


def test_precond_wrapper_runs_in_the_oracle_solvers(ko):
    n = 32
    kx, ky = _fields(n, n, 1, contrast=100.0)
    Ao = ko.aniso_var_fn(kx, ky)
    r = np.random.default_rng(2).standard_normal(n * n)
    z = ko.apply_precond(twin.precond_fn(ko, kx, ky, 3), Ao, r, (0.05, 2.0), n)
    assert np.array_equal(z, twin.jacobi_cheb(kx, ky, r, 3, (0.05, 2.0), n, n))
    Ao = ko.aniso_var_fn(kx, ky)
    b = ko.manufactured_rhs(Ao, n)
    plain = ko.cg_omp(Ao, b, 1e-9, 20000)
    pre = ko.pcg_omp(Ao, b, 1e-9, 20000, twin.precond_fn(ko, kx, ky, 3), (0.05, 2.0))
    assert np.abs(pre.x - 1.0).max() < 1e-6 and pre.iter < plain.iter
