"""CPU tests of the CSR twin (tests/csr_twin.c) and of the host-side checks of kl.csr (no GPU needed).

The twin defines the evaluation order of KL_OP_CSR that the GPU kernels are held to bit for bit
(tests/test_gpu_csr.py); here it is held to scipy's A @ x within rounding, on every lane width W.
"""
import numpy as np
import pytest
import scipy.sparse as sp

import csr_twin as twin


def _rand(n, per_row, seed, unsorted=True, dups=True):
    """n rows of 0..2*per_row-1 entries (exactly one for per_row = 1, so that W = 1) with random columns (duplicates kept
    unless dups=False), storage order random"""
    rng = np.random.default_rng(seed)
    lens = rng.integers(0, 2 * per_row, n) if per_row > 1 else np.ones(n, dtype=np.int64)
    indptr = np.zeros(n + 1, dtype=np.int64)
    indptr[1:] = np.cumsum(lens)
    nnz = int(indptr[-1])
    cols = rng.integers(0, n, nnz).astype(np.int32)
    if not dups:
        for i in range(n):
            a, b = indptr[i], indptr[i + 1]
            cols[a:b] = rng.choice(n, b - a, replace=False)
    if not unsorted:
        for i in range(n):
            cols[indptr[i]:indptr[i + 1]].sort()
    return indptr, cols, rng.standard_normal(nnz)


def _scipy(ip, ix, dv, n):
    # duplicates summed by scipy when it converts; the product is the same matrix
    return sp.csr_matrix((dv, ix, ip), shape=(n, n))


def _rel(a, b):
    return np.abs(a - b).max() / max(np.abs(b).max(), 1e-300)


@pytest.mark.parametrize("per_row", [1, 2, 3, 4, 7, 8, 12, 16, 25, 32, 60])
def test_twin_matches_scipy_every_width(per_row):
    n = 3000
    ip, ix, dv = _rand(n, per_row, per_row)
    x = np.random.default_rng(per_row + 100).standard_normal(n)
    ref = _scipy(ip, ix, dv, n) @ x
    y = twin.spmv((ip, ix, dv), x)
    # error bound of a sum of up to 2*per_row products: a few units of rounding of the row's magnitude
    mag = np.abs(_scipy(ip, ix, np.abs(dv), n) @ np.abs(x)).max()
    assert np.abs(y - ref).max() <= 1e-14 * mag * 2 * per_row
    assert _rel(y, ref) < 1e-13


def test_every_width_is_reached():
    n = 3000
    seen = {twin.width(n, _rand(n, p, p)[0][-1]) for p in (1, 2, 3, 4, 7, 8, 12, 16, 25, 32, 60)}
    assert seen == {1, 2, 4, 8, 16, 32}


def test_width_rule_on_hand_built_cases():
    assert twin.width(10, 0) == 1           # no entries
    assert twin.width(10, 10) == 1          # ceil(1) = 1
    assert twin.width(10, 11) == 2          # ceil(1.1) = 2
    assert twin.width(10, 20) == 2
    assert twin.width(10, 21) == 4          # ceil(2.1) = 3 -> 4
    assert twin.width(10, 40) == 4
    assert twin.width(10, 41) == 8
    assert twin.width(10, 160) == 16
    assert twin.width(10, 161) == 32
    assert twin.width(10, 320) == 32
    assert twin.width(10, 10 ** 6) == 32    # clamped
    assert twin.width(16777216, 83869696) == 8    # CSR Poisson 4096^2: 4.999 per row


def test_hand_built_rows():
    # row 0 empty, row 1 one entry, row 2 unsorted with a duplicate column, row 3 longer than W (nnz 11 over 4 rows:
    # ceil(2.75) = 3 -> W = 4)
    ip = np.array([0, 0, 1, 5, 11])
    ix = np.array([2, 3, 0, 3, 0, 0, 1, 2, 3, 1, 0], dtype=np.int32)
    dv = np.array([2.0, 1.5, -1.0, 0.25, 4.0, 1.0, 2.0, 3.0, 4.0, 5.0, 6.0])
    x = np.array([1.0, 2.0, 3.0, 4.0])
    y = twin.spmv((ip, ix, dv), x)
    assert y[0] == 0.0
    assert y[1] == 2.0 * 3.0
    assert y[2] == 1.5 * 4.0 - 1.0 * 1.0 + 0.25 * 4.0 + 4.0 * 1.0
    # W = 4: lanes take k = 5+l, 9+l: lane0 = fma(5, 2, fma(1, 1, 0)) = 11, lane1 = fma(6, 1, 2*2) = 10, lane2 = 9,
    # lane3 = 16; butterfly off 2: (11+9, 10+16, ...), off 1: 20 + 26 = 46
    assert twin.width(4, 11) == 4
    assert y[3] == 46.0
    assert np.array_equal(twin.diag((ip, ix, dv)), np.array([0.0, 0.0, 0.0, 4.0]))     # only row 3 stores (3, 3)


def test_duplicates_and_unsorted_columns_add_up():
    n = 500
    ip, ix, dv = _rand(n, 9, 7)
    A = _scipy(ip, ix, dv, n)
    x = np.random.default_rng(8).standard_normal(n)
    assert _rel(twin.spmv((ip, ix, dv), x), A @ x) < 1e-13
    d = twin.diag((ip, ix, dv))
    assert np.abs(d - A.diagonal()).max() <= 1e-14 * np.abs(dv).max() * 4


def test_poisson_matrix_is_the_stencil():
    ns = 37
    A = twin.poisson5(ns)
    assert A.nnz == 5 * ns * ns - 4 * ns
    x = np.random.default_rng(1).standard_normal(ns * ns)
    X = x.reshape(ns, ns)              # [j, i]
    P = np.pad(X, 1)
    ref = (4 * X - P[1:-1, :-2] - P[1:-1, 2:] - P[:-2, 1:-1] - P[2:, 1:-1]).reshape(-1)
    assert _rel(twin.spmv(A, x), ref) < 1e-14


def test_jacobi_cheb_degree0_and_recurrence():
    n = 400
    ip, ix, dv = twin.irregular(n, 3, long_rows=2, long_len=300, max_len=20)
    A = _scipy(ip, ix, dv, n)
    r = np.random.default_rng(4).standard_normal(n)
    assert np.array_equal(twin.jacobi_cheb((ip, ix, dv), r, 0, ()), r * (1.0 / twin.diag((ip, ix, dv))))
    # degree k: the Chebyshev polynomial of D^-1 A applied to D^-1 r; compare with a float64 numpy restatement
    Dinv = 1.0 / A.diagonal()
    a, b = 0.05, 1.9
    theta, delta = (a + b) / 2, (b - a) / 2
    sigma = theta / delta
    rho = 1 / sigma
    d = Dinv * r / theta
    z = d.copy()
    for _ in range(5):
        rn = 1 / (2 * sigma - rho)
        d = rn * rho * d + 2 * rn / delta * (Dinv * (r - A @ z))
        z = z + d
        rho = rn
    assert _rel(twin.jacobi_cheb((ip, ix, dv), r, 5, (a, b)), z) < 1e-12


# ---- kl.csr: host-side checks ----------------------------------------------------------------------------------------
@pytest.fixture
def no_device(monkeypatch):
    """any attempt of kl.csr to reach a device fails the test"""
    import torch

    class Touched(Exception):
        pass

    def boom(*a, **k):
        raise Touched("kl.csr reached the device")

    monkeypatch.setattr(torch.cuda, "current_device", boom)
    monkeypatch.setattr(torch.Tensor, "to", boom)
    monkeypatch.setattr(torch.Tensor, "cuda", boom)
    return Touched


def _bad_inputs():
    ip, ix, dv = np.array([0, 2, 3, 4]), np.array([0, 1, 1, 2], dtype=np.int32), np.array([4.0, -1.0, 4.0, 4.0])
    yield "non-square", (sp.csr_matrix(np.ones((3, 4))),), "square"
    yield "indptr not starting at 0", ((np.array([1, 2, 3, 4]), ix, dv), 3), "indptr"
    yield "indptr decreasing", ((np.array([0, 3, 2, 4]), ix, dv), 3), "indptr"
    yield "indptr not ending at nnz", ((np.array([0, 2, 3, 3]), ix, dv), 3), "indptr"
    yield "indptr length", ((np.array([0, 2, 4]), ix, dv), 3), "indptr"
    yield "column out of range", ((ip, np.array([0, 1, 3, 2], dtype=np.int32), dv), 3), "column"
    yield "negative column", ((ip, np.array([0, -1, 1, 2], dtype=np.int32), dv), 3), "column"
    yield "NaN value", ((ip, ix, np.array([4.0, np.nan, 4.0, 4.0])), 3), "finite"
    yield "inf value", ((ip, ix, np.array([4.0, np.inf, 4.0, 4.0])), 3), "finite"
    yield "non-numeric values", ((ip, ix, np.array(["a", "b", "c", "d"])), 3), "float64"
    yield "indices/values length", ((ip, ix[:3], dv), 3), "column indices"
    yield "n >= 2^31", ((ip, ix, dv), 2 ** 31), "2\\^31"
    yield "n < 2", ((np.array([0, 1]), np.array([0], dtype=np.int32), np.array([1.0])), 1), "2 <= n"
    yield "tuple without n", ((ip, ix, dv),), "needs n"
    yield "dense array", (np.eye(3),), "expected"


@pytest.mark.parametrize("case", list(_bad_inputs()), ids=lambda c: c[0])
def test_csr_rejects_malformed_input_before_the_device(no_device, case):
    import gmres_b200 as kl
    _, args, msg = case
    with pytest.raises(kl.KrylovError, match=msg):
        kl.csr(*args)


def test_csr_accepts_valid_input_up_to_the_upload(no_device):
    import gmres_b200 as kl
    A = twin.poisson5(8)
    for args in ((A,), (A.tocoo(),), ((A.indptr, A.indices, A.data), 64), ((A.indptr.astype(np.int64),
                                                                           A.indices.astype(np.int64), A.data), 64)):
        with pytest.raises(no_device):
            kl.csr(*args)
