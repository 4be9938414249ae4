"""ctypes loader of the CPU twin of KL_OP_CSR and of KL_PC_JACOBI_CHEB on it (tests/csr_twin.c; test infrastructure
only), and builders of the test matrices.

The library is compiled on first use into a temporary directory (removed at exit), with the oracle's flags, so that
the source tree may be read-only.  The arrays of the matrix last set are kept alive here while the twin holds pointers
to them.
"""
import ctypes as C
import os
import subprocess
import tempfile

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
_dp = C.POINTER(C.c_double)
_lib = None
_dir = None
_keep = None


def lib():
    global _lib, _dir
    if _lib is None:
        _dir = tempfile.TemporaryDirectory(prefix="csr_twin_")
        so = os.path.join(_dir.name, "libcsr_twin.so")
        subprocess.check_call(["gcc", "-O3", "-fopenmp", "-march=x86-64-v3", "-funroll-loops", "-ffp-contract=off",
                               "-fPIC", "-std=gnu11", "-shared", "-o", so, os.path.join(_HERE, "csr_twin.c"), "-lm"])
        _lib = C.CDLL(so)
        _lib.csr_set.argtypes = [C.c_int64, C.c_int64, C.c_void_p, C.c_void_p, C.c_void_p]
        _lib.csr_width.argtypes = [C.c_int64, C.c_int64]
    return _lib


def _p(a):
    return a.ctypes.data_as(_dp)


def set_matrix(indptr, indices, data):
    global _keep
    rp = np.ascontiguousarray(indptr, dtype=np.int64)
    ci = np.ascontiguousarray(indices, dtype=np.int32)
    v = np.ascontiguousarray(data, dtype=np.float64)
    _keep = (rp, ci, v)
    lib().csr_set(rp.size - 1, v.size, rp.ctypes.data, ci.ctypes.data, v.ctypes.data)


def _arrays(A):
    """(indptr, indices, data) of a scipy.sparse matrix (its storage order kept) or of such a tuple"""
    if hasattr(A, "tocsr"):
        M = A.tocsr()
        return M.indptr, M.indices, M.data
    return A


def width(n, nnz):
    return lib().csr_width(int(n), int(nnz))


def spmv(A, x):
    """y = A x in the kernels' order"""
    set_matrix(*_arrays(A))
    x = np.ascontiguousarray(x, dtype=np.float64)
    y = np.zeros_like(x)
    lib().csr_spmv(_p(x), _p(y))
    return y


def diag(A):
    """diag(A) as the kernels sum it"""
    ip, ix, dv = _arrays(A)
    set_matrix(ip, ix, dv)
    out = np.zeros(len(ip) - 1)
    lib().csr_diag(_p(out))
    return out


def jacobi_cheb(A, r, degree, params):
    """z = M^-1 r of KL_PC_JACOBI_CHEB of the given degree"""
    set_matrix(*_arrays(A))
    lib().csr_set_degree(int(degree))
    r = np.ascontiguousarray(r, dtype=np.float64)
    z = np.zeros_like(r)
    aux = np.zeros_like(r)
    prm = np.ascontiguousarray(params if len(params) else (0.0, 0.0), dtype=np.float64)
    lib().csr_jacobi_cheb(_p(r), _p(z), _p(aux), _p(prm))
    return z


def stencil_fn(ko, A):
    """the twin as an operator of the oracle solvers (`ko` = oracle.oracle)"""
    set_matrix(*_arrays(A))
    return ko.STENCIL_FN(C.cast(lib().csr_apply, C.c_void_p).value)


def precond_fn(ko, A, degree):
    """the twin's Jacobi-Chebyshev as a preconditioner of the oracle solvers; also sets A as the twin's matrix"""
    set_matrix(*_arrays(A))
    lib().csr_set_degree(int(degree))
    return ko.PRECOND_FN(C.cast(lib().csr_precond, C.c_void_p).value)


# ---- test matrices -------------------------------------------------------------------------------------------------
def poisson5(ns):
    """the 5-point Poisson matrix of KL_OP_POISSON5 on an ns x ns grid (idx = i + j*ns), rows sorted by column"""
    import scipy.sparse as sp
    t = sp.diags([-np.ones(ns - 1), 4.0 * np.ones(ns), -np.ones(ns - 1)], [-1, 0, 1])
    e = sp.diags([-np.ones(ns - 1), -np.ones(ns - 1)], [-1, 1])
    i = sp.identity(ns)
    A = (sp.kron(i, t) + sp.kron(e, i)).tocsr()
    A.sort_indices()
    return A


def stencil5(w, nx, ny):
    """the matrix of KL_OP_STENCIL5 with weights w = (c, wl, wr, wd, wu), storage order l, r, d, u, c per row"""
    import scipy.sparse as sp
    c, wl, wr, wd, wu = (float(v) for v in w)
    n = nx * ny
    idx = np.arange(n)
    i, j = idx % nx, idx // nx
    rows, cols, vals = [], [], []
    for ok, off, wgt in ((i > 0, -1, -wl), (i < nx - 1, 1, -wr), (j < ny - 1, nx, -wd), (j > 0, -nx, -wu)):
        rows.append(idx[ok]); cols.append(idx[ok] + off); vals.append(np.full(ok.sum(), wgt))
    rows.append(idx); cols.append(idx); vals.append(np.full(n, c))
    A = sp.csr_matrix((np.concatenate(vals), (np.concatenate(rows), np.concatenate(cols))), shape=(n, n))
    A.sort_indices()
    return A


def aniso_var(kx, ky, nx, ny):
    """the matrix of KL_OP_ANISO5_VAR (face weights as in ko_aniso_var)"""
    import scipy.sparse as sp
    n = nx * ny
    idx = np.arange(n)
    i, j = idx % nx, idx // nx
    kx = np.asarray(kx, dtype=np.float64); ky = np.asarray(ky, dtype=np.float64)
    wl = np.where(i > 0, 0.5 * (kx + np.roll(kx, 1)), kx)
    wr = np.where(i < nx - 1, 0.5 * (kx + np.roll(kx, -1)), kx)
    wu = np.where(j > 0, 0.5 * (ky + np.roll(ky, nx)), ky)
    wd = np.where(j < ny - 1, 0.5 * (ky + np.roll(ky, -nx)), ky)
    dg = ((wl + wr) + wd) + wu
    rows, cols, vals = [idx], [idx], [dg]
    for ok, off, wgt in ((i > 0, -1, wl), (i < nx - 1, 1, wr), (j < ny - 1, nx, wd), (j > 0, -nx, wu)):
        rows.append(idx[ok]); cols.append(idx[ok] + off); vals.append(-wgt[ok])
    A = sp.csr_matrix((np.concatenate(vals), (np.concatenate(rows), np.concatenate(cols))), shape=(n, n))
    A.sort_indices()
    return A


def irregular(n, seed, long_rows=4, long_len=10000, max_len=64):
    """n rows of 1..max_len random off-diagonal entries (unsorted, duplicates possible) plus the diagonal, and a few
    rows of about long_len entries; diagonally dominant, so Jacobi is defined"""
    rng = np.random.default_rng(seed)
    lens = rng.integers(1, max_len + 1, n)
    lens[rng.choice(n, long_rows, replace=False)] = long_len
    nnz = int(lens.sum()) + n
    indptr = np.zeros(n + 1, dtype=np.int64)
    indptr[1:] = np.cumsum(lens + 1)
    cols = rng.integers(0, n, nnz).astype(np.int32)
    vals = rng.uniform(-1.0, 1.0, nnz)
    first = indptr[:-1]
    cols[first] = np.arange(n, dtype=np.int32)           # the diagonal first in every row
    vals[first] = 0.0
    absrow = np.add.reduceat(np.abs(vals), first)
    vals[first] = absrow + 1.0
    return indptr, cols, vals
