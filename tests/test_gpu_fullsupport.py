"""Kernels and solvers on right-hand sides with support on the whole grid, at the benchmark's grid sizes.

Most other GPU tests feed b = A*1, which for the 5-point operator is zero away from the boundary lines: after k
iterations the Krylov vectors are still zero outside a band of about k lines along each edge, so the CTAs inside
the grid multiply zeros and contribute zero partials, and a wrong halo line, tile height or lost partial sum there
changes no bit of the output.  Here every input is a seeded standard normal vector generated on the device, and

  * point-wise kernels (operators, cbpr2, cheb(k)) are compared BIT FOR BIT with the CPU oracle (square grids) or a
    torch restatement in the kernel's summation order (any grid), over the geometry options and edge shapes;
  * reductions and solvers are compared with restatements of the reference recurrences run in np.longdouble (CPU,
    up to 1024^2) or in FP64 torch on the GPU (bench sizes), the latter calibrated against the former in the same run;
  * options changed on a warm handle must give what a fresh handle with the option set gives (CUDA-graph keys).

`_defect` gives the reference operators a one-CTA error (the upper halo line of one interior CTA dropped); the
sensitivity tests show that these inputs and bars see such an error deep inside the grid.

The bars (history point-wise relative, x relative to max |x|) are below; each test prints what it observes
(pytest -s).
"""
import contextlib

import numpy as np
import pytest

from parity import hist_rel
from test_gpu_large import t_apply, t_cbpr2

gpu = pytest.mark.gpu
P = (8.2, 0.2)          # tests/test_poisson_mf.f90:38, the benchmark's preconditioner parameters

# include/krylov_b200.h
MAX_RESTARTS, VERR, CHECK_EVERY, HH_MODE = 2, 3, 4, 6
TMA, REORTH_ETA, CHAIN, ROWS, PDL, TAIL, STAGGER, REVERSE, PERSISTENT, CG_ONEPASS = 9, 11, 12, 13, 15, 17, 18, 19, 21, 22

# bars: >= 10x the largest deviation observed on a B200 (1000 W power limit), and >= 10x the FP64 torch reference's own
# deviation from np.longdouble (test_cg_1024_three_modes_vs_longdouble, test_solvers_small_vs_longdouble)
BAR_CG = 1e-13          # plain and preconditioned CG, history and x: observed <= 1.4e-15
BAR_RED1 = 1e-14        # history[0] of CG (one reduction of r = b - alpha0 A b) against a longdouble sum: observed <= 4.4e-16
BAR_RED2 = 1e-14        # history[1] (predicted beta, the pass's four fused sums): observed <= 5.6e-16
BAR_BICG = 1e-13        # BiCGSTAB, 12 iterations: observed <= 3.2e-15 (the b = A*1 test's bars are 1e-9 / 1e-5)
BAR_GMRES = 1e-12       # one GMRES-MGSR cycle (always-twice CGS2): observed <= 2.9e-14; the FP64 reference's own
                        # deviation from longdouble reaches 1.3e-14 at 256^2
BAR_GMRES_SEL = 1e-11   # selective reorthogonalisation skips second passes (||I - V^T V|| ~ 1e-12 instead of 1e-15), so
                        # how far it sits from the always-twice reference depends on which passes it skips: observed 2.3e-14
BAR_HH = 1e-10          # Householder GMRES against the (multi-threaded) oracle: observed <= 8.8e-12


# ---------------------------------------------------------------------------------------------------------------
# references
# ---------------------------------------------------------------------------------------------------------------
def _defect(nx, ny):
    """(line, first column, end column) of one interior CTA-sized patch whose upper halo line a defective operator
    drops: 240 columns (the chain kernel's strip for L <= 2) on a line in the middle of the grid"""
    c0 = (nx // 2) // 240 * 240
    return ny // 2, c0, min(c0 + 240, nx)


def np_op(nx, ny, ex=1.0, ey=1.0, poisson=True, defect=None):
    """numpy restatement of the 5-point operators (idx = i + j*nx, zero Dirichlet) in any float dtype"""
    def A(x):
        X = x.reshape(ny, nx)
        Pd = np.pad(X, 1)
        l, r, dn, up = Pd[1:-1, :-2], Pd[1:-1, 2:], Pd[2:, 1:-1], Pd[:-2, 1:-1]
        if poisson:
            y = 4 * X - (((l + r) + dn) + up)
        else:
            y = 2 * (ex + ey) * X - (ex * (l + r) + ey * (dn + up))
        if defect:
            j, c0, c1 = defect
            y[j, c0:c1] += (1.0 if poisson else ey) * up[j, c0:c1]
        return y.reshape(-1)
    return A


def t_op(torch, nx, ny, ex=1.0, ey=1.0, poisson=True, defect=None):
    """the same on torch tensors (t_apply of test_gpu_large.py, bit-exact for the Poisson operator)"""
    def A(x):
        y = t_apply(torch, x, nx, ny, ex, ey, poisson)
        if defect:
            j, c0, c1 = defect
            y.view(ny, nx)[j, c0:c1] += (1.0 if poisson else ey) * x.view(ny, nx)[j - 1, c0:c1]
        return y
    return A


def cbpr2_ref(A, params=P):
    return lambda r: t_cbpr2(None, A, r, params)


def cheb_ref(A, k, params=P):
    """oracle/krylov_extras.c ko_cheb (Saad, Alg. 12.1), params in either order"""
    ea, eb = params
    theta, delta = (eb + ea) / 2.0, abs(eb - ea) / 2.0
    sigma = theta / delta

    def M(r):
        rho_prev = 1.0 / sigma
        d = r / theta
        z = d
        for _ in range(k):
            rho = 1.0 / (2.0 * sigma - rho_prev)
            d = (rho * rho_prev) * d + (2.0 * rho / delta) * (r - A(z))
            z = z + d
            rho_prev = rho
        return z
    return M


class NpOps:
    """vector operations of the reference recurrences on numpy arrays (pairwise sums in the array's dtype)"""
    @staticmethod
    def dot(a, b):
        return (a * b).sum()

    @staticmethod
    def zeros2(rows, like):
        return np.zeros((rows, like.size), dtype=like.dtype)

    @staticmethod
    def host(v):
        return np.asarray(v)

    @staticmethod
    def dev(v, like):
        return np.asarray(v, dtype=like.dtype)


class TorchOps:
    @staticmethod
    def dot(a, b):
        import torch
        return torch.dot(a, b)

    @staticmethod
    def zeros2(rows, like):
        return like.new_zeros((rows, like.numel()))

    @staticmethod
    def host(v):
        return v.cpu().numpy()

    @staticmethod
    def dev(v, like):
        import torch
        return torch.from_numpy(np.ascontiguousarray(v, dtype=np.float64)).to(like.device)


def ref_cg(ops, A, b, iters, M=None):
    """cg.f90:83-152 (M None) / :154-231 (pcg): residual history ||r_k|| and x"""
    x = b * 0.0
    r = b * 1.0
    z = M(r) if M else r
    p = z * 1.0
    rz = ops.dot(r, z)
    hist = []
    for _ in range(iters):
        ap = A(p)
        alpha = rz / ops.dot(ap, p)
        x += alpha * p
        r = r - alpha * ap
        hist.append(float(ops.dot(r, r) ** 0.5))
        z = M(r) if M else r
        rz_new = ops.dot(r, z)
        p = z + (rz_new / rz) * p
        rz = rz_new
    return np.array(hist), x


def ref_bicgstab(ops, A, b, iters, M):
    """bicgstab.f90:91-182"""
    x = b * 0.0
    r, r0, p = b * 1.0, b * 1.0, b * 1.0
    hist = []
    for _ in range(iters):
        z1 = M(p)
        ap = A(z1)
        rr0 = ops.dot(r, r0)
        alpha = rr0 / ops.dot(ap, r0)
        s = r - alpha * ap
        z2 = M(s)
        as_ = A(z2)
        omega = ops.dot(as_, s) / ops.dot(as_, as_)
        x += alpha * z1
        x += omega * z2
        r = s - omega * as_
        hist.append(float(ops.dot(r, r) ** 0.5))
        p = r + ((ops.dot(r, r0) / rr0) * (alpha / omega)) * (p - omega * ap)
    return np.array(hist), x


def ref_gmres_cycle(ops, A, b, m, M):
    """one restart cycle of gmres_mgsr.f90:277-391 with the left preconditioner M, orthogonalised twice (classical
    Gram-Schmidt twice; equal to MGS twice in exact arithmetic).  Returns final_err (|g_{j+1}| / ||b||) and x."""
    beta0 = float(ops.dot(b, b) ** 0.5)
    w = M(b)
    beta = ops.dot(w, w) ** 0.5
    V = ops.zeros2(m + 1, b)
    V[0] = w / beta
    hv0 = ops.host(beta)
    ft = np.longdouble if hv0.dtype == np.longdouble else np.float64
    H = np.zeros((m + 1, m), dtype=ft)
    g = np.zeros(m + 1, dtype=ft)
    g[0] = ft(hv0)
    cs, sn = np.zeros(m, dtype=ft), np.zeros(m, dtype=ft)
    fe = []
    for j in range(m):
        w = M(A(V[j]))
        for _ in range(2):
            hc = V[: j + 1] @ w
            w = w - hc @ V[: j + 1]
            H[: j + 1, j] += ops.host(hc).astype(ft)
        hn = ops.dot(w, w) ** 0.5
        H[j + 1, j] = ft(ops.host(hn))
        for i in range(j):
            t = H[i, j]
            H[i, j] = cs[i] * t + sn[i] * H[i + 1, j]
            H[i + 1, j] = -sn[i] * t + cs[i] * H[i + 1, j]
        ds = np.hypot(H[j + 1, j], H[j, j])
        cs[j], sn[j] = H[j, j] / ds, H[j + 1, j] / ds
        H[j, j] = cs[j] * H[j, j] + sn[j] * H[j + 1, j]
        H[j + 1, j] = 0
        t = g[j]
        g[j], g[j + 1] = cs[j] * t + sn[j] * g[j + 1], -sn[j] * t + cs[j] * g[j + 1]
        fe.append(float(abs(g[j + 1])) / beta0)
        V[j + 1] = w / hn
    y = np.zeros(m, dtype=ft)
    for i in range(m - 1, -1, -1):
        y[i] = (g[i] - H[i, i + 1:m] @ y[i + 1:]) / H[i, i]
    return np.array(fe), ops.dev(y, b) @ V[:m]


def ld_ok():
    return np.finfo(np.longdouble).nmant > np.finfo(np.float64).nmant


needs_ld = pytest.mark.skipif(not ld_ok(), reason="np.longdouble is no wider than float64 on this platform")


def ld(v):
    """a float64 vector (numpy or torch) as np.longdouble"""
    v = v.cpu().numpy() if hasattr(v, "cpu") else np.asarray(v)
    return v.astype(np.longdouble)


def xrel(x, xr):
    """max |x - xr| / max |xr| in float64 (x, xr numpy or torch, any dtype)"""
    if hasattr(x, "cpu") and hasattr(xr, "cpu"):
        return float((x - xr).abs().max() / xr.abs().max())
    x, xr = np.asarray(x.cpu() if hasattr(x, "cpu") else x), np.asarray(xr.cpu() if hasattr(xr, "cpu") else xr)
    return float(np.abs(x.astype(np.longdouble) - xr).max() / np.abs(xr).max())


def hrel(a, b):
    a, b = np.asarray(a, dtype=np.float64), np.asarray(b, dtype=np.float64)
    assert a.size == b.size
    return float(np.abs(a / b - 1).max())


# ---------------------------------------------------------------------------------------------------------------
# CPU: both references against the oracle (64^2, random b)
# ---------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("kind", ["torch", "longdouble"])
def test_references_match_oracle(ko, kind):
    if kind == "longdouble" and not ld_ok():
        pytest.skip("np.longdouble is no wider than float64 on this platform")
    ns, n = 64, 64 * 64
    b = np.random.default_rng(64).standard_normal(n)
    if kind == "torch":
        import torch
        ops, bv = TorchOps, torch.from_numpy(b.copy())
        A, Ad = t_op(torch, ns, ns), t_op(torch, ns, ns, defect=_defect(ns, ns))
        Aa = t_op(torch, ns, ns, 1.0, 0.01, poisson=False)
    else:
        ops, bv = NpOps, b.astype(np.longdouble)
        A, Ad = np_op(ns, ns), np_op(ns, ns, defect=_defect(ns, ns))
        Aa = np_op(ns, ns, 1.0, 0.01, poisson=False)
    out = {}
    o = ko.cg_omp(ko.stvec_fn(), b, 0.0, 60)
    out["cg"] = (ref_cg(ops, A, bv, 60), o)
    o = ko.pcg_omp(ko.stvec_fn(), b, 0.0, 30, ko.cbpr2_fn(), P)
    out["pcg cbpr2"] = (ref_cg(ops, A, bv, 30, cbpr2_ref(A)), o)
    o = ko.pcg_omp(ko.stvec_fn(), b, 0.0, 20, ko.cheb_fn(4), P)
    out["pcg cheb4"] = (ref_cg(ops, A, bv, 20, cheb_ref(A, 4)), o)
    o = ko.pbicgstab_omp(ko.aniso_fn(1.0, 0.01), b, 0.0, 12, ko.cbpr2_fn(), P)
    out["bicgstab aniso"] = (ref_bicgstab(ops, Aa, bv, 12, cbpr2_ref(Aa)), o)
    o = ko.gmres_mgsr_omp(ko.stvec_fn(), b, 40, 0.0, ko.cbpr2_fn(), P, max_restarts=1, skip_verr=True)
    out["gmres cbpr2"] = (ref_gmres_cycle(ops, A, bv, 40, cbpr2_ref(A)), o)
    for name, ((hist, x), o) in out.items():
        d, dx = hrel(hist, o.history), xrel(x, o.x)
        print(f"{kind} reference vs oracle, {name} at 64^2: history {d:.2e}, x {dx:.2e}")
        assert d < 1e-12 and dx < 1e-12, name
    # and the defect is visible
    hist, _ = ref_cg(ops, Ad, bv, 60)
    assert hrel(hist, out["cg"][1].history) > 1e-6


# ---------------------------------------------------------------------------------------------------------------
# GPU fixtures
# ---------------------------------------------------------------------------------------------------------------
@pytest.fixture(scope="module")
def env():
    import torch
    import gmres_b200 as kl
    h = kl.Handle(0)
    h.set_option(VERR, 0)
    yield kl, h, torch
    h.close()
    torch.cuda.empty_cache()


@contextlib.contextmanager
def opts(h, **kv):
    """set options by name (module constants) and restore them afterwards"""
    keys = {globals()[k]: v for k, v in kv.items()}
    old = {k: h.get_option(k) for k in keys}
    try:
        for k, v in keys.items():
            h.set_option(k, v)
        yield
    finally:
        for k, v in old.items():
            h.set_option(k, v)


def randn(torch, n, seed):
    g = torch.Generator(device="cuda")
    g.manual_seed(seed)
    return torch.randn(n, generator=g, dtype=torch.float64, device="cuda")


@contextlib.contextmanager
def oracle_threads(ko):
    ko.set_threads(ko.max_threads())
    try:
        yield
    finally:
        ko.set_threads(1)


def _free(torch):
    import gc
    gc.collect()
    torch.cuda.empty_cache()


# ---------------------------------------------------------------------------------------------------------------
# point-wise kernels, bit-exact
# ---------------------------------------------------------------------------------------------------------------
@gpu
@pytest.mark.parametrize("n", [16384, 8192])
def test_operators_bench_size_vs_oracle(env, ko, n):
    kl, h, torch = env
    x = randn(torch, n * n, n)
    xh = x.cpu().numpy()
    with oracle_threads(ko):
        for op, fo in ((kl.stvec, ko.stvec_fn()), (kl.stv_poisson, ko.stv_poisson_fn()),
                       (kl.aniso(1.0, 0.01), ko.aniso_fn(1.0, 0.01))):
            y = h.apply(op, x, n, n).cpu().numpy()
            yo = ko.apply(fo, xh, n, parallel=True)
            assert np.array_equal(y, yo), (n, op.kind, np.abs(y - yo).max())
            del y, yo
        if n == 16384:
            z = h.apply_precond(kl.cbpr2, kl.stvec, x, P, n, n).cpu().numpy()
            zo = ko.apply_precond(ko.cbpr2_fn(), ko.stvec_fn(), xh, P, n, parallel=True)
            assert np.array_equal(z, zo), np.abs(z - zo).max()
            del z, zo
        else:
            for k in (1, 2, 3, 4, 5, 6, 8, 13):     # one chain, continuation chunks, the LEAN interior march
                z = h.apply_precond(kl.cheb(k), kl.stvec, x, P, n, n).cpu().numpy()
                zo = ko.apply_precond(ko.cheb_fn(k), ko.stvec_fn(), xh, P, n, parallel=True)
                assert np.array_equal(z, zo), (k, np.abs(z - zo).max())
                del z, zo
    del x, xh
    _free(torch)


@gpu
@pytest.mark.parametrize("what", ["stvec", "cbpr2", "cheb4"])
def test_geometry_option_sweep_8192(env, ko, what):
    """Every combination of the stencil kernels' geometry options gives the oracle's bits.  Rows = 8 makes
    33 x 1024 tiles, more than the reduction buffer's 16384 slots: the TMA kernel loops over several tiles per CTA
    and the register-pipelined one (TMA = 0) takes stencil_geometry's fallback."""
    kl, h, torch = env
    n = 8192
    x = randn(torch, n * n, 3)
    xh = x.cpu().numpy()
    with oracle_threads(ko):
        if what == "stvec":
            ref = ko.apply(ko.stvec_fn(), xh, n, parallel=True)
            run = lambda: h.apply(kl.stvec, x, n, n)
        else:
            M, Mo = (kl.cbpr2, ko.cbpr2_fn()) if what == "cbpr2" else (kl.cheb(4), ko.cheb_fn(4))
            ref = ko.apply_precond(Mo, ko.stvec_fn(), xh, P, n, parallel=True)
            run = lambda: h.apply_precond(M, kl.stvec, x, P, n, n)
    ref = torch.from_numpy(ref).cuda()
    bad = []
    for tma in (1, 0):
        for pers in (0, 1):
            for stag in (0, 1):
                for tail in (-1, 0, 3, 7):
                    for rows in (0, 8, 13, 61, 128):
                        with opts(h, TMA=tma, PERSISTENT=pers, STAGGER=stag, TAIL=tail, ROWS=rows):
                            y = run()
                        if not torch.equal(y, ref):
                            bad.append((tma, pers, stag, tail, rows, float((y - ref).abs().max())))
    assert not bad, bad
    del x, xh, ref
    _free(torch)


EDGE_NX = [63, 64, 65, 66, 226, 240, 242, 254, 256, 257, 542, 4112]
EDGE_NY = [1, 2, 3, 5, 25, 49, 301]


def _t_stv_poisson(torch, x, nx, ny):
    """poisson.f90:79-96 in its own order: (((4x - x_{i-1}) - x_{i+1}) - x_{j-1}) - x_{j+1}, missing neighbours 0"""
    X = x.view(ny, nx)
    Pd = torch.nn.functional.pad(X, (1, 1, 1, 1))
    return ((((4.0 * X - Pd[1:-1, :-2]) - Pd[1:-1, 2:]) - Pd[:-2, 1:-1]) - Pd[2:, 1:-1]).reshape(-1)


@gpu
@pytest.mark.parametrize("nx", EDGE_NX)
def test_edge_shapes_pointwise(env, nx):
    """Shapes around the strip widths (kTmaStrip = 252; chain STRIP 240 / 224 / 208; the 64-column warp window),
    odd nx (scalar path) and short grids.  The operators against the torch restatement (any grid); cbpr2, cheb(k)
    and the anisotropic operator, whose fmas torch cannot restate, chained / TMA against the one-kernel-per-
    application, register-pipelined path.  A shape the library rejects must raise, not return wrong numbers."""
    kl, h, torch = env
    rejected = []
    for ny in EDGE_NY:
        x = randn(torch, nx * ny, nx * 1000 + ny)
        try:
            y = h.apply(kl.stvec, x, nx, ny)
        except kl.api.KrylovError as e:
            rejected.append((ny, str(e)))
            continue
        assert torch.equal(y, t_apply(torch, x, nx, ny)), (nx, ny)
        assert torch.equal(h.apply(kl.stv_poisson, x, nx, ny), _t_stv_poisson(torch, x, nx, ny)), (nx, ny)
        ya = h.apply(kl.aniso(1.0, 0.01), x, nx, ny)
        with opts(h, TMA=0):
            assert torch.equal(ya, h.apply(kl.aniso(1.0, 0.01), x, nx, ny)), (nx, ny)
        for M in [kl.cbpr2] + [kl.cheb(k) for k in (1, 2, 3, 4, 5, 6, 8, 13)]:
            for op in (kl.stvec, kl.aniso(1.0, 0.01)):
                z = h.apply_precond(M, op, x, P, nx, ny)
                with opts(h, CHAIN=0, TMA=0):
                    zs = h.apply_precond(M, op, x, P, nx, ny)
                assert torch.equal(z, zs), (nx, ny, M, op.kind, float((z - zs).abs().max()))
    print(f"nx {nx}: rejected {rejected}")
    assert all(ny < 25 for ny, _ in rejected), rejected


@gpu
@pytest.mark.parametrize("ns", [63, 64, 65, 66, 226, 240, 242, 254, 256, 257, 542])
def test_edge_shapes_square_vs_oracle(env, ko, ns):
    kl, h, torch = env
    x = randn(torch, ns * ns, ns)
    xh = x.cpu().numpy()
    for op, fo in ((kl.stvec, ko.stvec_fn()), (kl.stv_poisson, ko.stv_poisson_fn()),
                   (kl.aniso(1.0, 0.01), ko.aniso_fn(1.0, 0.01))):
        assert np.array_equal(h.apply(op, x, ns, ns).cpu().numpy(), ko.apply(fo, xh, ns)), (ns, op.kind)
    for M, Mo in [(kl.cbpr2, ko.cbpr2_fn())] + [(kl.cheb(k), None) for k in (1, 2, 3, 4, 5, 6, 8, 13)]:
        Mo = Mo or ko.cheb_fn(M.degree)
        z = h.apply_precond(M, kl.stvec, x, P, ns, ns).cpu().numpy()
        assert np.array_equal(z, ko.apply_precond(Mo, ko.stvec_fn(), xh, P, ns)), (ns, M)


# ---------------------------------------------------------------------------------------------------------------
# reductions against an extended-precision sum
# ---------------------------------------------------------------------------------------------------------------
def _ld_first_residual(b, ab, chunk=1 << 24):
    """||b - alpha0 A b||, alpha0 = b.b / b.Ab, with every sum in np.longdouble (host, chunked)"""
    bb = bab = np.longdouble(0)
    for s in range(0, b.numel(), chunk):
        bc, ac = ld(b[s:s + chunk]), ld(ab[s:s + chunk])
        bb += (bc * bc).sum()
        bab += (bc * ac).sum()
    alpha = bb / bab
    rr = np.longdouble(0)
    for s in range(0, b.numel(), chunk):
        rc = ld(b[s:s + chunk]) - alpha * ld(ab[s:s + chunk])
        rr += (rc * rc).sum()
    return float(np.sqrt(rr))


@gpu
@needs_ld
@pytest.mark.parametrize("nx,ny", [(16384, 16384), (8192, 8192), (4112, 301), (542, 49), (256, 25), (66, 5),
                                   (240, 1000), (257, 49), (4096, 4096)])
def test_cg_reductions_vs_longdouble(env, nx, ny):
    """history[0] = ||b - alpha0 A b|| through one reduction of each CG mode; at 16384^2 one lost or duplicated CTA
    partial (of 16 215) moves r.r by ~6e-5.  history[1] goes through the predicted beta and the pass's four fused
    sums; it is compared with the FP64 torch reference of two iterations."""
    kl, h, torch = env
    b = randn(torch, nx * ny, 7 * nx + ny)
    want0 = _ld_first_residual(b, t_apply(torch, b, nx, ny))
    want = ref_cg(TorchOps, t_op(torch, nx, ny), b, 2)[0]
    for mode in (0, 1, 2):
        with opts(h, CG_ONEPASS=mode):
            g1 = h.cg_omp(kl.stvec, b, 0.0, 1, nx=nx, ny=ny)
            g2 = h.cg_omp(kl.stvec, b, 0.0, 2, nx=nx, ny=ny)
        d0, d1 = abs(g1.history[0] / want0 - 1), abs(g2.history[1] / want[1] - 1)
        print(f"cg reductions {nx}x{ny} mode {mode}: history[0] {d0:.2e} (bar {BAR_RED1:.0e}), "
              f"history[1] {d1:.2e} (bar {BAR_RED2:.0e})")
        assert g1.history.size == 1 and g2.history.size == 2 and g2.history[0] == g1.history[0]
        assert d0 < BAR_RED1 and d1 < BAR_RED2, (mode, d0, d1)
    del b
    _free(torch)


# ---------------------------------------------------------------------------------------------------------------
# the FP64 torch reference calibrated against the longdouble one; solvers against longdouble at 1024^2 / 512^2
# ---------------------------------------------------------------------------------------------------------------
@gpu
@needs_ld
def test_cg_1024_three_modes_vs_longdouble(env):
    """CG at 1024^2 (the largest size for the longdouble reference): the kernels in all three modes and the FP64
    torch reference against np.longdouble.  The torch reference's own deviation is what bounds the bars used at the
    bench sizes, so it must sit well below them."""
    kl, h, torch = env
    n, its = 1024, 40
    b = randn(torch, n * n, 1024)
    hl, xl = ref_cg(NpOps, np_op(n, n), ld(b), its)
    ht, xt = ref_cg(TorchOps, t_op(torch, n, n), b, its)
    dt, dxt = hrel(ht, hl), xrel(xt.cpu().numpy(), xl)
    print(f"cg 1024^2 FP64 torch reference vs longdouble: history {dt:.2e}, x {dxt:.2e}")
    assert dt < BAR_CG / 10 and dxt < BAR_CG / 10
    for mode in (0, 1, 2):
        for ce in (8, 5):
            with opts(h, CG_ONEPASS=mode, CHECK_EVERY=ce):
                g = h.cg_omp(kl.stvec, b, 0.0, its, nx=n, ny=n)
            d, dx = hrel(g.history, hl), xrel(g.x.cpu().numpy(), xl)
            print(f"cg 1024^2 mode {mode} check_every {ce} vs longdouble: history {d:.2e}, x {dx:.2e}")
            assert d < BAR_CG and dx < BAR_CG, (mode, ce, d, dx)


@gpu
@needs_ld
def test_solvers_small_vs_longdouble(env):
    """PCG (cbpr2, cheb(4)), BiCGSTAB and one GMRES-MGSR cycle against np.longdouble, and the FP64 torch
    reference's own deviation from it (which bounds the bars of the bench-size tests)."""
    kl, h, torch = env
    n = 1024
    b = randn(torch, n * n, 11)
    A, At = np_op(n, n), t_op(torch, n, n)
    Aa, Aat = np_op(n, n, 1.0, 0.01, poisson=False), t_op(torch, n, n, 1.0, 0.01, poisson=False)
    cases = [
        ("pcg cbpr2", BAR_CG, lambda: h.pcg_omp(kl.stvec, b, 0.0, 20, kl.cbpr2, P, nx=n, ny=n),
         lambda o, A_, b_: ref_cg(o, A_, b_, 20, cbpr2_ref(A_)), A, At),
        ("pcg cheb4", BAR_CG, lambda: h.pcg_omp(kl.stvec, b, 0.0, 12, kl.cheb(4), P, nx=n, ny=n),
         lambda o, A_, b_: ref_cg(o, A_, b_, 12, cheb_ref(A_, 4)), A, At),
        ("bicgstab aniso cbpr2", BAR_BICG, lambda: h.pbicgstab_omp(kl.aniso(1.0, 0.01), b, 0.0, 12, kl.cbpr2, P, nx=n, ny=n),
         lambda o, A_, b_: ref_bicgstab(o, A_, b_, 12, cbpr2_ref(A_)), Aa, Aat),
    ]
    with opts(h, CHECK_EVERY=32):
        for name, bar, gpu_run, ref, An, Atn in cases:
            hl, xl = ref(NpOps, An, ld(b))
            ht, xt = ref(TorchOps, Atn, b)
            g = gpu_run()
            dt, dxt = hrel(ht, hl), xrel(xt.cpu().numpy(), xl)
            d, dx = hrel(g.history, hl), xrel(g.x.cpu().numpy(), xl)
            print(f"{name} 1024^2 vs longdouble: kernels history {d:.2e} x {dx:.2e}; torch reference {dt:.2e} {dxt:.2e}")
            assert dt < bar / 10 and dxt < bar / 10, name
            assert d < bar and dx < bar, name
    # GMRES: 256^2 (the longdouble Gram-Schmidt is the slow part)
    n, m = 256, 95
    b = randn(torch, n * n, 12)
    A, At = np_op(n, n), t_op(torch, n, n)
    fl, xl = ref_gmres_cycle(NpOps, A, ld(b), m, cbpr2_ref(A))
    ft, xt = ref_gmres_cycle(TorchOps, At, b, m, cbpr2_ref(At))
    with opts(h, MAX_RESTARTS=1):
        g = h.gmres_mgsr_omp(kl.stvec, b, m, 0.0, kl.cbpr2, P, nx=n, ny=n)
    d, dx, dt, dxt = hrel(g.history, fl), xrel(g.x.cpu().numpy(), xl), hrel(ft, fl), xrel(xt.cpu().numpy(), xl)
    print(f"gmres cbpr2 256^2 m 95 vs longdouble: kernels history {d:.2e} x {dx:.2e}; torch reference {dt:.2e} {dxt:.2e}")
    assert g.n_out == m and dt < BAR_GMRES / 10 and dxt < BAR_GMRES / 10
    assert d < BAR_GMRES and dx < BAR_GMRES
    _free(torch)


# ---------------------------------------------------------------------------------------------------------------
# every bench workload with random b at its bench size, against the FP64 torch reference
# ---------------------------------------------------------------------------------------------------------------
@gpu
@pytest.mark.parametrize("n", [16384, 4096])
def test_cg_bench_size_all_modes(env, n):
    """cg16384 (and 4096^2, exactly the 2^24-unknown pair threshold): pairs (auto), one pass and two kernels, with
    graph capture and replay (24 iterations, polls every 8) and with batches that start on a pass B and a run that
    ends with the x flush (25 iterations, polls every 5)."""
    kl, h, torch = env
    b = randn(torch, n * n, 16384 + n)
    A = t_op(torch, n, n)
    refs = {its: ref_cg(TorchOps, A, b, its) for its in (24, 25)}
    worst = 0.0
    for mode in (-1, 1, 0):
        for its, ce in ((24, 8), (25, 5)):
            with opts(h, CG_ONEPASS=mode, CHECK_EVERY=ce):
                g = h.cg_omp(kl.stvec, b, 0.0, its, nx=n, ny=n)
            hr, xr = refs[its]
            d, dx = hrel(g.history, hr), xrel(g.x, xr)
            worst = max(worst, d, dx)
            print(f"cg {n}^2 mode {mode} its {its} check_every {ce}: history {d:.2e}, x {dx:.2e} (bar {BAR_CG:.0e})")
            assert g.iter == its and d < BAR_CG and dx < BAR_CG, (mode, its, d, dx)
            del g
    if n == 16384:
        hd, xd = ref_cg(TorchOps, t_op(torch, n, n, defect=_defect(n, n)), b, 24)
        sh, sx = hrel(hd, refs[24][0]), xrel(xd, refs[24][1])
        print(f"cg 16384^2 one-CTA defect: history {sh:.2e}, x {sx:.2e}: {min(sh, sx) / BAR_CG:.1e} x the bar")
        assert min(sh, sx) > 100 * BAR_CG
        del hd, xd
    del b, refs
    _free(torch)


@gpu
@pytest.mark.parametrize("case", ["pcg16384", "pcg8192cheb4", "bicgstab8192"])
def test_pcg_bicgstab_bench_size(env, case):
    kl, h, torch = env
    n = 16384 if case == "pcg16384" else 8192
    b = randn(torch, n * n, {"pcg16384": 1, "pcg8192cheb4": 2, "bicgstab8192": 3}[case])
    if case == "bicgstab8192":
        A = t_op(torch, n, n, 1.0, 0.01, poisson=False)
        hr, xr = ref_bicgstab(TorchOps, A, b, 12, cbpr2_ref(A))
        run = lambda: h.pbicgstab_omp(kl.aniso(1.0, 0.01), b, 0.0, 12, kl.cbpr2, P, nx=n, ny=n)
        bar = BAR_BICG
    else:
        A = t_op(torch, n, n)
        M, Mr, its = (kl.cbpr2, cbpr2_ref(A), 20) if case == "pcg16384" else (kl.cheb(4), cheb_ref(A, 4), 12)
        hr, xr = ref_cg(TorchOps, A, b, its, Mr)
        run = lambda: h.pcg_omp(kl.stvec, b, 0.0, its, M, P, nx=n, ny=n)
        bar = BAR_CG
    with opts(h, CHECK_EVERY=8):
        g = run()
    d, dx = hrel(g.history, hr), xrel(g.x, xr)
    print(f"{case}: history {d:.2e}, x {dx:.2e} (bar {bar:.0e})")
    assert d < bar and dx < bar
    del b, g, xr
    _free(torch)


@gpu
@pytest.mark.parametrize("case", ["gmres4096", "gmres4096sel", "gmres4096cheb4"])
def test_gmres_bench_size_one_cycle(env, case):
    kl, h, torch = env
    n, m = 4096, 95
    b = randn(torch, n * n, 4096 + len(case))
    A = t_op(torch, n, n)
    M, Mr = (kl.cheb(4), cheb_ref(A, 4)) if case.endswith("cheb4") else (kl.cbpr2, cbpr2_ref(A))
    fr, xr = ref_gmres_cycle(TorchOps, A, b, m, Mr)
    sel = case == "gmres4096sel"
    with opts(h, MAX_RESTARTS=1, REORTH_ETA=300):
        h.set_ortho(2 if sel else 1)
        try:
            g = h.gmres_mgsr_omp(kl.stvec, b, m, 0.0, M, P, nx=n, ny=n)
        finally:
            h.set_ortho(1)
    bar = BAR_GMRES_SEL if sel else BAR_GMRES
    d, dx = hrel(g.history, fr), xrel(g.x, xr)
    print(f"{case}: history {d:.2e}, x {dx:.2e} (bar {bar:.0e})")
    assert g.n_out == m and d < bar and dx < bar
    if case == "gmres4096":
        fd, xd = ref_gmres_cycle(TorchOps, t_op(torch, n, n, defect=_defect(n, n)), b, m, cbpr2_ref(
            t_op(torch, n, n, defect=_defect(n, n))))
        sh, sx = hrel(fd, fr), xrel(xd, xr)
        print(f"gmres4096 one-CTA defect: history {sh:.2e}, x {sx:.2e}: {min(sh, sx) / bar:.1e} x the bar")
        assert min(sh, sx) > 100 * bar
        del xd
    del b, g, xr
    _free(torch)


@gpu
def test_hh1024_vs_oracle(env, ko):
    kl, h, torch = env
    ns, m = 1024, 95
    b = np.random.default_rng(1024).standard_normal(ns * ns)
    with oracle_threads(ko):
        o = ko.gmres_hh(ko.stvec_fn(), b, m, 0.0, None, max_stages=1, skip_verr=True)
    with opts(h, MAX_RESTARTS=1):
        for mode in (1, 0):
            with opts(h, HH_MODE=mode):
                g = h.gmres_hh_omp(kl.stvec, b, m, 0.0)
            d, dx = hist_rel(g.history, o.history), xrel(g.x, o.x)
            print(f"hh1024 mode {mode}: history {d:.2e}, x {dx:.2e} (bar {BAR_HH:.0e})")
            assert (g.n_out, g.restart_out) == (m, 1) and d < BAR_HH and dx < BAR_HH


# ---------------------------------------------------------------------------------------------------------------
# options take effect on a warm handle
# ---------------------------------------------------------------------------------------------------------------
WARM = [("TMA", 0), ("PERSISTENT", 1), ("STAGGER", 1), ("TAIL", 3), ("ROWS", 13), ("PDL", 0), ("REVERSE", 1)]


def _solve(kl, h, solver, b, n):
    if solver == "cg":          # two-kernel path (REVERSE applies to its second kernel), batches replayed as graphs
        with opts(h, CG_ONEPASS=0, CHECK_EVERY=16):
            return h.cg_omp(kl.stvec, b, 0.0, 64, nx=n, ny=n)
    if solver == "gmres":
        with opts(h, MAX_RESTARTS=3):
            return h.gmres_mgsr_omp(kl.stvec, b, 30, 0.0, kl.cbpr2, P, nx=n, ny=n)
    with opts(h, MAX_RESTARTS=3):
        return h.gmres_hh_omp(kl.stvec, b, 20, 0.0, nx=n, ny=n)


@gpu
@pytest.mark.parametrize("solver,n", [("cg", 2048), ("gmres", 2048), ("hh", 512)])
@pytest.mark.parametrize("opt,value", WARM)
def test_option_takes_effect_on_warm_handle(env, solver, n, opt, value):
    """Solve with the defaults, set the option, solve again on the same handle: bit-identical to a fresh handle
    that had the option before its first solve (a CUDA graph captured under the old setting must not be replayed).
    2048^2: enough tiles that PERSISTENT changes the CTA grid and with it the partition of the partial sums."""
    kl, h0, torch = env
    b = randn(torch, n * n, n + 5)
    warm, fresh = kl.Handle(0), kl.Handle(0)
    try:
        for hd in (warm, fresh):
            hd.set_option(VERR, 0)
        d0 = _solve(kl, warm, solver, b, n)
        _solve(kl, warm, solver, b, n)
        warm.set_option(globals()[opt], value)
        w = _solve(kl, warm, solver, b, n)
        fresh.set_option(globals()[opt], value)
        f = _solve(kl, fresh, solver, b, n)
        f2 = _solve(kl, fresh, solver, b, n)
    finally:
        warm.close()
        fresh.close()
    same = lambda a, c: np.array_equal(a.history, c.history) and torch.equal(a.x, c.x)
    print(f"{solver} {n}^2 {opt}={value}: result differs from the default's: {not same(f, d0)}")
    assert same(f, f2)
    assert same(w, f), (opt, hrel(w.history, f.history))
