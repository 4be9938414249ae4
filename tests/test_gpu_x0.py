"""KL_OPT_X0: every solver entry started from a caller-supplied initial guess x0 (the `x0=` argument of the Python
mirror).

  1. x0 = 0 with the option on is bit-identical to the option off (x, history, counts, status) in every mode;
  2. CG, PCG and BiCGSTAB from a random x0 run exactly the recurrence of a cold solve of b' = b - A x0 (the
     recurrences never read x): identical histories and counts, and x_warm = x0 + x_cold up to rounding;
  3. a GMRES solve split in two (c1 cycles, then c2 more from the returned x) equals the uninterrupted solve bit for bit;
  4. x0 that already meets the stopping test returns at once: KL_OK, zero iterations, x = x0 bit for bit;
  5. maxit = 0 returns x0 unchanged;
  6. warm-started solves on a handle with cached CUDA graphs equal a fresh handle's;
  7. the Python mirror's and the C ABI's edges.

Right-hand sides and initial guesses are seeded normal vectors generated on the device (support on the whole grid).
"""
import contextlib
import ctypes as C

import numpy as np
import pytest

from test_oracle import _dense_poisson

pytestmark = pytest.mark.gpu
P = (8.2, 0.2)          # tests/test_poisson_mf.f90:38

# include/krylov_b200.h
ORTHO, MAX_RESTARTS, VERR, CHECK_EVERY, HH_MODE, FUSE, CG_ONEPASS, X0 = 1, 2, 3, 4, 6, 7, 22, 23
OPTS = dict(ORTHO=ORTHO, MAX_RESTARTS=MAX_RESTARTS, VERR=VERR, CHECK_EVERY=CHECK_EVERY, HH_MODE=HH_MODE, FUSE=FUSE,
            CG_ONEPASS=CG_ONEPASS)
KL_OK, KL_NOT_CONVERGED, KL_ERR_INVALID = 0, 1, -1

# x_warm - (x0 + x_cold), relative to max |x_warm|: the two differ only in where x0 enters the sum of the alpha*p
# updates.  Bar: >= 10x the largest value observed on a B200 (1000 W power limit): 7.2e-16 over every case of
# test_warm_equals_cold_of_shifted_rhs.
BAR_SHIFT = 1e-14


@pytest.fixture(scope="module")
def env():
    import torch
    import gmres_b200 as kl
    h = kl.Handle(0)
    aux = kl.Handle(0)          # applies the 5-point operator for the KL_OP_USER callback
    yield kl, h, aux, torch
    h.close()
    aux.close()
    torch.cuda.empty_cache()


@contextlib.contextmanager
def opts(h, **kv):
    keys = {OPTS[k]: v for k, v in kv.items()}
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


def user_stvec(kl, aux):
    """stvec as a KL_OP_USER callback: the second handle applies the built-in operator on the solver's stream"""
    o, _ = kl.stvec._c()

    def fn(dx, dy, nx, nyl, stream):
        L = aux._L
        assert L.kl_set_stream(aux._h, C.c_void_p(stream)) == 0
        assert L.kl_set_pointer_mode(aux._h, kl.api.KL_POINTER_DEVICE) == 0
        assert L.kl_apply_operator(aux._h, C.byref(o), C.c_void_p(dx), C.c_void_p(dy), nx, nyl) == 0
    return kl.Operator(kl.api.KL_OP_USER, fn=fn)


def solve(env, kind, b, n, x0=None, tol=0.0, its=30, **kw):
    """one solver call by name; n = grid side (stencil) or matrix order (dense: b's length is n)"""
    kl, h, aux, torch = env
    k = kind.split(":")
    if k[0] == "cg":
        with opts(h, CG_ONEPASS=int(k[1]), **kw):
            return h.cg_omp(kl.stvec, b, tol, its, nx=n, ny=n, x0=x0)
    if k[0] == "pcg":
        M = kl.cheb(4) if k[1] == "cheb4" else kl.cbpr2
        A = user_stvec(kl, aux) if k[1] == "user" else kl.stvec
        with opts(h, FUSE=0 if k[1] == "nofuse" else 1, **kw):
            return h.pcg_omp(A, b, tol, its, M, P, nx=n, ny=n, x0=x0)
    if k[0] == "bicgstab":
        with opts(h, **kw):
            if k[1] == "plain":
                return h.bicgstab(kl.stvec, b, tol, its, nx=n, ny=n, x0=x0)
            return h.pbicgstab_omp(kl.stvec, b, tol, its, kl.cbpr2, P, nx=n, ny=n, x0=x0)
    if k[0] == "gmres":             # gmres:omp|mf:ortho:none|cbpr2|cheb4
        M = {"none": None, "cbpr2": kl.cbpr2, "cheb4": kl.cheb(4)}[k[3]]
        f = h.gmres_mgsr_omp if k[1] == "omp" else h.gmres_mgsr_mf
        with opts(h, ORTHO=int(k[2]), VERR=0, **kw):
            return f(kl.stvec, b, its, tol, M, P if M else None, nx=n, ny=n, x0=x0)
    if k[0] == "hh":                # hh:omp|prec:mode
        with opts(h, HH_MODE=int(k[2]), VERR=0, **kw):
            if k[1] == "omp":
                return h.gmres_hh_omp(kl.stvec, b, its, tol, nx=n, ny=n, x0=x0)
            return h.gmres_hh_prec_omp(kl.stvec, b, its, tol, kl.cbpr2, P, nx=n, ny=n, x0=x0)
    if k[0] == "dense":             # dense:mgsr|hh on the 400-unknown Poisson matrix
        A = _dense_poisson(20)
        with opts(h, **kw):
            f = h.gmres_mgsr_dense if k[1] == "mgsr" else h.gmres_hh_dense
            return f(A, b, its, tol, x0=x0)
    raise ValueError(kind)


def xeq(torch, a, c):
    if isinstance(a, np.ndarray):
        return isinstance(c, np.ndarray) and np.array_equal(a, c)
    return torch.equal(a, c)


def same(torch, a, c):
    """bit-identical results: x, history, status and every count"""
    ok = xeq(torch, a.x, c.x) and np.array_equal(a.history, c.history) and a.status == c.status
    if hasattr(a, "iter"):
        return ok and a.iter == c.iter and np.array_equal([a.res], [c.res])
    return (ok and (a.n_out, a.restart_out) == (c.n_out, c.restart_out) and np.array_equal(a.final_err, c.final_err)
            and np.array_equal(a.v_err, c.v_err))


def is_gmres(kind):
    return kind.split(":")[0] in ("gmres", "hh", "dense")


# ---------------------------------------------------------------------------------------------------------------
# 1. x0 = 0 with the option on == option off
# ---------------------------------------------------------------------------------------------------------------
ZERO_CASES = (
    [("cg:0", 2048), ("cg:1", 2048), ("cg:2", 2048), ("cg:-1", 16384)]
    + [(f"pcg:{p}", 2048) for p in ("cbpr2", "cheb4", "nofuse", "user")]
    + [("bicgstab:plain", 2048), ("bicgstab:cbpr2", 2048)]
    + [(f"gmres:{v}:{o}:{p}", n) for n in (300, 2048) for v in ("omp", "mf") for o in (0, 1, 2)
       for p in ("none", "cbpr2", "cheb4")]
    + [(f"hh:{v}:{mode}", 1024) for v in ("omp", "prec") for mode in (0, 1)]
    + [("dense:mgsr", 20), ("dense:hh", 20)]
)


@pytest.mark.parametrize("kind,n", ZERO_CASES)
def test_zero_x0_is_cold(env, kind, n):
    kl, h, aux, torch = env
    dense = kind.startswith("dense")
    nn = n * n
    b = randn(torch, nn, 7 + n)
    if dense:
        b = b.cpu().numpy()
    x0 = np.zeros(nn) if dense else torch.zeros_like(b)
    gm = is_gmres(kind)
    kw = dict(its=20, MAX_RESTARTS=2) if gm else dict(its=24 if n == 16384 else 31, CHECK_EVERY=8)
    cold = solve(env, kind, b, n, **kw)
    warm = solve(env, kind, b, n, x0=x0, **kw)
    assert same(torch, cold, warm), kind
    assert not np.isnan(cold.history).any()


# ---------------------------------------------------------------------------------------------------------------
# 2. CG / PCG / BiCGSTAB from x0 = the cold solve of b - A x0
# ---------------------------------------------------------------------------------------------------------------
def _first_drops(hist):
    """indices k where history[k] is below every earlier entry: tol just above history[k] converges at k + 1"""
    run = np.minimum.accumulate(hist)
    return [k for k in range(1, hist.size) if hist[k] < run[k - 1]]


SHIFT_CASES = [f"cg:{m}" for m in (0, 1, 2)] + ["pcg:cbpr2", "bicgstab:plain", "bicgstab:cbpr2"]
_shift_worst = [0.0]


@pytest.mark.parametrize("kind", SHIFT_CASES)
@pytest.mark.parametrize("host", [False, True])
@pytest.mark.parametrize("ce", [16, 5])
def test_warm_equals_cold_of_shifted_rhs(env, kind, host, ce):
    """odd and even maxit without convergence, then convergence at an odd and at an even iteration; CHECK_EVERY 16
    replays graphs, 5 makes the pair mode's batches start on a second pass"""
    kl, h, aux, torch = env
    n = 1024
    b = randn(torch, n * n, 11)
    x0 = randn(torch, n * n, 12)
    bs = b - h.apply(kl.stvec, x0, n, n)
    if host:
        b, x0, bs = b.cpu().numpy(), x0.cpu().numpy(), bs.cpu().numpy()
    x0_keep = x0.copy() if host else x0.clone()
    full = solve(env, kind, bs, n, its=61, CHECK_EVERY=ce)
    drops = _first_drops(full.history)
    odd = [k for k in drops if (k + 1) % 2 == 1 and k > 8]
    even = [k for k in drops if (k + 1) % 2 == 0 and k > 8]
    assert odd and even, drops
    runs = [(0.0, 40), (0.0, 41)] + [(float(np.nextafter(full.history[k], np.inf)), 61) for k in (odd[0], even[0])]
    for tol, its in runs:
        c = solve(env, kind, bs, n, tol=tol, its=its, CHECK_EVERY=ce)
        w = solve(env, kind, b, n, x0=x0, tol=tol, its=its, CHECK_EVERY=ce)
        assert (w.status, w.iter) == (c.status, c.iter) and np.array_equal([w.res], [c.res]), (tol, its)
        assert np.array_equal(w.history, c.history), (tol, its)
        if tol > 0:
            assert w.status == KL_OK and w.iter in (odd[0] + 1, even[0] + 1)
        xw = torch.as_tensor(w.x, device="cuda")
        xs = torch.as_tensor(x0, device="cuda") + torch.as_tensor(c.x, device="cuda")
        d = float((xw - xs).abs().max() / xw.abs().max())
        _shift_worst[0] = max(_shift_worst[0], d)
        assert d < BAR_SHIFT, (tol, its, d)
    assert xeq(torch, x0, x0_keep)
    print(f"{kind} host={host} check_every={ce}: |x_warm - (x0 + x_cold)| / max|x_warm| up to {_shift_worst[0]:.2e} "
          f"(bar {BAR_SHIFT:.0e})")


# ---------------------------------------------------------------------------------------------------------------
# 3. a GMRES solve split in two == the uninterrupted solve
# ---------------------------------------------------------------------------------------------------------------
SPLIT_CASES = ([(f"gmres:omp:{o}:cbpr2", 2048, 30, 2, 2) for o in (0, 1, 2)]
               + [("gmres:mf:1:cbpr2", 2048, 30, 1, 2), ("gmres:omp:1:cbpr2", 4096, 95, 1, 1),
                  ("gmres:omp:2:cbpr2", 4096, 95, 1, 1)]
               + [(f"hh:omp:{mode}", 1024, 20, 2, 1) for mode in (0, 1)])


@pytest.mark.parametrize("kind,n,m,c1,c2", SPLIT_CASES)
def test_gmres_resume_equals_uninterrupted(env, kind, n, m, c1, c2):
    kl, h, aux, torch = env
    b = randn(torch, n * n, 3 * n + m)
    full = solve(env, kind, b, n, its=m, MAX_RESTARTS=c1 + c2)
    first = solve(env, kind, b, n, its=m, MAX_RESTARTS=c1)
    second = solve(env, kind, b, n, x0=first.x, its=m, MAX_RESTARTS=c2)
    k = second.history.size
    assert full.status == second.status == KL_NOT_CONVERGED
    assert (full.restart_out, second.restart_out, first.restart_out) == (c1 + c2, c2, c1)
    assert full.n_out == second.n_out
    assert full.history.size == first.history.size + k
    assert np.array_equal(full.history[-k:], second.history)
    assert np.array_equal(full.history[:-k], first.history)
    assert torch.equal(full.x, second.x)


# ---------------------------------------------------------------------------------------------------------------
# 4. zero-step return, 5. maxit = 0
# ---------------------------------------------------------------------------------------------------------------
ALL_KINDS = (["cg:0", "cg:1", "cg:2", "pcg:cbpr2", "pcg:cheb4", "pcg:nofuse", "pcg:user", "bicgstab:plain",
              "bicgstab:cbpr2"]
             + [f"gmres:{v}:{o}:{p}" for v in ("omp", "mf") for o in (0, 1, 2) for p in ("none", "cbpr2")]
             + ["gmres:omp:1:cheb4"] + [f"hh:{v}:{mode}" for v in ("omp", "prec") for mode in (0, 1)]
             + ["dense:mgsr", "dense:hh"])


def _check_zero_step(torch, kind, r, x0, res_pos, tol):
    assert r.status == KL_OK and r.history.size == 0, (kind, r.status, r.history.size)
    assert xeq(torch, r.x, x0), kind
    if is_gmres(kind):
        assert (r.n_out, r.restart_out) == (0, 1) and not r.final_err.any() and not r.v_err.any()
        assert (r.restart_out - 1) * 30 + r.n_out == 0       # the drivers' count (tests/test_poisson_mf.f90:78)
    else:
        assert r.iter == 0 and not np.isnan(r.res)
        assert (0.0 < r.res < tol) if res_pos else r.res == 0.0, (kind, r.res)


@pytest.mark.parametrize("kind", ALL_KINDS)
def test_zero_step_return(env, kind):
    """x0 = 1 with b = A*1 (r0 = 0 exactly), and x0 = 1 + 1e-9 noise (0 < ||r0|| < tol)"""
    kl, h, aux, torch = env
    dense = kind.startswith("dense")
    n = 20 if dense else 256
    ones = torch.ones(n * n, dtype=torch.float64, device="cuda")
    if dense:
        A = _dense_poisson(n)
        b = h.dense_matvec(A, np.ones(n * n))
        x0s = [np.ones(n * n), np.ones(n * n) + 1e-9 * randn(torch, n * n, 5).cpu().numpy()]
    else:
        b = h.apply(kl.stvec, ones, n, n)
        x0s = [ones, ones + 1e-9 * randn(torch, n * n, 5)]
    for res_pos, x0 in zip((False, True), x0s):
        r = solve(env, kind, b, n, x0=x0, tol=1e-3, its=30, MAX_RESTARTS=5) if is_gmres(kind) else solve(
            env, kind, b, n, x0=x0, tol=1e-3, its=30)
        _check_zero_step(torch, kind, r, x0, res_pos, 1e-3)
    # the handle still solves cold afterwards (the early return left nothing behind)
    r = solve(env, kind, b, n, tol=1e-3, its=30, MAX_RESTARTS=2) if is_gmres(kind) else solve(
        env, kind, b, n, tol=1e-3, its=100)
    assert r.status in (KL_OK, KL_NOT_CONVERGED) and r.history.size > 0 and not np.isnan(r.history).any()


@pytest.mark.parametrize("kind", ["cg:0", "cg:1", "cg:2", "pcg:cbpr2", "pcg:nofuse", "bicgstab:cbpr2"])
@pytest.mark.parametrize("host", [False, True])
def test_maxit_zero_returns_x0(env, kind, host):
    kl, h, aux, torch = env
    n = 512
    b, x0 = randn(torch, n * n, 21), randn(torch, n * n, 22)
    if host:
        b, x0 = b.cpu().numpy(), x0.cpu().numpy()
    r = solve(env, kind, b, n, x0=x0, its=0)
    assert r.status == KL_NOT_CONVERGED and r.iter == 0 and r.history.size == 0
    assert xeq(torch, r.x, x0)


# ---------------------------------------------------------------------------------------------------------------
# 6. warm-started solves on a handle that holds CUDA graphs of cold solves
# ---------------------------------------------------------------------------------------------------------------
WARM_SOLVES = [("cg:0", 2048, dict(its=64, CHECK_EVERY=16)), ("cg:2", 2048, dict(its=64, CHECK_EVERY=16)),
               ("pcg:cbpr2", 2048, dict(its=48, CHECK_EVERY=16)),
               ("gmres:omp:1:cbpr2", 2048, dict(its=30, MAX_RESTARTS=3)), ("hh:omp:1", 512, dict(its=20, MAX_RESTARTS=3))]


def test_warm_start_on_warm_handle(env):
    kl, h0, aux, torch = env
    warm, fresh = kl.Handle(0), kl.Handle(0)
    try:
        for kind, n, kw in WARM_SOLVES:
            b, x0 = randn(torch, n * n, 31), randn(torch, n * n, 32)
            run = lambda hd, x0=None: solve((kl, hd, aux, torch), kind, b, n, x0=x0, **kw)
            run(warm)
            run(warm)                       # graphs captured and replayed by cold solves
            w1, w2 = run(warm, x0), run(warm)
            f1, f2 = run(fresh, x0), run(fresh)
            assert same(torch, w1, f1) and same(torch, w2, f2), kind
            assert not same(torch, w1, w2)
    finally:
        warm.close()
        fresh.close()


# ---------------------------------------------------------------------------------------------------------------
# 7. edges of the Python mirror and the C ABI
# ---------------------------------------------------------------------------------------------------------------
class _NoLibrary:
    def __getattr__(self, name):
        def call(*args):
            raise AssertionError(f"library called: {name}")
        return call


def test_api_edges(env):
    kl, h, aux, torch = env
    n = 256
    b = randn(torch, n * n, 41)
    x0 = randn(torch, n * n, 42)
    keep = x0.clone()
    # the caller's x0 is not written (device and host mode, CG and GMRES, also into a set_output_buffer buffer)
    r = h.cg_omp(kl.stvec, b, 1e-9, 20, nx=n, ny=n, x0=x0)
    assert torch.equal(x0, keep) and not torch.equal(r.x, x0)
    out = torch.empty_like(b)
    h.set_output_buffer(out)
    r = h.gmres_mgsr_omp(kl.stvec, b, 20, 1e-9, kl.cbpr2, P, nx=n, ny=n, x0=x0)
    assert r.x is out and torch.equal(x0, keep)
    bh, x0h = b.cpu().numpy(), x0.cpu().numpy()
    keep_h = x0h.copy()
    r = h.bicgstab(kl.stvec, bh, 1e-9, 20, nx=n, ny=n, x0=x0h)
    assert np.array_equal(x0h, keep_h) and not np.array_equal(r.x, x0h)
    # a mismatched kind or length raises before any call into the library
    L = h._L
    h._L = _NoLibrary()
    try:
        for bb, xx in ((b, x0h), (bh, x0), (b, x0.float()), (b, x0[:-1]), (bh, x0h[:-1]), (bh, list(x0h))):
            with pytest.raises(kl.KrylovError):
                h.cg_omp(kl.stvec, bb, 1e-9, 20, nx=n, ny=n, x0=xx)
            with pytest.raises(kl.KrylovError):
                h.gmres_hh_omp(kl.stvec, bb, 20, 1e-9, nx=n, ny=n, x0=xx)
    finally:
        h._L = L
    # C ABI: the option's values, x == b in device mode
    v = C.c_int()
    assert L.kl_set_option(h._h, X0, 2) == KL_ERR_INVALID
    assert L.kl_set_option(h._h, X0, 1) == KL_OK and L.kl_get_option(h._h, X0, C.byref(v)) == KL_OK and v.value == 1
    assert L.kl_set_pointer_mode(h._h, kl.api.KL_POINTER_DEVICE) == KL_OK
    o, _ = kl.stvec._c()
    it, res = C.c_int(20), C.c_double()
    xb = b.clone()
    assert L.kl_cg(h._h, C.byref(o), C.c_void_p(xb.data_ptr()), C.c_void_p(xb.data_ptr()), n, n, 1e-9, C.byref(it),
                   C.byref(res)) == KL_ERR_INVALID
    fe, ve, no, ro = np.zeros(20), np.zeros(21), C.c_int(), C.c_int()
    assert L.kl_gmres_hh_omp(h._h, C.byref(o), C.c_void_p(xb.data_ptr()), C.c_void_p(xb.data_ptr()), n, n, 20, 1e-9,
                             fe.ctypes.data_as(C.POINTER(C.c_double)), ve.ctypes.data_as(C.POINTER(C.c_double)),
                             C.byref(no), C.byref(ro)) == KL_ERR_INVALID
    assert torch.equal(xb, b)
    # the mirror sets the option on every call: a value left on the handle does not make a call without x0 warm
    cold = h.cg_omp(kl.stvec, b, 1e-9, 50, nx=n, ny=n)
    assert h.get_option(X0) == 0
    h.set_option(X0, 1)
    again = h.cg_omp(kl.stvec, b, 1e-9, 50, nx=n, ny=n)
    assert same(torch, cold, again)
