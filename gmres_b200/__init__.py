"""gmres_b200 -- B200-native (sm_100a) Krylov hot path behind the reference's plug-in API.

Host-side Python mirror of the reference's module procedures (AlexanderGSC/gmres):
same names, argument order and meaning as the Fortran interfaces, over the C ABI in
include/krylov_b200.h (libkrylov_b200.so, hand-written CUDA).  There is NO CPU
fallback: importing works without a GPU (so that the ABI can be inspected), but
creating a Handle or running anything requires the CUDA library and a device and
fails loudly otherwise.

    import gmres_b200 as kl
    h = kl.Handle()
    b = h.apply(kl.stvec, np.ones(n * n), n, n)              # call stvec(x, b, nsize)
    r = h.gmres_mgsr_omp(kl.stvec, b, 95, 1e-8, kl.cbpr2, (8.2, 0.2))
    r.x, r.final_err, r.v_err, r.n_out, r.restart_out       # the reference's outputs
"""
from . import api  # noqa: F401
from .api import (  # noqa: F401
    Handle,
    KrylovError,
    Operator,
    Precond,
    GmresResult,
    CgResult,
    stvec,
    stv_poisson,
    aniso,
    aniso_var,
    stencil5,
    convdiff,
    stencil5_spectrum,
    cbpr2,
    cheb,
    jacobi_cheb,
    no_precond,
    ORTHO_MGS2,
    ORTHO_CGS2,
    ORTHO_CGS2_SELECTIVE,
    HH_SEQUENTIAL,
    HH_BLOCKED,
    library_path,
    load_library,
    KL_OPT_FUSE,
    KL_OPT_TMA,
    KL_OPT_CHAIN,
    KL_OPT_STENCIL_ROWS,
    KL_OPT_PROFILE,
    KL_OPT_CHECK_EVERY,
    KL_OPT_X0,
    KL_PC_JACOBI_CHEB,
    KL_OP_STENCIL5,
)

__all__ = [
    "Handle", "KrylovError", "Operator", "Precond", "GmresResult", "CgResult", "stvec",
    "stv_poisson", "aniso", "stencil5", "convdiff", "stencil5_spectrum", "cbpr2", "cheb", "jacobi_cheb", "no_precond", "library_path", "load_library",
]
