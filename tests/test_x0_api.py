"""CPU-only: the x0 argument of the Python mirror (KL_OPT_X0) is validated before any call into the library, and the
option is declared in the C header with the value the mirror uses."""
import os
import re

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


class _NoLibrary:
    def __getattr__(self, name):
        def call(*args):
            raise AssertionError(f"library called: {name}")
        return call


@pytest.fixture
def handle():
    """a Handle whose library must not be reached (no device is needed to get this far)"""
    import gmres_b200 as kl
    h = kl.Handle.__new__(kl.Handle)
    h._L, h._h = _NoLibrary(), None
    return h


def test_option_value_matches_header():
    import gmres_b200 as kl
    hdr = open(os.path.join(ROOT, "include", "krylov_b200.h")).read()
    assert int(re.search(r"KL_OPT_X0\s*=\s*(\d+)", hdr).group(1)) == kl.KL_OPT_X0 == 23
    assert int(re.search(r"#define KL_VERSION (\d+)", hdr).group(1)) == 101


@pytest.mark.parametrize("x0", [list(np.zeros(64)), np.zeros(63), np.zeros((2, 64))])
def test_bad_x0_raises_before_the_library(handle, x0):
    import gmres_b200 as kl
    b = np.ones(64)
    calls = [lambda: handle.cg(kl.stvec, b, 1e-9, 10, x0=x0),
             lambda: handle.pbicgstab_omp(kl.stvec, b, 1e-9, 10, kl.cbpr2, (8.2, 0.2), x0=x0),
             lambda: handle.gmres_mgsr_omp(kl.stvec, b, 5, 1e-9, x0=x0),
             lambda: handle.gmres_hh_omp(kl.stvec, b, 5, 1e-9, x0=x0),
             lambda: handle.gmres_mgsr_dense(np.eye(64), b, 5, 1e-9, x0=x0)]
    for call in calls:
        with pytest.raises(kl.KrylovError):
            call()
