"""The many-mode field reference (tests/many_modes_ref.py) on the CPU: it is the oracle's solve wherever the oracle can
hold the mode set, and it reproduces field_test's analytic answer with every mode 1 .. nx/2 kept."""
import numpy as np
import pytest

from many_modes_ref import ManyModeField, field_test_expected
from oracle import oracle as O


@pytest.mark.parametrize("nx,modes", [(192, range(1, 65)), (256, [1, 2, 3, 7]), (1000, [3, -5, 64, 499])])
def test_reference_is_the_oracle_solve_up_to_64_modes(nx, modes):
    modes = list(modes)
    op = O.default_params(nx=nx, nmode=len(modes), modes=modes)
    o = O.Oracle(op)
    rho = np.random.default_rng(nx).standard_normal(nx) * 1e-4
    E, mre, mim = o.field_solve(rho)
    ref = ManyModeField(nx, op.lx, modes)
    E2, mre2, mim2 = ref.solve(rho)
    assert np.array_equal(ref.F_re.ravel(), o.F_re) and np.array_equal(ref.F_im.ravel(), o.F_im)
    assert np.array_equal(ref.grad_inv, o.grad_inv)
    assert np.array_equal(E2, E) and np.array_equal(mre2, mre) and np.array_equal(mim2, mim)


def test_chunks_keep_each_mode_column():
    """Tables of 512 modes built 64 at a time equal the oracle's tables of any 64-mode subset, column for column."""
    nx, lx = 1024, O.default_params().lx
    ref = ManyModeField(nx, lx, range(1, 513))
    sub = [5, 70, 133, 200, 511]
    o = O.Oracle(O.default_params(nx=nx, nmode=len(sub), modes=sub))
    cols = [m - 1 for m in sub]
    assert np.array_equal(ref.F_re[:, cols].ravel(), o.F_re) and np.array_equal(ref.F_im[:, cols].ravel(), o.F_im)
    assert np.array_equal(ref.grad_inv[cols], o.grad_inv)


@pytest.mark.parametrize("m0", [1, 2, 64, 65, 200, 511])
def test_field_test_analytic_all_modes_kept(m0):
    """field_test (src/pic1dp_field.F90:276-309) with every mode 1 .. 512 of nx = 1024 kept: rho_j = cos(2 pi m0 j / nx)
    gives E_j = sin(2 pi m0 j / nx) / k_m0, whichever m0, and only mode m0 is excited."""
    nx, lx = 1024, O.default_params().lx
    ref = ManyModeField(nx, lx, range(1, nx // 2 + 1))
    rho, E_exact = field_test_expected(nx, lx, m0)
    E, mre, mim = ref.solve(rho)
    assert np.max(np.abs(E - E_exact)) < 1e-12
    assert abs(mim[m0 - 1] * (2.0 * np.pi * m0 / lx) + 0.5) < 1e-12   # -(1/nx) sum cos^2 = -1/2, times 1/k
    others = np.delete(np.abs(mim), m0 - 1).max() + np.abs(mre).max()
    assert others * (2.0 * np.pi / lx) < 1e-12
