"""Reference field solve for any number of kept modes, built from the oracle's C restatement.

orc_params holds up to 64 modes.  Every column of the partial-DFT tables and every projection depends on its own mode
alone, so the oracle's orc_field_init and orc_field_solve run 64 modes at a time give the tables, mode_re and mode_im
of the whole set unchanged.  Only the synthesis E_j = 2 (sum_m F_re[j,m] re[m] + sum_m F_im[j,m] im[m]) sums over
modes; it is done here left to right over the whole set, one IEEE add and multiply per term like MatMult /
MatMultAdd (numpy evaluates each elementwise product and sum separately, never fused).
"""
from __future__ import annotations

import ctypes as C

import numpy as np

from oracle import oracle as O

CHUNK = O.MAX_MODES


def _dp(a):
    return a.ctypes.data_as(C.POINTER(C.c_double))


class ManyModeField:
    def __init__(self, nx: int, lx: float, modes):
        self.nx, self.lx, self.modes = nx, lx, [int(m) for m in modes]
        M = len(self.modes)
        self.F_re, self.F_im, self.grad_inv = np.empty((nx, M)), np.empty((nx, M)), np.empty(M)
        self.chunks = []
        for c in range(0, M, CHUNK):
            ms = self.modes[c:c + CHUNK]
            o = O.Oracle(O.default_params(nx=nx, lx=lx, nmode=len(ms), modes=ms))
            self.F_re[:, c:c + len(ms)] = o.F_re.reshape(nx, len(ms))
            self.F_im[:, c:c + len(ms)] = o.F_im.reshape(nx, len(ms))
            self.grad_inv[c:c + len(ms)] = o.grad_inv
            self.chunks.append((c, o))

    def solve(self, rho):
        """(E, mode_re, mode_im) of field_solve_electric in the sequential (one-rank SeqAIJ) order."""
        rho = np.ascontiguousarray(rho, dtype=np.float64)
        M = len(self.modes)
        mre, mim = np.empty(M), np.empty(M)
        for c, o in self.chunks:
            E, r, i = o.field_solve(rho)
            mre[c:c + r.size], mim[c:c + i.size] = r, i
        s = np.zeros(self.nx)
        for m in range(M):
            s = s + self.F_re[:, m] * mre[m]   # MatMult(F_re, mode_re)   src/pic1dp_field.F90:251
        for m in range(M):
            s = s + self.F_im[:, m] * mim[m]   # MatMultAdd(F_im, mode_im) :253
        return s * 2.0, mre, mim               # :256


def field_test_expected(nx: int, lx: float, m0: int):
    """field_test with rho_j = cos(2 pi m0 j / nx): E_j = sin(2 pi m0 j / nx) / k_m0, k_m0 = 2 pi m0 / lx."""
    j = np.arange(nx)
    return np.cos(2.0 * np.pi * m0 * j / nx), np.sin(2.0 * np.pi * m0 * j / nx) / (2.0 * np.pi * m0 / lx)
