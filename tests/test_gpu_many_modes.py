"""Field solve with any number of kept modes (pic1dp_gpu_set_modes), up to every mode 1 .. nx/2 the grid resolves:
the many-mode kernels against the oracle's operators and solve order (tests/many_modes_ref.py), the unchanged
single-CTA path, the time loop, the unfiltered bump-on-tail growth rate, the host driver's modes= and the refusals."""
import ctypes as C
import subprocess

import numpy as np
import pytest

import pic1dp_b200 as P
from pic1dp_b200 import _capi
from helpers import ChunkedOracleRun, copy_state, make_params, rel_err, synth_markers
from many_modes_ref import ManyModeField
from test_gpu_physics import GAMMA_ANALYTIC, quiet_start
from tools_py3.runinfo import growthrate_energy_fit

pytestmark = pytest.mark.gpu

TOL_SUM = 1e-12   # rho, E: relative to max|.|, as in test_gpu_parity.py


def _solve(gp, modes, rho):
    with P.Pic1dGpu(gp) as g:
        g.set_modes(modes)
        g.set_field(chargeden=rho)
        g.solve_field()
        f = g.get_field()
        ops = g.get_operators()
    return f, ops


@pytest.mark.parametrize("nx,modes", [(192, range(1, 97)), (1024, range(1, 513)), (4096, range(1, 2049)),
                                      (4096, range(1, 1001, 3))])
def test_solve_matches_oracle(nx, modes):
    """SEQUENTIAL: E, mode_re, mode_im bit-identical to the oracle's sequential solve of the same rho, and the tables
    bit-identical to field_init's; TREE: within 1e-13 of max|.| (it runs the same order above 64 modes: identical)."""
    modes = list(modes)
    op, gp = make_params(nx=nx, capacity=16, field_mode=P.FIELD_SEQUENTIAL)
    ref = ManyModeField(nx, op.lx, modes)
    rho = np.random.default_rng(nx + len(modes)).standard_normal(nx) * 1e-4
    E, mre, mim = ref.solve(rho)
    f, (Fre, Fim, ginv) = _solve(gp, modes, rho)
    assert np.array_equal(Fre, ref.F_re) and np.array_equal(Fim, ref.F_im) and np.array_equal(ginv, ref.grad_inv)
    assert np.array_equal(f["electric"], E)
    assert np.array_equal(f["mode_re"], mre) and np.array_equal(f["mode_im"], mim)
    _, gp_tree = make_params(nx=nx, capacity=16, field_mode=P.FIELD_TREE)
    ft, _ = _solve(gp_tree, modes, rho)
    scale = max(np.abs(mre).max(), np.abs(mim).max())
    assert rel_err(ft["electric"], E) < 1e-13
    assert rel_err(ft["mode_re"], mre, scale) < 1e-13 and rel_err(ft["mode_im"], mim, scale) < 1e-13
    assert all(np.array_equal(ft[k], f[k]) for k in ("electric", "mode_re", "mode_im"))


def test_set_modes_with_create_time_set_is_bitwise_unchanged():
    """A handle created with modes {1, 2, 3} and one given the same set through set_modes: identical rho, E and
    markers after 10 steps."""
    op, gp = make_params(nx=256, nmode=3, modes=[1, 2, 3], capacity=200000, deposit_mode=P.DEPOSIT_FIXED)
    _, gp1 = make_params(nx=256, capacity=200000, deposit_mode=P.DEPOSIT_FIXED)
    st = synth_markers(op, 200000, seed=21)
    outs = []
    for params, modes in ((gp, None), (gp1, [1, 2, 3])):
        with P.Pic1dGpu(params) as g:
            if modes:
                g.set_modes(modes)
            g.set_markers(0, st["x"], st["v"], st["p"], st["w"])
            g.collect_charge()
            g.solve_field()
            g.step(10)
            outs.append((g.get_field(), g.get_markers(0)))
    for k in ("electric", "chargeden", "mode_re", "mode_im"):
        assert np.array_equal(outs[0][0][k], outs[1][0][k]), k
    for k in ("x", "v", "p", "w"):
        assert np.array_equal(outs[0][1][k], outs[1][1][k]), k


class _ManyModeRun(ChunkedOracleRun):
    """The oracle's time loop with the field solved over any mode set."""

    def __init__(self, op, st, nchunks, modes):
        super().__init__(op, st, nchunks)
        self.set_modes(modes)

    def set_modes(self, modes):
        self.field = ManyModeField(self.op.nx, self.op.lx, modes)

    def solve_field(self):
        self.E, self.mode_re, self.mode_im = self.field.solve(self.rho)


def test_time_loop_unfiltered_nx1024():
    """1e6 markers, nx = 1024, modes 1 .. 512, 10 steps against the oracle, with the set changed to modes 1 .. 256
    after step 5: cell indices bit-exact at every substep, rho and E within TOL_SUM, x, v, w within 1e-12; step(1)
    replayed from the captured graph equals step(1) with no_step_graph = 1 bit for bit."""
    n, nx, nsteps, switch = 1_000_000, 1024, 10, 5
    full, half = list(range(1, nx // 2 + 1)), list(range(1, nx // 4 + 1))
    op, gp = make_params(nx=nx, capacity=n)
    st = synth_markers(op, n, seed=22)
    ref = _ManyModeRun(op, copy_state(st), 8, full)
    ref.init_field()
    with P.Pic1dGpu(gp) as g:   # the reference driver's calls, one substep at a time
        g.set_modes(full)
        g.set_markers(0, st["x"], st["v"], st["p"], st["w"])
        g.collect_charge()
        g.solve_field()
        for it in range(nsteps):
            if it == switch:
                ref.set_modes(half)
                g.set_modes(half)
            for irk in (1, 2):
                ref.push(irk)
                ref.collect_charge()
                ref.solve_field()
                g.push(irk)
                g.collect_charge()
                g.solve_field()
                f = g.get_field()
                assert np.array_equal(g.get_shape_x(0)[0], ref.cell_index()), (it, irk)
                assert rel_err(f["chargeden"], ref.rho) < TOL_SUM, (it, irk)
                assert rel_err(f["electric"], ref.E) < TOL_SUM, (it, irk)
        assert f["mode_re"].size == len(half)
    stepped = []
    for no_graph in (0, 1):
        _, gps = make_params(nx=nx, capacity=n, no_step_graph=no_graph)
        with P.Pic1dGpu(gps) as g:
            g.set_modes(full)
            g.set_markers(0, st["x"], st["v"], st["p"], st["w"])
            g.collect_charge()
            g.solve_field()
            for it in range(nsteps):
                if it == switch:
                    g.set_modes(half)
                g.step(1)
            stepped.append((g.get_field(), g.get_markers(0), g.counters().graph_replays))
    assert stepped[0][2] == nsteps and stepped[1][2] == 0
    for k in ("electric", "chargeden", "mode_re", "mode_im"):
        assert np.array_equal(stepped[0][0][k], stepped[1][0][k]), k
    for k in ("x", "v", "w"):
        assert np.array_equal(stepped[0][1][k], stepped[1][1][k]), k
        assert rel_err(stepped[0][1][k], ref.full[k]) < 1e-12, k
    assert rel_err(stepped[0][0]["chargeden"], ref.rho) < TOL_SUM and rel_err(stepped[0][0]["electric"], ref.E) < TOL_SUM


def test_bump_on_tail_growth_rate_unfiltered():
    """The default bump-on-tail run at nx = 192 with every mode 1 .. 96 kept, 4e6 quiet-start markers, t = 0..60: the
    growth rate of mode 1's energy |mode_1|^2, fitted on [20, 50], within 3 % of the analytic root."""
    op, gp = make_params(nx=192, capacity=4_000_000)
    st = quiet_start(op, 2000, 2000)
    with P.Pic1dGpu(gp) as g:
        g.set_modes(range(1, 97))
        g.set_markers(0, st["x"], st["v"], st["p"], st["w"])
        g.collect_charge()
        g.solve_field()
        t, en = [], []
        for it in range(120):
            g.step(10)
            f = g.get_field()
            t.append(op.dt * 10 * (it + 1))
            en.append(f["mode_re"][0] ** 2 + f["mode_im"][0] ** 2)
        assert g.counters().oob_markers == 0
    gamma = growthrate_energy_fit(np.array(t), np.array(en), 20.0, 50.0) / 2.0
    assert abs(gamma / GAMMA_ANALYTIC - 1.0) < 0.03, gamma


def test_cpp_host_driver_modes_range(tmp_path):
    """host/pic1dp_host modes=1:96 writes a pic1dp.out with all 96 modes; its records agree with the text trace."""
    from pic1dp_b200 import build
    from tools_py3.output_data import OutputData
    exe = build.build_host()
    out, pout = tmp_path / "energy.txt", tmp_path / "pic1dp.out"
    r = subprocess.run([exe, "nparticle_max=300000", "nx=192", "time_max=2", "seed_type=1", "modes=1:96", f"out={out}",
                        f"petsc_out={pout}"], capture_output=True, text=True, timeout=600)
    assert r.returncode == 0, r.stdout + r.stderr
    rows = np.loadtxt(out)
    od = OutputData(str(pout))
    assert (od.nmode, od.nx) == (96, 192) and list(od.mode) == list(range(1, 97)) and od.ntime == rows.shape[0]
    sc, md = od.get_scalar_t(), od.get_mode_t()
    assert np.allclose(sc[0], rows[:, 0]) and np.array_equal(sc[1], rows[:, 1])
    assert np.array_equal(md[0], rows[:, 2]) and np.array_equal(md[96], rows[:, 3])
    bad = subprocess.run([exe, "modes=0:3"], capture_output=True, text=True, timeout=600)
    assert bad.returncode != 0


def test_refusals_leave_the_handle_usable():
    """nmode = 0, a mode 0, a NULL modes pointer and tables past PIC1DP_MAX_FIELD_TABLE_BYTES are refused with their
    codes; the handle keeps its mode set and solves as before."""
    nx = 8192
    op, gp = make_params(nx=nx, capacity=16, field_mode=P.FIELD_SEQUENTIAL)
    modes = list(range(1, 101))
    rho = np.random.default_rng(23).standard_normal(nx) * 1e-4
    with P.Pic1dGpu(gp) as g:
        g.set_modes(modes)
        g.set_field(chargeden=rho)
        g.solve_field()
        before = g.get_field()
        L = g.L
        one = (C.c_int32 * 1)(1)
        assert L.pic1dp_gpu_set_modes(g._h, 0, one) == _capi.EINVAL
        assert L.pic1dp_gpu_set_modes(g._h, 1, None) == _capi.EINVAL
        assert L.pic1dp_gpu_set_modes(g._h, 3, (C.c_int32 * 3)(1, 0, 2)) == _capi.EINVAL
        too_many = _capi.MAX_FIELD_TABLE_BYTES // (32 * nx) + 1
        big = (C.c_int32 * too_many)(*range(1, too_many + 1))
        assert L.pic1dp_gpu_set_modes(g._h, too_many, big) == _capi.EUNSUPPORTED
        assert "PIC1DP_MAX_FIELD_TABLE_BYTES" in L.pic1dp_gpu_last_error(g._h).decode()
        with pytest.raises(P.Pic1dpError):
            g.set_modes([])
        assert g.modes == modes
        g.set_field(chargeden=rho)
        g.solve_field()
        after = g.get_field()
    for k in ("electric", "mode_re", "mode_im"):
        assert np.array_equal(before[k], after[k]), k
