"""Stratosphere-adjusted forcing of the line-by-line path (rcm_lbl_adjusted_forcing / Solver.lbl_adjusted_forcing): the
adjustment dT of the stratospheric layers 0 .. ntrop - 1 that restores their heating rates after a VMR perturbation, and the
forcing at TOA and at the tropopause before (IRF) and after (SARF) it, without changing anything.

Checker: an independent solve on the C port (rcmo_lbl_tau + rcmo_lbl_radiative_transfer) at the state the next LBL step
radiates, dT added to the radiated profile of the stratospheric layers, and scipy's hybr for dE_l(perturbed, T + dT) =
dE_l(base, T), l < ntrop.
"""
import ctypes as C
import subprocess

import numpy as np
import pytest

from conftest import GOLDEN, table_path  # noqa: F401
from test_gpu_adjusted_forcing import FdhColumn
from test_gpu_adjusted_forcing_configs import kernel_solve
from test_gpu_lbl_diagnostics import _p, case, make, port_rt, port_tau  # noqa: F401 (case is a fixture)
from test_gpu_lbl_flux_jacobian import lbl_driver_case
from test_gpu_lbl_radiative_kernels import Port, case200, solver  # noqa: F401 (case200 is a fixture)

pytestmark = pytest.mark.gpu

NLAY, NLEV = 20, 21
CO2_2X, CO2_4X = [1.0, 2.0, 1.0, 1.0, 1.0], [1.0, 4.0, 1.0, 1.0, 1.0]
NTROP_CYCLE = (0, 2, 4, 7, 12)
KEYS = ("F", "dT_adj", "E_down", "E_up", "iters")


class LblColumn(FdhColumn):
    """The fixed-dynamical-heating problem of column col on the port: fluxes(f, dT) with the factors f (None: unscaled) and
    dT added to the radiated temperature of layers 0 .. len(dT) - 1; tau does not depend on T."""

    def __init__(self, P, col, f):
        self.P, self.col, self._tau = P, col, {}
        super().__init__(None, f)

    def tau(self, f):
        key = None if f is None else tuple(f)
        if key not in self._tau:
            t = port_tau(self.P.port, self.P.c, self.P.h2o, self.col, f)
            if self.P.cloud is not None:
                t[:, 17] = t[:, 17] - 1.0 + self.P.cloud[self.col]
            self._tau[key] = np.ascontiguousarray(t)
        return self._tau[key]

    def fluxes(self, f, dT=()):
        T = self.P.T[self.col].copy()
        T[:len(dT)] += dT
        return port_rt(self.P.port, self.P.p, self.tau(f), self.P.lo, self.P.hi, T, self.P.Ts[self.col])


def ntrop_of(n):
    return np.array([NTROP_CYCLE[c % len(NTROP_CYCLE)] for c in range(n)])


def check_against_port(port, s, c, steps, f, cols, cloud=None):
    ntrop = ntrop_of(s.ncol)
    d = s.lbl_adjusted_forcing(f, ntrop, tol=1e-9)
    assert np.all(d["converged"]), d["iters"]
    P = Port(port, c, s.get_state(), steps, None, cloud=cloud)
    for col in cols:
        m = ntrop[col]
        dT, F = LblColumn(P, col, f).solve(m)
        assert np.all(d["dT_adj"][col, m:] == 0.0), col
        assert np.abs(d["dT_adj"][col] - dT).max() <= 1e-6, (col, m, d["dT_adj"][col] - dT)
        assert np.abs(d["F"][col] - F).max() <= 1e-8, (col, m, d["F"][col] - F)
    return d


# ---- 1. against an independent solve on the port ----------------------------------------------------------------------------
@pytest.mark.parametrize("nwvl", [1500, 200])
@pytest.mark.parametrize("steps", [0, 3])
@pytest.mark.parametrize("f", [CO2_2X, CO2_4X], ids=["2xCO2", "4xCO2"])
def test_adjustment_equals_the_port_solution(rcm, port, case, case200, nwvl, steps, f):
    c = case if nwvl == 1500 else case200
    s = solver(rcm, c)
    if steps:
        s.advance(steps)
    d = check_against_port(port, s, c, steps, f, range(10))
    s.close()
    print(f"nwvl {nwvl}, steps {steps}, CO2 x{f[1]:g}: iters {np.bincount(d['iters'])}, "
          f"IRF_toa {d['IRF_toa'].mean():.4f}, SARF_toa {d['SARF_toa'].mean():.4f}")


@pytest.mark.parametrize("f", [[1.5, 1, 1, 1, 1], [1, 1, 0.5, 1, 1], [1, 1, 1, 2, 3], [1.2, 2, 0.8, 1.5, 1.1]],
                         ids=["h2o", "o3", "ch4_n2o", "all"])
def test_other_perturbations_against_the_port(rcm, port, case, f):
    """H2O and O3 through the scale kernel, CH4 and N2O through the composed plane, and all together"""
    s = solver(rcm, case)
    s.advance(2)
    check_against_port(port, s, case, 2, f, range(5, 15))
    s.close()


def test_column_cloud_against_the_port(rcm, port, case):
    s = solver(rcm, case)
    n = case["ncol"]
    tau_s = np.linspace(0.5, 4.0, n)
    s.set_column_solar(tau_s=tau_s, mu_s=np.linspace(0.3, 0.9, n), cloud_from_tau_s=True)
    s.advance(1)
    check_against_port(port, s, case, 1, CO2_2X, range(0, n, 3), cloud=tau_s / 2.0)
    s.close()


# ---- 2. exact cases ----------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("steps", [0, 2])
def test_exact_cases(rcm, case, steps):
    s = make(rcm, case)
    if steps:
        s.advance(steps)
    base = s.lbl_diagnose_fluxes()
    n = s.ncol
    # no perturbation: nothing to adjust, the base fluxes, which are the next step's
    d = s.lbl_adjusted_forcing([1, 1, 1, 1, 1], 7)
    assert np.all(d["iters"] == 0) and np.all(d["dT_adj"] == 0.0) and np.all(d["F"] == 0.0)
    assert np.array_equal(d["E_down"], base["E_down"]) and np.array_equal(d["E_up"], base["E_up"])
    for f in (CO2_4X, [1.5, 1, 0.5, 2, 3]):
        pert = s.lbl_diagnose_fluxes(vmr_scale=f)
        Nb, Np = base["E_down"] - base["E_up"], pert["E_down"] - pert["E_up"]
        # no stratosphere: SARF = IRF, the fluxes of the perturbed state
        d = s.lbl_adjusted_forcing(f, 0)
        assert np.all(d["iters"] == 0) and np.all(d["dT_adj"] == 0.0)
        assert np.array_equal(d["F"][:, 0], Np[:, 0] - Nb[:, 0]) and np.array_equal(d["F"][:, 0], d["F"][:, 2])
        assert np.array_equal(d["E_down"], pert["E_down"]) and np.array_equal(d["E_up"], pert["E_up"])
        # any stratosphere: iterate 0's IRF is the flux call's, bit for bit; SARF from the call's own fluxes
        k = np.arange(n)
        ntrop = np.array([NTROP_CYCLE[c % len(NTROP_CYCLE)] + c % 3 for c in k])
        d = s.lbl_adjusted_forcing(f, ntrop)
        assert np.array_equal(d["F"][:, 0], Np[:, 0] - Nb[:, 0]) and np.array_equal(d["F"][:, 1], Np[k, ntrop] - Nb[k, ntrop])
        Na = d["E_down"] - d["E_up"]
        assert np.array_equal(d["F"][:, 2], Na[:, 0] - Nb[:, 0]) and np.array_equal(d["F"][:, 3], Na[k, ntrop] - Nb[k, ntrop])
        for c in k:
            assert np.all(d["dT_adj"][c, ntrop[c]:] == 0.0), c
    s.advance(1)   # and the base state is the next step's
    g = s.get_state(want=("E_down", "E_up"))
    assert np.array_equal(g["E_down"], base["E_down"]) and np.array_equal(g["E_up"], base["E_up"])
    s.close()


@pytest.mark.parametrize("f", [CO2_4X, [1, 2, 1, 1.5, 2]])
def test_one_newton_step_is_the_solve_of_the_jacobian_block(rcm, case, f):
    """max_iter = 1 at a tolerance no update meets: dT_adj[c, :m] solves lbl_flux_jacobian(f)'s block against the flux
    calls' residual, in the Newton kernel's operation order"""
    s = make(rcm, case)
    s.advance(2)
    n = s.ncol
    ntrop = 1 + np.arange(n) % 19
    d = s.lbl_adjusted_forcing(f, ntrop, tol=1e-300, max_iter=1)
    H = s.lbl_flux_jacobian(vmr_scale=f)["dE_jac"]
    r = s.lbl_diagnose_fluxes(vmr_scale=f)["dE"] - s.lbl_diagnose_fluxes()["dE"]
    s.close()
    assert np.all(d["iters"] == -1)
    for c in range(n):
        m = ntrop[c]
        x = kernel_solve(H[c, :m, :m], -r[c, :m])
        assert np.array_equal(d["dT_adj"][c, :m], x), c
        assert np.all(d["dT_adj"][c, m:] == 0.0)


# ---- 3. self-consistency ------------------------------------------------------------------------------------------------------
def test_stratospheric_budget_and_convergence(rcm, case):
    s = make(rcm, case)
    s.advance(3)
    for tol in (1e-6, 1e-9):
        for m in (4, 9, 12):
            d = s.lbl_adjusted_forcing(CO2_2X, m, tol=tol)
            assert np.all(d["converged"]), d["iters"]
            assert d["iters"].max() <= 6, d["iters"]
            gap = np.abs(d["SARF_toa"] - d["SARF_trop"])
            assert np.all(gap <= m * tol + 1e-10), gap.max()
    s.close()


def test_unconverged_columns_are_reported(rcm, case):
    s = make(rcm, case)
    s.advance(2)
    ntrop = ntrop_of(s.ncol)
    full = s.lbl_adjusted_forcing(CO2_4X, ntrop, tol=1e-9)
    short = s.lbl_adjusted_forcing(CO2_4X, ntrop, tol=1e-9, max_iter=1)
    s.close()
    assert np.all(full["converged"])
    bad = short["iters"] == -1
    assert np.array_equal(bad, full["iters"] > 1) and bad.any() and (~bad).any()
    for k in KEYS:   # a column that converges within max_iter has the full call's results
        assert np.array_equal(short[k][~bad], full[k][~bad]), k


# ---- 4. determinism and no side effects ----------------------------------------------------------------------------------------
def test_three_chunks_and_a_reused_slot(rcm, case200):
    """16,400 columns = 8,192 + 8,192 + 16: chunk 1 has no stratosphere, so its slot finishes at iterate 0 and takes chunk 2
    while chunk 0 iterates.  Whole range = each chunk alone = single columns."""
    c, n, ch = case200, 16400, 8192
    s = make(rcm, c, 1.0, rep=n // c["ncol"] + 1, n=n)
    s.advance(1)
    ntrop = (np.arange(n) * 7) % 20
    ntrop[ch:2 * ch] = 0
    whole = s.lbl_adjusted_forcing(CO2_4X, ntrop, tol=1e-9)
    assert np.all(whole["converged"]) and np.all(whole["iters"][ch:2 * ch] == 0) and whole["iters"][:ch].max() > 0
    for c0 in (0, ch, 2 * ch):
        part = s.lbl_adjusted_forcing(CO2_4X, ntrop[c0:c0 + ch], col0=c0, ncol=min(ch, n - c0), tol=1e-9)
        for k in KEYS:
            assert np.array_equal(whole[k][c0:c0 + ch], part[k]), (c0, k)
    for col in (0, 8191, 8192, 16383, 16384, 16399):
        one = s.lbl_adjusted_forcing(CO2_4X, ntrop[col:col + 1], col0=col, ncol=1, tol=1e-9)
        for k in KEYS:
            assert np.array_equal(whole[k][col:col + 1], one[k]), (col, k)
    s.close()


def test_the_call_changes_nothing(rcm, case, tmp_path):
    a, b = make(rcm, case), make(rcm, case)
    for s in (a, b):
        s.advance(2)
    a.lbl_adjusted_forcing(CO2_2X, 4)
    a.lbl_adjusted_forcing([1.5, 2, 0.5, 2, 2], ntrop_of(a.ncol))
    a.lbl_adjusted_forcing(CO2_4X, 7, col0=5, ncol=7, max_iter=1)
    for s, p in ((a, "a.ck"), (b, "b.ck")):
        s.save_checkpoint(str(tmp_path / p))
    assert open(tmp_path / "a.ck", "rb").read() == open(tmp_path / "b.ck", "rb").read()
    for s in (a, b):
        s.advance(2)
    ga, gb = a.get_state(), b.get_state()
    for k in ga:
        assert np.array_equal(ga[k], gb[k]), k
    a.close(); b.close()


def test_errors_leave_the_solver_usable(rcm, case):
    L = rcm.load_library()
    ref = make(rcm, case)
    ref.advance(1)
    ref_next = ref.get_state()
    ref.close()
    s = make(rcm, case)
    h = s._h

    def call(col0=0, ncol=24, sc=CO2_2X, nt=4, tol=1e-6, max_iter=20, ntrop=True, h=h):
        scv = None if sc is None else np.ascontiguousarray(sc, dtype=np.float64)
        ntv = np.full(max(ncol, 1), nt, dtype=np.int32)
        F = np.zeros(max(ncol, 1) * 4)
        return L.rcm_lbl_adjusted_forcing(h, C.c_int(col0), C.c_int(ncol), None if scv is None else _p(scv),
                                          _p(ntv) if ntrop else None, C.c_double(tol), C.c_int(max_iter), _p(F), None, None,
                                          None, None)

    assert call() == 0 and call(sc=None) == 0
    assert call(col0=-1) == 1 and call(col0=20, ncol=5) == 1 and call(ncol=0) == 1
    for bad in ([-1, 1, 1, 1, 1], [1, np.nan, 1, 1, 1], [1, 1, np.inf, 1, 1]):
        assert call(sc=bad) == 1
    assert call(ntrop=False) == 1 and call(nt=-1) == 1 and call(nt=20) == 1
    for tol in (0.0, -1e-6, np.nan, np.inf):
        assert call(tol=tol) == 1
    assert call(max_iter=0) == 1
    nt = np.full(24, 4, dtype=np.int32)
    assert L.rcm_adjusted_forcing(h, 0, 24, None, _p(nt), C.c_double(1e-6), 20, _p(np.zeros(96)), None, None, None, None) == 2
    s.advance(1)
    got = s.get_state()
    for key in got:
        assert np.array_equal(got[key], ref_next[key]), key
    s.close()
    st = case["st"]
    r = rcm.Solver(0)
    r.set_repwvl_table_from(rcm.Table(table_path(10)))
    r.set_columns(case["pl"], st["Tlayer"], case["Tsurf"], st["vmr9"], st["rel_hum"])
    assert call(h=r._h) == 2
    r.close()
    e = rcm.Solver(0)
    e.set_lbl_tables(case["wvl"], case["tau5"], case["h2o_ref"], case["o3_ref"], 1.0)
    assert call(h=e._h, ncol=1) == 2
    e.close()


# ---- 5. the C++ driver -------------------------------------------------------------------------------------------------------
def test_driver_lbl_forcing_file(rcm, tmp_path):
    dc = lbl_driver_case(rcm, tmp_path)
    exe, common, pl = dc["exe"], dc["common"], dc["pl"]
    f1 = str(tmp_path / "f1.csv")
    r = subprocess.run([exe, *common, "--out", str(tmp_path / "o1.txt"), "--lbl-forcing-out", f1], capture_output=True,
                       text=True, timeout=300)
    assert r.returncode == 0, r.stderr
    s = dc["solver"]()
    d = s.lbl_adjusted_forcing(CO2_2X, 4)   # the driver's defaults: 1,2,1,1,1, 4 layers, tol 1e-6, 20 updates
    s.close()
    dT, F = np.zeros(NLAY), np.zeros(4)
    for c in range(d["F"].shape[0]):   # column order, then one division: the driver's arithmetic
        dT = dT + d["dT_adj"][c]
        F = F + d["F"][c]
    n = d["F"].shape[0]
    lines = open(f1).read().splitlines()
    assert lines[0] == "layer,p_layer,dT_adj" and len(lines) == 1 + NLAY + 5
    rows = [l.split(",") for l in lines[1:]]
    assert [r[0] for r in rows] == [str(l) for l in range(NLAY)] + ["IRF_toa", "IRF_trop", "SARF_toa", "SARF_trop",
                                                                     "unconverged"]
    assert np.array_equal([float(r[1]) for r in rows[:NLAY]], (pl[:NLAY] + pl[1:]) / 2.0)
    assert np.array_equal([float(r[2]) for r in rows[:NLAY]], dT / n)
    assert np.array_equal([float(r[2]) for r in rows[NLAY:NLAY + 4]], F / n)
    assert int(rows[-1][2]) == int(np.sum(d["iters"] < 0))
    # other factors and stratosphere
    f3 = str(tmp_path / "f3.csv")
    r = subprocess.run([exe, *common, "--out", str(tmp_path / "o3.txt"), "--lbl-forcing-out", f3, "--forcing-scale",
                        "1,4,1,1,1", "--trop-layers", "0"], capture_output=True, text=True, timeout=300)
    assert r.returncode == 0, r.stderr
    rows3 = [l.split(",") for l in open(f3).read().splitlines()[1:]]
    assert all(float(x[2]) == 0.0 for x in rows3[:NLAY]) and rows3[NLAY][2] == rows3[NLAY + 2][2]
    # refused with a repwvl table; --forcing-out still refused with --lbl; bad arguments
    r = subprocess.run([exe, "--atm", str(GOLDEN) + "/column21.atm", "--table", table_path(10), "--max-steps", "1",
                        "--lbl-forcing-out", str(tmp_path / "x.csv")], capture_output=True, text=True)
    assert r.returncode == 1 and "--lbl-forcing-out" in r.stderr
    r = subprocess.run([exe, *common, "--forcing-out", str(tmp_path / "x.csv")], capture_output=True, text=True)
    assert r.returncode == 1 and "--forcing-out" in r.stderr and "--lbl-forcing-out" in r.stderr
    for bad in (["--trop-layers", "20"], ["--forcing-scale", "1,2,1,1"]):
        r = subprocess.run([exe, *common, "--lbl-forcing-out", str(tmp_path / "x.csv"), *bad], capture_output=True, text=True)
        assert r.returncode == 1 and bad[0] in r.stderr, bad
    if rcm.device_count() < 2:
        pytest.skip("the --gpus 2 half needs two GPUs")
    f2 = str(tmp_path / "f2.csv")
    r = subprocess.run([exe, *common, "--out", str(tmp_path / "o2.txt"), "--lbl-forcing-out", f2, "--gpus", "2"],
                       capture_output=True, text=True, timeout=300)
    assert r.returncode == 0, r.stderr
    assert open(f1, "rb").read() == open(f2, "rb").read()
