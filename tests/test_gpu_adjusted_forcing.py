"""Stratosphere-adjusted forcing by fixed dynamical heating (rcm_adjusted_forcing / Solver.adjusted_forcing): the adjustment
dT of the stratospheric layers 0 .. ntrop - 1 that restores their heating rates after a VMR perturbation, and the forcing at
TOA and at the tropopause before (IRF) and after (SARF) it, without changing anything.

Checker: an independent solve on the C port of the reference (oracle/rcm_oracle.c).  Per column the port's read_tau and
radiative_transfer evaluate dE at the inputs the next step radiates with (test_gpu_radiative_kernels.radiated_inputs), dT
added to the stratospheric layers of both the profile tau is interpolated at and the radiated profile, and
scipy.optimize.root (hybr) solves dE_l(perturbed, T + dT) = dE_l(base, T) for l < ntrop.
"""
import ctypes as C
import os

import numpy as np
import pytest
from scipy.optimize import root

from conftest import GOLDEN, table_path
from test_gpu_diagnostics import CO2_2X, ensemble, solver, status_of
from test_gpu_radiative_kernels import driver, radiated_inputs

pytestmark = pytest.mark.gpu
NLAY, NLEV = 20, 21
CO2_4X = [1.0, 4.0, 1.0, 1.0, 1.0]
NTROP_CYCLE = (0, 2, 4, 7, 12)
OPT_PATH = 5


@pytest.fixture(scope="module")
def ens21(rcm):
    return ensemble(rcm, 21, 2024)


# ---- the port's fixed-dynamical-heating solve -----------------------------------------------------------------------------
class PortColumn:
    """One column of the port: fluxes of the base state and of the perturbed state at T + dT (dT on layers 0 .. m - 1)."""

    def __init__(self, port, tab, st, T, vmr9, rel_hum, Tsurf, first, co2_scale, tau_s):
        self.port, self.tab, self.pl, self.Tsurf, self.tau_s = port, tab, st["plevel"], Tsurf, tau_s
        self.tau_T, self.Trad, self.v0 = radiated_inputs(port, st, T, vmr9, rel_hum, first)
        self.v1 = radiated_inputs(port, st, T, vmr9, rel_hum, first, co2_scale=co2_scale)[2]

    def fluxes(self, v9, dT=()):
        d = np.zeros(NLAY)
        d[:len(dT)] = dT
        tau, _, _ = self.port.read_tau(self.tab, self.pl, self.tau_T + d, v9, tau_s=self.tau_s)
        return self.port.radiative_transfer(tau, self.tab["wvl"], self.tab["weight"], self.Trad + d, self.Tsurf, 0.0)

    def solve(self, m):
        """-> dT [20], F [4] of the port's own solution (tight hybr tolerance, from dT = 0)."""
        Ed0, Eu0, dE0 = self.fluxes(self.v0)
        Ed1, Eu1, _ = self.fluxes(self.v1)
        x = np.zeros(0)
        if m:
            x = root(lambda x: self.fluxes(self.v1, x)[2][:m] - dE0[:m], np.zeros(m), method="hybr",
                     options=dict(xtol=1e-14)).x
            assert self.residual(m, x) <= 1e-10, (m, self.residual(m, x))
        Ed2, Eu2, _ = self.fluxes(self.v1, x)
        N0, N1, N2 = Ed0 - Eu0, Ed1 - Eu1, Ed2 - Eu2
        dT = np.zeros(NLAY)
        dT[:m] = x
        return dT, np.array([N1[0] - N0[0], N1[m] - N0[m], N2[0] - N0[0], N2[m] - N0[m]])

    def residual(self, m, dT):
        """max_{l < m} |dE_l(perturbed, T + dT) - dE_l(base, T)| on the port."""
        if m == 0:
            return 0.0
        return np.abs(self.fluxes(self.v1, dT[:m])[2][:m] - self.fluxes(self.v0)[2][:m]).max()


def check_against_port(port, s, st, tab, nsteps_done, vmr_scale, tau_s=None):
    ntrop = np.array([NTROP_CYCLE[c % len(NTROP_CYCLE)] for c in range(s.ncol)])
    d = s.adjusted_forcing(vmr_scale, ntrop, tol=1e-9)
    assert np.all(d["converged"]), d["iters"]
    g = s.get_state(("Tlayer", "Tsurf"))
    for c in range(s.ncol):
        m = ntrop[c]
        col = PortColumn(port, tab, st, g["Tlayer"][c], st["vmr9"][c], st["rel_hum"][c], g["Tsurf"][c], nsteps_done == 0,
                         vmr_scale[1], 2.0 if tau_s is None else tau_s[c])
        dT, F = col.solve(m)
        assert np.all(d["dT_adj"][c, m:] == 0.0), c
        assert np.abs(d["dT_adj"][c] - dT).max() <= 1e-6, (c, m, d["dT_adj"][c] - dT)
        assert np.abs(d["F"][c] - F).max() <= 1e-8, (c, m, d["F"][c] - F)
        assert col.residual(m, d["dT_adj"][c]) <= 1e-8, (c, m, col.residual(m, d["dT_adj"][c]))
    return d


# ---- 1. against an independent solve on the port ----------------------------------------------------------------------------
@pytest.mark.parametrize("nsteps", [3, 0])
@pytest.mark.parametrize("vmr_scale", [CO2_2X, CO2_4X], ids=["2xCO2", "4xCO2"])
def test_adjustment_equals_the_port_solution(rcm, port, ens21, nsteps, vmr_scale):
    """21 columns (a ragged second tile), Reduced20, ntrop cycling over 0, 2, 4, 7, 12."""
    tab = port.load_rcmtab(table_path(20))
    s = solver(rcm, 20, ens21)
    if nsteps:
        s.advance(nsteps)
    d = check_against_port(port, s, ens21, tab, nsteps, vmr_scale)
    s.close()
    print(f"nsteps {nsteps}, CO2 x{vmr_scale[1]:g}: iters {np.bincount(d['iters'])}")


def test_column_cloud(rcm, port, ens21):
    tab = port.load_rcmtab(table_path(20))
    s = solver(rcm, 20, ens21)
    s.advance(1)
    rng = np.random.default_rng(5)
    tau_s, mu_s = rng.uniform(0.5, 4.0, s.ncol), rng.uniform(0.3, 0.8, s.ncol)
    s.set_column_solar(None, tau_s, mu_s, None, cloud_from_tau_s=True)
    check_against_port(port, s, ens21, tab, 1, CO2_2X, tau_s=tau_s)
    s.close()


# ---- 2. exact cases ----------------------------------------------------------------------------------------------------------
def test_exact_cases(rcm, ens21):
    s = solver(rcm, 100, ens21)
    s.advance(2)
    base = s.diagnose_fluxes(spectral=False)
    pert = s.diagnose_fluxes(vmr_scale=CO2_2X, spectral=False)
    # no perturbation: nothing to adjust, the base fluxes
    d = s.adjusted_forcing(None, 7)
    assert np.all(d["iters"] == 0) and np.all(d["dT_adj"] == 0.0) and np.all(d["F"] == 0.0)
    assert np.array_equal(d["E_down"], base["E_down"]) and np.array_equal(d["E_up"], base["E_up"])
    # no stratosphere: SARF = IRF, the fluxes of the perturbed state
    d = s.adjusted_forcing(CO2_2X, 0)
    irf_toa = (pert["E_down"][:, 0] - pert["E_up"][:, 0]) - (base["E_down"][:, 0] - base["E_up"][:, 0])
    assert np.all(d["iters"] == 0) and np.all(d["dT_adj"] == 0.0)
    assert np.array_equal(d["F"][:, 0], d["F"][:, 2]) and np.array_equal(d["F"][:, 0], irf_toa)
    assert np.array_equal(d["E_down"], pert["E_down"]) and np.array_equal(d["E_up"], pert["E_up"])
    # any stratosphere: the IRF columns are those of the two diagnostic calls
    k = np.arange(s.ncol)
    ntrop = np.array([NTROP_CYCLE[c % len(NTROP_CYCLE)] + c % 3 for c in k])
    d = s.adjusted_forcing(CO2_2X, ntrop)
    s.close()
    Nb, Np = base["E_down"] - base["E_up"], pert["E_down"] - pert["E_up"]
    assert np.array_equal(d["F"][:, 0], irf_toa) and np.array_equal(d["F"][:, 1], Np[k, ntrop] - Nb[k, ntrop])
    # and the SARF columns those of the call's own fluxes
    Na = d["E_down"] - d["E_up"]
    assert np.array_equal(d["F"][:, 2], Na[:, 0] - Nb[:, 0]) and np.array_equal(d["F"][:, 3], Na[k, ntrop] - Nb[k, ntrop])
    for c in k:
        assert np.all(d["dT_adj"][c, ntrop[c]:] == 0.0), c


# ---- 3. self-consistency ------------------------------------------------------------------------------------------------------
def test_stratospheric_budget_and_cooling(rcm):
    st = ensemble(rcm, 2000, 31)
    s = solver(rcm, 100, st)
    s.advance(3)
    tol = 1e-6
    for m in (4, 9):
        d = s.adjusted_forcing(CO2_2X, m, tol=tol)
        ok = d["converged"]
        assert ok.mean() > 0.99, np.bincount(d["iters"] + 1)
        # summed over the stratosphere the heating-rate changes telescope to Delta N_0 - Delta N_trop
        gap = np.abs(d["SARF_toa"][ok] - d["SARF_trop"][ok])
        assert np.all(gap <= m * tol + 1e-10), gap.max()
        assert d["dT_adj"][:, 0].mean() < 0.0  # 2xCO2 cools the stratosphere
        assert np.all(d["dT_adj"][:, m:] == 0.0)
    s.close()


# ---- 4. determinism and no side effects -----------------------------------------------------------------------------------------
def test_results_do_not_depend_on_the_range_or_the_chunks(rcm):
    """8,200 columns: two chunks of the whole-range call (8,192 + 8), a sub-range in one chunk, single columns."""
    st = ensemble(rcm, 8200, 13)
    s = solver(rcm, 100, st)
    s.advance(2)
    ntrop = (np.arange(8200) * 7) % 20
    whole = s.adjusted_forcing(CO2_2X, ntrop)
    part = s.adjusted_forcing(CO2_2X, ntrop[4000:], col0=4000)
    keys = ("F", "dT_adj", "E_down", "E_up", "iters")
    for k in keys:
        assert np.array_equal(whole[k][4000:], part[k]), k
    for c in (0, 15, 16, 4000, 4321, 8183, 8191, 8192, 8195, 8199):
        one = s.adjusted_forcing(CO2_2X, ntrop[c:c + 1], col0=c, ncol=1)
        for k in keys:
            assert np.array_equal(whole[k][c:c + 1], one[k]), (c, k)
    s.close()


def test_the_call_changes_nothing(rcm, ens21, tmp_path):
    a, b = solver(rcm, 20, ens21), solver(rcm, 20, ens21)
    b.adjusted_forcing(CO2_2X, 4)
    sa = [a.advance(2)]
    sb = [b.advance(2)]
    b.adjusted_forcing(CO2_4X, np.arange(21) % 20, col0=0, ncol=21)
    b.adjusted_forcing(CO2_2X, 6, col0=3, ncol=5)
    sa.append(a.advance(2))
    sb.append(b.advance(2))
    for x, y in zip(sa, sb):
        assert np.array_equal(x, y)
    ga, gb = a.get_state(), b.get_state()
    for k in ga:
        assert np.array_equal(ga[k], gb[k]), k
    a.save_checkpoint(str(tmp_path / "a.ckpt"))
    b.save_checkpoint(str(tmp_path / "b.ckpt"))
    assert open(tmp_path / "a.ckpt", "rb").read() == open(tmp_path / "b.ckpt", "rb").read()
    a.close()
    b.close()


# ---- 5. non-convergence and errors ----------------------------------------------------------------------------------------------
def test_unconverged_columns_are_reported(rcm, port, ens21):
    """max_iter = 1 at a tolerance one update cannot meet: RCM_OK, iters -1, outputs of the last evaluated iterate."""
    tab = port.load_rcmtab(table_path(20))
    s = solver(rcm, 20, ens21)
    s.advance(1)
    base = s.diagnose_fluxes(spectral=False)
    d = s.adjusted_forcing(CO2_4X, 12, tol=1e-12, max_iter=1)
    g = s.get_state(("Tlayer", "Tsurf"))
    s.close()
    assert np.any(d["iters"] == -1) and np.all((d["iters"] == -1) | (d["iters"] == 0) | (d["iters"] == 1))
    assert np.all(np.isfinite(d["F"])) and np.all(np.isfinite(d["dT_adj"])) and np.any(d["dT_adj"] != 0.0)
    Nb = base["E_down"] - base["E_up"]
    assert np.array_equal(d["SARF_toa"], (d["E_down"][:, 0] - d["E_up"][:, 0]) - Nb[:, 0])
    assert np.array_equal(d["SARF_trop"], (d["E_down"][:, 12] - d["E_up"][:, 12]) - Nb[:, 12])
    for c in np.flatnonzero(d["iters"] == -1)[:5]:  # E_down / E_up are the port's fluxes at the reported dT_adj
        col = PortColumn(port, tab, ens21, g["Tlayer"][c], ens21["vmr9"][c], ens21["rel_hum"][c], g["Tsurf"][c], False, 4.0,
                         2.0)
        Ed, Eu, _ = col.fluxes(col.v1, d["dT_adj"][c, :12])
        sc = np.abs(Eu).max()
        assert np.abs(d["E_down"][c] - Ed).max() <= 1e-10 * sc and np.abs(d["E_up"][c] - Eu).max() <= 1e-10 * sc, c


def test_errors_leave_the_solver_usable(rcm, ens21):
    s = solver(rcm, 20, ens21)
    for col0, ncol in ((-1, 3), (0, 0), (20, 2), (0, 22)):
        assert status_of(rcm, lambda: s.adjusted_forcing(CO2_2X, np.zeros(max(ncol, 0), int), col0, ncol)) == 1, (col0, ncol)
    for bad in (-1.0, np.nan, np.inf):
        assert status_of(rcm, lambda: s.adjusted_forcing([1.0, bad, 1.0, 1.0, 1.0], 4)) == 1, bad
    for bad in (-1, 20):
        nt = np.full(21, 4)
        nt[17] = bad
        assert status_of(rcm, lambda: s.adjusted_forcing(CO2_2X, nt)) == 1, bad
    for tol in (0.0, -1e-6, np.nan, np.inf):
        assert status_of(rcm, lambda: s.adjusted_forcing(CO2_2X, 4, tol=tol)) == 1, tol
    assert status_of(rcm, lambda: s.adjusted_forcing(CO2_2X, 4, max_iter=0)) == 1
    L = rcm.load_library()
    F = np.zeros((21, 4))
    st = L.rcm_adjusted_forcing(s._h, C.c_int(0), C.c_int(21), None, None, C.c_double(1e-6), C.c_int(20),
                                rcm.capi._p(F), None, None, None, None)
    assert st == 1 and "ntrop" in L.rcm_last_error(s._h).decode()
    with pytest.raises(ValueError):
        s.adjusted_forcing([2.0], 4)
    with pytest.raises(ValueError):
        s.adjusted_forcing(CO2_2X, np.full(20, 4))
    s.set_option(OPT_PATH, 1)
    assert status_of(rcm, lambda: s.adjusted_forcing(CO2_2X, 4)) == 2
    s.set_option(OPT_PATH, 0)
    ref = s.adjusted_forcing(CO2_2X, 4)
    s.advance(1)
    assert np.all(ref["converged"]) and np.all(s.adjusted_forcing(CO2_2X, 4)["converged"])
    s.close()

    p = rcm.default_params()
    p.species_mask = 0x0F
    m = solver(rcm, 20, ens21, params=p)
    assert status_of(rcm, lambda: m.adjusted_forcing(None, 4)) == 2
    m.advance(1)
    m.close()

    st = ens21
    lb = rcm.Solver(0)
    wvl, tau5 = rcm.make_lbl_tables(300, 7, st["plevel"], st["vmr9"][0, 0], st["vmr9"][0, 2])
    lb.set_lbl_tables(wvl, tau5, st["vmr9"][0, 0], st["vmr9"][0, 2])
    lb.set_columns(st["plevel"], st["Tlayer"], st["Tsurf"], st["vmr9"], st["rel_hum"])
    assert status_of(rcm, lambda: lb.adjusted_forcing(CO2_2X, 4)) == 2
    lb.advance(1)
    assert np.isfinite(lb.get_state(("E_up",))["E_up"]).all()
    lb.close()


# ---- 6. the driver's --forcing-out -------------------------------------------------------------------------------------------------
def test_driver_forcing_out(rcm, tmp_path):
    ck, ff = str(tmp_path / "run.ckpt"), str(tmp_path / "forcing.csv")
    common = ["--table", table_path(100), "--ncol", "64", "--seed", "9", "--max-steps", "3", "--steps-exact"]
    r = driver(rcm, *common, "--out", str(tmp_path / "o.txt"), "--checkpoint", ck, "--forcing-out", ff)
    assert r.returncode == 0, r.stderr
    lines = open(ff).read().splitlines()
    assert lines[0] == "layer,p_layer,dT_adj" and len(lines) == 1 + NLAY + 5
    rows = [l.split(",") for l in lines[1:]]
    assert [r[0] for r in rows] == [str(l) for l in range(NLAY)] + ["IRF_toa", "IRF_trop", "SARF_toa", "SARF_trop",
                                                                     "unconverged"]
    assert all(r[1] == "" for r in rows[NLAY:])

    s = rcm.Solver(0)
    s.set_repwvl_table_from(rcm.Table(table_path(100)))
    s.load_checkpoint(ck)
    d = s.adjusted_forcing(CO2_2X, 4)  # the driver's defaults: 1,2,1,1,1, 4 layers, tol 1e-6, 20 updates
    s.close()
    dT, F = np.zeros(NLAY), np.zeros(4)
    for c in range(d["F"].shape[0]):  # column order, then one division: the driver's arithmetic
        dT = dT + d["dT_adj"][c]
        F = F + d["F"][c]
    n = d["F"].shape[0]
    atm = rcm.read_atm(os.path.join(GOLDEN, "column21.atm"))
    pl = atm[:, 1]
    assert np.array_equal([float(r[1]) for r in rows[:NLAY]], (pl[:NLAY] + pl[1:]) / 2.0)
    assert np.array_equal([float(r[2]) for r in rows[:NLAY]], dT / n)
    assert np.array_equal([float(r[2]) for r in rows[NLAY:NLAY + 4]], F / n)
    assert int(rows[-1][2]) == int(np.sum(d["iters"] < 0))

    # no stratosphere: SARF = IRF, no adjustment
    r = driver(rcm, *common, "--out", str(tmp_path / "o3.txt"), "--forcing-out", str(tmp_path / "f3.csv"),
               "--forcing-scale", "1,4,1,1,1", "--trop-layers", "0")
    assert r.returncode == 0, r.stderr
    rows3 = [l.split(",") for l in open(tmp_path / "f3.csv").read().splitlines()[1:]]
    assert all(float(x[2]) == 0.0 for x in rows3[:NLAY]) and rows3[NLAY][2] == rows3[NLAY + 2][2]
    assert float(rows3[NLAY][2]) > 0.0 and rows3[-1][2] == "0"

    d = tmp_path / "lbl"
    d.mkdir()
    r = driver(rcm, "--lbl", str(d), "--forcing-out", ff, "--max-steps", "1")
    assert r.returncode == 1 and "--forcing-out" in r.stderr
    for bad in (["--trop-layers", "x"], ["--trop-layers", "4x"], ["--trop-layers", "20"], ["--forcing-scale", "1,2,1,1"]):
        r = driver(rcm, *common, "--out", str(tmp_path / "o4.txt"), "--forcing-out", ff, *bad)
        assert r.returncode == 1 and bad[0] in r.stderr, bad

    if rcm.device_count() < 2:
        pytest.skip("--gpus 2 needs two GPUs")
    ff2 = str(tmp_path / "forcing2.csv")
    r = driver(rcm, *common, "--out", str(tmp_path / "o2.txt"), "--forcing-out", ff2, "--gpus", "2")
    assert r.returncode == 0, r.stderr
    assert open(ff).read() == open(ff2).read()
