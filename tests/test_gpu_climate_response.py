"""Equilibrium climate response (rcm_climate_response / Solver.climate_response): the response dT of the stratospheric layers
0 .. ntrop - 1 and the uniform potential-temperature increment dTs of the troposphere and the surface that restore the
stratospheric heating rates and the net flux at the tropopause after a VMR perturbation, with the water-vapour feedback at
fixed relative humidity or at fixed absolute humidity, without changing anything.

Checker: an independent solve on the C port of the reference (oracle/rcm_oracle.c).  Per column the port's read_tau and
radiative_transfer evaluate the fluxes at the inputs the next step radiates with (test_gpu_radiative_kernels.radiated_inputs),
dT added to both the profile tau is interpolated at and the radiated profile, T_surf + dTs, with fixed RH the H2O of the port's
feedback at T + dT times the H2O factor, and scipy.optimize.root (hybr) solves the ntrop + 1 equations.
"""
import ctypes as C
import os

import numpy as np
import pytest
from scipy.linalg import lu_factor
from scipy.optimize import root

from conftest import GOLDEN, table_path
from test_gpu_adjusted_forcing_configs import one_step_case
from test_gpu_diagnostics import CO2_2X, ensemble, feedback, solver, status_of, theta_sort
from test_gpu_radiative_kernels import driver, radiated_inputs

pytestmark = pytest.mark.gpu
NLAY, NLEV, NE = 20, 21, 41
CO2_4X = [1.0, 4.0, 1.0, 1.0, 1.0]
NTROP_CYCLE = (0, 2, 4, 7, 12)
OPT_PATH = 5
KEYS = ("F", "dT", "dTs", "E_down", "E_up", "iters")


@pytest.fixture(scope="module")
def ens21(rcm):
    return ensemble(rcm, 21, 2024)


def ntrop_of(n):
    return np.array([NTROP_CYCLE[c % len(NTROP_CYCLE)] for c in range(n)])


def gamma(T):
    """d ln q / dT of the feedback's Magnus formula"""
    x = T - 273.15 + 243.04
    return 17.625 * 243.04 / (x * x)


# ---- the port's response solve ------------------------------------------------------------------------------------------------
class EcsColumn:
    """The climate-response problem of one column on the port: fluxes(x) of the perturbed state at the unknowns x = (dT_0 ..
    dT_{m-1}, dTs) (None: the base state), dT_l = dTs / conv_l below the tropopause, the surface at T_surf + dTs."""

    def __init__(self, port, tab, st, T, vmr9, rel_hum, Tsurf, first, f, fixed_rh, m, tau_s=2.0):
        self.port, self.tab, self.pl, self.Tsurf, self.tau_s = port, tab, st["plevel"], Tsurf, tau_s
        self.conv, self.player, self.rel_hum = st["conv"], st["player"], rel_hum
        self.f, self.fixed_rh, self.m = f, fixed_rh, m
        self.tau_T, self.Trad, self.v0 = radiated_inputs(port, st, T, vmr9, rel_hum, first)
        self.v1 = radiated_inputs(port, st, T, vmr9, rel_hum, first, h2o_scale=f[0], co2_scale=f[1])[2]

    def profile(self, x):
        m = self.m
        d = np.zeros(NLAY)
        d[:m] = x[:m]
        d[m:] = x[m] / self.conv[m:]
        return d

    def fluxes(self, x=None):
        if x is None:
            tau, _, _ = self.port.read_tau(self.tab, self.pl, self.tau_T, self.v0, tau_s=self.tau_s)
            return self.port.radiative_transfer(tau, self.tab["wvl"], self.tab["weight"], self.Trad, self.Tsurf, 0.0)
        d = self.profile(x)
        v = self.v1.copy()
        if self.fixed_rh:
            v[0] = feedback(self.port, self.Trad + d, self.rel_hum, self.player) * self.f[0]
        tau, _, _ = self.port.read_tau(self.tab, self.pl, self.tau_T + d, v, tau_s=self.tau_s)
        return self.port.radiative_transfer(tau, self.tab["wvl"], self.tab["weight"], self.Trad + d, self.Tsurf + x[self.m], 0.0)

    def residual(self, x):
        m = self.m
        Ed0, Eu0, dE0 = self.base
        Ed, Eu, dE = self.fluxes(x)
        return np.append(dE[:m] - dE0[:m], (Ed[m] - Eu[m]) - (Ed0[m] - Eu0[m]))

    def solve(self):
        """-> dT [20], dTs, F [2] of the port's own solution (tight hybr tolerance, from 0)."""
        self.base = self.fluxes()
        x = root(self.residual, np.zeros(self.m + 1), method="hybr", options=dict(xtol=1e-14)).x
        assert np.abs(self.residual(x)).max() <= 1e-10, (self.m, self.residual(x))
        Ed0, Eu0, _ = self.base
        Ed1, Eu1, _ = self.fluxes(np.zeros(self.m + 1))
        N0, N1, m = Ed0 - Eu0, Ed1 - Eu1, self.m
        return self.profile(x), x[m], np.array([N1[0] - N0[0], N1[m] - N0[m]])


def check_against_port(port, s, st, tab, nsteps_done, f, fixed_rh):
    ntrop = ntrop_of(s.ncol)
    d = s.climate_response(f, ntrop, fixed_rh=fixed_rh, tol=1e-9)
    assert np.all(d["converged"]), d["iters"]
    g = s.get_state(("Tlayer", "Tsurf"))
    for c in range(s.ncol):
        m = ntrop[c]
        col = EcsColumn(port, tab, st, g["Tlayer"][c], st["vmr9"][c], st["rel_hum"][c], g["Tsurf"][c], nsteps_done == 0, f,
                        fixed_rh, m)
        dT, dTs, F = col.solve()
        assert np.abs(d["dT"][c] - dT).max() <= 1e-6, (c, m, d["dT"][c] - dT)
        assert abs(d["dTs"][c] - dTs) <= 1e-6, (c, m, d["dTs"][c] - dTs)
        assert np.abs(d["F"][c] - F).max() <= 1e-8, (c, m, d["F"][c] - F)
        x = np.append(d["dT"][c, :m], d["dTs"][c])
        assert np.abs(col.residual(x)).max() <= 1e-8, (c, m, col.residual(x))
    return d


# ---- 1. against an independent solve on the port ------------------------------------------------------------------------------
@pytest.mark.parametrize("nsteps,fixed_rh", [(3, True), (3, False), (0, False)], ids=["rh", "q", "q_step0"])
@pytest.mark.parametrize("f", [CO2_2X, CO2_4X], ids=["2xCO2", "4xCO2"])
def test_response_equals_the_port_solution(rcm, port, ens21, nsteps, fixed_rh, f):
    """21 columns (a ragged second tile), Reduced20, ntrop cycling over 0, 2, 4, 7, 12."""
    tab = port.load_rcmtab(table_path(20))
    s = solver(rcm, 20, ens21)
    if nsteps:
        s.advance(nsteps)
    d = check_against_port(port, s, ens21, tab, nsteps, f, fixed_rh)
    s.close()
    print(f"nsteps {nsteps}, fixed_rh {fixed_rh}, CO2 x{f[1]:g}: iters {np.bincount(d['iters'])}, dTs {d['dTs'].mean():.4f}")


# ---- 2. exact cases -----------------------------------------------------------------------------------------------------------
def newton_matrix(J, H, T, m, fixed_rh, conv):
    """A [m + 1][m + 1] of one column, assembled from flux_jacobian's J [2][21][41] and dE_jac [20][41] as the call defines it"""
    D = np.vstack([H[:m], J[0, m] - J[1, m]])
    g = gamma(T) if fixed_rh else np.zeros(NLAY)
    A = np.zeros((m + 1, m + 1))
    A[:, :m] = D[:, :m] + g[:m] * D[:, NLAY + 1:NLAY + 1 + m]
    A[:, m] = D[:, NLAY] + ((D[:, m:NLAY] + g[m:] * D[:, NLAY + 1 + m:]) / conv[m:]).sum(axis=1)
    return A


def test_exact_cases(rcm, port, ens21):
    s = solver(rcm, 100, ens21)
    s.advance(2)
    n = s.ncol
    base = s.diagnose_fluxes(spectral=False)
    pert = s.diagnose_fluxes(vmr_scale=CO2_2X, spectral=False)
    # no perturbation: nothing responds, the base fluxes
    for rh in (True, False):
        d = s.climate_response(None, 7, fixed_rh=rh)
        assert np.all(d["iters"] == 0) and np.all(d["dT"] == 0.0) and np.all(d["dTs"] == 0.0) and np.all(d["F"] == 0.0)
        assert np.array_equal(d["E_down"], base["E_down"]) and np.array_equal(d["E_up"], base["E_up"])
    # F: the IRF of adjusted_forcing and of the two diagnostic calls, bit for bit
    k = np.arange(n)
    ntrop = np.array([NTROP_CYCLE[c % len(NTROP_CYCLE)] + c % 3 for c in k])
    tol = 1e-6
    d = s.climate_response(CO2_2X, ntrop, tol=tol)
    a = s.adjusted_forcing(CO2_2X, ntrop)
    Nb, Np = base["E_down"] - base["E_up"], pert["E_down"] - pert["E_up"]
    assert np.array_equal(d["F"], a["F"][:, :2])
    assert np.array_equal(d["F"][:, 0], Np[:, 0] - Nb[:, 0]) and np.array_equal(d["F"][:, 1], Np[k, ntrop] - Nb[k, ntrop])
    # at the solution the TOA net flux is back to the base's: the heating rates telescope
    assert np.all(d["converged"]), d["iters"]
    Na = d["E_down"] - d["E_up"]
    assert np.all(np.abs(Na[:, 0] - Nb[:, 0]) <= (ntrop + 1) * tol + 1e-10)
    for c in k:
        m = ntrop[c]
        assert np.array_equal(d["dT"][c, m:], d["dTs"][c] / ens21["conv"][m:]), c
    # one Newton update: a NumPy solve of A assembled from flux_jacobian at iterate 0
    g = s.get_state(("Tlayer",))
    for rh in (True, False):
        one = s.climate_response(CO2_4X, ntrop, fixed_rh=rh, tol=1e-12, max_iter=1)
        assert np.all(one["iters"] == -1)
        fj = s.flux_jacobian(vmr_scale=CO2_4X)
        p4 = s.diagnose_fluxes(vmr_scale=CO2_4X, spectral=False)
        for c in k:
            m = ntrop[c]
            Tb = theta_sort(port, g["Tlayer"][c], ens21["conv"])
            A = newton_matrix(fj["J"][c], fj["dE_jac"][c], Tb, m, rh, ens21["conv"])
            r = np.append(p4["dE"][c, :m] - base["dE"][c, :m],
                          (p4["E_down"][c, m] - p4["E_up"][c, m]) - (base["E_down"][c, m] - base["E_up"][c, m]))
            delta = np.linalg.solve(A, -r)
            got = np.append(one["dT"][c, :m], one["dTs"][c])
            assert np.abs(got - delta).max() <= 1e-12 * np.abs(delta).max(), (c, m, got - delta)
    s.close()


def test_one_update_with_row_exchanges(rcm, port):
    """The edge ensemble's cold-layer columns give Newton matrices that need a row exchange: one update (max_iter = 1) is
    still numpy's solve of A, within a few (m + 1) eps cond(A)."""
    s, st, _, _, _ = one_step_case(rcm, port, "edge")
    n = s.ncol
    ntrop = 1 + np.arange(n) % 19
    pl = st["plevel"]
    conv = (1000.0 / ((pl[:-1] + pl[1:]) / 2.0)) ** (2.0 / 7.0)
    base = s.diagnose_fluxes(spectral=False)
    p4 = s.diagnose_fluxes(vmr_scale=CO2_4X, spectral=False)
    fj = s.flux_jacobian(vmr_scale=CO2_4X)
    one = s.climate_response(CO2_4X, ntrop, fixed_rh=False, tol=1e-300, max_iter=1)
    s.close()
    exchanged, compared = 0, 0
    for c in range(n):
        m = ntrop[c]
        A = newton_matrix(fj["J"][c], fj["dE_jac"][c], None, m, False, conv)
        r = np.append(p4["dE"][c, :m] - base["dE"][c, :m],
                      (p4["E_down"][c, m] - p4["E_up"][c, m]) - (base["E_down"][c, m] - base["E_up"][c, m]))
        if not (np.isfinite(A).all() and np.isfinite(r).all()) or one["iters"][c] != -1:
            continue
        delta = np.linalg.solve(A, -r)
        got = np.append(one["dT"][c, :m], one["dTs"][c])
        err = np.abs(got - delta).max() / np.abs(delta).max()
        assert err <= 4 * (m + 1) * 2.2e-16 * np.linalg.cond(A, np.inf), (c, m, err)
        exchanged += int(np.any(lu_factor(A)[1] != np.arange(m + 1)))
        compared += 1
    print(f"edge: {exchanged} of {compared} compared Newton matrices need a row exchange")
    assert compared > n // 2 and exchanged > 0


# ---- 3. physics ---------------------------------------------------------------------------------------------------------------
def test_physics(rcm):
    st = ensemble(rcm, 500, 31)
    s = solver(rcm, 100, st)
    s.advance(3)
    m = 4
    rh2 = s.climate_response(CO2_2X, m)
    q2 = s.climate_response(CO2_2X, m, fixed_rh=False)
    rh4 = s.climate_response(CO2_4X, m)
    for d in (rh2, q2, rh4):
        assert d["converged"].mean() > 0.99, np.bincount(d["iters"] + 1)
    ok = rh2["converged"] & q2["converged"] & rh4["converged"]
    ecs_rh, ecs_q, ecs4 = rh2["dTs"][ok].mean(), q2["dTs"][ok].mean(), rh4["dTs"][ok].mean()
    print(f"dTs 2xCO2: fixed RH {ecs_rh:.4f} K, fixed q {ecs_q:.4f} K; 4xCO2 fixed RH {ecs4:.4f} K")
    assert ecs_q > 0.0 and ecs_rh > ecs_q           # warming, amplified by the water-vapour feedback
    assert rh2["dT"][ok, 0].mean() < 0.0            # the stratosphere cools
    assert 1.6 < ecs4 / ecs_rh < 2.4                 # about proportional to ln(CO2)
    # linear consistency: for a small forcing dTs = -SARF_trop / lambda, lambda the Schur complement of A at the base state
    # (at fixed q: the adjustment of adjusted_forcing keeps q fixed)
    f = [1.0, 1.01, 1.0, 1.0, 1.0]
    d = s.climate_response(f, m, fixed_rh=False, tol=1e-10)
    a = s.adjusted_forcing(f, m, tol=1e-12)
    fj = s.flux_jacobian()
    lam = np.zeros(s.ncol)
    for c in range(s.ncol):
        A = newton_matrix(fj["J"][c], fj["dE_jac"][c], None, m, False, st["conv"])
        lam[c] = A[m, m] - A[m, :m] @ np.linalg.solve(A[:m, :m], A[:m, m])
    ok = d["converged"] & a["converged"]
    lin = (-a["SARF_trop"][ok] / lam[ok]).mean()
    print(f"CO2 x1.01: dTs {d['dTs'][ok].mean():.6f} K, -SARF_trop / lambda {lin:.6f} K")
    assert abs(d["dTs"][ok].mean() - lin) <= 0.02 * abs(lin)
    s.close()


# ---- 4. determinism and no side effects ---------------------------------------------------------------------------------------
@pytest.mark.parametrize("ncol", [8200, 16400])
def test_results_do_not_depend_on_the_range_or_the_chunks(rcm, ncol):
    """two resp. three chunks of the whole-range call, a sub-range, single columns on both sides of every chunk boundary"""
    st = ensemble(rcm, ncol, 13)
    s = solver(rcm, 100, st)
    s.advance(2)
    ntrop = (np.arange(ncol) * 7) % 20
    whole = s.climate_response(CO2_2X, ntrop)
    assert whole["converged"].mean() > 0.99
    part = s.climate_response(CO2_2X, ntrop[4000:], col0=4000)
    for k in KEYS:
        assert np.array_equal(whole[k][4000:], part[k]), k
    for c in (0, 15, 16, 4000, 8191, 8192, 8199, ncol - 1) + ((16383, 16384) if ncol > 16384 else ()):
        one = s.climate_response(CO2_2X, ntrop[c:c + 1], col0=c, ncol=1)
        for k in KEYS:
            assert np.array_equal(whole[k][c:c + 1], one[k]), (c, k)
    s.close()


def test_the_call_changes_nothing(rcm, ens21, tmp_path):
    a, b = solver(rcm, 20, ens21), solver(rcm, 20, ens21)
    b.climate_response(CO2_2X, 4, fixed_rh=False)
    sa = [a.advance(2)]
    sb = [b.advance(2)]
    b.climate_response(CO2_4X, np.arange(21) % 20, col0=0, ncol=21)
    b.climate_response(CO2_2X, 6, col0=3, ncol=5, fixed_rh=False)
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
    # two solvers with different tables share the constant bank
    c = solver(rcm, 100, ens21)
    c.advance(2)
    ra = a.climate_response(CO2_2X, 4)
    rc = c.climate_response(CO2_2X, 4)
    assert np.array_equal(ra["dTs"], a.climate_response(CO2_2X, 4)["dTs"])
    assert np.array_equal(rc["dTs"], c.climate_response(CO2_2X, 4)["dTs"])
    for x in (a, b, c):
        x.close()


# ---- 5. non-convergence and errors --------------------------------------------------------------------------------------------
def test_unconverged_columns_are_reported(rcm, ens21):
    """max_iter = 1 at a tolerance one update cannot meet: RCM_OK, iters -1, outputs of the last evaluated iterate."""
    s = solver(rcm, 20, ens21)
    s.advance(1)
    base = s.diagnose_fluxes(spectral=False)
    d = s.climate_response(CO2_4X, 12, tol=1e-12, max_iter=1)
    assert np.all(d["iters"] == -1) and np.all(np.isfinite(d["dTs"])) and np.all(d["dTs"] != 0.0)
    Nb = base["E_down"] - base["E_up"]
    assert np.all(np.isfinite(d["E_down"] - d["E_up"] - Nb))
    s.close()


def test_errors_leave_the_solver_usable(rcm, ens21):
    s = solver(rcm, 20, ens21)
    for col0, ncol in ((-1, 3), (0, 0), (20, 2), (0, 22)):
        assert status_of(rcm, lambda: s.climate_response(CO2_2X, np.zeros(max(ncol, 0), int), False, col0, ncol)) == 1
    for bad in (-1.0, np.nan, np.inf):
        assert status_of(rcm, lambda: s.climate_response([1.0, bad, 1.0, 1.0, 1.0], 4, False)) == 1, bad
    for bad in (-1, 20):
        nt = np.full(21, 4)
        nt[17] = bad
        assert status_of(rcm, lambda: s.climate_response(CO2_2X, nt, False)) == 1, bad
    for tol in (0.0, -1e-6, np.nan, np.inf):
        assert status_of(rcm, lambda: s.climate_response(CO2_2X, 4, False, tol=tol)) == 1, tol
    assert status_of(rcm, lambda: s.climate_response(CO2_2X, 4, False, max_iter=0)) == 1
    # fixed RH at step 0: the step applies no feedback there
    assert status_of(rcm, lambda: s.climate_response(CO2_2X, 4, True)) == 2
    assert np.all(s.climate_response(CO2_2X, 4, False)["converged"])
    L = rcm.load_library()
    F = np.zeros((21, 2))
    st = L.rcm_climate_response(s._h, C.c_int(0), C.c_int(21), None, None, C.c_int(0), C.c_double(1e-6), C.c_int(20),
                                rcm.capi._p(F), None, None, None, None, None)
    assert st == 1 and "ntrop" in L.rcm_last_error(s._h).decode()
    with pytest.raises(ValueError):
        s.climate_response([2.0], 4)
    s.advance(1)
    s.set_option(OPT_PATH, 1)
    assert status_of(rcm, lambda: s.climate_response(CO2_2X, 4)) == 2
    s.set_option(OPT_PATH, 0)
    assert np.all(s.climate_response(CO2_2X, 4)["converged"])
    s.close()

    p = rcm.default_params()
    p.species_mask = 0x1E  # no H2O
    m = solver(rcm, 20, ens21, params=p)
    m.advance(1)
    assert status_of(rcm, lambda: m.climate_response(None, 4)) == 2
    m.advance(1)
    m.close()

    st = ens21
    lb = rcm.Solver(0)
    wvl, tau5 = rcm.make_lbl_tables(300, 7, st["plevel"], st["vmr9"][0, 0], st["vmr9"][0, 2])
    lb.set_lbl_tables(wvl, tau5, st["vmr9"][0, 0], st["vmr9"][0, 2])
    lb.set_columns(st["plevel"], st["Tlayer"], st["Tsurf"], st["vmr9"], st["rel_hum"])
    lb.advance(1)
    assert status_of(rcm, lambda: lb.climate_response(CO2_2X, 4)) == 2
    lb.advance(1)
    assert np.isfinite(lb.get_state(("E_up",))["E_up"]).all()
    lb.close()


# ---- 6. the driver's --response-out -------------------------------------------------------------------------------------------
def read_rows(path):
    lines = open(path).read().splitlines()
    assert lines[0] == "layer,p_layer,dT" and len(lines) == 1 + NLAY + 4
    return [l.split(",") for l in lines[1:]]


def test_driver_response_out(rcm, tmp_path):
    ck, rf = str(tmp_path / "run.ckpt"), str(tmp_path / "response.csv")
    common = ["--table", table_path(100), "--ncol", "64", "--seed", "9", "--max-steps", "3", "--steps-exact"]
    r = driver(rcm, *common, "--out", str(tmp_path / "o.txt"), "--checkpoint", ck, "--response-out", rf)
    assert r.returncode == 0, r.stderr
    rows = read_rows(rf)
    assert [x[0] for x in rows] == [str(l) for l in range(NLAY)] + ["dTs", "IRF_toa", "IRF_trop", "unconverged"]
    assert all(x[1] == "" for x in rows[NLAY:])
    r = driver(rcm, *common, "--out", str(tmp_path / "oq.txt"), "--response-out", str(tmp_path / "q.csv"), "--fixed-q",
               "--forcing-scale", "1,4,1,1,1", "--trop-layers", "2")
    assert r.returncode == 0, r.stderr
    rows_q = read_rows(tmp_path / "q.csv")

    s = rcm.Solver(0)
    s.set_repwvl_table_from(rcm.Table(table_path(100)))
    s.load_checkpoint(ck)
    atm = rcm.read_atm(os.path.join(GOLDEN, "column21.atm"))
    pl = atm[:, 1]
    for rws, d in ((rows, s.climate_response(CO2_2X, 4)), (rows_q, s.climate_response(CO2_4X, 2, fixed_rh=False))):
        dT, dTs, F = np.zeros(NLAY), 0.0, np.zeros(2)
        for c in range(d["F"].shape[0]):  # column order, then one division: the driver's arithmetic
            dT = dT + d["dT"][c]
            dTs = dTs + d["dTs"][c]
            F = F + d["F"][c]
        n = d["F"].shape[0]
        assert np.array_equal([float(x[1]) for x in rws[:NLAY]], (pl[:NLAY] + pl[1:]) / 2.0)
        assert np.array_equal([float(x[2]) for x in rws[:NLAY]], dT / n)
        assert float(rws[NLAY][2]) == dTs / n and np.array_equal([float(x[2]) for x in rws[NLAY + 1:NLAY + 3]], F / n)
        assert int(rws[-1][2]) == int(np.sum(d["iters"] < 0))
    s.close()

    d = tmp_path / "lbl"
    d.mkdir()
    r = driver(rcm, "--lbl", str(d), "--response-out", rf, "--max-steps", "1")
    assert r.returncode == 1 and "--response-out" in r.stderr
    r = driver(rcm, *common, "--out", str(tmp_path / "o5.txt"), "--lbl-response-out", rf)
    assert r.returncode == 1 and "--lbl-response-out" in r.stderr
    for bad in (["--trop-layers", "x"], ["--trop-layers", "20"], ["--forcing-scale", "1,2,1,1"]):
        r = driver(rcm, *common, "--out", str(tmp_path / "o4.txt"), "--response-out", rf, *bad)
        assert r.returncode == 1 and bad[0] in r.stderr, bad

    if rcm.device_count() < 2:
        pytest.skip("--gpus 2 needs two GPUs")
    rf2 = str(tmp_path / "response2.csv")
    r = driver(rcm, *common, "--out", str(tmp_path / "o2.txt"), "--response-out", rf2, "--gpus", "2")
    assert r.returncode == 0, r.stderr
    assert open(rf).read() == open(rf2).read()
