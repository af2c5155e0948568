"""Equilibrium climate response of the line-by-line path (rcm_lbl_climate_response / Solver.lbl_climate_response): the
stratospheric response dT_l, l < ntrop, and the uniform potential-temperature increment dTs of the troposphere and the surface
that restore the stratospheric heating rates and the net flux at the tropopause, at fixed relative or absolute humidity.

Checker: an independent solve on the C port (rcmo_lbl_tau + rcmo_lbl_radiative_transfer) at the state the next LBL step
radiates: dT added to the radiated profile, T_surf + dTs, with fixed RH the H2O of the port's feedback at T + dT times the H2O
factor in s_H2O, and scipy's hybr for the ntrop + 1 equations.
"""
import subprocess

import numpy as np
import pytest
from scipy.optimize import root

from conftest import GOLDEN, table_path  # noqa: F401
from test_gpu_climate_response import NTROP_CYCLE, newton_matrix, ntrop_of
from test_gpu_diagnostics import feedback, status_of
from test_gpu_lbl_diagnostics import case, make, port_rt, port_tau  # noqa: F401 (case is a fixture)
from test_gpu_lbl_flux_jacobian import lbl_driver_case
from test_gpu_lbl_radiative_kernels import Port, case200, solver  # noqa: F401 (case200 is a fixture)

pytestmark = pytest.mark.gpu

NLAY, NLEV = 20, 21
CO2_2X, CO2_4X = [1.0, 2.0, 1.0, 1.0, 1.0], [1.0, 4.0, 1.0, 1.0, 1.0]
KEYS = ("F", "dT", "dTs", "E_down", "E_up", "iters")


class LblEcsColumn:
    """The climate-response problem of column col on the port: fluxes(x) at x = (dT_0 .. dT_{m-1}, dTs), None: the base."""

    def __init__(self, P, c, col, f, fixed_rh, m):
        self.P, self.c, self.col, self.f, self.fixed_rh, self.m = P, c, col, f, fixed_rh, m
        pl = c["pl"]
        self.player = (pl[:-1] + pl[1:]) / 2.0
        self.conv = (1000.0 / self.player) ** (2.0 / 7.0)

    def profile(self, x):
        d = np.zeros(NLAY)
        d[:self.m] = x[:self.m]
        d[self.m:] = x[self.m] / self.conv[self.m:]
        return d

    def fluxes(self, x=None):
        P, col = self.P, self.col
        T = P.T[col].copy()
        if x is None:
            return port_rt(P.port, P.p, port_tau(P.port, self.c, P.h2o, col, None), P.lo, P.hi, T, P.Ts[col])
        d = self.profile(x)
        h2o = P.h2o.copy()
        if self.fixed_rh:
            h2o[col] = feedback(P.port, T + d, self.c["st"]["rel_hum"][col], self.player)
        tau = port_tau(P.port, self.c, h2o, col, self.f)
        return port_rt(P.port, P.p, tau, P.lo, P.hi, T + d, P.Ts[col] + x[self.m])

    def residual(self, x):
        m = self.m
        Ed0, Eu0, dE0 = self.base
        Ed, Eu, dE = self.fluxes(x)
        return np.append(dE[:m] - dE0[:m], (Ed[m] - Eu[m]) - (Ed0[m] - Eu0[m]))

    def solve(self):
        self.base = self.fluxes()
        x = root(self.residual, np.zeros(self.m + 1), method="hybr", options=dict(xtol=1e-14)).x
        assert np.abs(self.residual(x)).max() <= 1e-10, (self.m, self.residual(x))
        Ed0, Eu0, _ = self.base
        Ed1, Eu1, _ = self.fluxes(np.zeros(self.m + 1))
        N0, N1, m = Ed0 - Eu0, Ed1 - Eu1, self.m
        return self.profile(x), x[m], np.array([N1[0] - N0[0], N1[m] - N0[m]])


# ---- 1. against an independent solve on the port ------------------------------------------------------------------------------
@pytest.mark.parametrize("steps,fixed_rh", [(3, True), (3, False), (0, False)], ids=["rh", "q", "q_step0"])
@pytest.mark.parametrize("f", [CO2_2X, CO2_4X], ids=["2xCO2", "4xCO2"])
def test_response_equals_the_port_solution(rcm, port, case, steps, fixed_rh, f):
    s = solver(rcm, case)
    if steps:
        s.advance(steps)
    ntrop = ntrop_of(s.ncol)
    d = s.lbl_climate_response(f, ntrop, fixed_rh=fixed_rh, tol=1e-9)
    assert np.all(d["converged"]), d["iters"]
    P = Port(port, case, s.get_state(), steps, None)
    s.close()
    for col in range(10):
        m = ntrop[col]
        pc = LblEcsColumn(P, case, col, f, fixed_rh, m)
        dT, dTs, F = pc.solve()
        assert np.abs(d["dT"][col] - dT).max() <= 1e-6, (col, m, d["dT"][col] - dT)
        assert abs(d["dTs"][col] - dTs) <= 1e-6, (col, m, d["dTs"][col] - dTs)
        assert np.abs(d["F"][col] - F).max() <= 1e-8, (col, m, d["F"][col] - F)
        assert np.abs(pc.residual(np.append(d["dT"][col, :m], d["dTs"][col]))).max() <= 1e-8, col
    print(f"steps {steps}, fixed_rh {fixed_rh}, CO2 x{f[1]:g}: iters {np.bincount(d['iters'])}, dTs {d['dTs'].mean():.4f}")


# ---- 2. exact cases -----------------------------------------------------------------------------------------------------------
def test_exact_cases(rcm, case):
    s = make(rcm, case)
    s.advance(2)
    n = s.ncol
    base = s.lbl_diagnose_fluxes()
    for rh in (True, False):
        d = s.lbl_climate_response([1, 1, 1, 1, 1], 7, fixed_rh=rh)
        assert np.all(d["iters"] == 0) and np.all(d["dT"] == 0.0) and np.all(d["dTs"] == 0.0) and np.all(d["F"] == 0.0)
        assert np.array_equal(d["E_down"], base["E_down"]) and np.array_equal(d["E_up"], base["E_up"])
    k = np.arange(n)
    ntrop = np.array([NTROP_CYCLE[c % len(NTROP_CYCLE)] + c % 3 for c in k])
    tol = 1e-6
    for f in (CO2_4X, [1.5, 1, 0.5, 2, 3]):
        pert = s.lbl_diagnose_fluxes(vmr_scale=f)
        Nb, Np = base["E_down"] - base["E_up"], pert["E_down"] - pert["E_up"]
        d = s.lbl_climate_response(f, ntrop, tol=tol)
        a = s.lbl_adjusted_forcing(f, ntrop)
        assert np.array_equal(d["F"], a["F"][:, :2])
        assert np.array_equal(d["F"][:, 0], Np[:, 0] - Nb[:, 0]) and np.array_equal(d["F"][:, 1], Np[k, ntrop] - Nb[k, ntrop])
        assert np.all(d["converged"]), d["iters"]
        Na = d["E_down"] - d["E_up"]
        assert np.all(np.abs(Na[:, 0] - Nb[:, 0]) <= (ntrop + 1) * tol + 1e-10)
    # one Newton update: a NumPy solve of A assembled from lbl_flux_jacobian at iterate 0
    g = s.get_state()
    for rh in (True, False):
        one = s.lbl_climate_response(CO2_4X, ntrop, fixed_rh=rh, tol=1e-12, max_iter=1)
        assert np.all(one["iters"] == -1)
        fj = s.lbl_flux_jacobian(vmr_scale=CO2_4X)
        p4 = s.lbl_diagnose_fluxes(vmr_scale=CO2_4X)
        pl = case["pl"]
        conv = (1000.0 / ((pl[:-1] + pl[1:]) / 2.0)) ** (2.0 / 7.0)
        for c in k:
            m = ntrop[c]
            Tb = np.sort(g["Tlayer"][c] * conv)[::-1] / conv
            A = newton_matrix(fj["J"][c], fj["dE_jac"][c], Tb, m, rh, conv)
            r = np.append(p4["dE"][c, :m] - base["dE"][c, :m],
                          (p4["E_down"][c, m] - p4["E_up"][c, m]) - (base["E_down"][c, m] - base["E_up"][c, m]))
            delta = np.linalg.solve(A, -r)
            got = np.append(one["dT"][c, :m], one["dTs"][c])
            assert np.abs(got - delta).max() <= 1e-12 * np.abs(delta).max(), (c, m, got - delta)
    s.close()


# ---- 3. physics and determinism -----------------------------------------------------------------------------------------------
def test_physics(rcm, case):
    s = make(rcm, case)
    s.advance(3)
    rh = s.lbl_climate_response(CO2_2X, 4)
    q = s.lbl_climate_response(CO2_2X, 4, fixed_rh=False)
    assert np.all(rh["converged"]) and np.all(q["converged"])
    print(f"LBL dTs 2xCO2: fixed RH {rh['dTs'].mean():.4f} K, fixed q {q['dTs'].mean():.4f} K")
    assert q["dTs"].mean() > 0.0 and rh["dTs"].mean() > q["dTs"].mean()
    assert rh["dT"][:, 0].mean() < 0.0
    s.close()


def test_three_chunks(rcm, case200):
    """16,400 columns = 8,192 + 8,192 + 16: whole range = each chunk alone = single columns."""
    c, n, ch = case200, 16400, 8192
    s = make(rcm, c, 1.0, rep=n // c["ncol"] + 1, n=n)
    s.advance(1)
    ntrop = (np.arange(n) * 7) % 20
    whole = s.lbl_climate_response(CO2_4X, ntrop, tol=1e-9)
    assert whole["converged"].mean() > 0.99
    for c0 in (0, ch, 2 * ch):
        part = s.lbl_climate_response(CO2_4X, ntrop[c0:c0 + ch], col0=c0, ncol=min(ch, n - c0), tol=1e-9)
        for k in KEYS:
            assert np.array_equal(whole[k][c0:c0 + ch], part[k]), (c0, k)
    for col in (0, 8191, 8192, 16383, 16384, 16399):
        one = s.lbl_climate_response(CO2_4X, ntrop[col:col + 1], col0=col, ncol=1, tol=1e-9)
        for k in KEYS:
            assert np.array_equal(whole[k][col:col + 1], one[k]), (col, k)
    s.close()


def test_the_call_changes_nothing(rcm, case, tmp_path):
    a, b = make(rcm, case), make(rcm, case)
    for s in (a, b):
        s.advance(2)
    b.lbl_climate_response(CO2_2X, 4)
    b.lbl_climate_response([1.5, 2, 0.5, 1, 1], np.arange(a.ncol) % 20, fixed_rh=False)
    sa, sb = a.advance(2), b.advance(2)
    assert np.array_equal(sa, sb)
    ga, gb = a.get_state(), b.get_state()
    for k in ga:
        assert np.array_equal(ga[k], gb[k]), k
    a.save_checkpoint(str(tmp_path / "a.ckpt"))
    b.save_checkpoint(str(tmp_path / "b.ckpt"))
    assert open(tmp_path / "a.ckpt", "rb").read() == open(tmp_path / "b.ckpt", "rb").read()
    a.close()
    b.close()


# ---- 4. errors ----------------------------------------------------------------------------------------------------------------
def test_errors_leave_the_solver_usable(rcm, case):
    s = make(rcm, case)
    n = s.ncol
    for col0, ncol in ((-1, 3), (0, 0), (n, 2), (0, n + 1)):
        assert status_of(rcm, lambda: s.lbl_climate_response(CO2_2X, np.zeros(max(ncol, 0), int), False, col0, ncol)) == 1
    for bad in (-1.0, np.nan, np.inf):
        assert status_of(rcm, lambda: s.lbl_climate_response([1.0, bad, 1.0, 1.0, 1.0], 4, False)) == 1, bad
    nt = np.full(n, 4)
    nt[5] = 20
    assert status_of(rcm, lambda: s.lbl_climate_response(CO2_2X, nt, False)) == 1
    assert status_of(rcm, lambda: s.lbl_climate_response(CO2_2X, 4, False, tol=0.0)) == 1
    assert status_of(rcm, lambda: s.lbl_climate_response(CO2_2X, 4, False, max_iter=0)) == 1
    assert status_of(rcm, lambda: s.lbl_climate_response(CO2_2X, 4, True)) == 2  # fixed RH at step 0
    assert np.all(s.lbl_climate_response(CO2_2X, 4, False)["converged"])
    s.advance(1)
    assert np.all(s.lbl_climate_response(CO2_2X, 4)["converged"])
    s.close()
    r = rcm.Solver(0)
    r.set_repwvl_table_from(rcm.Table(table_path(20)))
    st = case["st"]
    r.set_columns(case["pl"], st["Tlayer"], case["Tsurf"], st["vmr9"], st["rel_hum"])
    r.advance(1)
    assert status_of(rcm, lambda: r.lbl_climate_response(CO2_2X, 4)) == 2
    r.advance(1)
    r.close()


# ---- 5. the C++ driver --------------------------------------------------------------------------------------------------------
def test_driver_lbl_response_file(rcm, tmp_path):
    dc = lbl_driver_case(rcm, tmp_path)
    exe, common, pl = dc["exe"], dc["common"], dc["pl"]
    f1 = str(tmp_path / "r1.csv")
    r = subprocess.run([exe, *common, "--out", str(tmp_path / "o1.txt"), "--lbl-response-out", f1, "--fixed-q"],
                       capture_output=True, text=True, timeout=300)
    assert r.returncode == 0, r.stderr
    s = dc["solver"]()
    d = s.lbl_climate_response(CO2_2X, 4, fixed_rh=False)
    s.close()
    dT, dTs, F = np.zeros(NLAY), 0.0, np.zeros(2)
    for c in range(d["F"].shape[0]):   # column order, then one division: the driver's arithmetic
        dT = dT + d["dT"][c]
        dTs = dTs + d["dTs"][c]
        F = F + d["F"][c]
    n = d["F"].shape[0]
    lines = open(f1).read().splitlines()
    assert lines[0] == "layer,p_layer,dT" and len(lines) == 1 + NLAY + 4
    rows = [l.split(",") for l in lines[1:]]
    assert [x[0] for x in rows] == [str(l) for l in range(NLAY)] + ["dTs", "IRF_toa", "IRF_trop", "unconverged"]
    assert np.array_equal([float(x[1]) for x in rows[:NLAY]], (pl[:NLAY] + pl[1:]) / 2.0)
    assert np.array_equal([float(x[2]) for x in rows[:NLAY]], dT / n)
    assert float(rows[NLAY][2]) == dTs / n
    assert np.array_equal([float(x[2]) for x in rows[NLAY + 1:NLAY + 3]], F / n)
    assert int(rows[-1][2]) == int(np.sum(d["iters"] < 0))
    if rcm.device_count() < 2:
        return
    f2 = str(tmp_path / "r2.csv")
    r = subprocess.run([exe, *common, "--out", str(tmp_path / "o2.txt"), "--lbl-response-out", f2, "--fixed-q", "--gpus", "2"],
                       capture_output=True, text=True, timeout=300)
    assert r.returncode == 0, r.stderr
    assert open(f1).read() == open(f2).read()
