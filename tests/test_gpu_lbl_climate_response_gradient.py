"""Climate-response gradients of the line-by-line path (rcm_lbl_climate_response_gradient /
Solver.lbl_climate_response_gradient): the derivatives of lbl_climate_response's dTs in every species' ln VMR in every layer of
the perturbed state and in an imposed forcing term of every equation, at its solution.

Checkers as test_gpu_climate_response_gradient: lbl_flux_jacobian and lbl_flux_gradient at zero forcing (both Planck branches,
other angle schedules, both tau-clamp placements), central differences of the C port's own solve with one layer's share of
tau or one equation perturbed, uniform differences of lbl_climate_response.
"""
import ctypes as C

import numpy as np
import pytest
from scipy.optimize import root

from conftest import table_path
from test_gpu_climate_response import ntrop_of
from test_gpu_climate_response_gradient import NS, check_uniform_differences, check_zero_forcing, entries_of
from test_gpu_diagnostics import feedback, status_of
from test_gpu_lbl_climate_response import CO2_2X, CO2_4X, LblEcsColumn
from test_gpu_lbl_diagnostics import _p, case, make, port_rt  # noqa: F401 (case is a fixture)
from test_gpu_lbl_radiative_kernels import Port, case200, solver  # noqa: F401 (case200 is a fixture)

pytestmark = pytest.mark.gpu
NLAY = 20


def conv_of(c):
    pl = c["pl"]
    return (1000.0 / ((pl[:-1] + pl[1:]) / 2.0)) ** (2.0 / 7.0)


def planck_profiles(s, c):
    conv = conv_of(c)
    T = s.get_state(("Tlayer",))["Tlayer"]
    return np.array([np.sort(t * conv)[::-1] / conv for t in T])


# ---- 1. zero forcing ----------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("nwvl", [1500, 200])
@pytest.mark.parametrize("steps,fixed_rh", [(0, False), (3, True), (3, False)], ids=["q_step0", "rh", "q"])
def test_zero_forcing_against_the_jacobian_and_the_flux_gradient(rcm, case, case200, nwvl, steps, fixed_rh):
    """1,500 wavelengths: the Simpson branch of the Planck source; 200: the series"""
    c = case if nwvl == 1500 else case200
    s = solver(rcm, c)
    if steps:
        s.advance(steps)
    check_zero_forcing(s, ntrop_of(s.ncol), fixed_rh, conv_of(c), planck_profiles(s, c), lbl=True)
    s.close()


@pytest.mark.parametrize("nangle,cubes,pairs", [(7, 1, 1), (30, 0, 0)])
def test_zero_forcing_on_other_angle_schedules(rcm, case, nangle, cubes, pairs):
    """(30, 0, 0): without cube chains the exp clamps tau instead of the layer"""
    p = rcm.default_params()
    p.nangle = nangle
    s = solver(rcm, case, p, cubes, pairs)
    s.advance(2)
    check_zero_forcing(s, (np.arange(s.ncol) * 5) % 20, True, conv_of(case), planck_profiles(s, case), lbl=True)
    s.close()


def test_zero_forcing_with_column_cloud(rcm, case):
    s = solver(rcm, case)
    n = case["ncol"]
    s.set_column_solar(tau_s=np.linspace(0.5, 4.0, n), mu_s=np.linspace(0.3, 0.9, n), cloud_from_tau_s=True)
    s.advance(2)
    check_zero_forcing(s, ntrop_of(n), True, conv_of(case), planck_profiles(s, case), lbl=True)
    s.close()


# ---- 2. against central differences of the port's own solve -------------------------------------------------------------------
def port_tau_layer(port, c, h2o, col, f, pert):
    """port_tau (test_gpu_lbl_diagnostics) with species sp's share of tau in layer l scaled by fac, pert = (sp, l, fac)"""
    f = [float(x) for x in f]
    t5 = c["tau5"]
    hs = (f[0] * h2o[col]) / c["h2o_ref"]
    os_ = (f[2] * c["st"]["vmr9"][col, 2]) / c["o3_ref"]
    co2, ch4, n2o = t5[1].copy(), f[4] * t5[3], f[3] * t5[4]
    if pert is not None:
        sp, l, fac = pert
        (hs, co2, os_, n2o, ch4)[sp][..., l] *= fac
    hs, os_, co2, ch4, n2o = (np.ascontiguousarray(a) for a in (hs, os_, co2, ch4, n2o))
    tau = np.zeros((c["nwvl"], 20))
    port.lib().rcmo_lbl_tau(C.c_int(c["nwvl"]), C.c_int(20), _p(t5[0]), _p(co2), _p(t5[2]), _p(ch4), _p(n2o), _p(hs),
                            C.c_double(f[1] * 1.0), _p(os_), _p(tau))
    tau[:, 17] += 1.0
    return tau


class PerturbedLblEcsColumn(LblEcsColumn):
    pert = None
    q = None

    def fluxes(self, x=None):
        if x is None:
            return super().fluxes(None)
        P, col = self.P, self.col
        T = P.T[col].copy()
        d = self.profile(x)
        h2o = P.h2o.copy()
        if self.fixed_rh:
            h2o[col] = feedback(P.port, T + d, self.c["st"]["rel_hum"][col], self.player)
        tau = port_tau_layer(P.port, self.c, h2o, col, self.f, self.pert)
        return port_rt(P.port, P.p, tau, P.lo, P.hi, T + d, P.Ts[col] + x[self.m])

    def residual(self, x):
        r = super().residual(x)
        return r if self.q is None else r + self.q


@pytest.mark.parametrize("steps,fixed_rh", [(3, True), (3, False), (0, False)], ids=["rh", "q", "q_step0"])
@pytest.mark.parametrize("f", [CO2_2X, CO2_4X], ids=["2xCO2", "4xCO2"])
def test_against_central_differences_of_the_port(rcm, port, case, steps, fixed_rh, f):
    """five columns (ntrop 0, 2, 4, 7, 12), every species in one stratospheric and one tropospheric layer, every equation;
    h = 1e-4 in ln x, 1e-3 W/m2 in q"""
    s = solver(rcm, case)
    if steps:
        s.advance(steps)
    ntrop = ntrop_of(s.ncol)
    d = s.lbl_climate_response_gradient(f, ntrop, fixed_rh=fixed_rh, tol=1e-9)
    r = s.lbl_climate_response(f, ntrop, fixed_rh=fixed_rh, tol=1e-9)
    assert np.array_equal(d["dTs"], r["dTs"]) and np.array_equal(d["iters"], r["iters"])
    assert np.all(d["converged"]), d["iters"]
    P = Port(port, case, s.get_state(), steps, None)
    s.close()
    worst = 0.0
    for col in range(5):
        m = ntrop[col]
        pc = PerturbedLblEcsColumn(P, case, col, f, fixed_rh, m)
        pc.base = pc.fluxes()
        x0 = np.append(r["dT"][col, :m], r["dTs"][col])
        dTs = lambda: root(pc.residual, x0, method="hybr", options=dict(xtol=1e-14)).x[m]
        gx = d["dTs_dlnx"][col].ravel()
        scale = np.abs(gx).max()
        for e in entries_of(m, col)[::3] + [sp * NLAY + (m + col) % NLAY for sp in range(NS)]:
            v = []
            for fac in (np.exp(1e-4), np.exp(-1e-4)):
                pc.pert = (e // NLAY, e % NLAY, fac)
                v.append(dTs())
            pc.pert = None
            fd = (v[0] - v[1]) / 2e-4
            err = abs(gx[e] - fd) / scale
            worst = max(worst, err)
            assert err <= 1e-5, (col, m, e, gx[e], fd)
        gq = np.append(d["dTs_dF"][col, :m], d["dTs_dF"][col, NLAY])
        for i in range(m + 1):
            v = []
            for sgn in (1.0, -1.0):
                pc.q = np.zeros(m + 1)
                pc.q[i] = sgn * 1e-3
                v.append(dTs())
            pc.q = None
            err = abs(gq[i] - (v[0] - v[1]) / 2e-3) / np.abs(gq).max()
            worst = max(worst, err)
            assert err <= 1e-5, (col, m, i)
    print(f"steps {steps}, fixed_rh {fixed_rh}, CO2 x{f[1]:g}: worst error {worst:.2e} of the row's largest |entry|")


# ---- 3. uniform differences on the device --------------------------------------------------------------------------------------
@pytest.mark.parametrize("fixed_rh", [True, False], ids=["rh", "q"])
def test_species_sums_against_uniform_differences(rcm, case, fixed_rh):
    s = solver(rcm, case)
    s.advance(3)
    check_uniform_differences(s, [1.5, 2.0, 0.5, 2.0, 1.3], ntrop_of(s.ncol), fixed_rh, lbl=True)
    s.close()


# ---- 4. determinism, failures and no side effects ------------------------------------------------------------------------------
def test_ranges_chunks_and_shards_give_the_same_rows(rcm, case200):
    c, n = case200, 8200
    s = make(rcm, c, 1.0, rep=n // c["ncol"] + 1, n=n)
    s.advance(1)
    ntrop = (np.arange(n) * 7) % 20
    keys = ("dTs", "dTs_dF", "dTs_dlnx", "iters")
    whole = s.lbl_climate_response_gradient(CO2_4X, ntrop, tol=1e-9)
    assert whole["converged"].mean() > 0.99
    part = s.lbl_climate_response_gradient(CO2_4X, ntrop[4000:], col0=4000, tol=1e-9)
    for k in keys:
        assert np.array_equal(whole[k][4000:], part[k], equal_nan=k != "iters"), k
    for col in (0, 8191, 8192, n - 1):
        one = s.lbl_climate_response_gradient(CO2_4X, ntrop[col:col + 1], col0=col, ncol=1, tol=1e-9)
        for k in keys:
            assert np.array_equal(whole[k][col:col + 1], one[k], equal_nan=k != "iters"), (col, k)
    s.close()
    st, rep = c["st"], n // c["ncol"] + 1
    tile = lambda a: np.tile(a, (rep,) + (1,) * (a.ndim - 1))[8000:n]   # make()'s columns 8000 .. n - 1 alone
    shard = rcm.Solver(0)
    shard.set_lbl_tables(c["wvl"], c["tau5"], c["h2o_ref"], c["o3_ref"], 1.0)
    shard.set_columns(c["pl"], tile(st["Tlayer"]), tile(c["Tsurf"]), tile(st["vmr9"]), tile(st["rel_hum"]))
    shard.advance(1)
    sh = shard.lbl_climate_response_gradient(CO2_4X, ntrop[8000:], tol=1e-9)
    for k in keys:
        assert np.array_equal(whole[k][8000:], sh[k], equal_nan=k != "iters"), k
    shard.close()


def test_failed_columns_give_nan_rows(rcm, case):
    s = make(rcm, case)
    s.advance(1)
    n = s.ncol
    for max_iter, tol in ((1, 1e-12), (2, 1e-9)):
        d = s.lbl_climate_response_gradient(CO2_4X, ntrop_of(n), tol=tol, max_iter=max_iter)
        r = s.lbl_climate_response(CO2_4X, ntrop_of(n), tol=tol, max_iter=max_iter)
        assert np.array_equal(d["iters"], r["iters"]) and np.array_equal(d["dTs"], r["dTs"])
        bad = d["iters"] == -1
        if max_iter == 1:
            assert np.all(bad)
        for k in ("dTs_dF", "dTs_dlnx"):
            rows = d[k].reshape(n, -1)
            assert np.all(np.isnan(rows[bad])) and np.all(np.isfinite(rows[~bad])), k
    s.close()


def test_the_call_changes_nothing(rcm, case, tmp_path):
    a, b = make(rcm, case), make(rcm, case)
    for s in (a, b):
        s.advance(2)
    b.lbl_climate_response_gradient(CO2_2X, 4)
    b.lbl_climate_response_gradient([1.5, 2, 0.5, 1, 1], np.arange(a.ncol) % 20, fixed_rh=False)
    assert np.array_equal(a.advance(2), b.advance(2))
    ga, gb = a.get_state(), b.get_state()
    for k in ga:
        assert np.array_equal(ga[k], gb[k]), k
    a.save_checkpoint(str(tmp_path / "a.ckpt"))
    b.save_checkpoint(str(tmp_path / "b.ckpt"))
    assert open(tmp_path / "a.ckpt", "rb").read() == open(tmp_path / "b.ckpt", "rb").read()
    a.close()
    b.close()


def test_errors_leave_the_solver_usable(rcm, case):
    s = make(rcm, case)
    n = s.ncol
    g = s.lbl_climate_response_gradient
    for col0, ncol in ((-1, 3), (0, 0), (n, 2), (0, n + 1)):
        assert status_of(rcm, lambda: g(CO2_2X, np.zeros(max(ncol, 0), int), False, col0, ncol)) == 1
    for bad in (-1.0, np.nan, np.inf):
        assert status_of(rcm, lambda: g([1.0, bad, 1.0, 1.0, 1.0], 4, False)) == 1, bad
    nt = np.full(n, 4)
    nt[5] = 20
    assert status_of(rcm, lambda: g(CO2_2X, nt, False)) == 1
    assert status_of(rcm, lambda: g(CO2_2X, 4, False, tol=0.0)) == 1
    assert status_of(rcm, lambda: g(CO2_2X, 4, False, max_iter=0)) == 1
    assert status_of(rcm, lambda: g(CO2_2X, 4, True)) == 2  # fixed RH at step 0
    L = rcm.load_library()
    n0 = s.launch_count()
    assert L.rcm_lbl_climate_response_gradient(s._h, C.c_int(0), C.c_int(n), None, _p(np.full(n, 4, dtype=np.int32)),
                                               C.c_int(0), C.c_double(1e-6), C.c_int(20), None, None, None, None) == 0
    assert s.launch_count() == n0
    assert np.all(g(CO2_2X, 4, False)["converged"])
    s.close()
    p = rcm.default_params()
    p.species_mask = 0x1F
    m = solver(rcm, case, p)
    m.advance(1)
    assert status_of(rcm, lambda: m.lbl_climate_response_gradient(None, 4, fixed_rh=False)) == 2
    m.advance(1)
    m.close()
    r = rcm.Solver(0)
    r.set_repwvl_table_from(rcm.Table(table_path(20)))
    st = case["st"]
    r.set_columns(case["pl"], st["Tlayer"], case["Tsurf"], st["vmr9"], st["rel_hum"])
    r.advance(1)
    assert status_of(rcm, lambda: r.lbl_climate_response_gradient(CO2_2X, 4)) == 2
    r.advance(1)
    r.close()
