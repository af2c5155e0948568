"""Climate-response gradients (rcm_climate_response_gradient / Solver.climate_response_gradient): the derivatives of the
equilibrium surface warming dTs of climate_response in every species' ln VMR in every layer of the perturbed state and in an
imposed forcing term of every equation, by one adjoint solve of the converged Newton system and one reverse sweep.

Checkers: at zero forcing (the solution is iterate 0) the transpose solve of the Newton matrix assembled from flux_jacobian and
the flux gradient with the cotangents the call defines, bit for bit; central differences of the C port's own Newton solve with
one layer's VMR or one equation perturbed; uniform differences of climate_response along each species' factor.
"""
import ctypes as C

import numpy as np
import pytest
from scipy.optimize import root

from conftest import table_path
from test_gpu_climate_response import CO2_4X, EcsColumn, gamma, newton_matrix, ntrop_of
from test_gpu_diagnostics import CO2_2X, ensemble, feedback, solver, status_of, theta_sort

pytestmark = pytest.mark.gpu
NLAY, NLEV, NS = 20, 21, 5
VMR9_ROW = (0, 1, 2, 3, 5)   # rows of vmr9 of the species of vmr_scale (H2O, CO2, O3, N2O, CH4)


@pytest.fixture(scope="module")
def ens21(rcm):
    return ensemble(rcm, 21, 2024)


# ---- shared checks (also used by the line-by-line file) ----------------------------------------------------------------------
def adjoint_cotangents(dF, ntrop):
    """the level cotangents the call defines from its own dTs_dF: w_dE[i] = s_i, w_E_down[ntrop] = s_m, w_E_up[ntrop] = -s_m"""
    n = dF.shape[0]
    wEd, wEu = np.zeros((n, NLEV)), np.zeros((n, NLEV))
    k = np.arange(n)
    wEd[k, ntrop] = dF[:, NLAY]
    wEu[k, ntrop] = -dF[:, NLAY]
    return wEd, wEu, dF[:, :NLAY].copy()


def check_zero_forcing(s, ntrop, fixed_rh, conv, Tb, lbl=False):
    """vmr_scale None: the solution is iterate 0, at the state flux_jacobian and flux_gradient differentiate"""
    call = s.lbl_climate_response_gradient if lbl else s.climate_response_gradient
    d = call(None, ntrop, fixed_rh=fixed_rh)
    n = s.ncol
    assert np.all(d["iters"] == 0) and np.all(d["dTs"] == 0.0)
    fj = s.lbl_flux_jacobian() if lbl else s.flux_jacobian()
    dF = d["dTs_dF"]
    mag = []   # |s|^T |A| of every column: the magnitude of the terms of s^T A
    for c in range(n):
        m = ntrop[c]
        A = newton_matrix(fj["J"][c], fj["dE_jac"][c], Tb[c], m, fixed_rh, conv)
        e = np.zeros(m + 1)
        e[m] = 1.0
        ref = -np.linalg.solve(A.T, e)
        got = np.append(dF[c, :m], dF[c, NLAY])
        assert np.abs(got - ref).max() <= 1e-10 * np.abs(ref).max(), (c, m, got - ref)
        assert np.all(dF[c, m:NLAY] == 0.0) and not np.signbit(dF[c, m:NLAY]).any(), c
        mag.append(np.abs(got) @ np.abs(A))
    wEd, wEu, wdE = adjoint_cotangents(dF, ntrop)
    fg = (s.lbl_flux_gradient if lbl else s.flux_gradient)(wEd, wEu, wdE)
    assert np.array_equal(d["dTs_dlnx"].reshape(n, NS * NLAY), fg["grad"][:, NLEV:])
    # the adjoint identity s^T A = -e_m^T on the gradient's T, T_surf and ln q entries
    g = fg["grad"]
    for c in range(n):
        m = ntrop[c]
        gm = gamma(Tb[c]) if fixed_rh else np.zeros(NLAY)
        sa = np.append(g[c, :m] + gm[:m] * g[c, NLEV:NLEV + m],
                       g[c, NLAY] + ((g[c, m:NLAY] + gm[m:] * g[c, NLEV + m:NLEV + NLAY]) / conv[m:]).sum())
        sa[m] += 1.0
        assert np.all(np.abs(sa) <= 1e-9 * mag[c]), (c, m, sa, mag[c])
    return d


def check_uniform_differences(s, f, ntrop, fixed_rh, lbl=False, h=1e-3):
    """sum_l dTs_dlnx[s] against central differences of climate_response along species s's factor, at tol 1e-10"""
    grad = s.lbl_climate_response_gradient if lbl else s.climate_response_gradient
    resp = s.lbl_climate_response if lbl else s.climate_response
    d = grad(f, ntrop, fixed_rh=fixed_rh, tol=1e-10)
    assert np.all(d["converged"]), d["iters"]
    tot = d["dTs_dlnx"].sum(axis=2)
    worst = 0.0
    for sp in range(NS):
        fp, fm = np.array(f, dtype=float), np.array(f, dtype=float)
        fp[sp] *= np.exp(h)
        fm[sp] *= np.exp(-h)
        a, b = resp(fp, ntrop, fixed_rh=fixed_rh, tol=1e-10), resp(fm, ntrop, fixed_rh=fixed_rh, tol=1e-10)
        assert np.all(a["converged"]) and np.all(b["converged"])
        fd = (a["dTs"] - b["dTs"]) / (2 * h)
        err = np.abs(tot[:, sp] - fd) / np.abs(tot).max(axis=1)
        worst = max(worst, err.max())
        assert np.all(err <= 1e-5), (sp, err.max())
    print(f"uniform differences (h {h:g}): worst error {worst:.2e} of the row's largest |entry|")


# ---- 1. zero forcing: the Newton matrix and the flux gradient -----------------------------------------------------------------
@pytest.mark.parametrize("nwvl", [20, 100])
@pytest.mark.parametrize("nsteps,fixed_rh", [(0, False), (3, True), (3, False)], ids=["q_step0", "rh", "q"])
def test_zero_forcing_against_the_jacobian_and_the_flux_gradient(rcm, port, ens21, nwvl, nsteps, fixed_rh):
    s = solver(rcm, nwvl, ens21)
    if nsteps:
        s.advance(nsteps)
    conv = ens21["conv"]
    T = s.get_state(("Tlayer",))["Tlayer"]
    Tb = np.array([theta_sort(port, t, conv) for t in T])
    check_zero_forcing(s, ntrop_of(s.ncol), fixed_rh, conv, Tb)
    s.close()


def test_zero_forcing_with_column_cloud(rcm, port, ens21):
    s = solver(rcm, 100, ens21)
    n = s.ncol
    s.set_column_solar(tau_s=np.linspace(0.5, 4.0, n), mu_s=np.linspace(0.3, 0.9, n), cloud_from_tau_s=True)
    s.advance(2)
    conv = ens21["conv"]
    T = s.get_state(("Tlayer",))["Tlayer"]
    Tb = np.array([theta_sort(port, t, conv) for t in T])
    check_zero_forcing(s, (np.arange(n) * 3) % 20, True, conv, Tb)
    s.close()


# ---- 2. against central differences of the port's own solve -------------------------------------------------------------------
class PerturbedEcsColumn(EcsColumn):
    """EcsColumn with one layer's VMR of the perturbed state scaled (row, layer, factor) and a forcing term q on the residual"""

    pert = None
    q = None

    def fluxes(self, x=None):
        if x is None:
            return super().fluxes(None)
        d = self.profile(x)
        v = self.v1.copy()
        if self.fixed_rh:
            v[0] = feedback(self.port, self.Trad + d, self.rel_hum, self.player) * self.f[0]
        if self.pert is not None:
            row, l, fac = self.pert
            v[row, l] = v[row, l] * fac
        tau, _, _ = self.port.read_tau(self.tab, self.pl, self.tau_T + d, v, tau_s=self.tau_s)
        return self.port.radiative_transfer(tau, self.tab["wvl"], self.tab["weight"], self.Trad + d, self.Tsurf + x[self.m], 0.0)

    def residual(self, x):
        r = super().residual(x)
        return r if self.q is None else r + self.q

    def dTs(self, x0):
        return root(self.residual, x0, method="hybr", options=dict(xtol=1e-14)).x[self.m]


def port_derivatives(col, x0, entries, h_lnx=1e-4, h_q=1e-3):
    """central differences of the port's dTs: {e: d/dln x_e} for e in entries, and d/dq_i for every equation"""
    m = col.m
    col.base = col.fluxes()
    out_x, out_q = {}, np.zeros(m + 1)
    for e in entries:
        sp, l = divmod(e, NLAY)
        v = []
        for fac in (np.exp(h_lnx), np.exp(-h_lnx)):
            col.pert = (VMR9_ROW[sp], l, fac)
            v.append(col.dTs(x0))
        col.pert = None
        out_x[e] = (v[0] - v[1]) / (2 * h_lnx)
    for i in range(m + 1):
        v = []
        for sgn in (1.0, -1.0):
            col.q = np.zeros(m + 1)
            col.q[i] = sgn * h_q
            v.append(col.dTs(x0))
        col.q = None
        out_q[i] = (v[0] - v[1]) / (2 * h_q)
    return out_x, out_q


def entries_of(m, c):
    """every species in one stratospheric (if any) and two tropospheric layers, varied with the column"""
    layers = ([c % m] if m else []) + [m + (c % (NLAY - m)), NLAY - 1 - (c % 3)]
    return [sp * NLAY + l for sp in range(NS) for l in layers]


@pytest.mark.parametrize("nsteps,fixed_rh", [(3, True), (3, False), (0, False)], ids=["rh", "q", "q_step0"])
@pytest.mark.parametrize("f", [CO2_2X, CO2_4X], ids=["2xCO2", "4xCO2"])
def test_against_central_differences_of_the_port(rcm, port, ens21, nsteps, fixed_rh, f):
    """21 columns, Reduced20, ntrop cycling over 0, 2, 4, 7, 12; h = 1e-4 in ln x, 1e-3 W/m2 in q"""
    tab = port.load_rcmtab(table_path(20))
    s = solver(rcm, 20, ens21)
    if nsteps:
        s.advance(nsteps)
    ntrop = ntrop_of(s.ncol)
    d = s.climate_response_gradient(f, ntrop, fixed_rh=fixed_rh, tol=1e-9)
    r = s.climate_response(f, ntrop, fixed_rh=fixed_rh, tol=1e-9)
    assert np.array_equal(d["dTs"], r["dTs"]) and np.array_equal(d["iters"], r["iters"])
    assert np.all(d["converged"]), d["iters"]
    g = s.get_state(("Tlayer", "Tsurf"))
    s.close()
    worst = 0.0
    for c in range(ens21["Tlayer"].shape[0]):
        m = ntrop[c]
        col = PerturbedEcsColumn(port, tab, ens21, g["Tlayer"][c], ens21["vmr9"][c], ens21["rel_hum"][c], g["Tsurf"][c],
                                 nsteps == 0, f, fixed_rh, m)
        x0 = np.append(r["dT"][c, :m], r["dTs"][c])
        ex = entries_of(m, c)
        fx, fq = port_derivatives(col, x0, ex)
        gx = d["dTs_dlnx"][c].ravel()
        scale = np.abs(gx).max()
        for e in ex:
            err = abs(gx[e] - fx[e]) / scale
            worst = max(worst, err)
            assert err <= 1e-5, (c, m, e, gx[e], fx[e])
        gq = np.append(d["dTs_dF"][c, :m], d["dTs_dF"][c, NLAY])
        err = np.abs(gq - fq).max() / np.abs(gq).max()
        worst = max(worst, err)
        assert err <= 1e-5, (c, m, gq, fq)
    print(f"nsteps {nsteps}, fixed_rh {fixed_rh}, CO2 x{f[1]:g}: worst error {worst:.2e} of the row's largest |entry|")


# ---- 3. uniform differences on the device --------------------------------------------------------------------------------------
@pytest.mark.parametrize("fixed_rh", [True, False], ids=["rh", "q"])
def test_species_sums_against_uniform_differences(rcm, ens21, fixed_rh):
    s = solver(rcm, 100, ens21)
    s.advance(3)
    check_uniform_differences(s, CO2_2X, ntrop_of(s.ncol), fixed_rh)
    s.close()


# ---- 4. determinism, failures and no side effects ------------------------------------------------------------------------------
def test_ranges_chunks_and_shards_give_the_same_rows(rcm):
    ncol = 8200
    st = ensemble(rcm, ncol, 13)
    s = solver(rcm, 100, st)
    s.advance(2)
    ntrop = (np.arange(ncol) * 7) % 20
    keys = ("dTs", "dTs_dF", "dTs_dlnx", "iters")
    whole = s.climate_response_gradient(CO2_2X, ntrop)
    assert whole["converged"].mean() > 0.99
    part = s.climate_response_gradient(CO2_2X, ntrop[4000:], col0=4000)
    for k in keys:
        assert np.array_equal(whole[k][4000:], part[k], equal_nan=k != "iters"), k
    for c in (0, 15, 16, 8191, 8192, ncol - 1):
        one = s.climate_response_gradient(CO2_2X, ntrop[c:c + 1], col0=c, ncol=1)
        for k in keys:
            assert np.array_equal(whole[k][c:c + 1], one[k], equal_nan=k != "iters"), (c, k)
    s.close()
    shard = solver(rcm, 100, st, sl=slice(8184, ncol))
    shard.advance(2)
    sh = shard.climate_response_gradient(CO2_2X, ntrop[8184:])
    for k in keys:
        assert np.array_equal(whole[k][8184:], sh[k], equal_nan=k != "iters"), k
    shard.close()


def test_failed_columns_give_nan_rows(rcm, ens21):
    s = solver(rcm, 20, ens21)
    s.advance(1)
    for max_iter, tol in ((1, 1e-12), (2, 1e-9)):
        d = s.climate_response_gradient(CO2_4X, ntrop_of(s.ncol), fixed_rh=True, tol=tol, max_iter=max_iter)
        r = s.climate_response(CO2_4X, ntrop_of(s.ncol), fixed_rh=True, tol=tol, max_iter=max_iter)
        assert np.array_equal(d["iters"], r["iters"]) and np.array_equal(d["dTs"], r["dTs"])
        bad = d["iters"] == -1
        if max_iter == 1:
            assert np.all(bad)
        for k in ("dTs_dF", "dTs_dlnx"):
            rows = d[k].reshape(s.ncol, -1)
            assert np.all(np.isnan(rows[bad])) and np.all(np.isfinite(rows[~bad])), k
    s.close()


def test_the_call_changes_nothing(rcm, ens21, tmp_path):
    a, b = solver(rcm, 20, ens21), solver(rcm, 20, ens21)
    for x in (a, b):
        x.advance(2)
    b.climate_response_gradient(CO2_2X, 4)
    b.climate_response_gradient(CO2_4X, np.arange(21) % 20, fixed_rh=False)
    b.climate_response_gradient(CO2_2X, 6, col0=3, ncol=5)
    assert np.array_equal(a.advance(2), b.advance(2))
    ga, gb = a.get_state(), b.get_state()
    for k in ga:
        assert np.array_equal(ga[k], gb[k]), k
    a.save_checkpoint(str(tmp_path / "a.ckpt"))
    b.save_checkpoint(str(tmp_path / "b.ckpt"))
    assert open(tmp_path / "a.ckpt", "rb").read() == open(tmp_path / "b.ckpt", "rb").read()
    for x in (a, b):
        x.close()


def test_errors_leave_the_solver_usable(rcm, ens21):
    s = solver(rcm, 20, ens21)
    g = s.climate_response_gradient
    for col0, ncol in ((-1, 3), (0, 0), (20, 2), (0, 22)):
        assert status_of(rcm, lambda: g(CO2_2X, np.zeros(max(ncol, 0), int), False, col0, ncol)) == 1
    for bad in (-1.0, np.nan, np.inf):
        assert status_of(rcm, lambda: g([1.0, bad, 1.0, 1.0, 1.0], 4, False)) == 1, bad
    for bad in (-1, 20):
        nt = np.full(21, 4)
        nt[17] = bad
        assert status_of(rcm, lambda: g(CO2_2X, nt, False)) == 1, bad
    for tol in (0.0, -1e-6, np.nan, np.inf):
        assert status_of(rcm, lambda: g(CO2_2X, 4, False, tol=tol)) == 1, tol
    assert status_of(rcm, lambda: g(CO2_2X, 4, False, max_iter=0)) == 1
    assert status_of(rcm, lambda: g(CO2_2X, 4, True)) == 2   # fixed RH at step 0
    L = rcm.load_library()
    nt = np.full(21, 4, dtype=np.int32)
    args = (s._h, C.c_int(0), C.c_int(21), None)
    assert L.rcm_climate_response_gradient(*args, None, C.c_int(0), C.c_double(1e-6), C.c_int(20), None,
                                           rcm.capi._p(np.zeros((21, 21))), None, None) == 1
    n0 = s.launch_count()
    assert L.rcm_climate_response_gradient(*args, rcm.capi._p(nt), C.c_int(0), C.c_double(1e-6), C.c_int(20),
                                           None, None, None, None) == 0
    assert s.launch_count() == n0
    assert np.all(g(CO2_2X, 4, False)["converged"])
    s.close()

    for mask in (0x0F, 0x3E, 0x1F):   # 0x1F: five active species with H2O, not the default; refused by the mask check
        p = rcm.default_params()
        p.species_mask = mask
        m = solver(rcm, 20, ens21, params=p)
        m.advance(1)
        assert status_of(rcm, lambda: m.climate_response_gradient(None, 4, fixed_rh=False)) == 2, mask
        m.advance(1)
        m.close()
    lb = rcm.Solver(0)
    wvl, tau5 = rcm.make_lbl_tables(300, 7, ens21["plevel"], ens21["vmr9"][0, 0], ens21["vmr9"][0, 2])
    lb.set_lbl_tables(wvl, tau5, ens21["vmr9"][0, 0], ens21["vmr9"][0, 2])
    lb.set_columns(ens21["plevel"], ens21["Tlayer"], ens21["Tsurf"], ens21["vmr9"], ens21["rel_hum"])
    lb.advance(1)
    assert status_of(rcm, lambda: lb.climate_response_gradient(CO2_2X, 4)) == 2
    lb.close()
