"""Flux Jacobians of the line-by-line path (rcm_lbl_flux_jacobian / Solver.lbl_flux_jacobian): analytic derivatives of every
level's E_down and E_up of the next LBL step, and of its heating rates, in T_l, T_surf and ln q_l, against central differences
of the C port (rcmo_lbl_tau + rcmo_lbl_radiative_transfer), against the LBL radiative kernels and the flux call, column by
column, without moving the state.
"""
import ctypes as C
import os
import subprocess

import numpy as np
import pytest

from conftest import GOLDEN, table_path
from test_gpu_lbl_diagnostics import _p, case, make, port_rt  # noqa: F401 (case is a fixture)
from test_gpu_lbl_radiative_kernels import BAR, SCALED, Port, case200, series_regime, simpson_order, solver  # noqa: F401

pytestmark = pytest.mark.gpu

NLAY, NLEV, NE = 20, 21, 41
HT, HQ = 1e-4, 1e-4   # central-difference steps in T and ln q; in T small enough that few columns see the port's B jump


class JPort(Port):
    """All 42 level fluxes of one column by the port, and their central differences in the 41 entries: Port.K at 21 levels."""

    def fluxes(self, col, tau, T, Ts):
        Ed, Eu, _ = port_rt(self.port, self.p, tau, self.lo, self.hi, T, Ts)
        return np.stack([Ed, Eu])

    def J(self, col):
        """[2][21][41] central differences"""
        T, Ts = self.T[col], self.Ts[col]
        tau0 = self.tau(col, self.h2o)
        J = np.zeros((2, NLEV, NE))
        for l in range(NLAY):
            Tp, Tm = T.copy(), T.copy()
            Tp[l] += HT
            Tm[l] -= HT
            J[:, :, l] = (self.fluxes(col, tau0, Tp, Ts) - self.fluxes(col, tau0, Tm, Ts)) / (2 * HT)
            hp, hm = self.h2o.copy(), self.h2o.copy()
            hp[col, l] *= np.exp(HQ)
            hm[col, l] *= np.exp(-HQ)
            J[:, :, NLAY + 1 + l] = (self.fluxes(col, self.tau(col, hp), T, Ts) - self.fluxes(col, self.tau(col, hm), T, Ts)) / (2 * HQ)
        J[:, :, NLAY] = (self.fluxes(col, tau0, T, Ts + HT) - self.fluxes(col, tau0, T, Ts - HT)) / (2 * HT)
        return J

    def smooth(self, col):
        """True when the port's B has no jump (Simpson order, series pieces) within +-HT of any of the column's temperatures:
        then every central difference is a derivative"""
        for t in list(self.T[col]) + [self.Ts[col]]:
            if np.any(simpson_order(self.lo, self.hi, t - HT) != simpson_order(self.lo, self.hi, t + HT)):
                return False
            if np.any(series_regime(self.lo, self.hi, t - HT) != series_regime(self.lo, self.hi, t + HT)):
                return False
        return True


def assert_rows(got, ref, what, bar):
    """every row (output, level) within bar of its largest |entry|"""
    for o in range(2):
        for k in range(NLEV):
            scale = np.max(np.abs(ref[o, k]))
            err = np.max(np.abs(got[o, k] - ref[o, k]))
            assert err <= bar * scale, (what, o, k, err, scale)


def compare(P, J, cols, what, bar, want=2):
    """the first `want` smooth columns of cols against the port"""
    done = 0
    for col in cols:
        if done == want:
            break
        if not P.smooth(col):
            continue
        assert_rows(J[col], P.J(col), (what, col), bar)
        done += 1
    assert done == want, (what, done)


def structure(J, H):
    """exact zeros of every column's J, and dE_jac restated from J entry by entry"""
    Jd, Ju = J[:, 0], J[:, 1]
    assert np.all(Jd[:, 0] == 0.0) and np.all(Jd[:, :, NLAY] == 0.0)
    for k in range(NLEV):
        for l in range(NLAY):
            if l >= k:
                assert np.all(Jd[:, k, l] == 0.0) and np.all(Jd[:, k, NLAY + 1 + l] == 0.0), (k, l)
            else:
                assert np.all(Ju[:, k, l] == 0.0) and np.all(Ju[:, k, NLAY + 1 + l] == 0.0), (k, l)
    ref = Jd[:, :-1] - Jd[:, 1:] + Ju[:, 1:] - Ju[:, :-1]
    ref[:, NLAY - 1] += Jd[:, NLAY] - Ju[:, NLAY]
    assert np.array_equal(H, ref)


# ---- against the port -----------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("nwvl", [1500, 200])
@pytest.mark.parametrize("steps", [0, 3])
@pytest.mark.parametrize("scaled", [False, True])
def test_every_entry_against_port_central_differences(rcm, port, case, case200, nwvl, steps, scaled):
    """1,500 wavelengths: the Simpson branch; 200: the series of cplkavg_dev (bar as the radiative-kernel tests)."""
    c = case if nwvl == 1500 else case200
    s = solver(rcm, c)
    if steps:
        s.advance(steps)
    g = s.get_state()
    f = SCALED if scaled else None
    d = s.lbl_flux_jacobian(vmr_scale=f)
    structure(d["J"], d["dE_jac"])
    compare(JPort(port, c, g, steps, f), d["J"], range(c["ncol"]), (nwvl, steps, scaled), BAR[nwvl])
    s.close()


def test_per_column_cloud_and_solar_against_the_port(rcm, port, case):
    c = case
    s = solver(rcm, c)
    n = c["ncol"]
    tau_s = np.linspace(0.5, 4.0, n)
    s.set_column_solar(tau_s=tau_s, mu_s=np.linspace(0.3, 0.9, n), cloud_from_tau_s=True)
    s.advance(2)
    g = s.get_state()
    d = s.lbl_flux_jacobian()
    structure(d["J"], d["dE_jac"])
    compare(JPort(port, c, g, 2, None, cloud=tau_s / 2.0), d["J"], range(1, n), "cloud", 1e-6)
    s.close()


@pytest.mark.parametrize("nangle,cubes,pairs", [(20, 1, 1), (7, 1, 1)])
def test_angle_schedules_against_the_port(rcm, port, case, nangle, cubes, pairs):
    c = case
    p = rcm.default_params()
    p.nangle = nangle
    s = solver(rcm, c, p, cubes, pairs)
    s.advance(2)
    g = s.get_state()
    d = s.lbl_flux_jacobian(vmr_scale=SCALED)
    compare(JPort(port, c, g, 2, SCALED, nangle=nangle), d["J"], range(3, c["ncol"]), (nangle, cubes, pairs), 1e-6)
    s.close()


# ---- against the other LBL calls ------------------------------------------------------------------------------------------
@pytest.mark.parametrize("steps", [0, 3])
def test_rows_are_the_radiative_kernels(rcm, case, steps):
    """rows E_up[0] and E_down[20] are rcm_lbl_radiative_kernels' K: the same terms, summed per level instead of per
    wavelength"""
    s = make(rcm, case)
    if steps:
        s.advance(steps)
    for f in (None, [1.2, 2, 0.7, 1.5, 1.1]):
        J = s.lbl_flux_jacobian(vmr_scale=f)["J"]
        K = s.lbl_radiative_kernels(vmr_scale=f)["K"]
        for o, row in ((0, J[:, 1, 0]), (1, J[:, 0, NLAY])):
            scale = np.max(np.abs(K[:, o]), axis=1)
            assert np.all(np.abs(row - K[:, o]).max(axis=1) <= 1e-12 * scale), (steps, f, o)
    s.close()


def test_ln_q_sum_against_the_flux_call(rcm, case):
    """sum over l of d/dln q_l = d/dln f_H2O: central differences of lbl_diagnose_fluxes with the factor e^(+-h)"""
    s = make(rcm, case)
    s.advance(3)
    J = s.lbl_flux_jacobian()["J"]
    eps = 1e-4
    up = s.lbl_diagnose_fluxes(vmr_scale=[np.exp(eps), 1, 1, 1, 1])
    dn = s.lbl_diagnose_fluxes(vmr_scale=[np.exp(-eps), 1, 1, 1, 1])
    for o, key in ((0, "E_down"), (1, "E_up")):
        dq = (up[key] - dn[key]) / (2 * eps)
        got = J[:, o, :, NLAY + 1:].sum(axis=2)
        scale = np.max(np.abs(J[:, o]), axis=2)
        assert np.all(np.abs(got - dq) <= 1e-6 * scale + 1e-300), o
    s.close()


# ---- invariance and side effects ------------------------------------------------------------------------------------------
def test_ranges_columns_and_chunks_give_the_same_rows(rcm, case200):
    """8,200 columns: two chunks of 8,192 + 8 for the whole range"""
    c, n = case200, 8200
    s = make(rcm, c, 1.0, rep=n // c["ncol"] + 1, n=n)
    s.advance(2)
    f = [1, 1.5, 1, 2, 1.3]
    whole = s.lbl_flux_jacobian(vmr_scale=f)
    for col0, m in ((0, 24), (8190, 5), (8199, 1), (11, 1), (1000, 7200)):
        sub = s.lbl_flux_jacobian(col0=col0, ncol=m, vmr_scale=f)
        for key in ("J", "dE_jac"):
            assert np.array_equal(sub[key], whole[key][col0:col0 + m]), (key, col0)
    assert np.array_equal(whole["J"][3], whole["J"][8160 + 3])   # replicated columns
    s.close()


def test_calls_move_nothing(rcm, case, tmp_path):
    a, b = make(rcm, case), make(rcm, case)
    for s in (a, b):
        s.advance(2)
    a.lbl_flux_jacobian()
    a.lbl_flux_jacobian(vmr_scale=[1.5, 2, 0.5, 2, 2])
    a.lbl_flux_jacobian(col0=5, ncol=7, vmr_scale=[1, 3, 1, 1, 1])
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

    def call(col0=0, ncol=24, sc=None, want=True):
        scv = None if sc is None else np.ascontiguousarray(sc, dtype=np.float64)
        J = np.zeros(max(ncol, 1) * 2 * NLEV * NE)
        H = np.zeros(max(ncol, 1) * NLAY * NE)
        return L.rcm_lbl_flux_jacobian(h, C.c_int(col0), C.c_int(ncol), None if scv is None else _p(scv),
                                       _p(J) if want else None, _p(H) if want else None)

    assert call() == 0
    assert call(col0=-1) == 1 and call(col0=20, ncol=5) == 1 and call(ncol=0) == 1
    for bad in ([-1, 1, 1, 1, 1], [1, np.nan, 1, 1, 1], [1, 1, np.inf, 1, 1]):
        assert call(sc=bad) == 1
    assert call(want=False) == 0                                     # nothing wanted
    assert L.rcm_flux_jacobian(h, 0, 24, None, None, _p(np.zeros(24 * NLAY * NE))) == 2   # the repwvl call refuses LBL
    s.advance(1)
    got = s.get_state()
    for key in got:
        assert np.array_equal(got[key], ref_next[key]), key
    s.close()
    st = case["st"]
    r = rcm.Solver(0)
    r.set_repwvl_table_from(rcm.Table(table_path(10)))
    r.set_columns(case["pl"], st["Tlayer"], case["Tsurf"], st["vmr9"], st["rel_hum"])
    assert L.rcm_lbl_flux_jacobian(r._h, 0, 24, None, None, _p(np.zeros(24 * NLAY * NE))) == 2
    r.advance(1)
    r.close()
    e = rcm.Solver(0)
    e.set_lbl_tables(case["wvl"], case["tau5"], case["h2o_ref"], case["o3_ref"], 1.0)
    assert L.rcm_lbl_flux_jacobian(e._h, 0, 1, None, None, _p(np.zeros(NLAY * NE))) == 2
    e.close()
    p = rcm.default_params()
    p.species_mask = 0b111
    m = rcm.Solver(0, p)
    m.set_lbl_tables(case["wvl"], case["tau5"], case["h2o_ref"], case["o3_ref"], 1.0)
    m.set_columns(case["pl"], st["Tlayer"], case["Tsurf"], st["vmr9"], st["rel_hum"])
    assert L.rcm_lbl_flux_jacobian(m._h, 0, 24, None, None, _p(np.zeros(24 * NLAY * NE))) == 2
    m.advance(1)
    m.close()


# ---- the C++ driver -----------------------------------------------------------------------------------------------------
def lbl_driver_case(rcm, tmp_path, ncol=6, seed=77, nwvl=700):
    """the driver's LBL inputs in a directory, and the solver state they start from"""
    lbl_atm = os.path.join(GOLDEN, "column21.lbl.atm")
    atm = rcm.read_atm(lbl_atm)
    pl = atm[:, 1].copy()
    vbase = np.stack([atm[:, 4], atm[:, 5], np.full(21, 400.0), np.full(21, 1.7), np.full(21, 0.315)])
    Tlev, vlev = rcm.make_ensemble(ncol, seed, pl, atm[:, 2].copy(), vbase)
    st = rcm.init_columns(pl, Tlev, vlev)
    h2o_ref, o3_ref = st["vmr9"][0, 0].copy(), st["vmr9"][0, 2].copy()
    wvl, tau5 = rcm.make_lbl_tables(nwvl, 777, pl, h2o_ref, o3_ref)
    d = tmp_path / "lbl"
    d.mkdir()
    for k, nm in enumerate(["h2o", "co2", "o3", "ch4", "n2o"]):
        rcm.write_lbl_asc(str(d / f"lbl.{nm}.asc"), wvl, tau5[k])
    common = ["--atm", lbl_atm, "--lbl", str(d), "--ncol", str(ncol), "--seed", str(seed), "--max-steps", "2", "--steps-exact"]

    def solver_after_run():
        s = rcm.Solver(0)
        s.set_lbl_tables(wvl, tau5, h2o_ref, o3_ref, 1.0)
        s.set_columns(pl, st["Tlayer"], 288.2, st["vmr9"], st["rel_hum"])
        s.advance(2)
        return s
    return dict(pl=pl, common=common, solver=solver_after_run, exe=os.path.join(os.path.dirname(rcm.library_path()), "rcm_rce"))


def test_driver_lbl_jacobian_file(rcm, tmp_path):
    dc = lbl_driver_case(rcm, tmp_path)
    exe, common, pl = dc["exe"], dc["common"], dc["pl"]
    f1 = str(tmp_path / "j1.csv")
    r = subprocess.run([exe, *common, "--out", str(tmp_path / "o1.txt"), "--lbl-jacobian-out", f1], capture_output=True,
                       text=True, timeout=300)
    assert r.returncode == 0, r.stderr
    s = dc["solver"]()
    H = s.lbl_flux_jacobian()["dE_jac"]
    s.close()
    acc = np.zeros((NLAY, NE))
    for row in H:             # column order, then one division: the driver's arithmetic
        acc = acc + row
    mean = acc / H.shape[0]
    lines = open(f1).read().splitlines()
    head = ["layer", "p_layer"] + [f"dT_{l}" for l in range(NLAY)] + ["dT_surf"] + [f"dlnq_{l}" for l in range(NLAY)]
    assert lines[0].split(",") == head and len(lines) == NLAY + 1
    rows = np.array([[float(x) for x in l.split(",")[1:]] for l in lines[1:]])
    assert np.array_equal(rows[:, 0], (pl[:NLAY] + pl[1:]) / 2.0)
    assert np.array_equal(rows[:, 1:], mean)
    # refused with a repwvl table; --jacobian-out still refused with --lbl
    r = subprocess.run([exe, "--atm", os.path.join(GOLDEN, "column21.atm"), "--table", table_path(10), "--max-steps", "1",
                        "--lbl-jacobian-out", str(tmp_path / "x.csv")], capture_output=True, text=True)
    assert r.returncode == 1 and "--lbl-jacobian-out" in r.stderr
    r = subprocess.run([exe, *common, "--jacobian-out", str(tmp_path / "x.csv")], capture_output=True, text=True)
    assert r.returncode == 1 and "--jacobian-out" in r.stderr and "--lbl-jacobian-out" in r.stderr
    if rcm.device_count() < 2:
        pytest.skip("the --gpus 2 half needs two GPUs")
    f2 = str(tmp_path / "j2.csv")
    r = subprocess.run([exe, *common, "--out", str(tmp_path / "o2.txt"), "--lbl-jacobian-out", f2, "--gpus", "2"],
                       capture_output=True, text=True, timeout=300)
    assert r.returncode == 0, r.stderr
    assert open(f1, "rb").read() == open(f2, "rb").read()
