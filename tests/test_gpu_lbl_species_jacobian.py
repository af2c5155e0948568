"""Species Jacobians of the line-by-line path (rcm_lbl_species_jacobian / Solver.lbl_species_jacobian): analytic derivatives of
every level's E_down and E_up of the next LBL step, and of its heating rates, with respect to the ln VMR of each of the five
species in each layer, against central differences of the C port's radiative transfer (rcmo_lbl_radiative_transfer) on tau
composed in numpy with one species' share in one layer scaled by exp(+-h), against lbl_flux_jacobian and lbl_diagnose_fluxes,
without moving the state.
"""
import ctypes as C
import os
import subprocess

import numpy as np
import pytest

from conftest import GOLDEN, table_path
from test_gpu_lbl_diagnostics import _p, case, make, port_rt, port_state  # noqa: F401 (case is a fixture)
from test_gpu_lbl_flux_jacobian import lbl_driver_case
from test_gpu_lbl_radiative_kernels import case200, solver  # noqa: F401 (case200 is a fixture)
from test_gpu_species_jacobian import check_species_file, structural_zeros

pytestmark = pytest.mark.gpu

NLAY, NLEV, NS = 20, 21, 5
NE = NS * NLAY
HQ = 1e-4
SCALED = [1.5, 2.0, 0.5, 2.0, 1.3]   # every species scaled (ascending species index)


class SPort:
    """The shares of tau of one column as rcm_lbl_diagnose_fluxes composes them, and the port's fluxes of their sum."""

    def __init__(self, port, c, g, steps, f=None, nangle=30, cloud=None):
        self.port, self.c = port, c
        self.f = [1.0] * NS if f is None else [float(x) for x in f]
        self.T, self.h2o = port_state(port, c, g, steps)
        self.Ts = g["Tsurf"]
        self.lo, self.hi = port.lbl_bin_edges(c["wvl"])
        self.p = port.default_params(0.0)
        self.p.nangle = nangle
        self.cloud = cloud

    def shares(self, col):
        """[5][nwvl][20] in ascending species index (tau5 is H2O, CO2, O3, CH4, N2O; co2_factor 1)"""
        c, f, t5 = self.c, self.f, self.c["tau5"]
        hs = (f[0] * self.h2o[col]) / c["h2o_ref"]
        os_ = (f[2] * c["st"]["vmr9"][col, 2]) / c["o3_ref"]
        return np.stack([t5[0] * hs, (f[1] * 1.0) * t5[1], t5[2] * os_, f[3] * t5[4], f[4] * t5[3]])

    def fluxes(self, col, sh):
        tau = sh.sum(axis=0)
        tau[:, 17] += 1.0 if self.cloud is None else self.cloud[col]
        Ed, Eu, _ = port_rt(self.port, self.p, np.ascontiguousarray(tau), self.lo, self.hi, self.T[col], self.Ts[col])
        return np.stack([Ed, Eu])

    def J(self, col):
        """[2][21][100] central differences"""
        sh = self.shares(col)
        J = np.zeros((2, NLEV, NE))
        for s in range(NS):
            for l in range(NLAY):
                up, dn = sh.copy(), sh.copy()
                up[s, :, l] *= np.exp(HQ)
                dn[s, :, l] *= np.exp(-HQ)
                J[:, :, s * NLAY + l] = (self.fluxes(col, up) - self.fluxes(col, dn)) / (2 * HQ)
        return J


def assert_rows(got, ref, what, bar=1e-6):
    """every row (output, level) within bar of its largest |entry|"""
    for o in range(2):
        for k in range(NLEV):
            scale = np.max(np.abs(ref[o, k]))
            err = np.max(np.abs(got[o, k] - ref[o, k]))
            assert err <= bar * scale, (what, o, k, err, scale)


def heating(J):
    Jd, Ju = J[:, 0], J[:, 1]
    ref = Jd[:, :-1] - Jd[:, 1:] + Ju[:, 1:] - Ju[:, :-1]
    ref[:, NLAY - 1] += Jd[:, NLAY] - Ju[:, NLAY]
    return ref


# ---- against the port -----------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("nwvl", [1500, 200])
@pytest.mark.parametrize("steps", [0, 3])
@pytest.mark.parametrize("scaled", [False, True])
def test_every_entry_against_port_central_differences(rcm, port, case, case200, nwvl, steps, scaled):
    """1,500 wavelengths: the Simpson branch of the Planck source; 200: the series.  T is fixed, so neither branch moves."""
    c = case if nwvl == 1500 else case200
    s = solver(rcm, c)
    if steps:
        s.advance(steps)
    g = s.get_state()
    f = SCALED if scaled else None
    d = s.lbl_species_jacobian(vmr_scale=f)
    structural_zeros(d["J"])
    assert np.array_equal(d["dE_jac"], heating(d["J"]))
    P = SPort(port, c, g, steps, f)
    for col in (0, 13):
        assert_rows(d["J"][col], P.J(col), (nwvl, steps, scaled, col))
    s.close()


def test_per_column_cloud_and_solar_against_the_port(rcm, port, case):
    c = case
    s = solver(rcm, c)
    n = c["ncol"]
    tau_s = np.linspace(0.5, 4.0, n)
    s.set_column_solar(tau_s=tau_s, mu_s=np.linspace(0.3, 0.9, n), cloud_from_tau_s=True)
    s.advance(2)
    g = s.get_state()
    d = s.lbl_species_jacobian()
    P = SPort(port, c, g, 2, None, cloud=tau_s / 2.0)
    for col in (1, 20):
        assert_rows(d["J"][col], P.J(col), ("cloud", col))
    s.close()


@pytest.mark.parametrize("nangle,cubes,pairs", [(20, 1, 1), (7, 1, 1)])
def test_angle_schedules_against_the_port(rcm, port, case, nangle, cubes, pairs):
    c = case
    p = rcm.default_params()
    p.nangle = nangle
    s = solver(rcm, c, p, cubes, pairs)
    s.advance(2)
    g = s.get_state()
    d = s.lbl_species_jacobian(vmr_scale=SCALED)
    P = SPort(port, c, g, 2, SCALED, nangle=nangle)
    for col in (3, 17):
        assert_rows(d["J"][col], P.J(col), (nangle, cubes, pairs, col))
    s.close()


# ---- against the other LBL calls ------------------------------------------------------------------------------------------
@pytest.mark.parametrize("steps", [0, 3])
def test_h2o_block_equals_the_flux_jacobian(rcm, case, steps):
    s = make(rcm, case)
    if steps:
        s.advance(steps)
    for f in (None, SCALED, [1, 2, 1, 1, 1]):
        d = s.lbl_species_jacobian(vmr_scale=f)
        j = s.lbl_flux_jacobian(vmr_scale=f)
        assert np.array_equal(d["J"][..., :NLAY], j["J"][..., NLAY + 1:]), f
        assert np.array_equal(d["dE_jac"][..., :NLAY], j["dE_jac"][..., NLAY + 1:]), f
    s.close()


def test_layer_sums_against_the_flux_call(rcm, case):
    """sum_l d/dln x_{s,l} = d/dln f_s: Richardson-extrapolated central differences of lbl_diagnose_fluxes, h = 1e-3"""
    s = make(rcm, case)
    s.advance(3)
    d = s.lbl_species_jacobian()

    def D(k, h):
        f = np.ones(NS)
        f[k] = np.exp(h)
        up = s.lbl_diagnose_fluxes(vmr_scale=f)
        f[k] = np.exp(-h)
        dn = s.lbl_diagnose_fluxes(vmr_scale=f)
        return {key: (up[key] - dn[key]) / (2 * h) for key in ("E_down", "E_up", "dE")}

    h = 1e-3
    for k in range(NS):
        d1, d2 = D(k, h), D(k, h / 2)
        blk = slice(k * NLAY, (k + 1) * NLAY)
        for an_all, key in ((d["J"][:, 0], "E_down"), (d["J"][:, 1], "E_up"), (d["dE_jac"], "dE")):
            fd = (4 * d2[key] - d1[key]) / 3
            an = an_all[..., blk].sum(axis=-1)
            tol = 1e-7 * np.abs(an_all).max(axis=-1) + 1e-300
            assert np.all(np.abs(an - fd) <= tol), (k, key, np.max(np.abs(an - fd) / tol))
    s.close()


# ---- structure -----------------------------------------------------------------------------------------------------------
def test_zero_vmr_and_clamped_layers_give_zero(rcm, port, case):
    c = case
    s = make(rcm, c)   # step 0: no feedback, the H2O set here is what the step uses
    v = np.array(c["st"]["vmr9"][:, [0, 1, 2, 3, 5]], dtype=np.float64)
    zero = [(0, 4), (0, 15), (2, 1), (2, 9)]   # (species, layer): H2O and O3
    for k, l in zero:
        v[:, k, l] = 0.0
    s.update_columns(vmr_active=v)
    d = s.lbl_species_jacobian()
    for k, l in zero:
        e = k * NLAY + l
        assert np.all(d["J"][..., e] == 0.0) and np.all(d["dE_jac"][..., e] == 0.0), (k, l)
    assert np.any(d["J"][:, 1, 0, 5] != 0.0)
    # H2O and O3 x1e12: layers whose tau is clamped at every wavelength have every entry exactly 0.0
    f = [1e12, 1, 1e12, 1, 1]
    cl = s.lbl_species_jacobian(vmr_scale=f)
    g = s.get_state()
    P = SPort(port, c, g, 0, f)
    hits = 0
    for col in (0, 9):
        tau = P.shares(col).sum(axis=0)
        full = np.all(tau > 999 * np.log(2.0) * 1.001, axis=0)   # [20] layers clamped at every wavelength
        hits += full.sum()
        for l in np.nonzero(full)[0]:
            assert np.all(cl["J"][col][..., l::NLAY] == 0.0), (col, l)
    assert hits > 0
    s.close()


# ---- invariance and side effects ------------------------------------------------------------------------------------------
def test_ranges_columns_and_chunks_give_the_same_rows(rcm, case200):
    """8,200 columns: two chunks of 8,192 + 8 for the whole range"""
    c, n = case200, 8200
    s = make(rcm, c, 1.0, rep=n // c["ncol"] + 1, n=n)
    s.advance(2)
    f = [1, 1.5, 1, 2, 1.3]
    whole = s.lbl_species_jacobian(vmr_scale=f)
    for col0, m in ((0, 24), (8190, 5), (8199, 1), (11, 1), (1000, 7200)):
        sub = s.lbl_species_jacobian(col0=col0, ncol=m, vmr_scale=f)
        for key in ("J", "dE_jac"):
            assert np.array_equal(sub[key], whole[key][col0:col0 + m]), (key, col0)
    assert np.array_equal(whole["J"][3], whole["J"][8160 + 3])   # replicated columns
    s.close()


def test_calls_move_nothing(rcm, case, tmp_path):
    a, b = make(rcm, case), make(rcm, case)
    for s in (a, b):
        s.advance(2)
    a.lbl_species_jacobian()
    a.lbl_species_jacobian(vmr_scale=[1.5, 2, 0.5, 2, 2])
    a.lbl_species_jacobian(col0=5, ncol=7, vmr_scale=[1, 3, 1, 1, 1])
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
        return L.rcm_lbl_species_jacobian(h, C.c_int(col0), C.c_int(ncol), None if scv is None else _p(scv),
                                          _p(J) if want else None, _p(H) if want else None)

    assert call() == 0
    assert call(col0=-1) == 1 and call(col0=20, ncol=5) == 1 and call(ncol=0) == 1
    for bad in ([-1, 1, 1, 1, 1], [1, np.nan, 1, 1, 1], [1, 1, 1, 1, np.inf]):
        assert call(sc=bad) == 1
    assert call(want=False) == 0                                      # nothing wanted
    assert L.rcm_species_jacobian(h, 0, 24, None, None, _p(np.zeros(24 * NLAY * NE))) == 2   # the repwvl call refuses LBL
    s.advance(1)
    got = s.get_state()
    for key in got:
        assert np.array_equal(got[key], ref_next[key]), key
    s.close()
    st = case["st"]
    r = rcm.Solver(0)
    r.set_repwvl_table_from(rcm.Table(table_path(10)))
    r.set_columns(case["pl"], st["Tlayer"], case["Tsurf"], st["vmr9"], st["rel_hum"])
    assert L.rcm_lbl_species_jacobian(r._h, 0, 24, None, None, _p(np.zeros(24 * NLAY * NE))) == 2
    r.advance(1)
    r.close()
    e = rcm.Solver(0)
    e.set_lbl_tables(case["wvl"], case["tau5"], case["h2o_ref"], case["o3_ref"], 1.0)
    assert L.rcm_lbl_species_jacobian(e._h, 0, 1, None, None, _p(np.zeros(NLAY * NE))) == 2
    e.close()
    p = rcm.default_params()
    p.species_mask = 0b111
    m = rcm.Solver(0, p)
    m.set_lbl_tables(case["wvl"], case["tau5"], case["h2o_ref"], case["o3_ref"], 1.0)
    m.set_columns(case["pl"], st["Tlayer"], case["Tsurf"], st["vmr9"], st["rel_hum"])
    assert L.rcm_lbl_species_jacobian(m._h, 0, 24, None, None, _p(np.zeros(24 * NLAY * NE))) == 2
    m.advance(1)
    m.close()


# ---- the C++ driver -----------------------------------------------------------------------------------------------------
def test_driver_lbl_species_file(rcm, tmp_path):
    dc = lbl_driver_case(rcm, tmp_path)
    exe, common, pl = dc["exe"], dc["common"], dc["pl"]
    f1 = str(tmp_path / "s1.csv")
    r = subprocess.run([exe, *common, "--out", str(tmp_path / "o1.txt"), "--lbl-species-jacobian-out", f1], capture_output=True,
                       text=True, timeout=300)
    assert r.returncode == 0, r.stderr
    s = dc["solver"]()
    d = s.lbl_species_jacobian()
    s.close()
    check_species_file(f1, pl, d["J"], d["dE_jac"])
    # refused with a repwvl table; --species-jacobian-out refused with --lbl
    r = subprocess.run([exe, "--atm", os.path.join(GOLDEN, "column21.atm"), "--table", table_path(10), "--max-steps", "1",
                        "--lbl-species-jacobian-out", str(tmp_path / "x.csv")], capture_output=True, text=True)
    assert r.returncode == 1 and "--lbl-species-jacobian-out" in r.stderr
    r = subprocess.run([exe, *common, "--species-jacobian-out", str(tmp_path / "x.csv")], capture_output=True, text=True)
    assert r.returncode == 1 and "--species-jacobian-out" in r.stderr and "--lbl-species-jacobian-out" in r.stderr
    if rcm.device_count() < 2:
        pytest.skip("the --gpus 2 half needs two GPUs")
    f2 = str(tmp_path / "s2.csv")
    r = subprocess.run([exe, *common, "--out", str(tmp_path / "o2.txt"), "--lbl-species-jacobian-out", f2, "--gpus", "2"],
                       capture_output=True, text=True, timeout=300)
    assert r.returncode == 0, r.stderr
    assert open(f1, "rb").read() == open(f2, "rb").read()
