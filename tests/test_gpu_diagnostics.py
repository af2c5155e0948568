"""The diagnostic radiation call (rcm_diagnose_fluxes / Solver.diagnose_fluxes): the fluxes the next step of the resident
ensemble would compute, per wavelength, optionally with scaled VMRs, without changing anything.

Checker: the C port of the reference (oracle/rcm_oracle.c).  Its radiative_transfer called with ONE wavelength (nwvl = 1
and that wavelength's wvl, weight and tau row) is exactly that wavelength's contribution in the reference's arithmetic;
"the next step's inputs" are built with the port's theta_sort and water_vapor_feedback (main.cpp:536-540, :281-289).
"""
import ctypes as C
import os
import subprocess

import numpy as np
import pytest

from conftest import GOLDEN, table_path

pytestmark = pytest.mark.gpu
NLAY, NLEV = 20, 21
OPT_PATH, OPT_MULTI = 5, 6
CO2_2X = [1.0, 2.0, 1.0, 1.0, 1.0]  # active species of the default mask: H2O, CO2, O3, N2O, CH4


# ---- the port's step-preparation routines ---------------------------------------------------------------------------
def theta_sort(port, T, conv):
    out = np.array(T, dtype=np.float64, order="C")
    port.lib().rcmo_theta_sort(C.c_int(NLAY), port._p(out), port._p(np.ascontiguousarray(conv, dtype=np.float64)))
    return out


def feedback(port, T, rel_hum, player):
    h2o = np.zeros(NLAY)
    f = lambda a: port._p(np.ascontiguousarray(a, dtype=np.float64))
    port.lib().rcmo_water_vapor_feedback(C.c_int(NLAY), f(T), f(rel_hum), f(player), port._p(h2o))
    return h2o


def next_step_inputs(port, tab, pl, st, T, vmr9, first, h2o_scale=1.0, co2_scale=1.0, tau_s=2.0):
    """tau [nwvl][20] and the sorted profile the next step of one column radiates with (main.cpp:500-504, :536-572)."""
    v9 = np.array(vmr9, dtype=np.float64)
    Ts = theta_sort(port, T, st["conv"])
    if first:
        tau_T = np.array(T, dtype=np.float64)  # tau of the initial, unsorted profile
    else:
        tau_T = Ts
        v9[0] = feedback(port, Ts, st["rel_hum_c"], st["player"])
    v9[0] = v9[0] * h2o_scale
    v9[1] = v9[1] * co2_scale
    tau, _, _ = port.read_tau(tab, pl, tau_T, v9, tau_s=tau_s)
    return tau, Ts


def per_wavelength(port, tab, tau, T, Tsurf, solar):
    nw = tab["wvl"].size
    dn, up = np.zeros((nw, NLEV)), np.zeros((nw, NLEV))
    for w in range(nw):
        dn[w], up[w], _ = port.radiative_transfer(tau[w:w + 1], tab["wvl"][w:w + 1], tab["weight"][w:w + 1], T, Tsurf, solar)
    return dn, up


# ---- fixtures ---------------------------------------------------------------------------------------------------------
def ensemble(rcm, ncol, seed):
    atm = rcm.read_atm(os.path.join(GOLDEN, "column21.atm"))
    pl = atm[:, 1].copy()
    Tlev, vlev = rcm.make_ensemble(ncol, seed, pl, atm[:, 2].copy(), atm[:, 4:9].T.copy())
    st = rcm.init_columns(pl, Tlev, vlev)
    st["plevel"], st["Tsurf"] = pl, Tlev[:, 20].copy()
    return st


def solver(rcm, n, st, sl=slice(None), params=None):
    s = rcm.Solver(0, params)
    s.set_repwvl_table_from(rcm.Table(table_path(n)))
    s.set_columns(st["plevel"], st["Tlayer"][sl], st["Tsurf"][sl], st["vmr9"][sl], st["rel_hum"][sl])
    return s


@pytest.fixture(scope="module")
def ens21(rcm):
    return ensemble(rcm, 21, 2024)


@pytest.fixture(scope="module")
def ens5000(rcm):
    return ensemble(rcm, 5000, 77)


def scale_of(ref):
    return np.max(np.abs(ref), axis=tuple(range(1, ref.ndim)), keepdims=True)


def check_against_port(port, s, st, tab, nsteps_done, solar_col=None, tau_s=None, h2o_scale=1.0):
    vs = None if h2o_scale == 1.0 else [h2o_scale, 1.0, 1.0, 1.0, 1.0]
    d = s.diagnose_fluxes(vmr_scale=vs)
    g = s.get_state(("Tlayer", "Tsurf"))
    ncol = s.ncol
    for c in range(ncol):
        cs = dict(st, rel_hum_c=st["rel_hum"][c])
        tau, Tsorted = next_step_inputs(port, tab, st["plevel"], cs, g["Tlayer"][c], st["vmr9"][c], nsteps_done == 0,
                                        h2o_scale=h2o_scale, tau_s=2.0 if tau_s is None else tau_s[c])
        solar = s.params.solar_irr if solar_col is None else solar_col[c]
        dn, up = per_wavelength(port, tab, tau, Tsorted, g["Tsurf"][c], solar)
        sc = max(np.abs(dn).max(), np.abs(up).max())
        assert np.abs(d["E_down_spec"][c] - dn).max() <= 1e-10 * sc, c
        assert np.abs(d["E_up_spec"][c] - up).max() <= 1e-10 * sc, c
        Ed, Eu, dE = port.radiative_transfer(tau, tab["wvl"], tab["weight"], Tsorted, g["Tsurf"][c], solar)
        sb = np.abs(Eu).max()
        for got, ref in ((d["E_down"][c], Ed), (d["E_up"][c], Eu), (d["dE"][c], dE)):
            assert np.abs(got - ref).max() <= 1e-10 * sb, c
    return d


# ---- 1. every wavelength against the port --------------------------------------------------------------------------
@pytest.mark.parametrize("nsteps", [3, 0])
def test_each_wavelength_equals_the_port(rcm, port, ens21, nsteps):
    """21 columns (a ragged second tile), Reduced20: after three steps (feedback and re-sort) and at step 0 (tau of the
    initial, unsorted profile)."""
    tab = port.load_rcmtab(table_path(20))
    s = solver(rcm, 20, ens21)
    if nsteps:
        s.advance(nsteps)
    d = check_against_port(port, s, ens21, tab, nsteps)
    assert d["E_down_spec"].shape == (21, 20, NLEV) and np.all(d["E_down_spec"][:, :, 0] == 0.0)
    s.close()


# ---- 2. golden anchors -----------------------------------------------------------------------------------------------
def test_golden_olr_and_2xco2_forcing(rcm, golden):
    """Base column of column21.atm, Reduced100, step 0: SURVEY 8(c)'s OLR, and the 2xCO2 instantaneous forcing of the port
    (CO2 row x 2) at the top and at the surface."""
    s = rcm.Solver(0)
    s.set_repwvl_table_from(rcm.Table(table_path(100)))
    g = golden
    s.set_columns(g["plevel"], g["Tlayer"][:1], g["Tsurf"][:1], g["vmr9"][:1], g["rel_hum"][:1])
    one = s.diagnose_fluxes()
    two = s.diagnose_fluxes(vmr_scale=CO2_2X)
    olr = one["E_up"][0, 0]
    assert abs(olr - 246.6782921988) <= 1e-10 * 246.6782921988
    irf_spec = one["E_up_spec"][0, :, 0] - two["E_up_spec"][0, :, 0]
    irf = olr - two["E_up"][0, 0]
    assert abs(irf - 2.977632560369) < 1e-9, irf
    assert abs(irf_spec.sum() - irf) < 1e-9
    assert abs((two["E_down"][0, 20] - one["E_down"][0, 20]) - 0.7239591259) < 1e-8
    s.close()


# ---- 3. internal consistency -----------------------------------------------------------------------------------------
def test_broadband_is_the_sequential_sum_of_the_spectrum(rcm, ens21):
    s = solver(rcm, 100, ens21)
    s.advance(2)
    d = s.diagnose_fluxes()
    for k, sk in (("E_down", "E_down_spec"), ("E_up", "E_up_spec")):
        acc = np.zeros((s.ncol, NLEV))
        for w in range(s.nwvl):
            acc = acc + d[sk][:, w]
        assert np.array_equal(acc, d[k]), k
    Ed, Eu = d["E_down"], d["E_up"]
    dE = Ed[:, :NLAY] - Ed[:, 1:] + Eu[:, 1:] - Eu[:, :NLAY]  # main.cpp:337-341
    dE[:, NLAY - 1] = dE[:, NLAY - 1] + (s.params.solar_irr + Ed[:, NLAY] - Eu[:, NLAY])
    assert np.array_equal(dE, d["dE"])
    ones = s.diagnose_fluxes(vmr_scale=np.ones(5))
    for k in d:
        assert np.array_equal(ones[k], d[k]), k
    bb = s.diagnose_fluxes(spectral=False)
    assert set(bb) == {"E_down", "E_up", "dE"} and all(np.array_equal(bb[k], d[k]) for k in bb)
    s.close()


# ---- 4. the step that follows -----------------------------------------------------------------------------------------
@pytest.mark.parametrize("nsteps", [0, 2])
def test_fluxes_are_those_of_the_next_step(rcm, ens21, nsteps):
    s = solver(rcm, 100, ens21)
    if nsteps:
        s.advance(nsteps)
    d = s.diagnose_fluxes(spectral=False)
    s.advance(1)
    g = s.get_state(("E_down", "E_up", "dE"))
    sc = np.abs(g["E_up"]).max(axis=1, keepdims=True)
    for k in ("E_down", "E_up", "dE"):
        assert np.max(np.abs(d[k] - g[k]) / sc) <= 1e-12, k
    s.close()


# ---- 5. nothing changes ----------------------------------------------------------------------------------------------
@pytest.mark.parametrize("multi", [2, 0])
def test_the_call_changes_nothing(rcm, ens21, tmp_path, multi):
    a, b = solver(rcm, 20, ens21), solver(rcm, 20, ens21)
    for s in (a, b):
        s.set_option(OPT_MULTI, multi)
    sa = [a.advance(2), a.advance(3)]
    b.diagnose_fluxes()
    sb = [b.advance(2)]
    b.diagnose_fluxes(vmr_scale=CO2_2X)
    b.diagnose_fluxes(col0=3, ncol=5, spectral=False)
    sb.append(b.advance(3))
    b.diagnose_fluxes()
    for x, y in zip(sa, sb):
        assert np.array_equal(x, y)
    ga, gb = a.get_state(), b.get_state()
    for k in ga:
        assert np.array_equal(ga[k], gb[k]), k
    a.save_checkpoint(str(tmp_path / "a.ckpt"))
    b.save_checkpoint(str(tmp_path / "b.ckpt"))
    assert open(tmp_path / "a.ckpt", "rb").read() == open(tmp_path / "b.ckpt", "rb").read()
    assert np.array_equal(a.advance(1), b.advance(1))
    a.close()
    b.close()


# ---- 6. shard invariance -----------------------------------------------------------------------------------------------
def test_results_do_not_depend_on_the_range(rcm, ens5000):
    s = solver(rcm, 100, ens5000)
    s.advance(2)
    whole = s.diagnose_fluxes()
    halves = [s.diagnose_fluxes(0, 2500), s.diagnose_fluxes(2500, 2500)]
    one = s.diagnose_fluxes(4321, 1)
    s.close()
    part = solver(rcm, 100, ens5000, slice(4000, 5000))
    part.advance(2)
    tail = part.diagnose_fluxes()
    part.close()
    for k in whole:
        assert np.array_equal(whole[k], np.concatenate([h[k] for h in halves])), k
        assert np.array_equal(whole[k][4321:4322], one[k]), k
        assert np.array_equal(whole[k][4000:], tail[k]), k


# ---- 7. per-column forcing and scaled VMRs --------------------------------------------------------------------------------
def test_per_column_cloud_and_solar_and_h2o_scale(rcm, port, ens21):
    tab = port.load_rcmtab(table_path(20))
    s = solver(rcm, 20, ens21)
    rng = np.random.default_rng(3)
    tau_s, mu_s = rng.uniform(0.5, 4.0, s.ncol), rng.uniform(0.3, 0.8, s.ncol)
    forc = s.set_column_solar(None, tau_s, mu_s, None, cloud_from_tau_s=True)
    s.advance(1)
    check_against_port(port, s, ens21, tab, 1, solar_col=forc["solar_irr"], tau_s=tau_s)
    check_against_port(port, s, ens21, tab, 1, solar_col=forc["solar_irr"], tau_s=tau_s, h2o_scale=1.25)
    s.close()


# ---- 8. errors -----------------------------------------------------------------------------------------------------------
def status_of(rcm, fn):
    with pytest.raises(rcm.RcmError) as e:
        fn()
    return int(str(e.value).split("rcm status ")[1].split(":")[0])


def test_errors_leave_the_solver_usable(rcm, ens21):
    s = solver(rcm, 20, ens21)
    for col0, ncol in ((-1, 3), (0, 0), (20, 2), (0, 22)):
        assert status_of(rcm, lambda: s.diagnose_fluxes(col0, ncol)) == 1, (col0, ncol)
    for bad in (-1.0, np.nan, np.inf):
        assert status_of(rcm, lambda: s.diagnose_fluxes(vmr_scale=[1.0, bad, 1.0, 1.0, 1.0])) == 1, bad
    with pytest.raises(ValueError):
        s.diagnose_fluxes(vmr_scale=[2.0])
    s.set_option(OPT_PATH, 1)
    assert status_of(rcm, lambda: s.diagnose_fluxes()) == 2
    s.set_option(OPT_PATH, 0)
    ref = s.diagnose_fluxes()
    s.advance(1)
    assert np.isfinite(s.diagnose_fluxes()["E_up"]).all() and np.isfinite(ref["E_up"]).all()
    s.close()

    p = rcm.default_params()
    p.species_mask = 0x0F
    m = solver(rcm, 20, ens21, params=p)
    assert status_of(rcm, lambda: m.diagnose_fluxes()) == 2
    m.advance(1)
    m.close()

    st = ens21
    lb = rcm.Solver(0)
    wvl, tau5 = rcm.make_lbl_tables(300, 7, st["plevel"], st["vmr9"][0, 0], st["vmr9"][0, 2])
    lb.set_lbl_tables(wvl, tau5, st["vmr9"][0, 0], st["vmr9"][0, 2])
    lb.set_columns(st["plevel"], st["Tlayer"], st["Tsurf"], st["vmr9"], st["rel_hum"])
    assert status_of(rcm, lambda: lb.diagnose_fluxes()) == 2
    lb.advance(1)
    assert np.isfinite(lb.get_state(("E_up",))["E_up"]).all()
    lb.close()

    empty = rcm.Solver(0)
    assert status_of(rcm, lambda: empty.diagnose_fluxes(0, 1)) == 2
    empty.close()


# ---- 9. the driver's --spectral-out ------------------------------------------------------------------------------------
def driver(rcm, *args):
    exe = os.path.join(os.path.dirname(rcm.library_path()), "rcm_rce")
    return subprocess.run([exe, "--atm", os.path.join(GOLDEN, "column21.atm"), *args], capture_output=True, text=True,
                          timeout=300)


def means_of(rcm, ckpt, n):
    s = rcm.Solver(0)
    s.set_repwvl_table_from(rcm.Table(table_path(n)))
    s.load_checkpoint(ckpt)
    d = s.diagnose_fluxes()
    s.close()
    olr, sfc = np.zeros(d["E_up_spec"].shape[1]), np.zeros(d["E_up_spec"].shape[1])
    for c in range(d["E_up_spec"].shape[0]):  # column order, then one division: the driver's arithmetic
        olr = olr + d["E_up_spec"][c, :, 0]
        sfc = sfc + d["E_down_spec"][c, :, NLEV - 1]
    return olr / d["E_up_spec"].shape[0], sfc / d["E_up_spec"].shape[0]


def test_driver_spectral_out(rcm, port, tmp_path):
    ck, spec = str(tmp_path / "run.ckpt"), str(tmp_path / "spectrum.csv")
    common = ["--table", table_path(100), "--ncol", "64", "--seed", "9", "--max-steps", "3", "--steps-exact"]
    r = driver(rcm, *common, "--out", str(tmp_path / "o.txt"), "--checkpoint", ck, "--spectral-out", spec)
    assert r.returncode == 0, r.stderr
    lines = open(spec).read().splitlines()
    assert lines[0] == "wvl_nm,weight,olr,surface_down" and len(lines) == 101
    rows = np.array([[float(x) for x in l.split(",")] for l in lines[1:]])
    tab = port.load_rcmtab(table_path(100))
    olr, sfc = means_of(rcm, ck, 100)
    assert np.array_equal(rows[:, 0], tab["wvl"]) and np.array_equal(rows[:, 1], tab["weight"])
    assert np.array_equal(rows[:, 2], olr) and np.array_equal(rows[:, 3], sfc)

    d = tmp_path / "lbl"
    d.mkdir()
    r = driver(rcm, "--lbl", str(d), "--spectral-out", spec, "--max-steps", "1")
    assert r.returncode == 1 and "--spectral-out" in r.stderr

    if rcm.device_count() < 2:
        pytest.skip("--gpus 2 needs two GPUs")
    spec2 = str(tmp_path / "spectrum2.csv")
    r = driver(rcm, *common, "--out", str(tmp_path / "o2.txt"), "--spectral-out", spec2, "--gpus", "2")
    assert r.returncode == 0, r.stderr
    assert open(spec).read() == open(spec2).read()
