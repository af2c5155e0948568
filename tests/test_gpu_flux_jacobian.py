"""Flux Jacobians of the resident ensemble (rcm_flux_jacobian / Solver.flux_jacobian): analytic derivatives of every level's
broadband E_down and E_up of the next step, and of its heating rates dE, with respect to every layer's temperature, the
surface temperature and every layer's ln(H2O VMR), without changing anything.

Checker: central differences of the C port of the reference (oracle/rcm_oracle.c) for all 42 fluxes, around the inputs the
next step radiates with (test_gpu_radiative_kernels.radiated_inputs), with that file's step sizes and its rule for layers
whose T +- h would change the port's table interval (skipped and counted).
"""
import os

import numpy as np
import pytest

from conftest import GOLDEN, table_path
from test_gpu_diagnostics import CO2_2X, ensemble, solver, status_of
from test_gpu_radiative_kernels import EPS, H, driver, radiated_inputs

pytestmark = pytest.mark.gpu
NLAY, NLEV, NE = 20, 21, 41


@pytest.fixture(scope="module")
def ens21(rcm):
    return ensemble(rcm, 21, 2024)


@pytest.fixture(scope="module")
def ens5000(rcm):
    return ensemble(rcm, 5000, 77)


def heating_jacobian(J):
    """dE_jac from J as dE from E (main.cpp:337-341), the solar term constant: the call's operation order."""
    Jd, Ju = J[:, 0], J[:, 1]
    Hj = Jd[:, :NLAY] - Jd[:, 1:] + Ju[:, 1:] - Ju[:, :NLAY]
    Hj[:, NLAY - 1] = Hj[:, NLAY - 1] + (Jd[:, NLAY] - Ju[:, NLAY])
    return Hj


# ---- the port's central differences ------------------------------------------------------------------------------------
def port_jacobian(port, tab, pl, tau_T, Trad, Tsurf, v9, tau_s=2.0):
    """-> J [2][21][41] by central differences, and the layers skipped for a change of lowpos_t."""
    def F(tT, Tr, Ts, v):
        tau, _, _ = port.read_tau(tab, pl, tT, v, tau_s=tau_s)
        Ed, Eu, _ = port.radiative_transfer(tau, tab["wvl"], tab["weight"], Tr, Ts, 0.0)
        return np.array([Ed, Eu])

    _, _, lt0 = port.read_tau(tab, pl, tau_T, v9, tau_s=tau_s)
    J = np.zeros((2, NLEV, NE))
    skipped = []
    for l in range(NLAY):
        tp, tm, rp, rm = tau_T.copy(), tau_T.copy(), Trad.copy(), Trad.copy()
        tp[l] += H
        tm[l] -= H
        rp[l] += H
        rm[l] -= H
        if any(not np.array_equal(port.read_tau(tab, pl, t, v9, tau_s=tau_s)[2], lt0) for t in (tp, tm)):
            skipped.append(l)
            continue
        J[..., l] = (F(tp, rp, Tsurf, v9) - F(tm, rm, Tsurf, v9)) / (2 * H)
    J[..., NLAY] = (F(tau_T, Trad, Tsurf + H, v9) - F(tau_T, Trad, Tsurf - H, v9)) / (2 * H)
    for l in range(NLAY):
        vp, vm = v9.copy(), v9.copy()
        vp[0, l] *= np.exp(EPS)
        vm[0, l] *= np.exp(-EPS)
        J[..., NLAY + 1 + l] = (F(tau_T, Trad, Tsurf, vp) - F(tau_T, Trad, Tsurf, vm)) / (2 * EPS)
    return J, skipped


def check_against_port(port, s, st, tab, nsteps_done, vmr_scale=None, tau_s=None):
    h2o_scale = 1.0 if vmr_scale is None else vmr_scale[0]
    co2_scale = 1.0 if vmr_scale is None else vmr_scale[1]
    d = s.flux_jacobian(vmr_scale=vmr_scale)
    g = s.get_state(("Tlayer", "Tsurf"))
    nskip = 0
    mask = np.ones(NE, dtype=bool)
    for c in range(s.ncol):
        tau_T, Trad, v9 = radiated_inputs(port, st, g["Tlayer"][c], st["vmr9"][c], st["rel_hum"][c], nsteps_done == 0,
                                          h2o_scale, co2_scale)
        ts = 2.0 if tau_s is None else tau_s[c]
        ref, skipped = port_jacobian(port, tab, st["plevel"], tau_T, Trad, g["Tsurf"][c], v9, tau_s=ts)
        nskip += len(skipped)
        mask[:] = True
        mask[skipped] = False
        for o in range(2):  # <= 1e-6 of the column's max |entry| of the E_down resp. E_up block
            sc = np.abs(ref[o]).max()
            err = np.abs(d["J"][c, o][:, mask] - ref[o][:, mask]).max()
            assert err <= 1e-6 * sc, (c, o, err, sc)
    assert nskip <= 0.1 * NLAY * s.ncol, nskip  # a layer within 1e-2 K of a table node is rare
    return d, nskip


# ---- 1. against the port's central differences ---------------------------------------------------------------------------
@pytest.mark.parametrize("nsteps", [3, 0])
def test_jacobian_equals_central_differences_of_the_port(rcm, port, ens21, nsteps):
    """21 columns (a ragged second tile), Reduced20, after three steps and at step 0, all 42 fluxes."""
    tab = port.load_rcmtab(table_path(20))
    s = solver(rcm, 20, ens21)
    if nsteps:
        s.advance(nsteps)
    d, nskip = check_against_port(port, s, ens21, tab, nsteps)
    print(f"nsteps {nsteps}: {nskip} layer temperatures skipped (table node within {H} K)")
    assert d["J"].shape == (21, 2, NLEV, NE) and d["dE_jac"].shape == (21, NLAY, NE)
    s.close()


def test_co2_scale_and_column_cloud(rcm, port, ens21):
    tab = port.load_rcmtab(table_path(20))
    s = solver(rcm, 20, ens21)
    s.advance(1)
    check_against_port(port, s, ens21, tab, 1, vmr_scale=CO2_2X)
    rng = np.random.default_rng(5)
    tau_s, mu_s = rng.uniform(0.5, 4.0, s.ncol), rng.uniform(0.3, 0.8, s.ncol)
    s.set_column_solar(None, tau_s, mu_s, None, cloud_from_tau_s=True)
    check_against_port(port, s, ens21, tab, 1, tau_s=tau_s)
    s.close()


# ---- 2.-4. structure, agreement with the radiative kernels, dE_jac -------------------------------------------------------
@pytest.mark.parametrize("vmr_scale", [None, CO2_2X])
def test_structure_kernels_and_heating_rates(rcm, ens21, vmr_scale):
    s = solver(rcm, 100, ens21)
    s.advance(2)
    d = s.flux_jacobian(vmr_scale=vmr_scale)
    K = s.radiative_kernels(vmr_scale=vmr_scale)["K"]
    s.close()
    J = d["J"]
    # structural zeros, exactly 0.0
    assert np.all(J[:, 0, 0] == 0.0)
    for k in range(NLEV):
        for l in range(NLAY):
            sl = [l, NLAY + 1 + l]
            if l >= k:
                assert np.all(J[:, 0, k, sl] == 0.0), (k, l)
            else:
                assert np.all(J[:, 1, k, sl] == 0.0), (k, l)
    assert np.all(J[:, 0, :, NLAY] == 0.0)
    assert np.all(J[:, 1, NLEV - 1, :NLAY] == 0.0) and np.all(J[:, 1, NLEV - 1, NLAY + 1:] == 0.0)
    assert np.all(J[:, 1, NLEV - 1, NLAY] > 0.0) and np.all(J[:, 1, 0, NLAY] > 0.0)
    # rows E_up[0] and E_down[20] are the radiative kernels' outputs 0 and 1
    for row, o in ((J[:, 1, 0], 0), (J[:, 0, NLEV - 1], 1)):
        sc = np.abs(K[:, o]).max(axis=1, keepdims=True)
        assert np.all(np.abs(row - K[:, o]) <= 1e-12 * sc), (o, np.max(np.abs(row - K[:, o]) / sc))
    # dE_jac is the numpy expression of J, bit for bit
    assert np.array_equal(d["dE_jac"], heating_jacobian(J))


# ---- 5. identity through the existing API -----------------------------------------------------------------------------------
def test_water_vapour_sum_equals_difference_of_diagnosed_fluxes(rcm, ens5000):
    """Sum_l dF/dln q_l is the derivative for H2O x e^eps in every layer: two diagnose_fluxes calls, all 42 fluxes and dE."""
    s = solver(rcm, 100, ens5000)
    s.advance(4)
    d = s.flux_jacobian()
    up = s.diagnose_fluxes(vmr_scale=[np.exp(EPS), 1, 1, 1, 1], spectral=False)
    dn = s.diagnose_fluxes(vmr_scale=[np.exp(-EPS), 1, 1, 1, 1], spectral=False)
    s.close()
    for an_all, key in ((d["J"][:, 0], "E_down"), (d["J"][:, 1], "E_up"), (d["dE_jac"], "dE")):
        fd = (up[key] - dn[key]) / (2 * EPS)
        an = an_all[..., NLAY + 1:].sum(axis=-1)
        tol = 1e-6 * np.maximum(np.abs(an_all[..., NLAY + 1:]).sum(axis=-1), 1e-3)
        assert np.all(np.abs(an - fd) <= tol), (key, np.max(np.abs(an - fd) / tol))


# ---- 6. invariance and no side effects -------------------------------------------------------------------------------------
def test_results_do_not_depend_on_the_range(rcm, ens5000):
    s = solver(rcm, 100, ens5000)
    s.advance(2)
    whole = s.flux_jacobian()
    halves = [s.flux_jacobian(0, 2500), s.flux_jacobian(2500, 2500)]
    one = s.flux_jacobian(4321, 1)
    few = s.flux_jacobian(4317, 9)
    s.close()
    part = solver(rcm, 100, ens5000, slice(4000, 5000))
    part.advance(2)
    tail = part.flux_jacobian()
    part.close()
    for k in ("J", "dE_jac"):
        assert np.array_equal(whole[k], np.concatenate([h[k] for h in halves])), k
        assert np.array_equal(whole[k][4321:4322], one[k]) and np.array_equal(few[k][4:5], one[k]), k
        assert np.array_equal(whole[k][4000:], tail[k]), k


def test_chunks_of_the_call_do_not_change_results(rcm):
    """Two chunks of the whole-ensemble call (8,192 + 108 columns) against a range that starts inside a tile and covers
    the chunk boundary in one chunk of its own."""
    st = ensemble(rcm, 8300, 11)
    s = solver(rcm, 20, st)
    s.advance(1)
    whole = s.flux_jacobian()
    cross = s.flux_jacobian(8185, 20)
    s.close()
    for k in ("J", "dE_jac"):
        assert np.array_equal(whole[k][8185:8205], cross[k]), k


@pytest.mark.parametrize("multi", [2, 0])
def test_the_call_changes_nothing(rcm, ens21, tmp_path, multi):
    OPT_MULTI = 6
    a, b = solver(rcm, 20, ens21), solver(rcm, 20, ens21)
    for s in (a, b):
        s.set_option(OPT_MULTI, multi)
    b.flux_jacobian()
    sa = [a.advance(2), a.advance(3)]
    sb = [b.advance(2)]
    b.flux_jacobian(vmr_scale=CO2_2X)
    b.flux_jacobian(col0=3, ncol=5)
    sb.append(b.advance(3))
    b.flux_jacobian()
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


# ---- 7. errors ---------------------------------------------------------------------------------------------------------------
def test_errors_leave_the_solver_usable(rcm, ens21):
    OPT_PATH = 5
    s = solver(rcm, 20, ens21)
    for col0, ncol in ((-1, 3), (0, 0), (20, 2), (0, 22)):
        assert status_of(rcm, lambda: s.flux_jacobian(col0, ncol)) == 1, (col0, ncol)
    for bad in (-1.0, np.nan, np.inf):
        assert status_of(rcm, lambda: s.flux_jacobian(vmr_scale=[1.0, bad, 1.0, 1.0, 1.0])) == 1, bad
    with pytest.raises(ValueError):
        s.flux_jacobian(vmr_scale=[2.0])
    s.set_option(OPT_PATH, 1)
    assert status_of(rcm, lambda: s.flux_jacobian()) == 2
    s.set_option(OPT_PATH, 0)
    ref = s.flux_jacobian()
    s.advance(1)
    assert np.isfinite(s.flux_jacobian()["J"]).all() and np.isfinite(ref["J"]).all()
    s.close()

    p = rcm.default_params()
    p.species_mask = 0x0F
    m = solver(rcm, 20, ens21, params=p)
    assert status_of(rcm, lambda: m.flux_jacobian()) == 2
    m.advance(1)
    m.close()

    # five active species without H2O: no water-vapour entries to differentiate
    p = rcm.default_params()
    p.species_mask = 0x3E  # CO2, O3, species 4, N2O, CH4
    w = solver(rcm, 20, ens21, params=p)
    assert status_of(rcm, lambda: w.flux_jacobian()) == 2
    w.advance(1)
    w.close()

    st = ens21
    lb = rcm.Solver(0)
    wvl, tau5 = rcm.make_lbl_tables(300, 7, st["plevel"], st["vmr9"][0, 0], st["vmr9"][0, 2])
    lb.set_lbl_tables(wvl, tau5, st["vmr9"][0, 0], st["vmr9"][0, 2])
    lb.set_columns(st["plevel"], st["Tlayer"], st["Tsurf"], st["vmr9"], st["rel_hum"])
    assert status_of(rcm, lambda: lb.flux_jacobian()) == 2
    lb.advance(1)
    assert np.isfinite(lb.get_state(("E_up",))["E_up"]).all()
    lb.close()


# ---- 8. the driver's --jacobian-out ----------------------------------------------------------------------------------------
def test_driver_jacobian_out(rcm, tmp_path):
    ck, jf = str(tmp_path / "run.ckpt"), str(tmp_path / "jacobian.csv")
    common = ["--table", table_path(100), "--ncol", "64", "--seed", "9", "--max-steps", "3", "--steps-exact"]
    r = driver(rcm, *common, "--out", str(tmp_path / "o.txt"), "--checkpoint", ck, "--jacobian-out", jf)
    assert r.returncode == 0, r.stderr
    lines = open(jf).read().splitlines()
    head = ["layer", "p_layer"] + [f"dT_{l}" for l in range(NLAY)] + ["dT_surf"] + [f"dlnq_{l}" for l in range(NLAY)]
    assert lines[0].split(",") == head and len(lines) == NLAY + 1
    assert [l.split(",")[0] for l in lines[1:]] == [str(l) for l in range(NLAY)]
    rows = np.array([[float(x) for x in l.split(",")[1:]] for l in lines[1:]])

    s = rcm.Solver(0)
    s.set_repwvl_table_from(rcm.Table(table_path(100)))
    s.load_checkpoint(ck)
    Hj = s.flux_jacobian()["dE_jac"]
    s.close()
    acc = np.zeros((NLAY, NE))
    for c in range(Hj.shape[0]):  # column order, then one division: the driver's arithmetic
        acc = acc + Hj[c]
    mean = acc / Hj.shape[0]
    atm = rcm.read_atm(os.path.join(GOLDEN, "column21.atm"))
    pl = atm[:, 1]
    assert np.array_equal(rows[:, 0], (pl[:NLAY] + pl[1:]) / 2.0)
    assert np.array_equal(rows[:, 1:], mean)

    d = tmp_path / "lbl"
    d.mkdir()
    r = driver(rcm, "--lbl", str(d), "--jacobian-out", jf, "--max-steps", "1")
    assert r.returncode == 1 and "--jacobian-out" in r.stderr

    if rcm.device_count() < 2:
        pytest.skip("--gpus 2 needs two GPUs")
    jf2 = str(tmp_path / "jacobian2.csv")
    r = driver(rcm, *common, "--out", str(tmp_path / "o2.txt"), "--jacobian-out", jf2, "--gpus", "2")
    assert r.returncode == 0, r.stderr
    assert open(jf).read() == open(jf2).read()

