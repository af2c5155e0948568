"""Radiative kernels of the resident ensemble (rcm_radiative_kernels / Solver.radiative_kernels): analytic derivatives of the
next step's OLR and surface downward flux with respect to every layer's temperature, the surface temperature and every
layer's ln(H2O VMR), per wavelength and broadband, without changing anything.

Checker: central differences of the C port of the reference (oracle/rcm_oracle.c) around the inputs the next step
radiates with, built as in test_gpu_diagnostics.py (the port's theta_sort and water_vapor_feedback).  d/dT_l moves layer
l's temperature both where its tau is interpolated (at step 0 the initial, unsorted profile) and in the radiated profile;
d/dln q_l multiplies the layer's H2O VMR by exp(+-eps) at fixed T.  Layers whose T +- h would change the port's table
interval (lowpos_t) have no central difference there and are skipped (and counted).
"""
import os
import subprocess

import numpy as np
import pytest

from conftest import GOLDEN, table_path
from test_gpu_diagnostics import CO2_2X, ensemble, feedback, solver, status_of, theta_sort

pytestmark = pytest.mark.gpu
NLAY, NLEV, NE = 20, 21, 41
H, EPS = 1e-2, 1e-4


@pytest.fixture(scope="module")
def ens21(rcm):
    return ensemble(rcm, 21, 2024)


@pytest.fixture(scope="module")
def ens5000(rcm):
    return ensemble(rcm, 5000, 77)


# ---- the port's central differences ------------------------------------------------------------------------------------
def radiated_inputs(port, st, T, vmr9, rel_hum, first, h2o_scale=1.0, co2_scale=1.0):
    """(profile tau is interpolated at, radiated profile, vmr9) of the next step of one column."""
    v9 = np.array(vmr9, dtype=np.float64)
    Ts = theta_sort(port, T, st["conv"])
    if first:
        tau_T = np.array(T, dtype=np.float64)
    else:
        tau_T = Ts.copy()
        v9[0] = feedback(port, Ts, rel_hum, st["player"])
    v9[0] = v9[0] * h2o_scale
    v9[1] = v9[1] * co2_scale
    return tau_T, Ts, v9


def port_kernels(port, tab, pl, tau_T, Trad, Tsurf, v9, tau_s=2.0, spectral=False):
    """-> K [2][41] (spectral: [nwvl][2][41]) by central differences, and the layers skipped for a change of lowpos_t."""
    nw = tab["wvl"].size

    def F(tT, Tr, Ts, v):
        tau, _, _ = port.read_tau(tab, pl, tT, v, tau_s=tau_s)
        if not spectral:
            Ed, Eu, _ = port.radiative_transfer(tau, tab["wvl"], tab["weight"], Tr, Ts, 0.0)
            return np.array([Eu[0], Ed[NLEV - 1]])
        out = np.zeros((nw, 2))
        for w in range(nw):
            Ed, Eu, _ = port.radiative_transfer(tau[w:w + 1], tab["wvl"][w:w + 1], tab["weight"][w:w + 1], Tr, Ts, 0.0)
            out[w] = Eu[0], Ed[NLEV - 1]
        return out

    _, _, lt0 = port.read_tau(tab, pl, tau_T, v9, tau_s=tau_s)
    K = np.zeros(((nw,) if spectral else ()) + (2, NE))
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
        K[..., l] = (F(tp, rp, Tsurf, v9) - F(tm, rm, Tsurf, v9)) / (2 * H)
    K[..., NLAY] = (F(tau_T, Trad, Tsurf + H, v9) - F(tau_T, Trad, Tsurf - H, v9)) / (2 * H)
    for l in range(NLAY):
        vp, vm = v9.copy(), v9.copy()
        vp[0, l] *= np.exp(EPS)
        vm[0, l] *= np.exp(-EPS)
        K[..., NLAY + 1 + l] = (F(tau_T, Trad, Tsurf, vp) - F(tau_T, Trad, Tsurf, vm)) / (2 * EPS)
    return K, skipped


def compare(got, ref, skipped, what):
    """<= 1e-6 of the column's max |K| per output; skipped layers' T entries left out."""
    mask = np.ones(ref.shape[-1], dtype=bool)
    mask[skipped] = False
    for o in range(2):
        sc = np.abs(ref[..., o, :]).max()
        err = np.abs(got[..., o, mask] - ref[..., o, mask]).max()
        assert err <= 1e-6 * sc, (what, o, err, sc)


def check_against_port(port, s, st, tab, nsteps_done, vmr_scale=None, tau_s=None, spectral_cols=()):
    h2o_scale = 1.0 if vmr_scale is None else vmr_scale[0]
    co2_scale = 1.0 if vmr_scale is None else vmr_scale[1]
    d = s.radiative_kernels(vmr_scale=vmr_scale, spectral=bool(spectral_cols))
    g = s.get_state(("Tlayer", "Tsurf"))
    nskip = 0
    for c in range(s.ncol):
        tau_T, Trad, v9 = radiated_inputs(port, st, g["Tlayer"][c], st["vmr9"][c], st["rel_hum"][c], nsteps_done == 0,
                                          h2o_scale, co2_scale)
        ts = 2.0 if tau_s is None else tau_s[c]
        ref, skipped = port_kernels(port, tab, st["plevel"], tau_T, Trad, g["Tsurf"][c], v9, tau_s=ts)
        nskip += len(skipped)
        compare(d["K"][c], ref, skipped, c)
        if c in spectral_cols:
            ref_s, skipped = port_kernels(port, tab, st["plevel"], tau_T, Trad, g["Tsurf"][c], v9, tau_s=ts, spectral=True)
            for w in range(s.nwvl):
                compare(d["K_spec"][c, w], ref_s[w], skipped, (c, w))
    assert nskip <= 0.1 * NLAY * s.ncol, nskip  # a layer within 1e-2 K of a table node is rare
    return d, nskip


# ---- 1. against the port's central differences ---------------------------------------------------------------------------
@pytest.mark.parametrize("nsteps", [3, 0])
def test_kernels_equal_central_differences_of_the_port(rcm, port, ens21, nsteps):
    """21 columns (a ragged second tile), Reduced20, after three steps and at step 0; every wavelength for three columns."""
    tab = port.load_rcmtab(table_path(20))
    s = solver(rcm, 20, ens21)
    if nsteps:
        s.advance(nsteps)
    d, nskip = check_against_port(port, s, ens21, tab, nsteps, spectral_cols=(0, 7, 20))
    print(f"nsteps {nsteps}: {nskip} layer temperatures skipped (table node within {H} K)")
    assert d["K"].shape == (21, 2, NE) and d["K_spec"].shape == (21, 20, 2, NE)
    s.close()


# ---- 2. base-column anchors --------------------------------------------------------------------------------------------
def test_base_column_anchors(rcm, port, golden):
    """Base column of column21.atm, Reduced100, step 0 (OLR 246.6782921988): Planck response, surface and cloud-layer
    terms, water-vapour sums - against the port's live differences, and near the published values."""
    tab = port.load_rcmtab(table_path(100))
    g = golden
    s = rcm.Solver(0)
    s.set_repwvl_table_from(rcm.Table(table_path(100)))
    s.set_columns(g["plevel"], g["Tlayer"][:1], g["Tsurf"][:1], g["vmr9"][:1], g["rel_hum"][:1])
    d = s.radiative_kernels()
    assert abs(s.diagnose_fluxes(spectral=False)["E_up"][0, 0] - 246.6782921988) <= 1e-10 * 246.6782921988
    tau_T = np.array(g["Tlayer"][0], dtype=np.float64)  # step 0: tau of the initial profile, the sorted one radiates
    Trad = theta_sort(port, tau_T, g["conv"])
    ref, skipped = port_kernels(port, tab, g["plevel"], tau_T, Trad, float(g["Tsurf"][0]), np.array(g["vmr9"][0]))
    assert not skipped
    K = d["K"][0]
    compare(K, ref, [], "base column")
    live = dict(planck=ref[0, :NLAY + 1].sum(), ts=ref[0, NLAY], cloud=ref[0, 17], olr_q=ref[0, NLAY + 1:].sum(),
                sfc_T=ref[1, :NLAY].sum(), sfc_q=ref[1, NLAY + 1:].sum())
    gpu = dict(planck=K[0, :NLAY + 1].sum(), ts=K[0, NLAY], cloud=K[0, 17], olr_q=K[0, NLAY + 1:].sum(),
               sfc_T=K[1, :NLAY].sum(), sfc_q=K[1, NLAY + 1:].sum())
    published = dict(planck=3.8047, ts=0.2914, cloud=1.1446, olr_q=-13.768, sfc_T=4.7804, sfc_q=8.558)
    for k in live:
        assert abs(gpu[k] - live[k]) <= 1e-6 * max(abs(live[k]), 1.0), (k, gpu[k], live[k])
        assert abs(live[k] - published[k]) <= 6e-4 * max(abs(published[k]), 1.0), (k, live[k], published[k])
    s.close()


# ---- 3. structure --------------------------------------------------------------------------------------------------------
def test_broadband_is_the_sequential_sum_of_the_spectrum(rcm, ens21):
    s = solver(rcm, 100, ens21)
    s.advance(2)
    d = s.radiative_kernels(spectral=True)
    acc = np.zeros((s.ncol, 2, NE))
    for w in range(s.nwvl):
        acc = acc + d["K_spec"][:, w]
    assert np.array_equal(acc, d["K"])
    assert np.all(d["K"][:, 1, NLAY] == 0.0) and np.all(d["K_spec"][:, :, 1, NLAY] == 0.0)
    assert np.all(d["dOLR_dTs"] > 0.0) and np.all(d["dOLR_dT"].sum(axis=1) + d["dOLR_dTs"] > 0.0)
    for k, v in (("dOLR_dT", d["K"][:, 0, :NLAY]), ("dOLR_dTs", d["K"][:, 0, NLAY]), ("dOLR_dlnq", d["K"][:, 0, NLAY + 1:]),
                 ("dSFC_dT", d["K"][:, 1, :NLAY]), ("dSFC_dlnq", d["K"][:, 1, NLAY + 1:])):
        assert np.array_equal(d[k], v), k
    bb = s.radiative_kernels()
    assert "K_spec" not in bb and np.array_equal(bb["K"], d["K"])
    assert np.array_equal(s.radiative_kernels(vmr_scale=np.ones(5))["K"], d["K"])
    s.close()


# ---- 4. identity through the existing API -----------------------------------------------------------------------------------
def test_water_vapour_sum_equals_difference_of_diagnosed_fluxes(rcm, ens5000):
    """Sum_l dF/dln q_l is the derivative for H2O x e^eps in every layer: two diagnose_fluxes calls, device only."""
    s = solver(rcm, 100, ens5000)
    s.advance(4)
    K = s.radiative_kernels()["K"]
    up = s.diagnose_fluxes(vmr_scale=[np.exp(EPS), 1, 1, 1, 1], spectral=False)
    dn = s.diagnose_fluxes(vmr_scale=[np.exp(-EPS), 1, 1, 1, 1], spectral=False)
    s.close()
    for o, (lev, key) in enumerate(((0, "E_up"), (NLEV - 1, "E_down"))):
        fd = (up[key][:, lev] - dn[key][:, lev]) / (2 * EPS)
        an = K[:, o, NLAY + 1:].sum(axis=1)
        tol = 1e-6 * np.abs(K[:, o, NLAY + 1:]).sum(axis=1)
        assert np.all(np.abs(an - fd) <= tol), (o, np.max(np.abs(an - fd) / tol))


# ---- 5. invariance and no side effects -------------------------------------------------------------------------------------
def test_results_do_not_depend_on_the_range(rcm, ens5000):
    s = solver(rcm, 100, ens5000)
    s.advance(2)
    whole = s.radiative_kernels()["K"]
    halves = np.concatenate([s.radiative_kernels(0, 2500)["K"], s.radiative_kernels(2500, 2500)["K"]])
    one = s.radiative_kernels(4321, 1, spectral=True)
    few = s.radiative_kernels(4317, 9, spectral=True)
    s.close()
    part = solver(rcm, 100, ens5000, slice(4000, 5000))
    part.advance(2)
    tail = part.radiative_kernels()["K"]
    part.close()
    assert np.array_equal(whole, halves)
    assert np.array_equal(whole[4321:4322], one["K"]) and np.array_equal(few["K_spec"][4:5], one["K_spec"])
    assert np.array_equal(whole[4000:], tail)


@pytest.mark.parametrize("multi", [2, 0])
def test_the_call_changes_nothing(rcm, ens21, tmp_path, multi):
    OPT_MULTI = 6
    a, b = solver(rcm, 20, ens21), solver(rcm, 20, ens21)
    for s in (a, b):
        s.set_option(OPT_MULTI, multi)
    b.radiative_kernels()
    sa = [a.advance(2), a.advance(3)]
    sb = [b.advance(2)]
    b.radiative_kernels(vmr_scale=CO2_2X, spectral=True)
    b.radiative_kernels(col0=3, ncol=5)
    sb.append(b.advance(3))
    b.radiative_kernels()
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


# ---- 6. variants against the port -----------------------------------------------------------------------------------------
def test_co2_scale_column_cloud_and_h2o_scale(rcm, port, ens21):
    tab = port.load_rcmtab(table_path(20))
    s = solver(rcm, 20, ens21)
    s.advance(1)
    check_against_port(port, s, ens21, tab, 1, vmr_scale=CO2_2X)
    rng = np.random.default_rng(5)
    tau_s, mu_s = rng.uniform(0.5, 4.0, s.ncol), rng.uniform(0.3, 0.8, s.ncol)
    s.set_column_solar(None, tau_s, mu_s, None, cloud_from_tau_s=True)
    check_against_port(port, s, ens21, tab, 1, tau_s=tau_s)
    check_against_port(port, s, ens21, tab, 1, vmr_scale=[1.25, 1.0, 1.0, 1.0, 1.0], tau_s=tau_s, spectral_cols=(5,))
    s.close()


# ---- 7. errors ---------------------------------------------------------------------------------------------------------------
def test_errors_leave_the_solver_usable(rcm, ens21):
    OPT_PATH = 5
    s = solver(rcm, 20, ens21)
    for col0, ncol in ((-1, 3), (0, 0), (20, 2), (0, 22)):
        assert status_of(rcm, lambda: s.radiative_kernels(col0, ncol)) == 1, (col0, ncol)
    for bad in (-1.0, np.nan, np.inf):
        assert status_of(rcm, lambda: s.radiative_kernels(vmr_scale=[1.0, bad, 1.0, 1.0, 1.0])) == 1, bad
    with pytest.raises(ValueError):
        s.radiative_kernels(vmr_scale=[2.0])
    s.set_option(OPT_PATH, 1)
    assert status_of(rcm, lambda: s.radiative_kernels()) == 2
    s.set_option(OPT_PATH, 0)
    ref = s.radiative_kernels()
    s.advance(1)
    assert np.isfinite(s.radiative_kernels()["K"]).all() and np.isfinite(ref["K"]).all()
    s.close()

    p = rcm.default_params()
    p.species_mask = 0x0F
    m = solver(rcm, 20, ens21, params=p)
    assert status_of(rcm, lambda: m.radiative_kernels()) == 2
    m.advance(1)
    m.close()

    st = ens21
    lb = rcm.Solver(0)
    wvl, tau5 = rcm.make_lbl_tables(300, 7, st["plevel"], st["vmr9"][0, 0], st["vmr9"][0, 2])
    lb.set_lbl_tables(wvl, tau5, st["vmr9"][0, 0], st["vmr9"][0, 2])
    lb.set_columns(st["plevel"], st["Tlayer"], st["Tsurf"], st["vmr9"], st["rel_hum"])
    assert status_of(rcm, lambda: lb.radiative_kernels()) == 2
    lb.advance(1)
    assert np.isfinite(lb.get_state(("E_up",))["E_up"]).all()
    lb.close()

    empty = rcm.Solver(0)
    assert status_of(rcm, lambda: empty.radiative_kernels(0, 1)) == 2
    empty.close()


# ---- 8. the driver's --kernels-out -----------------------------------------------------------------------------------------
def driver(rcm, *args):
    exe = os.path.join(os.path.dirname(rcm.library_path()), "rcm_rce")
    return subprocess.run([exe, "--atm", os.path.join(GOLDEN, "column21.atm"), *args], capture_output=True, text=True,
                          timeout=300)


def test_driver_kernels_out(rcm, tmp_path):
    ck, kf = str(tmp_path / "run.ckpt"), str(tmp_path / "kernels.csv")
    common = ["--table", table_path(100), "--ncol", "64", "--seed", "9", "--max-steps", "3", "--steps-exact"]
    r = driver(rcm, *common, "--out", str(tmp_path / "o.txt"), "--checkpoint", ck, "--kernels-out", kf)
    assert r.returncode == 0, r.stderr
    lines = open(kf).read().splitlines()
    assert lines[0] == "layer,p_layer,dOLR_dT,dOLR_dlnq,dSFC_dT,dSFC_dlnq" and len(lines) == NLAY + 2
    rows = np.array([[float(x) for x in l.split(",")[1:]] for l in lines[1:]])
    assert [l.split(",")[0] for l in lines[1:]] == [str(l) for l in range(NLAY)] + ["surface"]

    s = rcm.Solver(0)
    s.set_repwvl_table_from(rcm.Table(table_path(100)))
    s.load_checkpoint(ck)
    K = s.radiative_kernels()["K"]
    s.close()
    acc = np.zeros((2, NE))
    for c in range(K.shape[0]):  # column order, then one division: the driver's arithmetic
        acc = acc + K[c]
    mean = acc / K.shape[0]
    atm = rcm.read_atm(os.path.join(GOLDEN, "column21.atm"))
    pl = atm[:, 1]
    assert np.array_equal(rows[:NLAY, 0], (pl[:NLAY] + pl[1:]) / 2.0) and rows[NLAY, 0] == pl[NLAY]
    assert np.array_equal(rows[:NLAY, 1], mean[0, :NLAY]) and np.array_equal(rows[:NLAY, 2], mean[0, NLAY + 1:])
    assert np.array_equal(rows[:NLAY, 3], mean[1, :NLAY]) and np.array_equal(rows[:NLAY, 4], mean[1, NLAY + 1:])
    assert np.array_equal(rows[NLAY, 1:], [mean[0, NLAY], 0.0, 0.0, 0.0])

    d = tmp_path / "lbl"
    d.mkdir()
    r = driver(rcm, "--lbl", str(d), "--kernels-out", kf, "--max-steps", "1")
    assert r.returncode == 1 and "--kernels-out" in r.stderr

    if rcm.device_count() < 2:
        pytest.skip("--gpus 2 needs two GPUs")
    kf2 = str(tmp_path / "kernels2.csv")
    r = driver(rcm, *common, "--out", str(tmp_path / "o2.txt"), "--kernels-out", kf2, "--gpus", "2")
    assert r.returncode == 0, r.stderr
    assert open(kf).read() == open(kf2).read()
