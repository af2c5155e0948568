"""The diagnostic radiation call of the line-by-line path (rcm_lbl_diagnose_fluxes / Solver.lbl_diagnose_fluxes): the fluxes
the next LBL step would compute, bit for bit against that step, per wavelength and band against the C port
(rcmo_lbl_tau + rcmo_lbl_radiative_transfer), with scaled species, without moving the state.
"""
import ctypes as C
import os
import subprocess

import numpy as np
import pytest

from conftest import GOLDEN, table_path

pytestmark = pytest.mark.gpu

# vmr_scale order: ascending species index H2O, CO2, O3, N2O, CH4 (tau5 is H2O, CO2, O3, CH4, N2O)
SCALES = {"none": None, "h2o": [1.5, 1, 1, 1, 1], "co2": [1, 2, 1, 1, 1], "o3": [1, 1, 0.5, 1, 1],
          "n2o": [1, 1, 1, 2, 1], "ch4": [1, 1, 1, 1, 2]}


@pytest.fixture(scope="module")
def case(rcm, tmp_path_factory):
    atm = rcm.read_atm(os.path.join(GOLDEN, "column21.lbl.atm"))
    full = rcm.read_atm(os.path.join(GOLDEN, "column21.atm"))
    pl = atm[:, 1].copy()
    ncol, nwvl = 24, 1500
    Tlev, vlev = rcm.make_ensemble(ncol, 4242, pl, atm[:, 2].copy(), full[:, 4:9].T.copy())
    st = rcm.init_columns(pl, Tlev, vlev)
    h2o_ref, o3_ref = st["vmr9"][0, 0].copy(), st["vmr9"][0, 2].copy()
    wvl, tau5 = rcm.make_lbl_tables(nwvl, 777, pl, h2o_ref, o3_ref)
    d = tmp_path_factory.mktemp("lbldiag")
    back = []
    for k, nm in enumerate(["h2o", "co2", "o3", "ch4", "n2o"]):
        path = str(d / f"lbl.{nm}.asc")
        rcm.write_lbl_asc(path, wvl, tau5[k])
        stt, x, y = rcm.ascii_file2xy2D(path)
        assert stt == 0 and np.array_equal(x, wvl) and np.array_equal(y, tau5[k])
        back.append(y)
    return dict(pl=pl, st=st, Tsurf=Tlev[:, 20].copy(), wvl=wvl, tau5=np.stack(back), h2o_ref=h2o_ref, o3_ref=o3_ref,
                ncol=ncol, nwvl=nwvl)


def make(rcm, c, co2_factor=1.0, rep=1, n=None):
    st = c["st"]
    tile = lambda a: np.tile(a, (rep,) + (1,) * (a.ndim - 1))[:n]
    s = rcm.Solver(0)
    s.set_lbl_tables(c["wvl"], c["tau5"], c["h2o_ref"], c["o3_ref"], co2_factor)
    s.set_columns(c["pl"], tile(st["Tlayer"]), tile(c["Tsurf"]), tile(st["vmr9"]), tile(st["rel_hum"]))
    return s


def next_step(s):
    s.advance(1)
    g = s.get_state(want=("E_down", "E_up", "dE"))
    return g["E_down"], g["E_up"], g["dE"]


def assert_next_step(s, **kw):
    d = s.lbl_diagnose_fluxes(**kw)
    Ed, Eu, dE = next_step(s)
    assert np.array_equal(d["E_down"], Ed) and np.array_equal(d["E_up"], Eu) and np.array_equal(d["dE"], dE)


@pytest.mark.parametrize("co2_factor", [1.0, 2.0])
def test_broadband_is_the_next_step_bit_for_bit(rcm, case, co2_factor):
    s = make(rcm, case, co2_factor)
    assert_next_step(s)                # step 0: no feedback
    s.advance(2)
    assert_next_step(s)                # after 3 steps: sort and feedback
    s.close()


def test_next_step_with_per_column_solar_and_cloud(rcm, case):
    s = make(rcm, case)
    n = case["ncol"]
    s.set_column_solar(tau_s=np.linspace(0.5, 4.0, n), mu_s=np.linspace(0.3, 0.9, n), cloud_from_tau_s=True)
    assert_next_step(s)
    s.advance(2)
    assert_next_step(s, bands=[0, 700, case["nwvl"]])   # with the band pass on too: the same broadband
    s.close()


def test_calls_move_nothing(rcm, case, tmp_path):
    nw = case["nwvl"]
    a, b = make(rcm, case), make(rcm, case)
    for s in (a, b):
        s.advance(2)
    a.lbl_diagnose_fluxes()
    a.lbl_diagnose_fluxes(vmr_scale=[1.5, 2, 0.5, 2, 2], bands=[0, 1, 128, 129, nw])
    a.lbl_diagnose_fluxes(col0=5, ncol=7, vmr_scale=[1, 3, 1, 1, 1], bands=np.arange(nw + 1))
    for s, p in ((a, "a.ck"), (b, "b.ck")):
        s.save_checkpoint(str(tmp_path / p))
    assert open(tmp_path / "a.ck", "rb").read() == open(tmp_path / "b.ck", "rb").read()
    for s in (a, b):
        s.advance(2)
    ga, gb = a.get_state(), b.get_state()
    for k in ga:
        assert np.array_equal(ga[k], gb[k]), k
    a.close(); b.close()


# ---- the C port ---------------------------------------------------------------------------------------------------------
def _p(a):
    return a.ctypes.data_as(C.c_void_p)


def port_state(port, c, g, step):
    """The state the next LBL step radiates: sorted T and the feedback's H2O (none at step 0), from the solver's state g."""
    L = port.lib()
    pl = c["pl"]
    player = (pl[:-1] + pl[1:]) / 2.0
    conv = (1000.0 / player) ** (2.0 / 7.0)
    T = np.array(g["Tlayer"], order="C")
    h2o = np.array(g["h2o"], order="C")
    rh = np.ascontiguousarray(c["st"]["rel_hum"])
    for k in range(T.shape[0]):
        L.rcmo_theta_sort(C.c_int(20), _p(T[k]), _p(conv))
        if step:
            L.rcmo_water_vapor_feedback(C.c_int(20), _p(T[k]), _p(rh[k]), _p(player), _p(h2o[k]))
    return T, h2o


def port_tau(port, c, h2o, col, f):
    """tau of column col by the definitions of rcm_lbl_diagnose_fluxes, scaled planes and scales in numpy, grey cloud added."""
    f = [1.0] * 5 if f is None else [float(x) for x in f]
    t5 = c["tau5"]
    hs = np.ascontiguousarray((f[0] * h2o[col]) / c["h2o_ref"])
    os_ = np.ascontiguousarray((f[2] * c["st"]["vmr9"][col, 2]) / c["o3_ref"])
    ch4 = np.ascontiguousarray(f[4] * t5[3])
    n2o = np.ascontiguousarray(f[3] * t5[4])
    tau = np.zeros((c["nwvl"], 20))
    port.lib().rcmo_lbl_tau(C.c_int(c["nwvl"]), C.c_int(20), _p(t5[0]), _p(t5[1]), _p(t5[2]), _p(ch4), _p(n2o), _p(hs),
                            C.c_double(f[1] * 1.0), _p(os_), _p(tau))
    tau[:, 17] += 1.0     # default grey cloud: layer 17, tau_s / 2
    return tau


def port_rt(port, p, tau, lo, hi, T, Ts):
    Ed, Eu, dE = np.zeros(21), np.zeros(21), np.zeros(20)
    port.lib().rcmo_lbl_radiative_transfer(C.byref(p), C.c_int(tau.shape[0]), _p(tau), _p(lo), _p(hi), _p(T), C.c_double(Ts),
                                           _p(Ed), _p(Eu), _p(dE))
    return Ed, Eu, dE


@pytest.mark.parametrize("steps", [0, 2])
def test_per_wavelength_and_broadband_against_the_port(rcm, port, case, steps):
    c = case
    nw = c["nwvl"]
    s = make(rcm, c)
    if steps:
        s.advance(steps)
    g = s.get_state()
    T, h2o = port_state(port, c, g, steps)
    lo, hi = port.lbl_bin_edges(c["wvl"])
    p = port.default_params(rcm.solar_setup()["solar_irr"])
    cols = [0, 13]
    for name, f in SCALES.items():
        d = s.lbl_diagnose_fluxes(vmr_scale=f, bands=np.arange(nw + 1))
        for col in cols:
            tau = port_tau(port, c, h2o, col, f)
            Ed, Eu, dE = port_rt(port, p, tau, lo, hi, T[col], g["Tsurf"][col])
            scale = np.max(np.abs(Eu))
            assert np.max(np.abs(d["E_up"][col] - Eu)) < 1e-10 * scale, name
            assert np.max(np.abs(d["E_down"][col] - Ed)) < 1e-10 * scale, name
            assert np.max(np.abs(d["dE"][col] - dE)) < 1e-10 * scale, name
            wd, wu = np.zeros((nw, 21)), np.zeros((nw, 21))
            for w in range(nw):
                wd[w], wu[w], _ = port_rt(port, p, tau[w:w + 1], lo[w:w + 1], hi[w:w + 1], T[col], g["Tsurf"][col])
            assert np.max(np.abs(d["E_down_band"][col] - wd)) < 1e-10 * scale, name
            assert np.max(np.abs(d["E_up_band"][col] - wu)) < 1e-10 * scale, name
    s.close()


def test_co2_factor_scale_equals_a_doubled_table(rcm, case, tmp_path):
    a, b = make(rcm, case, 1.0), make(rcm, case, 2.0)
    a.advance(2)
    a.save_checkpoint(str(tmp_path / "a.ck"))
    b.load_checkpoint(str(tmp_path / "a.ck"))       # the same state under the doubled table
    da = a.lbl_diagnose_fluxes(vmr_scale=[1, 2, 1, 1, 1])
    db = b.lbl_diagnose_fluxes()
    Ed, Eu, dE = next_step(b)
    for k, ref in (("E_down", Ed), ("E_up", Eu), ("dE", dE)):
        assert np.array_equal(da[k], db[k]) and np.array_equal(da[k], ref), k
    assert np.all(da["E_up"][:, 0] < a.lbl_diagnose_fluxes()["E_up"][:, 0])   # 2xCO2 lowers the OLR
    a.close(); b.close()


def test_bands_are_sequential_sums_of_the_wavelengths(rcm, case):
    nw = case["nwvl"]
    s = make(rcm, case)
    s.advance(3)
    f = [1.2, 2, 0.7, 1.5, 1.1]
    w = s.lbl_diagnose_fluxes(vmr_scale=f, bands=np.arange(nw + 1))
    rng = np.random.default_rng(5)
    parts = [[0, nw], [0, 1, 2, 3, nw], [0, 127, 128, 129, 300, 511, 513, nw - 1, nw],
             np.unique(np.concatenate([[0, nw], rng.choice(np.arange(1, nw), 40, replace=False)]))]
    for bs in parts:
        bs = np.asarray(bs)
        d = s.lbl_diagnose_fluxes(vmr_scale=f, bands=bs)
        for k in ("E_down_band", "E_up_band"):
            ref = np.stack([np.cumsum(w[k][:, a:b], axis=1)[:, -1] for a, b in zip(bs[:-1], bs[1:])], axis=1)
            assert np.array_equal(d[k], ref), (k, bs[:5])
    one = s.lbl_diagnose_fluxes(vmr_scale=f, bands=[0, nw])
    scale = np.max(np.abs(one["E_up"]), axis=1, keepdims=True)
    assert np.max(np.abs(one["E_up_band"][:, 0] - one["E_up"]) / scale) < 1e-12
    assert np.max(np.abs(one["E_down_band"][:, 0] - one["E_down"]) / scale) < 1e-12
    s.close()


def test_ranges_columns_and_chunks_give_the_same_rows(rcm, case):
    nw = case["nwvl"]
    n = 8200                                # > 8,192 (broadband chunk) and > 3,968 (band chunk at 1,500 wavelengths); ragged
    s = make(rcm, case, 2.0, rep=n // case["ncol"] + 1, n=n)
    s.advance(2)
    bands = [0, 100, 129, 1000, nw]
    f = [1, 1, 1, 2, 1]
    whole = s.lbl_diagnose_fluxes(vmr_scale=f, bands=bands)
    for col0, m in ((0, 24), (8190, 10), (3960, 17), (8199, 1), (11, 1)):
        sub = s.lbl_diagnose_fluxes(col0=col0, ncol=m, vmr_scale=f, bands=bands)
        for k in sub:
            assert np.array_equal(sub[k], whole[k][col0:col0 + m]), (k, col0)
    per = whole["E_up_band"]
    assert np.array_equal(per[0], per[case["ncol"]]) and np.array_equal(per[5], per[8184 + 5])   # replicated columns
    assert_next_step(s)
    s.close()


def test_errors_leave_the_solver_usable(rcm, case):
    nw = case["nwvl"]
    L = rcm.load_library()
    ref = make(rcm, case)
    ref_next = next_step(ref)
    ref.close()
    s = make(rcm, case)
    h = s._h

    def call(col0=0, ncol=24, sc=None, nband=2, bs=(0, 10, nw), bands=True):
        scv = None if sc is None else np.ascontiguousarray(sc, dtype=np.float64)
        bsv = None if bs is None else np.ascontiguousarray(bs, dtype=np.int32)
        out = np.zeros((ncol if ncol > 0 else 1) * max(nband, 1) * 21)
        o2 = np.zeros((ncol if ncol > 0 else 1) * 21)
        return L.rcm_lbl_diagnose_fluxes(h, C.c_int(col0), C.c_int(ncol), None if scv is None else _p(scv), C.c_int(nband),
                                         None if bsv is None else _p(bsv), _p(out) if bands else None, None, _p(o2), None, None)

    assert call() == 0
    assert call(col0=-1) == 1 and call(col0=20, ncol=5) == 1 and call(ncol=0) == 1
    for bad in ([-1, 1, 1, 1, 1], [1, np.nan, 1, 1, 1], [1, 1, np.inf, 1, 1]):
        assert call(sc=bad) == 1
    assert call(nband=0, bs=(0,)) == 1
    assert call(bs=None) == 1
    assert call(bs=(0, 10, 10)) == 1 and call(bs=(0, 20, 10)) == 1
    assert call(bs=(1, 10, nw)) == 1 and call(bs=(0, 10, nw - 1)) == 1 and call(bs=(0, 10, nw + 1)) == 1
    assert call(bs=None, bands=False) == 0                       # band_start is read only for band outputs
    got = next_step(s)
    assert all(np.array_equal(x, y) for x, y in zip(got, ref_next))
    s.close()
    # not on the LBL path; no columns; another species_mask
    r = rcm.Solver(0)
    r.set_repwvl_table_from(rcm.Table(table_path(10)))
    st = case["st"]
    r.set_columns(case["pl"], st["Tlayer"], case["Tsurf"], st["vmr9"], st["rel_hum"])
    assert L.rcm_lbl_diagnose_fluxes(r._h, 0, 24, None, 0, None, None, None, _p(np.zeros(24 * 21)), None, None) == 2
    r.close()
    e = rcm.Solver(0)
    e.set_lbl_tables(case["wvl"], case["tau5"], case["h2o_ref"], case["o3_ref"], 1.0)
    assert L.rcm_lbl_diagnose_fluxes(e._h, 0, 1, None, 0, None, None, None, _p(np.zeros(21)), None, None) == 2
    e.close()
    p = rcm.default_params()
    p.species_mask = 0b111
    m = rcm.Solver(0, p)
    m.set_lbl_tables(case["wvl"], case["tau5"], case["h2o_ref"], case["o3_ref"], 1.0)
    m.set_columns(case["pl"], st["Tlayer"], case["Tsurf"], st["vmr9"], st["rel_hum"])
    assert L.rcm_lbl_diagnose_fluxes(m._h, 0, 24, None, 0, None, None, None, _p(np.zeros(24 * 21)), None, None) == 2
    m.advance(1)
    m.close()


# ---- the C++ driver -----------------------------------------------------------------------------------------------------
def test_driver_band_file(rcm, tmp_path):
    exe = os.path.join(os.path.dirname(rcm.library_path()), "rcm_rce")
    lbl_atm = os.path.join(GOLDEN, "column21.lbl.atm")
    atm = rcm.read_atm(lbl_atm)
    pl = atm[:, 1].copy()
    vbase = np.stack([atm[:, 4], atm[:, 5], np.full(21, 400.0), np.full(21, 1.7), np.full(21, 0.315)])
    ncol, seed, nwvl, K = 6, 77, 700, 64
    Tlev, vlev = rcm.make_ensemble(ncol, seed, pl, atm[:, 2].copy(), vbase)
    st = rcm.init_columns(pl, Tlev, vlev)
    h2o_ref, o3_ref = st["vmr9"][0, 0].copy(), st["vmr9"][0, 2].copy()
    wvl, tau5 = rcm.make_lbl_tables(nwvl, 777, pl, h2o_ref, o3_ref)
    d = tmp_path / "lbl"
    d.mkdir()
    for k, nm in enumerate(["h2o", "co2", "o3", "ch4", "n2o"]):
        rcm.write_lbl_asc(str(d / f"lbl.{nm}.asc"), wvl, tau5[k])
    common = ["--atm", lbl_atm, "--lbl", str(d), "--ncol", str(ncol), "--seed", str(seed), "--max-steps", "2", "--steps-exact",
              "--band-size", str(K), "--forcing-scale", "1,2,1,1,1.5"]
    f1 = str(tmp_path / "bands1.csv")
    r = subprocess.run([exe, *common, "--out", str(tmp_path / "o1.txt"), "--lbl-bands-out", f1], capture_output=True, text=True,
                       timeout=300)
    assert r.returncode == 0, r.stderr
    s = rcm.Solver(0)
    s.set_lbl_tables(wvl, tau5, h2o_ref, o3_ref, 1.0)
    s.set_columns(pl, st["Tlayer"], 288.2, st["vmr9"], st["rel_hum"])
    s.advance(2)
    bs = np.append(np.arange(0, nwvl, K), nwvl)
    u = s.lbl_diagnose_fluxes(bands=bs)
    v = s.lbl_diagnose_fluxes(bands=bs, vmr_scale=[1, 2, 1, 1, 1.5])
    s.close()
    dl = np.diff(wvl)
    lo = wvl - np.concatenate([[dl[0]], dl]) / 2.0
    hi = wvl + np.concatenate([dl, [dl[-1]]]) / 2.0

    def mean(x):            # summed in column order, divided once
        acc = np.zeros(x.shape[1:])
        for row in x:
            acc = acc + row
        return acc / x.shape[0]

    cols = [mean(u["E_up_band"][:, :, 0]), mean(u["E_down_band"][:, :, 20]), mean(v["E_up_band"][:, :, 0]),
            mean(v["E_down_band"][:, :, 20])]
    lines = open(f1).read().splitlines()
    assert lines[0] == "wvl_lo_nm,wvl_hi_nm,olr,surface_down,olr_scaled,surface_down_scaled"
    assert len(lines) == len(bs)
    for b, line in enumerate(lines[1:]):
        vals = [float(x) for x in line.split(",")]
        assert vals[0] == lo[bs[b]] and vals[1] == hi[bs[b + 1] - 1]
        assert vals[2:] == [cols[q][b] for q in range(4)], b
    # refused with a repwvl table
    r = subprocess.run([exe, "--atm", os.path.join(GOLDEN, "column21.atm"), "--table", table_path(10), "--max-steps", "1",
                        "--lbl-bands-out", str(tmp_path / "x.csv")], capture_output=True, text=True)
    assert r.returncode == 1 and "--lbl-bands-out" in r.stderr
    # the same bytes on two GPUs
    if rcm.device_count() < 2:
        pytest.skip("the --gpus 2 half needs two GPUs")
    f2 = str(tmp_path / "bands2.csv")
    r = subprocess.run([exe, *common, "--out", str(tmp_path / "o2.txt"), "--lbl-bands-out", f2, "--gpus", "2"],
                       capture_output=True, text=True, timeout=300)
    assert r.returncode == 0, r.stderr
    assert open(f1, "rb").read() == open(f2, "rb").read()
