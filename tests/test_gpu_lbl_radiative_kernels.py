"""Radiative kernels of the line-by-line path (rcm_lbl_radiative_kernels / Solver.lbl_radiative_kernels): analytic derivatives
of the next LBL step's OLR and surface downward flux in T_l, T_surf and ln q_l, broadband and per band, against central
differences of the C port (rcmo_lbl_tau + rcmo_lbl_radiative_transfer), against central differences of the GPU flux call, as
sequential sums, column by column, without moving the state.
"""
import ctypes as C
import os
import subprocess

import numpy as np
import pytest

from conftest import GOLDEN, table_path
from test_gpu_lbl_diagnostics import _p, case, make, port_rt, port_state, port_tau  # noqa: F401 (case is a fixture)

pytestmark = pytest.mark.gpu

NLAY, NE = 20, 41
HT, HQ = 1e-2, 1e-4          # central-difference steps: K in T, ln q
OPT_CUBES, OPT_PAIRS = 0, 4
SCALED = [1.5, 2, 1, 1, 1]   # H2O x1.5, CO2 x2 (ascending species index)


def make_case(rcm, nwvl, seed=4242, ncol=24):
    """case of test_gpu_lbl_diagnostics with another number of wavelengths (no ASCII round trip)."""
    atm = rcm.read_atm(os.path.join(GOLDEN, "column21.lbl.atm"))
    full = rcm.read_atm(os.path.join(GOLDEN, "column21.atm"))
    pl = atm[:, 1].copy()
    Tlev, vlev = rcm.make_ensemble(ncol, seed, pl, atm[:, 2].copy(), full[:, 4:9].T.copy())
    st = rcm.init_columns(pl, Tlev, vlev)
    h2o_ref, o3_ref = st["vmr9"][0, 0].copy(), st["vmr9"][0, 2].copy()
    wvl, tau5 = rcm.make_lbl_tables(nwvl, 777, pl, h2o_ref, o3_ref)
    return dict(pl=pl, st=st, Tsurf=Tlev[:, 20].copy(), wvl=wvl, tau5=np.ascontiguousarray(tau5), h2o_ref=h2o_ref,
                o3_ref=o3_ref, ncol=ncol, nwvl=nwvl)


@pytest.fixture(scope="module")
def case200(rcm):
    return make_case(rcm, 200)


def solver(rcm, c, params=None, cubes=None, pairs=None):
    st = c["st"]
    s = rcm.Solver(0, params) if params is not None else rcm.Solver(0)
    s.set_lbl_tables(c["wvl"], c["tau5"], c["h2o_ref"], c["o3_ref"], 1.0)
    s.set_columns(c["pl"], st["Tlayer"], c["Tsurf"], st["vmr9"], st["rel_hum"])
    if cubes is not None:
        s.set_option(OPT_CUBES, cubes)
    if pairs is not None:
        s.set_option(OPT_PAIRS, pairs)
    return s


# ---- the port's central differences ---------------------------------------------------------------------------------------
def simpson_order(lo, hi, T):
    """n at which the port's cplkavg (rcm_oracle.c) stops its Simpson loop for each bin [lo, hi] at T; 0 off that branch."""
    c2, vmax = 1.438786, np.log(np.finfo(float).max)
    whi, wlo = 1.0e7 / lo, 1.0e7 / hi
    v0, v1 = c2 * wlo / T, c2 * whi / T
    simp = (v0 > np.finfo(float).eps) & (v1 < vmax) & ((whi - wlo) / whi < 1e-2)
    f = lambda x: x ** 3 / np.expm1(x)
    hh = v1 - v0
    n_at = np.zeros(lo.size, dtype=int)
    old = np.zeros(lo.size)
    for n in range(1, 11):
        d = hh / (2 * n)
        val = f(v0) + f(v1)
        for k in range(1, 2 * n):
            val = val + 2 * (1 + k % 2) * f(v0 + k * d)
        val = val * d / 3.0
        stop = (n_at == 0) & (np.abs((val - old) / val) <= 1e-6)
        n_at[stop] = n
        old = val
    n_at[(n_at == 0) & simp] = 10
    return np.where(simp, n_at, 0)


VCP = np.array([10.25, 5.7, 3.9, 2.9, 2.3, 1.9])   # the series' term-count thresholds (rcm_oracle.c)


def series_regime(lo, hi, T):
    """per bin which pieces the port's series branch uses at T: the polynomial below v = 1.5, else the number of terms"""
    c2 = 1.438786
    reg = lambda v: np.where(v < 1.5, 0, 1 + (v[:, None] < VCP[None, :]).sum(axis=1))
    return 100 * reg(c2 * (1.0e7 / hi) / T) + reg(c2 * (1.0e7 / lo) / T)


# The port's series branch (wide bins) is a piecewise approximation of the integral: its B agrees with the integral's own
# derivative, 4B/T - K T^3 (v1 f(v1) - v0 f(v0)), only to 8.3e-4 of dB/dT per bin on the 200-wavelength tables (worst at the
# polynomial / series seam v = 1.5), while on the Simpson branch dB/dT is the exact derivative of the port's value.
BAR = {1500: 1e-6, 200: 1e-3}


class Port:
    """F = (E_up[0], E_down[20]) of one column by the port, and its central differences in the 41 entries."""

    def __init__(self, port, c, g, steps, f=None, nangle=30, cloud=None):
        self.port, self.c, self.f = port, c, f
        self.T, self.h2o = port_state(port, c, g, steps)
        self.Ts = g["Tsurf"]
        self.lo, self.hi = port.lbl_bin_edges(c["wvl"])
        self.p = port.default_params(0.0)
        self.p.nangle = nangle
        self.cloud = cloud            # per-column cloud tau on layer 17, or None (the default grey cloud, 1.0)

    def tau(self, col, h2o):
        t = port_tau(self.port, self.c, h2o, col, self.f)
        if self.cloud is not None:
            t[:, 17] = t[:, 17] - 1.0 + self.cloud[col]
        return t

    def F(self, col, w, tau, T, Ts):
        sl = slice(None) if w is None else (slice(w, w + 1) if np.isscalar(w) else w)
        Ed, Eu, _ = port_rt(self.port, self.p, np.ascontiguousarray(tau[sl]), np.ascontiguousarray(self.lo[sl]),
                            np.ascontiguousarray(self.hi[sl]), T, Ts)
        return np.array([Eu[0], Ed[20]])

    def K(self, col, w=None):
        """[2][41] central differences; w: one wavelength (index), an index array, or None for all."""
        T, Ts = self.T[col], self.Ts[col]
        tau0 = self.tau(col, self.h2o)
        K = np.zeros((2, NE))
        for l in range(NLAY):
            Tp, Tm = T.copy(), T.copy()
            Tp[l] += HT
            Tm[l] -= HT
            K[:, l] = (self.F(col, w, tau0, Tp, Ts) - self.F(col, w, tau0, Tm, Ts)) / (2 * HT)
            hp, hm = self.h2o.copy(), self.h2o.copy()
            hp[col, l] *= np.exp(HQ)
            hm[col, l] *= np.exp(-HQ)
            K[:, NLAY + 1 + l] = (self.F(col, w, self.tau(col, hp), T, Ts) - self.F(col, w, self.tau(col, hm), T, Ts)) / (2 * HQ)
        K[:, NLAY] = (self.F(col, w, tau0, T, Ts + HT) - self.F(col, w, tau0, T, Ts - HT)) / (2 * HT)
        return K

    def order_changes(self, col):
        """[nwvl] True where the port's Simpson order, or the pieces of its series, differ between T - h and T + h for a
        layer or the surface: its B jumps there and a central difference is no derivative."""
        out = np.zeros(self.lo.size, dtype=bool)
        for t in list(self.T[col]) + [self.Ts[col]]:
            out |= simpson_order(self.lo, self.hi, t - HT) != simpson_order(self.lo, self.hi, t + HT)
            out |= series_regime(self.lo, self.hi, t - HT) != series_regime(self.lo, self.hi, t + HT)
        return out


def assert_rows(got, ref, what, bar=1e-6):
    """every entry within bar of the max |K| of its output"""
    for o in range(2):
        scale = np.max(np.abs(ref[..., o, :]))
        err = np.max(np.abs(got[..., o, :] - ref[..., o, :]))
        assert err <= bar * scale, (what, o, err, scale)


@pytest.mark.parametrize("nwvl", [1500, 200])
@pytest.mark.parametrize("steps", [0, 3])
@pytest.mark.parametrize("scaled", [False, True])
def test_broadband_against_port_central_differences(rcm, port, case, case200, nwvl, steps, scaled):
    """1,500 wavelengths: narrow bins, the Simpson branch; 200: relative bin width 1.6e-2, the series of cplkavg_dev."""
    c = case if nwvl == 1500 else case200
    s = solver(rcm, c)
    if steps:
        s.advance(steps)
    g = s.get_state()
    f = SCALED if scaled else None
    k = s.lbl_radiative_kernels(vmr_scale=f, bands=np.arange(nwvl + 1))
    P = Port(port, c, g, steps, f)
    lo, hi = P.lo, P.hi
    narrow = simpson_order(lo, hi, 250.0) > 0
    assert narrow.all() if nwvl == 1500 else not narrow.any()
    skipped = 0
    for col in (0, 7, 13):
        moved = P.order_changes(col)
        skipped += int(moved.sum())
        if moved.any():   # both sides over the other wavelengths: the GPU's one-wavelength bands summed in index order
            keep = np.flatnonzero(~moved)
            got = np.cumsum(k["K_band"][col, keep], axis=0)[-1]
            assert_rows(got, P.K(col, keep), (nwvl, steps, scaled, col), BAR[nwvl])
        else:
            assert_rows(k["K"][col], P.K(col), (nwvl, steps, scaled, col), BAR[nwvl])
        assert k["K"][col, 1, NLAY] == 0.0
    # a wavelength whose port B jumps within +-h (Simpson order, series pieces) is counted and bounded
    assert skipped <= 0.02 * 3 * nwvl, skipped
    s.close()


@pytest.mark.parametrize("nwvl", [1500, 200])
def test_one_wavelength_bands_against_port_differences(rcm, port, case, case200, nwvl):
    c = case if nwvl == 1500 else case200
    s = solver(rcm, c)
    s.advance(3)
    g = s.get_state()
    kb = s.lbl_radiative_kernels(vmr_scale=SCALED, bands=np.arange(c["nwvl"] + 1))["K_band"]
    P = Port(port, c, g, 3, SCALED)
    ws = np.arange(0, c["nwvl"], 7 if nwvl == 1500 else 1)
    excluded = 0
    for col in (2, 19):
        moved = P.order_changes(col)
        keep = [w for w in ws if not moved[w]]
        excluded += len(ws) - len(keep)
        ref = np.stack([P.K(col, w) for w in keep])
        assert_rows(kb[col, keep], ref, (nwvl, col), BAR[nwvl])
        assert np.all(kb[col, :, 1, NLAY] == 0.0)
    # a wavelength whose port B jumps within +-h has no central difference to compare with: counted, bounded
    assert excluded <= 0.02 * 2 * len(ws), excluded
    s.close()


def test_per_column_cloud_and_solar_against_the_port(rcm, port, case):
    c = case
    s = solver(rcm, c)
    n = c["ncol"]
    tau_s = np.linspace(0.5, 4.0, n)
    s.set_column_solar(tau_s=tau_s, mu_s=np.linspace(0.3, 0.9, n), cloud_from_tau_s=True)
    s.advance(2)
    g = s.get_state()
    k = s.lbl_radiative_kernels()
    P = Port(port, c, g, 2, None, cloud=tau_s / 2.0)
    for col in (1, 22):
        assert_rows(k["K"][col], P.K(col), col)
    s.close()


# (nangle, cube chains, pair units): other quadratures than the default 30 angles with both
@pytest.mark.parametrize("nangle,cubes,pairs", [(20, 1, 1), (30, 0, 1), (30, 1, 0), (7, 1, 1)])
def test_angle_schedules_against_the_port(rcm, port, case, nangle, cubes, pairs):
    c = case
    p = rcm.default_params()
    p.nangle = nangle
    s = solver(rcm, c, p, cubes, pairs)
    s.advance(2)
    g = s.get_state()
    k = s.lbl_radiative_kernels(vmr_scale=SCALED)
    P = Port(port, c, g, 2, SCALED, nangle=nangle)
    for col in (0, 17):
        assert_rows(k["K"][col], P.K(col), (nangle, cubes, pairs, col))
    s.close()


def test_sums_in_a_fixed_order(rcm, case):
    nw = case["nwvl"]
    s = make(rcm, case)
    s.advance(3)
    f = [1.2, 2, 0.7, 1.5, 1.1]
    one = s.lbl_radiative_kernels(vmr_scale=f, bands=np.arange(nw + 1))
    whole = s.lbl_radiative_kernels(vmr_scale=f, bands=[0, nw])
    assert np.array_equal(whole["K"], whole["K_band"][:, 0]) and np.array_equal(whole["K"], one["K"])
    assert np.all(whole["K"][:, 1, NLAY] == 0.0)
    rng = np.random.default_rng(5)
    parts = [[0, 1, 2, 3, nw], [0, 127, 128, 129, 300, 511, 513, nw - 1, nw],
             np.unique(np.concatenate([[0, nw], rng.choice(np.arange(1, nw), 40, replace=False)]))]
    for bs in parts:
        bs = np.asarray(bs)
        d = s.lbl_radiative_kernels(vmr_scale=f, bands=bs)
        ref = np.stack([np.cumsum(one["K_band"][:, a:b], axis=1)[:, -1] for a, b in zip(bs[:-1], bs[1:])], axis=1)
        assert np.array_equal(d["K_band"], ref), bs[:5]
        assert np.array_equal(d["K"], whole["K"])
    acc = np.zeros_like(whole["K"])
    for w in range(nw):
        acc = acc + one["K_band"][:, w]
    assert np.array_equal(acc, whole["K"])
    s.close()


def test_ranges_columns_and_chunks_give_the_same_rows(rcm, case):
    nw = case["nwvl"]
    n = 4200                     # the call's chunk at 1,500 wavelengths: 2e9 / (1500 x 82 x 8) -> 2,032 columns; three chunks
    s = make(rcm, case, 1.0, rep=n // case["ncol"] + 1, n=n)
    s.advance(2)
    bands = [0, 100, 129, 1000, nw]
    f = [1, 1, 1, 2, 1.3]
    whole = s.lbl_radiative_kernels(vmr_scale=f, bands=bands)
    for col0, m in ((0, 24), (2030, 10), (4060, 17), (4199, 1), (11, 1), (1000, 3100)):
        sub = s.lbl_radiative_kernels(col0=col0, ncol=m, vmr_scale=f, bands=bands)
        for key in ("K", "K_band"):
            assert np.array_equal(sub[key], whole[key][col0:col0 + m]), (key, col0)
    per = whole["K_band"]
    assert np.array_equal(per[0], per[case["ncol"]]) and np.array_equal(per[5], per[4176 + 5])   # replicated columns
    s.close()


def test_calls_move_nothing(rcm, case, tmp_path):
    nw = case["nwvl"]
    a, b = make(rcm, case), make(rcm, case)
    for s in (a, b):
        s.advance(2)
    a.lbl_radiative_kernels()
    a.lbl_radiative_kernels(vmr_scale=[1.5, 2, 0.5, 2, 2], bands=[0, 1, 128, 129, nw])
    a.lbl_radiative_kernels(col0=5, ncol=7, vmr_scale=[1, 3, 1, 1, 1], bands=np.arange(nw + 1))
    for s, p in ((a, "a.ck"), (b, "b.ck")):
        s.save_checkpoint(str(tmp_path / p))
    assert open(tmp_path / "a.ck", "rb").read() == open(tmp_path / "b.ck", "rb").read()
    for s in (a, b):
        s.advance(2)
    ga, gb = a.get_state(), b.get_state()
    for k in ga:
        assert np.array_equal(ga[k], gb[k]), k
    a.close(); b.close()


def test_self_consistency_with_the_flux_call_on_the_bench_workload(rcm):
    """4,096 columns x 20,000 wavelengths (bench.py's LBL case) at step 0: the kernels' sums against central differences of
    rcm_lbl_diagnose_fluxes - in ln q through f_H2O = e^(+-eps), in T on two solvers with every layer and the surface
    shifted by +-h."""
    c = make_case(rcm, 20000, 4242, 4096)
    st = c["st"]
    s = solver(rcm, c)
    k = s.lbl_radiative_kernels()["K"]
    eps, h = 1e-4, 1e-2
    up = s.lbl_diagnose_fluxes(vmr_scale=[np.exp(eps), 1, 1, 1, 1])
    dn = s.lbl_diagnose_fluxes(vmr_scale=[np.exp(-eps), 1, 1, 1, 1])
    F = lambda d: np.stack([d["E_up"][:, 0], d["E_down"][:, 20]], axis=1)
    dq = (F(up) - F(dn)) / (2 * eps)
    scale = np.max(np.abs(k), axis=2)
    assert np.all(np.abs(k[:, :, NLAY + 1:].sum(axis=2) - dq) <= 1e-6 * scale)
    s.close()
    Fs = []
    for sign in (1, -1):
        t = rcm.Solver(0)
        t.set_lbl_tables(c["wvl"], c["tau5"], c["h2o_ref"], c["o3_ref"], 1.0)
        t.set_columns(c["pl"], st["Tlayer"] + sign * h, c["Tsurf"] + sign * h, st["vmr9"], st["rel_hum"])
        Fs.append(F(t.lbl_diagnose_fluxes()))
        t.close()
    dT = (Fs[0] - Fs[1]) / (2 * h)
    pl = c["pl"]
    conv = (1000.0 / ((pl[:-1] + pl[1:]) / 2.0)) ** (2.0 / 7.0)
    ident = lambda T: np.all(np.diff(T * conv, axis=1) < 0, axis=1)   # theta falls with the layer index: the sort moves nothing
    ok = ident(st["Tlayer"]) & ident(st["Tlayer"] + h) & ident(st["Tlayer"] - h)
    skipped = int((~ok).sum())
    assert skipped <= st["Tlayer"].shape[0] // 2, skipped
    got = k[:, :, :NLAY + 1].sum(axis=2)
    assert np.all(np.abs(got - dT)[ok] <= 1e-6 * scale[ok])


def test_clamped_layers_have_zero_ln_q_entries(rcm, port, case):
    """The default schedule (30 angles, cube chains and pair units) clamps tau in front of the sweep (clampk = 0: its
    tau_clamp x min(1/mu) exceeds 92.2; without cube chains the exp clamps instead, test_gpu_diagnostic_configs).  With H2O
    x1e6 some tau exceed 999 ln2 >= tau_clamp: those (wavelength, layer) ln q entries are exactly 0.0."""
    c = case
    s = make(rcm, c)
    f = [1e6, 1, 1, 1, 1]
    kb = s.lbl_radiative_kernels(vmr_scale=f, bands=np.arange(c["nwvl"] + 1))["K_band"]
    g = s.get_state()
    T, h2o = port_state(port, c, g, 0)
    for col in (0, 9):
        tau = port_tau(port, c, h2o, col, f)
        hit = tau > 999 * np.log(2.0) * 1.001
        assert hit.sum() > 0
        for o in range(2):
            assert np.all(kb[col, :, o, NLAY + 1:][hit] == 0.0)
        assert np.any(kb[col, :, 0, NLAY + 1:][~hit] != 0.0)
    s.close()


def test_errors_leave_the_solver_usable(rcm, case):
    nw = case["nwvl"]
    L = rcm.load_library()
    ref = make(rcm, case)
    ref.advance(1)
    ref_next = ref.get_state()
    ref.close()
    s = make(rcm, case)
    h = s._h

    def call(col0=0, ncol=24, sc=None, nband=2, bs=(0, 10, nw), bands=True, broad=True):
        scv = None if sc is None else np.ascontiguousarray(sc, dtype=np.float64)
        bsv = None if bs is None else np.ascontiguousarray(bs, dtype=np.int32)
        kb = np.zeros(max(ncol, 1) * max(nband, 1) * 82)
        k = np.zeros(max(ncol, 1) * 82)
        return L.rcm_lbl_radiative_kernels(h, C.c_int(col0), C.c_int(ncol), None if scv is None else _p(scv), C.c_int(nband),
                                           None if bsv is None else _p(bsv), _p(kb) if bands else None, _p(k) if broad else None)

    assert call() == 0
    assert call(col0=-1) == 1 and call(col0=20, ncol=5) == 1 and call(ncol=0) == 1
    for bad in ([-1, 1, 1, 1, 1], [1, np.nan, 1, 1, 1], [1, 1, np.inf, 1, 1]):
        assert call(sc=bad) == 1
    assert call(nband=0, bs=(0,)) == 1
    assert call(bs=None) == 1
    assert call(bs=(0, 10, 10)) == 1 and call(bs=(0, 20, 10)) == 1
    assert call(bs=(1, 10, nw)) == 1 and call(bs=(0, 10, nw - 1)) == 1 and call(bs=(0, 10, nw + 1)) == 1
    assert call(bs=None, bands=False) == 0                       # band_start is read only for K_band
    assert call(bs=None, nband=0, bands=False, broad=False) == 0  # nothing wanted
    assert L.rcm_radiative_kernels(h, 0, 24, None, None, _p(np.zeros(24 * 82))) == 2   # the repwvl call refuses LBL
    s.advance(1)
    got = s.get_state()
    for key in got:
        assert np.array_equal(got[key], ref_next[key]), key
    s.close()
    r = rcm.Solver(0)
    r.set_repwvl_table_from(rcm.Table(table_path(10)))
    st = case["st"]
    r.set_columns(case["pl"], st["Tlayer"], case["Tsurf"], st["vmr9"], st["rel_hum"])
    assert L.rcm_lbl_radiative_kernels(r._h, 0, 24, None, 0, None, None, _p(np.zeros(24 * 82))) == 2
    r.close()
    e = rcm.Solver(0)
    e.set_lbl_tables(case["wvl"], case["tau5"], case["h2o_ref"], case["o3_ref"], 1.0)
    assert L.rcm_lbl_radiative_kernels(e._h, 0, 1, None, 0, None, None, _p(np.zeros(82))) == 2
    e.close()
    p = rcm.default_params()
    p.species_mask = 0b111
    m = rcm.Solver(0, p)
    m.set_lbl_tables(case["wvl"], case["tau5"], case["h2o_ref"], case["o3_ref"], 1.0)
    m.set_columns(case["pl"], st["Tlayer"], case["Tsurf"], st["vmr9"], st["rel_hum"])
    assert L.rcm_lbl_radiative_kernels(m._h, 0, 24, None, 0, None, None, _p(np.zeros(24 * 82))) == 2
    m.advance(1)
    m.close()


# ---- the C++ driver -----------------------------------------------------------------------------------------------------
def test_driver_lbl_kernels_file(rcm, tmp_path):
    exe = os.path.join(os.path.dirname(rcm.library_path()), "rcm_rce")
    lbl_atm = os.path.join(GOLDEN, "column21.lbl.atm")
    atm = rcm.read_atm(lbl_atm)
    pl = atm[:, 1].copy()
    vbase = np.stack([atm[:, 4], atm[:, 5], np.full(21, 400.0), np.full(21, 1.7), np.full(21, 0.315)])
    ncol, seed, nwvl = 6, 77, 700
    Tlev, vlev = rcm.make_ensemble(ncol, seed, pl, atm[:, 2].copy(), vbase)
    st = rcm.init_columns(pl, Tlev, vlev)
    h2o_ref, o3_ref = st["vmr9"][0, 0].copy(), st["vmr9"][0, 2].copy()
    wvl, tau5 = rcm.make_lbl_tables(nwvl, 777, pl, h2o_ref, o3_ref)
    d = tmp_path / "lbl"
    d.mkdir()
    for k, nm in enumerate(["h2o", "co2", "o3", "ch4", "n2o"]):
        rcm.write_lbl_asc(str(d / f"lbl.{nm}.asc"), wvl, tau5[k])
    common = ["--atm", lbl_atm, "--lbl", str(d), "--ncol", str(ncol), "--seed", str(seed), "--max-steps", "2", "--steps-exact"]
    f1 = str(tmp_path / "k1.csv")
    r = subprocess.run([exe, *common, "--out", str(tmp_path / "o1.txt"), "--lbl-kernels-out", f1], capture_output=True,
                       text=True, timeout=300)
    assert r.returncode == 0, r.stderr
    s = rcm.Solver(0)
    s.set_lbl_tables(wvl, tau5, h2o_ref, o3_ref, 1.0)
    s.set_columns(pl, st["Tlayer"], 288.2, st["vmr9"], st["rel_hum"])
    s.advance(2)
    K = s.lbl_radiative_kernels()["K"]
    s.close()
    acc = np.zeros((2, NE))
    for row in K:             # column order, then one division: the driver's arithmetic
        acc = acc + row
    mean = acc / K.shape[0]
    lines = open(f1).read().splitlines()
    assert lines[0] == "layer,p_layer,dOLR_dT,dOLR_dlnq,dSFC_dT,dSFC_dlnq" and len(lines) == NLAY + 2
    assert [l.split(",")[0] for l in lines[1:]] == [str(l) for l in range(NLAY)] + ["surface"]
    rows = np.array([[float(x) for x in l.split(",")[1:]] for l in lines[1:]])
    assert np.array_equal(rows[:NLAY, 0], (pl[:NLAY] + pl[1:]) / 2.0) and rows[NLAY, 0] == pl[NLAY]
    assert np.array_equal(rows[:NLAY, 1], mean[0, :NLAY]) and np.array_equal(rows[:NLAY, 2], mean[0, NLAY + 1:])
    assert np.array_equal(rows[:NLAY, 3], mean[1, :NLAY]) and np.array_equal(rows[:NLAY, 4], mean[1, NLAY + 1:])
    assert np.array_equal(rows[NLAY, 1:], [mean[0, NLAY], 0.0, 0.0, 0.0])
    # refused with a repwvl table
    r = subprocess.run([exe, "--atm", os.path.join(GOLDEN, "column21.atm"), "--table", table_path(10), "--max-steps", "1",
                        "--lbl-kernels-out", str(tmp_path / "x.csv")], capture_output=True, text=True)
    assert r.returncode == 1 and "--lbl-kernels-out" in r.stderr
    if rcm.device_count() < 2:
        pytest.skip("the --gpus 2 half needs two GPUs")
    f2 = str(tmp_path / "k2.csv")
    r = subprocess.run([exe, *common, "--out", str(tmp_path / "o2.txt"), "--lbl-kernels-out", f2, "--gpus", "2"],
                       capture_output=True, text=True, timeout=300)
    assert r.returncode == 0, r.stderr
    assert open(f1, "rb").read() == open(f2, "rb").read()
