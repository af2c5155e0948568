"""The diagnostic, kernel and Jacobian calls (diagnose_fluxes, radiative_kernels, flux_jacobian) away from the configuration
their own files test: other angle schedules (both instances of every kernel's exponent clamp, padding chains, a schedule of
one pair unit and no chain, MAX_ANGLE), other cloud layers and none, the 10- and 100-wavelength tables, profiles at the edges
of the table (tau below the kernels' floor, extrapolated cross sections, tau above the upper clamp), the chunk boundary, and
the __constant__ bank shared by several solvers on one device.

Checker: the C port of the reference (oracle/rcm_oracle.c) with the schedule's nangle and cloud layer.  Its fluxes are taken
per wavelength and their central differences once per column (port_derivatives); the radiative kernels K are the rows
E_up[0] and E_down[20] of the same differences.  On the edge profiles the reference is the port's tau floored at TAU_FLOOR,
the kernels' documented model (DESIGN.md section 4; it equals the plain port's tau wherever tau >= -8), radiated by
two_stream: behind a layer with tau < 0 the port's 1 - alpha form loses transmissions that still matter (see two_stream).
"""
import os

import numpy as np
import pytest

from conftest import GOLDEN, table_path
from test_gpu_diagnostics import ensemble, solver
from test_gpu_flux_jacobian import heating_jacobian
from test_gpu_radiative_kernels import EPS, H, radiated_inputs

pytestmark = pytest.mark.gpu
NLAY, NLEV, NE = 20, 21, 41
OPT_CUBES, OPT_PAIRS = 0, 4
TAU_FLOOR = -8.0
RATE = 1e-2  # largest change of any exponent tau / mu over one difference step (see port_derivatives)


# ---- the port's fluxes and their central differences -------------------------------------------------------------------
def planck(wvl_nm, weight, T):
    """rcmo_planck (main.cpp:186-204) on arrays"""
    h, c, kB = 6.62607e-34, 299792458.0, 1.380649e-23
    wvl = wvl_nm * 1e-9
    return weight * 2 * h * c ** 2 / (wvl ** 5 * (np.exp(h * c / (wvl * kB * T)) - 1)) / 1e9


def two_stream(tau, wvl, weight, T, Ts, nangle):
    """Per-wavelength E_down, E_up [nwvl][2][21] of main.cpp:291-318 with the transmission t = exp(-tau / mu) where the
    reference writes 1 - alpha, alpha = 1 - exp(-tau / mu): L = t (L - B) + B, as the kernels.  The same expression, but
    1 - alpha is exactly 0 for t < 2^-53, and behind a layer with tau < 0 (t up to e^480 at the floor) the radiance that such a
    t passes on is not negligible: there the port keeps B alone where the kernels and this function keep t (L - B) + B."""
    mu = (0.5 + np.arange(nangle)) / nangle  # main.cpp:482
    cw = 2 * np.pi * mu / nangle
    B = planck(wvl[:, None], weight[:, None], T[None, :])
    out = np.zeros((tau.shape[0], 2, NLEV))
    with np.errstate(over="ignore", invalid="ignore"):
        t = np.exp(-tau[:, :, None] / mu)
        L = np.zeros((tau.shape[0], nangle))
        for l in range(NLAY):
            L = t[:, l] * (L - B[:, l, None]) + B[:, l, None]
            out[:, 0, l + 1] = L @ cw
        L = np.repeat(planck(wvl, weight, Ts)[:, None], nangle, axis=1)
        out[:, 1, NLAY] = L @ cw
        for l in range(NLAY - 1, -1, -1):
            L = t[:, l] * (L - B[:, l, None]) + B[:, l, None]
            out[:, 1, l] = L @ cw
    return out


class PortColumn:
    """One column's next-step radiation in the port: tau from the table at tau_T (cloud in cloud_layer, floored at
    tau_floor if given), fluxes of Trad and Tsurf with nangle angles - from the port's radiative_transfer, or with
    stable from two_stream."""

    def __init__(self, port, tab, pl, tau_T, Trad, Tsurf, v9, nangle=30, cloud_layer=17, tau_floor=None, stable=False):
        self.port, self.tab, self.pl = port, tab, pl
        self.tau_T, self.Trad, self.Tsurf, self.v9 = tau_T, Trad, float(Tsurf), v9
        self.nangle, self.cloud_layer, self.tau_floor, self.stable = nangle, cloud_layer, tau_floor, stable

    def tau(self, tT, v, floor=True):
        return self.port.read_tau(self.tab, self.pl, tT, v, cloud_on=self.cloud_layer >= 0, cloud_layer=self.cloud_layer,
                                  tau_floor=self.tau_floor if floor else None)

    def fluxes(self, tT=None, Tr=None, Ts=None, v=None, spectral=True):
        """-> [nwvl][2][21] per wavelength (spectral) or [2][21] broadband: E_down, E_up"""
        tT = self.tau_T if tT is None else tT
        Tr = self.Trad if Tr is None else Tr
        Ts = self.Tsurf if Ts is None else Ts
        v = self.v9 if v is None else v
        tab, tau = self.tab, self.tau(tT, v)[0]
        if self.stable:
            out = two_stream(tau, tab["wvl"], tab["weight"], Tr, Ts, self.nangle)
            return out if spectral else out.sum(axis=0)
        if not spectral:
            return np.array(self.port.radiative_transfer(tau, tab["wvl"], tab["weight"], Tr, Ts, 0.0, nangle=self.nangle)[:2])
        out = np.zeros((tab["wvl"].size, 2, NLEV))
        for w in range(tab["wvl"].size):
            Ed, Eu, _ = self.port.radiative_transfer(tau[w:w + 1], tab["wvl"][w:w + 1], tab["weight"][w:w + 1], Tr, Ts, 0.0,
                                                     nangle=self.nangle)
            out[w] = Ed, Eu
        return out

    def broadband(self, solar, tT=None, Tr=None, v=None):
        """-> E_down, E_up, dE of all wavelengths, with the solar term (main.cpp:337-341); tT, Tr, v as in fluxes"""
        tT = self.tau_T if tT is None else tT
        Tr = self.Trad if Tr is None else Tr
        v = self.v9 if v is None else v
        if not self.stable:
            tab = self.tab
            return self.port.radiative_transfer(self.tau(tT, v)[0], tab["wvl"], tab["weight"], Tr, self.Tsurf, solar,
                                                nangle=self.nangle)
        Ed, Eu = self.fluxes(tT, Tr, None, v, spectral=False)
        dE = Ed[:NLAY] - Ed[1:] + Eu[1:] - Eu[:NLAY]
        dE[NLAY - 1] += solar + Ed[NLAY] - Eu[NLAY]
        return Ed, Eu, dE


def port_derivatives(pc, spectral=False):
    """Central differences of the port's fluxes -> J [2][21][41] (spectral: per wavelength, [nwvl][2][21][41]), and the
    mask of the 41 entries that have one.

    Entry x_e moves tau_T and Trad (T_l), Tsurf, or H2O by exp(+-s) (ln q_l).  The fluxes are sums of exp(-tau / mu), whose
    third derivative is r^2 times the first, r = |d tau / d x_e| / mu.  The step is H (EPS in ln q), cut down to RATE / r
    with r at the largest that matters (see step): where tau < 0 that is at the smallest mu, e^(-tau / mu) up to e^480.
    Richardson extrapolation (4 D(s/2) - D(s)) / 3 leaves an error of order RATE^4.  No difference exists - the entry is
    left out - where T_l +- H changes the layer's table interval (lowpos_t; the derivative jumps there), or where tau +- its
    change crosses tau_floor (the floored tau has a kink there)."""
    tab = pc.tab
    mu_min = 0.5 / pc.nangle
    _, _, lt0 = pc.tau(pc.tau_T, pc.v9)
    J = np.zeros(((tab["wvl"].size,) if spectral else ()) + (2, NLEV, NE))
    mask = np.ones(NE, dtype=bool)

    def F(**kw):
        return pc.fluxes(spectral=spectral, **kw)

    def difference(move, s):
        d1 = (F(**move(s)) - F(**move(-s))) / (2 * s)
        d2 = (F(**move(s / 2)) - F(**move(-s / 2))) / s
        return (4 * d2 - d1) / 3

    def step(s0, tp, tm):
        # the largest rate of change of an exponent tau / mu that matters: exp(-tau / mu) (tau / mu)^3 peaks at
        # tau / mu = 3, so a tau > 3 mu_min is weighed at mu = tau / 3 (smaller mu give terms below e^-3)
        tau = (tp + tm) / 2
        r = (np.abs(tp - tm) / (2 * s0) / np.maximum(tau / 3, mu_min)).max()
        return min(s0, RATE / r) if r > 0 else s0

    def crosses(tp, tm):
        return pc.tau_floor is not None and np.any((tp < pc.tau_floor) != (tm < pc.tau_floor))

    for l in range(NLAY):
        def move_T(s, l=l):
            tT, Tr = pc.tau_T.copy(), pc.Trad.copy()
            tT[l] += s
            Tr[l] += s
            return dict(tT=tT, Tr=Tr)

        tp, _, ltp = pc.tau(move_T(H)["tT"], pc.v9, floor=False)
        tm, _, ltm = pc.tau(move_T(-H)["tT"], pc.v9, floor=False)
        if not (np.array_equal(ltp, lt0) and np.array_equal(ltm, lt0)):
            mask[l] = False
            continue
        s = step(H, tp[:, l], tm[:, l])
        if s < H:
            tp, _, _ = pc.tau(move_T(s)["tT"], pc.v9, floor=False)
            tm, _, _ = pc.tau(move_T(-s)["tT"], pc.v9, floor=False)
        if crosses(tp[:, l], tm[:, l]):
            mask[l] = False
            continue
        J[..., l] = difference(move_T, s)
    J[..., NLAY] = difference(lambda s: dict(Ts=pc.Tsurf + s), H)
    for l in range(NLAY):
        def move_q(s, l=l):
            v = pc.v9.copy()
            v[0, l] *= np.exp(s)
            return dict(v=v)

        tp = pc.tau(pc.tau_T, move_q(EPS)["v"], floor=False)[0][:, l]
        tm = pc.tau(pc.tau_T, move_q(-EPS)["v"], floor=False)[0][:, l]
        s = step(EPS, tp, tm)
        if s < EPS:
            tp = pc.tau(pc.tau_T, move_q(s)["v"], floor=False)[0][:, l]
            tm = pc.tau(pc.tau_T, move_q(-s)["v"], floor=False)[0][:, l]
        if crosses(tp, tm):
            mask[NLAY + 1 + l] = False
            continue
        J[..., NLAY + 1 + l] = difference(move_q, s)
    return J, mask


def rows_of_K(J):
    """K [..][2][41] from J [..][2][21][41]: output 0 = E_up[0], output 1 = E_down[20]"""
    return np.stack([J[..., 1, 0, :], J[..., 0, NLEV - 1, :]], axis=-2)


def assert_close(got, ref, mask, what, rtol=1e-6):
    """|got - ref| <= rtol * max |ref| of each output (K: a row [41], J: a block [21][41]), entries with a difference"""
    sc = np.abs(ref).max(axis=-1, keepdims=True)
    if ref.shape[-3:-1] == (2, NLEV):
        sc = sc.max(axis=-2, keepdims=True)
    err = np.abs(got[..., mask] - ref[..., mask])
    assert np.all(err <= rtol * sc), (what, float(np.max(err / sc)))


def assert_structure(d, K, J, cols):
    """What holds by construction, on the columns cols: the zeros of J and K exactly 0.0, J's rows E_up[0] and E_down[20]
    equal to K to 1e-12 of the row's largest entry, dE_jac the numpy expression of J bit for bit."""
    J, Kb, Ks, Hj = J["J"][cols], K["K"][cols], K["K_spec"][cols], J["dE_jac"][cols]
    assert np.all(J[:, 0, 0] == 0.0) and np.all(J[:, 0, :, NLAY] == 0.0)
    for k in range(NLEV):
        for l in range(NLAY):
            sl = [l, NLAY + 1 + l]
            assert np.all(J[:, 0 if l >= k else 1, k, sl] == 0.0), (k, l)
    assert np.all(J[:, 1, NLEV - 1, :NLAY] == 0.0) and np.all(J[:, 1, NLEV - 1, NLAY + 1:] == 0.0)
    assert np.all(Kb[:, 1, NLAY] == 0.0) and np.all(Ks[:, :, 1, NLAY] == 0.0)
    for row, o in ((J[:, 1, 0], 0), (J[:, 0, NLEV - 1], 1)):
        sc = np.abs(Kb[:, o]).max(axis=1, keepdims=True)
        assert np.all(np.abs(row - Kb[:, o]) <= 1e-12 * sc), (o, float(np.max(np.abs(row - Kb[:, o]) / sc)))
    assert np.array_equal(Hj, heating_jacobian(J))
    acc = np.zeros_like(Kb)
    for w in range(Ks.shape[1]):
        acc = acc + Ks[:, w]
    assert np.array_equal(acc, Kb)


def run_calls(s):
    return s.diagnose_fluxes(), s.radiative_kernels(spectral=True), s.flux_jacobian()


def port_columns(port, g, st, tab, nsteps_done, cols, **cfg):
    """(c, PortColumn) of the columns cols of the state g (get_state's Tlayer and Tsurf) nsteps_done steps after st"""
    for c in cols:
        tau_T, Trad, v9 = radiated_inputs(port, st, g["Tlayer"][c], st["vmr9"][c], st["rel_hum"][c], nsteps_done == 0)
        yield c, PortColumn(port, tab, st["plevel"], tau_T, Trad, g["Tsurf"][c], v9, **cfg)


def check_column(c, pc, d, K, J, solar, spectral):
    """One column of the three calls against the port: fluxes per wavelength to 1e-10 of the wavelength's largest, broadband
    to 1e-10 of the column's largest, J (and K, K_spec) against the central differences to 1e-6 of the column's largest
    entry per output.  -> the number of entries without a difference."""
    spec, (Ed, Eu, dE) = pc.fluxes(), pc.broadband(solar)
    sc = np.abs(spec).max(axis=(1, 2))
    assert np.all(np.abs(d["E_down_spec"][c] - spec[:, 0]).max(axis=1) <= 1e-10 * sc), (c, "E_down_spec")
    assert np.all(np.abs(d["E_up_spec"][c] - spec[:, 1]).max(axis=1) <= 1e-10 * sc), (c, "E_up_spec")
    sb = np.abs(Eu).max()
    for k, got, ref in (("E_down", d["E_down"][c], Ed), ("E_up", d["E_up"][c], Eu), ("dE", d["dE"][c], dE)):
        assert np.abs(got - ref).max() <= 1e-10 * sb, (c, k)
    if spectral:
        Js, mask = port_derivatives(pc, spectral=True)
        assert_close(K["K_spec"][c], rows_of_K(Js), mask, (c, "K_spec"))
        Jref = Js.sum(axis=0)
    else:
        Jref, mask = port_derivatives(pc)
    assert_close(J["J"][c], Jref, mask, (c, "J"))
    assert_close(K["K"][c], rows_of_K(Jref), mask, (c, "K"))
    return int(NE - mask.sum())


# ---- 1. angle schedules and cloud layers -----------------------------------------------------------------------------------
# (nangle, cubes, pairs, cloud layer, steps done).  Without cube chains tau_clamp * min(1/mu) stays below 92.2 and exp
# clamps its exponent itself (clampk = 1, the <true> instances): at 30 angles tau_clamp = 11.5, at 20 angles 17.3, so the
# <false> instance's clamp of tau would leave transmissions of e^-12 and e^-18 (at 12 angles e^-30, below any tolerance
# against the port).  3 angles are one pair unit and no chain; 1, 7 and 64 angles have an odd number of chains and so a
# padding slot with zero weight; 64 is MAX_ANGLE.
SCHEDULES = [(30, 0, 1, 17, 2), (30, 0, 1, 17, 0), (20, 0, 1, -1, 2), (30, 1, 0, 17, 2), (3, 1, 1, 17, 2), (1, 1, 1, 0, 2),
             (7, 1, 1, 3, 2), (64, 1, 1, 19, 2)]


@pytest.mark.parametrize("nangle,cubes,pairs,cloud,nsteps", SCHEDULES)
def test_schedules_and_cloud_layers_against_the_port(rcm, port, nangle, cubes, pairs, cloud, nsteps):
    """21 columns (a ragged second tile), Reduced20: every wavelength's fluxes, K, J and K_spec of two columns."""
    tab = port.load_rcmtab(table_path(20))
    st = ensemble(rcm, 21, 500 + nangle)
    p = rcm.default_params()
    p.nangle, p.cloud_layer = nangle, cloud
    s = solver(rcm, 20, st, params=p)
    s.set_option(OPT_CUBES, cubes)
    s.set_option(OPT_PAIRS, pairs)
    if nsteps:
        s.advance(nsteps)
    d, K, J = run_calls(s)
    if nangle == 3:  # the step itself on this schedule, as test_other_quadratures_and_clouds_against_the_port
        ref = port.advance(tab, st["plevel"], st["rel_hum"], s.params.solar_irr, st["Tlayer"], st["Tsurf"], st["vmr9"],
                           nsteps, nangle=nangle, cloud_layer=cloud)
        got = s.get_state(("Tlayer", "E_up", "E_down"))
        sc = np.abs(ref["E_up"]).max(axis=1, keepdims=True)
        for k in ("E_up", "E_down"):
            assert np.max(np.abs(got[k] - ref[k]) / sc) < 1e-9, k
        np.testing.assert_allclose(got["Tlayer"], ref["Tlayer"], rtol=1e-10)
    g = s.get_state(("Tlayer", "Tsurf"))
    s.close()
    assert_structure(d, K, J, slice(None))
    nskip = 0
    for c, pc in port_columns(port, g, st, tab, nsteps, range(st["Tlayer"].shape[0]), nangle=nangle, cloud_layer=cloud):
        nskip += check_column(c, pc, d, K, J, p.solar_irr, spectral=c in (0, 20))
    assert nskip <= 0.1 * NLAY * st["Tlayer"].shape[0], nskip  # a layer within 1e-2 K of a table node is rare


# ---- 2. the 10- and 100-wavelength tables -------------------------------------------------------------------------------
@pytest.mark.parametrize("n", [10, 100])
def test_other_tables_against_the_port(rcm, port, n):
    """Reduced10 (10 wavelengths: the last round of 4-wavelength groups has two padding groups and a partial store) on
    every column and wavelength, K the sequential sum of K_spec; Reduced100 on five columns."""
    tab = port.load_rcmtab(table_path(n))
    st = ensemble(rcm, 21, 600 + n)
    s = solver(rcm, n, st)
    s.advance(2)
    d, K, J = run_calls(s)
    g = s.get_state(("Tlayer", "Tsurf"))
    s.close()
    assert d["E_up_spec"].shape == (21, n, NLEV) and K["K_spec"].shape == (21, n, 2, NE)
    assert_structure(d, K, J, slice(None))
    cols = range(21) if n == 10 else (0, 4, 9, 15, 20)
    nskip = 0
    for c, pc in port_columns(port, g, st, tab, 2, cols):
        nskip += check_column(c, pc, d, K, J, s.params.solar_irr, spectral=n == 10)
    assert nskip <= 0.1 * NLAY * len(cols), nskip


# ---- 3. profiles at the edges of the table ----------------------------------------------------------------------------------
def edge_ensemble(rcm, port, tab):
    """32 columns as test_other_species_masks_and_extreme_profiles (offsets of -55 .. +60 K with vertical structure, VMRs
    x 10^U(-1, 1), no ozone in some columns), the 16 wild columns of test_row_staging_fallback_and_equivalence (110 K across
    one tile) and 8 columns with one layer 122 .. 180 K below its pressure's reference temperature: below the table's
    lowest temperature node, where LowerPos takes the last interval and the cross sections are extrapolated to tau < 0."""
    atm = rcm.read_atm(os.path.join(GOLDEN, "column21.atm"))
    pl = atm[:, 1].copy()
    rng = np.random.default_rng(11)
    n = 32
    Tlev = (atm[:, 2][None, :] + rng.uniform(-55, 60, (n, 1))
            + 15 * np.sin(np.linspace(0, 3, 21))[None, :] * rng.uniform(-1, 1, (n, 1)))
    vlev = np.tile(atm[:, 4:9].T[None], (n, 1, 1)) * 10 ** rng.uniform(-1, 1, (n, 5, 1))
    vlev[::7, 1] = 0.0
    wild, wv = rcm.make_ensemble(16, 5, pl, atm[:, 2].copy(), atm[:, 4:9].T.copy())
    cold, cv = rcm.make_ensemble(8, 13, pl, atm[:, 2].copy(), atm[:, 4:9].T.copy())
    Tlev = np.concatenate([Tlev, wild + np.linspace(-55.0, 55.0, 16)[:, None], cold])
    st = rcm.init_columns(pl, Tlev, np.concatenate([vlev, wv, cv]))
    st["plevel"], st["Tsurf"] = pl, Tlev[:, 20].copy()
    _, lp, _ = port.read_tau(tab, pl, st["Tlayer"][0], st["vmr9"][0])
    t_ref = tab["t_ref"][lp[::-1]]  # of every layer's pressure (lowpos_p is bottom-up)
    for c, (l, dT) in enumerate(zip((2, 6, 10, 14, 18, 4, 8, 12), (-122, -130, -140, -150, -160, -170, -180, -125))):
        st["Tlayer"][48 + c, l] = t_ref[l] + dT
    return st


def edge_regimes(pc):
    """-> (a layer below its lowest temperature node, a tau in (-8, 0), a tau < -8, a tau above every upper clamp) of the
    port's unfloored tau; tau_clamp = 999 ln2 / max(1/mu) < 999 ln2 for every schedule.  A layer's temperature nodes are
    t_ref[ip] + t_pert with ip its lowpos_p, no interpolation in p (rcm_oracle.c:69-71); below the lowest one LowerPos takes
    the last interval."""
    tab = pc.tab
    raw, lp, lt = pc.tau(pc.tau_T, pc.v9, floor=False)
    below = (pc.tau_T < tab["t_ref"][lp[::-1]] + tab["t_pert"][0]) & (lt[::-1] == tab["t_pert"].size - 2)
    return np.array([below.any(), ((raw > TAU_FLOOR) & (raw < 0)).any(), (raw < TAU_FLOOR).any(),
                     (raw > 999 * np.log(2)).any()])


@pytest.mark.parametrize("n", [20, 100])
def test_edge_profiles_against_the_floored_port(rcm, port, n):
    """Step 0 of the edge ensemble: fluxes, K, J (and K_spec of the cold-layer columns) against the port's tau floored at
    TAU_FLOOR with two_stream's fluxes, on the columns where they are finite; the compared columns reach every regime of
    tau.  two_stream equals the port's radiative_transfer on every column without tau < 0.

    On the cold-layer columns (tau < 0) fluxes and derivatives reach 1e100 .. 1e207 at some levels and wavelengths, and the
    tolerances are relative to the largest entry of each output (per wavelength for the fluxes): there the comparison pins
    the largest, amplified entries, not values of physical size.  The columns without tau < 0, at least half of them, carry
    the comparison at physical sizes."""
    tab = port.load_rcmtab(table_path(n))
    st = edge_ensemble(rcm, port, tab)
    ncol = st["Tlayer"].shape[0]
    s = solver(rcm, n, st)
    d, K, J = run_calls(s)
    g = s.get_state(("Tlayer", "Tsurf"))
    s.close()
    compared, reached, nskip, nplain = [], np.zeros(4, dtype=bool), 0, 0
    for c, pc in port_columns(port, g, st, tab, 0, range(ncol), tau_floor=TAU_FLOOR, stable=True):
        spec = pc.fluxes()
        if not np.isfinite(spec).all():  # several layers near the floor: e^(480 k) overflows, here as in the kernels
            continue
        if pc.tau(pc.tau_T, pc.v9)[0].min() >= 0.0:
            plain = PortColumn(port, tab, st["plevel"], pc.tau_T, pc.Trad, pc.Tsurf, pc.v9, tau_floor=TAU_FLOOR)
            sc = np.abs(spec).max(axis=(1, 2), keepdims=True)
            assert np.all(np.abs(plain.fluxes() - spec) <= 1e-12 * sc), c
            nplain += 1
        nskip += check_column(c, pc, d, K, J, s.params.solar_irr, spectral=c >= 48)
        reached |= edge_regimes(pc)
        compared.append(c)
    print(f"Reduced{n}: {ncol - len(compared)} of {ncol} columns overflow, {len(compared) - nplain} compared columns with "
          f"tau < 0, {nskip} entries without a difference")
    assert len(compared) >= ncol - 4, ncol - len(compared)
    assert nplain >= ncol // 2, nplain
    assert reached.all(), reached  # below the lowest node, tau in (-8, 0), tau < -8, tau above the upper clamp
    assert_structure(d, K, J, compared)
    assert nskip <= 0.1 * NLAY * len(compared), nskip


# ---- 4. chunks ---------------------------------------------------------------------------------------------------------------
def test_chunks_of_the_diagnostic_and_kernel_calls(rcm):
    """Two chunks of the whole-ensemble call (8,192 + 108 columns) against a range across the chunk boundary in one chunk
    of its own, as test_chunks_of_the_call_do_not_change_results for flux_jacobian."""
    st = ensemble(rcm, 8300, 11)
    s = solver(rcm, 20, st)
    s.advance(1)
    whole, cross = s.diagnose_fluxes(), s.diagnose_fluxes(8185, 20)
    kwhole, kcross = s.radiative_kernels(spectral=True), s.radiative_kernels(8185, 20, spectral=True)
    s.close()
    for k in whole:
        assert np.array_equal(whole[k][8185:8205], cross[k]), k
    for k in ("K", "K_spec"):
        assert np.array_equal(kwhole[k][8185:8205], kcross[k]), k


# ---- 5. the shared constant bank --------------------------------------------------------------------------------------------
def schedule_7(rcm):
    p = rcm.default_params()
    p.nangle = 7  # cube chains, one pair unit and a padding chain
    return p


def assert_same(x, y, what):
    for k in x:
        assert np.array_equal(x[k], y[k]), (what, k)


def test_two_solvers_on_one_device(rcm):
    """Two solvers on the same table and device, at 30 and at 7 angles: every call refreshes the __constant__ bank, so
    interleaved calls give each solver's results alone, bit for bit."""
    st = ensemble(rcm, 21, 2024)
    alone = {}
    for name, p in (("30", None), ("7", schedule_7(rcm))):
        s = solver(rcm, 20, st, params=p)
        s.advance(2)
        alone[name] = run_calls(s)
        s.close()
    for x, y in zip(alone["30"], alone["7"]):
        assert all(not np.array_equal(x[k], y[k]) for k in x)
    a, b = solver(rcm, 20, st), solver(rcm, 20, st, params=schedule_7(rcm))
    a.advance(2)
    b.advance(2)
    calls = (lambda s: s.diagnose_fluxes(), lambda s: s.radiative_kernels(spectral=True), lambda s: s.flux_jacobian())
    for first, second in (((a, "30"), (b, "7")), ((b, "7"), (a, "30"))):
        for i, call in enumerate(calls):
            for s, name in (first, second):
                assert_same(call(s), alone[name][i], (name, i))
    a.close()
    b.close()


def test_set_params_on_a_live_solver(rcm, tmp_path):
    """set_params(nangle = 7) after calls at 30 angles: the next calls equal those of a fresh 7-angle solver that loaded
    the live solver's checkpoint."""
    st = ensemble(rcm, 21, 2024)
    s = solver(rcm, 20, st)
    s.advance(2)
    at30 = run_calls(s)
    ck = str(tmp_path / "live.ckpt")
    s.save_checkpoint(ck)
    s.set_params(schedule_7(rcm))
    live = run_calls(s)
    s.close()
    f = rcm.Solver(0, schedule_7(rcm))
    f.set_repwvl_table_from(rcm.Table(table_path(20)))
    f.load_checkpoint(ck)
    fresh = run_calls(f)
    f.close()
    for i in range(3):
        assert_same(live[i], fresh[i], i)
        assert not np.array_equal(live[i][next(iter(live[i]))], at30[i][next(iter(at30[i]))])
