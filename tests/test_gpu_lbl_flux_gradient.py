"""Adjoint flux gradients of the line-by-line path (rcm_lbl_flux_gradient / Solver.lbl_flux_gradient): the derivatives of one
weighted sum of each column's broadband fluxes and heating rates of the next LBL step in T_l, T_surf and every species' ln VMR
per layer, by one reverse sweep, without moving the state.

Checkers: the contraction of lbl_flux_jacobian and lbl_species_jacobian with the same cotangents (Simpson and series branches
of the Planck source, other angle schedules, both tau-clamp placements); the LBL radiative kernels for unit cotangents;
central differences of the C port's fluxes; Richardson-extrapolated differences of lbl_diagnose_fluxes with one species scaled.
"""
import ctypes as C

import numpy as np
import pytest

from conftest import table_path
from test_gpu_diagnostics import status_of
from test_gpu_flux_gradient import NE, assert_contraction, check_contraction, contract, cotangents, full_jacobian
from test_gpu_flux_jacobian import heating_jacobian
from test_gpu_lbl_diagnostics import _p, case, make  # noqa: F401 (case is a fixture)
from test_gpu_lbl_flux_jacobian import JPort
from test_gpu_lbl_radiative_kernels import case200, solver  # noqa: F401 (case200 is a fixture)
from test_gpu_lbl_species_jacobian import SPort

pytestmark = pytest.mark.gpu

NLAY, NLEV, NS = 20, 21, 5
SCALED = [1.5, 2.0, 0.5, 2.0, 1.3]   # every species scaled (ascending species index)


# ---- 1. the contraction of the Jacobians ---------------------------------------------------------------------------------
@pytest.mark.parametrize("nwvl", [1500, 200])
@pytest.mark.parametrize("steps", [0, 3])
@pytest.mark.parametrize("scaled", [False, True])
def test_contraction_of_the_jacobians(rcm, case, case200, nwvl, steps, scaled):
    """1,500 wavelengths: the Simpson branch of the Planck source; 200: the series"""
    s = solver(rcm, case if nwvl == 1500 else case200)
    if steps:
        s.advance(steps)
    check_contraction(s, SCALED if scaled else None, seed=steps + 10 * nwvl, lbl=True)
    s.close()


def test_contraction_with_column_cloud_and_solar(rcm, case):
    s = solver(rcm, case)
    n = case["ncol"]
    s.set_column_solar(tau_s=np.linspace(0.5, 4.0, n), mu_s=np.linspace(0.3, 0.9, n), cloud_from_tau_s=True)
    s.advance(2)
    check_contraction(s, [1.0, 2.0, 0.5, 1.0, 1.0], seed=3, lbl=True)
    s.close()


@pytest.mark.parametrize("nangle,cubes,pairs", [(20, 1, 1), (7, 1, 1), (30, 0, 0)])
def test_contraction_on_other_angle_schedules(rcm, case, nangle, cubes, pairs):
    """(20, 1, 1) and (7, 1, 1): other schedules; (30, 0, 0): without cube chains the exp clamps tau instead of the layer
    (the kernel's other CLAMPK instance, test_gpu_lbl_radiative_kernels)"""
    p = rcm.default_params()
    p.nangle = nangle
    s = solver(rcm, case, p, cubes, pairs)
    s.advance(2)
    check_contraction(s, SCALED, seed=nangle, lbl=True)
    s.close()


# ---- 2. unit cotangents are the radiative kernels -------------------------------------------------------------------------
@pytest.mark.parametrize("steps", [0, 3])
def test_unit_cotangents_give_the_radiative_kernels(rcm, case, steps):
    s = make(rcm, case)
    if steps:
        s.advance(steps)
    K = s.lbl_radiative_kernels(vmr_scale=SCALED)["K"]
    n = s.ncol
    for o, key, k in ((0, "w_E_up", 0), (1, "w_E_down", NLAY)):
        w = np.zeros((n, NLEV))
        w[:, k] = 1.0
        g = s.lbl_flux_gradient(vmr_scale=SCALED, **{key: w})["grad"]
        scale = np.abs(K[:, o]).max(axis=1)
        assert np.all(np.abs(g[:, :2 * NLAY + 1] - K[:, o]).max(axis=1) <= 1e-12 * scale), (steps, o)
    s.close()


# ---- 3. central differences of the port ------------------------------------------------------------------------------------
def test_every_entry_against_central_differences_of_the_port(rcm, port, case):
    """the port's J in T, T_surf and ln q (JPort) and in the species (SPort), contracted with the cotangents, on columns
    whose Planck source has no jump within the T step"""
    s = solver(rcm, case)
    s.advance(2)
    g = s.get_state()
    w = cotangents(s.ncol, 9)
    got = s.lbl_flux_gradient(vmr_scale=SCALED, **w)["grad"]
    jp, sp = JPort(port, case, g, 2, SCALED), SPort(port, case, g, 2, SCALED)
    done = 0
    for col in range(s.ncol):
        if done == 3:
            break
        if not jp.smooth(col):
            continue
        J = np.concatenate([jp.J(col), sp.J(col)[..., NLAY:]], axis=-1)[None]
        ref, _ = contract({k: v[col:col + 1] for k, v in w.items()}, J, heating_jacobian(J))
        assert np.abs(got[col] - ref[0]).max() <= 1e-6 * np.abs(ref[0]).max(), col
        done += 1
    assert done == 3
    s.close()


# ---- 4. directional derivatives against the flux call ------------------------------------------------------------------------
def test_species_directions_against_the_flux_call(rcm, case):
    """sum_l dPhi/dln x_{s,l} = dPhi/dln f_s: Richardson-extrapolated central differences of lbl_diagnose_fluxes"""
    s = make(rcm, case)
    s.advance(3)
    w = cotangents(s.ncol, 12)
    d = s.lbl_flux_gradient(**w)
    J, H = full_jacobian(s, lbl=True)
    _, scale = contract(w, J, H)

    def phi(f):
        r = s.lbl_diagnose_fluxes(vmr_scale=f)
        return (np.sum(w["w_E_down"] * r["E_down"], axis=1) + np.sum(w["w_E_up"] * r["E_up"], axis=1)
                + np.sum(w["w_dE"] * r["dE"], axis=1))

    def D(k, h):
        f = np.ones(NS)
        f[k] = np.exp(h)
        up = phi(f)
        f[k] = np.exp(-h)
        return (up - phi(f)) / (2 * h)

    h = 1e-3
    for k in range(NS):
        fd = (4 * D(k, h / 2) - D(k, h)) / 3
        an = d["dlnx"][:, k].sum(axis=1)
        assert np.all(np.abs(an - fd) <= 1e-6 * NLAY * scale), (k, np.max(np.abs(an - fd) / scale))
    s.close()


# ---- 5. exact zeros, linearity ----------------------------------------------------------------------------------------------
def test_exact_zeros_and_linearity(rcm, case):
    s = make(rcm, case)
    s.advance(1)
    n = s.ncol
    L = rcm.load_library()
    before = L.rcm_launch_count(s._h)
    g = np.full((n, NE), 7.0)
    assert L.rcm_lbl_flux_gradient(s._h, C.c_int(0), C.c_int(n), None, None, None, None, _p(g)) == 0
    assert np.all(g == 0.0) and L.rcm_launch_count(s._h) == before
    for k in (0, 1, 7, 19, 20):
        w = np.zeros((n, NLEV))
        w[:, k] = 1.0
        got = s.lbl_flux_gradient(w_E_down=w)["grad"]
        layers = np.arange(NLAY) >= k
        cols = np.concatenate([layers, [True], np.tile(layers, NS)])
        assert np.all(got[:, cols] == 0.0), k
    w = cotangents(n, 13)   # a zero factor zeroes that species' entries
    z = s.lbl_flux_gradient(vmr_scale=[1.0, 0.0, 1.0, 0.0, 1.0], **w)   # no CO2, no N2O
    assert np.all(z["dlnx"][:, 1] == 0.0) and np.all(z["dlnx"][:, 3] == 0.0) and np.any(z["dlnx"][:, 4] != 0.0)
    w1, w2, a = cotangents(n, 14), cotangents(n, 15), 3.25
    g1, g2 = s.lbl_flux_gradient(**w1)["grad"], s.lbl_flux_gradient(**w2)["grad"]
    g12 = s.lbl_flux_gradient(**{k: a * w1[k] + w2[k] for k in w1})["grad"]
    J, H = full_jacobian(s, lbl=True)
    _, s1 = contract(w1, J, H)
    _, s2 = contract(w2, J, H)
    assert np.all(np.abs(g12 - (a * g1 + g2)).max(axis=1) <= 1e-12 * (a * s1 + s2))
    s.close()


# ---- 6. invariance and no side effects --------------------------------------------------------------------------------------
def test_ranges_columns_and_chunks_give_the_same_rows(rcm, case200):
    """8,208 columns of 200 wavelengths: two chunks (8,192 + 16); ranges inside one chunk and across the boundary"""
    n = 8208
    s = make(rcm, case200, rep=(n + case200["ncol"] - 1) // case200["ncol"], n=n)
    s.advance(1)
    w = cotangents(n, 16)
    whole = s.lbl_flux_gradient(vmr_scale=SCALED, **w)["grad"]
    for col0, m in ((0, 24), (8185, 15), (8207, 1), (11, 1), (1000, 7200)):
        sub = s.lbl_flux_gradient(col0=col0, ncol=m, vmr_scale=SCALED, **{k: v[col0:col0 + m] for k, v in w.items()})
        assert np.array_equal(sub["grad"], whole[col0:col0 + m]), col0
    s.close()


def test_calls_move_nothing(rcm, case, tmp_path):
    a, b = make(rcm, case), make(rcm, case)
    w = cotangents(case["ncol"], 17)
    b.lbl_flux_gradient(**w)
    sa = [a.advance(2), a.advance(2)]
    sb = [b.advance(2)]
    b.lbl_flux_gradient(vmr_scale=SCALED, **w)
    sb.append(b.advance(2))
    for x, y in zip(sa, sb):
        assert np.array_equal(x, y)
    ga, gb = a.get_state(), b.get_state()
    for k in ga:
        assert np.array_equal(ga[k], gb[k]), k
    a.save_checkpoint(str(tmp_path / "a.ckpt"))
    b.save_checkpoint(str(tmp_path / "b.ckpt"))
    assert open(tmp_path / "a.ckpt", "rb").read() == open(tmp_path / "b.ckpt", "rb").read()
    a.close()
    b.close()


# ---- 7. errors ---------------------------------------------------------------------------------------------------------------
def test_errors_leave_the_solver_usable(rcm, case):
    s = make(rcm, case)
    w = cotangents(case["ncol"], 18)
    for col0, ncol in ((-1, 3), (0, 0), (20, 5), (0, 25)):
        assert status_of(rcm, lambda: s.lbl_flux_gradient(col0=col0, ncol=ncol)) == 1, (col0, ncol)
    for key in ("w_E_down", "w_E_up", "w_dE"):
        for bad in (np.nan, np.inf):
            v = w[key].copy()
            v[2, 4] = bad
            assert status_of(rcm, lambda: s.lbl_flux_gradient(**{**w, key: v})) == 1, (key, bad)
    for bad in ([-1, 1, 1, 1, 1], [1, np.nan, 1, 1, 1]):
        assert status_of(rcm, lambda: s.lbl_flux_gradient(vmr_scale=bad, **w)) == 1
    assert status_of(rcm, lambda: s.flux_gradient(**w)) == 2   # the repwvl call refuses LBL
    J, H = full_jacobian(s, lbl=True)
    assert_contraction(s.lbl_flux_gradient(**w)["grad"], w, J, H)
    s.close()
    st = case["st"]
    r = rcm.Solver(0)
    r.set_repwvl_table_from(rcm.Table(table_path(10)))
    r.set_columns(case["pl"], st["Tlayer"], case["Tsurf"], st["vmr9"], st["rel_hum"])
    assert status_of(rcm, lambda: r.lbl_flux_gradient(**w)) == 2
    r.advance(1)
    r.close()
    p = rcm.default_params()
    p.species_mask = 0x3F
    m = rcm.Solver(0, p)
    m.set_lbl_tables(case["wvl"], case["tau5"], case["h2o_ref"], case["o3_ref"], 1.0)
    m.set_columns(case["pl"], st["Tlayer"], case["Tsurf"], st["vmr9"], st["rel_hum"])
    assert status_of(rcm, lambda: m.lbl_flux_gradient(**w)) == 2
    m.advance(1)
    m.close()
