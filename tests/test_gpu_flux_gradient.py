"""Adjoint flux gradients of the resident ensemble (rcm_flux_gradient / Solver.flux_gradient): the derivatives of one weighted
sum of each column's broadband fluxes and heating rates of the next step in T_l, T_surf and every species' ln VMR per layer,
by one reverse sweep, without changing anything.

Checkers: the contraction of rcm_flux_jacobian and rcm_species_jacobian with the same cotangents; the radiative kernels for a
unit cotangent on the OLR or the surface downward flux; central differences of the C port's fluxes; Richardson-extrapolated
differences of the objective from diagnose_fluxes with one species scaled.
"""
import ctypes as C

import numpy as np
import pytest

from conftest import table_path
from test_gpu_diagnostics import CO2_2X, ensemble, solver, status_of
from test_gpu_flux_jacobian import heating_jacobian, port_jacobian
from test_gpu_radiative_kernels import radiated_inputs
from test_gpu_species_jacobian import V9_ROW, port_species_jacobian

pytestmark = pytest.mark.gpu
NLAY, NLEV, NS = 20, 21, 5
NE = NLEV + NS * NLAY   # 121
O3_HALF = [1.0, 1.0, 0.5, 1.0, 1.0]
SUBSETS = ("all", "E_down", "E_up", "dE")


@pytest.fixture(scope="module")
def ens21(rcm):
    return ensemble(rcm, 21, 2024)


def cotangents(n, seed, which="all"):
    rng = np.random.default_rng(seed)
    w = dict(w_E_down=rng.normal(size=(n, NLEV)), w_E_up=rng.normal(size=(n, NLEV)), w_dE=rng.normal(size=(n, NLAY)))
    if which != "all":
        w = {k: (v if k == "w_" + which else None) for k, v in w.items()}
    return w


def full_jacobian(s, vmr_scale=None, lbl=False):
    """J [n][2][21][121], H [n][20][121]: the flux Jacobian's 41 entries, then the species Jacobian's CO2..CH4 blocks"""
    f = (s.lbl_flux_jacobian if lbl else s.flux_jacobian)(vmr_scale=vmr_scale)
    sp = (s.lbl_species_jacobian if lbl else s.species_jacobian)(vmr_scale=vmr_scale)
    return (np.concatenate([f["J"], sp["J"][..., NLAY:]], axis=-1),
            np.concatenate([f["dE_jac"], sp["dE_jac"][..., NLAY:]], axis=-1))


def contract(w, J, H):
    """-> the reference gradient [n][121] and each column's largest sum |w| |J| over the entries"""
    ref = np.zeros((J.shape[0], NE))
    mag = np.zeros((J.shape[0], NE))
    for key, M in (("w_E_down", J[:, 0]), ("w_E_up", J[:, 1]), ("w_dE", H)):
        if w[key] is not None:
            ref += np.einsum("nk,nke->ne", w[key], M)
            mag += np.einsum("nk,nke->ne", np.abs(w[key]), np.abs(M))
    return ref, mag.max(axis=1)


def assert_contraction(got, w, J, H, bar=1e-11, what=None):
    ref, scale = contract(w, J, H)
    err = np.abs(got - ref).max(axis=1)
    assert np.all(err <= bar * scale), (what, np.max(err / scale))


def check_contraction(s, vmr_scale=None, seed=1, lbl=False):
    J, H = full_jacobian(s, vmr_scale, lbl)
    fn = s.lbl_flux_gradient if lbl else s.flux_gradient
    for i, which in enumerate(SUBSETS):
        w = cotangents(s.ncol, seed + i, which)
        d = fn(vmr_scale=vmr_scale, **w)
        assert d["grad"].shape == (s.ncol, NE)
        assert_contraction(d["grad"], w, J, H, what=(vmr_scale, which))
        assert np.array_equal(d["dT"], d["grad"][:, :NLAY]) and np.array_equal(d["dTs"], d["grad"][:, NLAY])
        assert np.array_equal(d["dlnx"], d["grad"][:, NLEV:].reshape(s.ncol, NS, NLAY))


# ---- 1. the contraction of the Jacobians ---------------------------------------------------------------------------------
@pytest.mark.parametrize("nsteps", [0, 3])
@pytest.mark.parametrize("vmr_scale", [None, CO2_2X, O3_HALF])
def test_contraction_of_the_jacobians(rcm, ens21, nsteps, vmr_scale):
    s = solver(rcm, 20, ens21)
    if nsteps:
        s.advance(nsteps)
    check_contraction(s, vmr_scale)
    s.close()


def test_contraction_reduced100_and_column_cloud(rcm, ens21):
    s = solver(rcm, 100, ens21)
    s.advance(2)
    check_contraction(s, O3_HALF, seed=7)
    rng = np.random.default_rng(5)
    s.set_column_solar(None, rng.uniform(0.5, 4.0, s.ncol), rng.uniform(0.3, 0.8, s.ncol), None, cloud_from_tau_s=True)
    check_contraction(s, CO2_2X, seed=11)
    s.close()


# ---- 2. unit cotangents are the radiative kernels -------------------------------------------------------------------------
def test_unit_cotangents_give_the_radiative_kernels(rcm, ens21):
    s = solver(rcm, 100, ens21)
    s.advance(2)
    K = s.radiative_kernels()["K"]
    n = s.ncol
    for o, key, k in ((0, "w_E_up", 0), (1, "w_E_down", NLAY)):
        w = np.zeros((n, NLEV))
        w[:, k] = 1.0
        g = s.flux_gradient(**{key: w})["grad"]
        scale = np.abs(K[:, o]).max(axis=1)
        assert np.all(np.abs(g[:, :2 * NLAY + 1] - K[:, o]).max(axis=1) <= 1e-12 * scale), o
    s.close()


# ---- 3. central differences of the port ------------------------------------------------------------------------------------
def test_every_entry_against_central_differences_of_the_port(rcm, port, ens21):
    """21 columns (a ragged second tile), Reduced20, after two steps: the port's J in T, T_surf, ln q and the species, with
    the cotangents; T entries of a layer near a table node (skipped by port_jacobian) are left out."""
    tab = port.load_rcmtab(table_path(20))
    s = solver(rcm, 20, ens21)
    s.advance(2)
    w = cotangents(s.ncol, 3)
    got = s.flux_gradient(**w)["grad"]
    g = s.get_state(("Tlayer", "Tsurf"))
    st = ens21
    for c in range(s.ncol):
        tau_T, Trad, v9 = radiated_inputs(port, st, g["Tlayer"][c], st["vmr9"][c], st["rel_hum"][c], False)
        J41, skipped = port_jacobian(port, tab, st["plevel"], tau_T, Trad, g["Tsurf"][c], v9)
        Jsp = port_species_jacobian(port, tab, st["plevel"], tau_T, Trad, g["Tsurf"][c], v9)
        J = np.concatenate([J41, Jsp[..., NLAY:]], axis=-1)[None]
        H = heating_jacobian(J)
        ref, _ = contract({k: v[c:c + 1] for k, v in w.items()}, J, H)
        mask = np.ones(NE, dtype=bool)
        mask[skipped] = False
        scale = np.abs(ref[0]).max()
        assert np.abs(got[c, mask] - ref[0, mask]).max() <= 1e-6 * scale, c


# ---- 4. directional derivatives against the flux call ------------------------------------------------------------------------
def test_species_directions_against_the_flux_call(rcm, ens21):
    """sum_l dPhi/dln x_{s,l} = dPhi/dln f_s: Richardson-extrapolated central differences of diagnose_fluxes, h = 1e-3"""
    s = solver(rcm, 100, ens21)
    s.advance(3)
    w = cotangents(s.ncol, 21)
    d = s.flux_gradient(**w)
    J, H = full_jacobian(s)
    _, scale = contract(w, J, H)

    def phi(f):
        r = s.diagnose_fluxes(vmr_scale=f, spectral=False)
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


# ---- 5. exact zeros ----------------------------------------------------------------------------------------------------------
def test_exact_zeros(rcm, ens21):
    s = solver(rcm, 20, ens21)
    s.advance(1)
    n = s.ncol
    L = rcm.load_library()
    launches = L.rcm_launch_count(s._h)
    z = s.flux_gradient(w_E_down=np.zeros((n, NLEV)))["grad"]   # non-NULL zeros still run (and give 0)
    assert np.all(z == 0.0)
    before = L.rcm_launch_count(s._h)
    g = np.full((n, NE), 7.0)
    assert L.rcm_flux_gradient(s._h, C.c_int(0), C.c_int(n), None, None, None, None, g.ctypes.data_as(C.c_void_p)) == 0
    assert np.all(g == 0.0) and L.rcm_launch_count(s._h) == before and before > launches
    assert L.rcm_flux_gradient(s._h, C.c_int(0), C.c_int(n), None, None, None, None, None) == 0
    for k in range(NLEV):   # a cotangent on E_down[k] alone: E_down[k] depends on no layer l >= k and not on T_surf
        w = np.zeros((n, NLEV))
        w[:, k] = np.linspace(0.5, 2.0, n)
        g = s.flux_gradient(w_E_down=w)["grad"]
        layers = np.arange(NLAY) >= k
        cols = np.concatenate([layers, [True], np.tile(layers, NS)])
        assert np.all(g[:, cols] == 0.0), k
        if k > 0:
            assert np.any(g[:, ~cols] != 0.0), k
    # zero VMRs and clamped tau
    v = np.array(ens21["vmr9"][:, list(V9_ROW)], dtype=np.float64)
    zero = [(1, 3), (1, 12), (4, 7), (3, 19), (2, 0)]
    for k, l in zero:
        v[:, k, l] = 0.0
    s.update_columns(vmr_active=v)
    w = cotangents(n, 4)
    g = s.flux_gradient(**w)
    for k, l in zero:
        assert np.all(g["dlnx"][:, k, l] == 0.0), (k, l)
    assert np.any(g["dlnx"][:, 4, 8] != 0.0)
    c = s.flux_gradient(vmr_scale=[1e12] * NS, **w)
    assert np.all(c["dlnx"] == 0.0)
    s.close()


# ---- 6. linearity ------------------------------------------------------------------------------------------------------------
def test_linearity(rcm, ens21):
    s = solver(rcm, 100, ens21)
    s.advance(2)
    w1, w2, a = cotangents(s.ncol, 31), cotangents(s.ncol, 32), -2.5
    g1, g2 = s.flux_gradient(**w1)["grad"], s.flux_gradient(**w2)["grad"]
    g = s.flux_gradient(**{k: a * w1[k] + w2[k] for k in w1})["grad"]
    J, H = full_jacobian(s)
    _, s1 = contract(w1, J, H)
    _, s2 = contract(w2, J, H)
    assert np.all(np.abs(g - (a * g1 + g2)).max(axis=1) <= 1e-12 * (abs(a) * s1 + s2))
    s.close()


# ---- 7. invariance ----------------------------------------------------------------------------------------------------------
def test_ranges_columns_and_chunks_give_the_same_rows(rcm):
    """8,200 columns: two chunks (8,192 + 8) for the whole range; ranges inside one chunk and across the boundary; a shard"""
    st = ensemble(rcm, 8200, 11)
    s = solver(rcm, 20, st)
    s.advance(1)
    w = cotangents(8200, 5)
    whole = s.flux_gradient(vmr_scale=O3_HALF, **w)["grad"]
    for col0, m in ((0, 24), (8185, 15), (8199, 1), (11, 1), (1000, 7200)):
        sub = s.flux_gradient(col0=col0, ncol=m, vmr_scale=O3_HALF, **{k: v[col0:col0 + m] for k, v in w.items()})["grad"]
        assert np.array_equal(sub, whole[col0:col0 + m]), col0
    s.close()
    part = solver(rcm, 20, st, slice(4000, 4100))
    part.advance(1)
    tail = part.flux_gradient(vmr_scale=O3_HALF, **{k: v[4000:4100] for k, v in w.items()})["grad"]
    part.close()
    assert np.array_equal(whole[4000:4100], tail)


# ---- 8. no side effects --------------------------------------------------------------------------------------------------------
def test_the_call_changes_nothing(rcm, ens21, tmp_path):
    a, b = solver(rcm, 20, ens21), solver(rcm, 20, ens21)
    w = cotangents(21, 6)
    b.flux_gradient(**w)
    sa = [a.advance(2), a.advance(3)]
    sb = [b.advance(2)]
    b.flux_gradient(vmr_scale=CO2_2X, **w)
    b.flux_gradient(col0=3, ncol=5, w_dE=w["w_dE"][3:8])
    sb.append(b.advance(3))
    b.flux_gradient(**w)
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


# ---- 9. errors ---------------------------------------------------------------------------------------------------------------
def test_errors_leave_the_solver_usable(rcm, ens21):
    OPT_PATH = 5
    L = rcm.load_library()
    s = solver(rcm, 20, ens21)
    w = cotangents(21, 8)
    for col0, ncol in ((-1, 3), (0, 0), (20, 2), (0, 22)):
        assert status_of(rcm, lambda: s.flux_gradient(col0=col0, ncol=ncol)) == 1, (col0, ncol)
    for key in ("w_E_down", "w_E_up", "w_dE"):
        for bad in (np.nan, np.inf, -np.inf):
            v = w[key].copy()
            v[5, 3] = bad
            assert status_of(rcm, lambda: s.flux_gradient(**{**w, key: v})) == 1, (key, bad)
    with pytest.raises(ValueError):
        s.flux_gradient(w_E_down=np.zeros((21, NLAY)))
    with pytest.raises(ValueError):
        s.flux_gradient(w_dE=np.zeros((20, NLAY)))
    s.set_option(OPT_PATH, 1)
    assert status_of(rcm, lambda: s.flux_gradient(**w)) == 2
    s.set_option(OPT_PATH, 0)
    J, H = full_jacobian(s)
    assert_contraction(s.flux_gradient(**w)["grad"], w, J, H)
    s.close()

    for mask in (0x0F, 0x3E, 0x1F):
        p = rcm.default_params()
        p.species_mask = mask
        m = solver(rcm, 20, ens21, params=p)
        assert status_of(rcm, lambda: m.flux_gradient(**w)) == 2, mask
        m.advance(1)
        m.close()

    st = ens21
    lb = rcm.Solver(0)
    wvl, tau5 = rcm.make_lbl_tables(300, 7, st["plevel"], st["vmr9"][0, 0], st["vmr9"][0, 2])
    lb.set_lbl_tables(wvl, tau5, st["vmr9"][0, 0], st["vmr9"][0, 2])
    lb.set_columns(st["plevel"], st["Tlayer"], st["Tsurf"], st["vmr9"], st["rel_hum"])
    assert status_of(rcm, lambda: lb.flux_gradient(**w)) == 2
    assert np.isfinite(lb.lbl_flux_gradient(**w)["grad"]).all()
    lb.close()
