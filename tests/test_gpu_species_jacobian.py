"""Species Jacobians of the resident ensemble (rcm_species_jacobian / Solver.species_jacobian): analytic derivatives of every
level's broadband E_down and E_up of the next step, and of its heating rates, with respect to the ln VMR of each of the five
species (H2O, CO2, O3, N2O, CH4) in each layer, without changing anything.

Checker: central differences of the C port of the reference (oracle/rcm_oracle.c) for all 42 fluxes, one species in one layer
multiplied by exp(+-eps), around the inputs the next step radiates with (test_gpu_radiative_kernels.radiated_inputs); the
H2O block against rcm_flux_jacobian bit for bit; the layer sums against diagnose_fluxes with the species' factor.
"""
import os

import numpy as np
import pytest

from conftest import GOLDEN, table_path
from test_gpu_diagnostics import CO2_2X, ensemble, solver, status_of
from test_gpu_flux_jacobian import heating_jacobian
from test_gpu_radiative_kernels import EPS, driver, radiated_inputs

pytestmark = pytest.mark.gpu
NLAY, NLEV, NS = 20, 21, 5
NE = NS * NLAY
V9_ROW = (0, 1, 2, 3, 5)   # rows of vmr9 of H2O, CO2, O3, N2O, CH4 (the default species_mask 0x2F)
O3_HALF = [1.0, 1.0, 0.5, 1.0, 1.0]


@pytest.fixture(scope="module")
def ens21(rcm):
    return ensemble(rcm, 21, 2024)


@pytest.fixture(scope="module")
def ens5000(rcm):
    return ensemble(rcm, 5000, 77)


# ---- the port's central differences ------------------------------------------------------------------------------------
def port_species_jacobian(port, tab, pl, tau_T, Trad, Tsurf, v9, tau_s=2.0):
    """-> J [2][21][100] by central differences: entry 20 s + l multiplies species s's VMR in layer l by exp(+-EPS)"""
    def F(v):
        tau, _, _ = port.read_tau(tab, pl, tau_T, v, tau_s=tau_s)
        Ed, Eu, _ = port.radiative_transfer(tau, tab["wvl"], tab["weight"], Trad, Tsurf, 0.0)
        return np.array([Ed, Eu])

    J = np.zeros((2, NLEV, NE))
    for s, row in enumerate(V9_ROW):
        for l in range(NLAY):
            vp, vm = v9.copy(), v9.copy()
            vp[row, l] *= np.exp(EPS)
            vm[row, l] *= np.exp(-EPS)
            J[..., s * NLAY + l] = (F(vp) - F(vm)) / (2 * EPS)
    return J


def check_against_port(port, s, st, tab, nsteps_done, vmr_scale=None, tau_s=None, cols=None):
    f = [1.0] * NS if vmr_scale is None else list(vmr_scale)
    d = s.species_jacobian(vmr_scale=vmr_scale)
    g = s.get_state(("Tlayer", "Tsurf"))
    for c in range(s.ncol) if cols is None else cols:
        tau_T, Trad, v9 = radiated_inputs(port, st, g["Tlayer"][c], st["vmr9"][c], st["rel_hum"][c], nsteps_done == 0, f[0], f[1])
        for k in (2, 3, 4):
            v9[V9_ROW[k]] = v9[V9_ROW[k]] * f[k]
        ts = 2.0 if tau_s is None else tau_s[c]
        ref = port_species_jacobian(port, tab, st["plevel"], tau_T, Trad, g["Tsurf"][c], v9, tau_s=ts)
        for o in range(2):  # <= 1e-6 of the column's max |entry| of the E_down resp. E_up block (test_gpu_flux_jacobian's bar)
            sc = np.abs(ref[o]).max()
            err = np.abs(d["J"][c, o] - ref[o]).max()
            assert err <= 1e-6 * sc, (c, o, err, sc)
    return d


# ---- 1. against the port's central differences ---------------------------------------------------------------------------
@pytest.mark.parametrize("nsteps", [3, 0])
def test_every_entry_against_central_differences_of_the_port(rcm, port, ens21, nsteps):
    """21 columns (a ragged second tile), Reduced20, after three steps and at step 0 (tau from the unsorted profile)."""
    tab = port.load_rcmtab(table_path(20))
    s = solver(rcm, 20, ens21)
    if nsteps:
        s.advance(nsteps)
    d = check_against_port(port, s, ens21, tab, nsteps)
    assert d["J"].shape == (21, 2, NLEV, NE) and d["dE_jac"].shape == (21, NLAY, NE)
    s.close()


def test_scales_other_table_and_column_cloud(rcm, port, ens21):
    """CO2 x2 and O3 x0.5 on Reduced20, O3 x0.5 on Reduced100, per-column cloud and solar"""
    tab = port.load_rcmtab(table_path(20))
    s = solver(rcm, 20, ens21)
    s.advance(1)
    check_against_port(port, s, ens21, tab, 1, vmr_scale=CO2_2X)
    check_against_port(port, s, ens21, tab, 1, vmr_scale=O3_HALF, cols=range(0, 21, 4))
    rng = np.random.default_rng(5)
    tau_s, mu_s = rng.uniform(0.5, 4.0, s.ncol), rng.uniform(0.3, 0.8, s.ncol)
    s.set_column_solar(None, tau_s, mu_s, None, cloud_from_tau_s=True)
    check_against_port(port, s, ens21, tab, 1, tau_s=tau_s, cols=range(1, 21, 3))
    s.close()
    tab = port.load_rcmtab(table_path(100))
    s = solver(rcm, 100, ens21)
    s.advance(2)
    check_against_port(port, s, ens21, tab, 2, vmr_scale=O3_HALF, cols=(0, 7, 20))
    s.close()


# ---- 2. the H2O block is the flux Jacobian's ln q block --------------------------------------------------------------------
@pytest.mark.parametrize("vmr_scale", [None, CO2_2X, [1.3, 1.0, 0.5, 2.0, 1.5]])
def test_h2o_block_equals_the_flux_jacobian(rcm, ens21, vmr_scale):
    s = solver(rcm, 100, ens21)
    s.advance(2)
    d = s.species_jacobian(vmr_scale=vmr_scale)
    f = s.flux_jacobian(vmr_scale=vmr_scale)
    s.close()
    assert np.array_equal(d["J"][..., :NLAY], f["J"][..., NLAY + 1:])
    assert np.array_equal(d["dE_jac"][..., :NLAY], f["dE_jac"][..., NLAY + 1:])
    assert np.array_equal(d["J_h2o"], f["J"][..., NLAY + 1:])


# ---- 3. layer sums against the flux call -------------------------------------------------------------------------------------
def test_layer_sums_against_the_flux_call(rcm, ens21):
    """sum_l d/dln x_{s,l} = d/dln f_s: Richardson-extrapolated central differences of diagnose_fluxes, h = 1e-3"""
    s = solver(rcm, 100, ens21)
    s.advance(3)
    d = s.species_jacobian()

    def D(k, h):
        f = np.ones(NS)
        f[k] = np.exp(h)
        up = s.diagnose_fluxes(vmr_scale=f, spectral=False)
        f[k] = np.exp(-h)
        dn = s.diagnose_fluxes(vmr_scale=f, spectral=False)
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


# ---- 4. structure ----------------------------------------------------------------------------------------------------------
def structural_zeros(J):
    for k in range(NLEV):
        for l in range(NLAY):
            cols = [s * NLAY + l for s in range(NS)]
            if l >= k:
                assert np.all(J[:, 0, k][:, cols] == 0.0), (k, l)
            else:
                assert np.all(J[:, 1, k][:, cols] == 0.0), (k, l)


@pytest.mark.parametrize("vmr_scale", [None, CO2_2X])
def test_structure_and_heating_rates(rcm, ens21, vmr_scale):
    s = solver(rcm, 100, ens21)
    s.advance(2)
    d = s.species_jacobian(vmr_scale=vmr_scale)
    s.close()
    J = d["J"]
    structural_zeros(J)
    assert np.array_equal(d["dE_jac"], heating_jacobian(J))
    for name_k, name in enumerate(("h2o", "co2", "o3", "n2o", "ch4")):
        assert np.array_equal(d[f"J_{name}"], J[..., name_k * NLAY:(name_k + 1) * NLAY])
    # more CO2 in the column lowers the OLR: its layer sum is negative in every column
    assert np.all(J[:, 1, 0, NLAY:2 * NLAY].sum(axis=-1) < 0.0)


def test_zero_vmr_and_clamped_layers_give_zero(rcm, ens21):
    s = solver(rcm, 20, ens21)
    s.advance(1)
    v = np.array(ens21["vmr9"][:, list(V9_ROW)], dtype=np.float64)   # [ncol][5][20] the active species
    zero = [(1, 3), (1, 12), (4, 7), (3, 19), (2, 0)]                  # (species, layer)
    for k, l in zero:
        v[:, k, l] = 0.0
    s.update_columns(vmr_active=v)
    d = s.species_jacobian()
    for k, l in zero:
        e = k * NLAY + l
        assert np.all(d["J"][..., e] == 0.0) and np.all(d["dE_jac"][..., e] == 0.0), (k, l)
    assert np.any(d["J"][:, 1, 0, NLAY + 4] != 0.0)
    # every species x1e12: tau is clamped (or floored) at every wavelength of every layer
    c = s.species_jacobian(vmr_scale=[1e12] * NS)
    assert np.all(c["J"] == 0.0) and np.all(c["dE_jac"] == 0.0)
    s.close()


# ---- 5. invariance and no side effects -------------------------------------------------------------------------------------
def test_ranges_columns_and_chunks_give_the_same_rows(rcm):
    """8,200 columns: two chunks (8,192 + 8) for the whole range; ranges inside one chunk and across the boundary"""
    st = ensemble(rcm, 8200, 11)
    s = solver(rcm, 20, st)
    s.advance(1)
    whole = s.species_jacobian(vmr_scale=O3_HALF)
    for col0, m in ((0, 24), (8185, 15), (8199, 1), (11, 1), (1000, 7200)):
        sub = s.species_jacobian(col0, m, vmr_scale=O3_HALF)
        for key in ("J", "dE_jac"):
            assert np.array_equal(sub[key], whole[key][col0:col0 + m]), (key, col0)
    s.close()
    part = solver(rcm, 20, st, slice(4000, 4100))
    part.advance(1)
    tail = part.species_jacobian(vmr_scale=O3_HALF)
    part.close()
    for key in ("J", "dE_jac"):
        assert np.array_equal(whole[key][4000:4100], tail[key]), key


def test_the_call_changes_nothing(rcm, ens21, tmp_path):
    a, b = solver(rcm, 20, ens21), solver(rcm, 20, ens21)
    b.species_jacobian()
    sa = [a.advance(2), a.advance(3)]
    sb = [b.advance(2)]
    b.species_jacobian(vmr_scale=CO2_2X)
    b.species_jacobian(col0=3, ncol=5)
    sb.append(b.advance(3))
    b.species_jacobian()
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


# ---- 6. errors ---------------------------------------------------------------------------------------------------------------
def test_errors_leave_the_solver_usable(rcm, ens21):
    import ctypes as C
    OPT_PATH = 5
    L = rcm.load_library()
    s = solver(rcm, 20, ens21)
    for col0, ncol in ((-1, 3), (0, 0), (20, 2), (0, 22)):
        assert status_of(rcm, lambda: s.species_jacobian(col0, ncol)) == 1, (col0, ncol)
    for bad in (-1.0, np.nan, np.inf):
        assert status_of(rcm, lambda: s.species_jacobian(vmr_scale=[1.0, 1.0, bad, 1.0, 1.0])) == 1, bad
    with pytest.raises(ValueError):
        s.species_jacobian(vmr_scale=[2.0])
    assert L.rcm_species_jacobian(s._h, C.c_int(0), C.c_int(21), None, None, None) == 0   # nothing wanted
    s.set_option(OPT_PATH, 1)
    assert status_of(rcm, lambda: s.species_jacobian()) == 2
    s.set_option(OPT_PATH, 0)
    ref = s.species_jacobian()
    s.advance(1)
    assert np.isfinite(s.species_jacobian()["J"]).all() and np.isfinite(ref["J"]).all()
    s.close()

    for mask in (0x0F, 0x3E, 0x1F):   # four species; no H2O; five species but not the default's (species 4 for CH4)
        p = rcm.default_params()
        p.species_mask = mask
        m = solver(rcm, 20, ens21, params=p)
        assert status_of(rcm, lambda: m.species_jacobian()) == 2, mask
        m.advance(1)
        m.close()

    st = ens21
    lb = rcm.Solver(0)
    wvl, tau5 = rcm.make_lbl_tables(300, 7, st["plevel"], st["vmr9"][0, 0], st["vmr9"][0, 2])
    lb.set_lbl_tables(wvl, tau5, st["vmr9"][0, 0], st["vmr9"][0, 2])
    lb.set_columns(st["plevel"], st["Tlayer"], st["Tsurf"], st["vmr9"], st["rel_hum"])
    assert status_of(rcm, lambda: lb.species_jacobian()) == 2
    lb.advance(1)
    assert np.isfinite(lb.get_state(("E_up",))["E_up"]).all()
    lb.close()


# ---- 7. the driver's --species-jacobian-out -----------------------------------------------------------------------------------
def species_means(J, H):
    """the driver's rows [100][3]: column order, then one division"""
    acc = np.zeros((NE, 3))
    for c in range(J.shape[0]):
        row = np.stack([J[c, 1, 0], J[c, 0, NLEV - 1], H[c][np.arange(NE) % NLAY, np.arange(NE)]], axis=1)
        acc = acc + row
    return acc / J.shape[0]


def check_species_file(path, pl, J, H):
    lines = open(path).read().splitlines()
    assert lines[0] == "species,layer,p_layer,dOLR_dlnx,dSFC_dlnx,dHeat_dlnx" and len(lines) == NE + 1
    names = [l.split(",")[0] for l in lines[1:]]
    assert names == [n for n in ("h2o", "co2", "o3", "n2o", "ch4") for _ in range(NLAY)]
    assert [int(l.split(",")[1]) for l in lines[1:]] == list(range(NLAY)) * NS
    rows = np.array([[float(x) for x in l.split(",")[2:]] for l in lines[1:]])
    assert np.array_equal(rows[:, 0], np.tile((pl[:NLAY] + pl[1:]) / 2.0, NS))
    assert np.array_equal(rows[:, 1:], species_means(J, H))


def test_driver_species_jacobian_out(rcm, tmp_path):
    ck, sf = str(tmp_path / "run.ckpt"), str(tmp_path / "species.csv")
    common = ["--table", table_path(100), "--ncol", "64", "--seed", "9", "--max-steps", "3", "--steps-exact"]
    r = driver(rcm, *common, "--out", str(tmp_path / "o.txt"), "--checkpoint", ck, "--species-jacobian-out", sf)
    assert r.returncode == 0, r.stderr
    s = rcm.Solver(0)
    s.set_repwvl_table_from(rcm.Table(table_path(100)))
    s.load_checkpoint(ck)
    d = s.species_jacobian()
    s.close()
    pl = rcm.read_atm(os.path.join(GOLDEN, "column21.atm"))[:, 1]
    check_species_file(sf, pl, d["J"], d["dE_jac"])

    d = tmp_path / "lbl"
    d.mkdir()
    r = driver(rcm, "--lbl", str(d), "--species-jacobian-out", sf, "--max-steps", "1")
    assert r.returncode == 1 and "--species-jacobian-out" in r.stderr and "--lbl-species-jacobian-out" in r.stderr

    if rcm.device_count() < 2:
        pytest.skip("--gpus 2 needs two GPUs")
    sf2 = str(tmp_path / "species2.csv")
    r = driver(rcm, *common, "--out", str(tmp_path / "o2.txt"), "--species-jacobian-out", sf2, "--gpus", "2")
    assert r.returncode == 0, r.stderr
    assert open(sf).read() == open(sf2).read()
