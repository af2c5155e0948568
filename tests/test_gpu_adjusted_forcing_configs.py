"""Stratosphere-adjusted forcing (adjusted_forcing) away from the configuration test_gpu_adjusted_forcing tests: every angle
schedule and cloud layer of test_gpu_diagnostic_configs, the 10- and 100-wavelength tables, ntrop up to 19, other species
scaled, one Newton step reproduced exactly, the convergence rate, layers that change table interval between iterates, the
step-0 rule on a theta inversion, non-finite columns, three chunks with a reused stream slot and the shared __constant__ bank.

Checker: the C port of the reference (oracle/rcm_oracle.c) through test_gpu_diagnostic_configs.PortColumn, solved by
test_gpu_adjusted_forcing.FdhColumn (scipy's hybr); for the Newton step itself the kernel's Gaussian elimination restated in
exact arithmetic (kernel_solve), with numpy / scipy for the condition and the pivots.
"""
from fractions import Fraction

import numpy as np
import pytest
import scipy.linalg

from conftest import table_path
from test_gpu_adjusted_forcing import FdhColumn
from test_gpu_diagnostic_configs import (OPT_CUBES, OPT_PAIRS, SCHEDULES, TAU_FLOOR, assert_same, edge_ensemble,
                                         port_columns, schedule_7)
from test_gpu_diagnostics import ensemble, solver, theta_sort

pytestmark = pytest.mark.gpu
NLAY, NLEV = 20, 21
EPS = np.finfo(np.float64).eps
CO2_4X = [1.0, 4.0, 1.0, 1.0, 1.0]
ACTIVE_ROWS = [0, 1, 2, 3, 5]  # vmr9 rows of the default mask's species H2O, CO2, O3, N2O, CH4: vmr_scale's order
NTROP21 = (np.arange(21) * 7) % 20  # 21 columns: every ntrop 0 .. 19
TOL = 1e-9
MAX_ITERS = 6  # Newton updates to TOL at 4xCO2 on every ordinary column (see test_schedules_against_the_port)
KEYS = ("F", "dT_adj", "E_down", "E_up", "iters")


def scaled(v9, vmr_scale):
    """v9 with the active species' rows times vmr_scale: rcm_diag_scale_kernel's scaling, after the feedback"""
    v = np.array(v9, dtype=np.float64)
    v[ACTIVE_ROWS] = v[ACTIVE_ROWS] * np.asarray(vmr_scale, dtype=np.float64)[:, None]
    return v


def fdh_column(pc, vmr_scale):
    """The FdhColumn of a port column pc (schedule, cloud layer, floor as configured): base VMRs pc.v9, perturbed scaled"""
    def fluxes(v, dT=()):
        d = np.zeros(NLAY)
        d[:len(dT)] = dT
        return pc.broadband(0.0, tT=pc.tau_T + d, Tr=pc.Trad + d, v=v)

    return FdhColumn(pc.v9, scaled(pc.v9, vmr_scale), fluxes)


def check_against_port(d, cols, ntrop, vmr_scale):
    """dT to 1e-6 K, F to 1e-8 W/m2 of the port's own solution, the port's residual at the call's dT to 1e-8 W/m2"""
    for c, pc in cols:
        m = ntrop[c]
        fc = fdh_column(pc, vmr_scale)
        dT, F = fc.solve(m)
        assert np.all(d["dT_adj"][c, m:] == 0.0), c
        assert np.abs(d["dT_adj"][c] - dT).max() <= 1e-6, (c, m, d["dT_adj"][c] - dT)
        assert np.abs(d["F"][c] - F).max() <= 1e-8, (c, m, d["F"][c] - F)
        assert fc.residual(m, d["dT_adj"][c]) <= 1e-8, (c, m, fc.residual(m, d["dT_adj"][c]))


def assert_converged(d, what):
    hist = np.bincount(d["iters"] + 1)
    print(f"{what}: iters -1.. {hist.tolist()}")
    assert np.all(d["converged"]), (what, hist)
    assert d["iters"].max() <= MAX_ITERS, (what, hist)


def configured(rcm, n, st, nangle=30, cubes=None, pairs=None, cloud=17, nsteps=0):
    p = rcm.default_params()
    p.nangle, p.cloud_layer = nangle, cloud
    s = solver(rcm, n, st, params=p)
    if cubes is not None:
        s.set_option(OPT_CUBES, cubes)
        s.set_option(OPT_PAIRS, pairs)
    if nsteps:
        s.advance(nsteps)
    return s


# ---- 1. schedules, cloud layers, tables, species -----------------------------------------------------------------------------
@pytest.mark.parametrize("nangle,cubes,pairs,cloud,nsteps", SCHEDULES)
def test_schedules_against_the_port(rcm, port, nangle, cubes, pairs, cloud, nsteps):
    """21 columns, Reduced20, 4xCO2, ntrop 0 .. 19: a wrong angle weight in the Newton step's Jacobian (steps 30 / nangle
    times too long or too short) leaves columns unconverged or over MAX_ITERS."""
    tab = port.load_rcmtab(table_path(20))
    st = ensemble(rcm, 21, 900 + nangle)
    s = configured(rcm, 20, st, nangle, cubes, pairs, cloud, nsteps)
    d = s.adjusted_forcing(CO2_4X, NTROP21, tol=TOL)
    g = s.get_state(("Tlayer", "Tsurf"))
    s.close()
    assert_converged(d, f"nangle {nangle} cubes {cubes} pairs {pairs} cloud {cloud} steps {nsteps}")
    check_against_port(d, port_columns(port, g, st, tab, nsteps, range(21), nangle=nangle, cloud_layer=cloud), NTROP21,
                       CO2_4X)


@pytest.mark.parametrize("n", [10, 100])
def test_other_tables_against_the_port(rcm, port, n):
    """Reduced10 on every column, Reduced100 on five (ntrop 7, 2, 17, 19, 0)"""
    tab = port.load_rcmtab(table_path(n))
    st = ensemble(rcm, 21, 950 + n)
    s = configured(rcm, n, st, nsteps=2)
    d = s.adjusted_forcing(CO2_4X, NTROP21, tol=TOL)
    g = s.get_state(("Tlayer", "Tsurf"))
    s.close()
    assert_converged(d, f"Reduced{n}")
    cols = range(21) if n == 10 else (1, 6, 11, 17, 20)
    check_against_port(d, port_columns(port, g, st, tab, 2, cols), NTROP21, CO2_4X)


@pytest.mark.parametrize("vmr_scale", [[1.0, 0.5, 1.0, 1.0, 1.0], [1.5, 1.0, 1.0, 1.0, 1.0], [1.0, 1.0, 0.5, 1.0, 1.0],
                                       [1.2, 3.0, 0.8, 1.1, 1.3]], ids=["CO2x0.5", "H2Ox1.5", "O3x0.5", "combined"])
def test_other_perturbations_against_the_port(rcm, port, vmr_scale):
    tab = port.load_rcmtab(table_path(20))
    st = ensemble(rcm, 21, 977)
    s = configured(rcm, 20, st, nsteps=2)
    d = s.adjusted_forcing(vmr_scale, NTROP21, tol=TOL)
    g = s.get_state(("Tlayer", "Tsurf"))
    s.close()
    assert_converged(d, str(vmr_scale))
    if vmr_scale[1] == 0.5:  # less CO2: negative forcing, and the stratosphere warms
        assert np.all(d["IRF_toa"] < 0.0) and d["dT_adj"][NTROP21 > 0, 0].min() > 0.0
    check_against_port(d, port_columns(port, g, st, tab, 2, range(21)), NTROP21, vmr_scale)


# ---- 2. one Newton step ------------------------------------------------------------------------------------------------------
def fms(c, a, b):
    """c - a * b rounded once: the DFMA the kernel's elimination and back substitution compile to"""
    return float(Fraction(c) - Fraction(a) * Fraction(b))


def kernel_solve(A, b):
    """rcm_fdh_newton_kernel's elimination in its operation order: pivot the largest |A[r][k]|, r >= k (the lowest row on
    ties), rows below updated as A[r][j] - f A[k][j] with f = A[r][k] / A[k][k], back substitution v - A[r][j] x[j] in
    ascending j, then v / A[r][r].  -> x"""
    m = len(b)
    M = [[float(x) for x in row] + [float(y)] for row, y in zip(A, b)]
    for k in range(m):
        p = max(range(k, m), key=lambda r: (abs(M[r][k]), -r))
        M[k][k:], M[p][k:] = M[p][k:], M[k][k:]
        for r in range(k + 1, m):
            f = M[r][k] / M[k][k]
            for j in range(k + 1, m + 1):
                M[r][j] = fms(M[r][j], f, M[k][j])
    x = [0.0] * m
    for r in range(m - 1, -1, -1):
        v = M[r][m]
        for j in range(r + 1, m):
            v = fms(v, M[r][j], x[j])
        x[r] = v / M[r][r]
    return np.array(x)


def one_step_case(rcm, port, case):
    """-> solver, ensemble, table, steps done, port-column options of the case"""
    if case == "edge":
        tab = port.load_rcmtab(table_path(20))
        st = edge_ensemble(rcm, port, tab)
        return solver(rcm, 20, st), st, tab, 0, dict(tau_floor=TAU_FLOOR, stable=True)
    n = int(case[1:])
    tab = port.load_rcmtab(table_path(n))
    st = ensemble(rcm, 38, 1000 + n)
    s = solver(rcm, n, st)
    s.advance(2)
    return s, st, tab, 2, {}


@pytest.mark.parametrize("case", ["R20", "R100", "edge"])
def test_one_newton_step_is_the_solve_of_the_jacobian_block(rcm, port, case):
    """max_iter = 1 at a tolerance no update meets: dT_adj[c, :m] is the solution of dE_jac[c, :m, :m] delta = -(dE_pert -
    dE_base)[c, :m] with flux_jacobian's and diagnose_fluxes' values (iterate 0 is those calls bit for bit), equal to the
    kernel's elimination restated exactly, with a backward error of a few m eps and within m eps cond of numpy's solve; E_down,
    E_up the port's at that delta.  Every m in 1 .. 19.  The blocks of ordinary columns are diagonally dominant; the edge
    ensemble's cold-layer columns give blocks that need a row exchange."""
    s, st, tab, nsteps, cfg = one_step_case(rcm, port, case)
    ncol = st["Tlayer"].shape[0]
    ntrop = 1 + np.arange(ncol) % 19
    base = s.diagnose_fluxes(spectral=False)
    pert = s.diagnose_fluxes(vmr_scale=CO2_4X, spectral=False)
    H = s.flux_jacobian(vmr_scale=CO2_4X)["dE_jac"]
    d = s.adjusted_forcing(CO2_4X, ntrop, tol=1e-300, max_iter=1)
    g = s.get_state(("Tlayer", "Tsurf"))
    s.close()
    compared, exchanged, worst = set(), 0, 0.0
    for c, pc in port_columns(port, g, st, tab, nsteps, range(ncol), **cfg):
        m = ntrop[c]
        A, r = H[c, :m, :m], -(pert["dE"][c, :m] - base["dE"][c, :m])
        if not (np.isfinite(A).all() and np.isfinite(r).all()):
            continue
        x = d["dT_adj"][c, :m]
        assert d["iters"][c] == -1 and np.all(d["dT_adj"][c, m:] == 0.0), c
        assert np.array_equal(x, kernel_solve(A, r)), (c, m)
        back = np.abs(A @ x - r).max() / (np.abs(A) @ np.abs(x) + np.abs(r)).max()
        assert back <= 4 * m * EPS, (c, m, back)
        ref = np.linalg.solve(A, r)
        err = np.abs(x - ref).max() / np.abs(ref).max()
        assert err <= 4 * m * EPS * np.linalg.cond(A, np.inf), (c, m, err)
        worst = max(worst, back / (m * EPS))
        Ed, Eu, _ = fdh_column(pc, CO2_4X).fluxes(scaled(pc.v9, CO2_4X), x)
        if np.isfinite(Ed).all() and np.isfinite(Eu).all():  # (cold layers: e^(480 k) may overflow at deeper levels)
            sc = np.abs(Eu).max()
            assert np.abs(d["E_down"][c] - Ed).max() <= 1e-10 * sc and np.abs(d["E_up"][c] - Eu).max() <= 1e-10 * sc, c
        exchanged += int(np.any(scipy.linalg.lu_factor(A)[1] != np.arange(m)))
        compared.add(m)
    print(f"{case}: {exchanged} of the compared blocks need a row exchange; backward error <= {worst:.2f} m eps")
    assert compared == set(range(1, 20)), compared
    if case == "edge":
        assert exchanged > 0


# ---- 3. convergence rate ----------------------------------------------------------------------------------------------------
FLOOR = 1e-10  # W/m2: the port's residual at the kernels' converged dT


@pytest.mark.parametrize("m", [4, 12, 19])
def test_convergence_is_superlinear(rcm, port, m):
    """Iterates 1 .. 4 (max_iter = K from dT = 0): the port's residual at iterate K falls quadratically to the floor the
    port and the kernels agree to; a Jacobian with a stale Planck profile converges only linearly."""
    tab = port.load_rcmtab(table_path(20))
    st = ensemble(rcm, 21, 1234)
    s = solver(rcm, 20, st)
    s.advance(2)
    dT = [s.adjusted_forcing(CO2_4X, m, tol=1e-300, max_iter=K)["dT_adj"] for K in (1, 2, 3, 4)]
    g = s.get_state(("Tlayer", "Tsurf"))
    s.close()
    worst = np.zeros(3)
    for c, pc in port_columns(port, g, st, tab, 2, range(21)):
        fc = fdh_column(pc, CO2_4X)
        r = [fc.residual(m, x[c]) for x in dT]
        worst = np.maximum(worst, [r[1] / r[0], r[2] / max(r[1], FLOOR), r[3] / max(r[2], FLOOR)])
        assert r[1] <= 1e-2 * r[0], (c, r)
        assert r[2] <= max(1e-3 * r[1], FLOOR), (c, r)
        assert r[3] <= max(1e-3 * r[2], FLOOR), (c, r)
    print(f"m {m}: largest r2/r1, r3/max(r2, floor), r4/max(r3, floor): {worst}")


# ---- 4. profiles that move the table interval and the step-0 rule -------------------------------------------------------------
def layer_t_ref(port, tab, st):
    _, lp, _ = port.read_tau(tab, st["plevel"], st["Tlayer"][0], st["vmr9"][0])
    return tab["t_ref"][lp[::-1]]  # the reference temperature of every layer's pressure (lowpos_p is bottom-up)


def test_layers_that_cross_a_table_node(rcm, port):
    """Step 0, stable columns whose stratospheric layers sit 0.05 .. 0.5 K above a temperature node of their pressure: the
    4xCO2 adjustment cools them below it, so the interval (TBI_IT) changes between the iterates."""
    tab = port.load_rcmtab(table_path(20))
    st = ensemble(rcm, 21, 4321)
    t_ref, rng = layer_t_ref(port, tab, st), np.random.default_rng(8)
    ntrop = 4 + np.arange(21) % 6
    for c in range(21):
        T, th = st["Tlayer"][c], st["Tlayer"][c] * st["conv"]
        for l in range(ntrop[c]):  # the node nearest to T_l that keeps theta decreasing downward
            cand = t_ref[l] + tab["t_pert"] + rng.uniform(0.05, 0.5)
            ok = (cand * st["conv"][l] > th[l + 1]) & ((cand * st["conv"][l] < th[l - 1]) if l else True)
            if ok.any():
                T[l] = cand[ok][np.argmin(np.abs(cand[ok] - T[l]))]
                th[l] = T[l] * st["conv"][l]
        assert np.allclose(theta_sort(port, st["Tlayer"][c], st["conv"]), st["Tlayer"][c], rtol=1e-15, atol=0), c
    s = solver(rcm, 20, st)
    d = s.adjusted_forcing(CO2_4X, ntrop, tol=TOL)
    g = s.get_state(("Tlayer", "Tsurf"))
    s.close()
    assert_converged(d, "node columns")
    moved = 0
    for c, pc in port_columns(port, g, st, tab, 0, range(21)):
        lt0 = pc.tau(pc.tau_T, pc.v9)[2][::-1]
        lt1 = pc.tau(pc.tau_T + d["dT_adj"][c], pc.v9)[2][::-1]
        moved += int(np.sum(lt0[:ntrop[c]] != lt1[:ntrop[c]]))
    print(f"{moved} of {ntrop.sum()} stratospheric layers change interval")
    assert moved >= ntrop.sum() // 2, moved
    check_against_port(d, port_columns(port, g, st, tab, 0, range(21)), ntrop, CO2_4X)


def test_step_0_with_a_theta_inversion(rcm, port):
    """Step 0 with a 4 .. 8 K warm bump at layers 8 .. 16 and ntrop 17 .. 19: the sorted profile (the Planck source) and
    the unsorted one (tau) differ inside the stratosphere, and dT moves both."""
    tab = port.load_rcmtab(table_path(20))
    st = ensemble(rcm, 21, 5678)
    st["Tlayer"][:, 8:17] += np.random.default_rng(3).uniform(4.0, 8.0, (21, 1))
    ntrop = 17 + np.arange(21) % 3
    for c in range(21):
        Ts = theta_sort(port, st["Tlayer"][c], st["conv"])
        assert np.any(np.abs(Ts - st["Tlayer"][c])[:ntrop[c]] > 1.0), c
    s = solver(rcm, 20, st)
    d = s.adjusted_forcing(CO2_4X, ntrop, tol=TOL)
    g = s.get_state(("Tlayer", "Tsurf"))
    s.close()
    assert_converged(d, "theta inversion")
    check_against_port(d, port_columns(port, g, st, tab, 0, range(21)), ntrop, CO2_4X)


# ---- 5. non-finite columns ---------------------------------------------------------------------------------------------------
def test_edge_ensemble(rcm, port):
    """Step 0 of the edge ensemble on Reduced20, four of its wild columns with every other layer 150 K below its
    pressure's reference temperature (tau below the floor in many layers: the fluxes overflow): RCM_OK; a column whose
    residual is not finite freezes at -1; every column equals a call on it alone; the finite, converged columns with
    tau >= 0 match the port."""
    tab = port.load_rcmtab(table_path(20))
    st = edge_ensemble(rcm, port, tab)
    t_ref = layer_t_ref(port, tab, st)
    for c in range(40, 44):
        st["Tlayer"][c, 1:19:2] = t_ref[1:19:2] - 150.0
    ncol = st["Tlayer"].shape[0]
    ntrop = np.where((np.arange(ncol) >= 48) | ((np.arange(ncol) >= 40) & (np.arange(ncol) < 44)), 19,
                     1 + np.arange(ncol) % 19)
    s = solver(rcm, 20, st)
    base = s.diagnose_fluxes(spectral=False)
    pert = s.diagnose_fluxes(vmr_scale=CO2_4X, spectral=False)
    d = s.adjusted_forcing(CO2_4X, ntrop, tol=TOL)
    for c in range(ncol):
        one = s.adjusted_forcing(CO2_4X, ntrop[c:c + 1], col0=c, ncol=1, tol=TOL)
        for k in KEYS:
            assert np.array_equal(d[k][c:c + 1], one[k], equal_nan=True), (c, k)
    g = s.get_state(("Tlayer", "Tsurf"))
    s.close()
    bad = [c for c in range(ncol) if not (np.isfinite(base["dE"][c, :ntrop[c]]).all()
                                          and np.isfinite(pert["dE"][c, :ntrop[c]]).all())]
    assert bad and np.all(d["iters"][bad] == -1), (bad, d["iters"][bad])
    plain = []
    for c, pc in port_columns(port, g, st, tab, 0, range(ncol), tau_floor=TAU_FLOOR, stable=True):
        if c not in bad and d["converged"][c] and pc.tau(pc.tau_T, pc.v9)[0].min() >= 0.0:
            plain.append((c, pc))
    print(f"{len(bad)} non-finite columns, {int(np.sum(~d['converged']))} unconverged, {len(plain)} compared")
    assert len(plain) >= ncol // 2, len(plain)
    check_against_port(d, plain, ntrop, CO2_4X)


# ---- 6. three chunks -----------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("fast", [1, 0])
def test_three_chunks_and_a_reused_slot(rcm, fast):
    """16,400 columns = 8,192 + 8,192 + 16.  fast = 1: chunk 1 has no stratosphere, its slot finishes at iterate 0 and
    takes chunk 2 while chunk 0 iterates.  fast = 0: chunk 0 has one stratospheric layer and needs no more updates than
    chunk 1, so its slot (checked first) finishes after iterating and takes chunk 2 with its iterate count reset.  Whole
    range = each chunk alone = single columns."""
    n, ch = 16400, 8192
    st = ensemble(rcm, n, 31 + fast)
    s = solver(rcm, 20, st)
    s.advance(1)
    ntrop = (np.arange(n) * 7) % 20
    ntrop[fast * ch:(fast + 1) * ch] = 1 - fast
    whole = s.adjusted_forcing(CO2_4X, ntrop, tol=TOL)
    it = whole["iters"]
    if fast == 0:
        assert 1 <= it[:ch].max() <= it[ch:2 * ch].max(), (it[:ch].max(), it[ch:2 * ch].max())
    for c0 in (0, ch, 2 * ch):
        part = s.adjusted_forcing(CO2_4X, ntrop[c0:c0 + ch], col0=c0, ncol=min(ch, n - c0), tol=TOL)
        for k in KEYS:
            assert np.array_equal(whole[k][c0:c0 + ch], part[k]), (c0, k)
    for c in (0, 8191, 8192, 16383, 16384, 16399):
        one = s.adjusted_forcing(CO2_4X, ntrop[c:c + 1], col0=c, ncol=1, tol=TOL)
        for k in KEYS:
            assert np.array_equal(whole[k][c:c + 1], one[k]), (c, k)
    s.close()
    assert np.all(whole["converged"])


# ---- 7. the shared constant bank -----------------------------------------------------------------------------------------------
def test_two_solvers_on_one_device(rcm):
    """A 30-angle and a 7-angle solver on one device, calls interleaved: each equals its solver alone, bit for bit."""
    st = ensemble(rcm, 21, 2024)
    call = lambda s: s.adjusted_forcing(CO2_4X, NTROP21, tol=TOL)
    alone = {}
    for name, p in (("30", None), ("7", schedule_7(rcm))):
        s = solver(rcm, 20, st, params=p)
        s.advance(2)
        alone[name] = call(s)
        s.close()
    assert not np.array_equal(alone["30"]["F"], alone["7"]["F"])
    a, b = solver(rcm, 20, st), solver(rcm, 20, st, params=schedule_7(rcm))
    a.advance(2)
    b.advance(2)
    for s, name in ((a, "30"), (b, "7"), (a, "30"), (b, "7")):
        assert_same(call(s), alone[name], name)
    a.close()
    b.close()


def test_set_params_on_a_live_solver(rcm, tmp_path):
    """set_params(nangle = 7) after a 30-angle call equals a fresh 7-angle solver that loaded the live one's checkpoint"""
    st = ensemble(rcm, 21, 2024)
    call = lambda s: s.adjusted_forcing(CO2_4X, NTROP21, tol=TOL)
    s = solver(rcm, 20, st)
    s.advance(2)
    at30 = call(s)
    ck = str(tmp_path / "live.ckpt")
    s.save_checkpoint(ck)
    s.set_params(schedule_7(rcm))
    live = call(s)
    s.close()
    f = rcm.Solver(0, schedule_7(rcm))
    f.set_repwvl_table_from(rcm.Table(table_path(20)))
    f.load_checkpoint(ck)
    fresh = call(f)
    f.close()
    assert_same(live, fresh, "live")
    assert not np.array_equal(live["F"], at30["F"])
