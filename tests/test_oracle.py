"""The CPU oracles against the reference's own artefacts (no GPU).

* output.txt of the reference (the only committed numbers): solar setup for three cloud optical
  depths and the t=0 profile rows;
* golden vectors produced by the UNMODIFIED reference (tools/make_golden.py): the plain-C port
  (oracle/rcm_oracle.c) must reproduce them bit for bit;
* the reference-built oracle (oracle/_ref) is re-run live when it is present.
"""
import os

import numpy as np
import pytest

from conftest import GOLDEN, table_path
from oracle import refcpu as R

needs_ref = pytest.mark.skipif(not R.available(), reason="oracle/_ref not built (no /root/reference)")


def test_solar_setup_matches_committed_reference_output(port):
    # /root/reference/output.txt:3-6 and :30-33 (values printed with %f), and the committed tau_s = 2.0
    for tau_s, albedo, rdir, sdir, tdir, solar in [(2.07672, 0.309331, 0.237519, 0.226157, 0.536324, 235.000099),
                                                   (2.05, 0.307414, 0.235182, 0.224178, 0.540641, 235.652433),
                                                   (2.0, 0.303798, None, None, None, 236.882897)]:
        s = port.solar_setup(tau_s=tau_s)
        assert f"{s['r_total']:.6f}" == f"{albedo:.6f}"
        assert f"{s['solar_irr']:.6f}" == f"{solar:.6f}"
        if rdir is not None:
            assert f"{s['r_dir']:.6f}" == f"{rdir:.6f}"
            assert f"{s['s_dir']:.6f}" == f"{sdir:.6f}"
            assert f"{s['t_dir']:.6f}" == f"{tdir:.6f}"
        assert abs(s["r_dir"] + s["s_dir"] + s["t_dir"] - 1.0) < 1e-6  # "sum: 1.000000", output.txt:5


def test_initial_profile_rows_match_committed_reference_output(port, golden):
    # /root/reference/output.txt:8-27: layer,player,Tlayer,theta,time at t=0
    rows = """0,25.000000,221.393000,635.177801 1,75.000000,221.393000,464.060873 2,125.000000,221.393000,401.041758
    3,175.000000,221.393000,364.282852 4,225.000000,221.393000,339.042853 5,275.000000,225.299500,325.799855
    6,325.000000,232.616500,320.702550 7,375.000000,239.063000,316.386335 8,425.000000,244.842000,312.651495
    9,475.000000,250.091000,309.365099 10,525.000000,254.908000,306.434706 11,575.000000,259.365500,303.793542
    12,625.000000,263.518000,301.391001 13,675.000000,267.409000,299.189516 14,725.000000,271.073000,297.159548
    15,775.000000,274.537000,295.276557 16,825.000000,277.824000,293.521596 17,875.000000,280.953500,291.879487
    18,925.000000,283.941500,290.337186 19,975.000000,286.801000,288.883142""".split()
    st = port.init_columns(golden["plevel"], golden["Tlevel"][:1], golden["vmr_ppm_level"][:1])
    T = st["Tlayer"][0].copy()
    theta = T * st["conv"]
    assert np.all(np.diff(theta) < 0), "theta-sort is a no-op on the initial profile"
    for i, row in enumerate(rows):
        assert row == f"{i},{st['player'][i]:f},{T[i]:f},{theta[i]:f}"


def test_lowerpos_truth_table(port, golden_misc):
    asc, desc = [0.0, 1.0, 2.0, 3.0], [3.0, 2.0, 1.0, 0.0]
    xs = golden_misc["lp_x"]
    assert [port.lowerpos(asc, x) for x in xs] == list(golden_misc["lp_asc"])
    assert [port.lowerpos(desc, x) for x in xs] == list(golden_misc["lp_desc"])
    # SURVEY.md Appendix A.1: out of range on either side -> last interval; exact hit -> lower neighbour
    assert port.lowerpos(asc, -1) == 2 and port.lowerpos(asc, 4) == 2 and port.lowerpos(asc, 2) == 1


@pytest.mark.parametrize("n", [10, 20, 100])
def test_port_reproduces_reference_golden_bitwise(port, golden, n):
    g = golden
    tab = port.load_rcmtab(table_path(n))
    for c in (0, 3, 14, 15):
        tau, lp, lt = port.read_tau(tab, g["plevel"], g["Tlayer"][c], g["vmr9"][c])
        assert np.array_equal(tau, g[f"tau{n}"][c])
        assert np.array_equal(lp, g[f"lowpos_p{n}"][c]) and np.array_equal(lt, g[f"lowpos_t{n}"][c])
    r1 = port.advance(tab, g["plevel"], g["rel_hum"], float(g["solar_irr"]), g["Tlayer"], g["Tsurf"], g["vmr9"], 1)
    for k in ("E_down", "E_up", "dE", "dt", "Tlayer", "Tsurf", "time_h"):
        assert np.array_equal(r1[k], g[f"s1_{k}_{n}"]), k
    r5 = port.advance(tab, g["plevel"], g["rel_hum"], float(g["solar_irr"]), g["Tlayer"], g["Tsurf"], g["vmr9"], 5,
                      want_trace=True)
    for k in ("E_down", "E_up", "dE", "dt", "Tlayer", "Tsurf", "time_h", "trace"):
        assert np.array_equal(r5[k], g[f"s5_{k}_{n}"]), k


def test_port_chunked_advance_equals_single_run(port, golden):
    g = golden
    tab = port.load_rcmtab(table_path(20))
    a = port.advance(tab, g["plevel"], g["rel_hum"], float(g["solar_irr"]), g["Tlayer"], g["Tsurf"], g["vmr9"], 2)
    b = port.advance(tab, g["plevel"], g["rel_hum"], float(g["solar_irr"]), a["Tlayer"], a["Tsurf"], a["vmr9"], 3,
                     first_step=2, time_h=a["time_h"])
    for k in ("E_down", "E_up", "dE", "Tlayer", "Tsurf", "time_h"):
        assert np.array_equal(b[k], g[f"s5_{k}_20"]), k


def test_port_edge_members(port, golden_edge):
    e = golden_edge
    for n in (10, 100):
        tab = port.load_rcmtab(table_path(n))
        for c in range(4):
            tau, lp, lt = port.read_tau(tab, e["plevel"], e["Tlayer"][c], e["vmr9"][c])
            assert np.array_equal(tau, e[f"tau{n}"][c])
            assert np.array_equal(lt, e[f"lowpos_t{n}"][c])


def test_port_cplkavg_matches_reference_samples(port, golden_misc):
    m = golden_misc
    got = np.array([port.cplkavg(a, b, t)[0] for a, b, t in zip(m["cpl_lo"], m["cpl_hi"], m["cpl_T"])])
    assert np.array_equal(got, m["cpl_val"])
    # full spectrum integrates to sigma T^4 / pi (libRadtran constant SIGMA = 5.67032e-8)
    v, st = port.cplkavg(1.0, 1e9, 300.0)
    assert st == 0 and abs(v - 5.67032e-8 * 300.0 ** 4 / np.pi) / v < 1e-6
    assert port.cplkavg(500.0, 400.0, 300.0)[1] == 1  # bad arguments: the reference exits here


def test_golden_survey_anchor_values(golden):
    # SURVEY.md section 8(c) / BASELINE.md section 4: step-0 fluxes of the base column
    for n, olr, ed, eu in [(10, 248.7241813688, 356.7120946431, 391.0613779498),
                           (20, 246.3964328153, 354.7132735806, 390.4620643786),
                           (100, 246.6782921988, 354.5377453745, 390.3394841235)]:
        assert abs(golden[f"s1_E_up_{n}"][0, 0] - olr) < 5e-10
        assert abs(golden[f"s1_E_down_{n}"][0, 20] - ed) < 5e-10
        assert abs(golden[f"s1_E_up_{n}"][0, 20] - eu) < 5e-10
    assert abs(golden["s1_dt_100"][0] - 13205.7) < 0.05 and abs(golden["s1_Tsurf_100"][0] - 293.919442) < 1e-6


def test_reference_live_equals_golden_and_port(port, golden, golden_misc):
    """The reference-built oracle when oracle/_ref is built; otherwise the outputs the reference stored in the golden files
    (solar setup, initial state) stand in for it and the port's run is the one checked."""
    g = golden
    if R.available():
        sol = R.solar()
    else:
        sol = {k: float(golden_misc["solar_" + k]) for k in port.solar_setup()}
    assert sol == port.solar_setup() and sol["solar_irr"] == float(g["solar_irr"])
    args = (g["plevel"], g["rel_hum"][:3], sol["solar_irr"], g["Tlayer"][:3], g["Tsurf"][:3], g["vmr9"][:3], 5)
    r = R.advance(table_path(100), *args) if R.available() else port.advance(port.load_rcmtab(table_path(100)), *args)
    for k in ("E_down", "E_up", "dE", "Tlayer", "Tsurf"):
        assert np.array_equal(r[k], g[f"s5_{k}_100"][:3]), k
    if R.available():
        st = R.init_columns(g["plevel"], g["Tlevel"], g["vmr_ppm_level"])
    else:
        st = {k: g["init_" + k] if "init_" + k in g.files else g[k] for k in ("Tlayer", "vmr9", "rel_hum", "player", "conv")}
    sp = port.init_columns(g["plevel"], g["Tlevel"], g["vmr_ppm_level"])
    for k in st:
        assert np.array_equal(st[k], sp[k]) and np.array_equal(st[k][:14] if st[k].ndim > 1 else st[k],
                                                                g["init_" + k] if "init_" + k in g.files else g[k])


@needs_ref
def test_lbl_composition_uses_reference_components(port):
    """LBL step: the port's sweep structure with tau given must equal the reference's radiative_transfer
    when the band Planck source is replaced consistently - checked through linearity in the source."""
    rng = np.random.default_rng(5)
    nw = 40
    wvl = np.sort(10 ** rng.uniform(3.7, 4.9, nw))
    lo, hi = port.lbl_bin_edges(wvl)
    assert np.all(hi > lo) and np.allclose(hi[:-1], lo[1:])
    assert np.array_equal(np.array([R.cplkavg(a, b, 250.0) for a, b in zip(lo, hi)]),
                          np.array([port.cplkavg(a, b, 250.0)[0] for a, b in zip(lo, hi)]))


@needs_ref
def test_lbl_step_sweeps_equal_the_reference_radiative_transfer_by_linearity(port, golden):
    """Path-level pin of the LBL composition's sweep / accumulation structure to the REFERENCE's radiative_transfer
    (main.cpp:320-344).  Fluxes are linear in the sources (B_0 .. B_19, B_surface) for a given tau.  The reference ties its
    source to T through the monochromatic Planck function times a spectral weight, so one source at a time is handed to
    it: layer l at its temperature with weights w_i = cplkavg(lo_i, hi_i, T_l) / planck(lambda_i, 1, T_l) - then the
    reference's w_i * planck(lambda_i, T_l) IS the band-integrated source of the LBL step - and every other layer and the
    surface at 1 K (their Planck source is exactly 0).  The 21 reference runs add up to the LBL port's step."""
    rng = np.random.default_rng(5)
    nw = 24
    wvl = np.sort(10 ** rng.uniform(3.7, 4.9, nw))
    lo, hi = port.lbl_bin_edges(wvl)
    pl, conv = golden["plevel"], golden["conv"]
    T0 = golden["Tlayer"][3] + rng.uniform(-2, 2, 20)
    Ts = 291.3
    Tsorted = -np.sort(-(T0 * conv)) / conv                      # main.cpp:536-540, as the step does first
    tau = 10 ** rng.uniform(-4, 1.3, (nw, 20))
    tau5 = np.zeros((5, nw, 20))
    tau5[3] = tau                                                # the unscaled CH4 slot carries the whole optical depth
    h2o_ref = golden["vmr9"][3, 0]
    got = port.lbl_advance(wvl, tau5, pl, golden["rel_hum"][3:4], h2o_ref, np.ones((1, 20)), 1.0, 0.0, T0[None], Ts,
                           h2o_ref[None], 1, cloud_on=False)
    L = port.lib()
    Ed, Eu = np.zeros(21), np.zeros(21)
    for src in range(21):
        Tsrc = Ts if src == 20 else Tsorted[src]
        w = np.array([R.cplkavg(a, b, Tsrc) / L.rcmo_planck(float(x), 1.0, float(Tsrc)) for a, b, x in zip(lo, hi, wvl)])
        Tl = np.full(20, 1.0)
        if src < 20:
            Tl[src] = Tsrc
        ed, eu, _ = R.radiative_transfer(tau, wvl, w, Tl, Ts if src == 20 else 1.0, 0.0)
        Ed += ed
        Eu += eu
    scale = np.abs(Eu).max()
    assert np.max(np.abs(got["E_down"][0] - Ed)) < 1e-12 * scale and np.max(np.abs(got["E_up"][0] - Eu)) < 1e-12 * scale
    assert Eu[0] > 1.0 and Ed[20] > 1.0                          # a real thermal spectrum, not zeros


def test_port_reaches_the_reference_equilibrium_for_a_perturbed_member(port, golden, golden_eq):
    """The C port over 6,000 iterations == the unmodified reference (tests/golden/ref_equilibrium.npz), bit for bit, for the
    most strongly perturbed member of the fixture (T_surface 297.8 K at equilibrium)."""
    c = int(np.argmax(golden_eq["Tsurf"]))
    assert c not in (0, 14, 15)
    r = port.advance(port.load_rcmtab(table_path(100)), golden["plevel"], golden["rel_hum"][c:c + 1], float(golden["solar_irr"]),
                     golden["Tlayer"][c:c + 1], golden["Tsurf"][c:c + 1], golden["vmr9"][c:c + 1], int(golden_eq["nsteps"]))
    assert np.array_equal(r["Tlayer"][0], golden_eq["Tlayer"][c]) and r["Tsurf"][0] == golden_eq["Tsurf"][c]
