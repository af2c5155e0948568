"""Cost and physics of the climate-response calls (rcm_climate_response, rcm_lbl_climate_response) on one GPU.

  repwvl: 65,536 columns on Reduced100 after 5 steps; medians of alternated synchronous calls: a step (rcm_advance(1)), the flux
          Jacobian (dE_jac only) and the 2xCO2 response with ntrop = 4 at fixed RH, tol 1e-6 W/m2, at most 20 updates.
  LBL:    the bench.py LBL workload, 4,096 columns x 20,000 synthetic wavelengths after 2 steps; the same three calls.
For both: the histogram of Newton updates and the ensemble means of dTs at fixed RH and at fixed q, of the IRF and of dT in the
stratosphere.  As information, not a test: on a few hundred repwvl columns the Tsurf difference of two time-stepped
rcm_run_to_equilibrium runs at co2_factor 1 and 2 next to the dTs of the response call at the first run's equilibrium.

    python tools/response_probe.py [--ncol 65536] [--lbl-ncol 4096] [--nwvl 20000] [--reps 5] [--eq-ncol 256] [--out FILE]
"""
import argparse
import os
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.dirname(ROOT))
import our_first_climate_model_b200 as rcm  # noqa: E402
from lbl_diag_probe import lbl_case  # noqa: E402

G = os.path.join(os.path.dirname(ROOT), "tests", "golden")
CO2_2X, NTROP, TOL = [1.0, 2.0, 1.0, 1.0, 1.0], 4, 1e-6


def repwvl_solver(ncol, co2_factor=1.0):
    atm = rcm.read_atm(os.path.join(G, "column21.atm"))
    pl = atm[:, 1].copy()
    Tlev, vlev = rcm.make_ensemble(ncol, 12345, pl, atm[:, 2].copy(), atm[:, 4:9].T.copy())
    st = rcm.init_columns(pl, Tlev, vlev, co2_factor)
    s = rcm.Solver(0)
    s.set_repwvl_table_from(rcm.Table(os.path.join(G, "Reduced100Forcing.rcmtab")))
    s.set_columns(pl, st["Tlayer"], np.full(ncol, 288.2), st["vmr9"], st["rel_hum"])
    return s


def timings(calls, reps):
    for f in calls.values():  # warm-up: modules, scratch allocation
        f()
    times = {k: [] for k in calls}
    for _ in range(reps):
        for k, f in calls.items():
            t0 = time.perf_counter()
            f()
            times[k].append(time.perf_counter() - t0)
    step = np.median(times["step"])
    jac = np.median(times["flux_jacobian"])
    return [f"{k:17s} median {1e3 * np.median(v):10.2f} ms   min {1e3 * np.min(v):10.2f} ms   "
            f"{np.median(v) / step:7.2f} x step   {np.median(v) / jac:6.3f} x flux_jacobian" for k, v in times.items()]


def physics(rh, q):
    lines = []
    for name, d in (("fixed RH", rh), ("fixed q", q)):
        it = d["iters"]
        ok = it >= 0
        lines.append(f"{name:8s}: Newton updates per column: " + ", ".join(f"{k}: {n}" for k, n in enumerate(np.bincount(it[ok])))
                     + f"; unconverged: {int((~ok).sum())}; mean dTs {d['dTs'][ok].mean():.6f} K, mean IRF_toa "
                     f"{d['IRF_toa'].mean():.6f} W/m2, mean dT of layers 0..{NTROP - 1}: "
                     + ", ".join(f"{x:.4f}" for x in d["dT"][ok].mean(axis=0)[:NTROP]) + " K")
    return lines


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--ncol", type=int, default=65536)
    ap.add_argument("--lbl-ncol", type=int, default=4096)
    ap.add_argument("--nwvl", type=int, default=20000)
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--eq-ncol", type=int, default=256)
    ap.add_argument("--out", default=None, help="also write the report here")
    a = ap.parse_args()
    card = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader", "-i", "0"],
                          capture_output=True, text=True).stdout.strip()
    lines = [f"card: {card}"]

    s = repwvl_solver(a.ncol)
    s.advance(5)
    rh, q = s.climate_response(CO2_2X, NTROP, tol=TOL), s.climate_response(CO2_2X, NTROP, fixed_rh=False, tol=TOL)

    def step():
        s.advance(1, want_scalars=False)
        s.synchronize()

    lines.append(f"repwvl: {a.ncol} columns, Reduced100 ({s.nwvl} wavelengths), 2xCO2, ntrop {NTROP}, tol {TOL:g} W/m2; physics at "
                 f"the state after 5 steps, then {a.reps} alternated reps (the state moves one step per rep)")
    lines += physics(rh, q)
    lines += timings({"step": step, "flux_jacobian": lambda: s.flux_jacobian(),
                      "climate_response": lambda: s.climate_response(CO2_2X, NTROP, tol=TOL)}, a.reps)
    s.close()

    c = lbl_case(a.lbl_ncol, a.nwvl, 4242)
    s = rcm.Solver(0)
    s.set_lbl_tables(c["wvl"], c["tau5"], c["h2o_ref"], c["o3_ref"], 1.0)
    st = c["st"]
    s.set_columns(c["pl"], st["Tlayer"], c["Tsurf"], st["vmr9"], st["rel_hum"])
    s.advance(2)
    rh, q = s.lbl_climate_response(CO2_2X, NTROP, tol=TOL), s.lbl_climate_response(CO2_2X, NTROP, fixed_rh=False, tol=TOL)
    lines.append(f"LBL: {a.lbl_ncol} columns x {a.nwvl} wavelengths (bench.py LBL case, after 2 steps), 2xCO2, ntrop {NTROP}, "
                 f"tol {TOL:g} W/m2; {max(2, a.reps // 2)} alternated reps")
    lines += physics(rh, q)
    lines += timings({"step": step, "flux_jacobian": lambda: s.lbl_flux_jacobian(),
                      "climate_response": lambda: s.lbl_climate_response(CO2_2X, NTROP, tol=TOL)}, max(2, a.reps // 2))
    s.close()

    eq = []
    for f in (1.0, 2.0):
        e = repwvl_solver(a.eq_ncol, f)
        done, last = e.run_to_equilibrium(40000, 100)
        eq.append((e, done, last))
    e1, e2 = eq[0][0], eq[1][0]
    dTs_run = e2.get_state(("Tsurf",))["Tsurf"] - e1.get_state(("Tsurf",))["Tsurf"]
    r = e1.climate_response(CO2_2X, NTROP, tol=TOL)
    ok = r["converged"]
    lines.append(f"time-stepped equilibrium, {a.eq_ncol} repwvl columns (Reduced100): co2_factor 1 after {eq[0][1]} steps "
                 f"({int(eq[0][2][2])} stationary), co2_factor 2 after {eq[1][1]} steps ({int(eq[1][2][2])} stationary); mean Tsurf "
                 f"difference {dTs_run.mean():.6f} K; climate_response at the first run's equilibrium (2xCO2, ntrop {NTROP}, fixed RH): "
                 f"mean dTs {r['dTs'][ok].mean():.6f} K ({int(ok.sum())} converged); mean |difference| per column "
                 f"{np.abs(r['dTs'][ok] - dTs_run[ok]).mean():.6f} K")
    for e, _, _ in eq:
        e.close()
    text = "\n".join(lines)
    print(text)
    if a.out:
        with open(a.out, "w") as fh:
            fh.write(text + "\n")


if __name__ == "__main__":
    main()
