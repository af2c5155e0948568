"""Cost of the line-by-line flux-Jacobian and adjusted-forcing calls (rcm_lbl_flux_jacobian, rcm_lbl_adjusted_forcing) on the
bench.py LBL workload: 4,096 columns x 20,000 synthetic wavelengths, after two steps.  Medians of alternated calls: one LBL
step (rcm_advance(1)), the flux Jacobian, and the adjusted forcing of 2xCO2 with 4 stratospheric layers at tol 1e-6 W/m2.
Also prints the Newton-update counts, the ensemble-mean IRF and SARF at TOA and at the tropopause, the ensemble-mean dT_adj
per stratospheric layer, and the card's name and power limit read in the same run.

    python tools/lbl_forcing_probe.py [--ncol 4096] [--nwvl 20000] [--reps 5] [--out FILE]
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

CO2_2X, NTROP, TOL = [1.0, 2.0, 1.0, 1.0, 1.0], 4, 1e-6


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--ncol", type=int, default=4096)
    ap.add_argument("--nwvl", type=int, default=20000)
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--out", default=None, help="also write the report here")
    a = ap.parse_args()
    card = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader", "-i", "0"],
                          capture_output=True, text=True).stdout.strip()
    rcm.load_library()
    c = lbl_case(a.ncol, a.nwvl, 4242)
    s = rcm.Solver(0)
    s.set_lbl_tables(c["wvl"], c["tau5"], c["h2o_ref"], c["o3_ref"], 1.0)
    st = c["st"]
    s.set_columns(c["pl"], st["Tlayer"], c["Tsurf"], st["vmr9"], st["rel_hum"])
    s.advance(2)

    def step():
        s.advance(1, want_scalars=False)
        s.synchronize()

    calls = {"step": step, "flux_jacobian": lambda: s.lbl_flux_jacobian(),
             "adjusted_forcing": lambda: s.lbl_adjusted_forcing(CO2_2X, NTROP, tol=TOL)}
    for f in calls.values():  # warm-up: modules, scratch allocation
        f()
    times = {k: [] for k in calls}
    for _ in range(a.reps):
        for k, f in calls.items():
            t0 = time.perf_counter()
            f()
            times[k].append(time.perf_counter() - t0)
    d = s.lbl_adjusted_forcing(CO2_2X, NTROP, tol=TOL)
    s.close()
    lines = [f"card: {card}",
             f"workload: {a.ncol} columns x {a.nwvl} wavelengths (bench.py LBL case, co2_factor 1, after 2 steps, then "
             f"{a.reps} alternated reps of each call; the state moves one step per rep)"]
    step_ms = 1e3 * np.median(times["step"])
    for name in calls:
        med = 1e3 * np.median(times[name])
        lines.append(f"{name:17s} median {med:10.2f} ms   min {1e3 * np.min(times[name]):10.2f} ms   {med / step_ms:7.2f} x step")
    it = d["iters"]
    lines.append(f"forcing: 2xCO2, ntrop {NTROP}, tol {TOL:g} W/m2; Newton updates per column: "
                 + ", ".join(f"{k}: {n}" for k, n in enumerate(np.bincount(it[it >= 0]))) + f"; unconverged: {int((it < 0).sum())}")
    lines.append(f"ensemble mean: IRF_toa {d['IRF_toa'].mean():.6f}, IRF_trop {d['IRF_trop'].mean():.6f}, "
                 f"SARF_toa {d['SARF_toa'].mean():.6f}, SARF_trop {d['SARF_trop'].mean():.6f} W/m2")
    lines.append("ensemble-mean dT_adj per layer (K): " + ", ".join(f"{x:.6f}" for x in d["dT_adj"].mean(axis=0)[:NTROP]))
    text = "\n".join(lines)
    print(text)
    if a.out:
        with open(a.out, "w") as f:
            f.write(text + "\n")


if __name__ == "__main__":
    main()
