"""Cost of the line-by-line diagnostic call (rcm_lbl_diagnose_fluxes) on the bench.py LBL workload: 4,096 columns x 20,000
synthetic wavelengths.  Medians of alternated calls: one LBL step (rcm_advance(1)), the broadband call, and the call with
bands of 100 wavelengths (broadband outputs off).  Also prints the ensemble-mean 2xCO2 instantaneous forcing at TOA and at the
surface of the present-day tables (co2_factor 1), and the card's name and power limit read in the same run.

    python tools/lbl_diag_probe.py [--ncol 4096] [--nwvl 20000] [--reps 5]
"""
import argparse
import os
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import our_first_climate_model_b200 as rcm  # noqa: E402

GOLDEN = os.path.join(ROOT, "tests", "golden")


def lbl_case(ncol, nwvl, seed):  # bench.py's build_lbl_case
    atm = rcm.read_atm(os.path.join(GOLDEN, "column21.lbl.atm"))
    full = rcm.read_atm(os.path.join(GOLDEN, "column21.atm"))
    pl = atm[:, 1].copy()
    Tlev, vlev = rcm.make_ensemble(ncol, seed, pl, atm[:, 2].copy(), full[:, 4:9].T.copy())
    st = rcm.init_columns(pl, Tlev, vlev, 1.0)
    base = rcm.init_columns(pl, atm[None, :, 2].copy(), full[None, :, 4:9].transpose(0, 2, 1).copy(), 1.0)
    h2o_ref, o3_ref = base["vmr9"][0, 0].copy(), base["vmr9"][0, 2].copy()
    wvl, tau5 = rcm.make_lbl_tables(nwvl, 777, pl, h2o_ref, o3_ref)
    return dict(pl=pl, st=st, Tsurf=Tlev[:, 20].copy(), wvl=wvl, tau5=tau5, h2o_ref=h2o_ref, o3_ref=o3_ref)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--ncol", type=int, default=4096)
    ap.add_argument("--nwvl", type=int, default=20000)
    ap.add_argument("--reps", type=int, default=5)
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
    bands = np.append(np.arange(0, a.nwvl, 100), a.nwvl)

    def step():
        s.advance(1, want_scalars=False)
        s.synchronize()

    calls = {"step": step, "broadband": lambda: s.lbl_diagnose_fluxes(),
             "bands100": lambda: s.lbl_diagnose_fluxes(bands=bands)}
    for f in calls.values():  # warm-up: modules, scratch allocation
        f()
    times = {k: [] for k in calls}
    for _ in range(a.reps):
        for k, f in calls.items():
            t0 = time.perf_counter()
            f()
            times[k].append(time.perf_counter() - t0)
    u = s.lbl_diagnose_fluxes()
    v = s.lbl_diagnose_fluxes(vmr_scale=[1, 2, 1, 1, 1])
    irf_toa = float(np.mean(u["E_up"][:, 0] - v["E_up"][:, 0]))
    irf_sfc = float(np.mean((v["E_down"][:, 20] - v["E_up"][:, 20]) - (u["E_down"][:, 20] - u["E_up"][:, 20])))
    s.close()
    print(f"card: {card}")
    print(f"workload: {a.ncol} columns x {a.nwvl} wavelengths (bench.py LBL case, co2_factor 1), {a.reps} alternated reps")
    for k in calls:
        print(f"{k:10s} median {1e3 * np.median(times[k]):9.2f} ms   min {1e3 * np.min(times[k]):9.2f} ms")
    print(f"band pass output: {len(bands) - 1} bands, staging {a.nwvl * 42 * 8 / 1e6:.2f} MB per column")
    print(f"2xCO2 IRF (ensemble mean): TOA {irf_toa:.4f} W/m2, surface {irf_sfc:.4f} W/m2")


if __name__ == "__main__":
    main()
