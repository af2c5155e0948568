"""Cost of the line-by-line radiative-kernel call (rcm_lbl_radiative_kernels) on the bench.py LBL workload: 4,096 columns x
20,000 synthetic wavelengths.  Medians of alternated calls: one LBL step (rcm_advance(1)), the broadband flux call
(rcm_lbl_diagnose_fluxes), the broadband kernels, and the kernels with bands of 100 wavelengths (K_band only).  Also prints
the ensemble-mean dOLR/dT_surf, sum_l dOLR/dT_l and sum_l dOLR/dln q_l, and the card's name and power limit read in the same
run.

    python tools/lbl_kernel_probe.py [--ncol 4096] [--nwvl 20000] [--reps 5]
"""
import argparse
import ctypes
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
    L = rcm.load_library()
    nb = len(bands) - 1
    Kb = np.zeros((a.ncol, nb, 2, 41))
    bs = np.ascontiguousarray(bands, dtype=np.int32)

    def step():
        s.advance(1, want_scalars=False)
        s.synchronize()

    def kernels_bands():  # K_band alone (the Python wrapper always asks for K too)
        p = lambda x: x.ctypes.data_as(ctypes.c_void_p)
        assert L.rcm_lbl_radiative_kernels(s._h, 0, a.ncol, None, nb, p(bs), p(Kb), None) == 0

    calls = {"step": step, "fluxes": lambda: s.lbl_diagnose_fluxes(), "kernels": lambda: s.lbl_radiative_kernels(),
             "kernels_bands100": kernels_bands}
    for f in calls.values():  # warm-up: modules, scratch allocation
        f()
    times = {k: [] for k in calls}
    for _ in range(a.reps):
        for k, f in calls.items():
            t0 = time.perf_counter()
            f()
            times[k].append(time.perf_counter() - t0)
    k = s.lbl_radiative_kernels()
    s.close()
    print(f"card: {card}")
    print(f"workload: {a.ncol} columns x {a.nwvl} wavelengths (bench.py LBL case, co2_factor 1, after 2 steps), {a.reps} alternated reps")
    step_ms = 1e3 * np.median(times["step"])
    for name in calls:
        med = 1e3 * np.median(times[name])
        print(f"{name:17s} median {med:9.2f} ms   min {1e3 * np.min(times[name]):9.2f} ms   {med / step_ms:6.2f} x step")
    print(f"staging {a.nwvl * 82 * 8 / 1e6:.2f} MB per column; {nb} bands")
    print(f"ensemble mean: dOLR/dT_surf {np.mean(k['dOLR_dTs']):.6f} W/m2/K, sum_l dOLR/dT_l {np.mean(k['dOLR_dT'].sum(1)):.6f} "
          f"W/m2/K, sum_l dOLR/dln q_l {np.mean(k['dOLR_dlnq'].sum(1)):.6f} W/m2")


if __name__ == "__main__":
    main()
